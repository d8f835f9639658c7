#!/usr/bin/env python
"""Conversion with and without global variance (GV) on the configs[4] shape: 128 mixtures,
1 200 utterances x 600 frames, bench.py's generator and seeds.  Prints one JSON line:
device-resident time (CUDA events, median of --reps calls after --warmup) and transform_packed
time (host clock around a synchronised call) for no GV, gv_iter = 0 (variance-scaling postfilter)
and gv_iter = 20; the bytes the GV stage must move at least (band rebuild + GV kernel) and the
HBM floor they imply at 7.7 TB/s; the card name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

N_MIX, UTT_FRAMES, HBM_BYTES_PER_S = 128, 600, 7.7e12


def card():
    import torch
    info = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm',
                            '--format=csv,noheader', '-i', '0'], capture_output=True, text=True,
                           timeout=30)
        info['power_limit_and_max_sm_clock'] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info['power_limit_and_max_sm_clock'] = f'unavailable: {e}'
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--utts', type=int, default=1200)
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--precision', default='auto')
    args = ap.parse_args()
    import torch
    import kwiiyatta_b200 as kw
    from kwiiyatta_b200 import synth
    from kwiiyatta_b200.delta import delta_features_device
    from kwiiyatta_b200.mlpg import MLPG
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device')
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    n = args.utts
    w, m, c = synth.make_joint_gmm(N_MIX, seed=0)
    model = type('M', (), dict(weights_=w, means_=m, covariances_=c, covariance_type='full'))
    base = synth.make_source_utterances(8, frames=UTT_FRAMES, seed0=synth.SEED0)
    rng = np.random.default_rng(1000)
    statics = np.concatenate([base[i % 8] + rng.normal(0, 0.02, base[0].shape)
                              for i in range(n)])
    off = torch.arange(0, (n + 1) * UTT_FRAMES, UTT_FRAMES, dtype=torch.int64, device=dev)
    src = delta_features_device(torch.from_numpy(statics).to(dev), off, n)
    plain = MLPG(model, device=dev, precision=args.precision)
    y0 = plain.transform_device(src, off, n, UTT_FRAMES)
    est = kw.estimate_gv((y0, off))
    gv = (1.5 * est.mean, est.var)          # a GV above the over-smoothed output's, as in use
    variants = {'no_gv': plain,
                'gv_iter_0': MLPG(model, device=dev, precision=args.precision, gv=gv, gv_iter=0),
                'gv_iter_20': MLPG(model, device=dev, precision=args.precision, gv=gv,
                                   gv_iter=20)}
    src_pin = src.cpu().pin_memory()
    out_pin = torch.empty((n * UTT_FRAMES, 24), dtype=torch.float64).pin_memory()
    lens = [UTT_FRAMES] * n
    res = {}
    for name, pg in variants.items():
        for _ in range(args.warmup):
            pg.transform_device(src, off, n, UTT_FRAMES)
            pg.transform_packed(src_pin, lens, out=out_pin)
        torch.cuda.synchronize()
        dev_ms, e2e_ms = [], []
        for _ in range(args.reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            pg.transform_device(src, off, n, UTT_FRAMES)
            b.record()
            b.synchronize()
            dev_ms.append(a.elapsed_time(b))
        for _ in range(args.reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pg.transform_packed(src_pin, lens, out=out_pin)
            torch.cuda.synchronize()
            e2e_ms.append((time.perf_counter() - t0) * 1e3)
        res[name] = {'device_ms_median': float(np.median(dev_ms)),
                     'device_ms_min': float(np.min(dev_ms)),
                     'packed_ms_median': float(np.median(e2e_ms))}
    total, sd, dh = n * UTT_FRAMES, 24, 72
    rebuild = 8 * total * (dh + 4 * sd)          # band kernel: E in, four band planes out
    kernel = 8 * total * sd * (4 + 2)            # GV kernel: four planes + y in, y out
    res['gv_stage_bytes_min'] = rebuild + kernel
    res['gv_stage_hbm_floor_ms'] = (rebuild + kernel) / HBM_BYTES_PER_S * 1e3
    res['gv_kernel_hbm_floor_ms'] = kernel / HBM_BYTES_PER_S * 1e3
    res['config'] = {'workload': f'configs[4] shape: {N_MIX} mixtures, {n} x {UTT_FRAMES} '
                                 'frames, bench.py seeds; GV mean 1.5 x that of the plain output',
                     'precision': args.precision, 'reps': args.reps, 'warmup': args.warmup,
                     'card': card()}
    print(json.dumps(res))


if __name__ == '__main__':
    main()
