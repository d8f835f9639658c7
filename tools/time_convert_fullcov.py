#!/usr/bin/env python
"""Conversion with the diagonal and the full conditional covariance on the configs[4] shape:
128 mixtures, 1 200 utterances x 600 frames, bench.py's generator and seeds.  Prints one JSON
line (and writes it to --out when given): device-resident time (CUDA events, median of --reps
calls after --warmup) and transform_packed time (host clock around a synchronised call) for
both; the per-stage split of the full path (hard sequence, right-hand side, block solve) from
a torch.profiler pass of its own; max |y_full - y_diag|; the card name and power limit read in
the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

N_MIX, UTT_FRAMES, SD = 128, 600, 24


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


def stage(name):
    """The stage of the full path a kernel belongs to."""
    if 'convert_fullcov_solve_kernel' in name:
        return 'block_solve'
    if 'convert_condmean_kernel' in name:
        return 'rhs'
    return 'hard_sequence'          # E-step (label mode), histogram, scan, scatter, memsets


def stage_split(torch, pg, src, off, n, reps):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            pg.transform_device(src, off, n, UTT_FRAMES)
        torch.cuda.synchronize()
    split = {}
    for ev in prof.key_averages():
        us = getattr(ev, 'device_time_total', None)
        if us is None:
            us = ev.cuda_time_total
        if us <= 0:
            continue
        s = stage(ev.key)
        split[s] = split.get(s, 0.0) + us / 1e3 / reps
    return {k: round(v, 4) for k, v in sorted(split.items())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--utts', type=int, default=1200)
    ap.add_argument('--reps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--precision', default='auto')
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    from kwiiyatta_b200 import _lib, synth
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
    variants = {'diagonal': MLPG(model, device=dev, precision=args.precision),
                'full': MLPG(model, device=dev, precision=args.precision,
                             conditional_covariance='full')}
    src_pin = src.cpu().pin_memory()
    out_pin = torch.empty((n * UTT_FRAMES, SD), dtype=torch.float64).pin_memory()
    lens = [UTT_FRAMES] * n
    res, outs = {}, {}
    for name, pg in variants.items():
        for _ in range(args.warmup):
            pg.transform_device(src, off, n, UTT_FRAMES)
            pg.transform_packed(src_pin, lens, out=out_pin)
        torch.cuda.synchronize()
        dev_ms, e2e_ms = [], []
        for _ in range(args.reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            y = pg.transform_device(src, off, n, UTT_FRAMES)
            b.record()
            b.synchronize()
            dev_ms.append(a.elapsed_time(b))
        outs[name] = y.cpu().numpy()
        for _ in range(args.reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            pg.transform_packed(src_pin, lens, out=out_pin)
            torch.cuda.synchronize()
            e2e_ms.append((time.perf_counter() - t0) * 1e3)
        assert np.array_equal(out_pin.numpy(), outs[name]), f'{name}: packed != device'
        res[name] = {'device_ms_median': float(np.median(dev_ms)),
                     'device_ms_min': float(np.min(dev_ms)),
                     'packed_ms_median': float(np.median(e2e_ms))}
    res['full_stage_ms'] = stage_split(torch, variants['full'], src, off, n, args.reps)
    res['max_abs_full_minus_diagonal'] = float(np.abs(outs['full'] - outs['diagonal']).max())
    res['mean_abs_full_minus_diagonal'] = float(np.abs(outs['full'] - outs['diagonal']).mean())
    total = n * UTT_FRAMES
    res['full_block_solve_flop'] = 9.0e4 * total      # ~9e4 FP64 flop per frame at sd = 24
    res['full_workspace_bytes'] = int(_lib.lib().kw_convert_fullcov_workspace_bytes(
        total, N_MIX, 3 * SD, variants['full'].precision))
    res['config'] = {'workload': f'configs[4] shape: {N_MIX} mixtures, {n} x {UTT_FRAMES} '
                                 'frames, bench.py seeds',
                     'precision': args.precision, 'reps': args.reps, 'warmup': args.warmup,
                     'card': card()}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
