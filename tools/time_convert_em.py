#!/usr/bin/env python
"""EM conversion over all mixture sequences (MLPG(em_iter=)) on the configs[4] shape: 128
mixtures, 1 200 utterances x 600 frames, bench.py's generator and seeds.  Prints one JSON line:
device-resident time (CUDA events, median of --reps calls after --warmup) and transform_packed
time (host clock around a synchronised call) for em_iter in {0, 1, 5, 10} at each precision;
per-stage kernel times of one em_iter = 1 call from torch.profiler (run separately from the timed
calls); the mean number of mixtures active (posterior above 1e-14 for some frame) per 32-frame
tile at the start and after 10 iterations; the objective trace summed over utterances;
max |y_tc - y_fp64|; the card name and power limit read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools.time_convert_gv import N_MIX, UTT_FRAMES, card  # noqa: E402

STAGES = {  # kernel-name substring -> stage (first match wins)
    'convert_em_frames': 'joint_frames', 'colstats': 'joint_frames', 'pack_x': 'joint_frames',
    'gmm_estep': 'estep', 'estep_tc': 'estep', 'pack_l': 'estep', 'lse_kernel': 'estep',
    'reduce_fixed': 'estep', 'convert_em_loglik': 'estep',
    'convert_soft_kernel': 'accumulate',
    'convert_band_kernel': 'band_solve', 'convert_mlpg': 'band_solve',
}


def stage_times(torch, model, precision, src, off, n):
    """Kernel time per stage of the EM iteration, from one profiled em_iter = 1 call minus one
    profiled em_iter = 0 call (which is the hard-sequence start both share)."""
    from torch.profiler import ProfilerActivity, profile

    def kernels(p):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            p.transform_device(src, off, n, UTT_FRAMES)
            torch.cuda.synchronize()
        out = {}
        for e in prof.events():
            if e.device_type.name != 'CUDA':
                continue
            out[e.name] = out.get(e.name, 0.0) + e.device_time / 1e3
        return out
    from kwiiyatta_b200.mlpg import MLPG
    one = kernels(MLPG(model, device=src.device, precision=precision, em_iter=1))
    zero = kernels(MLPG(model, device=src.device, precision=precision))
    res = {}
    for name, ms in one.items():
        ms -= zero.get(name, 0.0)
        stage = next((s for k, s in STAGES.items() if k in name), 'other')
        res[stage] = res.get(stage, 0.0) + ms
    return {k: round(v, 4) for k, v in res.items() if abs(v) > 1e-6}


def active_per_tile(torch, model, src, y, diff=False):
    """Mean number of mixtures with a posterior above 1e-14 in a 32-frame tile (tiles cut at
    multiples of 32 frames of the whole batch, as convert_soft_kernel cuts them)."""
    from oracle import mlpg_em_ref as em
    cond = em.conditional(model.weights_, model.means_, model.covariances_, diff)
    means, pc = em.joint_model(cond)
    dev = src.device
    t = y.shape[0] // UTT_FRAMES
    yy = y.view(t, UTT_FRAMES, -1)
    zero = torch.zeros_like(yy[:, :1])
    ym = torch.cat([zero, yy[:, :-1]], 1)
    yp = torch.cat([yy[:, 1:], zero], 1)
    wy = torch.cat([yy, 0.5 * (yp - ym), ym - 2 * yy + yp], 2).reshape(y.shape[0], -1)
    z = torch.cat([src, wy], 1)
    pc_t = torch.from_numpy(pc).to(dev)
    b = torch.einsum('kd,kde->ke', torch.from_numpy(means).to(dev), pc_t)
    logdet = torch.log(torch.diagonal(pc_t, dim1=1, dim2=2)).sum(1)
    lw = torch.log(torch.from_numpy(model.weights_).to(dev))
    wlp = torch.empty((z.shape[0], len(lw)), dtype=torch.float64, device=dev)
    for k in range(len(lw)):
        q = ((z @ pc_t[k] - b[k]) ** 2).sum(1)
        wlp[:, k] = -0.5 * (z.shape[1] * np.log(2 * np.pi) + q) + logdet[k] + lw[k]
    gamma = torch.softmax(wlp, 1)
    n = gamma.shape[0] // 32 * 32
    act = (gamma[:n].view(-1, 32, gamma.shape[1]) > 1e-14).any(1).sum(1).double()
    return float(act.mean())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--utts', type=int, default=1200)
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=2)
    args = ap.parse_args()
    import torch
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
    src_pin = src.cpu().pin_memory()
    out_pin = torch.empty((n * UTT_FRAMES, 24), dtype=torch.float64).pin_memory()
    lens = [UTT_FRAMES] * n
    res, outs = {}, {}
    for prec in ('fp64', 'tc'):
        for em_iter in (0, 1, 5, 10):
            pg = MLPG(model, device=dev, precision=prec, em_iter=em_iter)
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
            entry = {'device_ms_median': float(np.median(dev_ms)),
                     'device_ms_min': float(np.min(dev_ms)),
                     'packed_ms_median': float(np.median(e2e_ms))}
            if em_iter:
                y, trace = pg.transform_device(src, off, n, UTT_FRAMES, return_em_info=True)
                entry['objective_trace_sum'] = trace.sum(0).cpu().tolist()
                outs[(prec, em_iter)] = y
            else:
                outs[(prec, 0)] = pg.transform_device(src, off, n, UTT_FRAMES)
            res[f'{prec}_em_iter_{em_iter}'] = entry
        res[f'{prec}_stage_ms_per_iteration'] = stage_times(torch, model, prec, src, off, n)
    res['max_abs_y_tc_minus_fp64'] = {
        str(k): float((outs[('tc', k)] - outs[('fp64', k)]).abs().max()) for k in (0, 1, 5, 10)}
    res['max_abs_y_fp64'] = float(outs[('fp64', 10)].abs().max())
    res['active_mixtures_per_32_frame_tile'] = {
        'start': active_per_tile(torch, model, src, outs[('fp64', 0)]),
        'after_10': active_per_tile(torch, model, src, outs[('fp64', 10)])}
    res['config'] = {'workload': f'configs[4] shape: {N_MIX} mixtures, {n} x {UTT_FRAMES} '
                                 'frames, bench.py seeds',
                     'reps': args.reps, 'warmup': args.warmup, 'card': card()}
    print(json.dumps(res))


if __name__ == '__main__':
    main()
