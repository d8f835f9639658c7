#!/usr/bin/env python
"""EM iteration time of covariance_type='diagonal_blocks' next to 'full' on the configs[1]
training matrix (the joint frames of bench.py's 503 synthetic pairs, K = 64, D = 144).

Prints one JSON line (and writes it to --out when given):
  * device time per EM iteration (CUDA events around --reps em_iteration_async calls after
    --warmup), for 'diagonal_blocks' (FP64), 'full' at precision 'auto' (what bench.py fits) and
    'full' at FP64;
  * per-kernel device time per iteration of 'diagonal_blocks' from a torch.profiler pass of its
    own, and the achieved FLOP/s of its E-step and statistics kernels from the algorithmic counts
    (7 flop per feature pair and (frame, component) in the E-step, 8 in the statistics);
  * held-out score (mean log-likelihood per frame) of both model types trained on a few
    synthetic utterances (a report, not a gate);
  * the card name and power limit, read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import warnings

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

K = 64


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


def joint_frames(first, n_pairs):
    import kwiiyatta_b200 as kw
    from kwiiyatta_b200 import synth
    padded = [synth.make_padded_pair(i) for i in range(first, first + n_pairs)]
    return kw.joint_array_from_pairs(padded, pad_silence=True, pad_len=synth.PAD_LEN)


def model(kind, precision, **kwargs):
    from kwiiyatta_b200.gmm import GaussianMixture
    return GaussianMixture(n_components=K, covariance_type=kind, precision=precision,
                           random_state=0, **kwargs)


def ms_per_iteration(torch, kind, precision, xd, warmup, reps):
    gm = model(kind, precision)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        x = gm.initialize(xd)
        for _ in range(warmup):
            gm.em_iteration_async(x)
        gm.last_lower_bound()
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        for _ in range(reps):
            gm.em_iteration_async(x)
        stop.record()
        torch.cuda.synchronize()
        lb = gm.last_lower_bound()
    return start.elapsed_time(stop) / reps, lb, gm.precision


def kernel_split(torch, xd, reps):
    from torch.profiler import ProfilerActivity, profile
    gm = model('diagonal_blocks', 'fp64')
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        x = gm.initialize(xd)
        gm.em_iteration(x)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                gm.em_iteration_async(x)
            torch.cuda.synchronize()
    split = {}
    for ev in prof.key_averages():
        us = getattr(ev, 'device_time_total', None)
        if us is None:
            us = ev.cuda_time_total
        if us > 0:
            split[ev.key] = round(us / 1e3 / reps, 5)
    return split


def held_out_scores(train_pairs, test_first, test_pairs, k):
    from kwiiyatta_b200.gmm import GaussianMixture
    x = joint_frames(0, train_pairs)
    y = joint_frames(test_first, test_pairs)
    out = {'train_frames': int(len(x)), 'test_frames': int(len(y)), 'components': k}
    for kind in ('full', 'diagonal_blocks'):
        try:
            with warnings.catch_warnings():
                warnings.simplefilter('ignore')
                gm = GaussianMixture(n_components=k, covariance_type=kind, precision='fp64',
                                     random_state=0).fit(x)
        except ValueError as e:         # e.g. an ill-defined covariance of the full model
            out[kind] = {'error': str(e)}
            continue
        out[kind] = {'train_score': gm.score(x), 'held_out_score': gm.score(y),
                     'n_iter': gm.n_iter_}
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    import kwiiyatta_b200 as kw
    from kwiiyatta_b200 import synth
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device')
    torch.cuda.set_device(0)
    kw.hooks.bind(pad_silence=lambda f, n: f, feature=synth.feature, resample=synth.resample)
    x = joint_frames(0, 503)
    xd = torch.from_numpy(x).cuda()
    n, d = x.shape
    res = {'tool': 'tools/time_gmm_diagblocks.py', 'card': card(),
           'workload': f'configs[1] training matrix: {n} joint frames x {d}, K = {K}',
           'reps': args.reps, 'warmup': args.warmup, 'em_iteration_ms': {}, 'lower_bound': {}}
    for label, kind, precision, reps in (('diagonal_blocks', 'diagonal_blocks', 'fp64',
                                          args.reps),
                                         ('full_auto', 'full', 'auto', args.reps),
                                         ('full_fp64', 'full', 'fp64', max(2, args.reps // 4))):
        ms, lb, used = ms_per_iteration(torch, kind, precision, xd, args.warmup, reps)
        res['em_iteration_ms'][label] = round(ms, 4)
        res['lower_bound'][label] = lb
        res.setdefault('precision_used', {})[label] = used
    split = kernel_split(torch, xd, args.reps)
    res['kernel_ms_per_iteration'] = split
    pairs = n * K * (d // 2)
    flops = {'gmm_db_estep_kernel': 7.0 * pairs, 'gmm_db_mstats_kernel': 8.0 * pairs}
    res['algorithmic_flop'] = flops
    res['achieved_tflops'] = {}
    for name, f in flops.items():
        ms = sum(v for key, v in split.items() if name in key)
        if ms > 0:
            res['achieved_tflops'][name] = round(f / (ms * 1e-3) / 1e12, 3)
    res['full_model_flop_per_iteration'] = 4.0 * n * K * d * d
    res['quality'] = held_out_scores(8, 400, 8, 8)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
