#!/usr/bin/env python
"""Low-delay conversion (MLPG.stream) with a K = 128 model (synth.make_joint_gmm(128)) at
n_slots in {1, 64, 1024, 8192} and delay in {0, 20, 40}.  Per configuration, after --warmup
pushes, over --pushes pushes:
  * device time per push: CUDA events recorded around each push_device;
  * host wall time per push: pinned host frames in, host frames out, synchronised (p50, p99);
  * frames per second (n_slots / p50 wall time);
and per delay the largest n_slots whose p99 push fits the 5 ms frame period.  Also the accuracy
table of the fixed-lag output against the offline conversion (max and mean |out - offline|) for
a random model (synth.make_joint_gmm(32, seed=3)) and for a 16-mixture
kw.GaussianMixture trained on the synthetic corpus, on the two synthetic utterances 0 and 1.
Reads the card name and power limit in the same run; fails without a GPU.  Prints one JSON line
and writes it to --out when given."""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

FRAME_PERIOD_MS = 5.0


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


class _Model:
    covariance_type = 'full'

    def __init__(self, w, m, c):
        self.weights_, self.means_, self.covariances_ = w, m, c


def time_config(torch, paramgen, pool, n_slots, delay, warmup, pushes):
    """pool: (P, n_slots, 24) pinned host frames, cycled."""
    stream = paramgen.stream(n_slots, delay)
    slots = np.arange(n_slots, dtype=np.int32)
    hout = torch.empty((n_slots, 24), dtype=torch.float64).pin_memory()
    hidx = torch.empty(n_slots, dtype=torch.int64).pin_memory()
    cur = torch.cuda.current_stream()
    dev_ms, wall_ms = [], []
    for i in range(warmup + pushes):
        frames = pool[i % len(pool)]
        t0 = time.perf_counter()
        x = frames.to('cuda', non_blocking=True)
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(cur)
        out, idx = stream.push_device(slots, x)
        ev1.record(cur)
        hout.copy_(out, non_blocking=True)
        hidx.copy_(idx, non_blocking=True)
        cur.synchronize()
        t1 = time.perf_counter()
        if i >= warmup:
            dev_ms.append(ev0.elapsed_time(ev1))
            wall_ms.append(1e3 * (t1 - t0))
    stream.end(slots)
    dev, wall = np.array(dev_ms), np.array(wall_ms)
    return {'n_slots': n_slots, 'delay': delay,
            'device_ms_per_push_p50': float(np.median(dev)),
            'device_ms_per_push_p99': float(np.percentile(dev, 99)),
            'wall_ms_per_push_p50': float(np.median(wall)),
            'wall_ms_per_push_p99': float(np.percentile(wall, 99)),
            'frames_per_s': float(n_slots / (np.median(wall) * 1e-3))}


def accuracy(kw, model, utts, delays):
    """max / mean |out - offline| over the utterances, out from the device stream."""
    paramgen = kw.MLPG(model)
    offline = paramgen.transform_many([kw_delta(u) for u in utts])
    rows = []
    for delay in delays:
        stream = paramgen.stream(len(utts), delay)
        outs = [[] for _ in utts]
        slots = np.arange(len(utts))
        for t in range(max(len(u) for u in utts)):
            live = [i for i, u in enumerate(utts) if t < len(u)]
            o, idx = stream.push(slots[live], np.stack([utts[i][t] for i in live]))
            for r, i in enumerate(live):
                if idx[r] >= 0:
                    outs[i].append(o[r])
        tails = stream.end(slots)
        errs = [np.abs(np.vstack(o + [tl]) - y) for o, tl, y in zip(outs, tails, offline)]
        rows.append({'delay': delay, 'max_per_utt': [float(e.max()) for e in errs],
                     'mean': float(np.mean(np.concatenate([e.ravel() for e in errs]))),
                     'offline_abs_max': float(max(np.abs(y).max() for y in offline))})
    return rows


def kw_delta(statics):
    from oracle import delta_ref
    return delta_ref.delta_features(statics)


def trained_model(kw, synth):
    pairs = [synth.make_padded_pair(i) for i in range(10)]
    kw.set_pad_silence(lambda f, n: f)   # the synthetic features are already padded
    x = kw.joint_array_from_pairs(pairs, pad_silence=True, pad_len=synth.PAD_LEN)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        return kw.GaussianMixture(n_components=16, max_iter=30, random_state=0).fit(x), len(x)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--warmup', type=int, default=50)
    ap.add_argument('--pushes', type=int, default=300)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('time_convert_stream needs a CUDA device')
    import kwiiyatta_b200 as kw
    from kwiiyatta_b200 import synth
    torch.cuda.set_device(0)
    res = {'card': card(), 'model': 'synth.make_joint_gmm(128): K = 128, dim_half = 72',
           'frame_period_ms': FRAME_PERIOD_MS, 'warmup': args.warmup, 'pushes': args.pushes}
    paramgen = kw.MLPG(_Model(*synth.make_joint_gmm(128)))
    res['precision'] = {0: 'fp64', 1: 'tc'}[paramgen.precision]
    utts = synth.make_source_utterances(16, frames=64, order=24)
    rows = []
    for n_slots in (1, 64, 1024, 8192):
        pool = torch.from_numpy(np.stack([
            np.stack([utts[(s + p) % 16][(p + s) % 64] for s in range(n_slots)])
            for p in range(64)])).pin_memory()
        for delay in (0, 20, 40):
            rows.append(time_config(torch, paramgen, pool, n_slots, delay, args.warmup,
                                    args.pushes))
            print(json.dumps(rows[-1]), file=sys.stderr)
    res['timing'] = rows
    res['max_slots_within_frame_period'] = {
        str(d): max([r['n_slots'] for r in rows
                     if r['delay'] == d and r['wall_ms_per_push_p99'] <= FRAME_PERIOD_MS],
                    default=0)
        for d in (0, 20, 40)}
    corpus = [synth.make_pair(u)[0].mel_cepstrum.data[:, 1:] for u in range(2)]
    delays = (0, 5, 10, 20, 40)
    res['accuracy_random_model'] = accuracy(kw, _Model(*synth.make_joint_gmm(32, seed=3)), corpus,
                                            delays)
    gm, n_frames = trained_model(kw, synth)
    res['trained_model'] = f'kw.GaussianMixture(16, max_iter=30) on {n_frames} joint frames'
    res['accuracy_trained_model'] = accuracy(kw, gm, corpus, delays)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
