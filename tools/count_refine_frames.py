"""Near-ties of the tensor-core hard labels on the configs[4] conversion workload.

Builds bench.py's conversion input (1 200 utterances x 600 frames, the K = 128 joint model,
rank 0), computes the tensor-core weighted log-probabilities of the 72-dimensional source
marginal, and counts the frames the label kernel re-checks in FP64: with the runner-up (two
components within 0.05 nat of the best), with the runner-up and the third (three), and over all
components (four or more).  Also times kw_gmm_hard_labels (precision 1, with its re-checks) with
CUDA events.  Prints one JSON line, with the card's name and power limit.

    python tools/count_refine_frames.py
"""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NEAR_TIE = 0.05          # the label kernel's re-check window (gmm_tc.cu estep_tc)


def main():
    import torch

    from kwiiyatta_b200 import _lib, synth
    from kwiiyatta_b200.delta import delta_features_device
    from kwiiyatta_b200.gmm import GaussianMixture
    n_utts, frames = 1200, 600
    w, m, c = synth.make_joint_gmm(128, seed=0)
    base = synth.make_source_utterances(8, frames=frames, seed0=synth.SEED0)
    rng = np.random.default_rng(1000)
    statics = np.concatenate([base[i % 8] + rng.normal(0, 0.02, base[0].shape)
                              for i in range(n_utts)])
    off = torch.arange(0, (n_utts + 1) * frames, frames, dtype=torch.int64, device='cuda')
    src = delta_features_device(torch.from_numpy(statics).cuda(), off, n_utts)
    n, dh = src.shape
    gm = GaussianMixture(n_components=128, precision='tc', reorder_every=0)
    gm._alloc(torch, n, dh, src.device)
    gm.set_parameters(w, m[:, :dh], c[:, :dh, :dh])
    gm._x_src, gm._x_used = src, None
    gm._pack(torch, src)
    gm._estep(torch, src, for_mstep=True)
    top = torch.topk(gm._resp[:, :n], 4, dim=0).values
    near = [int(((top[0] - top[i]) < NEAR_TIE).sum()) for i in (1, 2, 3)]
    labels = torch.empty(n, dtype=torch.int32, device='cuda')
    args = (n, src, 128, dh, gm._means[0], gm._pc, gm._aux, labels, 1, gm._ws, gm._ws_bytes,
            _lib.stream_ptr(torch))
    for _ in range(5):
        _lib.call('kw_gmm_hard_labels', *args)
    reps = 50
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(reps):
        _lib.call('kw_gmm_hard_labels', *args)
    t1.record()
    torch.cuda.synchronize()
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                       capture_output=True, text=True).stdout.strip().splitlines()
    print(json.dumps({'frames': n, 'components': 128, 'dim': dh,
                      'two_within': near[0] - near[1], 'three_within': near[1] - near[2],
                      'four_or_more_within': near[2],
                      'hard_labels_ms': t0.elapsed_time(t1) / reps,
                      'gpu': q[0] if q else torch.cuda.get_device_name()}))


if __name__ == '__main__':
    main()
