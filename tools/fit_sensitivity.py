#!/usr/bin/env python
"""The bench's user-level fit (KMeans initialisation on the device, tol = 1e-3, max_iter = 100):
final lower bound per precision -- how far 100 iterations carry rounding-level differences of
the M-step."""
import os, sys, warnings
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import kwiiyatta_b200 as kw
from kwiiyatta_b200 import synth
kw.hooks.bind(pad_silence=lambda f, n: f, feature=synth.feature, resample=synth.resample)
padded = [synth.make_padded_pair(i) for i in range(503)]
x = kw.joint_array_from_pairs(padded, pad_silence=True, pad_len=synth.PAD_LEN)
dev = torch.device('cuda', 0)
for prec in ('tc', 'fp64'):
    conv = kw.B200GMMFeatureConverter(components=64, random_state=0, verbose=0, device=dev,
                                      precision=prec)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        conv._train(x)
    g = conv.gmm
    lbs = np.asarray(g.lower_bounds_)
    print(f'{prec}: n_iter {g.n_iter_} lower bound {g.lower_bound_:.6f}; after 1/10/50 '
          f'iterations {lbs[0]:.6f} {lbs[9]:.6f} {lbs[49]:.6f}; smallest n_k '
          f'{g.weights_.min() * len(x):.1f}')
