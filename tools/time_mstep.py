#!/usr/bin/env python
"""CUDA-event time of kw_gmm_mstep_accumulate on the dense synthetic workload of prof_stage.py
(every tile carries weight for every component).  KW_CLOCKS=1 also samples the SM clock, the
power draw and the clock-event reasons with nvidia-smi over 1500 calls."""
import os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import kwiiyatta_b200 as kw
dev = torch.device('cuda', 0)
rng = np.random.default_rng(0)
n, d, k = 176323, 144, 64
centres = rng.standard_normal((k, d)) * 0.5
x = centres[rng.integers(0, k, n)] + 0.6 * rng.standard_normal((n, d))
lab = rng.integers(0, k, n)
resp0 = torch.zeros((n, k), dtype=torch.float64, device=dev)
resp0[torch.arange(n, device=dev), torch.from_numpy(lab).to(dev)] = 1.0
kw.GaussianMixture._check_info = lambda self: None          # experiments may produce garbage
kw.GaussianMixture._raise_ill_defined = staticmethod(lambda: None)
gm = kw.GaussianMixture(n_components=k, max_iter=1, tol=0.0, resp_init=resp0, precision='tc', device=dev, reorder_every=0)
xd = gm.initialize(x)
gm.em_iteration(xd)
gm._estep(torch, xd)
cen = gm._means[gm._cur]
for _ in range(2):
    gm._accumulate(torch, xd, cen)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(5):
    gm._accumulate(torch, xd, cen)
e1.record(); e1.synchronize()
print(f'mstep_accumulate {e0.elapsed_time(e1) / 5:.3f} ms (dense)')
if os.environ.get('KW_CLOCKS'):
    import subprocess, threading, time
    samples = []
    stop = threading.Event()
    def poll():
        while not stop.is_set():
            out = subprocess.run(['nvidia-smi', '--id=0', '--query-gpu=clocks.sm,power.draw,clocks_event_reasons.sw_power_cap,clocks_event_reasons.hw_slowdown,clocks_event_reasons.sw_thermal_slowdown', '--format=csv,noheader,nounits'], capture_output=True, text=True).stdout.strip()
            samples.append(out)
            stop.wait(0.05)
    th = threading.Thread(target=poll); th.start()
    e0.record()
    for _ in range(1500):
        gm._accumulate(torch, xd, cen)
    e1.record(); e1.synchronize()
    stop.set(); th.join()
    print(f'1500 calls: {e0.elapsed_time(e1) / 1500:.3f} ms each')
    print('clock samples:', samples[:3], '...', samples[len(samples) // 2], '...', samples[-2:])
