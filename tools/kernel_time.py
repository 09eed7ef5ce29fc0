#!/usr/bin/env python
"""Time one ensemble kernel configuration (developer tool; also the command profiled under ncu).

    python tools/kernel_time.py --model decomp --precision fp64-collapsed --spectra 2368 --walkers 256 --steps 500
    BISIP_B200_LIB=bisip_b200/csrc/libbisip_b200_dbg.so python tools/kernel_time.py ...   # per-phase cycle counters

Synthetic spectra of the benchmark shape (bisip_b200/synthetic.py), kernel alone with CUDA events, best of --reps.
"""
import argparse
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
from bisip_b200 import _lib, engine, synthetic  # noqa: E402
from bisip_b200.batch import BatchInversion  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--model", default="decomp")
ap.add_argument("--precision", default="fp64")
ap.add_argument("--spectra", type=int, default=2368)
ap.add_argument("--walkers", type=int, default=256)
ap.add_argument("--steps", type=int, default=500)
ap.add_argument("--n-freq", type=int, default=64)
ap.add_argument("--n-tau", type=int, default=64)
ap.add_argument("--poly-deg", type=int, default=4)
ap.add_argument("--n-modes", type=int, default=1)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--keep", type=int, default=10, help="thin of the kept chain (discard = steps/2)")
a = ap.parse_args()

dev = _lib.require_cuda()
f, w = synthetic.frequencies(a.n_freq)
kw = dict(poly_deg=a.poly_deg, n_tau=a.n_tau, n_modes=a.n_modes)
probe = BatchInversion(a.model, w, np.zeros((1, 2, a.n_freq)), np.ones((1, 2, a.n_freq)), device=dev, **kw)
fwd = lambda th, ww: engine.forward(probe._spec(), _lib.dev_f64(th[:, None, :], dev), _lib.dev_f64(ww, dev))[:, 0].cpu().numpy()
nsyn = min(a.spectra, 592)
syn = synthetic.make(a.model, 0, nsyn, fwd, N=a.n_freq, poly_deg=a.poly_deg, n_modes=a.n_modes, n_tau=a.n_tau)
reps = -(-a.spectra // nsyn)
zn = np.tile(syn['zn'], (reps, 1, 1))[:a.spectra]
ze = np.tile(syn['zn_err'], (reps, 1, 1))[:a.spectra]
inv = BatchInversion(a.model, w, zn, ze, nwalkers=a.walkers, nsteps=a.steps, precision=a.precision, seed=7, device=dev, **kw)
spec = inv._spec()
p0 = _lib.dev_f64(inv.draw_p0(0, a.spectra), dev)
w_d, y_d, ye_d, b_d = _lib.dev_f64(w, dev), _lib.dev_f64(zn, dev), _lib.dev_f64(ze, dev), _lib.dev_f64(inv.param_bounds, dev)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
import time
best, times = 1e30, []
t_start = time.perf_counter()
rep = 0
while True:       # warm up for >= 0.4 s (module load, clock ramp from idle), then time a.reps launches
    warm = time.perf_counter() - t_start < 0.4
    c = p0.clone()
    e0.record()
    res = engine.ensemble_run(spec, c, w_d, y_d, ye_d, b_d, nsteps=a.steps, seed=7, discard=a.steps // 2, thin=a.keep,
                              store_chain=True, store_logp=False)
    e1.record()
    torch.cuda.synchronize()
    if not warm:
        times.append(e0.elapsed_time(e1))
        rep += 1
        if rep >= a.reps:
            break
best = min(times)
kind = engine.decomp_kernel_kind(spec, a.n_freq, a.walkers) if a.model == 'decomp' else a.model
print(json.dumps({"model": a.model, "precision": a.precision, "kernel": kind, "spectra": a.spectra, "walkers": a.walkers,
                  "steps": a.steps, "n_freq": a.n_freq, "n_tau": a.n_tau, "n_modes": a.n_modes, "ms": best, "ms_median": float(np.median(times)),
                  "evals_per_s": a.spectra * a.walkers * (a.steps + 1) / (best * 1e-3),
                  "acceptance": float(res['accepted'].double().mean().item() / a.steps),
                  "nan_flags": int((res['flags'] != 0).sum().item())}))
