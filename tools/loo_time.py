#!/usr/bin/env python
"""Cost of fit(..., loo=True) on a C5 shard (developer tool).

One collapsed-FP64 fit_device(keep_chain=True) leaves a C5-shaped kept chain on the device (12,500 spectra x 100 kept
steps x 256 walkers x 6 parameters = 15.4 GB, far past the 126 MB L2, so every pass reads HBM).  On it, psis_loo and
waic are timed with CUDA events after warm-up, alternating, over the whole shard, and the timed PSIS-LOO is checked
against the fit's own keys.  The whole shard through BatchInversion.fit_device is timed without and with loo
(alternating, median of --fit-reps).  Prints and appends one JSON line to --out, with the card name and power limit
read in the same run."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from bisip_b200 import _lib, engine, synthetic
from bisip_b200.batch import BatchInversion

N_FREQ, N_TAU, POLY_DEG, WALKERS, NSTEPS, DISCARD, THIN = 64, 64, 4, 256, 2000, 1000, 10
SEED = 0xB151B


def gpu_info():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unavailable'


def spread(ms):
    ms = np.asarray(ms)
    return {'median': float(np.median(ms)), 'min': float(ms.min()), 'max': float(ms.max())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--spectra', type=int, default=12500)
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--fit-reps', type=int, default=3)
    ap.add_argument('--out', default=os.path.join('profiles', 'r03_loo_time.json'))
    a = ap.parse_args()
    dev = _lib.require_cuda()
    card = gpu_info()
    print('gpu:', card, file=sys.stderr)
    B = a.spectra
    probe = BatchInversion('decomp', synthetic.frequencies(N_FREQ)[1], np.zeros((1, 2, N_FREQ)), np.ones((1, 2, N_FREQ)),
                           poly_deg=POLY_DEG, n_tau=N_TAU, device=dev)

    def cuda_forward(theta, w):
        return engine.forward(probe._spec(), _lib.dev_f64(theta[:, None, :], dev), _lib.dev_f64(w, dev))[:, 0].cpu().numpy()
    syn = synthetic.make('decomp', 0, B, cuda_forward, N=N_FREQ, poly_deg=POLY_DEG, n_tau=N_TAU)
    inv = BatchInversion('decomp', syn['w'], syn['zn'], syn['zn_err'], nwalkers=WALKERS, nsteps=NSTEPS, poly_deg=POLY_DEG,
                         n_tau=N_TAU, precision='fp64-collapsed', seed=SEED, device=dev)
    res = inv.fit_device(discard=DISCARD, thin=THIN, keep_chain=True, loo=True)
    chain = res['chain']
    nk, ndim = chain.shape[1], chain.shape[3]
    flat = chain.reshape(B, nk * WALKERS, ndim)
    spec, w = inv._spec(), _lib.dev_f64(syn['w'], dev)
    y, ye = _lib.dev_f64(syn['zn'], dev), _lib.dev_f64(syn['zn_err'], dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    for _ in range(3):                                            # warm-up of every shape
        lo = engine.psis_loo(spec, flat, w, y, ye)
        engine.waic(spec, flat, w, y, ye)
    torch.cuda.synchronize()
    loo_ms, waic_ms = [], []
    for _ in range(a.reps):
        ev[0].record()
        lo = engine.psis_loo(spec, flat, w, y, ye)
        ev[1].record()
        engine.waic(spec, flat, w, y, ye)
        ev[2].record()
        torch.cuda.synchronize()
        loo_ms.append(ev[0].elapsed_time(ev[1]))
        waic_ms.append(ev[1].elapsed_time(ev[2]))
    same = bool(torch.equal(lo['elpd'], res['elpd_loo']) and torch.equal(lo['p_loo'], res['p_loo'])
                and torch.equal(lo['se'], res['se_elpd_loo']) and torch.equal(lo['n_high_k'], res['loo_n_high_k'])
                and torch.equal(lo['elpd_i'], res['loo_pointwise'])
                and torch.equal(lo['pareto_k'].nan_to_num(), res['pareto_k'].nan_to_num()))
    k = res['pareto_k']
    k_bands = {'k<0.5': int((k < 0.5).sum()), '0.5<=k<=0.7': int(((k >= 0.5) & (k <= 0.7)).sum()),
               'k>0.7': int((k > 0.7).sum()), 'nan': int(k.isnan().sum())}
    n_high = int((res['loo_n_high_k'] > 0).sum())
    del chain, flat, res, lo
    torch.cuda.empty_cache()
    fit_ms = {'plain': [], 'loo': []}
    flags = {'plain': {}, 'loo': {'loo': True}}
    for _ in range(a.fit_reps):
        for key, f in flags.items():
            torch.cuda.synchronize()
            ev[0].record()
            inv.fit_device(discard=DISCARD, thin=THIN, **f)
            ev[1].record()
            torch.cuda.synchronize()
            fit_ms[key].append(ev[0].elapsed_time(ev[1]))
    n = nk * WALKERS
    pairs = B * n * N_FREQ                                        # (sample, frequency) pairs, each evaluated once
    chain_bytes = B * n * ndim * 8
    line = {
        'tool': 'tools/loo_time.py', 'gpu': card, 'torch': torch.__version__,
        'shape': [B, nk, WALKERS, ndim], 'chain_GB': chain_bytes / 1e9, 'reps': a.reps, 'n_freq': N_FREQ,
        'n_tau': N_TAU, 'psis_loo_ms': spread(loo_ms), 'waic_ms': spread(waic_ms),
        'sample_frequency_pairs': pairs, 'column_ctas': B * N_FREQ,
        'us_per_column_cta': float(np.median(loo_ms)) * 1e3 / (B * N_FREQ),
        'pair_evaluations_per_s': pairs / (float(np.median(loo_ms)) / 1e3),
        'fit_device_ms': {key: spread(v) for key, v in fit_ms.items()},
        'pareto_k_bands': k_bands, 'spectra_with_high_k': n_high,
        'timed_results_equal_fit_results': same,
    }
    line['psis_loo_over_waic'] = line['psis_loo_ms']['median'] / line['waic_ms']['median']
    print(json.dumps(line))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'a') as f:
        f.write(json.dumps(line) + '\n')
    sys.exit(0 if same else 1)


if __name__ == '__main__':
    main()
