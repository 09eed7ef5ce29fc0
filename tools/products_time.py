#!/usr/bin/env python
"""Cost of fit(..., rtd=True, model_curves=True) on a C5 shard (developer tool).

One collapsed-FP64 fit_device(keep_chain=True) leaves a C5-shaped kept chain on the device (12,500 spectra x 100 kept
steps x 256 walkers x 6 parameters = 15.4 GB, far past the 126 MB L2, so every pass reads HBM).  On it, column_stats,
rtd_stats and model_percentile are timed with CUDA events after warm-up, alternating, over the whole shard, and the
timed results are checked against the fit's own products.  The whole shard through BatchInversion.fit_device is timed
without and with rtd / model_curves (alternating, median of --fit-reps).  Prints and appends one JSON line to --out,
with the card name and power limit read in the same run."""
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
PCT = (2.5, 50, 97.5)
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
    ap.add_argument('--out', default=os.path.join('profiles', 'r03_products_time.json'))
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
    res = inv.fit_device(discard=DISCARD, thin=THIN, keep_chain=True, rtd=True, model_curves=True)
    chain = res['chain']
    nk, ndim = chain.shape[1], chain.shape[3]
    flat = chain.reshape(B, nk * WALKERS, ndim)
    spec, w = inv._spec(), _lib.dev_f64(syn['w'], dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    for _ in range(3):                                            # warm-up of every shape
        engine.column_stats(flat, p=list(PCT), want_mean=True, want_std=True)
        rs = engine.rtd_stats(flat, spec.log_taus, p=list(PCT), want_mean=True, want_std=True)
        mp = engine.model_percentile(spec, flat, w, list(PCT))
    torch.cuda.synchronize()
    stats_ms, rtd_ms, curve_ms = [], [], []
    for _ in range(a.reps):
        ev[0].record()
        engine.column_stats(flat, p=list(PCT), want_mean=True, want_std=True)
        ev[1].record()
        rs = engine.rtd_stats(flat, spec.log_taus, p=list(PCT), want_mean=True, want_std=True)
        ev[2].record()
        mp = engine.model_percentile(spec, flat, w, list(PCT))
        ev[3].record()
        torch.cuda.synchronize()
        stats_ms.append(ev[0].elapsed_time(ev[1]))
        rtd_ms.append(ev[1].elapsed_time(ev[2]))
        curve_ms.append(ev[2].elapsed_time(ev[3]))
    S = N_TAU
    same = bool(torch.equal(rs['pct'][:, :, :S], res['rtd_percentiles']) and torch.equal(rs['mean'][:, S],
                res['total_chargeability_mean']) and torch.equal(mp, res['model_percentiles']))
    del chain, flat, res, rs, mp
    torch.cuda.empty_cache()
    fit_ms = {'plain': [], 'rtd': [], 'rtd_model_curves': []}
    flags = {'plain': {}, 'rtd': {'rtd': True}, 'rtd_model_curves': {'rtd': True, 'model_curves': True}}
    for _ in range(a.fit_reps):
        for k, f in flags.items():
            torch.cuda.synchronize()
            ev[0].record()
            inv.fit_device(discard=DISCARD, thin=THIN, **f)
            ev[1].record()
            torch.cuda.synchronize()
            fit_ms[k].append(ev[0].elapsed_time(ev[1]))
    cols_stats, cols_rtd, cols_curve = B * ndim, B * (N_TAU + 1), B * 2 * N_FREQ
    line = {
        'tool': 'tools/products_time.py', 'gpu': card, 'torch': torch.__version__,
        'shape': [B, nk, WALKERS, ndim], 'chain_GB': B * nk * WALKERS * ndim * 8 / 1e9, 'reps': a.reps,
        'n_tau': N_TAU, 'n_freq': N_FREQ,
        'column_stats_ms': spread(stats_ms), 'rtd_stats_ms': spread(rtd_ms), 'model_percentile_ms': spread(curve_ms),
        'columns': {'column_stats': cols_stats, 'rtd_stats': cols_rtd, 'model_percentile': cols_curve},
        'us_per_column': {'column_stats': 1e3 * float(np.median(stats_ms)) / cols_stats,
                          'rtd_stats': 1e3 * float(np.median(rtd_ms)) / cols_rtd,
                          'model_percentile': 1e3 * float(np.median(curve_ms)) / cols_curve},
        'fit_device_ms': {k: spread(v) for k, v in fit_ms.items()},
        'timed_results_equal_fit_results': same,
    }
    line['rtd_column_over_stats_column'] = line['us_per_column']['rtd_stats'] / line['us_per_column']['column_stats']
    print(json.dumps(line))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'a') as f:
        f.write(json.dumps(line) + '\n')
    sys.exit(0 if same else 1)


if __name__ == '__main__':
    main()
