#!/usr/bin/env python
"""Cost of fit(..., autocorr=True) on a C5 shard (developer tool).

One collapsed-FP64 fit_device(keep_chain=True) leaves a C5-shaped kept chain on the device (12,500 spectra x 100 kept
steps x 256 walkers x 6 parameters = 15.4 GB, far past the 126 MB L2, so every pass reads HBM).  On it, column_stats
and autocorr_time are timed with CUDA events after warm-up, alternating, and 256 spectra are checked against
sampler.integrated_time_batch.  The end-to-end fit with and without autocorr is timed too (alternating).  Prints and
appends one JSON line to --out, with the card name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from bisip_b200 import _lib, engine, sampler, synthetic
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
    ap.add_argument('--check', type=int, default=256)
    ap.add_argument('--out', default=os.path.join('profiles', 'r03_autocorr_time.json'))
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
    res = inv.fit_device(discard=DISCARD, thin=THIN, keep_chain=True, autocorr=True)
    chain = res['chain']
    nk, ndim = chain.shape[1], chain.shape[3]
    flat = chain.reshape(B, nk * WALKERS, ndim)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    for _ in range(3):                                            # warm-up of both shapes
        engine.column_stats(flat, p=list(PCT), want_mean=True, want_std=True)
        tau = engine.autocorr_time(chain)
    torch.cuda.synchronize()
    stats_ms, acf_ms = [], []
    for _ in range(a.reps):
        ev[0].record()
        engine.column_stats(flat, p=list(PCT), want_mean=True, want_std=True)
        ev[1].record()
        tau = engine.autocorr_time(chain)
        ev[2].record()
        torch.cuda.synchronize()
        stats_ms.append(ev[0].elapsed_time(ev[1]))
        acf_ms.append(ev[1].elapsed_time(ev[2]))
    same_as_fit = bool(torch.equal(THIN * tau, res['autocorr_time']))
    # check against the FFT implementation on evenly spaced spectra, in sub-batches
    idx = np.linspace(0, B - 1, min(a.check, B)).astype(np.int64)
    got = tau[torch.from_numpy(idx).to(dev)].cpu().numpy()
    ref = np.concatenate([sampler.integrated_time_batch(chain[torch.from_numpy(idx[i:i + 32]).to(dev)], c=5).cpu().numpy()
                          for i in range(0, len(idx), 32)])
    noise = np.abs(ref) < 1e-6                                    # window at the last lag: tau is rounding noise
    rel = np.abs(got - ref)[~noise] / np.abs(ref)[~noise]
    t_all = tau.cpu().numpy()
    del chain, flat, res
    torch.cuda.empty_cache()
    fit_ms = {False: [], True: []}
    for _ in range(a.fit_reps):
        for ac in (False, True):
            torch.cuda.synchronize()
            ev[0].record()
            inv.fit_device(discard=DISCARD, thin=THIN, autocorr=ac)
            ev[1].record()
            torch.cuda.synchronize()
            fit_ms[ac].append(ev[0].elapsed_time(ev[1]))
    line = {
        'tool': 'tools/autocorr_time.py', 'gpu': card, 'torch': torch.__version__,
        'shape': [B, nk, WALKERS, ndim], 'chain_GB': B * nk * WALKERS * ndim * 8 / 1e9, 'reps': a.reps,
        'column_stats_ms': spread(stats_ms), 'autocorr_time_ms': spread(acf_ms),
        'autocorr_over_stats': float(np.median(acf_ms) / np.median(stats_ms)),
        'fit_device_ms': {'autocorr_false': spread(fit_ms[False]), 'autocorr_true': spread(fit_ms[True])},
        'tau_kept_steps': {'median': float(np.nanmedian(t_all)), 'max': float(np.nanmax(t_all)),
                           'nan': int(np.isnan(t_all).sum())},
        'check': {'spectra': int(len(idx)), 'max_rel_err_vs_integrated_time_batch': float(rel.max()) if rel.size else None,
                  'last_lag_columns': int(noise.sum()),
                  'max_abs_err_last_lag': float(np.abs(got - ref)[noise].max()) if noise.any() else None,
                  'timed_result_equals_fit_result': same_as_fit},
    }
    print(json.dumps(line))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'a') as f:
        f.write(json.dumps(line) + '\n')
    ok = same_as_fit and (not rel.size or rel.max() <= 1e-10)
    sys.exit(0 if ok else 1)


if __name__ == '__main__':
    main()
