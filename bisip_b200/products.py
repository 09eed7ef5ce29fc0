"""Derived products and result tables — the steps right after the hot path (SURVEY.md §8f-2/3).

* Relaxation-time distribution and total chargeability of a polynomial decomposition
  (reference ``docs/tutorials/decomposition.ipynb`` cells 25-29, the ``get_m`` helper).
* CSV export of parameter percentiles in the layout of the reference's quickstart
  (``docs/tutorials/quickstart.ipynb`` cells 31-34, ``quickstart_results.csv``): one header
  line with the comma-joined parameter names, one row per percentile, ``%.18e`` numbers.

Host-side NumPy on tiny arrays; nothing here is on the sampled path.
"""
import numpy as np


def relaxation_time_distribution(a, log_taus):
    """m[..., l] = sum_i a[..., i] * log_tau_l**i.

    a: (..., poly_deg+1) polynomial coefficients in ascending powers (theta[1:]);
    log_taus: (poly_deg+1, n_tau) power table (``PolynomialDecomposition.log_taus``).
    Accumulates power by power in ascending order like the tutorial's loop."""
    a = np.asarray(a, dtype=np.float64)
    log_taus = np.asarray(log_taus, dtype=np.float64)
    if a.shape[-1] != log_taus.shape[0]:
        raise ValueError(f"expected {log_taus.shape[0]} coefficients, got {a.shape[-1]}")
    m = np.zeros(a.shape[:-1] + (log_taus.shape[1],))
    for i in range(log_taus.shape[0]):
        m = m + a[..., i, None] * log_taus[i]
    return m


def total_chargeability(a, log_taus):
    """Sum of the RTD over the tau grid (the tutorial's ``total_m``)."""
    return relaxation_time_distribution(a, log_taus).sum(-1)


def save_percentiles_csv(path, param_names, results):
    """Write a (n_percentiles, ndim) table exactly like the reference quickstart does:
    ``np.savetxt(path, results, header=','.join(param_names), delimiter=',', comments='')``."""
    results = np.atleast_2d(np.asarray(results, dtype=np.float64))
    if results.shape[1] != len(param_names):
        raise ValueError("results must have one column per parameter")
    np.savetxt(path, results, header=','.join(param_names), delimiter=',', comments='')


def load_percentiles_csv(path):
    """Inverse of ``save_percentiles_csv``: (param_names, (n, ndim) array)."""
    with open(path) as f:
        names = f.readline().strip().split(',')
    return names, np.atleast_2d(np.loadtxt(path, delimiter=',', skiprows=1))


def batch_table(param_names, results, ids=None, percentiles=(2.5, 50, 97.5)):
    """Flatten ``BatchInversion.results`` into (column names, 2-D array): one row per spectrum with
    id, acceptance fraction, flags, then mean / std / each percentile of every parameter, and — when the results hold
    ``autocorr_time`` (``fit(..., autocorr=True)``) — one ``<name>_tau`` column per parameter, then — when they hold the
    total chargeability (``fit(..., rtd=True)``) — ``total_m_mean``, ``total_m_std`` and one ``total_m_p<q>`` per
    percentile.  The RTD and model-curve arrays stay in ``results``."""
    B = results['mean'].shape[0]
    ids = np.arange(B) if ids is None else np.asarray(ids)
    cols = ['spectrum', 'acceptance_fraction', 'flags']
    blocks = [np.asarray(ids, dtype=np.float64)[:, None], results['acceptance_fraction'][:, None],
              results['flags'].astype(np.float64)[:, None]]
    for tag, arr in (('mean', results['mean']), ('std', results['std'])):
        cols += [f'{n}_{tag}' for n in param_names]
        blocks.append(arr)
    for k, q in enumerate(percentiles):
        cols += [f'{n}_p{q:g}' for n in param_names]
        blocks.append(results['percentiles'][:, k])
    if 'autocorr_time' in results:
        cols += [f'{n}_tau' for n in param_names]
        blocks.append(results['autocorr_time'])
    if 'total_chargeability_mean' in results:
        cols += ['total_m_mean', 'total_m_std'] + [f'total_m_p{q:g}' for q in percentiles]
        blocks += [results['total_chargeability_mean'][:, None], results['total_chargeability_std'][:, None],
                   results['total_chargeability_percentiles']]
    return cols, np.concatenate(blocks, axis=1)
