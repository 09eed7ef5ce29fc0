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
    percentile, then — when they hold the WAIC (``fit(..., waic=True)``) — ``elpd_waic``, ``p_waic``, ``se_elpd_waic``
    and ``waic_n_high_p``, then — when they hold PSIS-LOO (``fit(..., loo=True)``) — ``elpd_loo``, ``p_loo``,
    ``se_elpd_loo`` and ``loo_n_high_k``.  The RTD, model-curve, pointwise WAIC / LOO and Pareto-k arrays stay in
    ``results``."""
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
    if 'elpd_waic' in results:
        cols += ['elpd_waic', 'p_waic', 'se_elpd_waic', 'waic_n_high_p']
        blocks += [results['elpd_waic'][:, None], results['p_waic'][:, None], results['se_elpd_waic'][:, None],
                   results['waic_n_high_p'].astype(np.float64)[:, None]]
    if 'elpd_loo' in results:
        cols += ['elpd_loo', 'p_loo', 'se_elpd_loo', 'loo_n_high_k']
        blocks += [results['elpd_loo'][:, None], results['p_loo'][:, None], results['se_elpd_loo'][:, None],
                   results['loo_n_high_k'].astype(np.float64)[:, None]]
    return cols, np.concatenate(blocks, axis=1)


def compare_waic(res_a, res_b):
    """Spectrum-by-spectrum WAIC comparison of two fits (``fit(..., waic=True)`` results, or ``get_waic`` dicts):
    ``elpd_diff`` = elpd_waic_a - elpd_waic_b (positive: model a is expected to predict the data better) and
    ``se_diff`` = sqrt(N var_j(pointwise_a - pointwise_b, ddof=1)), the standard error of that difference (Vehtari,
    Gelman & Gabry 2017), each of shape (B,) (scalars for single-spectrum dicts).  The comparison is only meaningful for
    two fits of the same ``zn`` / ``zn_err``: the pointwise terms are paired by frequency.  Raises ``ValueError`` when
    the shapes differ."""
    return _compare_elpd(res_a, res_b, 'compare_waic', 'elpd_waic', 'waic_pointwise')


def compare_loo(res_a, res_b):
    """Spectrum-by-spectrum PSIS-LOO comparison of two fits (``fit(..., loo=True)`` results, or ``get_loo`` dicts):
    ``elpd_diff`` = elpd_loo_a - elpd_loo_b (positive: model a is expected to predict the data better) and ``se_diff``
    = sqrt(N var_j(loo_pointwise_a - loo_pointwise_b, ddof=1)), the standard error of that difference (Vehtari, Gelman &
    Gabry 2017), each of shape (B,) (scalars for single-spectrum dicts).  As ``compare_waic``: only meaningful for two
    fits of the same ``zn`` / ``zn_err``; raises ``ValueError`` when the shapes differ.  Check ``pareto_k`` first: a
    frequency with a high k makes its elpd_loo term unreliable."""
    return _compare_elpd(res_a, res_b, 'compare_loo', 'elpd_loo', 'loo_pointwise')


def _compare_elpd(res_a, res_b, name, total, pointwise):
    """elpd difference and its standard error from the per-spectrum totals and the per-frequency pointwise terms."""
    ea, eb = np.asarray(res_a[total], dtype=np.float64), np.asarray(res_b[total], dtype=np.float64)
    pa = np.asarray(res_a[pointwise], dtype=np.float64)
    pb = np.asarray(res_b[pointwise], dtype=np.float64)
    if ea.shape != eb.shape or pa.shape != pb.shape or pa.shape[:-1] != ea.shape:
        raise ValueError(f"{name}: shapes differ ({total} {ea.shape} vs {eb.shape}, "
                         f"{pointwise} {pa.shape} vs {pb.shape})")
    d = pa - pb
    N = d.shape[-1]
    return {'elpd_diff': ea - eb, 'se_diff': np.sqrt(N * np.var(d, axis=-1, ddof=1))}
