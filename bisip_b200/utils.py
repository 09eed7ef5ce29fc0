"""Chain post-processing and data ingest mixin — host-side mirror of reference ``utils.py``.

Same method names, argument meaning, warnings and errors as the reference
(``utils.py:17-146``); the reductions themselves run on the GPU:

* ``get_param_percentile / mean / std`` -> ``bisip_column_stats`` (exact order statistics
  with NumPy's 'linear' rule, so percentiles are bit-identical to ``np.percentile``)
* ``get_model_percentile`` -> ``bisip_model_percentile``: one CTA per model column evaluates the forward
  model for the whole flat chain into shared memory and selects there (the reference loops ``forward`` in
  Python once per sample, ``utils.py:32-34``); chains longer than ~27,000 samples fall back to one batched
  ``bisip_forward`` + ``bisip_column_stats``.
"""
import warnings

import numpy as np

from . import _lib, engine


class utils(object):

    # ---------------------------------------------------------------- percentiles of the model
    def get_model_percentile(self, p=[2.5, 50, 97.5], chain=None, **kwargs):
        """Percentiles of the forward model over an MCMC chain -> (len(p), 2, N).
        Mirrors reference ``utils.py:17-35``."""
        chain = self.parse_chain(chain, **kwargs)
        dev = _lib.require_cuda(getattr(self, "device", None))
        th = _lib.dev_f64(chain, dev).reshape(1, -1, chain.shape[-1])
        w = _lib.dev_const(self.data['w'], dev)
        out = engine.model_percentile(self._spec(dev), th, w, p)          # fused: forward + select per model column
        if out is None:                                                  # chain longer than a CTA's shared memory
            Z = engine.forward(self._spec(dev), th, w)                   # (1, n, 2, N)
            n, N = Z.shape[1], Z.shape[3]
            out = engine.column_stats(Z.reshape(1, n, 2 * N), p=p)["pct"].reshape(1, -1, 2, N)
        res = out[0].cpu().numpy()
        return res if np.ndim(p) else res[0]

    def get_waic(self, chain=None, **kwargs):
        """WAIC of the fit over an MCMC chain (Watanabe's widely applicable information criterion, as in Vehtari,
        Gelman & Gabry 2017), for comparing models fitted to the same data: a dict of ``elpd_waic``, ``p_waic``,
        ``se_elpd_waic`` (floats), ``waic_pointwise`` (N,) = lppd - p per frequency and ``waic_n_high_p`` (the number
        of frequencies with p > 0.4).  The kernel behind ``BatchInversion.fit(..., waic=True)`` (``engine.waic``), FP64
        for every precision.  ``chain`` / ``discard`` / ``thin`` as in ``get_model_percentile``."""
        chain = self.parse_chain(chain, **kwargs)
        dev = _lib.require_cuda(getattr(self, "device", None))
        th = _lib.dev_f64(chain, dev).reshape(1, -1, chain.shape[-1])
        w = _lib.dev_const(self.data['w'], dev)
        y = _lib.dev_f64(self.data['zn'], dev).reshape(1, 2, -1)
        ye = _lib.dev_f64(self.data['zn_err'], dev).reshape(1, 2, -1)
        r = {k: v[0].cpu().numpy() for k, v in engine.waic(self._spec(dev), th, w, y, ye).items()}
        return {'elpd_waic': float(r['elpd']), 'p_waic': float(r['p_waic']), 'se_elpd_waic': float(r['se']),
                'waic_pointwise': r['lppd'] - r['p'], 'waic_n_high_p': int(r['n_high_p'])}

    def get_loo(self, chain=None, **kwargs):
        """PSIS-LOO of the fit over an MCMC chain: leave-one-out cross-validation by Pareto-smoothed importance sampling
        (Vehtari, Gelman & Gabry 2017; ArviZ's ``psislw`` with r_eff = 1), for comparing models fitted to the same data
        where WAIC is unreliable.  A dict of ``elpd_loo``, ``p_loo``, ``se_elpd_loo`` (floats), ``loo_pointwise`` (N,)
        = elpd_loo per frequency, ``pareto_k`` (N,), the Pareto shape of each frequency's importance ratios (inf for a
        tail of 4 samples or fewer), and ``loo_n_high_k``, the number of frequencies with k > min(1 - 1/log10 S, 0.7).
        The kernel behind ``BatchInversion.fit(..., loo=True)`` (``engine.psis_loo``), FP64 for every precision.
        ``chain`` / ``discard`` / ``thin`` as in ``get_model_percentile``."""
        chain = self.parse_chain(chain, **kwargs)
        dev = _lib.require_cuda(getattr(self, "device", None))
        th = _lib.dev_f64(chain, dev).reshape(1, -1, chain.shape[-1])
        w = _lib.dev_const(self.data['w'], dev)
        y = _lib.dev_f64(self.data['zn'], dev).reshape(1, 2, -1)
        ye = _lib.dev_f64(self.data['zn_err'], dev).reshape(1, 2, -1)
        r = {k: v[0].cpu().numpy() for k, v in engine.psis_loo(self._spec(dev), th, w, y, ye).items()}
        return {'elpd_loo': float(r['elpd']), 'p_loo': float(r['p_loo']), 'se_elpd_loo': float(r['se']),
                'loo_pointwise': r['elpd_i'], 'pareto_k': r['pareto_k'], 'loo_n_high_k': int(r['n_high_k'])}

    # ---------------------------------------------------------------- parameter statistics
    def _chain_stats(self, chain, p=None, mean=False, std=False):
        dev = _lib.require_cuda(getattr(self, "device", None))
        flat = _lib.dev_f64(chain, dev).reshape(1, -1, chain.shape[-1])
        return engine.column_stats(flat, p=p, want_mean=mean, want_std=std)

    def get_param_percentile(self, p=[2.5, 50, 97.5], chain=None, **kwargs):
        """Percentiles of the parameters over a chain -> (len(p), ndim).  Ref ``utils.py:37-53``."""
        chain = self.parse_chain(chain, **kwargs)
        res = self._chain_stats(chain, p=p)["pct"][0].cpu().numpy()
        return res if np.ndim(p) else res[0]

    def get_param_mean(self, chain=None, **kwargs):
        """Mean of the parameters over a chain -> (ndim,).  Ref ``utils.py:55-69``."""
        chain = self.parse_chain(chain, **kwargs)
        return self._chain_stats(chain, mean=True)["mean"][0].cpu().numpy()

    def get_param_std(self, chain=None, **kwargs):
        """Population standard deviation (ddof=0) -> (ndim,).  Ref ``utils.py:71-85``."""
        chain = self.parse_chain(chain, **kwargs)
        return self._chain_stats(chain, std=True)["std"][0].cpu().numpy()

    def save_results(self, path, p=[2.5, 50, 97.5], chain=None, **kwargs):
        """Write the parameter percentiles to a CSV in the layout of the reference quickstart
        (``quickstart.ipynb`` cells 31-34): header = comma-joined ``param_names``, one row per
        percentile.  Returns the (len(p), ndim) table."""
        from .products import save_percentiles_csv
        results = self.get_param_percentile(p=p, chain=chain, **kwargs)
        save_percentiles_csv(path, self.param_names, results)
        return results

    def parse_chain(self, chain, **kwargs):
        """Same contract as reference ``utils.py:87-106``."""
        if chain is None:
            kwargs['flat'] = True
            chain = self.get_chain(**kwargs)
            if 'discard' not in kwargs and 'thin' not in kwargs:
                warnings.warn(('No samples were discarded from the chain.\n'
                               'Pass discard and thin keywords to remove '
                               'burn-in samples and reduce autocorrelation.'),
                              UserWarning)
        else:
            if chain.ndim > 2:
                raise ValueError('Flatten chain by passing flat=True.')
            if 'discard' in kwargs or 'thin' in kwargs:
                raise ValueError('Please pass either a chain obtained with '
                                 'the get_chain() method or pass '
                                 'discard and thin keywords to parse '
                                 'the full chain. Do not pass both.')
        return chain

    # ---------------------------------------------------------------- data ingest
    def load_data(self, filename, headers=1, ph_units='mrad'):
        """Read one SIP spectrum (CSV: freq, amp, pha, amp_err, pha_err) and normalise it.
        Host NumPy code with the reference's arithmetic (``utils.py:108-146``)."""
        return prepare_data(np.loadtxt(f'{filename}', skiprows=headers, delimiter=','), ph_units)

    def print_latex_parameters(self, names, values, uncertainties, decimals=3):
        """Pretty-print parameters with LaTeX in a notebook (reference ``utils.py:148-187``).
        Unlike the reference, models without a symbol table print their plain names."""
        from IPython.display import display, Math
        symbols = {
            'PeltonColeCole': {'\\r0': '\\rho_0', '\\m': 'm_', '\\c': 'c_', '\\log_tau': '\\log\\tau_'},
            'Dias2000': {'\\r0': '\\rho_0', '\\m': 'm', '\\log_tau': '\\log\\tau'},
        }.get(type(self).__name__, {})
        for n, v, u in zip(names, values, uncertainties):
            txt = '\\{0}: {1:.{3}f} \\pm {2:.{3}f}'.format(n, v, u, decimals)
            for old, new in symbols.items():
                txt = txt.replace(old, new)
            display(Math(txt))


def prepare_data(table, ph_units='mrad'):
    """(n, 5) table of [freq, amp, pha, amp_err, pha_err] -> the reference's data dict.

    Keys (reference ``utils.py:121-144``): freq, amp, pha, amp_err, pha_err, Z, Z_err,
    norm_factor, zn, zn_err, N, w.  Error propagation and normalisation follow the
    reference operation by operation so that ``zn`` / ``zn_err`` are bit-identical.
    """
    table = np.asarray(table, dtype=np.float64)
    names = ['freq', 'amp', 'pha', 'amp_err', 'pha_err']
    data = {name: table[:, i] for i, name in enumerate(names)}
    if ph_units == 'mrad':
        data['pha'] = data['pha'] / 1000
        data['pha_err'] = data['pha_err'] / 1000
    if ph_units == 'deg':
        data['pha'] = np.radians(data['pha'])
        data['pha_err'] = np.radians(data['pha_err'])
    amp, pha = data['amp'], data['pha']
    data['Z'] = amp * (np.cos(pha) + 1j * np.sin(pha))
    err_im = np.sqrt(((amp * np.cos(pha) * data['pha_err']) ** 2) + (np.sin(pha) * data['amp_err']) ** 2)
    err_re = np.sqrt(((amp * np.sin(pha) * data['pha_err']) ** 2) + (np.cos(pha) * data['amp_err']) ** 2)
    data['Z_err'] = err_re + 1j * err_im
    data['norm_factor'] = max(abs(data['Z']))
    zn = data['Z'] / data['norm_factor']
    zn_e = data['Z_err'] / data['norm_factor']
    data['zn'] = np.array([zn.real, zn.imag])
    data['zn_err'] = np.array([zn_e.real, zn_e.imag])
    data['N'] = len(data['freq'])
    data['w'] = 2 * np.pi * data['freq']
    return data


def read_tables(filepaths, headers=1):
    """Read many data files of the reference's CSV format (``docs/user/data_format.rst``: freq, amp, pha, amp_err,
    pha_err) -> (B, N, 5) float64 with the values ``np.loadtxt(fp, skiprows=headers, delimiter=',')`` returns for each
    (the reference reads one file per model object, ``utils.py:116-118``).  The bodies are joined and parsed by ONE
    text-to-double pass (the same correctly rounded conversion), ~3.5x faster per file than a ``np.loadtxt`` call each;
    anything irregular (comment lines, files of different length, stray tokens) takes the per-file path, which raises
    NumPy's own errors."""
    bodies, nlines = [], set()
    for fp in filepaths:
        with open(f'{fp}', 'rb') as f:
            for _ in range(headers):
                f.readline()
            body = f.read()
        bodies.append(body)
        nlines.add(sum(1 for line in body.splitlines() if line.strip()))
    tables = None
    if len(nlines) == 1 and not any(b'#' in b for b in bodies):
        n = nlines.pop()
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter('error')      # a token that is not a number: fall back, let np.loadtxt explain
            try:
                flat = np.fromstring(b' '.join(bodies).replace(b',', b' '), dtype=np.float64, sep=' ')
                if n > 0 and flat.size == len(bodies) * n * 5:
                    tables = flat.reshape(len(bodies), n, 5)
            except (DeprecationWarning, ValueError):
                tables = None
    if tables is None:
        per_file = [np.loadtxt(f'{fp}', skiprows=headers, delimiter=',') for fp in filepaths]
        lengths = sorted({t.shape[0] for t in per_file})
        if len(lengths) != 1:
            raise ValueError(f'files with the same number of frequencies are needed, got N in {lengths}; '
                             'group the files by length')
        tables = np.stack(per_file)
    return tables


def prepare_data_batch(tables, ph_units='mrad'):
    """``prepare_data`` for a (B, N, 5) stack of tables in one vectorised pass: the same element-wise operations in the
    same order, so every array equals the per-file result bit for bit.  Returns a dict of arrays with a leading B axis
    (``zn`` / ``zn_err`` are (B, 2, N)); ``norm_factor`` is (B,), ``N`` an int."""
    tables = np.asarray(tables, dtype=np.float64)
    names = ['freq', 'amp', 'pha', 'amp_err', 'pha_err']
    data = {name: tables[:, :, i] for i, name in enumerate(names)}
    if ph_units == 'mrad':
        data['pha'] = data['pha'] / 1000
        data['pha_err'] = data['pha_err'] / 1000
    if ph_units == 'deg':
        data['pha'] = np.radians(data['pha'])
        data['pha_err'] = np.radians(data['pha_err'])
    amp, pha = data['amp'], data['pha']
    data['Z'] = amp * (np.cos(pha) + 1j * np.sin(pha))
    err_im = np.sqrt(((amp * np.cos(pha) * data['pha_err']) ** 2) + (np.sin(pha) * data['amp_err']) ** 2)
    err_re = np.sqrt(((amp * np.sin(pha) * data['pha_err']) ** 2) + (np.cos(pha) * data['amp_err']) ** 2)
    data['Z_err'] = err_re + 1j * err_im
    data['norm_factor'] = np.max(np.abs(data['Z']), axis=1)
    zn = data['Z'] / data['norm_factor'][:, None]
    zn_e = data['Z_err'] / data['norm_factor'][:, None]
    data['zn'] = np.stack([zn.real, zn.imag], axis=1)
    data['zn_err'] = np.stack([zn_e.real, zn_e.imag], axis=1)
    data['N'] = tables.shape[1]
    data['w'] = 2 * np.pi * data['freq']
    return data


class BatchData:
    """Per-file view of ``prepare_data_batch`` output: ``batch_data[i]`` is the reference's data dict of file ``i``
    (``utils.py:121-144``), built on access."""

    def __init__(self, arrays):
        self.arrays = arrays

    def __len__(self):
        return self.arrays['zn'].shape[0]

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(len(self)))]
        if not -len(self) <= i < len(self):
            raise IndexError(i)
        out = {k: v[i] for k, v in self.arrays.items() if k != 'N'}
        out['N'] = self.arrays['N']
        return out

    def __iter__(self):
        return (self[i] for i in range(len(self)))
