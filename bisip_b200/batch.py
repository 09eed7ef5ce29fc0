"""Survey-scale inversion: many independent spectra, one CTA each, sharded one block per GPU.

The reference handles batches as a serial Python loop over files
(``docs/tutorials/decomposition.ipynb`` cells 9-10: ``for fp in files: model = ...; model.fit()``).
``BatchInversion`` keeps the per-spectrum semantics of ``Inversion.fit`` +
``get_param_percentile / mean / std`` (reference ``models.py:84-119``, ``utils.py:37-85``) but
runs all spectra of a shard in one ``bisip_ensemble_run`` launch and reduces the kept chain to
summaries on the device (``bisip_column_stats``); chains never visit the host unless asked for.

Multi-GPU: spectra are independent, so rank ``r`` of ``G`` owns the contiguous block
``shard_range(B, r, G)`` and no collective runs during sampling.  The Philox counter carries
the *global* spectrum index, so results do not depend on ``G`` or on the sub-batch size.
``fit_sharded`` is the product-level entry point: full arrays in, complete result out on every rank
(``gather_packed``: one NCCL all-gather of the packed summaries; ``gather_chain_to_rank0``: optional chunked gather of
the kept chains).  ``gather`` is the per-tensor variant (NCCL on GPU tensors; gloo on CPU tensors in the unit tests).
"""
import os
from dataclasses import replace

import numpy as np
import torch

from . import _lib, engine

_MODEL_IDS = {'decomp': _lib.MODEL_DECOMP, 'colecole': _lib.MODEL_COLECOLE, 'dias': _lib.MODEL_DIAS,
              'shin': _lib.MODEL_SHIN}


def default_bounds(model, poly_deg=5, n_modes=1):
    """Default parameter boxes of the reference models (``models.py:212-213, 249-252, 287-291,
    325-331``) as ((names), (2, ndim) array)."""
    if model == 'decomp':
        names = ['r0'] + [f'a{i}' for i in range(poly_deg + 1)]
        box = [[0.9, 1.1]] + [[-1, 1]] * (poly_deg + 1)
    elif model == 'colecole':
        names = (['r0'] + [f'm{i+1}' for i in range(n_modes)] + [f'log_tau{i+1}' for i in range(n_modes)]
                 + [f'c{i+1}' for i in range(n_modes)])
        box = [[0.9, 1.1]] + [[0.0, 1.0]] * n_modes + [[-15, 5]] * n_modes + [[0.0, 1.0]] * n_modes
    elif model == 'dias':
        names = ['r0', 'm', 'log_tau', 'eta', 'delta']
        box = [[0.9, 1.1], [0, 1], [-20, 0], [0, 150], [0, 1]]
    elif model == 'shin':
        names = ['R1', 'R2', 'log_Q1', 'log_Q2', 'n1', 'n2']
        box = [[0.0, 1.0], [0.0, 1.0], [-15, -13], [-7, -5], [0, 1], [0, 1]]
    else:
        raise ValueError(f'unknown model {model!r}')
    return names, np.array(box, dtype=np.float64).T


def tau_grid(w, n_tau=None, poly_deg=5):
    """Relaxation-time grid and power table of PolynomialDecomposition (reference ``models.py:201-209``) for one
    frequency vector (N,) or a stack of them (B, N), vectorised over the stack with the same element-wise arithmetic (the
    rows equal the one-vector results bit for bit): (log_tau (..., S), taus (..., S), log_taus (..., poly_deg+1, S))."""
    w = np.asarray(w, dtype=np.float64)
    lw = np.log10(1. / w)
    lo = np.floor(lw.min(axis=-1) - 1)
    hi = np.floor(lw.max(axis=-1) + 1)
    log_tau = np.linspace(lo, hi, 2 * w.shape[-1] if n_tau is None else int(n_tau), axis=-1)
    log_taus = np.stack([log_tau ** i for i in range(poly_deg + 1)], axis=-2)
    return log_tau, 10 ** log_tau, log_taus


def shard_range(n, rank, world):
    """Contiguous block of spectrum indices owned by ``rank``: [lo, hi)."""
    per = -(-n // world)
    lo = min(n, rank * per)
    return lo, min(n, lo + per)


def gather(local, n_total, rank, world, group=None):
    """All-gather per-spectrum result tensors (dict name -> tensor with leading dim = local
    shard size) into full-length tensors ordered by global spectrum index."""
    import torch.distributed as dist
    per = -(-n_total // world)
    out = {}
    for key in sorted(local):
        t = local[key]
        pad = torch.zeros((per,) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        pad[:t.shape[0]] = t
        parts = [torch.empty_like(pad) for _ in range(world)]
        dist.all_gather(parts, pad, group=group)
        out[key] = torch.cat(parts, 0)[:n_total]
    return out


def gather_packed(local, n_total, rank, world, group=None):
    """``gather`` with ONE collective: every per-spectrum tensor is flattened to float64 columns of one
    (per, width) buffer, all-gathered once, and split again (int tensors are exact in float64 up to 2^53)."""
    import torch.distributed as dist
    per = -(-n_total // world)
    keys = sorted(local)
    first = local[keys[0]]
    n_loc = first.shape[0]
    # explicit widths: a rank whose shard is empty (fewer spectra than ranks) still takes part in the collective
    cols = [local[k].reshape(n_loc, int(np.prod(local[k].shape[1:], dtype=np.int64))).to(torch.float64) for k in keys]
    widths = [c.shape[1] for c in cols]
    pad = torch.zeros((per, sum(widths)), dtype=torch.float64, device=first.device)
    pad[:n_loc] = torch.cat(cols, 1)
    full = torch.empty((world * per, sum(widths)), dtype=torch.float64, device=first.device)
    dist.all_gather_into_tensor(full, pad, group=group)
    out, c0 = {}, 0
    for k, wd in zip(keys, widths):
        t = full[:n_total, c0:c0 + wd].reshape((n_total,) + tuple(local[k].shape[1:]))
        out[k] = t.to(local[k].dtype)
        c0 += wd
    return out


def gather_chain_to_rank0(chain, n_total, rank, world, group=None, chunk_bytes=1 << 28):
    """Chunked gather of per-spectrum chains (n_local, ...) to rank 0: at most ``chunk_bytes`` per rank in flight,
    so a survey's (thinned) chains never need a second device-resident copy.  Returns the (n_total, ...) host array
    on rank 0 and None elsewhere.  Every rank makes the same number of collective calls."""
    import torch.distributed as dist
    per = -(-n_total // world)
    item = int(np.prod(chain.shape[1:])) * chain.element_size()
    step = max(1, int(chunk_bytes // max(1, item)))
    out = np.empty((n_total,) + tuple(chain.shape[1:]), dtype=np.float64) if rank == 0 else None
    for c0 in range(0, per, step):
        c1 = min(per, c0 + step)
        buf = torch.zeros((c1 - c0,) + tuple(chain.shape[1:]), dtype=chain.dtype, device=chain.device)
        k = max(0, min(chain.shape[0], c1) - c0)
        if k > 0:
            buf[:k] = chain[c0:c0 + k]
        parts = [torch.empty_like(buf) for _ in range(world)] if rank == 0 else None
        dist.gather(buf, parts, dst=0, group=group)
        if rank == 0:
            for r in range(world):
                g0 = r * per + c0
                kk = max(0, min(n_total, r * per + c1) - g0)
                if kk > 0:
                    out[g0:g0 + kk] = parts[r][:kk].cpu().numpy()
    return out


def fit_sharded(model, w, zn, zn_err, discard=0, thin=1, percentiles=(2.5, 50, 97.5), p0=None, gather_chain=False,
                group=None, batch_size=None, autocorr=False, rtd=False, model_curves=False, **kwargs):
    """Invert a whole survey on all ranks of the current ``torch.distributed`` job (one process per GPU).

    The reference inverts a batch as a serial loop over files (``docs/tutorials/decomposition.ipynb`` cells 9-10);
    here every rank takes the FULL arrays (``w`` (N,) or (B, N); ``zn``, ``zn_err`` (B, 2, N); optional ``p0``
    (B, W, ndim)), inverts its contiguous block ``shard_range(B, rank, world)`` with ``BatchInversion`` (Philox
    counters carry the global spectrum index: the result does not depend on the number of ranks), and the
    per-spectrum summaries are all-gathered with one NCCL collective, so every rank returns the complete result:
    ``percentiles`` (B, len(p), ndim), ``mean``, ``std`` (B, ndim), ``acceptance_fraction``, ``flags`` (B,), with
    ``autocorr=True`` ``autocorr_time`` (B, ndim), and with ``rtd=True`` / ``model_curves=True`` the RTD,
    total-chargeability and model-curve keys (see ``BatchInversion.fit``).  With ``gather_chain=True`` the kept
    chains (``discard`` / ``thin``) are gathered to rank 0 in chunks (``chain`` (B, n_keep, W, ndim) on rank 0, None
    elsewhere).  Without an initialised process group it runs the
    whole survey on the current device.  ``kwargs`` go to ``BatchInversion`` (nwalkers, nsteps, poly_deg, ...)."""
    import torch.distributed as dist
    on = dist.is_available() and dist.is_initialized()
    rank = dist.get_rank(group) if on else 0
    world = dist.get_world_size(group) if on else 1
    B = int(zn.shape[0])
    lo, hi = shard_range(B, rank, world)
    w_arr = np.asarray(w, dtype=np.float64)
    inv = BatchInversion(model, w_arr if w_arr.ndim == 1 else w_arr[lo:hi], zn[lo:hi], zn_err[lo:hi],
                         spectrum_offset=lo + int(kwargs.pop('spectrum_offset', 0)), **kwargs)
    # the optional products are passed only when set, so fit_device overrides written for the older signature keep working
    extra = {k: True for k, on in (('autocorr', autocorr), ('rtd', rtd), ('model_curves', model_curves)) if on}
    dev_res = inv.fit_device(None if p0 is None else p0[lo:hi], discard, thin, percentiles, gather_chain, batch_size,
                             **extra)
    chain = dev_res.pop('chain', None)
    dev_res.pop('log_prob', None)
    if on and world > 1:
        full = gather_packed(dev_res, B, rank, world, group)
        chain_all = gather_chain_to_rank0(chain, B, rank, world, group) if gather_chain else None
    else:
        full = dev_res
        chain_all = chain.cpu().numpy() if gather_chain else None
    out = {k: v.cpu().numpy() for k, v in full.items()}
    if gather_chain:
        out['chain'] = chain_all
    out['shard'] = (lo, hi)
    inv.results, inv.percentiles = out, tuple(float(q) for q in percentiles)
    out['inversion'] = inv
    inv._apply_nan_policy(out['flags'])         # on the complete result: every rank warns / raises alike
    return out


class BatchInversion:
    """Invert ``B`` spectra that share a model (and its bounds) on one GPU.

    Args:
        model (str): 'decomp' (PolynomialDecomposition), 'colecole', 'dias' or 'shin'.
        w: angular frequencies, (N,) shared by all spectra or (B, N).
        zn, zn_err: normalised data and errors, (B, 2, N), rows [real; imag]
            (the ``data['zn']`` / ``data['zn_err']`` arrays of the reference, ``utils.py:141-142``).
        nwalkers, nsteps: as ``Inversion``.
        bounds: optional (2, ndim) override of the default parameter boxes.
        poly_deg, c_exp, n_tau, precision: PolynomialDecomposition options.
        n_modes: Cole-Cole modes.
        seed: Philox key.  spectrum_offset: global index of the first spectrum (for shards).
        nan_policy: what ``fit`` does when a spectrum's log-probability was NaN (``results['flags'] != 0``; emcee
            raises ``ValueError`` for a single spectrum): 'warn' (default), 'raise' or 'ignore'.
    """

    def __init__(self, model, w, zn, zn_err, nwalkers=32, nsteps=5000, bounds=None, poly_deg=5, c_exp=1.0,
                 n_tau=None, precision='fp64', n_modes=1, seed=0, spectrum_offset=0, a=2.0, device=None,
                 nan_policy='warn'):
        if model not in _MODEL_IDS:
            raise ValueError(f'unknown model {model!r}')
        self.model = model
        self.nwalkers, self.nsteps = int(nwalkers), int(nsteps)
        self.seed, self.spectrum_offset, self.a = int(seed), int(spectrum_offset), float(a)
        if nan_policy not in ('warn', 'raise', 'ignore'):
            raise ValueError("nan_policy must be 'warn', 'raise' or 'ignore'")
        self.nan_policy = nan_policy
        self.device = _lib.require_cuda(device)
        self.param_names, dflt = default_bounds(model, poly_deg, n_modes)
        self.param_bounds = dflt if bounds is None else np.asarray(bounds, dtype=np.float64)
        self.ndim = self.param_bounds.shape[1]
        self.w = np.asarray(w, dtype=np.float64)
        self._zn, self._zn_err = zn, zn_err
        self.n_spectra = int(zn.shape[0])
        self.poly_deg, self.c_exp, self.n_modes, self.precision = poly_deg, c_exp, n_modes, precision
        taus = log_taus = None
        if model == 'decomp':
            self.log_tau, taus, log_taus = tau_grid(self.w, n_tau, poly_deg)
        self.taus, self.log_taus = taus, log_taus
        self.results = None

    # ------------------------------------------------------------------ helpers
    def _spec(self, lo=None, hi=None):
        dev = self.device
        taus = log_taus = None
        if self.taus is not None:
            per_spectrum = self.taus.ndim == 2
            taus = _lib.dev_f64(self.taus[lo:hi] if per_spectrum else self.taus, dev)
            log_taus = _lib.dev_f64(self.log_taus[lo:hi] if per_spectrum else self.log_taus, dev)
        return engine.ModelSpec(model=_MODEL_IDS[self.model], ndim=self.ndim, n_modes=self.n_modes, taus=taus,
                                log_taus=log_taus, c_exp=float(self.c_exp), precision=_lib.PRECISIONS[self.precision])

    def _to_dev(self, a, lo, hi):
        if isinstance(a, torch.Tensor):
            return a[lo:hi].to(self.device, dtype=torch.float64, non_blocking=True).contiguous()
        return _lib.dev_f64(a[lo:hi], self.device)

    P0_BLOCK = 64

    def draw_p0(self, lo, hi):
        """Uniform starting positions inside the bounds, like ``Inversion.fit`` does with
        ``np.random.uniform`` (reference ``models.py:104-106``).  Spectra are drawn in blocks of 64 global indices
        from ``default_rng([seed, block])`` (one generator per block, not per spectrum: a 100,000-spectra survey
        needs 1,563 of them), so the positions of a spectrum depend on its global index only — not on sharding or
        sub-batching."""
        out = np.empty((hi - lo, self.nwalkers, self.ndim))
        lob, hib = self.param_bounds
        g0, g1 = self.spectrum_offset + lo, self.spectrum_offset + hi
        nb = self.P0_BLOCK

        def fill(blk):
            rng = np.random.default_rng([self.seed, blk])
            block = rng.uniform(lob, hib, (nb, self.nwalkers, self.ndim))
            a, b = max(g0, blk * nb), min(g1, (blk + 1) * nb)
            out[a - g0:b - g0] = block[a - blk * nb:b - blk * nb]

        blocks = range(g0 // nb, (g1 + nb - 1) // nb)
        # the blocks are independent generators writing disjoint rows and NumPy fills without the GIL: a shard's draw
        # (154 MB at the C5 shape) is host time in front of the first launch, so it runs on a few threads
        nthreads = min(8, len(blocks) // 4, max(1, (os.cpu_count() or 1) // max(1, int(os.environ.get('LOCAL_WORLD_SIZE', '1')))))
        if nthreads > 1:
            from concurrent.futures import ThreadPoolExecutor
            with ThreadPoolExecutor(nthreads) as ex:
                list(ex.map(fill, blocks))
        else:
            for blk in blocks:
                fill(blk)
        return out

    def _validate(self, p0):
        """The checks ``Inversion.fit`` inherits from emcee, for the whole batch at once."""
        if self.param_bounds.shape != (2, self.ndim) or len(self.param_names) != self.ndim:
            raise ValueError(f'bounds must be (2, {len(self.param_names)}) for model {self.model!r}, got {self.param_bounds.shape}')
        if self.nwalkers < 2 * self.ndim:
            raise RuntimeError("It is unadvisable to use a red-blue move with fewer walkers than "
                               "twice the number of dimensions.")
        if p0 is not None:
            if tuple(p0.shape) != (self.n_spectra, self.nwalkers, self.ndim):
                raise ValueError("incompatible input dimensions {0}".format(tuple(p0.shape)))

    def max_batch(self, n_keep, keep_chain):
        free, _ = torch.cuda.mem_get_info(self.device)
        # kept chain (+ log-prob when the chain is kept); the statistics read it in place: no workspace
        per = n_keep * self.nwalkers * (self.ndim + (1 if keep_chain else 0)) * 8 + self.nwalkers * self.ndim * 8 * 4 + 4096
        return max(1, min(65535, int(0.7 * free // per)))

    # ------------------------------------------------------------------ fit
    def fit(self, p0=None, discard=0, thin=1, percentiles=(2.5, 50, 97.5), keep_chain=False, batch_size=None,
            autocorr=False, rtd=False, model_curves=False):
        """Sample every spectrum and summarise the kept chain on the device.

        Returns (and stores in ``self.results``) a dict of host arrays:
        ``percentiles`` (B, len(p), ndim), ``mean`` (B, ndim), ``std`` (B, ndim),
        ``acceptance_fraction`` (B,), ``flags`` (B,), and with ``keep_chain`` the kept
        ``chain`` (B, n_keep, W, ndim) and ``log_prob`` (B, n_keep, W).
        With ``autocorr=True`` also ``autocorr_time`` (B, ndim): emcee's integrated autocorrelation time of every
        parameter in steps (``sampler.get_autocorr_time(discard=, thin=, quiet=True)`` of each spectrum), computed on
        the device from each sub-batch's kept chain before it is dropped; NaN where a walker's kept series is constant.
        With ``rtd=True`` (``'decomp'`` only) the relaxation-time distribution m_l = sum_i a_i log_tau_l^i and the total
        chargeability sum_l m_l of every kept sample are summarised like the parameters: ``rtd_percentiles``
        (B, len(p), n_tau), ``rtd_mean``, ``rtd_std`` (B, n_tau), ``total_chargeability_percentiles`` (B, len(p)),
        ``total_chargeability_mean``, ``total_chargeability_std`` (B,).  The RTD percentiles equal ``np.percentile`` of
        ``products.relaxation_time_distribution`` over the flat chain bit for bit.
        With ``model_curves=True`` also ``model_percentiles`` (B, len(p), 2, N): the percentiles of the forward model
        over the flat chain in normalised units, as ``get_model_percentile`` (FP64 for every ``precision``).
        Both are computed on the device from each sub-batch's kept chain before it is dropped.
        """
        dev_res = self.fit_device(p0, discard, thin, percentiles, keep_chain, batch_size, _chain_to_host=True,
                                  autocorr=autocorr, rtd=rtd, model_curves=model_curves)
        self.percentiles = tuple(float(q) for q in percentiles)
        self.results = {k: (v if isinstance(v, np.ndarray) else v.cpu().numpy()) for k, v in dev_res.items()}
        self._apply_nan_policy(self.results['flags'])
        return self.results

    def _apply_nan_policy(self, flags):
        bad = int(np.count_nonzero(flags))
        if bad and self.nan_policy != 'ignore':
            msg = (f"Probability function returned NaN for {bad} of {len(flags)} spectra "
                   "(results['flags'] != 0; emcee raises ValueError for a single spectrum)")
            if self.nan_policy == 'raise':
                raise ValueError(msg)
            import warnings
            warnings.warn(msg, RuntimeWarning)

    def fit_gathered(self, n_total, p0=None, discard=0, thin=1, percentiles=(2.5, 50, 97.5), group=None, batch_size=None,
                     autocorr=False, rtd=False, model_curves=False):
        """``fit`` for a shard-local inversion inside a ``torch.distributed`` job: this object holds spectra
        ``[spectrum_offset, spectrum_offset + n_spectra)`` of a survey of ``n_total`` sharded by ``shard_range``; after
        sampling, the summaries of all ranks are all-gathered (one NCCL collective) and the COMPLETE result
        (``n_total`` rows, host arrays) is returned on every rank.  Without a process group it equals ``fit``."""
        import torch.distributed as dist
        dev_res = self.fit_device(p0, discard, thin, percentiles, False, batch_size, autocorr=autocorr, rtd=rtd,
                                  model_curves=model_curves)
        if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
            dev_res = gather_packed(dev_res, int(n_total), dist.get_rank(group), dist.get_world_size(group), group)
        self.percentiles = tuple(float(q) for q in percentiles)
        self.results = {k: v.cpu().numpy() for k, v in dev_res.items()}
        self._apply_nan_policy(self.results['flags'])
        return self.results

    def fit_device(self, p0=None, discard=0, thin=1, percentiles=(2.5, 50, 97.5), keep_chain=False,
                   batch_size=None, _chain_to_host=False, autocorr=False, rtd=False, model_curves=False):
        """Same as ``fit`` but leaves the summaries on the GPU (for the NCCL gather).  With ``keep_chain`` the kept
        chains of all sub-batches stay on the device too (``fit`` moves each sub-batch's chain to the host instead)."""
        if rtd and self.model != 'decomp':
            raise ValueError("rtd=True is defined for the polynomial decomposition ('decomp') only")
        B, W, ndim = self.n_spectra, self.nwalkers, self.ndim
        nk = engine.n_keep(self.nsteps, discard, thin)
        if nk == 0:
            raise ValueError('discard/thin leave no samples')
        self._validate(p0)
        if B == 0:                              # an empty shard (fewer spectra than ranks): nothing to launch
            f64 = dict(dtype=torch.float64, device=self.device)
            out = {'percentiles': torch.empty((0, len(percentiles), ndim), **f64), 'mean': torch.empty((0, ndim), **f64),
                   'std': torch.empty((0, ndim), **f64), 'acceptance_fraction': torch.empty((0,), **f64),
                   'flags': torch.empty((0,), dtype=torch.int32, device=self.device)}
            if autocorr:
                out['autocorr_time'] = torch.empty((0, ndim), **f64)
            P = len(percentiles)
            if rtd:
                S = self.log_taus.shape[-1]
                out.update(rtd_percentiles=torch.empty((0, P, S), **f64), rtd_mean=torch.empty((0, S), **f64),
                           rtd_std=torch.empty((0, S), **f64), total_chargeability_percentiles=torch.empty((0, P), **f64),
                           total_chargeability_mean=torch.empty((0,), **f64),
                           total_chargeability_std=torch.empty((0,), **f64))
            if model_curves:
                out['model_percentiles'] = torch.empty((0, P, 2, self.w.shape[-1]), **f64)
            if keep_chain:
                out['chain'], out['log_prob'] = torch.empty((0, nk, W, ndim), **f64), torch.empty((0, nk, W), **f64)
                if _chain_to_host:
                    out['chain'], out['log_prob'] = out['chain'].numpy(force=True), out['log_prob'].numpy(force=True)
            return out
        bs = int(batch_size) if batch_size else self.max_batch(nk, keep_chain)
        bounds = _lib.dev_f64(self.param_bounds, self.device)
        shared_w = self.w.ndim == 1
        w_all = _lib.dev_f64(self.w, self.device) if shared_w else None
        acc = {k: [] for k in ('percentiles', 'mean', 'std', 'acceptance_fraction', 'flags')}
        if autocorr:
            acc['autocorr_time'] = []
        if rtd:
            for k in ('rtd_percentiles', 'rtd_mean', 'rtd_std', 'total_chargeability_percentiles',
                      'total_chargeability_mean', 'total_chargeability_std'):
                acc[k] = []
        if model_curves:
            acc['model_percentiles'] = []
        if keep_chain:
            acc['chain'], acc['log_prob'] = [], []
        for lo in range(0, B, bs):
            hi = min(B, lo + bs)
            y = self._to_dev(self._zn, lo, hi)
            ye = self._to_dev(self._zn_err, lo, hi)
            w = w_all if shared_w else _lib.dev_f64(self.w[lo:hi], self.device)
            if p0 is not None:
                coords = self._to_dev(p0, lo, hi).clone()
                # emcee's finiteness check, on the device copy (a host pass over a C5 shard's 154 MB costs more than the
                # upload) and before this sub-batch is sampled
                if not bool(torch.isfinite(coords).all()):
                    raise ValueError("At least one parameter value was infinite or NaN")
            else:
                coords = _lib.dev_f64(self.draw_p0(lo, hi), self.device)
            spec = self._spec(lo, hi)
            res = engine.ensemble_run(spec, coords, w, y, ye, bounds, nsteps=self.nsteps, seed=self.seed,
                                      spectrum0=self.spectrum_offset + lo, a=self.a, discard=discard, thin=thin,
                                      store_chain=True, store_logp=keep_chain)
            flat = res['chain'].reshape(hi - lo, nk * W, ndim)
            st = engine.column_stats(flat, p=list(percentiles), want_mean=True, want_std=True)
            acc['percentiles'].append(st['pct'])
            acc['mean'].append(st['mean'])
            acc['std'].append(st['std'])
            if autocorr:                           # emcee's default c = 5; in steps of the run
                acc['autocorr_time'].append(thin * engine.autocorr_time(res['chain'], 5.0))
            if rtd:                                # column n_tau of rtd_stats is the total chargeability
                S = spec.log_taus.shape[-1]
                rs = engine.rtd_stats(flat, spec.log_taus, p=list(percentiles), want_mean=True, want_std=True)
                acc['rtd_percentiles'].append(rs['pct'][:, :, :S])
                acc['rtd_mean'].append(rs['mean'][:, :S])
                acc['rtd_std'].append(rs['std'][:, :S])
                acc['total_chargeability_percentiles'].append(rs['pct'][:, :, S])
                acc['total_chargeability_mean'].append(rs['mean'][:, S])
                acc['total_chargeability_std'].append(rs['std'][:, S])
            if model_curves:
                acc['model_percentiles'].append(self._model_curves(spec, flat, w, percentiles))
            acc['acceptance_fraction'].append(res['accepted'].to(torch.float64).mean(1) / float(self.nsteps))
            acc['flags'].append(res['flags'])
            if keep_chain and _chain_to_host:      # sub-batching stays effective: nothing accumulates on the device
                acc['chain'].append(res['chain'].cpu().numpy())
                acc['log_prob'].append(res['log_prob'].cpu().numpy())
            elif keep_chain:
                acc['chain'].append(res['chain'])
                acc['log_prob'].append(res['log_prob'])
        return {k: (np.concatenate(v, 0) if isinstance(v[0], np.ndarray) else torch.cat(v, 0)) for k, v in acc.items()}

    MODEL_CURVE_BYTES = 1 << 30    # (n, 2N) model matrices of one group of the model-curve fallback

    def _model_curves(self, spec, flat, w, percentiles):
        """Percentiles of the forward model over every spectrum's flat chain, (k, len(p), 2, N): fused
        (``engine.model_percentile``), or for chains past one CTA's shared memory ``forward`` + ``column_stats`` on
        groups of spectra whose model matrices fit ``MODEL_CURVE_BYTES``.  FP64 on both paths, as the fused kernel."""
        p = list(percentiles)
        out = engine.model_percentile(spec, flat, w, p)
        if out is not None:
            return out
        if spec.precision not in (_lib.PREC_FP64, _lib.PREC_FP64_COLLAPSED):
            spec = replace(spec, precision=_lib.PREC_FP64)
        k, n, _ = flat.shape
        N = w.shape[-1]
        g = max(1, self.MODEL_CURVE_BYTES // (n * 2 * N * 8))
        parts = []
        for s0 in range(0, k, g):
            s1 = min(k, s0 + g)
            sub = spec if spec.tau_stride() == 0 else replace(spec, taus=spec.taus[s0:s1], log_taus=spec.log_taus[s0:s1])
            Z = engine.forward(sub, flat[s0:s1], w if w.dim() == 1 else w[s0:s1])
            parts.append(engine.column_stats(Z.reshape(s1 - s0, n, 2 * N), p=p)['pct'].reshape(s1 - s0, -1, 2, N))
        return torch.cat(parts, 0)

    # ------------------------------------------------------------------ results
    def rtd(self, stat='mean'):
        """Relaxation-time distribution of every spectrum from the fitted coefficients:
        ``stat`` = 'mean' or an index into the stored percentiles.  Returns (m (B, n_tau), total_m (B,))."""
        from .products import relaxation_time_distribution
        if self.model != 'decomp':
            raise ValueError('rtd() is defined for the polynomial decomposition only')
        if self.results is None:
            raise AssertionError('Model is not fitted! Fit the model to a dataset before attempting to plot results.')
        a = self.results['mean'] if stat == 'mean' else self.results['percentiles'][:, int(stat)]
        lt = self.log_taus
        if lt.ndim == 3 and a.shape[0] != lt.shape[0] and 'shard' in self.results:
            a = a[slice(*self.results['shard'])]      # after fit_sharded with per-spectrum grids: this rank's block
        m = (relaxation_time_distribution(a[:, 1:], lt) if lt.ndim == 2 else
             np.stack([relaxation_time_distribution(a[b, 1:], lt[b]) for b in range(a.shape[0])]))
        return m, m.sum(-1)

    def get_autocorr_time(self, c=5, thin=1):
        """Integrated autocorrelation time of every parameter of every spectrum, (B, ndim), from the kept chain of
        the last ``fit(..., keep_chain=True)`` (emcee's estimator; ``thin`` = the thinning that fit used, so the
        result is in steps).  Evaluated on the GPU in sub-batches by the kernel behind ``fit(..., autocorr=True)``."""
        if self.results is None or 'chain' not in self.results:
            raise AssertionError('get_autocorr_time needs fit(..., keep_chain=True)')
        ch = self.results['chain']
        out = np.empty((ch.shape[0], ch.shape[-1]))
        step = max(1, int(2 ** 27 // max(1, ch[0].size)))            # ~1 GB of float64 per sub-batch
        for lo in range(0, ch.shape[0], step):
            t = torch.from_numpy(ch[lo:lo + step]).to(self.device)
            out[lo:lo + step] = (thin * engine.autocorr_time(t, c)).cpu().numpy()
        return out

    def to_csv(self, path, ids=None):
        """One row per spectrum: id, acceptance, flags, mean/std/percentiles of every parameter."""
        from .products import batch_table
        if self.results is None:
            raise AssertionError('Model is not fitted! Fit the model to a dataset before attempting to plot results.')
        cols, table = batch_table(self.param_names, self.results, ids, self.percentiles)
        np.savetxt(path, table, header=','.join(cols), delimiter=',', comments='')
        return cols

    # ------------------------------------------------------------------ construction from files
    @classmethod
    def from_files(cls, model, filepaths, headers=1, ph_units='mrad', **kwargs):
        """Vectorised ingest of many data files (reference ``utils.py:108-146`` applied to each file: one text-to-double pass
        over all of them, one NumPy pass for the error propagation and the normalisation; ``zn`` / ``zn_err`` equal the
        per-file ``load_data`` result bit for bit).  The files must hold the SAME NUMBER of frequencies (one kernel launch
        has one n_freq); their frequency values may differ (then ``w`` is per spectrum).  Group files of different length
        and build one ``BatchInversion`` per group.  ``inv.data[i]`` is the reference's data dict of file ``i``.  Under
        ``torchrun`` give each rank its block: ``from_files(model, paths[lo:hi], spectrum_offset=lo, ...)`` with
        ``lo, hi = shard_range(len(paths), rank, world)``."""
        from .utils import BatchData, prepare_data_batch, read_tables
        try:
            tables = read_tables(filepaths, headers)
        except ValueError as e:
            if 'same number of frequencies' in str(e):
                raise ValueError('from_files needs ' + str(e)) from None
            raise
        arrays = prepare_data_batch(tables, ph_units)
        ws = arrays['w']
        w = ws[0] if np.all(ws == ws[0]) else ws
        inv = cls(model, w, arrays['zn'], arrays['zn_err'], **kwargs)
        inv.data = BatchData(arrays)
        return inv
