"""Inversion base class and the four SIP models — host-side mirror of reference ``models.py``.

Public surface kept identical to the reference (constructors ``models.py:41-42, 195, 243,
283, 321``; ``fit`` ``:84``; ``get_chain`` ``:121``; ``forward``; ``_log_likelihood`` ``:59``;
``_log_prior`` ``:64``; ``_log_probability`` ``:71``; properties ``:139-179``), so a script
written against ``bisip`` runs against ``bisip_b200`` unchanged.  What differs is where the
work happens: ``forward`` / ``_log_*`` call the batched CUDA kernels through the C ABI and
``fit`` runs the whole stretch-move chain on the GPU (``bisip_ensemble_run``) instead of
emcee + NumPy + Cython.  There is no CPU fallback.

Additive keyword arguments (absent from the reference): ``seed`` (Philox key; default is
drawn from NumPy's global generator at ``fit`` time so ``np.random.seed`` still makes runs
repeatable), ``device``, and for ``PolynomialDecomposition`` ``n_tau`` and ``precision``.
"""
import numpy as np

from . import _lib, engine
from . import plotlib as _plotlib
from . import utils as _utils
from .sampler import EnsembleSampler


class Inversion(_plotlib.plotlib, _utils.utils):
    """Abstract base of the SIP inversion models (reference ``models.py:22-179``).

    Args:
        filepath (str): path of the data file (CSV: freq, amp, pha, amp_err, pha_err).
        nwalkers (int): number of ensemble walkers. Defaults to 32.
        nsteps (int): number of MCMC steps. Defaults to 5000.
        headers (int): number of header lines in the file. Defaults to 1.
        ph_units (str): phase units, 'mrad', 'rad' or 'deg'. Defaults to 'mrad'.
        seed (int, optional): Philox key of the on-device sampler.
        device (optional): CUDA device. Defaults to the current one.
    """

    _model_id = None

    def __init__(self, filepath, nwalkers=32, nsteps=5000, headers=1, ph_units='mrad', seed=None,
                 device=None):
        self.filepath = filepath
        self.nwalkers = nwalkers
        self.nsteps = nsteps
        self.headers = headers
        self.ph_units = ph_units
        self.seed = seed
        self.device = device

        self._p0 = None
        self._params = {}
        self.__fitted = False
        self._data = self.load_data(self.filepath, self.headers, self.ph_units)

    # ---------------------------------------------------------------- device plumbing
    def _spec(self, dev):
        """ModelSpec (model constants as device tensors) for the C ABI."""
        return engine.ModelSpec(model=self._model_id, ndim=len(self.params))

    def _theta_batch(self, theta, dev):
        th = np.asarray(theta, dtype=np.float64)
        single = th.ndim == 1
        return _lib.dev_f64(th.reshape(1, -1, th.shape[-1]), dev), single

    def _is_own_forward(self, f):
        return getattr(f, '__self__', None) is self and getattr(f, '__func__', None) is type(self).forward

    def _user_loglike(self, theta, f, x, y, yerr):
        """``_log_likelihood`` for a user-supplied forward callable (reference ``models.py:59-62`` accepts any
        ``f(theta, x) -> (2, N)``): the callable runs where the user wrote it, on the host, once per parameter vector;
        the Gaussian reduction runs on the GPU (``bisip_gauss_loglike``).  There is still no CPU implementation of
        the likelihood or of the built-in models."""
        dev = _lib.require_cuda(self.device)
        th = np.asarray(theta, dtype=np.float64)
        single = th.ndim == 1
        rows = [np.asarray(f(t, x), dtype=np.float64) for t in th.reshape(-1, th.shape[-1])]
        shape = np.shape(y)
        for r in rows:
            if r.shape != shape:
                raise ValueError(f'forward callable returned shape {r.shape}, data has shape {shape}')
        Z = _lib.dev_f64(np.stack(rows).reshape(len(rows), 2, -1), dev)
        ll = engine.gauss_loglike(Z, _lib.dev_const(y, dev).reshape(2, -1),
                                  _lib.dev_const(yerr, dev).reshape(2, -1)).cpu().numpy()
        return float(ll[0]) if single else ll.reshape(th.shape[:-1])

    # ---------------------------------------------------------------- probabilities
    def forward(self, theta, w):
        """Complex resistivity of the model -> float64 (2, N), rows [real; imag]
        (or (n, 2, N) for a (n, ndim) batch of parameter vectors)."""
        dev = _lib.require_cuda(self.device)
        th, single = self._theta_batch(theta, dev)
        Z = engine.forward(self._spec(dev), th, _lib.dev_const(w, dev))[0].cpu().numpy()
        return Z[0] if single else Z

    def _log_probability(self, theta, model, bounds, x, y, yerr):
        """Bayes numerator: strict box prior + Gaussian log-likelihood, fused on the GPU
        (reference ``models.py:71-76``)."""
        if not self._is_own_forward(model):      # user callable: prior on the host, callable on the host, reduction on the GPU
            lp = self._log_prior(theta, bounds)
            if np.ndim(lp) == 0:
                return -np.inf if not np.isfinite(lp) else lp + self._log_likelihood(theta, model, x, y, yerr)
            out = np.full(np.shape(lp), -np.inf)
            ok = np.isfinite(lp)
            if ok.any():
                out[ok] = self._user_loglike(np.asarray(theta, dtype=np.float64)[ok], model, x, y, yerr)
            return out
        dev = _lib.require_cuda(self.device)
        th, single = self._theta_batch(theta, dev)
        lp = engine.log_probability(self._spec(dev), th, _lib.dev_const(x, dev),
                                    _lib.dev_const(y, dev).reshape(1, 2, -1),
                                    _lib.dev_const(yerr, dev).reshape(1, 2, -1),
                                    _lib.dev_const(bounds, dev))[0].cpu().numpy()
        return float(lp[0]) if single else lp

    def _log_likelihood(self, theta, f, x, y, yerr):
        """-0.5*sum((y-f)^2/sigma^2 + 2 ln sigma^2) (reference ``models.py:59-62``)."""
        if not self._is_own_forward(f):
            return self._user_loglike(theta, f, x, y, yerr)
        wide = np.array([[-np.inf] * len(self.params), [np.inf] * len(self.params)])
        return self._log_probability(theta, f, wide, x, y, yerr)

    def _log_prior(self, theta, bounds):
        """0 inside the open box, -inf outside or on its faces (reference ``models.py:64-69``)."""
        theta = np.asarray(theta)
        bounds = np.asarray(bounds)
        inside = np.logical_and((bounds[0] < theta).all(axis=-1), (theta < bounds[1]).all(axis=-1))
        if np.ndim(inside) == 0:
            return 0.0 if inside else -np.inf
        return np.where(inside, 0.0, -np.inf)

    def _check_if_fitted(self):
        if not self.fitted:
            raise AssertionError('Model is not fitted! Fit the model to a '
                                 'dataset before attempting to plot results.')

    # ---------------------------------------------------------------- sampling
    def fit(self, p0=None, pool=None, moves=None):
        """Sample the posterior with the on-device affine-invariant ensemble sampler.

        Args:
            p0 (ndarray): starting positions (nwalkers, ndim); drawn uniformly inside the
                parameter bounds with ``np.random.uniform`` if None (as the reference).
            pool, moves: accepted for signature compatibility (reference ``models.py:84``);
                only ``None`` is meaningful — walkers already run in parallel on the GPU and
                the move is emcee's default ``StretchMove(a=2)``.
        """
        if pool is not None or moves is not None:
            raise NotImplementedError('pool= / moves= have no GPU meaning: the CUDA sampler runs all '
                                      'walkers in parallel with the default stretch move')
        self._p0 = p0
        bounds = self.param_bounds          # read at fit() time: users edit params in between
        self.ndim = bounds.shape[1]
        if self._p0 is None:
            self._p0 = np.random.uniform(*bounds, (self.nwalkers, self.ndim))
        dev = _lib.require_cuda(self.device)
        self._sampler = EnsembleSampler(self.nwalkers, self.ndim, self._spec(dev), self._data['w'],
                                        self._data['zn'], self._data['zn_err'], bounds,
                                        seed=self.seed, device=dev)
        self._sampler.run_mcmc(self._p0, self.nsteps, progress=True)
        self.__fitted = True

    def get_chain(self, **kwargs):
        """MCMC chain of a fitted model.

        Keyword Args:
            discard (int): burn-in steps to drop.
            thin (int): keep every ``thin``-th step.
            flat (bool): False -> (nsteps, nwalkers, ndim); True -> (nsteps*nwalkers, ndim).
        """
        self._check_if_fitted()
        return self._sampler.get_chain(**kwargs)

    # ---------------------------------------------------------------- properties
    @property
    def p0(self):
        """ndarray: starting positions, (nwalkers, ndim)."""
        return self._p0

    @property
    def params(self):
        """dict: parameter name -> [lower, upper]."""
        return self._params

    @params.setter
    def params(self, var):
        self._params = var

    @property
    def sampler(self):
        """EnsembleSampler: emcee-compatible view of the on-device sampler."""
        self._check_if_fitted()
        return self._sampler

    @property
    def data(self):
        """dict: the input data."""
        return self._data

    @property
    def fitted(self):
        """bool: whether ``fit`` has been run."""
        return self.__fitted

    @property
    def param_names(self):
        """list of str: ordered parameter names."""
        return list(self.params.keys())

    @property
    def param_bounds(self):
        """ndarray (2, ndim): ordered lower / upper bounds."""
        return np.array(list(self.params.values())).T


class PolynomialDecomposition(Inversion):
    """Debye / Warburg polynomial decomposition (reference ``models.py:182-229``).

    Args:
        poly_deg (int): polynomial degree of the relaxation-time distribution. Defaults to 5.
        c_exp (float): 1.0 -> Debye, 0.5 -> Warburg. Defaults to 1.0.
        n_tau (int, optional): number of relaxation times; the reference hard-codes ``2*N``.
        precision (str): 'fp64' (two-stage contraction on DMMA tiles, the default), 'fp64-collapsed'
            (FP64, z = (L K) a with L K built once per spectrum: same 1e-12 parity, ~10x fewer flops),
            'tf32' or '3xtf32' (tcgen05 tensor cores, stated tolerance).
    """

    _model_id = _lib.MODEL_DECOMP

    def __init__(self, *args, poly_deg=5, c_exp=1.0, n_tau=None, precision='fp64', **kwargs):
        super().__init__(*args, **kwargs)
        self.c_exp = c_exp
        self.poly_deg = poly_deg
        self.precision = precision

        w = self._data['w']
        lo = np.floor(min(np.log10(1. / w)) - 1)
        hi = np.floor(max(np.log10(1. / w)) + 1)
        self.log_tau = np.linspace(lo, hi, 2 * self._data['N'] if n_tau is None else int(n_tau))
        # public, user-replaceable tables, exactly as the reference builds them (:207-209)
        self.log_taus = np.array([self.log_tau ** i for i in range(self.poly_deg + 1)])
        self.taus = 10 ** self.log_tau

        self.params.update({'r0': [0.9, 1.1]})
        self.params.update({f'a{i}': [-1, 1] for i in range(self.poly_deg + 1)})

    def _spec(self, dev):
        return engine.ModelSpec(model=self._model_id, ndim=1 + self.log_taus.shape[0],
                                taus=_lib.dev_const(self.taus, dev), log_taus=_lib.dev_const(self.log_taus, dev),
                                c_exp=float(self.c_exp), precision=_lib.PRECISIONS[self.precision])

    def forward(self, theta, w):
        """Polynomial-decomposition impedance; theta = [r0, a0, a1, ..., a_poly_deg]
        (ascending powers — the order the reference code uses, ``models.py:228-229``)."""
        return super().forward(theta, w)

    # ---- derived products: what decomposition users read off a fit (reference
    #      docs/tutorials/decomposition.ipynb cells 25-29: get_m / total_m) ------------------------
    def get_rtd(self, chain=None, p=None, **kwargs):
        """Relaxation-time distribution m(tau_l) = sum_i a_i log_tau_l^i over the tau grid.

        With ``p=None`` the RTD of the posterior-mean coefficients, shape ``(n_tau,)`` (the
        tutorial's ``get_m``); with percentiles ``p`` the per-tau percentiles of the RTD over
        the chain, shape ``(len(p), n_tau)`` (``bisip_rtd_stats`` on the uploaded chain, the kernel behind
        ``BatchInversion.fit(..., rtd=True)``; equal to ``np.percentile`` of the RTD of every sample bit for bit).
        ``chain`` / ``discard`` / ``thin`` as in ``get_param_mean``."""
        from .products import relaxation_time_distribution
        if p is None:
            return relaxation_time_distribution(self.get_param_mean(chain=chain, **kwargs)[1:], self.log_taus)
        chain = self.parse_chain(chain, **kwargs)
        dev = _lib.require_cuda(getattr(self, "device", None))
        th = _lib.dev_f64(chain, dev).reshape(1, -1, chain.shape[-1])
        out = engine.rtd_stats(th, _lib.dev_const(self.log_taus, dev), p=p)["pct"][0, :, :-1]    # the last column: total
        res = out.cpu().numpy()
        return res if np.ndim(p) else res[0]

    def get_total_chargeability(self, chain=None, **kwargs):
        """Sum of the RTD of the posterior-mean coefficients over the tau grid (the tutorial's
        ``total_m`` column)."""
        return float(np.sum(self.get_rtd(chain=chain, **kwargs)))


class PeltonColeCole(Inversion):
    """Generalised (multi-mode) Pelton Cole-Cole model (reference ``models.py:232-271``).

    Args:
        n_modes (int): number of Cole-Cole modes. Defaults to 1.
    """

    _model_id = _lib.MODEL_COLECOLE

    def __init__(self, *args, n_modes=1, **kwargs):
        super().__init__(*args, **kwargs)
        self.n_modes = n_modes
        modes = range(1, self.n_modes + 1)
        self.params.update({'r0': [0.9, 1.1]})
        self.params.update({f'm{i}': [0.0, 1.0] for i in modes})
        self.params.update({f'log_tau{i}': [-15, 5] for i in modes})
        self.params.update({f'c{i}': [0.0, 1.0] for i in modes})

    def _spec(self, dev):
        return engine.ModelSpec(model=self._model_id, ndim=1 + 3 * self.n_modes, n_modes=self.n_modes)

    def forward(self, theta, w):
        """Cole-Cole impedance; theta = [r0, m_1..m_K, log_tau_1..K (natural log), c_1..c_K]."""
        return super().forward(theta, w)


ColeCole = PeltonColeCole


class Dias2000(Inversion):
    """Dias (2000) model (reference ``models.py:274-305``); theta = [r0, m, log_tau, eta, delta]."""

    _model_id = _lib.MODEL_DIAS

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.params.update({'r0': [0.9, 1.1],
                            'm': [0, 1],
                            'log_tau': [-20, 0],
                            'eta': [0, 150],
                            'delta': [0, 1]})


class Shin2015(Inversion):
    """Shin (2015) double CPE model (reference ``models.py:308-349``);
    theta = [R1, R2, log_Q1, log_Q2, n1, n2].

    .. warning::
        The reference flags this model as "yielding unexpected results"; it is reproduced
        as is, not corrected.
    """

    _model_id = _lib.MODEL_SHIN

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.params.update({'R1': [0.0, 1.0],
                            'R2': [0.0, 1.0],
                            'log_Q1': [-15, -13],
                            'log_Q2': [-7, -5],
                            'n1': [0, 1],
                            'n2': [0, 1]})
