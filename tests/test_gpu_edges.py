"""Shape / edge-case sweep of the on-device sampler against the C oracle on the same Philox stream:
odd and minimal walker counts, walkers beyond the CTA size, odd frequency / tau counts, per-spectrum
(ragged-by-content) frequency and tau grids, every polynomial degree and mode count the kernels accept,
discard / thin corner cases, continuation with step0, a stretch scale that is not a power of two, and the
argument errors of the C ABI."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _spectrum(model, N, rng, **kw):
    """A smooth synthetic spectrum from the oracle forward at a central theta, 2 % noise."""
    from bisip_b200.batch import default_bounds, tau_grid
    from oracle import oracle
    w = 2 * np.pi * np.logspace(3.5, -1.5, N)
    _, bounds = default_bounds(model, kw.get('poly_deg', 4), kw.get('n_modes', 1))
    okw = {}
    if model == 'decomp':
        _, taus, log_taus = tau_grid(w, kw.get('n_tau'), kw.get('poly_deg', 4))
        okw = dict(taus=taus, log_taus=log_taus, c_exp=kw.get('c_exp', 1.0))
        th = np.concatenate([[1.0], 0.004 * rng.uniform(0.2, 1.0, bounds.shape[1] - 1) / 6.0 ** np.arange(bounds.shape[1] - 1)])
    else:
        okw = dict(n_modes=kw.get('n_modes', 1))
        th = 0.5 * (bounds[0] + bounds[1]) + 0.1 * (bounds[1] - bounds[0]) * rng.uniform(-1, 1, bounds.shape[1])
    prob0 = oracle.Problem(model, w, np.zeros((2, N)), np.ones((2, N)), bounds, **okw)
    Z = prob0.forward(th)
    sig = 0.02 * np.abs(Z[0] + 1j * Z[1]) * np.ones((2, 1))
    y = Z + sig * rng.standard_normal((2, N))
    nf = np.max(np.abs(y[0] + 1j * y[1]))
    return w, y / nf, sig / nf, bounds, okw


SHAPES = [
    # model, N, W, T, kwargs
    ('dias', 64, 10, 60, {}),                      # minimal ensemble: nwalkers = 2*ndim
    ('dias', 17, 31, 50, {}),                      # odd walkers (halves 16 / 15), odd N
    ('dias', 64, 300, 12, {}),                     # more walkers than threads in a CTA
    ('shin', 33, 130, 25, {}),                     # just above the 128-thread variant
    ('shin', 5, 12, 80, {}),                       # fewer frequencies than lanes per row
    ('colecole', 64, 64, 40, dict(n_modes=3)),
    ('colecole', 20, 52, 30, dict(n_modes=4)),
    ('colecole', 20, 64, 20, dict(n_modes=5)),     # generic (8-mode) kernel
    ('colecole', 12, 100, 15, dict(n_modes=8)),
    ('decomp', 64, 256, 10, dict(poly_deg=0, n_tau=64)),
    ('decomp', 20, 24, 60, dict(poly_deg=7, n_tau=40)),
    ('decomp', 64, 64, 30, dict(poly_deg=3, n_tau=33)),          # odd tau count (zero-padded k chunk)
    ('decomp', 7, 18, 50, dict(poly_deg=2, n_tau=9, c_exp=0.5)), # one k chunk, 2N = 14 columns
    ('decomp', 64, 40, 20, dict(poly_deg=4, n_tau=65)),          # smallest clustered (n_tau > 64) case
    ('decomp', 31, 258, 6, dict(poly_deg=5, n_tau=200, c_exp=0.7)),
    ('colecole', 33, 260, 8, dict(n_modes=1)),     # 1 mode beyond the warp-private kernel's 256 walkers
    ('colecole', 40, 140, 12, dict(n_modes=2)),    # 2 modes, > 128 walkers, > 32 frequencies: 256-thread variant
    ('decomp', 40, 270, 6, dict(poly_deg=3, n_tau=40)),          # 33-48 taus beyond the warp-private kernel's 256 walkers
]


@pytest.mark.parametrize("model,N,W,T,kw", SHAPES, ids=[f"{s[0]}-N{s[1]}-W{s[2]}-{i}" for i, s in enumerate(SHAPES)])
def test_shape_sweep_chain_matches_oracle(model, N, W, T, kw):
    from bisip_b200.batch import BatchInversion
    from oracle import oracle
    rng = np.random.default_rng(N * 1000 + W)
    w, zn, ze, bounds, okw = _spectrum(model, N, rng, **kw)
    inv = BatchInversion(model, w, zn[None], ze[None], nwalkers=W, nsteps=T, seed=99, spectrum_offset=7, **kw)
    p0 = inv.draw_p0(0, 1)
    res = inv.fit(p0=p0, keep_chain=True)
    ref = oracle.Problem(model, w, zn, ze, bounds, **okw).run(p0[0], T, seed=99, spectrum=7)
    assert res['flags'][0] == 0 and not ref['nan']
    np.testing.assert_array_equal(res['chain'][0], ref['chain'])
    fin = np.isfinite(ref['log_prob'])
    assert np.array_equal(fin, np.isfinite(res['log_prob'][0]))
    assert np.max(np.abs(res['log_prob'][0][fin] - ref['log_prob'][fin]) / np.maximum(1, np.abs(ref['log_prob'][fin]))) <= 1e-12
    assert res['acceptance_fraction'][0] == pytest.approx(ref['accepted'].mean() / T, abs=1e-15)


COLLAPSED_SHAPES = [
    # N, W, T, kwargs — every coefficient count the collapsed kernel is templated on (poly_deg 0..7), every work split:
    # one / two proposals per thread, 128- and 256-thread CTAs, fewer rows than a warp, more thread-rows than threads,
    # frequency groups that do not divide N, tau grids of any size (no cluster, no tau limit in this form)
    (64, 256, 10, dict(poly_deg=0, n_tau=64)),
    (20, 24, 60, dict(poly_deg=7, n_tau=40)),
    (64, 64, 30, dict(poly_deg=3, n_tau=33)),
    (7, 18, 50, dict(poly_deg=2, n_tau=9, c_exp=0.5)),
    (64, 40, 20, dict(poly_deg=4, n_tau=65)),
    (31, 258, 6, dict(poly_deg=5, n_tau=200, c_exp=0.7)),
    (37, 128, 20, dict(poly_deg=1, n_tau=50)),
    (64, 129, 12, dict(poly_deg=6, n_tau=128)),
    (5, 14, 40, dict(poly_deg=4, n_tau=12)),
    (64, 1100, 4, dict(poly_deg=4, n_tau=64)),
    (3, 600, 5, dict(poly_deg=2, n_tau=300)),
]


@pytest.mark.parametrize("N,W,T,kw", COLLAPSED_SHAPES, ids=[f"N{s[0]}-W{s[1]}-P{s[3]['poly_deg']}" for s in COLLAPSED_SHAPES])
def test_collapsed_shape_sweep_chain_matches_oracle(N, W, T, kw):
    """precision='fp64-collapsed' (csrc/decomp_collapsed.cuh) over the shape classes of its work split: the chain is
    the oracle's on the same Philox stream and the stored log-probabilities agree to 1e-12."""
    from bisip_b200 import engine
    from bisip_b200.batch import BatchInversion
    from oracle import oracle
    rng = np.random.default_rng(N * 1000 + W)
    w, zn, ze, bounds, okw = _spectrum('decomp', N, rng, **kw)
    inv = BatchInversion('decomp', w, zn[None], ze[None], nwalkers=W, nsteps=T, seed=99, spectrum_offset=7,
                         precision='fp64-collapsed', **kw)
    assert engine.decomp_kernel_kind(inv._spec(), N, W) == 'fp64-collapsed'
    p0 = inv.draw_p0(0, 1)
    res = inv.fit(p0=p0, keep_chain=True)
    ref = oracle.Problem('decomp', w, zn, ze, bounds, **okw).run(p0[0], T, seed=99, spectrum=7)
    assert res['flags'][0] == 0 and not ref['nan']
    np.testing.assert_array_equal(res['chain'][0], ref['chain'])
    fin = np.isfinite(ref['log_prob'])
    assert np.array_equal(fin, np.isfinite(res['log_prob'][0]))
    assert np.max(np.abs(res['log_prob'][0][fin] - ref['log_prob'][fin]) / np.maximum(1, np.abs(ref['log_prob'][fin]))) <= 1e-12
    # forward through the batched kernel on the chain's last ensemble (ragged chunk: W is rarely a multiple of 128)
    th = res['chain'][0][-1]
    Z = engine.forward(inv._spec(), inv._to_dev(th[None], 0, 1), inv._to_dev(w[None], 0, 1)[0]).cpu().numpy()[0]
    Zo = oracle.Problem('decomp', w, zn, ze, bounds, **okw).forward(th)
    assert (np.max(np.abs(Z - Zo), axis=(1, 2)) / np.max(np.abs(Zo), axis=(1, 2))).max() <= 1e-12


BIG_SHAPES = [
    # model, N, W, T, kwargs — beyond the tile shapes of the two-stage kernels: poly_deg 8..12 (collapsed FP64 tiles with
    # 2-4 k-steps, whatever FP64 precision is asked for) and 9..12 Cole-Cole modes (generic 16-mode kernel)
    ('decomp', 20, 32, 40, dict(poly_deg=8, n_tau=40)),
    ('decomp', 64, 64, 20, dict(poly_deg=9, n_tau=64)),
    ('decomp', 33, 100, 15, dict(poly_deg=10, n_tau=50, c_exp=0.5)),
    ('decomp', 64, 256, 8, dict(poly_deg=12, n_tau=128)),
    ('decomp', 12, 60, 20, dict(poly_deg=14, n_tau=30)),
    ('decomp', 20, 80, 10, dict(poly_deg=20, n_tau=40)),
    ('colecole', 20, 64, 20, dict(n_modes=9)),
    ('colecole', 33, 80, 12, dict(n_modes=12)),
    ('colecole', 12, 100, 10, dict(n_modes=16)),
]


@pytest.mark.parametrize("model,N,W,T,kw", BIG_SHAPES, ids=[f"{s[0]}-N{s[1]}-W{s[2]}-{i}" for i, s in enumerate(BIG_SHAPES)])
def test_unbounded_model_sizes_chain_forward_logprob(model, N, W, T, kw):
    """The reference accepts any poly_deg (models.py:195, 207-208) and any n_modes (models.py:243-252).  Chain identical
    to the oracle's on the same stream; batched forward / log-probability within 1e-12 of the oracle."""
    from bisip_b200 import engine
    from bisip_b200.batch import BatchInversion
    from oracle import oracle
    rng = np.random.default_rng(N * 1000 + W)
    w, zn, ze, bounds, okw = _spectrum(model, N, rng, **kw)
    inv = BatchInversion(model, w, zn[None], ze[None], nwalkers=W, nsteps=T, seed=99, spectrum_offset=7, **kw)
    p0 = inv.draw_p0(0, 1)
    res = inv.fit(p0=p0, keep_chain=True)
    prob = oracle.Problem(model, w, zn, ze, bounds, **okw)
    ref = prob.run(p0[0], T, seed=99, spectrum=7)
    assert res['flags'][0] == 0 and not ref['nan']
    np.testing.assert_array_equal(res['chain'][0], ref['chain'])
    fin = np.isfinite(ref['log_prob'])
    assert np.array_equal(fin, np.isfinite(res['log_prob'][0]))
    assert np.max(np.abs(res['log_prob'][0][fin] - ref['log_prob'][fin]) / np.maximum(1, np.abs(ref['log_prob'][fin]))) <= 1e-12
    th = np.concatenate([res['chain'][0][-1], p0[0][:7]])                 # posterior-ish and prior-wide thetas
    dev_th, dev_w = inv._to_dev(th[None], 0, 1), inv._to_dev(w[None], 0, 1)[0]
    Z = engine.forward(inv._spec(), dev_th, dev_w).cpu().numpy()[0]
    Zo = prob.forward(th)
    assert (np.max(np.abs(Z - Zo), axis=(1, 2)) / np.max(np.abs(Zo), axis=(1, 2))).max() <= 1e-12
    lp = engine.log_probability(inv._spec(), dev_th, dev_w, inv._to_dev(zn[None], 0, 1), inv._to_dev(ze[None], 0, 1),
                                inv._to_dev(bounds[None], 0, 1)[0]).cpu().numpy()[0]
    lpo = prob.log_probability(th)
    assert np.max(np.abs(lp - lpo) / np.maximum(1, np.abs(lpo))) <= 1e-12
    # model percentiles (fused kernel) for the same sizes
    mp = engine.model_percentile(inv._spec(), inv._to_dev(res['chain'][0][T // 2:].reshape(1, -1, th.shape[1]), 0, 1), dev_w, [50.0])
    want = np.percentile(prob.forward(res['chain'][0][T // 2:].reshape(-1, th.shape[1])), 50.0, axis=0)
    assert np.max(np.abs(mp.cpu().numpy()[0, 0] - want)) <= 1e-12 * np.max(np.abs(want))


def test_big_polynomial_limits():
    """poly_deg > 7 is an FP64-only, <= 256-walker path; beyond poly_deg 29 and for the TF32 modes the library says so."""
    from bisip_b200 import _lib
    from bisip_b200.batch import BatchInversion
    w = 2 * np.pi * np.logspace(3, -1, 16)
    zn, ze = np.zeros((1, 2, 16)), np.ones((1, 2, 16))
    with pytest.raises(_lib.BisipError, match='256 walkers'):
        BatchInversion('decomp', w, zn, ze, nwalkers=300, nsteps=3, poly_deg=9).fit()
    with pytest.raises(_lib.BisipError, match='poly_deg > 29'):
        BatchInversion('decomp', w, zn, ze, nwalkers=64, nsteps=3, poly_deg=30).fit()
    with pytest.raises(_lib.BisipError, match="needs precision"):
        BatchInversion('decomp', w, zn, ze, nwalkers=64, nsteps=3, poly_deg=9, precision='3xtf32').fit()
    with pytest.raises(_lib.BisipError, match=r"\[1,16\]"):
        BatchInversion('colecole', w, zn, ze, nwalkers=128, nsteps=3, n_modes=17).fit()


def test_per_spectrum_grids_and_non_pow2_scale():
    """w (B,N) and the tau grids differ per spectrum (w_stride / tau_stride paths); a = 2.5 takes the
    true-division branch of the stretch factor."""
    from bisip_b200.batch import BatchInversion, tau_grid
    from oracle import oracle
    rng = np.random.default_rng(5)
    N, W, T = 24, 36, 40
    specs = [_spectrum('decomp', N, rng, poly_deg=3, n_tau=30) for _ in range(3)]
    ws = np.stack([s[0] * (1.0 + 0.3 * i) for i, s in enumerate(specs)])           # three different grids
    zn, ze = np.stack([s[1] for s in specs]), np.stack([s[2] for s in specs])
    inv = BatchInversion('decomp', ws, zn, ze, nwalkers=W, nsteps=T, poly_deg=3, n_tau=30, seed=3, a=2.5)
    assert inv.taus.shape == (3, 30)
    p0 = inv.draw_p0(0, 3)
    res = inv.fit(p0=p0, keep_chain=True)
    for b in range(3):
        _, taus, log_taus = tau_grid(ws[b], 30, 3)
        ref = oracle.Problem('decomp', ws[b], zn[b], ze[b], inv.param_bounds, taus=taus, log_taus=log_taus).run(
            p0[b], T, seed=3, spectrum=b, a=2.5)
        np.testing.assert_array_equal(res['chain'][b], ref['chain'])


def test_discard_thin_corner_cases_and_continuation(data_files):
    """emcee slicing chain[discard+thin-1::thin] at the corners, and run_mcmc continuing a chain (step0)."""
    import bisip_b200 as bb
    from bisip_b200 import engine
    for d, t in ((0, 1), (9, 1), (10, 1), (0, 10), (0, 11), (3, 4), (5, 5), (2, 3)):
        assert engine.n_keep(10, d, t) == len(np.arange(10)[d + t - 1::t])
    m = bb.Dias2000(data_files['SIP-K389175'], nwalkers=16, nsteps=30, seed=8)
    p0 = np.random.default_rng(1).uniform(*m.param_bounds, (16, 5))
    m.fit(p0=p0)
    full = m.get_chain()
    np.testing.assert_array_equal(m.get_chain(discard=29), full[29:])
    np.testing.assert_array_equal(m.get_chain(thin=30), full[29::30])
    assert m.get_chain(discard=30).shape == (0, 16, 5)
    # continuing for 20 more steps == one 50-step run (the Philox counter carries the absolute step)
    m.sampler.run_mcmc(None, 20)
    assert m.sampler.iteration == 50 and m.get_chain().shape == (50, 16, 5)
    m2 = bb.Dias2000(data_files['SIP-K389175'], nwalkers=16, nsteps=50, seed=8)
    m2.fit(p0=p0)
    np.testing.assert_array_equal(m.get_chain(), m2.get_chain())
    np.testing.assert_array_equal(m.sampler.acceptance_fraction, m2.sampler.acceptance_fraction)
    from bisip_b200.batch import BatchInversion
    inv = BatchInversion('dias', m.data['w'], m.data['zn'][None], m.data['zn_err'][None], nwalkers=16, nsteps=10)
    with pytest.raises(ValueError):
        inv.fit(discard=10)                       # nothing left to summarise


def test_nan_data_sets_flags_and_raises(data_files):
    """A NaN in the data makes every log-probability NaN: emcee raises ValueError; the batch API flags it."""
    import bisip_b200 as bb
    from bisip_b200.batch import BatchInversion
    m = bb.PeltonColeCole(data_files['SIP-K389175'], nwalkers=16, nsteps=5)
    zn = np.stack([m.data['zn'], m.data['zn']])
    zn[1, 0, 3] = np.nan
    inv = BatchInversion('colecole', m.data['w'], zn, np.stack([m.data['zn_err']] * 2), nwalkers=16, nsteps=5)
    res = inv.fit()
    assert res['flags'][0] == 0 and res['flags'][1] != 0
    m._data['zn'] = zn[1]
    with pytest.raises(ValueError, match="NaN"):
        m.fit()


def test_c_abi_argument_errors():
    import ctypes as C
    from bisip_b200 import _lib
    lib = _lib.load()
    d = _lib.ModelDesc(_lib.MODEL_DIAS, 4, 8, 1, 0, 0, 0, 0, 1.0)                  # Dias with ndim 4
    assert lib.bisip_forward(C.byref(d), 1, 1, None, None, 0, None, None, 0, None, None) == -1
    assert b"ndim" in lib.bisip_last_error()
    d = _lib.ModelDesc(_lib.MODEL_DECOMP, 32, 8, 1, 16, 31, 0, 0, 1.0)              # poly_deg 30
    assert lib.bisip_forward(C.byref(d), 1, 1, None, None, 0, None, None, 0, None, None) == -2
    d = _lib.ModelDesc(_lib.MODEL_DECOMP, 10, 8, 1, 16, 9, _lib.PREC_3XTF32, 0, 1.0)  # poly_deg 8 in a TF32 mode
    assert lib.bisip_forward(C.byref(d), 1, 1, None, None, 0, None, None, 0, None, None) == -2
    d = _lib.ModelDesc(_lib.MODEL_COLECOLE, 52, 8, 17, 0, 0, 0, 0, 1.0)             # 17 modes
    assert lib.bisip_forward(C.byref(d), 1, 1, None, None, 0, None, None, 0, None, None) == -2
    d = _lib.ModelDesc(_lib.MODEL_DIAS, 5, 8, 1, 0, 0, 0, 0, 1.0)
    assert lib.bisip_forward(C.byref(d), 0, 1, None, None, 0, None, None, 0, None, None) == -1   # empty batch
    assert lib.bisip_forward(None, 1, 1, None, None, 0, None, None, 0, None, None) == -1
    assert lib.bisip_column_stats(None, 1, 1, 1, 0, None, None, None, None, None, None, 0, None) == -1
