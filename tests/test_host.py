"""CPU tests of the host layer: data ingest parity, chain slicing semantics, the percentile index
arithmetic, error contracts, the C-ABI exports, and the multi-rank shard/gather logic (gloo, 2 ranks)."""
import ctypes
import os
import re
import subprocess
import sys
import warnings

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_load_data_matches_reference(gold_ld, data_files):
    import bisip_b200 as bb
    for name in ('SIP-K389170', 'SIP-K389172', 'SIP-K389173', 'SIP-K389174', 'SIP-K389175', 'SIP-K389176'):
        d = bb.Dias2000(data_files[name]).data
        for k in ('zn', 'zn_err', 'w', 'Z', 'Z_err'):
            np.testing.assert_array_equal(d[k], gold_ld[f'{name}/{k}'])      # bit-identical
        assert d['norm_factor'] == gold_ld[f'{name}/norm_factor']
        assert d['N'] == 20 and d['zn'].shape == (2, 20)
    for units in ('rad', 'deg'):
        d = bb.Dias2000(data_files['SIP-K389175'], ph_units=units).data
        np.testing.assert_array_equal(d['zn'], gold_ld[f'units_{units}/zn'])
        np.testing.assert_array_equal(d['zn_err'], gold_ld[f'units_{units}/zn_err'])
    d = bb.PeltonColeCole(data_files['SIP-K389172'], headers=9).data
    np.testing.assert_array_equal(d['zn'], gold_ld['headers9/zn'])
    assert set(d) == {'freq', 'amp', 'pha', 'amp_err', 'pha_err', 'Z', 'Z_err', 'norm_factor', 'zn', 'zn_err', 'N', 'w'}


def test_from_files_vectorised_ingest_is_bit_identical(gold_ld, data_files, tmp_path, monkeypatch):
    """BatchInversion.from_files (one text-to-double pass + one vectorised prepare over all files) against the per-file
    load_data of the drop-in classes and the goldens generated from the reference; irregular inputs take NumPy's per-file
    path; ragged lengths raise."""
    import torch
    from bisip_b200 import _lib, utils
    from bisip_b200.batch import BatchInversion
    monkeypatch.setattr(_lib, 'require_cuda', lambda device=None: torch.device('cpu'))
    names = ['SIP-K389170', 'SIP-K389172', 'SIP-K389173', 'SIP-K389174', 'SIP-K389175', 'SIP-K389176']
    paths = [data_files[n] for n in names]
    for units in ('mrad', 'rad', 'deg'):
        inv = BatchInversion.from_files('dias', paths, ph_units=units, nwalkers=16, nsteps=10)
        assert inv.n_spectra == 6 and inv._zn.shape == (6, 2, 20) and len(inv.data) == 6
        for i, fp in enumerate(paths):
            one = utils.prepare_data(np.loadtxt(fp, skiprows=1, delimiter=','), units)
            d = inv.data[i]
            assert set(d) == set(one) and d['N'] == one['N'] == 20
            for k in one:
                np.testing.assert_array_equal(d[k], one[k], err_msg=f'{names[i]} {k} {units}')     # bit-identical
            np.testing.assert_array_equal(inv._zn[i], one['zn'])
            np.testing.assert_array_equal(inv._zn_err[i], one['zn_err'])
    inv = BatchInversion.from_files('dias', paths, nwalkers=16, nsteps=10)
    for i, n in enumerate(names):
        np.testing.assert_array_equal(inv._zn[i], gold_ld[f'{n}/zn'])
        np.testing.assert_array_equal(inv._zn_err[i], gold_ld[f'{n}/zn_err'])
    assert [d['norm_factor'] for d in inv.data][4] == gold_ld['SIP-K389175/norm_factor']
    assert inv.w.ndim == 1                                   # the bundled files share their frequency grid
    # the fast pass and the per-file path agree on what they parse
    np.testing.assert_array_equal(utils.read_tables(paths), np.stack([np.loadtxt(fp, skiprows=1, delimiter=',') for fp in paths]))
    # other header counts, per-spectrum frequency grids, irregular formatting (spaces, a comment line): per-file path
    body = open(paths[4]).read().splitlines()
    (tmp_path / 'h3.dat').write_text('\n'.join(['# a', '# b'] + body) + '\n')
    np.testing.assert_array_equal(BatchInversion.from_files('dias', [tmp_path / 'h3.dat'], headers=3, nwalkers=16, nsteps=10)._zn[0],
                                  gold_ld['SIP-K389175/zn'])
    rows = [r.split(',') for r in body[1:]]
    shifted = [body[0]] + [','.join([repr(float(r[0]) * 1.5)] + r[1:]) for r in rows]
    (tmp_path / 'shifted.dat').write_text('\n'.join(shifted) + '\n')
    inv2 = BatchInversion.from_files('dias', [paths[4], tmp_path / 'shifted.dat'], nwalkers=16, nsteps=10)
    assert inv2.w.shape == (2, 20)
    np.testing.assert_array_equal(inv2.w[1], 2 * np.pi * np.array([float(r[0]) * 1.5 for r in rows]))
    np.testing.assert_array_equal(inv2.w[0], gold_ld['SIP-K389175/w'])
    spaced = [body[0]] + [', '.join(r) for r in rows[:10]] + ['# comment'] + [', '.join(r) for r in rows[10:]]
    (tmp_path / 'spaced.dat').write_text('\n'.join(spaced) + '\n')
    np.testing.assert_array_equal(BatchInversion.from_files('dias', [tmp_path / 'spaced.dat'], nwalkers=16, nsteps=10)._zn[0],
                                  gold_ld['SIP-K389175/zn'])
    (tmp_path / 'short.dat').write_text('\n'.join(body[:-3]) + '\n')
    with pytest.raises(ValueError, match='same number of frequencies'):
        BatchInversion.from_files('dias', [paths[4], tmp_path / 'short.dat'], nwalkers=16, nsteps=10)
    (tmp_path / 'bad.dat').write_text('\n'.join(body[:5] + ['1.0,abc,3.0,4.0,5.0'] + body[6:]) + '\n')
    with pytest.raises(ValueError):
        BatchInversion.from_files('dias', [tmp_path / 'bad.dat'], nwalkers=16, nsteps=10)


def test_model_surface_matches_reference(data_files, gold_fl):
    import bisip_b200 as bb
    fp = data_files['SIP-K389175']
    pd = bb.PolynomialDecomposition(fp, poly_deg=4)
    assert pd.param_names == ['r0', 'a0', 'a1', 'a2', 'a3', 'a4']
    np.testing.assert_array_equal(pd.param_bounds, gold_fl['decomp_p4_debye/bounds'])
    np.testing.assert_array_equal(pd.taus, gold_fl['decomp_p4_debye/taus'])
    np.testing.assert_array_equal(pd.log_taus, gold_fl['decomp_p4_debye/log_taus'])
    np.testing.assert_array_equal(pd.log_tau, np.linspace(-6, 2, 40))
    assert (pd.nwalkers, pd.nsteps, pd.headers, pd.ph_units, pd.poly_deg, pd.c_exp) == (32, 5000, 1, 'mrad', 4, 1.0)
    assert bb.PolynomialDecomposition(fp).poly_deg == 5
    assert bb.PolynomialDecomposition(fp, n_tau=64).taus.shape == (64,)
    cc = bb.ColeCole(fp, n_modes=2)
    assert bb.ColeCole is bb.PeltonColeCole
    assert cc.param_names == ['r0', 'm1', 'm2', 'log_tau1', 'log_tau2', 'c1', 'c2']
    np.testing.assert_array_equal(cc.param_bounds, gold_fl['colecole_k2/bounds'])
    np.testing.assert_array_equal(bb.Dias2000(fp).param_bounds, gold_fl['dias/bounds'])
    np.testing.assert_array_equal(bb.Shin2015(fp).param_bounds, gold_fl['shin/bounds'])
    # bounds are read from the mutable params dict on every access (reference models.py:176-179)
    pd.params.update(a0=[-2, 2])
    assert pd.param_bounds[0, 1] == -2
    assert not pd.fitted and pd.p0 is None
    with pytest.raises(AssertionError, match='Model is not fitted'):
        pd.get_chain()
    with pytest.raises(AssertionError):
        pd.sampler
    with pytest.raises(AssertionError):
        pd.plot_traces()
    # prior is host logic: strict inequalities, NaN -> -inf
    b = pd.param_bounds
    assert pd._log_prior(np.array([1.0, 0, 0, 0, 0, 0]), b) == 0.0
    assert pd._log_prior(np.array([1.1, 0, 0, 0, 0, 0]), b) == -np.inf
    assert pd._log_prior(np.array([np.nan, 0, 0, 0, 0, 0]), b) == -np.inf
    assert set(bb.__all__) >= {'Inversion', 'PolynomialDecomposition', 'PeltonColeCole', 'Dias2000', 'Shin2015',
                               'plotlib', 'test_run', 'DataFiles'}
    assert sorted(bb.DataFiles()) == ['SIP-K389170', 'SIP-K389172', 'SIP-K389173', 'SIP-K389174', 'SIP-K389175', 'SIP-K389176']


def test_no_cpu_fallback(data_files):
    """Without a GPU the product path must fail loudly, never compute on the host."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    import bisip_b200 as bb
    from bisip_b200._lib import BisipError
    m = bb.Dias2000(data_files['SIP-K389175'], nwalkers=32, nsteps=10)
    with pytest.raises(BisipError, match='no CPU fallback'):
        m.forward(np.array([1.0, 0.25, -10, 5, 0.5]), m.data['w'])
    with pytest.raises(BisipError):
        m.fit()
    # a user forward callable runs on the host, but the likelihood reduction is a CUDA kernel: still no CPU path
    inside = m.param_bounds.mean(axis=0)
    with pytest.raises(BisipError, match='no CPU fallback'):
        m._log_probability(inside, lambda t, w: np.zeros((2, len(w))), m.param_bounds, m.data['w'], m.data['zn'],
                           m.data['zn_err'])
    # outside the prior box the reference returns -inf without calling the model (models.py:71-76)
    assert m._log_probability(np.zeros(5), lambda t, w: 1 / 0, m.param_bounds, m.data['w'], m.data['zn'],
                              m.data['zn_err']) == -np.inf


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, 'bisip_b200')
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                src = open(os.path.join(dp, f)).read()
                assert not re.search(r'^\s*(from|import)\s+oracle', src, re.M), f
                assert 'oracle/' not in src or f == 'data.py' or 'tests/golden' in src or 'same stream as oracle' in src.lower() \
                    or 'oracle/bisip_oracle.c' in src, f


def test_slice_chain_emcee_semantics():
    from bisip_b200.sampler import slice_chain
    T, W, D = 2000, 32, 4
    arr = np.arange(T * W * D, dtype=np.float64).reshape(T, W, D)
    assert slice_chain(arr, T, discard=500).shape == (1500, 32, 4)          # quickstart.ipynb:173
    flat = slice_chain(arr, T, discard=500, thin=2, flat=True)
    assert flat.shape == (24000, 4)                                          # quickstart.ipynb:192
    np.testing.assert_array_equal(flat, arr[501::2].reshape(-1, 4))
    np.testing.assert_array_equal(slice_chain(arr, T, thin=10), arr[9::10])
    assert slice_chain(arr, 100).shape == (100, 32, 4)                       # iteration bound
    from bisip_b200 import _lib
    lib = _lib.load()
    for (t, d, th) in [(2000, 500, 2), (2000, 0, 1), (2000, 1000, 10), (10, 9, 1), (10, 10, 1), (7, 0, 3), (7, 2, 5)]:
        assert lib.bisip_n_keep(t, d, th) == len(range(d + th - 1, t, th))


def test_percentile_indices_match_numpy():
    from bisip_b200._lib import percentile_indices
    rng = np.random.default_rng(0)
    for n in (1, 2, 3, 10, 999, 25600, 512000):
        x = np.sort(rng.standard_normal(n))
        p = np.array([0, 2.5, 16, 33.3, 50, 84, 97.5, 99.99, 100])
        lo, g = percentile_indices(n, p)
        hi = np.minimum(lo + 1, n - 1)
        a, b = x[lo], x[hi]
        d = b - a
        val = np.where(g >= 0.5, b - d * (1 - g), a + d * g)
        np.testing.assert_array_equal(val, np.percentile(x, p))
    with pytest.raises(ValueError):
        percentile_indices(10, [101])


def test_parse_chain_contract(data_files):
    import bisip_b200 as bb
    m = bb.Dias2000(data_files['SIP-K389175'])
    with pytest.raises(ValueError, match='Flatten chain'):
        m.parse_chain(np.zeros((4, 3, 2)))
    with pytest.raises(ValueError, match='Do not pass both'):
        m.parse_chain(np.zeros((4, 2)), discard=1)
    c = np.zeros((4, 2))
    assert m.parse_chain(c) is c
    with pytest.raises(AssertionError):          # chain=None -> get_chain -> not fitted
        m.parse_chain(None, discard=1)


def test_c_abi_exports_every_declared_symbol():
    from bisip_b200 import _lib
    hdr = open(os.path.join(ROOT, 'include', 'bisip_b200.h')).read()
    declared = set(re.findall(r'^\s*(?:const\s+char\s*\*\s*|int64_t\s+|int\s+)(bisip_\w+)\s*\(', hdr, re.M))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name
    assert _lib.load().bisip_abi_version() == _lib.ABI_VERSION == 2
    out = subprocess.run(['nm', '-D', '--defined-only', _lib.LIB_PATH], capture_output=True, text=True).stdout
    assert all(re.search(rf'\bT {n}\b', out) for n in declared)


def test_header_enums_match_python_constants():
    """The ctypes layer hard-codes the enum values of include/bisip_b200.h (models, precisions, kernel kinds)."""
    import re
    from bisip_b200 import _lib
    hdr = open(os.path.join(ROOT, 'include', 'bisip_b200.h')).read()
    val = {m.group(1): int(m.group(2)) for m in re.finditer(r'\b(BISIP_[A-Z0-9_]+)\s*=\s*(-?\d+)', hdr)}
    assert (val['BISIP_MODEL_COLECOLE'], val['BISIP_MODEL_DIAS'], val['BISIP_MODEL_SHIN'], val['BISIP_MODEL_DECOMP']) == \
        (_lib.MODEL_COLECOLE, _lib.MODEL_DIAS, _lib.MODEL_SHIN, _lib.MODEL_DECOMP)
    assert _lib.PRECISIONS == {'fp64': val['BISIP_PREC_FP64'], 'tf32': val['BISIP_PREC_TF32'], '3xtf32': val['BISIP_PREC_3XTF32'],
                               'tf32-mma': val['BISIP_PREC_TF32_MMA'], '3xtf32-mma': val['BISIP_PREC_3XTF32_MMA'],
                               'fp64-collapsed': val['BISIP_PREC_FP64_COLLAPSED']}
    assert _lib.KERNEL_KINDS == {val['BISIP_KERNEL_DMMA']: 'dmma', val['BISIP_KERNEL_DMMA_CLUSTER']: 'dmma-cluster',
                                 val['BISIP_KERNEL_MMA_TF32']: 'mma-tf32', val['BISIP_KERNEL_TCGEN05']: 'tcgen05',
                                 val['BISIP_KERNEL_TCGEN05_CLUSTER']: 'tcgen05-cluster',
                                 val['BISIP_KERNEL_FP64_COLLAPSED']: 'fp64-collapsed'}


def test_walkers_independent_and_autocorr():
    from bisip_b200.sampler import integrated_time, walkers_independent
    rng = np.random.default_rng(1)
    assert walkers_independent(rng.standard_normal((32, 5)))
    assert not walkers_independent(np.ones((32, 5)))
    x = rng.standard_normal((32, 5)); x[:, 1] = x[:, 0]
    assert not walkers_independent(x)
    # AR(1) with phi: tau = (1+phi)/(1-phi)
    phi, n = 0.8, 60000
    e = rng.standard_normal((n, 4))
    y = np.zeros((n, 4))
    for i in range(1, n):
        y[i] = phi * y[i - 1] + e[i]
    tau = integrated_time(y[:, :, None])
    assert abs(tau[0] - 9.0) < 1.0


def test_batched_autocorr_time_matches_the_per_chain_estimator():
    import torch
    from bisip_b200 import sampler
    rng = np.random.default_rng(3)
    B, T, W, D = 3, 600, 8, 2
    x = np.zeros((B, T, W, D))
    for b, phi in enumerate((0.5, 0.8, 0.95)):                       # AR(1) chains: tau = (1 + phi)/(1 - phi)
        e = rng.standard_normal((T, W, D))
        for t in range(1, T):
            x[b, t] = phi * x[b, t - 1] + e[t]
    got = sampler.integrated_time_batch(torch.from_numpy(x), c=5, thin=2).numpy()
    for b in range(B):
        ref = 2 * sampler.integrated_time(x[b], c=5, quiet=True)
        np.testing.assert_allclose(got[b], ref, rtol=1e-10)
    assert got[2].mean() > got[1].mean() > got[0].mean()


def test_synthetic_generator_is_shard_independent():
    from bisip_b200 import synthetic
    fwd = lambda th, w: np.stack([np.stack([np.outer(t[:1], np.ones_like(w))[0], -0.1 * t[1] * np.ones_like(w)]) for t in th])
    a = synthetic.make('dias', 0, 6, fwd, N=16)
    b = synthetic.make('dias', 3, 6, fwd, N=16)
    np.testing.assert_array_equal(a['zn'][3:], b['zn'])
    np.testing.assert_array_equal(a['theta_true'][3:], b['theta_true'])
    lo, hi = synthetic.true_box('decomp', 4)
    assert lo[0] == 0.95 and hi[0] == 1.05 and a['zn'].shape == (6, 2, 16)
    assert np.allclose(np.max(np.hypot(a['zn'][:, 0], a['zn'][:, 1]), axis=1), 1.0)


def test_draw_p0_depends_on_global_index_only(monkeypatch):
    """Starting positions of a spectrum are a function of (seed, global index): the same whatever the shard, the sub-batch
    or the number of host threads that drew them (BatchInversion.draw_p0 fills blocks of 64 indices in parallel)."""
    import torch
    from bisip_b200 import _lib
    from bisip_b200.batch import BatchInversion
    monkeypatch.setattr(_lib, 'require_cuda', lambda device=None: torch.device('cpu'))
    w = np.logspace(3, -1, 8)
    mk = lambda n, off: BatchInversion('dias', w, np.zeros((n, 2, 8)), np.ones((n, 2, 8)), nwalkers=12, nsteps=5, seed=3,
                                       spectrum_offset=off)
    monkeypatch.setenv('LOCAL_WORLD_SIZE', '1')
    full = mk(1000, 0).draw_p0(0, 1000)                  # 16 blocks: threaded
    lo, hi = mk(1, 0).param_bounds
    assert full.shape == (1000, 12, 5) and np.all(full >= lo) and np.all(full < hi)
    monkeypatch.setenv('LOCAL_WORLD_SIZE', '1000000')     # one thread
    np.testing.assert_array_equal(mk(1000, 0).draw_p0(0, 1000), full)
    np.testing.assert_array_equal(mk(300, 450).draw_p0(0, 300), full[450:750])       # another shard
    np.testing.assert_array_equal(mk(1000, 0).draw_p0(63, 130), full[63:130])         # a sub-batch across block edges
    assert not np.array_equal(full[0], full[64])


def test_tau_grid_matches_reference_tables_and_vectorises(data_files):
    """batch.tau_grid builds PolynomialDecomposition's log_tau / taus / log_taus (reference models.py:201-209) — the same
    tables the drop-in class holds (which test_model_surface_matches_reference pins to the reference's), and for a (B, N)
    stack of frequency vectors the rows are bit-identical to the one-vector results."""
    import bisip_b200 as bb
    from bisip_b200.batch import tau_grid
    m = bb.PolynomialDecomposition(data_files['SIP-K389175'], poly_deg=5)
    lt, taus, lts = tau_grid(m.data['w'], None, 5)
    np.testing.assert_array_equal(lt, m.log_tau)
    np.testing.assert_array_equal(taus, m.taus)
    np.testing.assert_array_equal(lts, m.log_taus)
    rng = np.random.default_rng(1)
    w = 2 * np.pi * 10 ** rng.uniform(-3, 5, (40, 33))
    stack = tau_grid(w, 40, 7)
    assert stack[0].shape == (40, 40) and stack[2].shape == (40, 8, 40)
    for i in range(40):
        for a, b in zip(stack, tau_grid(w[i], 40, 7)):
            np.testing.assert_array_equal(a[i], b)


def test_shard_range_partitions():
    from bisip_b200.batch import shard_range
    for n in (1, 7, 8, 100000, 12501):
        for world in (1, 2, 4, 8):
            spans = [shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            assert max(h - l for l, h in spans) == -(-n // world)


_GLOO_WORKER = r'''
import os, sys
sys.path.insert(0, os.environ["BISIP_ROOT"])
import numpy as np, torch, torch.distributed as dist
from bisip_b200.batch import shard_range, gather
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:" + os.environ["PORT"],
                        rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
rank, world = dist.get_rank(), dist.get_world_size()
n = 11
lo, hi = shard_range(n, rank, world)
idx = torch.arange(lo, hi, dtype=torch.float64)
local = {"mean": idx[:, None] * torch.ones(1, 3, dtype=torch.float64),
         "percentiles": idx[:, None, None] + torch.arange(6, dtype=torch.float64).reshape(1, 2, 3),
         "flags": torch.arange(lo, hi, dtype=torch.int32)}
full = gather(local, n, rank, world)
assert full["mean"].shape == (n, 3) and full["percentiles"].shape == (n, 2, 3)
assert torch.equal(full["mean"][:, 0], torch.arange(n, dtype=torch.float64))
assert torch.equal(full["flags"], torch.arange(n, dtype=torch.int32))
assert torch.equal(full["percentiles"][:, 1, 2], torch.arange(n, dtype=torch.float64) + 5)
dist.barrier()
dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_gather_two_ranks_gloo(tmp_path):
    """World-size-2 gloo run of the shard + all-gather logic that the N>1 GPU path uses with NCCL."""
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER)
    port = str(29600 + os.getpid() % 300)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", PORT=port, BISIP_ROOT=ROOT)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    for p in procs:
        out, _ = p.communicate(timeout=180)
        assert p.returncode == 0, out
        assert "ok" in out


def test_bench_reference_arm_prints_one_json_line():
    """`bench.py --impl reference` (the CPU arm the driver launches next to the GPU arm): stdout is exactly one JSON
    line with the contract's keys, whatever the workers or native libraries print; ranks other than 0 print nothing."""
    import json
    env = dict(os.environ, BISIP_BENCH_REF_STEPS='2')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '1'],
                         capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = out.stdout.splitlines()
    assert len(lines) == 1, lines
    j = json.loads(lines[0])
    assert j['impl'] == 'reference' and j['metric'] == 'log-prob evals/sec' and j['unit'] == 'evals/s'
    assert j['value'] > 0 and j['higher_is_better'] is True and j['vs_baseline'] is None
    assert j['cpu_baseline']['kind'] == 'reference' and j['cpu_baseline']['cores'] >= 1
    assert j['e2e'] == {'value': j['value'], 'unit': 'evals/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    quiet = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '1'],
                           capture_output=True, text=True, env=dict(env, RANK='1', WORLD_SIZE='2'), timeout=600)
    assert quiet.returncode == 0 and quiet.stdout == ''


def test_bench_dump_outputs_writes_seeded_float64_samples(tmp_path, monkeypatch):
    """`bench.py --dump-outputs`: float64 .npy files whose sampled rows are fixed by the seed and equal the rows of the
    step's results they name; the total is held under the limit."""
    import importlib.util
    import torch
    spec = importlib.util.spec_from_file_location('bench_under_test', os.path.join(ROOT, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    monkeypatch.setattr(bench, 'DUMP_MAX_SPECTRA', 30)
    g = torch.Generator().manual_seed(0)
    B, W = 40, 8
    out = {'percentiles': torch.rand(B, 3, 6, generator=g, dtype=torch.float64),
           'mean': torch.rand(B, 6, generator=g, dtype=torch.float64),
           'std': torch.rand(B, 6, generator=g, dtype=torch.float64),
           'acceptance_fraction': torch.rand(B, generator=g, dtype=torch.float64)}
    res = {'chain': torch.rand(B, 3, W, 6, generator=g, dtype=torch.float64),
           'accepted': torch.randint(0, 100, (B, W), generator=g, dtype=torch.int32)}
    bench.dump_outputs(torch, str(tmp_path / 'a'), out, res)
    bench.dump_outputs(torch, str(tmp_path / 'b'), out, res)
    names = sorted(os.listdir(tmp_path / 'a'))
    assert names == sorted(f'{k}.npy' for k in list(out) + ['spectra', 'chain', 'accepted', 'chain_spectra'])
    d = {n[:-4]: np.load(tmp_path / 'a' / n) for n in names}
    for n in names:
        assert d[n[:-4]].dtype == np.float64
        np.testing.assert_array_equal(d[n[:-4]], np.load(tmp_path / 'b' / n))
    rows, crow = d['spectra'].astype(int), d['chain_spectra'].astype(int)
    assert len(rows) == 30 and np.all(np.diff(rows) > 0) and len(crow) == bench.DUMP_CHAINS and np.all(np.diff(crow) > 0)
    for k in out:
        np.testing.assert_array_equal(d[k], out[k].numpy()[rows])
    np.testing.assert_array_equal(d['chain'], res['chain'].numpy()[crow])
    np.testing.assert_array_equal(d['accepted'], res['accepted'].numpy()[crow])
    monkeypatch.setattr(bench, 'DUMP_LIMIT', 1000)
    with pytest.raises(ValueError):
        bench.dump_outputs(torch, str(tmp_path / 'c'), out, res)


_SHARDED_WORKER = r'''
import os, sys
sys.path.insert(0, os.environ["BISIP_ROOT"])
import numpy as np, torch, torch.distributed as dist
import bisip_b200
from bisip_b200 import _lib, batch
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:" + os.environ["PORT"],
                        rank=int(os.environ["RANK"]), world_size=int(os.environ["WORLD_SIZE"]))
rank, world = dist.get_rank(), dist.get_world_size()
# the device work is stubbed: per-spectrum results are functions of the GLOBAL spectrum index, on CPU tensors
_lib.require_cuda = lambda device=None: torch.device("cpu")
def fake_fit_device(self, p0=None, discard=0, thin=1, percentiles=(2.5, 50, 97.5), keep_chain=False, batch_size=None,
                    _chain_to_host=False):
    g = torch.arange(self.spectrum_offset, self.spectrum_offset + self.n_spectra, dtype=torch.float64)
    assert p0 is None or p0.shape[0] == self.n_spectra
    out = {"percentiles": g[:, None, None] + torch.arange(len(percentiles) * self.ndim, dtype=torch.float64).reshape(1, len(percentiles), self.ndim),
           "mean": g[:, None] * torch.ones(1, self.ndim, dtype=torch.float64), "std": 0.5 * g[:, None] * torch.ones(1, self.ndim, dtype=torch.float64),
           "acceptance_fraction": 0.01 * g, "flags": (g % 3 == 0).to(torch.int32)}
    if keep_chain:
        out["chain"] = g[:, None, None, None] * torch.ones(1, 4, self.nwalkers, self.ndim, dtype=torch.float64)
        out["log_prob"] = torch.zeros(self.n_spectra, 4, self.nwalkers, dtype=torch.float64)
    return out
batch.BatchInversion.fit_device = fake_fit_device
B, N = 11, 8
w = np.logspace(3, -1, N)
zn = np.zeros((B, 2, N)); ze = np.ones((B, 2, N))
p0 = np.zeros((B, 12, 5))
res = bisip_b200.fit_sharded("dias", w, zn, ze, discard=2, thin=1, p0=p0, gather_chain=True, nwalkers=12, nsteps=10)
assert res["shard"] == batch.shard_range(B, rank, world)
assert res["mean"].shape == (B, 5) and res["percentiles"].shape == (B, 3, 5) and res["flags"].dtype == np.int32
np.testing.assert_array_equal(res["mean"][:, 0], np.arange(B))
np.testing.assert_array_equal(res["percentiles"][:, 2, 4], np.arange(B) + 14)
np.testing.assert_array_equal(res["flags"], (np.arange(B) % 3 == 0).astype(np.int32))
np.testing.assert_allclose(res["acceptance_fraction"], 0.01 * np.arange(B))
if rank == 0:
    assert res["chain"].shape == (B, 4, 12, 5)
    np.testing.assert_array_equal(res["chain"][:, 1, 3, 2], np.arange(B))
else:
    assert res["chain"] is None
# fewer spectra than ranks: rank 1 owns an empty block and still takes part in every collective
import warnings
with warnings.catch_warnings(record=True) as caught:
    warnings.simplefilter("always")
    one = bisip_b200.fit_sharded("dias", w, zn[:1], ze[:1], discard=2, p0=p0[:1], gather_chain=True, nwalkers=12, nsteps=10)
assert one["shard"] == ((0, 1) if rank == 0 else (1, 1))
assert one["mean"].shape == (1, 5) and one["percentiles"].shape == (1, 3, 5) and one["flags"].tolist() == [1]
assert (one["chain"].shape == (1, 4, 12, 5)) if rank == 0 else (one["chain"] is None)
assert any("returned NaN for 1 of 1" in str(c.message) for c in caught)      # nan_policy sees the complete result
# tiny chunks: several collective rounds, ragged last shard
ch = torch.arange(*batch.shard_range(B, rank, world), dtype=torch.float64)[:, None] * torch.ones(1, 7, dtype=torch.float64)
full = batch.gather_chain_to_rank0(ch, B, rank, world, chunk_bytes=2 * 7 * 8)
if rank == 0:
    np.testing.assert_array_equal(full[:, 3], np.arange(B))
dist.barrier()
dist.destroy_process_group()
print("rank", rank, "ok")
'''


def test_fit_sharded_two_ranks_gloo(tmp_path):
    """Product-level multi-GPU entry point (full arrays in, complete result on every rank, chains to rank 0) on a
    world-size-2 gloo group; the per-rank device work is stubbed so the test runs on CPU."""
    script = tmp_path / "worker_sharded.py"
    script.write_text(_SHARDED_WORKER)
    port = str(29900 + os.getpid() % 90)
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", PORT=port, BISIP_ROOT=ROOT)
        procs.append(subprocess.Popen([sys.executable, str(script)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    for p in procs:
        out, _ = p.communicate(timeout=180)
        assert p.returncode == 0, out
        assert "ok" in out


def test_cython_funcs_surface_and_argument_checks():
    """bisip_b200.cython_funcs exports the reference's four native names (cython_funcs.pyx:49-108) and applies Cython's
    typed-buffer checks BEFORE touching the GPU (so they are testable here)."""
    import inspect
    from bisip_b200 import cython_funcs as cf
    sig = {n: list(inspect.signature(getattr(cf, n)).parameters) for n in cf.__all__}
    assert sig == {'ColeCole_cyth': ['w', 'R0', 'm', 'lt', 'c'],
                   'Dias2000_cyth': ['w', 'R0', 'm', 'log_tau', 'eta', 'delta'],
                   'Decomp_cyth': ['w', 'taus', 'log_taus', 'c_exp', 'R0', 'a'],
                   'Shin2015_cyth': ['w', 'R', 'log_Q', 'n']}
    w = np.array([1.0, 2.0])
    with pytest.raises(ValueError, match='Buffer dtype mismatch'):
        cf.Dias2000_cyth(w.astype(np.float32), 1.0, 0.25, -10.0, 5.0, 0.5)
    with pytest.raises(ValueError, match='wrong number of dimensions'):
        cf.Decomp_cyth(w, np.ones(3), np.ones(3), 1.0, 1.0, np.ones(1))
    with pytest.raises(TypeError):
        cf.ColeCole_cyth([1.0, 2.0], 1.0, np.array([0.3]), np.array([-2.0]), np.array([0.5]))
    with pytest.raises(TypeError):
        cf.Shin2015_cyth(w, np.array([0.5, 0.5]), np.array([-14.0, -6.0]), 'n')


def test_batch_validation_and_run_mcmc_kwargs(monkeypatch):
    """emcee's up-front checks apply to batches too; unsupported run_mcmc keywords raise (no silent semantics change)."""
    import torch
    from bisip_b200 import _lib
    from bisip_b200.batch import BatchInversion
    from bisip_b200.sampler import EnsembleSampler
    monkeypatch.setattr(_lib, 'require_cuda', lambda device=None: torch.device('cpu'))
    w = np.logspace(3, -1, 8)
    zn, ze = np.zeros((3, 2, 8)), np.ones((3, 2, 8))
    with pytest.raises(RuntimeError):
        BatchInversion('dias', w, zn, ze, nwalkers=8, nsteps=10).fit_device()
    with pytest.raises(ValueError, match='bounds must be'):
        BatchInversion('dias', w, zn, ze, nwalkers=16, nsteps=10, bounds=np.zeros((2, 4))).fit_device()
    with pytest.raises(ValueError, match='incompatible input dimensions'):
        BatchInversion('dias', w, zn, ze, nwalkers=16, nsteps=10).fit_device(p0=np.zeros((3, 15, 5)))
    p0 = np.zeros((3, 16, 5)); p0[1, 2, 3] = np.nan
    with pytest.raises(ValueError, match='infinite or NaN'):
        BatchInversion('dias', w, zn, ze, nwalkers=16, nsteps=10).fit_device(p0=p0, batch_size=2)   # checked on the uploaded copy, per sub-batch, before any launch
    with pytest.raises(ValueError):
        BatchInversion('dias', w, zn, ze, nan_policy='maybe')
    empty = BatchInversion('dias', w, zn[:0], ze[:0], nwalkers=16, nsteps=10).fit_device(discard=4, keep_chain=True)
    assert empty['percentiles'].shape == (0, 3, 5) and empty['chain'].shape == (0, 6, 16, 5)
    assert empty['flags'].dtype == torch.int32 and empty['log_prob'].shape == (0, 6, 16)
    from bisip_b200 import engine
    s = EnsembleSampler(16, 5, engine.ModelSpec(model=_lib.MODEL_DIAS, ndim=5), w, zn[0], ze[0], np.zeros((2, 5)), seed=1)
    with pytest.raises(NotImplementedError, match='thin_by'):
        s.run_mcmc(np.zeros((16, 5)), 10, thin_by=2)


def test_exp_table_constants_and_accuracy():
    """The table-driven exp of csrc/models.cuh (exp_fast): every 2^(j/32) entry in the source is the correctly rounded
    value, the reduction / Taylor constants are the ones tools/exp_table_check.py evaluates, and that evaluation (exact
    rational arithmetic, one rounding per FMA) stays below 2e-16 relative — far inside the 1e-12 parity bar."""
    import importlib.util
    import re
    from decimal import Decimal, getcontext
    src = open(os.path.join(ROOT, 'bisip_b200', 'csrc', 'models.cuh')).read()
    tab = re.search(r'kExp2Tab\[32\] = \{(.*?)\};', src, re.S).group(1)
    vals = [float.fromhex(t) for t in re.findall(r'0x1\.[0-9a-f]+p[+-]\d+', tab)]
    assert len(vals) == 32
    getcontext().prec = 50
    ln2 = Decimal(2).ln()
    for j, v in enumerate(vals):
        assert v == float((ln2 * Decimal(j) / Decimal(32)).exp()), j
    spec = importlib.util.spec_from_file_location('exp_table_check', os.path.join(ROOT, 'tools', 'exp_table_check.py'))
    chk = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(chk)
    kt = re.search(r'kExpT\[8\] = \{(.*?)\};', src, re.S).group(1)
    consts = [float.fromhex(t) for t in re.findall(r'-?0x1\.[0-9a-f]+p[+-]\d+', kt)]
    assert consts == [chk.A, chk.H, chk.L] + chk.C
    assert chk.TAB == vals
    rng = np.random.default_rng(3)
    worst = 0.0
    for x in np.concatenate([rng.uniform(-700, 700, 300), rng.uniform(-40, 40, 300), [0.0, 1e-300, -1e-9, 699.9, -699.9]]):
        ex = Decimal(float(x)).exp()
        worst = max(worst, float(abs((Decimal(chk.exp_table(float(x))) - ex) / ex)))
    assert worst < 2e-16


def test_library_sass_uses_the_tensor_cores_it_claims():
    """The shipped sm_100a library holds the instructions DESIGN.md says the decomposition kernels issue: FP64 DMMA tiles
    (default and collapsed paths), tcgen05 MMAs with tensor-memory loads / stores (TF32 / 3xTF32 paths: UTCHMMA, LDTM, STTM)
    and the mma.sync TF32 tiles of the comparison arm.  cuobjdump runs on the CPU; no GPU needed."""
    import shutil
    exe = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    if not os.path.exists(exe):
        pytest.skip('cuobjdump not available')
    from bisip_b200 import _lib
    out = subprocess.run([exe, '-sass', _lib.LIB_PATH], capture_output=True, text=True, timeout=600).stdout
    assert 'sm_100a' in out
    count = lambda key: sum(1 for line in out.splitlines() if key in line)
    assert count('DMMA') >= 1000
    assert count('UTCHMMA') >= 100 and count('LDTM') >= 100 and count('STTM') >= 50
    assert count('HMMA.1688.F32.TF32') >= 100
