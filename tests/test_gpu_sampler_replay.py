"""Step-by-step replay of the reduced-precision decomposition samplers against their Philox stream and an FP64
reference log-probability (tests/replay.py).

A TF32 / 3xTF32 chain cannot be compared with the oracle's: the first accept decision that flips makes the chains
diverge.  The replay checks instead, step by step, what the stream determines: every walker is either unchanged or
bitwise its proposal, rejected walkers carry their lp bit for bit, accepted moves satisfy the accept inequality with
the kernel's own stored lp, rejected ones fail it with the FP64 reference lp (unless the margin is inside the
precision's stated error), and the accepted counts match.  Every stored lp and every initial lp is also compared with
the reference within the stated tolerance of the precision (tests/test_gpu_parity.py: log-prob relative 3e-3 for
TF32, 5e-5 for 3xTF32).  This reaches the evaluators as they run inside the sampler, which the batched entry point
does not: the 2-CTA tcgen05 cluster (real | imaginary column split, partial chi^2 exchanged over DSMEM) has no
batched form at all, and the single-CTA tcgen05 evaluator runs here under a tensor-memory allocation per CTA with
two CTAs per SM.  The FP64 'dmma' / 'dmma-cluster' rows are controls with no band on rejections: there the harness
and the kernels agree exactly.
"""
import time

import numpy as np
import pytest

import replay
from helpers import lp_err

pytestmark = pytest.mark.gpu

SEED = 2029
OFFSET = 5           # global index of the first spectrum: the Philox counter carries OFFSET + b

SHAPES = [  # (n_freq, n_tau, poly_deg, walkers, c_exp, precision, expected kernel, spectra, steps)
    (64, 64, 4, 256, 1.0, '3xtf32', 'tcgen05', 3, 30),      # C5 shape: one M=128 tile per half-step, two CTAs per SM
    (64, 64, 4, 256, 1.0, 'tf32', 'tcgen05', 3, 30),
    (20, 40, 4, 32, 1.0, '3xtf32', 'tcgen05', 3, 40),       # bundled-file shape: 16-row half-steps, padded columns / taus
    (33, 50, 3, 66, 0.5, '3xtf32', 'tcgen05', 3, 40),       # odd everything, Warburg
    (64, 8, 0, 14, 1.0, '3xtf32', 'tcgen05', 3, 40),        # a single K step, poly_deg 0
    (5, 3, 1, 8, 1.0, '3xtf32', 'tcgen05', 3, 40),          # fewer taus than a K step, fewer frequencies than a column group
    (9, 4, 5, 16, 1.0, 'tf32', 'tcgen05', 3, 40),           # more coefficients than taus
    (64, 64, 7, 254, 1.0, '3xtf32', 'tcgen05', 3, 30),      # poly_deg 7, 127-row half-steps
    (64, 128, 4, 256, 1.0, '3xtf32', 'tcgen05', 3, 30),     # two 64-tau chunks
    (64, 256, 4, 128, 1.0, 'tf32', 'tcgen05', 3, 30),       # four chunks
    (64, 256, 4, 128, 1.0, '3xtf32', 'tcgen05-cluster', 3, 30),   # real | imaginary columns over a 2-CTA cluster
    (64, 256, 4, 256, 0.5, '3xtf32', 'tcgen05-cluster', 3, 30),
    (40, 256, 5, 100, 1.0, '3xtf32', 'tcgen05-cluster', 3, 30),   # 48 columns per CTA
    (64, 512, 4, 64, 1.0, '3xtf32', 'mma-tf32', 3, 30),     # too large for the pair -> mma.sync tiles
    (64, 64, 4, 258, 1.0, '3xtf32', 'mma-tf32', 3, 30),     # 129-row half-steps
    (96, 64, 4, 64, 1.0, '3xtf32', 'mma-tf32', 3, 30),      # 192 columns
    (64, 64, 4, 256, 1.0, '3xtf32-mma', 'mma-tf32', 3, 30),
    (64, 64, 4, 256, 1.0, 'tf32-mma', 'mma-tf32', 3, 30),
    (64, 64, 4, 256, 1.0, '3xtf32', 'tcgen05', 320, 6),     # co-residency: several CTAs per SM, each with tensor memory
    (64, 64, 4, 256, 1.0, 'fp64', 'dmma', 3, 20),           # FP64 controls
    (64, 128, 4, 256, 1.0, 'fp64', 'dmma-cluster', 3, 20),
]

LP_TOL = {'tf32': 3e-3, 'tf32-mma': 3e-3, '3xtf32': 5e-5, '3xtf32-mma': 5e-5, 'fp64': 0.0}
# Largest fraction of decisions left unjudged (margin inside the band), twice the largest measured per precision.
# Measured (NVIDIA B200, 1,000 W power limit): 3xTF32 0.10-1.11 % per row (1.11 % with 96 frequencies on mma.sync,
# 1.10 % in the co-residency row; no accepted move was ever unjudged); TF32 5.8-20.4 % (the band is 3e-3 |lp| with
# |lp| ~ 1e3 at these spectra: ~3 nats); FP64 0: every decision judged.
UNJUDGED_MAX = {'tf32': 0.41, 'tf32-mma': 0.41, '3xtf32': 0.023, '3xtf32-mma': 0.023, 'fp64': 0.0}


def _replayed(B):
    """All spectra of a small batch; first, last, the uniform start (1) and evenly spaced ones of a large batch."""
    if B <= 8:
        return list(range(B))
    return sorted(set(np.linspace(0, B - 1, 38).round().astype(int)) | {0, 1, B - 1})


@pytest.mark.parametrize("N,S,P,W,c_exp,prec,kind,B,T", SHAPES,
                         ids=[f"{s[6]}-{s[5]}-N{s[0]}-S{s[1]}-P{s[2]}-W{s[3]}-B{s[7]}" for s in SHAPES])
def test_sampler_replay(N, S, P, W, c_exp, prec, kind, B, T):
    import torch
    from bisip_b200 import _lib, engine, synthetic
    from bisip_b200.batch import BatchInversion, tau_grid
    from oracle import oracle
    t0 = time.perf_counter()
    dev = _lib.require_cuda()
    _, w = synthetic.frequencies(N)
    _, taus, log_taus = tau_grid(w, S, P)
    ndim = P + 2

    def fwd(th, ww):
        return replay.DecompReference(ww, taus, log_taus, c_exp, np.zeros((2, N)), np.ones((2, N)), bounds).forward(th)

    inv = BatchInversion('decomp', w, np.zeros((1, 2, N)), np.ones((1, 2, N)), nwalkers=W, nsteps=T, poly_deg=P,
                         n_tau=S, c_exp=c_exp, precision=prec, seed=SEED, spectrum_offset=OFFSET, device=dev)
    bounds = inv.param_bounds
    syn = synthetic.make('decomp', OFFSET, OFFSET + B, fwd, N=N, poly_deg=P, n_tau=S)
    zn, ze = syn['zn'], syn['zn_err']
    spec = inv._spec()
    assert engine.decomp_kernel_kind(spec, N, W) == kind
    truth = syn['theta_true'].copy()
    truth[:, 0] /= syn['norm_factor']
    rng = np.random.default_rng(N * 1000 + W)
    p0 = truth[:, None, :] * (1 + 2e-3 * rng.standard_normal((B, W, ndim)))
    p0[1] = inv.draw_p0(1, 2)[0]                                            # one spectrum from uniform over the box
    args = (_lib.dev_f64(w, dev), _lib.dev_f64(zn, dev), _lib.dev_f64(ze, dev), _lib.dev_f64(bounds, dev))
    # the kernel's initial lp (the launch choice does not depend on nsteps), then the chain from the same p0
    lp0 = engine.ensemble_run(spec, _lib.dev_f64(p0, dev), *args, nsteps=0, seed=SEED, spectrum0=OFFSET)['lp'].cpu().numpy()
    res = engine.ensemble_run(spec, _lib.dev_f64(p0, dev), *args, nsteps=T, seed=SEED, spectrum0=OFFSET)
    chain, logp = res['chain'].cpu().numpy(), res['log_prob'].cpu().numpy()
    accepted, flags = res['accepted'].cpu().numpy(), res['flags'].cpu().numpy()
    assert np.all(flags == 0)
    np.testing.assert_array_equal(res['coords'].cpu().numpy(), chain[:, -1])
    np.testing.assert_array_equal(res['lp'].cpu().numpy(), logp[:, -1])

    tol = LP_TOL[prec]
    tot = dict(position=0, carry=0, accept=0, reject=0, count=0, decisions=0, unjudged_accept=0, unjudged_reject=0,
               ref_evals=0)
    errs = []
    for i, b in enumerate(_replayed(B)):
        ref = replay.DecompReference(w, taus, log_taus, c_exp, zn[b], ze[b], bounds)
        if i == 0:      # the NumPy reference is the oracle's log-probability
            th = np.concatenate([p0[b][:16], chain[b][-1][:16]])
            prob = oracle.Problem('decomp', w, zn[b], ze[b], bounds, taus=taus, log_taus=log_taus, c_exp=c_exp)
            assert lp_err(ref(th), prob.log_probability(th)).max() <= 1e-12
        r = replay.replay(SEED, OFFSET + b, 2.0, p0[b], lp0[b], chain[b], logp[b], accepted[b], ref, tol)
        for k in tot:
            tot[k] += r[k]
        # every stored lp: the initial ones, and the new lp of every move (a rejected walker carries its lp bitwise,
        # which the replay checks)
        prev = np.concatenate([p0[b][None], chain[b][:-1]])
        moved = np.any(chain[b] != prev, axis=-1)
        th = np.concatenate([p0[b], chain[b][moved]])
        got = np.concatenate([lp0[b], logp[b][moved]])
        want = ref(th)
        assert np.array_equal(np.isneginf(got), np.isneginf(want)), b
        errs.append(lp_err(got, want))
    errs = np.concatenate(errs)
    unjudged = tot['unjudged_accept'] + tot['unjudged_reject']
    frac = unjudged / tot['decisions']
    batched = ''
    if kind in ('tcgen05', 'mma-tf32') and prec != 'fp64':
        # The batched log-probability runs the same evaluator code, each tile row on its own: the stored lps are
        # bitwise its values (measured on every such row).  Except where only the sampler's half-step size forced
        # mma.sync (129 rows > the 128-lane tile): the batched path tiles by 128 rows and runs tcgen05 there (measured
        # max difference 1.0e-6 relative).  Not for the cluster rows: the batched path has no clustered form and runs
        # those shapes on mma.sync tiles.
        lpb = engine.log_probability(spec, _lib.dev_f64(chain.reshape(B, T * W, ndim), dev), *args).cpu().numpy()
        d = lp_err(lpb, logp.reshape(B, T * W))
        batched = f' batched: max {d.max():.3e} equal {np.array_equal(lpb, logp.reshape(B, T * W))}'
        if (W + 1) // 2 <= 128:
            np.testing.assert_array_equal(lpb, logp.reshape(B, T * W))
        assert d.max() <= tol
    print(f"\n[replay] {kind} {prec} N{N} S{S} P{P} W{W} B{B} T{T}: lp_err max {errs.max():.3e} median "
          f"{np.median(errs):.3e}; unjudged {unjudged}/{tot['decisions']} ({frac:.4%}; accept {tot['unjudged_accept']}); "
          f"ref evals {tot['ref_evals']}; {time.perf_counter() - t0:.2f} s{batched}")
    assert replay.violations(tot) == 0, tot
    assert errs.max() <= (1e-12 if tol == 0 else tol)
    if tol:
        assert errs.max() > 1e-9                                            # the reduced-precision path really ran
    assert frac <= UNJUDGED_MAX[prec], tot
