"""CPU tests of the chain replay harness (tests/replay.py): its Philox against the oracle's, a clean replay of
oracle chains over the models, walker counts, stretch scales and spectrum indices the GPU replays use, and negative
controls that each corruption of a chain is reported."""
import numpy as np
import pytest

import replay
from helpers import oracle_problem
from oracle import oracle

KAT = [((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
       ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
       ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
        (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1))]


def test_vectorised_philox_matches_oracle():
    for ctr, key, want in KAT:
        got = replay.philox4x32_10(*ctr, *key)
        assert tuple(int(v) for v in got) == want
    rng = np.random.default_rng(2)
    c = rng.integers(0, 2 ** 32, (10_000, 4), dtype=np.uint64)
    k = rng.integers(0, 2 ** 32, (10_000, 2), dtype=np.uint64)
    got = np.stack(replay.philox4x32_10(c[:, 0], c[:, 1], c[:, 2], c[:, 3], k[:, 0], k[:, 1]), axis=1)
    want = np.array([oracle.philox4x32_10(tuple(int(v) for v in c[i]), tuple(int(v) for v in k[i])) for i in range(len(c))],
                    dtype=np.uint64)
    np.testing.assert_array_equal(got, want)


def _problem(case, gold_fl, gold_ld):
    if case == 'decomp_p3_debye':            # the p3 tau table of the golden fixture with a Debye exponent
        ld = gold_ld
        return oracle.Problem('decomp', ld['SIP-K389175/w'], ld['SIP-K389175/zn'], ld['SIP-K389175/zn_err'],
                              gold_fl['decomp_p3_c07/bounds'], taus=gold_fl['decomp_p3_c07/taus'],
                              log_taus=gold_fl['decomp_p3_c07/log_taus'], c_exp=1.0)
    return oracle_problem(case, gold_fl, gold_ld)


def _oracle_run(case, W, a, spectrum, T, gold_fl, gold_ld, seed=77):
    prob = _problem(case, gold_fl, gold_ld)
    p0 = np.random.default_rng(W).uniform(prob.bounds[0], prob.bounds[1], (W, prob.ndim))
    run = prob.run(p0, T, seed=seed, spectrum=spectrum, a=a)
    assert not run['nan']
    return prob, p0, run


RUNS = [  # golden case, walkers, stretch scale, spectrum index, steps
    ('decomp_p4_debye', 12, 2.0, 0, 40),      # W = 2 ndim
    ('decomp_p4_debye', 32, 2.0, 3, 40),
    ('decomp_p3_debye', 31, 4.0, 9, 40),      # odd W, a a power of two other than 2
    ('dias', 31, 2.5, 0, 40),                 # odd W, a not a power of two
    ('dias', 300, 2.0, 5, 12),                # more walkers than a CTA has threads
    ('shin', 12, 2.0, 1, 40),
    ('colecole_k2', 70, 4.0, 12, 40),
]


@pytest.mark.parametrize("case,W,a,spec,T", RUNS, ids=[f"{r[0]}-W{r[1]}-a{r[2]}-s{r[3]}" for r in RUNS])
def test_replay_of_oracle_chain_is_clean(case, W, a, spec, T, gold_fl, gold_ld):
    prob, p0, run = _oracle_run(case, W, a, spec, T, gold_fl, gold_ld)
    r = replay.replay(77, spec, a, p0, prob.log_probability(p0), run['chain'], run['log_prob'], run['accepted'],
                      prob.log_probability, tol=0.0)
    assert replay.violations(r) == 0, r
    assert r['unjudged_accept'] == 0 and r['unjudged_reject'] == 0, r
    assert r['decisions'] == T * W
    assert 0 < run['accepted'].sum() < T * W


def test_decomp_reference_pinned_and_replays_oracle_chain(gold_fl, gold_ld):
    """The NumPy FP64 decomposition log-probability equals the oracle's to 1e-12, and as the replay's reference it
    judges an oracle chain clean."""
    from helpers import lp_err
    for case in ('decomp_p4_debye', 'decomp_p4_warburg', 'decomp_p3_c07'):
        prob = oracle_problem(case, gold_fl, gold_ld)
        ref = replay.DecompReference(prob.w, prob.taus, prob.log_taus, prob.c.c_exp, prob.y, prob.yerr, prob.bounds)
        rng = np.random.default_rng(4)
        th = rng.uniform(prob.bounds[0], prob.bounds[1], (300, prob.ndim))
        th[150:, 1:] *= 0.02
        th[0, 0] = prob.bounds[1, 0]                         # on a face: -inf
        want = prob.log_probability(th)
        got = ref(th)
        assert np.array_equal(np.isneginf(got), np.isneginf(want)) and np.isneginf(got[0])
        assert lp_err(got, want).max() <= 1e-12
    prob, p0, run = _oracle_run('decomp_p4_debye', 32, 2.0, 3, 40, gold_fl, gold_ld)
    ref = replay.DecompReference(prob.w, prob.taus, prob.log_taus, 1.0, prob.y, prob.yerr, prob.bounds)
    r = replay.replay(77, 3, 2.0, p0, prob.log_probability(p0), run['chain'], run['log_prob'], run['accepted'], ref,
                      tol=1e-12)
    assert replay.violations(r) == 0 and r['unjudged_reject'] + r['unjudged_accept'] == 0, r


@pytest.fixture(scope='module')
def dias_run(gold_fl, gold_ld):
    prob, p0, run = _oracle_run('dias', 31, 2.5, 4, 40, gold_fl, gold_ld)
    return prob, p0, run


def _replay(prob, p0, run, chain=None, log_prob=None, seed=77, spec=4):
    return replay.replay(seed, spec, 2.5, p0, prob.log_probability(p0),
                         run['chain'] if chain is None else chain, run['log_prob'] if log_prob is None else log_prob,
                         run['accepted'], prob.log_probability, tol=0.0)


def test_negative_control_one_ulp_in_one_position(dias_run):
    prob, p0, run = dias_run
    ch = run['chain'].copy()
    ch[17, 5, 2] = np.nextafter(ch[17, 5, 2], np.inf)
    assert _replay(prob, p0, run, chain=ch)['position'] > 0


def test_negative_control_two_walkers_swapped(dias_run):
    prob, p0, run = dias_run
    ch, lp = run['chain'].copy(), run['log_prob'].copy()
    ch[20, [3, 8]] = ch[20, [8, 3]]
    lp[20, [3, 8]] = lp[20, [8, 3]]
    assert _replay(prob, p0, run, chain=ch, log_prob=lp)['position'] > 0


def test_negative_control_stored_lp_changed_on_rejected_step(dias_run):
    prob, p0, run = dias_run
    ch = run['chain']
    t, k = next((t, k) for t in range(10, 40) for k in range(31) if np.array_equal(ch[t, k], ch[t - 1, k]))
    lp = run['log_prob'].copy()
    lp[t, k] = np.nextafter(lp[t, k], -np.inf)
    r = _replay(prob, p0, run, log_prob=lp)
    assert r['carry'] > 0 and r['position'] == 0


def test_negative_control_wrong_spectrum_and_seed(dias_run):
    prob, p0, run = dias_run
    assert _replay(prob, p0, run)['position'] == 0
    assert replay.violations(_replay(prob, p0, run, spec=5)) > 0
    assert replay.violations(_replay(prob, p0, run, seed=78)) > 0
