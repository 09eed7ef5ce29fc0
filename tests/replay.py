"""Step-by-step replay of a stretch-move chain against its Philox stream (host only, NumPy).

The sampler's random stream is fully specified (``oracle/bisip_oracle.c::oracle_ensemble_run``,
``bisip_b200/csrc/sampler.cuh``): counter = (index, step, spectrum, purpose), key = seed.  Given the ensemble before
a step and the one after it, the stream alone determines the red/blue split, every partner and stretch factor, hence
every proposal bit for bit (the proposal arithmetic is unfused on both sides), and every ln u.  What is left free is
the sampler's own log-probabilities, so a chain from a reduced-precision kernel, whose accept decisions cannot match
an FP64 run once one of them flips, can still be checked decision by decision:

* positions: after its half-step every walker is either bitwise unchanged or bitwise its proposal;
* carry: a rejected walker keeps its previous stored lp bit for bit;
* accepted: ``((ndim-1) ln zz + lp') - lp > ln u`` holds with the sampler's own stored lp';
* rejected: the same inequality is false with the reference lp'(q) (the rejected lp' is not stored);
* counts: the accepted count of every walker equals the sampler's.

A decision whose margin is within the band of what the check cannot resolve is counted as unjudged instead: for an
accepted move ``1e-9 + 2^-46 max(|lp'|, |lp|)`` (host / device ``log`` ulps and the FP32 pre-filter of the kernel's
accept step, which hands every margin below 2^-12 to FP64 logarithms), for a rejected one that plus
``tol * max(1, |lp_ref(q)|)``, the stated error of the precision that computed lp'.
"""
import numpy as np

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
_LO = np.uint64(0xFFFFFFFF)
_S32 = np.uint64(32)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (Random123) over broadcastable integer arrays of 32-bit values; returns four uint64 arrays
    holding the 32-bit output words."""
    c0, c1, c2, c3, k0, k1 = (np.asarray(v, dtype=np.uint64) & _LO for v in (c0, c1, c2, c3, k0, k1))
    for _ in range(10):
        p0, p1 = _M0 * c0, _M1 * c2                      # 32 x 32 -> 64 bits: exact in uint64
        c0, c1, c2, c3 = (p1 >> _S32) ^ c1 ^ k0, p1 & _LO, (p0 >> _S32) ^ c3 ^ k1, p0 & _LO
        k0, k1 = (k0 + _W0) & _LO, (k1 + _W1) & _LO
    return c0, c1, c2, c3


def u53(a, b):
    """NumPy legacy random_sample bit recipe, as the kernel and the oracle assemble it (exact in float64)."""
    return ((a >> np.uint64(5)).astype(np.float64) * 67108864.0 + (b >> np.uint64(6)).astype(np.float64)) / 9007199254740992.0


def split(seed, spectrum, t, W):
    """Walker indices by rank for step t: ranks [0, H0) form split 0, [H0, W) split 1."""
    i = np.arange(W, dtype=np.uint64)
    words = philox4x32_10(i >> np.uint64(2), t, spectrum, 0, seed & 0xFFFFFFFF, seed >> 32)
    word = np.choose((i & np.uint64(3)).astype(np.intp), words)
    kmask = np.uint64((1 << max(0, int(W - 1).bit_length())) - 1)
    keys = (word & ~kmask & _LO) | i                      # unique: the low bits carry the walker index
    return np.argsort(keys, kind='stable')


def draws(seed, spectrum, t, s, Hs, Nc, a):
    """Stretch factors, partner ranks (into the complementary split) and ln u of the Hs proposals of half-step s."""
    x0, x1, x2, x3 = philox4x32_10(np.arange(Hs), t, spectrum, 1 + s, seed & 0xFFFFFFFF, seed >> 32)
    u = u53(x0, x1)
    zr = (a - 1.0) * u + 1.0
    zz = zr * zr / a
    partner = ((x2 * np.uint64(Nc)) >> _S32).astype(np.intp)
    lu = np.log(u53(x3, ((x2 << np.uint64(16)) & _LO) | np.uint64(0x8000)))
    return zz, partner, lu


def _bits(x):
    return np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)


def replay(seed, spectrum, a, p0, lp0, chain, log_prob, accepted, lp_ref, tol, step0=0):
    """Replay a chain kept with discard=0, thin=1: p0 (W, ndim) and lp0 (W,) the ensemble and stored lps before
    step ``step0``; chain (T, W, ndim), log_prob (T, W), accepted (W,) as the sampler returned them; ``lp_ref``
    maps thetas (n, ndim) to FP64 reference log-probabilities (n,); ``tol`` the relative error band of the sampler's
    log-probabilities (0 for FP64).

    Returns counts: violations ``position``, ``carry``, ``accept``, ``reject`` (decisions contradicted by the stream),
    ``count`` (walkers whose accepted count differs), and ``decisions``, ``unjudged_accept``, ``unjudged_reject``,
    ``ref_evals`` (rows handed to ``lp_ref``)."""
    seed, spectrum = int(seed), int(spectrum)
    chain = np.asarray(chain, dtype=np.float64)
    log_prob = np.asarray(log_prob, dtype=np.float64)
    T, W, ndim = chain.shape
    H0 = (W + 1) // 2
    out = dict(position=0, carry=0, accept=0, reject=0, count=0, decisions=0, unjudged_accept=0, unjudged_reject=0,
               ref_evals=0)
    n_acc = np.zeros(W, dtype=np.int64)
    cur = np.array(p0, dtype=np.float64)
    cur_lp = np.array(lp0, dtype=np.float64)
    for it in range(T):
        t = step0 + it
        after, after_lp = chain[it], log_prob[it]
        order = split(seed, spectrum, t, W)
        for s in range(2):
            off, Hs = (H0, W - H0) if s else (0, H0)
            coff, Nc = (0, H0) if s else (H0, W - H0)
            zz, partner, lu = draws(seed, spectrum, t, s, Hs, Nc, a)
            k = order[off:off + Hs]
            cj = cur[order[coff + partner]]
            q = cj - (cj - cur[k]) * zz[:, None]
            fac = (ndim - 1.0) * np.log(zz)
            lpo = cur_lp[k]
            new, new_lp = after[k], after_lp[k]
            moved = np.all(_bits(new) == _bits(q), axis=1)
            kept = np.all(_bits(new) == _bits(cur[k]), axis=1)
            acc = moved & ~kept
            out['position'] += int(np.count_nonzero(~moved & ~kept))
            rej = ~acc
            out['carry'] += int(np.count_nonzero(rej & (_bits(new_lp) != _bits(lpo))))
            out['decisions'] += Hs
            with np.errstate(invalid='ignore', over='ignore'):
                # accepted: judged with the sampler's own lp'
                la, lo_a = new_lp[acc], lpo[acc]
                margin = ((fac[acc] + la) - lo_a) - lu[acc]
                fin = np.isfinite(la) & np.isfinite(lo_a)
                band = 1e-9 + np.where(fin, 2.0 ** -46 * np.maximum(np.abs(np.where(fin, la, 0)), np.abs(np.where(fin, lo_a, 0))), 0)
                unj = np.abs(margin) <= band                 # NaN margin: judged (emcee's nan > x is False)
                out['unjudged_accept'] += int(np.count_nonzero(unj))
                out['accept'] += int(np.count_nonzero(~unj & ~(margin > 0)))
                # rejected: judged with the reference lp'(q)
                if np.any(rej):
                    lr = np.asarray(lp_ref(q[rej]), dtype=np.float64)
                    out['ref_evals'] += int(lr.shape[0])
                    lo_r = lpo[rej]
                    margin = ((fac[rej] + lr) - lo_r) - lu[rej]
                    fin = np.isfinite(lr) & np.isfinite(lo_r)
                    big = np.maximum(np.abs(np.where(fin, lr, 0)), np.abs(np.where(fin, lo_r, 0)))
                    band = np.where(fin, 1e-9 + 2.0 ** -46 * big + tol * np.maximum(1.0, np.abs(np.where(fin, lr, 0))), 0)
                    unj = np.abs(margin) <= band
                    out['unjudged_reject'] += int(np.count_nonzero(unj))
                    out['reject'] += int(np.count_nonzero(~unj & (margin > 0)))
            n_acc[k[acc]] += 1
            cur[k] = new                                     # half-step 1 proposes from the updated split 0
            cur_lp[k] = new_lp
    out['count'] = int(np.count_nonzero(n_acc != np.asarray(accepted)))
    return out


def violations(r):
    return r['position'] + r['carry'] + r['accept'] + r['reject'] + r['count']


class DecompReference:
    """FP64 log-probability of the polynomial decomposition for one spectrum (NumPy restatement of
    ``oracle/bisip_oracle.c``: Debye kernel matrix K from complex arithmetic, M = a @ log_taus,
    Z = R0 (1 - M K), Gaussian sum, strict box).  Vectorised over thetas, for replays that need ~10^5 evaluations
    at 256-512 taus where the oracle's S x N cpow calls per evaluation are too slow.  Pinned to
    ``oracle.Problem.log_probability`` by the tests that use it."""

    def __init__(self, w, taus, log_taus, c_exp, y, yerr, bounds):
        K = 1 - 1 / (1 + (1j * np.asarray(w)[None, :] * np.asarray(taus)[:, None]) ** c_exp)     # (S, N)
        self.Kre, self.Kim = np.ascontiguousarray(K.real), np.ascontiguousarray(K.imag)
        self.log_taus = np.asarray(log_taus, dtype=np.float64)                                  # (D, S)
        self.y = np.asarray(y, dtype=np.float64).reshape(2, -1)
        s2 = np.asarray(yerr, dtype=np.float64).reshape(2, -1) ** 2
        self.s2 = s2
        self.llc = np.sum(2 * np.log(s2))
        self.bounds = np.asarray(bounds, dtype=np.float64)

    def forward(self, theta):
        th = np.atleast_2d(np.asarray(theta, dtype=np.float64))
        M = th[:, 1:] @ self.log_taus
        R0 = th[:, :1]
        return np.stack([R0 * (1 - M @ self.Kre), -R0 * (M @ self.Kim)], axis=1)                 # (n, 2, N)

    def __call__(self, theta):
        th = np.atleast_2d(np.asarray(theta, dtype=np.float64))
        out = np.full(th.shape[0], -np.inf)
        inside = np.all((self.bounds[0] < th) & (th < self.bounds[1]), axis=1)
        for c0 in range(0, th.shape[0], 4096):
            sel = np.flatnonzero(inside[c0:c0 + 4096]) + c0
            if sel.size:
                r = self.y - self.forward(th[sel])
                out[sel] = -0.5 * (np.sum(r * r / self.s2, axis=(1, 2)) + self.llc)
        return out
