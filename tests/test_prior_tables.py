"""The prior kernels and code-point tables against exact references, at every depth up to VBQ_MAX_DEPTH = 20.

Every other search test checks the kernels on the table the kernel itself built, so a wrong table would pass them
all.  Here the tables, the inverse CDFs, the CDF and the Gaussian quantiles are compared with the arbitrary-precision
reference of tests/prior_reference.py (mpmath, CPU) on samples of every depth, and with float64 certificates on whole
tables; then the searches that read the deepest tables (raw-length quantize, intervals, the float64 embedding search)
are compared with the NumPy oracle on the same table.

Tolerances: a correct float64 computation followed by one rounding to float32 returns the correctly rounded float32
of the true value, except when the true value lies within the float64 computation's own error of a float32 rounding
boundary.  That error (the "band") is derived per entry in prior_reference.solver_band from the solver's stopping rule
and an a-priori bound of the float64 evaluation; only inside it may the kernel return the other neighbour."""
import os

import numpy as np
import pytest
import torch

import prior_reference as R
from oracle import vbq_oracle as O
import vbq_test_helpers as H

pytestmark = pytest.mark.gpu

mpmath = R.mpmath
DEV = "cuda"
N_MAX = 20
DEPTHS = (0, 1, 10, 11, 13, 16, 20)
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "%s.npz")


def _dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def heap_xi(Q):
    """xi of heap entries 0..Q-1: (i + 1/2) 2^-n, exact in float64 (what heap_xi() in priors.cu computes)."""
    h = np.arange(Q, dtype=np.int64)
    n = np.floor(np.log2(h + 1)).astype(np.int64)
    n -= (1 << n) > h + 1                                     # guard the float log2 at powers of two
    n += (1 << (n + 1)) <= h + 1
    return (h + 1 - (1 << n) + 0.5) * np.exp2(-n.astype(np.float64))


def xi_of(h):
    """heap_xi of one entry."""
    n = int(h + 1).bit_length() - 1
    return (h + 1 - (1 << n) + 0.5) * 2.0 ** -n


def sorted_order(N):
    """Heap index of every sorted position: sorted rank of (n, i) is (2i + 1) 2^(N-n) - 1."""
    n = np.repeat(np.arange(N + 1), [1 << k for k in range(N + 1)])
    i = np.arange((1 << (N + 1)) - 1) - ((1 << n) - 1)
    return np.argsort(O.heap_to_sorted_rank(n, i, N))


def depth_sample(N, rng, n_random):
    """Both ends and the middle of every depth 0..N, plus `n_random` uniformly drawn heap entries."""
    hs = []
    for n in range(N + 1):
        base, w = (1 << n) - 1, 1 << n
        hs += [base, base + w // 2, base + w - 1]
    hs += list(rng.integers(0, (1 << (N + 1)) - 1, n_random))
    return np.unique(np.asarray(hs, dtype=np.int64))


# ----------------------------------------------------------------------------------------------------------------------
# the prior zoo: trained priors, the reference initialisation at three scales, gates from off to strongly non-linear,
# a prior far off zero, and channel counts that are not multiples of 16
# ----------------------------------------------------------------------------------------------------------------------
def _golden(name):
    g = np.load(GOLDEN % name)
    return O.LearnedPriorNP([g["matrix%d" % k] for k in range(4)], [g["bias%d" % k] for k in range(4)],
                            [g["factor%d" % k] for k in range(3)])


def _shifted(C=5, median=300.0):
    """init_scale 0.01 moved to `median` by the first-layer bias: depth-20 quantiles ~1e-8 apart at z ~ 300, where
    one float32 ulp is 3e-5, so many adjacent float32 entries are equal."""
    pr = H.make_prior(C, seed=41, factor_std=0.5, init_scale=0.01)
    pr.biases[0] = (pr.biases[0] - pr.matrices[0] * np.float32(median)).astype(np.float32)
    return pr


ZOO = {
    "golden_c6_n10": lambda: _golden("learned_c6_n10"),
    "golden_c20_n6_gated": lambda: _golden("learned_c20_n6_gated"),
    "scale0.01_c1": lambda: H.make_prior(1, seed=31, factor_std=0.5, init_scale=0.01),
    "scale1000_c5": lambda: H.make_prior(5, seed=32, factor_std=0.5, init_scale=1000.0),
    "fs0_c16": lambda: H.make_prior(16, seed=33, factor_std=0.0, init_scale=10.0),
    "fs3_c17": lambda: H.make_prior(17, seed=34, factor_std=3.0, init_scale=10.0),
    "fs0.5_c33": lambda: H.make_prior(33, seed=35, factor_std=0.5, init_scale=10.0),
    "shifted300_c5": _shifted,
}

_CACHE = {}


def zoo(name):
    """Per-module cache: the prior, its packed parameters, the kernel's depth-20 table (host) and mpmath roots."""
    if name not in _CACHE:
        import vbq_b200
        pr = ZOO[name]()
        packed = pr.packed()
        t20 = vbq_b200.ops.build_code_points_learned(_dev(packed), N_MAX).cpu().numpy()
        _CACHE[name] = dict(pr=pr, packed=packed, t20=t20, roots={})
    return _CACHE[name]


def mp_root(z, c, h):
    """mpmath quantile of heap entry h of channel c (cached); the kernel's value only seeds the bracket."""
    key = (c, int(h))
    if key not in z["roots"]:
        xi = xi_of(int(h))
        z["roots"][key] = R.inverse_cdf(z["packed"][c], xi, guess=float(z["t20"][c, h]))
    return z["roots"][key]


def check_correctly_rounded(z, c, hs, got):
    """got[k] is the float32 of heap entry hs[k]: it must be the correctly rounded quantile outside the band."""
    bad = []
    for h, g in zip(hs, got):
        root = mp_root(z, c, h)
        want, dist = R.f32_correctly_rounded(root)
        if g != want and not dist <= R.solver_band(z["packed"][c], root, xi_of(int(h))):
            bad.append((c, int(h), float(g), float(want), dist))
    assert not bad, "not correctly rounded outside the band: %s" % bad[:5]


def certify_f64(pr, c, xi, t):
    """Float64 certificate that each float32 t is the correctly rounded root of logits_c = logit(xi) up to the band:
    logits at the midpoints to both float32 neighbours must straddle the target, except by at most the float64
    evaluation error of those logits (prior_reference.logits_error_bound, u = 2^-53) plus the band's other terms
    (2 ulps of the target, the 1e-14 |x| stopping rule times the slope).  Returns the number of entries that are
    inside that allowance on the wrong side (i.e. inside the band)."""
    t = np.asarray(t, dtype=np.float32)
    assert np.all(np.isfinite(t))
    lo = 0.5 * (t.astype(np.float64) + np.nextafter(t, np.float32(-np.inf)).astype(np.float64))
    hi = 0.5 * (t.astype(np.float64) + np.nextafter(t, np.float32(np.inf)).astype(np.float64))
    target = np.log(xi) - np.log1p(-xi)
    one = O.LearnedPriorNP([m[c:c + 1] for m in pr.matrices], [b[c:c + 1] for b in pr.biases],
                           [f[c:c + 1] for f in pr.factors])
    p = pr.packed()[c]
    Llo, Lhi = one.logits(lo[:, None])[:, 0], one.logits(hi[:, None])[:, 0]
    slope = (Lhi - Llo) / (hi - lo)
    tol_lo = R.logits_error_bound(p, lo, R.U64, 2) + 4 * R.U64 * np.abs(target) + 1e-14 * np.abs(lo) * slope
    tol_hi = R.logits_error_bound(p, hi, R.U64, 2) + 4 * R.U64 * np.abs(target) + 1e-14 * np.abs(hi) * slope
    ok = (Llo - target <= tol_lo) & (Lhi - target >= -tol_hi)
    assert ok.all(), "channel %d: %d entries are not the rounded root, e.g. heap %s" % (
        c, (~ok).sum(), np.flatnonzero(~ok)[:5])
    return int(((Llo > target) | (Lhi < target)).sum())


# ----------------------------------------------------------------------------------------------------------------------
# 1. learned tables at every depth
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(ZOO))
def test_learned_tables_every_depth(name):
    import vbq_b200
    z = zoo(name)
    pr, packed, t20 = z["pr"], z["packed"], z["t20"]
    C = pr.channels
    params = _dev(packed)
    # the xi of heap entry h does not depend on N: every depth's table is a prefix of the depth-20 one
    for N in DEPTHS[:-1]:
        tN = vbq_b200.ops.build_code_points_learned(params, N).cpu().numpy()
        assert tN.shape == (C, (1 << (N + 1)) - 1)
        assert np.array_equal(tN, t20[:, :tN.shape[1]]), N
    # full tables of depth <= 10 against the float64 bisection oracle: equal, or neighbours inside the band
    Q10 = (1 << 11) - 1
    xi10 = heap_xi(Q10)
    want = pr.inverse_cdf_f64(np.repeat(xi10[:, None], C, axis=1)).T
    diff = np.argwhere(want != t20[:, :Q10])
    ulp = np.abs(want.view(np.int32).astype(np.int64) - t20[:, :Q10].view(np.int32).astype(np.int64))
    assert ulp.max() <= 1
    if len(diff):
        for c, h in diff[:50]:
            check_correctly_rounded(z, int(c), [int(h)], [t20[c, h]])
    # full tables of depth <= 13 (every channel) and of depth 20 (first and last channel): float64 certificate
    Q13 = (1 << 14) - 1
    xi13, xi20 = heap_xi(Q13), heap_xi(t20.shape[1])
    band = 0
    for c in range(C):
        band += certify_f64(pr, c, xi13, t20[c, :Q13])
    for c in sorted({0, C - 1}):
        band += certify_f64(pr, c, xi20, t20[c])
    print("%s: %d certified entries inside the band" % (name, band))
    # mpmath: ends and middle of every depth of the first and last channel, and 1000 random (channel, entry) pairs
    rng = np.random.default_rng(7)
    for c in sorted({0, C - 1}):
        hs = depth_sample(N_MAX, rng, 0)
        check_correctly_rounded(z, c, hs, t20[c, hs])
    cs = rng.integers(0, C, 1000)
    hs = rng.integers(0, t20.shape[1], 1000)
    for c in range(C):
        sel = cs == c
        check_correctly_rounded(z, c, hs[sel], t20[c, hs[sel]])
    # the same device routine behind learned_inverse_cdf: bit-identical on the same xi, at every depth
    xi_rep = torch.from_numpy(xi20).to(DEV).reshape(-1, 1).expand(-1, C).contiguous()
    inv = vbq_b200.ops.learned_inverse_cdf(params, xi_rep)
    assert torch.equal(inv.t(), torch.from_numpy(t20).to(DEV))
    del xi_rep, inv


# ----------------------------------------------------------------------------------------------------------------------
# 2. table structure
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(ZOO))
def test_table_structure(name):
    z = zoo(name)
    t20 = z["t20"]
    s = t20[:, sorted_order(N_MAX)]
    d = np.diff(s, axis=1)
    assert np.all(d >= 0), "sorted order decreases"
    # every heap node lies between its two children (the search kernels walk the heap as a binary search tree)
    Qp = (1 << N_MAX) - 1
    h = np.arange(Qp)
    assert np.all(t20[:, 2 * h + 1] <= t20[:, h]) and np.all(t20[:, h] <= t20[:, 2 * h + 2])
    # equal adjacent entries only where the exact quantiles are within one float32 ulp of each other
    order = sorted_order(N_MAX)
    cs, ks = np.nonzero(d == 0)
    rng = np.random.default_rng(3)
    pick = rng.permutation(len(cs))[:40]
    for c, k in zip(cs[pick], ks[pick]):
        a, b = mp_root(z, c, order[k]), mp_root(z, c, order[k + 1])
        with mpmath.workdps(R.DPS):
            assert abs(b - a) <= mpmath.mpf(float(np.spacing(np.abs(s[c, k])))), (c, k)
    if name.startswith("shifted"):
        # the collided case is real: the searches below run on a table with equal adjacent entries
        assert len(cs) > 1000, len(cs)
        print("%s: %d equal adjacent float32 entries at depth 20" % (name, len(cs)))


# ----------------------------------------------------------------------------------------------------------------------
# 3. inverse CDF at the edges of its domain
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["golden_c6_n10", "scale1000_c5", "fs3_c17", "shifted300_c5"])
def test_inverse_cdf_edges(name):
    import vbq_b200
    z = zoo(name)
    C = z["pr"].channels
    special = np.array([0.0, -0.0, 1.0, np.nan, -0.1, 1.1, -np.inf, np.inf])
    finite = np.array([5e-324, 1e-300, 2.0 ** -60, 2.0 ** -21, 0.5, 1 - 2.0 ** -21, 1 - 2.0 ** -53])
    xi = np.concatenate([special, finite])
    got = vbq_b200.ops.learned_inverse_cdf(_dev(z["packed"]), _dev(np.repeat(xi[:, None], C, axis=1))).cpu().numpy()
    # solve_inverse_cdf: xi == 0 -> -inf, xi == 1 -> +inf, anything else outside (0, 1) (and NaN) -> NaN
    want = np.array([-np.inf, -np.inf, np.inf, np.nan, np.nan, np.nan, np.nan, np.nan], dtype=np.float32)
    assert np.array_equal(got[:len(special)], np.repeat(want[:, None], C, axis=1), equal_nan=True)
    fin = got[len(special):]
    assert np.all(np.diff(fin, axis=0) >= 0), "not monotone in xi"
    for c in range(C):
        for k, x in enumerate(finite):
            root = R.inverse_cdf(z["packed"][c], x, guess=float(fin[k, c]) if np.isfinite(fin[k, c]) else None)
            want32, dist = R.f32_correctly_rounded(root)
            # +-inf only where the true root is beyond the float32 range (want32 is then +-inf too)
            assert fin[k, c] == want32 or dist <= R.solver_band(z["packed"][c], root, x), (c, x, fin[k, c], want32)


# ----------------------------------------------------------------------------------------------------------------------
# 4. CDF accuracy, tails included
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["golden_c6_n10", "golden_c20_n6_gated", "scale0.01_c1", "scale1000_c5", "fs3_c17",
                                  "shifted300_c5"])
def test_learned_cdf_against_mpmath(name):
    import vbq_b200
    z = zoo(name)
    pr, packed = z["pr"], z["packed"]
    C = pr.channels
    cs = range(C) if C <= 6 else (0, 1, C // 2, C - 1)
    rows = []
    # exact quantiles from the lower tail (CDF 1e-38, above the flush to 0 at logits -88.7) through the body to the
    # upper tail (1 - 1e-7, below the saturation at 1 - 2^-24), one past it, then steps out from the median in units
    # of the prior's own width (so narrow and off-centre priors get as many unsaturated points as wide ones) and out
    # to the float32 range
    xis = np.concatenate([np.logspace(-38, -1, 19), [0.5], 1 - np.logspace(-1, -7, 7), [1 - 1e-12]])
    steps = np.logspace(-3, 38, 42)
    for c in cs:
        med = float(z["t20"][c, 0])
        width = float(z["t20"][c, 2]) - float(z["t20"][c, 1])          # interquartile range (heap entries 1, 2)
        guess = pr.inverse_cdf_f64(np.repeat(xis[:, None], C, axis=1))[:, c]
        q = [float(R.inverse_cdf(packed[c], p, guess=float(g))) for p, g in zip(xis, guess)]
        with np.errstate(over="ignore"):
            off_ = np.float32(width) * steps.astype(np.float32)
        off_ = off_[np.isfinite(off_)]
        mag = np.concatenate([np.logspace(-6, 38, 45), [3.4e38]]).astype(np.float32)
        xs = np.concatenate([q, med + off_, med - off_, mag, -mag]).astype(np.float32)
        xs = xs[np.isfinite(xs)]
        col = np.full((len(xs), C), med, dtype=np.float32)
        col[:, c] = xs
        rows.append((c, col))
    x = np.concatenate([r[1] for r in rows])
    got = vbq_b200.ops.learned_cdf(_dev(packed), _dev(x)).cpu().numpy()
    ref32 = pr.cdf(x)                                  # the reference's float32 formula (learned_prior.py:109-148)
    off = 0
    n_checked = 0
    for c, col in rows:
        for k in range(col.shape[0]):
            xv = col[k, c]
            g, r32 = got[off + k, c], ref32[off + k, c]
            exact = R.cdf(packed[c], float(xv))
            lg = R.logits(packed[c], float(xv))
            # float32 logits: forward error bound with u = 2^-24 and CUDA's 2-ulp tanhf
            EL = float(R.logits_error_bound(packed[c], float(xv), R.U32, 2))
            if g in (0.0, 1.0) or r32 in (0.0, 1.0):
                # flushed to 0 (expf(-logits) overflows: logits < -88.72) or saturated to 1 (1 + expf(-logits)
                # rounds to 1: logits > 16.64): the reference's float32 formula must do the same, except where the
                # exact logits are within the float32 logits error of that threshold
                near = min(abs(float(lg) + 88.7228391), abs(float(lg) - 16.6355324)) <= EL + 1e-3
                assert g == r32 or near, (name, c, xv, g, r32, float(lg))
                continue
            # |d cdf| <= cdf (1 - cdf) |d logits| e^|d logits| for the logits error, plus expf (2 ulps), 1 + e and the
            # IEEE division (half an ulp each): 8 u relative; 2^-149 absolute for subnormal results
            with mpmath.workdps(R.DPS):
                bound = exact * ((1 - exact) * EL * np.exp(min(EL, 1.0)) + 8 * R.U32) + mpmath.mpf(2) ** -149
                assert abs(mpmath.mpf(float(g)) - exact) <= bound, (name, c, xv, g, float(exact), EL)
            n_checked += 1
        off += col.shape[0]
    # every row has at least the 26 unsaturated quantiles plus the steps inside the prior's width
    assert n_checked > 30 * len(rows)


# ----------------------------------------------------------------------------------------------------------------------
# 5. Gaussian quantiles and tables
# ----------------------------------------------------------------------------------------------------------------------
# CUDA documents normcdfinv (double) to at most 8 ulps (CUDA C++ Programming Guide, Mathematical Functions,
# double-precision table; the header refers to it with \note_accuracy_double).
NORMCDFINV_ULPS = 8
_NDTRI = {}


def mp_ndtri(xi):
    if xi not in _NDTRI:
        _NDTRI[xi] = R.ndtri(xi)
    return _NDTRI[xi]


def gaussian_bound(q, s, p, zf):
    """|fl(fl(normcdfinv(xi) s) + m) - (q s + m)| <= 8 ulp(q) s + ulp(p)/2 + ulp(z)/2: the documented quantile error
    scaled by s, then the two float64 roundings of scipy's `ndtri(q) * scale + loc` (p = the product, z = the sum)."""
    return NORMCDFINV_ULPS * np.spacing(abs(q)) * s + 0.5 * np.spacing(abs(p)) + 0.5 * np.spacing(abs(zf))


MEANS = np.array([3e-6, -2.5e-3, 0.1, -1.0, 12.0, -300.0, 1e3])
STDS = np.array([1e-6, 1e-3, 0.37, 1.0, 5.5, 100.0, 1e3])


@pytest.mark.parametrize("N", [10, 16, 20])
def test_gaussian_tables_against_mpmath(N):
    import vbq_b200
    C = len(MEANS)
    Q = (1 << (N + 1)) - 1
    table = vbq_b200.ops.build_code_points_gaussian(_dev(MEANS), _dev(STDS), N).cpu().numpy()
    xi = heap_xi(Q)
    z64 = vbq_b200.ops.gaussian_inverse_cdf(torch.from_numpy(xi).to(DEV).reshape(-1, 1).expand(-1, C).contiguous(),
                                            _dev(MEANS), _dev(STDS)).cpu().numpy()
    # the table is the float32 cast of the float64 quantile (quantizer.py:34): same routine, every entry
    assert np.array_equal(table, z64.astype(np.float32).T)
    hs = depth_sample(N, np.random.default_rng(N), 1000)
    bad = []
    for h in hs:
        q = mp_ndtri(float(xi[h]))
        for c in range(C):
            with mpmath.workdps(R.DPS):
                exact = q * mpmath.mpf(STDS[c]) + mpmath.mpf(MEANS[c])
                err = float(abs(mpmath.mpf(float(z64[h, c])) - exact))
            b = gaussian_bound(float(q), STDS[c], float(q) * STDS[c], z64[h, c])
            if not err <= b:
                bad.append(("f64", c, int(h), err, b))
            want32, dist = R.f32_correctly_rounded(exact)
            if table[c, h] != want32 and not dist * abs(float(exact)) <= b:
                bad.append(("f32", c, int(h), float(table[c, h]), float(want32)))
    assert not bad, bad[:5]


@pytest.mark.parametrize("N", [10, 11, 12])
def test_gaussian_codebook_codepoints(N):
    import vbq_b200
    std = 1.2329
    cb = vbq_b200.GaussianCodebook(std, N)
    Q = (1 << (N + 1)) - 1
    xi = heap_xi(Q)
    assert np.array_equal(cb.lengths, np.repeat(np.arange(N + 1), [1 << n for n in range(N + 1)]))
    hs = depth_sample(N, np.random.default_rng(100 + N), 1500)
    for h in hs:
        q = mp_ndtri(float(xi[h]))
        with mpmath.workdps(R.DPS):
            exact = q * mpmath.mpf(std)
            err = float(abs(mpmath.mpf(float(cb.codepoints[h])) - exact))
        assert err <= gaussian_bound(float(q), std, cb.codepoints[h], cb.codepoints[h]), (h, err)
    # the float32 search table is the cast of the float64 code points
    assert np.array_equal(cb._table[0].cpu().numpy(), cb.codepoints.astype(np.float32))


# ----------------------------------------------------------------------------------------------------------------------
# 6. searches that read the deep tables
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["fs0.5_c17", "shifted300_c5"])
@pytest.mark.parametrize("N", [11, 14, 20])
def test_quantize_on_deep_tables(name, N):
    import vbq_b200
    from vbq_b200 import ops
    if name == "fs0.5_c17":
        pr = H.make_prior(17, seed=36, factor_std=0.5)
        table = ops.build_code_points_learned(_dev(pr.packed()), N).cpu().numpy()
    else:
        z = zoo(name)
        pr = z["pr"]
        table = z["t20"][:, :(1 << (N + 1)) - 1].copy()
    C = pr.channels
    rows = 2000
    mu, sigma, _ = H.make_latents(pr, rows, seed=N, table=table)
    # a third of the rows with sigma small enough that the deepest depths win
    sigma[rows // 3: 2 * rows // 3] *= np.float32(1e-5)
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N)
    q.set_code_points(_dev(table))
    oq = O.QuantizerNP(C, N)
    oq.set_code_points(table, build_grids=N <= 14)
    lambs = [2.0 ** -8, 0.5]
    out = q.quantize(_dev(mu), _dev(sigma), lambs,
                     outputs=ops.OUT_ZHAT | ops.OUT_QIDX | ops.OUT_LEVEL | ops.OUT_BITS | ops.OUT_TOTALS)
    Zo, Bo = oq.compress_batch_channel_latents(mu, sigma, lambs)
    for i, l in enumerate(lambs):
        zk, lk = out["zhat"][i].cpu().numpy(), out["level"][i].cpu().numpy()
        assert np.array_equal(zk, Zo[l]), "lambda=%g: %d z_hat differ" % (l, (zk != Zo[l]).sum())
        assert np.array_equal(lk, Bo[l])
        assert np.array_equal(out["qidx"][i].cpu().numpy(), oq.sorted_index(Zo[l]))
        bits, dist = O.rd_totals(mu, sigma, zk, Bo[l])
        tot = out["totals"][i].cpu().numpy()
        assert tot[0] == bits
        assert abs(tot[3] - dist) <= 1e-6 * max(dist, 1.0)   # float64 sums of float32 terms
    # entropy-model bits are looked up at the same searchsorted index (quantizer.py:223-225), also on equal entries
    rng = np.random.default_rng(N)
    q.entropy_models = {l: rng.uniform(1.0, 30.0, (C, q.quantization_levels)).astype(np.float32) for l in lambs}
    out = q.quantize(_dev(mu), _dev(sigma), lambs, outputs=ops.OUT_QIDX | ops.OUT_TOTALS, entropy_bits=True)
    for i, l in enumerate(lambs):
        I = oq.sorted_index(Zo[l])
        assert np.array_equal(out["qidx"][i].cpu().numpy(), I)
        want = np.take_along_axis(q.entropy_models[l].T, I, axis=0)
        assert np.array_equal(out["em_bits"][i].cpu().numpy(), want)
        # float64 sum of the same float32 terms in another order: 1e-12 relative
        assert abs(out["totals"][i, 2].item() - want.sum(dtype=np.float64)) <= 1e-12 * want.sum(dtype=np.float64)
    if N > 14:
        return
    # the stand-alone bracket operator at the same depth against the literal edge-padded searchsorted
    left, right = q.get_all_N_bit_intervals(mu)
    lo, ro = oq.get_all_N_bit_intervals(mu)
    assert np.array_equal(left.cpu().numpy(), lo) and np.array_equal(right.cpu().numpy(), ro)


@pytest.mark.parametrize("name", ["fs0.5_c17", "shifted300_c5"])
def test_intervals_depth_20(name):
    import vbq_b200
    if name == "fs0.5_c17":
        pr = H.make_prior(17, seed=36, factor_std=0.5)
        table = vbq_b200.ops.build_code_points_learned(_dev(pr.packed()), N_MAX).cpu().numpy()
    else:
        z = zoo(name)
        pr, table = z["pr"], z["t20"]
    mu, _, _ = H.make_latents(pr, 500, seed=5, table=table)
    q = vbq_b200.ChannelwisePriorCDFQuantizer(pr.channels, N_MAX)
    q.set_code_points(_dev(table))
    oq = O.QuantizerNP(pr.channels, N_MAX)
    oq.set_code_points(table, build_grids=False)
    left, right = q.get_all_N_bit_intervals(mu)
    # the padded grids would be (C, 21, 2^20): the fast restatement has the same edge semantics (quantizer.py:57)
    lo, ro = oq.get_all_N_bit_intervals_fast(mu)
    assert np.array_equal(left.cpu().numpy(), lo) and np.array_equal(right.cpu().numpy(), ro)


# ----------------------------------------------------------------------------------------------------------------------
# 7. the float64 embedding search at its depth limit
# ----------------------------------------------------------------------------------------------------------------------
def _notebook_search(means, stds, beta, codepoints, bitlengths, chunk=2000):
    """ipynb:429-443 literally, beta as given: NumPy's own promotion decides the precision of (2 beta) stds^2
    (float32 for a Python float, float64 for a NumPy float64 under NumPy >= 2).  Exhaustive, first minimum."""
    m, s = means.ravel(), stds.ravel()
    idx = np.empty(m.size, dtype=np.int64)
    for i in range(0, m.size, chunk):
        se = (codepoints[None, :] - m[i:i + chunk, None]) ** 2
        wp = (2 * beta) * s[i:i + chunk, None] ** 2 * bitlengths[None, :]
        idx[i:i + chunk] = np.argmin(se + wp, axis=1)
    return codepoints[idx].astype(means.dtype).reshape(means.shape), idx


@pytest.mark.parametrize("N", [11, 12])
def test_embedding_f64_search_deep(N):
    import vbq_b200
    from vbq_b200 import ops
    from vbq_b200.word_embeddings import _pen_f32
    rng = np.random.default_rng(N)
    means = rng.normal(-0.08, 1.2329, (200, 100)).astype(np.float32)
    stds = np.exp(rng.normal(np.log(0.04), 1.5, means.shape)).astype(np.float32)
    cb = vbq_b200.GaussianCodebook(1.2329, N)
    means[0, :10] = cb.codepoints[[0, 1, 2, 5, 2 ** N - 1, 2 ** N, 2 ** (N + 1) - 2, 3, 4, 6]].astype(np.float32)
    means[1, :4] = [-1e4, 1e4, 0.0, -0.0]
    for beta in (0.37, np.float64(12.5)):
        got, _ = cb.compress_coordinates(means, stds, beta, exact=True)
        if isinstance(beta, float):
            want, widx = O.compress_coordinates(means, stds, beta, cb.codepoints, cb.lengths, chunk=2000)
        else:
            want, widx = _notebook_search(means, stds, beta, cb.codepoints, cb.lengths)
        assert np.array_equal(got, want), "beta=%r: %d optima differ" % (beta, (got != want).sum())
        per_level = np.arange(N + 1, dtype=np.float64)
        _, heap, level = ops.compress_coordinates_f64(_dev(means), _dev(stds), _dev(cb.codepoints), _dev(per_level),
                                                      float(beta), _pen_f32(beta), want_index=True, want_level=True)
        assert np.array_equal(heap.cpu().numpy().ravel(), widx.ravel())
        assert np.array_equal(level.cpu().numpy().ravel(), cb.lengths[widx.ravel()])


def test_embedding_f64_search_refuses_depth_13():
    import vbq_b200
    cb = vbq_b200.GaussianCodebook(1.0, 13)
    means = np.zeros((4, 16), dtype=np.float32)
    with pytest.raises(vbq_b200._lib.VbqError, match="max_codepoint_length=13 > 12"):
        cb.compress_coordinates(means, np.ones_like(means), 1.0, exact=True)
