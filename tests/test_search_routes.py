"""The search against the oracle on every route the dispatcher of vbq_quantize_hp (csrc/quantize.cu) can take for the
calls a fitted model makes: corrected code lengths with entropy-model bits, log-variance inputs, depths past 10, the
entropy-model fit at depth and the host pipeline.

Each launcher of the chain returns -1 when it does not apply, so which kernel serves a call depends on N, raw or
corrected lengths, the entropy model, the number of lambdas, C % 4, the sign of the penalties and the output set.  ROUTES
names, for every row, the kernel(s) the dispatcher picks; `test_route_is_the_named_kernel` checks the names with
torch.profiler, so a dispatch change cannot silently drop a route from the matrix.  The oracle comparisons are bit-exact:
z_hat, depth, code length, sorted index and entropy-model bits on every coordinate.

Log-variance inputs: every kernel derives sigma with one helper (sigma_of_logvar, csrc/tree.cuh), whose bits
ops.selftest_sigma_from_logvar returns.  Given those sigmas the oracle must reproduce the FLAG_LOGVAR run exactly, and
the helper itself is checked against the correctly rounded sqrt(exp(lv))."""
import functools
import re

import numpy as np
import pytest
import torch

from oracle import vbq_oracle as O
import vbq_test_helpers as H

pytestmark = pytest.mark.gpu

DEV = "cuda"
OUT_ALL = ("zhat", "qidx", "level", "bits")


def _dev(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def _sigma_k(lv):
    """The kernels' sigma of log-variances lv (host float32 array)."""
    from vbq_b200 import ops
    return ops.selftest_sigma_from_logvar(_dev(np.asarray(lv, dtype=np.float32))).cpu().numpy()


# ----------------------------------------------------------------------------------------------------------------------
# a. sigma = sqrt(exp(lv)) against the correctly rounded value
# ----------------------------------------------------------------------------------------------------------------------
F32_MAX = float(np.finfo(np.float32).max)
LN_OVERFLOW = np.log(F32_MAX)           # exp(lv) > FLT_MAX beyond this
LN_SUBNORMAL = np.log(2.0 ** -126)      # exp(lv) subnormal below this
LN_ZERO = np.log(2.0 ** -150)           # exp(lv) rounds to 0 below this


def _around(x, k=48):
    """Every float32 within k ulps of x (both signs of zero included)."""
    out = [np.float32(x)]
    for d in (np.float32(np.inf), np.float32(-np.inf)):
        f = np.float32(x)
        for _ in range(k):
            f = np.nextafter(f, d)
            out.append(f)
    return np.array(out + ([np.float32(-0.0)] if x == 0 else []), dtype=np.float32)


def _f32_ulp(e):
    """Spacing of float32 at the (positive, real) value e: 2^(max(floor(log2 e), -126) - 23)."""
    with np.errstate(divide="ignore"):
        ex = np.floor(np.log2(np.maximum(e, 2.0 ** -1000)))
    return np.exp2(np.maximum(ex, -126.0) - 23.0)


def _rn_f32_exact(lv):
    """Correctly rounded float32 of sqrt(exp(lv)) for finite float32 lv: float64 sqrt(exp(.)) rounded once, and mpmath
    where the float64 value lies within 2^-20 float32 ulp of a float32 rounding boundary (the midpoint between two
    float32 neighbours), where float64's own error could decide the rounding."""
    import mpmath
    x = lv.astype(np.float64)
    with np.errstate(over="ignore"):
        s64 = np.sqrt(np.exp(x))
    ref = s64.astype(np.float32)
    ok = np.isfinite(s64) & (s64 > 0)
    lo = np.where(ok, ref, 0).astype(np.float32)
    lo = np.where(lo.astype(np.float64) > s64, np.nextafter(lo, np.float32(-np.inf)), lo)   # float32 below s64
    hi = np.nextafter(lo, np.float32(np.inf))
    mid = 0.5 * (lo.astype(np.float64) + hi.astype(np.float64))
    near = ok & (np.abs(s64 - mid) <= (hi.astype(np.float64) - lo.astype(np.float64)) * 2.0 ** -20)
    mpmath.mp.prec = 200
    for j in np.flatnonzero(near):
        exact = mpmath.sqrt(mpmath.exp(mpmath.mpf(float(x[j]))))
        ref[j] = hi[j] if exact > mpmath.mpf(float(mid[j])) else lo[j]
        assert exact != mpmath.mpf(float(mid[j]))     # sqrt(exp(x)) is transcendental for float x != 0
    return ref, int(near.sum())


def test_sigma_of_logvar_against_correctly_rounded():
    """Bound.  CUDA documents expf with at most 2 ulp error and sqrtf as correctly rounded (CUDA C Programming Guide,
    mathematical functions, non-fast-math build).  So the kernel's sigma is RN(sqrt(E)) for some E with
    |E - exp(lv)| <= 2 ulp32(exp(lv)).  As sqrt and RN are monotone, sigma lies in [RN(sqrt(e - 2u)), RN(sqrt(e + 2u))]
    with e = exp(lv), u = ulp32(e): checked on every input.  Where e is a normal float32 this gives a plain ulp bound:
    E = e (1 + d), |d| <= 2^-22, so sqrt(E) = sqrt(e) (1 + d/2 + O(d^2)) lies within 2^-23 sqrt(e) < 2 ulp of sqrt(e)
    (ulp32(s) > 2^-24 s); one correct rounding adds 1/2 ulp and the correctly rounded reference is 1/2 ulp from the
    exact value, so the two differ by less than 3 ulp, i.e. by at most 2 ulp.  In the subnormal range of exp(lv) the 2 ulp
    are absolute (2^-148) and only the interval applies; beyond log(FLT_MAX) the interval reaches inf.
    Special values (+-0, +-inf, NaN) must give what NumPy's np.exp(lv) ** 0.5 gives."""
    rng = np.random.default_rng(20)
    uni = rng.uniform(-110.0, 95.0, 4_000_000).astype(np.float32)
    edges = np.concatenate([_around(LN_OVERFLOW), _around(LN_SUBNORMAL), _around(LN_ZERO), _around(-149 * np.log(2)),
                            _around(0.0, 8)]).astype(np.float32)
    lv = np.concatenate([uni, edges])
    got = _sigma_k(lv)
    ref, n_mp = _rn_f32_exact(lv)

    # the interval of the documented bound, evaluated in float64 and widened by 2^-50 relative before its one rounding
    e = np.exp(lv.astype(np.float64))
    u = _f32_ulp(e)
    with np.errstate(over="ignore"):
        lo = (np.sqrt(np.maximum(e - 2 * u, 0.0)) * (1 - 2.0 ** -50)).astype(np.float32)
        hi = (np.sqrt(e + 2 * u) * (1 + 2.0 ** -50)).astype(np.float32)
    hi = np.where(e + 2 * u >= 2.0 ** 128, np.float32(np.inf), hi)
    lo = np.where(e - 2 * u >= 2.0 ** 128, np.float32(np.inf), lo)
    bad = ~((got >= lo) & (got <= hi))
    assert not bad.any(), "sigma outside the expf/sqrtf bound at lv=%s: got %s, want [%s, %s]" % (
        lv[bad][:5], got[bad][:5], lo[bad][:5], hi[bad][:5])
    normal = (e >= 2.0 ** -126) & (e <= F32_MAX)
    d_ulp = np.abs(got[normal].view(np.int32).astype(np.int64) - ref[normal].view(np.int32).astype(np.int64))
    assert d_ulp.max() <= 2, d_ulp.max()

    special = np.array([0.0, -0.0, np.inf, -np.inf, np.nan], dtype=np.float32)
    want = np.exp(special) ** np.float32(0.5)
    assert np.array_equal(_sigma_k(special), want, equal_nan=True)

    # how often the kernels' sigma differs from the reference's float32 NumPy sigma (quantizer.py:93, :198)
    npy = np.exp(uni) ** np.float32(0.5)
    mid = (uni > -20) & (uni < 20)
    n = len(uni)
    print("sigma_of_logvar: %d of %d (%.3g %%) differ from NumPy's float32 exp(lv) ** 0.5 over U(-110, 95), "
          "%.3g %% over (-20, 20); %.3g %% from the correctly rounded value; max %d ulp (normal range); %d resolved "
          "with mpmath" % ((got[:n] != npy).sum(), n, 100 * (got[:n] != npy).mean(), 100 * (got[:n][mid] != npy[mid]).mean(),
                           100 * (got[:n] != ref[:n]).mean(), d_ulp.max(), n_mp))


# ----------------------------------------------------------------------------------------------------------------------
# b / c. the route matrix
# ----------------------------------------------------------------------------------------------------------------------
_QK = r"vbq_quantize_kernel<%s, (true|false), true, %s, true, %s, 2, 640>"   # MODE, PRUNE, TOTALS, DEEP, EXTRAS, NT
DEEP_REF = _QK % (0, "true", 0)              # deep tables: reference mode, depths 11..N from global memory

# id: (N, C, L, mode, correction style, outputs, the kernel(s) the dispatcher launches)
ROUTES = {
    "tma_raw":            (10, 48, 1, "raw", None, ("zhat", "level"), [r"vbq_bisect_tma_kernel<false, 0,"]),
    "cpasync_raw":        (10, 21, 1, "raw", None, OUT_ALL, [r"vbq_bisect_kernel<(true|false), true, 10,"]),
    "bisect_sweep_raw":   (10, 48, 4, "raw", None, OUT_ALL, [r"vbq_bisect_sweep_kernel<true, true,"]),
    "tma_both_em":        (10, 48, 1, "em", "fitted", ("zhat", "bits"),
                           [r"vbq_bisect_tma_kernel<true, 2,", r"em_gather_kernel<true, true>"]),
    "both_sweep_em":      (10, 48, 3, "em", "noisy", OUT_ALL,
                           [r"vbq_both_sweep_kernel<true, true, false,", r"em_gather_kernel<true, false>"]),
    "bracket_sweep_neg":  (10, 48, 3, "em", "negative", OUT_ALL, [r"vbq_sweep_kernel<false, true,"]),
    "strict_nt10":        (10, 21, 1, "em", "fitted", OUT_ALL, [_QK % (1, "false", 10)]),
    "bracket_sweep_c21":  (10, 21, 3, "em", "noisy", OUT_ALL, [r"vbq_sweep_kernel<false, true,"]),
    "strict_nt0":         (6, 16, 1, "em", "noisy", OUT_ALL, [_QK % (1, "false", 0)]),
    "both_sweep_n6":      (6, 16, 3, "corrected", "fitted", OUT_ALL, [r"vbq_both_sweep_kernel<true, true, false,"]),
    "deep_n13_l1":        (13, 17, 1, "em", "fitted", OUT_ALL, [DEEP_REF]),
    "deep_n13_l3":        (13, 17, 3, "em", "noisy", OUT_ALL, [DEEP_REF]),
    "deep_n16_l2":        (16, 20, 2, "em", "fitted", OUT_ALL, [DEEP_REF]),
    "deep_bisect_raw":    (13, 17, 2, "raw", None, OUT_ALL, [r"vbq_bisect_kernel<(true|false), true, -1,"]),
    "deep_shifted300":    (14, 5, 2, "em", "noisy", OUT_ALL, [DEEP_REF]),
}
SWEEPS = ("vbq_sweep_kernel", "vbq_both_sweep_kernel", "vbq_bisect_sweep_kernel")


def _corrections(style, rng, L, C, N):
    """R_lambda[c, n] (L, C, N+1) in the shapes of test_gpu_tma._lengths: "fitted" (almost monotone, dips at shallow
    depths), "noisy" (every depth can have a cheaper deeper neighbour) and "negative" (noisy shifted below zero, so that
    some penalties are negative)."""
    n = np.arange(N + 1, dtype=np.float64)[None, None, :]
    if style == "fitted":
        R = 5.0 + 0.08 * (n - 3.0) ** 2 + rng.normal(0.0, 0.35, size=(L, C, N + 1))
    else:
        R = rng.gamma(2.0, 2.0, size=(L, C, N + 1)) - (4.0 + n if style == "negative" else 0.0)
    return R.astype(np.float32)


@functools.lru_cache(maxsize=None)
def _setup(rid):
    """Quantizer, oracle, latents and lambdas of one row (cached: the matrix and the route check share them)."""
    import vbq_b200
    from vbq_b200 import ops
    N, C, L, mode, style, outs, _ = ROUTES[rid]
    seed = 1000 + sum(map(ord, rid))
    if rid == "deep_shifted300":
        import test_prior_tables as PT
        z = PT.zoo("shifted300_c5")
        pr, table = z["pr"], z["t20"][:, :(1 << (N + 1)) - 1].copy()
    else:
        pr = H.make_prior(C, seed=seed)
        table = ops.build_code_points_learned(_dev(pr.packed()), N).cpu().numpy()
    rows = 1200 if N > 10 else 2400 + C % 7
    mu, _, lv = H.make_latents(pr, rows, seed + 1, table=table)
    rng = np.random.default_rng(seed + 2)
    srt = np.sort(table, axis=1)
    on = srt[np.arange(C)[None, :], rng.integers(0, srt.shape[1], (rows, C))]
    mu = np.where(rng.random((rows, C)) < 1 / 3, on, mu).astype(np.float32)      # a third exactly on code points
    mu[:16] = H.make_latents(pr, 16, seed + 1, table=table)[0]                    # keep the edge rows
    lambs = [float(l) for l in (2.0 ** np.linspace(-6, 3, L) if L > 1 else [0.5])]
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N)
    q.set_code_points(_dev(table))
    oq = O.QuantizerNP(C, N)
    oq.set_code_points(table, build_grids=False)
    if mode != "raw":
        R = _corrections(style, rng, L, C, N)
        rcl = {l: R[i] for i, l in enumerate(lambs)}
        q.raw_code_length_entropy_models = rcl
        oq.raw_code_length_entropy_models = rcl
    if mode == "em":
        em = {l: rng.gamma(2.0, 3.0, size=(C, q.quantization_levels)).astype(np.float32) for l in lambs}
        q.entropy_models = em
        oq.entropy_models = em
    sigma = np.exp(lv) ** np.float32(0.5)
    return dict(q=q, oq=oq, mu=mu, lv=lv, sigma=sigma, sigma_k=_sigma_k(lv), lambs=lambs, outs=outs, em=mode == "em")


def _kernel_run(s, scales, logvar):
    from vbq_b200 import ops
    bits = {"zhat": ops.OUT_ZHAT, "qidx": ops.OUT_QIDX, "level": ops.OUT_LEVEL, "bits": ops.OUT_BITS}
    outputs = functools.reduce(lambda a, k: a | bits[k], s["outs"], ops.OUT_TOTALS)
    out = s["q"].quantize(_dev(s["mu"]), _dev(scales), s["lambs"], logvar=logvar, outputs=outputs, entropy_bits=s["em"])
    keep = s["outs"] + (("em_bits",) if s["em"] else ()) + ("totals",)
    return {k: out[k].cpu().numpy() for k in keep}


def _expected(s, sigma):
    """The oracle's per-coordinate outputs and float64 totals for the given sigma."""
    oq, mu, lambs = s["oq"], s["mu"], s["lambs"]
    Zo, Bo, det = oq.compress_batch_channel_latents(mu, sigma, lambs, details=True)
    res = []
    for l in lambs:
        I = oq.sorted_index(Zo[l])
        level = det[l]["level"].astype(np.int32)
        bits = Bo[l].astype(np.float32)
        eb = np.take_along_axis(oq.entropy_models[l].T, I, axis=0) if s["em"] else None
        _, dist = O.rd_totals(mu, sigma, Zo[l], bits)
        tot = [float(level.sum(dtype=np.int64)), float(bits.sum(dtype=np.float64)),
               float(eb.sum(dtype=np.float64)) if s["em"] else None, dist]
        res.append(dict(zhat=Zo[l], level=level, bits=bits, qidx=I.astype(np.int32), em_bits=eb, totals=tot))
    return res


def _check_against_oracle(rid, got, want):
    rel = 2e-6 if any(k in "".join(ROUTES[rid][6]) for k in SWEEPS) else 1e-6
    for i, w in enumerate(want):
        for k in got:
            if k == "totals":
                continue
            assert np.array_equal(got[k][i], w[k]), "%s, lambda %d: %s differs on %d coordinates" % (
                rid, i, k, (got[k][i] != w[k]).sum())
        t = got["totals"][i]
        assert t[0] == w["totals"][0], (rid, i, t, w["totals"])            # depth sums are integers: exact
        for j in (1, 2, 3):
            if w["totals"][j] is None:
                continue
            # DESIGN §6 (C): float64 sums of float32 terms rounded to 2^-24 (sweeps: 2^-16 tiles), with an absolute floor
            assert abs(t[j] - w["totals"][j]) <= rel * abs(w["totals"][j]) + 5e-5 * (rel / 1e-6), (rid, i, j, t, w["totals"])


@pytest.mark.parametrize("rid", list(ROUTES))
def test_route_matrix_against_oracle(rid):
    """Given sigma, and given log-variances with FLAG_LOGVAR, every output of the route equals the oracle's on the
    sigma the kernel used (np.exp(lv) ** 0.5, resp. the kernels' own sigma of lv); the FLAG_LOGVAR run equals the run on
    the kernels' sigma exactly, totals included."""
    s = _setup(rid)
    got_s = _kernel_run(s, s["sigma"], False)
    got_lv = _kernel_run(s, s["lv"], True)
    got_k = _kernel_run(s, s["sigma_k"], False)
    assert got_lv.keys() == got_k.keys()
    for k in got_lv:
        assert np.array_equal(got_lv[k], got_k[k]), (rid, k)
    want = _expected(s, s["sigma"])
    _check_against_oracle(rid, got_s, want)
    if not np.array_equal(s["sigma_k"], s["sigma"]):
        want = _expected(s, s["sigma_k"])
    _check_against_oracle(rid, got_lv, want)


@pytest.mark.parametrize("rid", list(ROUTES))
def test_route_is_the_named_kernel(rid):
    """The dispatcher launches exactly the kernels ROUTES names for the row (read from the launchers' -1 conditions)."""
    from torch.profiler import ProfilerActivity, profile
    s = _setup(rid)
    _kernel_run(s, s["lv"], True)                      # warm: shared-memory attributes, cached tables
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _kernel_run(s, s["lv"], True)
        torch.cuda.synchronize()
    events = list(prof.events())
    names = [e.name for e in events if str(e.device_type).endswith("CUDA")] + \
        [k.name for e in events for k in getattr(e, "kernels", [])]
    names = sorted({n for n in names if re.search(r"vbq_|em_gather", n)})
    pats = ROUTES[rid][6]
    assert names and all(any(re.search(p, n) for p in pats) for n in names) and \
        all(any(re.search(p, n) for n in names) for p in pats), (rid, names, pats)


# ----------------------------------------------------------------------------------------------------------------------
# d. the entropy-model fit at depth (torch.bincount branch of _histograms), in several row chunks
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N", [11, 13])
def test_entropy_model_fit_at_depth(N):
    import vbq_b200
    from vbq_b200 import ops
    C, rows, lambs = 17, 1500, [2.0 ** -5, 0.5, 4.0]
    pr = H.make_prior(C, seed=60 + N)
    table = ops.build_code_points_learned(_dev(pr.packed()), N).cpu().numpy()
    mu, sigma, lv = H.make_latents(pr, rows, 61 + N, table=table)
    sk = _sigma_k(lv)

    def fit_kernel(stds):
        q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N)
        q.set_code_points(_dev(table))
        # at most 400 rows per chunk: four chunks of the search and of the histograms
        q._histograms = functools.partial(q._histograms, max_chunk_symbols=len(lambs) * C * 400)
        q.build_entropy_models_from_latents(mu, None if stds is not None else lv, lambs, 1, posterior_stds=stds)
        return q

    def fit_oracle(stds):
        oq = O.QuantizerNP(C, N)
        oq.set_code_points(table, build_grids=False)
        oq.build_entropy_models_from_latents(mu, lv, lambs, 1, posterior_stds=stds)
        return oq

    for qk, qo in ((fit_kernel(sigma), fit_oracle(None)), (fit_kernel(None), fit_oracle(sk))):
        for l in lambs:
            assert np.array_equal(qk.raw_code_length_entropy_models[l], qo.raw_code_length_entropy_models[l]), (N, l)
            assert np.array_equal(qk.entropy_models[l], qo.entropy_models[l]), (N, l)


# ----------------------------------------------------------------------------------------------------------------------
# e. the host pipeline (NumPy in, NumPy out: vbq_quantize_host) in several chunks against the oracle
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("N,C,n_lambda,corrected", [(10, 24, 1, False), (10, 24, 16, False), (10, 24, 1, True),
                                                    (10, 24, 3, True), (13, 17, 3, True)])
def test_host_pipeline_against_oracle(N, C, n_lambda, corrected):
    """compress_batch_channel_latents and compress_latents on NumPy arrays, 300-row chunks (the last one ragged).  With
    16 lambdas at N = 10, and with corrected lengths, the pipeline has no host copy of the penalties and runs other
    kernels than the device path; its totals, accumulated chunk by chunk, must still match the device path's (1e-12 when
    both run the same kernel family, else the tolerance between kernel families, DESIGN §6 (C))."""
    import vbq_b200
    from vbq_b200 import ops
    rows = 1111
    pr = H.make_prior(C, seed=80 + N + n_lambda)
    table = ops.build_code_points_learned(_dev(pr.packed()), N).cpu().numpy()
    mu, sigma, lv = H.make_latents(pr, rows, 81 + n_lambda, table=table)
    sk = _sigma_k(lv)
    lambs = [float(l) for l in (2.0 ** np.linspace(-8, 6, n_lambda) if n_lambda > 1 else [0.25])]
    rng = np.random.default_rng(n_lambda)
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N)
    q._HOST_CHUNK_ROWS = 300
    q.set_code_points(_dev(table))
    oq = O.QuantizerNP(C, N)
    oq.set_code_points(table, build_grids=False)
    em = {l: rng.gamma(2.0, 3.0, size=(C, q.quantization_levels)).astype(np.float32) for l in lambs}
    q.entropy_models = oq.entropy_models = em
    if corrected:
        R = _corrections("fitted", rng, n_lambda, C, N)
        q.raw_code_length_entropy_models = oq.raw_code_length_entropy_models = {l: R[i] for i, l in enumerate(lambs)}

    Zk, Bk = q.compress_batch_channel_latents(mu, sigma, lambs)
    Zo, Bo = oq.compress_batch_channel_latents(mu, sigma, lambs)
    for l in lambs:
        assert isinstance(Zk[l], np.ndarray) and np.array_equal(Zk[l], Zo[l]) and np.array_equal(Bk[l], Bo[l]), l
    shape = (1, 11, 101, C)
    out = q.compress_latents(mu.reshape(shape), lv.reshape(shape), lambs)
    want = oq.compress_latents(mu.reshape(shape), None, lambs, posterior_stds=sk)
    for l in lambs:
        for key in ("Z_hat", "raw_num_bits", "num_bits_cl", "num_bits"):
            if key in want and l in want[key]:
                assert np.array_equal(out[key][l], want[key][l]), (key, l)

    # totals of the chunked pipeline (VBQ_FLAG_ACCUMULATE_TOTALS) against the one-call device path
    outs = ops.OUT_ZHAT | ops.OUT_LEVEL | ops.OUT_BITS | ops.OUT_TOTALS
    h = q._quantize_host(mu, lv, lambs, outs, logvar=True, entropy_bits=True)
    d = q.quantize(_dev(mu), _dev(lv), lambs, logvar=True, outputs=outs, entropy_bits=True)
    for k in ("zhat", "level", "bits", "em_bits"):
        assert torch.equal(h[k], d[k].cpu()), k
    th, td = h["totals"], d["totals"].cpu()
    assert torch.equal(th[:, 0], td[:, 0])
    # one lambda, or N > 10: the pipeline and the device path run the same kernel (the single-lambda launchers do not
    # need the host copy at these output sets); otherwise the device path takes the both-ends sweep
    rel = 1e-12 if n_lambda == 1 or N > 10 else 2e-6
    assert torch.allclose(th, td, rtol=rel, atol=0), (th, td)
