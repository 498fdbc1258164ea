"""Query scores against VBQE blobs (vbq_rans_shared_row_scores, CompressedEmbedding.scores / topk): CPU tests of the
NumPy reference (an exact fma32, a hand-worked answer, the work split), ABI and argument validation; GPU tests of the
kernel against the reference bit for bit, of topk against the exact ranking, of the full 1 M x 300 plane, of topk's
workspace and of a corrupt group range."""
import ctypes
import random
from fractions import Fraction

import numpy as np
import pytest
import torch

import embedding_scores_reference as S
from vbq_b200 import serialize

F32 = np.float32


def _round_f32(x: Fraction) -> np.float32:
    """The float32 nearest to the rational x, ties to even, overflow to inf (IEEE round-to-nearest)."""
    if x == 0:
        return F32(0.0)
    big = Fraction(2) ** 128 - Fraction(2) ** 103              # the midpoint between FLT_MAX and 2^128
    if abs(x) >= big:
        return F32(np.inf) if x > 0 else F32(-np.inf)
    c = F32(float(x))
    if np.isinf(c):
        c = np.copysign(F32(S.F32_MAX), c).astype(F32)
    with np.errstate(over="ignore"):
        cands = {c, np.nextafter(c, F32(np.inf)), np.nextafter(c, F32(-np.inf))}
    cands = [v for v in cands if np.isfinite(v)]
    best = min(cands, key=lambda v: (abs(Fraction(float(v)) - x), int(np.array(v).view(np.int32)) & 1))
    return F32(best)


def _fma_exact(a, b, c):
    r = _round_f32(Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c)))
    return F32(0.0) if r == 0 else r          # the emulation's sign of an exact zero follows IEEE; compared by value


def _same_bits(a, b):
    a, b = np.asarray(a, F32), np.asarray(b, F32)
    return np.array_equal(a.view(np.int32), b.view(np.int32)) or (
        np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[~np.isnan(a)].view(np.int32),
                                                                    b[~np.isnan(b)].view(np.int32)))


# ---------------------------------------------------------------------------------------------------------------------
# the reference
# ---------------------------------------------------------------------------------------------------------------------
def test_fma32_matches_exact_rational_arithmetic():
    rng = np.random.default_rng(1)
    cases = []
    for scale in (1.0, 1e-20, 1e-38, 1e19, 1e-44):
        a = (rng.standard_normal(300) * scale).astype(F32)
        b = (rng.standard_normal(300)).astype(F32)
        c = (rng.standard_normal(300) * scale).astype(F32)
        cases += list(zip(a, b, c))
    one = F32(1.0)
    a = F32(1 + 2 ** -23)
    b = F32(2 ** -24 * (1 - 2 ** -23))
    # float64 sums that land exactly on a float32 midpoint with a non-zero error on either side
    cases += [(a, b, F32(1 + 2 ** -23)), (a, -b, F32(1 + 3 * 2 ** -23)), (-a, b, F32(-(1 + 2 ** -23))),
              (a, -b, F32(-(1 + 2 ** -23)))]
    tiny = F32(2 ** -75)
    cases += [(tiny, F32(1.5 * 2 ** -75), F32(0)), (tiny, F32(1.5 * 2 ** -75), F32(2 ** -149)),       # subnormals
              (F32(2 ** -149), F32(0.5), F32(0)), (F32(2 ** -149), F32(1.5), F32(-2 ** -149)),
              (F32(2 ** 64), F32(2 ** 64), F32(0)), (F32(S.F32_MAX), one, F32(S.F32_MAX)),           # overflow
              (F32(S.F32_MAX), one, F32(2 ** 103)), (F32(S.F32_MAX), one, F32(2 ** 102)),
              (F32(-S.F32_MAX), F32(2), F32(S.F32_MAX)), (F32(3), F32(5), F32(-15))]
    for a, b, c in cases:
        got = S.fma32(a, b, c)
        want = _fma_exact(a, b, c)
        assert got == want or (np.isinf(got) and got == want), (a, b, c, got, want)
        assert got.dtype == F32
    # the vectorised form agrees with the scalar one
    a, b, c = (np.array([x[i] for x in cases], F32) for i in range(3))
    assert _same_bits(S.fma32(a, b, c), [S.fma32(x, y, z) for x, y, z in zip(a, b, c)])
    # a naive float64 product-sum rounded once to float32 gets the first midpoint case wrong
    a, b, c = F32(1 + 2 ** -23), F32(2 ** -24 * (1 - 2 ** -23)), F32(1 + 2 ** -23)
    assert F32(np.float64(a) * np.float64(b) + np.float64(c)) != S.fma32(a, b, c)


def test_reference_known_answer():
    """D = 5; row 0 = (1, 2, 3, 4, 5), row 1 = 0; q = (1, 1, 1, 1, 2).  a0 = 1 + 5 * 2 = 11, a1 = 2, a2 = 3, a3 = 4, so
    dot = (11 + 2) + (3 + 4) = 20; zz = (1 + 25) + 4 + 9 + 16 = 55, qq = (1 + 4) + 1 + 1 + 1 = 8, cosine = 20 /
    (sqrtf(55) sqrtf(8)); the zero row has dot 0 and cosine 0 (zero denominator)."""
    Z = np.array([[1, 2, 3, 4, 5], [0, 0, 0, 0, 0]], F32)
    Q = np.array([[1, 1, 1, 1, 2]], F32)
    assert S.scores(Z, Q, "dot").tolist() == [[20.0, 0.0]]
    cos = S.scores(Z, Q, "cosine")
    assert cos[0, 0] == F32(20) / (np.sqrt(F32(55)) * np.sqrt(F32(8))) and cos[0, 1] == 0
    # the order matters: a[d % 4] sums 1e8 and -1e8 in d = 0 and 4 before the 1 of d = 8 joins them
    Z = np.array([[1e8, 0, 0, 0, -1e8, 0, 0, 0, 1]], F32)
    assert S.scores(Z, np.ones((1, 9), F32))[0, 0] == 1.0


@pytest.mark.parametrize("D", [1, 7, 32, 33, 300])
@pytest.mark.parametrize("n_rows,seg,K", [(97, 1, 1), (97, 3, 2), (400, 40, 5), (400, 10 ** 6, 16), (1000, 64, 64),
                                          (1000, 7, 100)])
def test_work_split_scores_every_row_once(D, n_rows, seg, K):
    n = n_rows * D
    rows = -(-n // 32)
    S_ = max(1, min(seg, rows))
    k = min(K, S_)
    C1 = (S_ - 1) // k + 1
    T = -(-rows // S_) * C1
    rng = random.Random(D + n_rows + seg + K)
    ranges = [(0, n_rows), (0, 0), (5, 6), (n_rows - 1, n_rows)] + [tuple(sorted(rng.sample(range(n_rows + 1), 2)))
                                                                    for _ in range(4)]
    for ipw in (1, 2, 5):
        for a, b in ranges:
            cnt = np.zeros(n_rows, np.int64)
            for w in range(-(-T // ipw)):
                lo, hi = S.warp_rows(w, D, n, seg, K, ipw, a, b)
                cnt[lo:hi] += 1
                assert all(S.owner(e, D, S_, k, ipw) == w for e in range(lo, hi))
            assert (cnt[a:b] == 1).all() and cnt[:a].sum() == 0 and cnt[b:].sum() == 0, (ipw, a, b)
    # rows whose coder rows cross a segment boundary are scored by the warp of the first segment's interval
    cross = [e for e in range(n_rows) if (e * D // 32) // S_ != ((e + 1) * D - 1) // 32 // S_]
    for e in cross[:20]:
        assert S.owner(e, D, S_, k, 1) == S.interval(e * D // 32, S_, k)


# ---------------------------------------------------------------------------------------------------------------------
# ABI and argument validation (no device)
# ---------------------------------------------------------------------------------------------------------------------
def test_scores_abi_validation_needs_no_gpu():
    from vbq_b200 import _lib
    lib = _lib.load()
    mq = lib.vbq_rans_shared_score_max_queries
    assert mq(1) == 64 and mq(300) == 64 and mq(0) == 0 and mq(-5) == 0 and mq(10 ** 6) == 0
    assert 0 < mq(2000) < 64 and mq(2000) >= mq(2001)
    p, odd = ctypes.c_void_p(16), ctypes.c_void_p(18)
    fn = lib.vbq_rans_shared_row_scores

    def call(n=1000, seg=4, N=10, P=16, K=1, offs=p, D=10, lo=0, hi=100, q=p, B=3, metric=0, cp=p, out=p, words=p):
        return fn(words, 10, p, n, seg, N, P, p, K, offs, p, D, lo, hi, q, B, metric, cp, out, p, None)
    assert call(N=11) == 3
    assert call(P=11) == 2
    assert call(K=0) == 2
    assert call(D=0) == 2 and call(D=3) == 2                         # D < 1, D not dividing n
    assert call(lo=-1) == 2 and call(lo=5, hi=4) == 2 and call(hi=101) == 2
    assert call(B=-1) == 2 and call(B=65) == 2 and call(metric=2) == 2
    assert call(D=40_000, n=10 ** 6, B=1, hi=25) == 2                # a query of 40,000 floats: none fits
    assert call(q=None) == 1 and call(cp=None) == 1 and call(out=None) == 1 and call(offs=None) == 1
    assert call(words=None) == 1
    assert call(q=odd) == 7 and call(out=odd) == 7
    assert call(n=2 ** 36, seg=2 ** 31, D=2 ** 4, hi=10) == 2


def _bare(shape):
    from vbq_b200 import CompressedEmbedding
    ce = object.__new__(CompressedEmbedding)           # the attributes read before the first device operation
    ce._shape, ce._D, ce.device = shape, int(np.prod(shape[1:])), torch.device("cuda")
    return ce


def test_scores_and_topk_argument_errors_need_no_gpu():
    ce = _bare((200, 30))
    good = np.zeros((2, 30), np.float32)
    for f in (ce.scores, lambda q, **kw: ce.topk(q, 5, **kw)):
        for q in (np.zeros((2, 30), np.int64), [[1, 2, 3] * 10], torch.zeros(2, 30, dtype=torch.int32),
                  torch.zeros(30, dtype=torch.bool)):
            with pytest.raises(TypeError):
                f(q)
        for q in (np.zeros((2, 31), np.float32), np.zeros(29, np.float32), np.zeros((2, 3, 10), np.float32)):
            with pytest.raises(ValueError):
                f(q)
        with pytest.raises(ValueError, match="metric"):
            f(good, metric="l2")
    for a, b in ((-1, 5), (5, 4), (0, 201), (1.5, 3), (True, 3)):
        with pytest.raises(IndexError):
            ce.scores(good, a, b)
    with pytest.raises(ValueError):
        _bare((10, 40_000)).scores(np.zeros(40_000, np.float32))                # no query of 40,000 floats fits
    with pytest.raises(ValueError):
        ce.topk(good, 2.5)
    with pytest.raises(TypeError):
        ce.topk(good, 3, exclude=np.zeros((2, 3), np.float32))
    with pytest.raises(ValueError):
        ce.topk(good, 3, exclude=np.zeros((3, 3), np.int64))


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _posteriors(shape, seed):
    rng = np.random.default_rng(seed)
    means = (rng.standard_normal(shape) * 1.2329 - 0.08).astype(np.float32)
    stds = np.exp(rng.standard_normal(shape) * 0.7 + np.log(0.04)).astype(np.float32)
    return means, stds


def _queries(rng, B, D):
    """Random queries, with a zero query (cosine with a zero denominator), huge values (products overflow to inf) and
    subnormals where the batch has room."""
    q = rng.standard_normal((B, D)).astype(np.float32)
    if B >= 3:
        q[1] = 0
        q[2, ::2] = 1e-41
    if B >= 4:
        q[3, 0] = 3e38
    if B >= 5:
        q[4, -1] = -3e38
    return q


def _check(ce, full_np, q, metric, start, stop, ref=None):
    got = ce.scores(torch.from_numpy(q.reshape((q.shape[0],) + ce.shape[1:])).cuda(), start, stop, metric)
    assert got.dtype == torch.float32 and tuple(got.shape) == (q.shape[0], stop - start)
    want = S.scores(full_np[start:stop], q, metric) if ref is None else ref[:, start:stop]
    assert _same_bits(got.cpu().numpy(), want), (metric, start, stop)
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("D", [1, 7, 32, 33, 300])
def test_gpu_scores_match_reference(D):
    import vbq_b200
    cb = vbq_b200.GaussianCodebook(1.2356, 10)
    V = {1: 5001, 7: 1001, 32: 301, 33: 297, 300: 101}[D]
    shape = (V,) if D == 1 else (V, D)
    n = V * D
    m, s = _posteriors(shape, D)
    rng = np.random.default_rng(D)
    q3 = _queries(rng, 5, D)[[0, 1, 2]] if D > 1 else _queries(rng, 3, D)
    mq = vbq_b200.ops.rans_shared_score_max_queries(D)
    for seg in (1, 3, 10 ** 6):
        blob = cb.compress_to_bytes(m, s, [1.0], seg_rows=seg)[1.0]
        full = cb.decompress_from_bytes(blob).reshape(V, D).cpu().numpy()
        Sg = serialize.shared_seg_rows(n, seg)
        refs = {mt: S.scores(full, q3, mt) for mt in ("dot", "cosine")}
        for K in (1, 5, None, Sg + 1):
            ce = vbq_b200.CompressedEmbedding(blob, checkpoint_rows=K)
            for mt in ("dot", "cosine"):
                for a, b in ((0, V), (5, 5), (7, 8), (3, V - 2), (V - 1, V)):
                    _check(ce, full, q3, mt, a, b, refs[mt])
    # batch sizes around the launch's query tile, on one blob
    ce = vbq_b200.CompressedEmbedding(blob, checkpoint_rows=5)
    for B in (1, mq, mq + 1, 200):
        q = _queries(rng, B, D)
        for mt in ("dot", "cosine"):
            _check(ce, full, q, mt, 0, V)
    # a single query of shape shape[1:], as a list of floats from the host
    one = q3[0].reshape(shape[1:])
    got = ce.scores(one.tolist() if D > 1 else float(one), 0, V)
    assert _same_bits(got.cpu().numpy(), refs["dot"][:1])


@pytest.mark.gpu
def test_gpu_scores_are_independent_of_k_blocks_and_runs():
    import vbq_b200
    cb = vbq_b200.GaussianCodebook(1.2356, 10)
    V, D = 3000, 50
    m, s = _posteriors((V, D), 11)
    blob = cb.compress_to_bytes(m, s, [2.0], seg_rows=64)[2.0]
    q = torch.from_numpy(_queries(np.random.default_rng(3), 40, D)).cuda()
    a = vbq_b200.CompressedEmbedding(blob, checkpoint_rows=32)
    b = vbq_b200.CompressedEmbedding(blob, checkpoint_rows=7)
    for mt in ("dot", "cosine"):
        whole = a.scores(q, metric=mt)
        assert torch.equal(whole.view(torch.int32), b.scores(q, metric=mt).view(torch.int32))
        assert torch.equal(whole.view(torch.int32), a.scores(q, metric=mt).view(torch.int32))
        blocks = torch.cat([a.scores(q, e, min(e + 333, V), mt) for e in range(0, V, 333)], dim=1)
        assert torch.equal(whole.view(torch.int32), blocks.view(torch.int32))
        assert torch.equal(whole[5:6].view(torch.int32), a.scores(q[5], metric=mt).view(torch.int32))


def _ranking(sc, k, exclude=None):
    """Exact ranking of a (B, V) score array by (-score, id) with -0.0 = +0.0 and NaN last."""
    B, V = sc.shape
    out = []
    for bq in range(B):
        v = sc[bq].astype(np.float64)
        v = np.where(np.isnan(v), -np.inf, v)
        key = np.lexsort((np.arange(V), np.where(np.isnan(sc[bq]), 1, 0), -v))
        if exclude is not None:
            key = key[~np.isin(key, exclude[bq][exclude[bq] >= 0])]
        out.append(key[:k])
    return np.array(out)


@pytest.mark.gpu
def test_gpu_topk_equals_exact_ranking():
    import vbq_b200
    cb = vbq_b200.GaussianCodebook(1.2356, 10)
    V, D = 2000, 30
    m, s = _posteriors((V, D), 12)
    rng = np.random.default_rng(12)
    for beta in (1.0, 1e5):                                         # at 1e5 most rows are identical
        blob = cb.compress_to_bytes(m, s, [beta], seg_rows=128)[beta]
        ce = vbq_b200.CompressedEmbedding(blob)
        q = torch.from_numpy(_queries(rng, 6, D)).cuda()
        ex = rng.integers(-1, V, (6, 4))
        ex[0] = [3, 3, -1, 10]
        for mt in ("dot", "cosine"):
            sc = ce.scores(q, metric=mt)
            scn = sc.cpu().numpy()
            if beta == 1e5:
                assert np.unique(scn[0]).size < V // 10
            for k in (1, 10, V):
                vals, ids = ce.topk(q, k, metric=mt)
                assert vals.shape == (6, k) and ids.dtype == torch.int64
                assert np.array_equal(ids.cpu().numpy(), _ranking(scn, k)), (beta, mt, k)
                assert torch.equal(vals.view(torch.int32), sc.gather(1, ids).view(torch.int32))
            n_ex = max(np.unique(r[r >= 0]).size for r in ex)
            for k in (1, 10, V - n_ex):
                vals, ids = ce.topk(q, k, metric=mt, exclude=torch.from_numpy(ex).cuda())
                assert np.array_equal(ids.cpu().numpy(), _ranking(scn, k, ex)), (beta, mt, k)
                assert torch.equal(vals.view(torch.int32), sc.gather(1, ids).view(torch.int32))
            with pytest.raises(ValueError):
                ce.topk(q, V - n_ex + 1, metric=mt, exclude=ex)
            with pytest.raises(IndexError):
                ce.topk(q, 3, metric=mt, exclude=np.full((6, 1), V))
    with pytest.raises(ValueError, match="finite"):
        ce.topk(np.full(D, np.nan, np.float32), 3)
    with pytest.raises(ValueError, match="finite"):
        ce.scores(np.full(D, np.inf, np.float32))


@pytest.mark.gpu
def test_gpu_topk_workspace_does_not_grow_with_rows():
    """Extra device memory of topk stays within TOPK_WORKSPACE_BYTES plus a few (B, k) arrays for two tables whose row
    counts differ by 8x and both exceed one block."""
    import vbq_b200
    cb = vbq_b200.GaussianCodebook(1.2356, 10)
    B, k, D = 200, 10, 4
    peaks = []
    for V in (100_000, 800_000):
        m, s = _posteriors((V, D), 13)
        ce = vbq_b200.CompressedEmbedding(cb.compress_to_bytes(m, s, [1.0])[1.0])
        R = ce.TOPK_WORKSPACE_BYTES // (ce._TOPK_CELL_BYTES * B)
        assert R < V
        q = torch.randn(B, D, device="cuda")
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        vals, ids = ce.topk(q, k)
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - base
        assert peak <= ce.TOPK_WORKSPACE_BYTES + 8 * (8 + 4) * B * k + (1 << 20), (V, peak)
        peaks.append(peak)
        del ce
    assert peaks[1] <= peaks[0] * 1.05 + (1 << 20)


@pytest.mark.gpu
def test_gpu_full_embedding_plane():
    """1 M x 300 at one beta: sampled rows equal the reference, and the top 10 agree with a float64 ranking wherever the
    score margin exceeds the float32 error bound (D + 2) 2^-24 sum |z_d q_d|."""
    import vbq_b200
    g = torch.Generator(device="cuda")
    g.manual_seed(78)
    V, D = 1_000_000, 300
    means = torch.randn((V, D), generator=g, device="cuda") * 1.2329 - 0.08
    stds = torch.exp(torch.randn((V, D), generator=g, device="cuda") * 0.7 + float(np.log(0.04)))
    cb = vbq_b200.GaussianCodebook(1.2356, 10)
    blob = cb.compress_to_bytes(means, stds, [26.8])[26.8]
    del means, stds
    full = cb.decompress_from_bytes(blob)
    ce = vbq_b200.CompressedEmbedding(blob)
    q = torch.randn((4, D), generator=g, device="cuda")
    sc = ce.scores(q)
    rows = torch.randint(0, V, (2000,), generator=g, device="cuda")
    want = S.scores(full[rows].cpu().numpy(), q.cpu().numpy())
    assert _same_bits(sc[:, rows].cpu().numpy(), want)
    vals, ids = ce.topk(q, 10)
    assert torch.equal(vals.view(torch.int32), sc.gather(1, ids).view(torch.int32))
    f64 = full.double() @ q.double().T                                    # (V, B)
    bound = (D + 2) * 2.0 ** -24 * (full.double().abs() @ q.double().abs().T)
    for b in range(4):
        order = torch.argsort(f64[:, b], descending=True, stable=True)[:11]
        top = order[:10]
        # the top i + 1 are certain where the gap to the next row exceeds the bound of row i plus the largest bound
        bmax = bound[:, b].max()
        for i in range(10):
            gap = f64[order[i], b] - f64[order[i + 1], b]
            if gap > bound[order[i], b] + bmax:
                assert set(ids[b, :i + 1].tolist()) == set(top[:i + 1].tolist()), (b, i)
    del full


@pytest.mark.gpu
def test_gpu_corrupt_group_range_sets_status_4():
    import vbq_b200
    from vbq_b200 import ops
    cb = vbq_b200.GaussianCodebook(1.2356, 10)
    V, D = 1000, 30
    m, s = _posteriors((V, D), 14)
    ce = vbq_b200.CompressedEmbedding(cb.compress_to_bytes(m, s, [1.0], seg_rows=64)[1.0], checkpoint_rows=16)
    bounds = ce._bounds.clone()
    bounds[1, 1] = ce._words.numel() + 10 ** 6                    # group 1 ends far past the payload
    bounds[2, 0] = -5
    q = torch.randn(3, D, device="cuda")
    _, st = ops.rans_shared_row_scores(ce._words, bounds, ce._cum, ce._n, ce._seg, 10, ce._P, ce._k, ce._offsets,
                                       ce._states, D, 0, V, q, ce._code_points)
    assert int(st.item()) & 4
    _, st = ops.rans_shared_row_scores(ce._words, ce._bounds, ce._cum, ce._n, ce._seg, 10, ce._P, ce._k,
                                       ce._offsets, ce._states, D, 0, V, q, ce._code_points)
    assert int(st.item()) == 0
