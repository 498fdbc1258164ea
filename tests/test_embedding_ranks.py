"""Exact target ranks (vbq_score_ranks / vbq_pair_scores, vbq_b200.ranks, CompressedEmbedding.ranks, analogy_ranks,
analogy_metrics, GaussianCodebook.analogy_sweep): CPU tests of the NumPy reference against a brute-force ranking, a
hand-worked answer, the metrics, ABI and argument validation; GPU tests of the kernels against the reference, against
scores / topk, dense against compressed, the full 1 M x 300 plane and the analogy helpers."""
import ctypes

import numpy as np
import pytest
import torch

import embedding_ranks_reference as R
import embedding_scores_reference as S

F32 = np.float32


def _brute_ranks(Z, Q, targets, metric, exclude=None):
    """Rank by sorting the tie-free keys of CompressedEmbedding.topk: (key << 32) | (0xFFFFFFFF - id), descending,
    excluded rows removed; the rank is the target's position + 1."""
    sc = S.scores(Z, Q, metric)
    B, V = sc.shape
    out = []
    for b in range(B):
        full = (R.keys(sc[b]) << 32) | (0xFFFFFFFF - np.arange(V, dtype=np.int64))
        order = np.argsort(-full, kind="stable")
        if exclude is not None:
            order = order[~np.isin(order, exclude[b][exclude[b] >= 0])]
        out.append(int(np.nonzero(order == targets[b])[0][0]) + 1)
    return np.array(out, np.int64)


def _extreme_rows(rng, V, D):
    """Rows with duplicates (equal scores: the id decides), zero rows (+-0.0 scores), huge values (products overflow
    to +-inf, sums to NaN) and subnormals."""
    Z = rng.standard_normal((V, D)).astype(F32)
    if V >= 8:
        Z[3] = Z[1]
        Z[V - 1] = Z[1]
        Z[2] = 0
        Z[4] = -0.0
        Z[5, 0] = 3e38
        Z[6, :] = 3e38 * np.sign(rng.standard_normal(D)).astype(F32)
        Z[7, ::2] = 1e-41
    return Z


def _exclude_for(rng, targets, V, E):
    ex = rng.integers(-1, V, (len(targets), E))
    for b, t in enumerate(targets):
        ex[b][ex[b] == t] = -1
    if E >= 3 and len(targets):
        ex[0, :2] = ex[0, 2]                                    # duplicates count once
    return ex


# ---------------------------------------------------------------------------------------------------------------------
# the reference
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("metric", ["dot", "cosine"])
@pytest.mark.parametrize("D", [1, 3, 5])
def test_reference_matches_brute_force_ranking(metric, D):
    rng = np.random.default_rng(D)
    V, B = 24, 9
    Z = _extreme_rows(rng, V, D)
    Q = rng.standard_normal((B, D)).astype(F32)
    Q[1] = 0                                                    # every score 0: the id alone ranks
    Q[2] = Z[1]                                                 # the duplicated rows tie at the top
    Q[3, 0] = 2e38                                              # overflow against row 5 / row 6
    t = np.array([0, V - 1, 3, 6, 1, 2, 4, 5, V - 1])
    assert np.array_equal(R.ranks(Z, Q, t, metric), _brute_ranks(Z, Q, t, metric))
    ex = _exclude_for(rng, t, V, 5)
    assert np.array_equal(R.ranks(Z, Q, t, metric, ex), _brute_ranks(Z, Q, t, metric, ex))
    # an excluded row that beats the target lowers its rank by one
    sc = S.scores(Z, Q, metric)
    r0 = R.ranks(Z, Q, t, metric)
    b = 0
    beater = int(np.argsort(-((R.keys(sc[b]) << 32) | (0xFFFFFFFF - np.arange(V))), kind="stable")[0])
    if beater != t[b]:
        ex1 = np.full((B, 2), -1)
        ex1[b] = [beater, beater]
        assert R.ranks(Z, Q, t, metric, ex1)[b] == r0[b] - 1
    if metric == "dot":
        assert R.ranks(Z, Q, t, metric)[1] == V                # query 1 scores 0 everywhere: the id alone ranks
        assert R.ranks(Z, Q, np.zeros(B, np.int64), metric)[1] == 1


def test_reference_known_answer():
    """Rows (D = 2): z0 = (1, 0), z1 = (0, 1), z2 = (1, 0), z3 = (-1, 0), z4 = (0, 0); query q = (1, 0).  Dot scores
    1, 0, 1, -1, 0, so the order is 0, 2 (ties with 0, larger id), 1, 4 (ties with 1: 0.0), 3.  Ranks: target 2 ->
    2, target 4 -> 4, target 3 -> 5; excluding row 0 makes target 2 rank 1 and target 4 rank 3."""
    Z = np.array([[1, 0], [0, 1], [1, 0], [-1, 0], [0, 0]], F32)
    Q = np.array([[1, 0]] * 3, F32)
    assert R.ranks(Z, Q, [2, 4, 3]).tolist() == [2, 4, 5]
    assert R.ranks(Z, Q, [2, 4, 3], exclude=np.array([[0, -1], [0, 0], [-1, -1]])).tolist() == [1, 3, 5]
    # cosine with q = (2, 0): rows 0 and 2 score 1, row 3 scores -1, rows 1 and 4 score 0 (row 4 has zero norm)
    assert R.ranks(Z, 2 * Q, [2, 4, 3], "cosine").tolist() == [2, 4, 5]
    # -0.0 equals +0.0: q = (-1, 0) scores -0.0 on row 1 (fma(0, -1, +0) = +0 ... then +0 + -0) and +0.0 on row 4
    Zm = np.array([[0, 1], [-0.0, 0], [0, 0]], F32)
    assert R.ranks(Zm, np.array([[-1, 0]], F32), [2]).tolist() == [3]


def test_analogy_reference_and_metrics():
    import vbq_b200
    r = np.array([1, 2, 10, 11, 1, 100])
    m = vbq_b200.analogy_metrics(r)
    assert set(m) == {"mrr", "acc", "hits10"} and all(isinstance(v, np.float64) for v in m.values())
    assert m["mrr"] == np.mean([1, 0.5, 0.1, 1 / 11, 1, 0.01]) and m["acc"] == 2 / 6 and m["hits10"] == 4 / 6
    assert vbq_b200.analogy_metrics(torch.tensor([1, 1])) == {"mrr": 1.0, "acc": 1.0, "hits10": 1.0}
    assert R.metrics(r) == pytest.approx(m, abs=0)
    for bad, exc in (([], ValueError), ([0, 1], ValueError), ([1.0, 2.0], TypeError)):
        with pytest.raises(exc):
            vbq_b200.analogy_metrics(np.array(bad))
    # the analogy query is (z_b - z_a) + z_c with the target d; a, b and c are excluded
    Z = np.array([[1, 0], [0, 1], [1, 1], [0, 2], [2, 0]], F32)
    qs = np.array([[0, 1, 2, 3], [1, 0, 2, 4]])
    assert np.array_equal(R.analogy_queries(Z, qs), [[0, 2], [2, 0]])
    assert R.analogy_ranks(Z, qs).tolist() == [1, 1]


# ---------------------------------------------------------------------------------------------------------------------
# ABI and argument validation (no device)
# ---------------------------------------------------------------------------------------------------------------------
def test_ranks_abi_validation_needs_no_gpu():
    from vbq_b200 import _lib
    lib = _lib.load()
    p, odd = ctypes.c_void_p(16), ctypes.c_void_p(18)

    def ranks(rows=p, n=100, D=8, off=0, q=p, B=3, metric=0, thr=p, tgt=p, cnt=p):
        return lib.vbq_score_ranks(rows, n, D, off, q, B, metric, thr, tgt, cnt, None)
    assert ranks(D=0) == 2 and ranks(n=-1) == 2 and ranks(B=-1) == 2 and ranks(off=-1) == 2
    assert ranks(metric=2) == 2 and ranks(metric=-1) == 2 and ranks(B=2 ** 31) == 2
    assert ranks(n=2 ** 62, D=4) == 2 and ranks(off=2 ** 63 - 50) == 2
    assert ranks(rows=None) == 1 and ranks(q=None) == 1 and ranks(thr=None) == 1 and ranks(tgt=None) == 1
    assert ranks(cnt=None) == 1
    assert ranks(rows=None, n=0) == 0 and ranks(q=None, thr=None, tgt=None, cnt=None, B=0) == 0     # no work
    assert ranks(rows=odd) == 7 and ranks(tgt=ctypes.c_void_p(20)) == 7 and ranks(cnt=ctypes.c_void_p(20)) == 7

    def pairs(rows=p, n=100, D=8, q=p, B=3, pr=p, pq=p, P=5, metric=1, out=p):
        return lib.vbq_pair_scores(rows, n, D, q, B, pr, pq, P, metric, out, None)
    assert pairs(D=0) == 2 and pairs(n=-1) == 2 and pairs(B=-1) == 2 and pairs(P=-1) == 2 and pairs(metric=3) == 2
    assert pairs(rows=None) == 1 and pairs(q=None) == 1 and pairs(pr=None) == 1 and pairs(pq=None) == 1
    assert pairs(out=None) == 1
    assert pairs(rows=None, pr=None, pq=None, out=None, P=0) == 0
    assert pairs(out=odd) == 7 and pairs(pr=ctypes.c_void_p(20)) == 7
    assert b"metric=3" in (lib.vbq_last_error() if pairs(metric=3) else b"")


def test_rank_argument_errors_need_no_gpu():
    import vbq_b200
    from vbq_b200 import CompressedEmbedding
    ce = object.__new__(CompressedEmbedding)              # the attributes read before the first device operation
    ce._shape, ce._D, ce.device = (200, 30), 30, torch.device("cuda")
    good, t = np.zeros((2, 30), np.float32), np.array([0, 1])
    for q in (np.zeros((2, 30), np.int64), torch.zeros(2, 30, dtype=torch.int32)):
        with pytest.raises(TypeError):
            ce.ranks(q, t)
    for q in (np.zeros((2, 31), np.float32), np.zeros((2, 3, 10), np.float32)):
        with pytest.raises(ValueError):
            ce.ranks(q, t)
    with pytest.raises(ValueError, match="metric"):
        ce.ranks(good, t, metric="l2")
    with pytest.raises(TypeError):
        ce.ranks(good, np.array([0.0, 1.0]))
    for bad in (np.array([0, 1, 2]), np.array([[0, 1]]), 0):
        with pytest.raises(ValueError):
            ce.ranks(good, bad)
    with pytest.raises(TypeError):
        ce.ranks(good, t, exclude=np.zeros((2, 3), np.float32))
    with pytest.raises(ValueError):
        ce.ranks(good, t, exclude=np.zeros((3, 3), np.int64))
    with pytest.raises(ValueError):
        vbq_b200.analogy_ranks(ce, np.zeros((4, 3), np.int64))
    with pytest.raises(TypeError):
        vbq_b200.analogy_ranks(ce, np.zeros((4, 4), np.float32))
    # the dense form takes only float32 CUDA tensors with at least one coordinate per row
    for m in (torch.zeros(5, 3), np.zeros((5, 3), np.float32), [[0.0]]):
        with pytest.raises(TypeError):
            vbq_b200.ranks(m, np.zeros((1, 3), np.float32), [0])
        with pytest.raises(TypeError):
            vbq_b200.analogy_ranks(m, np.zeros((1, 4), np.int64))


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _posteriors(shape, seed):
    rng = np.random.default_rng(seed)
    means = (rng.standard_normal(shape) * 1.2329 - 0.08).astype(np.float32)
    stds = np.exp(rng.standard_normal(shape) * 0.7 + np.log(0.04)).astype(np.float32)
    return means, stds


@pytest.mark.gpu
@pytest.mark.parametrize("D", [1, 3, 4, 7, 32, 33, 100, 300])
def test_gpu_ranks_match_reference(D):
    import vbq_b200
    rng = np.random.default_rng(100 + D)
    for V, B in ((1, 1), (8, 5), (200, 65), (333, 130)):
        Z = _extreme_rows(rng, V, D)
        Q = rng.standard_normal((B, D)).astype(F32)
        if B >= 5:
            Q[1] = Z[1 % V]
            Q[2] = 0
            Q[3, 0] = 2e38
            Q[4, ::3] = 1e-40
        t = rng.integers(0, V, B)
        t[0], t[-1] = 0, V - 1
        Zd = torch.from_numpy(Z).cuda()
        for metric in ("dot", "cosine"):
            got = vbq_b200.ranks(Zd, torch.from_numpy(Q).cuda(), t, metric)
            assert got.dtype == torch.int64 and got.shape == (B,)
            assert np.array_equal(got.cpu().numpy(), R.ranks(Z, Q, t, metric)), (V, B, metric)
            if V > 1:
                ex = _exclude_for(rng, t, V, 4)
                got = vbq_b200.ranks(Zd, Q, torch.from_numpy(t).cuda(), metric, exclude=ex)
                assert np.array_equal(got.cpu().numpy(), R.ranks(Z, Q, t, metric, ex)), (V, B, metric)
    # a (V, *tail) matrix and a single query of the tail's shape
    Z = rng.standard_normal((50, D)).astype(F32)
    got = vbq_b200.ranks(torch.from_numpy(Z).cuda().reshape((50,) + ((D,) if D > 1 else ())), Z[7].reshape(
        (D,) if D > 1 else ()), [7])
    assert got.tolist() == R.ranks(Z, Z[7:8], [7]).tolist()


@pytest.mark.gpu
def test_gpu_ranks_agree_with_scores_and_topk():
    import vbq_b200
    cb = vbq_b200.GaussianCodebook(1.2356, 10)
    V, D, B = 3000, 40, 70
    m, s = _posteriors((V, D), 21)
    rng = np.random.default_rng(21)
    for beta in (1.0, 1e5):                                      # at 1e5 most rows are equal: the id decides
        blob = cb.compress_to_bytes(m, s, [beta], seg_rows=64)[beta]
        ce = vbq_b200.CompressedEmbedding(blob)
        dense = cb.decompress_from_bytes(blob)
        q = torch.from_numpy(rng.standard_normal((B, D)).astype(F32)).cuda()
        t = torch.from_numpy(rng.integers(0, V, B)).cuda()
        ex = torch.from_numpy(_exclude_for(rng, t.cpu().numpy(), V, 3)).cuda()
        for metric in ("dot", "cosine"):
            sc = ce.scores(q, metric=metric)
            k = torch.from_numpy(R.keys(sc.cpu().numpy())).cuda()
            kt = k.gather(1, t[:, None])
            ids = torch.arange(V, device="cuda")[None, :]
            want = 1 + ((k > kt) | ((k == kt) & (ids < t[:, None]))).sum(1)
            got = vbq_b200.ranks(dense, q, t, metric)
            assert torch.equal(got, want), (beta, metric)
            assert torch.equal(got, vbq_b200.ranks(dense, q, t, metric))          # repeatable
            for e in (None, ex):
                r = vbq_b200.ranks(dense, q, t, metric, exclude=e)
                _, top = ce.topk(q, 10, metric=metric, exclude=e)
                inside = (top == t[:, None]).any(1)
                assert torch.equal(inside, r <= 10), (beta, metric)
                sel = torch.nonzero(r <= 10)[:, 0]
                assert torch.equal(top[sel, r[sel] - 1], t[sel])


@pytest.mark.gpu
def test_gpu_dense_and_compressed_ranks_agree():
    import vbq_b200
    from vbq_b200 import CompressedEmbedding
    cb = vbq_b200.GaussianCodebook(1.2356, 10)
    rng = np.random.default_rng(31)
    for (V, D) in ((2000, 30), (1501, 7)):
        m, s = _posteriors((V, D), V)
        q = rng.standard_normal((67, D)).astype(F32)
        t = rng.integers(0, V, 67)
        ex = _exclude_for(rng, t, V, 3)
        for seg in (1, 37, None):
            blob = cb.compress_to_bytes(m, s, [2.0], seg_rows=seg)[2.0]
            dense = cb.decompress_from_bytes(blob)
            for metric in ("dot", "cosine"):
                want = vbq_b200.ranks(dense, q, t, metric, exclude=ex)
                for K in (1, 9, None):
                    ce = CompressedEmbedding(blob, checkpoint_rows=K)
                    assert torch.equal(ce.ranks(q, t, metric, exclude=ex), want), (V, D, seg, K, metric)
                ce.RANKS_WORKSPACE_BYTES = 97 * (4 * D + ce._RANKS_ROW_EXTRA_BYTES)   # 97-row blocks: many blocks
                assert torch.equal(ce.ranks(q, t, metric, exclude=ex), want), (V, D, seg, metric)
                assert torch.equal(ce.ranks(q, t, metric, exclude=ex), want)


@pytest.mark.gpu
def test_gpu_full_plane_ranks_against_block_scores():
    """1 M x 300, B = 1,024: CompressedEmbedding.ranks and dense ranks equal counts over CompressedEmbedding.scores."""
    import vbq_b200
    g = torch.Generator(device="cuda")
    g.manual_seed(79)
    V, D, B = 1_000_000, 300, 1024
    means = torch.randn((V, D), generator=g, device="cuda") * 1.2329 - 0.08
    stds = torch.exp(torch.randn((V, D), generator=g, device="cuda") * 0.7 + float(np.log(0.04)))
    cb = vbq_b200.GaussianCodebook(1.2356, 10)
    blob = cb.compress_to_bytes(means, stds, [26.8])[26.8]
    del means, stds
    ce = vbq_b200.CompressedEmbedding(blob)
    q = torch.randn((B, D), generator=g, device="cuda")
    t = torch.randint(0, V, (B,), generator=g, device="cuda")
    blocks = [(a, min(V, a + 100_000)) for a in range(0, V, 100_000)]
    for metric in ("dot", "cosine"):
        kt = torch.zeros(B, dtype=torch.int64, device="cuda")
        for a, b in blocks:                                      # the targets' keys
            k = _keys_t(ce.scores(q, a, b, metric))
            inb = (t >= a) & (t < b)
            kt = torch.where(inb, k.gather(1, (t - a).clamp(0, b - a - 1)[:, None])[:, 0], kt)
        want = torch.ones(B, dtype=torch.int64, device="cuda")
        for a, b in blocks:                                      # the rows that beat them
            k = _keys_t(ce.scores(q, a, b, metric))
            ids = torch.arange(a, b, device="cuda")[None, :]
            want += ((k > kt[:, None]) | ((k == kt[:, None]) & (ids < t[:, None]))).sum(1)
        assert torch.equal(ce.ranks(q, t, metric), want), metric
        dense = cb.decompress_from_bytes(blob)
        assert torch.equal(vbq_b200.ranks(dense, q, t, metric), want), metric
        del dense


def _keys_t(s):
    """embedding_ranks_reference.keys on a device tensor."""
    b = s.view(torch.int32).to(torch.int64)
    k = torch.where(b < 0, b ^ 0x7FFFFFFF, b)
    k = torch.where(s == 0, torch.zeros_like(k), k)
    return torch.where(torch.isnan(s), torch.full_like(k, -(1 << 31)), k)


@pytest.mark.gpu
def test_gpu_analogy_helpers():
    import vbq_b200
    cb = vbq_b200.GaussianCodebook(1.2356, 10)
    V, D, B = 1200, 24, 150
    m, s = _posteriors((V, D), 41)
    rng = np.random.default_rng(41)
    qs = np.stack([rng.choice(V, 4, replace=False) for _ in range(B)])
    blob = cb.compress_to_bytes(m, s, [1.0])[1.0]
    dense = cb.decompress_from_bytes(blob)
    ce = vbq_b200.CompressedEmbedding(blob)
    for metric in ("cosine", "dot"):
        Z = dense.cpu().numpy()
        q = R.analogy_queries(Z, qs)
        want = vbq_b200.ranks(dense, q, qs[:, 3], metric, exclude=qs[:, :3])
        got = vbq_b200.analogy_ranks(dense, torch.from_numpy(qs).cuda(), metric)
        assert torch.equal(got, want)
        assert torch.equal(vbq_b200.analogy_ranks(ce, qs, metric), want)
        assert np.array_equal(got.cpu().numpy(), R.analogy_ranks(Z, qs, metric))
    assert vbq_b200.analogy_ranks(dense, qs).dtype == torch.int64      # the default metric is the cosine
    bad = qs.copy()
    bad[0, 3] = bad[0, 1]
    with pytest.raises(ValueError, match="exclude"):
        vbq_b200.analogy_ranks(dense, bad)
    with pytest.raises(IndexError):
        vbq_b200.analogy_ranks(ce, np.array([[0, 1, 2, V]]))
    # analogy_sweep is the test_beta loop: quality per beta on compress_coordinates, bits from beta_sweep
    mt, st = torch.from_numpy(m).cuda(), torch.from_numpy(s).cuda()
    betas = [0.3, 3.0, 300.0]
    for exact in (True, False):
        table = cb.analogy_sweep(mt, st, betas, qs, exact=exact)
        assert table.shape == (3, 4) and table.dtype == np.float64
        assert np.array_equal(table[:, 3], cb.beta_sweep(mt, st, betas, exact=exact))
        for i, beta in enumerate(betas):
            zhat, _ = cb.compress_coordinates(mt, st, beta, exact=exact)
            met = vbq_b200.analogy_metrics(vbq_b200.analogy_ranks(zhat, qs))
            assert table[i, :3].tolist() == [met["mrr"], met["acc"], met["hits10"]], (exact, beta)


@pytest.mark.gpu
def test_gpu_rank_argument_errors():
    import vbq_b200
    V, D = 100, 8
    Z = torch.randn(V, D, device="cuda")
    q = torch.randn(3, D, device="cuda")
    t = torch.tensor([0, 5, V - 1], device="cuda")
    for bad in ([0, 5, V], [-1, 0, 0]):
        with pytest.raises(IndexError):
            vbq_b200.ranks(Z, q, bad)
    with pytest.raises(IndexError):
        vbq_b200.ranks(Z, q, t, exclude=np.array([[V], [0], [1]]))
    with pytest.raises(IndexError):
        vbq_b200.ranks(Z, q, t, exclude=np.array([[-2], [0], [1]]))
    with pytest.raises(ValueError, match="own exclude"):
        vbq_b200.ranks(Z, q, t, exclude=np.array([[3, -1], [1, 5], [2, 2]]))
    qn = q.clone()
    qn[1, 2] = float("nan")
    with pytest.raises(ValueError, match="finite"):
        vbq_b200.ranks(Z, qn, t)
    with pytest.raises(TypeError):
        vbq_b200.ranks(Z.double(), q, t)
    with pytest.raises(ValueError):
        vbq_b200.ranks(Z, torch.randn(3, D + 1, device="cuda"), t)
    assert vbq_b200.ranks(Z, torch.randn(0, D, device="cuda"), []).shape == (0,)
