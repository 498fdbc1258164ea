"""Row access into VBQE blobs (vbq_rans_shared_checkpoints / vbq_rans_shared_decode_rows, CompressedEmbedding): CPU
tests of the NumPy reference (checkpoints, decoding from them, the work list), the default checkpoint interval, ABI and
argument validation; GPU tests of the index against the reference bit for bit, of lookups against the full decode, of
reading only the needed segments and of bad work lists."""
import ctypes

import numpy as np
import pytest
import torch

import embedding_lookup_reference as E
import rans_shared_reference as R
from vbq_b200 import coding, serialize

Q10 = 2047


def _table(rng, Q=Q10, P=16):
    cnt = np.zeros(Q, np.int64)
    cnt[Q // 2 - 40:Q // 2 + 40] = rng.integers(1, 1000, 80)
    cnt[rng.integers(0, Q, 10)] = 1
    return coding.frequency_tables(cnt, P, keep_zeros=True)[0]


def _plane(rng, t, n):
    return rng.choice(t.size, size=n, p=t / t.sum()).astype(np.int32)


# ---------------------------------------------------------------------------------------------------------------------
# the reference
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,seg,K", [(1, 1, 1), (33, 2, 1), (1000, 3, 1), (1000, 5, 2), (5000, 40, 7),
                                     (5000, 40, 40), (5000, 40, 1000), (7007, 1000, 9), (9600, 300, 64)])
def test_reference_decoding_from_every_checkpoint_reproduces_the_full_decode(n, seg, K):
    rng = np.random.default_rng(n + seg + K)
    t = _table(rng)
    plane = _plane(rng, t, n)
    pay = R.rans_encode(plane[None], t[None], 16, seg)
    full = R.rans_decode(pay, 1, n, seg, t[None], 16)[0]
    offs, states = E.checkpoints(pay, n, seg, t, 16, K)
    assert offs.size == E.checkpoint_count(n, seg, K)
    S = max(1, min(seg, -(-n // 32)))
    k = min(K, S)
    rows = -(-n // 32)
    for g in range(-(-rows // S)):
        length = min(S, rows - g * S)
        for j in range((length - 1) // k + 1):
            first = g * S + j * k
            last = min(first + k, g * S + length) - 1
            sym = E.decode_from(pay, n, seg, t, 16, K, offs, states, g, j, last)
            want = np.full(sym.size, -1, np.int64)
            idx = np.arange(32 * first, 32 * (last + 1))
            want[idx < n] = full[idx[idx < n]]
            assert np.array_equal(sym.reshape(-1), want), (g, j)


def test_reference_checkpoint_known_answer():
    """The hand-worked stream of test_rans_embeddings (n = 33, one segment of two rows, f = (1, 0, 4095), P = 12) with
    K = 1: one checkpoint, before row 1.  Row 0: lane 0 (x = 2^24, slot 0, symbol 0, f = 1) drops to 4096 and reads the
    group's one word (0x0000): x = 2^28; lanes 1..31 (x = 0x00010011, slot 17, symbol 2) go to 4095 * 16 + 16 = 2^16
    and read nothing.  So the offset is 64 state words + 1 = 65 and the states are 2^28, then 31 x 2^16."""
    t = np.array([1, 0, 4095])
    pay = np.array([65, 0, 0x0000, 0x0100] + [0x0011, 0x0001] * 31 + [0x0000])
    offs, states = E.checkpoints(pay, 33, 2, t, 12, 1)
    assert offs.tolist() == [65]
    assert states.tolist() == [[1 << 28] + [1 << 16] * 31]
    assert E.decode_from(pay, 33, 2, t, 12, 1, offs, states, 0, 1, 1).tolist() == [[0] + [-1] * 31]


@pytest.mark.parametrize("D", [1, 7, 32, 33, 300])
@pytest.mark.parametrize("seg,K", [(1, 1), (3, 2), (40, 5), (10 ** 6, 16)])
def test_reference_work_list_covers_every_requested_symbol_once(D, seg, K):
    rng = np.random.default_rng(D * 7 + seg + K)
    V = 97
    n = V * D
    t = _table(rng)
    plane = _plane(rng, t, n)
    seg = serialize.shared_seg_rows(n, seg)                # the reference encoder loops over seg_rows rows
    pay = R.rans_encode(plane[None], t[None], 16, seg)
    full = plane.reshape(V, D)
    for ids in (rng.integers(0, V, 30), [0, V - 1], np.arange(V)[::-1], [5, 5, 5]):
        rows, out = E.gather(pay, n, seg, t, 16, K, ids, D)         # asserts that no element is written twice
        assert np.array_equal(out, full[rows]), ids
        _, items = E.work_list(ids, D, n, seg, K)
        assert (np.diff(items[:, 0] * (1 << 32) + items[:, 1]) > 0).all()   # one item per interval, in order


# ---------------------------------------------------------------------------------------------------------------------
# default K, ABI and argument validation (no device)
# ---------------------------------------------------------------------------------------------------------------------
def test_checkpoint_count_matches_the_reference():
    from vbq_b200 import ops
    for n, seg, K in [(0, 1, 1), (1, 1, 1), (33, 2, 1), (1000, 3, 1), (5000, 40, 7), (5000, 40, 39), (5000, 40, 40),
                      (5000, 40, 10 ** 9), (300_000_000, 9209, 64), (300_000_000, 5_000_000, 32)]:
        assert ops.rans_shared_checkpoint_count(n, seg, K) == E.checkpoint_count(n, seg, K), (n, seg, K)


def test_default_checkpoint_rows_rule():
    from vbq_b200 import ops
    from vbq_b200.word_embeddings import default_checkpoint_rows
    for n, seg, pay in [(300_000_000, 5146, 133_000_000), (300_000_000, 1018, 26_200_000),
                        (300_000_000, 4_687_500, 75_000), (3_000_000, 300, 10 ** 6), (1000, 32, 10), (10, 1, 4)]:
        S = serialize.shared_seg_rows(n, seg)
        K = default_checkpoint_rows(n, seg, pay)
        assert K >= 32
        assert 132 * 8 * ops.rans_shared_checkpoint_count(n, S, K) <= pay
        if K > 32:
            assert 132 * 8 * ops.rans_shared_checkpoint_count(n, S, K - 1) > pay
    # about 0.5 bits per coordinate of index at K = 64 rows (2,048 coordinates): 132 * 8 / 2048
    assert abs(132 * 8 / 2048 - 0.516) < 1e-3


def test_lookup_abi_validation_needs_no_gpu():
    from vbq_b200 import _lib
    lib = _lib.load()
    cnt = lib.vbq_rans_shared_checkpoint_count
    assert cnt(1000, 4, 1) == 24 and cnt(1000, 4, 2) == 8 and cnt(1000, 4, 4) == 0     # 8 segments of 4 rows
    assert cnt(1000, 4, 0) == -1 and cnt(-1, 4, 1) == -1 and cnt(1000, 0, 1) == -1
    assert cnt(2 ** 36, 2 ** 31, 1) == -1                                   # beyond the 32-bit offsets
    assert cnt(1000, 2 ** 62, 2 ** 62) == 0
    p, odd = ctypes.c_void_p(16), ctypes.c_void_p(18)
    ck = lib.vbq_rans_shared_checkpoints
    assert ck(p, 10, p, 1000, 4, 11, 16, p, 1, p, p, p, None) == 3           # N > 10
    assert ck(p, 10, p, 1000, 4, 10, 17, p, 1, p, p, p, None) == 2           # prob_bits
    assert ck(p, 10, p, 1000, 4, 10, 16, p, 0, p, p, p, None) == 2           # K < 1
    assert ck(p, -1, p, 1000, 4, 10, 16, p, 1, p, p, p, None) == 2
    assert ck(p, 10, p, 1000, 4, 10, 16, p, 1, None, p, p, None) == 1        # index missing
    assert ck(p, 10, p, 1000, 4, 10, 16, None, 1, p, p, p, None) == 1
    assert ck(p, 10, None, 1000, 4, 10, 16, p, 1, p, p, p, None) == 1
    assert ck(p, 10, p, 1000, 4, 10, 16, odd, 1, p, p, p, None) == 7
    assert ck(p, 10, p, 2 ** 36, 2 ** 31, 10, 16, p, 1, p, p, p, None) == 2   # shape beyond the offsets
    dr = lib.vbq_rans_shared_decode_rows

    def rows(n=1000, seg=4, N=10, P=16, K=1, offs=p, items=p, n_items=5, rws=p, n_req=3, D=10, cp=p, q=p, z=p):
        return dr(p, 10, p, n, seg, N, P, p, K, offs, p, items, n_items, rws, n_req, D, cp, q, z, p, None)
    assert rows(N=11) == 3
    assert rows(P=11) == 2
    assert rows(K=0) == 2
    assert rows(D=0) == 2 and rows(D=3) == 2                                 # D < 1, D not dividing n
    assert rows(n_req=-1) == 2 and rows(n_req=101) == 2                      # more rows than the plane has
    assert rows(n_items=-1) == 2
    assert rows(items=None) == 1 and rows(rws=None) == 1 and rows(offs=None) == 1
    assert rows(z=p, cp=None) == 1                                           # z_hat without code points
    assert rows(items=ctypes.c_void_p(20)) == 7 and rows(rws=ctypes.c_void_p(12)) == 7 and rows(z=odd) == 7
    assert rows(n=2 ** 36, seg=2 ** 31, D=2 ** 4) == 2


def _small_blob():
    rng = np.random.default_rng(9)
    t = _table(rng)
    plane = _plane(rng, t, 6000)
    hdr = serialize.embedding_header(10, 16, (200, 30), 40, 1.2356, 1.0, 1234, t)
    return hdr + R.rans_encode(plane[None], t[None], 16, 40).astype("<u2").tobytes()


def test_constructor_and_lookup_argument_errors_need_no_gpu():
    """Malformed blobs and a bad checkpoint_rows raise ValueError, non-integer ids TypeError and host ids outside the
    table IndexError, all before anything is uploaded or launched (on a machine without a GPU, reaching the device
    would raise something else)."""
    from vbq_b200 import CompressedEmbedding
    blob = _small_blob()
    for bad in (b"VBQ2" + blob[4:], blob[:-2], blob + b"\0\0", blob[:30]):
        with pytest.raises(ValueError):
            CompressedEmbedding(bad)
    for K in (0, -3, 2.5, True):
        with pytest.raises(ValueError, match="checkpoint_rows"):
            CompressedEmbedding(blob, checkpoint_rows=K)
    ce = object.__new__(CompressedEmbedding)           # the attributes lookup reads before the first device operation
    ce._shape, ce._D, ce.device = (200, 30), 30, torch.device("cuda")
    for ids in ([0.5, 1.0], np.array([1.0]), torch.tensor([1.0]), torch.tensor([True])):
        with pytest.raises(TypeError):
            ce.lookup(ids)
    for ids in ([200], [-1, 3], np.array([[0, 1], [2, 250]]), torch.tensor([0, 199, 200], dtype=torch.int32)):
        with pytest.raises(IndexError):
            ce.lookup(ids)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _posteriors(shape, seed):
    rng = np.random.default_rng(seed)
    means = (rng.standard_normal(shape) * 1.2329 - 0.08).astype(np.float32)
    stds = np.exp(rng.standard_normal(shape) * 0.7 + np.log(0.04)).astype(np.float32)
    return means, stds


@pytest.mark.gpu
@pytest.mark.parametrize("n,seg,K", [(1000, 1, 1), (7007, 3, 2), (9600, 40, 7), (300_300, 256, 5),
                                     (300_300, 256, 64), (300_300, 10 ** 6, 100)])
def test_gpu_checkpoint_index_matches_reference(n, seg, K):
    from vbq_b200 import ops
    rng = np.random.default_rng(n + K)
    t = _table(rng)
    plane = _plane(rng, t, n)
    pay = R.rans_encode(plane[None], t[None], 16, seg)
    S = serialize.shared_seg_rows(n, seg)
    bounds = serialize._offset_bounds(pay, [serialize.shared_nact(n, S)])
    w = torch.from_numpy(pay.view(np.int16).copy()).cuda()
    b = torch.from_numpy(np.ascontiguousarray(bounds, dtype=np.int64)).cuda()
    cum = torch.from_numpy(coding.cum_table_shared(t[None]).view(np.int32)).cuda()
    offs, states, status = ops.rans_shared_checkpoints(w, b, cum, n, S, 10, 16, min(K, S))
    assert int(status.item()) == 0
    ro, rs = E.checkpoints(pay, n, S, t, 16, K)
    assert np.array_equal(offs.cpu().numpy().view(np.uint32), ro)
    assert np.array_equal(states.cpu().numpy().view(np.uint32), rs)


def _boundary_rows(V, D, S, K, coder_rows):
    """Embedding rows that hold the first symbol of a segment or of a checkpoint interval, and their neighbours."""
    k = min(K, S)
    starts = (np.arange(0, coder_rows, S)[:, None] + np.arange(0, S, k)[None, :]).ravel()
    e = (32 * starts[starts < coder_rows]) // D
    e = np.unique(np.clip(np.concatenate([e - 1, e, e + 1]), 0, V - 1))
    return e[np.linspace(0, e.size - 1, min(e.size, 300)).astype(np.int64)]


@pytest.mark.gpu
@pytest.mark.parametrize("D", [1, 7, 32, 33, 300])
def test_gpu_lookup_equals_full_decode(D):
    import vbq_b200
    cb = vbq_b200.GaussianCodebook(1.2356, 10)
    V = {1: 5001, 7: 1001, 32: 1001, 33: 997, 300: 1001}[D]
    shape = (V,) if D == 1 else (V, D)
    n = V * D
    assert n % 32 or D == 32                       # the plane's last row is partial where it can be
    m, s = _posteriors(shape, D)
    rng = np.random.default_rng(D)
    coder_rows = -(-n // 32)
    for seg in (1, 3, 256, 10 ** 6):
        blob = cb.compress_to_bytes(m, s, [1.0], seg_rows=seg)[1.0]
        full = cb.decompress_from_bytes(blob)
        S = serialize.shared_seg_rows(n, seg)
        for K in (1, 5, 64, None, S + 1):
            ce = vbq_b200.CompressedEmbedding(blob, checkpoint_rows=K)
            assert ce.shape == shape and ce.beta == 1.0
            assert ce.checkpoint_rows == (K if K is not None else
                                          vbq_b200.word_embeddings.default_checkpoint_rows(n, S, 2 * ce._words.numel()))
            k = ce.checkpoint_rows
            rnd = rng.integers(0, V, 200)
            cases = [rnd, rnd[::-1].copy(), [0, V - 1], _boundary_rows(V, D, S, k, coder_rows),
                     rng.permutation(V), np.zeros(0, np.int64), rnd[:60].reshape(6, 10)]
            for i, ids in enumerate(cases):
                for conv in (lambda a: torch.from_numpy(np.asarray(a)).cuda(),
                             lambda a: torch.from_numpy(np.asarray(a).astype(np.int32)),
                             lambda a: np.asarray(a).tolist()):
                    got = ce.lookup(conv(ids))
                    want = full[torch.from_numpy(np.asarray(ids, dtype=np.int64)).cuda()]
                    assert got.dtype == torch.float32 and got.shape == want.shape, (seg, K, i)
                    assert torch.equal(got, want), (D, seg, K, i)
        assert torch.equal(ce(np.arange(V)), full)
        assert ce.nbytes >= 2 * ce._words.numel() + 132 * ce._offsets.numel()


@pytest.mark.gpu
def test_gpu_full_embedding_plane():
    """1 M x 300 at two betas, default segmentation and K: 4,096 random ids and all rows equal the full decode."""
    import vbq_b200
    g = torch.Generator(device="cuda")
    g.manual_seed(77)
    V, D = 1_000_000, 300
    means = torch.randn((V, D), generator=g, device="cuda") * 1.2329 - 0.08
    stds = torch.exp(torch.randn((V, D), generator=g, device="cuda") * 0.7 + float(np.log(0.04)))
    cb = vbq_b200.GaussianCodebook(1.2356, 10)
    betas = [0.518, 1931.0]
    blobs = cb.compress_to_bytes(means, stds, betas)
    del means, stds
    for beta in betas:
        full = cb.decompress_from_bytes(blobs[beta])
        ce = vbq_b200.CompressedEmbedding(blobs[beta])
        h = serialize.read_embedding_header(blobs[beta])
        assert 132 * 8 * ce._offsets.numel() <= 2 * h["words"].size
        ids = torch.randint(0, V, (4096,), device="cuda", generator=g)
        assert torch.equal(ce.lookup(ids), full[ids])
        assert torch.equal(ce.lookup(torch.arange(V, device="cuda")), full)
        del full, ce


@pytest.mark.gpu
def test_gpu_lookup_reads_only_the_segments_it_needs():
    """Corrupt the words of segment 2: the constructor rejects the blob, but an object built from the clean blob whose
    payload is then corrupted the same way still looks up every row outside segment 2 correctly."""
    import vbq_b200
    cb = vbq_b200.GaussianCodebook(1.2356, 10)
    V, D = 2000, 30
    m, s = _posteriors((V, D), 4)
    blob = cb.compress_to_bytes(m, s, [1.0], seg_rows=256)[1.0]
    h = serialize.read_embedding_header(blob)
    off = len(blob) - 2 * h["words"].size
    a, b = h["bounds"][2]
    bad = bytearray(blob)
    for i in range(a + 70, b, 7):
        bad[off + 2 * i] ^= 0x5A
    with pytest.raises(ValueError, match="corrupt"):
        vbq_b200.CompressedEmbedding(bytes(bad))
    full = cb.decompress_from_bytes(blob)
    ce = vbq_b200.CompressedEmbedding(blob, checkpoint_rows=16)
    ce._words.copy_(torch.from_numpy(np.frombuffer(bytes(bad), dtype="<i2", offset=off).copy()).cuda())
    seg_of_row = lambda e: (np.asarray(e) * D // 32 // 256, (np.asarray(e) * D + D - 1) // 32 // 256)
    ids = np.array([e for e in range(V) if 2 not in seg_of_row(e)])
    assert ids.size < V
    assert torch.equal(ce.lookup(ids), full[torch.from_numpy(ids).cuda()])


@pytest.mark.gpu
def test_gpu_bad_work_lists_set_status_8_and_write_nothing():
    import vbq_b200
    from vbq_b200 import _lib
    cb = vbq_b200.GaussianCodebook(1.2356, 10)
    V, D = 1000, 30
    m, s = _posteriors((V, D), 5)
    blob = cb.compress_to_bytes(m, s, [1.0], seg_rows=64)[1.0]
    ce = vbq_b200.CompressedEmbedding(blob, checkpoint_rows=16)
    u = torch.tensor([3, 40, 41], dtype=torch.int64, device="cuda")
    good = ce._work_list(u)[0]
    G = ce._bounds.shape[0]
    lib = _lib.load()
    guard = 1024

    def run(items, rows=u):
        out = torch.full((rows.numel() * D + guard,), -7.0, device="cuda")
        status = torch.zeros(1, dtype=torch.int32, device="cuda")
        items = items.contiguous()
        _lib.check(lib.vbq_rans_shared_decode_rows(
            ce._words.data_ptr(), ce._words.numel(), ce._bounds.data_ptr(), ce._n, ce._seg, 10, ce._P,
            ce._cum.data_ptr(), ce._k, ce._offsets.data_ptr(), ce._states.data_ptr(), items.data_ptr(),
            items.shape[0], rows.data_ptr(), rows.numel(), D, ce._code_points.data_ptr(), None, out.data_ptr(),
            status.data_ptr(), torch.cuda.current_stream().cuda_stream), "vbq_rans_shared_decode_rows")
        return int(status.item()), out
    st, out = run(good)
    assert st == 0 and torch.equal(out[:3 * D].reshape(3, D), cb.decompress_from_bytes(blob)[u])
    assert (out[3 * D:] == -7.0).all()
    per = (ce._seg - 1) // ce._k
    bads = []
    for field, value in ((0, G), (0, -1), (1, per + 1), (1, -1), (2, 10 ** 6), (2, -1), (3, -1), (4, 4), (3, 3)):
        it = good.clone()
        it[0, field] = value
        bads.append(it)
    it = good.clone()
    it[0, 2] = it[0, 0] * ce._seg + it[0, 1] * ce._k + ce._k          # one row past the interval
    bads.append(it)
    for it in bads:
        st, out = run(it[:1])
        assert st & 8, it[0].tolist()
        assert (out == -7.0).all(), it[0].tolist()
    # rows 40 and 41 share the second item's slice [1, 3); the first item (row 3) stays valid and writes row 0
    assert good[:, 3:].tolist() == [[0, 1], [1, 3]]
    for rows in (torch.tensor([3, 41, 40], dtype=torch.int64, device="cuda"),        # unsorted
                 torch.tensor([3, 40, 40], dtype=torch.int64, device="cuda"),        # repeated
                 torch.tensor([3, 40, V], dtype=torch.int64, device="cuda")):        # past the table
        st, out = run(good, rows)
        assert st & 8, rows.tolist()
        assert (out[D:] == -7.0).all(), rows.tolist()
