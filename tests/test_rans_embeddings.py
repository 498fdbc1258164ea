"""Entropy coding of word embeddings with the shared-table rANS coder (vbq_rans_shared_*, serialize VBQE,
GaussianCodebook.compress_to_bytes): CPU tests of the NumPy reference layout, the zero-preserving tables, the VBQE
header and the ABI; GPU tests of the kernels against the reference byte for byte, of corrupt streams, of the
end-to-end bytes -> optima path and of the rate."""
import ctypes
import hashlib
import struct

import numpy as np
import pytest
import torch

import rans_shared_reference as R
from vbq_b200 import coding, serialize

Q10 = 2047


def _table(rng, Q, P, where):
    """Zero-preserving table from random counts on a few symbol ranges: zeros at the front, middle and/or end."""
    cnt = np.zeros(Q, np.int64)
    if where == "front":
        cnt[Q // 2:] = rng.integers(1, 100, Q - Q // 2)
    elif where == "end":
        cnt[:Q // 3] = rng.integers(1, 100, Q // 3)
    elif where == "middle":
        cnt[:5] = rng.integers(1, 1000, 5)
        cnt[-5:] = rng.integers(1, 1000, 5)
    else:                                               # peaked with sparse tails, zeros everywhere
        cnt[rng.integers(0, Q, 40)] = rng.integers(1, 30, 40)
        cnt[Q // 2] = 100_000
    return coding.frequency_tables(cnt, P, keep_zeros=True)[0]


def _planes(rng, tables, n):
    return np.stack([rng.choice(t.size, size=n, p=t / t.sum()) for t in tables]).astype(np.int32)


def _xent_bits(planes, tables):
    P = int(np.log2(tables[0].sum()))
    return sum(float(-np.log2(t[p] / 2.0 ** P).sum()) for p, t in zip(planes, tables))


NS = [0, 1, 31, 32, 33, 1000]
WHERE = ["front", "middle", "end", "peaked"]


@pytest.mark.parametrize("n", NS)
@pytest.mark.parametrize("P", [12, 16])
def test_reference_round_trip(n, P):
    rng = np.random.default_rng(n * 100 + P)
    tables = np.stack([_table(rng, Q10, P, w) for w in WHERE])
    planes = _planes(rng, tables, n)
    for seg in ([1, 2, 3, 1000], [1000] * 4, [2] * 4):       # several segments (ragged last row), one segment
        pay = R.rans_encode(planes, tables, P, seg)
        assert np.array_equal(R.rans_decode(pay, 4, n, seg, tables, P), planes)


@pytest.mark.parametrize("P", [12, 16])
def test_reference_single_symbol_table(P):
    """f = 2^P for one symbol: the symbols cost nothing, the payload is the offsets and the untouched states."""
    t = np.zeros((1, 7), np.int64)
    t[0, 3] = 1 << P
    assert np.array_equal(coding.frequency_tables(np.array([[0, 0, 0, 9, 0, 0, 0]]), P, keep_zeros=True), t)
    planes = np.full((1, 1000), 3, np.int32)
    pay = R.rans_encode(planes, t, P, 1)                     # 32 rows -> 32 groups, the last one with 8 lanes
    G, lanes = 32, 1000
    assert pay.size == 2 * G + 2 * lanes
    assert (pay[2 * G:].reshape(-1, 2) == [0, 1]).all()      # every state is 2^16
    assert np.array_equal(R.rans_decode(pay, 1, 1000, 1, t, P), planes)


def test_reference_known_answer():
    """N = 1 (Q = 3), P = 12, f = (1, 0, 4095): symbol 1 has frequency 0.  n = 33, one group of two rows; row 1 holds
    lane 0 only.  Rows are coded last to first from x = 2^16 with x_max = f << 20:
      lane 0, symbols 0 (row 0), 0 (row 1):  x = 65536 -> 2^28; then 2^28 >= 1 << 20 emits 0x0000, x = 2^12 -> 2^24;
      lanes 1..31, symbol 2 (row 0):  x = ((65536 // 4095) << 12) + 65536 % 4095 + cum[2] = 65536 + 16 + 1 = 0x00010011.
    Payload: end offset 65 (64 state words + 1 word), lane 0's state (0x0000, 0x0100), 31 x (0x0011, 0x0001), 0x0000."""
    t = np.array([[1, 0, 4095]])
    planes = np.array([[0] + [2] * 31 + [0]])
    want = [65, 0, 0x0000, 0x0100] + [0x0011, 0x0001] * 31 + [0x0000]
    assert R.rans_encode(planes, t, 12, 2).tolist() == want
    assert R.rans_decode(np.array(want), 1, 33, 2, t, 12).tolist() == planes.tolist()
    with pytest.raises(ValueError, match="frequency 0"):
        R.rans_encode(np.array([[1]]), t, 12, 2)


def test_reference_rejects_corrupt_streams():
    rng = np.random.default_rng(5)
    t = _table(rng, Q10, 16, "middle")[None]
    planes = _planes(rng, t, 5000)
    pay = R.rans_encode(planes, t, 16, 40)                   # 157 rows -> 4 groups
    bad = pay.copy()
    bad[200] ^= 0x0100
    with pytest.raises(ValueError):
        R.rans_decode(bad, 1, 5000, 40, t, 16)
    with pytest.raises(ValueError):
        R.rans_decode(pay[:-1], 1, 5000, 40, t, 16)


# ---------------------------------------------------------------------------------------------------------------------
# zero-preserving tables
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("P", [12, 14, 16])
def test_zero_preserving_tables(P):
    rng = np.random.default_rng(P)
    cnt = rng.integers(0, 1000, (5, Q10)) ** 2
    cnt[cnt < 200_000] = 0                                   # about 55 % zeros
    cnt[1, :] = 0
    cnt[1, 77] = 5                                           # one used symbol
    cnt[2, :] = 1                                            # every symbol once: as many used symbols as possible
    cnt[3, :] = 0
    cnt[3, ::500] = 10 ** 9
    cnt[3, 1] = 1                                            # a symbol far below 2^-P still gets 1
    f = coding.frequency_tables(cnt, P, keep_zeros=True)
    assert f.dtype == np.int32 and f.shape == cnt.shape
    assert (f[cnt == 0] == 0).all() and (f[cnt > 0] >= 1).all()
    assert (f.sum(axis=1) == 2 ** P).all()
    assert f[1, 77] == 2 ** P
    assert np.array_equal(f, coding.frequency_tables(cnt.copy(), P, keep_zeros=True))     # deterministic
    with pytest.raises(ValueError, match="integer counts"):
        coding.frequency_tables(cnt.astype(np.float32), P, keep_zeros=True)


def test_frequency_tables_default_unchanged():
    """The default (every entry >= 1) gives the same tables as before keep_zeros existed: BLAKE2b-64 digests of its
    output on seeded entropy models and counts, recorded from the implementation without the keyword."""
    rng = np.random.default_rng(2024)
    em = -np.log2(np.maximum(rng.dirichlet(np.full(Q10, 0.05), size=4), 1e-30)).astype(np.float32)
    cnt = rng.integers(0, 1000, (3, Q10)) ** 2
    cnt[1, ::3] = 0
    cnt[2] = 0
    got = [hashlib.blake2b(coding.frequency_tables(m, P).astype("<i4").tobytes(), digest_size=8).hexdigest()
           for P in (12, 16) for m in (np.minimum(em, np.float32(60)), cnt)]
    assert got == ["98f347cbb25930fd", "dd89d35272aad09b", "defc8b2422e1a932", "0743b68ad906e8d0"]


def test_code_points_fingerprint_and_cum():
    cp = np.linspace(-3.0, 3.0, 7)
    assert coding.code_points_fingerprint(cp) == coding.code_points_fingerprint(cp.copy())
    cp2 = cp.copy()
    cp2[3] = np.nextafter(cp2[3], 1.0)
    assert coding.code_points_fingerprint(cp2) != coding.code_points_fingerprint(cp)
    assert coding.cum_table_shared(np.array([[0, 4096, 0]])).tolist() == [[0, 0, 4096, 4096]]


# ---------------------------------------------------------------------------------------------------------------------
# VBQE header and ABI validation (no device)
# ---------------------------------------------------------------------------------------------------------------------
def _cpu_blob(planes_1, table, P, seg, shape, std=1.25, beta=0.5, fp=1234):
    N = int(np.log2(table.size + 1)) - 1
    hdr = serialize.embedding_header(N, P, shape, seg, std, beta, fp, table)
    return hdr + R.rans_encode(planes_1, table[None], P, seg).astype("<u2").tobytes()


def _blob_case():
    rng = np.random.default_rng(9)
    t = _table(rng, Q10, 16, "middle")
    planes = _planes(rng, t[None], 6000)
    return t, planes, _cpu_blob(planes, t, 16, 40, (200, 30))


def test_embedding_header_parses():
    t, planes, blob = _blob_case()
    h = serialize.read_embedding_header(blob)
    assert (h["max_bits"], h["prob_bits"], h["shape"], h["seg_rows"]) == (10, 16, (200, 30), 40)
    assert (h["empirical_std"], h["beta"], h["fingerprint"]) == (1.25, 0.5, 1234)
    assert np.array_equal(h["table"], t)
    k = int((t > 0).sum())
    assert len(blob) == serialize._HDRE.size + 16 + serialize._HDRE2.size + 6 * k + 2 * h["words"].size


def test_embedding_header_rejects_malformed_blobs():
    t, planes, blob = _blob_case()
    k = int((t > 0).sum())
    tab = serialize._HDRE.size + 16 + serialize._HDRE2.size          # offset of the sparse table's symbols
    pay = tab + 6 * k
    with pytest.raises(ValueError, match="magic"):
        serialize.read_embedding_header(b"VBQ2" + blob[4:])
    for n in (3, serialize._HDRE.size + 5, tab - 1, tab + 7, pay + 2, len(blob) - 2, len(blob) - 1):
        with pytest.raises(ValueError):
            serialize.read_embedding_header(blob[:n])
    with pytest.raises(ValueError, match="after the last plane"):
        serialize.read_embedding_header(blob + b"\0\0")

    def patched(off, fmt, value):
        b = bytearray(blob)
        struct.pack_into(fmt, b, off, value)
        return bytes(b)
    f0 = struct.unpack_from("<I", blob, tab + 2 * k)[0]
    with pytest.raises(ValueError, match="sum"):
        serialize.read_embedding_header(patched(tab + 2 * k, "<I", f0 + 1))        # frequencies off by one
    s0, s1 = struct.unpack_from("<HH", blob, tab)
    with pytest.raises(ValueError, match="unsorted"):
        serialize.read_embedding_header(patched(tab, "<H", s1))                    # a repeated symbol
    with pytest.raises(ValueError, match="unsorted"):
        serialize.read_embedding_header(patched(tab + 2 * (k - 1), "<H", Q10))     # a symbol >= Q
    with pytest.raises(ValueError, match="offset table"):
        serialize.read_embedding_header(patched(pay + 2, "<H", 0x00FF))            # first group end far out
    with pytest.raises(ValueError, match="bad VBQE header"):
        serialize.read_embedding_header(patched(4, "<I", 11))                      # N > 10
    with pytest.raises(ValueError, match="bad VBQE header"):
        serialize.read_embedding_header(patched(8, "<I", 17))                      # prob_bits


def test_embedding_header_applies_the_coders_limits():
    """seg_rows beyond the plane's rows, and shapes whose worst case exceeds the coder's 32-bit offsets, are a
    ValueError on the host, before any allocation or launch."""
    t, planes, blob = _blob_case()
    tab = serialize._HDRE.size + 16

    def patched(off, fmt, value):
        b = bytearray(blob)
        struct.pack_into(fmt, b, off, value)
        return bytes(b)
    for seg in (0, 189, 2 ** 58, 2 ** 62):                     # 6000 symbols are 188 rows
        with pytest.raises(ValueError, match="bad VBQE header"):
            serialize.read_embedding_header(patched(tab, "<Q", seg))
    one = np.zeros(Q10, np.int64)
    one[3] = 1 << 16
    huge = serialize.embedding_header(10, 16, (2 ** 36,), 2 ** 31, 1.0, 1.0, 0, one) + bytes(2 * 66)
    with pytest.raises(ValueError, match="32-bit offsets"):
        serialize.read_embedding_header(huge)


def test_shared_abi_clamps_seg_rows():
    """A segment longer than the plane is the whole plane: sizes do not grow with seg_rows and do not wrap."""
    from vbq_b200 import _lib
    lib = _lib.load()

    def one(v):
        return (ctypes.c_longlong * 1)(v)
    for fn in (lib.vbq_rans_shared_workspace_bytes, lib.vbq_rans_shared_payload_bound):
        want = fn(1, 1000, one(32))
        for seg in (33, 10 ** 9, 2 ** 58, 2 ** 60, 2 ** 62, 2 ** 63 - 1):
            assert fn(1, 1000, one(seg)) == want, (fn, seg)
    need = lib.vbq_rans_shared_workspace_bytes(1, 1000, one(2 ** 60))
    p = ctypes.c_void_p(16)
    assert lib.vbq_rans_shared_encode(p, 1, 1000, one(2 ** 60), 10, 16, p, p, 1 << 30, p, p, p, need - 1, None) == 5


def test_shared_abi_validation_needs_no_gpu():
    from vbq_b200 import _lib
    lib = _lib.load()
    seg = (ctypes.c_longlong * 3)(4, 4, 1)
    assert lib.vbq_rans_shared_payload_bound(1, 1000, seg) == 2 * (2 * 8 + 1000 + 2 * 32 * 8)
    assert lib.vbq_rans_shared_payload_bound(1, 1000, (ctypes.c_longlong * 1)(1)) == 2 * (2 * 32 + 1000 + 2 * 1000)
    assert lib.vbq_rans_shared_payload_bound(0, 1000, seg) == -1
    assert lib.vbq_rans_shared_payload_bound(65, 1000, (ctypes.c_longlong * 65)(*[1] * 65)) == -1
    assert lib.vbq_rans_shared_payload_bound(1, 1000, None) == -1
    assert lib.vbq_rans_shared_workspace_bytes(3, 0, seg) >= 0
    assert lib.vbq_rans_shared_workspace_bytes(1, 10, (ctypes.c_longlong * 1)(0)) == -1
    one = ctypes.c_void_p(16)
    enc = lib.vbq_rans_shared_encode
    big = 1 << 30
    assert enc(one, 1, 1000, seg, 11, 16, one, one, big, one, one, one, big, None) == 3            # N > 10
    assert enc(one, 1, 1000, seg, 10, 17, one, one, big, one, one, one, big, None) == 2            # prob_bits
    assert enc(one, 1, 1000, seg, 10, 11, one, one, big, one, one, one, big, None) == 2
    assert enc(one, 1, 1000, None, 10, 16, one, one, big, one, one, one, big, None) == 1           # seg_rows
    assert enc(None, 1, 1000, seg, 10, 16, one, one, big, one, one, one, big, None) == 1
    assert enc(one, 1, 1000, seg, 10, 16, None, one, big, one, one, one, big, None) == 1
    assert enc(one, 1, 1000, seg, 10, 16, one, one, 16, one, one, one, big, None) == 5             # payload capacity
    assert enc(one, 1, 1000, seg, 10, 16, one, one, big, one, one, one, 8, None) == 5              # workspace
    odd = ctypes.c_void_p(18)
    assert enc(one, 1, 1000, seg, 10, 16, odd, one, big, one, one, one, big, None) == 7            # cum not 4-aligned
    dec = lib.vbq_rans_shared_decode
    assert dec(one, 10, one, 1, 1000, seg, 11, 16, one, one, one, one, one, None) == 3
    assert dec(one, 10, one, 1, 1000, seg, 10, 16, one, None, one, one, one, None) == 1            # z_hat w/o table
    assert dec(one, 10, None, 1, 1000, seg, 10, 16, one, one, one, one, one, None) == 1
    assert dec(one, -1, one, 1, 1000, seg, 10, 16, one, one, one, one, one, None) == 2
    assert dec(one, 10, one, 1, 1000, seg, 10, 16, one, one, one, odd, one, None) == 7


# ---------------------------------------------------------------------------------------------------------------------
# GPU: kernels against the reference, byte for byte
# ---------------------------------------------------------------------------------------------------------------------
def _gpu_encode(planes, tables, N, P, seg):
    from vbq_b200 import ops
    q = torch.from_numpy(np.ascontiguousarray(planes, dtype=np.int32)).cuda()
    cum = torch.from_numpy(coding.cum_table_shared(tables).view(np.int32)).cuda()
    pay, size, status = ops.rans_shared_encode(q, cum, N, P, seg)
    assert int(status.item()) == 0
    return pay[:int(size.item()) // 2].cpu().numpy().view(np.uint16)


def _gpu_decode(pay, n, tables, N, P, seg, cp=None):
    from vbq_b200 import ops
    bounds = serialize._offset_bounds(pay, [serialize.shared_nact(n, s) for s in seg])
    w = torch.from_numpy(pay.view(np.int16).copy()).cuda()
    b = torch.from_numpy(np.ascontiguousarray(bounds, dtype=np.int64)).cuda()
    cum = torch.from_numpy(coding.cum_table_shared(tables).view(np.int32)).cuda()
    q, z, status = ops.rans_shared_decode(w, b, cum, n, seg, N, P, cp)
    assert int(status.item()) == 0
    return q.cpu().numpy(), None if z is None else z.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("n", NS)
@pytest.mark.parametrize("P", [12, 16])
def test_gpu_kernels_match_reference(n, P):
    rng = np.random.default_rng(n * 100 + P)
    tables = np.stack([_table(rng, Q10, P, w) for w in WHERE[:3]])
    planes = _planes(rng, tables, n)
    cp = torch.sort(torch.randn(Q10, device="cuda")).values
    for sel, seg in (([0], [1]), ([1], [1000]), ([0, 1, 2], [1, 2, 1000]), ([2, 0, 1], [3, 3, 3])):
        ref = R.rans_encode(planes[sel], tables[sel], P, seg)
        assert np.array_equal(_gpu_encode(planes[sel], tables[sel], 10, P, seg), ref), (sel, seg)
        q, z = _gpu_decode(ref, n, tables[sel], 10, P, seg, cp)
        assert np.array_equal(q, planes[sel])
        assert np.array_equal(z, cp.cpu().numpy()[planes[sel]])


@pytest.mark.gpu
def test_gpu_single_symbol_and_small_depth():
    t = np.zeros((1, 7), np.int64)
    t[0, 3] = 1 << 16
    planes = np.full((1, 1000), 3, np.int32)
    ref = R.rans_encode(planes, t, 16, 4)
    assert np.array_equal(_gpu_encode(planes, t, 2, 16, [4]), ref)
    assert np.array_equal(_gpu_decode(ref, 1000, t, 2, 16, [4])[0], planes)


@pytest.mark.gpu
def test_gpu_full_embedding_shape_matches_reference():
    """1 M x 300 coordinates as one plane, the symbol statistics of a mid-rate beta, at the default segmentation."""
    import vbq_b200.word_embeddings as WE
    rng = np.random.default_rng(300)
    n = 1_000_000 * 300
    cnt = np.zeros(Q10, np.int64)
    cnt[1023 + np.arange(-60, 61)] = np.exp(-0.5 * (np.arange(-60, 61) / 12.0) ** 2) * 1e6 + 1
    t = coding.frequency_tables(cnt, 16, keep_zeros=True)
    planes = _planes(rng, t, n)
    seg = [WE.default_seg_rows(n, WE._entropy_of_counts(np.bincount(planes[0], minlength=Q10)))]
    ref = R.rans_encode(planes, t, 16, seg)
    assert np.array_equal(_gpu_encode(planes, t, 10, 16, seg), ref)
    assert np.array_equal(_gpu_decode(ref, n, t, 10, 16, seg)[0], planes)


@pytest.mark.gpu
def test_gpu_encoder_status_is_an_error():
    from vbq_b200 import ops
    t = np.array([[1 << 15, 0, 1 << 15]])
    zero = torch.tensor([[0, 2, 1, 0]], dtype=torch.int32, device="cuda")
    with pytest.raises(ValueError, match="frequency 0"):
        serialize.encode_embeddings(zero, t, 1, (4,), [1], 1.0, [1.0], 0)
    out = torch.tensor([[0, 2, 3, 0]], dtype=torch.int32, device="cuda")
    with pytest.raises(ValueError, match="outside"):
        serialize.encode_embeddings(out, t, 1, (4,), [1], 1.0, [1.0], 0)
    cum = torch.from_numpy(coding.cum_table_shared(t).view(np.int32)).cuda()
    assert int(ops.rans_shared_encode(out, cum, 1, 16, 1)[2].item()) == 1
    assert int(ops.rans_shared_encode(zero, cum, 1, 16, 1)[2].item()) == 2


@pytest.mark.gpu
def test_gpu_corrupt_payloads_are_reported_not_faulted():
    t, planes, blob = _blob_case()
    h = serialize.read_embedding_header(blob)
    off = len(blob) - 2 * h["words"].size
    G = h["bounds"].shape[0]
    flipped = bytearray(blob)
    flipped[off + 2 * (2 * G + 64 + 10) + 1] ^= 0x01                   # a byte inside the first group's words
    with pytest.raises(ValueError, match="corrupt"):
        serialize.decode_embedding(bytes(flipped))
    w = h["words"].copy()
    ends = w[0:2 * G:2].astype(np.int64) | (w[1:2 * G:2].astype(np.int64) << 16)

    def with_ends(e, data):
        tab = np.stack([e & 0xFFFF, e >> 16], axis=1).reshape(-1).astype("<u2")
        return blob[:off] + tab.tobytes() + data.astype("<u2").tobytes()
    # a truncated group: the last word of group 0 removed and the later offsets moved down by one
    with pytest.raises(ValueError, match="corrupt"):
        serialize.decode_embedding(with_ends(ends - 1, np.delete(w[2 * G:], ends[0] - 1)))
    # shifted offsets: group 0 claims the first word of group 1 (the table is still well-formed)
    shifted = ends.copy()
    shifted[0] += 1
    with pytest.raises(ValueError, match="corrupt"):
        serialize.decode_embedding(with_ends(shifted, w[2 * G:]))
    assert np.array_equal(serialize.decode_embedding(blob)["qidx"].cpu().numpy(), planes[0])


# ---------------------------------------------------------------------------------------------------------------------
# GPU: GaussianCodebook.compress_to_bytes / decompress_from_bytes
# ---------------------------------------------------------------------------------------------------------------------
def _posteriors(shape, seed):
    rng = np.random.default_rng(seed)
    means = (rng.standard_normal(shape) * 1.2329 - 0.08).astype(np.float32)
    stds = np.exp(rng.standard_normal(shape) * 0.7 + np.log(0.04)).astype(np.float32)
    return means, stds


@pytest.mark.gpu
@pytest.mark.parametrize("exact", [True, False])
def test_gpu_bytes_round_trip_equals_compress_coordinates(exact):
    import vbq_b200
    cb = vbq_b200.GaussianCodebook(1.2356, 10)
    for shape, as_torch in (((3000, 300), False), ((3000, 300), True), ((12345,), False), ((7, 11, 13), True)):
        m, s = _posteriors(shape, sum(shape))
        if as_torch:
            m, s = torch.from_numpy(m).cuda(), torch.from_numpy(s).cuda()
        betas = [0.01, np.float64(1.0), 300.0]
        blobs = cb.compress_to_bytes(m, s, betas, exact=exact)
        assert list(blobs) == betas
        for beta in betas:
            want = cb.compress_coordinates(m, s, beta, exact=exact)[0]
            want = want.cpu().numpy() if as_torch else want
            z = cb.decompress_from_bytes(blobs[beta])
            assert z.dtype == torch.float32 and tuple(z.shape) == shape
            assert np.array_equal(z.cpu().numpy(), want), (shape, beta)
    # a receiver with only the blob
    h = serialize.read_embedding_header(blobs[300.0])
    rx = vbq_b200.GaussianCodebook(h["empirical_std"], h["max_bits"])
    assert torch.equal(rx.decompress_from_bytes(blobs[300.0]), cb.decompress_from_bytes(blobs[300.0]))


@pytest.mark.gpu
def test_gpu_seg_rows_longer_than_the_plane():
    import vbq_b200
    cb = vbq_b200.GaussianCodebook(1.2356, 10)
    m, s = _posteriors((1000, 300), 2)
    big = cb.compress_to_bytes(m, s, [1.0], seg_rows=10 ** 9)[1.0]
    assert serialize.read_embedding_header(big)["seg_rows"] == -(-1000 * 300 // 32)
    assert big == cb.compress_to_bytes(m, s, [1.0], seg_rows=-(-1000 * 300 // 32))[1.0]
    assert np.array_equal(cb.decompress_from_bytes(big).cpu().numpy(), cb.compress_coordinates(m, s, 1.0)[0])
    with pytest.raises(ValueError, match="seg_rows"):
        cb.compress_to_bytes(m, s, [1.0], seg_rows=0)


@pytest.mark.gpu
def test_gpu_decompress_rejects_another_codebook():
    import vbq_b200
    cb = vbq_b200.GaussianCodebook(1.2356, 10)
    m, s = _posteriors((500, 30), 1)
    blob = cb.compress_to_bytes(m, s, [1.0], seg_rows=3)[1.0]
    for other in (vbq_b200.GaussianCodebook(1.2357, 10), vbq_b200.GaussianCodebook(1.2356, 9)):
        with pytest.raises(ValueError, match="another codebook"):
            other.decompress_from_bytes(blob)
    with pytest.raises(ValueError, match="N <= 10"):
        vbq_b200.GaussianCodebook(1.2356, 11).compress_to_bytes(m, s, [1.0])


@pytest.mark.gpu
def test_gpu_rate_near_empirical_entropy():
    """Seeded 100 k x 300 posteriors at three betas, default segmentation: the payload is within the cross-entropy
    under the integer table plus the flushed states and offsets (+0.1 %), and the blob within 1 % of empirical_entropy
    plus its header and table.  At the grid's lowest rate (beta = 1e5, about 0.002 bits per coordinate here) one
    segment's states alone are more than 1 % of the entropy; there the blob must be below the VBQ2 floor of 0.0458 bits
    per coordinate."""
    import vbq_b200
    from vbq_b200.word_embeddings import empirical_entropy
    cb = vbq_b200.GaussianCodebook(1.2356, 10)
    shape = (100_000, 300)
    n = shape[0] * shape[1]
    m, s = _posteriors(shape, 100)
    m, s = torch.from_numpy(m).cuda(), torch.from_numpy(s).cuda()
    betas = [0.01, 10.0, 1000.0, 1e5]
    blobs = cb.compress_to_bytes(m, s, betas)
    for beta in betas:
        blob = blobs[beta]
        h = serialize.read_embedding_header(blob)
        q = serialize.decode_embedding(blob)["qidx"].cpu().numpy()
        G = h["bounds"].shape[0]
        payload_bits = 16 * h["words"].size
        xent = _xent_bits(q[None], h["table"][None])
        assert payload_bits <= 1.001 * xent + 1024 * G + 32 * G, (beta, payload_bits, xent, G)
        ideal = empirical_entropy(cb.compress_coordinates(m, s, beta)[0])
        header_bits = 8 * (len(blob) - 2 * h["words"].size)
        if beta < 1e5:
            assert abs(8 * len(blob) - (ideal + header_bits)) <= 0.01 * ideal, (beta, 8 * len(blob), ideal, header_bits)
    assert 8 * len(blobs[1e5]) < 0.0458 * n
