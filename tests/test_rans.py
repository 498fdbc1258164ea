"""rANS entropy coding of the sorted quantile indices (csrc/rans.cu, serialize.encode / decode, compress_to_bytes):
CPU tests of the reference coder, the frequency tables, the ABI and the VBQ2 header; GPU tests of the kernels against
the reference, byte for byte, and of the quantizer's bytes -> z_hat path."""
import ctypes
import pickle

import numpy as np
import pytest
import torch

import rans_reference as R
from oracle import vbq_oracle as O
from vbq_b200 import coding, serialize


def _tables(rng, n_planes, C, Q, P, peaked):
    """Integer tables from random counts: peaked ones put most mass on a few symbols per channel."""
    if peaked:
        cnt = rng.integers(0, 3, (n_planes, C, Q))
        cnt[..., rng.integers(0, Q, 3)] += 10_000
    else:
        cnt = rng.integers(0, 50, (n_planes, C, Q)) ** 3
    return np.stack([coding.frequency_tables(cnt[p], P) for p in range(n_planes)])


def _planes(rng, tables, items, rows):
    n_planes, C, Q = tables.shape
    p = tables / tables.sum(-1, keepdims=True)
    out = np.zeros((n_planes, items, rows, C), np.int32)
    for i in range(n_planes):
        for c in range(C):
            out[i, :, :, c] = rng.choice(Q, size=(items, rows), p=p[i, c])
    return out


def _xent_bits(planes, tables):
    P = int(np.log2(tables[0, 0].sum()))
    bits = 0.0
    for i in range(planes.shape[0]):
        f = tables[i].T[planes[i].reshape(-1, planes.shape[-1]), np.arange(planes.shape[-1])]
        bits += float(-np.log2(f / 2.0 ** P).sum())
    return bits


# (n_planes, items, item_rows, C, N, seg_rows, prob_bits, peaked)
CASES = [(1, 1, 0, 5, 4, 1, 16, False), (1, 1, 1, 1, 0, 1, 12, False), (1, 2, 1, 37, 10, 1, 16, True),
         (1, 1, 1537, 32, 10, 1537, 16, False), (2, 3, 17, 5, 1, 5, 14, True), (1, 2, 300, 192, 10, 300, 16, True),
         (3, 2, 64, 37, 4, 20, 15, False), (1, 1, 1537, 1, 10, 512, 12, True), (3, 4, 33, 192, 10, 33, 16, False)]


def _case(n_planes, items, rows, C, N, seg, P, peaked):
    rng = np.random.default_rng(hash((n_planes, items, rows, C, N, seg, P, peaked)) % 2 ** 32)
    t = _tables(rng, n_planes, C, 2 ** (N + 1) - 1, P, peaked)
    return t, _planes(rng, t, items, rows)


@pytest.mark.parametrize("case", CASES)
def test_reference_round_trip(case):
    n_planes, items, rows, C, N, seg, P, peaked = case
    t, planes = _case(*case)
    pay = R.rans_encode(planes, t, P, seg)
    assert np.array_equal(R.rans_decode(pay, n_planes, items, rows, C, seg, t, P), planes)


def test_reference_known_answer():
    """Two lanes, three rows, N = 1, P = 12, worked by hand (rows coded last to first, x0 = 2^16, x_max = f << 20):
    channel 0, f = (2048, 1024, 1024), symbols 0 1 2:  x = 65536 -> 265216 -> 1062912 -> 2125824 = 0x00207000;
    channel 1, f = (1, 4094, 1), symbols 0 1 0:  x = 65536 -> 2^28 -> 268566593 = 0x10020041 >= 1 << 20 at row 0, so it
    emits 0x0041 and 0x1002 -> 0x01002000.  Payload: end offset 5 (two words), states (low, high), the one word."""
    t = np.array([[[2048, 1024, 1024], [1, 4094, 1]]])
    planes = np.array([[[[0, 0], [1, 1], [2, 0]]]])
    want = [5, 0, 0x7000, 0x0020, 0x2000, 0x0100, 0x0041]
    pay = R.rans_encode(planes, t, 12, 3)
    assert pay.tolist() == want
    assert R.rans_decode(np.array(want), 1, 1, 3, 2, 3, t, 12).tolist() == planes.tolist()


@pytest.mark.parametrize("peaked", [False, True])
def test_coded_bits_near_cross_entropy(peaked):
    rng = np.random.default_rng(7 + peaked)
    C, N, items, rows, P = 37, 10, 2, 2000, 16
    t = _tables(rng, 1, C, 2 ** (N + 1) - 1, P, peaked)
    planes = _planes(rng, t, items, rows)
    pay = R.rans_encode(planes, t, P, rows)
    groups = items * 2
    overhead = 32 * C * items + 32 * groups                  # a 32-bit state per lane and group, a 32-bit offset per group
    assert 16 * pay.size <= 1.003 * _xent_bits(planes, t) + overhead


def test_reference_rejects_corrupt_streams():
    t, planes = _case(1, 2, 200, 37, 10, 200, 16, False)
    pay = R.rans_encode(planes, t, 16, 200)
    bad = pay.copy()
    bad[20] ^= 0x0100                                        # one flipped byte inside the first group's words
    with pytest.raises(ValueError):
        R.rans_decode(bad, 1, 2, 200, 37, 200, t, 16)
    # drop the last word of group 0 and shift the later offsets: a group that runs out of words
    G = 4
    ends = (pay[0:2 * G:2].astype(np.int64) | (pay[1:2 * G:2].astype(np.int64) << 16))
    cut = ends.copy()
    cut -= 1
    tab = np.stack([cut & 0xFFFF, cut >> 16], axis=1).reshape(-1).astype(np.uint16)
    short = np.concatenate([tab, np.delete(pay[2 * G:], ends[0] - 1)])
    with pytest.raises(ValueError):
        R.rans_decode(short, 1, 2, 200, 37, 200, t, 16)


# ---------------------------------------------------------------------------------------------------------------------
# frequency tables
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("P", [12, 14, 15, 16])
def test_frequency_tables_sum_and_floor(P):
    rng = np.random.default_rng(P)
    Q = 2047
    em = -np.log2(np.maximum(rng.dirichlet(np.full(Q, 0.05), size=6), 1e-30)).astype(np.float32)
    em = np.minimum(em, np.float32(60))
    f = coding.frequency_tables(em, P)
    assert f.dtype == np.int32 and f.shape == (6, Q)
    assert (f >= 1).all() and (f.sum(1) == 2 ** P).all()
    assert np.array_equal(f, coding.frequency_tables(em.copy(), P))          # deterministic
    counts = rng.integers(0, 1000, (3, Q))
    counts[1] = 0                                                            # a channel without counts: uniform
    g = coding.frequency_tables(counts, P)
    assert (g >= 1).all() and (g.sum(1) == 2 ** P).all()
    assert g[1].max() - g[1].min() <= 1


def test_frequency_tables_extremes():
    Q = 2047
    one_hot = np.full((1, Q), 60.0, np.float32)
    one_hot[0, 5] = 0.0
    f = coding.frequency_tables(one_hot, 16)
    assert f[0, 5] == 2 ** 16 - (Q - 1) and (np.delete(f[0], 5) == 1).all()
    uni = coding.frequency_tables(np.full((2, Q), np.log2(Q), np.float32), 16)
    assert (uni.sum(1) == 2 ** 16).all() and uni.max() - uni.min() <= 1
    assert coding.frequency_tables(np.zeros((1, 1), np.float32), 12).tolist() == [[4096]]
    with pytest.raises(ValueError):
        coding.frequency_tables(one_hot, 11)
    with pytest.raises(ValueError):
        coding.frequency_tables(np.zeros((1, 4097)), 12)


def test_frequency_tables_near_ideal_on_quantized_latents():
    """Cross-entropy under the integer tables is within 0.25 % of the sum of num_bits (the fitted models' ideal code
    lengths) on latents quantized by the reference quantizer."""
    import vbq_test_helpers as H
    C, N = 8, 10
    pr = H.make_prior(C, seed=4)
    q = O.QuantizerNP(C, N)
    q.build_code_points(lambda xi: pr.inverse_cdf_f64(xi))
    mu, _, lv = H.make_latents(pr, 6000, 5, edge_cases=False)
    lambs = [2.0 ** -6, 0.5, 8.0]
    q.build_entropy_models_from_latents(mu[:3000], lv[:3000], lambs, 1)
    out = q.compress_latents(mu[3000:], lv[3000:], lambs)
    for l in lambs:
        I = q.sorted_index(out["Z_hat"][l].reshape(-1, C))
        ideal = float(out["num_bits"][l].astype(np.float64).sum())
        f = coding.frequency_tables(q.entropy_models[l], 16)
        xent = float(-np.log2(np.take_along_axis(f.T, I, 0) / 2.0 ** 16).sum())
        assert abs(xent - ideal) <= 0.0025 * ideal, (l, xent, ideal)


def test_fingerprint_and_cum():
    f = np.array([[1, 2, 4093], [4094, 1, 1]])
    assert coding.fingerprint(f) == R.fingerprint(f)
    g = f.copy()
    g[0, :2] = [2, 1]
    assert coding.fingerprint(g) != coding.fingerprint(f)
    assert coding.cum_table(f).tolist() == [[0, 1, 3], [0, 4094, 4095]]
    assert coding.prob_bits_of(f) == 12


# ---------------------------------------------------------------------------------------------------------------------
# ABI and header checks (no device)
# ---------------------------------------------------------------------------------------------------------------------
def test_abi_validation_needs_no_gpu():
    from vbq_b200 import _lib
    lib = _lib.load()
    assert lib.vbq_rans_payload_bound(1, 1, 1536, 192, 1536) == 2 * (2 * 6 + 192 * 1538)
    assert lib.vbq_rans_payload_bound(3, 24, 1536, 192, 1536) == 3 * 2 * (2 * 144 + 24 * 192 * 1538)
    assert lib.vbq_rans_workspace_bytes(1, 1, 0, 5, 1) >= 0
    assert lib.vbq_rans_payload_bound(0, 1, 1, 1, 1) == -1 and lib.vbq_rans_payload_bound(1, 1, 1, 0, 1) == -1
    assert lib.vbq_rans_workspace_bytes(1, 1, 8, 4, 0) == -1
    one = ctypes.c_void_p(16)
    enc = lib.vbq_rans_encode
    assert enc(one, 1, 1, 8, 4, 8, 11, 16, one, one, 1 << 30, one, one, one, 1 << 30, None) == 3     # N > 10
    assert enc(one, 1, 1, 8, 4, 8, 10, 17, one, one, 1 << 30, one, one, one, 1 << 30, None) == 2     # prob_bits
    assert enc(one, 1, 1, 8, 4, 8, 10, 11, one, one, 1 << 30, one, one, one, 1 << 30, None) == 2
    assert enc(one, 1, 1, -1, 4, 8, 10, 16, one, one, 1 << 30, one, one, one, 1 << 30, None) == 2    # rows
    assert enc(one, 1, 1, 8, 4, 0, 10, 16, one, one, 1 << 30, one, one, one, 1 << 30, None) == 2     # seg_rows
    assert enc(None, 1, 1, 8, 4, 8, 10, 16, one, one, 1 << 30, one, one, one, 1 << 30, None) == 1
    assert enc(one, 1, 1, 8, 4, 8, 10, 16, one, one, 16, one, one, one, 1 << 30, None) == 5          # payload capacity
    assert enc(one, 1, 1, 8, 4, 8, 10, 16, one, one, 1 << 30, one, one, one, 8, None) == 5           # workspace
    dec = lib.vbq_rans_decode
    assert dec(one, 10, one, 1, 1, 8, 4, 8, 11, 16, one, one, one, one, one, None) == 3
    assert dec(one, 10, one, 1, 1, 8, 4, 8, 1, 12, one, None, one, one, one, None) == 1               # z_hat w/o table
    assert dec(one, -1, one, 1, 1, 8, 4, 8, 1, 12, one, one, one, one, one, None) == 2
    assert dec(one, 10, one, 1, 1, 8, 4, 8, 2, 12, one, one, one, ctypes.c_void_p(18), one, None) == 7


def _cpu_blob(t, planes, P, seg, lambdas, embed=False, height=0):
    """A VBQ2 blob built from the reference payload (no device)."""
    n_planes, items, rows, C = planes.shape
    f = dict(N=int(np.log2(t.shape[-1] + 1)) - 1, C=C, P=P, n_planes=n_planes, items=items, item_rows=rows, seg_rows=seg)
    hdr = serialize._header(f, lambdas, [coding.fingerprint(x) for x in t], height, t if embed else None)
    return b"".join(hdr) + R.rans_encode(planes, t, P, seg).astype("<u2").tobytes()


def test_header_parsing_rejects_bad_streams():
    t, planes = _case(2, 2, 40, 37, 4, 40, 16, False)
    blob = _cpu_blob(t, planes, 16, 40, [0.5, 8.0], height=8)
    h = serialize.read_header(blob)
    assert (h["n_planes"], h["items"], h["item_rows"], h["C"], h["prob_bits"], h["height"]) == (2, 2, 40, 37, 16, 8)
    assert h["lambdas"] == [0.5, 8.0] and h["fingerprints"][1] == coding.fingerprint(t[1])
    with pytest.raises(ValueError, match="magic"):
        serialize.decode(b"VBQ1" + blob[4:], tables=list(t))
    for n in (10, serialize._HDR2.size + 3, len(blob) - 2, len(blob) - 1):
        with pytest.raises(ValueError):
            serialize.decode(blob[:n], tables=list(t))
    with pytest.raises(ValueError, match="after the last plane"):
        serialize.decode(blob + b"\0\0", tables=list(t))
    off = serialize._HDR2.size + 2 * serialize._PLANE2.size
    bad = bytearray(blob)
    bad[off + 2] = 0xFF                                        # high half of the first group's end offset
    with pytest.raises(ValueError, match="offset table"):
        serialize.decode(bytes(bad), tables=list(t))
    with pytest.raises(ValueError, match="fingerprint"):
        serialize.decode(blob, tables=[t[1], t[0]])
    with pytest.raises(ValueError, match="embeds no"):
        serialize.decode(blob)
    with pytest.raises(ValueError, match="no table for lambda"):
        serialize.decode(blob, tables={0.5: t[0]})
    emb = _cpu_blob(t, planes, 16, 40, [0.5, 8.0], embed=True)
    assert np.array_equal(serialize.read_header(emb)["tables"], t)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: kernels against the reference, byte for byte
# ---------------------------------------------------------------------------------------------------------------------
def _gpu_payload(planes, t, N, P, seg):
    from vbq_b200 import ops
    q = torch.from_numpy(np.ascontiguousarray(planes, dtype=np.int32)).cuda()
    cum = torch.from_numpy(coding.cum_table(t).view(np.int16)).cuda()
    pay, size, status = ops.rans_encode(q, cum, N, P, seg)
    assert int(status.item()) == 0
    return pay[:int(size.item()) // 2].cpu().numpy().view(np.uint16)


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES)
def test_gpu_encode_decode_match_reference(case):
    from vbq_b200 import ops
    n_planes, items, rows, C, N, seg, P, peaked = case
    t, planes = _case(*case)
    ref = R.rans_encode(planes, t, P, seg)
    assert np.array_equal(_gpu_payload(planes, t, N, P, seg), ref)
    lambdas = [0.25 * (i + 1) for i in range(n_planes)]
    blob = _cpu_blob(t, planes, P, seg, lambdas)
    cp = torch.sort(torch.randn(C, 2 ** (N + 1) - 1, device="cuda"), dim=1).values
    out = serialize.decode(blob, tables=list(t), code_points=cp)
    assert np.array_equal(out["qidx"].cpu().numpy(), planes)
    want = cp.cpu().numpy()[np.arange(C), planes]
    assert np.array_equal(out["zhat"].cpu().numpy(), want)
    assert out["lambdas"] == lambdas
    # serialize.encode is the same bytes as the reference blob
    q = torch.from_numpy(planes.reshape(n_planes, items * rows, C)).cuda()
    assert serialize.encode(q, t, N, items=items, seg_rows=seg, lambdas=lambdas) == blob
    del ops


def _kodak_case():
    """The Kodak-shaped batch of bench.py (24 images of 32 x 48 latents, C = 192, N = 10), three lambdas."""
    import vbq_b200
    from vbq_b200 import ops
    import vbq_test_helpers as H
    C, N, B, Hh, W = 192, 10, 24, 32, 48
    pr = H.make_prior(C, seed=11)
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N)
    q.set_code_points(ops.build_code_points_learned(torch.from_numpy(pr.packed()).cuda(), N))
    # the latents of H.make_latents (mu = F^-1(U(0.001, 0.999)), logvar ~ N(-3, 1.5^2)), with F^-1 on the device
    rng = np.random.default_rng(12)
    params = torch.from_numpy(pr.packed()).cuda()
    mu = ops.learned_inverse_cdf(params, torch.from_numpy(rng.uniform(0.001, 0.999, (2 * B * Hh * W, C))).cuda())
    mu = mu.cpu().numpy()
    lv = rng.normal(-3.0, 1.5, (2 * B * Hh * W, C)).astype(np.float32)
    lambs = [2.0 ** -6, 0.5, 8.0]
    q.build_entropy_models_from_latents(mu[:B * Hh * W], lv[:B * Hh * W], lambs, 1)
    return q, mu[B * Hh * W:].reshape(B, Hh, W, C), lv[B * Hh * W:].reshape(B, Hh, W, C), lambs


@pytest.mark.gpu
def test_gpu_kodak_shape_matches_reference():
    from vbq_b200 import ops
    q, mu, lv, lambs = _kodak_case()
    B, Hh, W, C = mu.shape
    out = q.quantize(torch.from_numpy(mu.reshape(-1, C)).cuda(), torch.from_numpy(lv.reshape(-1, C)).cuda(), lambs,
                     logvar=True, outputs=ops.OUT_QIDX)
    planes = out["qidx"].cpu().numpy().reshape(3, B, Hh * W, C)
    t = np.stack([q.rans_tables(l) for l in lambs])
    ref = R.rans_encode(planes, t, 16, Hh * W)
    assert np.array_equal(_gpu_payload(planes, t, 10, 16, Hh * W), ref)           # three planes, one launch
    assert np.array_equal(_gpu_payload(planes[1:2], t[1:2], 10, 16, Hh * W),
                          R.rans_encode(planes[1:2], t[1:2], 16, Hh * W))          # one plane
    blob = _cpu_blob(t, planes, 16, Hh * W, lambs)
    dec = serialize.decode(blob, tables=list(t), code_points=q.code_points_by_channel)
    assert np.array_equal(dec["qidx"].cpu().numpy(), planes)


@pytest.mark.gpu
def test_gpu_compress_to_bytes_end_to_end():
    """compress_to_bytes -> pickle the quantizer -> a fresh object -> decompress_from_bytes gives compress_latents'
    Z_hat bit for bit for every image and lambda, in about Σ num_bits plus the stated overhead."""
    import vbq_b200
    q, mu, lv, lambs = _kodak_case()
    B, Hh, W, C = mu.shape
    blobs = q.compress_to_bytes(mu, lv, lambs)
    ref = q.compress_latents(mu, lv, lambs)
    q2 = pickle.loads(pickle.dumps(q))
    assert isinstance(q2, vbq_b200.ChannelwisePriorCDFQuantizer)
    groups = (C + 31) // 32
    hdr_bits = 8 * (serialize._HDR2.size + serialize._PLANE2.size)
    for l in lambs:
        assert len(blobs[l]) == B
        for b in range(B):
            z = q2.decompress_from_bytes(blobs[l][b])
            assert tuple(z.shape) == (1, Hh, W, C)
            assert np.array_equal(z.cpu().numpy()[0], ref["Z_hat"][l][b])
            ideal = float(ref["num_bits"][l][b].astype(np.float64).sum())
            assert 8 * len(blobs[l][b]) <= 1.003 * ideal + 32 * C + 32 * groups + hdr_bits


@pytest.mark.gpu
def test_gpu_corrupt_payloads_are_reported_not_faulted():
    t, planes = _case(1, 2, 200, 37, 10, 200, 16, False)
    blob = bytearray(_cpu_blob(t, planes, 16, 200, [1.0]))
    off = serialize._HDR2.size + serialize._PLANE2.size
    flipped = bytearray(blob)
    flipped[off + 2 * 40 + 1] ^= 0x01                         # a byte inside the first group's words
    with pytest.raises(ValueError, match="corrupt"):
        serialize.decode(bytes(flipped), tables=list(t))
    # a truncated group: its last word removed and the later offsets moved down by one
    G = 4
    w = np.frombuffer(bytes(blob[off:]), dtype="<u2").copy()
    ends = w[0:2 * G:2].astype(np.int64) | (w[1:2 * G:2].astype(np.int64) << 16)
    cut = ends - 1
    tab = np.stack([cut & 0xFFFF, cut >> 16], axis=1).reshape(-1).astype("<u2")
    short = np.concatenate([tab, np.delete(w[2 * G:], ends[0] - 1)])
    with pytest.raises(ValueError, match="corrupt"):
        serialize.decode(bytes(blob[:off]) + short.astype("<u2").tobytes(), tables=list(t))
    # the intact stream still decodes after the failures
    assert np.array_equal(serialize.decode(bytes(blob), tables=list(t))["qidx"].cpu().numpy(), planes)


@pytest.mark.gpu
def test_gpu_embedded_tables_from_counts():
    """A stream coded from its own counts carries its tables."""
    from vbq_b200 import ops
    rng = np.random.default_rng(3)
    C, N, rows = 5, 4, 999
    qi = torch.from_numpy(rng.integers(0, 7, (rows, C)).astype(np.int32)).cuda()
    t = coding.frequency_tables(ops.symbol_histogram(qi, N).cpu().numpy(), 14)
    blob = serialize.encode(qi, t, N, embed_tables=True, seg_rows=100)
    out = serialize.decode(blob)
    assert torch.equal(out["qidx"][0, 0], qi)
    with pytest.raises(ValueError, match="outside"):
        serialize.encode(qi + 40, t, N)
