"""Many VBQ2 blobs in one launch (vbq_rans_decode_batch, serialize.decode_many, decompress_many): CPU tests of the work
list against the reference layout, of the checks made before any launch and of the ABI's argument validation; GPU tests
of decode_many against decode, bit for bit, of the quantizer's receiver path, of corrupt blobs and of bad raw units."""
import ctypes

import numpy as np
import pytest
import torch

import rans_reference as R
from vbq_b200 import coding, serialize


def _table(C, N, P, seed):
    rng = np.random.default_rng(seed)
    return coding.frequency_tables(rng.integers(0, 50, (C, 2 ** (N + 1) - 1)) ** 3, P)


def _symbols(rng, tables, items, rows):
    """(L, items, rows, C) symbols drawn from each plane's table (inverse CDF per channel)."""
    L, C, Q = tables.shape
    out = np.zeros((L, items, rows, C), np.int32)
    for p in range(L):
        cdf = np.cumsum(tables[p], axis=1) / tables[p].sum(axis=1, keepdims=True)
        u = rng.random((items * rows, C))
        for c in range(C):
            out[p, :, :, c] = np.minimum(np.searchsorted(cdf[c], u[:, c], side="right"), Q - 1).reshape(items, rows)
    return out


def _cpu_blob(t, planes, P, seg, lambdas, height=0):
    """A VBQ2 blob from the reference payload (no device)."""
    L, items, rows, C = planes.shape
    f = dict(N=int(np.log2(t.shape[-1] + 1)) - 1, C=C, P=P, n_planes=L, items=items, item_rows=rows, seg_rows=seg)
    hdr = serialize._header(f, lambdas, [coding.fingerprint(x) for x in t], height)
    return b"".join(hdr) + R.rans_encode(planes, t, P, seg).astype("<u2").tobytes()


# (n_planes, items, item_rows, seg_rows, height, table ids of the planes) of each blob; C = 37 or 1, N = 4
SPECS = [(1, 1, 12, 12, 3, [0]), (2, 3, 7, 3, 0, [1, 0]), (1, 2, 9, 1, 0, [2]), (3, 1, 5, 100, 5, [0, 1, 2]),
         (1, 1, 0, 4, 0, [1]), (1, 1, 33, 8, 0, [1])]


def _cpu_case(C, seed=0):
    N, P = 4, 14
    rng = np.random.default_rng(seed)
    tabs = [_table(C, N, P, seed + 10 + i) for i in range(3)]
    blobs, planes = [], []
    for L, items, rows, seg, height, ids in SPECS:
        t = np.stack([tabs[i] for i in ids])
        p = _symbols(rng, t, items, rows)
        blobs.append(_cpu_blob(t, p, P, seg, [float(i) for i in ids], height))
        planes.append(p)
    return tabs, blobs, planes, N, P


def _decode_unit(words, u, tables, C, P):
    """NumPy decoder of one work unit: (rows, nact) symbols of lanes 32 cg + j from the unit's word range alone."""
    start, end, out, rows, table, cg, blob = (int(v) for v in u)
    nact = min(32, C - 32 * cg)
    f = tables[table][32 * cg:32 * cg + nact].astype(np.int64)
    cum = np.cumsum(f, axis=1) - f
    w = words.astype(np.int64)
    x = w[start:start + 2 * nact:2] | (w[start + 1:start + 2 * nact:2] << 16)
    pos = start + 2 * nact
    sym = np.zeros((rows, nact), np.int64)
    lanes = np.arange(nact)
    for r in range(rows):
        slot = x & ((1 << P) - 1)
        s = np.array([np.searchsorted(cum[j], slot[j], side="right") - 1 for j in range(nact)])
        x = f[lanes, s] * (x >> P) + slot - cum[lanes, s]
        for j in np.flatnonzero(x < 1 << 16):
            assert pos < end
            x[j] = (x[j] << 16) | w[pos]
            pos += 1
        sym[r] = s
    assert (x == 1 << 16).all() and pos == end
    return sym


@pytest.mark.parametrize("C", [37, 1])
def test_batch_plan_against_reference(C):
    tabs, blobs, planes, N, P = _cpu_case(C)
    headers = [serialize.read_header(b) for b in blobs]
    payloads = [serialize._payload_words(b, h) for b, h in zip(blobs, headers)]
    plan = serialize.batch_plan(headers, payloads, [s[5] for s in SPECS])
    units, ctas, CG = plan["units"], plan["ctas"], -(-C // 32)
    # every group of every blob exactly once
    want = sorted((b, p, i, s, g) for b, (L, items, rows, seg, _, _) in enumerate(SPECS) for p in range(L)
                  for i in range(items) for s in range(-(-rows // seg)) for g in range(CG))
    got = []
    for u in units:
        b = int(u[6])
        L, items, rows, seg = SPECS[b][:4]
        e = (int(u[2]) - int(plan["offsets"][b]) - 32 * int(u[5])) // C
        p, rest = divmod(e, items * rows)
        i, r0 = divmod(rest, rows)
        assert r0 % seg == 0 and int(u[3]) == min(seg, rows - r0) and int(u[4]) == SPECS[b][5][p]
        got.append((b, p, i, r0 // seg, int(u[5])))
    assert sorted(got) == want and len(got) == len(set(got))
    # descriptors: consecutive, in order, at most 8 units of one (table, cg) each
    assert ctas[:, 0].tolist() == np.concatenate([[0], np.cumsum(ctas[:-1, 1])]).tolist()
    assert int(ctas[:, 1].sum()) == len(units) and (ctas[:, 1] >= 1).all() and (ctas[:, 1] <= 8).all()
    for first, count, table, cg in ctas:
        assert (units[first:first + count, 4] == table).all() and (units[first:first + count, 5] == cg).all()
    # the units' outputs tile [0, n_out) once, and their word ranges are disjoint
    cover = np.zeros(plan["n_out"], np.int64)
    for u in units:
        nact = min(32, C - 32 * int(u[5]))
        idx = int(u[2]) + np.arange(int(u[3]))[:, None] * C + np.arange(nact)[None, :]
        np.add.at(cover, idx.reshape(-1), 1)
    assert (cover == 1).all()
    r = units[np.argsort(units[:, 0])]
    assert (r[1:, 0] >= r[:-1, 1]).all()
    # decoding every unit from its fields alone gives the reference's symbols in the right place
    out = np.full(plan["n_out"], -1, np.int64)
    for u in units:
        sym = _decode_unit(plan["words"], u, tabs, C, P)
        nact = sym.shape[1]
        out[int(u[2]) + np.arange(int(u[3]))[:, None] * C + np.arange(nact)[None, :]] = sym
    for b, p in enumerate(planes):
        ref = R.rans_decode(payloads[b], *p.shape, SPECS[b][3], [tabs[i] for i in SPECS[b][5]], P)
        o, n = int(plan["offsets"][b]), int(plan["sizes"][b])
        assert np.array_equal(out[o:o + n].reshape(p.shape), ref) and np.array_equal(ref, p)


def test_decode_many_checks_before_any_launch():
    """Every failure here raises on the host, before an upload: the device given cannot even be reached."""
    tabs, blobs, planes, N, P = _cpu_case(37)
    tables = {float(i): tabs[i] for i in range(3)}
    no_device = "cuda:99"
    other_c = _cpu_case(1)[1][0]
    with pytest.raises(ValueError, match="blob 6 has C=1"):
        serialize.decode_many(blobs + [other_c], tables=tables, device=no_device)
    t5 = _table(37, 5, P, 3)
    p5 = _symbols(np.random.default_rng(1), t5[None], 1, 4)
    other_n = _cpu_blob(t5[None], p5, P, 4, [0.0])
    with pytest.raises(ValueError, match="blob 1 has C=37 N=5"):
        serialize.decode_many([blobs[0], other_n], tables={0.0: t5}, device=no_device)
    with pytest.raises(ValueError, match="blob 2: no table for lambda 2.0"):
        serialize.decode_many(blobs, tables={0.0: tabs[0], 1.0: tabs[1]}, device=no_device)
    swapped = {0.0: tabs[0], 1.0: tabs[2], 2.0: tabs[1]}
    with pytest.raises(ValueError, match="blob 1: the frequency table of plane 0 .lambda 1.0. has another fingerprint"):
        serialize.decode_many(blobs, tables=swapped, device=no_device)
    with pytest.raises(ValueError, match="blob 0 embeds no"):
        serialize.decode_many(blobs, device=no_device)
    for cut in (10, serialize._HDR2.size + 3, len(blobs[1]) - 2, len(blobs[1]) - 1):
        with pytest.raises(ValueError):
            serialize.decode_many([blobs[0], blobs[1][:cut]], tables=tables, device=no_device)
    with pytest.raises(ValueError, match="after the last plane"):
        serialize.decode_many([blobs[0], blobs[1] + b"\0\0"], tables=tables, device=no_device)
    assert serialize.decode_many([], device=no_device) == []


def test_decompress_many_checks_before_any_launch():
    import vbq_b200
    C, N = 37, 4
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N, device="cuda:99")
    rng = np.random.default_rng(5)
    q.entropy_models = {0.5: -np.log2(rng.dirichlet(np.ones(31), C)), 8.0: -np.log2(rng.dirichlet(np.ones(31), C))}
    t = {l: q.rans_tables(l) for l in (0.5, 8.0)}

    def blob(lam, Hh, W):
        p = _symbols(rng, t[lam][None], 1, Hh * W)
        return _cpu_blob(t[lam][None], p, 16, Hh * W, [lam], Hh)
    a, b = blob(0.5, 3, 4), blob(8.0, 4, 3)
    assert q.decompress_many([]) == []
    with pytest.raises(KeyError):
        q.decompress_many([a, blob(0.5, 3, 4).replace(np.float64(0.5).tobytes(), np.float64(2.0).tobytes(), 1)])
    with pytest.raises(ValueError, match="stack=True needs blobs of one shape"):
        q.decompress_many([a, b], stack=True)


def test_abi_validation_needs_no_gpu():
    from vbq_b200 import _lib
    lib = _lib.load()
    one = ctypes.c_void_p(16)
    dec = lib.vbq_rans_decode_batch

    def call(**kw):
        a = dict(payload=one, words=10, cum=one, pb=one, n_tables=1, C=4, N=4, units=one, n_units=1, ctas=one,
                 n_ctas=1, n_blobs=1, cp=one, n_out=10, q=one, z=one, status=one)
        a.update(kw)
        return dec(a["payload"], a["words"], a["cum"], a["pb"], a["n_tables"], a["C"], a["N"], a["units"],
                   a["n_units"], a["ctas"], a["n_ctas"], a["n_blobs"], a["cp"], a["n_out"], a["q"], a["z"],
                   a["status"], None)
    assert call(N=11) == 3 and call(N=-1) == 3
    for bad in (dict(C=0), dict(words=-1), dict(n_units=-1), dict(n_ctas=-1), dict(n_blobs=-1), dict(n_out=-1),
                dict(n_tables=-1), dict(n_units=0), dict(n_blobs=0), dict(n_tables=0), dict(n_ctas=1 << 31)):
        assert call(**bad) == 2, bad
    for bad in ("payload", "cum", "pb", "units", "ctas", "status", "cp"):
        assert call(**{bad: None}) == 1, bad
    for bad in ("payload", "pb", "units", "ctas", "cp", "q", "z", "status"):
        assert call(**{bad: ctypes.c_void_p(17 if bad == "payload" else 20 if bad in ("units", "ctas") else 18)}) == 7, bad
    assert call(cum=ctypes.c_void_p(17)) == 7
    # no work and no status entries: nothing to launch or clear, so no device is touched
    assert call(payload=None, cum=None, pb=None, units=None, n_units=0, ctas=None, n_ctas=0, n_blobs=0, cp=None, z=None,
                q=None, status=None) == 0


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _gpu_blob(rng, tables, lambdas, items, rows, seg, height=0):
    t = np.stack(tables)
    p = _symbols(rng, t, items, rows)
    q = torch.from_numpy(p.reshape(len(tables), items * rows, -1)).cuda()
    return serialize.encode(q, t, int(np.log2(t.shape[-1] + 1)) - 1, items=items, seg_rows=seg, lambdas=lambdas,
                            height=height)


def _assert_same(many, singles):
    assert len(many) == len(singles)
    for m, s in zip(many, singles):
        assert m.keys() == s.keys()
        for k in s:
            if isinstance(s[k], torch.Tensor):
                assert m[k].shape == s[k].shape and torch.equal(m[k], s[k]), k
            else:
                assert m[k] == s[k], k


def _mixed_case(C, N, n_tables, P, seed):
    """Blobs over n_tables tables (prob_bits P) with every seg_rows from 1 row to the whole item, heights h x w and
    w x h, odd item_rows, multi-plane and multi-item blobs, and one blob listed twice."""
    rng = np.random.default_rng(seed)
    tabs = {float(i): _table(C, N, P, seed + i) for i in range(n_tables)}
    lam = list(tabs)
    pick = lambda k: [lam[(k + j) % n_tables] for j in range(min(n_tables, 1 + k % 3))]
    blobs = []
    for k, (items, Hh, W, seg) in enumerate([(1, 4, 6, 24), (1, 6, 4, 24), (2, 4, 6, 1), (1, 3, 5, 7), (3, 1, 9, 4),
                                             (1, 5, 5, 25), (2, 2, 3, 2), (1, 7, 3, 100)]):
        ls = pick(k)
        blobs.append(_gpu_blob(rng, [tabs[l] for l in ls], ls, items, Hh * W, seg, Hh))
    blobs.insert(3, blobs[1])
    return tabs, blobs


@pytest.mark.gpu
@pytest.mark.parametrize("C,n_tables,P", [(1, 1, 12), (33, 2, 16), (192, 3, 16), (33, 3, 12), (192, 1, 12)])
def test_gpu_decode_many_equals_decode(C, n_tables, P):
    N = 10 if C == 192 else 4
    tabs, blobs = _mixed_case(C, N, n_tables, P, seed=C + n_tables + P)
    cp = torch.sort(torch.randn(C, 2 ** (N + 1) - 1, device="cuda"), dim=1).values
    for want_qidx, code_points in ((True, cp), (True, None), (False, cp)):
        many = serialize.decode_many(blobs, tables=tabs, code_points=code_points, want_qidx=want_qidx)
        _assert_same(many, [serialize.decode(b, tables=tabs, code_points=code_points, want_qidx=want_qidx)
                            for b in blobs])


@pytest.mark.gpu
def test_gpu_decode_many_prob_bits_mix_and_edges():
    """Tables of prob_bits 12 and 16 in one call, blobs with embedded tables, 1,000 tiny blobs and the empty list."""
    C, N = 33, 4
    rng = np.random.default_rng(7)
    t12, t16, t16b = _table(C, N, 12, 1), _table(C, N, 16, 2), _table(C, N, 16, 3)
    tabs = {0.0: t12, 1.0: t16, 2.0: t16b}
    blobs = [_gpu_blob(rng, [t12], [0.0], 2, 11, 5), _gpu_blob(rng, [t16], [1.0], 1, 13, 13),
             _gpu_blob(rng, [t16, t16b], [1.0, 2.0], 1, 6, 2)]   # one prob_bits per blob
    _assert_same(serialize.decode_many(blobs, tables=tabs), [serialize.decode(b, tables=tabs) for b in blobs])
    q = torch.from_numpy(_symbols(rng, t16[None], 1, 9)[0, 0]).cuda()
    emb = [serialize.encode(q, t16, N, embed_tables=True), serialize.encode(q[:4], t16, N, embed_tables=True)]
    _assert_same(serialize.decode_many(emb), [serialize.decode(b) for b in emb])
    tiny = [_gpu_blob(rng, [t16 if k % 3 else t12], [1.0 if k % 3 else 0.0], 1, 1 + k % 4, 1 + k % 2)
            for k in range(1000)]
    _assert_same(serialize.decode_many(tiny, tables=tabs), [serialize.decode(b, tables=tabs) for b in tiny])
    assert serialize.decode_many([]) == []


@pytest.mark.gpu
def test_gpu_decompress_many_end_to_end():
    """compress_to_bytes of a Kodak-shaped batch at three lambdas -> all 72 blobs in one decompress_many call equal
    compress_latents' Z_hat; stack=True gives the per-lambda stacks; both orientations mix in one call."""
    from test_rans import _kodak_case
    q, mu, lv, lambs = _kodak_case()
    B, Hh, W, C = mu.shape
    blobs = q.compress_to_bytes(mu, lv, lambs)
    ref = q.compress_latents(mu, lv, lambs)
    flat = [b for l in lambs for b in blobs[l]]
    zs = q.decompress_many(flat)
    assert len(zs) == 3 * B
    ptr = zs[0].untyped_storage().data_ptr()
    for i, l in enumerate(lambs):
        for b in range(B):
            z = zs[i * B + b]
            assert tuple(z.shape) == (1, Hh, W, C) and z.untyped_storage().data_ptr() == ptr
            assert np.array_equal(z.cpu().numpy()[0], ref["Z_hat"][l][b])
        st = q.decompress_many(blobs[l], stack=True)
        assert tuple(st.shape) == (B, Hh, W, C) and np.array_equal(st.cpu().numpy(), ref["Z_hat"][l])
    assert torch.equal(q.decompress_many(flat, stack=True), torch.cat(zs))
    assert torch.equal(q.decompress_many(flat[:1])[0], q.decompress_from_bytes(flat[0]))
    # the same latents transposed: 48 x 32 images next to 32 x 48 ones
    tr = q.compress_to_bytes(np.ascontiguousarray(mu.transpose(0, 2, 1, 3)),
                             np.ascontiguousarray(lv.transpose(0, 2, 1, 3)), lambs[1:2])[lambs[1]]
    mixed = [x for pair in zip(blobs[lambs[1]], tr) for x in pair]
    got = q.decompress_many(mixed)
    for g, blob in zip(got, mixed):
        assert torch.equal(g, q.decompress_from_bytes(blob))
    with pytest.raises(ValueError, match="stack=True"):
        q.decompress_many(mixed, stack=True)


def _flip_word(blob, k):
    b = bytearray(blob)
    off = serialize.read_header(blob)["payload_offset"]
    b[off + 2 * k] ^= 0x04
    return bytes(b)


def _bad_state(blob):
    """The first group's first state set below 2^16 (its high half zeroed)."""
    h = serialize.read_header(blob)
    G = -(-h["C"] // 32) * h["items"] * -(-h["item_rows"] // h["seg_rows"]) * h["n_planes"]
    k = h["payload_offset"] + 2 * (2 * G + 1)
    return blob[:k] + b"\0\0" + blob[k + 2:]


def _truncated_group(blob):
    """The first group's last word removed and the later offsets moved down by one."""
    h = serialize.read_header(blob)
    off = h["payload_offset"]
    G = -(-h["C"] // 32) * h["items"] * -(-h["item_rows"] // h["seg_rows"])
    w = np.frombuffer(blob[off:], dtype="<u2").copy()
    ends = w[0:2 * G:2].astype(np.int64) | (w[1:2 * G:2].astype(np.int64) << 16)
    cut = ends - 1
    tab = np.stack([cut & 0xFFFF, cut >> 16], axis=1).reshape(-1).astype("<u2")
    return blob[:off] + np.concatenate([tab, np.delete(w[2 * G:], ends[0] - 1)]).astype("<u2").tobytes()


def _plan_on_device(blobs, tables):
    headers = [serialize.read_header(b) for b in blobs]
    plan = serialize.batch_plan(headers, [serialize._payload_words(b, h) for b, h in zip(blobs, headers)],
                                [[0] * h["n_planes"] for h in headers])
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return (plan, dev(plan["words"].view(np.int16)), dev(coding.cum_table(tables[None]).view(np.int16)),
            torch.tensor([coding.prob_bits_of(tables)], dtype=torch.int32).cuda(), dev(plan["units"]), dev(plan["ctas"]))


@pytest.mark.gpu
def test_gpu_corrupt_blob_is_named():
    from vbq_b200 import ops
    C, N = 37, 10
    rng = np.random.default_rng(9)
    t = _table(C, N, 16, 4)
    good = [_gpu_blob(rng, [t], [1.0], 1, 200, 200) for _ in range(5)]
    cp = torch.sort(torch.randn(C, 2 ** (N + 1) - 1, device="cuda"), dim=1).values
    G = 2
    for k, bad, bits in ((3, _flip_word(good[3], 2 * G + 80), 1 | 2), (1, _truncated_group(good[1]), 1 | 2),
                         (4, _bad_state(good[4]), 4)):
        blobs = list(good)
        blobs[k] = bad
        with pytest.raises(ValueError, match=r"corrupt VBQ2 payload in blob %d \(blob %d: decoder status" % (k, k)):
            serialize.decode_many(blobs, tables=[t], code_points=cp)
        plan, w, cum, pb, units, ctas = _plan_on_device(blobs, t)
        _, _, status = ops.rans_decode_batch(w, cum, pb, units, ctas, len(blobs), N, plan["n_out"], cp)
        st = status.cpu().numpy()
        assert st[k] != 0 and (st[k] & ~bits) == 0 and (np.delete(st, k) == 0).all(), st
    _assert_same(serialize.decode_many(good, tables=[t], code_points=cp),
                 [serialize.decode(b, tables=[t], code_points=cp) for b in good])


@pytest.mark.gpu
def test_gpu_bad_units_set_bit_8_and_write_nothing():
    from vbq_b200 import _lib
    C, N = 37, 4
    rng = np.random.default_rng(10)
    t = _table(C, N, 14, 6)
    blobs = [_gpu_blob(rng, [t], [0.0], 2, 9, 4) for _ in range(3)]
    plan, w, cum, pb, units, ctas = _plan_on_device(blobs, t)
    n_out, guard = plan["n_out"], 4096
    cp = torch.sort(torch.randn(C, 2 ** (N + 1) - 1, device="cuda"), dim=1).values
    lib = _lib.load()
    U = units.shape[0]
    # (unit field, value) -> the blob whose status gets bit 8
    cases = [((0, 0), w.numel()), ((0, 0), -1), ((0, 1), w.numel() + 1), ((0, 4), 1), ((0, 4), -1), ((0, 5), 1),
             ((0, 2), n_out - 2), ((0, 2), -5), ((0, 3), 10 ** 12), ((0, 3), 0), ((0, 6), 7), ((0, 6), -1)]
    for (i, field), value in cases:
        bad = units.clone()
        bad[i, field] = value
        blob = int(units[i, 6]) if field != 6 else 0
        q = torch.full((n_out + 2 * guard,), -7, dtype=torch.int32, device="cuda")
        z = torch.full((n_out + 2 * guard,), -7.0, dtype=torch.float32, device="cuda")
        status = torch.full((len(blobs),), 99, dtype=torch.int32, device="cuda")
        _lib.check(lib.vbq_rans_decode_batch(w.data_ptr(), w.numel(), cum.data_ptr(), pb.data_ptr(), 1, C, N,
                                             bad.data_ptr(), U, ctas.data_ptr(), ctas.shape[0], len(blobs),
                                             cp.data_ptr(), n_out, q[guard:].data_ptr(), z[guard:].data_ptr(),
                                             status.data_ptr(), None), "vbq_rans_decode_batch")
        st = status.cpu().numpy()
        assert st[blob] & 8 and (np.delete(st, blob) & 8 == 0).all(), (field, value, st)
        assert (q[:guard] == -7).all() and (q[guard + n_out:] == -7).all()
        assert (z[:guard] == -7.0).all() and (z[guard + n_out:] == -7.0).all()
        # the bad unit wrote nothing into its own range either
        u = units[i].tolist()
        nact = min(32, C - 32 * u[5])
        idx = guard + u[2] + torch.arange(u[3])[:, None] * C + torch.arange(nact)[None, :]
        assert (q[idx.cuda()] == -7).all()
    for d in ([0, 9, 0, 0], [-1, 1, 0, 0], [U, 1, 0, 0], [0, 1, 1, 0], [0, 1, 0, 2]):
        bad = ctas.clone()
        bad[0] = torch.tensor(d)
        status = torch.zeros(len(blobs), dtype=torch.int32, device="cuda")
        q = torch.full((n_out + 2 * guard,), -7, dtype=torch.int32, device="cuda")
        _lib.check(lib.vbq_rans_decode_batch(w.data_ptr(), w.numel(), cum.data_ptr(), pb.data_ptr(), 1, C, N,
                                             units.data_ptr(), U, bad.data_ptr(), ctas.shape[0], len(blobs), None,
                                             n_out, q[guard:].data_ptr(), None, status.data_ptr(), None),
                   "vbq_rans_decode_batch")
        assert status.cpu().numpy()[0] & 8, d
        assert (q[:guard] == -7).all() and (q[guard + n_out:] == -7).all()
