"""Many images in one encode launch (vbq_rans_encode_batch, serialize.encode_many, compress_many): CPU tests of the work
list against the reference layout, of the checks made before any launch and of the ABI's argument validation; GPU tests
of encode_many against per-image encode_items, byte for byte, of the quantizer's sender path, of out-of-range symbols
and of bad raw units."""
import ctypes

import numpy as np
import pytest
import torch

import rans_reference as R
from vbq_b200 import coding, serialize


def _table(C, N, P, seed):
    rng = np.random.default_rng(seed)
    return coding.frequency_tables(rng.integers(0, 50, (C, 2 ** (N + 1) - 1)) ** 3, P)


def _symbols(rng, tables, rows):
    """(L, rows, C) symbols drawn from each plane's table (inverse CDF per channel)."""
    L, C, Q = tables.shape
    out = np.zeros((L, rows, C), np.int32)
    for p in range(L):
        cdf = np.cumsum(tables[p], axis=1) / tables[p].sum(axis=1, keepdims=True)
        u = rng.random((rows, C))
        for c in range(C):
            out[p, :, c] = np.minimum(np.searchsorted(cdf[c], u[:, c], side="right"), Q - 1)
    return out


# (H', W') of each image: both orientations, one row, odd row counts, an empty image
SHAPES = [(4, 6), (6, 4), (1, 1), (3, 5), (1, 9), (5, 5), (0, 3), (2, 3), (7, 3)]


def _encode_unit(sym, u, tables, C, P):
    """NumPy encoder of one work unit from its fields alone: the group's states, then its words in decoder order."""
    inp, rows, table, cg, group, scratch, blob = (int(v) for v in u)
    nact = min(32, C - 32 * cg)
    lanes = np.arange(nact)
    f = tables[table][32 * cg:32 * cg + nact].astype(np.uint64)
    cum = np.cumsum(f, axis=1) - f
    x = np.full(nact, 1 << 16, np.uint64)
    per_row = []
    for t in range(rows - 1, -1, -1):
        s = sym[inp + t * C + lanes]
        fs, cs = f[lanes, s], cum[lanes, s]
        emit = x >= fs << np.uint64(32 - P)
        per_row.append(x[emit] & np.uint64(0xFFFF))
        x = np.where(emit, x >> np.uint64(16), x)
        x = ((x // fs) << np.uint64(P)) + x % fs + cs
    states = np.stack([x & np.uint64(0xFFFF), x >> np.uint64(16)], axis=1).reshape(-1)
    return np.concatenate([states] + per_row[::-1]).astype(np.uint16)


@pytest.mark.parametrize("C,seg_rows", [(37, None), (37, 1), (1, 3), (70, 4)])
def test_encode_plan_against_reference(C, seg_rows):
    N, P = 4, 14
    rng = np.random.default_rng(C + (seg_rows or 0))
    tabs = [_table(C, N, P, 20 + i) for i in range(3)]
    table_ids = [2, 0, 2]
    rows = np.array([h * w for h, w in SHAPES])
    B, L, CG = len(SHAPES), len(table_ids), -(-C // 32)
    planes = _symbols(rng, np.stack([tabs[i] for i in table_ids]), int(rows.sum()))
    plan = serialize.encode_plan(rows, seg_rows, C, table_ids)
    units, ctas, bg = plan["units"], plan["ctas"], plan["blob_groups"]
    seg = np.maximum(1, rows if seg_rows is None else np.full(rows.size, seg_rows))
    assert plan["seg"].tolist() == seg.tolist()
    # every group of every blob exactly once, blob-major, and each unit's fields match its group
    n_segs = -(-rows // seg)
    assert bg.tolist() == np.concatenate([[0], np.cumsum(np.tile(n_segs * CG, L))]).tolist()
    assert sorted(units[:, 4].tolist()) == list(range(plan["n_groups"]))
    row0 = np.cumsum(rows) - rows
    for inp, r, table, cg, g, scratch, blob in units.tolist():
        p, b = divmod(blob, B)
        assert bg[blob] <= g < bg[blob + 1] and table == table_ids[p]
        s, c = divmod(g - bg[blob], CG)
        assert c == cg and r == min(seg[b], rows[b] - s * seg[b])
        assert inp == (p * rows.sum() + row0[b] + s * seg[b]) * C + 32 * cg
    # scratch ranges: disjoint, each nact (rows + 2) words, inside scratch_words; the payload bound
    nact = np.minimum(32, C - 32 * units[:, 3])
    r = np.argsort(units[:, 5])
    lo, hi = units[r, 5], units[r, 5] + nact[r] * (units[r, 1] + 2)
    assert (lo[1:] >= hi[:-1]).all() and lo[0] >= 0 and hi[-1] <= plan["scratch_words"]
    assert plan["payload_words"] == 2 * plan["n_groups"] + plan["scratch_words"]
    # descriptors: consecutive, in order, at most 8 units of one (table, cg) each; units sorted by (table, cg)
    assert ctas[:, 0].tolist() == np.concatenate([[0], np.cumsum(ctas[:-1, 1])]).tolist()
    assert int(ctas[:, 1].sum()) == len(units) and (ctas[:, 1] >= 1).all() and (ctas[:, 1] <= 8).all()
    for first, count, table, cg in ctas:
        assert (units[first:first + count, 2] == table).all() and (units[first:first + count, 3] == cg).all()
    assert (np.diff(units[:, 2] * CG + units[:, 3]) >= 0).all()
    # encoding every unit from its fields alone and laying the groups out per blob gives the reference's payload
    groups = {int(u[4]): _encode_unit(planes.reshape(-1), u, tabs, C, P) for u in units}
    for i in range(L * B):
        p, b = divmod(i, B)
        gs = [groups[g] for g in range(bg[i], bg[i + 1])]
        ends = np.cumsum([len(x) for x in gs]).astype(np.int64)
        tab = np.stack([ends & 0xFFFF, ends >> 16], axis=1).reshape(-1).astype(np.uint16)
        got = np.concatenate([tab] + gs).astype(np.uint16)
        img = planes[p, row0[b]:row0[b] + rows[b]][None, None]
        assert np.array_equal(got, R.rans_encode(img, tabs[table_ids[p]][None], P, int(seg[b]))), (p, b)


def test_encode_many_checks_before_any_launch():
    """Every failure here raises on the host: the symbols are a CPU tensor, which the kernel wrapper would refuse."""
    C, N, P = 33, 4, 16
    t = _table(C, N, P, 1)
    q = torch.zeros((2, 20, C), dtype=torch.int32)
    with pytest.raises(ValueError, match="do not sum to the 20 rows"):
        serialize.encode_many(q, t, N, [12, 7])
    with pytest.raises(ValueError, match="height 3 does not divide the 8 rows of image 1"):
        serialize.encode_many(q, t, N, [12, 8], heights=[4, 3])
    with pytest.raises(ValueError, match="2 heights for 3 images"):
        serialize.encode_many(q, t, N, [12, 4, 4], heights=[4, 2])
    with pytest.raises(ValueError, match=r"need \(C, Q\) = \(33, 31\)"):
        serialize.encode_many(q, [t, t[:, :15]], N, [12, 8])
    with pytest.raises(ValueError, match="3 tables for 2 planes"):
        serialize.encode_many(q, [t, t, t], N, [12, 8])
    with pytest.raises(ValueError, match="one .C, Q. table per plane"):
        serialize.encode_many(q, np.stack([t, t, t]), N, [12, 8])
    with pytest.raises(ValueError, match="3 lambdas for 2 planes"):
        serialize.encode_many(q, t, N, [12, 8], lambdas=[1, 2, 3])
    t0 = t.copy()
    t0[5, 0], t0[5, 1] = t0[5, 0] + t0[5, 1], 0
    with pytest.raises(ValueError, match="every frequency must be >= 1"):
        serialize.encode_many(q, [t, t0], N, [12, 8])
    with pytest.raises(ValueError, match="32-bit offset table"):
        serialize.encode_plan([1 << 27], None, 40, [0])
    # arguments that pass every check reach the kernel wrapper, which has no CPU fallback
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        serialize.encode_many(q, t, N, [12, 8], heights=[3, 2])


def test_compress_many_checks_before_any_launch():
    import vbq_b200
    C, N = 37, 4
    q = vbq_b200.ChannelwisePriorCDFQuantizer(C, N, device="cuda:99")
    img = np.zeros((3, 4, C), np.float32)
    with pytest.raises(TypeError, match="entropy_models not built"):
        q.compress_many([img], [img], [0.5])
    rng = np.random.default_rng(5)
    q.entropy_models = {0.5: -np.log2(rng.dirichlet(np.ones(31), C)), 8.0: -np.log2(rng.dirichlet(np.ones(31), C))}
    assert q.compress_many([], [], [0.5, 8.0]) == {0.5: [], 8.0: []}
    bad = np.zeros((3, 4, C + 1), np.float32)
    with pytest.raises(ValueError, match="image 1 has means"):
        q.compress_many([img, bad], [img, bad], [0.5])
    with pytest.raises(ValueError, match="image 0 has means"):
        q.compress_many([img[None, None]], [img[None, None]], [0.5])
    with pytest.raises(ValueError, match="1 means for 2 logvars"):
        q.compress_many([img], [img, img], [0.5])


def test_abi_validation_needs_no_gpu():
    from vbq_b200 import _lib
    lib = _lib.load()
    one = ctypes.c_void_p(16)
    enc = lib.vbq_rans_encode_batch

    def call(**kw):
        a = dict(inp=one, n_in=100, cum=one, pb=one, n_tables=1, C=4, N=4, units=one, n_units=1, ctas=one, n_ctas=1,
                 bg=one, n_blobs=1, n_groups=1, payload=one, payload_words=10, starts=one, status=one, ws=one,
                 ws_bytes=4096)
        a.update(kw)
        return enc(a["inp"], a["n_in"], a["cum"], a["pb"], a["n_tables"], a["C"], a["N"], a["units"], a["n_units"],
                   a["ctas"], a["n_ctas"], a["bg"], a["n_blobs"], a["n_groups"], a["payload"], a["payload_words"],
                   a["starts"], a["status"], a["ws"], a["ws_bytes"], None)
    assert call(N=11) == 3 and call(N=-1) == 3
    for bad in (dict(C=0), dict(C=32 * 65535 + 1), dict(n_in=-1), dict(n_units=-1), dict(n_ctas=-1),
                dict(n_ctas=1 << 31), dict(n_blobs=-1), dict(n_groups=-1), dict(n_groups=1 << 31),
                dict(payload_words=-1), dict(ws_bytes=-1), dict(n_tables=-1), dict(n_units=0), dict(n_tables=0),
                dict(n_groups=0), dict(n_blobs=0)):
        assert call(**bad) == 2, bad
    for bad in ("inp", "cum", "pb", "units", "ctas", "bg", "payload", "starts", "status", "ws"):
        assert call(**{bad: None}) == 1, bad
    for bad in ("inp", "pb", "units", "ctas", "bg", "starts", "status", "ws"):
        assert call(**{bad: ctypes.c_void_p(18 if bad in ("inp", "pb", "status") else 20)}) == 7, bad
    assert call(cum=ctypes.c_void_p(17)) == 7 and call(payload=ctypes.c_void_p(17)) == 7
    assert call(ws_bytes=255 * 3) == 5                 # smaller than the three index arrays of one group
    assert lib.vbq_rans_encode_batch_workspace_bytes(1, 10) == 3 * 256 + 256
    assert lib.vbq_rans_encode_batch_workspace_bytes(-1, 10) == -1
    assert lib.vbq_rans_encode_batch_workspace_bytes(1, -1) == -1


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _per_image(q, tables, N, rows, seg_rows, lambdas, heights):
    """encode_items of every (plane, image) on its own: the reference encode_many must equal byte for byte."""
    row0 = np.cumsum(rows) - rows
    return [[serialize.encode_items(q[p:p + 1, row0[b]:row0[b] + rows[b]], tables[p], N, items=1, seg_rows=seg_rows,
                                    lambdas=[lambdas[p]], height=heights[b])[0][0] for b in range(len(rows))]
            for p in range(q.shape[0])]


def _mixed_images(rng, tables, shapes):
    rows = np.array([h * w for h, w in shapes])
    sym = _symbols(rng, np.stack(tables), int(rows.sum()))
    return torch.from_numpy(sym).cuda(), rows, [h for h, _ in shapes]


@pytest.mark.gpu
@pytest.mark.parametrize("C,Ps,seg_rows", [(1, [12], None), (33, [16, 16], 1), (192, [16, 12, 16], 3),
                                           (33, [12, 16, 12], None), (192, [12], 7), (1, [16, 12], 1)])
def test_gpu_encode_many_equals_encode_items(C, Ps, seg_rows):
    N = 10 if C == 192 else 4
    rng = np.random.default_rng(C + len(Ps) + (seg_rows or 0))
    tables = [_table(C, N, P, 30 + i) for i, P in enumerate(Ps)]
    shapes = SHAPES + [SHAPES[3]]                      # a repeated shape with its own symbols
    q, rows, heights = _mixed_images(rng, tables, shapes)
    r0 = int(rows[:4].sum())
    q[:, -int(rows[-1]):] = q[:, r0 - int(rows[3]):r0]   # and the same image twice
    lam = [0.25 * (i + 1) for i in range(len(Ps))]
    got = serialize.encode_many(q, tables, N, rows, seg_rows=seg_rows, lambdas=lam, heights=heights)
    want = _per_image(q, tables, N, rows, seg_rows, lam, heights)
    assert got == want
    assert got[0][3] == got[0][-1]
    # an (L, C, Q) array of tables of one prob_bits, and a (C, Q) table broadcast to every plane
    if len(set(Ps)) == 1:
        assert serialize.encode_many(q, np.stack(tables), N, rows, seg_rows, lam, heights) == want
    assert serialize.encode_many(q, tables[0], N, rows, seg_rows, lam, heights) == \
        _per_image(q, [tables[0]] * len(Ps), N, rows, seg_rows, lam, heights)
    # the blobs decode back to the symbols in one decode_many call
    flat = [b for plane in got for b in plane]
    dec = serialize.decode_many(flat, tables={l: t for l, t in zip(lam, tables)})
    row0 = np.cumsum(rows) - rows
    for i, d in enumerate(dec):
        p, b = divmod(i, len(rows))
        assert torch.equal(d["qidx"].reshape(-1, C), q[p, row0[b]:row0[b] + rows[b]])


@pytest.mark.gpu
def test_gpu_encode_many_edges():
    """1,000 tiny images, one image, the empty list, and images of zero rows."""
    C, N = 33, 4
    rng = np.random.default_rng(3)
    t12, t16 = _table(C, N, 12, 1), _table(C, N, 16, 2)
    shapes = [(1 + k % 3, 1 + k % 2) for k in range(1000)]
    q, rows, heights = _mixed_images(rng, [t12, t16], shapes)
    got = serialize.encode_many(q, [t12, t16], N, rows, seg_rows=2, lambdas=[0.0, 1.0], heights=heights)
    assert got == _per_image(q, [t12, t16], N, rows, 2, [0.0, 1.0], heights)
    one = q[:, :7]
    assert serialize.encode_many(one, [t12, t16], N, [7]) == _per_image(one, [t12, t16], N, [7], None, [0.0, 0.0], [0])
    assert serialize.encode_many(q[:, :0], [t12, t16], N, []) == [[], []]
    empty = serialize.encode_many(q[:, :0], [t12, t16], N, [0, 0], heights=[0, 0])
    assert empty == _per_image(q[:, :0], [t12, t16], N, [0, 0], None, [0.0, 0.0], [0, 0])


@pytest.mark.gpu
def test_gpu_compress_many_kodak_mixed_orientation():
    """24 Kodak-shaped latents, 12 of 32 x 48 and 12 of 48 x 32, at three lambdas: compress_many equals the
    per-image compress_to_bytes byte for byte, with host and device inputs, and decompress_many of its output equals
    each image's compress_latents z_hat."""
    from test_rans import _kodak_case
    q, mu, lv, lambs = _kodak_case()
    B = mu.shape[0]
    tr = lambda a: np.ascontiguousarray(a.transpose(1, 0, 2))
    means = [mu[b] if b % 2 else tr(mu[b]) for b in range(B)]
    logvars = [lv[b] if b % 2 else tr(lv[b]) for b in range(B)]
    got = q.compress_many(means, logvars, lambs)
    assert list(got) == lambs and all(len(got[l]) == B for l in lambs)
    for b in range(B):
        one = q.compress_to_bytes(means[b][None], logvars[b][None], lambs)
        for l in lambs:
            assert got[l][b] == one[l][0], (b, l)
    dev = q.compress_many([torch.from_numpy(m[None]).cuda() for m in means],
                          [torch.from_numpy(v).cuda() for v in logvars], lambs)
    assert dev == got
    zs = q.decompress_many([x for l in lambs for x in got[l]])
    for b in range(B):
        ref = q.compress_latents(means[b][None], logvars[b][None], lambs)["Z_hat"]
        for i, l in enumerate(lambs):
            assert np.array_equal(zs[i * B + b].cpu().numpy(), ref[l]), (l, b)


@pytest.mark.gpu
def test_gpu_out_of_range_symbol_names_the_images():
    from vbq_b200 import ops
    C, N = 37, 4
    rng = np.random.default_rng(4)
    tables = [_table(C, N, 16, 5), _table(C, N, 14, 6)]
    q, rows, heights = _mixed_images(rng, tables, SHAPES)
    row0 = np.cumsum(rows) - rows
    bad = q.clone()
    bad[1, row0[3] + 2, 36] = 31                       # Q = 31
    bad[1, row0[8], 0] = -1
    bad[0, row0[8] + 5, 5] = 1 << 20
    with pytest.raises(ValueError, match=r"cannot encode images 3, 8 for max_bits=4 \(image 8 of plane 0 .*; "
                                         r"image 3 of plane 1 .*; image 8 of plane 1 "):
        serialize.encode_many(bad, tables, N, rows, heights=heights)
    plan = serialize.encode_plan(rows, None, C, [0, 1])
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    cum = dev(np.stack([coding.cum_table(t) for t in tables]).view(np.int16))
    pb = torch.tensor([16, 14], dtype=torch.int32).cuda()
    _, meta = ops.rans_encode_batch(bad, cum, pb, dev(plan["units"]), dev(plan["ctas"]), dev(plan["blob_groups"]),
                                    plan["n_groups"], N, plan["scratch_words"])
    LB = 2 * len(SHAPES)
    st = meta.cpu().numpy()[LB + 1:].view(np.int32)[:LB]
    want = np.zeros(LB, np.int32)
    want[[len(SHAPES) + 3, 8, len(SHAPES) + 8]] = 1
    assert st.tolist() == want.tolist()
    assert serialize.encode_many(q, tables, N, rows, heights=heights) == \
        _per_image(q, tables, N, rows, None, [0.0, 0.0], heights)


@pytest.mark.gpu
def test_gpu_bad_units_set_bit_8_and_stay_in_bounds():
    """Units, descriptors and blob group tables that the kernel's checks reject: bit 8 on the right blob, and the guard
    regions around the payload, the blob starts and the workspace untouched."""
    from vbq_b200 import _lib
    C, N = 37, 4
    rng = np.random.default_rng(10)
    t = _table(C, N, 14, 6)
    q, rows, _ = _mixed_images(rng, [t], [(3, 3), (2, 5), (4, 1)])
    plan = serialize.encode_plan(rows, 4, C, [0])
    dev = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    cum, pb = dev(coding.cum_table(t[None]).view(np.int16)), torch.tensor([14], dtype=torch.int32).cuda()
    units, ctas, bg = dev(plan["units"]), dev(plan["ctas"]), dev(plan["blob_groups"])
    U, n_blobs, n_groups, sw = units.shape[0], len(rows), plan["n_groups"], plan["scratch_words"]
    pw, guard = plan["payload_words"], 4096
    lib = _lib.load()
    ws_bytes = lib.vbq_rans_encode_batch_workspace_bytes(n_groups, sw)

    def run(u=units, c=ctas, g=bg):
        payload = torch.full((pw + 2 * guard,), -7, dtype=torch.int16, device="cuda")
        starts = torch.full((n_blobs + 1 + 2 * guard,), -7, dtype=torch.int64, device="cuda")
        status = torch.full((n_blobs,), 99, dtype=torch.int32, device="cuda")
        ws = torch.full((ws_bytes + 2 * guard,), 0x55, dtype=torch.uint8, device="cuda")
        _lib.check(lib.vbq_rans_encode_batch(q.data_ptr(), q.numel(), cum.data_ptr(), pb.data_ptr(), 1, C, N,
                                             u.data_ptr(), U, c.data_ptr(), c.shape[0], g.data_ptr(), n_blobs,
                                             n_groups, payload[guard:].data_ptr(), pw, starts[guard:].data_ptr(),
                                             status.data_ptr(), ws[guard:].data_ptr(), ws_bytes, None),
                   "vbq_rans_encode_batch")
        assert (payload[:guard] == -7).all() and (payload[guard + pw:] == -7).all()
        assert (starts[:guard] == -7).all() and (starts[guard + n_blobs + 1:] == -7).all()
        assert (ws[:guard] == 0x55).all() and (ws[guard + ws_bytes:] == 0x55).all()
        return status.cpu().numpy(), starts[guard:guard + n_blobs + 1].cpu().numpy()

    st, good_starts = run()
    assert (st == 0).all()
    u0 = plan["units"][0]
    n_in = q.numel()
    # (unit field, value): in, rows, table, cg, group, scratch, blob
    cases = [(0, -1), (0, n_in), (0, n_in - C), (1, 0), (1, 10 ** 12), (1, 10 ** 6), (2, 1), (2, -1), (3, 1),
             (3, -1), (4, n_groups), (4, -1), (5, -1), (5, sw), (5, sw - 5), (6, n_blobs), (6, -1)]
    for field, value in cases:
        bad = units.clone()
        bad[0, field] = value
        st, starts = run(u=bad)
        blob = int(u0[6]) if field != 6 else 0
        assert st[blob] & 8 and (np.delete(st, blob) & 8 == 0).all(), (field, value, st)
        # the bad unit coded nothing, so its group is left at size 0 and the payload is shorter
        assert starts[-1] < good_starts[-1], (field, value)
    for d in ([0, 9, 0, 0], [-1, 1, 0, 0], [U, 1, 0, 0], [0, 1, 1, 0], [0, 1, 0, 2]):
        bad = ctas.clone()
        bad[0] = torch.tensor(d)
        st, _ = run(c=bad)
        assert st[0] & 8, d
    for g in ([1, 2, 4, n_groups], [0, 3, 2, n_groups], [0, 2, 4, n_groups + 1], [0, 2, 4, n_groups - 1]):
        st, starts = run(g=torch.tensor(g, dtype=torch.int64).cuda())
        assert st[0] & 8 and (starts == 0).all(), g
