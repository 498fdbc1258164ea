"""Plain NumPy restatement of row access into one shared-table plane (include/vbq_b200.h, vbq_rans_shared_checkpoints /
vbq_rans_shared_decode_rows, CompressedEmbedding): the checkpoint index, a decode from a checkpoint to a stop row, and
the work list for a set of embedding rows.  Built on rans_shared_reference (one plane, P-bit table, seg_rows rows per
segment); K is the checkpoint interval in coder rows, clamped to the segment length."""
import numpy as np

import rans_shared_reference as R

L = R.L


def _plane(payload, n, seg, table):
    """(words, group starts, group ends, nact, cum, f) of a one-plane payload."""
    w = np.asarray(payload, dtype=np.uint16).astype(np.uint64)
    G = R._groups(n, seg)
    ends = (w[0:2 * G:2] | (w[1:2 * G:2] << np.uint64(16))).astype(np.int64)
    starts = np.concatenate([[0], ends[:-1]]).astype(np.int64) + 2 * G
    f = np.asarray(table, dtype=np.uint64)
    return w, starts, ends + 2 * G, R._row(n, seg, 0)[1].sum(axis=1), np.cumsum(f) - f, f


def _step(x, pos, w, a, f, cum, P):
    """One row for every group: the rule of rans_shared_reference.rans_decode.  Returns (symbols, x, pos)."""
    M = np.uint64(1 << P)
    slot = x & (M - np.uint64(1))
    s = np.searchsorted(cum, slot, side="right") - 1
    x = np.where(a, f[s] * (x >> np.uint64(P)) + slot - cum[s], x)
    need = a & (x < L)
    off = pos[:, None] + np.cumsum(need, axis=1) - need
    x = np.where(need, (x << np.uint64(16)) | w[np.minimum(off, w.size - 1)], x)
    return s, x, pos + need.sum(axis=1)


def checkpoint_count(n, seg_rows, K):
    seg = max(1, min(int(seg_rows), -(-n // 32)))
    k = min(int(K), seg)
    rows = -(-n // 32)
    lens = [min(seg, rows - g * seg) for g in range(R._groups(n, seg))]
    return sum((ln - 1) // k for ln in lens)


def checkpoints(payload, n, seg_rows, table, P, K):
    """The index: offsets (M,) uint32 from the group's start word and states (M, 32) uint32, entry
    g ((seg - 1) // K) + j - 1 for checkpoint j >= 1 of segment g (before row g seg + j K)."""
    seg = max(1, min(int(seg_rows), -(-n // 32)))
    k = min(int(K), seg)
    w, starts, ends, nact, cum, f = _plane(payload, n, seg, table)
    G = starts.size
    rows = -(-n // 32)
    per = (seg - 1) // k
    M = checkpoint_count(n, seg, k)
    offsets = np.zeros(M, np.uint32)
    states = np.zeros((M, 32), np.uint32)
    x = np.full((G, 32), L, dtype=np.uint64)
    for g in range(G):
        b = starts[g]
        x[g, :nact[g]] = w[b:b + 2 * nact[g]:2] | (w[b + 1:b + 2 * nact[g]:2] << np.uint64(16))
    pos = starts + 2 * nact
    lens = np.minimum(seg, rows - seg * np.arange(G))
    for t in range(seg):
        if t and t % k == 0:
            for g in np.flatnonzero(t < lens):
                c = g * per + t // k - 1
                offsets[c] = pos[g] - starts[g]
                states[c] = x[g]
        _, x, pos = _step(x, pos, w, R._row(n, seg, t)[1], f, cum, P)
    return offsets, states


def decode_from(payload, n, seg_rows, table, P, K, offsets, states, segment, j, last_row):
    """Symbols of coder rows [segment seg + j K, last_row] decoded from checkpoint j of `segment` (j = 0: the segment's
    start): (rows, 32) int64, -1 where a lane holds no symbol."""
    seg = max(1, min(int(seg_rows), -(-n // 32)))
    k = min(int(K), seg)
    w, starts, ends, nact, cum, f = _plane(payload, n, seg, table)
    g = segment
    if j == 0:
        b = starts[g]
        x = np.full((1, 32), L, dtype=np.uint64)
        x[0, :nact[g]] = w[b:b + 2 * nact[g]:2] | (w[b + 1:b + 2 * nact[g]:2] << np.uint64(16))
        pos = np.array([b + 2 * nact[g]])
    else:
        c = g * ((seg - 1) // k) + j - 1
        x = states[c].astype(np.uint64)[None]
        pos = np.array([starts[g] + int(offsets[c])])
    first = g * seg + j * k
    out = []
    for r in range(first, last_row + 1):
        kk = r * 32 + np.arange(32)
        a = (kk < n)[None]
        s, x, pos = _step(x, pos, w, a, f, cum, P)
        out.append(np.where(a[0], s[0], -1))
    return np.array(out, dtype=np.int64).reshape(-1, 32)


def work_list(ids, D, n, seg_rows, K):
    """(rows, items): the sorted unique rows of ids and the (n_items, 5) int64 work list [segment, checkpoint, last_row,
    lo, hi]: one item per checkpoint interval that a requested row touches, decoding up to the last coder row any
    requested row needs in it, with the slice of rows that touch it."""
    seg = max(1, min(int(seg_rows), -(-n // 32)))
    k = min(int(K), seg)
    coder_rows = -(-n // 32)
    rows = np.unique(np.asarray(ids, dtype=np.int64).reshape(-1))
    by_interval = {}
    for u, e in enumerate(rows):
        for r in range(e * D // 32, (e * D + D - 1) // 32 + 1):
            g, t = divmod(r, seg)
            key = (g, t // k)
            lo, hi, last = by_interval.get(key, (u, u + 1, r))
            by_interval[key] = (min(lo, u), max(hi, u + 1), max(last, r))
    items = [[g, j, last, lo, hi] for (g, j), (lo, hi, last) in sorted(by_interval.items())]
    assert all(last < min(g * seg + (j + 1) * k, (g + 1) * seg, coder_rows) for g, j, last, _, _ in items)
    return rows, np.array(items, dtype=np.int64).reshape(-1, 5)


def gather(payload, n, seg_rows, table, P, K, ids, D):
    """Execute the work list on the reference decoder: (n_req, D) int64 symbols of the unique sorted rows, -1 where no
    item wrote (there should be none)."""
    offsets, states = checkpoints(payload, n, seg_rows, table, P, K)
    rows, items = work_list(ids, D, n, seg_rows, K)
    seg = max(1, min(int(seg_rows), -(-n // 32)))
    k = min(int(K), seg)
    out = np.full((rows.size, D), -1, np.int64)
    for g, j, last, lo, hi in items:
        sym = decode_from(payload, n, seg, table, P, k, offsets, states, g, j, last)
        first = g * seg + j * k
        t = (first + np.arange(sym.shape[0]))[:, None] * 32 + np.arange(32)
        for u in range(lo, hi):
            m = (t // D == rows[u]) & (sym >= 0)
            assert (out[u, t[m] - rows[u] * D] == -1).all(), "two items wrote the same element"
            out[u, t[m] - rows[u] * D] = sym[m]
    return rows, out
