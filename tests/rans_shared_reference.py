"""Plain NumPy restatement of the shared-table rANS layout of include/vbq_b200.h (vbq_rans_shared_*, csrc/rans.cu): the
byte-exact reference the tests compare the kernels with.  Vectorised over the groups of a plane, looping over rows.

planes (n_planes, n) symbols; tables (n_planes, Q) integer frequencies (entries >= 0, rows summing to 2^P); seg_rows
one per plane.  Symbol k sits at row k // 32, lane k % 32; a group is a segment of seg_rows rows.  Payload = uint16
words: per plane the group end offset table (uint32 per group, low half first) and the groups (the states of the lanes
that hold a symbol, low half first, then the words in decoder order: rows ascending, lanes ascending)."""
import numpy as np

L = 1 << 16


def _groups(n, seg_rows):
    return -(-(-(-n // 32)) // seg_rows)


def _row(n, seg_rows, t):
    """(G, 32) symbol index of every lane of row t of each group, and whether that symbol exists."""
    k = (np.arange(_groups(n, seg_rows), dtype=np.int64)[:, None] * seg_rows + t) * 32 + np.arange(32)
    return k, k < n


def _segs(seg_rows, n_planes):
    return [int(seg_rows)] * n_planes if np.isscalar(seg_rows) else [int(s) for s in seg_rows]


def rans_encode(planes, tables, P, seg_rows):
    """Raises ValueError for a symbol outside [0, Q) or of frequency 0 (the encoder's status bits 1 and 2)."""
    planes = np.asarray(planes)
    n_planes, n = planes.shape
    out = []
    for p, seg in enumerate(_segs(seg_rows, n_planes)):
        f = np.asarray(tables[p], dtype=np.uint64)
        Q = f.size
        cum = np.cumsum(f) - f
        if ((planes[p] < 0) | (planes[p] >= Q)).any():
            raise ValueError("symbol outside [0, Q)")
        if (f[planes[p]] == 0).any():
            raise ValueError("symbol of frequency 0")
        G = _groups(n, seg)
        sym = np.zeros(G * seg * 32, np.int32)
        sym[:n] = planes[p]
        sym = sym.reshape(G, seg, 32)
        x = np.full((G, 32), L, dtype=np.uint64)
        E = np.full((G, seg, 32), -1, dtype=np.int32)
        for t in range(seg - 1, -1, -1):               # rows last to first
            a = _row(n, seg, t)[1]
            fs, cs = f[sym[:, t]], cum[sym[:, t]]
            emit = a & (x >= (fs << np.uint64(32 - P)))
            E[:, t] = np.where(emit, (x & np.uint64(0xFFFF)).astype(np.int32), -1)
            x = np.where(emit, x >> np.uint64(16), x)
            x = np.where(a, ((x // np.maximum(fs, 1)) << np.uint64(P)) + x % np.maximum(fs, 1) + cs, x)
        nact = _row(n, seg, 0)[1].sum(axis=1)
        groups = []
        for g in range(G):
            na = nact[g]
            st = np.stack([x[g, :na] & np.uint64(0xFFFF), x[g, :na] >> np.uint64(16)], axis=1).reshape(-1)
            w = E[g].reshape(-1)
            groups.append(np.concatenate([st.astype(np.uint16), w[w >= 0].astype(np.uint16)]))
        ends = np.cumsum([len(gr) for gr in groups]).astype(np.uint64)
        out.append(np.stack([ends & np.uint64(0xFFFF), ends >> np.uint64(16)], axis=1).reshape(-1).astype(np.uint16))
        out.extend(groups)
    return np.concatenate(out).astype(np.uint16) if out else np.zeros(0, np.uint16)


def rans_decode(payload, n_planes, n, seg_rows, tables, P):
    """Inverse of rans_encode; raises ValueError on an offset table outside the payload, a group that runs out of
    words, a final state other than 2^16 or words left over."""
    w = np.asarray(payload, dtype=np.uint16).astype(np.uint64)
    out = np.zeros((n_planes, n), dtype=np.int32)
    pos0 = 0
    M = np.uint64(1 << P)
    for p, seg in enumerate(_segs(seg_rows, n_planes)):
        G = _groups(n, seg)
        nact = _row(n, seg, 0)[1].sum(axis=1)
        if pos0 + 2 * G > w.size:
            raise ValueError("payload truncated in an offset table")
        ends = (w[pos0:pos0 + 2 * G:2] | (w[pos0 + 1:pos0 + 2 * G:2] << np.uint64(16))).astype(np.int64)
        data0 = pos0 + 2 * G
        starts = np.concatenate([[0], ends[:-1]]).astype(np.int64)
        if G and ((ends - starts < 2 * nact).any() or data0 + ends[-1] > w.size):
            raise ValueError("offset table outside the payload")
        f = np.asarray(tables[p], dtype=np.uint64)
        cum = np.cumsum(f) - f
        x = np.full((G, 32), L, dtype=np.uint64)
        for g in range(G):
            b = data0 + starts[g]
            x[g, :nact[g]] = w[b:b + 2 * nact[g]:2] | (w[b + 1:b + 2 * nact[g]:2] << np.uint64(16))
        if (x < L).any():
            raise ValueError("initial state below 2^16")
        pos = data0 + starts + 2 * nact
        end = data0 + ends
        for t in range(seg):
            k, a = _row(n, seg, t)
            slot = x & (M - np.uint64(1))
            s = np.searchsorted(cum, slot, side="right") - 1          # the largest s with cum[s] <= slot
            xn = f[s] * (x >> np.uint64(P)) + slot - cum[s]
            x = np.where(a, xn, x)
            need = a & (x < L)
            kk = need.sum(axis=1)
            if (pos + kk > end).any():
                raise ValueError("a group ran out of words")
            off = pos[:, None] + np.cumsum(need, axis=1) - need
            word = w[np.minimum(off, w.size - 1)] if w.size else np.zeros_like(x)
            x = np.where(need, (x << np.uint64(16)) | word, x)
            pos = pos + kk
            out[p, k[a]] = s[a]
        if (x != L).any() or (G and (pos != end).any()):
            raise ValueError("integrity check failed: final state != 2^16 or words left over")
        pos0 = data0 + (int(ends[-1]) if G else 0)
    if pos0 != w.size:
        raise ValueError("trailing words after the last plane")
    return out
