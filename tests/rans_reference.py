"""Plain NumPy restatement of the rANS stream layout of include/vbq_b200.h (csrc/rans.cu): the byte-exact reference the
tests compare the kernels with.  Vectorised over lanes (all groups of a plane at once), looping over rows.

planes (n_planes, items, item_rows, C) symbols, tables (n_planes, C, Q) integer frequencies (entries >= 1, rows summing
to 2^P); payload = uint16 words: per plane the group end offset table (uint32 per group, low half first) and the
groups (active-lane states, low half first, then the words in decoder order)."""
import hashlib
import struct

import numpy as np

L = 1 << 16


def fingerprint(f):
    t = np.asarray(f)
    C, Q = t.shape
    h = hashlib.blake2b(struct.pack("<II", C, Q) + np.ascontiguousarray(t, dtype="<u4").tobytes(), digest_size=8)
    return int.from_bytes(h.digest(), "little")


def _layout(items, item_rows, C, seg_rows):
    n_segs = -(-item_rows // seg_rows)
    CG = -(-C // 32)
    nact = np.minimum(32, C - 32 * np.arange(CG))
    lens = np.minimum(seg_rows, item_rows - seg_rows * np.arange(n_segs))
    return n_segs, CG, nact, lens


def _lanes(items, n_segs, CG, C, lens, seg_rows):
    """(t, items, n_segs, CG*32) mask of coded (row, lane) pairs and the channel of every lane."""
    ch = np.arange(CG * 32)
    act = (np.arange(seg_rows)[:, None, None, None] < lens[None, None, :, None]) & (ch < C)[None, None, None, :]
    return np.broadcast_to(act, (seg_rows, items, n_segs, CG * 32)), np.minimum(ch, C - 1)


def rans_encode(planes, tables, P, seg_rows):
    planes = np.asarray(planes)
    n_planes, items, item_rows, C = planes.shape
    n_segs, CG, nact, lens = _layout(items, item_rows, C, seg_rows)
    G = items * n_segs * CG
    out = []
    for p in range(n_planes):
        f = np.asarray(tables[p], dtype=np.uint64)
        cum = np.cumsum(f, axis=1) - f
        sym = np.zeros((items, n_segs * seg_rows, CG * 32), dtype=np.int64)
        sym[:, :item_rows, :C] = planes[p]
        sym = sym.reshape(items, n_segs, seg_rows, CG * 32)
        act, ch = _lanes(items, n_segs, CG, C, lens, seg_rows)
        x = np.full((items, n_segs, CG * 32), L, dtype=np.uint64)
        E = np.full((seg_rows, items, n_segs, CG * 32), -1, dtype=np.int64)
        for t in range(seg_rows - 1, -1, -1):           # rows last to first
            s = sym[:, :, t, :]
            a = act[t]
            fs, cs = f[ch, s], cum[ch, s]
            emit = a & (x >= (fs << np.uint64(32 - P)))
            E[t] = np.where(emit, (x & np.uint64(0xFFFF)).astype(np.int64), -1)
            x = np.where(emit, x >> np.uint64(16), x)
            x = np.where(a, ((x // fs) << np.uint64(P)) + x % fs + cs, x)
        E = E.reshape(seg_rows, G, 32).transpose(1, 0, 2).reshape(G, seg_rows * 32)   # groups in (item, seg, cg) order
        xs = x.reshape(G, 32)
        groups = []
        for g in range(G):
            na = nact[g % CG]
            st = np.stack([xs[g, :na] & np.uint64(0xFFFF), xs[g, :na] >> np.uint64(16)], axis=1).reshape(-1)
            w = E[g][E[g] >= 0]
            groups.append(np.concatenate([st.astype(np.uint16), w.astype(np.uint16)]))
        ends = np.cumsum([len(gr) for gr in groups]).astype(np.uint64)
        table = np.stack([ends & np.uint64(0xFFFF), ends >> np.uint64(16)], axis=1).reshape(-1).astype(np.uint16)
        out.append(table)
        out.extend(groups)
    return np.concatenate(out).astype(np.uint16) if out else np.zeros(0, np.uint16)


def rans_decode(payload, n_planes, items, item_rows, C, seg_rows, tables, P):
    """Inverse of rans_encode; raises ValueError on an offset table outside the payload, a group that runs out of
    words, a final state other than 2^16 or words left over."""
    w = np.asarray(payload, dtype=np.uint16).astype(np.uint64)
    n_segs, CG, nact, lens = _layout(items, item_rows, C, seg_rows)
    G = items * n_segs * CG
    out = np.zeros((n_planes, items, item_rows, C), dtype=np.int64)
    pos0 = 0
    M = np.uint64(1 << P)
    for p in range(n_planes):
        if pos0 + 2 * G > w.size:
            raise ValueError("payload truncated in an offset table")
        ends = (w[pos0:pos0 + 2 * G:2] | (w[pos0 + 1:pos0 + 2 * G:2] << np.uint64(16))).astype(np.int64)
        data0 = pos0 + 2 * G
        starts = np.concatenate([[0], ends[:-1]]).astype(np.int64)
        na_g = np.tile(nact, items * n_segs)
        if G and ((np.diff(ends) < 0).any() or (ends - starts < 2 * na_g).any() or data0 + ends[-1] > w.size):
            raise ValueError("offset table outside the payload")
        f = np.asarray(tables[p], dtype=np.uint64)
        cum = np.cumsum(f, axis=1) - f
        flat = (cum + np.arange(C, dtype=np.uint64)[:, None] * M).reshape(-1)      # monotone over (channel, symbol)
        act, ch = _lanes(items, n_segs, CG, C, lens, seg_rows)
        act = act.reshape(seg_rows, G, 32)
        ch = ch.reshape(CG, 32)[np.arange(G) % CG]
        lane_on = (np.arange(CG * 32) < C).reshape(CG, 32)[np.arange(G) % CG]
        x = np.full((G, 32), L, dtype=np.uint64)
        for g in range(G):
            na = nact[g % CG]
            b = data0 + starts[g]
            x[g, :na] = w[b:b + 2 * na:2] | (w[b + 1:b + 2 * na:2] << np.uint64(16))
        if (x < L).any():
            raise ValueError("initial state below 2^16")
        pos = data0 + starts + 2 * na_g
        end = data0 + ends if G else np.zeros(0, np.int64)
        dec = np.zeros((seg_rows, G, 32), dtype=np.int64)
        for t in range(seg_rows):
            a = act[t]
            slot = x & (M - np.uint64(1))
            key = ch.astype(np.uint64) * M + slot
            gi = np.searchsorted(flat, key, side="right") - 1
            s = gi - ch * f.shape[1]
            fs, cs = f[ch, s], cum[ch, s]
            xn = fs * (x >> np.uint64(P)) + slot - cs
            x = np.where(a, xn, x)
            need = a & (x < L)
            k = need.sum(axis=1)
            if (pos + k > end).any():
                raise ValueError("a group ran out of words")
            off = pos[:, None] + np.cumsum(need, axis=1) - need
            word = w[np.minimum(off, w.size - 1)] if w.size else np.zeros_like(x)
            x = np.where(need, (x << np.uint64(16)) | word, x)
            pos = pos + k
            dec[t] = np.where(a, s, 0)
        if ((x != L) & lane_on).any() or (G and (pos != end).any()):
            raise ValueError("integrity check failed: final state != 2^16 or words left over")
        d = dec.reshape(seg_rows, items, n_segs, CG * 32).transpose(1, 2, 0, 3).reshape(items, n_segs * seg_rows, CG * 32)
        out[p] = d[:, :item_rows, :C]
        pos0 = data0 + (int(ends[-1]) if G else 0)
    if pos0 != w.size:
        raise ValueError("trailing words after the last plane")
    return out
