"""Wire formats for the emitted symbols (SURVEY §8 row f4).

The reference stops at counting its sorted quantile indices per channel (quantizer.py:135-146) and reporting ideal
code lengths (ipynb:452-455).  This module turns the kernel's `qidx` output into bytes and reads them back, in two
formats:

VBQ1 (`dumps` / `loads`): a fixed-width bit stream (max_bits_per_coord+1 bits per symbol, packed on the GPU) plus,
optionally, the per-channel counts an external entropy coder needs.  Layout (little endian):  magic b"VBQ1" |
uint32 N, C, L, flags | uint64 rows | [flags & 1: L*C*Q uint32 counts] | L streams, each ceil(rows*C*(N+1)/32) uint32
words (symbols in (row, channel) order).

VBQ2 (`encode` / `decode`): entropy coded with the GPU rANS coder of csrc/rans.cu, one integer frequency table per
(plane, channel) (`coding.frequency_tables`).  Layout (little endian):  magic b"VBQ2" | uint32 N, C, prob_bits,
n_planes, items | uint64 item_rows, seg_rows | uint32 height, flags | per plane: float64 lambda, uint64 fingerprint of
its table (`coding.fingerprint`) | [flags & 1: the tables, n_planes*C*Q uint16 entries f-1] | the rANS payload of
include/vbq_b200.h (per plane: uint32 group end offsets, then the groups' 16-bit words).  `height` is H' of an
item of H' x W' = item_rows latent rows (0 if unknown).

VBQE (`encode_embeddings` / `decode_embedding`, behind `GaussianCodebook.compress_to_bytes`): one plane of word-embedding
coordinates coded with the shared-table rANS coder (`vbq_rans_shared_*`), one table for all coordinates.  Layout
(little endian):  magic b"VBQE" | uint32 N, prob_bits, ndim | ndim uint64 extents of the tensor | uint64 seg_rows |
float64 empirical_std, beta | uint64 fingerprint of the codebook's float64 code points (`coding.code_points_fingerprint`)
| the sparse table: uint32 k, k ascending uint16 symbols, k uint32 frequencies (those of every other symbol are 0) |
the rANS payload (uint32 group end offsets, then the groups' 16-bit words).
"""
from __future__ import annotations

import math
import struct

import numpy as np
import torch

from . import coding, ops, utils

MAGIC = b"VBQ1"
_HDR = struct.Struct("<4sIIIIQ")


def dumps(qidx, max_bits: int, with_counts: bool = False) -> bytes:
    """qidx: (rows, C) or (L, rows, C) int32 CUDA tensor of sorted quantile indices -> bytes."""
    q = qidx if qidx.dim() == 3 else qidx.unsqueeze(0)
    L, rows, C = q.shape
    Q = ops.num_levels(max_bits)
    out = [_HDR.pack(MAGIC, max_bits, C, L, 1 if with_counts else 0, rows)]
    if with_counts:
        for i in range(L):
            counts = ops.symbol_histogram(q[i], max_bits)
            out.append(counts.to(torch.int32).cpu().numpy().astype("<u4").tobytes())
    for i in range(L):
        out.append(ops.pack_indices(q[i], max_bits).cpu().numpy().astype("<i4").tobytes())
    return b"".join(out)


def loads(data: bytes, device="cuda"):
    """Inverse of dumps: dict(max_bits, qidx (L, rows, C) int32 on `device`, counts (L, C, Q) int64 or None)."""
    magic, N, C, L, flags, rows = _HDR.unpack_from(data, 0)
    if magic != MAGIC:
        raise ValueError("vbq_b200.serialize: bad magic %r" % magic)
    Q = ops.num_levels(N)
    pos = _HDR.size
    counts = None
    if flags & 1:
        n = L * C * Q
        counts = torch.from_numpy(np.frombuffer(data, dtype="<u4", count=n, offset=pos).astype(np.int64))
        counts = counts.reshape(L, C, Q)
        pos += 4 * n
    n_sym = rows * C
    n_words = ops.packed_index_words(n_sym, N)
    qs = []
    for _ in range(L):
        w = np.frombuffer(data, dtype="<i4", count=n_words, offset=pos)
        pos += 4 * n_words
        words = torch.from_numpy(w.copy()).to(device)
        qs.append(ops.unpack_indices(words, n_sym, N).reshape(rows, C))
    return dict(max_bits=N, qidx=torch.stack(qs) if qs else torch.empty((0, rows, C), dtype=torch.int32, device=device),
                counts=counts)


def ideal_code_length_bits(counts) -> float:
    """Σ_c [ n_c log2 n_c - Σ_s k_cs log2 k_cs ]: the length of an ideal adaptive-free entropy code with one frequency
    table per channel (the per-channel analogue of ipynb:452-455)."""
    c = counts.double()
    tot = c.sum(dim=-1)
    t1 = torch.where(tot > 0, tot * torch.log2(tot.clamp(min=1)), torch.zeros_like(tot)).sum()
    t2 = torch.where(c > 0, c * torch.log2(c.clamp(min=1)), torch.zeros_like(c)).sum()
    return float(t1 - t2)


# ------------------------------------------------------------------------------------------------------
# VBQ2: rANS-coded planes
# ------------------------------------------------------------------------------------------------------
MAGIC2 = b"VBQ2"
_HDR2 = struct.Struct("<4sIIIIIQQII")
_PLANE2 = struct.Struct("<dQ")
FLAG_TABLES = 1


def _as_tables(tables, n_planes):
    t = np.asarray(tables)
    if t.ndim == 2:
        t = np.broadcast_to(t, (n_planes,) + t.shape)
    if t.ndim != 3 or t.shape[0] != n_planes:
        raise ValueError("vbq_b200.serialize: need one (C, Q) table per plane, got shape %s" % (t.shape,))
    return t


def _encode_payload(qidx, tables, max_bits, items, seg_rows):
    """-> (header fields, host payload as uint16 words, tables int64)."""
    q = qidx if qidx.dim() == 3 else qidx.unsqueeze(0)
    L, rows, C = q.shape
    items = int(items)
    if items < 1 or rows % items:
        raise ValueError("vbq_b200.serialize: %d rows do not split into %d items" % (rows, items))
    item_rows = rows // items
    seg = max(1, item_rows if seg_rows is None else int(seg_rows))
    t = _as_tables(tables, L)
    P = coding.prob_bits_of(t)
    t = coding.check_tables(t, P)
    if t.shape[1:] != (C, ops.num_levels(max_bits)):
        raise ValueError("vbq_b200.serialize: tables are %s, need (C, Q) = (%d, %d)" % (t.shape[1:], C,
                                                                                     ops.num_levels(max_bits)))
    cum = torch.from_numpy(coding.cum_table(t).view(np.int16)).to(q.device)
    payload, size, status = ops.rans_encode(q.contiguous().reshape(L, items, item_rows, C), cum, max_bits, P, seg)
    if int(status.item()) != 0:
        raise ValueError("vbq_b200.serialize: a symbol lies outside [0, Q) for max_bits=%d" % max_bits)
    n = int(size.item()) // 2
    words = payload[:n].cpu().numpy().view(np.uint16)
    return dict(N=max_bits, C=C, P=P, n_planes=L, items=items, item_rows=item_rows, seg_rows=seg), words, t


def _header(f, lambdas, fingerprints, height, tables=None):
    out = [_HDR2.pack(MAGIC2, f["N"], f["C"], f["P"], f["n_planes"], f["items"], f["item_rows"], f["seg_rows"],
                      int(height), FLAG_TABLES if tables is not None else 0)]
    out += [_PLANE2.pack(float(l), fp) for l, fp in zip(lambdas, fingerprints)]
    if tables is not None:
        out.append(np.ascontiguousarray(tables - 1, dtype="<u2").tobytes())
    return out


def _lambdas(lambdas, L):
    lam = [0.0] * L if lambdas is None else [float(l) for l in lambdas]
    if len(lam) != L:
        raise ValueError("vbq_b200.serialize: %d lambdas for %d planes" % (len(lam), L))
    return lam


def encode(qidx, tables, max_bits: int, items: int = 1, seg_rows=None, embed_tables: bool = False, lambdas=None,
           height: int = 0) -> bytes:
    """Entropy-code sorted quantile indices into one VBQ2 blob (one kernel launch for all planes).

    qidx: (rows, C) or (L, rows, C) int32 CUDA tensor, rows = items * item_rows (each item, e.g. one image, in row
    order).  tables: (C, Q) or (L, C, Q) integer frequency tables (`coding.frequency_tables`).  seg_rows: rows per
    coded segment (default: the whole item); every segment of every 32-channel group costs a 32-bit state per channel.
    embed_tables: store the tables in the blob (for streams coded from their own counts).  lambdas: the plane labels
    recorded in the header (default 0.0).  height: H' of an item of H' x W' latent rows, recorded for the receiver."""
    f, words, t = _encode_payload(qidx, tables, max_bits, items, seg_rows)
    fps = [coding.fingerprint(t[i]) for i in range(f["n_planes"])]
    out = _header(f, _lambdas(lambdas, f["n_planes"]), fps, height, t if embed_tables else None)
    out.append(words.astype("<u2").tobytes())
    return b"".join(out)


def encode_items(qidx, tables, max_bits: int, items: int, seg_rows=None, lambdas=None, height: int = 0):
    """Like `encode` (one launch for every plane and item), but returns one separately decodable VBQ2 blob per
    (plane, item): a list over planes of lists over items of bytes."""
    f, words, t = _encode_payload(qidx, tables, max_bits, items, seg_rows)
    lam = _lambdas(lambdas, f["n_planes"])
    G = f["items"] * -(-f["item_rows"] // f["seg_rows"]) * -(-f["C"] // 32)
    per_item = G // f["items"] if f["items"] else 0
    one = dict(f, n_planes=1, items=1)
    out, pos = [], 0
    for p in range(f["n_planes"]):
        ends = words[pos:pos + 2 * G].astype(np.uint64)
        ends = ends[0::2] | (ends[1::2] << np.uint64(16))
        data = words[pos + 2 * G:pos + 2 * G + (int(ends[-1]) if G else 0)]
        pos += 2 * G + (int(ends[-1]) if G else 0)
        hdr = b"".join(_header(one, [lam[p]], [coding.fingerprint(t[p])], height))
        blobs = []
        for i in range(f["items"]):
            a = int(ends[i * per_item - 1]) if i and per_item else 0
            b = int(ends[(i + 1) * per_item - 1]) if per_item else 0
            e = ends[i * per_item:(i + 1) * per_item] - np.uint64(a)
            tab = np.stack([e & np.uint64(0xFFFF), e >> np.uint64(16)], axis=1).reshape(-1).astype("<u2")
            blobs.append(hdr + tab.tobytes() + data[a:b].astype("<u2").tobytes())
        out.append(blobs)
    return out


def read_header(data: bytes) -> dict:
    """Parse and check a VBQ2 header (host only): N, C, prob_bits, n_planes, items, item_rows, seg_rows, height,
    flags, lambdas, fingerprints, embedded tables or None, and the byte offset of the payload.  Raises ValueError."""
    data = memoryview(data)
    if len(data) < _HDR2.size:
        raise ValueError("vbq_b200.serialize: %d bytes are too short for a VBQ2 header" % len(data))
    magic, N, C, P, L, items, item_rows, seg_rows, height, flags = _HDR2.unpack_from(data, 0)
    if magic != MAGIC2:
        raise ValueError("vbq_b200.serialize: bad magic %r (expected %r)" % (bytes(magic), MAGIC2))
    if N > 10 or C < 1 or L < 1 or seg_rows < 1 or not 12 <= P <= 16 or flags & ~FLAG_TABLES:
        raise ValueError("vbq_b200.serialize: bad VBQ2 header (N=%d C=%d prob_bits=%d planes=%d seg_rows=%d flags=%d)"
                         % (N, C, P, L, seg_rows, flags))
    if height and item_rows % height:
        raise ValueError("vbq_b200.serialize: height %d does not divide %d rows" % (height, item_rows))
    Q = ops.num_levels(N)
    pos = _HDR2.size + L * _PLANE2.size
    if len(data) < pos:
        raise ValueError("vbq_b200.serialize: truncated plane table")
    planes = [_PLANE2.unpack_from(data, _HDR2.size + i * _PLANE2.size) for i in range(L)]
    tables = None
    if flags & FLAG_TABLES:
        n = L * C * Q
        if len(data) < pos + 2 * n:
            raise ValueError("vbq_b200.serialize: truncated frequency tables")
        tables = np.frombuffer(data, dtype="<u2", count=n, offset=pos).astype(np.int64).reshape(L, C, Q) + 1
        pos += 2 * n
    return dict(max_bits=N, C=C, prob_bits=P, n_planes=L, items=items, item_rows=item_rows, seg_rows=seg_rows,
                height=height, flags=flags, lambdas=[p[0] for p in planes], fingerprints=[p[1] for p in planes],
                tables=tables, payload_offset=pos)


def _group_bounds(words, h):
    """The group word ranges of a VBQ2 payload (see _offset_bounds)."""
    C, items = h["C"], h["items"]
    n_segs = -(-h["item_rows"] // h["seg_rows"])
    CG = -(-C // 32)
    nact = np.tile(np.minimum(32, C - 32 * np.arange(CG)), items * n_segs).astype(np.int64)
    return _offset_bounds(words, [nact] * h["n_planes"])


def _offset_bounds(words, nacts):
    """Check the offset tables of a payload whose planes have groups of nacts[p] state lanes each (monotone, every group
    holding at least its states, inside the payload, nothing left over) -> (all groups, 2) int64 word ranges."""
    bounds, pos = [], 0
    for nact in nacts:
        G = nact.size
        if pos + 2 * G > words.size:
            raise ValueError("vbq_b200.serialize: payload truncated in an offset table")
        e = words[pos:pos + 2 * G].astype(np.int64)
        ends = e[0::2] | (e[1::2] << 16)
        starts = np.concatenate([[0], ends[:-1]])[:G].astype(np.int64)
        base = pos + 2 * G
        if G and ((ends - starts < 2 * nact).any() or base + ends[-1] > words.size):
            raise ValueError("vbq_b200.serialize: offset table out of range")
        bounds.append(np.stack([base + starts, base + ends], axis=1))
        pos = base + (int(ends[-1]) if G else 0)
    if pos != words.size:
        raise ValueError("vbq_b200.serialize: %d bytes after the last plane" % (2 * (words.size - pos)))
    return np.concatenate(bounds) if bounds else np.zeros((0, 2), np.int64)


def decode(data: bytes, tables=None, code_points=None, device="cuda", want_qidx: bool = True) -> dict:
    """Inverse of `encode`.  tables: one (C, Q) integer table per plane (a sequence, an (L, C, Q) array, or a dict
    keyed by the header's lambdas); default: the tables embedded in the blob.  Every table must have the fingerprint
    the header records.  code_points: (C, Q) ascending code points (`code_points_by_channel`) to produce z_hat.

    Returns dict(qidx, zhat: (n_planes, items, item_rows, C) device tensors or None, and the header fields).  A
    malformed header or offset table, or a table with the wrong fingerprint, raises ValueError before any launch; a
    payload that fails the decoder's integrity check raises ValueError after it."""
    h = read_header(data)
    L, C, P, N = h["n_planes"], h["C"], h["prob_bits"], h["max_bits"]
    if tables is None:
        if h["tables"] is None:
            raise ValueError("vbq_b200.serialize: the blob embeds no frequency tables; pass `tables`")
        tables = h["tables"]
    elif isinstance(tables, dict):
        try:
            tables = [tables[lam] for lam in h["lambdas"]]
        except KeyError as e:
            raise ValueError("vbq_b200.serialize: no table for lambda %r" % (e.args[0],))
    t = _as_tables([np.asarray(x) for x in tables] if isinstance(tables, (list, tuple)) else tables, L)
    if t.shape[1:] != (C, ops.num_levels(N)):
        raise ValueError("vbq_b200.serialize: tables are %s, the blob needs (%d, %d)" % (t.shape[1:], C, ops.num_levels(N)))
    for i in range(L):
        if coding.fingerprint(t[i]) != h["fingerprints"][i]:
            raise ValueError("vbq_b200.serialize: the frequency table of plane %d (lambda %r) has another fingerprint "
                             "than the one the stream was coded with" % (i, h["lambdas"][i]))
    t = coding.check_tables(t, P)
    words = _payload_words(data, h)
    bounds = _group_bounds(words, h)
    dev = torch.device(device)
    w = torch.from_numpy(words.view(np.int16).copy()).to(dev)
    b = torch.from_numpy(np.ascontiguousarray(bounds, dtype=np.int64)).to(dev)
    cum = torch.from_numpy(coding.cum_table(t).view(np.int16)).to(dev)
    cp = None if code_points is None else code_points.to(device=dev, dtype=torch.float32).contiguous()
    q, z, status = ops.rans_decode(w, b, cum, h["items"], h["item_rows"], h["seg_rows"], N, P, cp, want_qidx)
    st = int(status.item())
    if st:
        raise ValueError("vbq_b200.serialize: corrupt VBQ2 payload (decoder status %d: %s)" % (st, _status_text(st)))
    out = {k: v for k, v in h.items() if k not in ("tables", "payload_offset")}
    out.update(qidx=q, zhat=z)
    return out


def _payload_words(data, h):
    rest = len(data) - h["payload_offset"]
    if rest % 2:
        raise ValueError("vbq_b200.serialize: payload of odd length")
    return np.frombuffer(data, dtype="<u2", count=rest // 2, offset=h["payload_offset"])


_STATUS_BITS = ((1, "a group ran out of words"), (2, "integrity check failed"), (4, "bad group range or initial state"),
                (8, "bad work unit"))


def _status_text(st):
    return ", ".join(m for bit, m in _STATUS_BITS if st & bit)


# ------------------------------------------------------------------------------------------------------
# many VBQ2 blobs in one launch (vbq_rans_decode_batch)
# ------------------------------------------------------------------------------------------------------
BATCH_CTA_UNITS = 8         # units per CTA descriptor: the decoder's warps per CTA


def batch_plan(headers, payloads, table_ids):
    """The work list of `decode_many` (host only).  headers: `read_header` dicts of blobs sharing C; payloads: each
    blob's payload as uint16 words; table_ids: per blob, the table index of each plane.  Checks every offset table and
    returns dict(words: the payloads back to back, units (U, 7) int64 (vbq_rans_batch_unit: start, end, out, rows,
    table, cg, blob), ctas (K, 4) int64 (vbq_rans_batch_cta: first, count, table, cg), offsets: each blob's first output
    element, sizes: its element count, n_out).  Blob b's output block is (n_planes, items, item_rows, C) at
    offsets[b].  Units are ordered by (table, cg), then blob, plane, item, segment, and each descriptor takes up to
    BATCH_CTA_UNITS consecutive units of one (table, cg)."""
    B = len(headers)
    C = headers[0]["C"] if B else 1
    CG = -(-C // 32)
    f = {k: np.array([h[k] for h in headers], dtype=np.int64) for k in ("n_planes", "items", "item_rows", "seg_rows")}
    L, items, item_rows, seg = f["n_planes"], f["items"], f["item_rows"], f["seg_rows"]
    n_segs = -(-item_rows // seg)
    G = L * items * n_segs * CG
    sizes = L * items * item_rows * C
    offsets = np.cumsum(sizes) - sizes
    lens = np.array([p.size for p in payloads], dtype=np.int64)
    bases = np.cumsum(lens) - lens
    # group ranges of every blob, in (plane, item, segment, cg) order, moved to the concatenated payload
    bounds = [_group_bounds(p, h) + base for p, h, base in zip(payloads, headers, bases)]
    bounds = np.concatenate(bounds) if B else np.zeros((0, 2), np.int64)
    blob = np.repeat(np.arange(B, dtype=np.int64), G)
    g = np.arange(int(G.sum()), dtype=np.int64) - np.repeat(np.cumsum(G) - G, G)
    cg = g % CG
    rest = g // CG
    sg = rest % n_segs[blob]
    rest //= n_segs[blob]
    item = rest % items[blob]
    plane = rest // items[blob]
    r0 = sg * seg[blob]
    rows = np.minimum(seg[blob], item_rows[blob] - r0)
    out = offsets[blob] + ((plane * items[blob] + item) * item_rows[blob] + r0) * C + 32 * cg
    tids = np.array([t for ids in table_ids for t in ids], dtype=np.int64)
    table = tids[(np.cumsum(L) - L)[blob] + plane]
    units = np.stack([bounds[:, 0], bounds[:, 1], out, rows, table, cg, blob], axis=1)
    units, ctas = _into_ctas(units, table, cg, CG)
    words = np.concatenate(payloads) if B else np.zeros(0, np.uint16)
    return dict(words=words, units=units, ctas=ctas, offsets=offsets, sizes=sizes, n_out=int(sizes.sum()))


def _into_ctas(units, table, cg, CG):
    """Units (rows of an int64 array) sorted stably by (table, cg), and the CTA descriptors (K, 4) int64 (first, count,
    table, cg) that take up to BATCH_CTA_UNITS consecutive units of one (table, cg) each."""
    U = units.shape[0]
    order = np.lexsort((np.arange(U), cg, table))
    units, table, cg = units[order], table[order], cg[order]
    key = table * CG + cg
    new_run = np.ones(U, bool)
    new_run[1:] = key[1:] != key[:-1]
    run_starts = np.flatnonzero(new_run)
    run = np.cumsum(new_run) - 1
    pos = np.arange(U) - run_starts[run]
    first = np.flatnonzero(pos % BATCH_CTA_UNITS == 0)
    run_ends = np.append(run_starts[1:], U)
    count = np.minimum(BATCH_CTA_UNITS, run_ends[run[first]] - first)
    ctas = np.stack([first, count, table[first], cg[first]], axis=1).astype(np.int64)
    return np.ascontiguousarray(units), ctas


def _resolve_tables(h, tables, b):
    """The tables argument of `decode_many` for blob b: per plane a (key, table) pair, where equal keys mean the same
    table object (fingerprinted once)."""
    L = h["n_planes"]
    if tables is None:
        if h["tables"] is None:
            raise ValueError("vbq_b200.serialize: blob %d embeds no frequency tables; pass `tables`" % b)
        return [(("blob", b, i), h["tables"][i]) for i in range(L)]
    if isinstance(tables, dict):
        try:
            return [(("obj", id(tables[lam])), tables[lam]) for lam in h["lambdas"]]
        except KeyError as e:
            raise ValueError("vbq_b200.serialize: blob %d: no table for lambda %r" % (b, e.args[0]))
    if isinstance(tables, (list, tuple)):
        if len(tables) != L:
            raise ValueError("vbq_b200.serialize: blob %d has %d planes, got %d tables" % (b, L, len(tables)))
        return [(("obj", id(t)), t) for t in tables]
    t = np.asarray(tables)
    if t.ndim == 2:
        return [(("obj", id(tables)), t)] * L
    t = _as_tables(t, L)
    return [(("obj", id(tables), i), t[i]) for i in range(L)]


def decode_blobs(blobs, headers, plane_tables, code_points=None, device="cuda", want_qidx: bool = True):
    """`decode_many` with parsed headers and resolved tables (plane_tables: per blob a list of (key, table) pairs as
    `_resolve_tables` makes them).  Returns (list of result dicts, flat qidx or None, flat zhat or None): every result
    tensor is a view into the flat buffers, in blob order."""
    if not blobs:
        return [], None, None
    C, N = headers[0]["C"], headers[0]["max_bits"]
    for b, h in enumerate(headers):
        if (h["C"], h["max_bits"]) != (C, N):
            raise ValueError("vbq_b200.serialize: blob %d has C=%d N=%d, blob 0 has C=%d N=%d; one call decodes "
                             "blobs of one quantizer" % (b, h["C"], h["max_bits"], C, N))
    Q = ops.num_levels(N)
    ids, distinct, table_ids = {}, [], []
    for b, (h, pt) in enumerate(zip(headers, plane_tables)):
        row = []
        for i, (key, table) in enumerate(pt):
            if key not in ids:
                t = np.asarray(table)
                if t.shape != (C, Q):
                    raise ValueError("vbq_b200.serialize: blob %d: tables are %s, the blob needs (%d, %d)"
                                     % (b, t.shape, C, Q))
                P = coding.prob_bits_of(t)
                ids[key] = len(distinct)
                distinct.append((coding.check_tables(t, P), coding.fingerprint(t), P))
            tid = ids[key]
            if distinct[tid][1] != h["fingerprints"][i] or distinct[tid][2] != h["prob_bits"]:
                raise ValueError("vbq_b200.serialize: blob %d: the frequency table of plane %d (lambda %r) has another "
                                 "fingerprint than the one the stream was coded with" % (b, i, h["lambdas"][i]))
            row.append(tid)
        table_ids.append(row)
    plan = batch_plan(headers, [_payload_words(d, h) for d, h in zip(blobs, headers)], table_ids)
    dev = torch.device(device)
    w = torch.from_numpy(plan["words"].view(np.int16)).to(dev)
    cum = torch.from_numpy(np.stack([coding.cum_table(t) for t, _, _ in distinct]).view(np.int16)).to(dev)
    pb = torch.tensor([P for _, _, P in distinct], dtype=torch.int32).to(dev)
    units = torch.from_numpy(plan["units"]).to(dev)
    ctas = torch.from_numpy(plan["ctas"]).to(dev)
    cp = None if code_points is None else code_points.to(device=dev, dtype=torch.float32).contiguous()
    q, z, status = ops.rans_decode_batch(w, cum, pb, units, ctas, len(blobs), N, plan["n_out"], cp, want_qidx)
    st = status.cpu().numpy()
    bad = np.flatnonzero(st)
    if bad.size:
        raise ValueError("vbq_b200.serialize: corrupt VBQ2 payload in blob%s %s (%s)" % (
            "s" if bad.size > 1 else "", ", ".join(str(b) for b in bad),
            "; ".join("blob %d: decoder status %d: %s" % (b, st[b], _status_text(int(st[b]))) for b in bad)))
    outs = []
    for h, o, n in zip(headers, plan["offsets"].tolist(), plan["sizes"].tolist()):
        shape = (h["n_planes"], h["items"], h["item_rows"], C)
        r = {k: v for k, v in h.items() if k not in ("tables", "payload_offset")}
        r.update(qidx=None if q is None else q[o:o + n].view(shape), zhat=None if z is None else z[o:o + n].view(shape))
        outs.append(r)
    return outs, q, z


def decode_many(blobs, tables=None, code_points=None, device="cuda", want_qidx: bool = True) -> list:
    """`decode` of every blob of a list in one kernel launch: a list of dicts, one per blob, each equal to what
    `decode` returns for that blob (qidx / zhat are views into one device buffer each).  The blobs may differ in
    lambda, prob_bits, seg_rows, item_rows, height, n_planes and items, and must share C and N.  tables: as for
    `decode`, applied to every blob.  Every header, table fingerprint and offset table is checked before anything is
    uploaded; a payload that fails the decoder's integrity check raises ValueError naming the failing blobs and their
    status bits, and no result is returned."""
    blobs = list(blobs)
    headers = [read_header(d) for d in blobs]
    plane_tables = [_resolve_tables(h, tables, b) for b, h in enumerate(headers)]
    return decode_blobs(blobs, headers, plane_tables, code_points, device, want_qidx)[0]


# ------------------------------------------------------------------------------------------------------
# many images in one launch (vbq_rans_encode_batch)
# ------------------------------------------------------------------------------------------------------
def encode_plan(item_rows, seg_rows, C: int, table_ids) -> dict:
    """The work list of `encode_many` (host only), the mirror of `batch_plan`.  item_rows: (B,) rows of each image, the
    images back to back in each of the L = len(table_ids) planes; seg_rows: rows per segment (None: the whole image);
    table_ids: the table index of each plane.  Blob p B + b is image b of plane p, its groups in (segment, cg) order.
    Returns dict(units (U, 7) int64 (vbq_rans_encode_unit: in, rows, table, cg, group, scratch, blob) sorted stably by
    (table, cg), ctas (K, 4) int64 (vbq_rans_batch_cta), blob_groups (L B + 1,) int64, seg (B,) the seg_rows each blob
    records, n_groups, scratch_words (every unit its own range of nact (rows + 2) words) and payload_words, the
    payload bound 2 n_groups + scratch_words).  Raises ValueError for an image whose worst case exceeds the 32-bit
    offset table."""
    R = np.asarray(item_rows, dtype=np.int64).reshape(-1)
    tids = np.asarray(table_ids, dtype=np.int64).reshape(-1)
    B, L, CG = R.size, tids.size, -(-C // 32)
    seg = np.maximum(1, R if seg_rows is None else np.full(B, int(seg_rows), np.int64))
    n_segs = -(-R // seg)
    worst = C * (R + 2 * n_segs)                   # an image's group data if every lane emitted a word on every row
    if (worst >= 2 ** 32).any():
        b = int(np.flatnonzero(worst >= 2 ** 32)[0])
        raise ValueError("vbq_b200.serialize: image %d of %d rows x %d channels in segments of %d rows exceeds the "
                         "32-bit offset table" % (b, R[b], C, seg[b]))
    row0 = np.cumsum(R) - R
    G = np.tile(n_segs * CG, L)                    # groups of blob p B + b
    blob_groups = np.concatenate([[0], np.cumsum(G)]).astype(np.int64)
    n_groups = int(blob_groups[-1])
    blob = np.repeat(np.arange(L * B, dtype=np.int64), G)
    g = np.arange(n_groups, dtype=np.int64)
    local = g - blob_groups[blob]
    cg = local % CG
    plane, b = blob // max(B, 1), blob % max(B, 1)
    r0 = (local // CG) * seg[b]
    rows = np.minimum(seg[b], R[b] - r0)
    nact = np.minimum(32, C - 32 * cg)
    words = nact * (rows + 2)
    scratch = np.cumsum(words) - words
    table = tids[plane]
    units = np.stack([(plane * int(R.sum()) + row0[b] + r0) * C + 32 * cg, rows, table, cg, g, scratch, blob], axis=1)
    units, ctas = _into_ctas(units.astype(np.int64), table, cg, CG)
    scratch_words = int(words.sum())
    return dict(units=units, ctas=ctas, blob_groups=blob_groups, seg=seg, n_groups=n_groups,
                scratch_words=scratch_words, payload_words=2 * n_groups + scratch_words)


def encode_many(qidx, tables, max_bits: int, item_rows, seg_rows=None, lambdas=None, heights=None) -> list:
    """Entropy-code many images of different shapes in one launch each of encode, scan and compaction: one VBQ2 blob
    per (plane, image), as a list over planes of lists over images of bytes.

    qidx: (L, total_rows, C) int32 CUDA tensor (what `quantize` returns for images concatenated row-wise).  tables: one
    (C, Q) integer table per plane (an (L, C, Q) array, a (C, Q) array for every plane, or a sequence); planes may
    differ in prob_bits.  item_rows: each image's row count.  seg_rows: rows per coded segment (default: the whole
    image).  lambdas: the plane labels (default 0.0).  heights: each image's H' (default 0, unknown).  Blob [p][b] is
    byte-identical to `encode_items(qidx[p:p+1, rows of image b], tables[p], max_bits, items=1, seg_rows=seg_rows,
    lambdas=[lambdas[p]], height=heights[b])[0][0]`.

    Every table is checked and fingerprinted once.  Item rows that do not sum to the rows, a height that does not
    divide its image's rows and tables of the wrong shape raise ValueError before any launch.  The call synchronises
    with the host twice: once for one copy of the blob starts and statuses, and once for the copy of the payload.  A
    symbol outside [0, Q) raises ValueError naming the images it lies in."""
    q = qidx if qidx.dim() == 3 else qidx.unsqueeze(0)
    L, rows, C = q.shape
    R = np.asarray(item_rows, dtype=np.int64).reshape(-1)
    B = R.size
    if (R < 0).any() or int(R.sum()) != rows:
        raise ValueError("vbq_b200.serialize: item_rows %s do not sum to the %d rows" % (R.tolist(), rows))
    hs = np.zeros(B, np.int64) if heights is None else np.asarray(heights, dtype=np.int64).reshape(-1)
    if hs.size != B:
        raise ValueError("vbq_b200.serialize: %d heights for %d images" % (hs.size, B))
    for b in np.flatnonzero((hs < 0) | ((hs > 0) & (R % np.maximum(hs, 1) != 0))):
        raise ValueError("vbq_b200.serialize: height %d does not divide the %d rows of image %d" % (hs[b], R[b], b))
    lam = _lambdas(lambdas, L)
    Q = ops.num_levels(max_bits)
    if isinstance(tables, (list, tuple)):
        if len(tables) != L:
            raise ValueError("vbq_b200.serialize: %d tables for %d planes" % (len(tables), L))
        keyed = [(id(t), t) for t in tables]
    elif np.ndim(tables) == 2:
        keyed = [(id(tables), tables)] * L
    else:
        t = _as_tables(tables, L)
        keyed = [((id(tables), p), t[p]) for p in range(L)]
    ids, distinct, table_ids = {}, [], []
    for p, (key, table) in enumerate(keyed):
        if key not in ids:
            t = np.asarray(table)
            if t.shape != (C, Q):
                raise ValueError("vbq_b200.serialize: the table of plane %d is %s, need (C, Q) = (%d, %d)"
                                 % (p, t.shape, C, Q))
            P = coding.prob_bits_of(t)
            ids[key] = len(distinct)
            distinct.append((coding.check_tables(t, P), coding.fingerprint(t), P))
        table_ids.append(ids[key])
    plan = encode_plan(R, seg_rows, C, table_ids)
    if B == 0:
        return [[] for _ in range(L)]
    dev = q.device
    U, K, LB = plan["units"].shape[0], plan["ctas"].shape[0], L * B
    index = torch.from_numpy(np.concatenate([plan["units"].reshape(-1), plan["ctas"].reshape(-1),
                                             plan["blob_groups"]])).to(dev)      # one upload for the work list
    units = index[:7 * U].view(U, 7)
    ctas = index[7 * U:7 * U + 4 * K].view(K, 4)
    cum = torch.from_numpy(np.stack([coding.cum_table(t) for t, _, _ in distinct]).view(np.int16)).to(dev)
    pb = torch.tensor([P for _, _, P in distinct], dtype=torch.int32).to(dev)
    payload, meta = ops.rans_encode_batch(q.contiguous(), cum, pb, units, ctas, index[7 * U + 4 * K:],
                                          plan["n_groups"], max_bits, plan["scratch_words"])
    m = utils.to_host_numpy(meta)
    starts, status = m[:LB + 1], m[LB + 1:].view(np.int32)[:LB]
    bad = np.flatnonzero(status)
    if bad.size:
        where = "; ".join("image %d of plane %d (lambda %r): %s" % (i % B, i // B, lam[i // B],
                                                                   _encode_status_text(int(status[i]))) for i in bad)
        raise ValueError("vbq_b200.serialize: cannot encode image%s %s for max_bits=%d (%s)" % (
            "s" if len(set((bad % B).tolist())) > 1 else "", ", ".join(str(b) for b in sorted(set((bad % B).tolist()))),
            max_bits, where))
    words = utils.to_host_numpy(payload[:int(starts[-1])]).view(np.uint16).astype("<u2", copy=False)
    out = []
    for p in range(L):
        _, fp, P = distinct[table_ids[p]]
        blobs = []
        for b in range(B):
            f = dict(N=max_bits, C=C, P=P, n_planes=1, items=1, item_rows=int(R[b]), seg_rows=int(plan["seg"][b]))
            i = p * B + b
            blobs.append(b"".join(_header(f, [lam[p]], [fp], int(hs[b]))) + words[starts[i]:starts[i + 1]].tobytes())
        out.append(blobs)
    return out


def _encode_status_text(st):
    return ", ".join(m for bit, m in ((1, "a symbol lies outside [0, Q)"), (8, "bad work unit")) if st & bit)


# ------------------------------------------------------------------------------------------------------
# VBQE: rANS-coded word embeddings, one shared table per blob
# ------------------------------------------------------------------------------------------------------
MAGIC_E = b"VBQE"
_HDRE = struct.Struct("<4sIII")       # magic, N, prob_bits, ndim; then ndim uint64 extents
_HDRE2 = struct.Struct("<QddQI")      # seg_rows, empirical_std, beta, code-point fingerprint, used symbols k
_MAX_NDIM = 32


def shared_seg_rows(n: int, seg_rows: int) -> int:
    """seg_rows as the shared-table coder uses it: a segment longer than the plane is the whole plane."""
    return max(1, min(int(seg_rows), -(-int(n) // 32)))


def shared_nact(n: int, seg_rows: int) -> np.ndarray:
    """State lanes of every group of a plane of n symbols in the shared-table layout: 32, except for a group that
    starts on the plane's last, partial row."""
    seg = shared_seg_rows(n, seg_rows)
    G = -(-(-(-n // 32)) // seg)
    return np.minimum(32, n - 32 * seg * np.arange(G, dtype=np.int64))


def embedding_header(max_bits, prob_bits, shape, seg_rows, empirical_std, beta, fingerprint, table) -> bytes:
    """The VBQE header and sparse table of one plane (table: (Q,) integer frequencies)."""
    t = np.asarray(table, dtype=np.int64)
    used = np.flatnonzero(t)
    return b"".join([_HDRE.pack(MAGIC_E, int(max_bits), int(prob_bits), len(shape)),
                     struct.pack("<%dQ" % len(shape), *[int(d) for d in shape]),
                     _HDRE2.pack(int(seg_rows), float(empirical_std), float(beta), int(fingerprint), used.size),
                     used.astype("<u2").tobytes(), t[used].astype("<u4").tobytes()])


def encode_embeddings(qidx, tables, max_bits: int, shape, seg_rows, empirical_std: float, betas, fingerprint: int):
    """Entropy-code L planes of symbols with the shared-table coder in one launch; one VBQE blob per plane.

    qidx: (L, n) int32 CUDA tensor of sorted quantile indices, n = prod(shape).  tables: (L, Q) integer frequencies
    (`coding.frequency_tables(counts, keep_zeros=True)`).  seg_rows: one per plane.  empirical_std, betas and the
    code-point fingerprint are recorded for the receiver.  Raises ValueError for a symbol outside [0, Q) or one whose
    frequency is 0."""
    L, n = qidx.shape
    if n != math.prod(shape):
        raise ValueError("vbq_b200.serialize: %d symbols do not fill shape %s" % (n, tuple(shape)))
    Q = ops.num_levels(max_bits)
    t = np.asarray(tables)
    if t.shape != (L, Q):
        raise ValueError("vbq_b200.serialize: tables are %s, need (%d, %d)" % (t.shape, L, Q))
    P = coding.prob_bits_of(t)
    t = coding.check_shared_tables(t, P)
    if any(int(x) < 1 for x in seg_rows):
        raise ValueError("vbq_b200.serialize: seg_rows must be >= 1, got %s" % (list(seg_rows),))
    seg = [shared_seg_rows(n, x) for x in seg_rows]
    cum = torch.from_numpy(coding.cum_table_shared(t).view(np.int32)).to(qidx.device)
    payload, size, status = ops.rans_shared_encode(qidx, cum, max_bits, P, seg)
    st = int(status.item())
    if st:
        raise ValueError("vbq_b200.serialize: " + " and ".join(
            m for bit, m in ((1, "a symbol lies outside [0, Q) for max_bits=%d" % max_bits),
                             (2, "a symbol has frequency 0 in its table")) if st & bit))
    words = payload[:int(size.item()) // 2].cpu().numpy().view(np.uint16)
    out, pos = [], 0
    for p in range(L):
        G = shared_nact(n, seg[p]).size
        e = words[pos:pos + 2 * G].astype(np.int64)
        end = pos + 2 * G + (int(e[-2] | (e[-1] << 16)) if G else 0)
        hdr = embedding_header(max_bits, P, shape, seg[p], empirical_std, betas[p], fingerprint, t[p])
        out.append(hdr + words[pos:end].astype("<u2").tobytes())
        pos = end
    return out


def read_embedding_header(data: bytes) -> dict:
    """Parse and check a VBQE blob on the host: max_bits, prob_bits, shape, seg_rows, empirical_std, beta,
    fingerprint, table ((Q,) int64 frequencies), and the payload's group word ranges `bounds` and `words`.  Raises
    ValueError for a bad magic, a truncated blob, a table that is unsorted, out of range or does not sum to
    2^prob_bits, a malformed offset table or bytes after the payload."""
    data = memoryview(data)
    if len(data) < _HDRE.size:
        raise ValueError("vbq_b200.serialize: %d bytes are too short for a VBQE header" % len(data))
    magic, N, P, ndim = _HDRE.unpack_from(data, 0)
    if magic != MAGIC_E:
        raise ValueError("vbq_b200.serialize: bad magic %r (expected %r)" % (bytes(magic), MAGIC_E))
    if N > 10 or not 12 <= P <= 16 or ndim > _MAX_NDIM:
        raise ValueError("vbq_b200.serialize: bad VBQE header (N=%d prob_bits=%d ndim=%d)" % (N, P, ndim))
    pos = _HDRE.size
    if len(data) < pos + 8 * ndim + _HDRE2.size:
        raise ValueError("vbq_b200.serialize: truncated VBQE header")
    shape = tuple(struct.unpack_from("<%dQ" % ndim, data, pos))
    pos += 8 * ndim
    seg_rows, std, beta, fp, k = _HDRE2.unpack_from(data, pos)
    pos += _HDRE2.size
    Q = ops.num_levels(N)
    n = math.prod(shape)
    if not 1 <= seg_rows <= max(1, -(-n // 32)) or not 1 <= k <= Q:
        raise ValueError("vbq_b200.serialize: bad VBQE header (seg_rows=%d, %d symbols, %d used)" % (seg_rows, n, k))
    if n + 66 * -(-n // (32 * seg_rows)) >= 2 ** 32:       # the coder's limit: a plane's worst case in 32-bit offsets
        raise ValueError("vbq_b200.serialize: %d symbols in segments of %d rows exceed the coder's 32-bit offsets"
                         % (n, seg_rows))
    if len(data) < pos + 6 * k:
        raise ValueError("vbq_b200.serialize: truncated frequency table")
    sym = np.frombuffer(data, dtype="<u2", count=k, offset=pos).astype(np.int64)
    freq = np.frombuffer(data, dtype="<u4", count=k, offset=pos + 2 * k).astype(np.int64)
    pos += 6 * k
    if (np.diff(sym) <= 0).any() or sym[-1] >= Q:
        raise ValueError("vbq_b200.serialize: table symbols unsorted or outside [0, %d)" % Q)
    if (freq < 1).any() or freq.sum() != 1 << P:
        raise ValueError("vbq_b200.serialize: table frequencies do not sum to 2^%d" % P)
    table = np.zeros(Q, np.int64)
    table[sym] = freq
    rest = len(data) - pos
    if rest % 2:
        raise ValueError("vbq_b200.serialize: payload of odd length")
    words = np.frombuffer(data, dtype="<u2", count=rest // 2, offset=pos)
    if 2 * -(-n // (32 * seg_rows)) > words.size:      # checked before the per-group arrays are built
        raise ValueError("vbq_b200.serialize: payload truncated in an offset table")
    bounds = _offset_bounds(words, [shared_nact(n, seg_rows)])
    return dict(max_bits=N, prob_bits=P, shape=shape, seg_rows=seg_rows, empirical_std=std, beta=beta,
                fingerprint=fp, table=table, words=words, bounds=bounds)


def decode_embedding(data: bytes, code_points=None, device="cuda", want_qidx: bool = True) -> dict:
    """Inverse of `encode_embeddings` for one blob: the header fields of `read_embedding_header` plus qidx and zhat,
    flat (n,) device tensors or None (zhat = code_points[q] for a (Q,) ascending table).  A malformed blob raises
    ValueError before any launch; a payload that fails the decoder's integrity check raises ValueError after it."""
    h = read_embedding_header(data)
    n = math.prod(h["shape"])
    dev = torch.device(device)
    w = torch.from_numpy(h["words"].view(np.int16).copy()).to(dev)
    b = torch.from_numpy(np.ascontiguousarray(h["bounds"], dtype=np.int64)).to(dev)
    cum = torch.from_numpy(coding.cum_table_shared(h["table"][None]).view(np.int32)).to(dev)
    cp = None if code_points is None else code_points.to(device=dev, dtype=torch.float32).contiguous()
    q, z, status = ops.rans_shared_decode(w, b, cum, n, h["seg_rows"], h["max_bits"], h["prob_bits"], cp, want_qidx)
    st = int(status.item())
    if st:
        raise ValueError("vbq_b200.serialize: corrupt VBQE payload (decoder status %d: %s)" % (
            st, ", ".join(m for bit, m in ((1, "a group ran out of words"), (2, "integrity check failed"),
                                            (4, "bad group range or initial state")) if st & bit)))
    out = {k: v for k, v in h.items() if k not in ("words", "bounds")}
    out.update(qidx=None if q is None else q[0], zhat=None if z is None else z[0])
    return out
