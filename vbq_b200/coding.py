"""Integer frequency tables for the rANS coder (csrc/rans.cu): from a fitted entropy model or from counts to a (C, Q)
table whose rows hold only entries >= 1 and sum to exactly 2^prob_bits, plus the table's fingerprint and cum form.

The tables are a deterministic NumPy function of the model, so a receiver that holds the same quantizer rebuilds the
sender's tables bit for bit; the 64-bit fingerprint in every VBQ2 header catches a receiver whose tables differ."""
from __future__ import annotations

import hashlib
import heapq
import math
import struct

import numpy as np

DEFAULT_PROB_BITS = 16


def _normalise_row(f, p, M):
    """Fix the sum of one rounded row greedily: each unit goes where it costs the least cross-entropy
    (sum_s p_s * -log2(f_s / M)); ties go to the lower symbol.  Entries of 0 stay 0 and entries of 1 stay >= 1."""
    d = M - int(f.sum())
    if d > 0:
        heap = [(-ps * math.log2((fs + 1) / fs), s) for s, (ps, fs) in enumerate(zip(p.tolist(), f.tolist())) if fs > 0]
        heapq.heapify(heap)
        for _ in range(d):
            _, s = heapq.heappop(heap)
            f[s] += 1
            heapq.heappush(heap, (-p[s] * math.log2((f[s] + 1) / f[s]), s))
    elif d < 0:
        heap = [(ps * math.log2(fs / (fs - 1)), s) for s, (ps, fs) in enumerate(zip(p.tolist(), f.tolist())) if fs > 1]
        heapq.heapify(heap)
        for _ in range(-d):
            _, s = heapq.heappop(heap)
            f[s] -= 1
            if f[s] > 1:
                heapq.heappush(heap, (p[s] * math.log2(f[s] / (f[s] - 1)), s))


def frequency_tables(model, prob_bits: int = DEFAULT_PROB_BITS, keep_zeros: bool = False) -> np.ndarray:
    """(C, Q) int32 frequency tables for the rANS coder.

    ``model`` is either an entropy model (float: -log2 p per channel and symbol, what ``entropy_models[lambda]`` holds)
    or integer counts (what ``ops.symbol_histogram`` returns; a channel without counts gets a uniform table).  Each
    row is p * 2^prob_bits rounded, clamped to >= 1, and brought to a sum of exactly 2^prob_bits by greedy unit
    changes of least cross-entropy cost.  12 <= prob_bits <= 16 and Q <= 2^prob_bits.

    ``keep_zeros=True`` (integer counts only) is the table of the shared-table coder (`vbq_rans_shared_*`), which codes
    the very symbols it was counted on: a symbol with count 0 gets frequency 0, every counted symbol at least 1, and
    a single counted symbol all of 2^prob_bits, so no probability mass is spent on symbols that never occur."""
    m = np.asarray(model)
    if m.ndim == 1:
        m = m[None]
    if m.ndim != 2 or m.shape[1] < 1:
        raise ValueError("vbq_b200.coding: model must be (C, Q), got shape %s" % (m.shape,))
    C, Q = m.shape
    prob_bits = int(prob_bits)
    if not 12 <= prob_bits <= 16 or Q > (1 << prob_bits):
        raise ValueError("vbq_b200.coding: prob_bits=%d (need 12..16 with Q=%d <= 2^prob_bits)" % (prob_bits, Q))
    if keep_zeros and not np.issubdtype(m.dtype, np.integer):
        raise ValueError("vbq_b200.coding: keep_zeros needs integer counts")
    if np.issubdtype(m.dtype, np.integer):
        counts = m.astype(np.float64)
        if (counts < 0).any():
            raise ValueError("vbq_b200.coding: negative counts")
        tot = counts.sum(axis=1, keepdims=True)
        p = np.where(tot > 0, counts / np.maximum(tot, 1), 1.0 / Q)
    else:
        mf = m.astype(np.float64)
        if not np.isfinite(mf).all():
            raise ValueError("vbq_b200.coding: entropy model has non-finite code lengths")
        p = np.exp2(-(mf - mf.min(axis=1, keepdims=True)))
        p /= p.sum(axis=1, keepdims=True)
    M = 1 << prob_bits
    f = np.maximum(1, np.rint(p * M)).astype(np.int64)
    if keep_zeros:
        f[p == 0] = 0
    for c in range(C):
        _normalise_row(f[c], p[c], M)
    return f.astype(np.int32)


def check_tables(f, prob_bits: int) -> np.ndarray:
    """Validate (C, Q) or (L, C, Q) integer tables (entries >= 1, rows summing to 2^prob_bits); returns them as int64."""
    t = np.asarray(f)
    if not np.issubdtype(t.dtype, np.integer):
        raise ValueError("vbq_b200.coding: frequency tables must be integer")
    t = t.astype(np.int64)
    if (t < 1).any() or (t.sum(axis=-1) != (1 << prob_bits)).any():
        raise ValueError("vbq_b200.coding: every frequency must be >= 1 and every row must sum to 2^%d" % prob_bits)
    return t


def prob_bits_of(f) -> int:
    """prob_bits of a table from its row sum (a power of two between 2^12 and 2^16)."""
    t = np.asarray(f, dtype=np.int64)
    tot = int(t.reshape(-1, t.shape[-1])[0].sum())
    P = tot.bit_length() - 1
    if tot != 1 << P or not 12 <= P <= 16:
        raise ValueError("vbq_b200.coding: table rows sum to %d, not 2^prob_bits with 12 <= prob_bits <= 16" % tot)
    return P


def cum_table(f) -> np.ndarray:
    """The kernels' table form: cum[..., s] = f[..., 0] + ... + f[..., s-1] as uint16 (cum[Q] = 2^prob_bits implicit)."""
    t = np.asarray(f, dtype=np.int64)
    return np.ascontiguousarray((np.cumsum(t, axis=-1) - t).astype(np.uint16))


def fingerprint(f) -> int:
    """64-bit fingerprint of one (C, Q) integer table: BLAKE2b-64 of uint32 C, Q and the entries as little-endian
    uint32, read as a little-endian integer."""
    t = np.asarray(f)
    C, Q = t.shape
    h = hashlib.blake2b(struct.pack("<II", C, Q) + np.ascontiguousarray(t, dtype="<u4").tobytes(), digest_size=8)
    return int.from_bytes(h.digest(), "little")


def check_shared_tables(f, prob_bits: int) -> np.ndarray:
    """Validate (L, Q) integer tables of the shared-table coder (entries >= 0, rows summing to 2^prob_bits); returns
    them as int64."""
    t = np.asarray(f)
    if not np.issubdtype(t.dtype, np.integer):
        raise ValueError("vbq_b200.coding: frequency tables must be integer")
    t = t.astype(np.int64)
    if (t < 0).any() or (t.sum(axis=-1) != (1 << prob_bits)).any():
        raise ValueError("vbq_b200.coding: every frequency must be >= 0 and every row must sum to 2^%d" % prob_bits)
    return t


def cum_table_shared(f) -> np.ndarray:
    """The shared-table coder's form: cum[..., s] = f[..., 0] + ... + f[..., s-1] for s = 0..Q as uint32, so
    cum[..., Q] = 2^prob_bits is explicit and a single symbol may hold the whole range."""
    t = np.asarray(f, dtype=np.int64)
    z = np.zeros(t.shape[:-1] + (1,), np.int64)
    return np.ascontiguousarray(np.concatenate([z, np.cumsum(t, axis=-1)], axis=-1).astype(np.uint32))


def code_points_fingerprint(code_points) -> int:
    """64-bit fingerprint of a (Q,) float64 code-point table: BLAKE2b-64 of uint32 Q and the values as little-endian
    float64, read as a little-endian integer.  Sender and receiver must quantize to the same code points bit for bit."""
    c = np.ascontiguousarray(code_points, dtype="<f8").reshape(-1)
    h = hashlib.blake2b(struct.pack("<I", c.size) + c.tobytes(), digest_size=8)
    return int.from_bytes(h.digest(), "little")
