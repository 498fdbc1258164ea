"""Plain NumPy restatement of query scoring against one shared-table plane (include/vbq_b200.h,
vbq_rans_shared_row_scores, CompressedEmbedding.scores / topk): the float32 numerics contract with an exact fma32, and
the work split that gives every embedding row to one warp."""
import numpy as np

F32_MAX = float(np.finfo(np.float32).max)


def fma32(a, b, c):
    """IEEE float32 fmaf(a, b, c) with round-to-nearest-even, elementwise.  The float64 product of two float32 values is
    exact; TwoSum gives the float64 sum s and its exact error; s rounds to float32 correctly unless it lies exactly on a
    float32 midpoint with a non-zero error, where the true value is on the error's side of the midpoint."""
    a, b, c = (np.asarray(v, dtype=np.float32) for v in (a, b, c))
    p = a.astype(np.float64) * b.astype(np.float64)
    c64 = c.astype(np.float64)
    with np.errstate(over="ignore", invalid="ignore"):
        s = p + c64
        bb = s - p
        err = (p - (s - bb)) + (c64 - bb)
        r = s.astype(np.float32)
        r64 = np.where(np.isinf(r), np.copysign(2.0 ** 128, s), r.astype(np.float64))   # inf as 2^128 for the test
        toward = np.where(r64 < s, np.float32(np.inf), np.float32(-np.inf)).astype(np.float32)
        nb = np.nextafter(np.where(np.isinf(r), np.copysign(np.float32(F32_MAX), r), r), toward).astype(np.float32)
        nb = np.where(np.isinf(r), np.copysign(np.float32(F32_MAX), r), nb)
        mid = np.isfinite(s) & (r64 != s) & ((r64 + nb.astype(np.float64)) * 0.5 == s) & (err != 0) & np.isfinite(err)
        # on a midpoint the error's sign picks the neighbour: r if r lies on that side, else nb
        pick_r = (err > 0) == (r64 > s)
    out = np.where(mid & ~pick_r, nb, r).astype(np.float32)
    return out.reshape(np.broadcast(a, b, c).shape)


def _sum4(a):
    return (a[0] + a[1]) + (a[2] + a[3])          # float32 adds


def scores(Z, Q, metric="dot"):
    """(B, V) float32 scores of queries Q (B, D) against rows Z (V, D) (the decoded float32 matrix) under the contract:
    a[d % 4] = fma32(z_d, q_d, a[d % 4]) in d order, dot = (a0 + a1) + (a2 + a3); cosine = dot / (sqrtf(zz) *
    sqrtf(qq)) if that product is > 0, else 0."""
    Z = np.asarray(Z, np.float32).reshape(np.shape(Z)[0], -1)
    Q = np.asarray(Q, np.float32).reshape(np.shape(Q)[0], -1)
    V, D = Z.shape
    B = Q.shape[0]
    acc = np.zeros((4, B, V), np.float32)
    zz = np.zeros((4, V), np.float32)
    qq = np.zeros((4, B), np.float32)
    for d in range(D):
        acc[d % 4] = fma32(Z[None, :, d], Q[:, d, None], acc[d % 4])
        zz[d % 4] = fma32(Z[:, d], Z[:, d], zz[d % 4])
        qq[d % 4] = fma32(Q[:, d], Q[:, d], qq[d % 4])
    with np.errstate(over="ignore", invalid="ignore", divide="ignore"):
        dot = _sum4(acc)
        if metric == "dot":
            return dot
        den = np.sqrt(_sum4(zz))[None, :] * np.sqrt(_sum4(qq))[:, None]
        return np.where(den > 0, dot / np.where(den > 0, den, np.float32(1)), np.float32(0)).astype(np.float32)


def interval(r, seg, K):
    """Checkpoint interval of coder row r: segment C1 + j with C1 = (seg - 1) // K + 1 slots per segment."""
    C1 = (seg - 1) // K + 1
    return (r // seg) * C1 + (r % seg) // K


def owner(e, D, seg, K, ipw):
    """The warp that scores embedding row e: the one whose intervals hold e's first coder row floor(e D / 32)."""
    return interval(e * D // 32, seg, K) // ipw


def warp_rows(w, D, n, seg, K, ipw, row_begin, row_end):
    """[e_lo, e_hi): the rows of [row_begin, row_end) that warp w scores, from the shape alone (as the kernel derives
    them): its intervals' coder rows [ra, rb) hold the first coder rows of rows ceil(32 ra / D) .. ceil(32 rb / D) - 1."""
    rows = -(-n // 32)
    seg = max(1, min(seg, rows))
    K = min(K, seg)
    C1 = (seg - 1) // K + 1
    T = -(-rows // seg) * C1
    I0 = w * ipw
    if I0 >= T:
        return 0, 0
    I1 = min(I0 + ipw, T)
    ra = min((I0 // C1) * seg + (I0 % C1) * K, rows)
    rb = min((I1 // C1) * seg + (I1 % C1) * K, rows)
    lo, hi = max(-(-32 * ra // D), row_begin), min(-(-32 * rb // D), row_end)
    return (lo, hi) if ra < rb and lo < hi else (0, 0)
