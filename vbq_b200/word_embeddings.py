"""Word-embedding VBQ: the notebook cells of the reference's
word-embeddings/compress-trained-word-embeddings.ipynb:373-390 (code points) and :429-443
(`compress_coordinates`), on the GPU.

All coordinates share one zero-mean Gaussian prior N(0, empirical_std^2).  The shared code-point tree is
replicated over 16 virtual channels so the same sm_100a kernel as the image path walks it
(bank-conflict-free interleaving, include/vbq_b200.h)."""
from __future__ import annotations

import math

import numpy as np
import torch

from . import coding, ops, serialize

_VC = 16  # virtual channels = VBQ_GROUP
_FLUSH_BUDGET = 0.005   # default segmentation: flushed states cost at most this share of the plane's entropy
_MIN_SEG_ROWS = 256


def empirical_std(means):
    """ipynb:373-374: sqrt(mean(mu^2))."""
    m = means if isinstance(means, torch.Tensor) else torch.as_tensor(np.asarray(means))
    return float(torch.sqrt(torch.mean(m.double().reshape(-1) ** 2)))


def empirical_entropy(values):
    """ipynb:452-455: total_counts*log2(total_counts) - sum(counts*log2(counts)) over the distinct values, i.e. the
    bit length of an ideal entropy code of the quantized coordinates.  Device tensors stay on the device."""
    t = values if isinstance(values, torch.Tensor) else torch.as_tensor(np.asarray(values))
    _, counts = torch.unique(t.reshape(-1), return_counts=True)
    c = counts.double()
    total = c.sum()
    return float(total * torch.log2(total) - (c * torch.log2(c)).sum())


def _entropy_of_counts(counts):
    """ipynb:452-455 from a count table (the last axis): total log2 total - sum counts log2 counts."""
    c = np.asarray(counts, dtype=np.float64)
    total = c.sum(axis=-1)
    plogp = np.where(c > 0, c * np.log2(np.maximum(c, 1.0)), 0.0).sum(axis=-1)
    return np.where(total > 0, total * np.log2(np.maximum(total, 1.0)), 0.0) - plogp


def default_seg_rows(n: int, entropy_bits: float) -> int:
    """Rows per segment of the shared-table coder for a plane of n symbols: the most segments whose flushed states
    (32 lanes x 32 bits per segment) cost at most 0.5 % of the plane's ideal code length, but no segment shorter than
    256 rows.  More segments mean more warps decoding in parallel."""
    rows = -(-int(n) // 32)
    segs = max(1, int(_FLUSH_BUDGET * float(entropy_bits) // 1024))
    return max(1, min(rows, max(_MIN_SEG_ROWS, -(-rows // segs))))


def _pen_f32(beta):
    """Whether the notebook forms (2 beta) sigma^2 in float32: always, unless beta is a NumPy float64 scalar, which
    NumPy >= 2 promotes to float64."""
    return not (isinstance(beta, np.floating) and np.lib.NumpyVersion(np.__version__) >= "2.0.0")


def _query_matrix(queries, metric, tail):
    """queries (B, *tail) or tail -> (B, prod(tail)) on their own device; TypeError / ValueError before anything
    reaches a device."""
    if metric not in ops.SCORE_METRICS:
        raise ValueError("vbq_b200: metric must be one of %s, got %r" % (sorted(ops.SCORE_METRICS), metric))
    if isinstance(queries, torch.Tensor):
        if not queries.dtype.is_floating_point:
            raise TypeError("vbq_b200: queries must be floating point, got %s" % queries.dtype)
        t = queries
    else:
        a = np.asarray(queries)
        if a.dtype.kind != "f":
            raise TypeError("vbq_b200: queries must be floating point, got %s" % a.dtype)
        t = torch.from_numpy(np.ascontiguousarray(a))
    if tuple(t.shape) == tail:
        t = t.reshape((1,) + tail)
    if t.dim() != len(tail) + 1 or tuple(t.shape[1:]) != tail:
        raise ValueError("vbq_b200: queries must have shape (B, %s) or %s, got %s"
                         % (", ".join(map(str, tail)), tail, tuple(t.shape)))
    return t.reshape(t.shape[0], math.prod(tail))


def _int_tensor(x, name):
    """An integer tensor (any device) from a tensor, array or list; TypeError for anything else."""
    if isinstance(x, torch.Tensor):
        t = x
    else:
        a = np.asarray(x)
        if a.size == 0 and not isinstance(x, np.ndarray):
            a = a.astype(np.int64)
        if a.dtype.kind not in "iu":
            raise TypeError("vbq_b200: %s must be integers, got %s" % (name, a.dtype))
        t = torch.from_numpy(a.astype(np.int64, copy=False))
    if t.dtype not in (torch.int8, torch.int16, torch.int32, torch.int64, torch.uint8):
        raise TypeError("vbq_b200: %s must be an integer tensor, got %s" % (name, t.dtype))
    return t


def _rank_inputs(queries, targets, metric, exclude, tail, V, device):
    """Validates the arguments of the rank functions before any launch: returns (q (B, D) float32, t (B,) int64,
    ex (B, E) int64) on `device`.  One host synchronisation reads the finiteness, the id ranges and the
    target-in-its-exclude-row flag together (none for B = 0)."""
    q = _query_matrix(queries, metric, tail)
    B = q.shape[0]
    t = _int_tensor(targets, "targets")
    if tuple(t.shape) != (B,):
        raise ValueError("vbq_b200: targets must be (%d,), got %s" % (B, tuple(t.shape)))
    if exclude is None:
        ex = torch.full((B, 0), -1, dtype=torch.int64)
    else:
        ex = _int_tensor(exclude, "exclude")
        if ex.dim() != 2 or ex.shape[0] != B:
            raise ValueError("vbq_b200: exclude must be (%d, E), got %s" % (B, tuple(ex.shape)))
    q = q.to(device=device, dtype=torch.float32).contiguous()
    t = t.to(device=device, dtype=torch.int64).contiguous()
    ex = ex.to(device=device, dtype=torch.int64).contiguous()
    if B == 0:
        return q, t, ex
    checks = [torch.isfinite(q).all().to(torch.int64), t.min(), t.max()]
    if ex.shape[1]:
        checks += [ex.min(), ex.max(), (ex == t[:, None]).any().to(torch.int64)]
    got = torch.stack(checks).tolist()
    if not got[0]:
        raise ValueError("vbq_b200: queries must be finite")
    if got[1] < 0 or got[2] >= V:
        raise IndexError("vbq_b200: target %d outside [0, %d)" % (got[1] if got[1] < 0 else got[2], V))
    if ex.shape[1]:
        if got[3] < -1 or got[4] >= V:
            raise IndexError("vbq_b200: exclude id %d outside [-1, %d)" % (got[3] if got[3] < -1 else got[4], V))
        if got[5]:
            raise ValueError("vbq_b200: a target is listed in its own exclude row")
    return q, t, ex


def _score_keys(s):
    """int64 keys of float32 scores in the order of CompressedEmbedding.topk: the order-preserving map of the bits,
    -0.0 as +0.0, NaN lowest."""
    bits = s.view(torch.int32)
    k = torch.where(bits < 0, bits ^ 0x7FFFFFFF, bits)
    k = k.masked_fill(s == 0, 0).masked_fill(torch.isnan(s), -(1 << 31))
    return k.to(torch.int64)


def _excluded_beaters(s, ids, valid, thr, t):
    """(B,) number of distinct excluded rows that beat the target: s (B, E) their scores, ids (B, E) their ids, valid
    marks the first occurrence of each id >= 0, thr (B,) the targets' scores, t (B,) the targets."""
    ks, kt = _score_keys(s), _score_keys(thr)[:, None]
    beats = (ks > kt) | ((ks == kt) & (ids < t[:, None]))
    return (beats & valid).sum(dim=1)


def _distinct_excluded(ex):
    """(sorted ids (B, E), mask of the first occurrence of every id >= 0)."""
    srt = ex.sort(dim=1).values
    valid = srt >= 0
    valid[:, 1:] &= srt[:, 1:] != srt[:, :-1]
    return srt, valid


def _dense_rows(matrix):
    """A (V, *tail) float32 CUDA tensor -> (V, D) contiguous; TypeError / ValueError otherwise."""
    if not isinstance(matrix, torch.Tensor) or not matrix.is_cuda or matrix.dtype != torch.float32:
        raise TypeError("vbq_b200: the embedding must be a float32 CUDA tensor or a CompressedEmbedding")
    if matrix.dim() < 1 or math.prod(matrix.shape[1:]) < 1:
        raise ValueError("vbq_b200: the embedding must be (V, *tail) with at least one coordinate per row, got %s"
                         % (tuple(matrix.shape),))
    return matrix.reshape(matrix.shape[0], -1).contiguous()


def ranks(matrix, queries, targets, metric="dot", exclude=None):
    """Exact rank of each query's target among the rows of a dense embedding: int64 (B,) tensor, 1 = the best row.

    matrix: a (V, *tail) float32 CUDA tensor (`compress_coordinates` or `decompress_from_bytes` output, or any
    matrix).  queries and metric as for `CompressedEmbedding.scores` (values must be finite).  targets: (B,) integer
    ids in [0, V) on any device.  exclude: an optional (B, E) integer array as for `CompressedEmbedding.topk` (-1 pads,
    duplicates count once); a target in its own exclude row is a ValueError.

    Scores follow the numerics contract of include/vbq_b200.h and rows are ordered as `topk` orders them (score key
    descending, then id ascending), so rank_i = 1 + the number of rows not excluded that beat t_i, and rank_i <= k
    exactly when `topk(q_i, k, exclude=exclude_i)` returns t_i, at position rank_i.  The count runs in the
    vbq_score_ranks kernel without writing a score; excluded rows are subtracted afterwards from their scores
    (vbq_pair_scores).  A non-empty call makes one host synchronisation (the argument checks)."""
    Z = _dense_rows(matrix)
    V = Z.shape[0]
    q, t, ex = _rank_inputs(queries, targets, metric, exclude, tuple(matrix.shape[1:]), V, Z.device)
    B = q.shape[0]
    if B == 0:
        return torch.empty(0, dtype=torch.int64, device=Z.device)
    ar = torch.arange(B, device=Z.device)
    thr = ops.pair_scores(Z, q, t, ar, metric)
    counts = torch.ones(B, dtype=torch.int64, device=Z.device)
    if ex.shape[1]:
        srt, valid = _distinct_excluded(ex)
        s = ops.pair_scores(Z, q, srt.clamp_min(0).reshape(-1), ar[:, None].expand_as(srt).reshape(-1), metric)
        counts -= _excluded_beaters(s.view(srt.shape), srt, valid, thr, t)
    return ops.score_ranks(Z, q, metric, thr, t, counts)


def analogy_ranks(embedding, questions, metric="cosine"):
    """Ranks of the answers of analogy questions a : b :: c : d (3CosAdd on the stored rows): int64 (B,) tensor.

    embedding: a dense (V, *tail) float32 CUDA tensor or a `CompressedEmbedding`.  questions: (B, 4) integer ids
    a, b, c, d (any device).  The query of a question is (z_b - z_a) + z_c in float32 with round-to-nearest, its target
    is d, and a, b and c are excluded (`ranks` / `CompressedEmbedding.ranks`), so a question whose d equals a, b or c
    is a ValueError.  Raises TypeError / ValueError for a bad questions array and IndexError for an id outside
    [0, V), before any launch."""
    compressed = isinstance(embedding, CompressedEmbedding)
    if compressed:
        V, tail, dev = embedding.shape[0], embedding.shape[1:], embedding.device
    else:
        Z = _dense_rows(embedding)
        V, tail, dev = Z.shape[0], tuple(embedding.shape[1:]), Z.device
    qs = _int_tensor(questions, "questions")
    if qs.dim() != 2 or qs.shape[1] != 4:
        raise ValueError("vbq_b200: questions must be (B, 4), got %s" % (tuple(qs.shape),))
    qs = qs.to(device=dev, dtype=torch.int64)
    B = qs.shape[0]
    if B:
        lo, hi = torch.stack([qs.min(), qs.max()]).tolist()
        if lo < 0 or hi >= V:
            raise IndexError("vbq_b200: question id %d outside [0, %d)" % (lo if lo < 0 else hi, V))
    abc = qs[:, :3].contiguous()
    rows = embedding.lookup(abc).reshape(B, 3, math.prod(tail)) if compressed else Z[abc]
    query = ((rows[:, 1] - rows[:, 0]) + rows[:, 2]).reshape((B,) + tuple(tail))
    if compressed:
        return embedding.ranks(query, qs[:, 3], metric, exclude=abc)
    return ranks(embedding, query, qs[:, 3], metric, exclude=abc)


def analogy_metrics(ranks):
    """The quality columns of the notebook's `test_beta` from analogy ranks: {"mrr": mean(1 / rank), "acc":
    mean(rank == 1), "hits10": mean(rank <= 10)} as float64.  ranks: a non-empty integer array (any device) of
    values >= 1."""
    r = (ranks.detach().cpu().numpy() if isinstance(ranks, torch.Tensor) else np.asarray(ranks)).reshape(-1)
    if r.size and r.dtype.kind not in "iu":
        raise TypeError("vbq_b200: ranks must be integers, got %s" % r.dtype)
    if r.size == 0 or r.min() < 1:
        raise ValueError("vbq_b200: ranks must be a non-empty array of values >= 1")
    r = r.astype(np.float64)
    return {"mrr": np.float64(np.mean(1.0 / r)), "acc": np.float64(np.mean(r == 1)),
            "hits10": np.float64(np.mean(r <= 10))}


class GaussianCodebook:
    """`codepoints` / `lengths` of the notebook (heap order, float64 / int64) plus the device tables."""

    def __init__(self, empirical_std, max_codepoint_length=10, device="cuda"):
        self.max_codepoint_length = int(max_codepoint_length)
        self.empirical_std = float(empirical_std)
        self.device = torch.device(device)
        N = self.max_codepoint_length
        # codepoint_xi = np.arange(0.5**(length+1), 1, 0.5**length), length-major (ipynb:383-388)
        xi = np.concatenate([np.arange(0.5 ** (n + 1), 1, 0.5 ** n) for n in range(N + 1)])
        xi_d = torch.from_numpy(xi).to(self.device).reshape(-1, 1)
        std_d = torch.tensor([self.empirical_std], dtype=torch.float64, device=self.device)
        pts = ops.gaussian_inverse_cdf(xi_d, None, std_d).reshape(-1)          # norm.ppf(xi, scale=std), float64
        self.codepoints = pts.cpu().numpy()
        self.lengths = np.concatenate([np.full(2 ** n, n, dtype=np.int64) for n in range(N + 1)])
        self._ascending = torch.sort(pts).values.to(torch.float32)                       # (Q,): z_hat of sorted index q
        self._table = pts.to(torch.float32).reshape(1, -1).repeat(_VC, 1).contiguous()   # (16, Q)
        self._packed = ops.pack_code_points(self._table, N)
        torch.cuda.current_stream(self._table.device).synchronize()
        ops.stable_packed(self._packed)

    def _level_lengths(self, bitlengths):
        N = self.max_codepoint_length
        bl = np.asarray(bitlengths)
        per_level = np.array([bl[2 ** n - 1] for n in range(N + 1)], dtype=np.float64)
        if not np.array_equal(np.repeat(per_level, [2 ** n for n in range(N + 1)]), bl.astype(np.float64)):
            raise NotImplementedError("bitlengths must be constant within a bit depth for the bracketing search")
        return per_level

    def quantize(self, means, stds, betas, bitlengths=None, outputs=ops.OUT_ZHAT, flags=0):
        """means, stds: float32 CUDA tensors of equal shape -> dict of (len(betas),) + means.shape tensors."""
        N = self.max_codepoint_length
        per_level = self._level_lengths(self.lengths if bitlengths is None else bitlengths).astype(np.float32)
        pen = np.stack([np.float32(b) * per_level for b in betas])[:, None, :]
        pen = ops.with_host_copy(pen, self.device)   # channel-independent: launch constants of the TMA kernel
        # the notebook's default lengths are the bit depths themselves: no length table, which lets vbq_quantize use
        # the certified-bisection kernels (raw code lengths); custom bitlengths go through the length-table path
        length = None
        if bitlengths is not None and not np.array_equal(per_level, np.arange(N + 1, dtype=np.float32)):
            length = torch.from_numpy(np.broadcast_to(per_level, (len(betas), 1, N + 1)).copy()).to(self.device)
        m = means.reshape(-1)
        s = stds.reshape(-1)
        n = m.numel()
        pad = (-n) % _VC
        if pad:
            m = torch.cat([m, m.new_zeros(pad)])
            s = torch.cat([s, s.new_ones(pad)])
        z, q, lv, b, _, tot = ops.quantize(m.reshape(-1, _VC).contiguous(), s.reshape(-1, _VC).contiguous(),
                                           self._table, self._packed, pen, length, None, N, outputs,
                                           ops.search_flags(betas, flags))
        L = len(betas)

        def unpad(t):
            return t.reshape(L, -1)[:, :n].reshape((L,) + tuple(means.shape)) if t.numel() else t

        return dict(zhat=unpad(z), qidx=unpad(q), level=unpad(lv), bits=unpad(b), totals=tot)

    def _sorted_index(self, heap, level):
        """Heap index h of depth d -> sorted index (2 i + 1) 2^(N-d) - 1 with i = h - (2^d - 1)."""
        i_in = heap - ((1 << level) - 1)
        return ((2 * i_in + 1) << (self.max_codepoint_length - level)) - 1

    def _add_counts(self, q, counts):
        """Add the symbols of q (int32 CUDA tensor) to counts (16, Q) int64: `vbq_symbol_histogram` over 16 virtual
        channels, the ragged tail (fewer than 16 symbols) by bincount."""
        N = self.max_codepoint_length
        q = q.reshape(-1)
        k = (q.numel() // _VC) * _VC
        if k:
            ops.symbol_histogram(q[:k].reshape(-1, _VC).contiguous(), N, counts)
        if k < q.numel():
            counts[0] += torch.bincount(q[k:].long(), minlength=counts.shape[1])

    def beta_sweep(self, means, stds, betas, exact=False, reduce_fn=None, max_chunk_symbols=1 << 29):
        """The rate side of the notebook's beta sweep (ipynb:464-473, :1102-1103: `test_beta` for every beta of
        `np.exp(np.linspace(np.log(0.01), np.log(100000), 50))`): compresses all coordinates with every beta and
        returns the `compressed_bitlength` = `empirical_entropy(compressed)` (ipynb:452-455) of each, as a float64
        array (the quality columns of `test_beta` come from `analogy_sweep`, which takes its rates from this method).

        The coordinates are walked ONCE for all betas (sweep kernel) in row chunks of at most ``max_chunk_symbols``
        (beta, coordinate) pairs; the symbols of a chunk are counted on the device (`vbq_symbol_histogram`) and only the
        (len(betas), Q) count table leaves the loop.  ``exact=True`` runs the notebook's float64 search once per beta
        instead.  ``reduce_fn`` (optional) all-reduces the int64 counts over row-sharded ranks
        (`vbq_b200.sharding.all_reduce_counts`) before the entropies are formed."""
        N, Q = self.max_codepoint_length, 2 ** (self.max_codepoint_length + 1) - 1
        m = (means if isinstance(means, torch.Tensor) else torch.as_tensor(np.asarray(means)))
        s = (stds if isinstance(stds, torch.Tensor) else torch.as_tensor(np.asarray(stds)))
        m = m.to(device=self.device, dtype=torch.float32).reshape(-1)
        s = s.to(device=self.device, dtype=torch.float32).reshape(-1)
        betas = [float(b) for b in betas]
        L, n = len(betas), m.numel()
        counts = torch.zeros((L, _VC, Q), dtype=torch.int64, device=self.device)
        if exact:
            cp = torch.from_numpy(self.codepoints).to(self.device)
            per_level = torch.from_numpy(self._level_lengths(self.lengths).astype(np.float64)).to(self.device)
            step = max(_VC, (max_chunk_symbols // _VC) * _VC)
            for i, beta in enumerate(betas):
                for a in range(0, n, step):
                    b = min(n, a + step)
                    _, heap, level = ops.compress_coordinates_f64(m[a:b], s[a:b], cp, per_level, beta, True,
                                                                  want_index=True, want_level=True)
                    self._add_counts(self._sorted_index(heap, level), counts[i])
        else:
            step = max(_VC, (max_chunk_symbols // max(L, 1) // _VC) * _VC)
            for a in range(0, n, step):
                b = min(n, a + step)
                q = self.quantize(m[a:b], s[a:b], betas, outputs=ops.OUT_QIDX)['qidx']        # (L, b - a)
                for i in range(L):
                    self._add_counts(q[i], counts[i])
        counts = counts.sum(dim=1)
        if reduce_fn is not None:
            counts = reduce_fn(counts)
        c = counts.double()
        total = c.sum(dim=1)
        plogp = torch.where(c > 0, c * torch.log2(c.clamp_min(1.0)), torch.zeros_like(c)).sum(dim=1)
        return (total * torch.log2(total) - plogp).cpu().numpy()

    def compress_coordinates(self, means, stds, beta, bitlengths=None, exact=True):
        """Notebook signature (ipynb:429-443): returns (optima shaped and typed like `means`, None).
        Minimises (c - mu)^2 + 2 beta sigma^2 len(c) over the code points.

        ``exact=True`` (default) runs the float64 kernel that reproduces the notebook's arithmetic bit for bit
        (float64 code points and losses; `(2*beta)*stds**2` in float32 unless `beta` is a NumPy float64 scalar, which
        NumPy >= 2 promotes to float64).  ``exact=False`` runs the float32 image-path kernel (lambda = beta), which
        is faster and differs only on near-ties."""
        is_np = not isinstance(means, torch.Tensor)
        m = torch.as_tensor(np.asarray(means)) if is_np else means
        s = torch.as_tensor(np.asarray(stds)) if is_np else stds
        m32 = m.to(device=self.device, dtype=torch.float32).contiguous()
        s32 = s.to(device=self.device, dtype=torch.float32).contiguous()
        if exact:
            per_level = self._level_lengths(self.lengths if bitlengths is None else bitlengths)
            out, _, _ = ops.compress_coordinates_f64(
                m32, s32, torch.from_numpy(self.codepoints).to(self.device),
                torch.from_numpy(per_level.astype(np.float64)).to(self.device), float(beta), _pen_f32(beta))
        else:
            out = self.quantize(m32, s32, [beta], bitlengths)['zhat'][0]
        if is_np:
            return out.cpu().numpy().astype(np.asarray(means).dtype), None
        return out.to(means.dtype), None

    def analogy_sweep(self, means, stds, betas, questions, metric="cosine", exact=True):
        """The notebook's `test_beta` loop (ipynb:464-473): for every beta, the analogy quality of the quantized
        embedding and its rate.  Returns a (len(betas), 4) float64 array with the columns mrr, acc, hits10, bits.

        means, stds: (V, *tail) posteriors (tensors or arrays).  questions: (B, 4) ids a, b, c, d as for
        `analogy_ranks`.  For each beta, z_hat = `compress_coordinates(means, stds, float(beta), exact=exact)` stays on
        the device (one at a time), `analogy_ranks(z_hat, questions, metric)` ranks the questions on it and
        `analogy_metrics` gives the first three columns.  The bits column is one `beta_sweep(means, stds, betas,
        exact=exact)` call, which takes every beta as a Python float too, so rate and quality come from the same
        quantization."""
        bits = self.beta_sweep(means, stds, betas, exact=exact)
        m = means if isinstance(means, torch.Tensor) else torch.as_tensor(np.asarray(means))
        s = stds if isinstance(stds, torch.Tensor) else torch.as_tensor(np.asarray(stds))
        m = m.to(device=self.device, dtype=torch.float32).contiguous()
        s = s.to(device=self.device, dtype=torch.float32).contiguous()
        out = np.empty((len(betas), 4), dtype=np.float64)
        for i, beta in enumerate(betas):
            zhat, _ = self.compress_coordinates(m, s, float(beta), exact=exact)
            met = analogy_metrics(analogy_ranks(zhat, questions, metric))
            del zhat
            out[i] = (met["mrr"], met["acc"], met["hits10"], bits[i])
        return out

    def compress_to_bytes(self, means, stds, betas, exact=True, prob_bits=coding.DEFAULT_PROB_BITS, seg_rows=None):
        """Entropy-code the coordinates that `compress_coordinates(means, stds, beta, exact=exact)` chooses, for every
        beta: returns {beta: bytes}, each a separately decodable VBQE blob (`serialize.read_embedding_header`) that
        `decompress_from_bytes` turns back into those optima as float32.

        The symbols (sorted quantile indices) are counted on the device, every beta gets one table that gives unused
        symbols frequency 0 (`coding.frequency_tables(counts, keep_zeros=True)`), and all betas are coded in one launch
        of the shared-table rANS coder.  ``seg_rows`` (rows of 32 coordinates per independently decodable segment)
        defaults per beta to `default_seg_rows`.  The coder holds N <= 10."""
        N = self.max_codepoint_length
        if N > 10:
            raise ValueError("vbq_b200: compress_to_bytes codes N <= 10, this codebook has N=%d" % N)
        m = means if isinstance(means, torch.Tensor) else torch.as_tensor(np.asarray(means))
        s = stds if isinstance(stds, torch.Tensor) else torch.as_tensor(np.asarray(stds))
        shape = tuple(m.shape)
        m32 = m.to(device=self.device, dtype=torch.float32).contiguous().reshape(-1)
        s32 = s.to(device=self.device, dtype=torch.float32).contiguous().reshape(-1)
        n = m32.numel()
        Q = ops.num_levels(N)
        if exact:
            cp = torch.from_numpy(self.codepoints).to(self.device)
            per_level = torch.from_numpy(self._level_lengths(self.lengths).astype(np.float64)).to(self.device)
        planes = torch.empty((len(betas), n), dtype=torch.int32, device=self.device)
        counts = torch.zeros((len(betas), _VC, Q), dtype=torch.int64, device=self.device)
        for i, beta in enumerate(betas):
            if exact:
                _, heap, level = ops.compress_coordinates_f64(m32, s32, cp, per_level, float(beta), _pen_f32(beta),
                                                              want_index=True, want_level=True)
                planes[i] = self._sorted_index(heap, level)
            else:
                planes[i] = self.quantize(m32, s32, [beta], outputs=ops.OUT_QIDX)['qidx'][0]
            self._add_counts(planes[i], counts[i])
        counts = counts.sum(dim=1).cpu().numpy()
        tables = np.stack([coding.frequency_tables(c, prob_bits, keep_zeros=True)[0] for c in counts])
        if seg_rows is None:
            seg = [default_seg_rows(n, h) for h in _entropy_of_counts(counts)]
        else:
            seg = [int(seg_rows)] * len(betas)
        blobs = serialize.encode_embeddings(planes, tables, N, shape, seg, self.empirical_std,
                                            [float(b) for b in betas], coding.code_points_fingerprint(self.codepoints))
        return dict(zip(betas, blobs))

    def decompress_from_bytes(self, blob):
        """The float32 optima of a `compress_to_bytes` blob as a device tensor of the original shape.  Raises
        ValueError if the blob was made with another N, empirical_std or code points, or is malformed or corrupt.  A
        receiver that has only the blob builds the codebook from it:
        ``h = serialize.read_embedding_header(blob); GaussianCodebook(h["empirical_std"], h["max_bits"])``."""
        h = serialize.read_embedding_header(blob)
        if (h["max_bits"] != self.max_codepoint_length or h["empirical_std"] != self.empirical_std
                or h["fingerprint"] != coding.code_points_fingerprint(self.codepoints)):
            raise ValueError("vbq_b200: the blob was coded with another codebook (N=%d, empirical_std=%r) than this "
                             "one (N=%d, empirical_std=%r) or with other code points"
                             % (h["max_bits"], h["empirical_std"], self.max_codepoint_length, self.empirical_std))
        out = serialize.decode_embedding(blob, self._ascending, self.device, want_qidx=False)
        return out["zhat"].reshape(h["shape"])


_CHECKPOINT_BYTES = 4 + 32 * 4          # one index entry: the word offset and 32 lane states
_INDEX_SHARE = 8                        # default K: the index takes at most 1/8 of the payload bytes
_MIN_CHECKPOINT_ROWS = 32


def default_checkpoint_rows(n: int, seg_rows: int, payload_bytes: int) -> int:
    """Checkpoint interval of `CompressedEmbedding` for a plane of n symbols in segments of seg_rows rows: the smallest
    number of coder rows (rows of 32 symbols), at least 32, for which the checkpoint index (132 bytes per checkpoint)
    takes at most 1/8 of the payload bytes.  The checkpoint count only falls as the interval grows, and an interval of
    a whole segment has none, so a bisection finds it."""
    seg = serialize.shared_seg_rows(n, seg_rows)
    lo, hi = _MIN_CHECKPOINT_ROWS, max(_MIN_CHECKPOINT_ROWS, seg)
    while lo < hi:
        mid = (lo + hi) // 2
        if _INDEX_SHARE * _CHECKPOINT_BYTES * ops.rans_shared_checkpoint_count(n, seg, mid) <= payload_bytes:
            hi = mid
        else:
            lo = mid + 1
    return lo


class CompressedEmbedding:
    """Row access into a `GaussianCodebook.compress_to_bytes` blob without decoding all of it.

    The payload, its frequency table and the ascending code points stay on the device, together with a checkpoint
    index: every ``checkpoint_rows`` coder rows (rows of 32 coordinates) of each segment, the decoder's word position
    and 32 lane states (132 bytes, include/vbq_b200.h).  A lookup starts each needed piece of the stream at the
    checkpoint before it, so its cost is about ``checkpoint_rows`` decoded rows per touched interval instead of the
    whole matrix.  The blob and its rate are unchanged; a smaller ``checkpoint_rows`` trades device memory for latency.

    ``CompressedEmbedding(blob, device="cuda", checkpoint_rows=None)`` parses the blob (every `ValueError` of
    `serialize.read_embedding_header` comes before anything is uploaded), rebuilds the codebook from its header, checks
    the code-point fingerprint and runs one full decode pass that builds the index and applies the coder's integrity
    check, so a corrupt payload raises `ValueError` here.  ``checkpoint_rows`` defaults to `default_checkpoint_rows`;
    a value of at least the segment length means no checkpoints.  Not an `nn.Module`; no gradients."""

    def __init__(self, blob, device="cuda", checkpoint_rows=None):
        h = serialize.read_embedding_header(blob)
        if len(h["shape"]) < 1:
            raise ValueError("vbq_b200: a 0-d VBQE blob has no rows to look up")
        if checkpoint_rows is not None and (isinstance(checkpoint_rows, bool) or int(checkpoint_rows) != checkpoint_rows
                                            or checkpoint_rows < 1):
            raise ValueError("vbq_b200: checkpoint_rows must be an integer >= 1, got %r" % (checkpoint_rows,))
        self.device = torch.device(device)
        self._shape = tuple(int(d) for d in h["shape"])
        self._beta = h["beta"]
        self._n = math.prod(self._shape)
        self._D = math.prod(self._shape[1:])
        self._seg = serialize.shared_seg_rows(self._n, h["seg_rows"])
        self._N, self._P = h["max_bits"], h["prob_bits"]
        payload_bytes = 2 * h["words"].size
        K = default_checkpoint_rows(self._n, self._seg, payload_bytes) if checkpoint_rows is None else int(checkpoint_rows)
        self._K = K
        self._k = min(K, self._seg)                  # what the kernels use: an interval never spans two segments
        cb = GaussianCodebook(h["empirical_std"], self._N, device=self.device)
        if coding.code_points_fingerprint(cb.codepoints) != h["fingerprint"]:
            raise ValueError("vbq_b200: the blob's code-point fingerprint does not match the codebook rebuilt from its "
                             "header (N=%d, empirical_std=%r)" % (self._N, h["empirical_std"]))
        self._code_points = cb._ascending
        self._words = torch.from_numpy(h["words"].view(np.int16).copy()).to(self.device)
        self._bounds = torch.from_numpy(np.ascontiguousarray(h["bounds"], dtype=np.int64)).to(self.device)
        self._cum = torch.from_numpy(coding.cum_table_shared(h["table"][None]).view(np.int32)).to(self.device)
        self._offsets, self._states, status = ops.rans_shared_checkpoints(
            self._words, self._bounds, self._cum, self._n, self._seg, self._N, self._P, self._k)
        st = int(status.item())
        if st:
            raise ValueError("vbq_b200: corrupt VBQE payload (decoder status %d: %s)" % (
                st, ", ".join(m for bit, m in ((1, "a group ran out of words"), (2, "integrity check failed"),
                                                (4, "bad group range or initial state")) if st & bit)))

    @property
    def shape(self):
        return self._shape

    @property
    def beta(self):
        return self._beta

    @property
    def checkpoint_rows(self):
        return self._K

    @property
    def nbytes(self):
        """Device bytes held: payload, checkpoint index, group ranges, cum table and code points."""
        return sum(t.numel() * t.element_size() for t in (self._words, self._offsets, self._states, self._bounds,
                                                          self._cum, self._code_points))

    def _ids(self, ids):
        """ids -> flat int64 tensor and its shape; TypeError / IndexError before anything runs on the device for
        host ids (device ids are range-checked with the work list's size)."""
        t = _int_tensor(ids, "ids")
        flat = t.reshape(-1)
        if not flat.is_cuda and flat.numel():
            lo, hi = int(flat.min()), int(flat.max())
            if lo < 0 or hi >= self._shape[0]:
                raise IndexError("vbq_b200: id %d outside [0, %d)" % (lo if lo < 0 else hi, self._shape[0]))
        return flat.to(device=self.device, dtype=torch.int64), tuple(t.shape)

    def _work_list(self, u, flat=None):
        """Sorted unique rows u -> (items (n_items, 5) int64, whether the requested ids `flat` already equal u), built
        on the device; one host synchronisation reads the id range, the list's size and that flag together."""
        D, S, K = self._D, self._seg, self._k
        C1 = (S - 1) // K + 1                        # interval slots per segment: interval I = segment C1 + j
        coder_rows = -(-self._n // 32)
        rf, rl = (u * D) // 32, (u * D + D - 1) // 32
        a = (rf // S) * C1 + (rf % S) // K
        b = (rl // S) * C1 + (rl % S) // K
        cnt = b - a + 1
        n_u = u.numel()
        total = cnt.sum()
        same = (u == flat).all() if flat is not None and flat.numel() == n_u else torch.zeros((), dtype=torch.bool,
                                                                                              device=u.device)
        lo_id, hi_id, n_pairs, n_items, same = torch.stack(
            [u[0], u[-1], total, total - (a[1:] == b[:-1]).sum(), same.to(torch.int64)]).tolist()
        if lo_id < 0 or hi_id >= self._shape[0]:
            raise IndexError("vbq_b200: id %d outside [0, %d)" % (lo_id if lo_id < 0 else hi_id, self._shape[0]))
        # one (row, interval) pair per interval a row touches; rows are sorted, so intervals are too
        row = torch.repeat_interleave(torch.arange(n_u, device=u.device), cnt, output_size=n_pairs)
        first = torch.cumsum(cnt, 0) - cnt
        I = a[row] + torch.arange(n_pairs, device=u.device) - first[row]
        new = torch.ones(n_pairs, dtype=torch.bool, device=u.device)
        new[1:] = I[1:] != I[:-1]
        item = torch.cumsum(new, 0) - 1
        seg, j = I // C1, I % C1
        r_end = torch.clamp(torch.minimum(seg * S + j * K + K, seg * S + S), max=coder_rows)
        last = torch.minimum(rl[row], r_end - 1)

        def reduce(v, how):
            return torch.zeros(n_items, dtype=torch.int64, device=u.device).scatter_reduce(0, item, v, how,
                                                                                            include_self=False)
        items = torch.stack([reduce(seg, "amax"), reduce(j, "amax"), reduce(last, "amax"), reduce(row, "amin"),
                             reduce(row, "amax") + 1], dim=1).contiguous()
        return items, bool(same)

    def lookup(self, ids):
        """float32 z_hat of the embedding rows `ids`: shape ids.shape + shape[1:], bit-identical to
        ``GaussianCodebook.decompress_from_bytes(blob)[ids]``.  ids: an integer tensor (any device), array or list, in
        any order and with duplicates.  Raises TypeError for non-integer ids and IndexError for an id outside
        [0, shape[0]) before the gather runs.  The work list (unique sorted rows, the checkpoint interval of every
        piece of each row, per-item slices) is built on the device with torch ops.  Sorted unique ids are gathered
        straight into the result; other ids are gathered once per distinct row and then indexed.

        A non-empty call makes three host synchronisations: one inside `torch.unique` (it sizes its output), one that
        reads the id range and the work list's size together, and one that reads the gather's status."""
        flat, shape = self._ids(ids)
        out_shape = shape + self._shape[1:]
        if flat.numel() == 0:
            return torch.empty(out_shape, dtype=torch.float32, device=self.device)
        u, inv = torch.unique(flat, sorted=True, return_inverse=True)
        items, sorted_unique = self._work_list(u, flat)
        _, z, status = ops.rans_shared_decode_rows(self._words, self._bounds, self._cum, self._n, self._seg, self._N,
                                                   self._P, self._k, self._offsets, self._states, items, u, self._D,
                                                   self._code_points)
        st = int(status.item())
        if st:
            raise RuntimeError("vbq_b200: row gather failed (status %d)" % st)
        if sorted_unique:                            # the gather wrote the answer in place
            return z.reshape(out_shape)
        return z[inv].reshape(out_shape)

    __call__ = lookup

    # -- scoring queries against every row -------------------------------------------------------------------------
    TOPK_WORKSPACE_BYTES = 256 << 20    # topk's row-block workspace; the block shrinks as the batch grows
    _TOPK_CELL_BYTES = 48               # device bytes per (query, block row) cell: scores, keys, values, temporaries

    def _queries(self, queries, metric):
        """queries -> (B, D) on their own device; TypeError / ValueError before anything reaches this device."""
        t = _query_matrix(queries, metric, self._shape[1:])
        if ops.rans_shared_score_max_queries(self._D) < 1:
            raise ValueError("vbq_b200: a query of %d coordinates does not fit the scoring kernel's shared memory"
                             % self._D)
        return t

    def _upload(self, q):
        return q.to(device=self.device, dtype=torch.float32).contiguous()

    def _scores_into(self, q, start, stop, metric, out, status):
        """Scores of q (B, D) against rows [start, stop) into out (B, stop - start), one launch per query tile; the
        launches' status bits are ORed into `status` on the device."""
        tile = ops.rans_shared_score_max_queries(self._D)
        for b0 in range(0, q.shape[0], tile):
            b1 = min(b0 + tile, q.shape[0])
            _, st = ops.rans_shared_row_scores(self._words, self._bounds, self._cum, self._n, self._seg, self._N,
                                               self._P, self._k, self._offsets, self._states, self._D, start, stop,
                                               q[b0:b1], self._code_points, metric, out=out[b0:b1])
            status.bitwise_or_(st)

    def _check_status(self, status):
        st = int(status.item())
        if st:
            raise RuntimeError("vbq_b200: scoring decode failed (status %d)" % st)

    def scores(self, queries, start=0, stop=None, metric="dot"):
        """float32 scores (B, stop - start) of every query against the embedding rows [start, stop), computed while
        the rows are decoded from the blob; the dense matrix is never built.

        queries: (B, *shape[1:]) or shape[1:] (one query, B = 1); a float tensor on any device, an array or a list of
        floats; values are cast to float32.  metric: "dot" or "cosine".  Each score is the float32 value of the numerics
        contract of include/vbq_b200.h (four accumulators stepped in coordinate order, fmaf with round-to-nearest; a
        cosine with a zero norm is 0), so it is bit-reproducible and independent of the range, the batch and
        checkpoint_rows.  Batches above ``ops.rans_shared_score_max_queries(D)`` queries run as several launches.

        Raises TypeError for non-float queries, ValueError for a wrong trailing shape, an unknown metric or a
        non-finite query, and IndexError unless 0 <= start <= stop <= shape[0].  A call makes two host
        synchronisations: the finiteness check and the status read."""
        V = self._shape[0]
        stop = V if stop is None else stop
        if (isinstance(start, bool) or isinstance(stop, bool) or int(start) != start or int(stop) != stop
                or not 0 <= int(start) <= int(stop) <= V):
            raise IndexError("vbq_b200: row range [%r, %r) outside [0, %d]" % (start, stop, V))
        start, stop = int(start), int(stop)
        q = self._upload(self._queries(queries, metric))
        if not bool(torch.isfinite(q).all()):
            raise ValueError("vbq_b200: queries must be finite")
        out = torch.empty((q.shape[0], stop - start), dtype=torch.float32, device=self.device)
        status = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._scores_into(q, start, stop, metric, out, status)
        self._check_status(status)
        return out

    def topk(self, queries, k, metric="dot", exclude=None):
        """The k best rows of every query: (values (B, k) float32, ids (B, k) int64), ordered by score descending and
        then by id ascending, so ties between equal rows resolve the same way on every run.  values are the `scores` of
        the returned ids, bit for bit.

        queries and metric as for `scores`.  exclude: an optional (B, E) integer array (any device) of rows that query b
        must skip, -1 for padding (for an analogy query, the three words of the question).  1 <= k <= shape[0] minus the
        most distinct rows any query excludes.

        The plane is scanned in blocks of R rows.  A block's scores become int64 keys: the order-preserving map of the
        float32 bits (-0.0 as +0.0, NaN lowest) in the high half and 0xFFFFFFFF - id in the low half, excluded rows get
        the minimum, and `torch.topk` over the block's keys and the running top k is an exact, tie-free selection.  R is
        chosen so that the block's scores, keys and temporaries take at most TOPK_WORKSPACE_BYTES (256 MiB) whatever
        shape[0] is; besides that the call holds a few (B, k) arrays.  A call makes two host synchronisations: one reads
        the finiteness and exclude checks together, one reads the decode status."""
        q = self._queries(queries, metric)
        V = self._shape[0]
        B = q.shape[0]
        if isinstance(k, bool) or int(k) != k:
            raise ValueError("vbq_b200: k must be an integer, got %r" % (k,))
        k = int(k)
        dev = self.device
        if not 1 <= k <= V:
            raise ValueError("vbq_b200: k=%d outside [1, %d]" % (k, V))
        if exclude is None:
            ex = torch.full((B, 0), -1, dtype=torch.int64, device=dev)
        else:
            ex = exclude if isinstance(exclude, torch.Tensor) else torch.from_numpy(np.asarray(exclude))
            if ex.dtype.is_floating_point or ex.dtype.is_complex or ex.dtype == torch.bool:
                raise TypeError("vbq_b200: exclude must be integers, got %s" % ex.dtype)
            if ex.dim() != 2 or ex.shape[0] != B:
                raise ValueError("vbq_b200: exclude must be (%d, E), got %s" % (B, tuple(ex.shape)))
            ex = ex.to(device=dev, dtype=torch.int64).contiguous()
        q = self._upload(q)
        checks = [torch.isfinite(q).all().to(torch.int64)]
        if ex.shape[1]:
            srt = ex.sort(dim=1).values
            new = torch.ones_like(srt, dtype=torch.bool)
            new[:, 1:] = srt[:, 1:] != srt[:, :-1]
            checks += [srt[:, 0].min(), srt[:, -1].max(), ((srt >= 0) & new).sum(dim=1).max()]
        got = torch.stack(checks).tolist()
        if not got[0]:
            raise ValueError("vbq_b200: queries must be finite")
        n_ex = 0
        if ex.shape[1]:
            if got[1] < -1 or got[2] >= V:
                raise IndexError("vbq_b200: exclude id %d outside [-1, %d)" % (got[1] if got[1] < -1 else got[2], V))
            n_ex = got[3]
        if not 1 <= k <= V - n_ex:
            raise ValueError("vbq_b200: k=%d outside [1, %d]" % (k, V - n_ex))

        R = max(1, min(V, self.TOPK_WORKSPACE_BYTES // (self._TOPK_CELL_BYTES * B)))
        buf = torch.empty(B * R, dtype=torch.float32, device=dev)
        keys = torch.full((B, k + R + 1), torch.iinfo(torch.int64).min, dtype=torch.int64, device=dev)   # last: scratch
        vals = torch.zeros((B, k + R), dtype=torch.float32, device=dev)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        brow = torch.arange(B, device=dev)[:, None].expand_as(ex)
        low = 0xFFFFFFFF - torch.arange(R, dtype=torch.int64, device=dev)
        for start in range(0, V, R):
            Rb = min(R, V - start)
            s = buf[:B * Rb].view(B, Rb)
            self._scores_into(q, start, start + Rb, metric, s, status)
            vals[:, k:k + Rb] = s
            bits = s.view(torch.int32)
            hi = torch.where(bits < 0, bits ^ 0x7FFFFFFF, bits)              # order-preserving on the float's bits
            hi.masked_fill_(s == 0, 0)                                       # -0.0 ties with +0.0
            hi.masked_fill_(torch.isnan(s), -(1 << 31))                      # NaN (after an overflow) is lowest
            kb = keys[:, k:k + Rb]
            kb.copy_(hi)
            kb.bitwise_left_shift_(32).bitwise_or_(low[:Rb] - start)
            if ex.shape[1]:
                inb = (ex >= start) & (ex < start + Rb)
                keys.index_put_((brow, torch.where(inb, ex - start + k, k + R)),
                                torch.tensor(torch.iinfo(torch.int64).min, device=dev))
            tk, ti = torch.topk(keys[:, :k + Rb], k, dim=1)
            tv = vals.gather(1, ti)
            keys[:, :k] = tk
            vals[:, :k] = tv
        self._check_status(status)
        ids = 0xFFFFFFFF - (keys[:, :k] & 0xFFFFFFFF)
        return vals[:, :k].clone(), ids

    # -- exact target ranks ----------------------------------------------------------------------------------------
    RANKS_WORKSPACE_BYTES = 256 << 20   # ranks' decoded row block (and its work list)
    _RANKS_ROW_EXTRA_BYTES = 128        # device bytes per block row besides its D floats: the work list's temporaries

    def ranks(self, queries, targets, metric="dot", exclude=None):
        """Exact rank of each query's target among the rows of this embedding: int64 (B,) tensor, equal to
        `vbq_b200.ranks(decompress_from_bytes(blob), queries, targets, metric, exclude)` (arguments as there; queries as
        for `scores`).

        The target rows and the excluded rows are read with `lookup` and scored with vbq_pair_scores.  Then the plane
        is decoded in blocks of R consecutive rows, each block straight into one buffer by the row gather, and
        vbq_score_ranks adds each block's counts; R is chosen so that a block takes at most RANKS_WORKSPACE_BYTES
        (256 MiB) whatever shape[0] is, so the dense matrix is never whole.  The counts are integers, so the result does
        not depend on R.  A non-empty call makes 5 + (number of blocks) host synchronisations: the argument checks,
        three in `lookup`, one per block for its work list and one for the decode status."""
        V = self._shape[0]
        q, t, ex = _rank_inputs(queries, targets, metric, exclude, self._shape[1:], V, self.device)
        B, D, dev = q.shape[0], self._D, self.device
        if B == 0:
            return torch.empty(0, dtype=torch.int64, device=dev)
        ar = torch.arange(B, device=dev)
        srt, valid = _distinct_excluded(ex)
        E = srt.shape[1]
        rows = self.lookup(torch.cat([t, srt.clamp_min(0).reshape(-1)])).reshape(B + B * E, D)
        thr = ops.pair_scores(rows, q, ar, ar, metric)
        counts = torch.ones(B, dtype=torch.int64, device=dev)
        if E:
            s = ops.pair_scores(rows, q, B + torch.arange(B * E, device=dev), ar[:, None].expand(B, E).reshape(-1),
                                metric)
            counts -= _excluded_beaters(s.view(B, E), srt, valid, thr, t)
        del rows
        R = max(1, min(V, self.RANKS_WORKSPACE_BYTES // (4 * D + self._RANKS_ROW_EXTRA_BYTES)))
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        for start in range(0, V, R):
            u = torch.arange(start, min(V, start + R), device=dev)
            items, _ = self._work_list(u)
            _, z, st = ops.rans_shared_decode_rows(self._words, self._bounds, self._cum, self._n, self._seg, self._N,
                                                   self._P, self._k, self._offsets, self._states, items, u, D,
                                                   self._code_points)
            status.bitwise_or_(st)
            ops.score_ranks(z, q, metric, thr, t, counts, row_offset=start)
            del z, items, u
        st = int(status.item())
        if st:
            raise RuntimeError("vbq_b200: row gather failed (status %d)" % st)
        return counts
