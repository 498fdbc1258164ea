"""Plain NumPy restatement of exact target ranks (include/vbq_b200.h, vbq_score_ranks / vbq_pair_scores,
vbq_b200.ranks, CompressedEmbedding.ranks, analogy_ranks / analogy_metrics): scores under the numerics contract of
embedding_scores_reference, the order of CompressedEmbedding.topk, and the analogy query."""
import numpy as np

import embedding_scores_reference as S


def keys(s):
    """int64 keys of float32 scores: the order-preserving map of the bits, -0.0 as +0.0, NaN lowest."""
    s = np.asarray(s, np.float32)
    b = s.view(np.int32).astype(np.int64)
    k = np.where(b < 0, b ^ 0x7FFFFFFF, b)
    k = np.where(s == 0, 0, k)
    return np.where(np.isnan(s), -(1 << 31), k)


def ranks(Z, Q, targets, metric="dot", exclude=None):
    """(B,) int64: 1 + #{j not excluded : key(s_ij) > key(s_it), or equal keys and j < t_i}."""
    sc = S.scores(Z, Q, metric)
    B, V = sc.shape
    t = np.asarray(targets, np.int64)
    k = keys(sc)
    kt = k[np.arange(B), t][:, None]
    ids = np.arange(V)[None, :]
    beats = (k > kt) | ((k == kt) & (ids < t[:, None]))
    if exclude is not None:
        for b in range(B):
            e = np.unique(np.asarray(exclude[b])[np.asarray(exclude[b]) >= 0])
            assert t[b] not in e
            beats[b, e] = False
    return 1 + beats.sum(axis=1).astype(np.int64)


def analogy_queries(Z, questions):
    """(z_b - z_a) + z_c in float32 for questions (B, 4) a, b, c, d."""
    Z = np.asarray(Z, np.float32).reshape(np.shape(Z)[0], -1)
    qs = np.asarray(questions, np.int64)
    return (Z[qs[:, 1]] - Z[qs[:, 0]]) + Z[qs[:, 2]]


def analogy_ranks(Z, questions, metric="cosine"):
    qs = np.asarray(questions, np.int64)
    return ranks(Z, analogy_queries(Z, qs), qs[:, 3], metric, exclude=qs[:, :3])


def metrics(r):
    r = np.asarray(r, np.float64)
    return {"mrr": np.mean(1.0 / r), "acc": np.mean(r == 1), "hits10": np.mean(r <= 10)}
