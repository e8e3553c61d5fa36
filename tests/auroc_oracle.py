"""TEST INFRASTRUCTURE ONLY.  Float64 numpy restatement of ``jamie_b200.evaluation.imputation_auroc`` (which computes it on
the GPU through jb_metric_feature_auroc): the reference's AUROC panel (jamie/evaluation.py:468-490), sklearn
``roc_auc_score(measured[:, j] > threshold, float32(imputed[:, j]))``, as the Mann-Whitney statistic in integers.

Rows are grouped by equal score in ascending order (-0.0 and +0.0 are one score); for group g with pos_g positives, neg_g
negatives and negbefore_g negatives in all lower groups, 2U = sum_g pos_g (2 negbefore_g + neg_g), and
AUROC = 2U / (2 P N), nan when P = 0 or N = 0 (where sklearn raises).
"""
import numpy as np


def u2_of(scores, labels):
    """2U of one column: float32-representable scores [n], boolean labels [n] (an int, exact)."""
    s = np.asarray(scores, np.float64) + 0.0          # -0.0 + 0.0 = +0.0
    y = np.asarray(labels, bool)
    _, g = np.unique(s, return_inverse=True)          # group index in ascending score order
    G = int(g.max()) + 1 if g.size else 0
    pos = np.bincount(g[y], minlength=G).astype(np.int64)
    neg = np.bincount(g[~y], minlength=G).astype(np.int64)
    negbefore = np.cumsum(neg) - neg
    return int((pos * (2 * negbefore + neg)).sum())


def finish(u2, n_pos, n):
    """AUROC = 2U / (2 P N) per column as one correctly rounded division (Python ints); nan for one class."""
    return np.array([u / (2 * p * (n - p)) if 0 < p < n else np.nan for u, p in zip(np.asarray(u2).tolist(),
                                                                                   np.asarray(n_pos).tolist())])


def imputation_auroc(imputed, measured, threshold=0.0):
    """(u2 uint64 [d], n_pos int64 [d], auroc float64 [d]) of dense [n, d] imputed and measured."""
    s = np.asarray(imputed).astype(np.float32)
    lab = np.asarray(measured) > threshold
    n, d = s.shape
    u2 = np.array([u2_of(s[:, j], lab[:, j]) for j in range(d)], np.uint64)
    n_pos = lab.sum(axis=0).astype(np.int64)
    return u2, n_pos, finish(u2, n_pos, n)
