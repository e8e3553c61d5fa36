"""TEST INFRASTRUCTURE ONLY.  Float64 numpy restatement of ``jamie_b200.evaluation.silhouette_samples`` (which runs its
pair work on the GPU through jb_silhouette): sklearn's ``silhouette_samples`` with euclidean distances.

Rows are rounded to float32 first. Distances are the sqrt of sums of squared float64 differences over the columns (no
``|a|^2 + |b|^2 - 2 a.b`` cancellation). Per row, the distances to every row are summed per label with ``np.bincount``;
``sums`` returns sklearn's ``_silhouette_reduce`` pair (intra, inter) and ``finish`` is sklearn's own arithmetic after it.
"""
import numpy as np


def encode(labels):
    """sklearn's LabelEncoder: (codes int64 [n], label frequencies)."""
    _, codes = np.unique(np.asarray(labels), return_inverse=True)
    codes = codes.ravel()
    return codes, np.bincount(codes)


def sums(x, codes, rows=None):
    """(intra, inter) float64 [n] (or of the given rows only): the sum of the distances to the row's own label, and the
    least mean distance to another label."""
    X = np.asarray(x, np.float32).astype(np.float64)
    freq = np.bincount(codes)
    rows = np.arange(X.shape[0]) if rows is None else np.asarray(rows)
    intra, inter = np.empty(len(rows)), np.empty(len(rows))
    for r, i in enumerate(rows):
        S = np.bincount(codes, weights=np.sqrt(((X[i] - X) ** 2).sum(1)), minlength=len(freq))
        intra[r] = S[codes[i]]
        S[codes[i]] = np.inf
        inter[r] = (S / freq).min()
    return intra, inter


def finish(intra, inter, codes, freq):
    """sklearn's silhouette_samples after _silhouette_reduce, in its order."""
    intra = intra / (freq - 1).take(codes, mode='clip')   # a singleton label divides 0 by 0: nan, then 0
    with np.errstate(divide='ignore', invalid='ignore'):
        s = (inter - intra) / np.maximum(intra, inter)
    return np.nan_to_num(s)


def silhouette_samples(x, labels):
    codes, freq = encode(labels)
    with np.errstate(divide='ignore', invalid='ignore'):
        return finish(*sums(x, codes), codes, freq)
