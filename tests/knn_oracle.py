"""TEST INFRASTRUCTURE ONLY.  Float64 numpy restatement of ``jamie_b200.evaluation.kneighbors`` / ``knn_impute`` (which
run on the GPU through jb_knn and jb_knn_average): sklearn's brute-force ``NearestNeighbors.kneighbors`` and
``KNeighborsRegressor.predict`` with euclidean distances.

Rows are rounded to float32 first. Squared distances are sums of squared float64 differences over the columns in order
(no ``|a|^2 + |b|^2 - 2 a.b`` cancellation); each query's neighbours are the first k of a stable argsort, so equal
distances go to the lowest reference index. 'distance' weights follow sklearn: 1 / d, and a row with a zero distance
weighs its zero-distance neighbours 1 and the others 0. Averages sum the weighted values in list order, then divide.
"""
import numpy as np

PAIRS = 1 << 22   # query rows x reference rows per chunk of the distance matrix


def sq_dists(query, reference):
    """[nq, nr] float64 squared distances of float32-rounded rows."""
    q = np.asarray(query, np.float32).astype(np.float64)
    r = np.asarray(reference, np.float32).astype(np.float64)
    D = np.zeros((q.shape[0], r.shape[0]))
    for c in range(q.shape[1]):
        D += (q[:, None, c] - r[None, :, c]) ** 2
    return D


def kneighbors(query, reference, k):
    """(dist float64 [nq, k], idx int64 [nq, k]) in ascending (distance, index) order."""
    nq, nr = np.shape(query)[0], np.shape(reference)[0]
    rows = max(1, PAIRS // nr)
    dist, idx = np.empty((nq, k)), np.empty((nq, k), np.int64)
    for q0 in range(0, nq, rows):
        D = sq_dists(query[q0:q0 + rows], reference)
        o = np.argsort(D, axis=1, kind='stable')[:, :k]
        idx[q0:q0 + rows] = o
        dist[q0:q0 + rows] = np.sqrt(np.take_along_axis(D, o, axis=1))
    return dist, idx


def weights_of(dist, weights):
    """sklearn's neighbour weights: all ones for 'uniform'; 1 / d, or the zero-distance rule, for 'distance'."""
    if weights == 'uniform':
        return np.ones_like(dist)
    w = np.empty_like(dist)
    for i, d in enumerate(dist):
        w[i] = (d == 0).astype(np.float64) if (d == 0).any() else 1.0 / d
    return w


def average(idx, w, values):
    """out[q] = sum_t w[q, t] values[idx[q, t]] / sum_t w[q, t], summed in list order."""
    V = np.asarray(values, np.float64)
    num = np.zeros((idx.shape[0], V.shape[1]))
    den = np.zeros(idx.shape[0])
    for t in range(idx.shape[1]):
        num += w[:, t, None] * V[idx[:, t]]
        den += w[:, t]
    return num / den[:, None]


def knn_impute(query, reference, values, k, weights='uniform'):
    dist, idx = kneighbors(query, reference, k)
    return average(idx, weights_of(dist, weights), values)
