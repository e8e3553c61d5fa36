"""CPU tests of kneighbors / knn_impute: the float64 reference (tests/knn_oracle.py) against sklearn's brute-force
NearestNeighbors and KNeighborsRegressor, and the host driver (jamie_b200/evaluation.py: batches, sparse values, the
zero-distance rule, refusals) with a numpy stand-in for jb_knn and jb_knn_average."""
import numpy as np
import pytest
import scipy.sparse as sp
from sklearn.neighbors import KNeighborsRegressor, NearestNeighbors

from jamie_b200 import evaluation
from tests import knn_oracle as K


def _data(nq, nr, L, d, seed):
    rng = np.random.default_rng(seed)
    q = rng.standard_normal((nq, L)).astype(np.float32)
    r = rng.standard_normal((nr, L)).astype(np.float32)
    return q, r, rng.standard_normal((nr, d))


class NumpyKnn:
    """Numpy jb_knn / jb_knn_average: splits the queries and the value columns into batches under batch_bytes by the
    engine's per-row and per-column byte counts, and computes each batch with the reference."""
    searches, slabs = [], []

    @classmethod
    def search(cls, query, reference, k, batch_bytes, device):
        assert query.dtype == reference.dtype == np.float32 and query.flags.c_contiguous and reference.flags.c_contiguous
        rows = max(1, batch_bytes // (4 * query.shape[1] + 40 * k + 8))
        parts = [K.kneighbors(query[q0:q0 + rows], reference, k) for q0 in range(0, query.shape[0], rows)]
        cls.searches.append(len(parts))
        return np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts])

    @classmethod
    def average(cls, idx, weights, values, batch_bytes, device):
        assert idx.dtype == np.int64 and values.dtype == np.float64 and values.flags.c_contiguous
        assert weights is None or (weights.dtype == np.float64 and weights.shape == idx.shape)
        w = np.ones(idx.shape) if weights is None else weights
        ws = max(1, batch_bytes // (8 * (values.shape[0] + idx.shape[0])))
        cols = range(0, values.shape[1], ws)
        cls.slabs.append(len(cols))
        return np.concatenate([K.average(idx, w, values[:, c0:c0 + ws]) for c0 in cols], axis=1)


def _impute(*a, **kw):
    return evaluation.knn_impute(*a, backend=NumpyKnn, **kw)


@pytest.mark.parametrize('nq,nr,L,k', [(1, 1, 2, 1), (40, 70, 3, 5), (63, 200, 33, 64), (100, 65, 8, 65)])
def test_oracle_matches_nearest_neighbors(nq, nr, L, k):
    q, r, _ = _data(nq, nr, L, 1, nq + nr)
    dist, idx = K.kneighbors(q, r, k)
    sd, si = NearestNeighbors(n_neighbors=k, algorithm='brute').fit(r.astype(np.float64)).kneighbors(q.astype(np.float64))
    np.testing.assert_array_equal(idx, si)
    np.testing.assert_allclose(dist, sd, rtol=1e-12, atol=0)
    assert np.all(np.diff(dist, axis=1) >= 0)


@pytest.mark.parametrize('weights', ['uniform', 'distance'])
@pytest.mark.parametrize('k', [1, 5, 30])
def test_oracle_matches_kneighbors_regressor(weights, k):
    q, r, v = _data(50, 120, 6, 7, k)
    got = K.knn_impute(q, r, v, k, weights)
    want = KNeighborsRegressor(n_neighbors=k, weights=weights, algorithm='brute').fit(r.astype(np.float64), v) \
        .predict(q.astype(np.float64))
    np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-13)


def test_oracle_ties_go_to_the_lowest_index():
    r = np.array([[1, 0], [0, 1], [-1, 0], [0, -1], [0, 0], [0, 0]], np.float32)
    dist, idx = K.kneighbors(np.zeros((1, 2), np.float32), r, 6)
    np.testing.assert_array_equal(idx[0], [4, 5, 0, 1, 2, 3])
    np.testing.assert_array_equal(dist[0], [0, 0, 1, 1, 1, 1])


def test_driver_equals_the_oracle_and_batches_change_nothing(monkeypatch):
    q, r, v = _data(70, 90, 5, 11, 3)
    want = K.knn_impute(q, r, v, 7, 'distance')
    np.testing.assert_allclose(_impute(q, r, v, k=7, weights='distance'), want, rtol=1e-15, atol=0)
    dist, idx = evaluation.kneighbors(q, r, 7, backend=NumpyKnn)
    kd, ki = K.kneighbors(q, r, 7)
    np.testing.assert_array_equal(idx, ki)
    np.testing.assert_array_equal(dist, kd)
    NumpyKnn.searches.clear()
    NumpyKnn.slabs.clear()
    monkeypatch.setattr(evaluation, 'KNN_BATCH_BYTES', 8 * (90 + 70) * 3)   # 3 value columns a slab, 12 query rows a batch
    small = _impute(q, r, v, k=7, weights='distance')
    assert NumpyKnn.searches == [6] and NumpyKnn.slabs == [4]
    np.testing.assert_array_equal(small, _impute(q, r, v, k=7, weights='distance'))
    np.testing.assert_allclose(small, want, rtol=1e-15, atol=0)


@pytest.mark.parametrize('fmt', [sp.csr_matrix, sp.csc_matrix, sp.coo_matrix])
def test_sparse_values_give_the_dense_result(fmt, monkeypatch):
    rng = np.random.default_rng(5)
    q, r, _ = _data(30, 80, 4, 1, 5)
    V = np.where(rng.random((80, 50)) < 0.05, rng.random((80, 50)) + 0.5, 0.0)
    dense = _impute(q, r, V, k=4)
    np.testing.assert_array_equal(_impute(q, r, fmt(V), k=4), dense)
    monkeypatch.setattr(evaluation, 'KNN_BATCH_BYTES', 8 * (80 + 30) * 7)   # 8 slabs of at most 7 columns
    NumpyKnn.slabs.clear()
    np.testing.assert_array_equal(_impute(q, r, fmt(V), k=4), dense)
    assert NumpyKnn.slabs == [1] * 8                                          # one device call per densified slab
    coo = sp.coo_matrix((np.array([1.0, 2.0]), (np.array([3, 3]), np.array([0, 0]))), shape=(80, 2))   # duplicates add up
    np.testing.assert_array_equal(_impute(q, r, coo, k=4), _impute(q, r, coo.toarray(), k=4))


def test_zero_distance_rule():
    r = np.array([[0, 0], [0, 0], [3, 0], [0, 4]], np.float32)
    v = np.array([[1.0], [3.0], [100.0], [1000.0]])
    q = np.array([[0, 0], [1, 0]], np.float32)
    got = _impute(q, r, v, k=3, weights='distance')
    assert got[0, 0] == 2.0                                         # only the two zero-distance neighbours, weight 1 each
    np.testing.assert_allclose(got[1, 0], (1 + 3 + 100 / 2) / (1 + 1 + 1 / 2), rtol=1e-15)
    want = KNeighborsRegressor(n_neighbors=3, weights='distance', algorithm='brute').fit(r, v).predict(q)
    np.testing.assert_allclose(got, want, rtol=1e-12)
    np.testing.assert_array_equal(evaluation.knn_weights(np.array([[0.0, 0.0, 2.0], [1.0, 2.0, 4.0]]), 'distance'),
                                  [[1.0, 1.0, 0.0], [1.0, 0.5, 0.25]])
    assert evaluation.knn_weights(np.ones((2, 3)), 'uniform') is None


def test_refusals():
    q, r, v = _data(5, 9, 3, 2, 0)
    bad = [
        (dict(query=q[:, :2]), 'one width'),
        (dict(query=q[0]), 'one width'),
        (dict(values=v[:8]), 'one row per reference row'),
        (dict(values=v[:, 0]), 'one row per reference row'),
        (dict(k=0), '1 <= k'),
        (dict(k=10), '1 <= k'),
        (dict(k=2.0), 'integer'),
        (dict(weights='gaussian'), 'weights'),
        (dict(query=np.where(np.arange(15).reshape(5, 3) == 4, np.nan, q)), 'query has non-finite'),
        (dict(reference=np.where(np.arange(27).reshape(9, 3) == 4, np.inf, r)), 'reference has non-finite'),
        (dict(query=q.astype(np.float64) * 1e300), 'query has non-finite'),
        (dict(values=np.where(np.arange(18).reshape(9, 2) == 1, np.nan, v)), 'values has non-finite'),
        (dict(values=sp.csr_matrix(np.where(np.arange(18).reshape(9, 2) == 1, np.inf, v))), 'values has non-finite'),
        (dict(query=np.zeros((0, 3), np.float32)), 'need rows'),
    ]
    for kw, msg in bad:
        args = dict(query=q, reference=r, values=v, k=3, weights='uniform')
        args.update(kw)
        with pytest.raises(ValueError, match=msg):
            _impute(**args)
    big = np.zeros((1100, 2), np.float32)
    with pytest.raises(ValueError, match='1024'):
        evaluation.kneighbors(big[:3], big, 1025, backend=NumpyKnn)
    with pytest.raises(ValueError, match='1 <= k'):
        evaluation.kneighbors(q, r, -1, backend=NumpyKnn)
