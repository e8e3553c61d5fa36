"""kneighbors / knn_impute / JAMIE.knn_predict on the GPU (jb_knn, jb_knn_average: csrc/knn.cuh): the device's neighbour
lists equal the float64 reference's (tests/knn_oracle.py) across tile, range and batch edges, with exact ties and
duplicate rows; agreement with sklearn's brute-force NearestNeighbors and KNeighborsRegressor; bit-identical reruns,
batch splits and sparse values; the memory refusal; and a trained model's knn_predict end to end."""
import ctypes as C
import os

import numpy as np
import pytest
import scipy.sparse as sp
from sklearn.neighbors import KNeighborsRegressor, NearestNeighbors

from tests import knn_oracle as K

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'mmdma.npz')


def _rows(kind, n, L, rng):
    if kind == 'normal':
        return rng.standard_normal((n, L)).astype(np.float32)
    if kind == 'grid':                                   # exact ties everywhere
        return rng.integers(-2, 3, (n, L)).astype(np.float32)
    if kind == 'duplicates':                             # each row repeated, in scattered places
        base = rng.standard_normal((max(1, n // 3), L)).astype(np.float32)
        return base[rng.integers(0, base.shape[0], n)]
    raise ValueError(kind)


def _search(q, r, k, batch_bytes=1 << 30):
    from jamie_b200.evaluation import DeviceKnn
    return DeviceKnn.search(np.ascontiguousarray(q, np.float32), np.ascontiguousarray(r, np.float32), k, batch_bytes, None)


def _check_lists(q, r, k, **kw):
    dist, idx = _search(q, r, k, **kw)
    kd, ki = K.kneighbors(q, r, k)
    np.testing.assert_array_equal(idx, ki)
    np.testing.assert_allclose(dist, kd, rtol=1e-12, atol=0)
    return dist, idx


# nq and nr each in {1, 63, 64, 65, 1000, 70000}; L in {2, 32, 33, 100}; k in {1, 5, 64, 1024, nr}
SHAPES = [
    (1, 1, 2, 1), (1, 63, 32, 'nr'), (63, 64, 33, 5), (64, 65, 100, 64), (65, 63, 2, 'nr'), (64, 64, 32, 64),
    (1000, 1000, 32, 5), (1000, 1000, 33, 1000), (1000, 65, 100, 1), (63, 1000, 2, 64), (65, 1024, 32, 1024),
    (1, 70000, 32, 5), (63, 70000, 33, 1024), (65, 70000, 2, 64), (70000, 64, 32, 5), (70000, 1, 100, 1),
]


@pytest.mark.parametrize('nq,nr,L,k', SHAPES)
@pytest.mark.parametrize('kind', ['normal', 'grid'])
def test_lists_equal_the_reference(nq, nr, L, k, kind):
    rng = np.random.default_rng(nq * 7 + nr + L)
    k = nr if k == 'nr' else k
    _check_lists(_rows(kind, nq, L, rng), _rows(kind, nr, L, rng), k)


@pytest.mark.parametrize('k', [1, 5, 64, 1000])
def test_duplicates_and_query_is_reference(k):
    rng = np.random.default_rng(k)
    r = _rows('duplicates', 1000, 32, rng)
    dist, idx = _check_lists(r, r, k)
    first = {tuple(row): i for i, row in reversed(list(enumerate(r.tolist())))}
    np.testing.assert_array_equal(idx[:, 0], [first[tuple(row)] for row in r.tolist()])   # the lowest equal row
    assert np.all(dist[:, 0] == 0)
    g = _rows('grid', 1000, 2, rng)                        # 25 distinct rows, 40 copies each
    _check_lists(g, g, k)


def test_small_batch_against_many_references():
    rng = np.random.default_rng(3)
    r = _rows('grid', 200000, 3, rng)
    for k in (5, 1024):
        _check_lists(_rows('grid', 100, 3, rng), r, k)


def test_kneighbors_matches_sklearn():
    from jamie_b200.evaluation import kneighbors
    rng = np.random.default_rng(4)
    q, r = _rows('normal', 1000, 32, rng), _rows('normal', 3000, 32, rng)
    for k in (1, 5, 50):
        dist, idx = kneighbors(q, r, k)
        sd, si = NearestNeighbors(n_neighbors=k, algorithm='brute').fit(r).kneighbors(q)
        np.testing.assert_array_equal(idx, si)
        np.testing.assert_allclose(dist, sd, rtol=1e-6, atol=0)


@pytest.mark.parametrize('weights,rtol', [('uniform', 1e-12), ('distance', 1e-6)])
def test_knn_impute_matches_sklearn(weights, rtol):
    from jamie_b200.evaluation import knn_impute
    rng = np.random.default_rng(5)
    q, r = _rows('normal', 700, 16, rng), _rows('normal', 2500, 16, rng)
    V = rng.standard_normal((2500, 300))
    for k in (1, 5, 30):
        got = knn_impute(q, r, V, k=k, weights=weights)
        want = KNeighborsRegressor(n_neighbors=k, weights=weights, algorithm='brute').fit(r, V).predict(q)
        np.testing.assert_allclose(got, want, rtol=rtol, atol=rtol * np.abs(V).max())   # sklearn's fp32 distance error
        np.testing.assert_allclose(got, K.knn_impute(q, r, V, k, weights), rtol=1e-12, atol=1e-13)


def test_bit_identical_reruns_batches_and_sparse(monkeypatch):
    from jamie_b200 import evaluation
    rng = np.random.default_rng(6)
    q, r = _rows('grid', 3000, 33, rng), _rows('normal', 20000, 33, rng)
    q = np.concatenate([q, _rows('normal', 1000, 33, rng)])
    for k in (5, 64):
        ref = _search(q, r, k)
        for bb in (1 << 30, 1, 40 * k * 100, 40 * k * 1000):   # one batch; one query row; ~100 and ~1000 rows a batch
            dist, idx = _search(q, r, k, batch_bytes=bb)
            np.testing.assert_array_equal(idx, ref[1])
            np.testing.assert_array_equal(dist, ref[0])
    V = np.where(rng.random((20000, 500)) < 0.05, rng.random((20000, 500)), 0.0)
    for weights in ('uniform', 'distance'):
        want = evaluation.knn_impute(q, r, V, k=7, weights=weights)
        np.testing.assert_array_equal(evaluation.knn_impute(q, r, V, k=7, weights=weights), want)
        np.testing.assert_array_equal(evaluation.knn_impute(q, r, sp.csr_matrix(V), k=7, weights=weights), want)
        with monkeypatch.context() as m:
            m.setattr(evaluation, 'KNN_BATCH_BYTES', 8 * (20000 + 4000) * 37)   # 14 column slabs; 1 GB / 8 k query rows
            np.testing.assert_array_equal(evaluation.knn_impute(q, r, V, k=7, weights=weights), want)
            np.testing.assert_array_equal(evaluation.knn_impute(q, r, sp.csc_matrix(V), k=7, weights=weights), want)


def test_refuses_a_problem_larger_than_free_memory():
    import torch
    from jamie_b200 import _lib
    from jamie_b200.evaluation import knn_impute
    lib = _lib.load()
    p = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
    free0 = torch.cuda.mem_get_info()[0]
    z = np.zeros(16, np.float32)
    idx, dist = np.zeros(4, np.int64), np.zeros(4)
    rc = lib.jb_knn(p(z), 1, p(z), (1 << 31) - 1, 1 << 20, 1, 1 << 30, 0, p(idx), p(dist))   # 9 PB of reference rows
    assert rc != 0
    msg = lib.jb_last_error().decode()
    assert 'GB' in msg and 'free' in msg, msg
    out = np.zeros(4)
    rc = lib.jb_knn_average(p(idx), None, 1, 1, p(out), 1 << 40, 1, 1, 1 << 30, 0, p(out))     # one column: 8.8 TB
    assert rc != 0
    msg = lib.jb_last_error().decode()
    assert 'GB' in msg and 'free' in msg, msg
    rc = lib.jb_knn(p(z), 1, p(z), 4, 4, 5, 1 << 30, 0, p(idx), p(dist))
    assert rc != 0 and 'k = 5' in lib.jb_last_error().decode()
    assert abs(torch.cuda.mem_get_info()[0] - free0) < (64 << 20)
    rng = np.random.default_rng(0)
    q, r, V = _rows('normal', 50, 4, rng), _rows('normal', 80, 4, rng), rng.standard_normal((80, 3))
    np.testing.assert_allclose(knn_impute(q, r, V), K.knn_impute(q, r, V, 5), rtol=1e-12)


def test_end_to_end_knn_predict():
    from jamie import JAMIE
    from jamie.evaluation import imputation_correlation
    g = np.load(GOLD)
    data = [g['data1'].astype(np.float32), g['data2'].astype(np.float32)]
    np.random.seed(1)
    jm = JAMIE(output_dim=8, batch_size=64, pca_dim=[20, 16], epoch_DNN=20, min_epochs=1, use_f_tilde=False, manual_seed=5)
    jm.fit_transform(dataset=[x.copy() for x in data], P=np.eye(data[0].shape[0]))
    try:
        e0, e1 = jm.transform_one(data[0], 0), jm.transform_one(data[1], 1)
        for weights in ('uniform', 'distance'):
            got = jm.knn_predict(data[0], 0, data[1], k=5, weights=weights)
            assert got.shape == data[1].shape and got.dtype == np.float64
            want = KNeighborsRegressor(n_neighbors=5, weights=weights, algorithm='brute') \
                .fit(np.float32(e1), data[1].astype(np.float64)).predict(np.float32(e0))
            np.testing.assert_allclose(got, want, rtol=1e-6, atol=1e-6 * np.abs(data[1]).max())
            np.testing.assert_allclose(got, K.knn_impute(e0, e1, data[1], 5, weights), rtol=1e-12, atol=1e-12)
        np.testing.assert_array_equal(jm.knn_predict(data[0], 0, sp.csr_matrix(data[1])), jm.knn_predict(data[0], 0, data[1]))
        back = jm.knn_predict(data[1], 1, data[0])
        np.testing.assert_allclose(back, K.knn_impute(e1, e0, data[0], 5), rtol=1e-12, atol=1e-12)
        r_knn = imputation_correlation(jm.knn_predict(data[0], 0, data[1]), data[1])
        r_dec = imputation_correlation(jm.modal_predict(data[0], 0), data[1])
        assert r_knn.shape == r_dec.shape == (data[1].shape[1],)
        assert np.isfinite(np.nanmean(r_knn)) and np.isfinite(np.nanmean(r_dec))
    finally:
        jm.engine.close()
