"""The F-estimation distances on the GPU (jb_dist_*, csrc/distances.cuh; SURVEY.md 8f row N2): the device arithmetic pinned
against a float64 numpy restatement (direct differences, no dot-product expansion), the kNN lists and the geodesic
all-pairs shortest paths against scipy on the GPU's own lists, the host path users get today, and
``JAMIE(distances='gpu')`` end to end."""
import contextlib
import io
import warnings

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.csgraph as csg
from scipy import stats

from jamie_b200 import correspondence as CR

pytestmark = pytest.mark.gpu

ZERO_DIAGONAL = ('geodesic', 'euclidean', 'l2', 'sqeuclidean', 'cityblock', 'l1', 'manhattan', 'cosine', 'correlation')


def restated(X, mode):
    """float64 restatement of every GPU mode but geodesic, from the definitions"""
    X = np.asarray(X, np.float64)
    n = len(X)
    if mode in ('euclidean', 'l2', 'sqeuclidean', 'cityblock', 'l1', 'manhattan'):
        D = np.empty((n, n))
        for i in range(n):
            diff = X - X[i]
            D[i] = np.abs(diff).sum(1) if mode in ('cityblock', 'l1', 'manhattan') else (diff * diff).sum(1)
        return np.sqrt(D) if mode in ('euclidean', 'l2') else D
    if mode == 'spearman':
        X = stats.rankdata(X, axis=1)
    if mode != 'cosine':
        X = X - X.mean(1, keepdims=True)
    norm = np.sqrt((X * X).sum(1))
    if mode == 'cosine':
        norm[norm == 0] = 1
    with np.errstate(invalid='ignore', divide='ignore'):
        U = X / norm[:, None]
    G = U @ U.T
    with np.errstate(invalid='ignore'):
        if mode in ('cosine', 'correlation'):
            D = np.clip(1 - G, 0, 2)
            np.fill_diagonal(D, 0)
            return D
        return (1 - np.clip(G, -1, 1)) / 2


def _data(n, d, kind='float64', variant='plain', seed=0):
    rng = np.random.default_rng(seed + 1000 * n + d)
    X = rng.standard_normal((n, d))
    if variant == 'offset':
        X += 100.0                     # rows far from the origin, like raw counts
    if kind == 'sparse':
        X[rng.random((n, d)) < 0.6] = 0.0
    if variant == 'duplicates' and n > 3:
        X[1] = X[0]
        X[n - 1] = X[n // 2]
    if kind == 'sparse':
        return sp.csr_matrix(X)
    return X.astype(np.float32) if kind == 'float32' else X


def _check_pairwise(got, X, mode):
    dense = X.toarray() if sp.issparse(X) else X
    ref = restated(np.asarray(dense, np.float64), mode)
    scale = np.nanmax(np.abs(ref)) if np.any(np.isfinite(ref)) else 1.0
    scale = scale if scale > 0 else 1.0
    g = got.astype(np.float64)
    # float32 outputs (what the host returns for float32 euclidean / cosine) carry their own rounding
    tol = 1e-12 * scale + (2.0 ** -24 * np.abs(ref) if got.dtype == np.float32 else 0)
    np.testing.assert_array_equal(np.isnan(g), np.isnan(ref))
    ok = np.isnan(ref) | (np.abs(g - ref) <= tol)
    assert ok.all(), (mode, np.nanmax(np.abs(g - ref)) / scale)
    assert np.array_equal(got, got.T, equal_nan=True)
    if mode in ZERO_DIAGONAL:
        assert np.all(np.diagonal(got) == 0)


GRID = [(n, d) for n in (1, 2, 5, 63, 64, 65) for d in (1, 3, 39)] + [(65, 300), (64, 2000), (1500, 300)]


@pytest.mark.parametrize('n, d', GRID)
@pytest.mark.parametrize('mode', ['euclidean', 'sqeuclidean', 'cityblock', 'cosine', 'correlation', 'pearson', 'spearman'])
def test_pairwise_modes_match_the_float64_restatement(mode, n, d):
    X = _data(n, d)
    fn = CR.gpu_distance_function(mode, 40)
    if n == 1 and mode in ('pearson', 'spearman'):
        np.testing.assert_array_equal(fn(X), CR.distance_function(mode, 40)(X))
        return
    ref = restated(X, mode)
    if mode == 'spearman' and np.isnan(ref).any():
        with pytest.raises(Exception, match='not well conditioned for spearman'):
            fn(X)
        return
    got = fn(X)
    assert got.shape == (n, n) and got.dtype == np.float64
    _check_pairwise(got, X, mode)
    np.testing.assert_array_equal(fn(X), got)      # bit-identical on a repeated run


@pytest.mark.parametrize('variant', ['plain', 'offset', 'duplicates'])
@pytest.mark.parametrize('kind', ['float32', 'sparse'])
@pytest.mark.parametrize('mode', ['euclidean', 'l2', 'sqeuclidean', 'cityblock', 'l1', 'manhattan', 'cosine', 'correlation',
                                  'pearson', 'spearman'])
def test_input_kinds_and_awkward_data(mode, kind, variant):
    X = _data(65, 39, kind, variant)
    got = CR.gpu_distance_function(mode, 40)(X)
    want_dtype = np.float32 if kind == 'float32' and mode in CR.KEEPS_FLOAT32 else np.float64
    assert got.dtype == want_dtype
    _check_pairwise(got, X.astype(np.float64) if kind == 'float32' else X, mode)
    if variant == 'duplicates' and mode in ('euclidean', 'l2', 'sqeuclidean', 'cityblock', 'l1', 'manhattan'):
        assert got[0, 1] == 0 and got[65 // 2, 64] == 0


def _geodesic_parts(X, kmax):
    """every stage of the GPU geodesic through the ABI: finished D, lists, k, geodesic matrix"""
    n = len(X)
    m = CR.DeviceDistances(n, 0)
    try:
        for slab in CR.prepared_slabs(X, None, 16):       # narrow slabs: many accumulate calls
            m.accumulate(0, slab)
        D = m.finish(1)
        idx, dist = m.knn(CR.knn_list_width(n, kmax))
        k = min(CR.connectivity_k(idx, kmax), n)
        G = m.geodesic(k)
    finally:
        m.close()
    return D, idx, dist, k, G


def _scipy_geodesic(idx, dist, k):
    n = len(idx)
    g = sp.csr_matrix((dist[:, :k].ravel(), idx[:, :k].ravel(), np.arange(0, n * k + 1, k)), shape=(n, n))
    S = csg.shortest_path(g, method='D', directed=False)   # explicit zeros (duplicate rows) are edges
    finite_max = np.nanmax(S[S != np.inf])
    S[S > finite_max] = 2 * finite_max
    return S


@pytest.mark.parametrize('case', ['manifold', 'clusters', 'duplicates', 'offset', 'n1', 'n2', 'n65'])
def test_geodesic_matches_scipy_on_the_gpu_lists(case):
    rng = np.random.default_rng(7)
    kmax = 40
    if case in ('manifold', 'duplicates', 'offset'):
        t = rng.random(700) * 8
        X = np.stack([np.cos(t) * t, np.sin(t) * t, 0.5 * t], 1) @ rng.standard_normal((3, 39)) + 0.01 * rng.standard_normal((700, 39))
        if case == 'duplicates':
            X[10:14] = X[9]
        if case == 'offset':
            X += 100.0
    elif case == 'clusters':
        X = np.concatenate([rng.standard_normal((90, 3)) + 100 * c for c in range(3)])
        kmax = 7
    else:
        X = rng.standard_normal(({'n1': 1, 'n2': 2, 'n65': 65}[case], 5))
    n = len(X)
    D, idx, dist, k, G = _geodesic_parts(X, kmax)
    K = CR.knn_list_width(n, kmax)
    _check_pairwise(D, X, 'euclidean')
    np.testing.assert_array_equal(idx, np.argsort(D, axis=1, kind='stable')[:, :K])
    np.testing.assert_array_equal(dist, np.take_along_axis(D, idx.astype(np.int64), 1))
    S = _scipy_geodesic(idx, dist, k)
    assert np.all(np.abs(G - S) <= 1e-12 * np.abs(S))
    assert np.array_equal(G, G.T)
    if case == 'clusters':
        finite = G[G < G.max()].max()
        assert G.max() == 2 * finite and np.all(G[:90, 90:] == G.max())
    if case == 'duplicates':
        assert np.all(G[9, 10:14] == 0)      # the zero-weight edges connect the duplicates
        np.testing.assert_allclose(G[13], G[9], rtol=1e-12, atol=0)
    D2, idx2, dist2, k2, G2 = _geodesic_parts(X, kmax)
    assert k2 == k and np.array_equal(D2, D) and np.array_equal(idx2, idx) and np.array_equal(G2, G)


@pytest.mark.parametrize('mode', sorted(CR.GPU_DISTANCE_MODES))
def test_matches_the_host_path(mode):
    """Centred data without duplicate rows: sklearn's formulas are exact to ~1e-14 there, so the paths agree to 1e-9."""
    rng = np.random.default_rng(11)
    if mode == 'geodesic':
        t = rng.random(400) * 6
        X = np.stack([np.cos(t), np.sin(t), t], 1) @ rng.standard_normal((3, 60)) + 0.01 * rng.standard_normal((400, 60))
    else:
        X = rng.standard_normal((300, 60))
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        want = CR.distance_function(mode, 40)(X)
    got = CR.gpu_distance_function(mode, 40)(X)
    assert got.shape == want.shape and got.dtype == want.dtype
    scale = np.abs(want).max()
    if mode == 'geodesic':
        from sklearn.neighbors import NearestNeighbors
        D, idx, _, k, _ = _geodesic_parts(X, 40)
        host_graph = NearestNeighbors(n_neighbors=k).fit(X).kneighbors_graph(X).tocsr()
        host_graph.sort_indices()
        assert np.array_equal(host_graph.indices.reshape(len(X), k), np.sort(idx[:, :k], 1))   # identical kNN edge sets
        np.testing.assert_allclose(got, want, rtol=1e-9, atol=0)
    else:
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-9 * scale)


@pytest.mark.parametrize('mode', ['euclidean', 'geodesic', 'cosine', 'pearson'])
def test_offset_and_duplicate_rows_against_the_host_path(mode):
    """Offset data (+100) and duplicate rows: sklearn's euclidean is |x|^2 - 2 x.y + |y|^2, whose cancellation leaves
    identical rows up to ~1e-6 of the scale apart (the GPU sums (x - y)^2 directly and is pinned to 1e-12 above), so the
    two paths are compared at 1e-5 of the scale."""
    rng = np.random.default_rng(12)
    t = rng.random(300) * 6
    X = np.stack([np.cos(t), np.sin(t), t], 1) @ rng.standard_normal((3, 60)) + 0.01 * rng.standard_normal((300, 60)) + 100.0
    X[5:8] = X[4]
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        want = CR.distance_function(mode, 40)(X)
    got = CR.gpu_distance_function(mode, 40)(X)
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-5 * np.abs(want).max())


def test_handle_errors():
    import ctypes as C
    from jamie_b200 import _lib
    lib = _lib.load()
    h = C.c_void_p()
    with pytest.raises(RuntimeError, match='float64 distance matrix'):
        _lib.check(lib.jb_dist_create(2_000_000, 0, C.byref(h)))      # 32 TB
    m = CR.DeviceDistances(10, 0)
    try:
        with pytest.raises(RuntimeError, match='needs the neighbour lists'):
            m.geodesic(3)
        with pytest.raises(RuntimeError, match='neighbours of 10 rows'):
            m.knn(11)
    finally:
        m.close()


def _fit(distances):
    from jamie import JAMIE
    rng = np.random.default_rng(2)
    t = rng.random(96)
    lat = np.stack([t, np.sin(4 * t), t ** 2], 1)
    data = [lat @ rng.normal(size=(3, 40)) + 0.02 * rng.normal(size=(96, 40)),
            lat @ rng.normal(size=(3, 28)) + 0.02 * rng.normal(size=(96, 28))]
    jm = JAMIE(output_dim=8, batch_size=96, pca_dim=None, epoch_pd=200, log_pd=100, epoch_DNN=60, min_epochs=20, log_DNN=30,
               distances=distances)
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        emb = jm.fit_transform(dataset=data)
    jm.engine.close()
    return jm, emb, buf.getvalue()


def test_jamie_gpu_distances_end_to_end():
    """The small default-constructor setup of test_gpu_correspondence.py with distances='gpu' and 'host'."""
    def lines(out):    # everything up to the end of matching but Prime_Dual's numbers
        head = out.split('Finished Matching!')[0]
        return [ln for ln in head.splitlines() if not ln.startswith('epoch:[')]
    jg, eg, og = _fit('gpu')
    jh, eh, oh = _fit('host')
    assert lines(og) == lines(oh)
    assert [ln.split()[0] for ln in og.splitlines() if ln.startswith('epoch:[')] == \
        [ln.split()[0] for ln in oh.splitlines() if ln.startswith('epoch:[')]
    for g, h in zip(jg.dist, jh.dist):
        assert g.shape == h.shape and g.dtype == h.dtype == np.float64
        np.testing.assert_allclose(g, h, rtol=1e-9)
    Fg, Fh = jg.match_result[0], jh.match_result[0]
    assert np.linalg.norm(Fg - Fh) / np.linalg.norm(Fh) < 1e-4
    assert all(np.all(np.isfinite(e)) for e in eg)
