"""The host side of the GPU distances (``correspondence.gpu_distance_function``, ``JAMIE(distances='gpu')``) with a numpy
stand-in for the device matrix: slab streaming, row preparation, output dtypes, the k-connectivity loop of
``geodesic_distances``, the host fallback and the keyword. The device arithmetic itself is pinned by
tests/test_gpu_distances.py."""
import warnings

import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.csgraph as csg

from jamie_b200 import correspondence as CR


class NumpyMatrix:
    """Same methods as correspondence.DeviceDistances, in float64 numpy."""
    last = None

    def __init__(self, n, device):
        self.D = np.zeros((n, n))
        self.slabs = 0
        self.k = None
        NumpyMatrix.last = self

    def accumulate(self, kind, slab):
        assert slab.dtype == np.float64 and slab.flags.c_contiguous and slab.shape[0] == len(self.D)
        self.slabs += 1
        if kind == 2:
            self.D += slab @ slab.T
        else:
            for i in range(len(slab)):
                diff = slab - slab[i]
                self.D[i] += (diff * diff).sum(1) if kind == 0 else np.abs(diff).sum(1)

    def finish(self, transform, copy=True):
        with np.errstate(invalid='ignore'):
            if transform == 1:
                self.D = np.sqrt(self.D)
            elif transform == 2:
                self.D = np.clip(1 - self.D, 0, 2)
                np.fill_diagonal(self.D, 0)
            elif transform == 3:
                self.D = (1 - np.clip(self.D, -1, 1)) / 2
        return self.D.copy() if copy else None

    def knn(self, k):
        idx = np.argsort(self.D, axis=1, kind='stable')[:, :k]
        self.lists = (idx, np.take_along_axis(self.D, idx, 1))
        return self.lists

    def geodesic(self, k, copy=True):
        idx, dist = self.lists
        n = len(idx)
        self.k = k
        g = sp.csr_matrix((dist[:, :k].ravel(), idx[:, :k].ravel(), np.arange(0, n * k + 1, k)), shape=(n, n))
        D = csg.shortest_path(g, method='D', directed=False)
        finite_max = np.nanmax(D[D != np.inf])
        D[D > finite_max] = 2 * finite_max
        self.D = D
        return D.copy() if copy else None

    def close(self):
        pass


def gpu_fn(mode, kmax=40):
    return CR.gpu_distance_function(mode, kmax, device=0, matrix=NumpyMatrix)


def _data(kind, n=48, d=23, seed=0):
    rng = np.random.default_rng(seed)
    if kind == 'sparse':
        return sp.random(n, d, density=0.35, random_state=seed, data_rvs=rng.standard_normal, format='csr')
    X = rng.standard_normal((n, d))
    return X.astype(np.float32) if kind == 'float32' else X


@pytest.mark.parametrize('kind', ['float64', 'float32', 'sparse'])
@pytest.mark.parametrize('mode', sorted(CR.GPU_DISTANCE_MODES))
def test_gpu_modes_match_host_function(mode, kind, monkeypatch):
    monkeypatch.setattr(CR, 'SLAB_BYTES', 8 * 48 * 5)     # 5-column slabs: several per matrix
    X = _data(kind)
    dense = X.toarray() if kind == 'sparse' else X
    host = CR.distance_function(mode, 40)
    want = host(dense)
    got = gpu_fn(mode)(X)
    assert NumpyMatrix.last.slabs == 5
    assert got.shape == want.shape and got.dtype == want.dtype, (got.dtype, want.dtype)
    if kind == 'float32':
        # sklearn computes cosine and NearestNeighbors in float32 for float32 input; the GPU path is float64 throughout, so
        # the values are compared with the host function on the same numbers in float64
        want = host(dense.astype(np.float64)).astype(want.dtype)
    scale = np.nanmax(np.abs(want))
    np.testing.assert_allclose(got, want, rtol=1e-9 if got.dtype == np.float64 else 2 ** -23, atol=1e-12 * scale)


def _recording_nearest_neighbors(monkeypatch):
    import sklearn.neighbors
    seen = []
    base = sklearn.neighbors.NearestNeighbors

    class Recording(base):
        def fit(self, X, y=None):
            seen.append(self.n_neighbors)
            return super().fit(X, y)
    Recording.__name__ = base.__name__
    monkeypatch.setattr(sklearn.neighbors, 'NearestNeighbors', Recording)
    return seen


def _clusters(sizes, d=4, gap=50.0, seed=0):
    rng = np.random.default_rng(seed)
    return np.concatenate([rng.standard_normal((m, d)) + gap * c for c, m in enumerate(sizes)])


@pytest.mark.parametrize('case, kmax, want_k', [
    ('manifold', 40, 5),          # connected at the first k
    ('three_clusters', 40, 13),   # 12 points each: connected once a list reaches the next cluster
    ('never', 10, 11),            # two far clusters of 50 points: k stops at the cap K' = 11, unreachable pairs remain
    ('tiny', 40, 5),              # n = 4 < k: every row lists all rows
    ('one_percent', 3, 7),        # 0.01 n = 6 > kmax sets the cap
])
def test_connectivity_loop_reaches_the_host_k(case, kmax, want_k, monkeypatch):
    rng = np.random.default_rng(1)
    if case == 'manifold':
        t = np.linspace(0, 6, 80)
        X = np.stack([np.cos(t), np.sin(t), t], 1) + 1e-3 * rng.standard_normal((80, 3))
    elif case == 'three_clusters':
        X = _clusters([12, 12, 12])
    elif case == 'never':
        X = _clusters([50, 50])
    elif case == 'tiny':
        X = rng.standard_normal((4, 3))
    else:
        X = _clusters([300, 300], d=3)
    seen = _recording_nearest_neighbors(monkeypatch)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        want = CR.geodesic_distances(X, kmax)
    got = gpu_fn('geodesic', kmax)(X)
    n = len(X)
    assert NumpyMatrix.last.k == seen[-1] == min(want_k, n)
    assert NumpyMatrix.last.k <= CR.knn_list_width(n, kmax)
    np.testing.assert_allclose(got, want, rtol=1e-9, atol=0)
    if case == 'never':
        finite = got[:50, :50].max()
        assert np.all(got[:50, 50:] == got.max()) and got.max() > finite


def test_knn_list_width_is_the_last_k_of_the_loop():
    for n, kmax, want in ((100, 40, 41), (100, 41, 43), (5000, 40, 51), (3, 40, 3), (9000, 40, 91)):
        assert CR.knn_list_width(n, kmax) == want


def test_row_preparations_edge_cases():
    X = np.random.default_rng(3).standard_normal((6, 9))
    X[2] = 0.0           # a zero row: cosine distance 1 to every other row, as sklearn gives
    X[4] = 7.0           # a constant row: NaN under pearson / correlation, as np.corrcoef / scipy give
    cos = gpu_fn('cosine')(X)
    assert np.all(cos[2, np.arange(6) != 2] == 1.0) and cos[2, 2] == 0.0
    for mode in ('pearson', 'correlation'):
        got, want = gpu_fn(mode)(X), CR.distance_function(mode, 40)(X)
        np.testing.assert_array_equal(np.isnan(got), np.isnan(want))
        assert np.isnan(got[4, 0]) and np.isnan(got[0, 4])
    with pytest.raises(Exception, match='not well conditioned for spearman'):
        gpu_fn('spearman')(X)


@pytest.mark.parametrize('mode', sorted(CR.GPU_DISTANCE_MODES))
def test_one_row_behaves_as_on_the_host(mode):
    X = np.random.default_rng(4).standard_normal((1, 5))
    want = CR.distance_function(mode, 40)(X)
    got = gpu_fn(mode)(X)
    assert got.shape == np.shape(want)
    np.testing.assert_array_equal(got, want)


def test_unsupported_mode_warns_and_runs_the_host_function():
    X = np.random.default_rng(5).standard_normal((10, 4))
    with pytest.warns(UserWarning, match="'chebyshev' has no GPU path"):
        fn = gpu_fn('chebyshev')
    np.testing.assert_array_equal(fn(X), CR.distance_function('chebyshev', 40)(X))


def test_distances_keyword():
    from jamie_b200.jamie import JAMIE
    assert JAMIE().distances == 'host'
    assert JAMIE(distances='gpu').distances == 'gpu'
    with pytest.raises(AssertionError, match="distances must be 'host' or 'gpu', not 'cuda'"):
        JAMIE(distances='cuda')


def test_compute_distances_routes_sparse_input_to_the_gpu_path(monkeypatch, capsys):
    from jamie_b200.jamie import JAMIE
    seen = []
    real = CR.gpu_distance_function

    def fake(mode, kmax, device=0):
        fn = real(mode, kmax, matrix=NumpyMatrix)

        def wrapped(df):
            seen.append((type(df), device))
            return fn(df)
        return wrapped
    monkeypatch.setattr(CR, 'gpu_distance_function', fake)
    monkeypatch.setattr(JAMIE, '_cuda_index', lambda self: 3)
    rng = np.random.default_rng(6)
    data = [sp.random(30, 12, density=0.5, random_state=1, data_rvs=rng.standard_normal, format='csr'), rng.standard_normal((25, 7))]
    runs = {}
    for how in ('host', 'gpu'):
        jm = JAMIE(distances=how)
        jm.dataset, jm.dataset_num = data, 2
        jm.compute_distances()
        runs[how] = (jm.dist, capsys.readouterr().out)
    assert seen == [(sp.csr_matrix, 3), (np.ndarray, 3)]
    assert runs['gpu'][1] == runs['host'][1]
    for g, h in zip(runs['gpu'][0], runs['host'][0]):
        assert g.shape == h.shape and g.dtype == h.dtype
        np.testing.assert_allclose(g, h, rtol=1e-9)
