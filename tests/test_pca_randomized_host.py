"""The randomized PCA fit driver (jamie_b200/pca_fit.py randomized_fit_transform) on the host: a float64 numpy stand-in for
the device operand runs the whole algorithm without a GPU, against sklearn's exact PCA."""
import numpy as np
import pytest
import scipy.sparse as sp


class NumpyOperator:
    """float64 numpy stand-in for pca_fit.DeviceOperator (same methods; counts the products)"""

    def __init__(self, X, device):
        self.X = X.tocsr().astype(np.float64) if sp.issparse(X) else np.asarray(X, np.float64)
        self.n, self.d = X.shape
        self.mean = np.zeros(self.d)
        self.calls = []

    def stats(self):
        X = self.X
        self.mean = np.asarray(X.mean(axis=0)).ravel()
        if sp.issparse(X):
            var = np.asarray(X.multiply(X).mean(axis=0)).ravel() - self.mean ** 2
        else:
            var = ((X - self.mean) ** 2).mean(axis=0)
        return self.mean.copy(), var

    def upload(self, a):
        return np.asarray(a, np.float64)

    def apply(self, trans, B):
        self.calls.append(trans)
        if trans:
            return np.asarray(self.X.T @ B) - np.outer(self.mean, B.sum(axis=0))
        return np.asarray(self.X @ B) - (self.mean @ B)[None, :]

    def orth(self, Y):
        return np.linalg.qr(Y)[0]

    def download(self, Y):
        return np.array(Y, np.float64)

    def close(self):
        pass


def _data(n, d, rank_like, seed):
    rng = np.random.default_rng(seed)
    lat = rng.normal(size=(n, rank_like)) * np.linspace(3.0, 0.5, rank_like)      # well separated spectrum
    X = lat @ rng.normal(size=(rank_like, d)) + 0.05 * rng.normal(size=(n, d)) + rng.normal(size=d) * 4   # non-zero means
    return X.astype(np.float32).astype(np.float64)


def _sparse_data(n, d, rank_like, seed):
    """sparse with a gapped spectrum: sparse loadings of sparse programs (rank rank_like, ~25 % nonzeros), plus small noise
    on the stored entries"""
    rng = np.random.default_rng(seed)
    lat = rng.normal(size=(n, rank_like)) * np.linspace(3.0, 0.5, rank_like) * (rng.random((n, rank_like)) < 0.3)
    X = lat @ (rng.normal(size=(rank_like, d)) * (rng.random((rank_like, d)) < 0.15) + 2.0 * (rng.random((rank_like, d)) < 0.05))
    nz = X != 0
    X[nz] += 0.05 * rng.normal(size=int(nz.sum()))
    return sp.csr_matrix(X.astype(np.float32).astype(np.float64))


def fit(X, k, seed=0, operator=NumpyOperator):
    from jamie_b200 import pca_fit
    return pca_fit.randomized_fit_transform(X, k, seed=seed, device=0, operator=operator)


def check_against_exact(X, k, pca, sample, cos_tol, var_rtol, sample_tol, noise_rtol=1e-6):
    from sklearn.decomposition import PCA
    Xd = X.toarray() if sp.issparse(X) else X
    ref = PCA(n_components=k, svd_solver='full')
    sample_ref = ref.fit_transform(Xd)
    dots = np.sum(pca.components_ * ref.components_, axis=1)
    assert dots.min() > 1 - cos_tol, dots.min()           # same vectors, same signs (v-based svd_flip)
    np.testing.assert_allclose(pca.explained_variance_, ref.explained_variance_, rtol=var_rtol)
    np.testing.assert_allclose(pca.singular_values_, ref.singular_values_, rtol=var_rtol)
    np.testing.assert_allclose(pca.explained_variance_ratio_, ref.explained_variance_ratio_, rtol=var_rtol)
    np.testing.assert_allclose(pca.mean_, ref.mean_, rtol=1e-12, atol=1e-12 * np.abs(Xd).max())
    np.testing.assert_allclose(pca.noise_variance_, ref.noise_variance_, rtol=noise_rtol)
    assert np.abs(sample - sample_ref).max() < sample_tol * np.abs(sample_ref).max()


@pytest.mark.parametrize('n,d,k,kind', [(400, 60, 12, 'dense'), (90, 300, 10, 'dense'), (300, 120, 16, 'sparse'),
                                        (80, 260, 12, 'sparse'), (70, 64, 60, 'dense'), (50, 90, 45, 'sparse')])
def test_matches_exact_pca(n, d, k, kind):
    """tall and wide (both transpose branches), dense and sparse, and k close to min(n, d)"""
    r = max(k + 4, 20) if k + 4 < min(n, d) else min(n, d)
    X = _sparse_data(n, d, r, n + d) if kind == 'sparse' else _data(n, d, r, n + d)
    pca, sample = fit(X, k)
    check_against_exact(X, k, pca, sample, 1e-9, 1e-7, 1e-7)


@pytest.mark.parametrize('n,d,k,n_iter', [(400, 60, 5, 7), (400, 60, 6, 4), (90, 300, 8, 7), (90, 300, 9, 4)])
def test_n_iter_rule_counts_products(n, d, k, n_iter, monkeypatch):
    """n_iter = 7 if k < 0.1 min(n, d) else 4; 2 n_iter + 2 products, alternating A @ Q and A^T @ Q"""
    ops = []

    class Counting(NumpyOperator):
        def __init__(self, X, device):
            super().__init__(X, device)
            ops.append(self)
    fit(_data(n, d, 20, 1), k, operator=Counting)
    calls = ops[0].calls
    assert len(calls) == 2 * n_iter + 2
    fwd = 1 if n < d else 0
    assert calls == [fwd, 1 - fwd] * (n_iter + 1)


def test_same_seed_same_output_and_seed_matters():
    X = _data(200, 80, 20, 2)
    a, sa = fit(X, 8, seed=3)
    b, sb = fit(X, 8, seed=3)
    np.testing.assert_array_equal(a.components_, b.components_)
    np.testing.assert_array_equal(sa, sb)
    # a different Omega: the same subspace up to round-off, but not the same bits
    c, _ = fit(X, 8, seed=4)
    assert not np.array_equal(a.components_, c.components_)
    np.testing.assert_allclose(np.abs(np.sum(a.components_ * c.components_, axis=1)), 1.0, atol=1e-9)


def test_returned_object_is_a_usable_sklearn_pca():
    from sklearn.decomposition import PCA
    X = _data(150, 40, 20, 5)
    pca, sample = fit(X, 6)
    assert isinstance(pca, PCA)
    assert pca._fit_svd_solver == 'randomized'
    assert pca.n_components_ == 6 and pca.n_samples_ == 150 and pca.n_features_in_ == 40
    assert pca.components_.shape == (6, 40) and sample.shape == (150, 6)
    for a in (pca.components_, pca.mean_, pca.explained_variance_, pca.explained_variance_ratio_, pca.singular_values_, sample):
        assert a.dtype == np.float64
    # sign convention: the largest-magnitude entry of every component is positive
    idx = np.argmax(np.abs(pca.components_), axis=1)
    assert np.all(pca.components_[np.arange(6), idx] > 0)
    np.testing.assert_allclose(pca.explained_variance_, pca.singular_values_ ** 2 / 149)
    # fit_transform's sample U S is the projection of the training rows, to the accuracy of the range finder (sklearn's
    # own randomized fit_transform returns U S as well)
    np.testing.assert_allclose(pca.transform(X), sample, atol=1e-4 * np.abs(sample).max())
    assert np.all(np.diff(pca.explained_variance_) <= 0)


def test_sparse_input_is_never_densified():
    X = _sparse_data(120, 50, 20, 6)
    seen = []

    class Recording(NumpyOperator):
        def __init__(self, X, device):
            seen.append(type(X))
            super().__init__(X, device)
    fit(X, 5, operator=Recording)
    fit(X.tocsc(), 5, operator=Recording)
    assert seen == [sp.csr_matrix, sp.csc_matrix]


def test_bad_n_components():
    X = _data(30, 20, 10, 7)
    for k in (0, 21):
        with pytest.raises(ValueError, match='n_components'):
            fit(X, k)


def test_pca_fit_keyword():
    from jamie import JAMIE
    for how in ('gpu', 'sklearn', 'randomized'):
        assert JAMIE(pca_fit=how).pca_fit == how
    with pytest.raises(AssertionError, match="pca_fit must be 'gpu', 'sklearn' or 'randomized', not 'eigh'"):
        JAMIE(pca_fit='eigh')


def test_sparse_create_refuses_inconsistent_csr():
    """checked on the host before the device is touched"""
    import ctypes as C
    from jamie_b200 import _lib
    if not __import__('os').path.exists(_lib.LIB_PATH):
        import __graft_entry__ as g
        g.build()
    lib = _lib.load()
    X = sp.csr_matrix(np.array([[1.0, 0.0, 2.0], [0.0, 3.0, 0.0]], np.float32))
    T = X.tocsc()

    def create(rp, ci, cp, ri, nnz=3):
        arrs = [np.asarray(rp, np.int64), np.asarray(ci, np.int32), X.data.astype(np.float32),
                np.asarray(cp, np.int64), np.asarray(ri, np.int32), T.data.astype(np.float32)]
        h = C.c_void_p()
        rc = lib.jb_pcaop_create_sparse(2, 3, nnz, *(a.ctypes.data_as(C.c_void_p) for a in arrs), 0, C.byref(h))
        assert rc != 0 and not h.value
        return lib.jb_last_error().decode()
    assert 'expected nnz' in create([0, 2, 2], X.indices, T.indptr, T.indices)          # row_ptr[n] != nnz
    assert 'out of range' in create(X.indptr, [0, 3, 1], T.indptr, T.indices)          # column index >= d
    assert 'out of range' in create(X.indptr, X.indices, T.indptr, [0, 2, 0])          # row index >= n
    assert 'decreases' in create([0, 4, 3], X.indices, T.indptr, T.indices)                # row_ptr not monotone
    assert 'expected nnz' in create(X.indptr, X.indices, [0, 1, 2, 2], T.indices)      # col_ptr[d] != nnz
