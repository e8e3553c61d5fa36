"""PCA fit with the Gram matrix on the GPU (jb_pca_colsum / jb_pca_gram + host eigh, jamie_b200/pca_fit.py; SURVEY.md 8
row N3) against the call the reference makes, ``sklearn.decomposition.PCA(n_components).fit_transform(data)``
(jamie/jamie.py:449-451), with every solver sklearn may pick for it."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _data(n, d, rank_like, seed):
    rng = np.random.default_rng(seed)
    lat = rng.normal(size=(n, rank_like)) * np.linspace(3.0, 0.5, rank_like)      # well separated spectrum
    X = lat @ rng.normal(size=(rank_like, d)) + 0.05 * rng.normal(size=(n, d)) + rng.normal(size=d) * 4   # non-zero means
    return X.astype(np.float32).astype(np.float64)


def _engine():
    from jamie_b200.engine import Engine
    return Engine([8, 8], 2, 8, 0.0)


@pytest.mark.parametrize('n,d,k,solver', [(400, 60, 12, 'full'), (3000, 130, 16, 'covariance_eigh'), (700, 1030, 24, 'randomized'),
                                          (20000, 257, 32, 'auto'), (90, 200, 10, 'full')])
def test_gram_pca_matches_sklearn(n, d, k, solver):
    from sklearn.decomposition import PCA
    from jamie_b200 import pca_fit
    X = _data(n, d, max(k + 4, 20), n + d)
    ref = PCA(n_components=k, svd_solver=solver, random_state=0)
    sample_ref = ref.fit_transform(X)
    eng = _engine()
    pca, sample = pca_fit.fit_transform(eng, X, k)
    eng.close()
    tol = 2e-3 if solver == 'randomized' else 2e-5            # the randomized solver is itself approximate
    np.testing.assert_allclose(pca.mean_, ref.mean_, rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(pca.explained_variance_, ref.explained_variance_, rtol=tol)
    np.testing.assert_allclose(pca.explained_variance_ratio_, ref.explained_variance_ratio_, rtol=tol, atol=1e-9)
    np.testing.assert_allclose(pca.singular_values_, ref.singular_values_, rtol=tol)
    # components: same vectors with the same sign convention (v-based svd_flip)
    cos = np.abs(np.sum(pca.components_ * ref.components_, axis=1))
    assert cos.min() > 1 - tol, cos.min()
    assert np.all(np.sum(pca.components_ * ref.components_, axis=1) > 0)
    scale = np.abs(sample_ref).max()
    assert np.abs(sample - sample_ref).max() < (50 * tol) * scale
    # the returned object is a genuine, usable sklearn PCA
    assert isinstance(pca, PCA)
    np.testing.assert_allclose(pca.transform(X[:7]), ref.transform(X[:7]), atol=(50 * tol) * scale)
    np.testing.assert_allclose(pca.inverse_transform(pca.transform(X[:7])), ref.inverse_transform(ref.transform(X[:7])),
                               atol=(50 * tol) * np.abs(X).max())


def test_gram_is_fp32_class_and_row_sharding_adds_up():
    """the Gram matrix against float64 numpy, and two half-shards (what two data-parallel ranks compute before their
    all-reduce) against the whole"""
    X = _data(5000, 96, 24, 3).astype(np.float32)
    eng = _engine()
    cs = eng.pca_colsum(X)
    np.testing.assert_allclose(cs, X.astype(np.float64).sum(0), rtol=1e-12, atol=1e-9)
    mean = cs / X.shape[0]
    G = eng.pca_gram(X, mean)
    Xc = X.astype(np.float64) - mean.astype(np.float32).astype(np.float64)
    want = Xc.T @ Xc
    assert np.abs(G - want).max() < 3e-6 * np.abs(want).max()
    G2 = eng.pca_gram(X[:2500], mean) + eng.pca_gram(X[2500:], mean)
    assert np.abs(G2 - want).max() < 3e-6 * np.abs(want).max()
    eng.close()


def test_fit_transform_uses_the_gpu_pca_fit_and_matches_the_host_fit():
    """JAMIE(pca_dim=...) end to end: same embeddings whether the PCA was fitted through the GPU Gram route or by the
    reference's sklearn call (same seeds; the fits agree to fp32 rounding, so do the trained models' inputs)."""
    from jamie import JAMIE
    data = [_data(300, 90, 24, 4), _data(300, 70, 24, 5)]     # separated spectra: the two fits pick the same basis
    pres = {}
    for how in ('gpu', 'sklearn'):
        np.random.seed(1)
        jm = JAMIE(output_dim=8, batch_size=64, pca_dim=[20, 16], epoch_DNN=3, min_epochs=1, use_f_tilde=False, manual_seed=5,
                   pca_fit=how)
        jm.fit_transform(dataset=[d.copy() for d in data])
        pres[how] = [np.asarray(jm.dataset[i]) for i in range(2)], [jm.model.preprocessing[i].__self__.pca for i in range(2)]
        jm.engine.close()
    from sklearn.decomposition import PCA
    for i in range(2):
        assert isinstance(pres['gpu'][1][i], PCA)
        np.testing.assert_allclose(pres['gpu'][0][i], pres['sklearn'][0][i], atol=2e-3)


def test_sparse_input_matches_dense_through_the_api():
    """AnnData-style scipy.sparse matrices: PCA fit and projection run block-wise (16 k densified rows at a time) and give
    what the dense matrices give."""
    import scipy.sparse as sp
    from jamie import JAMIE
    rng = np.random.default_rng(8)
    data = []
    for d, seed in ((90, 4), (70, 5)):
        X = _data(300, d, 24, seed)
        X[np.abs(X - X.mean(0)) < 0.4 * X.std(0)] = 0.0          # make it sparse-ish (structure survives)
        data.append(X.astype(np.float32).astype(np.float64))
    outs = {}
    for how in ('dense', 'sparse'):
        np.random.seed(1)
        jm = JAMIE(output_dim=8, batch_size=64, pca_dim=[20, 16], epoch_DNN=3, min_epochs=1, use_f_tilde=False, manual_seed=5)
        emb = jm.fit_transform(dataset=[(sp.csr_matrix(d) if how == 'sparse' else d.copy()) for d in data])
        outs[how] = [np.asarray(jm.dataset[i]) for i in range(2)], emb, jm.modal_predict(sp.csr_matrix(data[0]) if how == 'sparse' else data[0], 0)
        jm.engine.close()
    for i in range(2):
        np.testing.assert_allclose(outs['sparse'][0][i], outs['dense'][0][i], atol=1e-5)
        np.testing.assert_allclose(outs['sparse'][1][i], outs['dense'][1][i], atol=1e-4)
    np.testing.assert_allclose(outs['sparse'][2], outs['dense'][2], atol=1e-3)
