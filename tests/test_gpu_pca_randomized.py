"""Randomized PCA fit on the GPU (the jb_pcaop handle, csrc/pcaop.cuh; jamie_b200/pca_fit.py randomized_fit_transform):
the operand products and column statistics against float64 numpy, the fit against sklearn's exact PCA and against the
float64 host stand-in with the same seed, a wide sparse input out of the Gram route's reach, and JAMIE end to end."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

from tests.test_pca_randomized_host import NumpyOperator, _data, _sparse_data, check_against_exact

pytestmark = pytest.mark.gpu


def _operand_data(n, d, seed, density):
    """non-zero means, an empty row (3), an all-zero column (7), a column stored in every row (5: with n > 4096 its CSC
    row is cut into segments)"""
    rng = np.random.default_rng(seed)
    X = (rng.normal(size=(n, d)) + rng.normal(size=d) * 3) * (rng.random((n, d)) < density)
    X[:, 5] = rng.normal(size=n) + 2.0
    X[3, :] = 0.0
    X[:, 7] = 0.0
    return X.astype(np.float32)


def _op(X):
    from jamie_b200 import pca_fit
    return pca_fit.DeviceOperator(X, 0)


@pytest.mark.parametrize('kind,n,d,density', [('sparse', 5000, 203, 0.05), ('sparse', 301, 1030, 0.3),
                                              ('dense', 517, 203, 1.0), ('dense', 300, 9001, 1.0)])
def test_apply_and_stats_match_float64(kind, n, d, density):
    import torch
    X = _operand_data(n, d, n + d, density)
    op = _op(sp.csr_matrix(X) if kind == 'sparse' else X)
    try:
        mean, var = op.stats()
        X64 = X.astype(np.float64)
        want_mean, want_var = X64.mean(0), X64.var(0)
        np.testing.assert_allclose(mean, want_mean, rtol=1e-12, atol=1e-12 * np.abs(want_mean).max())
        np.testing.assert_allclose(var, want_var, rtol=1e-12, atol=1e-12 * want_var.max())
        assert var[7] == 0.0 and mean[7] == 0.0
        # the dense planes are centred with the fp32 mean (k_split_tf32); the sparse correction uses the float64 mean
        Xc = X64 - (mean.astype(np.float32).astype(np.float64) if kind == 'dense' else mean)
        tol = 1e-6 if kind == 'sparse' else 1e-5
        rng = np.random.default_rng(1)
        for l in (7, 37):
            for trans in (0, 1):
                B = rng.normal(size=(n if trans else d, l)).astype(np.float32)
                want = (Xc.T if trans else Xc) @ B.astype(np.float64)
                Bd = op.upload(B)
                Y = op.apply(trans, Bd)
                Y2 = op.apply(trans, Bd)
                torch.cuda.synchronize()
                got = Y.cpu().numpy()
                assert got.shape == want.shape
                err = np.abs(got - want).max() / np.abs(want).max()
                assert err <= tol, (l, trans, err)
                assert torch.equal(Y, Y2)                       # bit-reproducible
    finally:
        op.close()


@pytest.mark.parametrize('n,d,k,kind', [(400, 60, 12, 'dense'), (90, 300, 10, 'dense'), (300, 120, 16, 'sparse'),
                                        (80, 260, 12, 'sparse'), (2000, 700, 40, 'dense')])
def test_fit_matches_exact_pca_and_the_host_stand_in(n, d, k, kind):
    from jamie_b200 import pca_fit
    r = max(k + 4, 20)
    X = _sparse_data(n, d, r, n + d) if kind == 'sparse' else _data(n, d, r, n + d)
    pca, sample = pca_fit.randomized_fit_transform(X, k, seed=11, device=0)
    check_against_exact(X, k, pca, sample, 1e-6, 1e-4, 1e-4, noise_rtol=1e-3)   # noise: a difference of near totals
    host, host_sample = pca_fit.randomized_fit_transform(X, k, seed=11, device=0, operator=NumpyOperator)
    assert np.sum(pca.components_ * host.components_, axis=1).min() > 1 - 1e-6
    np.testing.assert_allclose(pca.explained_variance_, host.explained_variance_, rtol=1e-4)
    assert np.abs(sample - host_sample).max() < 1e-4 * np.abs(host_sample).max()
    again, again_sample = pca_fit.randomized_fit_transform(X, k, seed=11, device=0)
    np.testing.assert_array_equal(again.components_, pca.components_)
    np.testing.assert_array_equal(again_sample, sample)


def test_wide_sparse_fit_beyond_the_gram_route():
    """3 000 x 60 000 sparse: the Gram route would need a 60 000 x 60 000 eigensolve; checked against the exact SVD
    through the n x n kernel matrix Xc Xc^T"""
    from jamie_b200 import pca_fit
    n, d, r, k = 3000, 60000, 40, 32
    rng = np.random.default_rng(21)
    lat = sp.random(n, r, density=0.1, random_state=1, data_rvs=rng.standard_normal).tocsr() @ sp.diags(np.linspace(3.0, 0.5, r))
    W = sp.random(r, d, density=0.01, random_state=2, data_rvs=rng.standard_normal).tocsr()
    X = (lat @ W).tocsr()
    X.data += 0.05 * rng.normal(size=X.nnz)
    X = X.astype(np.float32).astype(np.float64)
    assert 0.002 < X.nnz / (n * d) < 0.05
    pca, sample = pca_fit.randomized_fit_transform(X, k, seed=0, device=0)
    mu = np.asarray(X.mean(axis=0)).ravel()
    Xm = np.asarray(X @ mu).ravel()
    G = (X @ X.T).toarray() - Xm[:, None] - Xm[None, :] + mu @ mu            # Xc Xc^T
    lam, U = np.linalg.eigh((G + G.T) / 2)
    lam, U = lam[::-1][:k], U[:, ::-1][:, :k]
    S = np.sqrt(lam)
    V = (np.asarray(X.T @ U) - np.outer(mu, U.sum(0))) / S                   # components (columns)
    np.testing.assert_allclose(pca.explained_variance_, lam / (n - 1), rtol=1e-4)
    cos = np.abs(np.sum(pca.components_ * V.T, axis=1))
    assert cos.min() > 1 - 1e-6, cos.min()
    np.testing.assert_allclose(np.abs(sample), np.abs(U * S), atol=1e-4 * np.abs(U * S).max())


def test_jamie_end_to_end_dense_and_sparse_and_checkpoint(tmp_path):
    """JAMIE(pca_fit='randomized') trains on the same PCA inputs as pca_fit='sklearn' (separated spectra), with dense and
    scipy.sparse inputs, and its checkpoint loads back"""
    from jamie import JAMIE
    data = [_data(300, 90, 24, 4), _data(300, 70, 24, 5)]
    sparse = [_sparse_data(300, 90, 24, 6), _sparse_data(300, 70, 24, 7)]
    for inputs in (data, sparse):
        pres = {}
        for how in ('randomized', 'sklearn'):
            np.random.seed(1)
            jm = JAMIE(output_dim=8, batch_size=64, pca_dim=[20, 16], epoch_DNN=3, min_epochs=1, use_f_tilde=False,
                       manual_seed=5, pca_fit=how)
            # sklearn's exact fit runs on the dense copy of the same matrices
            jm.fit_transform(dataset=[x.copy() if how == 'randomized' or not sp.issparse(x) else x.toarray() for x in inputs])
            pres[how] = [np.asarray(jm.dataset[i]) for i in range(2)]
            if how == 'randomized' and inputs is sparse:
                f = str(tmp_path / 'model.h5')
                jm.save_model(f)
                jm2 = JAMIE()
                jm2.load_model(f)
                for i in range(2):
                    np.testing.assert_array_equal(jm2.modal_predict(inputs[i], i), jm.modal_predict(inputs[i], i))
                jm2.engine.close()
            jm.engine.close()
        for i in range(2):
            np.testing.assert_allclose(pres['randomized'][i], pres['sklearn'][i], atol=2e-3)


def test_create_refuses_an_operand_that_does_not_fit():
    from jamie_b200 import _lib
    lib = _lib.load()
    h = C.c_void_p()
    X = np.zeros(16, np.float32)
    n = d = 400000                                             # 640 GB fp32, three copies
    rc = lib.jb_pcaop_create_dense(X.ctypes.data_as(C.c_void_p), n, d, 0, C.byref(h))
    assert rc != 0 and not h.value
    msg = lib.jb_last_error().decode()
    assert 'GB' in msg and 'free' in msg, msg
