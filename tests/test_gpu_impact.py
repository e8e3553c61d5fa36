"""JAMIE.feature_impact on the GPU (jb_feature_impact, csrc/impact.cuh) against the loop it replaces: modal_predict of
every ablated matrix scored with imputation_correlation (or transform_one for space='latent'). Also bit-identical reruns,
batch splits and sparse input, and the memory refusal."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

pytestmark = pytest.mark.gpu

EVAL_RTOL = 2e-3   # test_gpu_eval.py: the fp16 chain sees inputs that differ by fp32 rounding
FEATURES = [0, 3, 5, 8, 13, 21, 22, 30, 34, 37, 2, 11]


def _pair(n=300, d=(90, 40), seed=0):
    rng = np.random.default_rng(seed)
    Zs = rng.normal(size=(n, 6))
    X = [(Zs @ rng.normal(size=(6, d[i])) + 0.3 * rng.normal(size=(n, d[i])) + rng.normal(size=d[i])).astype(np.float32)
         for i in range(2)]
    return X


def _train(pca_dim):
    from jamie import JAMIE
    np.random.seed(1)
    data = _pair()
    jm = JAMIE(output_dim=8, batch_size=64, pca_dim=pca_dim, epoch_DNN=20, min_epochs=1, use_f_tilde=False, manual_seed=5)
    jm.fit_transform(dataset=[x.copy() for x in data])
    return jm, data


SIDES = {'pca-pca': [20, 16], 'pca-none': [20, None], 'none-pca': [None, 16]}


@pytest.fixture(scope='module', params=list(SIDES))
def trained(request):
    jm, data = _train(SIDES[request.param])
    yield jm, data
    jm.engine.close()


def _loop(jm, X, J, target=None, latent=False):
    from jamie_b200.evaluation import imputation_correlation
    from jamie_b200.impact import naive_feature_impact
    fills = X[:, J].astype(np.float64).mean(0)
    predict = (lambda A: jm.transform_one(A, 0)) if latent else (lambda A: jm.modal_predict(A, 0))
    return naive_feature_impact(predict, X, J, fills, target, pearson=imputation_correlation)


def _norm_rel(a, b):
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


def test_output_space_matches_the_loop(trained):
    jm, (X, T) = trained
    got = jm.feature_impact(X, 0, target=T, features=FEATURES)
    shift, base_r, r = _loop(jm, X, FEATURES, T)
    np.testing.assert_allclose(got.baseline_r, base_r, rtol=0, atol=1e-6)
    np.testing.assert_allclose(got.r, r, rtol=0, atol=EVAL_RTOL)
    assert _norm_rel(got.shift, shift) < EVAL_RTOL
    assert got.shift.shape == (len(FEATURES), T.shape[1]) and np.isfinite(got.impact).all()


def test_latent_space_matches_the_loop(trained):
    jm, (X, _) = trained
    got = jm.feature_impact(X, 0, features=FEATURES, space='latent')
    shift, _, _ = _loop(jm, X, FEATURES, latent=True)
    assert got.shift.shape == (len(FEATURES), jm.model.output_dim)
    assert _norm_rel(got.shift, shift) < EVAL_RTOL
    np.testing.assert_allclose(got.impact, got.shift.mean(1))


def test_bit_identical_reruns_batches_and_sparse(trained, monkeypatch):
    from jamie_b200 import impact
    jm, (X, T) = trained
    Xs = X.copy()
    Xs[np.abs(Xs) < 0.5] = 0.0
    ref = jm.feature_impact(Xs, 0, target=T, features=FEATURES)
    again = jm.feature_impact(Xs, 0, target=T, features=FEATURES)
    sparse = jm.feature_impact(sp.csr_matrix(Xs), 0, target=T, features=FEATURES)
    monkeypatch.setattr(impact, 'BATCH_BYTES', 1)     # one feature per batch, 32-row ranges
    small = jm.feature_impact(Xs, 0, target=T, features=FEATURES)
    for other in (again, sparse, small):
        for name in ('shift', 'impact', 'baseline_r', 'r'):
            np.testing.assert_array_equal(getattr(other, name), getattr(ref, name), err_msg=name)


def test_refuses_a_problem_larger_than_free_memory(trained):
    import torch
    from jamie_b200 import _lib
    jm, (X, T) = trained
    eng = jm._ensure_engine()
    lib = _lib.load()
    Z = np.zeros(16)
    out = np.zeros(16)
    free0 = torch.cuda.mem_get_info()[0]
    n = 1 << 36                                              # Z alone: 2^36 rows x dims[0] float64
    rc = lib.jb_feature_impact(eng.h, 0, 1, Z.ctypes.data_as(C.c_void_p), n, 1, Z.ctypes.data_as(C.c_void_p),
                               Z.ctypes.data_as(C.c_void_p), None, 0, None, None, 0.0, 1.0, None, None, eng.dims[1], None,
                               None, None, out.ctypes.data_as(C.c_void_p), 1 << 30, None)
    assert rc != 0
    msg = lib.jb_last_error().decode()
    assert 'GB' in msg and 'free' in msg, msg
    assert abs(torch.cuda.mem_get_info()[0] - free0) < (64 << 20)
    got = jm.feature_impact(X, 0, features=FEATURES[:2])        # the engine still works
    assert np.isfinite(got.shift).all()
