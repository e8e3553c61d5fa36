"""JAMIE.shap_values on the GPU (jb_shapley, csrc/shapley.cuh) against the estimator run through modal_predict one masked
batch at a time (naive_shap_values) with the same permutations, against exact Shapley values by coalition enumeration,
and against transform_one for space='latent'. Also efficiency, bit-identical reruns, batch splits and sparse input, and
the memory refusal."""
import ctypes as C
import itertools
import math

import numpy as np
import pytest
import scipy.sparse as sp

from tests.test_gpu_impact import SIDES, _norm_rel, _train

pytestmark = pytest.mark.gpu

EVAL_RTOL = 2e-3   # test_gpu_impact.py: the fp16 chain sees inputs that differ by fp32 rounding


@pytest.fixture(scope='module', params=list(SIDES))
def trained(request):
    jm, data = _train(SIDES[request.param])
    yield jm, data
    jm.engine.close()


def _predict(jm, O, latent=False):
    if latent:
        return lambda A: np.asarray(jm.transform_one(A, 0), np.float64)[:, O]
    return lambda A: np.asarray(jm.modal_predict(A, 0), np.float64)[:, O]


def test_output_space_matches_the_naive_estimator(trained):
    from jamie_b200 import shapley
    jm, (X, T) = trained
    O = np.array([0, 3, 7, 11, 25, 39])
    perms = shapley.draw_permutations(X.shape[1], 2, 7)
    got = shapley.shap_values(jm, X[:3], 0, X[100:120], outputs=O, perms=perms)
    values, base = shapley.naive_shap_values(_predict(jm, O), X[:3], X[100:120], perms)
    assert got.values.shape == (3, X.shape[1], len(O)) and np.array_equal(got.outputs, O)
    assert _norm_rel(got.values, values) < EVAL_RTOL
    assert _norm_rel(got.base_values, base) < 1e-5
    # the public call draws the same antithetic pairs from manual_seed
    pub = jm.shap_values(X[:3], 0, X[100:120], outputs=O, seed=7)
    np.testing.assert_array_equal(pub.values, got.values)


def test_efficiency_against_modal_predict(trained):
    jm, (X, T) = trained
    O = np.arange(T.shape[1])
    got = jm.shap_values(X[:5], 0, X[200:230], n_permutations=4)
    f = _predict(jm, O)
    want = f(X[:5]) - f(X[200:230]).mean(0)
    assert _norm_rel(got.values.sum(1), want) < EVAL_RTOL
    assert _norm_rel(got.base_values, f(X[200:230]).mean(0)) < 1e-5


def test_all_orders_give_exact_shapley_values(trained):
    from jamie_b200 import shapley
    jm, (X, T) = trained
    rng = np.random.default_rng(3)
    A = [2, 9, 17, 30, 51, 77]
    B = np.repeat(X[:1], 8, axis=0).astype(np.float64)
    B[:, A] += rng.normal(size=(8, len(A)))
    x = X[0].astype(np.float64)
    x[A] += rng.normal(size=len(A))
    base = rng.permutation(X.shape[1])
    slots = np.flatnonzero(np.isin(base, A))
    perms = []
    for order in itertools.permutations(A):
        p = base.copy()
        p[slots] = order
        perms.append(p)
    O = np.array([1, 4, 9, 20])
    got = shapley.shap_values(jm, x[None], 0, B, outputs=O, perms=np.array(perms))
    # exact: every coalition S of A, v(S) = mean over b of f(x on S, b elsewhere), through one modal_predict call
    coal = [S for r in range(7) for S in itertools.combinations(range(6), r)]
    M = np.concatenate([np.where(np.isin(np.arange(X.shape[1]), [A[q] for q in S])[None, :], x[None, :], B) for S in coal])
    v = dict(zip(coal, _predict(jm, O)(M).reshape(len(coal), 8, len(O)).mean(1)))
    exact = np.zeros((6, len(O)))
    for q in range(6):
        for S in coal:
            if q not in S:
                wt = math.factorial(len(S)) * math.factorial(5 - len(S)) / math.factorial(6)
                exact[q] += wt * (v[tuple(sorted(S + (q,)))] - v[S])
    assert _norm_rel(got.values[0, A], exact) < EVAL_RTOL
    assert np.all(np.delete(got.values[0], A, axis=0) == 0.0)


def test_latent_space_matches_transform_one(trained):
    from jamie_b200 import shapley
    jm, (X, T) = trained
    O = np.array([0, 2, 5])
    perms = shapley.draw_permutations(X.shape[1], 2, 1)
    got = shapley.shap_values(jm, X[10:12], 0, X[50:60], outputs=O, space='latent', perms=perms)
    values, base = shapley.naive_shap_values(_predict(jm, O, latent=True), X[10:12], X[50:60], perms)
    assert got.values.shape == (2, X.shape[1], 3)
    assert _norm_rel(got.values, values) < EVAL_RTOL
    assert _norm_rel(got.base_values, base) < 1e-5


def test_bit_identical_reruns_batches_and_sparse(trained, monkeypatch):
    from jamie_b200 import shapley
    jm, (X, T) = trained
    Xs = X.copy()
    Xs[np.abs(Xs) < 0.5] = 0.0
    Xs[:, 7] = 0.0                                     # a dummy feature: equal in every explained and background row
    args = (Xs[:4], 0, Xs[60:76])
    ref = jm.shap_values(*args, outputs=[0, 5, 6])
    again = jm.shap_values(*args, outputs=[0, 5, 6])
    sparse = jm.shap_values(sp.csr_matrix(Xs[:4]), 0, sp.csr_matrix(Xs[60:76]), outputs=[0, 5, 6])
    monkeypatch.setattr(shapley, 'BATCH_BYTES', 1)     # one segment per batch
    small = jm.shap_values(*args, outputs=[0, 5, 6])
    for other in (again, sparse, small):
        np.testing.assert_array_equal(other.values, ref.values)
        np.testing.assert_array_equal(other.base_values, ref.base_values)
    assert np.isfinite(ref.values).all() and np.all(ref.values[:, 7] == 0.0)


def test_refuses_a_problem_larger_than_free_memory(trained):
    import torch
    from jamie_b200 import _lib
    jm, (X, T) = trained
    eng = jm._ensure_engine()
    lib = _lib.load()
    z = np.zeros(16)
    perm = np.arange(16, dtype=np.int32)
    oc = np.zeros(1, np.int32)
    p = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
    free0 = torch.cuda.mem_get_info()[0]
    nx = 1 << 30                                       # the explained rows alone: 2^30 x 90 float64
    rc = lib.jb_shapley(eng.h, 0, 1, p(z), nx, p(z), 1, X.shape[1], p(z), p(perm), 1, p(z), None, 0, None, None, 0.0, 1.0,
                        None, None, p(oc), 1, p(z), p(z), None, 1 << 30, None)
    assert rc != 0
    msg = lib.jb_last_error().decode()
    assert 'GB' in msg and 'free' in msg, msg
    assert abs(torch.cuda.mem_get_info()[0] - free0) < (64 << 20)
    got = jm.shap_values(X[:1], 0, X[5:9], outputs=[0])    # the engine still works
    assert np.isfinite(got.values).all()
