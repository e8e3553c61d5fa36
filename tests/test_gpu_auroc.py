"""imputation_auroc on the GPU (jb_metric_feature_auroc, csrc/auroc.cuh): the device's 2U and P equal the integers of the
float64 reference (tests/auroc_oracle.py) on both sides of the shared-memory regime, AUROC equals sklearn's
roc_auc_score, sparse measured equals dense, results are bit-identical across reruns and batch splits, the memory
refusal, and a trained model's modal_predict scored end to end."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp
from sklearn.metrics import roc_auc_score

from tests import auroc_oracle as A

pytestmark = pytest.mark.gpu

RATES = [0.001, 0.01, 0.05, 0.2, 0.5, 0.8, 0.95, 0.99]


def _scores(kind, n, d, rng):
    if kind == 'continuous':
        return rng.standard_normal((n, d), dtype=np.float32)
    if kind == 'ties':
        return (rng.integers(-3, 4, (n, d)) * 0.5).astype(np.float32)
    if kind == 'signed_zeros':
        return rng.choice(np.array([-0.0, 0.0, -0.0, 1.0, -1.0], np.float32), (n, d))
    if kind == 'large':
        vals = np.array([-3.4e38, -1e30, -1e-30, -1e-45, -0.0, 0.0, 1e-45, 1e-38, 1e30, 3.4e38], np.float32)
        S = rng.choice(vals, (n, d))
        return np.where(rng.random((n, d)) < 0.5, S, rng.standard_normal((n, d), dtype=np.float32) * np.float32(1e37))
    raise ValueError(kind)


def _measured(n, d, rng):
    """Positive rates from 0.1 % to 99 % across the columns, positives > 0 and negatives 0; column 0 has no positives and
    column 1 no negatives."""
    rate = np.array(RATES)[np.arange(d) % len(RATES)]
    M = np.where(rng.random((n, d)) < rate, rng.random((n, d)) + 0.5, 0.0)
    M[:, 0] = 0.0
    if d > 1:
        M[:, 1] = 1.0
    return M


def _device_counts(scores, measured, batch_bytes=1 << 30):
    """(u2, n_pos) straight from jb_metric_feature_auroc."""
    from jamie_b200 import _lib, evaluation
    S = np.ascontiguousarray(scores, np.float32)
    ptr, rows = evaluation.positive_lists(measured, 0.0, batch_bytes)
    n, d = S.shape
    u2, n_pos = np.empty(d, np.uint64), np.empty(d, np.int64)
    p = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
    lib = _lib.load()
    _lib.check(lib.jb_metric_feature_auroc(p(S), n, d, p(ptr), p(rows), batch_bytes, 0, p(u2), p(n_pos)))
    return u2, n_pos


SHAPES = [(2, 16), (60, 64), (4301, 300), (70000, 8)]   # 70 000 rows: above the shared-memory regime (26 624)
KINDS = ['continuous', 'ties', 'signed_zeros', 'large']


@pytest.mark.parametrize('kind', KINDS)
@pytest.mark.parametrize('shape', SHAPES, ids=[f'{n}x{d}' for n, d in SHAPES])
def test_device_integers_equal_the_reference(shape, kind):
    n, d = shape
    rng = np.random.default_rng(n + d)
    S, M = _scores(kind, n, d, rng), _measured(n, d, rng)
    u2, n_pos = _device_counts(S, M)
    ru2, rpos, _ = A.imputation_auroc(S, M)
    np.testing.assert_array_equal(n_pos, rpos)
    np.testing.assert_array_equal(u2, ru2)


def test_wide_batches_equal_the_reference():
    rng = np.random.default_rng(11)
    n, d = 4301, 3000
    S, M = _scores('ties', n, d, rng), _measured(n, d, rng)
    u2, n_pos = _device_counts(S, M, batch_bytes=64 << 20)   # several column batches
    ru2, rpos, _ = A.imputation_auroc(S, M)
    np.testing.assert_array_equal(n_pos, rpos)
    np.testing.assert_array_equal(u2, ru2)


@pytest.mark.parametrize('n', [60, 4301, 70000])
def test_auroc_matches_sklearn(n):
    from jamie_b200.evaluation import imputation_auroc
    rng = np.random.default_rng(n)
    d = 24
    S = np.where(rng.random((n, d)) < 0.5, _scores('continuous', n, d, rng), _scores('ties', n, d, rng))
    M = _measured(n, d, rng)
    got = imputation_auroc(S.astype(np.float64), M)
    for j in range(d):
        y = M[:, j] > 0
        if 0 < y.sum() < n:
            assert abs(got[j] - roc_auc_score(y, S[:, j])) <= 1e-12, j
        else:
            assert np.isnan(got[j]), j
    assert np.isnan(got[0]) and np.isnan(got[1])


@pytest.mark.parametrize('fmt', [sp.csr_matrix, sp.csc_matrix])
def test_sparse_measured_equals_dense(fmt):
    from jamie_b200.evaluation import imputation_auroc
    rng = np.random.default_rng(5)
    n, d = 4301, 400
    S = _scores('continuous', n, d, rng)
    M = np.where(rng.random((n, d)) < 0.05, rng.random((n, d)) + 0.1, 0.0)
    M[rng.random((n, d)) < 0.01] = -0.5                    # stored values that are negatives
    np.testing.assert_array_equal(imputation_auroc(S, fmt(M)), imputation_auroc(S, M))


@pytest.mark.parametrize('n', [4301, 70000])
def test_bit_identical_reruns_and_batches(n, monkeypatch):
    from jamie_b200 import evaluation
    rng = np.random.default_rng(9)
    d = 64 if n < 10000 else 12
    S, M = _scores('ties', n, d, rng), _measured(n, d, rng)
    ref = evaluation.imputation_auroc(S, M)
    again = evaluation.imputation_auroc(S, M)
    ref_u2 = _device_counts(S, M)[0]
    monkeypatch.setattr(evaluation, 'BATCH_BYTES', 1)     # one column per batch
    small = evaluation.imputation_auroc(S, M)
    np.testing.assert_array_equal(_device_counts(S, M, batch_bytes=24 * n * 5)[0], ref_u2)
    for other in (again, small):
        np.testing.assert_array_equal(other, ref)


def test_refuses_a_problem_larger_than_free_memory():
    import torch
    from jamie_b200 import _lib, evaluation
    lib = _lib.load()
    z = np.zeros(16)
    u2, n_pos = np.zeros(4, np.uint64), np.zeros(4, np.int64)
    p = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
    free0 = torch.cuda.mem_get_info()[0]
    d = 1 << 40                                   # the per-column outputs alone: 16 TB
    rc = lib.jb_metric_feature_auroc(p(z), 4301, d, p(z), None, 1 << 30, 0, p(u2), p(n_pos))
    assert rc != 0
    msg = lib.jb_last_error().decode()
    assert 'GB' in msg and 'free' in msg, msg
    assert abs(torch.cuda.mem_get_info()[0] - free0) < (64 << 20)
    rng = np.random.default_rng(0)
    S, M = _scores('continuous', 100, 8, rng), _measured(100, 8, rng)
    np.testing.assert_array_equal(evaluation.imputation_auroc(S, M), A.imputation_auroc(S, M)[2])


def test_end_to_end_modal_predict():
    from jamie import JAMIE
    from jamie.evaluation import imputation_auroc
    np.random.seed(1)
    rng = np.random.default_rng(0)
    n, dims = 300, (90, 40)
    Zs = rng.normal(size=(n, 6))
    data = [(Zs @ rng.normal(size=(6, dims[i])) + 0.3 * rng.normal(size=(n, dims[i])) + rng.normal(size=dims[i]))
            .astype(np.float32) for i in range(2)]
    jm = JAMIE(output_dim=8, batch_size=64, pca_dim=[20, 16], epoch_DNN=20, min_epochs=1, use_f_tilde=False, manual_seed=5)
    jm.fit_transform(dataset=[x.copy() for x in data])
    try:
        imputed = jm.modal_predict(data[0], 0)
        measured = data[1]
        got = imputation_auroc(imputed, measured)
        want = np.array([roc_auc_score(measured[:, j] > 0, np.float32(imputed[:, j])) if 0 < (measured[:, j] > 0).sum() < n
                         else np.nan for j in range(dims[1])])
        assert np.isfinite(want).sum() > 10
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-12)
    finally:
        jm.engine.close()
