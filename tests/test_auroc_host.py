"""CPU tests of imputation_auroc: the float64 reference (tests/auroc_oracle.py) against sklearn's roc_auc_score and exact
rational arithmetic, and the host driver (jamie_b200/evaluation.py: labels, positive lists, batching, refusals) with a numpy
stand-in for jb_metric_feature_auroc."""
import ctypes as C
from fractions import Fraction

import numpy as np
import pytest
import scipy.sparse as sp
from sklearn.metrics import roc_auc_score

from jamie_b200 import _lib, evaluation
from tests import auroc_oracle as A


def _scores(kind, n, d, rng):
    if kind == 'continuous':
        return rng.standard_normal((n, d))
    if kind == 'ties':
        return rng.integers(-2, 3, (n, d)) * 0.25
    if kind == 'signed_zeros':
        return rng.choice([-0.0, 0.0, -1.5, 1.5, -3.0], (n, d))
    if kind == 'constant':
        return np.full((n, d), 0.7)
    raise ValueError(kind)


def _labels(n, d, rng):
    rates = np.array([0.02, 0.1, 0.5, 0.9, 0.98])[np.arange(d) % 5]
    return rng.random((n, d)) < rates


@pytest.mark.parametrize('kind', ['continuous', 'ties', 'signed_zeros', 'constant'])
@pytest.mark.parametrize('n', [2, 7, 60, 500])
def test_oracle_matches_roc_auc_score(kind, n):
    rng = np.random.default_rng(n)
    s, y = _scores(kind, n, 30, rng), _labels(n, 30, rng)
    u2, n_pos, auc = A.imputation_auroc(s, y.astype(np.float64), threshold=0.5)
    np.testing.assert_array_equal(n_pos, y.sum(0))
    for j in range(s.shape[1]):
        if 0 < n_pos[j] < n:
            assert abs(auc[j] - roc_auc_score(y[:, j], s[:, j].astype(np.float32))) <= 1e-12
            if kind == 'constant':
                assert auc[j] == 0.5
        else:
            assert np.isnan(auc[j])


def test_oracle_perfect_separation_and_n2():
    s = np.array([[0.1, 0.9], [0.9, 0.1]])
    y = np.array([[0.0, 0.0], [1.0, 1.0]])
    u2, n_pos, auc = A.imputation_auroc(s, y)
    np.testing.assert_array_equal(auc, [1.0, 0.0])
    np.testing.assert_array_equal(u2, [2, 0])
    np.testing.assert_array_equal(n_pos, [1, 1])
    s = np.array([[-0.0], [0.0]])                     # one score: 0.5
    assert A.imputation_auroc(s, np.array([[1.0], [0.0]]))[2][0] == 0.5


@pytest.mark.parametrize('kind', ['continuous', 'ties', 'signed_zeros'])
def test_oracle_u2_against_fractions(kind):
    rng = np.random.default_rng(3)
    n = 40
    s, y = _scores(kind, n, 12, rng).astype(np.float32), _labels(n, 12, rng)
    u2, n_pos, auc = A.imputation_auroc(s, y.astype(np.float64), threshold=0.5)
    for j in range(s.shape[1]):
        P = int(y[:, j].sum())
        pos, neg = s[y[:, j], j], s[~y[:, j], j]
        if not 0 < P < n:
            assert int(u2[j]) == 0 and np.isnan(auc[j])
            continue
        half = Fraction(1, 2)
        exact = sum(Fraction(1) if a > b else half if a == b else Fraction(0) for a in pos for b in neg) / (P * (n - P))
        assert Fraction(int(u2[j]), 2 * P * (n - P)) == exact
        assert auc[j] == float(exact)


class StandIn:
    """Numpy jb_metric_feature_auroc: reads the arguments through their pointers, splits the columns into batches as the
    engine does, and computes 2U and P with the reference from the positive lists."""

    def __init__(self):
        self.calls = []

    def jb_metric_feature_auroc(self, scores, n, d, ptr, rows, batch_bytes, device, u2, n_pos):
        def arr(p, ct, size):
            return np.ctypeslib.as_array(C.cast(p, C.POINTER(ct)), (size,)) if size else np.zeros(0)
        S = arr(scores, C.c_float, n * d).reshape(n, d)
        ptr_a = arr(ptr, C.c_longlong, d + 1).copy()
        rows_a = arr(rows, C.c_int, int(ptr_a[-1])).copy()
        out_u2, out_np = arr(u2, C.c_ulonglong, d), arr(n_pos, C.c_longlong, d)
        self.calls.append(dict(ptr=ptr_a, rows=rows_a, n=n, d=d, batch_bytes=batch_bytes))
        w = max(1, min(d, int(batch_bytes // (16 * n))))
        for j0 in range(0, d, w):
            for j in range(j0, min(d, j0 + w)):
                y = np.zeros(n, bool)
                y[rows_a[ptr_a[j]:ptr_a[j + 1]]] = True
                out_u2[j] = A.u2_of(S[:, j], y)
                out_np[j] = ptr_a[j + 1] - ptr_a[j]
        return 0


@pytest.fixture
def stand_in(monkeypatch):
    lib = StandIn()
    monkeypatch.setattr(_lib, 'load', lambda: lib)
    return lib


def _problem(n=90, d=23, seed=0, density=0.3):
    rng = np.random.default_rng(seed)
    imputed = rng.standard_normal((n, d)).astype(np.float32).astype(np.float64)
    imputed[:, 3] = np.round(imputed[:, 3])                          # ties
    vals = rng.random((n, d)) * 2.0
    measured = np.where(rng.random((n, d)) < density, vals, 0.0)
    measured[:, 5] = 0.0                                             # no positives
    measured[:, 6] = 1.0 + vals[:, 6]                                # no negatives
    return imputed, measured


def test_driver_matches_the_reference_and_sklearn(stand_in):
    imputed, measured = _problem()
    got = evaluation.imputation_auroc(imputed, measured, device=0)
    u2, n_pos, want = A.imputation_auroc(imputed, measured)
    np.testing.assert_array_equal(got, want)
    assert np.isnan(got[5]) and np.isnan(got[6]) and np.isfinite(np.delete(got, [5, 6])).all()
    for j in np.flatnonzero(np.isfinite(want)):
        assert abs(got[j] - roc_auc_score(measured[:, j] > 0, imputed[:, j])) <= 1e-12
    assert len(stand_in.calls) == 1 and stand_in.calls[0]['batch_bytes'] == evaluation.BATCH_BYTES


def test_positive_lists_identical_for_dense_and_sparse_formats(stand_in):
    imputed, measured = _problem(seed=1, density=0.05)
    measured[2, 0] = -1.0                                            # a stored negative value
    results = [evaluation.imputation_auroc(imputed, fmt(measured), device=0)
               for fmt in (np.asarray, sp.csr_matrix, sp.csc_matrix, sp.coo_matrix)]
    ref = stand_in.calls[0]
    for call, res in zip(stand_in.calls[1:], results[1:]):
        np.testing.assert_array_equal(call['ptr'], ref['ptr'])
        np.testing.assert_array_equal(call['rows'], ref['rows'])
        np.testing.assert_array_equal(res, results[0])
    assert ref['rows'].dtype == np.int32 and ref['ptr'].dtype == np.int64


def test_sparse_duplicates_and_explicit_zeros():
    rows, cols = np.array([0, 0, 3, 2, 2]), np.array([1, 1, 0, 0, 2])
    vals = np.array([0.4, 0.4, 0.0, 0.5, -0.5])                     # (0, 1) sums to 0.8; (2, 2) is stored, negative
    M = sp.coo_matrix((vals, (rows, cols)), shape=(5, 3))
    ptr, r = evaluation.positive_lists(M, 0.0, evaluation.BATCH_BYTES)
    ptr_d, r_d = evaluation.positive_lists(M.toarray(), 0.0, evaluation.BATCH_BYTES)
    np.testing.assert_array_equal(ptr, [0, 1, 2, 2])
    np.testing.assert_array_equal(r, [2, 0])
    np.testing.assert_array_equal(ptr, ptr_d)
    np.testing.assert_array_equal(r, r_d)
    ptr, r = evaluation.positive_lists(M, 0.45, evaluation.BATCH_BYTES)
    np.testing.assert_array_equal(ptr, [0, 1, 2, 2])


def test_threshold_semantics(stand_in):
    imputed, measured = _problem(seed=2)
    measured = np.round(measured, 1)
    for thr in (0.0, 0.5, 1.0, -0.25):                               # labels are measured > threshold, strictly
        got = evaluation.imputation_auroc(imputed, measured, threshold=thr, device=0)
        np.testing.assert_array_equal(got, A.imputation_auroc(imputed, measured, thr)[2])
        lab = measured > thr
        np.testing.assert_array_equal(np.diff(stand_in.calls[-1]['ptr']), lab.sum(0))
        if thr >= 0:
            np.testing.assert_array_equal(evaluation.imputation_auroc(imputed, sp.csr_matrix(measured), thr, device=0), got)
    # the comparison is in measured's own dtype: no rounding of measured before it
    m32 = np.full((4, 1), np.float32(0.1))
    m32[0, 0] = 0.0
    ptr, _ = evaluation.positive_lists(m32, 0.1, evaluation.BATCH_BYTES)
    assert ptr[-1] == int((m32 > 0.1).sum())
    ptr, _ = evaluation.positive_lists(m32.astype(np.float64), 0.1, evaluation.BATCH_BYTES)
    assert ptr[-1] == 3                                              # float64(float32(0.1)) > 0.1


@pytest.mark.parametrize('batch_bytes', [1, 4 * 90 * 3, 4 * 90 * 7 + 5, 1 << 30])
def test_batching_gives_the_same_lists_and_result(stand_in, monkeypatch, batch_bytes):
    imputed, measured = _problem(seed=4)
    ref = evaluation.imputation_auroc(imputed, measured, device=0)
    ref_call = stand_in.calls[-1]
    monkeypatch.setattr(evaluation, 'BATCH_BYTES', batch_bytes)
    got = evaluation.imputation_auroc(imputed, measured, device=0)
    np.testing.assert_array_equal(got, ref)
    np.testing.assert_array_equal(stand_in.calls[-1]['ptr'], ref_call['ptr'])
    np.testing.assert_array_equal(stand_in.calls[-1]['rows'], ref_call['rows'])
    assert stand_in.calls[-1]['batch_bytes'] == batch_bytes


def _bad_inputs():
    imputed, measured = _problem(n=12, d=8)
    nan_imp = imputed.copy()
    nan_imp[1, 2] = np.nan
    inf_meas = measured.copy()
    inf_meas[0, 0] = np.inf
    big = imputed.copy()
    big[0, 0] = 1e300                                                # finite in float64, inf in float32
    huge = np.broadcast_to(np.zeros((1, 1), np.float32), (1 << 31, 1))
    sp_nan = sp.csr_matrix(measured)
    sp_nan.data[0] = np.nan
    return [
        ((imputed, measured[:, :3]), {}, 'shape'),
        ((imputed[0], measured[0]), {}, 'shape'),
        ((sp.csr_matrix(imputed), measured), {}, 'dense'),
        ((nan_imp, measured), {}, 'non-finite'),
        ((big, measured), {}, 'non-finite'),
        ((imputed, inf_meas), {}, 'non-finite'),
        ((imputed, sp_nan), {}, 'non-finite'),
        ((imputed, measured), {'threshold': [0.0, 1.0]}, 'scalar'),
        ((imputed, measured), {'threshold': np.nan}, 'finite'),
        ((imputed, measured), {'threshold': 'zero'}, 'finite'),
        ((imputed, sp.csc_matrix(measured)), {'threshold': -0.5}, 'dense array'),
        ((huge, huge), {}, r'2\^31'),
        ((imputed[:0], measured[:0]), {}, 'one row'),
    ]


@pytest.mark.parametrize('case', range(len(_bad_inputs())))
def test_refusals_before_any_device_work(stand_in, case):
    args, kw, match = _bad_inputs()[case]
    with pytest.raises(ValueError, match=match):
        evaluation.imputation_auroc(*args, device=0, **kw)
    assert stand_in.calls == []


def test_reexported_by_the_reference_package():
    import jamie.evaluation
    assert jamie.evaluation.imputation_auroc is evaluation.imputation_auroc
