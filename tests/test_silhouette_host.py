"""CPU tests of silhouette_samples / silhouette_score: the float64 reference (tests/silhouette_oracle.py) against
sklearn's silhouette_samples, and the host driver (jamie_b200/evaluation.py: label encoding, the sort by label and its
inverse, sklearn's finish, the sample draw, refusals) with a numpy stand-in for jb_silhouette."""
import numpy as np
import pytest
import scipy.sparse as sp
from sklearn.metrics import silhouette_samples as sk_samples
from sklearn.metrics import silhouette_score as sk_score

from jamie_b200 import evaluation
from tests import silhouette_oracle as S


class NumpySilhouette:
    """Numpy jb_silhouette: checks the sorted layout the driver hands over and computes the sums with the reference."""
    calls = []

    @classmethod
    def sums(cls, x_sorted, label_off, batch_bytes, device):
        assert x_sorted.dtype == np.float32 and x_sorted.flags.c_contiguous and x_sorted.ndim == 2
        assert label_off.dtype == np.int64 and label_off[0] == 0 and label_off[-1] == x_sorted.shape[0]
        assert np.all(np.diff(label_off) > 0) and len(label_off) >= 3
        cls.calls.append((x_sorted.copy(), label_off.copy(), batch_bytes))
        codes = np.repeat(np.arange(len(label_off) - 1), np.diff(label_off))
        return S.sums(x_sorted, codes)


def _samples(X, labels, **kw):
    return evaluation.silhouette_samples(X, labels, backend=NumpySilhouette, **kw)


def _data(kind, n, L, rng):
    if kind == 'normal':
        return rng.standard_normal((n, L))
    if kind == 'clustered':
        centres = rng.standard_normal((6, L)) * 4
        return centres[rng.integers(0, 6, n)] + rng.standard_normal((n, L)) * 0.5
    if kind == 'offset':                                    # large common offset: cancellation in |a|^2 + |b|^2 - 2ab
        return rng.standard_normal((n, L)) + 50.0
    raise ValueError(kind)


@pytest.mark.parametrize('kind', ['normal', 'clustered', 'offset'])
def test_oracle_matches_sklearn(kind):
    rng = np.random.default_rng(len(kind))
    X = _data(kind, 3000, 8, rng).astype(np.float32).astype(np.float64)   # float32 rows, as the oracle reads them
    for labels in (rng.integers(0, 2, 3000), rng.integers(0, 20, 3000)):
        np.testing.assert_allclose(S.silhouette_samples(X, labels), sk_samples(X, labels), rtol=0, atol=1e-12)


@pytest.mark.parametrize('labels', [
    np.array(['b cell', 't cell', 'nk'] * 40),
    np.array([0.5, -1.25, 3.0, 0.5] * 30),
    np.array([7, -3, 100, 7, 7, 100] * 20),
], ids=['strings', 'floats', 'sparse-integers'])
def test_driver_encodes_sorts_and_unpermutes(labels):
    rng = np.random.default_rng(1)
    X = rng.standard_normal((120, 5)).astype(np.float32)
    NumpySilhouette.calls.clear()
    got = _samples(X, labels)
    assert got.dtype == np.float64 and got.shape == (120,)
    np.testing.assert_allclose(got, S.silhouette_samples(X, labels), rtol=0, atol=1e-14)
    np.testing.assert_allclose(got, sk_samples(X.astype(np.float64), labels), rtol=0, atol=1e-12)
    (xs, off, bb), = NumpySilhouette.calls                   # one device call, rows stably sorted by label code
    _, codes = np.unique(labels, return_inverse=True)
    np.testing.assert_array_equal(xs, X[np.argsort(codes, kind='stable')])
    np.testing.assert_array_equal(off, np.concatenate([[0], np.cumsum(np.bincount(codes))]))
    assert bb == evaluation.SILHOUETTE_BATCH_BYTES


def test_singletons_and_zero_distances_give_zero():
    X = np.array([[0, 0], [0, 0], [0, 0], [0, 0], [5, 5], [9, 1]], np.float32)
    labels = np.array([0, 0, 1, 1, 2, 3])                     # rows 0-3: a = b = 0; rows 4, 5 alone in their labels
    got = _samples(X, labels)
    np.testing.assert_array_equal(got, np.zeros(6))
    np.testing.assert_array_equal(got, sk_samples(X, labels))
    mixed = np.array([0, 1, 0, 1, 0, 1])
    np.testing.assert_allclose(_samples(X, mixed), sk_samples(X.astype(np.float64), mixed), rtol=0, atol=1e-12)


def test_float32_rounding_and_dtypes():
    rng = np.random.default_rng(2)
    X = rng.standard_normal((200, 7))
    labels = rng.integers(0, 4, 200)
    np.testing.assert_array_equal(_samples(X, labels), _samples(X.astype(np.float32), labels))
    np.testing.assert_array_equal(_samples(X, labels), _samples(np.asfortranarray(X), list(labels)))


@pytest.mark.parametrize('sample_size', [None, 1, 50, 199, 500])
def test_score_draws_rows_as_sklearn(sample_size):
    rng = np.random.default_rng(3)
    X = rng.standard_normal((300, 4)).astype(np.float32).astype(np.float64)
    labels = rng.integers(0, 3, 300)
    if sample_size == 1:                                     # one row has one label: refused with sklearn's message
        with pytest.raises(ValueError, match='Number of labels is 1'):
            evaluation.silhouette_score(X, labels, sample_size=sample_size, random_state=0, backend=NumpySilhouette)
        return
    for seed in (0, 12345):
        got = evaluation.silhouette_score(X, labels, sample_size=sample_size, random_state=seed, backend=NumpySilhouette)
        assert isinstance(got, float)
        assert abs(got - sk_score(X, labels, sample_size=sample_size, random_state=seed)) < 1e-12
        got = evaluation.silhouette_score(X, labels, sample_size=sample_size, random_state=np.random.RandomState(seed),
                                          backend=NumpySilhouette)
        assert abs(got - sk_score(X, labels, sample_size=sample_size, random_state=np.random.RandomState(seed))) < 1e-12
    np.random.seed(7)
    got = evaluation.silhouette_score(X, labels, sample_size=sample_size, backend=NumpySilhouette)
    np.random.seed(7)
    assert abs(got - sk_score(X, labels, sample_size=sample_size)) < 1e-12


def test_refusals():
    rng = np.random.default_rng(4)
    X = rng.standard_normal((10, 3))
    y = np.arange(10) % 3
    bad = [
        (dict(metric='cosine'), "'euclidean'"),
        (dict(metric='precomputed'), "'euclidean'"),
        (dict(X=sp.csr_matrix(X)), 'dense'),
        (dict(X=X[:, 0]), r'\[n, L\]'),
        (dict(X=X[None]), r'\[n, L\]'),
        (dict(labels=y[:9]), 'one label per row'),
        (dict(labels=y[:, None]), 'one label per row'),
        (dict(X=np.zeros((0, 3)), labels=y[:0]), 'rows and columns'),
        (dict(X=np.zeros((10, 0))), 'rows and columns'),
        (dict(X=np.where(np.arange(30).reshape(10, 3) == 4, np.nan, X)), 'non-finite'),
        (dict(X=np.where(np.arange(30).reshape(10, 3) == 4, np.inf, X)), 'non-finite'),
        (dict(X=X * 1e300), 'non-finite'),
        (dict(labels=np.zeros(10)), r'Number of labels is 1\. Valid values are 2 to n_samples - 1 \(inclusive\)'),
        (dict(labels=np.arange(10)), r'Number of labels is 10\. Valid values are 2 to n_samples - 1 \(inclusive\)'),
    ]
    NumpySilhouette.calls.clear()
    for kw, msg in bad:
        args = dict(X=X, labels=y)
        args.update(kw)
        with pytest.raises(ValueError, match=msg):
            _samples(**args)
        with pytest.raises(ValueError, match=msg):
            evaluation.silhouette_score(**args, backend=NumpySilhouette)
    for ss in (0, -3, 2.5, True):
        with pytest.raises(ValueError, match='sample_size'):
            evaluation.silhouette_score(X, y, sample_size=ss, backend=NumpySilhouette)
    with pytest.raises(ValueError, match='seed'):
        evaluation.silhouette_score(X, y, sample_size=5, random_state='seven', backend=NumpySilhouette)
    huge = np.broadcast_to(np.float32(0), (1 << 31, 1))       # views: no memory behind the 2^31 rows
    with pytest.raises(ValueError, match='2\\^31'):
        _samples(huge, np.broadcast_to(np.int64(0), (1 << 31,)))
    assert NumpySilhouette.calls == []                       # no refusal reached the device call
    labels9 = np.arange(10) % 9                              # n - 1 labels are allowed
    np.testing.assert_allclose(_samples(X, labels9), sk_samples(X.astype(np.float32).astype(np.float64), labels9),
                               rtol=0, atol=1e-12)
