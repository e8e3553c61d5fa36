"""CPU tests of the Shapley-value driver (jamie_b200/shapley.py): the estimator against exact Shapley values, efficiency,
dummy features, skipped steps, the permutation draw, sparse input, refusals, the zero-scale rule and the fallback, with a
float64 numpy stand-in for the device class built on the oracle's eval forward."""
import itertools
import math
import warnings

import numpy as np
import pytest
import scipy.sparse as sp

from oracle import jamie_oracle as O
from tests.test_impact_host import _data, _model, _oracle


@pytest.fixture(autouse=True)
def host_float64(monkeypatch):
    """The host arithmetic is pinned: no GPU projector, and the oracle's eval forward in float64."""
    from jamie_b200 import utilities as Ut
    monkeypatch.setattr(Ut, '_GPU_PROJECTOR', None)
    monkeypatch.setattr(O, 'F32', np.float64)


class NumpyShapley:
    """Float64 stand-in for shapley.DeviceShapley: the same walks (prefix sums from z_b, w and the raw rows, inactive
    steps skipped unless SKIP is False), evaluated with the oracle's eval forward."""
    calls = []
    SKIP = True

    def __init__(self, jm):
        self.orc = _oracle(jm)

    def run(self, frm, to, X, Bg, Zb, perms, w, w_col, out, out_cols, phi, base, stats, batch_bytes):
        NumpyShapley.calls.append(np.array(perms))
        d = X.shape[1]
        if w_col is None:
            W = np.asarray(w, np.float64)
        else:
            W = np.zeros((d, Zb.shape[1]))
            W[np.arange(d), w_col] = w

        def f(Z):
            y = np.asarray(self.orc.encode_mu(Z, frm) if to < 0 else self.orc.impute(Z, frm, to), np.float64)
            if out.kind == 'pca':
                return (y * out.s + out.m) @ np.asarray(out.comp, np.float64) + out.mean
            if out.kind == 'affine':
                y = y * out.scale + out.shift
            return y[:, out_cols]
        fb = f(Zb)
        for b in range(Bg.shape[0]):
            base += fb[b]
        nb, k = Zb.shape
        for i in range(X.shape[0]):
            for p in perms:
                Dp = (X[i][None, :] - Bg)[:, p]
                Z = Zb[:, None, :] + np.cumsum(Dp[:, :, None] * W[p][None], axis=1)
                Y = f(Z.reshape(-1, k)).reshape(nb, d, -1)
                active = Dp != 0 if NumpyShapley.SKIP else np.ones_like(Dp, bool)
                stats += [active.sum(), (~active).sum()]
                for b in range(nb):
                    ts = np.flatnonzero(active[b])
                    steps = np.diff(np.vstack([fb[b][None, :], Y[b, ts]]), axis=0)
                    phi[i, p[ts]] += steps


def _run(jm, X, m, B, **kw):
    from jamie_b200.shapley import shap_values
    NumpyShapley.calls = []
    return shap_values(jm, X, m, B, device=NumpyShapley, **kw)


def _f(jm, pres, m, O_, space='output'):
    """f on raw rows through the oracle in float64: the imputation (or embedding) restricted to the outputs O_."""
    orc = _oracle(jm)

    def f(A):
        A = A.toarray() if sp.issparse(A) else np.asarray(A, np.float64)
        Z = pres[m].transform(A)
        if space == 'latent':
            return np.asarray(orc.encode_mu(Z, m), np.float64)[:, O_]
        return np.asarray(pres[1 - m].inverse_transform(orc.impute(Z, m, 1 - m)), np.float64)[:, O_]
    return f


def _close(a, b, tol=1e-10):
    np.testing.assert_allclose(a, b, rtol=tol, atol=tol)


def _exact(f, x, B, A):
    """Exact Shapley values of the features A by coalition enumeration; x and every background row agree elsewhere."""
    k = len(A)
    v = {}
    for r in range(k + 1):
        for S in itertools.combinations(range(k), r):
            M = B.copy()
            M[:, [A[q] for q in S]] = x[[A[q] for q in S]]
            v[S] = f(M).mean(0)
    phi = np.zeros((k, len(v[()])))
    for q in range(k):
        for S in v:
            if q in S:
                continue
            T = tuple(sorted(S + (q,)))
            phi[q] += math.factorial(len(S)) * math.factorial(k - len(S) - 1) / math.factorial(k) * (v[T] - v[S])
    return phi


def walk_case(raw_m, A, nb=3, seed=4):
    """An x that differs from nb background rows in the features A only (the rows agree elsewhere)."""
    rng = np.random.default_rng(seed)
    B = np.repeat(raw_m[:1], nb, axis=0)
    B[:, A] += rng.normal(size=(nb, len(A)))
    x = raw_m[0].copy()
    x[A] += rng.normal(size=len(A))
    return x, B


def all_orders(d, A, seed=0):
    """Permutations of d features whose restrictions to A run through all len(A)! orders once."""
    base = np.random.default_rng(seed).permutation(d)
    slots = np.flatnonzero(np.isin(base, A))
    P = []
    for order in itertools.permutations(A):
        p = base.copy()
        p[slots] = order
        P.append(p)
    return np.array(P, np.int32)


@pytest.mark.parametrize('sides', [('pca', 'pca'), ('none', 'pca'), ('pca', 'none')])
def test_all_orders_give_exact_shapley_values(sides):
    jm, raw, pres = _model(sides)
    A = [1, 4, 6, 9, 12, 15]
    x, B = walk_case(raw[0], A)
    O_ = np.array([0, 2, 3])
    got = _run(jm, x[None], 0, B, outputs=O_, perms=all_orders(raw[0].shape[1], A))
    want = _exact(_f(jm, pres, 0, O_), x, B, A)
    _close(got.values[0, A], want)
    rest = np.setdiff1d(np.arange(raw[0].shape[1]), A)
    assert np.all(got.values[0, rest] == 0.0)


@pytest.mark.parametrize('sides,m,space', [(('pca', 'pca'), 0, 'output'), (('pca', 'none'), 0, 'output'),
                                           (('none', 'pca'), 0, 'output'), (('pca', 'none'), 1, 'output'),
                                           (('pca', 'pca'), 1, 'latent')])
def test_efficiency_and_agreement_with_the_naive_estimator(sides, m, space):
    from jamie_b200.shapley import naive_shap_values
    jm, raw, pres = _model(sides)
    X, B = raw[m][:3], raw[m][40:47]
    f = _f(jm, pres, m, slice(None), space)
    for seed in (0, 11):
        got = _run(jm, X, m, B, space=space, n_permutations=4, seed=seed)
        assert got.values.shape == (3, X.shape[1], f(X[:1]).shape[1])
        _close(got.values.sum(1), f(X) - got.base_values)
        _close(got.base_values, f(B).mean(0))
        values, base = naive_shap_values(f, X, B, NumpyShapley.calls[0])
        _close(got.values, values)
        _close(got.base_values, base)


def test_dummy_features_are_exactly_zero():
    jm, raw, pres = _model(('pca', 'pca'))
    X, B = raw[0][:2].copy(), raw[0][30:36].copy()
    B[:, [2, 7]] = 0.75
    X[:, [2, 7]] = 0.75
    got = _run(jm, X, 0, B, n_permutations=6, seed=3)
    assert np.all(got.values[:, [2, 7]] == 0.0)
    assert np.all(got.values[:, [0, 1, 3]] != 0.0)


def test_skipping_inactive_steps_changes_nothing(monkeypatch):
    jm, raw, pres = _model(('pca', 'none'))
    X, B = raw[0][:2].copy(), raw[0][20:25].copy()
    X[np.abs(X) < 0.9] = 0.0
    B[np.abs(B) < 0.9] = 0.0
    skip = _run(jm, X, 0, B, n_permutations=4)
    monkeypatch.setattr(NumpyShapley, 'SKIP', False)
    full = _run(jm, X, 0, B, n_permutations=4)
    _close(skip.values, full.values, 1e-12)
    _close(skip.base_values, full.base_values, 1e-12)


def test_antithetic_pairs_and_seeding():
    from jamie_b200.shapley import draw_permutations
    P = draw_permutations(23, 6, 9)
    assert P.shape == (6, 23) and P.dtype == np.int32
    for k in range(3):
        assert np.array_equal(np.sort(P[2 * k]), np.arange(23))
        assert np.array_equal(P[2 * k + 1], P[2 * k][::-1])
    rng = np.random.default_rng(9)
    assert np.array_equal(P[0], rng.permutation(23)) and np.array_equal(P[2], rng.permutation(23))
    assert np.array_equal(draw_permutations(23, 6, 9), P)
    assert not np.array_equal(draw_permutations(23, 6, 10), P)
    jm, raw, _ = _model(('pca', 'pca'))
    jm.manual_seed = 321
    X, B = raw[0][:1], raw[0][5:8]
    a = _run(jm, X, 0, B)
    assert np.array_equal(NumpyShapley.calls[0], draw_permutations(23, 2, 321))
    b = _run(jm, X, 0, B, seed=321)
    np.testing.assert_array_equal(a.values, b.values)
    _run(jm, X, 0, B, seed=5)
    assert np.array_equal(NumpyShapley.calls[0], draw_permutations(23, 2, 5))


def test_sparse_input_equals_dense(monkeypatch):
    from jamie_b200 import shapley
    jm, raw, _ = _model(('pca', 'pca'))
    X, B = raw[0][:5].copy(), raw[0][20:29].copy()
    X[np.abs(X) < 0.8] = 0.0
    B[np.abs(B) < 0.8] = 0.0
    dense = _run(jm, X, 0, B, outputs=[1, 5])
    monkeypatch.setattr(shapley, 'BACKGROUND_ROWS', 4)        # background blocks of 4 rows, one explained row per call
    monkeypatch.setattr(shapley, 'X_BLOCK_BYTES', 8 * X.shape[1])
    sparse = _run(jm, sp.csr_matrix(X), 0, sp.csr_matrix(B), outputs=[1, 5])
    assert len(NumpyShapley.calls) == 5 * 3
    _close(sparse.values, dense.values, 1e-12)
    _close(sparse.base_values, dense.base_values, 1e-12)
    assert np.array_equal(sparse.outputs, [1, 5])


def test_refusals(monkeypatch):
    from jamie_b200 import shapley
    jm, raw, _ = _model(('pca', 'pca'))
    X, B = raw[0][:4], raw[0][10:15]
    d = X.shape[1]
    bad = X.copy()
    bad[1, 3] = np.inf
    cases = [
        (X, B[:, :-1], {}), (X[:, :-1], B[:, :-1], {}), (X[0], B, {}), (X[:0], B, {}), (X, B[:0], {}),
        (bad, B, {}), (X, np.where(B > 0, np.nan, B), {}),
        (X, B, dict(n_permutations=3)), (X, B, dict(n_permutations=0)), (X, B, dict(n_permutations=-2)),
        (X, B, dict(n_permutations=2.0)),
        (X, B, dict(outputs=[0, 17])), (X, B, dict(outputs=[-1])), (X, B, dict(outputs=[2, 2])), (X, B, dict(outputs=[])),
        (X, B, dict(space='input')), (X, B, dict(space='latent', outputs=[6])),
        (X, B, dict(perms=np.zeros((2, d), int))),
    ]
    for A, Bk, kw in cases:
        with pytest.raises(ValueError):
            _run(jm, A, 0, Bk, **kw)
        assert NumpyShapley.calls == []
    monkeypatch.setattr(shapley, 'RESULT_BYTES', 4 * d * 17 * 8 - 1)
    with pytest.raises(ValueError, match='select fewer outputs'):
        _run(jm, X, 0, B)
    assert NumpyShapley.calls == []
    got = _run(jm, X, 0, B, outputs=[3])
    assert got.values.shape == (4, d, 1)


def test_zero_scale_features():
    jm, raw, pres = _model(('none', 'pca'))          # column 3 is constant (1.5) in the training data: its scale is 0
    X, B = raw[0][:3].copy(), raw[0][10:16].copy()
    got = _run(jm, X, 0, B, n_permutations=2)
    assert np.all(got.values[:, 3] == 0.0) and np.isfinite(got.values).all()
    f = _f(jm, pres, 0, slice(None))
    _close(got.values.sum(1), f(X) - f(B).mean(0))
    X[1, 3] = 2.0
    with pytest.raises(ValueError, match=r'\[3\]'):
        _run(jm, X, 0, B)
    X[:, 3] = B[:, 3] = 2.0                           # the same everywhere, but not the training value: input infinite
    with pytest.raises(ValueError, match='not finite'):
        _run(jm, X, 0, B)
    assert NumpyShapley.calls == []


def test_whitened_pca_takes_the_naive_path(monkeypatch):
    from jamie_b200.shapley import naive_shap_values
    jm, raw, pres = _model(('pca', 'pca'), whiten=True)
    orc = _oracle(jm)
    monkeypatch.setattr(jm, 'modal_predict',
                        lambda A, m: pres[1].inverse_transform(orc.impute(pres[0].transform(A), 0, 1)), raising=False)
    X, B = raw[0][:2], raw[0][10:14]
    with pytest.warns(UserWarning, match='one full prediction per masked batch'):
        got = _run(jm, X, 0, B, outputs=[0, 4], n_permutations=2, seed=1)
    assert NumpyShapley.calls == []
    from jamie_b200.shapley import draw_permutations
    f = _f(jm, pres, 0, [0, 4])
    values, base = naive_shap_values(f, X, B, draw_permutations(X.shape[1], 2, 1))
    _close(got.values, values)
    _close(got.base_values, base)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        _close(got.values.sum(1), f(X) - base)
