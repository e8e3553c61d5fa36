"""CPU tests of the feature-ablation driver (jamie_b200/impact.py): the rank-1 form of the ablated inputs, fill modes,
feature selection, sparse input, refusals, the fallback and the impact rule, with a float64 numpy stand-in for the
device class built on the oracle's eval forward."""
import warnings

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from oracle import jamie_oracle as O


@pytest.fixture(autouse=True)
def host_float64(monkeypatch):
    """The host arithmetic is pinned: no GPU projector, and the oracle's eval forward in float64."""
    from jamie_b200 import utilities as Ut
    monkeypatch.setattr(Ut, '_GPU_PROJECTOR', None)
    monkeypatch.setattr(O, 'F32', np.float64)


def _data(n, d, seed, const_col=None):
    rng = np.random.default_rng(seed)
    X = rng.normal(size=(n, d)) @ rng.normal(size=(d, d)) * 0.3 + rng.normal(size=d)
    if const_col is not None:
        X[:, const_col] = 1.5
    return X


def _model(sides, seed=0, L=6, n=80, d_raw=(23, 17), k=(7, 5), whiten=False):
    """A JAMIE with random weights (no training) whose input sides are 'pca' or 'none' (per-column standardisation)."""
    from sklearn.decomposition import PCA
    from jamie_b200.jamie import JAMIE
    from jamie_b200.model import edModelVar
    from jamie_b200.utilities import preclass
    raw = [_data(n, d_raw[i], seed + i, const_col=3 if sides[i] == 'none' else None) for i in range(2)]
    pres, dims = [], []
    for i in range(2):
        if sides[i] == 'pca':
            pca = PCA(k[i], whiten=whiten and i == 0)
            pres.append(preclass(pca.fit_transform(raw[i]), pca=pca))
            dims.append(k[i])
        else:
            pres.append(preclass(raw[i], axis=0))
            dims.append(d_raw[i])
    torch.manual_seed(seed)
    jm = JAMIE()
    jm.model = edModelVar(dims, L, preprocessing=[p.transform for p in pres],
                          preprocessing_inverse=[p.inverse_transform for p in pres])
    with torch.no_grad():   # non-trivial BatchNorm statistics
        g = torch.Generator().manual_seed(seed + 7)
        for name, b in jm.model.named_buffers():
            if name.endswith('running_mean'):
                b.copy_(torch.randn(b.shape, generator=g) * 0.1)
            elif name.endswith('running_var'):
                b.copy_(torch.rand(b.shape, generator=g) + 0.5)
    jm.dataset_num = 2
    return jm, raw, pres


def _oracle(jm):
    return O.OracleModel(jm.model.input_dims, jm.model.output_dim, params=jm.model.packed_parameters(),
                         buffers=jm.model.packed_buffers())


def _pearson(Y, T):
    """jb_metric_feature_pearson's formula in float64 (a constant column gives nan)."""
    Y, T = np.asarray(Y, np.float64), np.asarray(T, np.float64)
    N = Y.shape[0]
    with np.errstate(all='ignore'):
        cxy = (Y * T).sum(0) - Y.sum(0) * T.sum(0) / N
        return cxy / np.sqrt(((Y * Y).sum(0) - Y.sum(0) ** 2 / N) * ((T * T).sum(0) - T.sum(0) ** 2 / N))


class NumpyImpact:
    """Float64 stand-in for impact.DeviceImpact: the same inputs, evaluated with the oracle's eval forward."""
    calls = []

    def __init__(self, jm):
        self.orc = _oracle(jm)

    @staticmethod
    def inputs(Z, dz, w, w_col, q):
        if w_col is None:
            return Z + dz[q][:, None] * w[q][None, :]
        Zj = Z.copy()
        Zj[:, w_col[q]] += dz[q] * w[q]
        return Zj

    def run(self, frm, to, Z, dz, w, w_col, out, target, batch_bytes):
        NumpyImpact.calls.append((Z, dz, w, w_col))

        def pred(A):
            y = self.orc.encode_mu(A, frm) if to < 0 else self.orc.impute(A, frm, to)
            y = np.asarray(y, np.float64)
            if out.kind == 'pca':
                return (y * out.s + out.m) @ np.asarray(out.comp, np.float64) + out.mean
            if out.kind == 'affine':
                return y * out.scale + out.shift
            return y
        Y0 = pred(Z)
        shift = np.empty((dz.shape[0], out.d_out))
        r = None if target is None else np.empty_like(shift)
        for q in range(dz.shape[0]):
            Yj = pred(self.inputs(Z, dz, w, w_col, q))
            shift[q] = np.abs(Yj - Y0).mean(0)
            if target is not None:
                r[q] = _pearson(Yj, target)
        return shift, (None if target is None else _pearson(Y0, target)), r


def _loop(jm, pres, X, m, J, fills, target, space='output'):
    """The definition on the oracle: one full float64 prediction per feature."""
    from jamie_b200.impact import naive_feature_impact
    orc = _oracle(jm)
    to = 1 - m

    def predict(A):
        A = A.toarray() if sp.issparse(A) else A
        Zi = pres[m].transform(A)
        if space == 'latent':
            return orc.encode_mu(Zi, m)
        return pres[to].inverse_transform(orc.impute(Zi, m, to))
    return naive_feature_impact(predict, X, J, fills, target, pearson=_pearson)


def _run(jm, X, m, **kw):
    from jamie_b200.impact import feature_impact
    NumpyImpact.calls = []
    return feature_impact(jm, X, m, device=NumpyImpact, **kw)


def _close(a, b, tol=1e-10):
    np.testing.assert_allclose(a, b, rtol=tol, atol=tol)


@pytest.mark.parametrize('sides', [('pca', 'pca'), ('none', 'pca')])
def test_rank1_inputs_equal_transform_of_ablated_rows(sides):
    jm, raw, pres = _model(sides)
    X = raw[0][:40]
    J = np.array([0, 3, 5, 11])
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        _run(jm, X, 0, features=J, fill=0.25)
    Z, dz, w, w_col = NumpyImpact.calls[0]
    for q, j in enumerate(J):
        if w_col is not None and not pres[0].stats()[1][j] > 0:
            continue
        Xj = X.copy()
        Xj[:, j] = 0.25
        _close(NumpyImpact.inputs(Z, dz, w, w_col, q), pres[0].transform(Xj))


@pytest.mark.parametrize('sides,m', [(('pca', 'pca'), 0), (('pca', 'none'), 0), (('none', 'pca'), 0), (('pca', 'none'), 1)])
@pytest.mark.parametrize('fill', ['mean', 'scalar', 'array'])
def test_standin_equals_naive_loop(sides, m, fill):
    jm, raw, pres = _model(sides)
    X = raw[m]
    d = X.shape[1]
    fills = {'mean': X.mean(0), 'scalar': np.full(d, -0.5), 'array': np.linspace(-1, 1, d)}[fill]
    arg = {'mean': 'mean', 'scalar': -0.5, 'array': np.linspace(-1, 1, d)}[fill]
    T = _data(X.shape[0], raw[1 - m].shape[1], 99)
    T[:, 2] = 4.0                                   # a constant target column: nan r, skipped by impact
    J = np.array([1, 0, 4, 7])
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        got = _run(jm, X, m, target=T, features=J, fill=arg)
    shift, base_r, r = _loop(jm, pres, X, m, J, fills[J], T)
    undefined = sides[m] == 'none' and np.isin(J, [3])
    shift[undefined] = np.nan
    r[undefined] = np.nan
    _close(got.shift, shift)
    _close(got.baseline_r, base_r)
    _close(got.r, r)
    assert np.array_equal(got.features, J)
    keep = np.array([len(np.unique(c)) > 1 for c in T.T])
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        want = np.nanmean((base_r[None] - r)[:, keep], axis=1)
    _close(got.impact, want)


def test_latent_space_and_impact_without_target():
    jm, raw, pres = _model(('pca', 'pca'))
    X = raw[1]
    J = np.arange(X.shape[1])
    got = _run(jm, X, 1, space='latent')
    shift, _, _ = _loop(jm, pres, X, 1, J, X.mean(0)[J], None, space='latent')
    _close(got.shift, shift)
    assert got.shift.shape == (X.shape[1], jm.model.output_dim)
    assert got.r is None and got.baseline_r is None
    _close(got.impact, shift.mean(1))


def test_mask_selection_and_sparse_equal_dense():
    jm, raw, pres = _model(('pca', 'pca'))
    X = raw[0].copy()
    X[np.abs(X) < 0.8] = 0.0
    mask = np.zeros(X.shape[1], bool)
    mask[[2, 5, 9]] = True
    dense = _run(jm, X, 0, features=mask)
    assert np.array_equal(dense.features, [2, 5, 9])
    by_index = _run(jm, X, 0, features=[2, 5, 9])
    np.testing.assert_array_equal(dense.shift, by_index.shift)
    sparse = _run(jm, sp.csr_matrix(X), 0, features=mask)
    _close(sparse.shift, dense.shift, 1e-12)


def test_zero_scale_feature_is_nan_and_warns():
    jm, raw, pres = _model(('none', 'pca'))
    X = raw[0][:30]                         # column 3 is constant in the training data: its scale is 0
    T = _data(30, raw[1].shape[1], 5)
    with pytest.warns(UserWarning, match='zero standardisation scale'):
        got = _run(jm, X, 0, target=T, features=[2, 3, 4], fill=0.0)
    assert np.isnan(got.shift[1]).all() and np.isnan(got.r[1]).all() and np.isnan(got.impact[1])
    assert np.isfinite(got.shift[[0, 2]]).all() and np.isfinite(got.impact[[0, 2]]).all()


def test_refusals():
    jm, raw, pres = _model(('pca', 'pca'))
    X = raw[0][:20]
    d = X.shape[1]
    T = _data(20, raw[1].shape[1], 3)
    bad = X.copy()
    bad[4, 6] = np.nan
    cases = [
        dict(features=[0, d]), dict(features=[-1]), dict(features=[2, 2]), dict(features=np.ones(d - 1, bool)),
        dict(fill=np.inf), dict(fill=np.r_[np.zeros(d - 1), np.nan], features=[d - 1]), dict(fill=np.zeros(d + 1)),
        dict(fill='median'), dict(target=T[:, :-1]), dict(target=T[:-1]), dict(target=T, space='latent'),
        dict(space='input'),
    ]
    for kw in cases:
        with pytest.raises(ValueError):
            _run(jm, X, 0, **kw)
        assert NumpyImpact.calls == []
    with pytest.raises(ValueError, match='non-finite'):
        _run(jm, bad, 0, features=[6], fill=0.0)
    _run(jm, X, 0, fill=np.r_[np.zeros(d - 1), np.nan], features=[0])    # a non-finite fill of a column not ablated


def test_whitened_pca_takes_the_naive_loop(monkeypatch):
    jm, raw, pres = _model(('pca', 'pca'), whiten=True)
    orc = _oracle(jm)
    X, T = raw[0][:30], _data(30, raw[1].shape[1], 8)
    from jamie_b200 import evaluation
    monkeypatch.setattr(jm, 'modal_predict',
                        lambda A, m: pres[1].inverse_transform(orc.impute(pres[0].transform(A), 0, 1)), raising=False)
    monkeypatch.setattr(evaluation, 'imputation_correlation', _pearson)
    with pytest.warns(UserWarning, match='one full prediction per feature'):
        got = _run(jm, X, 0, target=T, features=[1, 4])
    assert NumpyImpact.calls == []
    shift, base_r, r = _loop(jm, pres, X, 0, [1, 4], X.mean(0)[[1, 4]], T)
    _close(got.shift, shift)
    _close(got.r, r)
    _close(got.baseline_r, base_r)


def test_impact_follows_the_column_rule():
    from jamie_b200.impact import impact_from
    T = np.array([[1., 2., 5.], [2., 2., 6.], [3., 2., 9.]])
    base = np.array([0.9, np.nan, 0.5])
    r = np.array([[0.7, 0.1, 0.2], [0.9, 0.3, np.nan]])
    np.testing.assert_allclose(impact_from(np.zeros((2, 3)), base, r, T), [(0.2 + 0.3) / 2, 0.0])
    np.testing.assert_allclose(impact_from(np.array([[1., 2., 3.]]), None, None, None), [2.0])
