"""Feature ablation analysis on the GPU: ``JAMIE.feature_impact`` (SURVEY.md 3.2).

The reference's notebooks rank input features by ablation: set one raw input feature to a fill value, rerun the imputation
(``modal_predict``) or the encoder (``transform_one``), score the result, and repeat for every feature. Run as a loop, each
feature pays a full host round trip over the raw matrix. Here the whole analysis runs on the device
(``jb_feature_impact``): with a linear input map an ablation of raw column j changes the network's input by a rank-1
term, Z(j) = Z + dz[:, j] w_j^T, so only Z, w and dz go to the device, and only the per-feature score matrices come back.

Definition (also what ``naive_feature_impact`` computes, one full call per feature): X(j) = X with column j set to f_j,
Y(j) = predict(X(j)), Y = predict(X).
  shift[j, c]   = mean over rows of |Y(j)[:, c] - Y[:, c]|
  baseline_r[c] = Pearson r(Y[:, c], target[:, c]),  r[j, c] = Pearson r(Y(j)[:, c], target[:, c])   (with a target)
  impact[j]     = mean of baseline_r - r[j] over the non-constant target columns (nan columns skipped, as
                  evaluation.mean_feature_r aggregates); without a target the mean over c of shift[j, c].
"""
import ctypes as C
import warnings
from dataclasses import dataclass
from typing import Optional

import numpy as np

from . import _lib, evaluation
from .utilities import preclass

# Upper bound of the device working set of one batch (ablated inputs, activations, predictions, sums), in bytes.
BATCH_BYTES = 2 << 30


@dataclass
class FeatureImpact:
    features: np.ndarray              # [F] raw input column indices, in the order asked for
    shift: np.ndarray                 # [F, d_out]
    impact: np.ndarray                # [F]
    baseline_r: Optional[np.ndarray]  # [d_out] or None without a target
    r: Optional[np.ndarray]           # [F, d_out] or None without a target


def _is_sparse(X):
    return hasattr(X, 'tocsc') and not isinstance(X, np.ndarray)


def _preclass_of(fn):
    """The preclass behind model.preprocessing[i] / preprocessing_inverse[i]; None for identity; False for anything else."""
    obj = getattr(fn, '__self__', None)
    if isinstance(obj, preclass):
        return obj
    if getattr(fn, '__name__', None) == 'identity':
        return None
    return False


def _linear_pca(pre):
    """(components_, mean_, m, s) of a preclass with a linear, non-whitened PCA and a usable scalar scale, else None."""
    lin = pre._linear()
    if lin is None:
        return None
    m, s = pre.stats()
    if not (np.isfinite(m) and np.isfinite(s) and s > 0):
        return None
    return np.asarray(lin[0], np.float64), np.asarray(lin[1], np.float64), float(m), float(s)


def _per_column(pre):
    """(m_c, s_c) of a preclass without PCA that standardises each column (axis=0), else None."""
    if pre.pca is not None or pre.axis != 0:
        return None
    m, s = pre.stats()
    return np.asarray(m, np.float64), np.asarray(s, np.float64)


def input_map(pre, d_in):
    """How an ablation of raw column j enters the network's input: ('dense', W [d_in, k]) with w_j = W[j], or ('column',
    scale [d_in]) with w_j = scale[j] e_j. None: no rank-1 form is known (whitened or non-linear PCA, ...)."""
    if pre is None:
        return 'column', np.ones(d_in)
    if pre is False:
        return None
    pca = _linear_pca(pre)
    if pca is not None:
        return 'dense', pca[0].T / pca[3]
    col = _per_column(pre)
    if col is not None:
        scale = np.full(d_in, np.nan)     # a zero scale: preclass.transform divides by zero, the ablation is undefined
        ok = col[1] > 0
        scale[ok] = 1.0 / col[1][ok]
        return 'column', scale
    return None


@dataclass
class OutputMap:
    kind: str                          # 'identity', 'pca' or 'affine'
    d_out: int
    comp: Optional[np.ndarray] = None  # pca: components_ [k, d_out], mean_ [d_out], scalar m, s (as jb_pca_inverse takes them)
    mean: Optional[np.ndarray] = None
    m: float = 0.0
    s: float = 1.0
    scale: Optional[np.ndarray] = None  # affine: y * scale[c] + shift[c]
    shift: Optional[np.ndarray] = None


def output_map(pre, width):
    if pre is None:
        return OutputMap('identity', width)
    if pre is False:
        return None
    lin = pre._linear()
    if lin is not None:
        m, s = pre.stats()
        return OutputMap('pca', int(np.shape(lin[0])[1]), comp=np.asarray(lin[0]), mean=np.asarray(lin[1]), m=float(m), s=float(s))
    col = _per_column(pre)
    if col is not None:
        return OutputMap('affine', width, scale=col[1], shift=col[0])
    return None


def dense_rows(X, fn, rows=16384):
    """fn applied to row blocks of X (a scipy.sparse X is densified one block at a time), stacked."""
    if not _is_sparse(X):
        return np.asarray(fn(X))
    Xr = X.tocsr()
    return np.concatenate([np.asarray(fn(Xr[r0:r0 + rows].toarray())) for r0 in range(0, X.shape[0], rows)], axis=0)


def ablated_columns(X, J):
    """X[:, J] as a dense float64 [n, |J|] array (CSC slicing for scipy.sparse: only these columns are densified)."""
    if _is_sparse(X):
        return np.asarray(X.tocsc()[:, J].toarray(), np.float64)
    return np.asarray(X[:, J], np.float64)


def _select(features, d_in):
    if features is None:
        return np.arange(d_in)
    f = np.asarray(features)
    if f.dtype == bool:
        if f.shape != (d_in,):
            raise ValueError(f'a feature mask needs {d_in} entries, got shape {f.shape}')
        return np.flatnonzero(f)
    if f.ndim != 1 or (f.size and not np.issubdtype(f.dtype, np.integer)):
        raise ValueError('features must be a 1-D array of column indices or a boolean mask')
    f = f.astype(np.int64)
    if f.size and (f.min() < 0 or f.max() >= d_in):
        raise ValueError(f'feature indices must lie in [0, {d_in})')
    if np.unique(f).size != f.size:
        raise ValueError('feature indices must be unique')
    return f


def _fills(fill, cols, J, d_in):
    """f_j of the selected features J; cols = X[:, J] (dense float64: 'mean' is the same for a sparse and a dense X)."""
    if isinstance(fill, str):
        if fill != 'mean':
            raise ValueError(f"fill must be 'mean', a scalar or an array of {d_in} values, not {fill!r}")
        return cols.mean(axis=0)
    f = np.asarray(fill, np.float64)
    if f.ndim == 0:
        return np.full(len(J), float(f))
    if f.shape != (d_in,):
        raise ValueError(f'fill needs {d_in} values, got shape {f.shape}')
    return f[J]


def impact_from(shift, baseline_r, r, target):
    """impact[j]: mean over the non-constant target columns of baseline_r - r[j] (nan skipped); else mean of shift[j]."""
    if target is None:
        return shift.mean(axis=1) if shift.shape[1] else np.full(shift.shape[0], np.nan)
    T = np.asarray(target)
    keep = np.array([len(np.unique(col)) > 1 for col in T.T], bool)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        return np.nanmean((baseline_r[None, :] - r)[:, keep], axis=1)


def naive_feature_impact(predict, X, J, fills, target=None, pearson=None):
    """The definition, one full predict call per feature: (shift, baseline_r, r). fills[q] is the fill of column J[q]; a
    scipy.sparse X stays sparse."""
    pearson = pearson or evaluation.imputation_correlation
    Y = np.asarray(predict(X), np.float64)
    base_r = None if target is None else np.asarray(pearson(Y, target), np.float64)
    shift = np.empty((len(J), Y.shape[1]))
    r = None if target is None else np.empty((len(J), Y.shape[1]))
    if _is_sparse(X):
        import scipy.sparse as sp
        Xc = X.tocsc()
    for q, j in enumerate(J):
        if _is_sparse(X):
            col = sp.csc_matrix(np.full((X.shape[0], 1), fills[q]))
            Xj = sp.hstack([Xc[:, :j], col, Xc[:, j + 1:]], format='csr')
        else:
            Xj = np.array(X, copy=True)
            Xj[:, j] = fills[q]
        Yj = np.asarray(predict(Xj), np.float64)
        shift[q] = np.abs(Yj - Y).mean(axis=0)
        if target is not None:
            r[q] = pearson(Yj, target)
    return shift, base_r, r


class DeviceImpact:
    """jb_feature_impact on the engine of a trained JAMIE (host tests substitute a numpy stand-in with the same run)."""

    def __init__(self, jm):
        import torch
        self.engine = jm._ensure_engine()
        self.stream = torch.cuda.current_stream().cuda_stream

    def run(self, frm, to, Z, dz, w, w_col, out, target, batch_bytes):
        """(shift [F, d_out], baseline_r [d_out] or None, r [F, d_out] or None)"""
        def p(a):
            return None if a is None else a.ctypes.data_as(C.c_void_p)
        F = dz.shape[0]
        Z = np.ascontiguousarray(Z, np.float64)
        dz = np.ascontiguousarray(dz, np.float64)
        w = np.ascontiguousarray(w, np.float64)
        w_col = None if w_col is None else np.ascontiguousarray(w_col, np.int32)
        kind = {'identity': 0, 'pca': 1, 'affine': 2}[out.kind]
        comp = mean = sc = sh = None
        if kind == 1:
            comp, mean = np.ascontiguousarray(out.comp, np.float32), np.ascontiguousarray(out.mean, np.float32)
        elif kind == 2:
            sc, sh = np.ascontiguousarray(out.scale, np.float64), np.ascontiguousarray(out.shift, np.float64)
        T = None if target is None else np.ascontiguousarray(target, np.float32)
        shift = np.empty((F, out.d_out))
        base_r = None if T is None else np.empty(out.d_out)
        r = None if T is None else np.empty((F, out.d_out))
        _lib.check(self.engine.lib.jb_feature_impact(
            self.engine.h, int(frm), int(to), p(Z), Z.shape[0], F, p(dz), p(w), p(w_col), kind, p(comp), p(mean),
            float(out.m), float(out.s), p(sc), p(sh), int(out.d_out), p(T), p(base_r), p(r), p(shift), int(batch_bytes),
            C.c_void_p(self.stream)))
        return shift, base_r, r


def feature_impact(jm, data, modality, target=None, features=None, fill='mean', space='output', device=DeviceImpact):
    """Ablation analysis of the raw input features of ``data`` (modality ``modality``); see the module docstring."""
    assert jm.model is not None, 'Model must be trained before feature impact analysis.'
    if space not in ('output', 'latent'):
        raise ValueError(f"space must be 'output' or 'latent', not {space!r}")
    if space == 'latent' and target is not None:
        raise ValueError("a target is only defined for space='output'")
    X = data if _is_sparse(data) else np.asarray(data)
    if X.ndim != 2:
        raise ValueError('data must be a 2-D [cells, features] matrix')
    n, d_in = X.shape
    J = _select(features, d_in)
    cols = ablated_columns(X, J)
    fills = _fills(fill, cols, J, d_in)
    if not np.all(np.isfinite(cols)):
        raise ValueError('data has non-finite values in an ablated column')
    if not np.all(np.isfinite(fills)):
        raise ValueError('fill values of the ablated features must be finite')
    dz = np.ascontiguousarray((fills[None, :] - cols).T)       # [F, n]

    model = jm.model
    to = (modality + 1) % jm.dataset_num if space == 'output' else -1
    pre_in = _preclass_of(model.preprocessing[modality])
    imap = input_map(pre_in, d_in)
    if space == 'output':
        omap = output_map(_preclass_of(model.preprocessing_inverse[to]), model.input_dims[to])
    else:
        omap = OutputMap('identity', model.output_dim)
    if target is not None:
        target = np.asarray(target.toarray() if _is_sparse(target) else target)
        d_want = omap.d_out if omap is not None else None
        if target.ndim != 2 or target.shape[0] != n or (d_want is not None and target.shape[1] != d_want):
            raise ValueError(f'target must be [{n}, {d_want}], got shape {target.shape}')

    undefined = np.zeros(len(J), bool)
    if imap is not None and imap[0] == 'column':
        undefined = ~np.isfinite(imap[1][J])
    if undefined.any():
        warnings.warn(f'{int(undefined.sum())} ablated feature(s) have a zero standardisation scale on the input side; '
                      'their ablation is undefined and reported as nan')

    if imap is None or omap is None:
        warnings.warn('the preprocessing of this model is not a linear PCA, a per-column standardisation or the identity: '
                      'feature impact runs one full prediction per feature')
        predict = (lambda A: jm.modal_predict(A, modality)) if space == 'output' else (lambda A: jm.transform_one(A, modality))
        shift, base_r, r = naive_feature_impact(predict, X, J, fills, target)
    else:
        Z = dense_rows(X, model.preprocessing[modality])
        if imap[0] == 'dense':
            w, w_col = imap[1][J], None
        else:
            w, w_col = np.where(undefined, 0.0, imap[1][J]), J
        shift, base_r, r = device(jm).run(modality, to, Z, dz, w, w_col, omap, target, BATCH_BYTES)
    shift = np.array(shift, np.float64)
    shift[undefined] = np.nan
    if r is not None:
        r = np.array(r, np.float64)
        r[undefined] = np.nan
    imp = impact_from(shift, base_r, r, target)
    imp[undefined] = np.nan
    return FeatureImpact(features=J, shift=shift, impact=imp, baseline_r=base_r, r=r)
