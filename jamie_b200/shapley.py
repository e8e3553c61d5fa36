"""Shapley-value attribution on the GPU: ``JAMIE.shap_values`` (SURVEY.md 3.2).

The reference's ``scMNC-Visual.ipynb`` wraps ``modal_predict`` in a lambda and hands it to a SHAP explainer to find the
genes that drive each imputed feature. A model-agnostic explainer calls the model once per masked batch, each a full host
round trip. Here the whole estimate runs on the device (``jb_shapley``): with a linear input map a walk from a background
row b to the explained row x, adding one raw feature per step, changes the network input by one rank-1 term per step, so
the walk's inputs are a prefix sum built on the device from z_b, w and the raw rows; only the attributions come back.

Definition (also what ``naive_shap_values`` computes, one predict call per masked batch): f is ``modal_predict``
restricted to the selected output columns (``space='output'``) or ``transform_one`` (``space='latent'``);
v(S) = mean over b of f(x on S, b elsewhere), the interventional Shapley game with an independent background.
Estimator: for every permutation pi and background row b, walk from b to x adding the features in the order pi and credit
each step's output difference to the feature it added; average over (permutation, b). The permutations come in antithetic
pairs (pi, reversed pi), drawn with ``np.random.default_rng(seed)``, and are shared by every explained and background row.
Σ_j values[i, j] = f(x_i) - base_values for every draw; with all orders of the differing features the values are exact.
"""
import ctypes as C
import warnings
from dataclasses import dataclass

import numpy as np

from . import _lib
from .impact import OutputMap, _is_sparse, _preclass_of, input_map, output_map

# Upper bound of the device working set of one batch (walk rows, activations, outputs, per-segment sums), in bytes.
BATCH_BYTES = 4 << 30
# Largest result (values, float64) computed without selecting outputs, in bytes.
RESULT_BYTES = 8 << 30
# Explained rows per device call: the rows of one call are densified together (a function of d only).
X_BLOCK_BYTES = 256 << 20
# Background rows per device call; each accumulator receives its terms in (background block, permutation, row) order.
BACKGROUND_ROWS = 1024
# Walk rows per predict call of naive_shap_values.
WALK_ROWS = 4096


@dataclass
class ShapValues:
    values: np.ndarray       # [n, d_in, |O|] float64
    base_values: np.ndarray  # [|O|]: mean over the background of f(b)
    outputs: np.ndarray      # [|O|] the selected raw output columns (or latent dims)


def draw_permutations(d, n_permutations, seed):
    """[n_permutations, d] int32: n_permutations / 2 permutations from np.random.default_rng(seed), each followed by its
    reverse."""
    rng = np.random.default_rng(seed)
    P = np.empty((n_permutations, d), np.int32)
    for k in range(n_permutations // 2):
        p = rng.permutation(d)
        P[2 * k], P[2 * k + 1] = p, p[::-1]
    return P


def _dense(A):
    return np.asarray(A.toarray() if _is_sparse(A) else A, np.float64)


def _blocks(A, rows):
    """(r0, dense float64 block) over row blocks of A (a scipy.sparse A is densified one block at a time)."""
    Ar = A.tocsr() if _is_sparse(A) else A
    for r0 in range(0, A.shape[0], rows):
        yield r0, _dense(Ar[r0:r0 + rows])


def _all_finite(A):
    return bool(np.all(np.isfinite(A.data if _is_sparse(A) else A)))


def _naive_sums(predict, X, Bg, perms, phi, base):
    """The estimator's sums with one predict call per masked batch (up to WALK_ROWS rows of one walk): phi [nx, d, |O|]
    += sum over (permutation, b) of the step differences, base += sum over b of f(b). Every step is evaluated."""
    fb = np.asarray(predict(Bg), np.float64)
    for b in range(Bg.shape[0]):
        base += fb[b]
    d = X.shape[1]
    rank = np.empty(d, np.int64)
    for i in range(X.shape[0]):
        x = X[i]
        for p in perms:
            rank[p] = np.arange(d)
            for b in range(Bg.shape[0]):
                prev = fb[b]
                for t0 in range(0, d, WALK_ROWS):
                    t = np.arange(t0, min(d, t0 + WALK_ROWS))
                    M = np.where(rank[None, :] <= t[:, None], x[None, :], Bg[b][None, :])
                    Y = np.asarray(predict(M), np.float64)
                    steps = np.diff(np.vstack([prev[None, :], Y]), axis=0)
                    phi[i, p[t]] += steps             # distinct features: one term each, in (permutation, b) order
                    prev = Y[-1]


def naive_shap_values(predict, X, background, perms):
    """The estimator with one full ``predict`` call per masked batch: (values [n, d, |O|], base_values [|O|]). ``predict``
    maps raw rows to the selected outputs; ``perms`` [P, d] as ``draw_permutations`` gives them."""
    X, Bg, perms = _dense(X), _dense(background), np.asarray(perms)
    n_out = np.asarray(predict(Bg[:1])).shape[1]
    phi = np.zeros((X.shape[0], X.shape[1], n_out))
    base = np.zeros(n_out)
    _naive_sums(predict, X, Bg, perms, phi, base)
    return phi / (len(perms) * Bg.shape[0]), base / Bg.shape[0]


class DeviceShapley:
    """jb_shapley on the engine of a trained JAMIE (host tests substitute a numpy stand-in with the same run)."""

    def __init__(self, jm):
        import torch
        self.engine = jm._ensure_engine()
        self.stream = torch.cuda.current_stream().cuda_stream

    def run(self, frm, to, X, Bg, Zb, perms, w, w_col, out, out_cols, phi, base, stats, batch_bytes):
        """phi [nx, d, |O|] += the step-difference sums, base [|O|] += sum over Bg of f(b), stats [2] += {chain rows,
        skipped steps}; all in place."""
        def p(a):
            return None if a is None else a.ctypes.data_as(C.c_void_p)
        X = np.ascontiguousarray(X, np.float64)
        Bg = np.ascontiguousarray(Bg, np.float64)
        Zb = np.ascontiguousarray(Zb, np.float64)
        perms = np.ascontiguousarray(perms, np.int32)
        w = np.ascontiguousarray(w, np.float64)
        w_col = None if w_col is None else np.ascontiguousarray(w_col, np.int32)
        kind = {'identity': 0, 'pca': 1, 'affine': 2}[out.kind]
        comp = mean = sc = sh = oc = None
        if kind == 1:
            comp, mean = np.ascontiguousarray(out.comp, np.float32), np.ascontiguousarray(out.mean, np.float32)
        else:
            oc = np.ascontiguousarray(out_cols, np.int32)
        if kind == 2:
            sc, sh = np.ascontiguousarray(out.scale, np.float64), np.ascontiguousarray(out.shift, np.float64)
        assert phi.flags.c_contiguous and phi.dtype == np.float64 and base.dtype == np.float64
        _lib.check(self.engine.lib.jb_shapley(
            self.engine.h, int(frm), int(to), p(X), X.shape[0], p(Bg), Bg.shape[0], X.shape[1], p(Zb), p(perms),
            perms.shape[0], p(w), p(w_col), kind, p(comp), p(mean), float(out.m), float(out.s), p(sc), p(sh), p(oc),
            phi.shape[2], p(phi), p(base), p(stats), int(batch_bytes), C.c_void_p(self.stream)))


def _input_width(pre, default):
    """The raw width preprocessing takes: components_'s columns (PCA), the sample's columns (per-column), else default."""
    if pre is None:
        return default
    if pre is False:
        return None
    comp = getattr(pre.pca, 'components_', None) if pre.pca is not None else None
    if comp is not None:
        return int(np.shape(comp)[1])
    return int(np.shape(pre.sample)[1]) if pre.pca is None and pre.axis == 0 else None


def _output_width(pre, omap, default):
    if omap is not None:
        return omap.d_out
    comp = getattr(getattr(pre, 'pca', None), 'components_', None)   # e.g. a whitened PCA: the fallback's raw width
    return int(np.shape(comp)[1]) if comp is not None else default


def _select_outputs(outputs, width, space):
    if outputs is None:
        return np.arange(width)
    o = np.asarray(outputs)
    if o.ndim != 1 or o.size == 0 or not np.issubdtype(o.dtype, np.integer):
        raise ValueError('outputs must be a non-empty 1-D array of output column indices')
    what = 'latent dimensions' if space == 'latent' else 'output columns'
    if o.min() < 0 or o.max() >= width:
        raise ValueError(f"outputs must lie in [0, {width}): space={space!r} has {width} {what}")
    if np.unique(o).size != o.size:
        raise ValueError('outputs must be unique')
    return o.astype(np.int64)


def _restricted(omap, O):
    """The output map restricted to the outputs O, and the chain columns the device reads for kinds identity / affine."""
    if omap.kind == 'pca':
        return OutputMap('pca', len(O), comp=np.asarray(omap.comp)[:, O], mean=np.asarray(omap.mean)[O], m=omap.m, s=omap.s), None
    return omap, O


def _zero_scale_differs(X, Bg, cols):
    """The columns among cols (zero standardisation scale) where some explained row differs from some background row."""
    bad = []
    for j in cols:
        vals = np.concatenate([_dense(X[:, [j]]).ravel(), _dense(Bg[:, [j]]).ravel()])
        if np.any(vals != vals[0]):
            bad.append(int(j))
    return bad


def shap_values(jm, data, modality, background, outputs=None, space='output', n_permutations=2, seed=None, perms=None,
                device=DeviceShapley):
    """Shapley values of the raw input features of ``data`` (modality ``modality``) against ``background``; see the module
    docstring. ``perms`` [P, d] replaces the drawn permutations (tests, exact enumeration)."""
    assert jm.model is not None, 'Model must be trained before Shapley values.'
    if space not in ('output', 'latent'):
        raise ValueError(f"space must be 'output' or 'latent', not {space!r}")
    X = data if _is_sparse(data) else np.asarray(data)
    Bg = background if _is_sparse(background) else np.asarray(background)
    if X.ndim != 2 or Bg.ndim != 2:
        raise ValueError('data and background must be 2-D [cells, features] matrices')
    n, d_in = X.shape
    if Bg.shape[1] != d_in:
        raise ValueError(f'background has {Bg.shape[1]} features, data has {d_in}')
    model = jm.model
    d_model = _input_width(_preclass_of(model.preprocessing[modality]), model.input_dims[modality])
    if d_model is not None and d_in != d_model:
        raise ValueError(f'data has {d_in} features, modality {modality} takes {d_model}')
    if n == 0 or Bg.shape[0] == 0:
        raise ValueError('data and background need at least one row each')
    if perms is None:
        if isinstance(n_permutations, bool) or not isinstance(n_permutations, (int, np.integer)) or n_permutations <= 0 \
                or n_permutations % 2:
            raise ValueError(f'n_permutations must be a positive even integer (antithetic pairs), not {n_permutations!r}')
    else:
        perms = np.asarray(perms)
        if perms.ndim != 2 or perms.shape[1] != d_in or perms.shape[0] == 0 or \
                not all(np.array_equal(np.sort(p), np.arange(d_in)) for p in perms):
            raise ValueError(f'perms must be [P, {d_in}] permutations of the raw features')
    if not _all_finite(X) or not _all_finite(Bg):
        raise ValueError('data and background must be finite')

    to = (modality + 1) % jm.dataset_num if space == 'output' else -1
    pre_in = _preclass_of(model.preprocessing[modality])
    imap = input_map(pre_in, d_in)
    if space == 'output':
        pre_out = _preclass_of(model.preprocessing_inverse[to])
        omap = output_map(pre_out, model.input_dims[to])
        width = _output_width(pre_out, omap, model.input_dims[to])
    else:
        omap = OutputMap('identity', model.output_dim)
        width = model.output_dim
    O = _select_outputs(outputs, width, space)
    if n * d_in * len(O) * 8 > RESULT_BYTES:
        raise ValueError(f'the result would be [{n}, {d_in}, {len(O)}] float64 ({n * d_in * len(O) * 8 / 1e9:.1f} GB, more '
                         f'than RESULT_BYTES = {RESULT_BYTES / 1e9:.1f} GB): select fewer outputs (or explain fewer rows)')

    w_col = None
    if imap is not None:
        if imap[0] == 'column':
            w = imap[1].copy()
            undefined = np.flatnonzero(~np.isfinite(w))
            bad = _zero_scale_differs(X, Bg, undefined)
            if bad:
                raise ValueError(f'raw feature(s) {bad} have a zero standardisation scale and differ between data and '
                                 'background: the network input is infinite on their walk steps')
            w[undefined] = 0.0          # never an active step: their values are 0
            w_col = np.arange(d_in)
        else:
            w = imap[1]
    if perms is None:
        perms = draw_permutations(d_in, int(n_permutations), jm.manual_seed if seed is None else seed)
    P = perms.shape[0]

    nb = Bg.shape[0]
    values = np.empty((n, d_in, len(O)))
    base = np.zeros(len(O))
    xrows = max(1, min(n, X_BLOCK_BYTES // (8 * d_in)))
    b_blocks = list(_blocks(Bg, BACKGROUND_ROWS))
    if imap is None or omap is None:
        warnings.warn('the preprocessing of this model is not a linear PCA, a per-column standardisation or the identity: '
                      'Shapley values run one full prediction per masked batch')
        if space == 'output':
            def predict(A):
                return np.asarray(jm.modal_predict(A, modality))[:, O]
        else:
            def predict(A):
                return np.asarray(jm.transform_one(A, modality))[:, O]
        for r0, xb in _blocks(X, xrows):
            phi = np.zeros((xb.shape[0], d_in, len(O)))
            acc = base if r0 == 0 else np.zeros(len(O))
            for _, bb in b_blocks:
                _naive_sums(predict, xb, bb, perms, phi, acc)
            values[r0:r0 + xb.shape[0]] = phi / (P * nb)
        return ShapValues(values=values, base_values=base / nb, outputs=O)

    zb = [np.asarray(model.preprocessing[modality](bb), np.float64) for _, bb in b_blocks]
    if not all(np.all(np.isfinite(z)) for z in zb):
        raise ValueError('the preprocessed background is not finite (a zero standardisation scale?)')
    out, out_cols = _restricted(omap, O)
    dev = device(jm)
    stats = np.zeros(2, np.int64)
    for r0, xb in _blocks(X, xrows):
        phi = np.zeros((xb.shape[0], d_in, len(O)))
        acc = base if r0 == 0 else np.zeros(len(O))
        for (_, bb), z in zip(b_blocks, zb):
            dev.run(modality, to, xb, bb, z, perms, w, w_col, out, out_cols, phi, acc, stats, BATCH_BYTES)
        values[r0:r0 + xb.shape[0]] = phi / (P * nb)
    return ShapValues(values=values, base_values=base / nb, outputs=O)
