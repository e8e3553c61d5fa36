"""The acceptance metrics the reference's notebooks report, with the reference's own definitions (same denominators,
same default k, same printed lines), computed on the GPU (SURVEY.md 8 row N4): the O(n^2 L) distance work of FOSCTTM and
of the kNN label transfer, and the per-feature correlation and AUROC of an imputed matrix, run as CUDA kernels behind the
C ABI (``jb_metric_foscttm``, ``jb_metric_knn_vote``, ``jb_metric_feature_pearson``: csrc/metrics.cuh;
``jb_metric_feature_auroc``: csrc/auroc.cuh), the exact kNN search and kNN regression that serve as the imputation
baseline (``jb_knn``, ``jb_knn_average``: csrc/knn.cuh), and the silhouette coefficients of an embedding under a labelling
(``jb_silhouette``: csrc/silhouette.cuh; sklearn's ``silhouette_samples`` / ``silhouette_score``), scored with cell types
for how well they separate and with the modality for how well the modalities mix.

Reference: FOSCTTM ``test_closer`` jamie/evaluation.py:65-85 (class method jamie/jamie.py:892-913), label-transfer
accuracy ``test_LabelTA`` jamie/evaluation.py:114-132 (class method jamie/jamie.py:943-961: k = None default), per-feature
imputation correlation jamie/evaluation.py:491-513 (sklearn ``r_regression``) and AUROC jamie/evaluation.py:468-490
(sklearn ``roc_auc_score`` on measured > threshold).

There is no host fallback: without the CUDA library these functions raise.  The only host-side distance computation left
is the reference's ``distance_metric=`` hook of ``test_closer`` (a user callable on the concatenated embeddings).
"""
import ctypes as C

import numpy as np

from . import _lib


def _f32(x):
    return np.ascontiguousarray(np.asarray(x), np.float32)


def _device(device):
    if device is not None:
        return int(device)
    import torch
    return torch.cuda.current_device() if torch.cuda.is_available() else 0


def test_closer(integrated_data, distance_metric=None, verbose=True, device=None):
    """Fraction of samples closer than the true match: raw_count / (2 size^2), both directions (lower is better)."""
    assert len(integrated_data) == 2, 'Two datasets are supported for FOSCTTM'
    size = np.asarray(integrated_data[0]).shape[0]
    if distance_metric is not None:   # the reference's signature: a callable on the concatenated embeddings
        a = np.asarray(integrated_data[0], np.float64)
        b = np.asarray(integrated_data[1], np.float64)
        distances = distance_metric(np.concatenate([a, b], axis=0))
        raw_count_closer = 0
        for i in range(size):
            local = distances[i][size:]
            raw_count_closer += int(np.sum(local < local[i]))
            local = distances[size + i][:size]
            raw_count_closer += int(np.sum(local < local[i]))
    else:
        a, b = _f32(integrated_data[0]), _f32(integrated_data[1])
        assert a.shape == b.shape and a.ndim == 2, 'FOSCTTM needs two [n, L] embeddings of matched rows'
        cnt = C.c_ulonglong(0)
        lib = _lib.load()
        _lib.check(lib.jb_metric_foscttm(a.ctypes.data_as(C.c_void_p), b.ctypes.data_as(C.c_void_p), a.shape[0], a.shape[1],
                                         _device(device), C.byref(cnt)))
        raw_count_closer = int(cnt.value)
    foscttm = raw_count_closer / (2 * size ** 2)
    if verbose:
        print(f'foscttm: {foscttm}')
    return foscttm


foscttm = test_closer   # name used by the tests of this repository


def default_k(datatype):
    """20 % of the average class size (jamie/jamie.py:946-950)."""
    total_size = min(*[len(d) for d in datatype])
    num_classes = len(np.unique(np.concatenate(datatype)).flatten())
    return int(.2 * total_size / num_classes)


def test_LabelTA(integrated_data, datatype, k=5, return_k=False, verbose=True, device=None):
    """kNN classifier (uniform votes, euclidean) fitted on modality 1's embedding and labels, scored on modality 0's."""
    if k is None:
        k = default_k(datatype)
    emb0, emb1 = _f32(integrated_data[0]), _f32(integrated_data[1])
    y0 = np.asarray(datatype[0]).ravel()
    y1 = np.asarray(datatype[1]).ravel()
    classes, y1c = np.unique(y1, return_inverse=True)   # sklearn: classes sorted, ties -> the lowest class
    y1c = np.ascontiguousarray(y1c, np.int32)
    pred = np.empty(emb0.shape[0], np.int32)
    lib = _lib.load()
    _lib.check(lib.jb_metric_knn_vote(emb0.ctypes.data_as(C.c_void_p), emb0.shape[0], emb1.ctypes.data_as(C.c_void_p),
                                      y1c.ctypes.data_as(C.c_void_p), emb1.shape[0], emb0.shape[1], int(k), len(classes),
                                      _device(device), pred.ctypes.data_as(C.c_void_p)))
    acc = float(np.sum(classes[pred] == y0)) / len(y0)
    if verbose:
        print(f'label transfer accuracy: {acc}')
    if return_k:
        return acc, k
    return acc


def label_transfer_accuracy(integrated_data, datatype, k=None, return_k=False):
    """The class method's form (jamie/jamie.py:943-961): k defaults to 20 % of the average class size, nothing printed."""
    return test_LabelTA(integrated_data, datatype, k=k, return_k=return_k, verbose=False)


def imputation_correlation(imputed, measured, device=None):
    """Per-feature Pearson r between imputed and measured values (constant features give nan and are skipped)."""
    x, y = _f32(imputed), _f32(measured)
    assert x.shape == y.shape and x.ndim == 2
    r = np.empty(x.shape[1], np.float64)
    lib = _lib.load()
    _lib.check(lib.jb_metric_feature_pearson(x.ctypes.data_as(C.c_void_p), y.ctypes.data_as(C.c_void_p), x.shape[0], x.shape[1],
                                             _device(device), r.ctypes.data_as(C.c_void_p)))
    return r


def mean_feature_r(imputed, measured):
    """Mean over the non-constant measured features, as ``_plot_correlation`` aggregates (jamie/evaluation.py:491-513)."""
    y = np.asarray(measured)
    keep = np.array([len(np.unique(col)) > 1 for col in y.T])
    return float(np.nanmean(imputation_correlation(imputed, measured)[keep]))


# Upper bound of the device working set of one column batch of imputation_auroc (and of the host's temporaries while it
# builds the positive lists of a dense ``measured``), in bytes.
BATCH_BYTES = 1 << 30


def _is_sparse(x):
    return hasattr(x, 'tocsc') and not isinstance(x, np.ndarray)


def positive_lists(measured, threshold, batch_bytes):
    """The rows with measured > threshold of every column as CSC lists: (int64 ptr [d + 1], int32 rows, increasing within
    a column). A scipy.sparse ``measured`` is read through its CSC form and never densified (threshold >= 0: implicit
    zeros are negatives); a dense one in column blocks of about batch_bytes / 4 elements. Raises ValueError for
    non-finite values."""
    n, d = measured.shape
    if _is_sparse(measured):
        M = measured.tocsc(copy=True)
        M.sum_duplicates()                      # the values a dense copy would hold, rows increasing within a column
        if not np.isfinite(M.data).all():
            raise ValueError('measured has non-finite values')
        keep = M.data > threshold
        ck = np.concatenate([[0], np.cumsum(keep, dtype=np.int64)])
        return ck[M.indptr], np.ascontiguousarray(M.indices[keep], np.int32)
    counts, rows = np.zeros(d + 1, np.int64), []
    cb = max(1, min(d, batch_bytes // (4 * max(n, 1))))
    for j0 in range(0, d, cb):
        blk = measured[:, j0:j0 + cb]
        if not np.isfinite(blk).all():
            raise ValueError('measured has non-finite values')
        m = np.ascontiguousarray((blk > threshold).T)    # [columns, n]: nonzeros by column, then row
        counts[j0 + 1:j0 + 1 + m.shape[0]] = m.sum(axis=1)
        rows.append((np.flatnonzero(m) % n).astype(np.int32))
    return np.cumsum(counts), np.concatenate(rows) if rows else np.zeros(0, np.int32)


def imputation_auroc(imputed, measured, threshold=0.0, device=None):
    """Per-feature AUROC of imputed values against the measured ones read as present / absent:
    roc_auc_score(measured[:, j] > threshold, float32(imputed[:, j])) for every column j (the AUROC panel of
    jamie/evaluation.py:468-490), computed on the GPU (``jb_metric_feature_auroc``) as the exact Mann-Whitney statistic
    2U in integers, then one float64 division 2U / (2 P N). A column with one class only gives nan.

    ``imputed`` is a dense [n, d] array (rounded to float32, as ``imputation_correlation`` does); ``measured`` is dense or
    any scipy.sparse format (never densified). Labels compare ``measured`` as given with ``threshold``."""
    if _is_sparse(imputed):
        raise ValueError('imputed must be a dense array')
    x = np.asarray(imputed)
    y = measured if _is_sparse(measured) else np.asarray(measured)
    if x.ndim != 2 or y.ndim != 2 or x.shape != y.shape:
        raise ValueError(f'imputed and measured must be two [n, d] matrices of one shape, got {x.shape} and {y.shape}')
    n, d = x.shape
    if n >= 1 << 31:
        raise ValueError(f'{n} rows: imputation_auroc takes fewer than 2^31')
    if np.ndim(threshold) != 0:
        raise ValueError('threshold must be a scalar')
    try:
        finite = np.isfinite(threshold)
    except TypeError:
        finite = False
    if not finite:
        raise ValueError(f'threshold must be a finite number, not {threshold!r}')
    if _is_sparse(y) and threshold < 0:
        raise ValueError('a sparse measured matrix with threshold < 0 would make every implicit zero positive: '
                         'pass a dense array')
    if n == 0:
        raise ValueError('imputation_auroc needs at least one row')
    with np.errstate(over='ignore'):
        scores = _f32(x)
    if not np.isfinite(scores).all():
        raise ValueError('imputed has non-finite values (after rounding to float32)')
    ptr, rows = positive_lists(y, threshold, BATCH_BYTES)
    if d == 0:
        return np.zeros(0, np.float64)
    u2 = np.empty(d, np.uint64)
    n_pos = np.empty(d, np.int64)
    lib = _lib.load()
    p = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
    _lib.check(lib.jb_metric_feature_auroc(p(scores), n, d, p(ptr), p(rows), int(BATCH_BYTES), _device(device), p(u2),
                                           p(n_pos)))
    # 2U and 2PN are exact integers; Python's int division rounds their quotient correctly
    return np.array([u / (2 * q * (n - q)) if 0 < q < n else np.nan for u, q in zip(u2.tolist(), n_pos.tolist())],
                    np.float64)


# Upper bound of the device working set of one query batch of kneighbors / knn_impute (the reference rows aside) and of
# one column slab of knn_impute's average, in bytes; a sparse ``values`` is densified on the host one such slab at a time.
KNN_BATCH_BYTES = 1 << 30
KNN_MAX_K = 1024   # the largest k of the device search (csrc/knn.cuh KN_MAXK)


class DeviceKnn:
    """The two device calls of kneighbors / knn_impute (host tests substitute a numpy stand-in with the same methods)."""

    @staticmethod
    def search(query, reference, k, batch_bytes, device):
        """jb_knn: (dist float64 [nq, k], idx int64 [nq, k]) of fp32 C-contiguous rows."""
        nq, nr = query.shape[0], reference.shape[0]
        idx = np.empty((nq, k), np.int64)
        dist = np.empty((nq, k), np.float64)
        p = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
        _lib.check(_lib.load().jb_knn(p(query), nq, p(reference), nr, query.shape[1], int(k), int(batch_bytes),
                                      _device(device), p(idx), p(dist)))
        return dist, idx

    @staticmethod
    def average(idx, weights, values, batch_bytes, device):
        """jb_knn_average: float64 [nq, w] for float64 ``values`` [nr, w] with unit column stride."""
        nq, k = idx.shape
        out = np.empty((nq, values.shape[1]), np.float64)
        p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)   # noqa: E731
        _lib.check(_lib.load().jb_knn_average(p(idx), p(weights), nq, int(k), p(values), values.shape[0], values.shape[1],
                                              values.strides[0] // 8, int(batch_bytes), _device(device), p(out)))
        return out


def _knn_rows(query, reference, k):
    """The query and reference rows as C-contiguous float32, checked; raises ValueError."""
    q, r = np.asarray(query), np.asarray(reference)
    if q.ndim != 2 or r.ndim != 2 or q.shape[1] != r.shape[1]:
        raise ValueError(f'query and reference must be [n, L] matrices of one width, got {q.shape} and {r.shape}')
    if q.shape[0] == 0 or r.shape[0] == 0 or q.shape[1] == 0:
        raise ValueError(f'query and reference need rows and columns, got {q.shape} and {r.shape}')
    if isinstance(k, bool) or not isinstance(k, (int, np.integer)):
        raise ValueError(f'k must be an integer, not {k!r}')
    if k < 1 or k > r.shape[0]:
        raise ValueError(f'k = {k} neighbours of {r.shape[0]} reference rows: 1 <= k <= {r.shape[0]}')
    if k > KNN_MAX_K:
        raise ValueError(f'k = {k}: the device search takes at most {KNN_MAX_K} neighbours')
    with np.errstate(over='ignore'):
        q32, r32 = _f32(q), _f32(r)
    for name, a in (('query', q32), ('reference', r32)):
        if not np.isfinite(a).all():
            raise ValueError(f'{name} has non-finite values (after rounding to float32)')
    return q32, r32


def kneighbors(query, reference, k, device=None, backend=DeviceKnn):
    """The k nearest reference rows of every query row in euclidean distance, searched exactly on the GPU (``jb_knn``):
    (dist float64 [nq, k], idx int64 [nq, k]), each row in ascending distance, equal distances by the lowest reference
    index. The same as ``NearestNeighbors(n_neighbors=k, algorithm='brute').fit(reference).kneighbors(query)`` on data
    without exact ties. Rows are rounded to float32, as ``test_closer`` and ``test_LabelTA`` do; distances are float64
    sums of squared differences, so they carry no cancellation. 1 <= k <= min(1024, nr)."""
    q32, r32 = _knn_rows(query, reference, k)
    return backend.search(q32, r32, int(k), KNN_BATCH_BYTES, device)


def knn_weights(dist, weights):
    """sklearn's neighbour weights: None for 'uniform'; for 'distance' 1 / d, except that a row with a zero distance
    weighs its zero-distance neighbours 1 and the others 0."""
    if weights == 'uniform':
        return None
    with np.errstate(divide='ignore'):
        w = 1.0 / dist
    inf = np.isinf(w)
    rows = inf.any(axis=1)
    w[rows] = inf[rows]
    return np.ascontiguousarray(w, np.float64)


def knn_impute(query, reference, values, k=5, weights='uniform', device=None, backend=DeviceKnn):
    """kNN regression on the GPU: for every query row the average of ``values`` over its k nearest ``reference`` rows
    (``kneighbors``), uniform or weighted by inverse distance (``weights='distance'``, sklearn's rules), float64 [nq, d].
    The same as ``KNeighborsRegressor(n_neighbors=k, weights=weights, algorithm='brute').fit(reference, values)
    .predict(query)``. ``values`` [nr, d] is a dense array (read as float64) or any scipy.sparse matrix; either goes to the
    device in column slabs, and a sparse one is densified one slab at a time."""
    if weights not in ('uniform', 'distance'):
        raise ValueError(f"weights must be 'uniform' or 'distance', not {weights!r}")
    q32, r32 = _knn_rows(query, reference, k)
    (nq, _), (nr, _) = q32.shape, r32.shape
    V = values if _is_sparse(values) else np.asarray(values, np.float64)
    if V.ndim != 2 or V.shape[0] != nr:
        raise ValueError(f'values must be [{nr}, d] (one row per reference row), got shape {V.shape}')
    d = V.shape[1]
    if _is_sparse(V):
        V = V.tocsc(copy=True)
        V.sum_duplicates()
        finite = np.isfinite(V.data).all()
    else:
        finite = np.isfinite(V).all()
    if not finite:
        raise ValueError('values has non-finite values')
    dist, idx = backend.search(q32, r32, int(k), KNN_BATCH_BYTES, device)
    w = knn_weights(dist, weights)
    if d == 0:
        return np.zeros((nq, 0), np.float64)
    if not _is_sparse(V):
        return backend.average(idx, w, np.ascontiguousarray(V), KNN_BATCH_BYTES, device)
    out = np.empty((nq, d), np.float64)
    cw = max(1, KNN_BATCH_BYTES // (8 * (nr + nq)))
    for c0 in range(0, d, cw):
        out[:, c0:c0 + cw] = backend.average(idx, w, np.ascontiguousarray(V[:, c0:c0 + cw].toarray(), np.float64),
                                             KNN_BATCH_BYTES, device)
    return out


# Upper bound of the device working set of one query batch of silhouette_samples (the rows aside), in bytes.
SILHOUETTE_BATCH_BYTES = 1 << 30


class DeviceSilhouette:
    """The device call of silhouette_samples (host tests substitute a numpy stand-in with the same method)."""

    @staticmethod
    def sums(x_sorted, label_off, batch_bytes, device):
        """jb_silhouette: (intra, inter) float64 [n] of fp32 C-contiguous rows sorted by label, label c holding rows
        label_off[c] .. label_off[c + 1]: the sum of the distances to the row's own label, and the least mean distance to
        another label."""
        n, L = x_sorted.shape
        off = np.ascontiguousarray(label_off, np.int64)
        intra, inter = np.empty(n, np.float64), np.empty(n, np.float64)
        p = lambda a: a.ctypes.data_as(C.c_void_p)   # noqa: E731
        _lib.check(_lib.load().jb_silhouette(p(x_sorted), n, L, p(off), len(off) - 1, int(batch_bytes), _device(device),
                                             p(intra), p(inter)))
        return intra, inter


def silhouette_samples(X, labels, metric='euclidean', device=None, backend=DeviceSilhouette):
    """The silhouette coefficient of every row, float64 [n]: the same as ``sklearn.metrics.silhouette_samples(X, labels)``
    with its O(n^2 L) pair work on the GPU (``jb_silhouette``). With a the mean distance of row i to the other rows of its
    label and b the least mean distance to the rows of another label, s = (b - a) / max(a, b); a row alone in its label,
    and a row with a = b = 0, gives 0. Rows are rounded to float32, as ``test_closer`` and ``kneighbors`` do; distances
    are the sqrt of float64 sums of squared differences, so they carry no cancellation. Scored with cell types as labels
    it measures how well types separate in a joint embedding; with the modality (0 / 1), how well the modalities mix."""
    if metric != 'euclidean':
        raise ValueError(f"metric must be 'euclidean', the only one supported, not {metric!r}")
    if _is_sparse(X):
        raise ValueError('X must be a dense array')
    x, lab = np.asarray(X), np.asarray(labels)
    if x.ndim != 2:
        raise ValueError(f'X must be an [n, L] matrix, got shape {x.shape}')
    if lab.ndim != 1 or lab.shape[0] != x.shape[0]:
        raise ValueError(f'labels must be one label per row of X ({x.shape[0]}), got shape {lab.shape}')
    n = x.shape[0]
    if n == 0 or x.shape[1] == 0:
        raise ValueError(f'X needs rows and columns, got shape {x.shape}')
    if n >= 1 << 31:
        raise ValueError(f'{n} rows: silhouette_samples takes fewer than 2^31')
    with np.errstate(over='ignore'):
        x32 = _f32(x)
    if not np.isfinite(x32).all():
        raise ValueError('X has non-finite values (after rounding to float32)')
    classes, codes = np.unique(lab, return_inverse=True)   # sklearn's LabelEncoder
    codes = codes.ravel()
    if not 1 < len(classes) < n:
        raise ValueError('Number of labels is %d. Valid values are 2 to n_samples - 1 (inclusive)' % len(classes))
    freq = np.bincount(codes)
    order = np.argsort(codes, kind='stable')
    label_off = np.concatenate([[0], np.cumsum(freq)]).astype(np.int64)
    intra_s, inter_s = backend.sums(np.ascontiguousarray(x32[order]), label_off, SILHOUETTE_BATCH_BYTES, device)
    intra, inter = np.empty(n, np.float64), np.empty(n, np.float64)
    intra[order], inter[order] = intra_s, inter_s
    # sklearn's own finish, in its order
    denom = (freq - 1).take(codes, mode='clip')
    with np.errstate(divide='ignore', invalid='ignore'):
        intra /= denom
    sil = inter - intra
    with np.errstate(divide='ignore', invalid='ignore'):
        sil /= np.maximum(intra, inter)
    return np.nan_to_num(sil)


def silhouette_score(X, labels, metric='euclidean', sample_size=None, random_state=None, device=None,
                     backend=DeviceSilhouette):
    """The mean silhouette coefficient, ``float(np.mean(silhouette_samples(X, labels)))``: the same as
    ``sklearn.metrics.silhouette_score``. With ``sample_size``, it scores the rows
    ``check_random_state(random_state).permutation(n)[:sample_size]``, as sklearn draws them."""
    if sample_size is not None:
        if isinstance(sample_size, bool) or not isinstance(sample_size, (int, np.integer)) or sample_size < 1:
            raise ValueError(f'sample_size must be a positive integer or None, not {sample_size!r}')
        if _is_sparse(X):
            raise ValueError('X must be a dense array')
        x, lab = np.asarray(X), np.asarray(labels)
        if x.ndim != 2 or lab.ndim != 1 or lab.shape[0] != x.shape[0]:
            raise ValueError(f'X must be an [n, L] matrix with one label per row, got shapes {x.shape} and {lab.shape}')
        idx = _random_state(random_state).permutation(x.shape[0])[:sample_size]
        X, labels = x[idx], lab[idx]
    return float(np.mean(silhouette_samples(X, labels, metric=metric, device=device, backend=backend)))


def _random_state(seed):
    """sklearn's check_random_state: numpy's global RandomState for None, a new one for an integer, or the instance."""
    if seed is None or seed is np.random:
        return np.random.mtrand._rand
    if isinstance(seed, (int, np.integer)) and not isinstance(seed, bool):
        return np.random.RandomState(seed)
    if isinstance(seed, np.random.RandomState):
        return seed
    raise ValueError(f'{seed!r} cannot be used to seed a numpy.random.RandomState instance')
