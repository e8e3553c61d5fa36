"""Distances and the correspondence estimate F (SURVEY 8f rows N2 / N1): what ``fit_transform`` runs before training when
``use_f_tilde=True`` and no ``match_result`` is supplied (jamie/jamie.py:160-175).

* ``distance_function`` / ``compute_distances`` -- jamie/jamie.py:839-890: per-dataset n x n distance matrix in the chosen
  ``distance_mode`` (host: sklearn / scipy, exactly the calls the reference makes).  The default mode 'geodesic' calls the
  third-party ``unioncom.utils.geodesic_distances`` (unioncom==0.4.0, NOT vendored in the reference): restated here from
  the published package -- kNN graph (k from 5 upwards in steps of 2 until connected or k > max(kmax, 0.01 n)), all-pairs
  shortest paths, unreachable pairs set to twice the largest finite distance.  PARITY UNPINNED for that function (no
  reference test or fixture covers it); the other modes and Prime_Dual are pinned by tests/golden/prime_dual.npz.
* ``gpu_distance_function`` -- the same distances on the GPU (``JAMIE(distances='gpu')``): the n^2 d accumulation over
  column slabs, the kNN selection and the all-pairs shortest paths run in csrc/distances.cuh behind the jb_dist handle;
  the host keeps the O(n d) row preparation, the slab iterator and the k-connectivity loop.
* ``prime_dual`` -- jamie/jamie.py:314-414: UnionCom's primal-dual Adam iteration for F on the GPU.  Dense n x n fp32
  algebra: four GEMMs per iteration through torch / cuBLAS (plain library GEMMs), everything else element-wise; the
  rank-one products of the reference (``Mu 1^T``, ``1 Lambda^T``, ``F 1 1^T``, ``1 1^T F``) are written as broadcasts of
  row / column sums.  Same update order, constants and printed lines as the reference.
"""
import warnings

import numpy as np


def geodesic_distances(X, kmax):
    """unioncom.utils.geodesic_distances (unioncom==0.4.0), restated; see the module docstring (parity unpinned)."""
    import scipy.sparse.csgraph as csg
    from sklearn.neighbors import NearestNeighbors
    X = np.asarray(X)
    n = len(X)
    k = 5

    def graph(k_):
        nb = NearestNeighbors(n_neighbors=min(k_, n), metric='euclidean').fit(X)
        return nb.kneighbors_graph(X, mode='distance')

    knn = graph(k)
    while csg.connected_components(knn, directed=False)[0] != 1:
        if k > max(kmax, 0.01 * n):
            break
        k += 2
        knn = graph(k)
    dist = csg.shortest_path(knn, method='D', directed=False)
    finite_max = np.nanmax(dist[dist != np.inf])
    dist[dist > finite_max] = 2 * finite_max
    return dist


def distance_function(distance_mode, kmax):
    """The per-dataset distance callable of jamie/jamie.py:851-884."""
    if distance_mode == 'geodesic':
        def fn(df):
            with warnings.catch_warnings():
                warnings.simplefilter('ignore')
                return np.array(geodesic_distances(df, kmax))
    elif distance_mode == 'spearman':
        def fn(df):
            from scipy import stats
            if df.shape[0] == 1:
                d = np.array([0])
            else:
                d, _ = stats.spearmanr(df, axis=1)
                if np.isnan(d).any():
                    raise Exception('Data is not well conditioned for spearman method '
                                    '(scipy.stats.spearmanr returned ``np.nan``)')
            if len(np.shape(d)) == 0:
                d = np.array([[1, d], [d, 1]])
            return (1 - np.array(d)) / 2
    elif distance_mode == 'pearson':
        def fn(df):
            if df.shape[0] == 1:
                return np.array([0])
            d = np.corrcoef(df.toarray() if hasattr(df, 'toarray') else df)
            if len(np.shape(d)) == 0:
                d = np.array([[1, d], [d, 1]])
            return (1 - np.array(d)) / 2
    else:
        def fn(df):
            from sklearn.metrics import pairwise_distances
            return pairwise_distances(df, metric=distance_mode)
    return fn


# ------------------------------------------------------------------------------------------------ distances on the GPU
# distance_mode -> (accumulated form, row preparation, finishing transform) of the jb_dist handle (csrc/distances.cuh).
# Forms: 0 = sum (a - b)^2, 1 = sum |a - b|, 2 = sum a b. Transforms: 0 = none, 1 = sqrt, 2 = 1 - g clipped to [0, 2] with a
# zero diagonal, 3 = (1 - clip(g, -1, 1)) / 2. Preparations (O(n d) on the host, streamed slab by slab): 'norm' = rows
# over their L2 norm (sklearn's normalize: a zero row stays zero), 'centre' = rows minus their mean over the L2 norm of
# that (a constant row becomes NaN, as np.corrcoef / scipy give), 'rank' = 'centre' on the row ranks (scipy.stats.rankdata,
# average ties: spearmanr's ranks).
GPU_DISTANCE_MODES = {
    'geodesic': (0, None, 1),
    'euclidean': (0, None, 1), 'l2': (0, None, 1),
    'sqeuclidean': (0, None, 0),
    'cityblock': (1, None, 0), 'l1': (1, None, 0), 'manhattan': (1, None, 0),
    'cosine': (2, 'norm', 2),
    'correlation': (2, 'centre', 2),
    'pearson': (2, 'centre', 3),
    'spearman': (2, 'rank', 3),
}
# modes whose host function keeps float32 input in float32 (sklearn's own euclidean / cosine); the others return float64
KEEPS_FLOAT32 = ('euclidean', 'l2', 'cosine')
SLAB_BYTES = 256 << 20    # float64 bytes of one column slab on its way to the device
SPEARMAN_NAN = 'Data is not well conditioned for spearman method (scipy.stats.spearmanr returned ``np.nan``)'


def _is_sparse(X):
    return hasattr(X, 'tocsc') and not isinstance(X, np.ndarray)


def column_slabs(X, width):
    """[n, <= width] C-contiguous float64 column slabs of X in column order. A scipy.sparse X is sliced from one CSC copy:
    only one slab is ever dense."""
    d = X.shape[1]
    if _is_sparse(X):
        X = X.tocsc()
    for c0 in range(0, d, width):
        c1 = min(d, c0 + width)
        if _is_sparse(X):
            yield np.ascontiguousarray(X[:, c0:c1].toarray(), np.float64)
        else:
            yield np.ascontiguousarray(X[:, c0:c1], np.float64)


def _rank_rows(X, rows=4096):
    from scipy import stats
    n = X.shape[0]
    R = np.empty(X.shape, np.float64)
    for r0 in range(0, n, rows):
        blk = X[r0:r0 + rows]
        R[r0:r0 + rows] = stats.rankdata(blk.toarray() if _is_sparse(blk) else np.asarray(blk), axis=1)
    return R


def prepared_slabs(X, prep, width):
    """The column slabs the handle accumulates: X itself, or X with every row normalised / centred / ranked (see
    GPU_DISTANCE_MODES). Row statistics take one pass over the slabs per statistic, in float64."""
    if prep == 'rank':
        X, prep = _rank_rows(X), 'centre'     # ranks are dense whatever the input
    if prep is None:
        yield from column_slabs(X, width)
        return
    n, d = X.shape
    shift = np.zeros(n)
    if prep == 'centre':
        for s in column_slabs(X, width):
            shift += s.sum(axis=1)
        shift /= d
    ss = np.zeros(n)
    for s in column_slabs(X, width):
        ss += ((s - shift[:, None]) ** 2).sum(axis=1)
    scale = np.sqrt(ss)
    if prep == 'norm':
        scale[scale == 0] = 1.0
    with np.errstate(invalid='ignore', divide='ignore'):
        for s in column_slabs(X, width):
            yield (s - shift[:, None]) / scale[:, None]


def knn_list_width(n, kmax):
    """K': the largest k the connectivity loop of geodesic_distances can reach (the first odd k >= 5 above
    max(kmax, 0.01 n)), capped at n."""
    k = 5
    while not k > max(kmax, 0.01 * n):
        k += 2
    return min(k, n)


def connectivity_k(idx, kmax):
    """The k at which geodesic_distances stops: from 5 in steps of 2 until the undirected graph of the first min(k, n)
    neighbours of every row is connected or k > max(kmax, 0.01 n). idx: [n, >= K'] neighbour lists, nearest first."""
    import scipy.sparse as sp
    import scipy.sparse.csgraph as csg
    n = idx.shape[0]

    def graph(k_):
        k_ = min(k_, n)
        return sp.csr_matrix((np.ones(n * k_), np.asarray(idx[:, :k_]).ravel(), np.arange(0, n * k_ + 1, k_)), shape=(n, n))

    k = 5
    while csg.connected_components(graph(k), directed=False)[0] != 1:
        if k > max(kmax, 0.01 * n):
            break
        k += 2
    return k


class DeviceDistances:
    """One n x n float64 distance matrix on a CUDA device: the jb_dist handle of the C ABI (include/jamie_b200.h)."""

    def __init__(self, n, device):
        import ctypes as C
        from . import _lib
        self._C, self._check, self.lib, self.n = C, _lib.check, _lib.load(), int(n)
        self.h = C.c_void_p()
        self._check(self.lib.jb_dist_create(self.n, int(device), C.byref(self.h)))

    def _ptr(self, a):
        return None if a is None else a.ctypes.data_as(self._C.c_void_p)

    def accumulate(self, kind, slab):
        slab = np.ascontiguousarray(slab, np.float64)
        assert slab.ndim == 2 and slab.shape[0] == self.n
        self._check(self.lib.jb_dist_accumulate(self.h, kind, self._ptr(slab), slab.shape[1], slab.shape[1]))

    def finish(self, transform, copy=True):
        out = np.empty((self.n, self.n)) if copy else None
        self._check(self.lib.jb_dist_finish(self.h, transform, self._ptr(out)))
        return out

    def knn(self, k):
        idx, dist = np.empty((self.n, k), np.int32), np.empty((self.n, k))
        self._check(self.lib.jb_dist_knn(self.h, int(k), self._ptr(idx), self._ptr(dist)))
        return idx, dist

    def geodesic(self, k, copy=True):
        out = np.empty((self.n, self.n)) if copy else None
        self._check(self.lib.jb_dist_geodesic(self.h, int(k), self._ptr(out)))
        return out

    def close(self):
        if self.h:
            self.lib.jb_dist_destroy(self.h)
            self.h = self._C.c_void_p()


def gpu_distance_function(distance_mode, kmax, device=0, matrix=DeviceDistances):
    """GPU counterpart of ``distance_function``: same shapes, dtypes and exceptions, with the n^2 d distance work, the
    kNN selection and the all-pairs shortest paths on the device (``matrix``: the device matrix class; a stand-in with
    the same methods runs the host side without a GPU). A mode without a GPU path warns and runs the host function."""
    if distance_mode not in GPU_DISTANCE_MODES:
        warnings.warn(f'distance_mode {distance_mode!r} has no GPU path: its distances are computed on the host')
        return distance_function(distance_mode, kmax)
    kind, prep, transform = GPU_DISTANCE_MODES[distance_mode]
    host_fn = distance_function(distance_mode, kmax)

    def fn(df):
        n, d = df.shape
        if n == 1 and distance_mode in ('pearson', 'spearman'):
            return host_fn(df)      # the host's one-element special case (O(d) work)
        m = matrix(n, device)
        try:
            for slab in prepared_slabs(df, prep, max(1, min(d, SLAB_BYTES // (8 * n)))):
                m.accumulate(kind, slab)
            if distance_mode == 'geodesic':
                m.finish(transform, copy=False)
                idx, _ = m.knn(knn_list_width(n, kmax))
                out = m.geodesic(min(connectivity_k(idx, kmax), n))
            else:
                out = m.finish(transform)
        finally:
            m.close()
        if distance_mode == 'spearman' and np.isnan(out).any():
            raise Exception(SPEARMAN_NAN)
        if df.dtype == np.float32 and distance_mode in KEEPS_FLOAT32:
            out = out.astype(np.float32)
        return out
    return fn


def prime_dual(Kx, Ky, dx, dy, epoch_pd=2000, epsilon=0.01, rho=10, delay=0, log_pd=100, verbose=True, device='cuda'):
    """F (m x n, fp32 ndarray) minimising ||a Kx - F Ky F^T|| under soft row / column constraints: jamie/jamie.py:314-414."""
    import torch
    if np.shape(Kx) == (1, 1) and np.shape(Ky) == (1, 1):
        warnings.warn('1x1 distance matrix, escaping...')
        return np.ones((1, 1), np.float32)
    N = int(max(np.shape(Kx)[0], np.shape(Ky)[0]))
    Kx = torch.from_numpy(np.asarray(Kx) / N).float().to(device)
    Ky = torch.from_numpy(np.asarray(Ky) / N).float().to(device)
    a = float(np.sqrt(dy / dx))
    m, n = Kx.shape[0], Ky.shape[0]
    F = torch.zeros((m, n), device=device)
    lam = torch.zeros((1, n), device=device)    # Lambda^T
    mu = torch.zeros((m, 1), device=device)
    S = torch.zeros((1, n), device=device)      # S^T
    m1 = torch.zeros_like(F)
    m2 = torch.zeros_like(F)
    b1, b2, delta = 0.9, 0.999, 10e-8
    trace_kk = torch.sum(Kx * Kx.t())           # trace(Kx Kx)
    for i in range(1, epoch_pd + 1):
        FKy = F @ Ky
        grad = (4.0 * (FKy @ (F.t() @ FKy)) - (4.0 * a) * (Kx @ FKy) + mu + lam
                + rho * (F.sum(dim=1, keepdim=True) + (F.sum(dim=0, keepdim=True) + (S - 2.0))))
        m1 = b1 * m1 + (1 - b1) * grad
        m2 = b2 * m2 + (1 - b2) * grad * grad
        step = (m1 / (1 - b1 ** i)) / (torch.sqrt(m2 / (1 - b2 ** i)) + delta)
        F = (1 - epsilon) * F + epsilon * torch.clamp(F - step, min=0)
        col = F.sum(dim=0, keepdim=True)        # (F^T 1)^T
        S = (1 - epsilon) * S + epsilon * torch.clamp(S - (lam + rho * (col - 1.0 + S)), min=0)
        mu = mu + epsilon * (F.sum(dim=1, keepdim=True) - 1.0)
        lam = lam + epsilon * (col - 1.0 + S)
        if i >= delay:
            FKyFt = (F @ Ky) @ F.t()
            a = torch.sum(Kx * FKyFt.t()) / trace_kk          # trace(Kx F Ky F^T) / trace(Kx Kx)
        if verbose and i % log_pd == 0:
            err = torch.norm(a * Kx - (F @ Ky) @ F.t())
            print('epoch:[{:d}/{:d}] err:{:.4f} alpha:{:.4f}'.format(i, epoch_pd, float(err), float(a)))
    return F.detach().cpu().numpy()
