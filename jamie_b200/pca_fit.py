"""PCA fit with its O(n d^2) work on the GPU (SURVEY.md 8 row N3; the reference calls sklearn's ``PCA(n_components=dim)
.fit_transform(data)`` on the host, jamie/jamie.py:436-452, which dominates "Setup" on large inputs).

The algorithm is sklearn's own ``covariance_eigh`` solver (sklearn/decomposition/_pca.py, ``_fit_full``): column means,
the centred Gram matrix C = (X - mean)^T (X - mean) / (n - 1), a symmetric eigendecomposition of the d x d matrix, the
leading eigenvectors as components with the v-based sign convention (``svd_flip(u_based_decision=False)``: the entry of
largest magnitude of every component is positive).  Here the two passes over the [n, d] matrix run on the GPU
(``jb_pca_colsum``, ``jb_pca_gram``: split fp32-class tensor-core GEMM, float64 accumulation over row chunks); only the
d x d eigenproblem (independent of n) is solved on the host with LAPACK.  With the rows sharded over data-parallel ranks
every rank reduces its own rows and the column sums / Gram matrices are all-reduced (one d-vector, one d x d matrix).

The result is returned as a genuine ``sklearn.decomposition.PCA`` object with its fitted attributes set, so that
``preclass`` pickles exactly like the reference's and a checkpoint written here still opens in the reference.
"""
import numpy as np


def _all_reduce_sum(arr, world, group=None):
    """Sum a float64 host array over the `world` ranks of an initialised torch.distributed group (no-op for one rank)."""
    if world <= 1:
        return arr
    try:
        import torch
        import torch.distributed as dist
    except Exception:   # pragma: no cover
        return arr
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return arr
    t = torch.from_numpy(np.ascontiguousarray(arr))
    if dist.get_backend(group) == 'nccl':
        t = t.cuda()
        dist.all_reduce(t, group=group)
        return t.cpu().numpy()
    dist.all_reduce(t, group=group)
    return t.numpy()


BLOCK_ROWS = 16384   # rows densified at a time when the input is a scipy.sparse matrix (AnnData.X)


def is_sparse(X):
    return hasattr(X, 'toarray') and not isinstance(X, np.ndarray)


def dense_blocks(X, lo=0, hi=None, rows=BLOCK_ROWS):
    """float32 row blocks of X[lo:hi]: the whole range at once for an ndarray, BLOCK_ROWS densified rows at a time for a
    scipy.sparse matrix (column sums, Gram matrices and projections are all additive / independent over row blocks, so a
    sparse single-cell matrix never has to exist densely on the host)."""
    hi = X.shape[0] if hi is None else hi
    if not is_sparse(X):
        if hi > lo:
            yield lo, np.ascontiguousarray(X[lo:hi], np.float32)
        return
    Xr = X.tocsr() if hasattr(X, 'tocsr') else X
    for r0 in range(lo, hi, rows):
        r1 = min(hi, r0 + rows)
        yield r0, np.ascontiguousarray(Xr[r0:r1].toarray(), np.float32)


def gram_pca_fit(engine, X, n_components, rank=0, world=1, group=None):
    """Fit on the rows of this rank's contiguous shard of X (ndarray or scipy.sparse), reduce over ranks; returns
    (components [k, d], mean [d], explained_variance [k], total_variance, n_samples), float64."""
    n, d = X.shape
    lo, hi = n * rank // world, n * (rank + 1) // world
    colsum = np.zeros(d)
    for _, blk in dense_blocks(X, lo, hi):
        colsum += engine.pca_colsum(blk)
    colsum = _all_reduce_sum(colsum, world, group)
    mean = colsum / n
    gram = np.zeros((d, d))
    for _, blk in dense_blocks(X, lo, hi):
        gram += engine.pca_gram(blk, mean)
    gram = _all_reduce_sum(gram, world, group)
    gram = (gram + gram.T) * 0.5                      # the tensor-core product is symmetric only to rounding
    C = gram / max(n - 1, 1)
    evals, evecs = np.linalg.eigh(C)                   # ascending
    evals = evals[::-1]
    evecs = evecs[:, ::-1]
    evals = np.maximum(evals, 0.0)                     # sklearn clips the round-off negatives the same way
    total_var = float(evals.sum())
    comps = evecs[:, :n_components].T.copy()
    # svd_flip(u_based_decision=False): sign of the largest-magnitude entry of every component row is positive
    idx = np.argmax(np.abs(comps), axis=1)
    signs = np.sign(comps[np.arange(comps.shape[0]), idx])
    signs[signs == 0] = 1
    comps *= signs[:, None]
    return comps, mean, evals[:n_components].copy(), total_var, n


def fit_sklearn_pca(engine, X, n_components, rank=0, world=1, group=None):
    """``PCA(n_components).fit(X)`` with the GPU Gram route; returns the fitted sklearn object."""
    from sklearn.decomposition import PCA
    comps, mean, ev, total_var, n = gram_pca_fit(engine, X, n_components, rank, world, group)
    d = comps.shape[1]
    pca = PCA(n_components=n_components)
    pca.n_samples_ = n
    pca.n_features_in_ = d
    pca.n_components_ = int(n_components)
    pca.components_ = comps
    pca.mean_ = mean
    pca.explained_variance_ = ev
    pca.explained_variance_ratio_ = ev / total_var if total_var > 0 else np.zeros_like(ev)
    pca.singular_values_ = np.sqrt(ev * max(n - 1, 1))
    rest = min(n, d) - n_components
    pca.noise_variance_ = float((total_var - ev.sum()) / rest) if rest > 0 else 0.0
    pca._fit_svd_solver = 'covariance_eigh'
    return pca


def fit_transform(engine, X, n_components, rank=0, world=1, group=None):
    """(fitted sklearn PCA, sample = the projected training matrix [n, k] float64): what ``pca.fit_transform(data)`` gives
    the reference (jamie/jamie.py:451); the projection is ``jb_pca_project`` without standardisation."""
    pca = fit_sklearn_pca(engine, X, n_components, rank, world, group)
    sample = np.empty((X.shape[0], int(n_components)), np.float64)
    for r0, blk in dense_blocks(X):
        sample[r0:r0 + blk.shape[0]] = engine.pca_project(blk, pca.components_, pca.mean_, 0.0, 1.0)
    return pca, sample


# ------------------------------------------------------------------------------------------------ randomized fit
# For wide inputs (tens of thousands of features) the d x d Gram matrix above no longer fits, and its host eigensolver
# takes hours. sklearn's own randomized solver, which ``PCA(n_components).fit_transform`` picks for such data
# (svd_solver='auto'), never forms it: it only multiplies the centred matrix and its transpose by thin [*, k + 10]
# matrices. Here those products run on the GPU (the jb_pcaop handle: 3xTF32 GEMM for a dense X, a CSR x dense kernel for
# a scipy.sparse X, which is never densified) and the small dense algebra around them stays plumbing.

class DeviceOperator:
    """The centred data operand Xc = X - 1 mean^T resident on one CUDA device: the jb_pcaop handle of the C ABI
    (include/jamie_b200.h). Arrays handed to and returned by ``apply`` are float32 torch tensors on that device."""

    def __init__(self, X, device):
        import ctypes as C
        import torch
        from . import _lib
        self._C, self._check, self.lib = C, _lib.check, _lib.load()
        self.torch, self.device = torch, torch.device('cuda', int(device))
        self.n, self.d = (int(s) for s in X.shape)
        self.h = C.c_void_p()
        p = lambda a: a.ctypes.data_as(C.c_void_p)
        if is_sparse(X):
            R, T = X.tocsr(), X.tocsc()
            parts = []
            for M in (R, T):
                if not M.has_canonical_format:    # sorted indices, no duplicates (without touching the caller's X)
                    M = M.copy()
                    M.sum_duplicates()
                parts += [np.ascontiguousarray(M.indptr, np.int64), np.ascontiguousarray(M.indices, np.int32),
                          np.ascontiguousarray(M.data, np.float32)]
            self._check(self.lib.jb_pcaop_create_sparse(self.n, self.d, int(parts[0][-1]), *(p(a) for a in parts),
                                                        int(device), C.byref(self.h)))
        else:
            Xf = np.ascontiguousarray(X, np.float32)
            self._check(self.lib.jb_pcaop_create_dense(p(Xf), self.n, self.d, int(device), C.byref(self.h)))

    def stats(self):
        """(mean [d], var [d]) float64, var with ddof 0; the mean is kept for the centring of ``apply``"""
        mean, var = np.empty(self.d), np.empty(self.d)
        self._check(self.lib.jb_pcaop_stats(self.h, mean.ctypes.data_as(self._C.c_void_p), var.ctypes.data_as(self._C.c_void_p)))
        return mean, var

    def upload(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(self.device)

    def apply(self, trans, B):
        """Xc @ B (trans 0, B [d, l]) or Xc.T @ B (trans 1, B [n, l])"""
        B = B.to(device=self.device, dtype=self.torch.float32).contiguous()
        rows, out = (self.n, self.d) if trans else (self.d, self.n)
        assert B.ndim == 2 and B.shape[0] == rows, (tuple(B.shape), trans)
        Y = self.torch.empty((out, B.shape[1]), dtype=self.torch.float32, device=self.device)
        stream = self.torch.cuda.current_stream(self.device).cuda_stream
        self._check(self.lib.jb_pcaop_apply(self.h, int(trans), B.data_ptr(), int(B.shape[1]), Y.data_ptr(), stream))
        return Y

    def orth(self, Y):
        """orthonormal basis of the columns of Y (economic QR; the column span is all the range finder needs)"""
        return self.torch.linalg.qr(Y, mode='reduced')[0]

    def download(self, Y):
        return Y.double().cpu().numpy()

    def close(self):
        if self.h:
            self.torch.cuda.synchronize(self.device)
            self.lib.jb_pcaop_destroy(self.h)
            self.h = self._C.c_void_p()


def _svd_flip_v(U, Vt):
    """sklearn's svd_flip(u_based_decision=False): the entry of largest magnitude of every row of Vt is positive"""
    idx = np.argmax(np.abs(Vt), axis=1)
    signs = np.sign(Vt[np.arange(Vt.shape[0]), idx])
    signs[signs == 0] = 1
    return U * signs[None, :], Vt * signs[:, None]


def randomized_fit_transform(X, n_components, seed, device=0, operator=DeviceOperator):
    """``PCA(n_components, svd_solver='randomized').fit_transform(X)`` (sklearn's ``_fit_truncated`` and
    ``_randomized_svd``: n_oversamples 10, n_iter 7 if k < 0.1 min(n, d) else 4, the transposed problem when n < d) with
    the products on the device. Omega is drawn with ``np.random.default_rng(seed)``, so the fit is reproducible; the power
    iterations are orthonormalised with a QR instead of sklearn's LU (the same column span in exact arithmetic).
    X: ndarray or any scipy.sparse matrix (never densified). ``operator``: the operand class (a stand-in with the same
    methods runs the driver without a GPU). Returns (fitted sklearn PCA, sample = U[:, :k] S[:k], float64 [n, k])."""
    import scipy.linalg
    from sklearn.decomposition import PCA
    n, d = X.shape
    k = int(n_components)
    if not 1 <= k <= min(n, d):
        raise ValueError(f'n_components={k} must be between 1 and min(n_samples, n_features)={min(n, d)}')
    l = min(k + 10, n, d)                        # the economic QR caps the sketch width at min(n, d)
    n_iter = 7 if k < 0.1 * min(n, d) else 4
    transpose = n < d                            # work on A = Xc^T [d, n] when the matrix is wide
    fwd, bwd = (1, 0) if transpose else (0, 1)   # A @ Q and A^T @ Q as operand products
    op = operator(X, device)
    try:
        mean, var = op.stats()
        omega = np.random.default_rng(seed).standard_normal((n if transpose else d, l), dtype=np.float32)
        Q = op.upload(omega)
        for _ in range(n_iter):
            Q = op.orth(op.apply(fwd, Q))
            Q = op.orth(op.apply(bwd, Q))
        Q = op.orth(op.apply(fwd, Q))
        Bt = op.download(op.apply(bwd, Q))       # B^T = A^T Q: [cols(A), l]
        Q = op.download(Q)
    finally:
        op.close()
    Uhat, S, Vt = scipy.linalg.svd(Bt.T, full_matrices=False, lapack_driver='gesdd')
    U = Q @ Uhat                                 # [rows(A), l]
    if transpose:                                # the SVD of Xc itself: U' = Vt^T, Vt' = U^T
        U, Vt = Vt.T, U.T
    U, Vt = _svd_flip_v(U, Vt)
    U, S, Vt = U[:, :k], S[:k], Vt[:k]
    ev = S ** 2 / max(n - 1, 1)
    total_var = float(var.sum() * n / max(n - 1, 1))
    pca = PCA(n_components=k, svd_solver='randomized', random_state=seed)
    pca.n_samples_ = n
    pca.n_features_in_ = d
    pca.n_components_ = k
    pca.components_ = np.ascontiguousarray(Vt)
    pca.mean_ = mean
    pca.explained_variance_ = ev
    pca.explained_variance_ratio_ = ev / total_var if total_var > 0 else np.zeros_like(ev)
    pca.singular_values_ = S.copy()
    pca.noise_variance_ = float((total_var - ev.sum()) / (min(n, d) - k)) if k < min(n, d) else 0.0
    pca._fit_svd_solver = 'randomized'
    return pca, U * S[None, :]
