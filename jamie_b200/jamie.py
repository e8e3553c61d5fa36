"""``JAMIE``: host-side mirror of the reference class (jamie/jamie.py:29-222, 416-837, 967-972) driving the CUDA engine.

Same constructor arguments, methods, attributes, printed lines and error messages as the reference for the hot path
(fit_transform -> project_jamie training loop, transform, transform_one, modal_predict, save_model, load_model).
Everything numeric runs in ``libjamie_b200.so``: the per-step work of the reference loop (batch gather, P/F blocks,
model forward, the four losses, backward, clip, Adam) is one CUDA-graph launch per optimizer step; the host keeps the
numpy batch sampler (same draws, same order as the reference, so a seeded run visits the same cells), the epoch
bookkeeping, early stopping and printing.

F estimation (``compute_distances`` + ``Prime_Dual``, jamie/jamie.py:224-414, 839-890) lives in ``correspondence.py``: the
distances on the host with the reference's own sklearn / scipy calls (``distances='gpu'``: on the GPU, csrc/distances.cuh),
the primal-dual iteration on the GPU.  Out of scope:
the tsne projection branch, ``corr_method='jamie'`` (marked WIP in the reference), ``model_pca='umap'``.
"""
import os
import time as _time
import warnings

import numpy as np
import torch

from .engine import Engine
from .model import edModelVar
from .unioncom_shim import UnionCom, init_random_seed
from .utilities import make_pca, preclass, time_logger

DISTANCE_MODES = [
    'euclidean', 'l2', 'l1', 'manhattan', 'cityblock', 'braycurtis', 'canberra', 'chebyshev', 'correlation', 'cosine',
    'dice', 'hamming', 'jaccard', 'kulsinski', 'mahalanobis', 'matching', 'minkowski', 'rogerstanimoto', 'russellrao',
    'seuclidean', 'sokalmichener', 'sokalsneath', 'sqeuclidean', 'yule', 'wminkowski', 'nan_euclidean', 'haversine',
    'geodesic', 'spearman', 'pearson',
]


def _dist_info():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_rows_apply(fn, data):
    """Row-sharded inference (SURVEY 8e: "inference shards trivially by rows"): under torch.distributed every rank calls
    this with the SAME ``data``; rank r runs ``fn`` on rows [n r / R, n (r + 1) / R) only and one all-gather hands every
    rank the full [n, d_out] result. No collective on the data path itself. One process: ``fn(data)``."""
    rank, world = _dist_info()
    if world == 1:
        return fn(data)
    import torch.distributed as dist
    n = len(data)
    lo, hi = (n * rank) // world, (n * (rank + 1)) // world
    part = np.ascontiguousarray(fn(data[lo:hi]))
    rows_max = -(-n // world)
    dev = 'cuda' if dist.get_backend() == 'nccl' else 'cpu'
    buf = torch.zeros((rows_max,) + part.shape[1:], dtype=torch.from_numpy(part).dtype, device=dev)
    buf[:hi - lo] = torch.from_numpy(part).to(dev)
    out = [torch.empty_like(buf) for _ in range(world)]
    dist.all_gather(out, buf)
    pieces = [out[r][:(n * (r + 1)) // world - (n * r) // world].cpu().numpy() for r in range(world)]
    return np.concatenate(pieces, axis=0)


class PriorSpec:
    """Correspondence prior in the most compact form that reproduces the reference's dense-matrix semantics."""

    def __init__(self, P, rows, method=None):
        # method: force the sampling method (data-parallel shards take the method of the GLOBAL prior)
        self.rows = rows
        self.diag = None      # 1-D mask m: P = diag(m)
        self.dense = None     # 2-D ndarray
        if P is None:
            # jamie/jamie.py:423-428: identity iff the datasets have the same number of rows, else zeros
            if rows[0] == rows[1]:
                self.diag = np.ones(rows[0], np.float32)
        else:
            if hasattr(P, 'toarray') and not isinstance(P, np.ndarray):   # scipy sparse
                d = np.asarray(P.diagonal()).ravel() if P.shape[0] == P.shape[1] else None
                if d is not None and P.count_nonzero() == np.count_nonzero(d):
                    P = d
                else:
                    P = P.toarray()
            P = np.asarray(P)
            if P.ndim == 1:
                assert rows[0] == rows[1] == P.shape[0], 'a 1-D prior is diag(m) and needs equally sized datasets'
                self.diag = P.astype(np.float32)
            else:
                assert P.shape == (rows[0], rows[1]), f'P must be {rows[0]} x {rows[1]}'
                if P.shape[0] == P.shape[1] and np.count_nonzero(P) == np.count_nonzero(np.diagonal(P)):
                    self.diag = np.diagonal(P).astype(np.float32)
                else:
                    self.dense = P.astype(np.float32)
        if self.diag is not None and not np.any(self.diag):
            self.diag = None
        # jamie/jamie.py:518-534
        if self.diag is not None and np.all(self.diag == 1):
            self.sampling_method = 'diag'
        elif self.diag is not None or (self.dense is not None and np.abs(self.dense).sum() != 0):
            self.sampling_method = 'hybrid'
        else:
            self.sampling_method = 'zeros'
            self.dense = None
        if method is not None and method != self.sampling_method:
            # a shard of a partially matched prior can be fully matched or empty: keep the global method where the shard
            # supports it ('hybrid' needs two positive entries, checked below), never a stricter one
            self.sampling_method = method if not (method == 'diag' and (self.diag is None or not np.all(self.diag == 1))) else self.sampling_method
        self.corr_samples = None
        if self.sampling_method == 'hybrid':
            # torch.argwhere(P > 0), of which the reference only ever reads rows 0 and 1 (jamie/jamie.py:525-526, 566)
            if self.diag is not None:
                nz = np.flatnonzero(self.diag > 0)[:2]
                self.corr_samples = np.stack([nz, nz], axis=1)
            else:
                self.corr_samples = np.argwhere(self.dense > 0)[:2]
            if len(self.corr_samples) < 2:
                if method is not None:      # a shard without two matched pairs samples uniformly
                    warnings.warn('this rank\'s shard of P has fewer than two positive entries: sampling uniformly')
                    self.sampling_method = 'zeros'
                    self.corr_samples = None
                else:
                    raise IndexError('hybrid sampling needs at least two positive entries in P')

    def upload(self, engine):
        if self.dense is not None:
            engine.set_prior_dense(self.dense)
        else:
            engine.set_prior_diag(self.diag)

    def to_dense(self):
        if self.dense is not None:
            return self.dense
        if self.diag is not None:
            return np.diag(self.diag)
        return np.zeros(self.rows, np.float32)


# Above this many rows numpy's legacy `np.random.choice(n, k, replace=False)` (a full permutation of n per call: 1.5 ms
# at n = 50k, 20 ms at n = 1M, measured) would starve the GPU step (0.27 ms), so `sampler='auto'` switches to an O(k) draw.
FAST_SAMPLER_ROWS = 16384


def sample_batch(method, rows, cols, batch_size, corr_samples=None, fast_rng=None):
    """Batch indices of one optimizer step: jamie/jamie.py:553-579, same numpy draws in the same order.

    fast_rng (a numpy Generator): draws without replacement come from `fast_rng.choice` instead of the legacy global
    `np.random.choice` -- the same distribution (a uniformly random k-subset in random order) in O(k) instead of O(n),
    but not the reference's random stream."""
    rep = min(ci for ci in cols) < batch_size

    def choice(n, k):
        if fast_rng is not None and not rep:
            return fast_rng.choice(n, k, replace=False)
        return np.random.choice(n, k, replace=rep)

    if method == 'diag':
        set_rand = choice(rows[0], batch_size) if fast_rng is not None else np.random.choice(range(rows[0]), batch_size, replace=rep)
        return [set_rand, set_rand]
    if method == 'hybrid':
        num_corr = len(corr_samples[0])   # == 2: the reference's self.num_corr (jamie/jamie.py:526)
        corr_sample_num = min(np.sum(np.random.rand(batch_size) < .8), num_corr)
        non_sample_num = batch_size - corr_sample_num
        corr_idx = np.random.choice(num_corr, corr_sample_num, replace=rep)
        out = []
        for i in range(2):
            head = np.asarray(corr_samples[i])[corr_idx]
            out.append(np.concatenate([head, choice(rows[i], non_sample_num)], axis=0))
        return out
    if method == 'zeros':
        if fast_rng is not None:
            return [choice(rows[i], batch_size) for i in range(2)]
        return [np.random.choice(range(rows[i]), batch_size, replace=rep) for i in range(2)]
    raise Exception(f'Sampling method {method} does not exist')


def chunk_epochs(first_epoch, streak_bound, min_epochs, max_steps_without_increment, use_early_stop, epoch_DNN,
                 len_dataloader, max_steps=4096):
    """How many epochs can be enqueued from `first_epoch` on without a host decision in between, given an upper bound of
    the early-stopping streak at that point: early stopping (jamie/jamie.py:777-792) is only evaluated once
    epoch > min_epochs, the streak then grows by at most one per epoch, and training stops when it reaches
    max_steps_without_increment -- so the earliest possible stop is always the LAST epoch of the chunk."""
    safe = max(1, (min_epochs + 1 - first_epoch) if first_epoch <= min_epochs else 0) \
        + max(0, max_steps_without_increment - streak_bound - 1) if use_early_stop else epoch_DNN
    return int(min(epoch_DNN - first_epoch, max(1, safe), max(1, max_steps // len_dataloader)))


class JAMIE(UnionCom):
    """
    Adaptation of https://github.com/caokai1073/UnionCom by caokai1073

    P: Correspondence prior matrix
    PF_Ratio: Ratio of priors:assumed correspondence; .5 is equal, 1 is only P
    in_place: Whether to do the calculation in place.  Will save memory but may
        alter original data
    """

    def __init__(self, match_result=None, PF_Ratio=None, corr_method='unioncom', dist_method='euclidean',
                 in_place=False, loss_weights=None, model_pca='pca', model_class=edModelVar, model_lr=1e-3,
                 dropout=None, pca_dim=2 * [512], batch_step=True, use_f_tilde=True, use_early_stop=True,
                 min_epochs=2500, min_increment=1e-8, max_steps_without_increment=500, debug=False, log_debug=100,
                 record_loss=True, enable_memory_logging=False, device='cpu', sampler='auto', pca_fit='gpu', distances='host',
                 **kwargs):
        # sampler (not in the reference): 'reference' = the reference's numpy draws call for call; 'fast' = the same
        # distribution from an O(batch) draw; 'auto' = 'reference' up to FAST_SAMPLER_ROWS cells, 'fast' above.
        assert sampler in ('auto', 'reference', 'fast'), f"sampler must be 'auto', 'reference' or 'fast', not {sampler!r}"
        self.sampler = sampler
        # pca_fit (not in the reference): 'gpu' = column sums + Gram matrix on the GPU, d x d eigensolver on the host (sklearn's
        # covariance_eigh algorithm, exact PCA); 'sklearn' = the reference's host call PCA(n_components).fit_transform(data);
        # 'randomized' = sklearn's randomized solver with its products on the GPU (wide and sparse inputs: no d x d matrix,
        # a scipy.sparse input is never densified; seeded with manual_seed).
        assert pca_fit in ('gpu', 'sklearn', 'randomized'), \
            f"pca_fit must be 'gpu', 'sklearn' or 'randomized', not {pca_fit!r}"
        self.pca_fit = pca_fit
        # distances (not in the reference): 'host' = compute_distances with the reference's sklearn / scipy calls; 'gpu' = the
        # same distances from the jb_dist kernels on the engine's device (correspondence.gpu_distance_function; a scipy.sparse
        # modality is streamed in column slabs, never densified whole).
        assert distances in ('host', 'gpu'), f"distances must be 'host' or 'gpu', not {distances!r}"
        self.distances = distances
        self.match_result = match_result
        self.PF_Ratio = PF_Ratio
        self.corr_method = corr_method
        self.dist_method = dist_method
        self.in_place = in_place
        self.loss_weights = loss_weights
        self.model_pca = model_pca
        self.model_class = model_class
        self.model_lr = model_lr
        self.dropout = dropout
        self.pca_dim = pca_dim
        self.batch_step = batch_step
        self.use_f_tilde = use_f_tilde
        self.use_early_stop = use_early_stop
        self.min_epochs = min_epochs
        self.min_increment = min_increment
        self.max_steps_without_increment = max_steps_without_increment
        self.debug = debug
        self.log_debug = log_debug
        self.record_loss = record_loss
        self.enable_memory_logging = enable_memory_logging
        # The reference defaults to 'cpu' and warns that its GPU path is incomplete (jamie/jamie.py:88-96).
        # This implementation has exactly one path, the CUDA engine: any value selects the process's CUDA device.
        self.device = device
        defaults = {'project_mode': 'jamie', 'log_pd': 500, 'lr': 1e-3, 'epoch_DNN': 10000, 'log_DNN': 500,
                    'batch_size': 512}
        for k, v in defaults.items():
            if k not in kwargs:
                kwargs[k] = v
        super().__init__(**kwargs)
        self.model = None
        self.engine = None
        self.P = None
        self.F = None
        self.dataset = None
        self.dataset_num = 2

    # ------------------------------------------------------------------------------------------------ device
    def _cuda_index(self):
        if not torch.cuda.is_available():
            raise RuntimeError('jamie_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback')
        dev = str(self.device)
        if dev.startswith('cuda:'):
            return int(dev.split(':')[1])
        return int(os.environ.get('LOCAL_RANK', torch.cuda.current_device()))

    @staticmethod
    def _stream():
        return torch.cuda.current_stream().cuda_stream

    # ------------------------------------------------------------------------------------------------ fit
    def fit_transform(self, dataset=None, P=None):
        """Fit function with ``nlma`` added"""
        self.P = P
        if self.integration_type not in ['MultiOmics']:
            raise Exception('integration_type error! Enter MultiOmics.')
        if self.distance_mode not in DISTANCE_MODES:
            raise Exception('distance_mode error! Enter a correct distance_mode.')
        if self.project_mode not in ('jamie', 'tsne'):
            raise Exception("Choose correct project_mode: 'nlma', 'tsne'.")
        assert self.model_pca in ('pca', 'umap')
        if self.project_mode == 'tsne':
            raise NotImplementedError("project_mode='tsne' (UnionCom's legacy projection) is outside this build's scope")
        if self.model_pca != 'pca':
            raise NotImplementedError("model_pca='umap' is outside this build's scope")

        time = time_logger(memory_usage=self.enable_memory_logging)
        init_random_seed(self.manual_seed)

        # Test for dataset type (must all be the same): AnnData inputs carry the matrix in .X
        self.dataset = dataset
        self.dataset_annotation = None
        if not isinstance(self.dataset[0], np.ndarray) and hasattr(self.dataset[0], 'X'):
            self.dataset = [d.X for d in self.dataset]
            self.dataset_annotation = dataset
        if not self.in_place:
            self.dataset = [d * 1 for d in self.dataset]
        self.dataset_num = len(self.dataset)
        self.col = []
        self.row = []
        for i in range(self.dataset_num):
            self.row.append(np.shape(self.dataset[i])[0])
            self.col.append(np.shape(self.dataset[i])[1])
        # Distances (jamie/jamie.py:160-166): needed only to estimate F
        need_dist = self.match_result is None and self.use_f_tilde
        self.compute_distances(save_dist=need_dist)
        time.log('Distance')

        # Correspondence between samples: supplied, zeros (use_f_tilde=False, jamie/jamie.py:172-173) or estimated with
        # Prime_Dual on the GPU. The reference's per-pair linear_sum_assignment (jamie/jamie.py:177-181) only feeds the
        # tsne branch: skipped.
        if not self.use_f_tilde:
            self.match_result = None
            self._F_dense = None
        else:
            if self.match_result is None:
                self.match_result = self.match()
            self._F_dense = np.asarray(self.match_result[0], np.float32)
        time.log('Correspondence')

        integrated_data = self.project_jamie(None)
        time.log('Mapping')

        print('-' * 33)
        print('JAMIE Done!')
        time.aggregate()
        print()
        return integrated_data

    # ------------------------------------------------------------------------------------------------ F estimation
    def compute_distances(self, save_dist=True):
        """Helper function to compute distances for each dataset (jamie/jamie.py:839-890)"""
        from .correspondence import distance_function, gpu_distance_function
        if save_dist:
            self.dist = []
        gpu_fn = None
        if save_dist and self.distances == 'gpu':
            gpu_fn = gpu_distance_function(self.distance_mode, self.kmax, device=self._cuda_index())
        print('Shape of Raw data')
        for i in range(self.dataset_num):
            print('Dataset {}:'.format(i), np.shape(self.dataset[i]))
            self.distance_function = gpu_fn or distance_function(self.distance_mode, self.kmax)
            if save_dist:
                data_i = self.dataset[i]
                if gpu_fn is None and hasattr(data_i, 'toarray') and not isinstance(data_i, np.ndarray):   # scipy.sparse (AnnData.X)
                    data_i = data_i.toarray()
                self.dist.append(self.distance_function(data_i))

    def match(self):
        """Find correspondence between multi-omics datasets (jamie/jamie.py:224-250)"""
        print('Device:', self.device)
        cor_pairs = []
        for i in range(self.dataset_num):
            for j in range(i + 1, self.dataset_num):
                print('-' * 33)
                print(f'Find correspondence between Dataset {i + 1} and Dataset {j + 1}')
                if self.corr_method == 'unioncom':
                    F = self.Prime_Dual([self.dist[i], self.dist[j]], dx=self.col[i], dy=self.col[j])
                elif self.corr_method == 'jamie':
                    raise NotImplementedError("corr_method='jamie' is marked WIP / unreliable in the reference "
                                              '(jamie/jamie.py:241-246) and is not built')
                else:
                    raise Exception(f'corr_method {self.corr_method!r} does not exist')
                cor_pairs.append(F)
        print('Finished Matching!')
        return cor_pairs

    def Prime_Dual(self, dist, dx=None, dy=None, verbose=True):
        """Prime dual combined with Adam algorithm to find the local optimal solution (jamie/jamie.py:314-414)"""
        from .correspondence import prime_dual
        dev = self._cuda_index()
        return prime_dual(dist[0], dist[1], dx, dy, epoch_pd=self.epoch_pd, epsilon=self.epsilon, rho=self.rho,
                          delay=self.delay, log_pd=self.log_pd, verbose=verbose, device=f'cuda:{dev}')

    # ------------------------------------------------------------------------------------------------ train
    def project_jamie(self, W=None):
        """Perform alignment using TSNE-like backend"""
        print('-' * 33)
        print('Train coupled autoencoders')
        assert self.dataset_num == 2, 'Currently only compatible with 2 modalities.'
        rank, world = _dist_info()
        timer = time_logger()

        # ---- preprocessing (jamie/jamie.py:433-469). The PCA fit runs its two passes over the [n, d] matrix on the GPU
        # (column sums + centred Gram matrix, rows sharded over the data-parallel ranks and all-reduced; pca_fit.py) and
        # only the d x d eigenproblem on the host -- sklearn's covariance_eigh algorithm, returned as a fitted sklearn PCA.
        # The projection + standardisation of the whole dataset runs on the GPU once the engine exists (below).
        pca_list, pca_inv_list, cols = [], [], []
        dims_req = self.pca_dim if self.pca_dim is not None else [None] * self.dataset_num
        fit_engine = None
        for i_mod, (dim, data) in enumerate(zip(dims_req, self.dataset)):
            if dim is not None:
                if min(*data.shape) < dim:
                    warnings.warn(
                        f'PCA dim must be lower than {min(*data.shape)}, found {dim}, '
                        f'adjusting to compensate.')
                    dim = min(*data.shape)
                if self.pca_fit == 'gpu':
                    from . import pca_fit
                    if fit_engine is None:   # a minimal handle: the PCA entry points only need its device and GEMM tables
                        dev0 = self._cuda_index()
                        torch.cuda.set_device(dev0)
                        fit_engine = Engine([8, 8], 2, 8, 0.0, device=dev0)
                    pca, sample = pca_fit.fit_transform(fit_engine, data if pca_fit.is_sparse(data) else np.asarray(data),
                                                        dim, rank, world)
                elif self.pca_fit == 'randomized':
                    # every rank runs the same seeded fit on all rows (no engine needed: the operand owns its device copy)
                    from . import pca_fit
                    dev0 = self._cuda_index()
                    torch.cuda.set_device(dev0)
                    pca, sample = pca_fit.randomized_fit_transform(data if pca_fit.is_sparse(data) else np.asarray(data), dim,
                                                                   seed=self.manual_seed, device=dev0)
                else:
                    pca = make_pca(dim)
                    sample = pca.fit_transform(data)
                pre = preclass(sample, pca=pca)
                cols.append(int(sample.shape[1]))
            else:
                if hasattr(data, 'toarray') and not isinstance(data, np.ndarray):   # no PCA on a sparse matrix: it is trained on as is
                    data = self.dataset[i_mod] = data.toarray()
                pre = preclass(data, axis=0)
                cols.append(int(np.shape(data)[1]))
            pca_list.append(pre.transform)
            pca_inv_list.append(pre.inverse_transform)
        if fit_engine is not None:
            fit_engine.close()
        self.col = cols

        # ---- model + optimizer state (jamie/jamie.py:471-481). The engine implements exactly edModelVar (the only model the
        # reference ships): another architecture passed as model_class would be built here and then trained as
        # something else, so it is rejected instead of silently ignored.
        if not (isinstance(self.model_class, type) and issubclass(self.model_class, edModelVar)):
            raise NotImplementedError(f'model_class={self.model_class!r}: the CUDA engine implements jamie.model.edModelVar '
                                      '(or a subclass that keeps its architecture)')
        self.model = self.model_class(self.col, self.output_dim, preprocessing=pca_list,
                                      preprocessing_inverse=pca_inv_list, dropout=self.dropout)
        # Batch size setup (jamie/jamie.py:510-514); with R data-parallel ranks an epoch is max(row)/(B*R) steps
        len_dataloader = int(np.max(self.row) / (self.batch_size * world))
        if len_dataloader == 0:
            len_dataloader = 1
            if world == 1:
                self.batch_size = int(np.max(self.row))
        self.PF_Ratio = 1 if self.PF_Ratio is None else self.PF_Ratio

        # ---- shard the cells over the data-parallel ranks (contiguous ranges; world == 1: everything)
        lo = [(r_ * rank) // world for r_ in self.row]
        hi = [(r_ * (rank + 1)) // world for r_ in self.row]
        prior_full = PriorSpec(self.P, self.row)
        self.sampling_method = prior_full.sampling_method
        self.P = prior_full   # compact prior; .to_dense() materialises the reference's matrix (small n only)
        if world == 1:
            prior = prior_full
            F_local = self._F_dense
        else:
            # rank r keeps the diagonal block P[lo_r:hi_r, lo_r:hi_r] (and the same block of F): correspondences between
            # cells of different ranks are not used by the data-parallel step (north_star: "each rank holding its P
            # sub-block for its batches")
            gm = prior_full.sampling_method
            if prior_full.diag is not None:
                prior = PriorSpec(prior_full.diag[lo[0]:hi[0]], [hi[0] - lo[0], hi[1] - lo[1]], method=gm)
            elif prior_full.dense is not None:
                prior = PriorSpec(prior_full.dense[lo[0]:hi[0], lo[1]:hi[1]], [hi[0] - lo[0], hi[1] - lo[1]], method=gm)
            else:
                prior = PriorSpec(np.zeros((hi[0] - lo[0], hi[1] - lo[1]), np.float32), [hi[0] - lo[0], hi[1] - lo[1]], method=gm)
            F_local = None if self._F_dense is None else self._F_dense[lo[0]:hi[0], lo[1]:hi[1]]
            if rank == 0:   # say so once when a dense P / F has correspondences that the sharding drops
                for name, M_ in (('P', prior_full.dense), ('F', self._F_dense)):
                    if M_ is None:
                        continue
                    kept = sum(int(np.count_nonzero(M_[(self.row[0] * r_) // world:(self.row[0] * (r_ + 1)) // world,
                                                      (self.row[1] * r_) // world:(self.row[1] * (r_ + 1)) // world]))
                               for r_ in range(world))
                    total_nz = int(np.count_nonzero(M_))
                    if kept < total_nz:
                        warnings.warn(f'data-parallel training over {world} ranks uses the diagonal blocks of {name} only: '
                                      f'{total_nz - kept} of its {total_nz} nonzero correspondences link cells of different '
                                      'ranks and are ignored')
        local_rows = [hi[i] - lo[i] for i in range(2)]
        self.F = F_local
        if world > 1 and min(local_rows) < self.batch_size and not (min(self.col) < self.batch_size):
            raise ValueError(f'data-parallel training over {world} ranks needs at least batch_size = {self.batch_size} cells per '
                             f'rank (sampling without replacement); this rank holds {min(local_rows)}. Lower batch_size or '
                             f'the number of ranks.')

        dev = self._cuda_index()
        torch.cuda.set_device(dev)
        if self.dist_method not in ('euclidean', 'cosine'):
            # the reference's sim_diff_func (jamie/jamie.py:484-504) has exactly these two branches; anything else leaves
            # it return None and the first step dies unpacking it
            raise ValueError(f"dist_method='{self.dist_method}': the training loss knows 'euclidean' and 'cosine'")
        self.engine = Engine(self.col, self.output_dim, self.batch_size, self.model.dropout_p, lr=self.model_lr,
                             loss_weights=self.loss_weights, pf_ratio=self.PF_Ratio,
                             seed=(self.manual_seed or 0) * 1000003 + rank, device=dev, world_size=world)
        eng = self.engine
        eng.set_dist_method(self.dist_method)
        self.model.attach_engine(eng)      # also routes preclass PCA projections through the engine (jb_pca_project)
        self.model.push_to_engine()
        # ingest: PCA projection + standardisation of every cell (jamie/jamie.py:458-459)
        self.dataset = [f(x) for f, x in zip(pca_list, self.dataset)]
        stream = self._stream()
        for i in range(2):
            eng.set_dataset(i, np.asarray(self.dataset[i][lo[i]:hi[i]], np.float32), stream)
        prior.upload(eng)
        eng.set_f_dense(F_local)
        if not self.batch_step:
            eng.set_grad_accumulate(False)
        if world > 1:
            import torch.distributed as dist
            from .dp import GradExchange
            gx = GradExchange(eng)   # NVLS multimem / peer-memory all-reduce on an NVSwitch box, else NCCL (gloo on CPU tests)
        self.model.train()
        # O(batch) sampler for large datasets; seeded from numpy's global generator, so np.random.seed(...) in the caller
        # still makes a run reproducible
        use_fast = self.sampler == 'fast' or (self.sampler == 'auto' and max(local_rows) > FAST_SAMPLER_ROWS)
        fast_rng = np.random.default_rng(np.random.randint(0, 2 ** 31 - 1, size=4)) if use_fast else None

        best_running_loss = np.inf
        streak = 0
        if self.record_loss:
            self.loss_history = {}
        names = ['KL', 'Rec', 'CosSim', 'F']
        lw = self.loss_weights
        c = (self.min_epochs / 2) if self.min_epochs > 0 else (self.epoch_DNN / 2)  # Midpoint (jamie/jamie.py:630)
        timer.log('Setup')

        epoch = 0
        stop = False
        t_sample = t_step = 0.0

        def build_chunk(first_epoch, streak_bound):
            """Sampling plan of the next chunk of epochs, starting at `first_epoch`, given an upper bound of the
            early-stopping streak at that point (chunk_epochs)."""
            nonlocal t_sample
            n = chunk_epochs(first_epoch, streak_bound, self.min_epochs, self.max_steps_without_increment,
                             self.use_early_stop, self.epoch_DNN, len_dataloader)
            t0 = _time.perf_counter()
            i0 = np.empty((n * len_dataloader, self.batch_size), np.int64)
            i1 = np.empty_like(i0)
            ann = np.empty(n * len_dataloader, np.float64)
            for e_ in range(n):
                kl_anneal = 1 / (1 + np.exp(-5 * ((first_epoch + e_) - c) / c))
                for b_ in range(len_dataloader):
                    rb = sample_batch(prior.sampling_method, local_rows, self.col, self.batch_size, prior.corr_samples, fast_rng)
                    i0[e_ * len_dataloader + b_] = rb[0]
                    i1[e_ * len_dataloader + b_] = rb[1]
                    ann[e_ * len_dataloader + b_] = kl_anneal
            t_sample += _time.perf_counter() - t0
            return n, i0, i1, ann

        chunk = build_chunk(0, 0) if self.epoch_DNN > 0 else None
        while chunk is not None and not stop:
            n_ep, idx0, idx1, anneal = chunk
            t1 = _time.perf_counter()
            eng.upload_plan(idx0, idx1, anneal, stream)
            nsteps = n_ep * len_dataloader
            if (world == 1 or gx.mode == 'kernel') and self.batch_step:
                eng.train_steps(nsteps, stream)          # (data-parallel: the step kernel exchanges the gradients itself)
            else:
                for s_ in range(nsteps):
                    if not self.batch_step:
                        eng.set_grad_accumulate(s_ % len_dataloader != 0)
                    eng.step_backward(stream)
                    last_of_epoch = (s_ + 1) % len_dataloader == 0
                    if self.batch_step or last_of_epoch:
                        if world > 1:
                            gx.all_reduce()
                        eng.step_update(stream)
            # The steps above are only enqueued: the next chunk's plan is sampled on the host while the GPU runs them.
            # Its size uses the largest streak this chunk can end with, so it never crosses an early-stop decision.
            t_enq = _time.perf_counter()
            chunk = build_chunk(epoch + n_ep, streak + n_ep) if epoch + n_ep < self.epoch_DNN else None
            t1 += _time.perf_counter() - t_enq                # sampling time is booked under 'Get subset samples'
            losses = eng.read_losses(nsteps, stream)          # one device->host read per chunk of epochs
            if world > 1:
                lt = torch.from_numpy(losses).cuda()
                dist.all_reduce(lt)
                losses = (lt / world).cpu().numpy()
            t_step += _time.perf_counter() - t1

            for e_ in range(n_ep):
                blk = losses[e_ * len_dataloader:(e_ + 1) * len_dataloader]
                tot = blk[:, 4].astype(np.float64)
                if not np.all(np.isfinite(tot)):
                    raise FloatingPointError(f'non-finite loss at epoch {epoch + 1}; your lr is likely too high')
                epoch_loss = float(tot.sum() / len_dataloader)
                best_batch_loss = float(tot.min())
                last = blk[-1]
                # Loss reporting: last batch of the epoch, weighted (jamie/jamie.py:752-761)
                if self.record_loss:
                    for k, name in enumerate(names):
                        self.loss_history.setdefault(name, []).append(float(last[k]) * (lw[k] if lw is not None else 1))
                if (epoch + 1) % self.log_debug == 0 and self.debug:
                    if lw is not None:
                        print(f'Epoch: {epoch + 1:d} - ' + '  '.join(
                            f'{names[k]}: {last[k] * lw[k]:.4f}' for k in range(4)))
                    else:
                        print('  '.join(f'{names[k]}: {last[k]:.4f}' for k in range(4)))
                if (epoch + 1) % self.log_DNN == 0:
                    print(f'epoch:[{epoch + 1:d}/{self.epoch_DNN}]: loss:{epoch_loss:4f}')
                # Early stopping (jamie/jamie.py:777-792)
                active_loss = best_batch_loss if self.batch_step else epoch_loss
                if epoch > self.min_epochs:
                    epsilon = best_running_loss - active_loss
                    if epsilon > self.min_increment:
                        best_running_loss = active_loss
                        streak = 0
                    else:
                        streak += 1
                    if streak >= self.max_steps_without_increment and self.use_early_stop:
                        stop = True
                        epoch += 1
                        assert e_ == n_ep - 1, 'early stop inside a chunk: the chunk bound is wrong'
                        break
                epoch += 1
        self.epochs_run = epoch
        timer.add('Get subset samples', t_sample, max(1, epoch * len_dataloader))
        timer.add('Step', t_step, max(1, epoch * len_dataloader))

        # ---- final encode (jamie/jamie.py:794-799): eval mode, z = mu; the n x n `corr` of the reference does not
        # influence the returned embeddings and is never built
        self.model.eval()
        if world > 1:
            self._average_bn_stats()
        self.model.pull_from_engine()
        # every rank encodes its own row range of each modality; one all-gather assembles the embeddings
        integrated_data = [shard_rows_apply(lambda x, i=i: eng.encode(i, np.asarray(x, np.float32), stream), self.dataset[i])
                           for i in range(2)]
        timer.log('Output')
        print("Finished Mapping!")
        if self.debug:
            timer.aggregate()
        return integrated_data

    def _average_bn_stats(self):
        import torch.distributed as dist
        world = dist.get_world_size()
        st = self.engine.get_bn_stats()
        keys = [k for k in st if not k.endswith('num_batches_tracked')]
        flat = torch.from_numpy(np.concatenate([st[k] for k in keys])).cuda()
        dist.all_reduce(flat)
        flat = (flat / world).cpu().numpy()
        o = 0
        for k in keys:
            st[k] = flat[o:o + st[k].size]
            o += st[k].size
        self.engine.set_bn_stats(st)

    # ------------------------------------------------------------------------------------------------ inference
    def _ensure_engine(self):
        assert self.model is not None, 'Model must be trained before modal prediction.'
        if self.model.engine() is None:
            dev = self._cuda_index()
            torch.cuda.set_device(dev)
            dims = self.model.input_dims
            eng = Engine(dims, self.model.output_dim, max(2, int(getattr(self, 'batch_size', 512) or 512)),
                         self.model.dropout_p, device=dev)
            self.model.attach_engine(eng)
            self.model.push_to_engine()
            self.engine = eng
        return self.model.engine()

    def modal_predict(self, data, modality, pre_transformed=False):
        """Predict the opposite modality from dataset ``data`` in modality ``modality``"""
        assert self.model is not None, 'Model must be trained before modal prediction.'
        eng = self._ensure_engine()
        to_modality = (modality + 1) % self.dataset_num

        def run(rows):
            if not pre_transformed:
                rows = self.model.preprocessing[modality](rows)
            decoded = eng.predict(modality, to_modality, np.asarray(rows, np.float32), self._stream())
            return np.array(self.model.preprocessing_inverse[to_modality](decoded))
        return shard_rows_apply(run, data)     # data-parallel: each rank imputes its own rows (pre- and post-processing too)

    def transform(self, dataset, corr=None, pre_transformed=False):
        """Transform data using an already trained model"""
        return [self.transform_one(d, i, pre_transformed=pre_transformed) for i, d in enumerate(dataset)]

    def transform_one(self, data, i, pre_transformed=False):
        """Transform data using an already trained model"""
        eng = self._ensure_engine()

        def run(rows):
            if not pre_transformed:
                rows = self.model.preprocessing[i](rows)
            return eng.encode(i, np.asarray(rows, np.float32), self._stream())
        return shard_rows_apply(run, data)

    def feature_impact(self, data, modality, target=None, features=None, fill='mean', space='output'):
        """Rank the raw input features of ``data`` (modality ``modality``) by ablation: each feature in turn set to ``fill``
        ('mean' of its column, a scalar or one value per feature), scored against ``target`` (the measured other modality)
        or by how far the predictions (``space='output'``) or embeddings (``space='latent'``) move. Runs on the GPU without
        a host round trip per feature; returns an ``impact.FeatureImpact``."""
        from .impact import feature_impact
        return feature_impact(self, data, modality, target=target, features=features, fill=fill, space=space)

    def shap_values(self, data, modality, background, outputs=None, space='output', n_permutations=2, seed=None):
        """Shapley values of the raw input features of ``data`` (modality ``modality``) for the imputed columns ``outputs``
        of the other modality (``space='output'``, default all) or the embedding dims (``space='latent'``), against the
        raw rows ``background``: antithetic permutation sampling with ``n_permutations`` permutations drawn from ``seed``
        (default ``manual_seed``). Runs on the GPU without a host round trip per masked batch; returns a
        ``shapley.ShapValues`` (values [n, d_in, |outputs|], base_values, outputs)."""
        from .shapley import shap_values
        return shap_values(self, data, modality, background, outputs=outputs, space=space, n_permutations=n_permutations,
                           seed=seed)

    def knn_predict(self, data, modality, reference, k=5, weights='uniform'):
        """Impute the other modality of ``data`` (raw rows of modality ``modality``) by nearest neighbours in the joint
        embedding: each row's imputation averages the measured raw rows of ``reference`` (the other modality, dense or
        scipy.sparse where ``transform_one`` takes it) over its k nearest reference rows, uniformly or by inverse distance
        (``weights='distance'``). The baseline that ``modal_predict``'s decoder imputation is judged against; float64
        [n, d_other_raw]. Exact search and averaging on the GPU (``evaluation.knn_impute``)."""
        from .evaluation import knn_impute
        other = (modality + 1) % self.dataset_num
        return knn_impute(self.transform_one(data, modality), self.transform_one(reference, other), reference, k=k,
                          weights=weights, device=self._cuda_index())

    # ------------------------------------------------------------------------------------------------ metrics
    def test_closer(self, integrated_data, distance_metric=None):
        """Test fraction of samples closer than the true match (jamie/jamie.py:892-913; prints ``foscttm: ...``)"""
        from .evaluation import test_closer
        return test_closer(integrated_data, distance_metric=distance_metric)

    def test_LabelTA(self, integrated_data, datatype, k=None, return_k=False):
        """Label transfer accuracy, k defaulting to 20% of the average class size (jamie/jamie.py:943-961)"""
        from .evaluation import label_transfer_accuracy
        return label_transfer_accuracy(integrated_data, datatype, k=k, return_k=return_k)

    # ------------------------------------------------------------------------------------------------ checkpoints
    def save_model(self, f):
        if self.model.engine() is not None:
            self.model.pull_from_engine()
        torch.save(self.model, f)

    def load_model(self, f):
        import jamie  # noqa: F401  (makes jamie.model / jamie.utilities importable for the unpickler)
        self.model = torch.load(f, weights_only=False)
        self.dataset_num = self.model.num_modalities
        self.engine = None
        self._ensure_engine()
