/* jamie_b200 -- C ABI of the B200-native JAMIE hot path (coupled-VAE train step + modal_predict / transform).
 *
 * The reference (Oafish1/JAMIE v4.4.5) is pure Python and has no FFI; these entry points are what a binding for its
 * hot path would call.  Each one names the reference code it replaces (paths relative to the reference root).
 * Binding stub (ctypes) and the Python-side mirror of the reference API: INTEGRATION.md, jamie_b200/_lib.py.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; jb_last_error() gives the message (thread-local).
 *     The Python wrapper raises RuntimeError / AssertionError with the reference's own messages where it has one.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream). All device work of a call is
 *     enqueued on it; calls do not synchronise the host unless stated.
 *   - the handle owns parameters, Adam moments, BatchNorm statistics, datasets and workspaces; the
 *     caller owns every buffer it passes in. A handle is bound to one device and is not thread-safe.
 *   - "packed" parameter order = edModelVar.named_parameters() order (jamie/model.py:147-220):
 *       sigma[2]; encoders.{0,1}.{0.weight,0.bias,1.weight,1.bias,4.weight,4.bias,5.weight,5.bias};
 *       fc_mus.{0,1}.{weight,bias}; fc_vars.{0,1}.{weight,bias};
 *       decoders.{0,1}.{0.weight,0.bias,1.weight,1.bias,4.weight,4.bias,5.weight,5.bias,8.weight,8.bias}
 *     "packed" BatchNorm order = encoders.0.1, encoders.0.5, encoders.1.1, encoders.1.5, decoders.0.1, decoders.0.5,
 *     decoders.1.1, decoders.1.5; for each layer running_mean[w] then running_var[w].
 */
#ifndef JAMIE_B200_H
#define JAMIE_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef struct jb_engine jb_engine;

typedef struct jb_config {
  int dims[2];          /* post-preprocessing widths D0, D1 (self.col, jamie/jamie.py:469) */
  int latent;           /* output_dim (jamie/jamie.py:475) */
  int max_batch;        /* largest batch size that will be stepped (batch_size, jamie/jamie.py:511-514) */
  float dropout;        /* resolved dropout probability (jamie/model.py:144-145) */
  float lr;             /* model_lr (jamie/jamie.py:481) */
  float beta1, beta2, adam_eps;   /* torch.optim.Adam defaults .9, .999, 1e-8 */
  float max_grad_norm;  /* clip_grad_norm_(..., 1) (jamie/jamie.py:739) */
  float loss_w[4];      /* loss_weights or 1s: KL, Rec, CosSim, F (jamie/jamie.py:723-728) */
  float pf_ratio;       /* PF_Ratio (None -> 1) (jamie/jamie.py:517, 604) */
  unsigned long long seed;   /* Philox key for dropout masks / eps when none are injected */
  int device;           /* CUDA device ordinal */
  int world_size;       /* data-parallel ranks; gradients are divided by it in jb_step_update */
} jb_config;

const char* jb_last_error(void);
int jb_version(void);

/* edModelVar.__init__ + optim.Adam(...) (jamie/model.py:121-220, jamie/jamie.py:472-481): allocates everything. */
int jb_create(const jb_config* cfg, jb_engine** out);
void jb_destroy(jb_engine* e);

/* number of packed parameters / packed BatchNorm floats */
long long jb_num_params(const jb_engine* e);
long long jb_num_bn_floats(const jb_engine* e);

/* state_dict I/O for save_model / load_model (jamie/jamie.py:967-972). Host pointers, packed order. Synchronous. */
int jb_set_params(jb_engine* e, const float* packed, long long n);
int jb_get_params(jb_engine* e, float* packed, long long n);
int jb_set_bn_stats(jb_engine* e, const float* packed, long long n, const long long num_batches_tracked[8]);
int jb_get_bn_stats(jb_engine* e, float* packed, long long n, long long num_batches_tracked[8]);
/* gradients of the last backward pass, packed order (parity tests; the reference reads p.grad) */
int jb_get_grads(jb_engine* e, float* packed, long long n);
/* Adam moments (packed order) and step count -- optional resume side-car; the reference never saves them. */
int jb_get_adam_state(jb_engine* e, float* m_packed, float* v_packed, long long n, long long* t);
int jb_set_adam_state(jb_engine* e, const float* m_packed, const float* v_packed, long long n, long long t);

/* self.dataset[i] after preprocessing (jamie/jamie.py:468, 507-508): n rows of dims[mod] floats, row pitch ld.
 * on_device != 0: X is a device pointer. The engine keeps its own copy (fp32). */
int jb_set_dataset(jb_engine* e, int mod, const float* X, long long n, long long ld, int on_device, void* stream);

/* Correspondence prior P (jamie/jamie.py:423-431) and F = match_result[0] (jamie/jamie.py:431).
 *   diag : P = diag(m), m[n] (identity, partially matched, or zeros) -- no n x n object is ever built
 *   dense: row-major [n0, n1] host matrix (small n only)
 *   F    : dense or absent (use_f_tilde=False -> zeros, jamie/jamie.py:172-173) */
int jb_set_prior_diag(jb_engine* e, const float* m, long long n);
int jb_set_prior_dense(jb_engine* e, const float* P, long long n0, long long n1);
int jb_set_f_dense(jb_engine* e, const float* F, long long n0, long long n1);   /* F == NULL: zeros */

/* Upload the sampling plan of the next `nsteps` optimizer steps (one epoch or more): batch indices per modality
 * (random_batch, jamie/jamie.py:553-583) and the KL anneal factor per step (jamie/jamie.py:630-631; the 0.032 and
 * loss weight are applied by the engine). Resets the plan cursor. idx*: [nsteps, batch] int64 host arrays. */
int jb_upload_plan(jb_engine* e, const long long* idx0, const long long* idx1, const double* kl_anneal,
                   int nsteps, int batch, void* stream);

/* Inject the randomness of the NEXT step only (parity tests): eps[i] = [batch, latent] fp32 (Normal.rsample,
 * jamie/model.py:239-240), masks[k] = [batch, width_k] uint8 keep-masks in draw order enc0 d1,d2; enc1 d1,d2;
 * dec0 d1,d2; dec1 d1,d2 (jamie/model.py:154,164,195,200). Host pointers. Without it the engine draws Philox. */
int jb_inject_randomness(jb_engine* e, const float* eps0, const float* eps1, const unsigned char* const masks[8],
                         void* stream);

/* Run `nsteps` full optimizer steps from the plan cursor: gather, P/F blocks, forward, 4 losses, backward,
 * clip_grad_norm_, Adam, zero_grad (jamie/jamie.py:549-742 with batch_step=True). Asynchronous; ONE launch of the
 * persistent step kernel for all `nsteps` steps (csrc/stepk.cuh), no host synchronisation. */
int jb_train_steps(jb_engine* e, int nsteps, void* stream);
/* Data-parallel split of one step: backward leaves the summed-loss gradients in the flat buffer returned by
 * jb_grad_buffer (the caller all-reduces it, e.g. NCCL sum), update divides by world_size, clips and applies Adam. */
int jb_step_backward(jb_engine* e, void* stream);
int jb_step_update(jb_engine* e, void* stream);
int jb_grad_buffer(jb_engine* e, float** dev_ptr, long long* n_floats);
/* Make the engine write its gradients into a caller-owned device buffer of at least the jb_grad_buffer size (16-byte
 * aligned), e.g. one allocated in NVLink symmetric / multicast memory so that the exchange can be a multimem all-reduce
 * instead of an NCCL call. dev_ptr = NULL returns to the engine's own buffer. The caller keeps the buffer alive. */
int jb_set_grad_buffer(jb_engine* e, float* dev_ptr, long long n_floats);
/* In-kernel gradient exchange over peer memory (NVLink / NVSwitch): grad_ptrs[q] = rank q's gradient buffer (each rank
 * passed its own to jb_set_grad_buffer; all of them mapped into this process, e.g. NVLink symmetric memory), flag_ptrs[q]
 * = rank q's zero-initialised scratch block of at least jb_exchange_scratch_bytes(). With an exchange configured the
 * step kernel sums the gradients across the ranks itself (reduce-scatter + all-gather + clip-norm partials inside the
 * persistent kernel, between WGRAD and ADAM): jb_train_steps(n) is ONE launch for n data-parallel optimizer steps and the
 * caller must not all-reduce jb_grad_buffer. All ranks must run the same number of steps in lockstep. world <= 1 or
 * NULL pointers turn it off. grad_multicast = the NVSwitch multicast address bound to all ranks' gradient buffers, or
 * NULL: with it the sum is taken inside the switch (multimem.ld_reduce) and broadcast with multimem.st. */
int jb_set_exchange(jb_engine* e, int rank, int world, float* const* grad_ptrs, unsigned int* const* flag_ptrs,
                    float* grad_multicast);
long long jb_exchange_scratch_bytes(void);
/* dist_method of sim_diff_func (jamie/jamie.py:484-502): 0 = 'euclidean' (the default: the "CosSim" loss is the row-wise
 * squared distance |z_i - c_i|^2), 1 = 'cosine' ((1 - cos(z_i, c_i))^2). Takes effect with the next step. */
int jb_set_dist_method(jb_engine* e, int method);
/* batch_step=False (jamie/jamie.py:744-749): accumulate gradients over several jb_step_backward calls, one
 * jb_step_update per epoch. accumulate != 0 makes the following backward passes add into the gradient buffer instead of
 * overwriting it (a device-side flag: no rebuild, no synchronisation). The optimizer step count (Adam bias correction)
 * advances per jb_step_update, the Philox stream per backward pass. */
int jb_set_grad_accumulate(jb_engine* e, int accumulate);

/* One optimizer step whose batch arrives from HOST memory (the reference keeps self.dataset wherever `device` says;
 * this is the end-to-end form for host-resident data): x0/x1 = the gathered rows data[i][idx_i] ([batch, dims[i]],
 * packed, ideally pinned), idx0/idx1 = their global cell ids (needed for the P/F blocks), kl_anneal as in
 * jb_upload_plan. Copies the batch in, runs the step graph, copies the 8 loss scalars out and synchronises. */
int jb_train_step_hostbatch(jb_engine* e, const float* x0, const float* x1, const long long* idx0, const long long* idx1,
                            int batch, double kl_anneal, float out_losses[8], void* stream);

/* Data-parallel form of the host-batch step: copy the batch in and run forward + backward only; the caller then
 * all-reduces jb_grad_buffer and calls jb_step_update. Host-batch steps alternate between two plan rows (slots): the
 * k-th host-batch step (k = 0, 1, ...) leaves its losses in row k & 1 of jb_read_losses(e, out, 2, stream). */
int jb_step_backward_hostbatch(jb_engine* e, const float* x0, const float* x1, const long long* idx0,
                               const long long* idx1, int batch, double kl_anneal, void* stream);

/* Asynchronous form of jb_train_step_hostbatch for a host loop that prepares batch k + 1 (the reference's
 * dataset[i][random_batch[i]] gather, jamie/jamie.py:583) while step k runs: submit enqueues the copies on an internal
 * copy stream and the step on `stream` and returns at once; wait blocks until the OLDEST submitted step has finished and
 * returns its 8 loss scalars. At most two steps may be in flight; x0 / x1 must stay valid (pinned) until the step's
 * jb_hostbatch_wait has returned. */
int jb_hostbatch_submit(jb_engine* e, const float* x0, const float* x1, const long long* idx0, const long long* idx1, int batch,
                        double kl_anneal, void* stream);
int jb_hostbatch_wait(jb_engine* e, float out_losses[8]);

/* Phases of the step kernel (csrc/stepk.cuh: StepPhase), in execution order. */
int jb_num_phases(void);
const char* jb_phase_name(int phase);

/* Benchmark hook: `iters` launches of the step kernel restricted to ONE phase, timed with CUDA events on `stream`.
 * Returns the average microseconds per launch (kernel set-up included: an upper bound of the phase's share of a step)
 * and, for GEMM phases, the FLOPs of one launch (0 otherwise). */
int jb_bench_stage(jb_engine* e, int phase, int iters, float* avg_us, double* flops, void* stream);

/* Profiling hook: runs `iters` (+1 warm-up) training steps in ONE launch of the persistent step kernel while CTA 0 records
 * the GPU global timer at every phase boundary; out_us[p] = average microseconds of phase p inside the kernel (its grid
 * barrier included), *n_launches = jb_num_phases(). Rewinds the plan cursor first (needs >= 2 plan rows) and takes
 * optimizer steps like jb_train_steps. */
int jb_profile_step(jb_engine* e, int iters, float* out_us, int cap, int* n_launches, void* stream);
/* Detail of the last jb_profile_step: out[4 p + k] for phase p, k = 0 total us (as above), 1 longest CTA work,
 * 2 mean CTA work, 3 barrier tail (end of the grid barrier - end of the last CTA's work). */
int jb_profile_detail(jb_engine* e, float* out, int cap);

/* Per-step results of the steps run since the last jb_upload_plan, in plan order. Synchronises `stream`.
 * out[s*8 + k]: k=0..3 the reference's `losses` list (KL incl. 0.032*anneal, Rec, 32*CosSim, F; unweighted by
 * loss_weights), k=4 weighted total (batch_loss), k=5 pre-clip gradient norm, k=6,7 reserved. */
int jb_read_losses(jb_engine* e, float* out, int nsteps, void* stream);

/* Eval-mode paths (BatchNorm running statistics folded into the weights, dropout off, z = mu).
 *   jb_encode : fc_mus[mod](encoders[mod](x))                      transform_one / transform / final encode
 *               (jamie/jamie.py:794-799, 817-837)
 *   jb_predict: decoders[to](fc_mus[from](encoders[from](x)))      edModelVar.impute (jamie/model.py:277-282)
 * X: [n, dims[from]] fp32 with row pitch ldx; out: [n, latent] or [n, dims[to]] with row pitch ldo.
 * on_device != 0: both are device pointers (no copies); else host pointers (pinned for full overlap) that are
 * streamed through the device in row chunks. Synchronous for host pointers, asynchronous for device pointers. */
int jb_encode(jb_engine* e, int mod, const float* X, long long n, long long ldx, float* out, long long ldo,
              int on_device, void* stream);
int jb_predict(jb_engine* e, int from, int to, const float* X, long long n, long long ldx, float* out,
               long long ldo, int on_device, void* stream);

/* preclass.transform / inverse_transform with PCA (jamie/utilities.py:660-678): out = ((X - mean) @ comp^T - m)/s
 * and out = (Z*s + m) @ comp + mean, fp32 on device (3xTF32 split for fp32-level accuracy).
 * comp: [k, d] row-major host matrix (pca.components_), mean: [d] (pca.mean_), m/s: scalar standardisation.
 * X/out host or device pointers as above. */
int jb_pca_project(jb_engine* e, const float* X, long long n, long long d, const float* comp, const float* mean,
                   int k, float m, float s, float* out, int on_device, void* stream);
int jb_pca_inverse(jb_engine* e, const float* Z, long long n, int k, const float* comp, const float* mean,
                   long long d, float m, float s, float* out, int on_device, void* stream);

/* Feature ablation (SURVEY.md 3.2: the notebooks' loops that replace one raw input feature, rerun modal_predict or
 * transform_one and score the result, once per feature; jamie_b200/impact.py). For every ablated feature j the network's
 * input is Z(j) = Z + dz[j] w_j^T, a rank-1 update of the unablated input Z = preprocessing[from](X):
 *   Z     [n, dims[from]] float64 host.   dz [n_feat][n] float64 host: f_j - X[:, j] per feature.
 *   w     w_col == NULL: [n_feat, dims[from]] (components_[:, j] / s of a PCA input side);
 *         else [n_feat] scalars added to column w_col[j] only (1 / s_j of a side standardised per column).
 * Y(j) = map(chain(Z(j))), chain = encoder -> mu (to = -1) or encoder -> mu -> decoder[to], in eval mode as jb_encode /
 * jb_predict; map_kind 0 = identity (d_out = the chain's width), 1 = the PCA inverse of jb_pca_inverse (comp [D_to, d_out],
 * mean [d_out], scalar m / s), 2 = fp32(y * aff_scale[c] + aff_shift[c]) (d_out = D_to). Y(-) is Y of the unablated Z.
 *   shift [n_feat, d_out] : mean over rows of |Y(j)[:, c] - Y(-)[:, c]|
 *   with target [n, d_out] fp32 (else NULL): base_r [d_out] = Pearson r(Y(-)[:, c], target[:, c]) and r [n_feat, d_out] the
 *   same for Y(j), finished as jb_metric_feature_pearson does (a constant column gives nan).
 * Works in batches of features x row ranges whose working set stays under batch_bytes (and the free memory): no
 * prediction leaves the device. Sums are float64 per 32-row slab at fixed absolute rows, folded in row order: results are
 * bit-identical across reruns and for any batch_bytes. Refuses, before any allocation, a problem whose smallest batch
 * (one feature, 32 rows) does not fit in free device memory. Host pointers; synchronous. */
int jb_feature_impact(jb_engine* e, int from, int to, const double* Z, long long n, long long n_feat, const double* dz,
                      const double* w, const int* w_col, int map_kind, const float* comp, const float* mean, float m, float s,
                      const double* aff_scale, const double* aff_shift, long long d_out, const float* target, double* base_r,
                      double* r, double* shift, long long batch_bytes, void* stream);

/* Shapley values by antithetic permutation walks (SURVEY.md 3.2: the notebooks' SHAP explainers around modal_predict;
 * jamie_b200/shapley.py). For every explained row x, permutation pi and background row b, the walk from b to x adds the
 * raw features in the order pi; with a linear input map its network inputs are z_t = z_{t-1} + (x_j - b_j) w_j, j = pi_t,
 * z_0 = z_b, built on the device in float64 and rounded once to fp32 per row. A step with x_j == b_j gets no chain row.
 *   X [nx, d], B [nb, d] float64 host: raw explained and background rows.  Zb [nb, dims[from]] float64: preprocessing[from](B).
 *   perms [n_perm, d] int32: permutations of the d raw features.
 *   w     w_col == NULL: [d, dims[from]] (components_[:, j] / s of a PCA input side);
 *         else [d] scalars added to column w_col[j] only (1 / s_j of a side standardised per column).
 * y = map(chain(z)), chain and output map as jb_feature_impact, restricted to n_out selected outputs: map_kind 1 takes comp
 * [D_to, n_out] and mean [n_out] already restricted to them; kinds 0 / 2 take out_cols [n_out] (columns of the chain's
 * output; kind 2's aff_scale / aff_shift have the chain's width).
 *   phi [nx, d, n_out] += sum over (permutation, background row) of y(z_t) - y(z_{t-1}), credited to feature pi_t.
 *   base [n_out] += sum over b of y(z_b).  stats [2] (or NULL) += {chain rows of the walks, inactive steps skipped}.
 * The caller divides by n_perm * nb. Works in batches of (explained row, background row) segments whose working set stays
 * under batch_bytes (and the free memory); no chain row leaves the device. Each accumulator of phi receives its terms one
 * at a time in float64, in (permutation, background row) order, without atomics: results are bit-identical across reruns
 * and for any batch_bytes. Refuses, before any allocation, a problem whose smallest batch (one segment of d active steps)
 * does not fit in free device memory. Host pointers; synchronous. */
int jb_shapley(jb_engine* e, int from, int to, const double* X, long long nx, const double* B, long long nb, long long d,
               const double* Zb, const int* perms, long long n_perm, const double* w, const int* w_col, int map_kind,
               const float* comp, const float* mean, float m, float s, const double* aff_scale, const double* aff_shift,
               const int* out_cols, long long n_out, double* phi, double* base, long long* stats, long long batch_bytes,
               void* stream);

/* PCA fit (jamie/jamie.py:436-452, sklearn PCA(n_components).fit with the covariance_eigh solver): the two O(n d) /
 * O(n d^2) passes over the [n, d] matrix run on the GPU -- column sums, then the centred Gram matrix
 * (X - mean)^T (X - mean) as a split (fp32-class) tensor-core GEMM accumulated over row chunks in float64. The caller
 * divides / all-reduces (rows sharded over ranks: sum colsum and n, then sum the Gram matrices) and solves the d x d
 * symmetric eigenproblem (host LAPACK: independent of n). X host or device pointer (packed rows); colsum [d], gram [d, d]
 * host float64. Synchronous. */
int jb_pca_colsum(jb_engine* e, const float* X, long long n, long long d, double* colsum, int on_device, void* stream);
int jb_pca_gram(jb_engine* e, const float* X, long long n, long long d, const double* mean, double* gram, int on_device,
                void* stream);

/* Evaluation metrics of the reference on the GPU (no engine handle needed; host pointers in, synchronous).
 *   jb_metric_foscttm: test_closer (jamie/evaluation.py:65-85, jamie/jamie.py:892-913) on two [n, L] embeddings with the
 *     euclidean distance: raw_count_closer = #{j: d(a_i, b_j) < d(a_i, b_i)} + #{j: d(b_i, a_j) < d(b_i, a_i)} summed over
 *     i; the caller divides by 2 n^2. Distances in float64.
 *   jb_metric_knn_vote: the kNN classifier of test_LabelTA (jamie/evaluation.py:114-132, jamie/jamie.py:943-961): for
 *     every query row the majority class (uniform votes; ties to the lowest class index) of its k nearest reference rows
 *     (euclidean; equal distances by the lowest row index). ref_class: class indices in [0, n_classes).
 *   jb_metric_feature_pearson: per-feature Pearson r of two [n, d] matrices (jamie/evaluation.py:491-513, sklearn
 *     r_regression); a constant feature gives nan.
 *   jb_metric_feature_auroc: per-feature AUROC of imputed scores against present / absent measured values (the AUROC
 *     panel of jamie/evaluation.py:468-490, sklearn roc_auc_score(measured[:, j] > threshold, imputed[:, j])). scores:
 *     [n, d] row-major fp32 (finite; -0.0 and +0.0 are one score). The positives of column j are the rows
 *     pos_row[pos_ptr[j] .. pos_ptr[j + 1]) (CSC lists: int64 pos_ptr [d + 1] from 0, int32 rows increasing in [0, n));
 *     every other row is a negative. Rows are grouped by equal score in ascending order; for group g with pos_g
 *     positives, neg_g negatives and negbefore_g negatives in all lower groups,
 *       u2[j] = 2U = sum_g pos_g (2 negbefore_g + neg_g)   (exact, uint64; n < 2^31),   n_pos[j] = P,
 *     and AUROC = 2U / (2 P N) with N = n - P (one float64 division by the caller; P = 0 or N = 0 has no AUROC).
 *     Integer arithmetic only: results do not depend on batch_bytes. Works in column batches whose working set stays
 *     under batch_bytes (and the free memory); refuses, before any allocation, a problem whose one-column batch does not
 *     fit in free device memory. */
int jb_metric_foscttm(const float* emb0, const float* emb1, long long n, int L, int device,
                      unsigned long long* raw_count_closer);
int jb_metric_knn_vote(const float* query, long long nq, const float* ref, const int* ref_class, long long nr, int L,
                       int k, int n_classes, int device, int* pred_class);
int jb_metric_feature_pearson(const float* x, const float* y, long long n, long long d, int device, double* r);
int jb_metric_feature_auroc(const float* scores, long long n, long long d, const long long* pos_ptr, const int* pos_row,
                            long long batch_bytes, int device, unsigned long long* u2, long long* n_pos);

/* Exact kNN search and kNN averaging on the GPU (csrc/knn.cuh; no engine handle; host pointers in, synchronous). They
 * replace sklearn's NearestNeighbors(algorithm='brute').kneighbors and KNeighborsRegressor(algorithm='brute').predict on
 * the host, whose search grows with nq * nr.
 *   jb_knn: for every query row the k nearest reference rows in euclidean distance. query [nq, L], ref [nr, L] row-major
 *     fp32; distances are float64 sums of squared fp32 differences (sequential over the columns, the tile arithmetic of
 *     jb_metric_foscttm). idx [nq, k] int64 and dist [nq, k] float64 (sqrt of the sum; NULL = not wanted) in ascending
 *     (squared sum, reference index) order: equal distances by the lowest index, as a stable argsort gives. 1 <= k <=
 *     min(1024, nr); nq, nr < 2^31. No [nq, nr] matrix is formed: the reference rows stay on the device, the queries go in
 *     batches whose lists fit in batch_bytes, and a small batch splits the reference rows into ranges whose lists are
 *     merged. No floating-point atomics: results do not depend on batch_bytes or the device.
 *   jb_knn_average: out[q, c] = sum_t w[q, t] values[idx[q, t], c] / sum_t w[q, t] in float64, summed in list order, for
 *     idx [nq, k] int64 in [0, nr) (the lists of jb_knn), weights [nq, k] float64 or NULL (all 1), values [nr, w] float64
 *     with row pitch ldv, out [nq, w] float64. The values go to the device in column slabs under batch_bytes.
 *   Both refuse, before any allocation, a problem whose smallest batch (one query row; one column) does not fit in free
 *   device memory. */
int jb_knn(const float* query, long long nq, const float* ref, long long nr, int L, int k, long long batch_bytes, int device,
           long long* idx, double* dist);
int jb_knn_average(const long long* idx, const double* weights, long long nq, int k, const double* values, long long nr,
                   long long w, long long ldv, long long batch_bytes, int device, double* out);

/* Silhouette sums on the GPU (csrc/silhouette.cuh; no engine handle; host pointers in, synchronous). They replace the
 * O(n^2 L) pair loop of sklearn's silhouette_samples on the host.
 *   x [n, L] row-major fp32, sorted by label: label c holds rows [label_off[c], label_off[c + 1]) (int64 label_off
 *   [n_labels + 1], 0 first, n last, every label non-empty; 2 <= n_labels <= n; n < 2^31). With d(i, j) the sqrt of the
 *   float64 sum of squared fp32 differences (the tile arithmetic of jb_metric_foscttm) and S[i, c] = sum over the rows
 *   j of label c of d(i, j):  intra[i] = S[i, l_i],  inter[i] = min over c != l_i of S[i, c] / n_c  (float64 [n], the two
 *   arrays of sklearn's _silhouette_reduce before the intra division). The rows stay on the device and the query rows go
 *   in batches whose workspace fits in batch_bytes. No floating-point atomics: results do not depend on batch_bytes or
 *   the device. Refuses, before any allocation, a problem whose rows and one query row's workspace do not fit in free
 *   device memory. */
int jb_silhouette(const float* x, long long n, int L, const long long* label_off, int n_labels, long long batch_bytes,
                  int device, double* intra, double* inter);

/* Distances of the F estimation (compute_distances, jamie/jamie.py:839-890; the default distance_mode 'geodesic' is
 * unioncom.utils.geodesic_distances of unioncom==0.4.0, restated and unpinned in jamie_b200/correspondence.py).
 * A jb_dist handle owns one n x n float64 matrix D on one device and a stream; host pointers throughout.
 *   jb_dist_create    : D = 0. Fails with a message when the 8 n^2 bytes of D do not fit in the device's free memory.
 *   jb_dist_accumulate: D[i, j] += sum_c f(slab[i, c], slab[j, c]) over a [n, w] float64 host slab with row pitch ld;
 *                       kind 0 = (a - b)^2, 1 = |a - b|, 2 = a b (the caller streams the columns of the data in slabs,
 *                       after row normalising / centring / ranking for the product forms). Columns are summed in order
 *                       (any slab widths give the same bits); D stays bitwise symmetric, diagonal exactly 0 for kinds 0
 *                       and 1. Asynchronous; `slab` may be reused when the call returns.
 *   jb_dist_finish    : transform 0 = none, 1 = sqrt (euclidean), 2 = 1 - g clipped to [0, 2] with a zero diagonal
 *                       (sklearn cosine_distances, scipy correlation), 3 = (1 - clip(g, -1, 1)) / 2 (np.corrcoef /
 *                       spearmanr for 'pearson' / 'spearman', jamie/jamie.py:851-884); NaN stays NaN. out [n, n] or NULL.
 *   jb_dist_knn       : per row the k nearest columns of D in ascending order, equal distances by the lowest column (a
 *                       stable argsort; the row itself counts, as in kneighbors_graph(X)). idx [n, k], dist [n, k] or
 *                       NULL. The lists stay on the device for jb_dist_geodesic. D must be non-negative.
 *   jb_dist_geodesic  : all-pairs shortest paths on the undirected graph of the first k (<= the jb_dist_knn k) neighbours
 *                       (blocked Floyd-Warshall in float64, overwriting D), then every pair above the largest finite
 *                       distance set to twice that distance. out [n, n] or NULL.
 * All but jb_dist_accumulate synchronise the handle's stream before they return. */
typedef struct jb_dist jb_dist;
int jb_dist_create(long long n, int device, jb_dist** out);
void jb_dist_destroy(jb_dist* h);
int jb_dist_accumulate(jb_dist* h, int kind, const double* slab, long long w, long long ld);
int jb_dist_finish(jb_dist* h, int transform, double* out);
int jb_dist_knn(jb_dist* h, int k, int* idx, double* dist);
int jb_dist_geodesic(jb_dist* h, int k, double* out);

/* Randomized PCA fit (sklearn's randomized solver, jamie_b200/pca_fit.py randomized_fit_transform): a jb_pcaop handle
 * holds one input matrix X [n, d] on one device and applies the implicitly centred Xc = X - 1 mu^T to thin dense
 * matrices, so that no d x d matrix is ever formed. It owns a stream; host data are copied with cudaMemcpyAsync on it.
 *   jb_pcaop_create_dense : dense fp32 rows [n, d] (host). Products: 3xTF32 split GEMM on hi/lo planes of Xc (the mean is
 *                           subtracted during the split), long reductions chunked and accumulated in float64.
 *   jb_pcaop_create_sparse: CSR of X and CSR of X^T (= CSC of X), host arrays: int64 indptr, int32 indices, fp32 values.
 *                           Products: one CSR x dense kernel for both directions, each output summing its row's nonzeros
 *                           in index order (fp32 values, float64 products and sums; long rows in fixed-size segments
 *                           added in order), then the centring as a float64 rank-1 correction before the one rounding to
 *                           fp32. No floating-point atomics: results are bit-reproducible.
 *   Both refuse, with a message and before any allocation, inconsistent CSR input and an operand (plus its workspaces)
 *   that does not fit in the device's free memory. mu = 0 until jb_pcaop_stats.
 *   jb_pcaop_stats  : per-column mean and variance (ddof 0), float64, two passes (sum, then centred squares; for sparse
 *                     input the (n - nnz_c) mu^2 of the zeros is added). mean [d], var [d] host or NULL. Stores mu in the
 *                     handle for the centring. Synchronous.
 *   jb_pcaop_apply  : trans 0: Y[n, l] = Xc B, with B [d, l].  trans 1: Y[d, l] = Xc^T B, with B [n, l].
 *                     Packed row-major fp32 DEVICE pointers, asynchronous on `stream` (ordered after the work already on
 *                     it; NULL = the legacy default stream). Workspaces for width l are allocated on first use; a width
 *                     whose workspaces do not fit is refused like an operand that does not fit. */
typedef struct jb_pcaop jb_pcaop;
int jb_pcaop_create_dense(const float* X, long long n, long long d, int device, jb_pcaop** out);
int jb_pcaop_create_sparse(long long n, long long d, long long nnz, const long long* row_ptr, const int* col_idx,
                           const float* row_val, const long long* col_ptr, const int* row_idx, const float* col_val,
                           int device, jb_pcaop** out);
int jb_pcaop_stats(jb_pcaop* h, double* mean, double* var);
int jb_pcaop_apply(jb_pcaop* h, int trans, const float* B, int l, float* Y, void* stream);
void jb_pcaop_destroy(jb_pcaop* h);

/* Debug / parity taps: copy a named intermediate of the last step to the host (synchronises).
 * Names: "x0","y1_0","h1_0","y2_0","h2_0","mulv0","z0","c0","xhat0", ... (see csrc/engine.cu: tap table),
 * "corr", "fblk", "grad" (padded flat), "theta". Returns the number of floats written, or -1. */
long long jb_debug_read(jb_engine* e, const char* name, float* out, long long cap);
/* number of kernel launches issued by the handle so far */
long long jb_launch_count(const jb_engine* e);

#ifdef __cplusplus
}
#endif
#endif /* JAMIE_B200_H */
