/*
 * polee_b200.h -- C ABI of libpolee_b200.so: the B200-native (sm_100a) replacement for the
 * prep-sample likelihood-approximation hot path of dcjones/polee.
 *
 * The reference has no FFI seam on this path (plain Julia calling plain Julia) and one real plugin
 * API (the TensorFlow custom-op ABI of src/tensorflow_ext/hsb_ops.cpp).  This header is the seam a
 * maintainer binds with `ccall` (julia/PoleeB200.jl) or from the rebuilt TF shim
 * (polee_b200/tf/hsb_ops_b200.cpp); INTEGRATION.md shows both bindings.  Each entry point cites the
 * reference function (file:line under the reference checkout) whose work it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; every host array is owned by the caller, copied inside the
 *     call and never retained; outputs are caller-allocated.
 *   - index arrays are passed EXACTLY as Julia stores them: 1-based UInt32 CSC arrays
 *     (SparseMatrixCSC{Float32,UInt32}, src/rnaseq_sample.jl:11) and 1-based Int32 tree arrays
 *     (node_parent_idxs / node_js, src/likelihood-approximation.jl:618-621).  The hsb_* entry points
 *     take the 0-based int32 left/right/leaf arrays of make_inverse_ptt_params (src/ptt.jl:293-309).
 *   - every function returns 0 on success or a POLEE_E* code; polee_last_error() gives the text.
 *     (Reference behaviour: @assert / error() exceptions -- the Julia glue turns codes into error().)
 *   - a handle is single-threaded; distinct handles are independent (one per GPU / Julia task).
 *   - there is NO CPU fallback: every compute entry point fails with POLEE_ECUDA when no sm_100
 *     device is usable.
 */
#ifndef POLEE_B200_H
#define POLEE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define POLEE_OK 0
#define POLEE_EINVAL 1      /* bad argument / call order */
#define POLEE_ECUDA 2       /* CUDA runtime error or no usable device */
#define POLEE_EBADTREE 3    /* node_parent_idxs / node_js do not describe a full binary tree */
#define POLEE_ENONFINITE 4  /* non-finite gradient (likelihood-approximation.jl:559 @assert all_finite) */
#define POLEE_ENCCL 5       /* NCCL error */
#define POLEE_ENOMEM 6

#define POLEE_APPROX_LOGIT_SKEW_NORMAL_PTT 0 /* LogitSkewNormalPTTApprox, likelihood-approximation.jl:395 */
#define POLEE_APPROX_OPTIMIZE_PTT 1          /* OptimizePTTApprox,        likelihood-approximation.jl:149 */

#define POLEE_NOISE_PHILOX 0   /* device Philox4x32-10 keyed (seed; node, draw, step) + Box-Muller */
#define POLEE_NOISE_INJECTED 1 /* caller supplies zs0[num_steps][K][n-1] (parity tests) */

typedef struct polee_handle polee_handle;

/* Options; defaults mirror src/constants.jl:53-65 and the keyword defaults at
 * likelihood-approximation.jl:395-401. */
typedef struct polee_opts {
    int32_t device;              /* CUDA device ordinal */
    int32_t approx;              /* POLEE_APPROX_* */
    int32_t num_steps;           /* LIKAP_NUM_STEPS = 500 */
    int32_t num_mc_samples;      /* LIKAP_NUM_MC_SAMPLES = 6 (K); 1..16 */
    int32_t gradonly;            /* Val(gradonly) = true: skip log-likelihood / ELBO values */
    int32_t use_efflen_jacobian; /* true */
    int32_t noise_mode;          /* POLEE_NOISE_* */
    int32_t exact_accumulation;  /* arithmetic of the two sparse products (src/sparse.jl:6-40):
                                  * 0 (default): class layout, Float32 FMAs inside a task (a row's <= 64 terms; <= 32
                                  *    rows per lane + a 5-level lane tree per column), Float64 across tasks;
                                  * 1: general layouts, Float32 products summed in Float64 in the reference's order
                                  *    (frag_probs bit-identical to the reference);
                                  * 2: class layout, every product and sum in Float64 */
    uint64_t seed;               /* Random.seed! default 123456789, main.jl:123-127 */
    double max_step_mu;          /* ss_max_mu_step    = 2e-1, likelihood-approximation.jl:421 */
    double max_step_omega;       /* ss_max_omega_step = 2e-1 */
    double max_step_alpha;       /* ss_max_alpha_step = 2e-2 */
    double max_step_z;           /* ss_max_z_step     = 1e-1 (OptimizePTTApprox :166) */
    int32_t use_cuda_graph;      /* capture one ADAM step and replay it (default 1) */
    int32_t reserved1;
} polee_opts;

/* ------------------------------------------------------------------ lifecycle */
int polee_opts_default(polee_opts *opts);
int polee_create(polee_handle **h, const polee_opts *opts);
int polee_destroy(polee_handle *h);
/* Device memory a destroyed handle used is kept in a per-process cache and handed to the next handle: `polee prep`
 * (src/main.jl:590-631) fits one sample after another, and cudaMalloc/cudaFree of the GB-sized layouts would cost
 * as much as ~100 ADAM steps per sample.  polee_trim_memory returns the cached blocks of `device` (-1: every device)
 * to the driver; POLEE_NO_CACHE=1 in the environment disables the cache. */
int polee_trim_memory(int32_t device);
/* text of the last error on this handle (or, with h == NULL, the last error of a failed create) */
const char *polee_last_error(const polee_handle *h);
/* library / device probe: returns POLEE_OK and fills what it can; sm = 100 on B200 */
int polee_device_info(int32_t device, int32_t *sm_major_minor, int32_t *num_sms, int64_t *hbm_bytes);

/* ------------------------------------------------------------------ inputs
 * polee_set_matrix_csc: RNASeqSample.X (src/rnaseq_sample.jl:11, built :390-524) for this rank's
 * rows; replaces `Xt = SparseMatrixCSC(transpose(X))` + `Model(m, n)`
 * (likelihood-approximation.jl:406-408).  ks (nullable) are the per-row counts of the factored
 * likelihood (likelihood.jl:59-85, salmon path).  Host pointers. */
int polee_set_matrix_csc(polee_handle *h, int64_t m, int64_t n, const uint32_t *colptr /* n+1, 1-based */,
                         const uint32_t *rowval /* nnz, 1-based */, const float *nzval /* nnz */,
                         const int64_t *ks /* m or NULL */);
/* same, arrays already resident in device memory on opts.device (synthetic generation on device) */
int polee_set_matrix_csc_device(polee_handle *h, int64_t m, int64_t n, const uint32_t *d_colptr,
                                const uint32_t *d_rowval, const float *d_nzval, const int64_t *d_ks);
/* sample.effective_lengths (Float32[n]) */
int polee_set_efflens(polee_handle *h, const float *efflens);
/* Optional: the gene -> transcripts map of `--gene-noninformative` (the `gene_transcripts` Dict built at
 * likelihood-approximation.jl:476-493), flattened: gene g owns transcripts[gene_ptr[g] .. gene_ptr[g+1]).  When set,
 * every draw adds gene_noninformative_prior! (likelihood.jl:114-159) to x_grad after the effective-length adjustment
 * (likelihood-approximation.jl:535-538).  Needs opts.use_efflen_jacobian (the reference's prior reads the `xls` that
 * adjustment fills) and the unweighted LogitSkewNormalPTTApprox fit.  num_genes == 0 clears the map (the default). */
int polee_set_gene_groups(polee_handle *h, int64_t num_genes, const int64_t *gene_ptr /* num_genes+1, 0-based offsets */,
                          const int32_t *transcripts /* 1-based transcript ids */);
/* PolyaTreeTransform(parent_idxs, output_idxs)  src/ptt.jl:89-116; 2n-1 entries each, as written to
 * .prep.h5 (node_parent_idxs, node_js).  Also computes the initial parameters
 * (likelihood-approximation.jl:451-456). */
int polee_set_tree(polee_handle *h, int64_t n, const int32_t *node_parent_idxs, const int32_t *node_js);
/* list_nodes(n) tree of PolyaTreeTransform(X, :sequential)  src/hclust.jl:477-489 */
int polee_set_tree_sequential(polee_handle *h, int64_t n);
/* The sample of one approximate_likelihood call in ONE call: polee_set_matrix_csc + polee_set_efflens + polee_set_tree
 * (the three inputs likelihood-approximation.jl:404-435 takes from the RNASeqSample and the PolyaTreeTransform), same
 * arguments, same resulting state.  The host-side tree preparation runs on a second host thread while the calling
 * thread uploads the matrix and the device builds its layout, so the set-up costs max(matrix, tree) instead of their
 * sum; a third short-lived thread loads the ADAM step's kernels meanwhile (CUDA loads a kernel lazily at its first
 * launch otherwise; POLEE_PRELOAD=0 turns that off).  Both helper threads are plain std::threads that touch nothing of
 * the caller's and are joined before the call returns.  A bad tree is reported (POLEE_EBADTREE) after the matrix has
 * been set. */
int polee_set_sample(polee_handle *h, int64_t m, int64_t n, const uint32_t *colptr, const uint32_t *rowval,
                     const float *nzval, const int64_t *ks /* m or NULL */, const float *efflens /* n */,
                     const int32_t *node_parent_idxs, const int32_t *node_js);

/* ------------------------------------------------------------------ the fit
 * approximate_likelihood(::LogitSkewNormalPTTApprox, sample; ...)  likelihood-approximation.jl:395-624
 * (and the factored variant :248-392 when ks were given).  Runs opts.num_steps ADAM steps of
 * opts.num_mc_samples draws on the device and returns mu / omega / alpha (Float32[n-1] each).
 * elbo_traj (nullable, num_steps doubles) receives the per-step mean ELBO when gradonly == 0.
 * noise (nullable unless noise_mode == INJECTED): zs0[num_steps][K][n-1] host floats. */
int polee_fit(polee_handle *h, float *mu, float *omega, float *alpha, double *elbo_traj, const float *noise);
/* approximate_likelihood(::OptimizePTTApprox, sample)["x"]  likelihood-approximation.jl:149-242 */
int polee_fit_optimize_ptt(polee_handle *h, float *xs /* n */);

/* finer-grained control of the same loop (bench / checkpointing, SURVEY section 5) */
int polee_init_params(polee_handle *h);                 /* :451-456, resets ADAM state and step counter */
int polee_run_steps(polee_handle *h, int32_t nsteps);   /* asynchronous: enqueue nsteps ADAM steps */
int polee_sync(polee_handle *h);                        /* wait + surface POLEE_ENONFINITE */
/* Progress of polee_run_steps / polee_fit: cb(steps_done, num_steps, user) is called on the calling thread each time
 * another `every` ADAM steps have FINISHED on the device (the steps are otherwise enqueued without waiting), so that
 * the reference's "Optimizing" progress bar (likelihood-approximation.jl:495, :574: next!(prog) once per step) keeps
 * moving.  cb == NULL removes it. */
typedef void (*polee_progress_fn)(int32_t steps_done, int32_t num_steps, void *user);
int polee_set_progress(polee_handle *h, polee_progress_fn cb, void *user, int32_t every);
int polee_get_params(polee_handle *h, float *mu, float *omega, float *alpha);
int polee_set_params(polee_handle *h, const float *mu, const float *omega, const float *alpha);
int polee_set_noise(polee_handle *h, const float *noise, int64_t num_steps); /* INJECTED mode buffer */
int polee_get_elbo(polee_handle *h, double *elbo_traj, int32_t nsteps);
/* stream the handle's kernels run on (cudaStream_t as void*), for CUDA-event timing by the caller */
void *polee_stream(polee_handle *h);
/* bytes one ADAM step streams with the device layouts in use, and its launch count (DESIGN.md section 3):
 * bytes_k1 = the likelihood pass (all of it when the equivalence-class or the fused layout is in use, then
 * bytes_k2 = 0; K1 / K2 of the split layout otherwise), bytes_k3 = tree + reparameterisation + ADAM */
int polee_step_stats(polee_handle *h, double *bytes_k1, double *bytes_k2, double *bytes_k3, int32_t *launches);
/* which device layouts hold the matrix (a1-a2: replaces Xt = SparseMatrixCSC(transpose(X)),
 * likelihood-approximation.jl:407): info[0..5] = rows, entries, classes, tasks, blob bytes, partials of the
 * equivalence-class layout; info[6..7] = rows, entries of the general layouts; info[8] = their kind (0 none,
 * 1 split, 2 fused); info[9] = padded row slots of the class layout; info[10] = the kernels the tree takes at the
 * draw count the work buffers were last sized for (0 chain scans, 1 DFS runs, 2 path products, 3 shared-memory
 * levels, 4 global-memory levels; -1 without a tree or before the first call that sizes them); info[11], info[12] =
 * programmatic edges (PDL launches of consecutive step kernels) in the captured one-step and multi-step graphs of
 * polee_run_steps, -1 while that graph is not captured.  count <= 13 values are written. */
int polee_layout_info(polee_handle *h, int64_t *info, int32_t count);
/* time (ms, CUDA events on the handle's stream) of `reps` launches of one named kernel group:
 * which = 1 (the likelihood pass; K1 alone on the pure split layout), 2 (K2 of the pure split layout),
 * 3 (K3 tree+reparam+ADAM), 4 (the class kernel alone, without the second stage that adds its partials) */
int polee_time_kernel(polee_handle *h, int32_t which, int32_t reps, float *ms_avg);

/* Random.rand!(als::ApproxLikelihoodSampler, xs)  src/approx-sampler.jl:37-44 (used by `polee sample`,
 * src/main.jl:845-855, and load_samples_hdf5's x0 init, src/estimate.jl:436-455): num_samples draws from the
 * approximation held by the handle (polee_set_tree + polee_set_params with omega = log(sigma)); xs[num_samples][n].
 * Device Philox noise keyed (seed; node, draw, batch). */
int polee_sample(polee_handle *h, int32_t num_samples, uint64_t seed, float *xs);

/* ------------------------------------------------------------------ piecewise (parity tests)
 * log_likelihood(frag_probs, log_frag_probs, X, Xt, xs, x_grad, Val(gradonly))  likelihood.jl:36-56
 * for K stacked xs vectors: xs[K][n] Float32 -> lp[K] (0 when gradonly), x_grad[K][n] Float64.
 * With ks set this is factored_log_likelihood (likelihood.jl:59-85). */
int polee_loglik_grad(polee_handle *h, const float *xs, int32_t K, int32_t gradonly, double *lp, double *x_grad);
/* frag_probs = Xt' * xs (pAt_mul_B!, sparse.jl:6-21) for one xs: returns 1/frag_probs as the device
 * stores it (Float32[m], original row order) */
int polee_frag_prob_recip(polee_handle *h, const float *xs, float *w);
/* transform!(t, ys, xs, Val(ladj))  ptt.jl:125-160 for K stacked ys[K][n-1] Float64 -> xs[K][n] Float32 */
int polee_ptt_transform(polee_handle *h, const double *ys, int32_t K, float *xs, double *ladj /* K or NULL */);
/* transform_gradients!(t, ys, y_grad, x_grad)  ptt.jl:167-209 (with_ladj=1) or
 * transform_gradients_no_ladj!  ptt.jl:217-251 (with_ladj=0); ys[K][n-1], x_grad[K][n] Float64 ->
 * y_grad[K][n-1] Float32 */
int polee_ptt_transform_gradients(polee_handle *h, const double *ys, const double *x_grad, int32_t K,
                                  int32_t with_ladj, float *y_grad);
/* inverse_transform!(t, xs, ys)  ptt.jl:257-285: xs[K][n] Float32 -> ys[K][n-1] Float64, ladj[K] */
int polee_ptt_inverse_transform(polee_handle *h, const float *xs, int32_t K, double *ys, double *ladj);
/* one ADAM step's K draws at the handle's current parameters with injected zs0[K][n-1]
 * (likelihood-approximation.jl:511-559): all outputs nullable; xs[K][n], ys[K][n-1], x_grad[K][n]
 * (after the effective-length adjustment), y_grad[K][n-1], and the draw-averaged mu/omega/alpha grads. */
int polee_lsn_draws(polee_handle *h, const float *zs0, int32_t K, float *xs, double *ys, double *x_grad,
                    float *y_grad, float *mu_grad, float *omega_grad, float *alpha_grad, double *elbo);

/* ------------------------------------------------------------------ hsb_ops (TF plugin boundary)
 * Device ordinal explicit; host pointers; left/right/leaf are [idx_batch][2n-1] with idx_batch == B
 * (a tree per row, as the reference op requires) or 1 (shared tree, broadcast). */
/* HSBOp::Compute       src/tensorflow_ext/hsb_ops.cpp:40-120  */
int polee_hsb(int32_t device, int64_t B, int64_t n, const float *y_logit /* [B][n-1] */, const int32_t *left,
              const int32_t *right, const int32_t *leaf, int64_t idx_batch, float *x /* [B][n] */);
/* InvHSBOp::Compute    src/tensorflow_ext/hsb_ops.cpp:153-249 */
int polee_inv_hsb(int32_t device, int64_t B, int64_t n, const float *x, const int32_t *left, const int32_t *right,
                  const int32_t *leaf, int64_t idx_batch, double *y /* [B][n-1] */, float *ladj /* [B] */);
/* InvHSBGradOp::Compute src/tensorflow_ext/hsb_ops.cpp:280-402 */
int polee_inv_hsb_grad(int32_t device, int64_t B, int64_t n, const double *y_grad, const float *ladj_grad,
                       const double *y, const int32_t *left, const int32_t *right, const int32_t *leaf,
                       int64_t idx_batch, float *backprops /* [B][n] */);
/* Plans: the validated + level-scheduled tree(s) resident on the device, for callers whose index
 * tensors are constant across calls (every training step of a TF model: src/estimate.jl:357-376). */
typedef struct polee_hsb_plan polee_hsb_plan;
int polee_hsb_plan_create(polee_hsb_plan **plan, int32_t device, int64_t n, int64_t idx_batch, const int32_t *left,
                          const int32_t *right, const int32_t *leaf);
int polee_hsb_plan_destroy(polee_hsb_plan *plan);
int polee_hsb_with_plan(const polee_hsb_plan *plan, int64_t B, const float *y_logit, float *x);
int polee_inv_hsb_with_plan(const polee_hsb_plan *plan, int64_t B, const float *x, double *y, float *ladj);
int polee_inv_hsb_grad_with_plan(const polee_hsb_plan *plan, int64_t B, const double *y_grad, const float *ladj_grad,
                                 const double *y, float *backprops);
/* Device-resident forms of the three ops: every tensor is a device pointer on the plan's device, the work is enqueued on
 * `stream` (a cudaStream_t; NULL = the legacy stream) and nothing is copied or allocated per call (scratch lives in the
 * plan).  This is what a DEVICE_GPU registration of the ops binds (the reference registers DEVICE_CPU only,
 * hsb_ops.cpp:120, 249, 402); polee_b200/tf/hsb_ops_b200.cpp registers both. */
int polee_hsb_device(const polee_hsb_plan *plan, int64_t B, const float *d_y_logit, float *d_x, void *stream);
int polee_inv_hsb_device(const polee_hsb_plan *plan, int64_t B, const float *d_x, double *d_y, float *d_ladj, void *stream);
int polee_inv_hsb_grad_device(const polee_hsb_plan *plan, int64_t B, const double *d_y_grad, const float *d_ladj_grad,
                              const double *d_y, float *d_backprops, void *stream);
/* log q(x) of the fitted LogitSkewNormalPTT approximation (definition: DESIGN.md K5) and d log q / dx (as InvHSBGrad
 * defines it).  x [B][n] on the simplex; mu/omega/alpha [param_batch][n-1], param_batch 1 or B; lp [B] Float64;
 * x_grad [B][n] Float32 or NULL (then only lp).  For each internal node k (numbered as the fit and the prep file
 * number them), with y_k = u_left / u_k from the tree inverse, sigma = Float64(expf(omega)),
 * z = log y - log1p(-y), s = (z - mu) / sigma, w = asinh(s) - alpha, z0 = sinh(w):
 *   log q(x) = sum_k [ -z0^2/2 - log(2 pi)/2 + log cosh w - log1p(s^2)/2 - log sigma - log y - log1p(-y) ] - sum_k log u_k
 * in Float64.  A row with some y_k exactly 0 or 1 gets lp = -inf (its x_grad is undefined); other rows are unaffected. */
int polee_approx_log_prob_with_plan(const polee_hsb_plan *plan, int64_t B, int64_t param_batch, const float *x,
                                    const float *mu, const float *omega, const float *alpha, double *lp, float *x_grad);
int polee_approx_log_prob_device(const polee_hsb_plan *plan, int64_t B, int64_t param_batch, const float *d_x,
                                 const float *d_mu, const float *d_omega, const float *d_alpha, double *d_lp,
                                 float *d_x_grad, void *stream);
/* HSBGrad, the gradient of HSB that the reference's op file leaves as a TODO (hsb_ops.cpp:123-125; DESIGN.md K4):
 * x_grad [B][n] = dL/dx, y_logit [B][n-1] as HSB took it, y_logit_grad [B][n-1] = dL/dy_logit.  With y_k =
 * 1 / (1 + exp(-y_logit_k)) and u_j (u_root = 1, u_left = y u_j, u_right = (1 - y) u_j) exactly as HSB makes them, in
 * Float64 without contraction: G = x_grad at a leaf, G_j = y G_l + (1 - y) G_r at internal node j (index k), and
 * y_logit_grad_k = Float32(((y (1 - y)) u_j) (G_l - G_r)).  The Float32 rounding of x is treated as the identity.  Every
 * value depends only on a node's parent or children, so the result does not depend on the schedule; no atomics.
 * Non-finite inputs propagate; n == 1 gives an empty output. */
int polee_hsb_grad(int32_t device, int64_t B, int64_t n, const float *x_grad, const float *y_logit, const int32_t *left,
                   const int32_t *right, const int32_t *leaf, int64_t idx_batch, float *y_logit_grad);
int polee_hsb_grad_with_plan(const polee_hsb_plan *plan, int64_t B, const float *x_grad, const float *y_logit,
                             float *y_logit_grad);
int polee_hsb_grad_device(const polee_hsb_plan *plan, int64_t B, const float *d_x_grad, const float *d_y_logit,
                          float *d_y_logit_grad, void *stream);
const char *polee_hsb_last_error(void);
/* make_inverse_ptt_params(node_parent_idxs, node_js)  src/ptt.jl:293-309 (host helper, exact ints) */
int polee_make_inverse_ptt_params(int64_t num_nodes, const int32_t *node_parent_idxs, const int32_t *node_js,
                                  int32_t *left_index, int32_t *right_index, int32_t *leaf_index);

/* PolyaTreeTransform(X, :cluster): the reference's tree heuristic, hclust + order_nodes (src/hclust.jl:193-319,
 * 361-389), on the host.  Output = the (node_parent_idxs, node_js) pair polee_set_tree takes (2n-1 entries each,
 * 1-based, DFS order with the right branch first).  Similarity ties are broken by an explicit rule (smaller node ids
 * first); the reference leaves them to unspecified library internals, so its exact tree cannot be reproduced (SURVEY
 * 8c) -- any valid tree gives a valid approximation.  No GPU needed. */
int polee_hclust(int64_t m, int64_t n, const uint32_t *colptr, const uint32_t *rowval, int32_t *node_parent_idxs,
                 int32_t *node_js);

/* Exact row de-duplication (tools/exact-factorization.jl:31-68): rows of X that agree in their transcript ids and
 * Float32 values bit for bit are merged; counts[u] = multiplicity of unique row u.  The compressed matrix + counts go
 * to polee_set_matrix_csc(..., ks = counts) (the factored likelihood, likelihood.jl:59-85) and give the same
 * likelihood and gradient as the original.  Unique rows are numbered by first occurrence (the reference's order is a
 * Julia Dict's iteration order, i.e. unspecified).  Host arrays in and out; rowval_out / nzval_out need room for nnz
 * entries, counts_out for m.  Runs on `device` (sorts + scans), standalone: no handle needed. */
int polee_exact_factorization(int32_t device, int64_t m, int64_t n, const uint32_t *colptr, const uint32_t *rowval,
                              const float *nzval, int64_t *m_unique, uint32_t *colptr_out /* n+1 */,
                              uint32_t *rowval_out, float *nzval_out, int64_t *counts_out, int64_t *nnz_out);

/* ------------------------------------------------------------------ multi-GPU (row-partitioned X)
 * Each rank holds a contiguous row block (equal nnz) and all n columns; one ncclAllReduce(sum) of the
 * transcript-length gradient g[n][K] (+K log-likelihoods) per ADAM step.  No reference counterpart
 * (the reference is single-process, SURVEY 2c). */
int polee_partition_rows(int64_t m, int64_t n, const uint32_t *colptr, const uint32_t *rowval, int32_t nparts,
                         int64_t *row_bounds /* nparts+1, 0-based half-open */);
int polee_comm_unique_id(char id[128]);
int polee_comm_init(polee_handle *h, int32_t nranks, int32_t rank, const char id[128]);
/* Optional, after polee_comm_init and once n is known (matrix or tree set), on a box whose GPUs reach each other over
 * NVLink / NVSwitch: the per-step all-reduce then runs as ONE kernel over peer memory (narrow, reduce-scatter by loads,
 * all-gather by stores, widen; all ranks get bit-identical sums) instead of narrow -> ncclAllReduce -> widen.  Every rank
 * calls polee_comm_peer_export (its CUDA IPC handle, 64 bytes), the host gathers the nranks handles in rank order by
 * whatever transport it has, every rank calls polee_comm_peer_import with all of them.  If the import fails (no peer
 * access) the NCCL path stays in use.  POLEE_ALLREDUCE=nccl | f64 selects the NCCL variants at run time. */
int polee_comm_peer_export(polee_handle *h, char handle[64]);
int polee_comm_peer_import(polee_handle *h, const char *handles /* nranks x 64 bytes; NULL: drop the mapping, back to NCCL */);

#ifdef __cplusplus
}
#endif
#endif /* POLEE_B200_H */
