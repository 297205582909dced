/*
 * evok.h -- C ABI of libevok.so: the sm_100a kernels behind the per-generation hot path of
 * EvoTorch's distribution-based searchers (PGPE / SNES / CEM / XNES / CMA-ES).
 *
 * The reference (nnaisense/evotorch @ cebcac4f) has no FFI: its "plugin interface" on this path is a
 * set of Python methods whose bodies are sequences of torch ops.  Each entry point below replaces the
 * body of one of those methods; the citation is `path:line` under /root/reference/src/evotorch.
 * INTEGRATION.md shows the ctypes stub a maintainer of the reference would add at each site.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in `_host`;
 *   - the caller owns all memory, including workspaces (query the *_workspace_bytes functions);
 *     the library never allocates, frees or synchronises (the one exception: evok_peer_alloc / open / close / free);
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, so every call is
 *     CUDA-graph capturable and re-entrant;
 *   - return value: 0 = ok, negative = argument error (EVOK_E_*), positive = cudaError_t;
 *   - populations are row-major fp32: X[i * ldx + j], i < n_rows, j < D.
 */
#ifndef EVOK_H_
#define EVOK_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EVOK_ABI_VERSION 1

#if defined(__GNUC__)
#define EVOK_API __attribute__((visibility("default")))
#else
#define EVOK_API
#endif

/* argument-error codes (negative return values) */
#define EVOK_E_NULLPTR (-1)
#define EVOK_E_BADSIZE (-2)
#define EVOK_E_BADENUM (-3)
#define EVOK_E_WORKSPACE (-4)
#define EVOK_E_ODDROWS (-5) /* symmetric sampling / gradients need an even number of rows */
#define EVOK_E_ALIGN (-6)

#define EVOK_MAX_PEERS 16 /* GPUs of one NVLink domain that can take part in a peer exchange */

/* objective functions with a fused evaluation kernel */
#define EVOK_OBJ_NONE 0      /* sample only */
#define EVOK_OBJ_SPHERE 1    /* sum x^2 */
#define EVOK_OBJ_RASTRIGIN 2 /* 10 D + sum(x^2 - 10 cos(2 pi x))  (reference README.md:86-89) */
#define EVOK_OBJ_ACKLEY 3    /* -20 exp(-0.2 sqrt(mean x^2)) - exp(mean cos(2 pi x)) + 20 + e */
#define EVOK_OBJ_COUNT 4

/* ranking methods (tools/ranking.py:186) */
#define EVOK_RANK_CENTERED 0
#define EVOK_RANK_LINEAR 1
#define EVOK_RANK_NES 2
#define EVOK_RANK_NORMALIZED 3
#define EVOK_RANK_RAW 4

/* gradient forms: S1_j = sum_r a_r eps_rj ; S2_j = sum_r b_r g(eps_rj) */
#define EVOK_GRAD_SEPARABLE 0 /* g = (eps^2 - sigma^2)/sigma; a=b=w_i; all rows      (distributions.py:548-579) */
#define EVOK_GRAD_SYMMETRIC 1 /* same g; a,b = (w+ -/+ w-)/2; even rows only           (distributions.py:708-773) */
#define EVOK_GRAD_EXP 2       /* g = (eps/sigma)^2 - 1; a=b=w_i                        (distributions.py:783-793) */
#define EVOK_GRAD_MOMENTS 3   /* g = eps^2; a=b=w_i (0/1 elite mask for CEM)           (distributions.py:538-546) */

int evok_abi_version(void);
/* number of kernels launched by this library since it was loaded (for bench.py's gpu_launches) */
uint64_t evok_launch_count(void);
const char* evok_error_string(int code);

/* ---------------------------------------------------------------------------------------------
 * K1 / K2: population sampling and evaluation.
 * Replaces: Distribution.sample -> SymmetricSeparableGaussian._fill / SeparableGaussian._fill
 *           (distributions.py:155-216, :514, :705) -> make_gaussian (tools/misc.py:1663-1755), and, for the
 *           built-in objectives, Problem._evaluate_batch (core.py:2602-2608).
 * Random numbers: Philox4x32-10 keyed by `seed`; the counter of a draw is a pure function of
 * (global row or direction index, column, `stream_id`), so the population does not depend on the launch
 * geometry nor on how rows are sharded over GPUs (`row0` = global index of the first local row).
 * symmetric != 0: rows 2k and 2k+1 are mu + sigma*z_k and mu - sigma*z_k (row0 and n_rows even).
 * X may be NULL when objective != NONE ("lazy population": evaluate without materialising).
 * f may be NULL when objective == NONE.
 * stream_offset_dev (nullable): device pointer to a 32-bit generation counter that is ADDED to the low word of
 * stream_id when the kernel runs -- a CUDA graph captured once then draws a fresh population at every replay
 * (the host increments the counter with an in-graph kernel); NULL = use stream_id as is.
 */
int evok_sample_eval(int objective, float* X, int64_t ldx, const float* mu, const float* sigma, int64_t row0,
                     int64_t n_rows, int64_t D, int symmetric, uint64_t seed, uint64_t stream_id,
                     const uint32_t* stream_offset_dev, float* f, void* stream);

/* K2 alone: f[i] = objective(X[i, :]) for an already materialised population (torch-RNG parity mode,
 * CMA-ES / XNES populations).  Replaces the user's vectorised torch objective at core.py:2604. */
int evok_eval(int objective, const float* X, int64_t ldx, int64_t n_rows, int64_t D, float* f, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K3: fitness -> utilities.  Replaces tools/ranking.py:24-183 (`rank` :189).
 * Sort semantics: STABLE (equal fitnesses keep ascending index order), -0 == +0, NaN largest;
 * identical to torch.argsort(f, descending=!higher_is_better, stable=True).
 * w: utilities (same length).  perm (nullable): the sorted order, worst first, as int64 (what
 * `argsort` returns).  ws: workspace of at least evok_rank_workspace_bytes(N) bytes.
 * Implementation: N <= 8192 -> ONE launch (rank by counting, utilities / flags / permutation written by the same kernel);
 * larger N -> stable LSD radix sort (4 passes x 8 bits) + a scatter kernel.  Both produce bit-identical results.
 * --------------------------------------------------------------------------------------------- */
size_t evok_rank_workspace_bytes(int64_t N);
int evok_rank(int method, const float* f, int64_t N, int higher_is_better, float* w, int64_t* perm, void* ws,
              size_t ws_bytes, void* stream);

/* Stable argsort of fp32 keys (SolutionBatch.argsort core.py:3827, CEM elite selection distributions.py:541,
 * CMA-ES cmaes.py:445).  Same workspace as evok_rank. */
int evok_argsort(const float* keys, int64_t N, int descending, int64_t* perm, void* ws, size_t ws_bytes,
                 void* stream);

/* out[i] = table[position of keys[i] in the stable sorted order] -- "the weight of a solution is weights[its rank]"
 * (CMA-ES get_population_weights, cmaes.py:445-451: argsort, inverse-permutation scatter and gather, in one call).
 * descending != 0: position 0 is the largest key.  Same workspace as evok_rank. */
int evok_rank_table(const float* keys, int64_t N, int descending, const float* table, float* out, void* ws, size_t ws_bytes, void* stream);

/* In-place weight post-processing on the N-vector (distributions.py:562-563, :722-723 `w - mean(w)`;
 * :784-785 `w / sum|w|`).  mode 1: subtract mean; mode 2: divide by sum of absolute values. */
int evok_weights_adjust(float* w, int64_t N, int mode, void* stream);

/* 0/1 mask of the `num_elites` largest weights, ties broken by ascending index (distributions.py:540-542).
 * Needs the rank workspace. */
int evok_elite_mask(const float* w, int64_t N, int64_t num_elites, float* mask, void* ws, size_t ws_bytes,
                    void* stream);

/* ---------------------------------------------------------------------------------------------
 * K4: utility-weighted column reductions over the population.
 * Replaces SeparableGaussian._compute_gradients (distributions.py:548-579),
 * SymmetricSeparableGaussian._compute_gradients (:708-773), ExpSeparableGaussian._compute_gradients
 * (:783-793) and the elite moments of _compute_gradients_via_parenthood_ratio (:538-546).
 *   out_mu[j]    = scale_mu    * sum_r a_r * (X[r,j] - mu[j])
 *   out_sigma[j] = scale_sigma * sum_r b_r * g(X[r,j] - mu[j])          (g, a, b per `form` above)
 * `w` holds the weights of the n_rows local rows (a slice of the global utility vector when the
 * population is sharded; the partial results of the shards then add up: all-reduce(sum)).
 * Deterministic (fixed two-stage reduction order, no atomics).
 * --------------------------------------------------------------------------------------------- */
size_t evok_grad_workspace_bytes(int64_t n_rows, int64_t D);
int evok_grad(int form, const float* X, int64_t ldx, const float* w, const float* mu, const float* sigma,
              int64_t n_rows, int64_t D, float scale_mu, float scale_sigma, float* out_mu, float* out_sigma,
              void* ws, size_t ws_bytes, void* stream);

/* K4 without a materialised population: regenerates eps from the Philox counters used by
 * evok_sample_eval(..., X = NULL) with the same (seed, stream_id, row0). */
int evok_grad_regen(int form, const float* w, const float* mu, const float* sigma, int64_t row0, int64_t n_rows,
                    int64_t D, uint64_t seed, uint64_t stream_id, const uint32_t* stream_offset_dev, float scale_mu,
                    float scale_sigma, float* out_mu, float* out_sigma, void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K5: D-vector updates (no host synchronisation; norms are reduced on the device).
 * --------------------------------------------------------------------------------------------- */
/* ClipUp.ascent (optimizers.py:319-357): v <- clip(momentum*v + stepsize*g/||g||, max_speed).
 * velocity is updated in place; step_out (nullable) receives the ascent step; mu (nullable) += step. */
int evok_clipup_step(const float* g, int64_t D, float* velocity, float stepsize, float momentum, float max_speed,
                     float* step_out, float* mu, void* stream);
/* Adam via TorchOptimizer.ascent (optimizers.py:60-91, :101-165): m, v updated in place; `t` is the 1-based
 * step count; step = lr * m_hat / (sqrt(v_hat) + eps). */
int evok_adam_step(const float* g, int64_t D, float* m, float* v, int64_t t, float lr, float beta1, float beta2,
                   float eps, float* step_out, float* mu, void* stream);
/* SGD with optional momentum (optimizers.py:168-228): buf <- momentum*buf + g (first step: buf = g). */
int evok_sgd_step(const float* g, int64_t D, float* buf, int first_step, float lr, float momentum, float* step_out,
                  float* mu, void* stream);
/* mu += lr * g  (Distribution._follow_gradient with a plain learning rate, distributions.py:385). */
int evok_axpy(const float* g, int64_t D, float lr, float* mu, void* stream);

/* sigma update + controlled clamp.  Replaces distributions.py:591-596 / :805-808 and modify_tensor
 * (tools/misc.py:711-816) as used by gaussian.py:404-416.
 *   exp_form == 0: target = sigma + lr*g          exp_form != 0: target = sigma * exp(0.5*lr*g)
 *   lo = max(lb, sigma - |sigma|*mc), hi = min(ub, sigma + |sigma|*mc); sigma <- min(max(target, lo), hi)
 * lb / ub / mc: device vectors (length D) or NULL; when NULL the scalar is used; a NaN scalar means
 * "not set" (-inf / +inf / no max-change limit). */
int evok_sigma_update(float* sigma, const float* g, int64_t D, float lr, int exp_form, const float* lb_vec,
                      float lb, const float* ub_vec, float ub, const float* mc_vec, float mc, void* stream);

/* CEM finalisation from elite moments (distributions.py:543-546): given S1 = sum eps, S2 = sum eps^2 over
 * the E elites, writes grad_mu = S1/E and grad_sigma = sqrt((S2 - S1^2/E)/(E-1)) - sigma. */
int evok_cem_finalize(const float* s1, const float* s2, const float* sigma, int64_t D, int64_t num_elites,
                      float* grad_mu, float* grad_sigma, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K8: batched flat-parameter MLP policy forward, one observation per policy.
 * Replaces Policy.__call__ (neuroevolution/net/vecrl.py:1240-1279: vmap(functional_call) over the rows of the
 * N x L parameter matrix set by set_parameters) for feed-forward nets made of Linear layers + activations.
 * Parameter row layout (net/functional.py:118-129): per layer W (out x in, row-major) then b (out).
 *   out[i, :] = layer_{n-1}(... act_0(W_0 obs[i, :] + b_0) ...)        acts: EVOK_ACT_* applied after each layer
 * dims_host: n_layers + 1 layer widths (host array); acts_host: n_layers activation ids (host array).
 * --------------------------------------------------------------------------------------------- */
#define EVOK_ACT_NONE 0
#define EVOK_ACT_TANH 1
#define EVOK_ACT_RELU 2
#define EVOK_ACT_SIGMOID 3
int64_t evok_mlp_parameter_length(int n_layers, const int32_t* dims_host);
int evok_mlp_forward(const float* params, int64_t ldp, const float* obs, int64_t ldo, float* out, int64_t ldout, int64_t N,
                     int n_layers, const int32_t* dims_host, const int32_t* acts_host, void* stream);

/* The same forward with the observation pre-processing of the rollout loop fused into the observation load
 * (vecgymne.py:604-660, :822-836; net/runningnorm.py:412-533): x = clamp((obs - mean) / stdev, clip_lo, clip_hi), where
 * mean = obs_sum / count and stdev = sqrt(max(obs_sumsq / count - mean^2, min_variance)) come from the RunningNorm sums on the
 * device (obs_sum == NULL: no normalisation; clip_* = NaN: no clipping).  `active` (N bytes, nullable): policies whose flag
 * is 0 are skipped -- their parameters are never read -- and receive zero actions.  `ws` (nullable, >= 4 bytes, 4-byte aligned):
 * with a mask, CTAs draw row chunks from a work counter kept there instead of a static round-robin (which leaves the number of
 * surviving policies per CTA binomially unbalanced). */
int evok_mlp_forward_prep(const float* params, int64_t ldp, const float* obs, int64_t ldo, float* out, int64_t ldout, int64_t N,
                          int n_layers, const int32_t* dims_host, const int32_t* acts_host, const float* obs_sum, const float* obs_sumsq,
                          const int64_t* obs_count_dev, float min_variance, float clip_lo, float clip_hi, const uint8_t* active,
                          void* ws, size_t ws_bytes, void* stream);

/* The forward of N networks on ONE shared input batch (B x dims[0]) -- a population scored on a common minibatch
 * (neuroevolution/supervisedne.py:337-347, where the reference loops over the solutions: parameterize_net + network(x), neproblem.py:342,
 * supervisedne.py:250).  Here the first layer of ALL networks is one tensor-core product of the stacked weight rows with the shared batch
 * (a persistent kernel gathers the weight rows from the flat parameter rows -- any 4-byte alignment -- straight into the swizzled
 * operand tiles, so every parameter is read from HBM once; bias and activation in the epilogue), the remaining (small, per-network)
 * layers run in a second kernel on the staged activations.  out: [N][B][dims[n_layers]].  n_layers >= 2, hidden widths <= 512,
 * X 16-byte aligned with ldx % 4 == 0. */
size_t evok_mlp_forward_shared_workspace_bytes(int64_t N, int64_t B, int n_layers, const int32_t* dims_host);
int evok_mlp_forward_shared(const float* params, int64_t ldp, int64_t N, const float* X, int64_t ldx, int64_t B, int n_layers,
                            const int32_t* dims_host, const int32_t* acts_host, float* out, void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K6 / K7: fp32-accurate tensor-core GEMM (tcgen05 + TMEM + TMA, 3xTF32 operand splitting).
 *   C[M x N] = A[M x K] * B[N x K]^T        A, B, C row-major fp32 (lda, ldb >= K; ldc >= N)
 *   optional C2[M x N] = alpha_dev[0] * (A B^T) + bias[col]    (C2 / alpha_dev / bias nullable)
 * Replaces the dense contractions of CMA-ES: `ys = (A @ zs.T).T`, `xs = m + sigma * ys` (cmaes.py:427-429; call with
 * A = zs, B = A_chol, C = ys, C2 = xs, alpha_dev = &sigma, bias = m) and the rank-mu update
 * sum_i w_i y_i y_i^T (cmaes.py:548; call with A = (w * Y)^T, B = Y^T built by evok_transpose_scale), and XNES'
 * `A z^T` / sum_i w_i z_i z_i^T (distributions.py:938, :980-984).
 * --------------------------------------------------------------------------------------------- */
size_t evok_gemm_workspace_bytes(int64_t M, int64_t N, int64_t K);
int evok_gemm_nt(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t M, int64_t N, int64_t K, float* C, int64_t ldc,
                 float* C2, int64_t ldc2, const float* alpha_dev, const float* bias, void* ws, size_t ws_bytes, void* stream);
/* The same product with a fused affine update of the output (no second pass over C):
 *   C[i][j] = k[0] * (A B^T)[i][j] + k[1] * E[i][j] + k[2] * u[i] * u[j]        k_dev: 3 device floats; E, u nullable (u needs M == N)
 * E may be C itself.  Replaces the covariance update of CMA-ES, cmaes.py:519-553:
 *   C <- C + c1a (pc pc^T - C) + c_mu (Y^T diag(w) Y - sum(w) C)   with k = (c_mu, 1 - c1a - c_mu sum(w), c1a * weighted_pc^2), u = p_c. */
int evok_gemm_nt_affine(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t M, int64_t N, int64_t K, float* C, int64_t ldc,
                        const float* k_dev, const float* E, int64_t lde, const float* u, void* ws, size_t ws_bytes, void* stream);
/* out[c, r] = (w ? w[r] : 1) * in[r, c]: builds the K-major operands of the weighted SYRK */
int evok_transpose_scale(const float* in, int64_t ldi, int64_t rows, int64_t cols, const float* w, float* out, int64_t ldo, void* stream);
/* both SYRK operands in one pass over `in`:  out_w[c, r] = w[r] * in[r, c],  out_p[c, r] = in[r, c] */
int evok_transpose_pair(const float* in, int64_t ldi, int64_t rows, int64_t cols, const float* w, float* out_w, float* out_p, int64_t ldo,
                        void* stream);

/* ---------------------------------------------------------------------------------------------
 * Batched searches: the functional ask / tell API with leading batch dimensions (algorithms/functional/funcpgpe.py:67, :301, :330,
 * funccem.py, funcclipup.py:95-108; `expects_ndim`, decorators.py:613).  n_items independent searches of the same shape run in ONE
 * launch per stage (grid y / z = item) instead of one launch chain per item.  Tensors are contiguous [items][...] unless an item
 * stride is given (stride 0 = the operand is shared by all items).  Per-item scalar hyper-parameters are HOST arrays (they travel in
 * the launch parameters).  Every stage computes exactly what its single-search entry point computes per item.
 * --------------------------------------------------------------------------------------------- */
/* K1: item b draws with Philox stream (stream_id0 + b): same bits as evok_sample_eval(..., stream_id = stream_id0 + b) per item */
int evok_sample_batched(float* X, int64_t item_stride_x, int64_t ldx, const float* mu, int64_t item_stride_mu, const float* sigma,
                        int64_t item_stride_sigma, int64_t n_items, int64_t n_rows, int64_t D, int symmetric, uint64_t seed, uint64_t stream_id0,
                        void* stream);
/* K3: f, w: [items][N].  ws: max(evok_rank_workspace_bytes(N), 8 * n_items + 256) bytes */
int evok_rank_batched(int method, const float* f, int64_t N, int64_t n_items, int higher_is_better, float* w, void* ws, size_t ws_bytes,
                      void* stream);
int evok_elite_mask_batched(const float* w, int64_t N, int64_t n_items, int64_t num_elites, float* mask, void* ws, size_t ws_bytes, void* stream);
int evok_weights_adjust_batched(float* w, int64_t N, int64_t n_items, int mode, void* stream);
/* K4: X [items][n_rows][D] (item stride / row pitch given), w [items][n_rows], out_mu / out_sigma [items][D] */
size_t evok_grad_batched_workspace_bytes(int64_t n_items, int64_t n_rows, int64_t D);
int evok_grad_batched(int form, const float* X, int64_t item_stride_x, int64_t ldx, const float* w, const float* mu, int64_t item_stride_mu,
                      const float* sigma, int64_t item_stride_sigma, int64_t n_items, int64_t n_rows, int64_t D, float scale_mu, float scale_sigma,
                      float* out_mu, float* out_sigma, void* ws, size_t ws_bytes, void* stream);
/* K5: g, velocity, center [items][D]; center += step.  sigma, g, lb / ub / mc vectors (nullable) [items][D] */
int evok_clipup_batched(const float* g, int64_t n_items, int64_t D, float* velocity, float* center, const float* stepsize_host,
                        const float* momentum_host, const float* max_speed_host, void* stream);
int evok_sigma_update_batched(float* sigma, const float* g, int64_t n_items, int64_t D, const float* lr_host, int exp_form, const float* lb_vec,
                              const float* ub_vec, const float* mc_vec, void* stream);

/* ---------------------------------------------------------------------------------------------
 * CMA-ES generation glue (algorithms/cmaes.py): the vector arithmetic between the dense contractions, fused.
 *   evok_cmaes_row_weights  : w_positive[i] = max(a_i, 0) (recombination weights, cmaes.py:468-475) and the active-CMA reweighting
 *       w_active[i] = a_i > 0 ? a_i : D * a_i / ||z_i||^2 (cmaes.py:531-535; active == 0: w_active = a).  One pass over Z.
 *   evok_cmaes_vector_update: one single-CTA kernel for update_m / update_p_sigma / update_sigma / _h_sig / update_p_c
 *       (cmaes.py:454-517, :31-46), all in place; k_out[0..2] = (c_mu, 1 - c1a - c_mu * sum(w), c1a * weighted_pc^2) are the
 *       coefficients of the covariance update for evok_gemm_nt_affine.  consts_host: 10 host floats
 *       (c_m, c_sigma, damp_sigma, c_c, c_1, c_mu, variance_discount_sigma, variance_discount_c, unbiased_expectation, sum(weights)).
 *       The generation counter of _h_sig comes from *steps_dev (then incremented by the kernel: CUDA-graph replay) or steps_host.
 * --------------------------------------------------------------------------------------------- */
int evok_cmaes_row_weights(const float* assigned_weights, const float* Z, int64_t ldz, int64_t N, int64_t D, int active, float* w_positive,
                           float* w_active, void* stream);
int evok_cmaes_vector_update(const float* local_disp, const float* shaped_disp, int64_t D, float* m, float* p_sigma, float* p_c, float* sigma_dev,
                             int64_t* steps_dev, int64_t steps_host, const float* consts_host, int csa_squared, float* k_out, float* h_sig_out,
                             void* stream);

/* Cholesky factorisation A = L L^T (fp32, lower; the strictly upper part of L is zeroed, like torch.linalg.cholesky).  Replaces
 * CMAES.decompose_C (cmaes.py:555-565, torch.linalg.cholesky -> cuSOLVER potrf).  ONE persistent kernel: 64 x 64 tiles, left-looking
 * tile dataflow with per-tile release / acquire flags instead of a launch (or grid barrier) per panel step.  Only the lower triangle
 * of A is read.  L must not alias A.  A matrix that is not positive definite yields NaNs (no error code: nothing is read back). */
size_t evok_cholesky_workspace_bytes(int64_t n);
int evok_cholesky(const float* A, int64_t lda, int64_t n, float* L, int64_t ldl, void* ws, size_t ws_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Peer exchange over NVLink / NVSwitch: the two collectives of the sharded generation (the reference's Ray round trip,
 * core.py:2762-3073 + algorithms/distributed/gaussian.py:199-272; evotorch_b200/distributed.py) done by libevok kernels.
 * One process per GPU; every rank owns one "exchange buffer" that all peers map (CUDA IPC).  The *_host tables are host
 * arrays of `world` device pointers, one per peer; peer_flags_host[p] = base of peer p's `world` 64-bit flags.
 *
 *   evok_peer_alloc / open / close / free : the only entry points that allocate.  `handle` is a 64-byte cudaIpcMemHandle_t
 *       to be passed to the other processes (any transport).  The buffer is zero-filled.
 *   evok_peer_push : the all-gather.  Runs behind the producer (evok_sample_eval into this rank's slice of the local fitness
 *       vector) and copies that slice to every peer, then raises flag[rank] = *epoch_dev + 1 in every peer's flag array.
 *   evok_peer_wait : one warp spins until all `world` local flags reach *epoch_dev + 1, then advances *epoch_dev.  After
 *       `timeout_ns` it gives up, sets *err_dev = 1 and advances anyway (no hang; the host checks err_dev when it likes).
 *   evok_grad_push : evok_grad / evok_grad_regen (X == NULL) whose finalisation writes this rank's (grad_mu | grad_sigma)
 *       into slot `rank` of every peer's slot array (peer_slots_host[p] = base of world x 2D floats) and raises the flags.
 *   evok_peer_reduce : waits like evok_peer_wait, then out[j] = sum over ranks (in rank order: bit-identical on every GPU)
 *       of slots[r * n + j] -- the all-reduce.
 * `done_dev` is a zero-initialised local uint32 per exchange point; `epoch_dev` a zero-initialised local uint64 per
 * exchange point.  Everything is stream-ordered and CUDA-graph capturable (the pointers are baked into the launch).
 * --------------------------------------------------------------------------------------------- */
/* Sharded ranking (round 2): the fitness all-gather + replicated global sort of the sharded generation replaced by a LOCAL
 * sort + an exchange of sorted keys.  Each GPU sorts only its own n_local fitnesses (stable LSD radix, 8 launches), pushes the
 * sorted orderable keys into every peer's key table (peer_keys_host[p] = base of peer p's N-entry uint32 table) together with
 * its local fitness sum (peer_fsum_host[p] = base of peer p's `world` doubles) and raises its flag; then, after all flags have
 * arrived, every local row finds its GLOBAL position = local position + sum over the other shards of the number of their keys
 * that precede it (binary searches over the L2-resident table; ties by global index exactly like the global stable sort) and
 * writes its utility.  Replaces, per GPU, tools/ranking.py:24-124 on the all-gathered vector (the Ray path ranks per actor,
 * core.py:3289).  Results are bit-identical to evok_rank on the gathered vector; methods: CENTERED, LINEAR, NES.
 * row_offsets_host: world + 1 global row offsets of the shards (host array); w_local: n_local utilities in local row order;
 * mean_out (nullable): global mean fitness.  done_dev: THREE zero-initialised uint32; ws: evok_rank_workspace_bytes(n_local). */
int evok_rank_sharded(int method, const float* f_local, int64_t N, int higher_is_better, int world, int rank,
                      const int64_t* row_offsets_host, void* const* peer_keys_host, void* const* peer_fsum_host,
                      void* const* peer_flags_host, uint64_t* epoch_dev, uint32_t* done_dev, uint32_t* err_dev, uint64_t timeout_ns,
                      float* w_local, float* mean_out, void* ws, size_t ws_bytes, void* stream);

int evok_peer_alloc(size_t bytes, void** dev_ptr_out_host, void* handle_out_64B_host);
int evok_peer_open(const void* handle_64B_host, void** dev_ptr_out_host);
int evok_peer_close(void* dev_ptr);
int evok_peer_free(void* dev_ptr);
/* evok_peer_push: the all-gather as ONE small kernel behind the producer: CTA p copies this rank's slice (n_bytes at src_local) to
 * offset dst_offset_bytes of peer p's buffer (peer_base_host[p]) with 16-byte stores, fences once and raises flag[rank] = *epoch_dev + 1
 * on that peer.  Consumer: evok_peer_wait. */
int evok_peer_push(const void* src_local, int64_t n_bytes, int64_t dst_offset_bytes, int world, int rank, void* const* peer_base_host,
                   void* const* peer_flags_host, const uint64_t* epoch_dev, void* stream);
int evok_peer_wait(const uint64_t* flags_local, int world, uint64_t* epoch_dev, uint32_t* err_dev, uint64_t timeout_ns, void* stream);
int evok_grad_push(int form, const float* X, int64_t ldx, const float* w, const float* mu, const float* sigma, int64_t row0,
                   int64_t n_rows, int64_t D, uint64_t seed, uint64_t stream_id, const uint32_t* stream_offset_dev, float scale_mu,
                   float scale_sigma, int world, int rank, void* const* peer_slots_host, void* const* peer_flags_host,
                   const uint64_t* epoch_dev, uint32_t* done_dev, void* ws, size_t ws_bytes, void* stream);
int evok_peer_reduce(const float* slots_local, int world, int64_t n, const uint64_t* flags_local, uint64_t* epoch_dev,
                     uint32_t* done_dev, uint32_t* err_dev, uint64_t timeout_ns, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* EVOK_H_ */
