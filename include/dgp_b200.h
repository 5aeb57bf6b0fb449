/* dgp_b200.h — C ABI of the B200-native doubly-stochastic DGP hot path.
 *
 * The reference (Hebbalali/dgp-toolbox) has no FFI layer: its boundary is the Python class API
 * (dgp_dace/utils/layers.py, dgp_dace/models/dgp.py, dgp_dace/Infill_criteria.py, dgp_dace/EHVI.py).  Each entry point
 * below names the reference method whose arithmetic it replaces; dgp_toolbox_b200/*.py binds them with ctypes and
 * keeps the reference's class/method names (see INTEGRATION.md).
 *
 * Conventions: every pointer is a DEVICE pointer on the ctx's device unless the name ends in _host; all arrays are
 * C-contiguous float64; calls are asynchronous on the ctx's stream; the caller pre-allocates every output; return
 * value 0 = success, negative = error (message via dgp_last_error).  One ctx per GPU per host thread.
 */
#ifndef DGP_B200_H
#define DGP_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef struct dgp_ctx dgp_ctx;

/* One SVGP layer = the state of reference SVGP_Layer (dgp_dace/utils/layers.py:181-224). */
typedef struct {
  int32_t D_in, D_out, M;
  int32_t white;              /* reference `white` flag (utils/layers.py:246,254-255,296-303): 1 = q(v) whitened, u = Lu v; 0 = default */
  int32_t mean_kind;          /* 0 Zero, 1 Identity, 2 Linear (utils/layer_initializations.py:27,42,52) */
  int32_t kernel_kind;        /* 0 SquaredExponential / RBF, 1 Matern32, 2 Matern52 (ARD; the kernels BO/SO_BO.py:190-197,237-244 offers) */
  const double* Z;            /* [M, D_in]   feature.Z */
  const double* lengthscales; /* [D_in]      kern.lengthscales (host side broadcasts an isotropic value) */
  const double* variance;     /* [1]         kern.variance */
  const double* q_mu;         /* [M, D_out] */
  const double* q_sqrt;       /* [D_out, M, M] lower triangular, dense storage */
  const double* mf_W;         /* [D_in, D_out] Linear.A or NULL */
  const double* mf_b;         /* [D_out] Linear.b or NULL */
  double jitter;              /* gpflow.default_jitter() = 1e-6 */
} dgp_layer_desc;

typedef struct {
  int32_t num_layers;
  const dgp_layer_desc* layers; /* HOST array of descriptors */
  const double* lik_variance;   /* [1] Gaussian likelihood variance */
} dgp_model_desc;

/* offsets (in doubles) into the flat ELBO/gradient buffer of dgp_elbo_grad */
typedef struct { int64_t dZ, dlengthscales, dvariance, dq_mu, dq_sqrt; } dgp_layer_grad_offsets;

int dgp_ctx_create(int device, void* cuda_stream, dgp_ctx** out);
void dgp_ctx_destroy(dgp_ctx* ctx);
const char* dgp_last_error(dgp_ctx* ctx);
int dgp_version(void);
int dgp_set_stream(dgp_ctx* ctx, void* cuda_stream);
/* Synchronises the ctx's stream and reports asynchronous numerical failures of the calls issued so far: DGP_ERR_NUMERIC (-4)
 * when a Kuu + jitter I was not positive definite (the asynchronous entry points dgp_elbo_grad / dgp_predict_moments / dgp_ei*
 * do not synchronise themselves). */
int dgp_check(dgp_ctx* ctx);
/* bytes of device workspace currently held by the ctx; the minibatch is processed in chunks of points sized so that the
 * workspace stays under the limit (default 24 GiB, env DGP_B200_WS_GB) */
int64_t dgp_workspace_bytes(dgp_ctx* ctx);
int dgp_set_workspace_limit(dgp_ctx* ctx, int64_t bytes);
/* number of kernels this ctx has launched (reset != 0 zeroes the counter afterwards) */
int64_t dgp_launch_count(dgp_ctx* ctx, int reset);

/* Per-category device time of the ctx's launches, measured with CUDA event pairs on the ctx's stream (bench.py's
 * live roofline figure). dgp_get_profile synchronises the stream; ms_out / launches_out have DGP_PROFILE_CATEGORIES entries. */
#define DGP_PROFILE_CATEGORIES 10
enum { DGP_CAT_PREP = 0,            /* Kuu build, Cholesky + inverse, KL, replicated M^3-class products, gradient assembly */
       DGP_CAT_KUF = 1,             /* Kuf tiles (covs.Kuf) */
       DGP_CAT_GEMM_FWD = 2,        /* V = Lu^-1 Kuf, A = Lu^-T V, T_d = q_sqrt_d^T A  (DMMA) */
       DGP_CAT_MOMENTS = 3,         /* mean / variance / sample epilogue */
       DGP_CAT_GEMM_BWD_DATA = 4,   /* dA' and W = Ku^-1 dA'  (DMMA) */
       DGP_CAT_RBF_BWD = 5,         /* RBF adjoint on the Kuf block */
       DGP_CAT_GEMM_BWD_PARAM = 6,  /* dKu, dq_sqrt, dq_mu, dZ contractions over the point-samples (DMMA) */
       DGP_CAT_OTHER = 7,           /* likelihood, upstream adjoints, acquisition epilogues */
       DGP_CAT_FUSED_FWD = 8,       /* fused conditional + sample kernel (Kuf, both solves, q_sqrt contraction, moments in one launch) */
       DGP_CAT_FUSED_BWD = 9 };     /* fused data-path adjoint (dV, K-bar = Lu^-T dV, kernel adjoint in one launch; V-form layers) */
int dgp_set_profiling(dgp_ctx* ctx, int on);
/* CUDA-graph replay (default 0). With on = 1 the model-level calls that draw their own Philox samples (dgp_elbo_grad,
 * dgp_predict_moments, dgp_ei, dgp_ei_grad; zs_host == NULL) capture their launch sequence -- ~70-130 small launches over the
 * per-layer side streams for a BO-sized problem -- into a CUDA graph the first time a call signature (every pointer, shape,
 * scalar and ctx flag; not the seed) is seen, and replay it afterwards: one seed store + one graph launch per call. The caller
 * keeps the buffers of a signature alive and in place (parameters updated in place, as dgp_adam_step does). Up to 16 signatures
 * are cached (LRU); growing the workspace or on = 0 drops them. Same kernels, same results bit for bit. */
int dgp_set_graph(dgp_ctx* ctx, int on);
/* on = 0 routes the conditional through the unfused GEMM pipeline (debug / A-B measurement); default 1 */
int dgp_set_fused(dgp_ctx* ctx, int on);
/* The first layer's input is X tiled over the S samples (models/dgp.py:49), so its conditional (and the adjoint's contractions)
 * are identical for every sample; on = 1 (default) evaluates them once per point and expands / reduces over S around them,
 * on = 0 evaluates every point-sample like the reference does. Results agree to summation order. */
int dgp_set_share_first_layer(dgp_ctx* ctx, int on);
/* The layers' replicated per-step work (Kuu build, operator packing, KL, M^3 glue, gradient assembly) runs on per-layer side
 * streams forked from and joined to the ctx's stream (default 1); 0 keeps every launch on the ctx's stream. */
int dgp_set_parallel_layers(dgp_ctx* ctx, int on);
/* V-form of the conditional (default on for both kinds of call): C_d = q_sqrt_d^T Lu^-T and beta = Lu^-1 q_mu are folded once per
 * call, T_d = C_d V, mean = V^T beta, var = s2 - |V|^2 + |T_d|^2, so the A = Lu^-T V pass disappears ((1 + D_out) M^2 instead of
 * (2 + D_out) M^2 flops per point-sample); the adjoint works on V as well (dV, K-bar = Lu^-T dV, contractions G1 = tril(dV V^T),
 * tril(V dT_d^T), V Gm) and maps back to (q_mu, q_sqrt, Ku) once per step through the Cholesky adjoint. 0 keeps the reference's
 * operation order (A = Ku^-1 Kuf explicitly) for the forward-only calls / for the ELBO+gradient calls. gradient_calls = 1 uses the
 * V-form adjoint when the call has >= 32768 point-samples (below that the ~8 extra M^3-class products per layer cost more than
 * they save), 2 always. Same results to rounding. */
int dgp_set_vform(dgp_ctx* ctx, int forward_calls, int gradient_calls);
int dgp_get_profile(dgp_ctx* ctx, double* ms_out, int64_t* launches_out, int reset);

/* kern.K(X, X2) of the GPflow stationary kernel the reference layers hold (utils/layers.py:221,230,243), K_out [n1, n2]:
 * kind 0: variance * exp(-r2 / 2); 1: variance (1 + sqrt3 r) exp(-sqrt3 r); 2: variance (1 + sqrt5 r + 5/3 r^2) exp(-sqrt5 r),
 * r2 = sum_j ((X[i,j] - X2[k,j]) / lengthscales[j])^2, r = sqrt(max(r2, 1e-36)). */
int dgp_kernel_K(dgp_ctx* ctx, int kernel_kind, int D, const double* lengthscales, const double* variance, const double* X, int64_t n1,
                 const double* X2, int64_t n2, double* K_out);

/* z[s,n,d] for one layer: the Philox-4x32-10 stream the fused path consumes when zs == NULL
 * (replaces tf.random.normal at utils/layers.py:113; counter = (n + n_offset, s, d, layer)). */
int dgp_philox_normal(dgp_ctx* ctx, uint64_t seed, int layer, int64_t S, int64_t N, int D, int64_t n_offset, double* z_out);

/* The raw Philox-4x32-10 words behind dgp_philox_normal, words_out [S, N, D, 4] uint32 (DEVICE): key = (seed_lo, seed_hi),
 * counter = (n + n_offset, s, d, layer). Integer plumbing, bit-exact against oracle.philox_uint32. */
int dgp_philox_raw(dgp_ctx* ctx, uint64_t seed, int layer, int64_t S, int64_t N, int D, int64_t n_offset, uint32_t* words_out);

/* SVGP_Layer.build_cholesky_if_needed (utils/layers.py:227-234): Ku [M,M] = Kuu + jitter I, Lu [M,M] = chol(Ku). */
int dgp_kuu_chol(dgp_ctx* ctx, const dgp_layer_desc* layer, double* Ku_out, double* Lu_out);

/* SVGP_Layer.conditional_ND (utils/layers.py:237-278), full_cov=False: X [P, D_in] -> mean, var [P, D_out]. */
int dgp_conditional_nd(dgp_ctx* ctx, const dgp_layer_desc* layer, const double* X, int64_t P, double* mean, double* var);

/* SVGP_Layer.KL (utils/layers.py:280-308) -> kl_out[1]. */
int dgp_kl(dgp_ctx* ctx, const dgp_layer_desc* layer, double* kl_out);

/* DGP_Base.propagate (models/dgp.py:34-63): X [N, D0] tiled S times, chained through the layers.
 * zs_host: HOST array of num_layers device pointers [S,N,D_out_l] (entries or the array itself may be NULL -> Philox).
 * Fs/Fmeans/Fvars_host: HOST arrays of num_layers device pointers [S,N,D_out_l]; entries (or arrays) may be NULL. */
int dgp_propagate(dgp_ctx* ctx, const dgp_model_desc* model, const double* X, int64_t N, int64_t S,
                  const double* const* zs_host, uint64_t seed, int64_t n_offset,
                  double* const* Fs_host, double* const* Fmeans_host, double* const* Fvars_host);

/* size (doubles) and layout of the flat buffer: [0] data term = scale * sum_n mean_s ve, [1] kl_weight * sum_l KL_l,
 * [2] d/d lik_variance, then per layer dZ, dlengthscales, dvariance, dq_mu, dq_sqrt (constrained space). ELBO = [0] - [1]. */
int64_t dgp_grad_size(const dgp_model_desc* model);
int dgp_grad_layout(const dgp_model_desc* model, dgp_layer_grad_offsets* offsets_host /* [num_layers] */);

/* DGP_Base.ELBO (models/dgp.py:89-100) and, when want_grad != 0, its gradient w.r.t. every parameter
 * (replaces tape.gradient at models/dgp.py:275). scale multiplies the data term (the reference's is 1);
 * kl_weight multiplies KL and its gradients (1/world_size on sharded runs so that a sum-allreduce restores them). */
int dgp_elbo_grad(dgp_ctx* ctx, const dgp_model_desc* model, const double* X, const double* Y, int64_t N, int64_t S,
                  double scale, double kl_weight, const double* const* zs_host, uint64_t seed, int64_t n_offset,
                  int want_grad, double* out_flat);

/* Same as dgp_elbo_grad with HOST X [N,D0], Y [N,Dy] and HOST result buffer: host<->device copies are part of the call. */
int dgp_elbo_grad_host(dgp_ctx* ctx, const dgp_model_desc* model, const double* X_host, const double* Y_host, int64_t N,
                       int64_t S, double scale, double kl_weight, uint64_t seed, int64_t n_offset, int want_grad,
                       double* out_flat_host);

/* One trainable parameter of the optimiser entry points below. */
typedef struct {
  double* value;          /* device, constrained space, updated in place (the array the layer descriptors point at) */
  int64_t count;          /* entries of value */
  int64_t grad_offset;    /* its gradient inside the dgp_elbo_grad buffer (dgp_grad_layout) */
  int64_t grad_count;     /* == count; or > count == 1: one scalar shared by grad_count gradient entries (non-ARD lengthscale) */
  int transform;          /* GPflow bijector: 0 identity, 1 softplus (positive()), 2 softplus + 1e-6 (likelihood variance),
                             3 FillTriangular over [count / M^2][M][M] (q_sqrt: entries above the diagonal are not variables) */
  int M;                  /* transform 3 only */
  double* mirror;         /* optional [mirror_count] broadcast of the updated scalar (the [D_in] vector a non-ARD lengthscale is */
  int64_t mirror_count;   /* expanded to for dgp_layer_desc.lengthscales), else NULL / 0 */
} dgp_adam_param;

/* tf.optimizers.Adam(lr, beta_1, beta_2, epsilon).apply_gradients on the unconstrained GPflow variables, minimising -ELBO
 * (models/dgp.py:132-154, 190-204): u = bijector^-1(value), g_u = -dELBO/dvalue * dvalue/du, m = b1 m + (1-b1) g_u,
 * v = b2 v + (1-b2) g_u^2, u -= lr sqrt(1-b2^t)/(1-b1^t) m / (sqrt(v) + epsilon), value = bijector(u); one launch for all
 * parameters. m_state / v_state: device [sum count] in params order, zero before the first step; t counts from 1.
 * params is a HOST array, n_params <= 48. */
int dgp_adam_step(dgp_ctx* ctx, const dgp_adam_param* params, int n_params, const double* grad_flat, double* m_state,
                  double* v_state, int64_t t, double lr, double beta1, double beta2, double epsilon);

/* `steps` iterations of the reference's training loop (models/dgp.py:146-154) without returning to the host: step k runs
 * dgp_elbo_grad(seed = seed0 + k * seed_stride mod 2^64) into out_flat and then dgp_adam_step(t = t0 + k). elbo_trace (device
 * [steps], or NULL) receives each step's ELBO estimate out[0] - out[1] (what the reference prints every `messages` steps). With
 * dgp_set_graph(1) a step is three launches: seed store, graph replay, Adam. */
int dgp_train_adam(dgp_ctx* ctx, const dgp_model_desc* model, const double* X, const double* Y, int64_t N, int64_t S, double scale,
                   double kl_weight, uint64_t seed0, uint64_t seed_stride, int64_t n_offset, const dgp_adam_param* params,
                   int n_params, double* m_state, double* v_state, int64_t t0, int64_t steps, double lr, double beta1,
                   double beta2, double epsilon, double* out_flat, double* elbo_trace);

/* ---- composite kernels and layers on supplied kernel matrices (SURVEY §8 f2: MF-DGP, MF_DGP.py:262-290) ----
 * k(x, y) = k_corr(x_a, y_a) (k_prev(x_b, y_b) + s_l^2 <x_b, y_b>) + k_in(x_a, y_a), + s_w^2 on the diagonal of K(X, X) and in K_diag;
 * a = the first Da of the D input columns, b = the rest. k_corr, k_prev: isotropic SquaredExponential; k_in: SquaredExponential, ARD
 * (in_ard = 1, Da lengthscales) or isotropic. has_prod = 0: k_in (+ White) alone. All pointers are DEVICE pointers to the parameter
 * values (scalars unless noted); white_variance / lin_variance may be NULL. */
typedef struct {
  int32_t D, Da, has_prod, has_linear, in_ard;
  const double* in_variance; const double* in_lengthscales;       /* [1], [Da] or [1] */
  const double* corr_variance; const double* corr_lengthscale;    /* [1], [1] */
  const double* prev_variance; const double* prev_lengthscale;    /* [1], [1] */
  const double* lin_variance; const double* white_variance;       /* [1] or NULL */
} dgp_comp_kernel;
#define DGP_COMP_THETA 7   /* d/d theta layout: in_var, corr_var, corr_ls, prev_var, prev_ls, lin_var, white_var, then in_ls[Da or 1] */

/* kern.K(X, X2) [P, P2] (X2 = NULL: K(X, X) [P, P] including the White diagonal) and kern.K_diag(X) [P] (gpflow Sum / Product /
 * SquaredExponential / Linear / White semantics with active_dims). */
int dgp_comp_K(dgp_ctx* ctx, const dgp_comp_kernel* k, const double* X, int64_t P, const double* X2, int64_t P2, double* K_out);
int dgp_comp_Kdiag(dgp_ctx* ctx, const dgp_comp_kernel* k, const double* X, int64_t P, double* out);
/* kern.K(X_b, X_b) for B blocks of N rows: X [B, N, D] -> K_out [B, N, N], the White variance on each block's diagonal, exactly as
 * dgp_comp_K with X2 = NULL gives for one block. One launch for all blocks: the K(X_s, X_s) of every sample of a layer application
 * (each sample of a layer >= 1 has its own augmented input [x, f_{l-1,s}]). Same descriptor checks and argument errors as dgp_comp_K. */
int dgp_comp_K_blocks(dgp_ctx* ctx, const dgp_comp_kernel* k, const double* X, int64_t B, int64_t N, double* K_out);
/* Adjoints: given Kbar = d loss / d K [P, P2] -> dX [P, D], dX2 [P2, D] (NULL with X2 = NULL: dX then carries both roles) and
 * dtheta [DGP_COMP_THETA + (in_ard ? Da : 1)]; given g = d loss / d K_diag [P] -> dX, dtheta. Deterministic reductions. */
int dgp_comp_K_grad(dgp_ctx* ctx, const dgp_comp_kernel* k, const double* X, int64_t P, const double* X2, int64_t P2,
                    const double* Kbar, double* dX, double* dX2, double* dtheta);
int dgp_comp_Kdiag_grad(dgp_ctx* ctx, const dgp_comp_kernel* k, const double* X, int64_t P, const double* g, double* dX, double* dtheta);

/* SVGP_Layer.conditional_ND + KL (utils/layers.py:237-308, white = False, no mean function) on supplied matrices: Ku [M, M] =
 * Kuu + jitter I, Kuf [M, P], Kdiag [P]; q_mu [M, D_out], q_sqrt [D_out, M, M]. -> mean, var [P, D_out], kl [1].
 * dgp_svgp_from_k_grad: adjoint for upstream gradients Gm = d loss / d mean, Gv = d loss / d var [P, D_out] and gkl = d loss / d kl:
 * dKu [M, M], dKuf [M, P], dKdiag [P], dq_mu [M, D_out], dq_sqrt [D_out, M, M] (lower triangle). The M^2 P contractions run in
 * the FP64 DMMA GEMM engine; the kernel matrices and their adjoints are the caller's (dgp_comp_K / dgp_comp_K_grad). */
int dgp_svgp_from_k(dgp_ctx* ctx, int M, int D_out, int64_t P, const double* Ku, const double* Kuf, const double* Kdiag,
                    const double* q_mu, const double* q_sqrt, double* mean, double* var, double* kl);
int dgp_svgp_from_k_grad(dgp_ctx* ctx, int M, int D_out, int64_t P, const double* Ku, const double* Kuf, const double* Kdiag,
                         const double* q_mu, const double* q_sqrt, const double* Gm, const double* Gv, double gkl,
                         double* dKu, double* dKuf, double* dKdiag, double* dq_mu, double* dq_sqrt);
/* The same two calls sharing the layer's replicated per-evaluation work. Inside one ELBO evaluation the reference applies a layer
 * several times to different inputs with the SAME Kuu, q_mu, q_sqrt (MF_DGP.py:38-44,98-132: Z_right sampling, one chain per fidelity;
 * MO_DGP.py:88-122: the cyclic chain); the factorisation, the M^3 products and the KL depend on those three only. `cache` is a caller-owned
 * DEVICE buffer of dgp_svgp_prep_cache_bytes(ctx, M, D_out) bytes: the first forward call (load = 0) factorises Kuu, forms the M^3
 * products and the KL and saves them; every later call with the same (Ku, q_mu, q_sqrt) -- forward with load = 1, and every adjoint --
 * restores them instead of recomputing. `stash` (may be NULL): a caller-owned DEVICE buffer of dgp_svgp_stash_bytes(M, D_out, P)
 * bytes per APPLICATION; the forward call leaves A = Ku^-1 Kuf and the T_d = q_sqrt_d^T A planes there and the adjoint call of the same
 * application reads them instead of running the three M^2 P forward products again. Results are identical to the uncached calls. */
int64_t dgp_svgp_prep_cache_bytes(dgp_ctx* ctx, int M, int D_out);
int64_t dgp_svgp_stash_bytes(int M, int D_out, int64_t P);
int dgp_svgp_from_k_cached(dgp_ctx* ctx, int M, int D_out, int64_t P, const double* Ku, const double* Kuf, const double* Kdiag,
                           const double* q_mu, const double* q_sqrt, double* mean, double* var, double* kl, double* cache,
                           int64_t cache_bytes, int load, double* stash);
int dgp_svgp_from_k_grad_cached(dgp_ctx* ctx, int M, int D_out, int64_t P, const double* Ku, const double* Kuf, const double* Kdiag,
                                const double* q_mu, const double* q_sqrt, const double* Gm, const double* Gv, double gkl,
                                double* dKu, double* dKuf, double* dKdiag, double* dq_mu, double* dq_sqrt, const double* cache,
                                int64_t cache_bytes, const double* stash);

/* SVGP_Layer.conditional_ND(full_cov=True) per sample and reparameterize(full_cov=True) (utils/layers.py:76-80,264-268,276;
 * utils/utils.py:43-52) on supplied matrices, white = False, no mean function (the MF / MO / EM layers). S samples of N points,
 * column p = s * N + n:
 *   Ku [M, M] = Kuu + jitter I, Kuf [M, S * N], Kff [Kff_batch, N, N] (Kff_batch = 1: one block shared by every sample, or S),
 *   q_mu [M, D_out], q_sqrt [D_out, M, M]  ->
 *   mean [S, N, D_out] (the mean dgp_svgp_from_k gives for the same Ku, Kuf, q);
 *   cov  [S, N, N, D_out] = Kff_s + A_s^T (q_sqrt_d q_sqrt_d^T - Ku) A_s, A_s = Ku^-1 Kuf_s      (may be NULL);
 *   F    [S, N, D_out]    = mean + chol(cov_sd + jitter I) z_sd                                   (may be NULL; F needs z [S, N, D_out]).
 * N <= 768 (one CTA factorises an N x N block), S * D_out <= 65535 blocks; M and D_out as dgp_svgp_from_k. Every argument and the workspace limit are checked
 * before the first launch. Forward only; factorises Ku itself (no prep cache). Synchronises; DGP_ERR_NUMERIC when Ku or a block
 * cov_sd + jitter I is not positive definite. */
int dgp_svgp_from_k_full_cov(dgp_ctx* ctx, int M, int D_out, int64_t N, int64_t S, const double* Ku, const double* Kuf,
                             const double* Kff, int64_t Kff_batch, const double* q_mu, const double* q_sqrt, const double* z,
                             double jitter, double* mean, double* cov, double* F);

/* ---- multi-GPU (SURVEY §8b/e): one process (or thread) and one ctx per GPU. The minibatch's points are sharded over the ranks by
 * the caller; parameters, Kuu, its Cholesky and the KL term are replicated; the path's only exchange step is ONE sum-allreduce of the
 * flat [data term, KL, gradients] buffer (NCCL over NVLink / NVSwitch, on the ctx's stream). NCCL is resolved at run time
 * (libnccl.so.2, or the path in DGP_B200_NCCL); DGP_ERR_UNSUPPORTED when it cannot be loaded.
 *   dgp_comm_unique_id: rank 0 creates the 128-byte ncclUniqueId and distributes it by any means (MPI, a file, torch.distributed).
 *   dgp_comm_init: collective over all ranks. dgp_allreduce_grads: in place, asynchronous on the ctx's stream.
 *   dgp_elbo_grad_sharded: dgp_elbo_grad on this rank's shard (n_offset = global index of its first point, so the Philox draws do
 *   not depend on the placement; KL weighted 1 / world) followed by the allreduce -- every rank ends with the full-batch buffer. */
int dgp_comm_unique_id(void* uid_out_128_bytes);
int dgp_comm_init(dgp_ctx* ctx, int rank, int world, const void* nccl_uid_128_bytes);
int dgp_allreduce_grads(dgp_ctx* ctx, double* elbo_and_grads, int64_t n_doubles);
int dgp_comm_destroy(dgp_ctx* ctx);
int dgp_elbo_grad_sharded(dgp_ctx* ctx, const dgp_model_desc* model, const double* X, const double* Y, int64_t N, int64_t S,
                          double scale, uint64_t seed, int64_t n_offset, int want_grad, double* out_flat);

/* GPflow NaturalGradient(gamma).minimize on the (q_mu, q_sqrt) pairs of the listed layers (models/dgp.py:188,218,312,343; default
 * XiNat parameterisation: theta <- theta - gamma d(-ELBO)/d eta, theta = (S^-1 mu, -S^-1/2), eta = (mu, S + mu mu^T), S = q_sqrt
 * q_sqrt^T), from the gradients a dgp_elbo_grad call left in grad_flat. Collapsed form, per output d: T = tril(q_sqrt_d^T G_R),
 * I + gamma (T + T^T - diag T) = U U^T (reverse Cholesky), q_sqrt_d <- q_sqrt_d U^-T, q_mu_d <- q_mu_d - gamma q_sqrt_d q_sqrt_d^T G_mu;
 * all on the device (batched over layers and outputs: triangular DMMA products, the Cholesky / triangular-inverse kernels of a1).
 * layer_ids: HOST array. The layers' q_mu / q_sqrt arrays are updated in place; nothing is written when a factorisation failed
 * (dgp_check reports it). */
int dgp_natgrad_step(dgp_ctx* ctx, const dgp_model_desc* model, const int* layer_ids, int n_layers, double gamma,
                     const double* grad_flat);

/* The same natural-gradient step on caller-supplied pairs (the multi-fidelity / multi-objective models, whose ELBO gradients come from
 * the supplied-matrix layer calls rather than from dgp_elbo_grad's flat buffer: MF_DGP.py:456,507, MF_DGP_EM.py, MO_DGP.py:446,487):
 * q_mu [M, D_out], q_sqrt [D_out, M, M] (lower) are updated in place from g_mu / g_sqrt = d ELBO / d q_mu, d ELBO / d q_sqrt (same
 * shapes; only the lower triangle of g_sqrt is read). M <= 768. HOST array of DEVICE pointers. */
typedef struct { double* q_mu; double* q_sqrt; const double* g_mu; const double* g_sqrt; int M; int D_out; } dgp_nat_pair;
int dgp_natgrad_pairs(dgp_ctx* ctx, const dgp_nat_pair* pairs, int n_pairs, double gamma);

/* `steps` iterations of part 2 of the reference's optimize_nat_adam (models/dgp.py:206-220,331-345) without returning to the host:
 * iteration k runs dgp_elbo_grad(seed0 + 2k seed_stride) + dgp_adam_step(t0 + k) on `params` (the non-variational parameters; n_params
 * may be 0), then dgp_elbo_grad(seed0 + (2k+1) seed_stride) + dgp_natgrad_step(nat_layers, gamma) -- two evaluations per iteration,
 * as NaturalGradient.minimize re-evaluates the objective. elbo_trace[k] = the first evaluation's ELBO estimate. */
int dgp_train_nat_adam(dgp_ctx* ctx, const dgp_model_desc* model, const double* X, const double* Y, int64_t N, int64_t S, double scale,
                       double kl_weight, uint64_t seed0, uint64_t seed_stride, int64_t n_offset, const dgp_adam_param* params,
                       int n_params, double* m_state, double* v_state, int64_t t0, int64_t steps, double lr, double beta1,
                       double beta2, double epsilon, const int* nat_layers, int n_nat, double gamma, double* out_flat,
                       double* elbo_trace);

/* Value and input gradient of a moment-based criterion (the gradient the reference's Adam-on-x stage takes with tape.gradient,
 * Infill_criteria.py:79-84,160-165): kind 0 = -EI on predict_f moments (== dgp_ei_grad), 1 = WB2 = -(EI - mean) and 2 = EV =
 * (mean - y) Phi + s phi, both on predict_y moments (+ sigma_n^2, Infill_criteria.py:124-133,249-257), 3 = WB2S = -(sigmoid(x_j) EI -
 * mean) per input column j (Infill_criteria.py:187-198; single-output model; value [N, D0]). value [N, D_L] otherwise,
 * d_value_dX [N, D0] = d sum(value) / dX. The adjoint chain runs without the parameter contractions.
 * kind 4 = adjoints supplied by the caller: `value` is an INPUT [N, D_L, 2] holding (dc/dmean, dc/dvar) of some criterion c w.r.t. the
 * mixture moments (y != 0: predict_y moments, y == 0: predict_f moments); d_value_dX = dc/dX. The same seed as the call that produced
 * the moments gives the same draws (EHVI: dgp_ehvi2d_grad, one kind-4 call per objective model). */
int dgp_acq_grad(dgp_ctx* ctx, const dgp_model_desc* model, int kind, const double* X, int64_t N, int64_t S,
                 const double* const* zs_host, uint64_t seed, int64_t n_offset, double y, double* value, double* d_value_dX);

/* ---- acquisition search (SURVEY §8 f3): the reference's `optimize` methods (Infill_criteria.py:61-87,142-168,207-233,290-316) run
 * tfp.optimizer.differential_evolution_minimize and then tf.optimizers.Adam on u, x = lw + (up - lw) / (1 + exp(u)). The criterion
 * itself is evaluated by the entry points below (dgp_ei, dgp_ei_grad, dgp_predict_moments + dgp_acq_moments); these four keep the
 * search state on the device between evaluations. All arrays are device pointers; lw / up have d entries. ----
 * dgp_de_propose: one "rand/1/bin" generation (TFP defaults: weight 0.5, crossover 0.9): candidate_i = pop[a] + weight (pop[b] -
 *   pop[c]) on the dimensions drawn with probability `crossover` (one dimension always), pop_i elsewhere; a, b, c distinct and != i.
 *   Random choices: Philox-4x32-10, key = seed, counter = (i, generation, slot, 0xDE) (csrc/acq.cuh states the word layout; the
 *   oracle reproduces it bit for bit). Writes the candidates in u-space and mapped into the box (the criterion's input). pop >= 4.
 * dgp_de_select: pop_i <- candidate_i where sum_k cand_val[i, k] < pop_val[i] (first != 0: take every candidate, initial evaluation).
 * dgp_box_from_u: x = lw + (up - lw) / (1 + exp(u)) for n rows.
 * dgp_adam_box_step: one tf.optimizers.Adam(lr, beta1, beta2, epsilon) step on u [n, d] from dx = d criterion / d x [n, d]
 *   (dx/du = -(up - lw) e^u / (1 + e^u)^2), t counts from 1; writes the new x [n, d]. n > 1 runs n searches side by side. */
int dgp_de_propose(dgp_ctx* ctx, const double* pop_u, int64_t pop, int d, const double* lw, const double* up, uint64_t seed,
                   int64_t generation, double weight, double crossover, double* cand_u, double* cand_x);
int dgp_de_select(dgp_ctx* ctx, double* pop_u, double* pop_val, const double* cand_u, const double* cand_val, int64_t pop, int d,
                  int ncol, int first);
int dgp_box_from_u(dgp_ctx* ctx, const double* u, const double* lw, const double* up, int64_t n, int d, double* x);
int dgp_adam_box_step(dgp_ctx* ctx, double* u, double* m_state, double* v_state, const double* dx, const double* lw,
                      const double* up, int64_t n, int d, int64_t t, double lr, double beta1, double beta2, double epsilon, double* x);

/* DGP_Base.predict_f / predict_y + DGP.predict mixture moments (models/dgp.py:66-77,113-124,362-366; also
 * Infill_criteria.py:39-41, EHVI.py:112-119): mean [N, D_L], var [N, D_L]; add_lik_var != 0 adds sigma_n^2 (predict_y). */
int dgp_predict_moments(dgp_ctx* ctx, const dgp_model_desc* model, const double* X, int64_t N, int64_t S,
                        const double* const* zs_host, uint64_t seed, int64_t n_offset, int add_lik_var,
                        double* mean, double* var);

/* DGP_Base.propagate(X, full_cov=True, S, zs) (models/dgp.py:34-63 with utils/layers.py:76-80,264-268,276 and utils/utils.py:43-52):
 * every layer's conditional is evaluated per sample with the full N x N covariance, samples are drawn with chol(var + jitter I) per
 * sample and output. Caller arrays (any may be NULL): Fs[l], Fmeans[l] [S, N, D_l]; Fvars[l] [S, N, N, D_l]. N <= 768 (one CTA
 * factorises an N x N block). Layers the fused conditional kernel takes build the K(X_s, X_s) term inside the covariance tiles;
 * other layers (dgp_set_fused(0), or a shape no fused configuration fits) run the unfused pipeline with the same covariance kernel,
 * except white=True layers, which need the fused kernel. zs / seed / n_offset as dgp_propagate. */
int dgp_propagate_full_cov(dgp_ctx* ctx, const dgp_model_desc* model, const double* X, int64_t N, int64_t S,
                           const double* const* zs_host, uint64_t seed, int64_t n_offset, double* const* Fs_host,
                           double* const* Fmeans_host, double* const* Fvars_host);

/* The same with the first layer's input given per sample: X [S, N, D_in] (Layer.conditional_SND / sample_from_conditional with
 * full_cov=True on per-sample inputs: one call for all S samples). */
int dgp_propagate_full_cov_snd(dgp_ctx* ctx, const dgp_model_desc* model, const double* X, int64_t N, int64_t S,
                               const double* const* zs_host, uint64_t seed, int64_t n_offset, double* const* Fs_host,
                               double* const* Fmeans_host, double* const* Fvars_host);

/* Grouped full_cov=True (batch acquisition): the N = G q points form G groups of q consecutive points, 1 <= q <= 32. Group g gets
 * what dgp_propagate_full_cov gives for X[g q : (g + 1) q] alone with n_offset + g q and the same seed: samples correlated within
 * the group, independent across groups. zs[l] [S, N, D_l] as dgp_propagate (group g uses columns g q ..). Caller arrays (any may
 * be NULL): Fs[l], Fmeans[l] [S, N, D_l]; Fcovs[l] [S, G, q, q, D_l]. No limit on N: whole groups run in chunks sized to the
 * workspace limit, with identical results. Refused before any launch: q outside 1 .. 32, N not a multiple of q. Forward only. */
int dgp_propagate_grouped_cov(dgp_ctx* ctx, const dgp_model_desc* model, const double* X, int64_t N, int64_t S, int q,
                              const double* const* zs_host, uint64_t seed, int64_t n_offset, double* const* Fs_host,
                              double* const* Fmeans_host, double* const* Fcovs_host);

/* Monte-Carlo q-EI of each group of dgp_propagate_grouped_cov: out [G, D_L] = -(1/S) sum_s max(y_min - min_j F_{s, g q + j}, 0)
 * on the last layer's jointly drawn samples (the sign convention of dgp_ei). The sum over s runs in a fixed order. Does not
 * synchronise (dgp_check reports a failed factorisation). */
int dgp_qei(dgp_ctx* ctx, const dgp_model_desc* model, const double* X, int64_t N, int64_t S, int q,
            const double* const* zs_host, uint64_t seed, int64_t n_offset, double y_min, double* out);

/* DGP_Base.E_log_p_Y (models/dgp.py:79-87): out [N, D_L] = mean over the S samples of the Gaussian variational expectations
 * (-0.5 log 2pi - 0.5 log s_n^2 - 0.5 ((Y - mu)^2 + var) / s_n^2, utils/utils.py:89-93) of the last layer's moments. */
int dgp_e_log_p_y(dgp_ctx* ctx, const dgp_model_desc* model, const double* X, const double* Y, int64_t N, int64_t S,
                  const double* const* zs_host, uint64_t seed, int64_t n_offset, double* out);

/* EI.run for a DGP (Infill_criteria.py:36-52): returns -EI [N,1]. analytic != 0: moment-matched closed form;
 * analytic == 0: Monte-Carlo mean_s max(y_min - F, 0) on the propagated samples. */
int dgp_ei(dgp_ctx* ctx, const dgp_model_desc* model, const double* X, int64_t N, int64_t S,
           const double* const* zs_host, uint64_t seed, int64_t n_offset, double y_min, int analytic, double* neg_ei);

/* EI.run (analytic) together with d sum(-EI) / dX [N, D_0]: what tape.gradient(loss, x) gives the reference's Adam-on-x search
 * (Infill_criteria.py:79-84). Runs the forward chain, the EI adjoints and the data path of the adjoint chain (no parameter
 * contractions). */
int dgp_ei_grad(dgp_ctx* ctx, const dgp_model_desc* model, const double* X, int64_t N, int64_t S, const double* const* zs_host,
                uint64_t seed, int64_t n_offset, double y_min, double* neg_ei, double* d_neg_ei_dX);

/* The other moment-based criteria of dgp_dace/Infill_criteria.py, evaluated on mixture moments (mean, var) [n] (DEVICE):
 * kind 0: -EI(y) (:43-47); 1: WB2 -(EI(y) - mean) (:124-133); 2: EV_one_constraint analytic with zero_c = y (:249-257);
 * 3: WB2S -(sigmoid(x) EI(y) - mean) with x [n, d] -> out [n, d] (:187-198); 4: probability of feasibility Phi((y - mean) / s)
 * (PoF, :318-341: the reference computes EI-style terms there and returns nothing; this is the quantity run_with_IC needs).
 * out [n] except for kind 3. */
int dgp_acq_moments(dgp_ctx* ctx, int kind, const double* mean, const double* var, int64_t n, double y, const double* x, int d,
                    double* out);
/* EV_one_constraint Monte-Carlo branch (:259-262): out [ND] = mean_s max(F[s] - zero_c, 0), F [S, ND]. */
int dgp_ev_mc(dgp_ctx* ctx, const double* F, int64_t S, int64_t ND, double zero_c, double* out);
/* Moment matching over the S samples of a propagated layer (models/dgp.py:362-366; EHVI.py:112-119 and the `mo_dgp` branch
 * :124-130, whose two objectives come out of ONE chain): Fmean, Fvar [S, ND] (DEVICE) -> mean [ND] = mean_s Fmean,
 * var [ND] = mean_s (Fvar + lik) + mean_s (Fmean - mean)^2 (centred: no cancellation at large |mean|); lik_variance (DEVICE, [1]) may be NULL (predict_f moments). */
int dgp_mixture_moments(dgp_ctx* ctx, const double* Fmean, const double* Fvar, int64_t S, int64_t ND, const double* lik_variance,
                        double* mean, double* var);

/* EHVI exact 2-objective strip sum (EHVI.py:102-104,154-157) from per-objective moments [N]; ynd0/ynd1: padded
 * Pareto front (EHVI.py:90-100), n entries each, DEVICE pointers. */
int dgp_ehvi2d(dgp_ctx* ctx, const double* m0, const double* v0, const double* m1, const double* v1, int64_t N,
               const double* ynd0, const double* ynd1, int n, double* out);
/* dgp_ehvi2d with its partial derivatives: grads [N][4] = (dE/dm0, dE/dv0, dE/dm1, dE/dv1). Chained to the candidates with
 * dgp_acq_grad kind 4 (one call per objective model), this is the gradient the Adam stage of optimize_EHVI takes with
 * tf.GradientTape (dgp_dace/EHVI.py:218-234). */
int dgp_ehvi2d_grad(dgp_ctx* ctx, const double* m0, const double* v0, const double* m1, const double* v1, int64_t N,
                    const double* ynd0, const double* ynd1, int n, double* out, double* grads);

/* Debug / test hook for the DMMA GEMM engine: C = alpha * A * op(B) + beta * C (row-major, tile-aligned shapes). */
int dgp_debug_gemm(dgp_ctx* ctx, int nt, int M, int N, int K, double alpha, const double* A, const double* B, double beta,
                   double* C, int a_tri, int c_lower, int batch, int splitk, const double* kscale);

#ifdef __cplusplus
}
#endif
#endif
