// C ABI of the B200-native doubly-stochastic DGP hot path (see include/dgp_b200.h for the contract and the
// reference methods each entry point replaces). Host orchestration only: every flop runs in the kernels of
// gemm.cuh (FP64 DMMA contractions), layer.cuh (streaming stages), prep.cuh / small.cuh (replicated M^2 / M^3 work)
// and acq.cuh (acquisition epilogues). There is no CPU fallback: without a CUDA device every call fails.
#include "../../include/dgp_b200.h"

#include <dlfcn.h>

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "acq.cuh"
#include "common.cuh"
#include "fused.cuh"
#include "fused_bwd.cuh"
#include "fullcov.cuh"
#include "extk.cuh"
#include "compkern.cuh"
#include "gemm.cuh"
#include "layer.cuh"
#include "philox.cuh"
#include "prep.cuh"
#include "small.cuh"

using namespace dgp;

struct dgp_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  std::string err;
  // bump arena for per-call device scratch; grown (never shrunk) between calls
  char* ws = nullptr;
  size_t cap = 0, used = 0;
  bool dry = false;
  bool replay = false;                  // allocate as usual but launch nothing: the caller restores the region from a saved copy (dgp_svgp_from_k_cached)
  size_t ws_limit = (size_t)24 << 30;   // chunks of the minibatch are sized to stay under this
  int num_sms = 148;
  bool chol_configured = false;
  int* d_info = nullptr;                // Cholesky failure flag
  // CUDA-graph replay of the ELBO+gradient step (dgp_set_graph): the step's launch sequence depends only on shapes, pointers
  // and flags, so it is captured once per distinct call signature and replayed; the Philox key is read from d_seed
  unsigned long long* d_seed = nullptr; // device slot holding the seed of a replayed step
  const unsigned long long* seed_ptr = nullptr;   // non-null while capturing: kernels read the seed from it
  bool use_graph = false;
  cudaStream_t cap_stream = nullptr;    // capture happens on a private stream (the caller's may be the legacy default stream)
  struct GraphEntry {
    std::vector<unsigned char> key;
    cudaGraphExec_t exec = nullptr;
    long launches = 0;
    std::vector<void*> pinned;          // host tables the captured copies read at every replay
    unsigned long last_use = 0;
  };
  std::vector<GraphEntry> graphs;
  unsigned long graph_tick = 0;
  std::vector<void*>* keep = nullptr;   // non-null while capturing
  double* h_pinned = nullptr;           // staging for the *_host entry points
  size_t h_pinned_bytes = 0;
  double* d_stage = nullptr;            // device side of that staging (outside the arena, which may be re-grown)
  size_t d_stage_bytes = 0;
  bool sync_launches = false;           // DGP_B200_SYNC_LAUNCHES: cudaDeviceSynchronize + error check after every launch (debugging)
  bool vform_forward_calls = true;      // forward-only calls fold q_sqrt_d^T Lu^-T once per step and skip the A pass
  bool use_vform_grad = true;           // ... and so does the ELBO+gradient path (V-form adjoint in backward_layer)
  long vform_grad_min_ps = 32768;       // fewer point-samples than this: keep the A-form adjoint (no Cholesky-adjoint glue)
  bool share_first_layer = true;        // evaluate the first layer once per point instead of once per point-sample
  bool use_fused = true;                // fused conditional kernel (fused.cuh); false -> unfused GEMM pipeline
  bool use_fused_bwd = true;            // fused data-path adjoint (fused_bwd.cuh) for V-form layers it supports
  bool warp_major_groups = false;       // fused kernels: the two warps of an SM sub-partition sit in different column groups
  int group_skew = 0;                   // ... which start this many clocks apart       // fused kernels: the two warps of an SM sub-partition sit in different column groups
  // the layers' replicated per-step work (Kuu build, operator packing, KL, M^3 glue, gradient assembly) is independent per
  // layer and made of tiny launches: it runs on per-layer side streams forked from / joined to the caller's stream
  static constexpr int kAux = 8;
  cudaStream_t aux[kAux] = {nullptr};
  cudaEvent_t ev_fork = nullptr, ev_join[kAux] = {nullptr};
  // per-layer work that only the adjoint / the KL sum consume (Kuu^-1, KL, its adjoint's products) keeps running on the side
  // streams while the forward chain starts; join_late() makes the ctx's stream wait for it
  cudaEvent_t ev_late[kAux] = {nullptr};
  int late_pending = 0;
  // a layer's parameter contractions keep running on the side streams while the next layer's data path of the adjoint chain
  // runs on the ctx's stream (two sets of adjoint temporaries alternate between the layers); join_param() waits for a set
  cudaEvent_t ev_param[2][4] = {{nullptr}};
  int param_pending[2] = {0, 0};
  bool parallel_layers = true;
  // NCCL communicator of the data-parallel step (dgp_comm_init); the library is resolved at run time (libnccl.so.2)
  void* nccl_comm = nullptr;
  int comm_rank = 0, comm_world = 1;
  long launches = 0;                    // kernels launched since the last dgp_reset_launch_count
  // optional per-category device timing (CUDA event pairs around every launch, on the ctx's stream)
  bool profiling = false;
  int cat = 0;
  std::vector<cudaEvent_t> ev_pool;
  struct Span { int cat; cudaEvent_t a, b; };
  std::vector<Span> spans;
  double cat_ms[DGP_PROFILE_CATEGORIES] = {0};
  long cat_launches[DGP_PROFILE_CATEGORIES] = {0};
};

namespace {

#define CK(expr)                                                                                   \
  do {                                                                                             \
    cudaError_t e__ = (expr);                                                                      \
    if (e__ != cudaSuccess) {                                                                      \
      c->err = std::string(#expr) + ": " + cudaGetErrorString(e__);                                \
      return DGP_ERR_CUDA;                                                                         \
    }                                                                                              \
  } while (0)
#define RC(expr)                 \
  do {                           \
    int rc__ = (expr);           \
    if (rc__ != DGP_OK) return rc__; \
  } while (0)
cudaEvent_t prof_event(dgp_ctx* c) {
  cudaEvent_t e = nullptr;
  if (!c->ev_pool.empty()) { e = c->ev_pool.back(); c->ev_pool.pop_back(); }
  else cudaEventCreate(&e);
  return e;
}
struct ProfScope {   // records an event pair around the launches issued during its lifetime
  dgp_ctx* c; cudaEvent_t a = nullptr;
  explicit ProfScope(dgp_ctx* ctx) : c(ctx) {
    if (c->profiling && !c->dry) { a = prof_event(c); cudaEventRecord(a, c->stream); }
  }
  ~ProfScope() {
    if (a) { cudaEvent_t b = prof_event(c); cudaEventRecord(b, c->stream); c->spans.push_back({c->cat, a, b}); }
  }
};
// kernel launch, skipped while planning the workspace
#define LAUNCH(kern, grid, block, smem, ...)                          \
  do {                                                                \
    if (!c->dry && !c->replay) {                                      \
      ProfScope ps__(c);                                              \
      kern<<<grid, block, smem, c->stream>>>(__VA_ARGS__);            \
      ++c->launches;                                                  \
      ++c->cat_launches[c->cat];                                      \
      CK(cudaGetLastError());                                         \
      if (c->sync_launches) {   /* DGP_B200_SYNC_LAUNCHES=1: find the launch that faults */ \
        cudaError_t es__ = cudaDeviceSynchronize();                   \
        if (es__ != cudaSuccess) {                                    \
          c->err = std::string(#kern) + " (line " + std::to_string(__LINE__) + "): " + cudaGetErrorString(es__); \
          fprintf(stderr, "dgp_b200: %s\n", c->err.c_str());          \
          return DGP_ERR_CUDA;                                        \
        }                                                             \
      }                                                               \
    }                                                                 \
  } while (0)
#define CAT(x) c->cat = (x)

double* walloc(dgp_ctx* c, size_t n_doubles) {
  size_t bytes = (n_doubles * sizeof(double) + 255) & ~(size_t)255;
  size_t off = c->used;
  c->used += bytes;
  if (c->dry) return nullptr;
  return reinterpret_cast<double*>(c->ws + off);
}

// Source pointer for a host->device table upload. While a step is being captured into a CUDA graph the copy node re-reads its
// source at every replay, so the table is moved into pinned memory owned by the graph entry.
const void* host_src(dgp_ctx* c, const void* p, size_t bytes) {
  if (!c->keep) return p;
  void* h = nullptr;
  if (cudaMallocHost(&h, bytes ? bytes : 1) != cudaSuccess) return nullptr;
  memcpy(h, p, bytes);
  c->keep->push_back(h);
  return h;
}
#define H2D(dst, src, bytes)                                                                       \
  do {                                                                                             \
    const void* s__ = host_src(c, (src), (bytes));                                                 \
    if (!s__) { c->err = "cudaMallocHost failed while capturing a graph"; return DGP_ERR_CUDA; }   \
    CK(cudaMemcpyAsync((dst), s__, (bytes), cudaMemcpyHostToDevice, c->stream));                   \
  } while (0)

struct LayerFork {   // fork the ctx's stream into per-layer side streams for a loop over layers, join afterwards
  dgp_ctx* c; cudaStream_t main; int n; bool active = false;
  LayerFork(dgp_ctx* ctx, int nlayers) : c(ctx), main(ctx->stream), n(nlayers < dgp_ctx::kAux ? nlayers : dgp_ctx::kAux) {
    // while profiling everything stays on one stream: an event pair around a launch that shares the SMs with launches of other
    // streams would time the sharing, not the kernel
    if (c->dry || nlayers < 2 || !c->parallel_layers || c->profiling) return;
    if (!c->ev_fork) {
      if (cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) != cudaSuccess) return;
      for (int i = 0; i < dgp_ctx::kAux; ++i) {
        if (cudaStreamCreateWithFlags(&c->aux[i], cudaStreamNonBlocking) != cudaSuccess) return;
        if (cudaEventCreateWithFlags(&c->ev_join[i], cudaEventDisableTiming) != cudaSuccess) return;
        if (cudaEventCreateWithFlags(&c->ev_late[i], cudaEventDisableTiming) != cudaSuccess) return;
      }
      for (int k = 0; k < 2; ++k)
        for (int i = 0; i < 4; ++i)
          if (cudaEventCreateWithFlags(&c->ev_param[k][i], cudaEventDisableTiming) != cudaSuccess) return;
    }
    if (cudaEventRecord(c->ev_fork, main) != cudaSuccess) return;
    for (int i = 0; i < n; ++i) cudaStreamWaitEvent(c->aux[i], c->ev_fork, 0);
    active = true;
  }
  void use(int l) { if (active) c->stream = c->aux[l % n]; }
  void join() {
    if (active) {
      for (int i = 0; i < n; ++i) { cudaEventRecord(c->ev_join[i], c->aux[i]); cudaStreamWaitEvent(main, c->ev_join[i], 0); }
      active = false;
    }
    c->stream = main;
  }
  void detach() {   // leave the side streams running; join_late() waits for them
    if (active) {
      for (int i = 0; i < n; ++i) cudaEventRecord(c->ev_late[i], c->aux[i]);
      c->late_pending = n;
      active = false;
    }
    c->stream = main;
  }
  void detach_param(int set) {   // leave the (<= 4) side streams running; join_param(set) waits for them
    if (active) {
      for (int i = 0; i < n; ++i) cudaEventRecord(c->ev_param[set][i], c->aux[i]);
      c->param_pending[set] = n;
      active = false;
    }
    c->stream = main;
  }
  ~LayerFork() { join(); }
};

void join_param(dgp_ctx* c, int set) {
  for (int i = 0; i < c->param_pending[set]; ++i) cudaStreamWaitEvent(c->stream, c->ev_param[set][i], 0);
  c->param_pending[set] = 0;
}

void join_late(dgp_ctx* c) {
  for (int i = 0; i < c->late_pending; ++i) cudaStreamWaitEvent(c->stream, c->ev_late[i], 0);
  c->late_pending = 0;
}
struct LateGuard {   // no exit from a model-level call leaves side-stream work unjoined (the next call reuses the arena)
  dgp_ctx* c;
  ~LateGuard() { join_late(c); join_param(c, 0); join_param(c, 1); }
};

void drop_graphs(dgp_ctx* c);

int ensure_ws(dgp_ctx* c, size_t need) {
  if (need <= c->cap) return DGP_OK;
  CK(cudaStreamSynchronize(c->stream));
  drop_graphs(c);   // captured steps point into the arena being replaced
  if (c->ws) CK(cudaFree(c->ws));
  c->ws = nullptr;
  c->cap = 0;
  size_t want = need + (need >> 3);
  cudaError_t e = cudaMalloc(&c->ws, want);
  if (e != cudaSuccess) {
    cudaGetLastError();
    want = need;
    CK(cudaMalloc(&c->ws, want));
  }
  c->cap = want;
  return DGP_OK;
}

// Planning half of planned(): runs `pass` dry (it lays the arena out and launches nothing), then grows the arena to fit.
template <typename F>
int plan(dgp_ctx* c, F&& pass) {
  c->dry = true; c->used = 0;
  const int rc = pass();
  c->dry = false;
  if (rc != DGP_OK) return rc;
  RC(ensure_ws(c, c->used));
  c->used = 0;
  return DGP_OK;
}

// Runs `pass` once to size the arena and once for real.
template <typename F>
int planned(dgp_ctx* c, F&& pass) {
  RC(plan(c, pass));
  return pass();
}

int gemm(dgp_ctx* c, GemmArgs g, bool nt) {
  if (c->dry || c->replay) return DGP_OK;
  ProfScope ps(c);
  cudaError_t e = gemm_launch(g, nt, c->stream);
  c->launches += g.splitk > 1 ? 2 : 1;
  c->cat_launches[c->cat] += g.splitk > 1 ? 2 : 1;
  if (e == cudaSuccess && c->sync_launches) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) {
    c->err = std::string("gemm_launch: ") + cudaGetErrorString(e);
    if (c->sync_launches)
      fprintf(stderr, "dgp_b200: %s (M %d N %d K %d batch %d nt %d splitk %d lower %d tri %d lda %ld ldb %ld ldc %ld)\n", c->err.c_str(), g.M, g.N,
              g.K, g.batch, (int)nt, g.splitk, g.c_lower, g.a_tri, g.lda, g.ldb, g.ldc);
    return DGP_ERR_CUDA;
  }
  return DGP_OK;
}

GemmArgs gargs(const double* A, long lda, const double* B, long ldb, double* C, long ldc, int M, int N, int K) {
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.A = A; g.lda = lda; g.B = B; g.ldb = ldb; g.C = C; g.ldc = ldc;
  g.M = M; g.N = N; g.K = K;
  g.alpha = 1.0; g.beta = 0.0; g.batch = 1; g.splitk = 1; g.kblocks = 1; g.kblk = K; g.bscale_mul = 1.0;
  return g;
}

// Split-K count for a contraction over the point-samples: the count (<= 64, >= 8 k-tiles per chunk, partial tiles within
// the scratch budget) whose CTA total fills whole waves best; ties go to the smaller count (less reduction traffic).
constexpr size_t kSplitkPartDoubles = (size_t)96 << 20;   // 768 MB of split-K partial tiles at most
constexpr int kSplitkMax = 64;    // most splits of a contraction over the point-samples (sizes the split-K scratch)
constexpr int kLowerWaves = 9;    // CTA waves a lower-only NT contraction is cut into
int pick_splitk(dgp_ctx* c, const GemmArgs& g, bool nt) {
  const GemmPlan p = gemm_plan(g, nt, c->num_sms);
  const size_t out_doubles = (size_t)g.batch * g.M * g.N;
  long smax = kSplitkMax;
  if ((size_t)smax * out_doubles > kSplitkPartDoubles) smax = (long)(kSplitkPartDoubles / out_doubles);
  const long ktiles = g.K / 16;
  if (smax > ktiles / 8) smax = ktiles / 8;
  if (smax < 1) smax = 1;
  if (p.tiles * smax < p.slots) {
    // Even the finest regular split leaves SMs idle: the product is latency-bound (one serial k-loop per CTA), not
    // throughput-bound. Cut K down to two k-steps per CTA, as far as the CTAs still fit in one wave.
    long s = ktiles / 4;
    if (s > 64) s = 64;
    if (s * p.tiles > p.slots) s = p.slots / p.tiles;
    if ((size_t)s * out_doubles > kSplitkPartDoubles) s = (long)(kSplitkPartDoubles / out_doubles);
    while (s > 1 && (s - 1) * ((ktiles + s - 1) / s) >= ktiles) --s;   // no empty last chunk
    return (int)(s < 1 ? 1 : s);
  }
  if (nt && g.c_lower && p.BM == 64 && gemm_small_bk32(g, nt)) {
    // lower-only NT product: its diagonal tiles run the 36-of-64-unit path and finish in ~0.56 of the time of the others, so
    // the CTAs are not uniform and many short CTAs pack better than whole waves of long ones (measured: 11 -> 33 splits, -10%)
    long s = (kLowerWaves * (long)p.slots + p.tiles - 1) / p.tiles;
    if (s > smax) s = smax;
    return (int)(s < 1 ? 1 : s);
  }
  int best = 1;
  double best_eff = -1.0;
  for (long s = 1; s <= smax; ++s) {
    const long chunk = (ktiles + s - 1) / s;
    if ((s - 1) * chunk >= ktiles) continue;   // an empty last chunk
    const long ctas = p.tiles * s;
    const long waves = (ctas + p.slots - 1) / p.slots;
    const double eff = (double)ctas / (double)(waves * p.slots);
    if (eff > best_eff + 0.02) { best_eff = eff; best = (int)s; }
  }
  return best;
}

template <typename F>
int dispatch_dmax(int D, F&& f) {
  if (D <= 1) return f(std::integral_constant<int, 1>());
  if (D <= 2) return f(std::integral_constant<int, 2>());
  if (D <= 4) return f(std::integral_constant<int, 4>());
  if (D <= 8) return f(std::integral_constant<int, 8>());
  if (D <= 16) return f(std::integral_constant<int, 16>());
  return f(std::integral_constant<int, 32>());
}

int check_layer(dgp_ctx* c, const dgp_layer_desc& L) {
  if (L.D_in < 1 || L.D_in > kMaxD - 1 || L.D_out < 1 || L.D_out > kMaxD || L.M < 1) {
    c->err = "layer widths must satisfy 1 <= D_in <= 31, 1 <= D_out <= 32, M >= 1";
    return DGP_ERR_ARG;
  }
  if (round_up(L.M, kTileM) > 768) { c->err = "M > 768 is not supported by the single-CTA Cholesky"; return DGP_ERR_UNSUPPORTED; }
  if (L.kernel_kind < 0 || L.kernel_kind > 2) { c->err = "kernel_kind must be 0 (SquaredExponential), 1 (Matern32) or 2 (Matern52)"; return DGP_ERR_UNSUPPORTED; }
  if (L.mean_kind < 0 || L.mean_kind > 2) { c->err = "mean_kind must be 0 (Zero), 1 (Identity) or 2 (Linear)"; return DGP_ERR_ARG; }
  if (L.mean_kind == 1 && L.D_in != L.D_out) { c->err = "Identity mean function needs D_in == D_out"; return DGP_ERR_ARG; }
  if (L.mean_kind == 2 && !L.mf_W) { c->err = "Linear mean function needs mf_W"; return DGP_ERR_ARG; }
  if (!L.Z || !L.lengthscales || !L.variance || !L.q_mu || !L.q_sqrt) { c->err = "null parameter pointer in layer descriptor"; return DGP_ERR_ARG; }
  return DGP_OK;
}

// ---------------------------------------------------------------------------------------------------------
// per-step replicated state of one layer (a1): everything derived from (Z, l, s2, q_mu, q_sqrt)
// ---------------------------------------------------------------------------------------------------------
struct LayerWs {
  int M = 0, Mp = 0, D_in = 0, D_out = 0;
  double *Ku = nullptr, *Knj = nullptr, *L = nullptr, *Linv = nullptr, *LinvT = nullptr;
  double *RpT = nullptr, *Rcat = nullptr, *qmuP = nullptr;
  // gradient / KL only
  double *Kinv = nullptr, *alpha = nullptr, *KRcat = nullptr, *LRcat = nullptr, *KSK = nullptr;
  // gradient accumulators over the chunks of the minibatch
  double *dKu = nullptr, *dR = nullptr, *dqmu = nullptr, *H = nullptr, *rbf_red = nullptr, *sgv = nullptr;
  double *dZk = nullptr, *kuu_part = nullptr, *kuu_red = nullptr, *kl = nullptr;
  // fused conditional kernel: scaled inducing inputs, packed operator stream, panel schedule
  double *Zs = nullptr, *zz = nullptr, *stream = nullptr;
  PanelDesc* sched = nullptr;
  int NP = 0, fcfg = -1;   // fcfg: index into the fused configurations, -1 = not available
  // V-form of the conditional (forward-only calls): C_d = q_sqrt_d^T Lu^-T [D][Mp][Mp] and beta = Lu^-1 q_mu [Mp][32]
  bool vform = false;
  bool white = false;   // whitened representation (utils/layers.py:246,254-255,296-303): C_d = q_sqrt_d^T, beta = q_mu, KL against N(0, I)
  double *Cmat = nullptr, *betaP = nullptr;
  // V-form adjoint: C_d^T side by side, L^T, accumulators over the chunks (Wacc = [tril(V diag(2 Gv_d) V^T)]_d, dbeta = V Gm) and
  // scratch of the once-per-step re-parameterisation back to (q_mu, q_sqrt, Ku): G1 = tril(dV V^T), DCt = [tril(V dT_d^T)]_d
  double *CTcat = nullptr, *G1 = nullptr, *DCt = nullptr, *Wacc = nullptr, *dbeta = nullptr, *dqmu2 = nullptr, *dRcat = nullptr;
  double *dLinv = nullptr, *sq1 = nullptr, *sq2 = nullptr;
  // fused data-path adjoint (fused_bwd.cuh): packed C_d^T / Lu^-T panel stream; bcfg: 0 = BM 256, 1 = BM 128, -1 = unfused GEMM pipeline
  double* bstream = nullptr; int bcfg = -1, NPb = 0;
  double* part_small = nullptr;   // split-K partials of this layer's long-K M^3-class products (per layer: the layers run concurrently)
};

// ---- fused kernel configurations ----
struct FusedChoice { int BM, PT; };
constexpr FusedChoice kFusedChoices[4] = {{128, 64}, {128, 32}, {64, 64}, {64, 32}};
constexpr size_t kMaxSmem = 227 * 1024;

size_t fused_smem(int cfg, int Mp, int D_in, int D_out) {
  switch (cfg) {
    case 0: return FusedCfg<128, 64, 4, 2>::smem_bytes(Mp, D_in, D_out);
    case 1: return FusedCfg<128, 32, 4, 2>::smem_bytes(Mp, D_in, D_out);
    case 2: return FusedCfg<64, 64, 2, 4>::smem_bytes(Mp, D_in, D_out);
    default: return FusedCfg<64, 32, 2, 4>::smem_bytes(Mp, D_in, D_out);
  }
}

int pick_fused_cfg(int Mp, int D_in, int D_out) {
  static const char* force = getenv("DGP_B200_FUSED_CFG");   // experiment hook: force one configuration
  if (force) { const int cfg = atoi(force); if (cfg >= 0 && cfg < 4 && Mp % kFusedChoices[cfg].BM == 0 && fused_smem(cfg, Mp, D_in, D_out) <= kMaxSmem) return cfg; }
  for (int cfg = 0; cfg < 4; ++cfg) {
    if (Mp % kFusedChoices[cfg].BM) continue;
    if (fused_smem(cfg, Mp, D_in, D_out) <= kMaxSmem) return cfg;
  }
  return -1;
}

// ---- fused data-path adjoint configurations ----
constexpr int kFusedBwdBM[2] = {128, 64};   // 128-row blocks (4 m-tiles per warp); 64-row blocks for Mp = 64, 192, ...
size_t fused_bwd_smem(int cfg, int Mp, int D_in, int D_out) {
  return cfg == 0 ? FusedBwdCfg<128, 64, 4, 2>::smem_bytes(Mp, D_in, D_out) : FusedBwdCfg<64, 64, 2, 4>::smem_bytes(Mp, D_in, D_out);
}
int pick_fused_bwd_cfg(int Mp, int D_in, int D_out) {
  if (D_in > 16) return -1;
  static const char* force = getenv("DGP_B200_FUSED_BWD_CFG");
  for (int cfg = force ? atoi(force) : 0; cfg < 2; ++cfg) {
    if (cfg < 0 || Mp % kFusedBwdBM[cfg]) continue;
    if (fused_bwd_smem(cfg, Mp, D_in, D_out) <= kMaxSmem) return cfg;
  }
  return -1;
}

std::vector<PanelDesc> build_schedule(int Mp, int BM, int D_out, bool vform) {
  std::vector<PanelDesc> v;
  const int nb = Mp / BM, kpb = BM / kPanelK, kt = Mp / kPanelK;
  for (int i = nb - 1; i >= 0; --i)
    for (int ks = 0; ks < (i + 1) * kpb; ++ks) {
      int fl = (ks == 0 ? kPanelFirst : 0) | (ks == (i + 1) * kpb - 1 ? kPanelLast : 0) | (ks * kPanelK >= i * BM ? kPanelClip : 0);
      if ((fl & kPanelLast) && i == 0) fl |= kPanelStageEnd;
      v.push_back(PanelDesc{0, 0, i, ks * kPanelK, fl, 0});
    }
  // upper-operator passes: A (A-form only), then the T_d passes two outputs at a time (the panels of d and d + 1 for the same row block
  // and k-range are adjacent: fused_forward_kernel multiplies both with one set of B fragments), a last single pass when D_out is odd
  auto upper = [&](int kind, int d0, int nd) {
    for (int i = 0; i < nb; ++i)
      for (int ks = i * kpb; ks < kt; ++ks) {
        int fl = (ks == i * kpb ? kPanelFirst : 0) | (ks == kt - 1 ? kPanelLast : 0) | (ks * kPanelK < (i + 1) * BM ? kPanelClip : 0);
        if ((fl & kPanelLast) && i == nb - 1) fl |= kPanelStageEnd;
        for (int d = d0; d < d0 + nd; ++d) v.push_back(PanelDesc{kind, d, i, ks * kPanelK, fl, 0});
      }
  };
  if (!vform) upper(1, 0, 1);
  for (int dp = 0; dp < D_out / 2; ++dp) upper(2, 2 * dp, 2);
  if (D_out & 1) upper(2, D_out - 1, 1);
  return v;
}

enum PrepLevel { PREP_FWD = 0, PREP_KL = 1, PREP_GRAD = 2 };

// What prep_layers lays out: the fused conditional kernel where a configuration fits (else the unfused GEMM pipeline), and the
// V-form for the fused non-white layers (white layers are always V-form).
struct LayerPath { bool fused, vform; };

// The path the ctx's settings select for a model-level call at `level` over `point_samples` point-samples.
LayerPath ctx_path(const dgp_ctx* c, PrepLevel level, long point_samples) {
  // the V-form adjoint pays ~8 extra M^3-class products per layer and step: worth it only when there are enough point-samples
  const bool vform = level == PREP_FWD ? c->vform_forward_calls
                                       : level == PREP_GRAD && c->use_vform_grad && point_samples >= c->vform_grad_min_ps;
  return {c->use_fused, vform};
}

// chol_inv_kernel / tri_inv_kernel opt in to the shared memory of the largest block they factorise (768), once per ctx (= device)
int chol_smem_optin(dgp_ctx* c) {
  if (c->chol_configured) return DGP_OK;
  CK(cudaFuncSetAttribute(chol_inv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)chol_smem_bytes(768)));
  CK(cudaFuncSetAttribute(tri_inv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tri_inv_smem_bytes(768)));
  c->chol_configured = true;
  return DGP_OK;
}

// An M^3-class product whose K runs over the D_out blocks of Mp: few output tiles, long K, so split K over the blocks.
void split_long_k(GemmArgs& g, int D, double* part) {
  g.splitk = D >= 16 ? 16 : (D >= 2 ? D : 1);
  g.part = part;
}

int prep_layers(dgp_ctx* c, const dgp_model_desc* model, std::vector<LayerWs>& lw, PrepLevel level, LayerPath path,
                bool defer_late = false, const double* const* Ku_ext = nullptr) {
  const int nl = model->num_layers;
  lw.assign(nl, LayerWs());
  std::vector<CholArgs> hargs(nl);
  int maxMp = 0;
  for (int l = 0; l < nl; ++l) {
    const dgp_layer_desc& d = model->layers[l];
    RC(check_layer(c, d));
    LayerWs& w = lw[l];
    w.M = d.M; w.Mp = (int)round_up(d.M, kTileM); w.D_in = d.D_in; w.D_out = d.D_out; w.white = d.white != 0;
    const size_t mm = (size_t)w.Mp * w.Mp;
    w.Ku = walloc(c, mm); w.Knj = walloc(c, mm); w.L = walloc(c, mm); w.Linv = walloc(c, mm); w.LinvT = walloc(c, mm);
    w.RpT = walloc(c, mm * w.D_out); w.Rcat = walloc(c, mm * w.D_out); w.qmuP = walloc(c, (size_t)w.Mp * 32);
    if (level >= PREP_KL) {
      w.Kinv = walloc(c, mm); w.alpha = walloc(c, (size_t)w.Mp * 32);
      w.LRcat = walloc(c, mm * w.D_out); w.kl = walloc(c, 1);
    }
    if (level >= PREP_GRAD) {
      w.KRcat = walloc(c, mm * w.D_out); w.KSK = walloc(c, mm); w.part_small = walloc(c, mm * 16);
      w.dKu = walloc(c, mm); w.dR = walloc(c, mm * w.D_out); w.dqmu = walloc(c, (size_t)w.Mp * 32);
      w.H = walloc(c, (size_t)w.Mp * 32); w.rbf_red = walloc(c, 32); w.sgv = walloc(c, 4);
      w.dZk = walloc(c, (size_t)w.M * w.D_in); w.kuu_part = walloc(c, (size_t)w.M * (w.D_in + 1)); w.kuu_red = walloc(c, 32);
    }
    if (w.Mp > maxMp) maxMp = w.Mp;
    hargs[l] = CholArgs{w.Ku, w.L, nullptr, nullptr, w.Mp, c->d_info};   // inverse: tri_inv_kernel
    w.fcfg = path.fused ? pick_fused_cfg(w.Mp, w.D_in, w.D_out) : -1;
    if (w.white && w.fcfg < 0) {
      c->err = "white=True layers run on the fused conditional kernel only (dgp_set_fused(1), and a layer shape it supports)";
      return DGP_ERR_UNSUPPORTED;
    }
    if (w.fcfg >= 0) {
      const int BM = kFusedChoices[w.fcfg].BM;
      const int nb = w.Mp / BM, kpb = BM / kPanelK;
      w.vform = w.white || path.vform;
      w.NP = ((w.vform ? 1 : 2) + w.D_out) * kpb * nb * (nb + 1) / 2;
      if (w.vform) { w.Cmat = walloc(c, mm * w.D_out); w.betaP = walloc(c, (size_t)w.Mp * 32); }
      if (w.vform && level == PREP_GRAD) {
        w.CTcat = walloc(c, mm * w.D_out); w.G1 = walloc(c, mm); w.DCt = walloc(c, mm * w.D_out); w.Wacc = walloc(c, mm * w.D_out);
        w.dbeta = walloc(c, (size_t)w.Mp * 32); w.dqmu2 = walloc(c, (size_t)w.Mp * 32); w.dRcat = walloc(c, mm * w.D_out);
        w.dLinv = walloc(c, mm); w.sq1 = walloc(c, mm); w.sq2 = walloc(c, mm);
        w.bcfg = c->use_fused_bwd ? pick_fused_bwd_cfg(w.Mp, w.D_in, w.D_out) : -1;
        if (w.bcfg >= 0) {
          const int BMb = kFusedBwdBM[w.bcfg], nbb = w.Mp / BMb;
          w.NPb = (w.D_out + 1) * (BMb / kPanelK) * nbb * (nbb + 1) / 2;
          w.bstream = walloc(c, (size_t)w.NPb * BMb * kPanelK);
        }
      }
      w.Zs = walloc(c, (size_t)w.M * w.D_in); w.zz = walloc(c, (size_t)w.Mp);
      w.stream = walloc(c, (size_t)w.NP * BM * kPanelK);
      w.sched = reinterpret_cast<PanelDesc*>(walloc(c, ((size_t)w.NP * sizeof(PanelDesc) + 7) / 8));
    }
  }
  CholArgs* dargs = reinterpret_cast<CholArgs*>(walloc(c, (sizeof(CholArgs) * nl + 7) / 8));
  double** dinv = reinterpret_cast<double**>(walloc(c, (size_t)nl));
  double** dinvT = reinterpret_cast<double**>(walloc(c, (size_t)nl));
  if (c->dry) return DGP_OK;
  std::vector<double*> hinv(nl), hinvT(nl);
  for (int l = 0; l < nl; ++l) { hinv[l] = lw[l].Linv; hinvT[l] = lw[l].LinvT; }
  H2D(dinv, hinv.data(), sizeof(double*) * nl);
  H2D(dinvT, hinvT.data(), sizeof(double*) * nl);

  CAT(DGP_CAT_PREP);
  // d_info is sticky: a failed factorisation stays flagged (and freezes the optimiser kernels) until dgp_check reads and clears it
  H2D(dargs, hargs.data(), sizeof(CholArgs) * nl);
  LayerFork forkA(c, nl);
  for (int l = 0; l < nl; ++l) {
    forkA.use(l);
    const dgp_layer_desc& d = model->layers[l];
    LayerWs& w = lw[l];
    const long mm = (long)w.Mp * w.Mp;
    if (Ku_ext && Ku_ext[l]) LAUNCH(pad_square_identity_kernel, (unsigned)((mm + 255) / 256), 256, 0, Ku_ext[l], w.M, w.Mp, w.Ku);   // caller's Kuu + jitter I
    else LAUNCH(kuu_build_kernel, (unsigned)((mm + 255) / 256), 256, 0, d.Z, d.lengthscales, d.variance, w.M, w.Mp, w.D_in, d.jitter, w.Ku, w.Knj, d.kernel_kind);
    const long np = mm * w.D_out > (long)w.Mp * 32 ? mm * w.D_out : (long)w.Mp * 32;
    LAUNCH(pad_params_kernel, (unsigned)((np + 255) / 256), 256, 0, d.q_sqrt, d.q_mu, w.M, w.Mp, w.D_out, w.RpT, w.Rcat, w.qmuP);
  }
  forkA.join();
  RC(chol_smem_optin(c));
  LAUNCH(chol_inv_kernel, nl, kCholThreads, chol_smem_bytes(maxMp), dargs);
  LAUNCH(tri_inv_kernel, dim3((unsigned)(maxMp / 32), (unsigned)nl), 256, tri_inv_smem_bytes(maxMp), dargs, dinv, dinvT);
  LayerFork forkB(c, nl);
  for (int l = 0; l < nl; ++l) {   // operator stream of the fused conditional kernel
    forkB.use(l);
    LayerWs& w = lw[l];
    if (w.fcfg < 0) continue;
    const dgp_layer_desc& d = model->layers[l];
    const int BM = kFusedChoices[w.fcfg].BM;
    if (w.white) {   // whitened: q(v) is given in the basis the solve already works in
      w.Cmat = w.RpT;
      w.betaP = w.qmuP;
    } else if (w.vform) {
      GemmArgs g = gargs(w.RpT, w.Mp, w.LinvT, w.Mp, w.Cmat, w.Mp, w.Mp, w.Mp, w.Mp);   // C_d = q_sqrt_d^T Lu^-T (upper x upper)
      g.a_tri = 2; g.batch = w.D_out; g.sA = (long)w.Mp * w.Mp; g.sB = 0; g.sC = (long)w.Mp * w.Mp;
      RC(gemm(c, g, false));
      g = gargs(w.Linv, w.Mp, w.qmuP, 32, w.betaP, 32, w.Mp, 32, w.Mp);                   // beta = Lu^-1 q_mu
      g.a_tri = 1;
      RC(gemm(c, g, false));
    }
    if (w.vform && level == PREP_GRAD) {
      const long nct = (long)w.D_out * w.Mp * w.Mp;
      LAUNCH(vform_transpose_kernel, (unsigned)((nct + 255) / 256), 256, 0, w.Cmat, w.Mp, w.D_out, w.CTcat);
      if (w.bcfg == 0) LAUNCH(pack_bwd_stream_kernel<128>, w.NPb, 256, 0, w.Cmat, w.LinvT, w.Mp, w.D_out, w.bstream);
      else if (w.bcfg == 1) LAUNCH(pack_bwd_stream_kernel<64>, w.NPb, 256, 0, w.Cmat, w.LinvT, w.Mp, w.D_out, w.bstream);
      // c_lower products leave the tiles above the diagonal unwritten: start the accumulators from zero
      CK(cudaMemsetAsync(w.Wacc, 0, (size_t)nct * sizeof(double), c->stream));
    }
    std::vector<PanelDesc> sch = build_schedule(w.Mp, BM, w.D_out, w.vform);
    if ((int)sch.size() != w.NP) { c->err = "internal: panel schedule size mismatch"; return DGP_ERR_ARG; }
    H2D(w.sched, sch.data(), sch.size() * sizeof(PanelDesc));
    LAUNCH(scale_z_kernel, (unsigned)((w.M * w.D_in + 255) / 256), 256, 0, d.Z, d.lengthscales, w.M, w.D_in, w.Zs);
    LAUNCH(zz_kernel, (unsigned)((w.Mp + 127) / 128), 128, 0, w.Zs, w.M, w.Mp, w.D_in, w.zz);
    const double* tsrc = w.vform ? w.Cmat : w.RpT;   // operator of the T_d passes
    if (BM == 128) LAUNCH(pack_stream_kernel<128>, w.NP, 256, 0, w.sched, w.Linv, w.LinvT, tsrc, w.Mp, w.stream);
    else LAUNCH(pack_stream_kernel<64>, w.NP, 256, 0, w.sched, w.Linv, w.LinvT, tsrc, w.Mp, w.stream);
  }
  forkB.join();
  if (level >= PREP_KL) {
    // consumed by the adjoint / the final KL sum only: with defer_late the forward chain does not wait for these
    LayerFork forkC(c, nl);
    for (int l = 0; l < nl; ++l) {
      forkC.use(l);
      LayerWs& w = lw[l];
      const int Mp = w.Mp, D = w.D_out;
      if (w.white) {   // KL(q(v) || N(0, I)) needs no product with Ku
        LAUNCH(kl_white_kernel, 1, 1024, 0, w.Rcat, w.qmuP, w.M, Mp, D, w.kl);
        continue;
      }
      GemmArgs g = gargs(w.LinvT, Mp, w.Linv, Mp, w.Kinv, Mp, Mp, Mp, Mp);   // Kinv = Linv^T Linv
      g.a_tri = 2;
      RC(gemm(c, g, false));
      g = gargs(w.Kinv, Mp, w.qmuP, 32, w.alpha, 32, Mp, 32, Mp);            // alpha = Kinv q_mu
      RC(gemm(c, g, false));
      g = gargs(w.Linv, Mp, w.Rcat, (long)D * Mp, w.LRcat, (long)D * Mp, Mp, D * Mp, Mp);   // Linv [R_1 .. R_D]
      g.a_tri = 1;
      RC(gemm(c, g, false));
      LAUNCH(kl_kernel, 1, 1024, 0, w.L, w.Rcat, w.LRcat, w.qmuP, w.alpha, w.M, Mp, D, w.kl);
      if (level >= PREP_GRAD) {
        g = gargs(w.Kinv, Mp, w.Rcat, (long)D * Mp, w.KRcat, (long)D * Mp, Mp, D * Mp, Mp);  // Kinv [R_1 .. R_D]
        RC(gemm(c, g, false));
        g = gargs(w.KRcat, (long)D * Mp, w.KRcat, (long)D * Mp, w.KSK, Mp, Mp, Mp, D * Mp);   // sum_d (Kinv R_d)(Kinv R_d)^T
        split_long_k(g, D, w.part_small);
        RC(gemm(c, g, true));
      }
    }
    // (not while profiling: an event pair around a launch that waits for SMs behind the forward chain would time the wait)
    if (defer_late && !c->profiling) forkC.detach();
  }
  return DGP_OK;
}

// ---------------------------------------------------------------------------------------------------------
// one chunk of the minibatch: Nc points x S samples, chained through the layers
// ---------------------------------------------------------------------------------------------------------
struct ChunkLayer {
  const double* Xin = nullptr; long xmod = 0;     // layer input [P][D_in] (layer 0: X rows, shared over S)
  double *F = nullptr, *Fmean = nullptr, *Fvar = nullptr, *z = nullptr;   // [P][D_out]
  double *A = nullptr, *T = nullptr;              // [Mp][Pp], [D_out][Mp][Pp]  (stash for the adjoint)
};

struct ChunkIO {   // caller-visible arrays [S][N][D_l], any may be null
  const double* const* zs = nullptr;
  double* const* Fs = nullptr;
  double* const* Fmeans = nullptr;
  double* const* Fvars = nullptr;
};

struct Temps { double *t0 = nullptr, *t1 = nullptr, *t2 = nullptr; };   // three [maxMp][Pp] planes

// q_mu is staged whole in shared memory by the unfused moments kernel
bool moments_fit(dgp_ctx* c, const LayerWs& w) {
  if (w.fcfg >= 0 || (size_t)w.M * w.D_out * sizeof(double) <= 160 * 1024) return true;
  c->err = "unfused conditional: M * D_out * 8 bytes of q_mu exceed the 160 KiB staged per CTA (fused path: M <= 256, D_out <= 16)";
  return false;
}

// ---- A-form GEMM pipeline of the conditional and its data-path adjoint, on [Mp][Pp] planes ----

// V = Lu^-1 Kuf, A = Lu^-T V, T_d = q_sqrt_d^T A
int aform_forward(dgp_ctx* c, const LayerWs& w, const double* K, double* V, double* A, double* T, long Pp) {
  const int Mp = w.Mp;
  GemmArgs g = gargs(w.Linv, Mp, K, Pp, V, Pp, Mp, (int)Pp, Mp);    // V = Lu^-1 Kuf            (layers.py:245)
  g.a_tri = 1;
  RC(gemm(c, g, false));
  g = gargs(w.LinvT, Mp, V, Pp, A, Pp, Mp, (int)Pp, Mp);            // A = Lu^-T V              (layers.py:247)
  g.a_tri = 2;
  RC(gemm(c, g, false));
  g = gargs(w.RpT, Mp, A, Pp, T, Pp, Mp, (int)Pp, Mp);              // T_d = q_sqrt_d^T A       (layers.py:257-271)
  g.a_tri = 2; g.batch = w.D_out; g.sA = (long)Mp * Mp; g.sB = 0; g.sC = (long)Mp * Pp;
  return gemm(c, g, false);
}

int forward_layer(dgp_ctx* c, const dgp_layer_desc& d, const LayerWs& w, ChunkLayer& cl, const Temps& tmp, bool stash,
                  double* Tshared, int layer, long Nc, long S, long N_total, long n0, unsigned long long seed, long n_offset,
                  const ChunkIO& io, bool need_sample) {
  const long P = Nc * S, Pp = round_up(P, kTileP);
  const int Mp = w.Mp, D = w.D_out;
  if (w.fcfg >= 0) {
    CAT(DGP_CAT_FUSED_FWD);
    FusedFwdArgs f;
    memset(&f, 0, sizeof(f));
    f.stream = w.stream; f.sched = w.sched; f.NP = w.NP; f.Zs = w.Zs; f.zz = w.zz; f.ls = d.lengthscales; f.var = d.variance;
    f.vform = w.vform ? 1 : 0; f.qmu = w.vform ? w.betaP : d.q_mu; f.qmu_ld = w.vform ? 32 : w.D_out;
    f.Xin = cl.Xin; f.xmod = cl.xmod; f.D_in = w.D_in; f.mfW = d.mf_W; f.mfb = d.mf_b; f.mean_kind = d.mean_kind; f.kind = d.kernel_kind;
    f.z_in = (io.zs && io.zs[layer]) ? io.zs[layer] : nullptr;
    f.seed = seed; f.seed_ptr = c->seed_ptr; f.layer = layer; f.Nc = Nc; f.N_total = N_total; f.n0 = n0; f.n_offset = n_offset;
    f.M = w.M; f.Mp = w.Mp; f.D_out = w.D_out; f.P = P; f.Pp = Pp; f.jitter = d.jitter;
    f.Fmean = cl.Fmean; f.Fvar = cl.Fvar; f.F = need_sample ? cl.F : nullptr; f.z = need_sample ? cl.z : nullptr;
    f.xFmean = (io.Fmeans && io.Fmeans[layer]) ? io.Fmeans[layer] : nullptr;
    f.xFvar = (io.Fvars && io.Fvars[layer]) ? io.Fvars[layer] : nullptr;
    f.xF = (io.Fs && io.Fs[layer]) ? io.Fs[layer] : nullptr;
    f.stashA = stash ? cl.A : nullptr; f.stashT = stash ? cl.T : nullptr;
    f.warp_major_groups = c->warp_major_groups ? 1 : 0; f.group_skew = c->group_skew;
    // few point-samples (a shared first layer, a BO-sized batch): halve the tile so that twice as many SMs share the launch;
    // the packed operator stream depends on BM only
    const int cfg = ((w.fcfg == 0 || w.fcfg == 2) && Pp / 64 <= c->num_sms / 2) ? w.fcfg + 1 : w.fcfg;
    const size_t smem = fused_smem(cfg, w.Mp, w.D_in, w.D_out);
    const long ntiles = Pp / kFusedChoices[cfg].PT;
    const long slots = (long)c->num_sms * ((cfg == 3 && smem <= 112 * 1024) ? 2 : 1);   // the small configuration fits two CTAs per SM
    const unsigned grid = (unsigned)(ntiles < slots ? ntiles : slots);
#define FUSED_LAUNCH(BM_, PT_, WM_, WN_)                                                                                   \
    do {                                                                                                                   \
      if (!c->dry) CK(cudaFuncSetAttribute(fused_forward_kernel<BM_, PT_, WM_, WN_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem)); \
      LAUNCH((fused_forward_kernel<BM_, PT_, WM_, WN_>), grid, (FusedCfg<BM_, PT_, WM_, WN_>::THREADS), smem, f);                                              \
    } while (0)
    switch (cfg) {
      case 0: FUSED_LAUNCH(128, 64, 4, 2); break;
      case 1: FUSED_LAUNCH(128, 32, 4, 2); break;
      case 2: FUSED_LAUNCH(64, 64, 2, 4); break;
      default: FUSED_LAUNCH(64, 32, 2, 4); break;
    }
#undef FUSED_LAUNCH
    return DGP_OK;
  }
  double* K = tmp.t0;
  double* V = tmp.t1;
  double* A = stash ? cl.A : tmp.t2;
  double* T = stash ? cl.T : Tshared;
  CAT(DGP_CAT_KUF);
  LAUNCH(kuf_kernel, dim3((unsigned)(Pp / kKufCols), (unsigned)(Mp / kKufRows)), 256, 0, cl.Xin, cl.xmod, d.Z, d.lengthscales,
         d.variance, w.M, Mp, w.D_in, P, Pp, K, d.kernel_kind);
  CAT(DGP_CAT_GEMM_FWD);
  RC(aform_forward(c, w, K, V, A, T, Pp));

  CAT(DGP_CAT_MOMENTS);
  MomentsArgs a;
  memset(&a, 0, sizeof(a));
  a.V = V; a.A = A; a.T = T; a.qmu = d.q_mu; a.var = d.variance;
  a.Xin = cl.Xin; a.xmod = cl.xmod; a.D_in = w.D_in;
  a.mfW = d.mf_W; a.mfb = d.mf_b; a.mean_kind = d.mean_kind;
  a.z_in = (io.zs && io.zs[layer]) ? io.zs[layer] : nullptr;
  a.seed = seed; a.seed_ptr = c->seed_ptr; a.layer = layer; a.Nc = Nc; a.N_total = N_total; a.n0 = n0; a.n_offset = n_offset;
  a.M = w.M; a.Mp = Mp; a.D_out = D; a.P = P; a.Pp = Pp; a.jitter = d.jitter;
  a.Fmean = cl.Fmean; a.Fvar = cl.Fvar; a.F = need_sample ? cl.F : nullptr; a.z = need_sample ? cl.z : nullptr;
  a.xFmean = (io.Fmeans && io.Fmeans[layer]) ? io.Fmeans[layer] : nullptr;
  a.xFvar = (io.Fvars && io.Fvars[layer]) ? io.Fvars[layer] : nullptr;
  a.xF = (io.Fs && io.Fs[layer]) ? io.Fs[layer] : nullptr;
  const size_t smem = (size_t)w.M * D * sizeof(double);
  if (!moments_fit(c, w)) return DGP_ERR_UNSUPPORTED;
  return dispatch_dmax(D, [&](auto dm) -> int {
    constexpr int DM = decltype(dm)::value;
    if (!c->dry) {
      CK(cudaFuncSetAttribute(moments_kernel<DM>, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    }
    LAUNCH(moments_kernel<DM>, (unsigned)((P + 127) / 128), 128, smem, a);
    return DGP_OK;
  });
}

struct Upstream { double *Gm, *GvT, *GmPad, *gq, *part; long nblocks; };

// The contractions over the point-samples that produce a layer's parameter gradients are independent of each other: they run
// side by side on the ctx's side streams, each with its own slice of the split-K scratch. On sub-wave calls that multiplies the
// occupied SMs; on full-size calls each kernel's tail wave is filled by the next kernel's CTAs (config 2: 100.9 -> 98.8 ms/step).
// `on_main` is issued on the caller's stream while they run.
struct ParamScratch {
  double* part = nullptr; size_t cap = 0;
  bool fixed = false; size_t off[4] = {0, 0, 0, 0}, room[4] = {0, 0, 0, 0};   // per-contraction regions that hold for every layer
  int defer_set = -1;   // >= 0: leave the contractions running and record their completion for join_param(defer_set)
};

template <typename F>
int param_gemms(dgp_ctx* c, GemmArgs* gs, const bool* nts, int n, const ParamScratch& ps, const int* slots, F&& on_main) {
  size_t off[8], total = 0;
  bool fixed = ps.fixed && n <= 4;
  auto slot = [&](int i) { return slots ? slots[i] : i; };   // which fixed scratch region contraction i uses
  for (int i = 0; i < n; ++i) {
    gs[i].splitk = pick_splitk(c, gs[i], nts[i]);
    off[i] = total;
    const size_t need = gs[i].splitk > 1 ? (size_t)gs[i].splitk * gs[i].batch * gs[i].M * gs[i].N : 0;
    total += (need + 31) & ~(size_t)31;
    if (fixed && need > ps.room[slot(i)]) fixed = false;
  }
  const bool par = fixed || total <= ps.cap;
  LayerFork fk(c, par ? n : 0);
  for (int i = 0; i < n; ++i) {
    fk.use(i);
    gs[i].part = ps.part + (fk.active ? (fixed ? ps.off[slot(i)] : off[i]) : 0);
    RC(gemm(c, gs[i], nts[i]));
  }
  if (fk.active) c->stream = fk.main;
  RC(on_main());
  // two layers' contractions may be in flight only with regions that do not depend on the layer; not while profiling (an event
  // pair around a launch that shares the SMs with another stream would time the sharing)
  if (fk.active && fixed && ps.defer_set >= 0 && !c->profiling) fk.detach_param(ps.defer_set);
  else fk.join();
  return DGP_OK;
}

// dA' = q_mu Gm^T + sum_d R_d (2 Gv_d o T_d), W = Ku^-1 dA'                          (SURVEY §9)
// With `split` (split-K scratch shared with the parameter contractions still in flight), few point-samples deal the D blocks of
// the second product out to splits.
int aform_adjoint(dgp_ctx* c, const LayerWs& w, const double* T, const double* GmPad, const double* GvT, double* dA, double* W,
                  long Pp, const ParamScratch* split) {
  const int Mp = w.Mp, D = w.D_out;
  GemmArgs g = gargs(w.qmuP, 32, GmPad, 32, dA, Pp, Mp, (int)Pp, 32);
  RC(gemm(c, g, true));
  g = gargs(w.Rcat, (long)D * Mp, T, Pp, dA, Pp, Mp, (int)Pp, D * Mp);
  g.a_tri = 1; g.kblocks = D; g.kblk = Mp; g.bscale = GvT; g.ld_bscale = Pp; g.bscale_mul = 2.0; g.beta = 1.0;
  if (D == 1) g.kblocks = 1;
  if (split && D > 1) {
    // few point-samples (a shared first layer): too few output tiles to occupy the GPU, so deal the D blocks out to splits
    const GemmPlan p = gemm_plan(g, false, c->num_sms);
    long s = p.tiles > 0 ? p.slots / (2 * p.tiles) : 1;
    if (s > D) s = D;
    if (s >= 2 && (size_t)s * Mp * Pp <= split->cap) {
      join_param(c, 0); join_param(c, 1);   // the scratch is shared with the parameter contractions still in flight
      g.splitk = (int)s; g.part = split->part;
    }
  }
  RC(gemm(c, g, false));
  g = gargs(w.Kinv, Mp, dA, Pp, W, Pp, Mp, (int)Pp, Mp);
  return gemm(c, g, false);
}

// The contractions over the point-samples that give the data parts of dKu, dq_sqrt and dq_mu (NT flags in kAformParamNT),
// accumulated onto the previous chunks' with `beta`.
constexpr bool kAformParamNT[3] = {true, true, false};
void aform_param_args(const LayerWs& w, const double* W, const double* A, const double* T, const double* GvT, const double* GmPad,
                      long Pp, double beta, GemmArgs pg[3]) {
  const int Mp = w.Mp;
  pg[0] = gargs(W, Pp, A, Pp, w.dKu, Mp, Mp, Mp, (int)Pp);          // dKu (data part) = -Wg A^T
  pg[0].alpha = -1.0; pg[0].beta = beta;
  pg[1] = gargs(A, Pp, T, Pp, w.dR, Mp, Mp, Mp, (int)Pp);           // dq_sqrt_d (data part) = tril(A diag(2 Gv_d) T_d^T)
  pg[1].alpha = 2.0; pg[1].beta = beta; pg[1].batch = w.D_out; pg[1].sA = 0; pg[1].sB = (long)Mp * Pp; pg[1].sC = (long)Mp * Mp;
  pg[1].c_lower = 1; pg[1].kscale = GvT; pg[1].sScale = Pp;
  pg[2] = gargs(A, Pp, GmPad, 32, w.dqmu, 32, Mp, 32, (int)Pp);     // dq_mu (data part) = A Gm
  pg[2].beta = beta;
}

// RBF adjoint on the Kuf block: W -> Wg (in place), Gbar, dXin, [X,1], partial sums for dl / ds2. VF: W is K-bar = dELBO/dKuf of
// the V-form and A is null; otherwise W = Ku^-1 dA' and A the stashed A plane. Sets `nb` to the blocks launched (one row of
// partial sums each, for reduce_partials_kernel).
template <bool VF>
int kernel_adjoint(dgp_ctx* c, const dgp_layer_desc& d, const LayerWs& w, const ChunkLayer& cl, const Upstream& up, double* W,
                   const double* A, double* Gbar, double* dXin, double* XaugPad, double* rbf_part, long P, long& nb) {
  const long Pp = round_up(P, kTileP);
  CAT(DGP_CAT_RBF_BWD);
  RbfBwdArgs r;
  memset(&r, 0, sizeof(r));
  r.W = W; r.A = A; r.gq = up.gq; r.Gbar = Gbar; r.Xin = cl.Xin; r.xmod = cl.xmod; r.Z = d.Z; r.ls = d.lengthscales;
  r.var = d.variance; r.M = w.M; r.Mp = w.Mp; r.D_in = w.D_in; r.P = P; r.Pp = Pp; r.Gm = up.Gm; r.D_out = w.D_out;
  r.mean_kind = d.mean_kind; r.mfW = d.mf_W; r.kind = d.kernel_kind; r.dXin = dXin; r.XaugPad = XaugPad; r.part = rbf_part;
  // latency-bound launch: 64-column blocks with 4 row groups, where their shared memory fits
  const bool small = Pp / 128 < 2L * c->num_sms && rbf_bwd_smem_bytes(w.M, w.D_in) <= kRbfBwdSmemMax;
  nb = small ? Pp / kRbfCols : Pp / 128;
  const size_t smem = small ? rbf_bwd_smem_bytes(w.M, w.D_in) : ((size_t)w.M * w.D_in + kMaxD + 32) * sizeof(double);
  return dispatch_dmax(w.D_in, [&](auto dm) -> int {
    constexpr int DM = decltype(dm)::value;
    if (small) {
      if (!c->dry) CK(cudaFuncSetAttribute((rbf_bwd2d_kernel<DM, VF>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kRbfBwdSmemMax));
      LAUNCH((rbf_bwd2d_kernel<DM, VF>), (unsigned)nb, 256, smem, r);
    } else {
      if (!c->dry) CK(cudaFuncSetAttribute((rbf_bwd_kernel<DM, VF>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kRbfBwdSmemMax));
      LAUNCH((rbf_bwd_kernel<DM, VF>), (unsigned)nb, 128, smem, r);
    }
    return DGP_OK;
  });
}

int backward_layer(dgp_ctx* c, const dgp_layer_desc& d, const LayerWs& w, const ChunkLayer& cl, const Temps& tmp,
                   const Upstream& up, double* dXin, double* XaugPad, double* rbf_part, const ParamScratch& ps, long Nc, long S, bool first_chunk,
                   bool params = true) {
  const long P = Nc * S, Pp = round_up(P, kTileP);
  const int Mp = w.Mp, D = w.D_out;
  const double beta = first_chunk ? 0.0 : 1.0;
  double* dA = tmp.t0;
  double* W = tmp.t1;
  double* Gbar = tmp.t2;
  if (w.vform) {
    // ---- V-form adjoint: cl.A holds V = Lu^-1 Kuf, T_d = C_d V, mean = V^T beta ----
    const double* V = cl.A;
    double* dV = dA;
    double* Kbar = W;
    const bool fused_bwd = w.bcfg >= 0;
    const long ntile64 = Pp / 64;
    long nbv = 0;
    if (fused_bwd) {
      // ---- one launch: dV, K-bar = Lu^-T dV and the kernel adjoint on resident tiles (fused_bwd.cuh) ----
      CAT(DGP_CAT_FUSED_BWD);
      FusedBwdArgs f;
      memset(&f, 0, sizeof(f));
      f.stream = w.bstream; f.V = V; f.T = cl.T; f.GvT = up.GvT; f.gq = up.gq; f.Gm = up.GmPad; f.gm_ld = 32; f.beta = w.betaP;
      f.Zs = w.Zs; f.zz = w.zz; f.ls = d.lengthscales; f.var = d.variance; f.Xin = cl.Xin; f.xmod = cl.xmod; f.D_in = w.D_in;
      f.mfW = d.mf_W; f.mean_kind = d.mean_kind; f.kind = d.kernel_kind; f.M = w.M; f.Mp = Mp; f.D_out = D; f.P = P; f.Pp = Pp;
      f.dV = nullptr;   // dV stays on chip: the parameter contractions below do not read it
      f.Gbar = Gbar; f.dXin = dXin; f.XaugPad = XaugPad; f.part = rbf_part;
      f.warp_major_groups = c->warp_major_groups ? 1 : 0; f.group_skew = c->group_skew;
      nbv = ntile64 * (w.bcfg == 0 ? 2 : 4);   // one row of partial sums per tile and column group
      const size_t smem = fused_bwd_smem(w.bcfg, Mp, w.D_in, D);
      const unsigned grid = (unsigned)(ntile64 < c->num_sms ? ntile64 : c->num_sms);
#define FUSED_BWD_LAUNCH(BM_, WM_, WN_, DM_)                                                                                \
      do {                                                                                                                  \
        if (!c->dry) CK(cudaFuncSetAttribute((fused_backward_kernel<BM_, 64, WM_, WN_, DM_>), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kMaxSmem)); \
        LAUNCH((fused_backward_kernel<BM_, 64, WM_, WN_, DM_>), grid, 384, smem, f);                                        \
      } while (0)
      if (w.bcfg == 0) { if (w.D_in <= 8) FUSED_BWD_LAUNCH(128, 4, 2, 8); else FUSED_BWD_LAUNCH(128, 4, 2, 16); }
      else { if (w.D_in <= 8) FUSED_BWD_LAUNCH(64, 2, 4, 8); else FUSED_BWD_LAUNCH(64, 2, 4, 16); }
#undef FUSED_BWD_LAUNCH
    } else {
    CAT(DGP_CAT_GEMM_BWD_DATA);
    // dV = beta Gm^T + sum_d C_d^T (2 Gv_d o T_d) - 2 V diag(sum_d Gv_d)          (gq = -sum_d Gv_d)
    GemmArgs g = gargs(w.betaP, 32, up.GmPad, 32, dV, Pp, Mp, (int)Pp, 32);
    RC(gemm(c, g, true));
    g = gargs(w.CTcat, (long)D * Mp, cl.T, Pp, dV, Pp, Mp, (int)Pp, D * Mp);
    g.a_tri = 1; g.kblocks = D; g.kblk = Mp; g.bscale = up.GvT; g.ld_bscale = Pp; g.bscale_mul = 2.0; g.beta = 1.0;
    if (D == 1) g.kblocks = 1;
    g.epi_plane = V; g.ld_epi = Pp; g.epi_col = up.gq; g.epi_mul = 2.0;
    RC(gemm(c, g, false));
    // K-bar = dELBO/dKuf = Lu^-T dV
    g = gargs(w.LinvT, Mp, dV, Pp, Kbar, Pp, Mp, (int)Pp, Mp);
    g.a_tri = 2;
    RC(gemm(c, g, false));
    RC(kernel_adjoint<true>(c, d, w, cl, up, Kbar, nullptr, Gbar, dXin, XaugPad, rbf_part, P, nbv));
    }
    if (!params) return DGP_OK;
    CAT(DGP_CAT_GEMM_BWD_PARAM);
    // Contractions over the point-samples. With dT_d = 2 Gv_d o (C_d V) and gq = -sum_d Gv_d both matrix accumulators of the V-form
    // are functions of the D_out symmetric matrices W_d = V diag(2 Gv_d) V^T:
    //   (dC_d)^T = V dT_d^T = W_d C_d^T,      dV V^T = beta (V Gm)^T + sum_d (C_d^T C_d - I) W_d,
    // so only tril(W_d) is accumulated here (D_out lower-only products instead of D_out + 1, and neither dV nor the T_d stash is
    // read again); the M^3-class products that turn W_d into G1 and DCt run once per step (run_model).
    GemmArgs pg[3];
    const bool pnt[3] = {true, false, false};
    const int slots[3] = {1, 2, 3};
    pg[0] = gargs(V, Pp, V, Pp, w.Wacc, (long)D * Mp, Mp, Mp, (int)Pp);
    pg[0].alpha = 2.0; pg[0].beta = beta; pg[0].batch = D; pg[0].sA = 0; pg[0].sB = 0; pg[0].sC = Mp; pg[0].c_lower = 1;
    pg[0].kscale = up.GvT; pg[0].sScale = Pp;
    // dbeta = V Gm ;  H = Gbar [X, 1]
    pg[1] = gargs(V, Pp, up.GmPad, 32, w.dbeta, 32, Mp, 32, (int)Pp);
    pg[1].beta = beta;
    pg[2] = gargs(Gbar, Pp, XaugPad, 32, w.H, 32, Mp, 32, (int)Pp);
    pg[2].beta = beta;
    RC(param_gemms(c, pg, pnt, 3, ps, slots, [&]() -> int {
      LAUNCH(reduce_partials_kernel, w.D_in + 1, 256, 0, rbf_part, nbv, w.D_in + 1, w.rbf_red, first_chunk ? 0 : 1);
      LAUNCH(reduce_partials_kernel, 3, 256, 0, up.part, up.nblocks, 3, w.sgv, first_chunk ? 0 : 1);
      return DGP_OK;
    }));
    return DGP_OK;
  }
  CAT(DGP_CAT_GEMM_BWD_DATA);
  RC(aform_adjoint(c, w, cl.T, up.GmPad, up.GvT, dA, W, Pp, &ps));
  long nb = 0;
  RC(kernel_adjoint<false>(c, d, w, cl, up, W, cl.A, Gbar, dXin, XaugPad, rbf_part, P, nb));
  if (!params) return DGP_OK;   // input gradient only (acquisition): the contractions over the point-samples are not needed
  CAT(DGP_CAT_GEMM_BWD_PARAM);
  GemmArgs pg[4];
  const bool pnt[4] = {kAformParamNT[0], kAformParamNT[1], kAformParamNT[2], false};
  aform_param_args(w, W, cl.A, cl.T, up.GvT, up.GmPad, Pp, beta, pg);
  pg[3] = gargs(Gbar, Pp, XaugPad, 32, w.H, 32, Mp, 32, (int)Pp);   // H = Gbar [X, 1]
  pg[3].beta = beta;
  RC(param_gemms(c, pg, pnt, 4, ps, nullptr, [&]() -> int {
    LAUNCH(reduce_partials_kernel, w.D_in + 1, 256, 0, rbf_part, nb, w.D_in + 1, w.rbf_red, first_chunk ? 0 : 1);
    LAUNCH(reduce_partials_kernel, 3, 256, 0, up.part, up.nblocks, 3, w.sgv, first_chunk ? 0 : 1);
    return DGP_OK;
  }));
  return DGP_OK;
}

struct RunOpts {
  bool want_grad = false, want_elbo = false;
  const double* Y = nullptr; int Dy = 0;
  double scale = 1.0, kl_weight = 1.0;
  double* out_flat = nullptr;            // elbo / gradient buffer (device)
  ChunkIO io;
  // prediction outputs
  double* pm = nullptr; double* pv = nullptr; int add_lik = 0;   // mixture moments [N][D_L]
  double* ve = nullptr;                                          // E_log_p_Y [N][D_L] (needs Y)
  double* ei = nullptr; double y_min = 0.0; int ei_analytic = 1; // -EI [N][D_L]
  bool need_last_sample = false;
  double* dx = nullptr;                                          // d sum(-EI) / dX [N][D0] (analytic EI only)
  int acq_kind = 0, acq_add_lik = 0;                             // criterion of the o.dx path (ei_upstream_kernel)
};

// Split-K scratch of the adjoint: four regions (the parameter contractions of a layer run side by side), sized for the widest
// layer so that the same layout serves every layer.
void splitk_regions(const std::vector<LayerWs>& lw, size_t room[4]) {
  size_t Mp = 0, D = 1;
  for (const LayerWs& w : lw) {
    if ((size_t)w.Mp > Mp) Mp = w.Mp;
    if ((size_t)w.D_out > D) D = w.D_out;
  }
  const size_t sm = kSplitkMax;
  room[0] = sm * Mp * Mp; room[1] = sm * D * Mp * Mp; room[2] = sm * Mp * 32; room[3] = sm * Mp * 32;
}
size_t max_splitk_part(const std::vector<LayerWs>& lw) {
  size_t room[4];
  splitk_regions(lw, room);
  const size_t m = room[0] + room[1] + room[2] + room[3] + 1024;
  return m < kSplitkPartDoubles ? m : kSplitkPartDoubles + ((size_t)32 * 1024 * 1024 / 8);
}

int check_chain(dgp_ctx* c, const dgp_model_desc* model, long N, long S) {
  const int nl = model->num_layers;
  if (nl < 1 || N < 1 || S < 1) { c->err = "need num_layers >= 1, N >= 1, S >= 1"; return DGP_ERR_ARG; }
  for (int l = 1; l < nl; ++l)
    if (model->layers[l].D_in != model->layers[l - 1].D_out) { c->err = "layer widths do not chain"; return DGP_ERR_ARG; }
  return DGP_OK;
}

// Runs the chain over all chunks. Returns via opts outputs. `plan` semantics are handled by c->dry.
int run_model(dgp_ctx* c, const dgp_model_desc* model, const double* X, long N, long S, unsigned long long seed, long n_offset,
              RunOpts& o) {
  RC(check_chain(c, model, N, S));
  const int nl = model->num_layers;
  const bool grad = o.want_grad;
  const bool adj = grad || o.dx;   // the adjoint chain runs (needs the A / T_d stash and Ku^-1)
  // first-layer sharing (see expand_first_layer_kernel): needs a later layer to consume the per-sample draws
  const bool share0 = c->share_first_layer && S > 1 && nl >= 2;
  if ((grad || o.want_elbo) && model->layers[nl - 1].D_out != o.Dy) { c->err = "Y width must equal the last layer's D_out"; return DGP_ERR_ARG; }
  if ((grad || o.want_elbo) && !model->lik_variance) { c->err = "lik_variance is null"; return DGP_ERR_ARG; }

  std::vector<LayerWs> lw;
  LateGuard late_guard{c};
  const PrepLevel level = adj ? PREP_GRAD : (o.want_elbo ? PREP_KL : PREP_FWD);
  RC(prep_layers(c, model, lw, level, ctx_path(c, level, N * S), true));
  for (const LayerWs& w : lw)   // refused in the planning pass, before any launch (the chunk loop below does not run there)
    if (!moments_fit(c, w)) return DGP_ERR_UNSUPPORTED;
  const size_t base_used = c->used;

  int maxMp = 0, maxD = 1;
  size_t pp_doubles = 0;   // workspace doubles per padded point-sample
  for (int l = 0; l < nl; ++l) {
    const LayerWs& w = lw[l];
    if (w.Mp > maxMp) maxMp = w.Mp;
    if (w.D_out > maxD) maxD = w.D_out;
    pp_doubles += 4 * (size_t)w.D_out;                              // F, Fmean, Fvar, z
    if (adj) pp_doubles += (size_t)(1 + w.D_out) * w.Mp;             // A, T stash
  }
  pp_doubles += 3 * (size_t)maxMp;                                   // temps
  if (!adj) pp_doubles += (size_t)maxD * maxMp;                      // shared T
  if (adj) pp_doubles += 2 * (size_t)maxD + 32 + 1 + 32 + 2 * 32;    // Gm, GvT, GmPad, gq, XaugPad, dX ping-pong
  if (adj && nl > 1) pp_doubles += 3 * (size_t)maxMp + 2 * (size_t)maxD + 32 + 1 + 32;   // second set of adjoint temporaries
  size_t fixed = base_used + (adj ? max_splitk_part(lw) * sizeof(double) : 0) + ((size_t)8 << 20);
  long Nc_max;
  {
    size_t avail = c->ws_limit > fixed ? c->ws_limit - fixed : 0;
    long pmax = (long)(avail / (pp_doubles * sizeof(double)));
    pmax = pmax / kTileP * kTileP - kTileP;
    Nc_max = pmax / S;
    if (Nc_max < 1) Nc_max = 1;
    if (Nc_max > N) Nc_max = N;
    // equalise the chunks
    long nchunks = (N + Nc_max - 1) / Nc_max;
    Nc_max = (N + nchunks - 1) / nchunks;
  }
  const long Ppmax = round_up(Nc_max * S, kTileP);

  // chunk-sized buffers (allocated once, reused by every chunk)
  std::vector<ChunkLayer> cls(nl);
  for (int l = 0; l < nl; ++l) {
    const LayerWs& w = lw[l];
    cls[l].F = walloc(c, (size_t)Ppmax * w.D_out);
    cls[l].Fmean = walloc(c, (size_t)Ppmax * w.D_out);
    cls[l].Fvar = walloc(c, (size_t)Ppmax * w.D_out);
    cls[l].z = walloc(c, (size_t)Ppmax * w.D_out);
    if (adj) {
      cls[l].A = walloc(c, (size_t)w.Mp * Ppmax);
      cls[l].T = walloc(c, (size_t)w.D_out * w.Mp * Ppmax);
    }
  }
  Temps tmp;
  tmp.t0 = walloc(c, (size_t)maxMp * Ppmax);
  tmp.t1 = walloc(c, (size_t)maxMp * Ppmax);
  tmp.t2 = walloc(c, (size_t)maxMp * Ppmax);
  double* Tshared = adj ? nullptr : walloc(c, (size_t)maxD * maxMp * Ppmax);
  Upstream up{nullptr, nullptr, nullptr, nullptr, nullptr, 0}, up1{nullptr, nullptr, nullptr, nullptr, nullptr, 0};
  Temps tmp1;
  double* XaugPad1 = nullptr;
  double *XaugPad = nullptr, *dXa = nullptr, *dXb = nullptr, *rbf_part = nullptr, *skpart = nullptr, *lik_part = nullptr;
  size_t skcap = 0;
  double* acc = nullptr;   // [0] data term, [1] d/d lik variance (accumulated over chunks)
  const long nbmax = Ppmax / 128;
  if (adj || o.want_elbo) {
    lik_part = walloc(c, (size_t)nbmax * 3);
    acc = walloc(c, 4);
  }
  if (adj) {
    up.Gm = walloc(c, (size_t)Ppmax * maxD);
    up.GvT = walloc(c, (size_t)Ppmax * maxD);
    up.GmPad = walloc(c, (size_t)Ppmax * 32);
    up.gq = walloc(c, (size_t)Ppmax);
    XaugPad = walloc(c, (size_t)Ppmax * 32);
    dXa = walloc(c, (size_t)Ppmax * 32);
    dXb = walloc(c, (size_t)Ppmax * 32);
    rbf_part = walloc(c, (size_t)nbmax * 8 * 20);   // one row of partials per 64-column block of rbf_bwd_kernel
    skcap = max_splitk_part(lw);
    skpart = walloc(c, skcap);
    if (nl > 1) {   // second set: layer l's parameter contractions read theirs while layer l-1's data path fills the other
      tmp1.t0 = walloc(c, (size_t)maxMp * Ppmax);
      tmp1.t1 = walloc(c, (size_t)maxMp * Ppmax);
      tmp1.t2 = walloc(c, (size_t)maxMp * Ppmax);
      up1.Gm = walloc(c, (size_t)Ppmax * maxD);
      up1.GvT = walloc(c, (size_t)Ppmax * maxD);
      up1.GmPad = walloc(c, (size_t)Ppmax * 32);
      up1.gq = walloc(c, (size_t)Ppmax);
      XaugPad1 = walloc(c, (size_t)Ppmax * 32);
    }
  }
  double* acq_direct = (o.dx && o.acq_kind == 3) ? walloc(c, (size_t)Nc_max * 32) : nullptr;
  ParamScratch ps;
  ps.part = skpart; ps.cap = skcap;
  if (adj) {
    splitk_regions(lw, ps.room);
    ps.off[0] = 0; ps.off[1] = ps.room[0]; ps.off[2] = ps.off[1] + ps.room[1]; ps.off[3] = ps.off[2] + ps.room[2];
    ps.fixed = ps.off[3] + ps.room[3] <= skcap;
  }
  if (c->dry) return DGP_OK;

  const int DL = model->layers[nl - 1].D_out;
  long n0 = 0;
  bool first = true;
  while (n0 < N) {
    const long Nc = (N - n0 < Nc_max) ? (N - n0) : Nc_max;
    const long P = Nc * S, Pp = round_up(P, kTileP);
    // ---- forward chain (models/dgp.py:49-61) ----
    for (int l = 0; l < nl; ++l) {
      const dgp_layer_desc& d = model->layers[l];
      ChunkLayer& cl = cls[l];
      if (l == 0) { cl.Xin = X + n0 * d.D_in; cl.xmod = Nc; }
      else { cl.Xin = cls[l - 1].F; cl.xmod = P; }
      const bool last = l == nl - 1;
      const bool need_sample = !last || o.need_last_sample || (o.io.Fs && o.io.Fs[l]);
      if (l == 0 && share0) {
        // the first layer sees the same X row for every sample: one conditional per point, expanded to the S samples
        RC(forward_layer(c, d, lw[0], cl, tmp, adj, Tshared, 0, Nc, 1, Nc, 0, seed, n_offset, ChunkIO(), false));
        CAT(DGP_CAT_MOMENTS);
        ExpandArgs e;
        memset(&e, 0, sizeof(e));
        e.mean0 = cl.Fmean; e.var0 = cl.Fvar; e.z_in = (o.io.zs && o.io.zs[0]) ? o.io.zs[0] : nullptr;
        e.seed = seed; e.seed_ptr = c->seed_ptr; e.layer = 0; e.Nc = Nc; e.N_total = N; e.n0 = n0; e.n_offset = n_offset; e.S = S; e.D = d.D_out;
        e.jitter = d.jitter; e.F = cl.F; e.z = cl.z;
        e.xFmean = (o.io.Fmeans && o.io.Fmeans[0]) ? o.io.Fmeans[0] : nullptr;
        e.xFvar = (o.io.Fvars && o.io.Fvars[0]) ? o.io.Fvars[0] : nullptr;
        e.xF = (o.io.Fs && o.io.Fs[0]) ? o.io.Fs[0] : nullptr;
        LAUNCH(expand_first_layer_kernel, (unsigned)((P * d.D_out + 255) / 256), 256, 0, e);
        continue;
      }
      RC(forward_layer(c, d, lw[l], cl, tmp, adj, Tshared, l, Nc, S, N, n0, seed, n_offset, o.io, need_sample));
    }
    const ChunkLayer& clL = cls[nl - 1];
    // adjoint chain over the layers, last to first; params = false stops at the input gradient (o.dx)
    auto run_backward = [&](bool params) -> int {
      join_late(c);   // Kuu^-1 and the other products deferred by prep_layers
      const long nb = Pp / 128;
      const int D0 = model->layers[0].D_in;
      double* dX_next = dXa;
      for (int l = nl - 1; l >= 0; --l) {
        const dgp_layer_desc& d = model->layers[l];
        CAT(DGP_CAT_OTHER);
        // the two sets of adjoint temporaries alternate: this layer's data path may start while the previous layer's parameter
        // contractions still read the other set; the contractions that read THIS set two layers ago must be done
        const int set = (nl > 1 && tmp1.t0) ? ((nl - 1 - l) & 1) : 0;
        const Temps& tm = set ? tmp1 : tmp;
        Upstream& us = set ? up1 : up;
        double* Xaug = set ? XaugPad1 : XaugPad;
        join_param(c, set);
        ParamScratch psl = ps;
        psl.defer_set = (params && l > 0 && tmp1.t0) ? set : -1;   // the first layer is the last one processed: nothing to overlap with
        if (l == 0 && share0) {
          // first-layer sharing: per-point upstream gradients = sums over the S samples, then a P = Nc adjoint
          const long Pp0 = round_up(Nc, kTileP), nb0 = Pp0 / 128;
          UpstreamOut uh{us.Gm, us.GvT, us.GmPad, us.gq, lik_part};
          LAUNCH(upstream_reduce_kernel, (unsigned)nb0, 128, 0, dX_next, cls[0].z, cls[0].Fvar, Nc, S, Pp0, d.D_out, d.jitter, uh);
          Upstream up0 = us;
          up0.part = lik_part; up0.nblocks = nb0;
          RC(backward_layer(c, d, lw[0], cls[0], tm, up0, o.dx ? o.dx + n0 * D0 : nullptr, Xaug, rbf_part, psl, Nc, 1, first, params));
          continue;
        }
        if (l < nl - 1) {
          // Gm = G_F, Gv = G_F z / (2 sqrt(var + jitter))                          (adjoint of utils/utils.py:40-41)
          UpstreamOut uh{us.Gm, us.GvT, us.GmPad, us.gq, lik_part};
          LAUNCH(upstream_kernel, (unsigned)nb, 128, 0, dX_next, cls[l].z, cls[l].Fvar, P, Pp, d.D_out, d.jitter, uh);
        }
        us.part = lik_part; us.nblocks = nb;
        double* dXin = (l > 0 || o.dx) ? (dX_next == dXa ? dXb : dXa) : nullptr;
        if (l == 0 && o.dx && S == 1) dXin = o.dx + n0 * D0;   // one sample: the per-point-sample gradient is the answer
        RC(backward_layer(c, d, lw[l], cls[l], tm, us, dXin, Xaug, rbf_part, psl, Nc, S, first, params));
        if (l == 0 && o.dx && S > 1) {
          CAT(DGP_CAT_OTHER);
          LAUNCH(sum_samples_kernel, (unsigned)((Nc * D0 + 255) / 256), 256, 0, dXin, Nc, S, D0, o.dx + n0 * D0);
        }
        if (dXin) dX_next = dXin;
      }
      join_param(c, 0); join_param(c, 1);   // the next chunk's forward chain reuses the temporaries
      return DGP_OK;
    };
    CAT(DGP_CAT_OTHER);
    // ---- prediction epilogues ----
    if (o.pm) {
      const long ND = Nc * DL;
      LAUNCH(mixture_moments_kernel, (unsigned)((ND + 255) / 256), 256, 0, clL.Fmean, clL.Fvar, S, ND, model->lik_variance,
             o.add_lik, o.pm + n0 * DL, o.pv + n0 * DL);
    }
    if (o.ve) {
      const long ND = Nc * DL;
      LAUNCH(ve_mean_kernel, (unsigned)((ND + 255) / 256), 256, 0, clL.Fmean, clL.Fvar, o.Y + n0 * DL, model->lik_variance, Nc, S, DL,
             o.ve + n0 * DL);
    }
    if (o.ei && !o.dx) {
      const long ND = Nc * DL;
      if (o.ei_analytic) {
        double* m = tmp.t0;
        double* v = tmp.t0 + ND;
        LAUNCH(mixture_moments_kernel, (unsigned)((ND + 255) / 256), 256, 0, clL.Fmean, clL.Fvar, S, ND, model->lik_variance, 0, m, v);
        LAUNCH(ei_analytic_kernel, (unsigned)((ND + 255) / 256), 256, 0, m, v, ND, o.y_min, o.ei + n0 * DL);
      } else {
        LAUNCH(ei_mc_kernel, (unsigned)((ND + 255) / 256), 256, 0, clL.F, S, ND, o.y_min, o.ei + n0 * DL);
      }
    }
    // ---- likelihood + adjoint chain ----
    if (grad || o.want_elbo) {
      UpstreamOut uo{up.Gm, up.GvT, up.GmPad, up.gq, lik_part};
      const long nb = Pp / 128;
      LAUNCH(likelihood_kernel, (unsigned)nb, 128, 0, clL.Fmean, clL.Fvar, o.Y + n0 * o.Dy, model->lik_variance, Nc, P, Pp, DL,
             o.scale / (double)S, grad ? 1 : 0, uo);
      LAUNCH(reduce_partials_kernel, 2, 256, 0, lik_part, nb, 3, acc, first ? 0 : 1);
      if (grad) {
        up.part = lik_part; up.nblocks = nb;
        RC(run_backward(true));
      }
    }
    if (o.dx) {
      // ---- d sum(-EI) / dX: EI upstream adjoints, then the data path of the adjoint chain (no parameter contractions) ----
      const long nb = Pp / 128;
      CK(cudaMemsetAsync(up.Gm, 0, (size_t)Pp * DL * sizeof(double), c->stream));
      CK(cudaMemsetAsync(up.GvT, 0, (size_t)Pp * DL * sizeof(double), c->stream));
      CK(cudaMemsetAsync(up.GmPad, 0, (size_t)Pp * 32 * sizeof(double), c->stream));
      CK(cudaMemsetAsync(up.gq, 0, (size_t)Pp * sizeof(double), c->stream));
      const int D0x = model->layers[0].D_in;
      const long vstride = o.acq_kind == 3 ? D0x : (o.acq_kind == 4 ? 2 * DL : DL);   // WB2S: one value per input column; 4: (dm, dv) pairs
      LAUNCH(ei_upstream_kernel, (unsigned)((Nc + 127) / 128), 128, 0, clL.Fmean, clL.Fvar, Nc, S, Pp, DL, o.y_min, o.ei + n0 * vstride,
             up.Gm, up.GvT, up.GmPad, up.gq, o.acq_kind, o.acq_add_lik ? model->lik_variance : nullptr, X + n0 * D0x, D0x, acq_direct);
      up.part = lik_part; up.nblocks = nb;
      RC(run_backward(false));
      if (o.acq_kind == 3) {
        CAT(DGP_CAT_OTHER);
        LAUNCH(add_inplace_kernel, (unsigned)((Nc * D0x + 255) / 256), 256, 0, o.dx + n0 * D0x, acq_direct, Nc * D0x);
      }
    }
    n0 += Nc;
    first = false;
  }

  // ---- replicated epilogue: KL, its adjoint, RBF adjoint on Kuu, gradient assembly ----
  join_late(c);
  CAT(DGP_CAT_PREP);
  if (grad || o.want_elbo) {
    double* out = o.out_flat;
    std::vector<dgp_layer_grad_offsets> offs(nl);
    dgp_grad_layout(model, offs.data());
    // out[0] = data term, out[2] = d/d lik variance, out[1] = kl_weight * sum KL
    CK(cudaMemcpyAsync(out, acc, sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
    CK(cudaMemcpyAsync(out + 2, acc + 1, sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
    std::vector<const double*> klp(nl);
    for (int l = 0; l < nl; ++l) klp[l] = lw[l].kl;
    double* klsum = acc + 2;
    CK(cudaMemsetAsync(klsum, 0, sizeof(double), c->stream));
    for (int l = 0; l < nl; ++l) LAUNCH(reduce_partials_kernel, 1, 256, 0, lw[l].kl, 1, 1, klsum, 1);
    LAUNCH(scale_copy_kernel, 1, 32, 0, klsum, o.kl_weight, out + 1);
    if (grad) {
      LayerFork forkE(c, nl);
      for (int l = 0; l < nl; ++l) {
        forkE.use(l);
        const dgp_layer_desc& d = model->layers[l];
        LayerWs& w = lw[l];
        const long mm = (long)w.Mp * w.Mp;
        if (w.vform) {
          // V-form accumulators (G1, DCt, dbeta) -> gradients w.r.t. q_mu, q_sqrt and Ku = Lu Lu^T
          const int Mp = w.Mp, D = w.D_out;
          const long nct = (long)D * mm;
          // W_d = V diag(2 Gv_d) V^T (lower triangles accumulated over the chunks) -> DCt_d = tril(W_d C_d^T),
          // G1 = tril(sum_d C_d^T (W_d C_d^T)^T + beta dbeta^T - sum_d W_d)                       (see backward_layer)
          GemmArgs g;
          LAUNCH(sym_fill_kernel, (unsigned)((nct + 255) / 256), 256, 0, w.Wacc, Mp, (long)D * Mp, D);
          g = gargs(w.Wacc, (long)D * Mp, w.CTcat, (long)D * Mp, w.DCt, (long)D * Mp, Mp, Mp, Mp);
          g.batch = D; g.sA = Mp; g.sB = Mp; g.sC = Mp;
          RC(gemm(c, g, false));
          g = gargs(w.CTcat, (long)D * Mp, w.DCt, (long)D * Mp, w.G1, Mp, Mp, Mp, D * Mp);
          split_long_k(g, D, w.part_small);
          RC(gemm(c, g, true));
          g = gargs(w.betaP, 32, w.dbeta, 32, w.G1, Mp, Mp, Mp, 32);
          g.beta = 1.0;
          RC(gemm(c, g, true));
          LAUNCH(g1_finish_kernel, (unsigned)((mm + 255) / 256), 256, 0, w.G1, w.Wacc, Mp, D);
          LAUNCH(tril_scale_kernel, (unsigned)((nct + 255) / 256), 256, 0, w.DCt, Mp, (long)D * Mp, D, 1.0);
          if (!w.white) {
            g = gargs(w.LinvT, Mp, w.dbeta, 32, w.dqmu2, 32, Mp, 32, Mp);              // dq_mu = Lu^-T dbeta
            g.a_tri = 2;
            RC(gemm(c, g, false));
            g = gargs(w.LinvT, Mp, w.DCt, (long)D * Mp, w.dRcat, (long)D * Mp, Mp, D * Mp, Mp);   // dq_sqrt_d = tril(Lu^-T dC_d^T)
            g.a_tri = 2;
            RC(gemm(c, g, false));
          }
          // dLu^-1 = tril(G1 Lu^T + sum_d dC_d^T q_sqrt_d^T + dbeta q_mu^T); whitened: C_d and beta do not involve Lu, G1 term only
          g = gargs(w.G1, Mp, w.L, Mp, w.dLinv, Mp, Mp, Mp, Mp);
          RC(gemm(c, g, true));
          if (!w.white) {
            g = gargs(w.DCt, (long)D * Mp, w.RpT, Mp, w.dLinv, Mp, Mp, Mp, D * Mp);
            g.beta = 1.0;
            split_long_k(g, D, w.part_small);
            RC(gemm(c, g, false));
            g = gargs(w.dbeta, 32, w.qmuP, 32, w.dLinv, Mp, Mp, Mp, 32);
            g.beta = 1.0;
            RC(gemm(c, g, true));
          }
          LAUNCH(tril_scale_kernel, (unsigned)((mm + 255) / 256), 256, 0, w.dLinv, Mp, (long)Mp, 1, 1.0);
          // Lu^-1 = X is a function of Ku = Lu Lu^T: dX = -Phi(X dKu X^T) X, hence (Phi is self-adjoint)
          //   dKu = -X^T sym(Phi(Xbar X^T)) X,  Xbar = dLu^-1,  Phi = lower triangle with halved diagonal
          g = gargs(w.dLinv, Mp, w.Linv, Mp, w.sq1, Mp, Mp, Mp, Mp);          // Q = Xbar X^T
          RC(gemm(c, g, true));
          LAUNCH(phi_sym_kernel, (unsigned)((mm + 255) / 256), 256, 0, w.sq1, Mp, w.sq2);
          g = gargs(w.LinvT, Mp, w.sq2, Mp, w.sq1, Mp, Mp, Mp, Mp);
          g.a_tri = 2;
          RC(gemm(c, g, false));
          g = gargs(w.sq1, Mp, w.Linv, Mp, w.dKu, Mp, Mp, Mp, Mp);
          g.alpha = -1.0;
          RC(gemm(c, g, false));
        }
        LAUNCH(dku_assemble_kernel, (unsigned)((mm + 255) / 256), 256, 0, w.dKu, w.Kinv, w.KSK, w.alpha, w.Knj, w.M, w.Mp, w.D_out,
               w.white ? 0.0 : o.kl_weight, 1);
        LAUNCH(kuu_bwd_kernel, w.M, 128, 0, w.dKu, d.Z, d.lengthscales, d.variance, w.M, w.Mp, w.D_in, w.dZk, w.kuu_part, d.kernel_kind);
        LAUNCH(reduce_partials_kernel, w.D_in + 1, 256, 0, w.kuu_part, (long)w.M, w.D_in + 1, w.kuu_red, 0);
        FinalizeArgs f;
        memset(&f, 0, sizeof(f));
        f.Gd = w.white ? w.DCt : (w.vform ? w.dRcat : w.dR); f.gd_cat = w.vform ? 1 : 0; f.KR = w.KRcat; f.Rcat = w.Rcat;
        f.dqmu = w.white ? w.dbeta : (w.vform ? w.dqmu2 : w.dqmu); f.alpha = w.alpha; f.H = w.H; f.dZk = w.dZk;
        f.white = w.white ? 1 : 0; f.qmuP = w.qmuP;
        f.rbf_red = w.rbf_red; f.kuu_red = w.kuu_red; f.sgv = w.sgv; f.Z = d.Z; f.ls = d.lengthscales;
        f.M = w.M; f.Mp = w.Mp; f.D_in = w.D_in; f.D_out = w.D_out; f.klw = o.kl_weight;
        f.dZ = out + offs[l].dZ; f.dls = out + offs[l].dlengthscales; f.dvar = out + offs[l].dvariance;
        f.dq_mu = out + offs[l].dq_mu; f.dq_sqrt = out + offs[l].dq_sqrt;
        const long nq = (long)w.D_out * w.M * w.M;
        LAUNCH(finalize_layer_kernel, (unsigned)((nq + 255) / 256), 256, 0, f);
      }
    }
  }
  return DGP_OK;
}

void drop_graphs(dgp_ctx* c) {
  for (auto& g : c->graphs) {
    if (g.exec) cudaGraphExecDestroy(g.exec);
    for (void* h : g.pinned) cudaFreeHost(h);
  }
  c->graphs.clear();
}

__global__ void set_seed_kernel(unsigned long long* slot, unsigned long long seed) { *slot = seed; }

template <typename T>
void key_put(std::vector<unsigned char>& k, const T& v) {
  const unsigned char* p = reinterpret_cast<const unsigned char*>(&v);
  k.insert(k.end(), p, p + sizeof(T));
}

// Everything the launch sequence of a step depends on, except the seed (read from c->d_seed by a replayed step).
std::vector<unsigned char> graph_key(dgp_ctx* c, const dgp_model_desc* model, const double* X, long N, long S, long n_offset,
                                     const RunOpts& o) {
  std::vector<unsigned char> k;
  k.reserve(512);
  key_put(k, model->num_layers); key_put(k, model->lik_variance);
  for (int l = 0; l < model->num_layers; ++l) {
    const dgp_layer_desc& d = model->layers[l];
    key_put(k, d.D_in); key_put(k, d.D_out); key_put(k, d.M); key_put(k, d.white); key_put(k, d.mean_kind); key_put(k, d.kernel_kind);
    key_put(k, d.Z); key_put(k, d.lengthscales); key_put(k, d.variance); key_put(k, d.q_mu); key_put(k, d.q_sqrt);
    key_put(k, d.mf_W); key_put(k, d.mf_b); key_put(k, d.jitter);
  }
  key_put(k, X); key_put(k, N); key_put(k, S); key_put(k, n_offset);
  key_put(k, o.want_grad); key_put(k, o.want_elbo); key_put(k, o.Y); key_put(k, o.Dy); key_put(k, o.scale); key_put(k, o.kl_weight);
  key_put(k, o.out_flat); key_put(k, o.ve); key_put(k, o.pm); key_put(k, o.pv); key_put(k, o.add_lik); key_put(k, o.ei); key_put(k, o.y_min);
  key_put(k, o.ei_analytic); key_put(k, o.need_last_sample); key_put(k, o.dx); key_put(k, o.acq_kind); key_put(k, o.acq_add_lik);
  key_put(k, c->use_fused); key_put(k, c->use_vform_grad); key_put(k, c->vform_forward_calls);
  key_put(k, c->vform_grad_min_ps); key_put(k, c->share_first_layer); key_put(k, c->parallel_layers); key_put(k, c->ws_limit);
  return k;
}

constexpr size_t kMaxGraphs = 16;

// Replay path of run_model_planned: capture the step once per call signature, then one seed store + one graph launch per call.
int run_model_graphed(dgp_ctx* c, const dgp_model_desc* model, const double* X, long N, long S, unsigned long long seed,
                      long n_offset, RunOpts& o) {
  std::vector<unsigned char> key = graph_key(c, model, X, N, S, n_offset, o);
  dgp_ctx::GraphEntry* hit = nullptr;
  for (auto& g : c->graphs)
    if (g.key == key) { hit = &g; break; }
  if (!hit) {
    // growing the arena may drop every cached graph (their nodes point into the old arena)
    RC(plan(c, [&] { return run_model(c, model, X, N, S, seed, n_offset, o); }));
    if (!c->cap_stream) CK(cudaStreamCreateWithFlags(&c->cap_stream, cudaStreamNonBlocking));
    if (!c->d_seed) CK(cudaMalloc(&c->d_seed, sizeof(unsigned long long)));
    if (c->graphs.size() >= kMaxGraphs) {   // evict the least recently used entry
      size_t lru = 0;
      for (size_t i = 1; i < c->graphs.size(); ++i)
        if (c->graphs[i].last_use < c->graphs[lru].last_use) lru = i;
      CK(cudaStreamSynchronize(c->stream));
      if (c->graphs[lru].exec) cudaGraphExecDestroy(c->graphs[lru].exec);
      for (void* h : c->graphs[lru].pinned) cudaFreeHost(h);
      c->graphs.erase(c->graphs.begin() + (long)lru);
    }
    dgp_ctx::GraphEntry e;
    e.key = std::move(key);
    cudaStream_t user = c->stream;
    const long launches0 = c->launches;
    CK(cudaStreamBeginCapture(c->cap_stream, cudaStreamCaptureModeRelaxed));
    c->stream = c->cap_stream; c->seed_ptr = c->d_seed; c->keep = &e.pinned;
    int rc = run_model(c, model, X, N, S, seed, n_offset, o);
    c->stream = user; c->seed_ptr = nullptr; c->keep = nullptr;
    cudaGraph_t graph = nullptr;
    cudaError_t ce = cudaStreamEndCapture(c->cap_stream, &graph);
    e.launches = c->launches - launches0;
    c->launches = launches0;
    if (rc == DGP_OK && ce != cudaSuccess) { c->err = std::string("cudaStreamEndCapture: ") + cudaGetErrorString(ce); rc = DGP_ERR_CUDA; }
    if (rc == DGP_OK) {
      ce = cudaGraphInstantiate(&e.exec, graph, 0);
      if (ce != cudaSuccess) { c->err = std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ce); rc = DGP_ERR_CUDA; }
    }
    if (graph) cudaGraphDestroy(graph);
    if (rc != DGP_OK) {
      cudaGetLastError();
      for (void* h : e.pinned) cudaFreeHost(h);
      return rc;
    }
    c->graphs.push_back(std::move(e));
    hit = &c->graphs.back();
  }
  hit->last_use = ++c->graph_tick;
  set_seed_kernel<<<1, 1, 0, c->stream>>>(c->d_seed, seed);
  CK(cudaGetLastError());
  CK(cudaGraphLaunch(hit->exec, c->stream));
  c->launches += hit->launches + 1;
  return DGP_OK;
}

// plan (dry) pass to size the arena, then the real pass
int run_model_planned(dgp_ctx* c, const dgp_model_desc* model, const double* X, long N, long S, unsigned long long seed,
                      long n_offset, RunOpts& o) {
  CK(cudaSetDevice(c->device));
  if (c->use_graph && !c->profiling && !o.io.zs && !o.io.Fs && !o.io.Fmeans && !o.io.Fvars)
    return run_model_graphed(c, model, X, N, S, seed, n_offset, o);
  return planned(c, [&] { return run_model(c, model, X, N, S, seed, n_offset, o); });
}

int check_chol(dgp_ctx* c, const char* what = nullptr) {
  int info = 0;
  CK(cudaMemcpyAsync(&info, c->d_info, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (info) {
    CK(cudaMemsetAsync(c->d_info, 0, sizeof(int), c->stream));   // reported once; later steps start clean
    c->err = what ? what : "Kuu + jitter I is not positive definite (Cholesky pivot <= 0); parameter updates were suspended from that step on";
    return DGP_ERR_NUMERIC;
  }
  return DGP_OK;
}

}  // namespace

// =========================================================================================================
// C ABI
// =========================================================================================================
extern "C" {

int dgp_version(void) { return 100; }

// ---- multi-GPU inside the C ABI (SURVEY §8b/e): points are sharded over ranks by the caller (n_offset = first global point of
// the shard, kl_weight = 1 / world); the one exchange step of the path is a sum-allreduce of the flat buffer over NVLink ----
namespace {
struct NcclUid { char internal[128]; };
struct NcclApi {
  int (*GetUniqueId)(NcclUid*) = nullptr;
  int (*CommInitRank)(void**, int, NcclUid, int) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
  bool ok = false;
  std::string why;
};
NcclApi& nccl_api() {
  static NcclApi api;
  static bool tried = false;
  if (tried) return api;
  tried = true;
  const char* names[] = {getenv("DGP_B200_NCCL"), "libnccl.so.2", "libnccl.so"};
  void* h = nullptr;
  for (const char* n : names) {
    if (!n) continue;
    h = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (h) break;
  }
  if (!h) { api.why = "libnccl.so.2 not found (set DGP_B200_NCCL to its path)"; return api; }
  api.GetUniqueId = reinterpret_cast<int (*)(NcclUid*)>(dlsym(h, "ncclGetUniqueId"));
  api.CommInitRank = reinterpret_cast<int (*)(void**, int, NcclUid, int)>(dlsym(h, "ncclCommInitRank"));
  api.AllReduce = reinterpret_cast<int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t)>(dlsym(h, "ncclAllReduce"));
  api.CommDestroy = reinterpret_cast<int (*)(void*)>(dlsym(h, "ncclCommDestroy"));
  api.GetErrorString = reinterpret_cast<const char* (*)(int)>(dlsym(h, "ncclGetErrorString"));
  api.ok = api.GetUniqueId && api.CommInitRank && api.AllReduce && api.CommDestroy && api.GetErrorString;
  if (!api.ok) api.why = "libnccl is missing a required symbol";
  return api;
}
constexpr int kNcclDouble = 8, kNcclSum = 0;
void nccl_comm_free(dgp_ctx* c) {
  if (c->nccl_comm) { nccl_api().CommDestroy(c->nccl_comm); c->nccl_comm = nullptr; c->comm_world = 1; c->comm_rank = 0; }
}
}  // namespace

int dgp_comm_unique_id(void* uid_out_128_bytes) {
  if (!uid_out_128_bytes) return DGP_ERR_ARG;
  NcclApi& n = nccl_api();
  if (!n.ok) return DGP_ERR_UNSUPPORTED;
  return n.GetUniqueId(reinterpret_cast<NcclUid*>(uid_out_128_bytes)) == 0 ? DGP_OK : DGP_ERR_CUDA;
}

int dgp_comm_init(dgp_ctx* c, int rank, int world, const void* nccl_uid_128_bytes) {
  if (!c || !nccl_uid_128_bytes || world < 1 || rank < 0 || rank >= world) return DGP_ERR_ARG;
  NcclApi& n = nccl_api();
  if (!n.ok) { c->err = n.why; return DGP_ERR_UNSUPPORTED; }
  CK(cudaSetDevice(c->device));
  if (c->nccl_comm) { n.CommDestroy(c->nccl_comm); c->nccl_comm = nullptr; }
  NcclUid uid;
  memcpy(&uid, nccl_uid_128_bytes, sizeof(uid));
  const int rc = n.CommInitRank(&c->nccl_comm, world, uid, rank);
  if (rc != 0) { c->err = std::string("ncclCommInitRank: ") + n.GetErrorString(rc); c->nccl_comm = nullptr; return DGP_ERR_CUDA; }
  c->comm_rank = rank; c->comm_world = world;
  return DGP_OK;
}

int dgp_allreduce_grads(dgp_ctx* c, double* elbo_and_grads, int64_t n_doubles) {
  if (!c || !elbo_and_grads || n_doubles < 1) return DGP_ERR_ARG;
  if (!c->nccl_comm) { c->err = "dgp_comm_init has not been called"; return DGP_ERR_ARG; }
  NcclApi& n = nccl_api();
  const int rc = n.AllReduce(elbo_and_grads, elbo_and_grads, (size_t)n_doubles, kNcclDouble, kNcclSum, c->nccl_comm, c->stream);
  if (rc != 0) { c->err = std::string("ncclAllReduce: ") + n.GetErrorString(rc); return DGP_ERR_CUDA; }
  return DGP_OK;
}

int dgp_comm_destroy(dgp_ctx* c) {
  if (!c) return DGP_ERR_ARG;
  nccl_comm_free(c);
  return DGP_OK;
}

// The data-parallel step in ONE call: this rank's shard of the minibatch (points [n_offset, n_offset + N) of the global batch),
// KL weighted 1 / world, then the sum-allreduce of the flat buffer on the ctx's stream.
int dgp_elbo_grad_sharded(dgp_ctx* c, const dgp_model_desc* model, const double* X, const double* Y, int64_t N, int64_t S, double scale,
                          uint64_t seed, int64_t n_offset, int want_grad, double* out_flat) {
  if (!c || !model) return DGP_ERR_ARG;
  const int world = c->nccl_comm ? c->comm_world : 1;
  RC(dgp_elbo_grad(c, model, X, Y, N, S, scale, 1.0 / world, nullptr, seed, n_offset, want_grad, out_flat));
  if (world > 1) RC(dgp_allreduce_grads(c, out_flat, want_grad ? dgp_grad_size(model) : 3));
  return DGP_OK;
}


int dgp_ctx_create(int device, void* cuda_stream, dgp_ctx** out) {
  if (!out) return DGP_ERR_ARG;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return DGP_ERR_CUDA;
  if (cudaSetDevice(device) != cudaSuccess) return DGP_ERR_CUDA;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return DGP_ERR_CUDA;
  if (prop.major != 10) return DGP_ERR_UNSUPPORTED;   // sm_100a only: no fallback path exists
  dgp_ctx* c = new dgp_ctx();
  c->device = device;
  c->num_sms = prop.multiProcessorCount;
  if (getenv("DGP_B200_UNFUSED")) c->use_fused = false;
  if (const char* e = getenv("DGP_B200_SYNC_LAUNCHES")) c->sync_launches = atoi(e) != 0;   // debugging: synchronise and check after every launch
  if (const char* e = getenv("DGP_B200_WARPMAP")) c->warp_major_groups = atoi(e) != 0;   // measurement hooks
  if (const char* e = getenv("DGP_B200_FUSED_BWD")) c->use_fused_bwd = atoi(e) != 0;
  if (const char* e = getenv("DGP_B200_SKEW")) c->group_skew = atoi(e);
  c->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
  if (cudaMalloc(&c->d_info, sizeof(int)) != cudaSuccess || cudaMemset(c->d_info, 0, sizeof(int)) != cudaSuccess) { delete c; return DGP_ERR_CUDA; }
  const char* lim = getenv("DGP_B200_WS_GB");
  if (lim && atof(lim) > 0.0) c->ws_limit = (size_t)(atof(lim) * (double)((size_t)1 << 30));
  *out = c;
  return DGP_OK;
}

void dgp_ctx_destroy(dgp_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  drop_graphs(c);
  nccl_comm_free(c);
  if (c->cap_stream) cudaStreamDestroy(c->cap_stream);
  if (c->d_seed) cudaFree(c->d_seed);
  if (c->ws) cudaFree(c->ws);
  if (c->d_info) cudaFree(c->d_info);
  if (c->h_pinned) cudaFreeHost(c->h_pinned);
  if (c->d_stage) cudaFree(c->d_stage);
  for (auto& s : c->spans) { cudaEventDestroy(s.a); cudaEventDestroy(s.b); }
  for (auto e : c->ev_pool) cudaEventDestroy(e);
  if (c->ev_fork) {
    cudaEventDestroy(c->ev_fork);
    for (int k = 0; k < 2; ++k) for (int i = 0; i < 4; ++i) if (c->ev_param[k][i]) cudaEventDestroy(c->ev_param[k][i]);
    for (int i = 0; i < dgp_ctx::kAux; ++i) { if (c->ev_join[i]) cudaEventDestroy(c->ev_join[i]); if (c->ev_late[i]) cudaEventDestroy(c->ev_late[i]); if (c->aux[i]) cudaStreamDestroy(c->aux[i]); }
  }
  delete c;
}

const char* dgp_last_error(dgp_ctx* c) { return c ? c->err.c_str() : "null ctx"; }

int dgp_set_stream(dgp_ctx* c, void* cuda_stream) {
  if (!c) return DGP_ERR_ARG;
  c->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
  return DGP_OK;
}

int64_t dgp_workspace_bytes(dgp_ctx* c) { return c ? (int64_t)c->cap : 0; }

int dgp_set_workspace_limit(dgp_ctx* c, int64_t bytes) {
  if (!c || bytes < ((int64_t)64 << 20)) return DGP_ERR_ARG;
  c->ws_limit = (size_t)bytes;
  return DGP_OK;
}

int dgp_set_parallel_layers(dgp_ctx* c, int on) {
  if (!c) return DGP_ERR_ARG;
  c->parallel_layers = on != 0;
  return DGP_OK;
}

int dgp_set_vform(dgp_ctx* c, int forward_calls, int gradient_calls) {
  if (!c) return DGP_ERR_ARG;
  c->use_vform_grad = gradient_calls != 0;
  c->vform_grad_min_ps = gradient_calls == 2 ? 0 : 32768;   // 2: always, 1: only with enough point-samples to amortise the glue
  c->vform_forward_calls = forward_calls != 0;
  return DGP_OK;
}

int dgp_check(dgp_ctx* c) {
  if (!c) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  return check_chol(c);
}

int dgp_set_share_first_layer(dgp_ctx* c, int on) {
  if (!c) return DGP_ERR_ARG;
  c->share_first_layer = on != 0;
  return DGP_OK;
}

int dgp_set_graph(dgp_ctx* c, int on) {
  if (!c) return DGP_ERR_ARG;
  c->use_graph = on != 0;
  if (!on) {
    CK(cudaSetDevice(c->device));
    CK(cudaStreamSynchronize(c->stream));
    drop_graphs(c);
  }
  return DGP_OK;
}

int dgp_set_fused(dgp_ctx* c, int on) {
  if (!c) return DGP_ERR_ARG;
  c->use_fused = on != 0;
  return DGP_OK;
}

int dgp_set_profiling(dgp_ctx* c, int on) {
  if (!c) return DGP_ERR_ARG;
  c->profiling = on != 0;
  return DGP_OK;
}

int dgp_get_profile(dgp_ctx* c, double* ms_out, int64_t* launches_out, int reset) {
  if (!c) return DGP_ERR_ARG;
  CK(cudaStreamSynchronize(c->stream));
  for (auto& s : c->spans) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, s.a, s.b) == cudaSuccess) c->cat_ms[s.cat] += ms;
    c->ev_pool.push_back(s.a);
    c->ev_pool.push_back(s.b);
  }
  c->spans.clear();
  for (int i = 0; i < DGP_PROFILE_CATEGORIES; ++i) {
    if (ms_out) ms_out[i] = c->cat_ms[i];
    if (launches_out) launches_out[i] = c->cat_launches[i];
    if (reset) { c->cat_ms[i] = 0.0; c->cat_launches[i] = 0; }
  }
  return DGP_OK;
}

int64_t dgp_launch_count(dgp_ctx* c, int reset) {
  if (!c) return 0;
  long v = c->launches;
  if (reset) c->launches = 0;
  return v;
}

int dgp_philox_normal(dgp_ctx* c, uint64_t seed, int layer, int64_t S, int64_t N, int D, int64_t n_offset, double* z_out) {
  if (!c || !z_out || S < 1 || N < 1 || D < 1) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  const long total = S * N * D;
  LAUNCH(philox_normal_kernel, (unsigned)((total + 255) / 256), 256, 0, (unsigned long long)seed, layer, (long)S, (long)N, D,
         (long)n_offset, z_out);
  return DGP_OK;
}

int dgp_philox_raw(dgp_ctx* c, uint64_t seed, int layer, int64_t S, int64_t N, int D, int64_t n_offset, uint32_t* words_out) {
  if (!c || !words_out || S < 1 || N < 1 || D < 1) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  const long total = S * N * D;
  LAUNCH(philox_raw_kernel, (unsigned)((total + 255) / 256), 256, 0, (unsigned long long)seed, layer, (long)S, (long)N, D, (long)n_offset,
         words_out);
  return DGP_OK;
}

int dgp_kernel_K(dgp_ctx* c, int kernel_kind, int D, const double* lengthscales, const double* variance, const double* X, int64_t n1,
                 const double* X2, int64_t n2, double* K_out) {
  if (!c || !X || !X2 || !K_out || D < 1 || D > kMaxD || n1 < 1 || n2 < 1 || kernel_kind < 0 || kernel_kind > 2) return DGP_ERR_ARG;
  if (n1 > 2147483647LL) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  LAUNCH(kuf_kernel, dim3((unsigned)((n2 + kKufCols - 1) / kKufCols), (unsigned)((n1 + kKufRows - 1) / kKufRows)), 256, 0, X2,
         (long)n2, X, lengthscales, variance, (int)n1, (int)n1, D, (long)n2, (long)n2, K_out, kernel_kind);
  return DGP_OK;
}

int dgp_kuu_chol(dgp_ctx* c, const dgp_layer_desc* layer, double* Ku_out, double* Lu_out) {
  if (!c || !layer) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  dgp_model_desc m{1, layer, nullptr};
  std::vector<LayerWs> lw;
  RC(planned(c, [&] { return prep_layers(c, &m, lw, PREP_FWD, ctx_path(c, PREP_FWD, 0)); }));
  const long mm = (long)layer->M * layer->M;
  if (Ku_out) LAUNCH(unpad_square_kernel, (unsigned)((mm + 255) / 256), 256, 0, lw[0].Ku, lw[0].M, lw[0].Mp, Ku_out);
  if (Lu_out) LAUNCH(unpad_square_kernel, (unsigned)((mm + 255) / 256), 256, 0, lw[0].L, lw[0].M, lw[0].Mp, Lu_out);
  return check_chol(c);
}

int dgp_kl(dgp_ctx* c, const dgp_layer_desc* layer, double* kl_out) {
  if (!c || !layer || !kl_out) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  dgp_model_desc m{1, layer, nullptr};
  std::vector<LayerWs> lw;
  RC(planned(c, [&] { return prep_layers(c, &m, lw, PREP_KL, ctx_path(c, PREP_KL, 0)); }));
  CK(cudaMemcpyAsync(kl_out, lw[0].kl, sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
  return check_chol(c);
}

int dgp_conditional_nd(dgp_ctx* c, const dgp_layer_desc* layer, const double* X, int64_t P, double* mean, double* var) {
  if (!c || !layer || !X || !mean || !var || P < 1) return DGP_ERR_ARG;
  dgp_model_desc m{1, layer, nullptr};
  RunOpts o;
  double* fm[1] = {mean};
  double* fv[1] = {var};
  o.io.Fmeans = fm; o.io.Fvars = fv;
  RC(run_model_planned(c, &m, X, P, 1, 0, 0, o));
  return check_chol(c);
}

int dgp_propagate(dgp_ctx* c, const dgp_model_desc* model, const double* X, int64_t N, int64_t S, const double* const* zs_host,
                  uint64_t seed, int64_t n_offset, double* const* Fs_host, double* const* Fmeans_host, double* const* Fvars_host) {
  if (!c || !model || !X) return DGP_ERR_ARG;
  RunOpts o;
  o.io.zs = zs_host; o.io.Fs = Fs_host; o.io.Fmeans = Fmeans_host; o.io.Fvars = Fvars_host;
  RC(run_model_planned(c, model, X, N, S, seed, n_offset, o));
  return check_chol(c);
}

namespace {
// propagate(full_cov=True): per layer the fused conditional (V-form, stash on) gives mean, V and T_d for all S samples at once;
// the S * D_out covariance blocks, their Cholesky factors and the correlated samples follow (fullcov.cuh).
int run_full_cov(dgp_ctx* c, const dgp_model_desc* model, const double* X, long N, long S, const double* const* zs_host,
                 unsigned long long seed, long n_offset, double* const* Fs_host, double* const* Fmeans_host,
                 double* const* Fvars_host) {
  RC(check_chain(c, model, N, S));
  const int nl = model->num_layers;
  const long Np = round_up(N, kTileM);
  if (Np > 768) { c->err = "full_cov=True: N > 768 is not supported (one CTA factorises an N x N block)"; return DGP_ERR_UNSUPPORTED; }
  std::vector<LayerWs> lw;
  RC(prep_layers(c, model, lw, PREP_FWD, {c->use_fused, true}));   // the covariance blocks are built from the V-form planes
  const long P = N * S, Pp = round_up(P, kTileP);
  int maxD = 1;
  for (int l = 0; l < nl; ++l) {
    if (lw[l].fcfg < 0 || !lw[l].vform) { c->err = "full_cov=True needs a layer shape the fused conditional kernel supports"; return DGP_ERR_UNSUPPORTED; }
    if (lw[l].D_out > maxD) maxD = lw[l].D_out;
  }
  std::vector<ChunkLayer> cls(nl);
  for (int l = 0; l < nl; ++l) {
    const LayerWs& w = lw[l];
    cls[l].F = walloc(c, (size_t)Pp * w.D_out); cls[l].Fmean = walloc(c, (size_t)Pp * w.D_out);
    cls[l].Fvar = walloc(c, (size_t)Pp * w.D_out); cls[l].z = walloc(c, (size_t)Pp * w.D_out);
  }
  // one set of planes and factor blocks, reused by every layer
  int maxMp = 0;
  for (int l = 0; l < nl; ++l) if (lw[l].Mp > maxMp) maxMp = lw[l].Mp;
  double* planeV = walloc(c, (size_t)maxMp * Pp);
  double* planeT = walloc(c, (size_t)maxD * maxMp * Pp);
  const size_t nblk = (size_t)S * maxD;
  double* cin = walloc(c, nblk * Np * Np);
  double* Lf = walloc(c, nblk * Np * Np);
  CholArgs* dargs = reinterpret_cast<CholArgs*>(walloc(c, (sizeof(CholArgs) * nblk + 7) / 8));
  Temps tmp;
  if (c->dry) return DGP_OK;
  std::vector<CholArgs> hargs(nblk);
  for (size_t i = 0; i < nblk; ++i) hargs[i] = CholArgs{cin + i * Np * Np, Lf + i * Np * Np, nullptr, nullptr, (int)Np, c->d_info};
  H2D(dargs, hargs.data(), sizeof(CholArgs) * nblk);
  RC(chol_smem_optin(c));
  for (int l = 0; l < nl; ++l) {
    const dgp_layer_desc& d = model->layers[l];
    const LayerWs& w = lw[l];
    ChunkLayer& cl = cls[l];
    if (l == 0) { cl.Xin = X; cl.xmod = N; } else { cl.Xin = cls[l - 1].F; cl.xmod = P; }
    cl.A = planeV; cl.T = planeT;
    ChunkIO io;   // means go straight to the caller; variances / samples are replaced by the full-covariance ones below
    std::vector<double*> fm(nl, nullptr);
    if (Fmeans_host && Fmeans_host[l]) { fm[l] = Fmeans_host[l]; io.Fmeans = fm.data(); }
    RC(forward_layer(c, d, w, cl, tmp, true, nullptr, l, N, S, N, 0, seed, n_offset, io, false));
    CAT(DGP_CAT_MOMENTS);
    FullCovArgs f;
    memset(&f, 0, sizeof(f));
    f.V = cl.A; f.T = cl.T; f.Xin = cl.Xin; f.xmod = cl.xmod; f.D_in = w.D_in; f.ls = d.lengthscales; f.var = d.variance;
    f.kind = d.kernel_kind; f.Mp = w.Mp; f.D = w.D_out; f.N = N; f.Np = Np; f.Pp = Pp; f.S = (int)S; f.jitter = d.jitter;
    f.var_out = (Fvars_host && Fvars_host[l]) ? Fvars_host[l] : nullptr; f.chol_in = cin;
    const unsigned nt = (unsigned)(Np / kFcTile), nb = (unsigned)(S * w.D_out);
    LAUNCH(fullcov_kernel, dim3(nt, nt, nb), 256, 0, f);
    const bool last = l == nl - 1;
    const bool want_sample = !last || (Fs_host && Fs_host[l]);
    if (!want_sample) continue;
    LAUNCH(chol_inv_kernel, nb, kCholThreads, chol_smem_bytes((int)Np), dargs);
    const double* z = (zs_host && zs_host[l]) ? zs_host[l] : nullptr;
    if (!z) {
      const long total = P * w.D_out;
      LAUNCH(philox_normal_kernel, (unsigned)((total + 255) / 256), 256, 0, seed, l, (long)S, (long)N, w.D_out, (long)n_offset, cl.z);
      z = cl.z;
    }
    LAUNCH(fullcov_sample_kernel, dim3((unsigned)((N + 127) / 128), nb), 128, 0, Lf, cl.Fmean, z, N, Np, w.D_out, (int)S, cl.F,
           (Fs_host && Fs_host[l]) ? Fs_host[l] : nullptr);
  }
  return DGP_OK;
}
}  // namespace

int dgp_propagate_full_cov(dgp_ctx* c, const dgp_model_desc* model, const double* X, int64_t N, int64_t S,
                           const double* const* zs_host, uint64_t seed, int64_t n_offset, double* const* Fs_host,
                           double* const* Fmeans_host, double* const* Fvars_host) {
  if (!c || !model || !X) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  RC(planned(c, [&] { return run_full_cov(c, model, X, N, S, zs_host, seed, n_offset, Fs_host, Fmeans_host, Fvars_host); }));
  return check_chol(c);
}

namespace {
CompK comp_view(const dgp_comp_kernel* k) {
  CompK v;
  v.D = k->D; v.Da = k->Da; v.has_prod = k->has_prod; v.has_linear = k->has_linear && k->lin_variance; v.in_ard = k->in_ard;
  v.in_var = k->in_variance; v.in_ls = k->in_lengthscales; v.corr_var = k->corr_variance; v.corr_ls = k->corr_lengthscale;
  v.prev_var = k->prev_variance; v.prev_ls = k->prev_lengthscale; v.lin_var = k->lin_variance; v.white_var = k->white_variance;
  return v;
}
int comp_check(dgp_ctx* c, const dgp_comp_kernel* k) {
  if (!k || k->D < 1 || k->D > kCompMaxD || k->Da < 1 || k->Da > k->D || !k->in_variance || !k->in_lengthscales) {
    c->err = "composite kernel: need 1 <= Da <= D <= 32 and the k_in parameters"; return DGP_ERR_ARG;
  }
  if (k->has_prod && (k->Da >= k->D || !k->corr_variance || !k->corr_lengthscale || !k->prev_variance || !k->prev_lengthscale)) {
    c->err = "composite kernel: the product part needs Da < D and the k_corr / k_prev parameters"; return DGP_ERR_ARG;
  }
  return DGP_OK;
}

// Prep of the supplied-matrix path: one layer on the A-form GEMM pipeline, Kuu = the caller's Ku. This also lays out the region
// that dgp_svgp_prep_cache_bytes sizes and the cached calls copy.
int svgp_prep(dgp_ctx* c, int M, int D, const double* Ku, const double* q_mu, const double* q_sqrt, PrepLevel level,
              std::vector<LayerWs>& lw) {
  // a descriptor that satisfies check_layer: the kernel fields are never read (Ku is supplied, the fused kernels are off)
  dgp_layer_desc d;
  memset(&d, 0, sizeof(d));
  d.D_in = 1; d.D_out = D; d.M = M; d.white = 0; d.mean_kind = 0; d.kernel_kind = 0;
  d.Z = Ku; d.lengthscales = Ku; d.variance = Ku; d.q_mu = q_mu; d.q_sqrt = q_sqrt; d.jitter = 0.0;
  dgp_model_desc model{1, &d, nullptr};
  const double* kext[1] = {Ku};
  return prep_layers(c, &model, lw, level, {false, false}, false, kext);
}

// The layer's conditional (and, with Gm, its adjoint) on supplied kernel matrices: A-form GEMM pipeline, one pass over all P.
int svgp_from_k_run(dgp_ctx* c, int M, int D, long P, const double* Ku, const double* Kuf, const double* Kdiag, const double* q_mu,
                    const double* q_sqrt, double* mean, double* var, double* kl, const double* Gm, const double* Gv, double gkl,
                    double* dKu, double* dKuf, double* dKdiag, double* dq_mu, double* dq_sqrt, double* cache = nullptr,
                    size_t cache_bytes = 0, bool cache_load = false, double* stash = nullptr) {
  const bool grad = Gm != nullptr;
  std::vector<LayerWs> lw;
  // With a cache the per-layer replicated work (Kuu factorisation, inverse, the M^3 products, KL) is done ONCE for all applications
  // of the layer inside one ELBO evaluation and their adjoints: the first call stores the prepared region of the arena, the others
  // lay the region out again without launching anything and copy it back (a few MB, device to device).
  const size_t prep_start = c->used;
  c->replay = cache != nullptr && cache_load;
  const int rc = svgp_prep(c, M, D, Ku, q_mu, q_sqrt, (grad || cache) ? PREP_GRAD : PREP_KL, lw);
  c->replay = false;
  RC(rc);
  if (cache && !c->dry) {
    const size_t prep_bytes = c->used - prep_start;
    if (prep_bytes > cache_bytes) { c->err = "dgp_svgp_from_k_cached: cache smaller than dgp_svgp_prep_cache_bytes"; return DGP_ERR_ARG; }
    if (cache_load) CK(cudaMemcpyAsync(c->ws + prep_start, cache, prep_bytes, cudaMemcpyDeviceToDevice, c->stream));
    else CK(cudaMemcpyAsync(cache, c->ws + prep_start, prep_bytes, cudaMemcpyDeviceToDevice, c->stream));
  }
  LayerWs& w = lw[0];
  const int Mp = w.Mp;
  const long Pp = round_up(P, kTileP);
  const size_t plane = (size_t)Mp * Pp;
  // `stash` (caller-owned, (1 + D) planes): the forward call leaves A and the T_d planes there and the adjoint call reads them back
  // instead of running the three forward products again
  const bool reuse = stash != nullptr && grad;
  const size_t nplanes = (reuse ? 0 : 2) + (stash ? 0 : 1 + (size_t)D) + (grad ? 2 : 0);
  if ((plane * nplanes + (size_t)Pp * 80) * sizeof(double) + c->used > c->ws_limit) {
    c->err = "dgp_svgp_from_k: P too large for the workspace limit (dgp_set_workspace_limit); split the points"; return DGP_ERR_UNSUPPORTED;
  }
  double *K = nullptr, *V = nullptr, *A = nullptr, *T = nullptr;
  if (!reuse) { K = walloc(c, plane); V = walloc(c, plane); }
  if (stash) { A = stash; T = stash + plane; }
  else { A = walloc(c, plane); T = walloc(c, plane * D); }
  double *dA = nullptr, *W = nullptr, *GvT = nullptr, *GmPad = nullptr, *gq = nullptr, *part = nullptr, *dummy = nullptr;
  size_t partcap = 0;
  if (grad) {
    dA = walloc(c, plane); W = walloc(c, plane);
    GvT = walloc(c, (size_t)D * Pp); GmPad = walloc(c, (size_t)Pp * 32); gq = walloc(c, (size_t)Pp);
    partcap = max_splitk_part(lw);
    part = walloc(c, partcap);
    dummy = walloc(c, 64);
  }
  if (c->dry) return DGP_OK;
  CAT(DGP_CAT_GEMM_FWD);
  if (!reuse) {
    LAUNCH(pad_plane_kernel, (unsigned)((plane + 255) / 256), 256, 0, Kuf, M, Mp, P, Pp, K);
    RC(aform_forward(c, w, K, V, A, T, Pp));
  }
  if (mean) {
    CAT(DGP_CAT_MOMENTS);
    LAUNCH(moments_ext_kernel, (unsigned)((P + 127) / 128), 128, 0, V, A, T, w.qmuP, Kdiag, M, Mp, D, P, Pp, mean, var);
  }
  if (kl) CK(cudaMemcpyAsync(kl, w.kl, sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
  if (!grad) return DGP_OK;
  // ---- adjoint (SURVEY §9, A-form) ----
  CAT(DGP_CAT_OTHER);
  LAUNCH(upstream_ext_kernel, (unsigned)(Pp / 128), 128, 0, Gm, Gv, P, Pp, D, GvT, GmPad, gq, dKdiag);
  CAT(DGP_CAT_GEMM_BWD_DATA);
  RC(aform_adjoint(c, w, T, GmPad, GvT, dA, W, Pp, nullptr));
  CAT(DGP_CAT_RBF_BWD);
  LAUNCH(kbar_ext_kernel, (unsigned)(((size_t)M * Pp + 255) / 256), 256, 0, W, A, gq, M, P, Pp, dKuf);
  CAT(DGP_CAT_GEMM_BWD_PARAM);
  GemmArgs pg[3];
  aform_param_args(w, W, A, T, GvT, GmPad, Pp, 0.0, pg);
  CK(cudaMemsetAsync(w.dR, 0, (size_t)D * Mp * Mp * sizeof(double), c->stream));   // c_lower leaves the upper tiles unwritten
  for (int i = 0; i < 3; ++i) {
    pg[i].splitk = pick_splitk(c, pg[i], kAformParamNT[i]);
    if (pg[i].splitk > 1 && (size_t)pg[i].splitk * pg[i].batch * pg[i].M * pg[i].N > partcap) pg[i].splitk = 1;
    pg[i].part = part;
    RC(gemm(c, pg[i], kAformParamNT[i]));
  }
  // ---- KL adjoint (weighted by gkl: the caller's d loss / d kl) and unpadding ----
  CAT(DGP_CAT_PREP);
  const long mm = (long)Mp * Mp;
  LAUNCH(dku_assemble_kernel, (unsigned)((mm + 255) / 256), 256, 0, w.dKu, w.Kinv, w.KSK, w.alpha, w.Knj, M, Mp, D, -gkl, 1);
  LAUNCH(unpad_square_kernel, (unsigned)(((long)M * M + 255) / 256), 256, 0, w.dKu, M, Mp, dKu);
  FinalizeArgs f;
  memset(&f, 0, sizeof(f));
  f.Gd = w.dR; f.gd_cat = 0; f.KR = w.KRcat; f.Rcat = w.Rcat; f.dqmu = w.dqmu; f.alpha = w.alpha; f.H = nullptr; f.dZk = dummy;
  f.rbf_red = nullptr; f.kuu_red = dummy; f.sgv = nullptr; f.Z = dummy; f.ls = dummy; f.M = M; f.Mp = Mp; f.D_in = 0; f.D_out = D;
  f.klw = -gkl; f.white = 0; f.qmuP = w.qmuP;
  f.dZ = dummy; f.dls = dummy; f.dvar = dummy + 32; f.dq_mu = dq_mu; f.dq_sqrt = dq_sqrt;
  const long nq = (long)D * M * M;
  LAUNCH(finalize_layer_kernel, (unsigned)((nq + 255) / 256), 256, 0, f);
  return DGP_OK;
}
}  // namespace

int dgp_comp_K(dgp_ctx* c, const dgp_comp_kernel* k, const double* X, int64_t P, const double* X2, int64_t P2, double* K_out) {
  if (!c || !X || !K_out || P < 1 || (X2 && P2 < 1)) return DGP_ERR_ARG;
  RC(comp_check(c, k));
  CK(cudaSetDevice(c->device));
  const long n2 = X2 ? P2 : P;
  CAT(DGP_CAT_KUF);
  LAUNCH(compk_K_kernel, (unsigned)((P * n2 + 255) / 256), 256, 0, comp_view(k), X, (long)P, X2, n2, K_out);
  return DGP_OK;
}

int dgp_comp_Kdiag(dgp_ctx* c, const dgp_comp_kernel* k, const double* X, int64_t P, double* out) {
  if (!c || !X || !out || P < 1) return DGP_ERR_ARG;
  RC(comp_check(c, k));
  CK(cudaSetDevice(c->device));
  CAT(DGP_CAT_KUF);
  LAUNCH(compk_Kdiag_kernel, (unsigned)((P + 255) / 256), 256, 0, comp_view(k), X, (long)P, out);
  return DGP_OK;
}

int dgp_comp_K_blocks(dgp_ctx* c, const dgp_comp_kernel* k, const double* X, int64_t B, int64_t N, double* K_out) {
  if (!c || !X || !K_out || B < 1 || N < 1) return DGP_ERR_ARG;
  RC(comp_check(c, k));
  CK(cudaSetDevice(c->device));
  const long nn = (long)N * N;
  CAT(DGP_CAT_KUF);
  LAUNCH(compk_K_blocks_kernel, dim3((unsigned)((nn + 255) / 256), (unsigned)(B < 65535 ? B : 65535)), 256, 0, comp_view(k), X, (long)B,
         (long)N, K_out);
  return DGP_OK;
}

int dgp_comp_K_grad(dgp_ctx* c, const dgp_comp_kernel* k, const double* X, int64_t P, const double* X2, int64_t P2,
                    const double* Kbar, double* dX, double* dX2, double* dtheta) {
  if (!c || !X || !Kbar || !dX || !dtheta || P < 1 || (X2 && (P2 < 1 || !dX2))) return DGP_ERR_ARG;
  RC(comp_check(c, k));
  CK(cudaSetDevice(c->device));
  const long n2 = X2 ? P2 : P;
  const int nt = kCompTheta + (k->in_ard ? k->Da : 1);
  // rows of X against column chunks of X2: enough CTAs to fill the machine when X is the M inducing inputs and X2 the point-samples
  int nsplit = 1;
  while (nsplit < 32 && (long)P * nsplit < 148L * 16 && n2 / (2 * nsplit) >= 1024) nsplit *= 2;
  const long chunk = (n2 + nsplit - 1) / nsplit;
  RC(ensure_ws(c, (size_t)P * nsplit * (nt + k->D) * sizeof(double)));
  double* part = reinterpret_cast<double*>(c->ws);
  double* dXp = nsplit > 1 ? part + (size_t)P * nsplit * nt : dX;
  CAT(DGP_CAT_RBF_BWD);
  if (k->D <= 8) {
    LAUNCH(compk_grad_rows_kernel<8>, dim3((unsigned)P, (unsigned)nsplit), 128, 0, comp_view(k), X, (long)P, X2, n2, chunk, Kbar, dXp, part);
  } else if (k->D <= 16) {
    LAUNCH(compk_grad_rows_kernel<16>, dim3((unsigned)P, (unsigned)nsplit), 128, 0, comp_view(k), X, (long)P, X2, n2, chunk, Kbar, dXp, part);
  } else {
    LAUNCH(compk_grad_rows_kernel<32>, dim3((unsigned)P, (unsigned)nsplit), 128, 0, comp_view(k), X, (long)P, X2, n2, chunk, Kbar, dXp, part);
  }
  if (nsplit > 1) LAUNCH(compk_sum_splits_kernel, (unsigned)((P * k->D + 255) / 256), 256, 0, dXp, nsplit, (long)P * k->D, dX);
  LAUNCH(reduce_partials_kernel, nt, 256, 0, part, (long)P * nsplit, nt, dtheta, 0);
  if (X2) {
    if (k->D <= 8) {
      LAUNCH(compk_grad_cols_kernel<8>, (unsigned)((P2 + 127) / 128), 128, 0, comp_view(k), X, (long)P, X2, (long)P2, Kbar, dX2);
    } else if (k->D <= 16) {
      LAUNCH(compk_grad_cols_kernel<16>, (unsigned)((P2 + 127) / 128), 128, 0, comp_view(k), X, (long)P, X2, (long)P2, Kbar, dX2);
    } else {
      LAUNCH(compk_grad_cols_kernel<32>, (unsigned)((P2 + 127) / 128), 128, 0, comp_view(k), X, (long)P, X2, (long)P2, Kbar, dX2);
    }
  }
  return DGP_OK;
}

int dgp_comp_Kdiag_grad(dgp_ctx* c, const dgp_comp_kernel* k, const double* X, int64_t P, const double* g, double* dX, double* dtheta) {
  if (!c || !X || !g || !dX || !dtheta || P < 1) return DGP_ERR_ARG;
  RC(comp_check(c, k));
  CK(cudaSetDevice(c->device));
  const int nt = kCompTheta + (k->in_ard ? k->Da : 1);
  const long nb = (P + 127) / 128;
  RC(ensure_ws(c, (size_t)nb * nt * sizeof(double)));
  double* part = reinterpret_cast<double*>(c->ws);
  CAT(DGP_CAT_RBF_BWD);
  LAUNCH(compk_Kdiag_grad_kernel, (unsigned)nb, 128, 0, comp_view(k), X, (long)P, g, dX, part);
  LAUNCH(reduce_partials_kernel, nt, 256, 0, part, nb, nt, dtheta, 0);
  return DGP_OK;
}

int dgp_svgp_from_k(dgp_ctx* c, int M, int D_out, int64_t P, const double* Ku, const double* Kuf, const double* Kdiag,
                    const double* q_mu, const double* q_sqrt, double* mean, double* var, double* kl) {
  if (!c || !Ku || !Kuf || !Kdiag || !q_mu || !q_sqrt || !mean || !var || M < 1 || D_out < 1 || D_out > kMaxD || P < 1) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  return planned(c, [&] {
    return svgp_from_k_run(c, M, D_out, P, Ku, Kuf, Kdiag, q_mu, q_sqrt, mean, var, kl, nullptr, nullptr, 0.0, nullptr, nullptr, nullptr,
                           nullptr, nullptr);
  });
}

int dgp_svgp_from_k_grad(dgp_ctx* c, int M, int D_out, int64_t P, const double* Ku, const double* Kuf, const double* Kdiag,
                         const double* q_mu, const double* q_sqrt, const double* Gm, const double* Gv, double gkl,
                         double* dKu, double* dKuf, double* dKdiag, double* dq_mu, double* dq_sqrt) {
  if (!c || !Ku || !Kuf || !Kdiag || !q_mu || !q_sqrt || !Gm || !Gv || !dKu || !dKuf || !dKdiag || !dq_mu || !dq_sqrt || M < 1 ||
      D_out < 1 || D_out > kMaxD || P < 1) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  return planned(c, [&] {
    return svgp_from_k_run(c, M, D_out, P, Ku, Kuf, Kdiag, q_mu, q_sqrt, nullptr, nullptr, nullptr, Gm, Gv, gkl, dKu, dKuf, dKdiag, dq_mu,
                           dq_sqrt);
  });
}

int64_t dgp_svgp_prep_cache_bytes(dgp_ctx* c, int M, int D_out) {
  if (!c || M < 1 || D_out < 1 || D_out > kMaxD) return -1;
  static const double unread = 0.0;      // the dry pass only lays the arena out: no pointer it is given is dereferenced
  std::vector<LayerWs> lw;
  const bool dry_saved = c->dry;
  const size_t used_saved = c->used;
  c->dry = true; c->used = 0;
  const int rc = svgp_prep(c, M, D_out, &unread, &unread, &unread, PREP_GRAD, lw);
  const size_t bytes = c->used;
  c->dry = dry_saved; c->used = used_saved;
  return rc == DGP_OK ? (int64_t)bytes : -1;
}

int64_t dgp_svgp_stash_bytes(int M, int D_out, int64_t P) {
  if (M < 1 || D_out < 1 || P < 1) return -1;
  return (int64_t)((size_t)(1 + D_out) * round_up(M, kTileM) * round_up(P, kTileP) * sizeof(double));
}

int dgp_svgp_from_k_cached(dgp_ctx* c, int M, int D_out, int64_t P, const double* Ku, const double* Kuf, const double* Kdiag,
                           const double* q_mu, const double* q_sqrt, double* mean, double* var, double* kl, double* cache,
                           int64_t cache_bytes, int load, double* stash) {
  if (!c || !Ku || !Kuf || !Kdiag || !q_mu || !q_sqrt || !mean || !var || !cache || cache_bytes < 1 || M < 1 || D_out < 1 ||
      D_out > kMaxD || P < 1) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  return planned(c, [&] {
    return svgp_from_k_run(c, M, D_out, P, Ku, Kuf, Kdiag, q_mu, q_sqrt, mean, var, kl, nullptr, nullptr, 0.0, nullptr, nullptr, nullptr,
                           nullptr, nullptr, cache, (size_t)cache_bytes, load != 0, stash);
  });
}

int dgp_svgp_from_k_grad_cached(dgp_ctx* c, int M, int D_out, int64_t P, const double* Ku, const double* Kuf, const double* Kdiag,
                                const double* q_mu, const double* q_sqrt, const double* Gm, const double* Gv, double gkl,
                                double* dKu, double* dKuf, double* dKdiag, double* dq_mu, double* dq_sqrt, const double* cache,
                                int64_t cache_bytes, const double* stash) {
  if (!c || !Ku || !Kuf || !Kdiag || !q_mu || !q_sqrt || !Gm || !Gv || !dKu || !dKuf || !dKdiag || !dq_mu || !dq_sqrt || !cache ||
      cache_bytes < 1 || M < 1 || D_out < 1 || D_out > kMaxD || P < 1) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  return planned(c, [&] {
    return svgp_from_k_run(c, M, D_out, P, Ku, Kuf, Kdiag, q_mu, q_sqrt, nullptr, nullptr, nullptr, Gm, Gv, gkl, dKu, dKuf, dKdiag, dq_mu,
                           dq_sqrt, const_cast<double*>(cache), (size_t)cache_bytes, true, const_cast<double*>(stash));
  });
}

namespace {
// full_cov=True on supplied matrices: the prep and the A-form planes of dgp_svgp_from_k over all S * N columns (so the mean is the
// same computation), then, as run_full_cov does on its V-form planes, the S * D_out covariance blocks, their factors and the samples.
int svgp_full_cov_run(dgp_ctx* c, int M, int D, long N, long S, const double* Ku, const double* Kuf, const double* Kff, long Kff_batch,
                      const double* q_mu, const double* q_sqrt, const double* z, double jitter, double* mean, double* cov, double* F) {
  std::vector<LayerWs> lw;
  RC(svgp_prep(c, M, D, Ku, q_mu, q_sqrt, PREP_FWD, lw));
  const LayerWs& w = lw[0];
  const int Mp = w.Mp;
  const long P = N * S, Pp = round_up(P, kTileP), Np = round_up(N, kTileM);
  const size_t plane = (size_t)Mp * Pp, nblk = (size_t)S * D, blk = (size_t)Np * Np;
  const bool blocks = cov || F;
  const size_t need = (plane * (3 + (size_t)D) + (size_t)P * (D + 1) + (blocks ? 1 : 0) * nblk * blk + (F ? 1 : 0) * nblk * blk) * sizeof(double);
  if (need + c->used > c->ws_limit) {
    c->err = "dgp_svgp_from_k_full_cov: S * N too large for the workspace limit (dgp_set_workspace_limit); split the samples";
    return DGP_ERR_UNSUPPORTED;
  }
  double* K = walloc(c, plane);
  double* V = walloc(c, plane);
  double* A = walloc(c, plane);
  double* T = walloc(c, plane * D);
  double* kzero = walloc(c, (size_t)P);           // K_diag of moments_ext_kernel: its variance is not used, the blocks carry it
  double* vscr = walloc(c, (size_t)P * D);
  double* cin = blocks ? walloc(c, nblk * blk) : nullptr;
  double* Lf = F ? walloc(c, nblk * blk) : nullptr;
  CholArgs* dargs = F ? reinterpret_cast<CholArgs*>(walloc(c, (sizeof(CholArgs) * nblk + 7) / 8)) : nullptr;
  if (c->dry) return DGP_OK;
  CAT(DGP_CAT_GEMM_FWD);
  LAUNCH(pad_plane_kernel, (unsigned)((plane + 255) / 256), 256, 0, Kuf, M, Mp, P, Pp, K);
  RC(aform_forward(c, w, K, V, A, T, Pp));
  CAT(DGP_CAT_MOMENTS);
  CK(cudaMemsetAsync(kzero, 0, (size_t)P * sizeof(double), c->stream));
  LAUNCH(moments_ext_kernel, (unsigned)((P + 127) / 128), 128, 0, V, A, T, w.qmuP, kzero, M, Mp, D, P, Pp, mean, vscr);
  if (!blocks) return DGP_OK;
  FullCovArgs f;
  memset(&f, 0, sizeof(f));
  f.V = V; f.T = T; f.Mp = Mp; f.D = D; f.N = N; f.Np = Np; f.Pp = Pp; f.S = (int)S; f.jitter = jitter;
  f.var_out = cov; f.chol_in = cin;
  const unsigned nt = (unsigned)(Np / kFcTile);
  LAUNCH(fullcov_ext_kernel, dim3(nt, nt, (unsigned)nblk), 256, 0, f, Kff, Kff_batch == 1 ? 0L : N * N);
  if (!F) return DGP_OK;
  std::vector<CholArgs> hargs(nblk);
  for (size_t i = 0; i < nblk; ++i) hargs[i] = CholArgs{cin + i * blk, Lf + i * blk, nullptr, nullptr, (int)Np, c->d_info};
  H2D(dargs, hargs.data(), sizeof(CholArgs) * nblk);
  RC(chol_smem_optin(c));
  LAUNCH(chol_inv_kernel, (unsigned)nblk, kCholThreads, chol_smem_bytes((int)Np), dargs);
  LAUNCH(fullcov_sample_kernel, dim3((unsigned)((N + 127) / 128), (unsigned)nblk), 128, 0, Lf, mean, z, N, Np, D, (int)S, F, nullptr);
  return DGP_OK;
}
}  // namespace

int dgp_svgp_from_k_full_cov(dgp_ctx* c, int M, int D_out, int64_t N, int64_t S, const double* Ku, const double* Kuf,
                             const double* Kff, int64_t Kff_batch, const double* q_mu, const double* q_sqrt, const double* z,
                             double jitter, double* mean, double* cov, double* F) {
  if (!c) return DGP_ERR_ARG;
  if (!Ku || !Kuf || !Kff || !q_mu || !q_sqrt || !mean || M < 1 || D_out < 1 || D_out > kMaxD || N < 1 || S < 1) {
    c->err = "dgp_svgp_from_k_full_cov: null input or output, or a size out of range (M >= 1, 1 <= D_out <= 32, N >= 1, S >= 1)";
    return DGP_ERR_ARG;
  }
  if (round_up(N, kTileM) > 768) {
    c->err = "dgp_svgp_from_k_full_cov: N > 768 is not supported (one CTA factorises an N x N block)"; return DGP_ERR_UNSUPPORTED;
  }
  if (Kff_batch != 1 && Kff_batch != S) { c->err = "dgp_svgp_from_k_full_cov: Kff_batch must be 1 (one shared block) or S"; return DGP_ERR_ARG; }
  if (F && !z) { c->err = "dgp_svgp_from_k_full_cov: F needs the draws z"; return DGP_ERR_ARG; }
  if (S * D_out > 65535) { c->err = "dgp_svgp_from_k_full_cov: S * D_out > 65535 covariance blocks"; return DGP_ERR_UNSUPPORTED; }
  CK(cudaSetDevice(c->device));
  RC(planned(c, [&] { return svgp_full_cov_run(c, M, D_out, N, S, Ku, Kuf, Kff, Kff_batch, q_mu, q_sqrt, z, jitter, mean, cov, F); }));
  return check_chol(c, "dgp_svgp_from_k_full_cov: Ku or a block cov + jitter I is not positive definite (Cholesky pivot <= 0)");
}

int64_t dgp_grad_size(const dgp_model_desc* model) {
  if (!model) return 0;
  int64_t n = 3;
  for (int l = 0; l < model->num_layers; ++l) {
    const dgp_layer_desc& d = model->layers[l];
    n += (int64_t)d.M * d.D_in + d.D_in + 1 + (int64_t)d.M * d.D_out + (int64_t)d.D_out * d.M * d.M;
  }
  return n;
}

int dgp_grad_layout(const dgp_model_desc* model, dgp_layer_grad_offsets* offs) {
  if (!model || !offs) return DGP_ERR_ARG;
  int64_t n = 3;
  for (int l = 0; l < model->num_layers; ++l) {
    const dgp_layer_desc& d = model->layers[l];
    offs[l].dZ = n; n += (int64_t)d.M * d.D_in;
    offs[l].dlengthscales = n; n += d.D_in;
    offs[l].dvariance = n; n += 1;
    offs[l].dq_mu = n; n += (int64_t)d.M * d.D_out;
    offs[l].dq_sqrt = n; n += (int64_t)d.D_out * d.M * d.M;
  }
  return DGP_OK;
}

int dgp_elbo_grad(dgp_ctx* c, const dgp_model_desc* model, const double* X, const double* Y, int64_t N, int64_t S, double scale,
                  double kl_weight, const double* const* zs_host, uint64_t seed, int64_t n_offset, int want_grad,
                  double* out_flat) {
  if (!c || !model || !X || !Y || !out_flat) return DGP_ERR_ARG;
  RunOpts o;
  o.want_grad = want_grad != 0; o.want_elbo = true;
  o.Y = Y; o.Dy = model->layers[model->num_layers - 1].D_out;
  o.scale = scale; o.kl_weight = kl_weight; o.out_flat = out_flat; o.io.zs = zs_host;
  return run_model_planned(c, model, X, N, S, seed, n_offset, o);
}

namespace {
int adam_table(dgp_ctx* c, const dgp_adam_param* params, int n_params, AdamTable& t) {
  if (!params || n_params < 1) { c->err = "no parameters to optimise"; return DGP_ERR_ARG; }
  if (n_params > kAdamMaxParams) { c->err = "more than 48 parameters in one Adam launch"; return DGP_ERR_UNSUPPORTED; }
  memset(&t, 0, sizeof(t));
  t.n = n_params;
  long start = 0;
  for (int i = 0; i < n_params; ++i) {
    const dgp_adam_param& p = params[i];
    if (!p.value || p.count < 1 || p.grad_offset < 0 || p.transform < 0 || p.transform > 3 ||
        (p.grad_count != p.count && p.count != 1) || p.grad_count < 1 ||
        (p.transform == 3 && (p.M < 1 || p.count % ((int64_t)p.M * p.M) != 0)) || (p.mirror && p.mirror_count < 1)) {
      c->err = "invalid dgp_adam_param";
      return DGP_ERR_ARG;
    }
    AdamSeg& sg = t.seg[i];
    sg.value = p.value; sg.mirror = p.mirror; sg.start = start; sg.count = p.count; sg.grad_offset = p.grad_offset;
    sg.grad_count = p.grad_count; sg.mirror_count = p.mirror ? p.mirror_count : 0; sg.transform = p.transform; sg.M = p.M > 0 ? p.M : 1;
    start += p.count;
  }
  t.total = start;
  return DGP_OK;
}

int adam_launch(dgp_ctx* c, const AdamTable& t, const double* grad, double* m, double* v, int64_t step, double lr, double b1,
                double b2, double eps, double* trace) {
  const double lr_t = lr * sqrt(1.0 - pow(b2, (double)step)) / (1.0 - pow(b1, (double)step));
  CAT(DGP_CAT_OTHER);
  LAUNCH(adam_kernel, (unsigned)((t.total + 255) / 256), 256, 0, t, grad, m, v, lr_t, b1, b2, eps, trace, c->d_info);
  return DGP_OK;
}
}  // namespace

int dgp_adam_step(dgp_ctx* c, const dgp_adam_param* params, int n_params, const double* grad_flat, double* m_state,
                  double* v_state, int64_t t, double lr, double beta1, double beta2, double epsilon) {
  if (!c || !grad_flat || !m_state || !v_state || t < 1) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  AdamTable tab;
  RC(adam_table(c, params, n_params, tab));
  return adam_launch(c, tab, grad_flat, m_state, v_state, t, lr, beta1, beta2, epsilon, nullptr);
}

int dgp_train_adam(dgp_ctx* c, const dgp_model_desc* model, const double* X, const double* Y, int64_t N, int64_t S, double scale,
                   double kl_weight, uint64_t seed0, uint64_t seed_stride, int64_t n_offset, const dgp_adam_param* params,
                   int n_params, double* m_state, double* v_state, int64_t t0, int64_t steps, double lr, double beta1,
                   double beta2, double epsilon, double* out_flat, double* elbo_trace) {
  if (!c || !model || !X || !Y || !out_flat || !m_state || !v_state || t0 < 1 || steps < 0) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  AdamTable tab;
  RC(adam_table(c, params, n_params, tab));
  for (int64_t k = 0; k < steps; ++k) {
    RC(dgp_elbo_grad(c, model, X, Y, N, S, scale, kl_weight, nullptr, seed0 + (uint64_t)k * seed_stride, n_offset, 1, out_flat));
    RC(adam_launch(c, tab, out_flat, m_state, v_state, t0 + k, lr, beta1, beta2, epsilon, elbo_trace ? elbo_trace + k : nullptr));
  }
  return DGP_OK;
}

namespace {
// One natural-gradient step on the listed layers from the gradients in grad_flat; all device work, batched over (layer, d).
// the (layer, d) outputs of one (q_mu [M, D], q_sqrt [D, M, M]) pair with its ELBO gradients, appended to `outs`
void natgrad_add_pair(std::vector<NatOut>& outs, long& off, int& maxMp, int& maxM, double* q_mu, double* q_sqrt, const double* g_mu,
                      const double* g_sqrt, int M, int D) {
  const int Mp = (int)round_up(M, kTileM);
  for (int j = 0; j < D; ++j) {
    NatOut o;
    o.q_sqrt = q_sqrt + (long)j * M * M; o.q_sqrt_out = const_cast<double*>(o.q_sqrt);
    o.g_sqrt = g_sqrt + (long)j * M * M;
    o.g_mu = g_mu; o.q_mu = q_mu;
    o.M = M; o.Mp = Mp; o.D = D; o.d = j; o.off = off;
    off += (long)Mp * Mp;
    outs.push_back(o);
  }
  if (Mp > maxMp) maxMp = Mp;
  if (M > maxM) maxM = M;
}

int natgrad_outs(dgp_ctx* c, const std::vector<NatOut>& outs, long off, int maxMp, int maxM, double gamma);

int natgrad_run(dgp_ctx* c, const dgp_model_desc* model, const int* layer_ids, int n_layers, double gamma, const double* grad_flat) {
  std::vector<dgp_layer_grad_offsets> offs(model->num_layers);
  dgp_grad_layout(model, offs.data());
  std::vector<NatOut> outs;
  int maxMp = 0, maxM = 0;
  long off = 0;
  for (int k = 0; k < n_layers; ++k) {
    const int l = layer_ids[k];
    if (l < 0 || l >= model->num_layers) { c->err = "natural gradient: layer index out of range"; return DGP_ERR_ARG; }
    const dgp_layer_desc& d = model->layers[l];
    RC(check_layer(c, d));
    natgrad_add_pair(outs, off, maxMp, maxM, const_cast<double*>(d.q_mu), const_cast<double*>(d.q_sqrt), grad_flat + offs[l].dq_mu,
                     grad_flat + offs[l].dq_sqrt, d.M, d.D_out);
  }
  return natgrad_outs(c, outs, off, maxMp, maxM, gamma);
}

int natgrad_pairs_run(dgp_ctx* c, const dgp_nat_pair* pairs, int n_pairs, double gamma) {
  std::vector<NatOut> outs;
  int maxMp = 0, maxM = 0;
  long off = 0;
  for (int k = 0; k < n_pairs; ++k) {
    const dgp_nat_pair& p = pairs[k];
    if (!p.q_mu || !p.q_sqrt || !p.g_mu || !p.g_sqrt || p.M < 1 || p.D_out < 1) { c->err = "natural gradient: null pointer or empty pair"; return DGP_ERR_ARG; }
    if (p.M > 768) { c->err = "natural gradient: M <= 768 (one CTA factorises an M x M block)"; return DGP_ERR_ARG; }
    natgrad_add_pair(outs, off, maxMp, maxM, p.q_mu, p.q_sqrt, p.g_mu, p.g_sqrt, p.M, p.D_out);
  }
  return natgrad_outs(c, outs, off, maxMp, maxM, gamma);
}

int natgrad_outs(dgp_ctx* c, const std::vector<NatOut>& outs, long off, int maxMp, int maxM, double gamma) {
  const int nout = (int)outs.size();
  if (nout == 0) return DGP_OK;
  double *R = walloc(c, off), *RT = walloc(c, off), *GR = walloc(c, off), *T = walloc(c, off), *Bf = walloc(c, off);
  double *Lf = walloc(c, off), *Linv = walloc(c, off), *LinvT = walloc(c, off), *UinvT = walloc(c, off), *Cm = walloc(c, off);
  NatOut* douts = reinterpret_cast<NatOut*>(walloc(c, (sizeof(NatOut) * nout + 7) / 8));
  CholArgs* dargs = reinterpret_cast<CholArgs*>(walloc(c, (sizeof(CholArgs) * nout + 7) / 8));
  double** dinv = reinterpret_cast<double**>(walloc(c, (size_t)nout));
  double** dinvT = reinterpret_cast<double**>(walloc(c, (size_t)nout));
  if (c->dry) return DGP_OK;
  std::vector<CholArgs> hargs(nout);
  std::vector<double*> hinv(nout), hinvT(nout);
  for (int i = 0; i < nout; ++i) {
    hargs[i] = CholArgs{Bf + outs[i].off, Lf + outs[i].off, nullptr, nullptr, outs[i].Mp, c->d_info};
    hinv[i] = Linv + outs[i].off; hinvT[i] = LinvT + outs[i].off;
  }
  CAT(DGP_CAT_PREP);
  H2D(douts, outs.data(), sizeof(NatOut) * nout);
  H2D(dargs, hargs.data(), sizeof(CholArgs) * nout);
  H2D(dinv, hinv.data(), sizeof(double*) * nout);
  H2D(dinvT, hinvT.data(), sizeof(double*) * nout);
  const unsigned gx = (unsigned)(((long)maxMp * maxMp + 255) / 256);
  LAUNCH(natgrad_prep_kernel, dim3(gx, (unsigned)nout), 256, 0, douts, R, RT, GR);
  for (int i = 0; i < nout; ++i) {   // T = R^T G_R (outputs of one layer share Mp; one launch per output keeps the shapes exact)
    const NatOut& o = outs[i];
    GemmArgs g = gargs(RT + o.off, o.Mp, GR + o.off, o.Mp, T + o.off, o.Mp, o.Mp, o.Mp, o.Mp);
    g.a_tri = 2;
    RC(gemm(c, g, false));
  }
  LAUNCH(natgrad_b_kernel, dim3(gx, (unsigned)nout), 256, 0, douts, T, gamma, Bf);
  RC(chol_smem_optin(c));
  LAUNCH(chol_inv_kernel, nout, kCholThreads, chol_smem_bytes(maxMp), dargs);
  LAUNCH(tri_inv_kernel, dim3((unsigned)(maxMp / 32), (unsigned)nout), 256, tri_inv_smem_bytes(maxMp), dargs, dinv, dinvT);
  LAUNCH(natgrad_flip_kernel, dim3(gx, (unsigned)nout), 256, 0, douts, LinvT, UinvT);
  for (int i = 0; i < nout; ++i) {   // C = R U^-T (lower x lower)
    const NatOut& o = outs[i];
    GemmArgs g = gargs(R + o.off, o.Mp, UinvT + o.off, o.Mp, Cm + o.off, o.Mp, o.Mp, o.Mp, o.Mp);
    g.a_tri = 1;
    RC(gemm(c, g, false));
  }
  LAUNCH(natgrad_finalize_kernel, nout, 256, 2 * (size_t)maxM * sizeof(double), douts, Cm, gamma, c->d_info);
  return DGP_OK;
}
}  // namespace

int dgp_natgrad_step(dgp_ctx* c, const dgp_model_desc* model, const int* layer_ids, int n_layers, double gamma,
                     const double* grad_flat) {
  if (!c || !model || !layer_ids || n_layers < 0 || !grad_flat) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  return planned(c, [&] { return natgrad_run(c, model, layer_ids, n_layers, gamma, grad_flat); });
}

int dgp_natgrad_pairs(dgp_ctx* c, const dgp_nat_pair* pairs, int n_pairs, double gamma) {
  if (!c || !pairs || n_pairs < 0) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  return planned(c, [&] { return natgrad_pairs_run(c, pairs, n_pairs, gamma); });
}

int dgp_train_nat_adam(dgp_ctx* c, const dgp_model_desc* model, const double* X, const double* Y, int64_t N, int64_t S, double scale,
                       double kl_weight, uint64_t seed0, uint64_t seed_stride, int64_t n_offset, const dgp_adam_param* params,
                       int n_params, double* m_state, double* v_state, int64_t t0, int64_t steps, double lr, double beta1,
                       double beta2, double epsilon, const int* nat_layers, int n_nat, double gamma, double* out_flat,
                       double* elbo_trace) {
  if (!c || !model || !X || !Y || !out_flat || !m_state || !v_state || !nat_layers || t0 < 1 || steps < 0) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  AdamTable tab;
  const bool have_adam = n_params > 0;
  if (have_adam) RC(adam_table(c, params, n_params, tab));
  for (int64_t k = 0; k < steps; ++k) {
    // models/dgp.py:338-343: Adam step on the non-variational parameters, then NaturalGradient.minimize with a FRESH evaluation
    RC(dgp_elbo_grad(c, model, X, Y, N, S, scale, kl_weight, nullptr, seed0 + (uint64_t)(2 * k) * seed_stride, n_offset, 1, out_flat));
    if (have_adam) RC(adam_launch(c, tab, out_flat, m_state, v_state, t0 + k, lr, beta1, beta2, epsilon, elbo_trace ? elbo_trace + k : nullptr));
    else if (elbo_trace) LAUNCH(scale_copy_diff_kernel, 1, 32, 0, out_flat, elbo_trace + k);
    RC(dgp_elbo_grad(c, model, X, Y, N, S, scale, kl_weight, nullptr, seed0 + (uint64_t)(2 * k + 1) * seed_stride, n_offset, 1, out_flat));
    RC(planned(c, [&] { return natgrad_run(c, model, nat_layers, n_nat, gamma, out_flat); }));
  }
  return DGP_OK;
}

int dgp_elbo_grad_host(dgp_ctx* c, const dgp_model_desc* model, const double* X_host, const double* Y_host, int64_t N,
                       int64_t S, double scale, double kl_weight, uint64_t seed, int64_t n_offset, int want_grad,
                       double* out_flat_host) {
  if (!c || !model || !X_host || !Y_host || !out_flat_host || N < 1) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  const int D0 = model->layers[0].D_in, Dy = model->layers[model->num_layers - 1].D_out;
  const int64_t gs = want_grad ? dgp_grad_size(model) : 3;
  const size_t nx = (size_t)N * D0, ny = (size_t)N * Dy;
  const size_t need = (nx + ny + (size_t)gs) * sizeof(double);
  if (c->h_pinned_bytes < need) {
    if (c->h_pinned) CK(cudaFreeHost(c->h_pinned));
    c->h_pinned = nullptr; c->h_pinned_bytes = 0;
    CK(cudaMallocHost(&c->h_pinned, need));
    c->h_pinned_bytes = need;
  }
  // device staging lives outside the arena (the arena may be re-grown by the call below)
  if (c->d_stage_bytes < need) {
    if (c->d_stage) CK(cudaFree(c->d_stage));
    c->d_stage = nullptr; c->d_stage_bytes = 0;
    CK(cudaMalloc(&c->d_stage, need));
    c->d_stage_bytes = need;
  }
  double* d_stage = c->d_stage;
  memcpy(c->h_pinned, X_host, nx * sizeof(double));
  memcpy(c->h_pinned + nx, Y_host, ny * sizeof(double));
  CK(cudaMemcpyAsync(d_stage, c->h_pinned, (nx + ny) * sizeof(double), cudaMemcpyHostToDevice, c->stream));
  double* d_out = d_stage + nx + ny;
  RC(dgp_elbo_grad(c, model, d_stage, d_stage + nx, N, S, scale, kl_weight, nullptr, seed, n_offset, want_grad, d_out));
  CK(cudaMemcpyAsync(c->h_pinned + nx + ny, d_out, (size_t)gs * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  memcpy(out_flat_host, c->h_pinned + nx + ny, (size_t)gs * sizeof(double));
  return check_chol(c);
}

int dgp_predict_moments(dgp_ctx* c, const dgp_model_desc* model, const double* X, int64_t N, int64_t S,
                        const double* const* zs_host, uint64_t seed, int64_t n_offset, int add_lik_var, double* mean, double* var) {
  if (!c || !model || !X || !mean || !var) return DGP_ERR_ARG;
  if (add_lik_var && !model->lik_variance) { c->err = "lik_variance is null"; return DGP_ERR_ARG; }
  RunOpts o;
  o.io.zs = zs_host; o.pm = mean; o.pv = var; o.add_lik = add_lik_var;
  return run_model_planned(c, model, X, N, S, seed, n_offset, o);
}

int dgp_e_log_p_y(dgp_ctx* c, const dgp_model_desc* model, const double* X, const double* Y, int64_t N, int64_t S,
                  const double* const* zs_host, uint64_t seed, int64_t n_offset, double* out) {
  if (!c || !model || !X || !Y || !out) return DGP_ERR_ARG;
  if (!model->lik_variance) { c->err = "lik_variance is null"; return DGP_ERR_ARG; }
  RunOpts o;
  o.io.zs = zs_host; o.ve = out; o.Y = Y; o.Dy = model->layers[model->num_layers - 1].D_out;
  return run_model_planned(c, model, X, N, S, seed, n_offset, o);
}

int dgp_ei(dgp_ctx* c, const dgp_model_desc* model, const double* X, int64_t N, int64_t S, const double* const* zs_host,
           uint64_t seed, int64_t n_offset, double y_min, int analytic, double* neg_ei) {
  if (!c || !model || !X || !neg_ei) return DGP_ERR_ARG;
  RunOpts o;
  o.io.zs = zs_host; o.ei = neg_ei; o.y_min = y_min; o.ei_analytic = analytic; o.need_last_sample = !analytic;
  return run_model_planned(c, model, X, N, S, seed, n_offset, o);
}

int dgp_ei_grad(dgp_ctx* c, const dgp_model_desc* model, const double* X, int64_t N, int64_t S, const double* const* zs_host,
                uint64_t seed, int64_t n_offset, double y_min, double* neg_ei, double* d_neg_ei_dX) {
  return dgp_acq_grad(c, model, 0, X, N, S, zs_host, seed, n_offset, y_min, neg_ei, d_neg_ei_dX);
}

int dgp_acq_grad(dgp_ctx* c, const dgp_model_desc* model, int kind, const double* X, int64_t N, int64_t S,
                 const double* const* zs_host, uint64_t seed, int64_t n_offset, double y, double* value, double* d_value_dX) {
  if (!c || !model || !X || !value || !d_value_dX || kind < 0 || kind > 4) return DGP_ERR_ARG;
  const bool add_lik = kind == 4 ? y != 0.0 : kind > 0;
  if (add_lik && !model->lik_variance) { c->err = "lik_variance is null"; return DGP_ERR_ARG; }
  if (kind == 3 && model->layers[model->num_layers - 1].D_out != 1) { c->err = "WB2S expects a single-output model"; return DGP_ERR_ARG; }
  RunOpts o;
  o.io.zs = zs_host; o.ei = value; o.y_min = y; o.ei_analytic = 1; o.dx = d_value_dX;
  o.acq_kind = kind; o.acq_add_lik = add_lik ? 1 : 0;
  return run_model_planned(c, model, X, N, S, seed, n_offset, o);
}

int dgp_acq_moments(dgp_ctx* c, int kind, const double* mean, const double* var, int64_t n, double y, const double* x, int d,
                    double* out) {
  if (!c || !mean || !var || !out || n < 1 || kind < 0 || kind > 4 || (kind == 3 && (!x || d < 1))) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  LAUNCH(acq_moments_kernel, (unsigned)((n + 255) / 256), 256, 0, kind, mean, var, (long)n, y, x, d, out);
  return DGP_OK;
}

int dgp_de_propose(dgp_ctx* c, const double* pop_u, int64_t pop, int d, const double* lw, const double* up, uint64_t seed,
                   int64_t generation, double weight, double crossover, double* cand_u, double* cand_x) {
  if (!c || !pop_u || !lw || !up || !cand_u || !cand_x || d < 1 || generation < 0) return DGP_ERR_ARG;
  if (pop < 4) { c->err = "differential evolution needs a population of at least 4"; return DGP_ERR_ARG; }
  CK(cudaSetDevice(c->device));
  CAT(DGP_CAT_OTHER);
  LAUNCH(de_propose_kernel, (unsigned)((pop * d + 127) / 128), 128, 0, pop_u, (long)pop, d, lw, up, (unsigned long long)seed,
         (const unsigned long long*)nullptr, (long)generation, weight, crossover, cand_u, cand_x);
  return DGP_OK;
}

int dgp_de_select(dgp_ctx* c, double* pop_u, double* pop_val, const double* cand_u, const double* cand_val, int64_t pop, int d,
                  int ncol, int first) {
  if (!c || !pop_u || !pop_val || !cand_u || !cand_val || pop < 1 || d < 1 || ncol < 1) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  CAT(DGP_CAT_OTHER);
  LAUNCH(de_select_kernel, (unsigned)((pop + 127) / 128), 128, 0, pop_u, pop_val, cand_u, cand_val, (long)pop, d, ncol, first);
  return DGP_OK;
}

int dgp_box_from_u(dgp_ctx* c, const double* u, const double* lw, const double* up, int64_t n, int d, double* x) {
  if (!c || !u || !lw || !up || !x || n < 1 || d < 1) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  CAT(DGP_CAT_OTHER);
  LAUNCH(box_from_u_kernel, (unsigned)((n * d + 127) / 128), 128, 0, u, lw, up, (long)n, d, x);
  return DGP_OK;
}

int dgp_adam_box_step(dgp_ctx* c, double* u, double* m_state, double* v_state, const double* dx, const double* lw,
                      const double* up, int64_t n, int d, int64_t t, double lr, double beta1, double beta2, double epsilon, double* x) {
  if (!c || !u || !m_state || !v_state || !dx || !lw || !up || !x || n < 1 || d < 1 || t < 1) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  CAT(DGP_CAT_OTHER);
  const double lr_t = lr * sqrt(1.0 - pow(beta2, (double)t)) / (1.0 - pow(beta1, (double)t));
  LAUNCH(adam_box_kernel, (unsigned)((n * d + 127) / 128), 128, 0, u, m_state, v_state, dx, lw, up, (long)n, d, lr_t, beta1, beta2,
         epsilon, x);
  return DGP_OK;
}

int dgp_ev_mc(dgp_ctx* c, const double* F, int64_t S, int64_t ND, double zero_c, double* out) {
  if (!c || !F || !out || S < 1 || ND < 1) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  LAUNCH(ev_mc_kernel, (unsigned)((ND + 255) / 256), 256, 0, F, (long)S, (long)ND, zero_c, out);
  return DGP_OK;
}

int dgp_mixture_moments(dgp_ctx* c, const double* Fmean, const double* Fvar, int64_t S, int64_t ND, const double* lik_variance,
                        double* mean, double* var) {
  if (!c || !Fmean || !Fvar || !mean || !var || S < 1 || ND < 1) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  LAUNCH(mixture_moments_kernel, (unsigned)((ND + 255) / 256), 256, 0, Fmean, Fvar, (long)S, (long)ND, lik_variance,
         lik_variance ? 1 : 0, mean, var);
  return DGP_OK;
}

int dgp_ehvi2d(dgp_ctx* c, const double* m0, const double* v0, const double* m1, const double* v1, int64_t N, const double* ynd0,
               const double* ynd1, int n, double* out) {
  if (!c || !m0 || !v0 || !m1 || !v1 || !ynd0 || !ynd1 || !out || N < 1 || n < 2 || n > 2048) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  LAUNCH(ehvi2d_kernel, (unsigned)((N + 127) / 128), 128, 2 * (size_t)n * sizeof(double), m0, v0, m1, v1, (long)N, ynd0, ynd1, n, out);
  return DGP_OK;
}

int dgp_ehvi2d_grad(dgp_ctx* c, const double* m0, const double* v0, const double* m1, const double* v1, int64_t N, const double* ynd0,
                    const double* ynd1, int n, double* out, double* grads) {
  if (!c || !m0 || !v0 || !m1 || !v1 || !ynd0 || !ynd1 || !out || !grads || N < 1 || n < 2 || n > 2048) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  LAUNCH(ehvi2d_grad_kernel, (unsigned)((N + 127) / 128), 128, 2 * (size_t)n * sizeof(double), m0, v0, m1, v1, (long)N, ynd0, ynd1, n, out,
         grads);
  return DGP_OK;
}

int dgp_debug_gemm(dgp_ctx* c, int nt, int M, int N, int K, double alpha, const double* A, const double* B, double beta,
                   double* C, int a_tri, int c_lower, int batch, int splitk, const double* kscale) {
  if (!c) return DGP_ERR_ARG;
  CK(cudaSetDevice(c->device));
  GemmArgs g = gargs(A, K, B, nt ? K : N, C, N, M, N, K);
  g.alpha = alpha; g.beta = beta; g.a_tri = a_tri; g.c_lower = c_lower; g.batch = batch < 1 ? 1 : batch;
  g.sA = (long)M * K; g.sB = nt ? (long)N * K : (long)K * N; g.sC = (long)M * N;
  g.kscale = kscale; g.sScale = K;
  g.splitk = splitk < 1 ? 1 : splitk;
  if (g.splitk > 1) {
    RC(ensure_ws(c, (size_t)g.splitk * g.batch * M * N * sizeof(double)));
    g.part = reinterpret_cast<double*>(c->ws);
  }
  return gemm(c, g, nt != 0);
}

}  // extern "C"
