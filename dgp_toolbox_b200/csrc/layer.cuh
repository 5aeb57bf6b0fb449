// Streaming kernels of the SVGP-layer conditional and its adjoint (SURVEY §8 a2-a8, §9).
// Layouts: inducing-major matrices are [Mp][Pp] row-major (point-sample index contiguous, both padded with zeros);
// point-major arrays are [P][D]. Point-sample index p = s * N + n (dgp_dace/utils/layers.py:82-85).
#pragma once
#include "common.cuh"
#include "philox.cuh"

namespace dgp {

// ---------------------------------------------------------------------------------------------------------
// a2: Kuf[m][p] = s2 * exp(-0.5 * sum_j ((z_mj - x_pj)/l_j)^2)   (covs.Kuf, utils/layers.py:243)
// X row of point-sample p is X[(p % xmod) * D + j]: layer 0 shares X over the S samples (models/dgp.py:49).
// ---------------------------------------------------------------------------------------------------------
constexpr int kKufCols = 128, kKufRows = 32;
__global__ void __launch_bounds__(256) kuf_kernel(const double* __restrict__ X, long xmod, const double* __restrict__ Z,
                                                  const double* __restrict__ ls, const double* __restrict__ var, int M, int Mp,
                                                  int D, long P, long Pp, double* __restrict__ K, int kind) {
  __shared__ double xs[kMaxD][kKufCols];
  __shared__ double zs[kKufRows][kMaxD + 1];
  __shared__ double il[kMaxD];
  const long p0 = (long)blockIdx.x * kKufCols;
  const int m0 = blockIdx.y * kKufRows;
  const int tid = threadIdx.x;
  if (tid < D) il[tid] = 1.0 / ls[tid];
  __syncthreads();
  for (int i = tid; i < kKufCols * D; i += 256) {
    int c = i / D, j = i % D;
    long p = p0 + c;
    xs[j][c] = (p < P) ? X[(p % xmod) * D + j] * il[j] : 0.0;
  }
  for (int i = tid; i < kKufRows * D; i += 256) {
    int r = i / D, j = i % D;
    zs[r][j] = (m0 + r < M) ? Z[(long)(m0 + r) * D + j] * il[j] : 0.0;
  }
  __syncthreads();
  const int c = tid & 127, rh = tid >> 7;
  const long p = p0 + c;
  const double s2 = var[0];
  for (int r = rh; r < kKufRows; r += 2) {
    double r2 = 0.0;
    for (int j = 0; j < D; ++j) {
      double t = zs[r][j] - xs[j][c];
      r2 = fma(t, t, r2);
    }
    double k = (m0 + r < M && p < P) ? kernel_value(kind, r2, s2) : 0.0;
    if (m0 + r < Mp && p < Pp) K[(long)(m0 + r) * Pp + p] = k;
  }
}

// ---------------------------------------------------------------------------------------------------------
// a3/a4/a6 epilogue: mean = A^T q_mu + mf(x), var = s2 - |V|^2 + sum_m T_d^2 (T_d = R_d^T A), F = mean + z sqrt(var + jitter)
// (utils/layers.py:249,271-278; utils/utils.py:40-41). One thread per point-sample, loop over inducing rows.
// Chunk-local index p = s * Nc + n; caller-visible arrays are [S][N_total][D] and use row s * N_total + n0 + n.
// ---------------------------------------------------------------------------------------------------------
struct MomentsArgs {
  const double* V; const double* A; const double* T;  // [Mp][Pp], [Mp][Pp], [D_out][Mp][Pp]
  const double* qmu;                                   // [M][D_out]
  const double* var;                                   // kernel variance
  const double* Xin; long xmod; int D_in;              // layer input (for the mean function)
  const double* mfW; const double* mfb; int mean_kind; // 0 zero, 1 identity, 2 linear
  const double* z_in;                                  // caller [S][N_total][D_out] or null -> Philox
  unsigned long long seed; const unsigned long long* seed_ptr; int layer; long Nc; long N_total; long n0; long n_offset;
  int M, Mp, D_out; long P, Pp;
  double jitter;
  double* Fmean; double* Fvar; double* F; double* z;       // chunk-local [P][D_out]; F / z may be null
  double* xFmean; double* xFvar; double* xF;               // caller-visible (global row mapping), any may be null
};

template <int DMAX>
__global__ void __launch_bounds__(128) moments_kernel(MomentsArgs a) {
  extern __shared__ double qs[];  // [M][D_out]
  for (int i = threadIdx.x; i < a.M * a.D_out; i += blockDim.x) qs[i] = a.qmu[i];
  __syncthreads();
  const long p = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= a.P) return;
  double mean[DMAX], del[DMAX], v2 = 0.0;
#pragma unroll
  for (int d = 0; d < DMAX; ++d) { mean[d] = 0.0; del[d] = 0.0; }
  const long plane = (long)a.Mp * a.Pp;
  for (int m = 0; m < a.M; ++m) {
    const long off = (long)m * a.Pp + p;
    const double v = a.V[off], am = a.A[off];
    v2 = fma(v, v, v2);
#pragma unroll
    for (int d = 0; d < DMAX; ++d)
      if (d < a.D_out) {
        const double t = a.T[(long)d * plane + off];
        mean[d] = fma(am, qs[m * a.D_out + d], mean[d]);
        del[d] = fma(t, t, del[d]);
      }
  }
  const double s2 = a.var[0];
  const double* x = a.Xin + (p % a.xmod) * a.D_in;
  const long s = p / a.Nc, n = p % a.Nc;
  const long xrow = s * a.N_total + a.n0 + n;
#pragma unroll
  for (int d = 0; d < DMAX; ++d)
    if (d < a.D_out) {
      double mf = 0.0;
      if (a.mean_kind == 1) mf = x[d];
      else if (a.mean_kind == 2) {
        for (int j = 0; j < a.D_in; ++j) mf = fma(x[j], a.mfW[j * a.D_out + d], mf);
        if (a.mfb) mf += a.mfb[d];
      }
      const double mu = mean[d] + mf;
      const double var = s2 - v2 + del[d];
      a.Fmean[p * a.D_out + d] = mu;
      a.Fvar[p * a.D_out + d] = var;
      if (a.xFmean) a.xFmean[xrow * a.D_out + d] = mu;
      if (a.xFvar) a.xFvar[xrow * a.D_out + d] = var;
      if (a.F) {
        const double z = a.z_in ? a.z_in[xrow * a.D_out + d]
                                : philox_normal(a.seed_ptr ? *a.seed_ptr : a.seed, (uint32_t)a.layer, (uint32_t)s, (uint32_t)(a.n0 + n + a.n_offset), (uint32_t)d);
        if (a.z) a.z[p * a.D_out + d] = z;
        const double f = mu + z * sqrt(var + a.jitter);
        a.F[p * a.D_out + d] = f;
        if (a.xF) a.xF[xrow * a.D_out + d] = f;
      }
    }
}

// ---------------------------------------------------------------------------------------------------------
// First-layer sharing. The first layer's input is X tiled over the S samples (models/dgp.py:49), so its conditional is
// the same for every sample: it is evaluated once per POINT (mean0, var0 [Nc][D]) and expanded here to the S samples,
// where the reparameterised draw F = mean + z sqrt(var + jitter) does differ per sample (utils/utils.py:40-41).
// ---------------------------------------------------------------------------------------------------------
struct ExpandArgs {
  const double* mean0; const double* var0;     // [Nc][D]
  const double* z_in;                          // caller [S][N_total][D] or null -> Philox
  unsigned long long seed; const unsigned long long* seed_ptr; int layer; long Nc; long N_total; long n0; long n_offset; long S; int D;
  double jitter;
  double* F; double* z;                        // chunk-local [S*Nc][D]
  double* xFmean; double* xFvar; double* xF;   // caller-visible, any may be null
};

__global__ void __launch_bounds__(256) expand_first_layer_kernel(ExpandArgs a) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= a.S * a.Nc * a.D) return;
  const int d = (int)(idx % a.D);
  const long p = idx / a.D;
  const long s = p / a.Nc, n = p % a.Nc;
  const double mu = a.mean0[n * a.D + d], var = a.var0[n * a.D + d];
  const long xrow = s * a.N_total + a.n0 + n;
  const double z = a.z_in ? a.z_in[xrow * a.D + d]
                          : philox_normal(a.seed_ptr ? *a.seed_ptr : a.seed, (uint32_t)a.layer, (uint32_t)s, (uint32_t)(a.n0 + n + a.n_offset), (uint32_t)d);
  const double f = mu + z * sqrt(var + a.jitter);
  a.F[idx] = f;
  a.z[idx] = z;
  if (a.xFmean) a.xFmean[xrow * a.D + d] = mu;
  if (a.xFvar) a.xFvar[xrow * a.D + d] = var;
  if (a.xF) a.xF[xrow * a.D + d] = f;
}

// Raw Philox-4x32-10 words of element (layer, s, n, d): the integer plumbing under the normal draws (bit-exact contract).
__global__ void philox_raw_kernel(unsigned long long seed, int layer, long S, long N, int D, long n_offset, uint32_t* out) {
  long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= S * N * D) return;
  int d = (int)(idx % D);
  long r = idx / D;
  long n = r % N, s = r / N;
  uint32_t w[4];
  philox4x32_10((uint32_t)(n + n_offset), (uint32_t)s, (uint32_t)d, (uint32_t)layer, (uint32_t)seed, (uint32_t)(seed >> 32), w);
  for (int k = 0; k < 4; ++k) out[idx * 4 + k] = w[k];
}

// Philox draws written out for the oracle / explicit-z callers.
__global__ void philox_normal_kernel(unsigned long long seed, int layer, long S, long N, int D, long n_offset, double* z) {
  long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= S * N * D) return;
  int d = (int)(idx % D);
  long r = idx / D;
  long n = r % N, s = r / N;
  z[idx] = philox_normal(seed, (uint32_t)layer, (uint32_t)s, (uint32_t)(n + n_offset), (uint32_t)d);
}

// ---------------------------------------------------------------------------------------------------------
// a8: Gaussian variational expectations + upstream adjoints of the last layer (utils/utils.py:89-93, models/dgp.py:79-100)
// ve = -0.5 log 2pi - 0.5 log sn2 - 0.5 ((Y - mu)^2 + var)/sn2 ; data term = (scale/S) sum ve.
// Writes per-block partial sums: part[block][0] = data term, [1] = d/d sn2, [2] = sum Gv.
// ---------------------------------------------------------------------------------------------------------
struct UpstreamOut {
  double* Gm;     // [Pp][D]   (rows >= P are zero)
  double* GvT;    // [D][Pp]
  double* GmPad;  // [Pp][32]
  double* gq;     // [Pp]  = -sum_d Gv
  double* part;   // [blocks][3]
};

__global__ void __launch_bounds__(128) likelihood_kernel(const double* __restrict__ Fmean, const double* __restrict__ Fvar,
                                                         const double* __restrict__ Y, const double* __restrict__ likvar,
                                                         long N, long P, long Pp, int D, double coef, int want_grad, UpstreamOut o) {
  __shared__ double red[32];
  const long p = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const double sn2 = likvar[0];
  double ve = 0.0, dsn = 0.0, sgv = 0.0;
  if (p < Pp) {
    double gq = 0.0;
    const long n = p % N;
    for (int d = 0; d < D; ++d) {
      double gm = 0.0, gv = 0.0;
      if (p < P) {
        const double mu = Fmean[p * D + d], var = Fvar[p * D + d];
        const double r = Y[n * D + d] - mu;
        const double q = fma(r, r, var);
        ve += -0.91893853320467274178 - 0.5 * log(sn2) - 0.5 * q / sn2;
        dsn += -0.5 / sn2 + 0.5 * q / (sn2 * sn2);
        gm = coef * r / sn2;
        gv = -0.5 * coef / sn2;
      }
      if (want_grad) {
        o.Gm[p * D + d] = gm;
        o.GvT[(long)d * Pp + p] = gv;
        o.GmPad[p * 32 + d] = gm;
        gq -= gv;
        sgv += gv;
      }
    }
    if (want_grad) {
      for (int d = D; d < 32; ++d) o.GmPad[p * 32 + d] = 0.0;
      o.gq[p] = gq;
    }
  }
  double t0 = block_sum(ve * coef, red);
  double t1 = block_sum(dsn * coef, red);
  double t2 = block_sum(sgv, red);
  if (threadIdx.x == 0) {
    o.part[(long)blockIdx.x * 3 + 0] = t0;
    o.part[(long)blockIdx.x * 3 + 1] = t1;
    o.part[(long)blockIdx.x * 3 + 2] = t2;
  }
}

// DGP_Base.E_log_p_Y (models/dgp.py:79-87): mean over the S samples of the Gaussian variational expectations
// (utils/utils.py:89-93), one value per point and output. Chunk-local moments [S * Nc][D] with p = s * Nc + n.
__global__ void __launch_bounds__(256) ve_mean_kernel(const double* __restrict__ Fmean, const double* __restrict__ Fvar,
                                                      const double* __restrict__ Y, const double* __restrict__ likvar, long Nc,
                                                      long S, int D, double* __restrict__ out) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= Nc * D) return;
  const double sn2 = likvar[0], y = Y[idx];
  const double c0 = -0.91893853320467274178 - 0.5 * log(sn2);
  double acc = 0.0;
  for (long s = 0; s < S; ++s) {
    const double r = y - Fmean[s * Nc * D + idx];
    acc += c0 - 0.5 * fma(r, r, Fvar[s * Nc * D + idx]) / sn2;
  }
  out[idx] = acc / (double)S;
}

// Hidden layer: G_F = d ELBO / d F (the next layer's input gradient); F = mean + z sqrt(var + jitter)
//   Gm = G_F, Gv = G_F z / (2 sqrt(var + jitter))          (adjoint of utils/utils.py:40-41)
__global__ void __launch_bounds__(128) upstream_kernel(const double* __restrict__ GF, const double* __restrict__ z,
                                                       const double* __restrict__ Fvar, long P, long Pp, int D, double jitter,
                                                       UpstreamOut o) {
  __shared__ double red[32];
  const long p = (long)blockIdx.x * blockDim.x + threadIdx.x;
  double sgv = 0.0;
  if (p < Pp) {
    double gq = 0.0;
    for (int d = 0; d < D; ++d) {
      double gm = 0.0, gv = 0.0;
      if (p < P) {
        gm = GF[p * D + d];
        gv = gm * z[p * D + d] / (2.0 * sqrt(Fvar[p * D + d] + jitter));
      }
      o.Gm[p * D + d] = gm;
      o.GvT[(long)d * Pp + p] = gv;
      o.GmPad[p * 32 + d] = gm;
      gq -= gv;
      sgv += gv;
    }
    for (int d = D; d < 32; ++d) o.GmPad[p * 32 + d] = 0.0;
    o.gq[p] = gq;
  }
  double t2 = block_sum(sgv, red);
  if (threadIdx.x == 0) {
    o.part[(long)blockIdx.x * 3 + 0] = 0.0;
    o.part[(long)blockIdx.x * 3 + 1] = 0.0;
    o.part[(long)blockIdx.x * 3 + 2] = t2;
  }
}

// First-layer sharing, adjoint side: the per-point upstream gradients are the sums over the S samples,
//   Gm[n] = sum_s G_F[s,n],  Gv[n] = sum_s G_F[s,n] z[s,n] / (2 sqrt(var0[n] + jitter)).
__global__ void __launch_bounds__(128) upstream_reduce_kernel(const double* __restrict__ GF, const double* __restrict__ z,
                                                              const double* __restrict__ var0, long Nc, long S, long Pp0, int D,
                                                              double jitter, UpstreamOut o) {
  __shared__ double red[32];
  const long n = (long)blockIdx.x * blockDim.x + threadIdx.x;
  double sgv = 0.0;
  if (n < Pp0) {
    double gq = 0.0;
    for (int d = 0; d < D; ++d) {
      double gm = 0.0, gv = 0.0;
      if (n < Nc) {
        double gz = 0.0;
        for (long s = 0; s < S; ++s) {
          const double g = GF[(s * Nc + n) * D + d];
          gm += g;
          gz = fma(g, z[(s * Nc + n) * D + d], gz);
        }
        gv = gz / (2.0 * sqrt(var0[n * D + d] + jitter));
      }
      o.Gm[n * D + d] = gm;
      o.GvT[(long)d * Pp0 + n] = gv;
      o.GmPad[n * 32 + d] = gm;
      gq -= gv;
      sgv += gv;
    }
    for (int d = D; d < 32; ++d) o.GmPad[n * 32 + d] = 0.0;
    o.gq[n] = gq;
  }
  double t2 = block_sum(sgv, red);
  if (threadIdx.x == 0) {
    o.part[(long)blockIdx.x * 3 + 0] = 0.0;
    o.part[(long)blockIdx.x * 3 + 1] = 0.0;
    o.part[(long)blockIdx.x * 3 + 2] = t2;
  }
}

// ---------------------------------------------------------------------------------------------------------
// RBF adjoint on the Kuf block (SURVEY §9): dK = W + 2 A diag(g_q); Gbar = dK o K;
//   Wg = W + A diag(g_q) (in place over W, feeds dKu = -Wg A^T); Gbar stored for dZ = -(z r - Gbar [X,1])/l^2;
//   dX[p][j] = sum_m Gbar (z_mj - x_pj)/l_j^2 (+ mean-function path); dl_j = sum Gbar (z-x)^2/l^3; ds2 = sum Gbar/s2.
// One thread per point-sample column, all inducing rows in a loop; per-block partials [blocks][D_in + 1].
// ---------------------------------------------------------------------------------------------------------
struct RbfBwdArgs {
  double* W;            // [Mp][Pp] in: W, out: Wg      (V-form, A == null: in: K-bar = dELBO/dKuf, left untouched)
  const double* A;      // [Mp][Pp] or null
  const double* gq;     // [Pp]
  double* Gbar;         // [Mp][Pp] out
  const double* Xin; long xmod; const double* Z; const double* ls; const double* var;
  int M, Mp, D_in; long P, Pp;
  const double* Gm; int D_out; int mean_kind; const double* mfW;   // mean-function path
  int kind;             // kernel kind (common.cuh: kernel_eval)
  double* dXin;         // [P][D_in] or null (layer 0)
  double* XaugPad;      // [Pp][32]: [x, 1, 0...]
  double* part;         // [blocks][D_in + 1]
};

constexpr int kRbfCols = 64, kRbfRowGroups = 4;   // 256 threads: 64 point-sample columns x 4 interleaved row groups
inline size_t rbf_bwd_smem_bytes(int M, int D_in) {
  return ((size_t)M * D_in + kMaxD + 32 + (size_t)kRbfRowGroups * kRbfCols * D_in) * sizeof(double);
}
// dynamic shared memory both kernel-adjoint variants opt into. The one-thread-per-column kernel needs at most
// (768 * 31 + 64) * 8 B = 186.5 KiB; the row-group kernel's extra partial sums do not fit with large M * D_in (M = 640,
// D_in = 31 needs 217.5 KiB), and such layers take the one-thread-per-column kernel at any size.
constexpr size_t kRbfBwdSmemMax = 200 * 1024;

// Small launches (fewer blocks than two waves of the one-thread-per-column kernel below): latency-bound, so each thread walks
// every 4th inducing row of its column and the row groups' partial input gradients are summed through shared memory.
template <int DMAX, bool VF>   // VF: V-form (no A plane, K-bar read-only)
__global__ void __launch_bounds__(256) rbf_bwd2d_kernel(RbfBwdArgs a) {
  extern __shared__ double sh[];
  double* zs = sh;                         // [M][D_in]  (unscaled)
  double* il = zs + (long)a.M * a.D_in;    // [D_in] 1/l
  double* red = il + kMaxD;                // [32]
  double* dxs = red + 32;                  // [row groups][cols][D_in] partial input gradients
  for (int i = threadIdx.x; i < a.M * a.D_in; i += blockDim.x) zs[i] = a.Z[i];
  if (threadIdx.x < a.D_in) il[threadIdx.x] = 1.0 / a.ls[threadIdx.x];
  __syncthreads();
  const int cl = threadIdx.x & (kRbfCols - 1), rg = threadIdx.x / kRbfCols;
  const long p = (long)blockIdx.x * kRbfCols + cl;  // < Pp
  const bool live = p < a.P;
  double x[DMAX], dx[DMAX], dl[DMAX], ds2 = 0.0;
#pragma unroll
  for (int j = 0; j < DMAX; ++j) {
    x[j] = (live && j < a.D_in) ? a.Xin[(p % a.xmod) * a.D_in + j] : 0.0;
    dx[j] = 0.0;
    dl[j] = 0.0;
  }
  const double s2 = a.var[0];
  const double g = a.gq[p];
  // each thread walks every 4th inducing row of its column (4x the parallelism of one thread per column: the loop is
  // latency-bound), in groups of 4 rows with all plane loads of a group issued up front (W is updated in place, so the
  // compiler cannot hoist the next rows' loads above the stores on its own)
  for (int mb = 0; mb < a.M; mb += 4 * kRbfRowGroups) {
    double wv[4], av[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int m = mb + u * kRbfRowGroups + rg;
      const long off = (long)m * a.Pp + p;
      wv[u] = (m < a.M) ? a.W[off] : 0.0;
      av[u] = (!VF && m < a.M) ? a.A[off] : 0.0;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int m = mb + u * kRbfRowGroups + rg;
      if (m < a.M) {
        const long off = (long)m * a.Pp + p;
        const double w = wv[u], am = av[u];
        double r2 = 0.0, t[DMAX];
#pragma unroll
        for (int j = 0; j < DMAX; ++j)
          if (j < a.D_in) {
            t[j] = (zs[m * a.D_in + j] - x[j]) * il[j];
            r2 = fma(t[j], t[j], r2);
          }
        double k = 0.0, gf = 0.0;
        if (live) kernel_eval(a.kind, r2, s2, k, gf);
        const double kbar = VF ? w : w + 2.0 * am * g;   // dELBO / dKuf[m][p]
        const double gb = kbar * gf;            // K-bar times -2 dk/d(r2): drives dX, dZ, dl
        if (!VF) a.W[off] = w + am * g;
        a.Gbar[off] = gb;
        ds2 += kbar * k;                        // d/d s2 = sum K-bar K / s2
#pragma unroll
        for (int j = 0; j < DMAX; ++j)
          if (j < a.D_in) {
            dx[j] = fma(gb * t[j], il[j], dx[j]);       // Gbar (z-x)/l^2
            dl[j] = fma(gb * t[j] * t[j], il[j], dl[j]);  // Gbar (z-x)^2/l^3
          }
      }
    }
  }
  // input gradient of the column: sum of the row groups' partials in a fixed order
#pragma unroll
  for (int j = 0; j < DMAX; ++j)
    if (j < a.D_in) dxs[((size_t)rg * kRbfCols + cl) * a.D_in + j] = dx[j];
  __syncthreads();
  if (rg == 0) {
#pragma unroll
    for (int j = 0; j < DMAX; ++j)
      if (j < a.D_in) {
        double v = 0.0;
        for (int q = 0; q < kRbfRowGroups; ++q) v += dxs[((size_t)q * kRbfCols + cl) * a.D_in + j];
        dx[j] = v;
      }
    if (p < a.Pp) {
#pragma unroll
      for (int j = 0; j < DMAX; ++j)
        if (j < a.D_in) a.XaugPad[p * 32 + j] = x[j];
      for (int j = a.D_in; j < 32; ++j) a.XaugPad[p * 32 + j] = (j == a.D_in && live) ? 1.0 : 0.0;
    }
    if (a.dXin && live) {
#pragma unroll
      for (int j = 0; j < DMAX; ++j)
        if (j < a.D_in) {
          double v = dx[j];
          if (a.mean_kind == 1) v += a.Gm[p * a.D_out + j];
          else if (a.mean_kind == 2) {
            for (int d = 0; d < a.D_out; ++d) v = fma(a.Gm[p * a.D_out + d], a.mfW[j * a.D_out + d], v);
          }
          a.dXin[p * a.D_in + j] = v;
        }
    }
  }
  for (int j = 0; j < a.D_in; ++j) {
    double v = 0.0;
#pragma unroll
    for (int jj = 0; jj < DMAX; ++jj)
      if (jj == j) v = dl[jj];
    double r = block_sum(v, red);
    if (threadIdx.x == 0) a.part[(long)blockIdx.x * (a.D_in + 1) + j] = r;
  }
  double r = block_sum(ds2 / s2, red);
  if (threadIdx.x == 0) a.part[(long)blockIdx.x * (a.D_in + 1) + a.D_in] = r;
}

// Large launches: one thread per point-sample column (bandwidth-friendlier 1 KB row segments per block).
template <int DMAX, bool VF>   // VF: V-form (no A plane, K-bar read-only)
__global__ void __launch_bounds__(128) rbf_bwd_kernel(RbfBwdArgs a) {
  extern __shared__ double sh[];
  double* zs = sh;                         // [M][D_in]  (unscaled)
  double* il = zs + (long)a.M * a.D_in;    // [D_in] 1/l
  double* red = il + kMaxD;                // [32]
  for (int i = threadIdx.x; i < a.M * a.D_in; i += blockDim.x) zs[i] = a.Z[i];
  if (threadIdx.x < a.D_in) il[threadIdx.x] = 1.0 / a.ls[threadIdx.x];
  __syncthreads();
  const long p = (long)blockIdx.x * blockDim.x + threadIdx.x;  // < Pp
  const bool live = p < a.P;
  double x[DMAX], dx[DMAX], dl[DMAX], ds2 = 0.0;
#pragma unroll
  for (int j = 0; j < DMAX; ++j) {
    x[j] = (live && j < a.D_in) ? a.Xin[(p % a.xmod) * a.D_in + j] : 0.0;
    dx[j] = 0.0;
    dl[j] = 0.0;
  }
  const double s2 = a.var[0];
  const double g = a.gq[p];
  // rows in groups of 4 with all eight plane loads of a group issued up front: W is updated in place, so the compiler
  // cannot hoist the next rows' loads above the stores on its own, and one row at a time is latency-bound
  for (int m0 = 0; m0 < a.M; m0 += 4) {
    double wv[4], av[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const long off = (long)(m0 + u) * a.Pp + p;
      wv[u] = (m0 + u < a.M) ? a.W[off] : 0.0;
      av[u] = (!VF && m0 + u < a.M) ? a.A[off] : 0.0;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int m = m0 + u;
      if (m < a.M) {
        const long off = (long)m * a.Pp + p;
        const double w = wv[u], am = av[u];
        double r2 = 0.0, t[DMAX];
#pragma unroll
        for (int j = 0; j < DMAX; ++j)
          if (j < a.D_in) {
            t[j] = (zs[m * a.D_in + j] - x[j]) * il[j];
            r2 = fma(t[j], t[j], r2);
          }
        double k = 0.0, gf = 0.0;
        if (live) kernel_eval(a.kind, r2, s2, k, gf);
        const double kbar = VF ? w : w + 2.0 * am * g;   // dELBO / dKuf[m][p]
        const double gb = kbar * gf;            // K-bar times -2 dk/d(r2): drives dX, dZ, dl
        if (!VF) a.W[off] = w + am * g;
        a.Gbar[off] = gb;
        ds2 += kbar * k;                        // d/d s2 = sum K-bar K / s2
#pragma unroll
        for (int j = 0; j < DMAX; ++j)
          if (j < a.D_in) {
            dx[j] = fma(gb * t[j], il[j], dx[j]);       // Gbar (z-x)/l^2
            dl[j] = fma(gb * t[j] * t[j], il[j], dl[j]);  // Gbar (z-x)^2/l^3
          }
      }
    }
  }
  if (p < a.Pp) {
#pragma unroll
    for (int j = 0; j < DMAX; ++j)
      if (j < a.D_in) a.XaugPad[p * 32 + j] = x[j];
    for (int j = a.D_in; j < 32; ++j) a.XaugPad[p * 32 + j] = (j == a.D_in && live) ? 1.0 : 0.0;
  }
  if (a.dXin && live) {
#pragma unroll
    for (int j = 0; j < DMAX; ++j)
      if (j < a.D_in) {
        double v = dx[j];
        if (a.mean_kind == 1) v += a.Gm[p * a.D_out + j];
        else if (a.mean_kind == 2) {
          for (int d = 0; d < a.D_out; ++d) v = fma(a.Gm[p * a.D_out + d], a.mfW[j * a.D_out + d], v);
        }
        a.dXin[p * a.D_in + j] = v;
      }
  }
  for (int j = 0; j < a.D_in; ++j) {
    double v = 0.0;
#pragma unroll
    for (int jj = 0; jj < DMAX; ++jj)
      if (jj == j) v = dl[jj];
    double r = block_sum(v, red);
    if (threadIdx.x == 0) a.part[(long)blockIdx.x * (a.D_in + 1) + j] = r;
  }
  double r = block_sum(ds2 / s2, red);
  if (threadIdx.x == 0) a.part[(long)blockIdx.x * (a.D_in + 1) + a.D_in] = r;
}

// out[c] = sum_b part[b][c]   -- one block per column, fixed-order tree (deterministic).
__global__ void __launch_bounds__(256) reduce_partials_kernel(const double* __restrict__ part, long nblocks, int ldp,
                                                              double* __restrict__ out, int accumulate) {
  __shared__ double red[32];
  const int c = blockIdx.x;
  double s = 0.0;
  for (long b = threadIdx.x; b < nblocks; b += blockDim.x) s += part[b * ldp + c];
  double r = block_sum(s, red);
  if (threadIdx.x == 0) out[c] = accumulate ? out[c] + r : r;
}

}  // namespace dgp
