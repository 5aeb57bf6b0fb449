// full_cov=True branches of the layer conditional and of the reparameterisation (SURVEY §8 f4):
//   conditional_SND's per-sample map (utils/layers.py:76-80), A_tiled^T B + kern.K(X) (:264-268), tf.transpose (:276),
//   reparameterize with chol(var + jitter I) per sample and output (utils/utils.py:43-52).
// In the V-form planes the forward kernel stashes (V = Lu^-1 Kuf [Mp][Pp], T_d = C_d V [D][Mp][Pp], columns p = s N + n):
//   cov_{s,d}[n][n'] = k(x_sn, x_sn') - sum_m V[m][sN+n] V[m][sN+n'] + sum_m T_d[m][sN+n] T_d[m][sN+n'].
// The N x N blocks are small (N <= 768: one CTA factorises a block), so the Gram products run as shared-memory tiled FP64 FMAs.
// The supplied-matrix path (dgp_svgp_from_k_full_cov) builds the same Gram on its A-form planes (V = Lu^-1 Kuf, T_d = q_sqrt_d^T A,
// so T_d^T T_d = A^T q_sqrt_d q_sqrt_d^T A and V^T V = A^T Ku A) with the k term read from the caller's Kff: fullcov_ext_kernel.
#pragma once
#include "common.cuh"

namespace dgp {

struct FullCovArgs {
  const double* V; const double* T;       // [Mp][Pp], [D][Mp][Pp]
  const double* Xin; long xmod; int D_in; // layer input rows (p % xmod)
  const double* ls; const double* var; int kind;
  int Mp, D; long N, Np, Pp; int S;
  double jitter;
  double* var_out;                        // caller [S][N][N][D] or null
  double* chol_in;                        // [S * D][Np][Np]: cov + jitter I, identity on the padding
};

constexpr int kFcTile = 32;

// One 32 x 32 tile of a covariance block. The K term is the layer's stationary kernel on the input rows, or (EXT) the caller's
// block Kff[s * kff_stride + i * N + j] (the supplied-matrix path: dgp_svgp_from_k_full_cov).
template <bool EXT>
__device__ __forceinline__ void fullcov_tile(const FullCovArgs& a, const double* __restrict__ Kff, long kff_stride) {
  __shared__ double vi[kFcTile][kFcTile + 1], vj[kFcTile][kFcTile + 1], ti[kFcTile][kFcTile + 1], tj[kFcTile][kFcTile + 1];
  const int s = blockIdx.z / a.D, d = blockIdx.z % a.D;
  const int i0 = blockIdx.y * kFcTile, j0 = blockIdx.x * kFcTile;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // ty in 0..7: rows ty, ty + 8, ...
  const double* Td = a.T + (long)d * a.Mp * a.Pp;
  const long c0 = (long)s * a.N;
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  for (int m0 = 0; m0 < a.Mp; m0 += kFcTile) {
    for (int r = ty; r < kFcTile; r += 8) {   // [m][column] tiles, coalesced along the point index
      const long row = (long)(m0 + r) * a.Pp + c0;
      const bool oki = i0 + tx < a.N, okj = j0 + tx < a.N;
      vi[r][tx] = oki ? a.V[row + i0 + tx] : 0.0;
      vj[r][tx] = okj ? a.V[row + j0 + tx] : 0.0;
      ti[r][tx] = oki ? Td[row + i0 + tx] : 0.0;
      tj[r][tx] = okj ? Td[row + j0 + tx] : 0.0;
    }
    __syncthreads();
#pragma unroll 8
    for (int m = 0; m < kFcTile; ++m) {
      const double vjm = vj[m][tx], tjm = tj[m][tx];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int r = ty + 8 * u;
        acc[u] = fma(ti[m][r], tjm, acc[u]);
        acc[u] = fma(-vi[m][r], vjm, acc[u]);
      }
    }
    __syncthreads();
  }
  const int j = j0 + tx;
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int i = i0 + ty + 8 * u;
    double out_pad = (i == j) ? 1.0 : 0.0;
    if (i < a.N && j < a.N) {
      double k;
      if (EXT) {
        k = Kff[(long)s * kff_stride + (long)i * a.N + j];
      } else {
        const double* xi = a.Xin + ((c0 + i) % a.xmod) * a.D_in;
        const double* xj = a.Xin + ((c0 + j) % a.xmod) * a.D_in;
        double r2 = 0.0;
        for (int q = 0; q < a.D_in; ++q) {
          const double t = (xi[q] - xj[q]) / a.ls[q];
          r2 = fma(t, t, r2);
        }
        k = kernel_value(a.kind, r2, a.var[0]);
      }
      const double cov = k + acc[u];
      if (a.var_out) a.var_out[(((long)s * a.N + i) * a.N + j) * a.D + d] = cov;
      out_pad = cov + (i == j ? a.jitter : 0.0);
    }
    if (i < a.Np && j < a.Np) a.chol_in[((long)blockIdx.z * a.Np + i) * a.Np + j] = out_pad;
  }
}

// grid: (Np / 32, Np / 32, S * D); block 32 x 8
__global__ void __launch_bounds__(256) fullcov_kernel(FullCovArgs a) { fullcov_tile<false>(a, nullptr, 0); }

// the same with the K term read from Kff [.][N][N]: kff_stride = N * N (one block per sample) or 0 (one block shared by all)
__global__ void __launch_bounds__(256) fullcov_ext_kernel(FullCovArgs a, const double* __restrict__ Kff, long kff_stride) {
  fullcov_tile<true>(a, Kff, kff_stride);
}

// F[s][n][d] = mean[s][n][d] + sum_{n' <= n} L_{s,d}[n][n'] z[s][n'][d]        (utils/utils.py:50)
__global__ void __launch_bounds__(128) fullcov_sample_kernel(const double* __restrict__ L, const double* __restrict__ mean,
                                                             const double* __restrict__ z, long N, long Np, int D, int S,
                                                             double* __restrict__ F, double* __restrict__ F_user) {
  const int s = blockIdx.y / D, d = blockIdx.y % D;
  const long n = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const double* Lm = L + ((long)blockIdx.y * Np + n) * Np;
  const double* zs = z + (long)s * N * D + d;
  double acc = 0.0;
  for (long k = 0; k <= n; ++k) acc = fma(Lm[k], zs[k * D], acc);
  const long o = ((long)s * N + n) * D + d;
  const double f = mean[o] + acc;
  F[o] = f;
  if (F_user) F_user[o] = f;
}

}  // namespace dgp
