// Grouped full_cov=True (batch acquisition): the N = G q points of a call form G groups of q consecutive points, and every group
// gets what propagate(full_cov=True) gives for those q points alone -- q x q covariance blocks per sample and output and samples
// correlated within the group, independent across groups. On the planes the conditional stashes (fullcov.cuh: V and T_d, columns
// p = s Nc + n) block (g, s, d) is
//   cov[i][j] = k(x_i, x_j) - sum_m V[m][c0 + i] V[m][c0 + j] + sum_m T_d[m][c0 + i] T_d[m][c0 + j],      c0 = s Nc + g q,
// then F = mean + chol(cov + jitter I) z (utils/utils.py:43-52). Blocks are at most 32 x 32: a sub-warp of QW lanes (the power of
// two >= q) owns one (group, sample) pair, lane i = row i. V^T V is formed once per pair and shared by the D outputs; the q x q
// Cholesky and the sample run in registers. The factorisation and the sample are chol_inv_kernel's first 32 x 32 diagonal block
// and fullcov_sample_kernel's sum, operation for operation: on the same block they give the same factor and sample bit for bit.
#pragma once
#include "common.cuh"

namespace dgp {

struct GroupCovArgs {
  const double* V; const double* T;        // [Mp][Pp], [D][Mp][Pp] planes of the chunk (columns p = s Nc + n)
  const double* Xin; long xmod; int D_in;  // layer input rows (p % xmod)
  const double* ls; const double* var; int kind;
  int Mp, D, q; long Nc, Pp, G; int S;     // G groups of q points in the chunk
  double jitter;
  const double* mean;                      // [P][D]
  const double* z; long z_ld;              // z[(s z_ld + n) D + d], n chunk-local; null: no sample
  double* F;                               // [P][D] (the next layer's input)
  double* F_user; long N_total, n0;        // caller [S][N_total][D] or null
  double* cov_user; long G_total, g0;      // caller [S][G_total][q][q][D] or null
  int* info;                               // sticky Cholesky failure flag
};

constexpr int kGcThreads = 128;

// sum over m of x_i x_j for the QW rows of a sub-warp, accumulated into acc[j] of lane i (x = 0 on rows >= q)
template <int QW>
__device__ __forceinline__ void group_gram(const double* __restrict__ plane, long Pp, int Mp, long col, bool row_ok,
                                           double (&acc)[QW]) {
#pragma unroll
  for (int j = 0; j < QW; ++j) acc[j] = 0.0;
  for (int m0 = 0; m0 < Mp; m0 += 4) {   // Mp is a multiple of 64
    double x[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) x[u] = row_ok ? plane[(long)(m0 + u) * Pp + col] : 0.0;
#pragma unroll
    for (int u = 0; u < 4; ++u)
#pragma unroll
      for (int j = 0; j < QW; ++j) acc[j] = fma(x[u], __shfl_sync(0xffffffffu, x[u], j, QW), acc[j]);
  }
}

// grid: ceil(G S / (kGcThreads / QW)) blocks of kGcThreads; pair = s G + g (adjacent groups share a warp: contiguous columns)
template <int QW>
__global__ void __launch_bounds__(kGcThreads, 1) grouped_cov_kernel(GroupCovArgs a) {
  const int lane = threadIdx.x & 31, i = lane & (QW - 1);
  const long pair = ((long)blockIdx.x * kGcThreads + threadIdx.x) / QW;
  const bool pair_ok = pair < a.G * a.S;   // the whole sub-warp agrees; every lane still takes part in the shuffles
  const long g = pair_ok ? pair % a.G : 0, s = pair_ok ? pair / a.G : 0;
  const bool row_ok = pair_ok && i < a.q;
  const long col = s * a.Nc + g * a.q + (row_ok ? i : 0);   // this lane's column of the planes
  // base = K - V^T V (row i), kept in shared memory ([j][thread]: conflict-free) to leave the registers to the T_d Gram and the factor
  __shared__ double base[QW][kGcThreads];
  double c[QW];
  group_gram<QW>(a.V, a.Pp, a.Mp, col, row_ok, c);
  {
    const double* xi = a.Xin + (col % a.xmod) * a.D_in;
    const long c0 = s * a.Nc + g * a.q;
#pragma unroll
    for (int j = 0; j < QW; ++j) {
      double k = 0.0;
      if (row_ok && j < a.q) {   // fullcov_tile's arithmetic: k(x_i, x_j) and k(x_j, x_i) are equal bit for bit
        const double* xj = a.Xin + ((c0 + j) % a.xmod) * a.D_in;
        double r2 = 0.0;
        for (int t = 0; t < a.D_in; ++t) {
          const double u = (xi[t] - xj[t]) / a.ls[t];
          r2 = fma(u, u, r2);
        }
        k = kernel_value(a.kind, r2, a.var[0]);
      }
      base[j][threadIdx.x] = k - c[j];
    }
  }
  for (int d = 0; d < a.D; ++d) {
    group_gram<QW>(a.T + (long)d * a.Mp * a.Pp, a.Pp, a.Mp, col, row_ok, c);
#pragma unroll
    for (int j = 0; j < QW; ++j) c[j] = base[j][threadIdx.x] + c[j];
    if (a.cov_user && row_ok) {
      double* o = a.cov_user + ((((s * a.G_total + a.g0 + g) * a.q + i) * a.q) * a.D + d);
#pragma unroll
      for (int j = 0; j < QW; ++j)
        if (j < a.q) o[(long)j * a.D] = c[j];
    }
    if (!a.z) continue;
    // Cholesky of cov + jitter I, right-looking on the unscaled rows as chol_inv_kernel does (rows >= q: identity padding)
#pragma unroll
    for (int j = 0; j < QW; ++j) c[j] = (i < a.q) ? c[j] + (i == j ? a.jitter : 0.0) : (i == j ? 1.0 : 0.0);
#pragma unroll
    for (int j = 0; j < QW; ++j) {
      if (j < a.q) {   // uniform over the warp (q is the same for every pair)
        const double djj = __shfl_sync(0xffffffffu, c[j], j, QW);
        const double inv = rsqrt(djj);
        if (pair_ok && i == 0 && !(djj > 0.0)) *a.info = 1;
        const double w = inv * inv;
        const double rj = -(c[j] * w);
#pragma unroll
        for (int cc = 1; cc < QW; ++cc) {
          if (cc > j) {
            const double cj = __shfl_sync(0xffffffffu, c[j], cc, QW);   // row cc, column j
            if (cc < a.q && i >= cc) c[cc] = fma(rj, cj, c[cc]);
          }
        }
        c[j] = i >= j ? c[j] * inv : 0.0;   // column j is final: L[i][j]
      }
    }
    // F = mean + L z, summed over k <= i in order as fullcov_sample_kernel does
    const long zrow = s * a.z_ld + g * a.q + (row_ok ? i : 0);
    const double zi = row_ok ? a.z[zrow * a.D + d] : 0.0;
    double acc = 0.0;
#pragma unroll
    for (int k = 0; k < QW; ++k) {
      const double zk = __shfl_sync(0xffffffffu, zi, k, QW);
      if (k <= i && k < a.q) acc = fma(c[k], zk, acc);
    }
    if (row_ok) {
      const long p = col;
      const double f = a.mean[p * a.D + d] + acc;
      a.F[p * a.D + d] = f;
      if (a.F_user) a.F_user[((s * a.N_total + a.n0 + g * a.q + i) * a.D) + d] = f;
    }
  }
}

// -q-EI of each group and output: out[g][d] = -(1/S) sum_s max(y_min - min_j F[s][g q + j][d], 0) on the chunk's last-layer samples
// F [S][Nc][D] (F = [P][D], p = s Nc + n). One warp per (g, d): lane l sums s = l, l + 32, ... in order, then a fixed shuffle tree,
// so the value does not depend on scheduling.
__global__ void __launch_bounds__(128) qei_reduce_kernel(const double* __restrict__ F, long S, long Nc, int q, long G, int D,
                                                         double y_min, double* __restrict__ out) {
  const long w = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (w >= G * D) return;   // whole warps leave together
  const long g = w / D;
  const int d = (int)(w % D);
  double acc = 0.0;
  for (long s = lane; s < S; s += 32) {
    const double* f = F + ((s * Nc + g * q) * D + d);
    double mn = f[0];
    for (int j = 1; j < q; ++j) mn = fmin(mn, f[(long)j * D]);
    acc += (mn - y_min) < 0.0 ? (y_min - mn) : 0.0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) out[g * D + d] = -(acc / (double)S);
}

}  // namespace dgp
