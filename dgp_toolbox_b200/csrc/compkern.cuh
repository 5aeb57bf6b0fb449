// Composite multi-fidelity kernel of the reference's MF / MO models (MF_DGP.py:262-290, MO_DGP.py likewise) and its adjoint:
//   k(x, y) = k_corr(x_a, y_a) * (k_prev(x_b, y_b) + s_l^2 <x_b, y_b>) + k_in(x_a, y_a)      (+ s_w^2 on the diagonal of K(X, X) / K_diag)
// a = the first Da columns (the model input), b = the remaining columns (the previous fidelity's output, augmented by the
// model: MF_DGP.py:125). k_corr, k_prev: isotropic SquaredExponential (GPflow RBF(active_dims=..., variance=1.0) has one
// lengthscale); k_in: SquaredExponential, ARD or isotropic. has_prod = 0 leaves k_in (+ White) alone: the first fidelity's kernel.
// GPflow semantics: RBF = s^2 exp(-r^2/2) on active_dims, Linear = s^2 <x, y> on active_dims, White = s^2 I for K(X) / K_diag only.
#pragma once
#include "common.cuh"

namespace dgp {

struct CompK {
  int D, Da, has_prod, has_linear, in_ard;
  const double *in_var, *in_ls, *corr_var, *corr_ls, *prev_var, *prev_ls, *lin_var, *white_var;
};
constexpr int kCompTheta = 7;   // in_var, corr_var, corr_ls, prev_var, prev_ls, lin_var, white_var; then in_ls[Da]

struct CompParts { double ki, kc, kp, kl, r2a, r2b, dot; };

__device__ __forceinline__ double compk_eval(const CompK& k, const double* __restrict__ x, const double* __restrict__ y, CompParts& q) {
  double ri = 0.0, r2a = 0.0;
  for (int j = 0; j < k.Da; ++j) {
    const double t = x[j] - y[j];
    const double il = 1.0 / k.in_ls[k.in_ard ? j : 0];
    ri = fma(t * il, t * il, ri);
    r2a = fma(t, t, r2a);
  }
  q.ki = k.in_var[0] * exp(-0.5 * ri);
  q.r2a = r2a; q.r2b = 0.0; q.dot = 0.0; q.kc = 0.0; q.kp = 0.0; q.kl = 0.0;
  if (!k.has_prod) return q.ki;
  for (int j = k.Da; j < k.D; ++j) {
    const double t = x[j] - y[j];
    q.r2b = fma(t, t, q.r2b);
    q.dot = fma(x[j], y[j], q.dot);
  }
  const double lc = k.corr_ls[0], lp = k.prev_ls[0];
  q.kc = k.corr_var[0] * exp(-0.5 * r2a / (lc * lc));
  q.kp = k.prev_var[0] * exp(-0.5 * q.r2b / (lp * lp));
  q.kl = k.has_linear ? k.lin_var[0] * q.dot : 0.0;
  return q.kc * (q.kp + q.kl) + q.ki;
}

// K [P][P2]; X2 == null: K(X, X) with the White variance on the diagonal
__global__ void compk_K_kernel(CompK k, const double* __restrict__ X, long P, const double* __restrict__ X2, long P2, double* __restrict__ K) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= P * P2) return;
  const long i = idx / P2, j = idx % P2;
  CompParts q;
  double v = compk_eval(k, X + i * k.D, (X2 ? X2 : X) + j * k.D, q);
  if (!X2 && i == j && k.white_var) v += k.white_var[0];
  K[idx] = v;
}

// K [B][N][N] = K(X_b, X_b) for the B blocks of X [B][N][D], White on each block's diagonal; grid (ceil(N^2 / 256), <= 65535),
// the y index walks the blocks
__global__ void compk_K_blocks_kernel(CompK k, const double* __restrict__ X, long B, long N, double* __restrict__ K) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= N * N) return;
  const long i = idx / N, j = idx % N;
  for (long b = blockIdx.y; b < B; b += gridDim.y) {
    const double* Xb = X + b * N * k.D;
    CompParts q;
    double v = compk_eval(k, Xb + i * k.D, Xb + j * k.D, q);
    if (i == j && k.white_var) v += k.white_var[0];
    K[b * N * N + idx] = v;
  }
}

__global__ void compk_Kdiag_kernel(CompK k, const double* __restrict__ X, long P, double* __restrict__ out) {
  const long p = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= P) return;
  double v = k.in_var[0] + (k.white_var ? k.white_var[0] : 0.0);
  if (k.has_prod) {
    double n2 = 0.0;
    for (int j = k.Da; j < k.D; ++j) n2 = fma(X[p * k.D + j], X[p * k.D + j], n2);
    v += k.corr_var[0] * (k.prev_var[0] + (k.has_linear ? k.lin_var[0] * n2 : 0.0));
  }
  out[p] = v;
}

constexpr int kCompMaxD = 32;

// The adjoint kernels keep per-thread accumulators (gx / gy [D], gt [7 + Da]) in REGISTERS: every loop over the columns is fully
// unrolled to MAXD with a predicate, so all array indices are compile-time constants (run-time loop bounds put the arrays in local
// memory: measured 5.8 ms + 3.3 ms per [256 x 524 288] Kuf adjoint before, see profiles/r02z_mo_dgp*.json). MAXD = 16 covers the
// multi-fidelity / multi-objective models (D = input dimension + 1); MAXD = 32 is the general instantiation.
// loop-invariant factors of the adjoint, computed once per thread (FP64 divisions cost as much as the exponentials)
struct CompInv { double hc, hp, ilc2, ilp2, sl, vin, vc, vp; };
__device__ __forceinline__ CompInv compk_inv(const CompK& k) {
  CompInv v;
  v.vin = k.in_var[0];
  v.ilc2 = k.has_prod ? 1.0 / (k.corr_ls[0] * k.corr_ls[0]) : 0.0;
  v.ilp2 = k.has_prod ? 1.0 / (k.prev_ls[0] * k.prev_ls[0]) : 0.0;
  v.hc = -0.5 * v.ilc2; v.hp = -0.5 * v.ilp2;
  v.sl = (k.has_prod && k.has_linear) ? k.lin_var[0] : 0.0;
  v.vc = k.has_prod ? k.corr_var[0] : 0.0;
  v.vp = k.has_prod ? k.prev_var[0] : 0.0;
  return v;
}

// x, y: the two input rows; ilv[j] = 1 / lengthscale of k_in for column j < Da (shared memory, computed once per block)
template <int MAXD>
__device__ __forceinline__ void compk_eval_t(const CompK& k, const CompInv& v, const double* __restrict__ x, const double (&y)[MAXD],
                                             const double* __restrict__ ilv, CompParts& q) {
  double ri = 0.0, r2a = 0.0, r2b = 0.0, dot = 0.0;
#pragma unroll
  for (int j = 0; j < MAXD; ++j) {
    if (j < k.Da) {
      const double t = x[j] - y[j];
      const double u = t * ilv[j];
      ri = fma(u, u, ri);
      r2a = fma(t, t, r2a);
    } else if (j < k.D) {
      const double t = x[j] - y[j];
      r2b = fma(t, t, r2b);
      dot = fma(x[j], y[j], dot);
    }
  }
  q.ki = v.vin * exp(-0.5 * ri);
  q.r2a = r2a; q.r2b = r2b; q.dot = dot; q.kc = 0.0; q.kp = 0.0; q.kl = 0.0;
  if (!k.has_prod) return;
  q.kc = v.vc * exp(v.hc * r2a);
  q.kp = v.vp * exp(v.hp * r2b);
  q.kl = v.sl * dot;
}

// accumulate w * d k(x, y) / d x into g (SIDE 0) or w * d k / d y into g (SIDE 1), and (THETA) the RAW theta sums into gt:
//   gt[0] += w ki, gt[1] += w kc (kp + kl), gt[2] += w kc (kp + kl) r2a, gt[3] += w kc kp, gt[4] += w kc kp r2b, gt[5] += w kc dot,
//   gt[7 + j] += w ki t_j^2 (ARD; gt[7] collects all columns otherwise) -- compk_theta_scale turns them into derivatives.
template <int MAXD, int SIDE, bool THETA>
__device__ __forceinline__ void compk_accumulate_t(const CompK& k, const CompInv& v, const double* __restrict__ x, const double (&y)[MAXD],
                                                   const double* __restrict__ ilv, const CompParts& q, double w, double (&g)[MAXD],
                                                   double (&gt)[kCompTheta + MAXD]) {
  const double sum = q.kp + q.kl;
  const double sg = SIDE == 0 ? -w : w;
  const double wki = sg * q.ki, wc = sg * sum * q.kc * v.ilc2;      // d/dx_j of the a-part = -(ki il_j^2 + (kp + kl) kc / lc^2) t_j
  const double wkc = w * q.kc, wp = wkc * q.kp * v.ilp2, wl = wkc * v.sl;
#pragma unroll
  for (int j = 0; j < MAXD; ++j) {
    if (j < k.Da) {
      const double t = x[j] - y[j];
      const double il = ilv[j];
      g[j] = fma(fma(wki, il * il, wc), t, g[j]);
      if (THETA) {
        const double c = w * q.ki * t * t;
        if (k.in_ard) gt[kCompTheta + j] += c;
        else gt[kCompTheta] += c;
      }
    } else if (j < k.D && k.has_prod) {
      const double t = x[j] - y[j];
      if (SIDE == 0) g[j] = fma(wl, y[j], fma(-wp, t, g[j]));
      else g[j] = fma(wl, x[j], fma(wp, t, g[j]));
    }
  }
  if (THETA) {
    gt[0] = fma(w, q.ki, gt[0]);
    if (k.has_prod) {
      gt[1] = fma(wkc, sum, gt[1]);
      gt[2] = fma(wkc * sum, q.r2a, gt[2]);
      gt[3] = fma(wkc, q.kp, gt[3]);
      gt[4] = fma(wkc * q.kp, q.r2b, gt[4]);
      if (k.has_linear) gt[5] = fma(wkc, q.dot, gt[5]);
    }
  }
}

// raw theta sum t (slot `slot`) -> derivative
__device__ __forceinline__ double compk_theta_scale(const CompK& k, int slot, double t) {
  switch (slot) {
    case 0: return t / k.in_var[0];
    case 1: return k.has_prod ? t / k.corr_var[0] : 0.0;
    case 2: return k.has_prod ? t / (k.corr_ls[0] * k.corr_ls[0] * k.corr_ls[0]) : 0.0;
    case 3: return k.has_prod ? t / k.prev_var[0] : 0.0;
    case 4: return k.has_prod ? t / (k.prev_ls[0] * k.prev_ls[0] * k.prev_ls[0]) : 0.0;
    case 5: case 6: return t;
    default: {
      const double l = k.in_ls[k.in_ard ? slot - kCompTheta : 0];
      return t / (l * l * l);
    }
  }
}

template <int MAXD>
__device__ __forceinline__ void compk_load_row(const CompK& k, const double* __restrict__ p, double (&v)[MAXD]) {
#pragma unroll
  for (int j = 0; j < MAXD; ++j) v[j] = j < k.D ? p[j] : 0.0;
}

// grid (P, nsplit): block (i, sp) handles row i of X against the columns [sp * chunk, (sp + 1) * chunk) of X2 (X when X2 == null):
//   dXp[sp][i][:] = sum_j Kbar[i][j] dk(x_i, y_j)/dx_i (+ sum_j Kbar[j][i] dk(x_j, x_i)/dx_i when X2 == null),
//   part[sp * P + i][:] = its share of d/d theta.  The splits are summed in order by compk_sum_splits_kernel / reduce_partials_kernel.
template <int MAXD>
__global__ void __launch_bounds__(128) compk_grad_rows_kernel(CompK k, const double* __restrict__ X, long P, const double* __restrict__ X2,
                                                              long P2, long chunk, const double* __restrict__ Kbar, double* __restrict__ dXp,
                                                              double* __restrict__ part) {
  __shared__ double red[32];
  __shared__ double xi[MAXD], ilv[MAXD];
  const long i = blockIdx.x, sp = blockIdx.y;
  const int nt = kCompTheta + (k.in_ard ? k.Da : 1);
  double gx[MAXD], gt[kCompTheta + MAXD], y[MAXD];
#pragma unroll
  for (int j = 0; j < MAXD; ++j) gx[j] = 0.0;
#pragma unroll
  for (int j = 0; j < kCompTheta + MAXD; ++j) gt[j] = 0.0;
  if (threadIdx.x < MAXD) {
    xi[threadIdx.x] = threadIdx.x < k.D ? X[i * k.D + threadIdx.x] : 0.0;
    ilv[threadIdx.x] = threadIdx.x < k.Da ? 1.0 / k.in_ls[k.in_ard ? threadIdx.x : 0] : 0.0;
  }
  __syncthreads();
  const double* Y = X2 ? X2 : X;
  const CompInv v = compk_inv(k);
  const long j1 = (sp + 1) * chunk < P2 ? (sp + 1) * chunk : P2;
  for (long j = sp * chunk + threadIdx.x; j < j1; j += blockDim.x) {
    CompParts q;
    compk_load_row<MAXD>(k, Y + j * k.D, y);
    compk_eval_t<MAXD>(k, v, xi, y, ilv, q);
    const double w = Kbar[i * P2 + j];
    compk_accumulate_t<MAXD, 0, true>(k, v, xi, y, ilv, q, w, gx, gt);
    if (!X2) {      // k is symmetric: d k(x_j, x_i)/d x_i = d k(x_i, x_j)/d x_i, so the column term shares the derivative
      double none[kCompTheta + MAXD];
      compk_accumulate_t<MAXD, 0, false>(k, v, xi, y, ilv, q, Kbar[j * P2 + i], gx, none);
      if (i == j && k.white_var) gt[6] += w;
    }
  }
#pragma unroll
  for (int j = 0; j < MAXD; ++j) {
    if (j < k.D) {
      const double r = block_sum(gx[j], red);
      if (threadIdx.x == 0) dXp[(sp * P + i) * k.D + j] = r;
    }
  }
#pragma unroll
  for (int j = 0; j < kCompTheta + MAXD; ++j) {
    if (j < nt) {
      const double r = block_sum(gt[j], red);
      if (threadIdx.x == 0) part[(sp * P + i) * nt + j] = compk_theta_scale(k, j, r);
    }
  }
}

// out[e] = sum_sp in[sp][e], e < n, in split order
__global__ void compk_sum_splits_kernel(const double* __restrict__ in, int nsplit, long n, double* __restrict__ out) {
  const long e = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  double s = 0.0;
  for (int sp = 0; sp < nsplit; ++sp) s += in[(long)sp * n + e];
  out[e] = s;
}

// One thread per row j of X2: dX2[j][:] = sum_i Kbar[i][j] dk(x_i, y_j)/dy_j   (the rows x_i are uniform across the warp)
template <int MAXD>
__global__ void __launch_bounds__(128) compk_grad_cols_kernel(CompK k, const double* __restrict__ X, long P, const double* __restrict__ X2,
                                                              long P2, const double* __restrict__ Kbar, double* __restrict__ dX2) {
  __shared__ double ilv[MAXD];
  if (threadIdx.x < MAXD) ilv[threadIdx.x] = threadIdx.x < k.Da ? 1.0 / k.in_ls[k.in_ard ? threadIdx.x : 0] : 0.0;
  __syncthreads();
  const long j = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= P2) return;
  double gy[MAXD], y[MAXD], none[kCompTheta + MAXD];
  const CompInv v = compk_inv(k);
#pragma unroll
  for (int d = 0; d < MAXD; ++d) gy[d] = 0.0;
  compk_load_row<MAXD>(k, X2 + j * k.D, y);
  for (long i = 0; i < P; ++i) {
    CompParts q;
    const double* x = X + i * k.D;      // uniform across the block: broadcast loads
    compk_eval_t<MAXD>(k, v, x, y, ilv, q);
    compk_accumulate_t<MAXD, 1, false>(k, v, x, y, ilv, q, Kbar[i * P2 + j], gy, none);
  }
#pragma unroll
  for (int d = 0; d < MAXD; ++d)
    if (d < k.D) dX2[j * k.D + d] = gy[d];
}

// K_diag adjoint: dX[p][b] = g[p] * 2 s_c^2 s_l^2 x_pb; per-block partial sums of d/d theta
__global__ void __launch_bounds__(128) compk_Kdiag_grad_kernel(CompK k, const double* __restrict__ X, long P, const double* __restrict__ g,
                                                               double* __restrict__ dX, double* __restrict__ part) {
  __shared__ double red[32];
  const long p = (long)blockIdx.x * blockDim.x + threadIdx.x;
  double t[kCompTheta];
  for (int j = 0; j < kCompTheta; ++j) t[j] = 0.0;
  if (p < P) {
    const double w = g[p];
    for (int j = 0; j < k.Da; ++j) dX[p * k.D + j] = 0.0;
    double n2 = 0.0;
    for (int j = k.Da; j < k.D; ++j) {
      const double x = X[p * k.D + j];
      n2 = fma(x, x, n2);
      dX[p * k.D + j] = (k.has_prod && k.has_linear) ? w * 2.0 * k.corr_var[0] * k.lin_var[0] * x : 0.0;
    }
    t[0] = w;
    t[6] = k.white_var ? w : 0.0;
    if (k.has_prod) {
      const double sl = k.has_linear ? k.lin_var[0] : 0.0;
      t[1] = w * (k.prev_var[0] + sl * n2);
      t[3] = w * k.corr_var[0];
      t[5] = k.has_linear ? w * k.corr_var[0] * n2 : 0.0;
    }
  }
  const int nt = kCompTheta + (k.in_ard ? k.Da : 1);
  for (int j = 0; j < nt; ++j) {
    const double r = block_sum(j < kCompTheta ? t[j] : 0.0, red);
    if (threadIdx.x == 0) part[(long)blockIdx.x * nt + j] = r;
  }
}

}  // namespace dgp
