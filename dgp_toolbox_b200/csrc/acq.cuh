// Acquisition epilogues (SURVEY §8 a11/a12): mixture moments over the S samples, EI (analytic + MC), exact 2-D EHVI.
// Reference: dgp_dace/models/dgp.py:362-366, dgp_dace/Infill_criteria.py:36-52, dgp_dace/EHVI.py:102-104,154-157.
#pragma once
#include "common.cuh"
#include "philox.cuh"

namespace dgp {

__device__ __forceinline__ double norm_cdf(double x) { return 0.5 * erfc(-x * 0.70710678118654752440); }
__device__ __forceinline__ double norm_pdf(double x) { return 0.39894228040143267794 * exp(-0.5 * x * x); }

// mean[n,d] = mean_s mu ; var[n,d] = mean_s (v + add) + mean_s (mu - mean)^2     (inputs [S,N,D])
// Centred second pass: the one-pass mean_s (v + mu^2) - mean^2 cancels when |mean| is large next to the spread and can come out
// zero or negative (then EI is NaN); this form has no cancellation and its error stays below S eps var.
__global__ void mixture_moments_kernel(const double* __restrict__ Fmean, const double* __restrict__ Fvar, long S, long ND,
                                       const double* __restrict__ likvar, int add_lik, double* __restrict__ mean,
                                       double* __restrict__ var) {
  long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ND) return;
  const double add = add_lik ? likvar[0] : 0.0;
  double sm = 0.0;
  for (long s = 0; s < S; ++s) sm += Fmean[s * ND + i];
  const double mu = sm / (double)S;
  double acc = 0.0;
  for (long s = 0; s < S; ++s) {
    const double d = Fmean[s * ND + i] - mu;
    acc += (Fvar[s * ND + i] + add) + d * d;
  }
  mean[i] = mu;
  var[i] = acc / (double)S;
}

// -EI from moments: Normal(mean, sqrt(var)); t1 = (y_min - mean) cdf(y_min); t2 = var * pdf(y_min)
__global__ void ei_analytic_kernel(const double* __restrict__ mean, const double* __restrict__ var, long n, double y_min,
                                   double* __restrict__ out) {
  long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double m = mean[i], v = var[i], s = sqrt(v);
  double u = (y_min - m) / s;
  double t1 = (y_min - m) * norm_cdf(u);
  double t2 = v * (norm_pdf(u) / s);
  out[i] = -(t1 + t2);
}

// -EI and its upstream adjoints w.r.t. the last layer's per-sample moments (for d(-EI)/dx, the gradient the reference's
// Adam-on-x acquisition search differentiates, Infill_criteria.py:79-84). With mbar = mean_s mu, vbar = mean_s v + mean_s (mu - mbar)^2
// (centred, as in mixture_moments_kernel), sigma = sqrt(vbar), u = (y_min - mbar)/sigma:  d(-EI)/d mbar = Phi(u),  d(-EI)/d vbar = -phi(u) / (2 sigma), hence
//   Gm[s] = Phi(u)/S - phi(u) (mu_s - mbar) / (sigma S),   Gv[s] = -phi(u) / (2 sigma S).
// One thread per candidate point; chunk-local p = s * Nc + n. Gm / GvT / GmPad / gq must be zero-filled beforehand.
// kind selects the criterion c(mbar, vbar) (and its partial derivatives) evaluated on the mixture moments; lik_var != null adds
// sigma_n^2 to vbar (predict_y moments, what WB2 / EV use; EI.run works on predict_f moments):
//   0  -EI(y)          u = (y - mbar)/sigma:  dc/dmbar = Phi(u),      dc/dvbar = -phi(u) / (2 sigma)
//   1  -(EI(y) - mbar) (WB2):                 dc/dmbar = Phi(u) + 1,  dc/dvbar as above
//   2  EV(y) = (mbar - y) Phi(t) + sigma phi(t), t = (mbar - y)/sigma:  dc/dmbar = Phi(t),  dc/dvbar = phi(t) / (2 sigma)
// Per sample: Gm[s] = dc/dmbar / S + 2 dc/dvbar (mu_s - mbar) / S,  Gv[s] = dc/dvbar / S.
__global__ void ei_upstream_kernel(const double* __restrict__ Fmean, const double* __restrict__ Fvar, long Nc, long S, long Pp, int D,
                                   double y_min, double* __restrict__ neg_ei, double* __restrict__ Gm, double* __restrict__ GvT,
                                   double* __restrict__ GmPad, double* __restrict__ gq, int kind, const double* __restrict__ lik_var,
                                   const double* __restrict__ Xc, int d0, double* __restrict__ direct) {
  // kind 3 (WB2S, Infill_criteria.py:187-198, single-output model): value[n][j] = -(sig(x_nj) EI - mbar), j < d0; the chain receives
  // the adjoints of sum_j value[n][j] (dc/dmbar = Phi(u) sum_j sig_j + d0, dc/dvbar = -phi(u) sum_j sig_j / (2 sigma)) and
  // `direct`[n][j] = -sig_j (1 - sig_j) EI is the explicit dependence on x, added to the input gradient by the caller.
  const long n = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= Nc) return;
  for (int d = 0; d < D; ++d) {
    double sm = 0.0;
    for (long s = 0; s < S; ++s) sm += Fmean[(s * Nc + n) * D + d];
    const double mbar = sm / (double)S;
    double acc = 0.0;
    for (long s = 0; s < S; ++s) {
      const double dm_s = Fmean[(s * Nc + n) * D + d] - mbar;
      acc += Fvar[(s * Nc + n) * D + d] + dm_s * dm_s;
    }
    const double vbar = acc / (double)S + (lik_var ? lik_var[0] : 0.0), sig = sqrt(vbar);
    double val = 0.0, dm, dv;
    if (kind == 4) {   // adjoints supplied by the caller (neg_ei holds (dc/dmbar, dc/dvbar) per candidate and output, read only)
      dm = neg_ei[(n * D + d) * 2];
      dv = neg_ei[(n * D + d) * 2 + 1];
    } else if (kind == 2) {
      const double t = (mbar - y_min) / sig, cdf = norm_cdf(t), pdf = norm_pdf(t);
      val = (mbar - y_min) * cdf + vbar * (pdf / sig);
      dm = cdf;
      dv = pdf / (2.0 * sig);
    } else {
      const double u = (y_min - mbar) / sig, cdf = norm_cdf(u), pdf = norm_pdf(u);
      val = -((y_min - mbar) * cdf + vbar * (pdf / sig));
      dm = cdf;
      dv = -pdf / (2.0 * sig);
      if (kind == 1) { val += mbar; dm += 1.0; }
      if (kind == 3) {
        const double ei = -val;
        double ssum = 0.0;
        for (int j = 0; j < d0; ++j) {
          const double sg = 1.0 / (1.0 + exp(-Xc[n * d0 + j]));
          ssum += sg;
          neg_ei[n * d0 + j] = -(sg * ei - mbar);
          direct[n * d0 + j] = -sg * (1.0 - sg) * ei;
        }
        dm = dm * ssum + (double)d0;
        dv = dv * ssum;
      }
    }
    if (kind != 3 && kind != 4) neg_ei[n * D + d] = val;
    const double gv = dv / (double)S;
    for (long s = 0; s < S; ++s) {
      const long p = s * Nc + n;
      const double gm = dm / (double)S + 2.0 * dv * (Fmean[p * D + d] - mbar) / (double)S;
      Gm[p * D + d] = gm;
      GmPad[p * 32 + d] = gm;
      GvT[(long)d * Pp + p] = gv;
      gq[p] -= gv;
    }
  }
}

// Moment-based criteria of dgp_dace/Infill_criteria.py on (mean, var) [n] (mixture moments of predict_y over the samples):
//   kind 0  -EI(y)                      (EI.run, :43-47,52)
//   kind 1  -(EI(y) - mean)             (WB2.run, :124-133)
//   kind 2  EV(c) = (mean - c) Phi((mean - c)/s) + s phi((mean - c)/s)   (EV_one_constraint.run analytic, :249-257)
//   kind 3  -(sigmoid(x[n][j]) EI(y) - mean)   -> out [n][d]            (WB2S.run, :187-198; S = 1/(1 + 1/exp(x)) elementwise in x)
//   kind 4  Phi((c - mean) / s): probability that the constraint value is below c     (PoF, :318-341 -- the reference computes the
//           EI-style terms there and returns nothing; this is the probability its name and its use in run_with_IC call for)
__global__ void acq_moments_kernel(int kind, const double* __restrict__ mean, const double* __restrict__ var, long n, double y,
                                   const double* __restrict__ x, int d, double* __restrict__ out) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double m = mean[i], v = var[i], s = sqrt(v);
  if (kind == 4) { out[i] = norm_cdf((y - m) / s); return; }
  if (kind == 2) {
    const double u = (m - y) / s;
    out[i] = (m - y) * norm_cdf(u) + v * (norm_pdf(u) / s);
    return;
  }
  const double u = (y - m) / s;
  const double ei = (y - m) * norm_cdf(u) + v * (norm_pdf(u) / s);
  if (kind == 0) out[i] = -ei;
  else if (kind == 1) out[i] = -(ei - m);
  else {
    for (int j = 0; j < d; ++j) {
      const double sg = 1.0 / (1.0 + 1.0 / exp(x[i * d + j]));
      out[i * d + j] = -(sg * ei - m);
    }
  }
}

// Monte-Carlo expected violation: mean_s where(F - c < 0, 0, F - c)     (EV_one_constraint.run, :259-262; F [S,N,D])
__global__ void ev_mc_kernel(const double* __restrict__ F, long S, long ND, double c, double* __restrict__ out) {
  long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ND) return;
  double acc = 0.0;
  for (long s = 0; s < S; ++s) {
    const double f = F[s * ND + i];
    acc += (f - c) < 0.0 ? 0.0 : (f - c);
  }
  out[i] = acc / (double)S;
}

// out[n][j] = sum_s in[(s * Nc + n)][j]
__global__ void sum_samples_kernel(const double* __restrict__ in, long Nc, long S, int D, double* __restrict__ out) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= Nc * D) return;
  double acc = 0.0;
  for (long s = 0; s < S; ++s) acc += in[s * Nc * D + idx];
  out[idx] = acc;
}

// -EI by Monte-Carlo: mean_s where(F - y_min < 0, y_min - F, 0)     (F [S,N,D])
__global__ void ei_mc_kernel(const double* __restrict__ F, long S, long ND, double y_min, double* __restrict__ out) {
  long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= ND) return;
  double acc = 0.0;
  for (long s = 0; s < S; ++s) {
    double f = F[s * ND + i];
    acc += (f - y_min) < 0.0 ? (y_min - f) : 0.0;
  }
  out[i] = -(acc / (double)S);
}

__device__ __forceinline__ double psi_fn(double a, double b, double mu, double sigma) {
  double u = (b - mu) / sigma;
  return sigma * norm_pdf(u) + (a - mu) * norm_cdf(u);
}

// Exact uncorrelated 2-objective EHVI strip sum over the padded front (n entries, staged in shared memory).
__global__ void ehvi2d_kernel(const double* __restrict__ m0, const double* __restrict__ v0, const double* __restrict__ m1,
                              const double* __restrict__ v1, long N, const double* __restrict__ ynd0,
                              const double* __restrict__ ynd1, int n, double* __restrict__ out) {
  extern __shared__ double sh[];
  double* y0 = sh;
  double* y1 = sh + n;
  for (int i = threadIdx.x; i < n; i += blockDim.x) { y0[i] = ynd0[i]; y1[i] = ynd1[i]; }
  __syncthreads();
  long c = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= N) return;
  const double mu0 = m0[c], s0 = sqrt(v0[c]), mu1 = m1[c], s1 = sqrt(v1[c]);
  const double cdf_last = norm_cdf((y0[n - 1] - mu0) / s0);
  double t1 = 0.0, t2 = 0.0;
  for (int i = 1; i < n; ++i) {
    const double d1 = psi_fn(y1[i], y1[i], mu1, s1) - psi_fn(y1[i], y1[0], mu1, s1);
    if (i < n - 1) t1 += (y0[i - 1] - y0[i]) * (norm_cdf((y0[i] - mu0) / s0) - cdf_last) * d1;
    t2 += (psi_fn(y0[i - 1], y0[i - 1], mu0, s0) - psi_fn(y0[i - 1], y0[i], mu0, s0)) * d1;
  }
  out[c] = t1 + t2;
}

// d psi / d mu and d psi / d sigma of psi(a, b, mu, sigma) = sigma phi(u) + (a - mu) Phi(u), u = (b - mu) / sigma
__device__ __forceinline__ void psi_grad(double a, double b, double mu, double sigma, double& val, double& dmu, double& dsig) {
  const double u = (b - mu) / sigma, pdf = norm_pdf(u), cdf = norm_cdf(u), q = (a - mu) * pdf / sigma;
  val = sigma * pdf + (a - mu) * cdf;
  dmu = u * pdf - cdf - q;
  dsig = pdf * (1.0 + u * u) - q * u;
}

// ehvi2d_kernel with its partial derivatives w.r.t. the four moments: grads[c] = (dE/dm0, dE/dv0, dE/dm1, dE/dv1)
// (the Adam stage of optimize_EHVI, EHVI.py:218-234, differentiates the criterion w.r.t. the candidate through them).
__global__ void ehvi2d_grad_kernel(const double* __restrict__ m0, const double* __restrict__ v0, const double* __restrict__ m1,
                                   const double* __restrict__ v1, long N, const double* __restrict__ ynd0,
                                   const double* __restrict__ ynd1, int n, double* __restrict__ out, double* __restrict__ grads) {
  extern __shared__ double sh[];
  double* y0 = sh;
  double* y1 = sh + n;
  for (int i = threadIdx.x; i < n; i += blockDim.x) { y0[i] = ynd0[i]; y1[i] = ynd1[i]; }
  __syncthreads();
  long c = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= N) return;
  const double mu0 = m0[c], s0 = sqrt(v0[c]), mu1 = m1[c], s1 = sqrt(v1[c]);
  const double ul = (y0[n - 1] - mu0) / s0, cdf_last = norm_cdf(ul), pdf_last = norm_pdf(ul);
  double e = 0.0, gm0 = 0.0, gs0 = 0.0, gm1 = 0.0, gs1 = 0.0;
  for (int i = 1; i < n; ++i) {
    double pa, pam, pas, pb, pbm, pbs;
    psi_grad(y1[i], y1[i], mu1, s1, pa, pam, pas);
    psi_grad(y1[i], y1[0], mu1, s1, pb, pbm, pbs);
    const double d1 = pa - pb, d1m = pam - pbm, d1s = pas - pbs;
    double f = 0.0, fm = 0.0, fs = 0.0;   // the objective-0 factor of the strip and its derivatives
    if (i < n - 1) {
      const double w = y0[i - 1] - y0[i], u = (y0[i] - mu0) / s0, pdf = norm_pdf(u);
      f += w * (norm_cdf(u) - cdf_last);
      fm += w * (-pdf + pdf_last) / s0;
      fs += w * (-u * pdf + ul * pdf_last) / s0;
    }
    psi_grad(y0[i - 1], y0[i - 1], mu0, s0, pa, pam, pas);
    psi_grad(y0[i - 1], y0[i], mu0, s0, pb, pbm, pbs);
    f += pa - pb; fm += pam - pbm; fs += pas - pbs;
    e += f * d1;
    gm0 += fm * d1; gs0 += fs * d1;
    gm1 += f * d1m; gs1 += f * d1s;
  }
  out[c] = e;
  grads[4 * c + 0] = gm0; grads[4 * c + 1] = gs0 / (2.0 * s0);
  grads[4 * c + 2] = gm1; grads[4 * c + 3] = gs1 / (2.0 * s1);
}

// ---------------------------------------------------------------------------------------------------------
// Acquisition search on the device (SURVEY §8 f3; reference Infill_criteria.py:61-87 and its copies for the other criteria):
// tfp.optimizer.differential_evolution_minimize ("rand/1/bin", differential weight 0.5, crossover probability 0.9) followed by
// tf.optimizers.Adam, both on u with x = lw + (up - lw) / (1 + exp(u)).
// Random choices come from Philox-4x32-10 with key = seed and counter = (member, generation, slot, 0xDE):
//   slot 0: words (w0, w1, w2, w3) -> three distinct partners a, b, c != member (w_k mod (pop-1-k), then skipping the excluded
//           indices in ascending order) and the forced crossover dimension w3 mod d;
//   slot 1 + j/4: word j%4 -> uniform (w + 0.5) / 2^32 of dimension j; the dimension takes the mutant when it is < crossover.
// ---------------------------------------------------------------------------------------------------------
__device__ inline int de_skip(int v, int e0, int e1, int e2, int n_excl) {   // v-th index not in the sorted exclusion list
  if (n_excl > 0 && v >= e0) ++v;
  if (n_excl > 1 && v >= e1) ++v;
  if (n_excl > 2 && v >= e2) ++v;
  return v;
}

__global__ void de_propose_kernel(const double* __restrict__ pop_u, long pop, int d, const double* __restrict__ lw,
                                  const double* __restrict__ up, unsigned long long seed, const unsigned long long* seed_ptr,
                                  long generation, double weight, double crossover, double* __restrict__ cand_u,
                                  double* __restrict__ cand_x) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= pop * d) return;
  const int i = (int)(idx / d), j = (int)(idx % d);
  const unsigned long long sd = seed_ptr ? *seed_ptr : seed;
  uint32_t w[4];
  philox4x32_10((uint32_t)i, (uint32_t)generation, 0u, 0xDEu, (uint32_t)sd, (uint32_t)(sd >> 32), w);
  const int a = de_skip((int)(w[0] % (uint32_t)(pop - 1)), i, 0, 0, 1);
  const int lo1 = min(i, a), hi1 = max(i, a);
  const int b = de_skip((int)(w[1] % (uint32_t)(pop - 2)), lo1, hi1, 0, 2);
  int e0 = lo1, e1 = hi1, e2 = b;   // sort {i, a, b}
  if (e2 < e1) { const int t = e1; e1 = e2; e2 = t; }
  if (e1 < e0) { const int t = e0; e0 = e1; e1 = t; }
  const int c = de_skip((int)(w[2] % (uint32_t)(pop - 3)), e0, e1, e2, 3);
  const int forced = (int)(w[3] % (uint32_t)d);
  uint32_t r[4];
  philox4x32_10((uint32_t)i, (uint32_t)generation, (uint32_t)(1 + j / 4), 0xDEu, (uint32_t)sd, (uint32_t)(sd >> 32), r);
  const double uni = ((double)r[j % 4] + 0.5) * (1.0 / 4294967296.0);
  const double mutant = pop_u[(long)a * d + j] + weight * (pop_u[(long)b * d + j] - pop_u[(long)c * d + j]);
  const double u = (uni < crossover || j == forced) ? mutant : pop_u[(long)i * d + j];
  cand_u[idx] = u;
  cand_x[idx] = lw[j] + (up[j] - lw[j]) / (1.0 + exp(u));
}

// Member i takes the candidate when it is strictly better (minimisation); values are summed over the ncol output columns.
__global__ void de_select_kernel(double* __restrict__ pop_u, double* __restrict__ pop_val, const double* __restrict__ cand_u,
                                 const double* __restrict__ cand_val, long pop, int d, int ncol, int first) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= pop) return;
  double v = 0.0;
  for (int k = 0; k < ncol; ++k) v += cand_val[i * ncol + k];
  if (first || v < pop_val[i]) {
    pop_val[i] = v;
    for (int j = 0; j < d; ++j) pop_u[i * d + j] = cand_u[i * d + j];
  }
}

__global__ void box_from_u_kernel(const double* __restrict__ u, const double* __restrict__ lw, const double* __restrict__ up,
                                  long n, int d, double* __restrict__ x) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * d) return;
  const int j = (int)(idx % d);
  x[idx] = lw[j] + (up[j] - lw[j]) / (1.0 + exp(u[idx]));
}

// One tf.optimizers.Adam step on u from dL/dx (Infill_criteria.py:79-84): dx/du = -(up - lw) e^u / (1 + e^u)^2; the new x is
// written back so that the next criterion evaluation reads it.
__global__ void adam_box_kernel(double* __restrict__ u, double* __restrict__ m_state, double* __restrict__ v_state,
                                const double* __restrict__ dx, const double* __restrict__ lw, const double* __restrict__ up, long n,
                                int d, double lr_t, double beta1, double beta2, double eps, double* __restrict__ x) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n * d) return;
  const int j = (int)(idx % d);
  const double span = up[j] - lw[j];
  double uu = u[idx];
  const double sg = 1.0 / (1.0 + exp(uu));              // x = lw + span * sg
  const double g = dx[idx] * (-span * sg * (1.0 - sg));
  const double m = beta1 * m_state[idx] + (1.0 - beta1) * g;
  const double v = beta2 * v_state[idx] + (1.0 - beta2) * g * g;
  m_state[idx] = m;
  v_state[idx] = v;
  uu -= lr_t * m / (sqrt(v) + eps);
  u[idx] = uu;
  x[idx] = lw[j] + span / (1.0 + exp(uu));
}

}  // namespace dgp

namespace dgp {
__global__ void add_inplace_kernel(double* __restrict__ dst, const double* __restrict__ src, long n) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] += src[i];
}
}  // namespace dgp
