// FP64 tensor-core (DMMA.8x8x4) GEMM engine used by every dense / triangular contraction on the DGP path.
//
//   NN:  C[b] = alpha * A[b] (M x K, row-major) * B[b] (K x N, row-major) + beta * C[b]
//   NT:  C[b] = alpha * A[b] (M x K) * diag(kscale[b]) * B[b]^T (B is N x K, row-major) + beta * C[b]
//
// Operands are staged global -> shared with a STAGES-deep cp.async ring; each warp owns a (BM/WM) x (BN/WN)
// sub-tile held as DMMA accumulator fragments. All dimensions are multiples of the tile sizes (buffers on the
// path are padded by construction), so there is no bounds checking in the inner loop.
//   a_tri = 1: A is lower triangular (K-range clipped at the row block), 2: upper triangular.
//   c_lower = 1: only tiles touching the lower triangle of C are computed (symmetric rank-k updates).
//   splitk > 1: K is cut into splitk chunks, partial tiles go to `part` and are summed in a fixed order
//               (deterministic, no atomics) by gemm_splitk_reduce.
#pragma once
#include <type_traits>

#include "common.cuh"

namespace dgp {

struct GemmArgs {
  const double* A; long lda; long sA;
  const double* B; long ldb; long sB;
  double* C; long ldc; long sC;
  int M, N, K;
  double alpha, beta;
  const double* kscale; long sScale;
  int a_tri;
  int c_lower;
  int batch;
  int splitk;
  double* part;
  // K-concatenation: K = kblocks * kblk; A is [M][kblocks*kblk], B is the row-stacked [kblocks*kblk][N] (NN only).
  // splitk > 1 (<= kblocks) deals whole blocks out to the splits.
  // With a_tri = 1 every block is lower triangular (its k-range is clipped at the row block). kblocks <= 1: plain GEMM.
  int kblocks; int kblk;
  // Optional column scale of B in NN mode: B[k][n] *= bscale_mul * bscale[(k / kblk) * ld_bscale + n].
  const double* bscale; long ld_bscale; double bscale_mul;
  // Optional epilogue term (non-split-K only): C[m][n] += epi_mul * epi_col[n] * epi_plane[m * ld_epi + n]
  const double* epi_plane; long ld_epi; const double* epi_col; double epi_mul;
};

template <int BM, int BN, int BK, int WM, int WN, bool NT, int STAGES>
struct GemmCfg {
  static constexpr int THREADS = WM * WN * 32;
  static constexpr int TM = BM / WM / 8, TN = BN / WN / 8;
  static constexpr int LDA = BK + 4;
  static constexpr int LDB = NT ? BK + 4 : BN + 4;
  static constexpr int A_STAGE = BM * LDA;
  static constexpr int B_STAGE = NT ? BN * LDB : BK * LDB;
  static constexpr size_t SMEM = (size_t)STAGES * (A_STAGE + B_STAGE + BK) * sizeof(double);
};

__device__ __forceinline__ bool gemm_tri_skip_enabled() { return true; }

// TSEL (lower-only products): 0 = every tile, 1 = strictly-lower tiles only and the diagonal-tile code compiled out (124 instead of
// 204 registers, so three CTAs fit an SM with a 2-stage ring), 2 = diagonal tiles only.
template <int BM, int BN, int BK, int WM, int WN, bool NT, int STAGES, int TSEL = 0>
__global__ void __launch_bounds__(WM* WN * 32) gemm_kernel(GemmArgs g) {
  using Cfg = GemmCfg<BM, BN, BK, WM, WN, NT, STAGES>;
  constexpr int THREADS = Cfg::THREADS, TM = Cfg::TM, TN = Cfg::TN, LDA = Cfg::LDA, LDB = Cfg::LDB;
  constexpr int A_STAGE = Cfg::A_STAGE, B_STAGE = Cfg::B_STAGE;
  extern __shared__ __align__(16) double smem[];
  double* As = smem;
  double* Bs = As + STAGES * A_STAGE;
  double* Ss = Bs + STAGES * B_STAGE;

  const int tid = threadIdx.x, lane = tid & 31;
  // Triangular A: inside a diagonal block a warp whose rows lie entirely above (lower A) / below (upper A) the k-tile has only
  // zeros to multiply and skips it. Warp w always runs on SM sub-partition w % 4, so the warp -> row-slot role rotates with the
  // CTA index to spread the lighter roles over the sub-partitions.
  const int warp = g.a_tri ? (int)(((tid >> 5) + blockIdx.x) % (WM * WN)) : (tid >> 5);
  const int g8 = lane >> 2, t4 = lane & 3;
  const int wm = warp / WN, wn = warp % WN;

  const int mt_count = g.M / BM, nt_count = g.N / BN;
  long bid = blockIdx.x;
  const int mt = (int)(bid % mt_count); bid /= mt_count;
  const int b = (int)(bid % g.batch); bid /= g.batch;
  const int nt = (int)(bid % nt_count); bid /= nt_count;
  const int split = (int)bid;
  const int m0 = mt * BM, n0 = nt * BN;
  if (g.c_lower && n0 >= m0 + BM) return;
  if (TSEL == 1 && n0 == m0) return;
  if (TSEL == 2 && n0 != m0) return;

  // split-K: chunks of whole k-tiles, the last one may be shorter (any split count works, so the launcher can pick the
  // count that fills whole waves of CTAs)
  const int kchunk = ((g.K / BK + g.splitk - 1) / g.splitk) * BK;
  int kbeg = min(split * kchunk, g.K), kend = min(kbeg + kchunk, g.K);
  if (g.a_tri == 1) kend = min(kend, m0 + BM);
  if (g.a_tri == 2) kbeg = max(kbeg, (m0 / BK) * BK);
  int ktiles = kend > kbeg ? (kend - kbeg) / BK : 0;
  int tpb = ktiles > 0 ? ktiles : 1;   // k-tiles per concatenated block
  const int kblk = g.kblocks > 1 ? g.kblk : 0;
  int blk0 = 0;   // first concatenated block of this CTA: with splitk > 1 the blocks (not the k-range) are dealt out to the splits
  if (g.kblocks > 1) {
    const int hi = g.a_tri == 1 ? min(g.kblk, m0 + BM) : g.kblk;
    int nblk = g.kblocks;
    if (g.splitk > 1) {
      const int bps = (g.kblocks + g.splitk - 1) / g.splitk;
      blk0 = split * bps;
      nblk = max(0, min(bps, g.kblocks - blk0));
    }
    kbeg = 0;
    tpb = hi / BK;
    ktiles = nblk * tpb;
  }
  auto koff = [&](int kt) { const int blk = kt / tpb; return (blk0 + blk) * kblk + kbeg + (kt - blk * tpb) * BK; };

  const double* Ab = g.A + (long)b * g.sA;
  const double* Bb = g.B + (long)b * g.sB;
  const double* Sb = g.kscale ? g.kscale + (long)b * g.sScale : nullptr;

  auto load_stage = [&](int stage, int k0) {
    double* as = As + stage * A_STAGE;
    double* bs = Bs + stage * B_STAGE;
    constexpr int A_CHUNKS = BM * BK / 2;
    for (int c = tid; c < A_CHUNKS; c += THREADS) {
      int r = c / (BK / 2), cc = c % (BK / 2);
      cp_async16(as + r * LDA + cc * 2, Ab + (long)(m0 + r) * g.lda + k0 + cc * 2);
    }
    if (NT) {
      constexpr int B_CHUNKS = BN * BK / 2;
      for (int c = tid; c < B_CHUNKS; c += THREADS) {
        int r = c / (BK / 2), cc = c % (BK / 2);
        cp_async16(bs + r * LDB + cc * 2, Bb + (long)(n0 + r) * g.ldb + k0 + cc * 2);
      }
    } else {
      constexpr int B_CHUNKS = BK * BN / 2;
      for (int c = tid; c < B_CHUNKS; c += THREADS) {
        int r = c / (BN / 2), cc = c % (BN / 2);
        cp_async16(bs + r * LDB + cc * 2, Bb + (long)(k0 + r) * g.ldb + n0 + cc * 2);
      }
    }
    if (Sb) {
      for (int c = tid; c < BK / 2; c += THREADS) cp_async16(Ss + stage * BK + c * 2, Sb + k0 + c * 2);
    }
  };

  // ---- diagonal tile of a lower-only NT product (contractions over the point-samples: tril(dV V^T), tril(V dT_d^T)) ----
  // Only the 36 of 64 accumulator units (8 x 8 each) on or below the diagonal are needed. Giving each warp a 32 x 32 quadrant
  // would leave one warp idle and two half-used while the CTA still takes the full time, so instead every warp computes ALL
  // 36 units for a quarter of each k-tile's k-steps; the four partial sums are added through shared memory at the end.
  // The CTA then takes 36/64 of the time of an off-diagonal tile.
  if constexpr (TSEL != 1 && NT && BM == 64 && BN == 64 && BK == 32 && WM * WN == 4) {
    if (g.c_lower && n0 == m0 && g.a_tri == 0 && g.kblocks <= 1) {
      const int w = tid >> 5;
      double d0[8][8], d1[8][8];
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) { d0[i][j] = 0.0; d1[i][j] = 0.0; }
#pragma unroll
      for (int s = 0; s < STAGES - 1; ++s) {
        if (s < ktiles) load_stage(s, koff(s));
        cp_async_commit();
      }
      for (int kt = 0; kt < ktiles; ++kt) {
        cp_async_wait<STAGES - 2>();
        __syncthreads();
        {
          int nk = kt + STAGES - 1;
          if (nk < ktiles) load_stage(nk % STAGES, koff(nk));
          cp_async_commit();
        }
        const int st = kt % STAGES;
        const double* as = As + st * A_STAGE + g8 * LDA + t4;
        const double* bs = Bs + st * B_STAGE + g8 * LDB + t4;
        const double* ss = Ss + st * BK + t4;
#pragma unroll
        for (int q = 0; q < BK / 16; ++q) {
          const int kk = w * (BK / 16) + q;   // this warp's k-steps of the tile
          double a[8], bb[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) a[i] = as[i * 8 * LDA + kk * 4];
          if (Sb) {
            const double sc = ss[kk * 4];
#pragma unroll
            for (int i = 0; i < 8; ++i) a[i] *= sc;
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) bb[j] = bs[j * 8 * LDB + kk * 4];
#pragma unroll
          for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j)
              if (j <= i) dmma884(d0[i][j], d1[i][j], a[i], bb[j]);
        }
      }
      cp_async_wait<0>();
      __syncthreads();
      // cross-warp sum in a fixed order through shared memory: red[w][unit][64]
      double* red = smem;
      static_assert((size_t)4 * 36 * 64 * sizeof(double) <= Cfg::SMEM, "reduction scratch fits in the operand ring");
      {
        int u = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
          for (int j = 0; j < 8; ++j)
            if (j <= i) {
              *reinterpret_cast<double2*>(red + ((size_t)(w * 36 + u) * 64) + g8 * 8 + 2 * t4) = make_double2(d0[i][j], d1[i][j]);
              ++u;
            }
      }
      __syncthreads();
      double* Pp = g.splitk > 1 ? g.part + ((long)split * g.batch + b) * (long)g.M * g.N : nullptr;
      double* Cb = g.C + (long)b * g.sC;
      for (int idx = tid; idx < 64 * 64; idx += THREADS) {
        const int r = idx >> 6, cc = idx & 63;
        const int i = r >> 3, j = cc >> 3;
        double v = 0.0;
        if (j <= i) {
          const int u = i * (i + 1) / 2 + j;
          const int e = (r & 7) * 8 + (cc & 7);
          v = ((red[(size_t)(0 * 36 + u) * 64 + e] + red[(size_t)(1 * 36 + u) * 64 + e]) + red[(size_t)(2 * 36 + u) * 64 + e]) +
              red[(size_t)(3 * 36 + u) * 64 + e];
        }
        if (Pp) Pp[(long)(m0 + r) * g.N + n0 + cc] = v;
        else {
          double* p = Cb + (long)(m0 + r) * g.ldc + n0 + cc;
          double o = g.alpha * v;
          if (g.beta != 0.0) o += g.beta * *p;
          *p = o;
        }
      }
      return;
    }
  }

  double c0[TM][TN], c1[TM][TN];
#pragma unroll
  for (int i = 0; i < TM; ++i)
#pragma unroll
    for (int j = 0; j < TN; ++j) { c0[i][j] = 0.0; c1[i][j] = 0.0; }

#pragma unroll
  for (int s = 0; s < STAGES - 1; ++s) {
    if (s < ktiles) load_stage(s, koff(s));
    cp_async_commit();
  }
  for (int kt = 0; kt < ktiles; ++kt) {
    cp_async_wait<STAGES - 2>();
    __syncthreads();
    {
      int nk = kt + STAGES - 1;
      if (nk < ktiles) load_stage(nk % STAGES, koff(nk));
      cp_async_commit();
    }
    const int st = kt % STAGES;
    const double* as = As + st * A_STAGE + (wm * TM * 8 + g8) * LDA + t4;
    const double* bs = NT ? Bs + st * B_STAGE + (wn * TN * 8 + g8) * LDB + t4
                          : Bs + st * B_STAGE + t4 * LDB + wn * TN * 8 + g8;
    const double* ss = Ss + st * BK + t4;
    double bsc[TN];
    if (!NT && g.bscale) {
      const double* bp = g.bscale + (long)(blk0 + kt / tpb) * g.ld_bscale + n0 + wn * TN * 8 + g8;
#pragma unroll
      for (int j = 0; j < TN; ++j) bsc[j] = g.bscale_mul * bp[j * 8];
    }
    // Two straight-line copies of the k-tile, with and without the operand scales: a predicated-off DMUL still queues on
    // the FP64 pipe the DMMAs use, so the unscaled products must not carry them at all.
    auto compute = [&](auto scaled) {
      constexpr bool SC = decltype(scaled)::value;
#pragma unroll
      for (int kk = 0; kk < BK / 4; ++kk) {
        double a[TM], bb[TN];
#pragma unroll
        for (int i = 0; i < TM; ++i) a[i] = as[i * 8 * LDA + kk * 4];
        if (SC && Sb) {
          double s = ss[kk * 4];
#pragma unroll
          for (int i = 0; i < TM; ++i) a[i] *= s;
        }
#pragma unroll
        for (int j = 0; j < TN; ++j) bb[j] = NT ? bs[j * 8 * LDB + kk * 4] : bs[kk * 4 * LDB + j * 8];
        if (SC && !NT && g.bscale) {
#pragma unroll
          for (int j = 0; j < TN; ++j) bb[j] *= bsc[j];
        }
#pragma unroll
        for (int i = 0; i < TM; ++i)
#pragma unroll
          for (int j = 0; j < TN; ++j) dmma884(c0[i][j], c1[i][j], a[i], bb[j]);
      }
    };
    bool skip = false;
    if (g.a_tri && gemm_tri_skip_enabled()) {
      const int kin = koff(kt) - (blk0 + kt / tpb) * kblk;   // k inside the (possibly concatenated) triangular block
      const int r0w = m0 + wm * TM * 8;               // first row of the warp
      skip = g.a_tri == 1 ? (kin > r0w + TM * 8 - 1) : (kin + BK - 1 < r0w);
    }
    if (skip) continue;
    if (Sb || (!NT && g.bscale)) compute(std::true_type());
    else compute(std::false_type());
  }
  cp_async_wait<0>();

  if (g.splitk > 1) {
    double* P = g.part + ((long)split * g.batch + b) * (long)g.M * g.N;
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
      for (int j = 0; j < TN; ++j) {
        int row = m0 + wm * TM * 8 + i * 8 + g8, col = n0 + wn * TN * 8 + j * 8 + 2 * t4;
        *reinterpret_cast<double2*>(P + (long)row * g.N + col) = make_double2(c0[i][j], c1[i][j]);
      }
  } else {
    double* Cb = g.C + (long)b * g.sC;
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
      for (int j = 0; j < TN; ++j) {
        int row = m0 + wm * TM * 8 + i * 8 + g8, col = n0 + wn * TN * 8 + j * 8 + 2 * t4;
        double2* p = reinterpret_cast<double2*>(Cb + (long)row * g.ldc + col);
        double2 v = make_double2(g.alpha * c0[i][j], g.alpha * c1[i][j]);
        if (g.beta != 0.0) { double2 o = *p; v.x += g.beta * o.x; v.y += g.beta * o.y; }
        if (g.epi_plane) {
          const double2 e = *reinterpret_cast<const double2*>(g.epi_plane + (long)row * g.ld_epi + col);
          v.x += g.epi_mul * g.epi_col[col] * e.x;
          v.y += g.epi_mul * g.epi_col[col + 1] * e.y;
        }
        *p = v;
      }
  }
}

// Sums split-K partials in split order (deterministic): C = alpha * sum_s part[s] + beta * C.
__global__ void gemm_splitk_reduce(GemmArgs g, int BM, int BN) {
  long total = (long)g.batch * g.M * g.N;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    int col = (int)(idx % g.N);
    long r = idx / g.N;
    int row = (int)(r % g.M);
    int b = (int)(r / g.M);
    if (g.c_lower && (col / BN) * BN >= (row / BM) * BM + BM) continue;
    double s = 0.0;
    for (int k = 0; k < g.splitk; ++k) s += g.part[((long)k * g.batch + b) * (long)g.M * g.N + (long)row * g.N + col];
    double* p = g.C + (long)b * g.sC + (long)row * g.ldc + col;
    double v = g.alpha * s;
    if (g.beta != 0.0) v += g.beta * *p;
    *p = v;
  }
}

template <int BM, int BN, int BK, int WM, int WN, bool NT, int STAGES, int TSEL = 0>
inline cudaError_t gemm_launch_cfg(const GemmArgs& g, cudaStream_t st, bool reduce = true) {
  using Cfg = GemmCfg<BM, BN, BK, WM, WN, NT, STAGES>;
  auto kern = gemm_kernel<BM, BN, BK, WM, WN, NT, STAGES, TSEL>;
  static bool configured[64] = {false};   // the opt-in shared-memory size is a per-device function attribute
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64 || !configured[dev]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64) configured[dev] = true;
  }
  long blocks = (long)(g.M / BM) * (g.N / BN) * g.batch * g.splitk;
  kern<<<(unsigned)blocks, Cfg::THREADS, Cfg::SMEM, st>>>(g);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  if (g.splitk > 1 && reduce) {
    long total = (long)g.batch * g.M * g.N;
    int rb = (int)((total + 255) / 256);
    if (rb > 148 * 8) rb = 148 * 8;
    gemm_splitk_reduce<<<rb, 256, 0, st>>>(g, BM, BN);
    e = cudaGetLastError();
  }
  return e;
}

// Tile shape the launcher will use and how many CTAs of it fit on the device at once (for wave-aware split-K choices).
struct GemmPlan { int BM, BN; long tiles; int slots; };

template <int BM, int BN, int BK, int WM, int WN, bool NT, int STAGES, int TSEL = 0>
inline int gemm_ctas_per_sm() {
  using Cfg = GemmCfg<BM, BN, BK, WM, WN, NT, STAGES>;
  static int cached = 0;
  if (!cached) {
    auto kern = gemm_kernel<BM, BN, BK, WM, WN, NT, STAGES, TSEL>;
    cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg::SMEM);
    int n = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, Cfg::THREADS, Cfg::SMEM) != cudaSuccess || n < 1) n = 1;
    cached = n;
  }
  return cached;
}

// NT products on 64x64 tiles (the contractions over the point-samples) run 32-deep k-tiles: half the barriers and loop
// bookkeeping per flop (measured -4% on the parameter adjoints; the short-K NN products are faster with 16)
inline bool gemm_small_bk32(const GemmArgs& g, bool nt) {
  if (!nt || g.K % 32) return false;
  if (g.kblocks > 1 && g.kblk % 32) return false;
  if (g.splitk > 1 && ((g.K / 32 + g.splitk - 1) / g.splitk) < 1) return false;
  return true;
}

// lower-only contraction over the point-samples on 64 x 64 x 32 tiles: strictly-lower and diagonal tiles as two launches (TSEL)
inline bool gemm_split_diag(const GemmArgs& g, bool nt) {
  return nt && g.c_lower && g.a_tri == 0 && g.kblocks <= 1 && g.M == g.N && g.M > 64 && g.K % 32 == 0 &&
         !((g.M % 128 == 0) && (g.N % 128 == 0) && ((long)g.M * g.N * g.batch >= 128L * 128 * 64));
}

inline bool gemm_uses_big_tiles(const GemmArgs& g) {
  return (g.M % 128 == 0) && (g.N % 128 == 0) && g.a_tri == 0 && ((long)g.M * g.N * g.batch >= 128L * 128 * 64);
}

inline GemmPlan gemm_plan(const GemmArgs& g, bool nt, int num_sms) {
  GemmPlan p;
  int per_sm;
  if (g.N == 32 && !nt) { p.BM = 64; p.BN = 32; per_sm = gemm_ctas_per_sm<64, 32, 16, 2, 1, false, 3>(); }
  else if (gemm_uses_big_tiles(g)) {
    p.BM = 128; p.BN = 128;
    per_sm = nt ? gemm_ctas_per_sm<128, 128, 16, 4, 4, true, 3>() : gemm_ctas_per_sm<128, 128, 16, 4, 4, false, 3>();
  } else {
    p.BM = 64; p.BN = 64;
    if (gemm_small_bk32(g, nt)) per_sm = nt ? gemm_ctas_per_sm<64, 64, 32, 2, 2, true, 3>() : gemm_ctas_per_sm<64, 64, 32, 2, 2, false, 3>();
    else per_sm = nt ? gemm_ctas_per_sm<64, 64, 16, 2, 2, true, 3>() : gemm_ctas_per_sm<64, 64, 16, 2, 2, false, 3>();
  }
  const long mt = g.M / p.BM, ntl = g.N / p.BN;
  long tiles = mt * ntl;
  if (g.c_lower) {
    tiles = 0;
    for (long i = 0; i < mt; ++i)
      for (long j = 0; j < ntl; ++j)
        if (j * p.BN < i * p.BM + p.BM) ++tiles;
  }
  if (p.BM == 64 && gemm_small_bk32(g, nt) && gemm_split_diag(g, nt)) {   // the wave that matters is the strictly-lower launch
    per_sm = gemm_ctas_per_sm<64, 64, 32, 2, 2, true, 2, 1>();
    tiles -= mt;
  }
  p.tiles = tiles * g.batch;
  p.slots = per_sm * num_sms;
  return p;
}

// Picks a tile configuration. Returns cudaErrorInvalidValue when the shape is not tile-aligned.
inline cudaError_t gemm_launch(const GemmArgs& g, bool nt, cudaStream_t st) {
  if (g.M % 64 || g.K % 16 || g.splitk < 1 || (g.splitk > 1 && !g.part)) return cudaErrorInvalidValue;
  if (g.epi_plane && (g.splitk != 1 || g.batch != 1)) return cudaErrorInvalidValue;
  if (g.kblocks > 1 && (nt || g.splitk > g.kblocks || g.kblk % 16 || g.kblocks * g.kblk != g.K || g.a_tri == 2)) return cudaErrorInvalidValue;
  if (g.N == 32 && !nt) return gemm_launch_cfg<64, 32, 16, 2, 1, false, 3>(g, st);
  if (g.N % 64) return cudaErrorInvalidValue;
  if (gemm_uses_big_tiles(g)) {
    return nt ? gemm_launch_cfg<128, 128, 16, 4, 4, true, 3>(g, st) : gemm_launch_cfg<128, 128, 16, 4, 4, false, 3>(g, st);
  }
  if (gemm_small_bk32(g, nt)) {
    // lower-only contraction over the point-samples: the strictly-lower tiles and the diagonal tiles as two launches (see TSEL)
    if (gemm_split_diag(g, nt)) {
      cudaError_t e = gemm_launch_cfg<64, 64, 32, 2, 2, true, 2, 1>(g, st, false);
      if (e != cudaSuccess) return e;
      return gemm_launch_cfg<64, 64, 32, 2, 2, true, 3, 2>(g, st, true);
    }
    return nt ? gemm_launch_cfg<64, 64, 32, 2, 2, true, 3>(g, st) : gemm_launch_cfg<64, 64, 32, 2, 2, false, 3>(g, st);
  }
  return nt ? gemm_launch_cfg<64, 64, 16, 2, 2, true, 3>(g, st) : gemm_launch_cfg<64, 64, 16, 2, 2, false, 3>(g, st);
}

}  // namespace dgp
