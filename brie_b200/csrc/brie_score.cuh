// Score-test parts of candidate cell covariates from one model's fitted posterior (DESIGN §2.3).
//
// With the model's W, b and sigma as fitted (the null model of the test), the posterior of Z factorises over
// (cell, event) and, per event g and candidate j,
//   r_cg = (Z_loc[c, g] - m_cg) / sigma^2                     posterior-mean residual, m_cg the prior mean
//   w_cg = max(sigma^2 - s_cg^2, 0) / sigma^4                 Louis' weight, as in the Wald pass (brie_wald.cuh)
//   U_gj = sum_c x_cj r_cg     A_gj = sum_c w_cg x_cj^2     B_gjk = sum_c w_cg x_cj x~_ck     Ut_gk = sum_c x~_ck r_cg
// x_cj is candidate j, x~_c the model's design row (Xc columns in mask order, then the intercept's 1 when it is
// per-event and trained).  The host turns these and I_g (brie_fit_wald_info) into the efficient score and its
// information (engine.score_from_parts).
//
// score_parts_kernel: CTA = 32 events (one per lane) x a block of JB candidates x a block of KB x~ columns x one
// chunk of cell rows (the Wald pass's chunks, a function of the cell count alone).  Each staged batch of kWaldBatch
// rows holds the block's candidate values and x~ columns in shared memory as float64; warp r takes rows r, r + 8, ...
// of a batch, computes r_cg and w_cg once in float64 (the prior mean too) and accumulates every part of the block in
// float64 registers.  The 8 warps' sums are added in warp order through shared memory and the CTA writes one partial
// per (chunk, output, event); score_reduce_kernel adds the chunks in chunk order.  No atomics: repeated calls are
// bit-identical, and so are event chunks and shards of a fit.  U and A are written by the CTAs of x~ block 0, Ut by
// those of candidate block 0.  FP64 on the CUDA cores: the sums over cells cancel, which TF32 / BF16 cannot carry.
#pragma once
#include <stdint.h>

#include "brie_kernels.cuh"
#include "brie_wald.cuh"

namespace brie {

constexpr int kScoreCols = 32;       // events per CTA
constexpr int kScoreRowGroups = 8;   // warps per CTA
constexpr int kScoreRed = 4;         // parts per round of the in-CTA reduction: 8 x 4 x 32 doubles

struct ScoreArgs {
  int64_t Nc, Ng, ld;
  int m;                // the model
  // prior_mean's fields (whole-fit buffers, indexed by m)
  const float* Xc; const float* Wc; const float* Wg; const float* Xg;
  int32_t KC, KG;
  const float* Zl; const float* Zs;   // (M, Nc, ld)
  const float* b;       // intercept: (M, ld) per event, or (M, Nc) per cell (cell_mode)
  const float* tau;     // sigma_log, laid out as b
  int cell_mode;
  const float* X;       // (Nc, ldx) candidates
  int64_t ldx;
  int J;                // candidates
  int width, wide, kt;  // x~: `width` Xc columns (wald_xc_col), kt = width + the intercept's 1
  uint32_t xc_mask;
  int64_t rows_per_chunk;
  int n_jblk, n_kblk;
  int64_t n_q;          // outputs per event: U (J), A (J), B (J kt, row-major), Ut (kt)
  double* part;         // (n_chunks, n_q, ld)
};

// Output index of accumulator v of the CTA at candidate block jblk, x~ block kblk, or -1 when another CTA writes it
// (or it lies past J / kt).  Accumulators: U (JB), A (JB), B (JB x KB, row-major), Ut (KB).
template <int JB, int KB>
__device__ __forceinline__ int64_t score_q(const ScoreArgs& a, int v, int jblk, int kblk) {
  const int j0 = jblk * JB, k0 = kblk * KB;
  if (v < 2 * JB) {
    const int j = j0 + (v % JB);
    if (kblk != 0 || j >= a.J) return -1;
    return v < JB ? j : (int64_t)a.J + j;
  }
  if (v < 2 * JB + JB * KB) {
    const int j = j0 + (v - 2 * JB) / KB, k = k0 + (v - 2 * JB) % KB;
    if (j >= a.J || k >= a.kt) return -1;
    return 2 * (int64_t)a.J + (int64_t)j * a.kt + k;
  }
  const int k = k0 + v - 2 * JB - JB * KB;
  if (jblk != 0 || k >= a.kt) return -1;
  return (int64_t)a.J * (a.kt + 2) + k;
}

template <int JB, int KB>
__global__ void __launch_bounds__(kScoreCols * kScoreRowGroups) score_parts_kernel(const ScoreArgs a) {
  constexpr int NV = JB * (2 + KB) + KB;
  constexpr int IU = 0, IA = JB, IB = 2 * JB, IT = 2 * JB + JB * KB;
  __shared__ double s_x[kWaldBatch][JB];
  __shared__ double s_t[kWaldBatch][KB];
  __shared__ double s_red[kScoreRowGroups * kScoreRed * kScoreCols];
  __shared__ int s_col[KB];   // Xc column of the block's x~ columns (-1: intercept, -2: none)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int bx = blockIdx.x;   // candidate blocks of one event tile are neighbours: they read the same Z planes
  const int jblk = bx % a.n_jblk;
  bx /= a.n_jblk;
  const int kblk = bx % a.n_kblk, tile = bx / a.n_kblk;
  const int j0 = jblk * JB, k0 = kblk * KB;
  const int64_t g = (int64_t)tile * kScoreCols + lane;
  const bool ev_ok = g < a.Ng;
  const int64_t c0 = (int64_t)blockIdx.y * a.rows_per_chunk;
  const int64_t c1 = min(c0 + a.rows_per_chunk, a.Nc);
  const int64_t xc_stride = a.KC > 0 ? a.KC : 1;
  const float* Xm = a.Xc + (int64_t)a.m * a.Nc * xc_stride;
  const int64_t zoff = (int64_t)a.m * a.Nc * a.ld;

  if (threadIdx.x < KB) {
    const int k = k0 + threadIdx.x;
    s_col[threadIdx.x] = k < a.kt ? wald_xc_col(a.width, a.wide, a.xc_mask, k) : -2;
  }

  double tau_e = 0.0, scale_e = 0.0, b_e = 0.0;   // per-event sigma and intercept, once
  if (!a.cell_mode && ev_ok) {
    tau_e = (double)a.tau[(int64_t)a.m * a.ld + g];
    scale_e = exp(-2.0 * tau_e);
    b_e = (double)a.b[(int64_t)a.m * a.ld + g];
  }
  double acc[NV];
#pragma unroll
  for (int v = 0; v < NV; ++v) acc[v] = 0.0;

  for (int64_t r0 = c0; r0 < c1; r0 += kWaldBatch) {
    __syncthreads();   // the previous batch is consumed (and s_col is written, first time round)
    for (int i = threadIdx.x; i < kWaldBatch * (JB + KB); i += blockDim.x) {
      const int r = i / (JB + KB), q = i % (JB + KB);
      const int64_t c = r0 + r;
      double v = 0.0;
      if (q < JB) {
        if (c < c1 && j0 + q < a.J) v = (double)a.X[c * a.ldx + j0 + q];
        s_x[r][q] = v;
      } else {
        const int ck = s_col[q - JB];
        if (c < c1 && ck > -2) v = ck >= 0 ? (double)Xm[c * xc_stride + ck] : 1.0;
        s_t[r][q - JB] = v;
      }
    }
    __syncthreads();
#pragma unroll 1
    for (int jj = 0; jj < kWaldBatch / kScoreRowGroups; ++jj) {
      const int r = warp + jj * kScoreRowGroups;
      const int64_t c = r0 + r;
      double res = 0.0, w = 0.0;
      if (c < c1 && ev_ok) {
        const double mu = (double)a.Zl[zoff + c * a.ld + g], lam = (double)a.Zs[zoff + c * a.ld + g];
        double tau = tau_e, scale = scale_e, base = b_e;
        if (a.cell_mode) {
          tau = (double)a.tau[(int64_t)a.m * a.Nc + c];
          scale = exp(-2.0 * tau);
          base = (double)a.b[(int64_t)a.m * a.Nc + c];
        }
        res = (mu - prior_mean(a, a.m, c, g, base)) * scale;
        w = fmax(-expm1(2.0 * (lam - tau)), 0.0) * scale;
      }
      double t[KB];
#pragma unroll
      for (int k = 0; k < KB; ++k) t[k] = s_t[r][k];
#pragma unroll
      for (int j = 0; j < JB; ++j) {
        const double x = s_x[r][j];
        const double wx = w * x;
        acc[IU + j] = fma(x, res, acc[IU + j]);
        acc[IA + j] = fma(wx, x, acc[IA + j]);
#pragma unroll
        for (int k = 0; k < KB; ++k) acc[IB + j * KB + k] = fma(wx, t[k], acc[IB + j * KB + k]);
      }
#pragma unroll
      for (int k = 0; k < KB; ++k) acc[IT + k] = fma(t[k], res, acc[IT + k]);
    }
  }

  // warps 0..7 added in order; kScoreRed parts per round
  double* out = a.part + (int64_t)blockIdx.y * a.n_q * a.ld;
#pragma unroll
  for (int v0 = 0; v0 < NV; v0 += kScoreRed) {
    __syncthreads();
#pragma unroll
    for (int i = 0; i < kScoreRed; ++i)
      if (v0 + i < NV) s_red[(warp * kScoreRed + i) * kScoreCols + lane] = acc[v0 + i];
    __syncthreads();
    if (threadIdx.x < kScoreRed * kScoreCols) {
      const int i = threadIdx.x / kScoreCols, e = threadIdx.x % kScoreCols;
      const int v = v0 + i;
      const int64_t ge = (int64_t)tile * kScoreCols + e;
      const int64_t q = v < NV ? score_q<JB, KB>(a, v, jblk, kblk) : -1;
      if (q >= 0 && ge < a.Ng) {
        double s = 0.0;
        for (int wp = 0; wp < kScoreRowGroups; ++wp) s += s_red[(wp * kScoreRed + i) * kScoreCols + e];
        out[q * a.ld + ge] = s;
      }
    }
  }
}

// Sum over chunks, in chunk order, of part[chunk, q, g] into U (Ng, J), A (Ng, J), B (Ng, J, kt), Ut (Ng, kt).
// Consecutive threads take consecutive events: the partials are read coalesced.
__global__ void __launch_bounds__(256) score_reduce_kernel(const double* __restrict__ part, int n_chunks, int64_t n_q,
                                                           int64_t ld, int64_t Ng, int J, int kt, double* U, double* A,
                                                           double* B, double* Ut) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Ng * n_q) return;
  const int64_t q = i / Ng, g = i % Ng;
  const int64_t plane = n_q * ld;
  double s = 0.0;
  for (int ch = 0; ch < n_chunks; ++ch) s += part[ch * plane + q * ld + g];
  const int64_t nb = (int64_t)J * kt;
  if (q < J) U[g * J + q] = s;
  else if (q < 2 * J) A[g * J + q - J] = s;
  else if (q < 2 * J + nb) B[g * nb + q - 2 * J] = s;
  else Ut[g * kt + q - 2 * J - nb] = s;
}

// Cross terms of the joint score test of a group of candidates (DESIGN §2.4): for a table of candidate pairs (j, j'),
//   A_gjj' = sum_c w_cg x_cj x_cj'
// with w_cg the Louis weight above.  The diagonal (j = j') is score_parts_kernel's A.
//
// score_cross_kernel: CTA = 32 events (one per lane) x one block of PB pairs x one chunk of cell rows (the Wald pass's
// chunks).  Each staged batch of kWaldBatch rows has its pair products x_cj x_cj' in shared memory (float64, exact for
// float32 inputs); warp r takes rows r, r + 8, ... of a batch, computes w_cg once per (row, event) and accumulates
// in float64 registers.  The 8 warps' sums are added in warp order and the CTA writes one partial per (chunk, pair,
// event); wald_reduce_kernel adds the chunks in chunk order.  No atomics: repeated calls, pair blocks, event chunks
// and shards give the same bits.
struct CrossArgs {
  int64_t Nc, Ng, ld;
  const float* Zs;      // (Nc, ld) Z_std_log of the model
  const float* tau;     // sigma_log of the model: (ld) per event, or (Nc) per cell (cell_tau)
  int cell_tau;
  const float* X;       // (Nc, ldx) candidates
  int64_t ldx;
  const int32_t* pairs; // (n_pairs, 2) candidate columns, device
  int n_pairs;
  int64_t rows_per_chunk;
  int n_tiles;
  double* part;         // (n_chunks, n_pairs, ld)
};

template <int PB>
__global__ void __launch_bounds__(kWaldCols * kWaldRowGroups) score_cross_kernel(const CrossArgs a) {
  static_assert(PB % kWaldRedPairs == 0 && PB <= kWaldMaxPairs, "pair block");
  __shared__ double s_buf[kWaldBatch * kWaldMaxPairs];   // staged pair products, then the reduction
  __shared__ int s_col[2][PB];                            // candidate columns of the block's pairs (-1: none)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int tile = blockIdx.x % a.n_tiles, pblk = blockIdx.x / a.n_tiles;
  const int p0 = pblk * PB;
  const int64_t g = (int64_t)tile * kWaldCols + lane;
  const bool ev_ok = g < a.Ng;
  const int64_t c0 = (int64_t)blockIdx.y * a.rows_per_chunk;
  const int64_t c1 = min(c0 + a.rows_per_chunk, a.Nc);

  if (threadIdx.x < PB) {
    const int p = p0 + threadIdx.x;
    s_col[0][threadIdx.x] = p < a.n_pairs ? a.pairs[2 * p] : -1;
    s_col[1][threadIdx.x] = p < a.n_pairs ? a.pairs[2 * p + 1] : -1;
  }

  double tau_w = 0.0, scale_w = 0.0;   // per-event sigma: tau and exp(-2 tau) once
  if (!a.cell_tau && ev_ok) {
    tau_w = (double)a.tau[g];
    scale_w = exp(-2.0 * tau_w);
  }
  double acc[PB];
#pragma unroll
  for (int p = 0; p < PB; ++p) acc[p] = 0.0;

  for (int64_t r0 = c0; r0 < c1; r0 += kWaldBatch) {
    __syncthreads();   // the previous batch is consumed (and s_col is written, first time round)
    for (int i = threadIdx.x; i < kWaldBatch * PB; i += blockDim.x) {
      const int r = i / PB, q = i % PB;
      const int64_t c = r0 + r;
      const int j = s_col[0][q], k = s_col[1][q];
      double v = 0.0;
      if (c < c1 && j >= 0) {
        const float* x = a.X + c * a.ldx;
        v = (double)x[j] * (double)x[k];
      }
      s_buf[r * PB + q] = v;
    }
    __syncthreads();
#pragma unroll
    for (int jj = 0; jj < kWaldBatch / kWaldRowGroups; ++jj) {
      const int r = warp + jj * kWaldRowGroups;
      const int64_t c = r0 + r;
      double w = 0.0;
      if (c < c1 && ev_ok) {
        const double lam = (double)a.Zs[c * a.ld + g];
        double tau = tau_w, scale = scale_w;
        if (a.cell_tau) {
          tau = (double)a.tau[c];
          scale = exp(-2.0 * tau);
        }
        w = fmax(-expm1(2.0 * (lam - tau)), 0.0) * scale;
      }
#pragma unroll
      for (int p = 0; p < PB; ++p) acc[p] = fma(w, s_buf[r * PB + p], acc[p]);
    }
  }

  // warps 0..7 added in order; kWaldRedPairs pairs per round
  const int64_t plane = (int64_t)a.n_pairs * a.ld;
  double* out = a.part + (int64_t)blockIdx.y * plane;
#pragma unroll
  for (int q0 = 0; q0 < PB; q0 += kWaldRedPairs) {
    __syncthreads();
#pragma unroll
    for (int i = 0; i < kWaldRedPairs; ++i) s_buf[(warp * kWaldRedPairs + i) * kWaldCols + lane] = acc[q0 + i];
    __syncthreads();
    if (threadIdx.x < kWaldRedPairs * kWaldCols) {
      const int i = threadIdx.x / kWaldCols, e = threadIdx.x % kWaldCols;
      const int p = p0 + q0 + i;
      const int64_t ge = (int64_t)tile * kWaldCols + e;
      double s = 0.0;
      for (int wp = 0; wp < kWaldRowGroups; ++wp) s += s_buf[(wp * kWaldRedPairs + i) * kWaldCols + e];
      if (p < a.n_pairs && ge < a.Ng) out[(int64_t)p * a.ld + ge] = s;
    }
  }
}

}  // namespace brie
