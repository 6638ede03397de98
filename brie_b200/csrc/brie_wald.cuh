// Observed information of one model's per-event regression parameters from its fitted posterior (DESIGN §2.2).
//
// Given W, b and sigma, the exact posterior of Z factorises over (cell, event), so Louis' missing-information
// formula gives the information of the coefficients of event g as
//   I_g = sum_c w_cg x~_c x~_c^T,   w_cg = max(sigma^2 - s_cg^2, 0) / sigma^4 = max(-expm1(2 (lambda - tau)), 0) exp(-2 tau)
// with s_cg = exp(Z_std_log[c, g]) and tau = sigma_log (the event's value, or the cell's in cell mode).
// x~_c is the model's design row: its Xc columns in mask order, then a 1 when the intercept is per-event and trained.
//
// wald_info_kernel: CTA = 32 events (one per lane) x one block of PB pairs (k <= l, row-major over x~) x one chunk
// of cell rows.  Each staged batch of kWaldBatch rows has its pair products x~_ck x~_cl in shared memory (float64,
// exact); warp r takes rows r, r + 8, ... of a batch and accumulates w_cg x~_ck x~_cl in float64 registers.  The
// 8 warps' sums are added in warp order through shared memory and the CTA writes one partial per (chunk, pair,
// event); wald_reduce_kernel adds the chunks in chunk order.  No atomics: repeated calls are bit-identical, and as the
// chunks depend on the number of cells alone, so is the same fit split into event chunks or shards.
// Z_std_log is read once per pair block, so the pass costs ceil(n_pairs / PB) reads of the model's (cells, events)
// plane.
#pragma once
#include <stdint.h>

namespace brie {

constexpr int kWaldCols = 32;       // events per CTA
constexpr int kWaldRowGroups = 8;   // warps per CTA
constexpr int kWaldBatch = 32;      // cell rows staged per batch
constexpr int kWaldMaxPairs = 36;   // widest pair block (the largest instantiation)
constexpr int kWaldRedPairs = 4;    // pairs per round of the in-CTA reduction: 8 x 4 x 32 doubles
constexpr int kWaldMinRows = 256;   // cell rows per chunk, at least ...
constexpr int kWaldMaxChunks = 64;  // ... and at most this many chunks (brie_fit_wald_info picks from n_cells alone)

struct WaldArgs {
  int64_t Nc, Ng, ld;
  const float* Zs;      // (Nc, ld) Z_std_log of the model
  const float* tau;     // sigma_log of the model: (ld) per event, or (Nc) per cell (cell_tau)
  const float* Xc;      // (Nc, xc_stride) design of the model
  int xc_stride;
  int width;            // x~ columns taken from Xc
  uint32_t xc_mask;     // !wide: x~ column j is Xc column (j-th set bit of xc_mask); wide: column j
  int wide;
  int has_b;            // x~ column `width` is the intercept's 1
  int n_pairs;          // kt (kt + 1) / 2, kt = width + has_b
  int cell_tau;
  int64_t rows_per_chunk;
  int n_tiles;          // event tiles of kWaldCols
  double* part;         // (n_chunks, n_pairs, ld)
};

// Xc column of x~ column j of a model whose x~ takes `width` Xc columns (!wide: the j-th set bit of xc_mask; wide:
// column j), or -1 for the intercept's 1.  Shared by the Wald and score passes (brie_score.cuh).
__device__ __forceinline__ int wald_xc_col(int width, int wide, uint32_t xc_mask, int j) {
  if (j >= width) return -1;
  if (wide) return j;
  int seen = 0;
  for (int k = 0; k < 32; ++k)
    if ((xc_mask >> k) & 1u) {
      if (seen == j) return k;
      ++seen;
    }
  return -1;
}

template <int PB>
__global__ void __launch_bounds__(kWaldCols * kWaldRowGroups) wald_info_kernel(const WaldArgs a) {
  static_assert(PB % kWaldRedPairs == 0 && PB <= kWaldMaxPairs, "pair block");
  __shared__ double s_buf[kWaldBatch * kWaldMaxPairs];   // staged pair products, then the reduction
  __shared__ int s_col[2][PB];                            // Xc columns of the block's pairs (-1: intercept, -2: none)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int tile = blockIdx.x % a.n_tiles, pblk = blockIdx.x / a.n_tiles;
  const int p0 = pblk * PB;
  const int64_t g = (int64_t)tile * kWaldCols + lane;
  const bool ev_ok = g < a.Ng;
  const int64_t c0 = (int64_t)blockIdx.y * a.rows_per_chunk;
  const int64_t c1 = min(c0 + a.rows_per_chunk, a.Nc);

  if (threadIdx.x < PB) {
    const int p = p0 + threadIdx.x;
    int ck = -2, cl = -2;
    if (p < a.n_pairs) {   // p -> (k, l), k <= l, row-major over the upper triangle
      const int kt = a.width + a.has_b;
      int k = 0, first = 0;
      while (p >= first + (kt - k)) {
        first += kt - k;
        ++k;
      }
      ck = wald_xc_col(a.width, a.wide, a.xc_mask, k);
      cl = wald_xc_col(a.width, a.wide, a.xc_mask, k + (p - first));
    }
    s_col[0][threadIdx.x] = ck;
    s_col[1][threadIdx.x] = cl;
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
      const int ck = s_col[0][q], cl = s_col[1][q];
      double v = 0.0;
      if (c < c1 && ck > -2) {
        const float* x = a.Xc + c * a.xc_stride;
        const double xk = ck >= 0 ? (double)x[ck] : 1.0;
        const double xl = cl >= 0 ? (double)x[cl] : 1.0;
        v = xk * xl;
      }
      s_buf[r * PB + q] = v;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < kWaldBatch / kWaldRowGroups; ++j) {
      const int r = warp + j * kWaldRowGroups;
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

// info[g * n_pairs + p] = sum over chunks, in chunk order, of part[chunk, p, g]
__global__ void __launch_bounds__(256) wald_reduce_kernel(const double* __restrict__ part, int n_chunks, int n_pairs,
                                                          int64_t ld, int64_t Ng, double* info) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= Ng * n_pairs) return;
  const int64_t g = i / n_pairs, p = i % n_pairs;
  const int64_t plane = (int64_t)n_pairs * ld;
  double s = 0.0;
  for (int ch = 0; ch < n_chunks; ++ch) s += part[ch * plane + p * ld + g];
  info[i] = s;
}

}  // namespace brie
