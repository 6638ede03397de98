// target = "marginLik" (SURVEY f4): the prior-sampled log-mean-exp objective of
// BRIE2.get_loss / logLik_MC (brie/models/model_TFProb.py:156-157, 188-189, 202-205):
//   loss = - sum_{c,g} log( (1/S) sum_s exp l(z_s) ),   z_s = m_cg + sigma * eps_s,
// m the prior mean (:118-127).  Only the prior's parameters are read inside loss_fn, so only
// intercept / sigma_log / Wc / Wg are trained; Z_loc and Z_std_log keep their initial values.
// An element without reads has l == 0 for every z: it contributes nothing to the loss or to
// any gradient, so only the 13-19 % of elements with reads do any work here and the pass reads
// the counts only (12 B per cell x event; no per-element state).
//
// With w_s = softmax_s(l_s), g_s = dl/dz:   d loss/d m = -sum_s w_s g_s =: -G,
// d loss/d sigma_log = -sigma sum_s w_s g_s eps_s =: -H; then the same per-event / per-cell
// reductions and Adam kernels as the ELBO step (event_update_kernel, cell_*_kernel).
#pragma once
#include "brie_kernels.cuh"

namespace brie {

struct MarginArgs {
  int64_t Nc, Ng, ld, event_offset;
  uint64_t seed;
  const float* c[3];
  const float* eff;
  const float* Xc; const float* Xg;
  const float* Wc; const float* b; const float* tau; const float* Wg;
  const uint8_t* active;
  float* part_ev;      // (n_row_chunks, M, NEV, ld)
  float* part_cell;    // (n_col_tiles, M, Nc, NCELL)
  uint32_t step, model_mask;
  int32_t M, S, rows_per_cta, KC, KG, cell_mode, NEV, NCELL;
  int32_t model_id[kMaxModels];
};

constexpr int kMarginTile = 128;   // events per CTA column tile: 4 segments of 32, lane = one event per segment
constexpr int kMarginMaxCell = BRIE_MAX_KG + 2;

// One element with reads: S prior samples, streaming log-sum-exp of the sample log-likelihoods
// with the softmax-weighted gradient sums carried along.  IEEE-accurate math.
__device__ __forceinline__ void margin_element(float pm, float sig, float c1, float c2, float n, float L1, float L2,
                                               float L3, bool eff, int S, uint32_t event, uint32_t cell,
                                               uint32_t step, uint32_t stream0, uint64_t seed, float& lme,
                                               float& G, float& H) {
  float mx = -INFINITY, Z = 0.f, A = 0.f, B = 0.f;
  const float ndL = n * (L1 - L2);
  for (int s0 = 0; s0 < S; s0 += 4) {
    float eps[4];
    brie_normals4(event, cell, step, stream0 + (uint32_t)(s0 >> 2), seed, eps);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (s0 + q < S) {
        const SampleLL r = sample_ll(fmaf(sig, eps[q], pm), c1, c2, n, L1, L2, L3, eff);
        const float gz = fmaf(c1, r.q, -c2 * r.psi) - ndL * (r.psi * r.q) / r.D;
        if (r.l > mx) {
          const float sc = expf(mx - r.l);   // 0 on the first sample
          Z *= sc; A *= sc; B *= sc;
          mx = r.l;
        }
        const float w = expf(r.l - mx);
        Z += w;
        A = fmaf(w, gz, A);
        B = fmaf(w * gz, eps[q], B);
      }
    }
  }
  lme = mx + logf(Z) - logf((float)S);
  G = A / Z;
  H = B / Z * sig;
}

// grid = (M, ceil(ld / 128), n_row_chunks), 8 warps; dynamic smem = 8 x NEV x 128 floats:
// every warp keeps its per-event partial sums in its own shared-memory slab (a lane only ever
// touches its own 4 columns, so no synchronisation until the end) -- they are updated for
// elements with reads only, which keeps the register budget independent of Kc.
__global__ void __launch_bounds__(kThreads) margin_step_kernel(const MarginArgs a) {
  const int m = blockIdx.x;
  if (!((a.model_mask >> m) & 1u)) return;
  const int tile = blockIdx.y, chunk = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t gbase = (int64_t)tile * kMarginTile;
  bool act[4];
  bool any = false;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int64_t g = gbase + j * 32 + lane;
    act[j] = g < a.Ng && a.active[(int64_t)m * a.ld + g] != 0;
    any |= act[j];
  }
  if (!__syncthreads_or(any)) return;

  extern __shared__ __align__(128) float smem[];
  float* acc = smem + warp * a.NEV * kMarginTile;
  for (int i = lane; i < a.NEV * kMarginTile; i += 32) acc[i] = 0.f;
  __syncwarp();

  const bool eff = a.eff != nullptr;
  const bool cell = a.cell_mode != 0;
  const int64_t row_begin = (int64_t)chunk * a.rows_per_cta;
  const int64_t row_end = min(row_begin + (int64_t)a.rows_per_cta, a.Nc);
  const uint32_t stream0 = brie_stream_word(BRIE_PHASE_TRAIN, (uint32_t)a.model_id[m], 0u);
  const int KC = a.KC, KG = a.KG;
  const int i_loss = a.NEV - 1;

  for (int64_t row = row_begin + warp; row < row_end; row += kWarps) {
    float cacc[kMarginMaxCell];
#pragma unroll
    for (int i = 0; i < kMarginMaxCell; ++i) cacc[i] = 0.f;
    const float* xrow = a.Xc + ((int64_t)m * a.Nc + row) * KC;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int col = j * 32 + lane;
      const int64_t g = gbase + col;
      if (!act[j]) continue;
      const int64_t off = row * a.ld + g;
      const float c1 = a.c[0][off], c2 = a.c[1][off], c3 = a.c[2] ? a.c[2][off] : 0.f;
      const float n = c1 + c2 + c3;
      if (!(n > 0.f)) continue;
      const float pm = prior_mean(a, m, row, g, cell ? a.b[(int64_t)m * a.Nc + row] : a.b[(int64_t)m * a.ld + g]);
      const float tj = cell ? a.tau[(int64_t)m * a.Nc + row] : a.tau[(int64_t)m * a.ld + g];
      float L1, L2, L3;
      event_lengths(a.eff, a.ld, g, L1, L2, L3);
      const float k0 = log_length_const(eff, c1, c2, c3, L1, L2, L3);
      float lme, G, H;
      margin_element(pm, expf(tj), c1, c2, n, L1, L2, L3, eff, a.S, (uint32_t)(a.event_offset + g), (uint32_t)row,
                     a.step, stream0, a.seed, lme, G, H);
      for (int k = 0; k < KC; ++k) acc[k * kMarginTile + col] = fmaf(-xrow[k], G, acc[k * kMarginTile + col]);
      if (!cell) {
        acc[KC * kMarginTile + col] -= G;
        acc[(KC + 1) * kMarginTile + col] -= H;
      }
      acc[i_loss * kMarginTile + col] -= lme + k0;
#pragma unroll
      for (int k = 0; k < BRIE_MAX_KG; ++k)
        if (k < KG) cacc[k] = fmaf(-a.Xg[g * KG + k], G, cacc[k]);
      if (cell) {
#pragma unroll
        for (int k = 0; k <= BRIE_MAX_KG; ++k)      // slots KG, KG + 1 (static indices keep cacc in registers)
          if (k == KG) { cacc[k] -= G; cacc[k + 1] -= H; }
      }
    }
    if (a.NCELL > 0) {
#pragma unroll
      for (int i = 0; i < kMarginMaxCell; ++i) {
        if (i < a.NCELL) {
          const float s = warp_sum(cacc[i]);
          if (lane == 0) a.part_cell[(((int64_t)tile * a.M + m) * a.Nc + row) * a.NCELL + i] = s;
        }
      }
    }
  }
  __syncthreads();
  if (threadIdx.x < kMarginTile && gbase + threadIdx.x < a.ld) {
    for (int i = 0; i < a.NEV; ++i) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) s += smem[(w * a.NEV + i) * kMarginTile + threadIdx.x];
      a.part_ev[(((int64_t)chunk * a.M + m) * a.NEV + i) * a.ld + gbase + threadIdx.x] = s;
    }
  }
}

}  // namespace brie
