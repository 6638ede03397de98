// Device kernels of the BRIE2 variational fit for sm_100a.
//
// Hot path replaced: one optimisation step of `tfp.math.minimize` over
// BRIE2.get_loss (brie/models/model_TFProb.py:194-211, 130-191, 118-127) plus the
// keras Adam update and the Variable constraints (:68-69, :80-81).  The reference
// materialises ~17 (S,Nc,Ng[,3]) tensors forward and as many backward; here one
// pass over the (cells, events) state does sampling, likelihood, KL, analytic
// gradients and Adam, reading 24 B + writing 24 B of state and reading 4 B of
// counts (packed dictionary codes; 12 B as float32 tiles) per cell x event
// (HBM-bound; see DESIGN.md).
//
// Layout: every (cells, events) array is row-major, events contiguous, leading
// dimension ld (ld % 4 == 0 is all the kernels need; the Python layer pads ld to 128
// floats so that rows start 512-byte aligned, +2-5 % on B200, profiles/r2_ab_rpi_tma.md).
// A warp owns a 128-event row segment (lane = 4
// consecutive events, one 16-byte load per array), a CTA of 8 warps owns
// rows_per_cta x 128 and walks its rows warp-interleaved.  Per-event sums over
// cells live in registers and leave the CTA as one partial per row chunk
// (deterministic two-stage reduction, no atomics); per-cell sums over events
// (gene-feature weights, per-cell intercept/sigma) are warp-shuffle reduced per
// row and leave as one partial per column tile.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "brie_philox.h"

namespace brie {

constexpr int kTileCols = 128;  // events per warp row segment
constexpr int kWarps = 8;
constexpr int kThreads = kWarps * 32;
constexpr int kMaxModels = 32;
constexpr int kMinCtas = 2;  // resident CTAs per SM the step kernel is register-budgeted for

constexpr float kB1c = 0.1f;     // 1 - beta_1 (keras Adam)
constexpr float kB2c = 0.001f;   // 1 - beta_2
constexpr float kAdamEps = 1e-7f;
constexpr float kZ975 = 1.959963984540054f;

struct StepArgs {
  int64_t Nc, Ng, ld, event_offset;
  uint64_t seed;
  const float* c[3];
  const float* eff;  // (3, ld) or null
  const float* Xc;   // (M, Nc, KC): per-model design matrix (unused columns are zero)
  const float* Xg;   // (Ng, KG)
  float* Zl;         // (M, Nc, ld)
  float* Zs;
  float* aZ;         // (4, M, Nc, ld)
  const float* Wc;   // (M, KC, ld)
  const float* b;    // (M, ld) | (M, Nc)
  const float* tau;
  const float* Wg;   // (M, Nc, KG)
  const uint8_t* active;  // (M, ld)
  float* part_ev;    // (n_row_chunks, M, NEV, ld)
  float* part_cell;  // (n_col_tiles, M, Nc, NCELL)
  float alpha;
  float inv_S;
  uint32_t step;
  // Two-step passes (PAIR instantiations, gene mode with per-event parameters only): the pass takes step `step` with
  // the parameters in `prev` ((M, KC + 2, ld): Wc rows, intercept, sigma_log) and `alpha`, then step `step` + 1 with
  // Wc / b / tau and `alpha2`, and leaves in part_st the statistics of the state it writes around Wc / b / tau
  // (pair_stat_rows, brie_fit_run_steps).
  float alpha2;
  const float* prev;
  float* part_st;    // (n_row_chunks, M, KC + 3, ld)
  uint32_t model_mask;  // bit m: model m has any active event
  int32_t M, S, rows_per_cta;
  int32_t model_id[kMaxModels];
  // Optional column compaction (extension rounds, when most reference batches have converged):
  // model m visits only the 8-event blocks blk_ids[m * blk_stride + 0 .. n_blk[m]) -- the blocks that
  // still hold an active event -- packed 4 * EPL to a tile.  Null = every column, in order.
  const int32_t* blk_ids;
  int64_t blk_stride;
  int32_t n_blk[kMaxModels];
  // Gathered sub-fit (brie_fit_buffers.event_ids): per-model column -> global event map and per-model
  // count / length tiles.  Null / 0 = columns are events event_offset + column, tiles shared by all models.
  const int32_t* ev_ids;   // (M, ld)
  int64_t c_mstride;       // floats between the count tiles of consecutive models
  int64_t eff_mstride;     // floats between the (3, ld) length tables of consecutive models
  // Wide designs (EXT instantiations): the covariate part of the prior mean, Xc Wc + Wg Xg^T, arrives as a dense
  // (M, Nc, ld) array computed by a GEMM before the launch, and r = (mu - m) / sigma^2 leaves as one, for the
  // GEMMs that turn it into d loss / d Wc = -Xc^T r and d loss / d Wg = -r Xg (brie_abi.cu).
  const float* PM;
  float* R;
  // Packed-code counts (CODE8 instantiations, brie_encode_counts): one word per element, byte l = index of layer l's
  // value in dict[l * 256 + .] (entry 0 is 0.0f, so word != 0 iff the element has reads).
  const uint32_t* codes;
  int64_t code_mstride;    // words between the code tiles of consecutive models (gathered sub-fits), 0 = shared
  const float* dict;       // (3, 256)
};

constexpr int kBlkCols = 8;   // events per compaction block = one 32-byte sector of every f32 array

__device__ __forceinline__ float sqrt_approx(float x) {
  float y;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ float lg2_approx(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;

// exp / log on the SFU (ex2/lg2.approx.ftz): 2 ulp-class, no denormal fix-up code
__device__ __forceinline__ float fast_exp(float x) { return ex2_approx(x * kLog2e); }
__device__ __forceinline__ float fast_log(float x) { return lg2_approx(x) * kLn2; }

__device__ __forceinline__ void cp_async16(uint32_t dst_smem, const void* src, bool valid) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst_smem), "l"(src), "r"(valid ? 16 : 0)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// keras Adam update_step (TF 2.15): m += (g-m)(1-b1); v += (g^2-v)(1-b2);
// x -= alpha_t * m / (sqrt(v) + eps)
__device__ __forceinline__ void adam_update(float& x, float& m, float& v, float g, float alpha) {
  m = fmaf(g - m, kB1c, m);
  v = fmaf(fmaf(g, g, -v), kB2c, v);
  x -= (m * alpha) * rcp_approx(sqrt_approx(v) + kAdamEps);
}

// Packed FP32 pairs (sm_100a FFMA2 / FADD2 / FMUL2: one issue slot, two IEEE-rounded results) in the dense phases
// and the Monte-Carlo samples of the step kernel.  A/B on one B200 against the scalar form, profiles/r2_ab_f32x2.md:
// C2 unchanged (0.936), C3 with loss trace 0.930 -> 0.949, C4 0.947 -> 0.958 / with loss trace 0.900 -> 0.923,
// Kc 16 0.730 -> 0.761 / 0.700 -> 0.742; the whole parity suite passed on either form.
#define BRIE_F2_BINARY(name, ptx)                                                                          \
  __device__ __forceinline__ float2 name(float2 a, float2 b) {                                             \
    float2 d;                                                                                              \
    asm("{.reg .b64 ra, rb, rd;\n\t mov.b64 ra, {%2, %3};\n\t mov.b64 rb, {%4, %5};\n\t" ptx               \
        " rd, ra, rb;\n\t mov.b64 {%0, %1}, rd;}"                                                          \
        : "=f"(d.x), "=f"(d.y)                                                                             \
        : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));                                                         \
    return d;                                                                                              \
  }
BRIE_F2_BINARY(f2_add, "add.rn.f32x2")
BRIE_F2_BINARY(f2_sub, "sub.rn.f32x2")
BRIE_F2_BINARY(f2_mul, "mul.rn.f32x2")
#undef BRIE_F2_BINARY
__device__ __forceinline__ float2 f2_fma(float2 a, float2 b, float2 c) {
  float2 d;
  asm("{.reg .b64 ra, rb, rc, rd;\n\t mov.b64 ra, {%2, %3};\n\t mov.b64 rb, {%4, %5};\n\t mov.b64 rc, {%6, %7};\n\t"
      "fma.rn.f32x2 rd, ra, rb, rc;\n\t mov.b64 {%0, %1}, rd;}"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
  return d;
}
__device__ __forceinline__ float2 f2_splat(float x) { return make_float2(x, x); }

// adam_update on a pair.  (g^2 - v is a multiply and a subtract here, not one fused multiply-add: there is no
// packed form with a negated addend; the difference is one rounding of g^2.)
__device__ __forceinline__ void adam_update2(float& x0, float& x1, float& m0, float& m1, float& v0, float& v1,
                                             float g0, float g1, float alpha) {
  const float2 g = make_float2(g0, g1);
  float2 m = make_float2(m0, m1), v = make_float2(v0, v1);
  m = f2_fma(f2_sub(g, m), f2_splat(kB1c), m);
  v = f2_fma(f2_sub(f2_mul(g, g), v), f2_splat(kB2c), v);
  const float2 den = f2_add(make_float2(sqrt_approx(v.x), sqrt_approx(v.y)), f2_splat(kAdamEps));
  const float2 step = f2_mul(f2_mul(m, f2_splat(alpha)), make_float2(rcp_approx(den.x), rcp_approx(den.y)));
  const float2 x = f2_sub(make_float2(x0, x1), step);
  x0 = x.x; x1 = x.y; m0 = m.x; m1 = m.y; v0 = v.x; v1 = v.y;
}

__device__ __forceinline__ float clip9(float x) { return fminf(fmaxf(x, -9.0f), 9.0f); }

// adam_update of one stored parameter *x with its moments *m, *v; `clip` applies the +-9 constraint to the result.
__device__ __forceinline__ void adam_at(float* x, float* m, float* v, float g, float alpha, bool clip = false) {
  float xx = *x, mm = *m, vv = *v;
  adam_update(xx, mm, vv, g, alpha);
  *x = clip ? clip9(xx) : xx; *m = mm; *v = vv;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// MC part of one element: S reparameterised samples z = mu + s*eps, the isoform
// likelihood of logLik_MC (model_TFProb.py:159-185) in the form
//   l = c1 log psi + c2 log(1-psi) + [c1 log L1 + c2 log L2 + c3 log L3] - n log D,
//   D = psi L1 + (1-psi) L2 + L3   (the binomial branch :162-167 is L = (1,1,0))
// and dl/dz = c1(1-psi) - c2 psi - n psi(1-psi)(L1-L2)/D.
// Returns sum_s g, sum_s g*eps and (LOSS) sum_s l without the bracket.
template <bool LOSS>
__device__ __forceinline__ void mc_samples(float mu, float s, float c1, float c2, float n,
                                           float L1, float L2, float L3, float dL, int S,
                                           uint32_t event, uint32_t cell, uint32_t step,
                                           uint32_t stream0, uint64_t seed, float& gsum,
                                           float& gesum, float& llsum) {
  gsum = 0.f; gesum = 0.f; llsum = 0.f;
  const float ndL = n * dL;
  for (int s0 = 0; s0 < S; s0 += 4) {
    float eps[4];
    brie_normals4(event, cell, step, stream0 + (uint32_t)(s0 >> 2), seed, eps);
    // two samples per instruction where both exist (S = 3: samples 0 and 1 as a pair, sample 2 alone)
#pragma unroll
    for (int j = 0; j < 4; j += 2) {
      if (s0 + j + 1 < S) {
        const float2 ep = make_float2(eps[j], eps[j + 1]);
        const float2 z = f2_fma(f2_splat(s), ep, f2_splat(mu));
        const float2 az = make_float2(fabsf(z.x), fabsf(z.y));
        const float2 ea = f2_mul(az, f2_splat(-kLog2e));
        const float2 e = make_float2(ex2_approx(ea.x), ex2_approx(ea.y));          // exp(-|z|)
        const float2 ope = f2_add(e, f2_splat(1.0f));
        const float2 inv = make_float2(rcp_approx(ope.x), rcp_approx(ope.y));
        const float2 lo = f2_mul(e, inv);
        const float2 psi = make_float2(z.x >= 0.f ? inv.x : lo.x, z.y >= 0.f ? inv.y : lo.y);
        const float2 q = make_float2(z.x >= 0.f ? lo.x : inv.x, z.y >= 0.f ? lo.y : inv.y);
        const float2 D = f2_fma(psi, f2_splat(L1), f2_fma(q, f2_splat(L2), f2_splat(L3)));
        const float2 rD = make_float2(rcp_approx(D.x), rcp_approx(D.y));
        const float2 t1 = f2_fma(f2_splat(c1), q, f2_mul(f2_splat(-c2), psi));
        const float2 t2 = f2_mul(f2_mul(f2_splat(ndL), f2_mul(psi, q)), rD);
        const float2 g = f2_sub(t1, t2);
        gsum += g.x;
        gsum += g.y;
        gesum = fmaf(g.x, ep.x, gesum);
        gesum = fmaf(g.y, ep.y, gesum);
        if (LOSS) {
          const float2 lsp = make_float2(fminf(z.x, 0.f) - fast_log(ope.x), fminf(z.y, 0.f) - fast_log(ope.y));
          const float2 u = f2_fma(f2_splat(c1), lsp, f2_mul(f2_splat(c2), f2_sub(lsp, z)));
          llsum += u.x - n * fast_log(D.x);
          llsum += u.y - n * fast_log(D.y);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if (s0 + j < S && !(s0 + (j | 1) < S)) {   // the unpaired last sample
        const float z = fmaf(s, eps[j], mu);
        const float e = ex2_approx(-kLog2e * fabsf(z));      // exp(-|z|)
        const float inv = rcp_approx(1.0f + e);
        const float lo = e * inv;
        const float psi = z >= 0.f ? inv : lo;
        const float q = z >= 0.f ? lo : inv;
        const float D = fmaf(psi, L1, fmaf(q, L2, L3));
        const float g = fmaf(c1, q, -c2 * psi) - ndL * (psi * q) * rcp_approx(D);
        gsum += g;
        gesum = fmaf(g, eps[j], gesum);
        if (LOSS) {
          const float lsp = fminf(z, 0.f) - fast_log(1.0f + e);  // log sigmoid(z)
          llsum += fmaf(c1, lsp, c2 * (lsp - z)) - n * fast_log(D);
        }
      }
    }
  }
}

template <int KC, int KG, bool CELL, bool LOSS, bool PAIR = false>
struct StepTraits {
  static constexpr int kGB = KC;                       // index of d/d intercept (gene mode)
  static constexpr int kGT = KC + 1;                   // index of d/d sigma_log (gene mode)
  static constexpr int kLoss = KC + (CELL ? 0 : 2);    // sum over cells of KL - loglik (PAIR: of each step in turn)
  static constexpr int NEV = KC + (CELL ? 0 : 2) + (LOSS ? (PAIR ? 2 : 1) : 0);
  static constexpr int NCELL = KG + (CELL ? 2 : 0);
};

// Events per lane of the step kernel: 4 (one 16-byte access per array) while the per-event
// accumulators and weights of a lane, 2 x KC x EPL registers, fit next to the rest; the wide
// covariate cases (KC = 16, and KC = 8 together with gene features, whose per-cell accumulators come on top)
// run with 2 events per lane (8-byte accesses, 64-event tiles) -- no instantiation spills to local memory.
__host__ __device__ constexpr int step_epl(int KC, int KG = 0) { return (KC > 8 || (KC == 8 && KG > 0)) ? 2 : 4; }

template <int EPL> struct LaneVec;
template <> struct LaneVec<4> { using type = float4; };
template <> struct LaneVec<2> { using type = float2; };
template <> struct LaneVec<1> { using type = float; };

template <int EPL>
__device__ __forceinline__ void vec_get(const typename LaneVec<EPL>::type& v, float (&x)[EPL]);
template <> __device__ __forceinline__ void vec_get<4>(const float4& v, float (&x)[4]) { x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w; }
template <> __device__ __forceinline__ void vec_get<2>(const float2& v, float (&x)[2]) { x[0] = v.x; x[1] = v.y; }
template <> __device__ __forceinline__ void vec_get<1>(const float& v, float (&x)[1]) { x[0] = v; }

template <int EPL>
__device__ __forceinline__ typename LaneVec<EPL>::type vec_make(const float (&x)[EPL]);
template <> __device__ __forceinline__ float4 vec_make<4>(const float (&x)[4]) { return make_float4(x[0], x[1], x[2], x[3]); }
template <> __device__ __forceinline__ float2 vec_make<2>(const float (&x)[2]) { return make_float2(x[0], x[1]); }
template <> __device__ __forceinline__ float vec_make<1>(const float (&x)[1]) { return x[0]; }

// cp.async of one lane's EPL floats; .cg (L2 only) needs 16 bytes, narrower copies use .ca
template <int BYTES>
__device__ __forceinline__ void cp_async_lane(uint32_t dst_smem, const void* src, bool valid) {
  if (BYTES == 16)
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst_smem), "l"(src), "r"(valid ? 16 : 0) : "memory");
  else if (BYTES == 8)
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(dst_smem), "l"(src), "r"(valid ? 8 : 0) : "memory");
  else
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst_smem), "l"(src), "r"(valid ? 4 : 0) : "memory");
}

// Fused ELBO forward + backward + Adam for the per-element variables.
// grid = (M, n_col_tiles, n_row_chunks): models fastest so the CTAs sharing a
// count tile are co-resident and the counts are fetched from HBM once.
//
// Each warp walks its rows of one (32 x EPL)-event segment through a private two-stage
// shared-memory ring filled with cp.async (EPL floats per lane per array, 9 arrays =
// 4.6 KB per row at EPL = 4): the next row streams in from HBM while the current one is
// processed, so loads in flight do not depend on register-resident state.  The row's
// warp-uniform constants (Xc[c, :], Wg[c, :], per-cell intercept / sigma_log) ride in the
// same commit group, one float per lane; one __syncwarp after the wait makes the stage
// readable by every lane of the warp (no CTA barrier in the row loop).
// One row is processed in three phases:
//   A (dense, lane = EPL events): KL terms and gradients, shared-parameter
//     accumulators; elements with reads (n > 0) push their tile column, compacted by
//     ballot/popc prefix, into the warp's shared-memory work queue;
//   B (compacted): lanes take queue items round-robin, read the element from the ring
//     stage, run the S Monte-Carlo samples (Philox + Box-Muller + likelihood gradient)
//     and leave the sums in the element's count slots -- zero-count elements, 80-87 % of
//     real data, cost nothing here and the lanes stay converged;
//   C (dense): owners subtract their slots (zeros where there were no reads),
//     Adam-update and store (16 B stores at EPL = 4).
// CODE8 (counts as packed dictionary codes, StepArgs.codes): the ring carries one code word per element in place of
// the three count arrays (7 arrays, 4 B of counts per element instead of 12), phase A's read test is word != 0,
// phase B decodes its items' counts from the (3, 256) dictionary in shared memory and leaves its sums in a per-warp
// scratch area, which the owners read only for their elements with reads.  The decoded values are the f32 tiles'
// bit patterns, so both forms compute the same bits.
constexpr int kQueueFields = 1;   // tile column of the element; its data is read from, and its results written to, the row's ring slots
constexpr int kRingArrays = 9;    // Z_loc, Z_std_log, c1, c2, c3, m_loc, v_loc, m_std, v_std
constexpr int kRingArraysCode8 = 7;   // Z_loc, Z_std_log, code, m_loc, v_loc, m_std, v_std
constexpr int kRingStages = 2;
constexpr int kDictSize = 256;    // values per layer of the count dictionary (code 0 = 0.0f)
__host__ __device__ constexpr int step_tile_cols(int KC, int KG = 0) { return 32 * step_epl(KC, KG); }
// Rows a warp processes per loop iteration.  The 2-events-per-lane instantiations take two adjacent rows at a time:
// their 64-event row holds ~10 elements with reads, a third of a warp, so the Monte-Carlo phase (Philox, Box-Muller,
// S likelihood samples: ~200 instructions whatever the number of items) ran mostly idle; the items of two rows
// share one pass.  Ring stages, queue and per-lane state then match the 4-events-per-lane kernels byte for byte.
// (16 covariates together with gene features keep one row per iteration: two rows' state next to 32 per-event and
// up to 10 per-cell accumulators would spill.)  A/B against one row per iteration: profiles/r2_ab_rpi_tma.md.
__host__ __device__ constexpr int step_rpi(int KC, int KG = 0) {
  return (step_epl(KC, KG) == 2 && !(KC > 8 && KG > 0)) ? 2 : 1;
}
// Per-event constants of a column tile (Wc rows, Xg columns, intercept, sigma_log, 1/sigma^2) stay in
// registers for narrow designs; wider ones (Kc + Kg >= 3) keep them in shared memory and re-read them
// every row, so they are not live across the Monte-Carlo phase (no spills).  A/B on one box
// (profiles/r1_ab_smem_consts.md, r1_ab_row_consts.md): C3 with loss trace +11 %, C4 +10 % / +23 %,
// Kc 15 +9 %; C3 without the loss trace runs 1 % slower from shared memory but spills from registers.
__host__ __device__ constexpr bool step_consts_in_smem(int KC, int KG) { return KC + KG >= 3; }
// Two-step passes keep both steps' constants in shared memory, whatever the width.
__host__ __device__ constexpr int step_n_consts(int KC, int KG, bool CELL, bool PAIR = false) {
  return PAIR ? 2 * (KC + 3) : (step_consts_in_smem(KC, KG) ? KC + KG + (CELL ? 0 : 3) : 0);
}
// Widest design stepped in two-step passes: above it the two steps' per-event sums and statistics no longer fit the
// register budget of two CTAs per SM (the Kc = 8 and 16 forms spill hundreds of bytes to local memory).
constexpr int kMaxPairKc = 4;
// Per-event statistics a two-step pass leaves per row chunk: R_k = sum_c x_ck d_c, R_0 = sum_c d_c, Q = sum_c d_c^2 and
// E = sum_c exp(2 (lam_c - tau)), d_c = mu_c - prior mean, of the state it writes, around the second step's parameters.
__host__ __device__ constexpr int pair_stat_rows(int KC) { return KC + 3; }
constexpr int kRowConstSlots = 32;   // per warp and ring stage: Xc[c, :], Wg[c, :], per-cell intercept / sigma_log of the row
// CODE8 or PAIR: per warp and row of an iteration, the Monte-Carlo sums d/dZ_loc, d/dZ_std_log and (LOSS) the
// log-likelihood (a two-step pass keeps the counts in the ring for its second step)
__host__ __device__ constexpr int step_n_scratch(bool LOSS) { return LOSS ? 3 : 2; }
__host__ __device__ constexpr int step_smem_bytes(int KC, int KG, bool CELL, bool LOSS, bool EXT = false,
                                                  bool CODE8 = false, bool PAIR = false) {
  return ((kWarps * kRingStages * ((CODE8 ? kRingArraysCode8 : kRingArrays) + (EXT ? 1 : 0)) +
           kWarps * kQueueFields + (CODE8 || PAIR ? kWarps * step_n_scratch(LOSS) : 0)) *
              step_rpi(KC, KG) +
          7 + step_n_consts(KC, KG, CELL, PAIR)) *
             step_tile_cols(KC, KG) * 4 +
         kWarps * kRingStages * step_rpi(KC, KG) * kRowConstSlots * 4 + (CODE8 ? 3 * kDictSize * 4 : 0);
}

// PAIR (two steps per pass, gene mode with per-event parameters only): after phase C of the first step the updated
// Z_loc, Z_std_log and moments go back into the row's ring slot instead of HBM, and phases A-C run again with the
// second step's constants, RNG step word and alpha; the Monte-Carlo queue is built once (it depends on the counts
// only).  The per-event gradient sums are those of the second step (the first step's came from the previous pass'
// statistics, or the sums-only pre-pass, kl_sums_kernel), and the state written is also summed into the statistics
// of pair_stat_rows around the second step's parameters, from which event_update_kernel forms the next step's sums.
template <int KC, int KG, bool CELL, bool LOSS, bool EXT = false, bool CODE8 = false, bool PAIR = false>
__global__ void __launch_bounds__(kThreads, kMinCtas) elbo_step_kernel(const StepArgs a) {
  static_assert(!EXT || (KC == 0 && KG == 0), "the wide-design form takes all covariates through PM / R");
  static_assert(!PAIR || (!CELL && KG == 0 && !EXT), "two-step passes need per-event parameters only");
  constexpr int NSTEP = PAIR ? 2 : 1;
  constexpr bool SCR = CODE8 || PAIR;                // Monte-Carlo sums go to the per-warp scratch, not the count slots
  constexpr int NK = KC + KG + (CELL ? 0 : 3);       // per-event constant rows of one step (kSm)
  constexpr int NST = PAIR ? pair_stat_rows(KC) : 0;
  // ring arrays per row slot (EXT: + the prior-mean tile) and the slots of the Adam moments / prior-mean tile in it
  constexpr int NRA = (CODE8 ? kRingArraysCode8 : kRingArrays) + (EXT ? 1 : 0);
  constexpr int IA = CODE8 ? 3 : 5;                  // m_loc, v_loc, m_std, v_std at IA .. IA + 3
  constexpr int IPM = IA + 4;
  constexpr int NSCR = step_n_scratch(LOSS);
  constexpr int RPI = step_rpi(KC, KG);              // rows per loop iteration = row slots per ring stage
  using T = StepTraits<KC, KG, CELL, LOSS, PAIR>;
  constexpr int NEV = T::NEV;
  constexpr int NCELL = T::NCELL;
  constexpr int EPL = step_epl(KC, KG);
  constexpr int TC = 32 * EPL;              // events per warp row segment (column tile)
  constexpr bool kSm = step_consts_in_smem(KC, KG) || PAIR;
  using Vec = typename LaneVec<EPL>::type;
  const int m = blockIdx.x;
  if (!((a.model_mask >> m) & 1u)) return;
  const int tile = blockIdx.y;
  const int chunk = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // column of this lane's first event, and of tile column threadIdx.x (per-event constants, partial sums)
  constexpr int LPB = kBlkCols / EPL;       // lanes per compaction block
  constexpr int BPT = TC / kBlkCols;        // blocks per tile
  int64_t g0 = (int64_t)tile * TC + lane * EPL;
  if (a.blk_ids != nullptr) {
    const int nblk = a.n_blk[m];
    if (tile * BPT >= nblk) return;
    const int bl = tile * BPT + lane / LPB;
    g0 = bl < nblk ? (int64_t)a.blk_ids[(int64_t)m * a.blk_stride + bl] * kBlkCols + (lane % LPB) * EPL : a.ld;
  }
  // recomputed where needed (constants load, final partial sums) rather than kept live across the row loop
  auto thread_col = [&]() -> int64_t {
    if (a.blk_ids == nullptr) return (int64_t)tile * TC + threadIdx.x;
    const int bt = tile * BPT + (int)(threadIdx.x / kBlkCols);
    return (threadIdx.x < TC && bt < a.n_blk[m])
               ? (int64_t)a.blk_ids[(int64_t)m * a.blk_stride + bt] * kBlkCols + (threadIdx.x % kBlkCols)
               : a.ld;
  };
  const bool in_ld = g0 < a.ld;             // ld % 4 == 0 and EPL divides 4: a lane is all in or all out

  uint32_t act = 0;                         // bit j: this lane's event j is still being optimised
  if (in_ld) {
#pragma unroll
    for (int j = 0; j < EPL; ++j) act |= (a.active[(int64_t)m * a.ld + g0 + j] != 0 ? 1u : 0u) << j;
  }
  extern __shared__ __align__(128) float smem[];
  constexpr int SLOT = NRA * TC;                     // floats of one row slot
  float* s_ring = smem + warp * (kRingStages * RPI * SLOT);
  uint32_t* q = reinterpret_cast<uint32_t*>(smem + kWarps * kRingStages * RPI * SLOT +
                                            warp * kQueueFields * RPI * TC);
  float(*s_L)[TC] = reinterpret_cast<float(*)[TC]>(smem + kWarps * kRingStages * RPI * SLOT +
                                                   kWarps * kQueueFields * RPI * TC);
  uint32_t* s_ev = reinterpret_cast<uint32_t*>(s_L + 6);   // global event id of each tile column (RNG counter word)
  float(*s_k)[TC] = s_L + 7;                // kSm: rows Wc[0..KC), Xg[0..KG), then (gene mode) b, tau, 1/sigma^2 (PAIR: per step)
  // Gene-feature slots are stored XOR-permuted per lane (slot i of lane L holds feature i ^ pk(L), pk = the top
  // log2(KG) lane bits reversed into a feature index) so that the per-cell reduction over the 32 lanes of
  // d loss / d Wg[c, :] is a halving butterfly without selects (see the end of the row loop).
  constexpr int KGB = KG == 8 ? 3 : (KG == 4 ? 2 : 0);
  static_assert(KG == 0 || (1 << KGB) == KG, "KG must be a power of two");
  int pk = 0;
#pragma unroll
  for (int t = 0; t < KGB; ++t) pk |= ((lane >> (4 - t)) & 1) << (KGB - 1 - t);
  constexpr int NRC = KC + KG + (CELL ? 2 : 0);   // per-row (cell) constants: Xc[c, :], Wg[c, :], b[c], tau[c]
  static_assert(NRC <= kRowConstSlots, "row constants must fit one slot per lane");
  constexpr int kRcBase = ((kWarps * kRingStages * NRA + kWarps * kQueueFields) * RPI + 7 +
                           step_n_consts(KC, KG, CELL, PAIR)) * TC;
  float* s_rc = smem + kRcBase + warp * (kRingStages * RPI * kRowConstSlots);
  // CODE8 or PAIR: this warp's Monte-Carlo sums (row r, sum k at (r * NSCR + k) * TC); CODE8: the count dictionary
  constexpr int kScrBase = kRcBase + kWarps * kRingStages * RPI * kRowConstSlots;
  float* const s_scr = smem + kScrBase + warp * (NSCR * RPI * TC);
  float* const s_dict = smem + kScrBase + kWarps * NSCR * RPI * TC;
  if (CODE8) {   // published by the barrier below
    for (int i = threadIdx.x; i < 3 * kDictSize; i += kThreads) s_dict[i] = a.dict[i];
  }

  // Per-event constants of the tile go to shared memory before the barrier that decides whether the tile has
  // any active event: their loads overlap the `active` loads and that barrier also publishes them.
  if (threadIdx.x < TC) {
    const int64_t g = thread_col();
    s_ev[threadIdx.x] = (a.ev_ids != nullptr && g < a.ld) ? (uint32_t)a.ev_ids[(int64_t)m * a.ld + g]
                                                          : (uint32_t)(a.event_offset + g);
    float l1 = 1.f, l2 = 1.f, l3 = 0.f;
    if (a.eff && g < a.ld) {
      const float* ef = a.eff + (int64_t)m * a.eff_mstride;
      l1 = ef[g]; l2 = ef[a.ld + g]; l3 = ef[2 * a.ld + g];
    }
    s_L[0][threadIdx.x] = l1; s_L[1][threadIdx.x] = l2; s_L[2][threadIdx.x] = l3;
    if (LOSS) {  // log lengths for the constant part of the log-likelihood (0 * log 0 never occurs: eff > 0)
      s_L[3][threadIdx.x] = logf(l1); s_L[4][threadIdx.x] = logf(l2);
      s_L[5][threadIdx.x] = a.eff ? logf(l3) : 0.f;
    }
    if (kSm) {
#pragma unroll
      for (int h = 0; h < NSTEP; ++h) {
        // PAIR: the first step's parameters of the real events come from `prev`
        const bool okc = g < a.ld, from_prev = PAIR && h == 0 && g < a.Ng;
        const float* wsrc = from_prev ? a.prev + (int64_t)m * (KC + 2) * a.ld : a.Wc + (int64_t)m * KC * a.ld;
        const float* bsrc = from_prev ? a.prev + ((int64_t)m * (KC + 2) + KC) * a.ld : a.b + (int64_t)m * a.ld;
        const float* tsrc = from_prev ? a.prev + ((int64_t)m * (KC + 2) + KC + 1) * a.ld : a.tau + (int64_t)m * a.ld;
        float(*sk)[TC] = s_k + h * NK;
#pragma unroll
        for (int k = 0; k < KC; ++k) sk[k][threadIdx.x] = okc ? wsrc[k * a.ld + g] : 0.f;
#pragma unroll
        for (int k = 0; k < KG; ++k) sk[KC + k][threadIdx.x] = g < a.Ng ? a.Xg[g * KG + k] : 0.f;
        if (!CELL) {
          const float t = okc ? tsrc[g] : 0.f;
          sk[KC + KG][threadIdx.x] = okc ? bsrc[g] : 0.f;
          sk[KC + KG + 1][threadIdx.x] = t;
          sk[KC + KG + 2][threadIdx.x] = fast_exp(-2.0f * t);
        }
      }
    }
  }
  if (!__syncthreads_or(act != 0)) return;
  const bool all_act = act == (1u << EPL) - 1u;

  const int64_t row_begin = (int64_t)chunk * a.rows_per_cta;
  const int n_rows = (int)(min(row_begin + (int64_t)a.rows_per_cta, a.Nc) - row_begin);
  const bool has_c3 = a.c[2] != nullptr;
  // Addresses = one warp-uniform 64-bit base per array (this model's plane at the CTA's first row: blockIdx and
  // kernel parameters only, so it lives in uniform registers) + a per-lane 32-bit element offset
  // (local row) * ld + column, which brie_fit_create keeps below 2^31 -- one wide multiply-add per access
  // instead of a 64-bit multiply-add chain per array and row.
  const int64_t plane = a.Nc * a.ld;
  const int64_t mplane = (int64_t)a.M * plane;
  const int64_t cta_off = (int64_t)m * plane + row_begin * a.ld;
  float* const bZl = a.Zl + cta_off;
  float* const bZs = a.Zs + cta_off;
  float* const bA0 = a.aZ + cta_off;
  float* const bA1 = a.aZ + mplane + cta_off;
  float* const bA2 = a.aZ + 2 * mplane + cta_off;
  float* const bA3 = a.aZ + 3 * mplane + cta_off;
  const float* const bPM = EXT ? a.PM + cta_off : nullptr;
  float* const bR = EXT ? a.R + cta_off : nullptr;
  const int64_t cnt_off = (int64_t)m * a.c_mstride + row_begin * a.ld;
  const float* const bC0 = a.c[0] + cnt_off;
  const float* const bC1 = a.c[1] + cnt_off;
  const float* const bC2 = has_c3 ? a.c[2] + cnt_off : a.c[0];
  const uint32_t* const bW = CODE8 ? a.codes + ((int64_t)m * a.code_mstride + row_begin * a.ld) : nullptr;
  const int64_t cell0 = (int64_t)m * a.Nc + row_begin;            // first cell of the CTA in the (M, Nc, .) row constants
  const uint32_t ld32 = (uint32_t)a.ld;
  const uint32_t col32 = in_ld ? (uint32_t)g0 : 0u;

  // ring producer: this lane's EPL-float column of each array, one commit group per row
  const uint32_t ring_lane = (uint32_t)__cvta_generic_to_shared(s_ring) + lane * (EPL * 4);
  // Lanes whose events are all frozen (converged reference batches) copy nothing: their ring slots are
  // zero-filled, they compute on zeros and store nothing, so a partly active tile only pays for the
  // 32-byte sectors that hold active events.
  const uint32_t rc_lane = (uint32_t)__cvta_generic_to_shared(s_rc) + lane * 4;
  auto issue_rows = [&](int lrb, int stage) {     // lrb: first of the RPI adjacent rows (index within the CTA)
#pragma unroll
    for (int r = 0; r < RPI; ++r) {
      const int lr = lrb + r;
      const bool ok = act != 0 && lr < n_rows;
      const uint32_t rel = ok ? (uint32_t)lr * ld32 + col32 : 0u;
      const uint32_t dst = ring_lane + (stage * RPI + r) * (SLOT * 4);
      cp_async_lane<EPL * 4>(dst + 0 * TC * 4, bZl + rel, ok);
      cp_async_lane<EPL * 4>(dst + 1 * TC * 4, bZs + rel, ok);
      if (CODE8) {
        cp_async_lane<EPL * 4>(dst + 2 * TC * 4, bW + rel, ok);
      } else {
        cp_async_lane<EPL * 4>(dst + 2 * TC * 4, bC0 + rel, ok);
        cp_async_lane<EPL * 4>(dst + 3 * TC * 4, bC1 + rel, ok);
        cp_async_lane<EPL * 4>(dst + 4 * TC * 4, bC2 + (has_c3 ? rel : 0u), ok && has_c3);
      }
      cp_async_lane<EPL * 4>(dst + (IA + 0) * TC * 4, bA0 + rel, ok);
      cp_async_lane<EPL * 4>(dst + (IA + 1) * TC * 4, bA1 + rel, ok);
      cp_async_lane<EPL * 4>(dst + (IA + 2) * TC * 4, bA2 + rel, ok);
      cp_async_lane<EPL * 4>(dst + (IA + 3) * TC * 4, bA3 + rel, ok);
      if (EXT) cp_async_lane<EPL * 4>(dst + IPM * TC * 4, bPM + rel, ok);
      if (NRC > 0) {
        // The row's warp-uniform constants ride in the same commit group, one float per lane.  (As plain
        // loads issued a row ahead they shared a scoreboard with the tile constants loaded before the loop,
        // and the first use of those waited for the prefetch every row: 23 % of the stall samples.)
        const bool okc = lane < NRC && lr < n_rows;
        const uint32_t rr = okc ? (uint32_t)lr : 0u;
        const float* src = a.Xc;
        if (lane < KC) src = a.Xc + cell0 * KC + (rr * KC + lane);
        else if (lane < KC + KG) src = a.Wg + cell0 * KG + (rr * KG + (lane - KC));
        else if (CELL && lane == KC + KG) src = a.b + cell0 + rr;
        else if (CELL) src = a.tau + cell0 + rr;
        cp_async_lane<4>(rc_lane + (stage * RPI + r) * (kRowConstSlots * 4), src, okc);
      }
    }
    cp_async_commit();                            // one group per iteration
  };
  issue_rows(warp * RPI, 0);

  float wc[KC > 0 ? KC : 1][EPL];
  float xg[KG > 0 ? KG : 1][EPL];
  float bb[EPL], tau[EPL], is2[EPL];
#pragma unroll
  for (int j = 0; j < EPL; ++j) {
    bb[j] = 0.f; tau[j] = 0.f; is2[j] = 1.f;
  }
#pragma unroll
  for (int k = 0; k < (KC > 0 ? KC : 1); ++k)
#pragma unroll
    for (int j = 0; j < EPL; ++j) wc[k][j] = 0.f;
#pragma unroll
  for (int k = 0; k < (KG > 0 ? KG : 1); ++k)
#pragma unroll
    for (int j = 0; j < EPL; ++j) xg[k][j] = 0.f;
  if (in_ld && !kSm) {
#pragma unroll
    for (int k = 0; k < KC; ++k)
      vec_get<EPL>(*reinterpret_cast<const Vec*>(a.Wc + ((int64_t)m * KC + k) * a.ld + g0), wc[k]);
#pragma unroll
    for (int j = 0; j < EPL; ++j) {
#pragma unroll
      for (int k = 0; k < KG; ++k) xg[k][j] = (g0 + j) < a.Ng ? a.Xg[(g0 + j) * KG + (k ^ pk)] : 0.f;
    }
    if (!CELL) {
      vec_get<EPL>(*reinterpret_cast<const Vec*>(a.b + (int64_t)m * a.ld + g0), bb);
      vec_get<EPL>(*reinterpret_cast<const Vec*>(a.tau + (int64_t)m * a.ld + g0), tau);
#pragma unroll
      for (int j = 0; j < EPL; ++j) is2[j] = fast_exp(-2.0f * tau[j]);
    }
  }

  float acc[NEV > 0 ? NEV : 1][EPL];
#pragma unroll
  for (int i = 0; i < (NEV > 0 ? NEV : 1); ++i)
#pragma unroll
    for (int j = 0; j < EPL; ++j) acc[i][j] = 0.f;
  float stat[NST > 0 ? NST : 1][EPL];       // PAIR: R_k (k < KC), R_0, Q, E of the lane's events
#pragma unroll
  for (int i = 0; i < (NST > 0 ? NST : 1); ++i)
#pragma unroll
    for (int j = 0; j < EPL; ++j) stat[i][j] = 0.f;

  const uint32_t stream0 = brie_stream_word(BRIE_PHASE_TRAIN, (uint32_t)a.model_id[m], 0u);
  const uint32_t lt_mask = (1u << lane) - 1u;

  // per-cell sums of one row over the 32 lanes -> one partial per column tile
  auto cell_reduce_store = [&](float (&cacc)[NCELL > 0 ? NCELL : 1], int64_t row) {
    float* pc = a.part_cell + (((int64_t)tile * a.M + m) * a.Nc + row) * NCELL;
    if (KG > 0) {
      // Halving butterfly: slot i of this lane holds feature i ^ pk, so at every step all lanes keep
      // the lower half of their slots and hand the upper half to the partner that keeps those features
      // (no selects); KG - 1 + log2(32 / KG) shuffles instead of 5 KG.
#pragma unroll
      for (int t = 0; t < KGB; ++t) {
        const int H = KG >> (t + 1);
#pragma unroll
        for (int i = 0; i < H; ++i) cacc[i] += __shfl_xor_sync(0xffffffffu, cacc[H + i], 16 >> t);
      }
      float sum = cacc[0];
#pragma unroll
      for (int o = 16 >> KGB; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      if ((lane & ((32 >> KGB) - 1)) == 0) pc[pk] = sum;
    }
    if (CELL) {  // d/d intercept and d/d sigma_log of the cell: two values, one per half-warp after the first step
      const bool hi = (lane & 16) != 0;
      const float keep = hi ? cacc[KG + 1] : cacc[KG], send = hi ? cacc[KG] : cacc[KG + 1];
      float sum = keep + __shfl_xor_sync(0xffffffffu, send, 16);
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      if ((lane & 15) == 0) pc[KG + (hi ? 1 : 0)] = sum;
    }
  };

  int stage = 0;
  for (int lrb = warp * RPI; lrb < n_rows; lrb += kWarps * RPI, stage ^= 1) {
    issue_rows(lrb + kWarps * RPI, stage ^ 1);   // prefetch the next rows (zero-size copies past the end)
    cp_async_wait<1>();                   // this iteration's group has landed
    __syncwarp();                         // other lanes read this lane's copies (row constants, Monte-Carlo items)
    float* const rs0 = s_ring + stage * (RPI * SLOT);                 // row slot r of this stage: rs0 + r * SLOT
    uint32_t nz = 0;                      // bit r * EPL + j: element j of row r has reads
    uint32_t bal[RPI * EPL];
    int n_items = 0;
#pragma unroll
    for (int h = 0; h < NSTEP; ++h) {     // PAIR: step `step` + h of the pass
    const float(*sk)[TC] = s_k + h * NK;
    const float alpha = h == 0 ? a.alpha : a.alpha2;
    // PAIR: the first step leaves nothing in the per-event gradient sums (only its loss)
    const bool grad_sums = !PAIR || h == NSTEP - 1;
    float mu[RPI][EPL], lam[RPI][EPL], gmu[RPI][EPL], glam[RPI][EPL];
    float cacc1[NCELL > 0 ? NCELL : 1];   // RPI == 1: kept until after phase C (as tuned for the gene-feature kernels)

    // ---- phase A: KL terms, shared-parameter accumulators, non-zero detection ----
#pragma unroll
    for (int r = 0; r < RPI; ++r) {
      const int lr = lrb + r;
      // In a chunk with an odd number of rows the second row of the last iteration does not exist.  Its slot and row
      // constants are zero-filled (mu = 0, log s = 0, x_c = 0), so its prior mean is the event's intercept b and it
      // would add b / sigma^2, 1 - (b^2 + 1) / sigma^2 and a KL term to the per-event intercept, sigma_log and loss
      // sums; those take zero for it (warp-uniform).  Its Wc terms are x_c * r = 0, and in cell mode (b = tau = 0
      // from the zero-filled row constants) every term is exactly 0.
      const bool real_row = RPI == 1 || CELL || lr < n_rows;
      const Vec* st = reinterpret_cast<const Vec*>(rs0 + r * SLOT) + lane;
      float xc[KC > 0 ? KC : 1], wg[KG > 0 ? KG : 1];
      float b_row = 0.f, tau_row = 0.f;
      if (NRC > 0) {
        const float* rc = s_rc + (stage * RPI + r) * kRowConstSlots;
#pragma unroll
        for (int k = 0; k < KC; ++k) xc[k] = rc[k];
#pragma unroll
        for (int k = 0; k < KG; ++k) wg[k] = rc[KC + (k ^ pk)];
        if (CELL) { b_row = rc[KC + KG]; tau_row = rc[KC + KG + 1]; }
        if (RPI == 1) __syncwarp();       // all lanes have read them before any lane's next prefetch overwrites the slot two iterations on
      }
      float c1[EPL], c2[EPL], c3[EPL], pmx[EPL];
#pragma unroll
      for (int j = 0; j < EPL; ++j) pmx[j] = 0.f;
      if (EXT) vec_get<EPL>(st[IPM * 32], pmx);
      vec_get<EPL>(st[0 * 32], mu[r]);
      vec_get<EPL>(st[1 * 32], lam[r]);
      vec_get<EPL>(st[2 * 32], c1);       // CODE8: the code words (as float bits)
      if (!CODE8) {
        vec_get<EPL>(st[3 * 32], c2);
        vec_get<EPL>(st[4 * 32], c3);
      }
      auto has_reads = [&](int j) {
        return CODE8 ? __float_as_uint(c1[j]) != 0u : c1[j] + c2[j] + c3[j] > 0.f;
      };
      float is2_row = 1.f;
      if (CELL) is2_row = fast_exp(-2.0f * tau_row);
      float caccr[NCELL > 0 ? NCELL : 1];
      float (&cacc)[NCELL > 0 ? NCELL : 1] = RPI == 1 ? cacc1 : caccr;
#pragma unroll
      for (int i = 0; i < (NCELL > 0 ? NCELL : 1); ++i) cacc[i] = 0.f;
      if (kSm) {  // this row's copy of the tile constants (dead again before the Monte-Carlo phase)
#pragma unroll
        for (int k = 0; k < KC; ++k) vec_get<EPL>(*reinterpret_cast<const Vec*>(&sk[k][lane * EPL]), wc[k]);
#pragma unroll
        for (int k = 0; k < KG; ++k)
          vec_get<EPL>(*reinterpret_cast<const Vec*>(&sk[KC + (k ^ pk)][lane * EPL]), xg[k]);
        if (!CELL) {
          vec_get<EPL>(*reinterpret_cast<const Vec*>(&sk[KC + KG][lane * EPL]), bb);
          vec_get<EPL>(*reinterpret_cast<const Vec*>(&sk[KC + KG + 1][lane * EPL]), tau);
          vec_get<EPL>(*reinterpret_cast<const Vec*>(&sk[KC + KG + 2][lane * EPL]), is2);
        }
      }
      static_assert(EPL % 2 == 0, "packed pairs need an even number of events per lane");
      float2 cacc2[NCELL > 0 ? NCELL : 1];
#pragma unroll
      for (int i = 0; i < (NCELL > 0 ? NCELL : 1); ++i) cacc2[i] = make_float2(0.f, 0.f);
#pragma unroll
      for (int p = 0; p < EPL / 2; ++p) {
        const int j0 = 2 * p, j1 = 2 * p + 1;
        const float2 tj = CELL ? f2_splat(tau_row) : make_float2(tau[j0], tau[j1]);
        const float2 i2 = CELL ? f2_splat(is2_row) : make_float2(is2[j0], is2[j1]);
        float2 pm = CELL ? f2_splat(b_row) : make_float2(bb[j0], bb[j1]);
        if (EXT) pm = f2_add(pm, make_float2(pmx[j0], pmx[j1]));
#pragma unroll
        for (int k = 0; k < KC; ++k) pm = f2_fma(f2_splat(xc[k]), make_float2(wc[k][j0], wc[k][j1]), pm);
#pragma unroll
        for (int k = 0; k < KG; ++k) pm = f2_fma(f2_splat(wg[k]), make_float2(xg[k][j0], xg[k][j1]), pm);
        const float2 d = f2_sub(make_float2(lam[r][j0], lam[r][j1]), tj);
        const float2 dd = f2_mul(d, f2_splat(2.0f * kLog2e));
        const float2 e2 = make_float2(ex2_approx(dd.x), ex2_approx(dd.y));   // s^2 / sigma^2
        const float2 diff = f2_sub(make_float2(mu[r][j0], mu[r][j1]), pm);
        const float2 rr = f2_mul(diff, i2);                                  // (mu - m) / sigma^2
        const float2 q2 = f2_mul(diff, rr);                                  // ((mu - m) / sigma)^2
        const float2 nr = make_float2(-rr.x, -rr.y);
        const float2 e2m1 = f2_add(e2, f2_splat(-1.0f));
        gmu[r][j0] = rr.x; gmu[r][j1] = rr.y;
        glam[r][j0] = e2m1.x; glam[r][j1] = e2m1.y;
        if (h == 0) {
          if (has_reads(j0)) nz |= 1u << (r * EPL + j0);
          if (has_reads(j1)) nz |= 1u << (r * EPL + j1);
        }
        const float2 gt = f2_sub(f2_sub(f2_splat(1.0f), q2), e2);            // d loss / d sigma_log
        if (grad_sums) {
#pragma unroll
          for (int k = 0; k < KC; ++k) {
            const float2 t = f2_fma(f2_splat(xc[k]), nr, make_float2(acc[k][j0], acc[k][j1]));
            acc[k][j0] = t.x; acc[k][j1] = t.y;
          }
        }
        const float2 rrs = real_row ? rr : f2_splat(0.f), gts = real_row ? gt : f2_splat(0.f);
        if (!CELL && grad_sums) {
          const float2 t = f2_sub(make_float2(acc[T::kGB][j0], acc[T::kGB][j1]), rrs);
          acc[T::kGB][j0] = t.x; acc[T::kGB][j1] = t.y;
          const float2 u = f2_add(make_float2(acc[T::kGT][j0], acc[T::kGT][j1]), gts);
          acc[T::kGT][j0] = u.x; acc[T::kGT][j1] = u.y;
        }
        if (LOSS) {                                                          // TFP _kl_normal_normal
          float2 kl = f2_sub(f2_fma(f2_splat(0.5f), q2, f2_mul(f2_splat(0.5f), e2m1)), d);
          if (!real_row) kl = f2_splat(0.f);
          const float2 t = f2_add(make_float2(acc[T::kLoss + h][j0], acc[T::kLoss + h][j1]), kl);
          acc[T::kLoss + h][j0] = t.x; acc[T::kLoss + h][j1] = t.y;
        }
        if (NCELL > 0) {
          const float2 nrm = make_float2((g0 + j0) < a.Ng ? nr.x : 0.f, (g0 + j1) < a.Ng ? nr.y : 0.f);
#pragma unroll
          for (int k = 0; k < KG; ++k) cacc2[k] = f2_fma(make_float2(xg[k][j0], xg[k][j1]), nrm, cacc2[k]);
          if (CELL) {
            const float2 gm = make_float2((g0 + j0) < a.Ng ? gt.x : 0.f, (g0 + j1) < a.Ng ? gt.y : 0.f);
            cacc2[KG] = f2_add(cacc2[KG], nrm);
            cacc2[KG + 1] = f2_add(cacc2[KG + 1], gm);
          }
        }
      }
#pragma unroll
      for (int i = 0; i < NCELL; ++i) cacc[i] = cacc2[i].x + cacc2[i].y;
      static_assert(!EXT || RPI == 1, "the wide-design store below writes every row of an iteration");
      if (EXT && act != 0)   // r = (mu - m) / sigma^2 of this row, for the gradient GEMMs (frozen lanes keep their old values: unused)
        __stcs(reinterpret_cast<Vec*>(bR + ((uint32_t)lr * ld32 + col32)), vec_make<EPL>(gmu[r]));
      if (RPI > 1 && NCELL > 0 && lr < n_rows) cell_reduce_store(cacc, row_begin + lr);
    }
    if (RPI > 1 && NRC > 0) __syncwarp(); // all lanes have read the row constants before the next prefetch of these slots

    // ---- phase B: compacted Monte-Carlo work (the items of all RPI rows share the passes) ----
    if (h == 0) {
#pragma unroll
      for (int j = 0; j < RPI * EPL; ++j) {
        bal[j] = __ballot_sync(0xffffffffu, nz & (1u << j));
        n_items += __popc(bal[j]);
      }
    }
    if (n_items > 0) {
      // The queue holds (row slot, tile column) only.  The rows' Z_loc, Z_std_log and counts are still in this stage
      // of the ring, so whichever lane takes an item reads them from there and leaves the Monte-Carlo sums in the
      // element's own count slots; an element without reads has zeros in those slots (counts are >= 0), so the
      // owners subtract their slots unconditionally afterwards.  (PAIR: the queue of the first step serves both; the
      // barrier below also publishes the first step's updated Z_loc / Z_std_log in the ring.)
      if (h == 0) {
        int base = 0;
#pragma unroll
        for (int j = 0; j < RPI * EPL; ++j) base += __popc(bal[j] & lt_mask);
#pragma unroll
        for (int j = 0; j < RPI * EPL; ++j)
          if ((nz >> j) & 1u)
            q[base + __popc(nz & ((1u << j) - 1u))] = (uint32_t)((j / EPL) * TC + lane * EPL + (j % EPL));
      }
      __syncwarp();
      for (int k = lane; k < n_items; k += 32) {
        const int item = (int)q[k];
        const int r = RPI > 1 ? item / TC : 0, col = RPI > 1 ? item % TC : item;
        float* rs = rs0 + r * SLOT;
        const float imu = rs[col], is = fast_exp(rs[TC + col]);
        float ic1, ic2, ic3;
        if (CODE8) {
          const uint32_t w = __float_as_uint(rs[2 * TC + col]);
          ic1 = s_dict[w & 255u];
          ic2 = s_dict[kDictSize + ((w >> 8) & 255u)];
          ic3 = s_dict[2 * kDictSize + ((w >> 16) & 255u)];
        } else {
          ic1 = rs[2 * TC + col]; ic2 = rs[3 * TC + col]; ic3 = rs[4 * TC + col];
        }
        const float in = ic1 + ic2 + ic3;
        const float l1 = s_L[0][col], l2 = s_L[1][col], l3 = s_L[2][col];
        float gs, ge, ls;
        mc_samples<LOSS>(imu, is, ic1, ic2, in, l1, l2, l3, l1 - l2, a.S, s_ev[col], (uint32_t)(row_begin + lrb + r),
                         a.step + (uint32_t)h, stream0, a.seed, gs, ge, ls);
        float* const out = SCR ? s_scr + r * (NSCR * TC) : rs + 2 * TC;
        out[col] = gs * a.inv_S;
        out[TC + col] = ge * is * a.inv_S;
        if (LOSS)
          out[2 * TC + col] = fmaf(ls, a.inv_S, fmaf(ic1, s_L[3][col], fmaf(ic2, s_L[4][col], ic3 * s_L[5][col])));
      }
      __syncwarp();
#pragma unroll
      for (int r = 0; r < RPI; ++r) {
        // SCR: the scratch holds sums only where this row had items, stale values elsewhere -- an element without
        // reads subtracts 0, as it subtracts its zero counts in the f32 form
        const Vec* st = SCR ? reinterpret_cast<const Vec*>(s_scr + r * (NSCR * TC)) + lane
                            : reinterpret_cast<const Vec*>(rs0 + r * SLOT + 2 * TC) + lane;
        float r1[EPL], r2[EPL];
        vec_get<EPL>(st[0 * 32], r1);
        vec_get<EPL>(st[1 * 32], r2);
        if (SCR) {
#pragma unroll
          for (int j = 0; j < EPL; ++j) {
            const bool hit = (nz >> (r * EPL + j)) & 1u;
            r1[j] = hit ? r1[j] : 0.f;
            r2[j] = hit ? r2[j] : 0.f;
          }
        }
#pragma unroll
        for (int j = 0; j < EPL; ++j) {
          gmu[r][j] -= r1[j];
          glam[r][j] -= r2[j];
        }
        if (LOSS) {
          float r3[EPL];
          vec_get<EPL>(st[2 * 32], r3);
#pragma unroll
          for (int j = 0; j < EPL; ++j) acc[T::kLoss + h][j] -= SCR && !((nz >> (r * EPL + j)) & 1u) ? 0.f : r3[j];
        }
      }
    }

    // ---- phase C: Adam on Z_loc / Z_std_log, clip, store (PAIR, first step: back into the ring slot) ----
#pragma unroll
    for (int r = 0; r < RPI; ++r) {
      const int lr = lrb + r;
      if (act != 0 && (RPI == 1 || lr < n_rows)) {
        const Vec* st = reinterpret_cast<const Vec*>(rs0 + r * SLOT) + lane;
        float m1[EPL], v1[EPL], m2[EPL], v2[EPL];
        vec_get<EPL>(st[(IA + 0) * 32], m1);
        vec_get<EPL>(st[(IA + 1) * 32], v1);
        vec_get<EPL>(st[(IA + 2) * 32], m2);
        vec_get<EPL>(st[(IA + 3) * 32], v2);
        if (all_act) {
#pragma unroll
          for (int p = 0; p < EPL / 2; ++p) {
            const int j0 = 2 * p, j1 = 2 * p + 1;
            adam_update2(mu[r][j0], mu[r][j1], m1[j0], m1[j1], v1[j0], v1[j1], gmu[r][j0], gmu[r][j1], alpha);
            adam_update2(lam[r][j0], lam[r][j1], m2[j0], m2[j1], v2[j0], v2[j1], glam[r][j0], glam[r][j1], alpha);
            mu[r][j0] = clip9(mu[r][j0]);  // Variable constraint (model_TFProb.py:80-81)
            mu[r][j1] = clip9(mu[r][j1]);
          }
        } else {
#pragma unroll
          for (int j = 0; j < EPL; ++j) {
            if ((act >> j) & 1u) {
              adam_update(mu[r][j], m1[j], v1[j], gmu[r][j], alpha);
              adam_update(lam[r][j], m2[j], v2[j], glam[r][j], alpha);
              mu[r][j] = clip9(mu[r][j]);
            }
          }
        }
        if (h < NSTEP - 1) {
          Vec* sw = reinterpret_cast<Vec*>(rs0 + r * SLOT) + lane;
          sw[0 * 32] = vec_make<EPL>(mu[r]);
          sw[1 * 32] = vec_make<EPL>(lam[r]);
          sw[(IA + 0) * 32] = vec_make<EPL>(m1);
          sw[(IA + 1) * 32] = vec_make<EPL>(v1);
          sw[(IA + 2) * 32] = vec_make<EPL>(m2);
          sw[(IA + 3) * 32] = vec_make<EPL>(v2);
        } else {
          const uint32_t rel = (uint32_t)lr * ld32 + col32;
          __stcs(reinterpret_cast<Vec*>(bZl + rel), vec_make<EPL>(mu[r]));
          __stcs(reinterpret_cast<Vec*>(bZs + rel), vec_make<EPL>(lam[r]));
          __stcs(reinterpret_cast<Vec*>(bA0 + rel), vec_make<EPL>(m1));
          __stcs(reinterpret_cast<Vec*>(bA1 + rel), vec_make<EPL>(v1));
          __stcs(reinterpret_cast<Vec*>(bA2 + rel), vec_make<EPL>(m2));
          __stcs(reinterpret_cast<Vec*>(bA3 + rel), vec_make<EPL>(v2));
        }
        if (PAIR && h == NSTEP - 1) {
          // statistics of the state just written around this step's parameters, centred there: the zero-count
          // elements' Z_loc sit close to the prior mean, so sums taken around 0 would cancel
          const float* rc = s_rc + (stage * RPI + r) * kRowConstSlots;
          float xs[KC > 0 ? KC : 1];
#pragma unroll
          for (int k = 0; k < KC; ++k) xs[k] = rc[k];
#pragma unroll
          for (int k = 0; k < KC; ++k) vec_get<EPL>(*reinterpret_cast<const Vec*>(&sk[k][lane * EPL]), wc[k]);
          vec_get<EPL>(*reinterpret_cast<const Vec*>(&sk[KC][lane * EPL]), bb);
          vec_get<EPL>(*reinterpret_cast<const Vec*>(&sk[KC + 1][lane * EPL]), tau);
#pragma unroll
          for (int j = 0; j < EPL; ++j) {
            float pm = bb[j];
#pragma unroll
            for (int k = 0; k < KC; ++k) pm = fmaf(xs[k], wc[k][j], pm);
            const float dv = mu[r][j] - pm;
#pragma unroll
            for (int k = 0; k < KC; ++k) stat[k][j] = fmaf(xs[k], dv, stat[k][j]);
            stat[KC][j] += dv;
            stat[KC + 1][j] = fmaf(dv, dv, stat[KC + 1][j]);
            stat[KC + 2][j] += ex2_approx((lam[r][j] - tau[j]) * (2.0f * kLog2e));
          }
        }
      }
    }
    if (RPI == 1 && NCELL > 0) cell_reduce_store(cacc1, row_begin + lrb);
    }
    if (PAIR) __syncwarp();   // all lanes have read this stage's row constants and ring slots before the next prefetch
  }
  cp_async_wait<0>();

  if (NEV > 0) {
    __syncthreads();  // all warps are done with their queues; reuse the memory for the reduction
    float(*red)[TC] = reinterpret_cast<float(*)[TC]>(smem + kWarps * kRingStages * RPI * SLOT);
    const int64_t gcol = thread_col();
#pragma unroll
    for (int i = 0; i < NEV; ++i) {
      *reinterpret_cast<Vec*>(&red[warp][lane * EPL]) = vec_make<EPL>(acc[i]);
      __syncthreads();
      if (threadIdx.x < TC && gcol < a.ld) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) s += red[w][threadIdx.x];
        a.part_ev[(((int64_t)chunk * a.M + m) * NEV + i) * a.ld + gcol] = s;
      }
      __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < NST; ++i) {
      *reinterpret_cast<Vec*>(&red[warp][lane * EPL]) = vec_make<EPL>(stat[i]);
      __syncthreads();
      if (threadIdx.x < TC && gcol < a.ld) {
        float s = 0.f;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) s += red[w][threadIdx.x];
        a.part_st[(((int64_t)chunk * a.M + m) * NST + i) * a.ld + gcol] = s;
      }
      __syncthreads();
    }
  }
}

// Per-event finalize: reduce the row-chunk partials in fixed order, Adam on Wc /
// per-event intercept / sigma_log (keras Adam + clip, model_TFProb.py:68-69), and
// write the pre-update per-event loss  sum_c KL - sum_c loglik  (:207-211).
struct EventArgs {
  int64_t ld, Ng;
  int32_t M, KC, NEV, n_chunks;
  int32_t idx_gb, idx_gt, idx_loss;  // -1 if absent
  int32_t train_b, train_tau, trace_slot, trace_cap;
  float alpha;
  const float* part_ev;
  float* Wc; float* b; float* tau;
  float* mom;          // (2, M, KC + 2, ld)
  const uint8_t* active;
  float* trace;
  uint32_t xc_mask[kMaxModels];
  // wide designs: d loss / d Wc comes from a GEMM as a dense (M, KC, ld) array, rows [0, xc_width[m]) in use
  const float* wc_grad;
  int32_t xc_width[kMaxModels];
  // Two-step passes (brie_fit_run_steps).  idx_loss2 >= 0: the row of the pass' second loss, for trace_slot + 1.
  // prev (M, KC + 2, ld), if set, receives the parameters the next pass takes its first step with: those before this
  // update, or with part_st those after the first of two updates.  part_st, if set: the pass' statistics
  // (pair_stat_rows), from which the look-ahead update with alpha2 takes its sums; gram (M, KC * KC + KC) holds
  // sum_c x_c x_c^T and sum_c x_c in float64, and Nc is the number of cells.
  int32_t idx_loss2;
  float* prev;
  const float* part_st;
  const double* gram;
  int64_t Nc;
  float alpha2;
};

constexpr int kMaxNEV = 20;  // BRIE_MAX_KC + 2 + 2 (two loss rows of a two-step pass)
constexpr int kMaxNST = 7;   // pair_stat_rows(kMaxPairKc)

// block = 8 warps x 32 events: warp w sums row chunks w, w+8, ... (coalesced 128-byte rows of the
// partial buffer), warp 0 combines the 8 sub-sums in fixed order (f64) and applies the updates.
__global__ void __launch_bounds__(256) event_update_kernel(const EventArgs a) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t g = (int64_t)blockIdx.x * 32 + lane;
  const int m = blockIdx.y;
  __shared__ float s_part[8][kMaxNEV + kMaxNST][32];
  const bool ok = g < a.Ng && a.active[(int64_t)m * a.ld + g] != 0;
  const int nst = a.part_st && a.KC <= kMaxPairKc ? pair_stat_rows(a.KC) : 0;
  if (ok) {
    for (int i = 0; i < a.NEV + nst; ++i) {
      const float* src = i < a.NEV ? a.part_ev + (int64_t)i * a.ld : a.part_st + (int64_t)(i - a.NEV) * a.ld;
      const int n = i < a.NEV ? a.NEV : nst;
      float s = 0.f;
      for (int c = w; c < a.n_chunks; c += 8) s += src[(((int64_t)c * a.M + m) * n) * a.ld + g];
      s_part[w][i][lane] = s;
    }
  }
  __syncthreads();
  if (w != 0 || g >= a.Ng) return;
  float* const wc = a.Wc + (int64_t)m * a.KC * a.ld + g;   // row k at wc[k * ld]
  float* const bp = a.b + (int64_t)m * a.ld + g;
  float* const tp = a.tau + (int64_t)m * a.ld + g;
  auto save_prev = [&]() {
    float* p = a.prev + (int64_t)m * (a.KC + 2) * a.ld + g;
    for (int k = 0; k < a.KC; ++k) p[k * a.ld] = wc[k * a.ld];
    p[a.KC * a.ld] = *bp;
    p[(a.KC + 1) * a.ld] = *tp;
  };
  // frozen events keep their parameters; the next pass still reads them
  if (!ok) { if (a.prev) save_prev(); return; }
  if (a.prev && !a.part_st) save_prev();
  // look-ahead (part_st set only for KC <= kMaxPairKc, brie_fit_create): the parameters before the update are its
  // reference point (w', b', tau'); fixed-size, fully unrolled, so they stay in registers
  const bool look_ahead = a.part_st != nullptr && a.KC <= kMaxPairKc;
  float w0[kMaxPairKc] = {};
  float b0 = 0.f, t0 = 0.f;
  if (look_ahead) {
#pragma unroll
    for (int k = 0; k < kMaxPairKc; ++k)
      if (k < a.KC) w0[k] = wc[k * a.ld];
    b0 = *bp; t0 = *tp;
  }
  auto red = [&](int i) {
    double s = 0.0;
#pragma unroll
    for (int ww = 0; ww < 8; ++ww) s += (double)s_part[ww][i][lane];
    return s;
  };
  const int64_t mstride = (int64_t)a.M * (a.KC + 2) * a.ld;
  auto adam_slot = [&](float* x, int slot, float grad, bool clip, float alpha) {
    const int64_t qi = ((int64_t)m * (a.KC + 2) + slot) * a.ld + g;
    adam_at(x, a.mom + qi, a.mom + mstride + qi, grad, alpha, clip);
  };
  auto trained = [&](int k) { return a.wc_grad ? k < a.xc_width[m] : ((a.xc_mask[m] >> k) & 1u) != 0; };
  for (int k = 0; k < a.KC; ++k) {
    if (!trained(k)) continue;
    const float grad = a.wc_grad ? a.wc_grad[((int64_t)m * a.KC + k) * a.ld + g] : (float)red(k);
    adam_slot(wc + k * a.ld, k, grad, false, a.alpha);
  }
  if (a.idx_gb >= 0 && a.train_b) adam_slot(bp, a.KC, (float)red(a.idx_gb), true, a.alpha);
  if (a.idx_gt >= 0 && a.train_tau) adam_slot(tp, a.KC + 1, (float)red(a.idx_gt), false, a.alpha);
  if (a.idx_loss >= 0 && a.trace_slot >= 0)
    a.trace[((int64_t)m * a.trace_cap + a.trace_slot) * a.ld + g] = (float)red(a.idx_loss);
  if (a.idx_loss2 >= 0 && a.trace_slot >= 0)
    a.trace[((int64_t)m * a.trace_cap + a.trace_slot + 1) * a.ld + g] = (float)red(a.idx_loss2);
  if (!look_ahead) return;

  // Look-ahead update.  The statistics R_k = sum_c x_ck d_c, R_0 = sum_c d_c, Q = sum_c d_c^2, E = sum_c exp(2 (lam_c
  // - tau')) with d_c = mu_c - p'_c were taken around the parameters (w', b', tau') the pass stepped with, which the
  // updates above moved by (dw, db, dtau).  Around the new ones, p_c = p'_c + x_c . dw + db, so
  //   sum_c x_ck (mu_c - p_c) = R_k - (G dw)_k - s_k db,   sum_c (mu_c - p_c) = R_0 - s . dw - n db,
  //   sum_c (mu_c - p_c)^2 = Q - 2 (dw . R + db R_0) + dw^T G dw + 2 db s . dw + n db^2,
  //   sum_c exp(2 (lam_c - tau)) = E exp(-2 dtau)
  // (G = sum_c x_c x_c^T, s = sum_c x_c, n cells), and the KL gradients of the next step follow exactly.
  save_prev();
  const int K = a.KC, i0 = a.NEV;      // statistic rows follow the a.NEV gradient / loss rows in s_part
  const double* G = a.gram + (int64_t)m * (K * K + K);
  const double* sv = G + K * K;
  const double n = (double)a.Nc;
  double dw[kMaxPairKc], Gdw[kMaxPairKc];
#pragma unroll
  for (int k = 0; k < kMaxPairKc; ++k) dw[k] = k < K ? (double)wc[k * a.ld] - (double)w0[k] : 0.0;   // 0 untrained
  const double db = (double)*bp - (double)b0, dt = (double)*tp - (double)t0;
  const double R0 = red(i0 + K), Q = red(i0 + K + 1), E = red(i0 + K + 2);
  double sdw = 0.0, wR = 0.0, wGw = 0.0;
#pragma unroll
  for (int k = 0; k < kMaxPairKc; ++k) {
    Gdw[k] = 0.0;
    if (k >= K) continue;
#pragma unroll
    for (int l = 0; l < kMaxPairKc; ++l)
      if (l < K) Gdw[k] += G[k * K + l] * dw[l];
    sdw += sv[k] * dw[k];
    wR += dw[k] * red(i0 + k);
    wGw += dw[k] * Gdw[k];
  }
  const double kappa = exp(-2.0 * (double)*tp);
#pragma unroll
  for (int k = 0; k < kMaxPairKc; ++k) {
    if (k >= K || !trained(k)) continue;
    adam_slot(wc + k * a.ld, k, (float)(-kappa * (red(i0 + k) - Gdw[k] - sv[k] * db)), false, a.alpha2);
  }
  const double S0 = R0 - sdw - n * db;
  const double S2 = Q - 2.0 * (wR + db * R0) + wGw + 2.0 * db * sdw + n * db * db;
  if (a.train_b) adam_slot(bp, K, (float)(-kappa * S0), true, a.alpha2);
  if (a.train_tau) adam_slot(tp, K + 1, (float)(n - kappa * S2 - E * exp(-2.0 * dt)), false, a.alpha2);
}

// Sums-only pre-pass of a run of two-step passes: the per-event gradient sums of one step (the KL terms, the only
// source of the per-event parameters' gradients in gene mode with Kg = 0) from Z_loc and Z_std_log, in
// elbo_step_kernel's row-chunk partial layout (KC + 2 rows), for event_update_kernel.  Lanes whose events are all
// frozen read nothing.
template <int KC>
__global__ void __launch_bounds__(kThreads) kl_sums_kernel(const StepArgs a) {
  constexpr int EPL = step_epl(KC), TC = 32 * EPL, NEV = KC + 2;
  using Vec = typename LaneVec<EPL>::type;
  const int m = blockIdx.x, tile = blockIdx.y, chunk = blockIdx.z;
  if (!((a.model_mask >> m) & 1u)) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t g0 = (int64_t)tile * TC + lane * EPL;
  bool act = false;
  if (g0 < a.ld) {
#pragma unroll
    for (int j = 0; j < EPL; ++j) act |= a.active[(int64_t)m * a.ld + g0 + j] != 0;
  }
  if (!__syncthreads_or(act)) return;
  float wc[KC > 0 ? KC : 1][EPL], bb[EPL], tau[EPL], is2[EPL], acc[NEV][EPL];
#pragma unroll
  for (int j = 0; j < EPL; ++j) {
    bb[j] = 0.f; tau[j] = 0.f;
#pragma unroll
    for (int k = 0; k < (KC > 0 ? KC : 1); ++k) wc[k][j] = 0.f;
#pragma unroll
    for (int i = 0; i < NEV; ++i) acc[i][j] = 0.f;
  }
  if (act) {
#pragma unroll
    for (int k = 0; k < KC; ++k) vec_get<EPL>(*reinterpret_cast<const Vec*>(a.Wc + ((int64_t)m * KC + k) * a.ld + g0), wc[k]);
    vec_get<EPL>(*reinterpret_cast<const Vec*>(a.b + (int64_t)m * a.ld + g0), bb);
    vec_get<EPL>(*reinterpret_cast<const Vec*>(a.tau + (int64_t)m * a.ld + g0), tau);
  }
#pragma unroll
  for (int j = 0; j < EPL; ++j) is2[j] = fast_exp(-2.0f * tau[j]);
  const int64_t row_begin = (int64_t)chunk * a.rows_per_cta;
  const int64_t row_end = min(row_begin + (int64_t)a.rows_per_cta, a.Nc);
  const int64_t plane = a.Nc * a.ld;
  for (int64_t row = row_begin + warp; act && row < row_end; row += kWarps) {
    float mu[EPL], lam[EPL], xc[KC > 0 ? KC : 1];
    const int64_t off = (int64_t)m * plane + row * a.ld + g0;
    vec_get<EPL>(__ldcs(reinterpret_cast<const Vec*>(a.Zl + off)), mu);
    vec_get<EPL>(__ldcs(reinterpret_cast<const Vec*>(a.Zs + off)), lam);
#pragma unroll
    for (int k = 0; k < KC; ++k) xc[k] = a.Xc[((int64_t)m * a.Nc + row) * KC + k];
#pragma unroll
    for (int j = 0; j < EPL; ++j) {
      float pm = bb[j];
#pragma unroll
      for (int k = 0; k < KC; ++k) pm = fmaf(xc[k], wc[k][j], pm);
      const float diff = mu[j] - pm, rr = diff * is2[j];
      const float e2 = ex2_approx((lam[j] - tau[j]) * (2.0f * kLog2e));
#pragma unroll
      for (int k = 0; k < KC; ++k) acc[k][j] = fmaf(xc[k], -rr, acc[k][j]);
      acc[KC][j] -= rr;
      acc[KC + 1][j] += (1.0f - diff * rr) - e2;
    }
  }
  __shared__ float red[kWarps][TC];
#pragma unroll
  for (int i = 0; i < NEV; ++i) {
    *reinterpret_cast<Vec*>(&red[warp][lane * EPL]) = vec_make<EPL>(acc[i]);
    __syncthreads();
    const int64_t g = (int64_t)tile * TC + threadIdx.x;
    if (threadIdx.x < TC && g < a.ld) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < kWarps; ++w) s += red[w][threadIdx.x];
      a.part_ev[(((int64_t)chunk * a.M + m) * NEV + i) * a.ld + g] = s;
    }
    __syncthreads();
  }
}

// gram[m] = (sum_c x_c x_c^T (K x K), sum_c x_c (K)) of model m's design rows, in float64 and a fixed order: one block
// per entry and model.
__global__ void __launch_bounds__(256) gram_kernel(const float* Xc, int64_t Nc, int K, double* gram) {
  const int e = blockIdx.x, m = blockIdx.y;
  const int i = e < K * K ? e / K : e - K * K, j = e < K * K ? e % K : -1;
  const float* X = Xc + (int64_t)m * Nc * K;
  double s = 0.0;
  for (int64_t c = threadIdx.x; c < Nc; c += blockDim.x)
    s += (double)X[c * K + i] * (j >= 0 ? (double)X[c * K + j] : 1.0);
  __shared__ double red[256];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) gram[(int64_t)m * (K * K + K) + e] = red[0];
}


// Per-cell gradient reduce over column tiles: G[m, c, i] = sum_tiles part_cell.
struct CellArgs {
  int64_t Nc;
  int32_t M, KG, NCELL, n_tiles;
  int32_t cell_mode, train_b, train_tau;
  uint32_t model_mask;
  float alpha;
  const float* part_cell;
  float* G;            // (M, Nc, NCELL)
  float* Wg; float* b; float* tau;
  float* mom;          // (2, M, Nc, KG + 2)
  int32_t n_part, part_off;   // the partials hold n_part values per cell, which land at G[.., part_off + j]
};

__global__ void __launch_bounds__(256) cell_reduce_kernel(const CellArgs a) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // over Nc * n_part
  const int m = blockIdx.y;
  if (i >= a.Nc * a.n_part) return;
  if (!((a.model_mask >> m) & 1u)) return;
  double s = 0.0;
  for (int t = 0; t < a.n_tiles; ++t)
    s += (double)a.part_cell[((int64_t)t * a.M + m) * a.Nc * a.n_part + i];
  const int64_t c = i / a.n_part, j = i % a.n_part;
  a.G[((int64_t)m * a.Nc + c) * a.NCELL + a.part_off + j] = (float)s;
}

__global__ void __launch_bounds__(256) cell_update_kernel(const CellArgs a) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int m = blockIdx.y;
  if (c >= a.Nc) return;
  if (!((a.model_mask >> m) & 1u)) return;
  const float* G = a.G + ((int64_t)m * a.Nc + c) * a.NCELL;
  const int64_t mstride = (int64_t)a.M * a.Nc * (a.KG + 2);
  float* mom = a.mom + ((int64_t)m * a.Nc + c) * (a.KG + 2);
  for (int k = 0; k < a.KG; ++k)
    adam_at(a.Wg + ((int64_t)m * a.Nc + c) * a.KG + k, mom + k, mom + mstride + k, G[k], a.alpha);
  if (a.cell_mode) {
    if (a.train_b)
      adam_at(a.b + (int64_t)m * a.Nc + c, mom + a.KG, mom + mstride + a.KG, G[a.KG], a.alpha, true);
    if (a.train_tau)
      adam_at(a.tau + (int64_t)m * a.Nc + c, mom + a.KG + 1, mom + mstride + a.KG + 1, G[a.KG + 1], a.alpha);
  }
}

// IEEE-accurate model terms of eval_loss_kernel, element_terms_kernel and margin_step_kernel (brie_margin.cuh).
// The fused step kernel has its own fast-math forms (mc_samples).
//
// Effective lengths of event g: the (3, ld) effLen table, or (1, 1, 0) -- the binomial branch,
// model_TFProb.py:162-167 -- without one.
__device__ __forceinline__ void event_lengths(const float* eff, int64_t ld, int64_t g, float& L1, float& L2,
                                              float& L3) {
  L1 = 1.f; L2 = 1.f; L3 = 0.f;
  if (eff) { L1 = eff[g]; L2 = eff[ld + g]; L3 = eff[2 * ld + g]; }
}

// The length constant c1 log L1 + c2 log L2 + c3 log L3 of the log-likelihood (0 without effLen).
__device__ __forceinline__ float log_length_const(bool eff, float c1, float c2, float c3, float L1, float L2,
                                                  float L3) {
  return eff ? fmaf(c1, logf(L1), fmaf(c2, logf(L2), c3 * logf(L3))) : 0.f;
}

// Prior mean intercept + Xc Wc + Wg Xg^T of (row, event g) for model m (model_TFProb.py:118-126); `base` is the
// intercept.  A is any argument struct with the fields Nc, ld, KC, KG, Xc, Wc, Wg, Xg.  T is the accumulation type:
// float for the model terms, double for the score pass (brie_score.cuh), whose residuals Z_loc - prior mean of cells
// without reads are far smaller than the float32 rounding of the sum.
template <class T, class A>
__device__ __forceinline__ T prior_mean(const A& a, int m, int64_t row, int64_t g, T base) {
  T pm = base;
  for (int k = 0; k < a.KC; ++k)
    pm = fma((T)a.Xc[((int64_t)m * a.Nc + row) * a.KC + k], (T)a.Wc[((int64_t)m * a.KC + k) * a.ld + g], pm);
  for (int k = 0; k < a.KG; ++k) pm = fma((T)a.Wg[((int64_t)m * a.Nc + row) * a.KG + k], (T)a.Xg[g * a.KG + k], pm);
  return pm;
}

// KL(N(mu, exp(lam)) || N(pm, exp(tau))) (model_TFProb.py:208).
__device__ __forceinline__ float kl_normal(float mu, float lam, float pm, float tau) {
  const float d = lam - tau;
  const float r0 = (mu - pm) * expf(-tau);
  return 0.5f * r0 * r0 + 0.5f * expm1f(2.0f * d) - d;
}

// Log-likelihood of one sample z (logLik_MC, model_TFProb.py:159-185) without the length constant:
//   l = c1 log psi + c2 log(1-psi) - n log D,   D = psi L1 + (1-psi) L2 + L3   (no n log D without effLen).
// psi, q = 1 - psi and D come back too, for dl/dz.
struct SampleLL { float l, psi, q, D; };
__device__ __forceinline__ SampleLL sample_ll(float z, float c1, float c2, float n, float L1, float L2, float L3,
                                              bool eff) {
  SampleLL r;
  const float e = expf(-fabsf(z));
  const float lsp = fminf(z, 0.f) - log1pf(e);
  const float inv = 1.0f / (1.0f + e);
  r.psi = z >= 0.f ? inv : e * inv;
  r.q = z >= 0.f ? e * inv : inv;
  r.D = fmaf(r.psi, L1, fmaf(r.q, L2, L3));
  r.l = fmaf(c1, lsp, c2 * (lsp - z)) - (eff ? n * logf(r.D) : 0.f);
  return r;
}

// Streaming log-mean-exp of sample log-likelihoods (tfp.math.reduce_logmeanexp, model_TFProb.py:188-189).
struct LogMeanExp {
  float mx = -INFINITY, Z = 0.f;
  __device__ __forceinline__ void add(float l) {
    if (l > mx) { Z *= expf(mx - l); mx = l; }
    Z += expf(l - mx);
  }
  __device__ __forceinline__ float value(int S) const { return mx + logf(Z) - logf((float)S); }
};

// Forward-only per-event loss with n_eval x S fresh-noise samples per element
// (the 500x get_loss(axis=0) loop of model_TFProb.py:261-264 in one pass).  Only
// elements with reads need samples: a zero-count element's log-lik is 0 for any z.
// IEEE-accurate math (this value feeds ELBO_gain, model_wrap.py:183-185).
struct EvalArgs {
  int64_t Nc, Ng, ld, event_offset;
  uint64_t seed;
  const float* c[3];
  const float* eff;
  const float* Xc; const float* Xg;
  const float* Zl; const float* Zs;
  const float* Wc; const float* b; const float* tau; const float* Wg;
  float* part_ev;      // (n_row_chunks, M, 2, ld)
  int32_t M, S, n_eval, rows_per_cta, KC, KG, cell_mode;
  int32_t margin;      // 1: target = "marginLik" -- samples from the prior, log-mean-exp per evaluation, no KL
  int32_t model_id[kMaxModels];
};

// One element with reads: its n_eval evaluations are spread over the 32 lanes (lane takes
// evaluations lane, lane+32, ...), so lane utilisation does not depend on the sparsity pattern;
// the warp sum is a fixed xor-shuffle tree (deterministic).  Returns sum over all samples of
// c1 log psi + c2 log(1-psi) - n log D  (without the constant sum_k c_k log L_k); with `margin`
// every evaluation contributes S x log-mean-exp of its S sample log-likelihoods instead
// (tfp.math.reduce_logmeanexp, model_TFProb.py:188-189), so the caller's 1/(n_eval S) applies to both.
__device__ __forceinline__ float eval_item(float mu, float s, float c1, float c2, float n, float L1, float L2,
                                           float L3, bool eff, bool margin, int n_eval, int S, uint32_t event,
                                           uint32_t cell, uint32_t stream0, uint64_t seed, int lane) {
  float acc = 0.f;
  for (int it = lane; it < n_eval; it += 32) {
    LogMeanExp lme;
    for (int s0 = 0; s0 < S; s0 += 4) {
      float eps[4];
      brie_normals4(event, cell, (uint32_t)it, stream0 + (uint32_t)(s0 >> 2), seed, eps);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (s0 + q < S) {
          const float l = sample_ll(fmaf(s, eps[q], mu), c1, c2, n, L1, L2, L3, eff).l;
          if (!margin) acc += l;
          else lme.add(l);
        }
      }
    }
    if (margin) acc += (float)S * lme.value(S);
  }
  return warp_sum(acc);
}

__global__ void __launch_bounds__(kThreads) eval_loss_kernel(const EvalArgs a) {
  const int m = blockIdx.x, tile = blockIdx.y, chunk = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t g0 = (int64_t)tile * kTileCols + lane * 4;
  const bool in_ld = g0 < a.ld;
  float kl[4] = {0.f, 0.f, 0.f, 0.f}, ll[4] = {0.f, 0.f, 0.f, 0.f};
  const int64_t row_begin = (int64_t)chunk * a.rows_per_cta;
  const int64_t row_end = min(row_begin + (int64_t)a.rows_per_cta, a.Nc);
  const int64_t plane = a.Nc * a.ld;
  const uint32_t stream0 = brie_stream_word(BRIE_PHASE_EVAL, (uint32_t)a.model_id[m], 0u);
  const float inv_n = 1.0f / ((float)a.n_eval * (float)a.S);
  const bool eff = a.eff != nullptr;
  float L1[4], L2[4], L3[4], bb[4], tau[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int64_t gj = g0 + j;
    L1[j] = 1.f; L2[j] = 1.f; L3[j] = 0.f; bb[j] = 0.f; tau[j] = 0.f;
    if (gj < a.ld) {
      event_lengths(a.eff, a.ld, gj, L1[j], L2[j], L3[j]);
      if (!a.cell_mode) { bb[j] = a.b[(int64_t)m * a.ld + gj]; tau[j] = a.tau[(int64_t)m * a.ld + gj]; }
    }
  }
  for (int64_t row = row_begin + warp; row < row_end; row += kWarps) {
    float mu[4] = {0.f, 0.f, 0.f, 0.f}, lam[4] = {0.f, 0.f, 0.f, 0.f};
    float c1[4] = {0.f, 0.f, 0.f, 0.f}, c2[4] = {0.f, 0.f, 0.f, 0.f}, c3[4] = {0.f, 0.f, 0.f, 0.f};
    if (in_ld) {
      const int64_t off = row * a.ld + g0;
      const float4 t0 = *reinterpret_cast<const float4*>(a.Zl + (int64_t)m * plane + off);
      const float4 t1 = *reinterpret_cast<const float4*>(a.Zs + (int64_t)m * plane + off);
      const float4 t2 = *reinterpret_cast<const float4*>(a.c[0] + off);
      const float4 t3 = *reinterpret_cast<const float4*>(a.c[1] + off);
      mu[0] = t0.x; mu[1] = t0.y; mu[2] = t0.z; mu[3] = t0.w;
      lam[0] = t1.x; lam[1] = t1.y; lam[2] = t1.z; lam[3] = t1.w;
      c1[0] = t2.x; c1[1] = t2.y; c1[2] = t2.z; c1[3] = t2.w;
      c2[0] = t3.x; c2[1] = t3.y; c2[2] = t3.z; c2[3] = t3.w;
      if (a.c[2]) {
        const float4 t4 = *reinterpret_cast<const float4*>(a.c[2] + off);
        c3[0] = t4.x; c3[1] = t4.y; c3[2] = t4.z; c3[3] = t4.w;
      }
    }
    float b_row = 0.f, tau_row = 0.f;
    if (a.cell_mode) { b_row = a.b[(int64_t)m * a.Nc + row]; tau_row = a.tau[(int64_t)m * a.Nc + row]; }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int64_t gj = g0 + j;
      const bool valid = gj < a.Ng;
      float n = 0.f;
      float zc = mu[j], zsl = lam[j];       // centre and log-scale the samples are drawn around
      if (valid) {
        const float tj = a.cell_mode ? tau_row : tau[j];
        const float pm = prior_mean(a, m, row, gj, a.cell_mode ? b_row : bb[j]);
        if (a.margin) { zc = pm; zsl = tj; }   // prior samples, no KL term (model_TFProb.py:156-157, 202-205)
        else kl[j] += kl_normal(mu[j], lam[j], pm, tj);
        n = c1[j] + c2[j] + c3[j];
      }
      // elements with reads, one at a time, all 32 lanes cooperating
      uint32_t todo = __ballot_sync(0xffffffffu, n > 0.f);
      while (todo) {
        const int src = __ffs(todo) - 1;
        todo &= todo - 1;
        const float imu = __shfl_sync(0xffffffffu, zc, src), ilam = __shfl_sync(0xffffffffu, zsl, src);
        const float ic1 = __shfl_sync(0xffffffffu, c1[j], src), ic2 = __shfl_sync(0xffffffffu, c2[j], src);
        const float in = __shfl_sync(0xffffffffu, n, src);
        const float l1 = __shfl_sync(0xffffffffu, L1[j], src), l2 = __shfl_sync(0xffffffffu, L2[j], src);
        const float l3 = __shfl_sync(0xffffffffu, L3[j], src);
        const uint32_t ev = (uint32_t)(a.event_offset + (int64_t)tile * kTileCols + src * 4 + j);
        const float tot = eval_item(imu, expf(ilam), ic1, ic2, in, l1, l2, l3, eff, a.margin != 0, a.n_eval, a.S, ev,
                                    (uint32_t)row, stream0, a.seed, lane);
        if (lane == src) ll[j] += fmaf(tot, inv_n, log_length_const(eff, c1[j], c2[j], c3[j], L1[j], L2[j], L3[j]));
      }
    }
  }
  __shared__ float red[kWarps][kTileCols];
  for (int i = 0; i < 2; ++i) {
    *reinterpret_cast<float4*>(&red[warp][lane * 4]) =
        i == 0 ? make_float4(kl[0], kl[1], kl[2], kl[3]) : make_float4(ll[0], ll[1], ll[2], ll[3]);
    __syncthreads();
    const int64_t gcol = (int64_t)tile * kTileCols + threadIdx.x;
    if (threadIdx.x < kTileCols && gcol < a.ld) {
      float s = 0.f;
      for (int w = 0; w < kWarps; ++w) s += red[w][threadIdx.x];
      a.part_ev[(((int64_t)chunk * a.M + m) * 2 + i) * a.ld + gcol] = s;
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(256) eval_reduce_kernel(const float* part_ev, int n_chunks, int M,
                                                          int64_t ld, int64_t Ng, float* out) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int m = blockIdx.y;
  if (g >= ld) return;
  double kl = 0.0, ll = 0.0;
  if (g < Ng) {
    for (int c = 0; c < n_chunks; ++c) {
      kl += (double)part_ev[(((int64_t)c * M + m) * 2 + 0) * ld + g];
      ll += (double)part_ev[(((int64_t)c * M + m) * 2 + 1) * ld + g];
    }
  }
  out[(int64_t)m * ld + g] = (float)(kl - ll);
}

// Element-wise terms of the public model API (BRIE2.logLik_MC, Z_prior, the KL inside get_loss;
// model_TFProb.py:118-127, 130-191, 208) for ONE model, written as dense (Nc, ld) arrays -- the reference
// returns exactly these (Nc, Ng) tensors.  One warp per 128-event row segment as in eval_loss_kernel; every
// element draws its own `S` samples (noise counter: phase EVAL, step = noise_step), IEEE-accurate math.
//   loglik[c, g]     mean_s l(z_s)                      z_s = Z_loc + Z_std eps_s          (:159, :191)
//                    or log mean_s exp l(z_s)           z_s = prior mean + sigma eps_s     (:157, :189)   (margin)
//   kl[c, g]         KL(N(Z_loc, Z_std) || N(prior mean, sigma))                                          (:208)
//   prior_mean[c, g] Xc Wc + Wg Xg^T + intercept                                                          (:118-126)
struct TermsArgs {
  int64_t Nc, Ng, ld, event_offset;
  uint64_t seed;
  const float* c[3];   // explicit count tiles (the caller's count_layers), c[2] may be null
  const float* eff;
  const float* Xc; const float* Xg;
  const float* Zl; const float* Zs;
  const float* Wc; const float* b; const float* tau; const float* Wg;
  float* loglik; float* kl; float* prior_mean;   // any may be null
  int32_t M, m, S, KC, KG, cell_mode, margin, model_id;
  uint32_t noise_step;
};

__global__ void __launch_bounds__(256) element_terms_kernel(const TermsArgs a) {
  const int64_t total = a.Nc * a.ld;
  const int m = a.m;
  const bool eff = a.eff != nullptr;
  const uint32_t stream0 = brie_stream_word(BRIE_PHASE_EVAL, (uint32_t)a.model_id, 0u);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t row = i / a.ld, g = i % a.ld;
    float o_ll = 0.f, o_kl = 0.f, o_pm = 0.f;
    if (g < a.Ng) {
      const float tj = a.cell_mode ? a.tau[(int64_t)m * a.Nc + row] : a.tau[(int64_t)m * a.ld + g];
      const float pm =
          prior_mean(a, m, row, g, a.cell_mode ? a.b[(int64_t)m * a.Nc + row] : a.b[(int64_t)m * a.ld + g]);
      o_pm = pm;
      const float mu = a.Zl[(int64_t)m * a.Nc * a.ld + i], lam = a.Zs[(int64_t)m * a.Nc * a.ld + i];
      if (a.kl) o_kl = kl_normal(mu, lam, pm, tj);
      if (a.loglik) {
        const float c1 = a.c[0][i], c2 = a.c[1][i], c3 = a.c[2] ? a.c[2][i] : 0.f;
        const float n = c1 + c2 + c3;
        float L1, L2, L3;
        event_lengths(a.eff, a.ld, g, L1, L2, L3);
        const float zc = a.margin ? pm : mu, zs = expf(a.margin ? tj : lam);
        const float k0 = log_length_const(eff, c1, c2, c3, L1, L2, L3);
        float acc = 0.f;
        LogMeanExp lme;
        if (n > 0.f || a.margin) {
          for (int s0 = 0; s0 < a.S; s0 += 4) {
            float eps[4];
            brie_normals4((uint32_t)(a.event_offset + g), (uint32_t)row, a.noise_step, stream0 + (uint32_t)(s0 >> 2),
                          a.seed, eps);
            for (int q = 0; q < 4 && s0 + q < a.S; ++q) {
              const float l = sample_ll(fmaf(zs, eps[q], zc), c1, c2, n, L1, L2, L3, eff).l + k0;
              if (!a.margin) acc += l;
              else lme.add(l);
            }
          }
          o_ll = a.margin ? lme.value(a.S) : acc / (float)a.S;
        }
      }
    }
    if (a.loglik) a.loglik[i] = o_ll;
    if (a.kl) a.kl[i] = o_kl;
    if (a.prior_mean) a.prior_mean[i] = o_pm;
  }
}

// Multinomial resampling of observed read depth (brie/models/simulator.py:54-73): for every cell x event,
// (c1, c2, c3) ~ Multinomial(total[c, g], Phi), Phi ~ [psi L1, (1 - psi) L2, L3] (:54-62), as two conditional
// binomials.  Exact Bernoulli counting up to 4096 reads per element, normal approximation beyond.
__device__ inline int resample_binomial(uint32_t event, uint32_t cell, uint32_t stream, uint64_t seed, uint32_t& ctr,
                                        int n, float p) {
  if (n <= 0 || p <= 0.f) return 0;
  if (p >= 1.f) return n;
  uint32_t buf[4];
  if (n > 4096) {
    brie_philox4x32_10(event, cell, ctr++, stream, (uint32_t)seed, (uint32_t)(seed >> 32), buf);
    float za, zb;
    brie_box_muller(buf[0], buf[1], &za, &zb);
    return min(n, max(0, (int)rintf(n * p + sqrtf(n * p * (1.f - p)) * za)));
  }
  int k = 0;
  for (int i = 0; i < n; i += 4) {
    brie_philox4x32_10(event, cell, ctr++, stream, (uint32_t)seed, (uint32_t)(seed >> 32), buf);
    for (int j = 0; j < 4 && i + j < n; ++j) k += brie_u01(buf[j]) < p;
  }
  return k;
}

__global__ void __launch_bounds__(256) resample_counts_kernel(uint64_t seed, int64_t Nc, int64_t Ng, int64_t ld,
                                                              int64_t event_offset, const float* total,
                                                              const float* psi, const float* eff, float* c1,
                                                              float* c2, float* c3) {
  const int64_t n_el = Nc * ld;
  const uint32_t stream = brie_stream_word(3u /* BRIE_PHASE_SIM */, 1u, 0u);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_el; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t c = i / ld, g = i % ld;
    float o1 = 0.f, o2 = 0.f, o3 = 0.f;
    const int n = g < Ng ? (int)rintf(total[i]) : 0;
    if (n > 0) {
      float L1, L2, L3;
      event_lengths(eff, ld, g, L1, L2, L3);
      const float ps = psi[i];
      const float p1 = ps * L1, p2 = (1.f - ps) * L2, D = p1 + p2 + L3;
      uint32_t ctr = 0;
      const int k1 = resample_binomial((uint32_t)(event_offset + g), (uint32_t)c, stream, seed, ctr, n, p1 / D);
      const int k2 = (D - p1) > 0.f
                         ? resample_binomial((uint32_t)(event_offset + g), (uint32_t)c, stream, seed, ctr, n - k1, p2 / (D - p1))
                         : 0;
      o1 = (float)k1; o2 = (float)k2; o3 = (float)(n - k1 - k2);
    }
    c1[i] = o1; c2[i] = o2;
    if (c3) c3[i] = o3;
  }
}

// Psi = sigmoid(Z_loc); Psi95CI = sigmoid(Z_loc + z975 s) - sigmoid(Z_loc - z975 s)
// (tfd.LogitNormal(...).quantile, model_TFProb.py:92-106); Z_std = exp(Z_std_log).
__device__ __forceinline__ float sigmoid_acc(float z) {
  const float e = expf(-fabsf(z));
  const float inv = 1.0f / (1.0f + e);
  return z >= 0.f ? inv : e * inv;
}

__global__ void __launch_bounds__(256) posterior_kernel(const float* Zl, const float* Zs, int64_t n,
                                                        float* Psi, float* CI, float* Zstd) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x) {
    const float mu = Zl[i], s = expf(Zs[i]);
    if (Psi) Psi[i] = sigmoid_acc(mu);
    if (CI) CI[i] = sigmoid_acc(fmaf(kZ975, s, mu)) - sigmoid_acc(fmaf(-kZ975, s, mu));
    if (Zstd) Zstd[i] = s;
  }
}

// out[s, r, c] = normal s of counter (col_offset + c, row_offset + r, step, stream).
__global__ void __launch_bounds__(256) normals_kernel(uint64_t seed, uint32_t phase, uint32_t model,
                                                      uint32_t step, int n_samples, int64_t n_rows,
                                                      int64_t n_cols, int64_t col_offset,
                                                      int64_t row_offset, int64_t ld_out, float* out) {
  const int64_t total = n_rows * n_cols;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / n_cols, c = i % n_cols;
    for (int s0 = 0; s0 < n_samples; s0 += 4) {
      float e[4];
      brie_normals4((uint32_t)(col_offset + c), (uint32_t)(row_offset + r), step,
                    brie_stream_word(phase, model, (uint32_t)(s0 >> 2)), seed, e);
      for (int q = 0; q < 4 && s0 + q < n_samples; ++q)
        out[((int64_t)(s0 + q) * n_rows + r) * ld_out + c] = e[q];
    }
  }
}

__global__ void __launch_bounds__(256) fill_kernel(float* p, int64_t n, float v) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * blockDim.x)
    p[i] = v;
}

// Sum the per-event loss trace over reference batches (global event groups).
__global__ void __launch_bounds__(128) group_trace_kernel(const float* trace, int trace_cap,
                                                          int64_t ld, int64_t Ng,
                                                          int64_t event_offset, int64_t group_size,
                                                          int64_t first_group, int64_t n_groups,
                                                          int n_slots, double* out) {
  const int slot = blockIdx.x, m = blockIdx.y;
  const float* row = trace + ((int64_t)m * trace_cap + slot) * ld;
  for (int64_t grp = threadIdx.x; grp < n_groups; grp += blockDim.x) {
    const int64_t lo = max((first_group + grp) * group_size - event_offset, (int64_t)0);
    const int64_t hi = min((first_group + grp + 1) * group_size - event_offset, Ng);
    double s = 0.0;
    for (int64_t g = lo; g < hi; ++g) s += (double)row[g];
    out[((int64_t)m * n_groups + grp) * n_slots + slot] = s;
  }
}

// Synthetic count generator (bench workloads too large for host RAM; SURVEY f3).
// Generative recipe of brie/models/simulator.py:54-73 with psi = logistic(N(., .)) as in
// simulator/simuPSI.py:129-130: z = mean_g + Xc[c,:] Wc[:,g] + sd_g N(0,1), clipped to +-9
// (simulator.py:38-39); n ~ Poisson(lam_g) * Bernoulli(cdr_g); (c1,c2,c3) ~ Multinomial(n, phi),
// phi ~ [psi L1, (1-psi) L2, L3]; pseudo-count as model_wrap.py:113-117.
#define BRIE_PHASE_SIM 3u

struct SimRng {
  uint32_t event, cell, stream, ctr;
  uint64_t seed;
  uint32_t buf[4];
  int have;
  __device__ uint32_t next() {
    if (have == 0) {
      brie_philox4x32_10(event, cell, ctr++, stream, (uint32_t)seed, (uint32_t)(seed >> 32), buf);
      have = 4;
    }
    --have;   // selects, not a dynamic index: the words stay in registers (no local memory)
    return have == 3 ? buf[3] : (have == 2 ? buf[2] : (have == 1 ? buf[1] : buf[0]));
  }
  __device__ float uniform() { return brie_u01(next()); }
  __device__ float normal() {
    float a, b;
    const uint32_t x = next(), y = next();
    brie_box_muller(x, y, &a, &b);
    return a;
  }
};

__device__ inline int sim_poisson(SimRng& r, float lam) {
  if (lam <= 0.f) return 0;
  if (lam > 40.f) return max(0, (int)rintf(lam + sqrtf(lam) * r.normal()));   // normal approximation in the tail
  const float limit = expf(-lam);                                            // Knuth's product method
  int k = 0;
  float p = r.uniform();
  while (p > limit && k < 400) { ++k; p *= r.uniform(); }
  return k;
}

__device__ inline int sim_binomial(SimRng& r, int n, float p) {
  if (n <= 0 || p <= 0.f) return 0;
  if (p >= 1.f) return n;
  if (n > 96) {
    const float mu = n * p, sd = sqrtf(n * p * (1.f - p));
    return min(n, max(0, (int)rintf(mu + sd * r.normal())));
  }
  int k = 0;
  for (int i = 0; i < n; ++i) k += r.uniform() < p;
  return k;
}

__global__ void __launch_bounds__(256) simulate_counts_kernel(uint64_t seed, int64_t Nc, int64_t Ng, int64_t ld,
                                                              int64_t event_offset, const float* mean,
                                                              const float* sd, const float* Xc, const float* Wc,
                                                              int Kc, const float* eff, const float* lam,
                                                              const float* cdr, float pseudo, float* c1,
                                                              float* c2, float* c3) {
  const int64_t total = Nc * ld;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t c = i / ld, g = i % ld;
    float o1 = 0.f, o2 = 0.f, o3 = 0.f;
    if (g < Ng) {
      SimRng r;
      r.event = (uint32_t)(event_offset + g); r.cell = (uint32_t)c; r.stream = brie_stream_word(BRIE_PHASE_SIM, 0u, 0u);
      r.ctr = 0; r.seed = seed; r.have = 0;
      const int n = (r.uniform() < cdr[g]) ? sim_poisson(r, lam[g]) : 0;
      if (n > 0) {
        float z = mean[g] + sd[g] * r.normal();
        for (int k = 0; k < Kc; ++k) z = fmaf(Xc[c * Kc + k], Wc[(int64_t)k * ld + g], z);
        z = fminf(fmaxf(z, -9.f), 9.f);
        const float psi = 1.f / (1.f + expf(-z));
        float L1, L2, L3;
        event_lengths(eff, ld, g, L1, L2, L3);
        const float p1 = psi * L1, p2 = (1.f - psi) * L2, D = p1 + p2 + L3;
        const int k1 = sim_binomial(r, n, p1 / D);
        const int k2 = sim_binomial(r, n - k1, p2 / (D - p1));
        o1 = (float)k1; o2 = (float)k2; o3 = (float)(n - k1 - k2);
        if (k1 + k2 > 0) { o1 += pseudo; o2 += pseudo; }
      }
    }
    c1[i] = o1; c2[i] = o2;
    if (c3) c3[i] = o3;
  }
}

}  // namespace brie
