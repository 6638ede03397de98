// Host side of the brie_b200 C ABI (include/brie_b200.h): argument checking,
// launch geometry, kernel dispatch.  No persistent device allocations.
#include <cublas_v2.h>
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <string>
#include <vector>

#include "../../include/brie_b200.h"
#include "brie_kernels.cuh"
#include "brie_margin.cuh"
#include "brie_wald.cuh"

#include "brie_host.h"

namespace {
thread_local std::string g_err;
}

struct brie_comm;
namespace brie {
int comm_allreduce_sum_f32(brie_comm* c, float* buf, int64_t n, cudaStream_t s);   // brie_comm.cu

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}
}  // namespace brie

struct brie_fit {
  brie_fit_desc d;
  brie_fit_sizes sz;
  brie_fit_buffers buf;
  bool bound = false;
  bool subfit = false;       // bound as a gathered sub-fit (event_ids or a per-model count / length stride)
  int nev_max = 0, ncell = 0;
  size_t off_part_ev = 0, off_part_cell = 0, off_G = 0;  // scratch carve-up (float offsets)
  size_t off_mom_cell = 0;   // adam_small: per-event moments (2, M, Kc + 2, ld) first, per-cell (2, M, Nc, Kg + 2) here
  bool stage_open = false;   // begin_stage has set the learning rate and cleared the Adam moments
  float lr = 0.f;
  int64_t t = 0;             // Adam step within the current stage
  uint32_t global_step = 0;  // RNG step word: counts every optimisation step of the fit
  float alpha = 0.f;
  int64_t launches = 0;
  bool step_open = false;    // phase 0 done, phase 1 pending
  // optional CUDA-event timing of the fused step kernel (bench.py roofline)
  std::vector<cudaEvent_t> ev0, ev1;
  int ev_used = 0;
  // column compaction of the step kernel (brie_fit_set_active_blocks); null = all columns
  const int32_t* blk_ids = nullptr;
  int64_t blk_stride = 0;
  int32_t n_blk[BRIE_MAX_MODELS] = {0};
  int blk_tiles = 0;
  brie_comm* comm = nullptr;   // event-sharded fit with shared per-cell parameters: G is all-reduced every step
  // wide designs (Kc > BRIE_MAX_KC or Kg > BRIE_MAX_KG): covariate contractions as GEMMs around the fused kernel
  bool wide = false;
  size_t off_PM = 0, off_R = 0, off_gWc = 0;   // (M, Nc, ld), (M, Nc, ld), (M, Kc, ld) in scratch
  cublasHandle_t blas = nullptr;
  // counts as packed dictionary codes (brie_fit_set_count_codes); null = the float32 tiles
  const uint32_t* codes = nullptr;
  int64_t code_mstride = 0;
  const float* code_dict = nullptr;
};

using namespace brie;

namespace {

constexpr int kMaxDevices = 64;

bool kc_supported(int k) { return k == 0 || k == 1 || k == 2 || k == 4 || k == 8 || k == 16; }
bool kg_supported(int k) { return k == 0 || k == 4 || k == 8; }

// Opt Kernel in to `bytes` of dynamic shared memory (needed above 48 KB) once per device: the attribute is per device.
template <auto* Kernel>
cudaError_t opt_in_smem(int bytes) {
  static bool configured[kMaxDevices] = {false};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const bool known = dev >= 0 && dev < kMaxDevices;
  if (known && configured[dev]) return cudaSuccess;
  e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess && known) configured[dev] = true;
  return e;
}

template <int KC, int KG, bool CELL, bool LOSS, bool EXT, bool CODE8>
cudaError_t launch_step(const StepArgs& a, dim3 grid, cudaStream_t s) {
  constexpr int smem = step_smem_bytes(KC, KG, CELL, LOSS, EXT, CODE8);
  cudaError_t e = opt_in_smem<elbo_step_kernel<KC, KG, CELL, LOSS, EXT, CODE8>>(smem);
  if (e != cudaSuccess) return e;
  elbo_step_kernel<KC, KG, CELL, LOSS, EXT, CODE8><<<grid, kThreads, smem, s>>>(a);
  return cudaGetLastError();
}

// the count form (f32 tiles or packed codes) is the innermost choice
template <int KC, int KG, bool CELL, bool LOSS, bool EXT>
cudaError_t launch_step_fmt(const StepArgs& a, dim3 grid, cudaStream_t s) {
  return a.codes ? launch_step<KC, KG, CELL, LOSS, EXT, true>(a, grid, s) : launch_step<KC, KG, CELL, LOSS, EXT, false>(a, grid, s);
}

const char* blas_status(cublasStatus_t st) {
  switch (st) {
    case CUBLAS_STATUS_SUCCESS: return "success";
    case CUBLAS_STATUS_NOT_INITIALIZED: return "not initialized";
    case CUBLAS_STATUS_ALLOC_FAILED: return "allocation failed";
    case CUBLAS_STATUS_INVALID_VALUE: return "invalid value";
    case CUBLAS_STATUS_ARCH_MISMATCH: return "arch mismatch";
    case CUBLAS_STATUS_EXECUTION_FAILED: return "execution failed";
    case CUBLAS_STATUS_INTERNAL_ERROR: return "internal error";
    case CUBLAS_STATUS_NOT_SUPPORTED: return "not supported";
    default: return "unknown";
  }
}
#define BRIE_BLAS(call)                                                                               \
  do {                                                                                                \
    cublasStatus_t st_ = (call);                                                                      \
    if (st_ != CUBLAS_STATUS_SUCCESS)                                                                 \
      return brie::fail(BRIE_ERR_CUDA, "%s failed: cuBLAS %s (%s:%d)", #call, blas_status(st_), __FILE__, __LINE__); \
  } while (0)

// Wide form, before the fused kernel: PM[m] (Nc x ld, row-major) = Xc[m] (Nc x Kc) Wc[m] (Kc x ld) + Wg[m] (Nc x Kg) Xg^T
// (Z_prior, model_TFProb.py:121-125).  Row-major arrays are handed to cuBLAS as their column-major transposes.
int wide_prior_mean(brie_fit* f, cudaStream_t s) {
  const brie_fit_desc& d = f->d;
  float* scratch = (float*)f->buf.scratch;
  const float one = 1.f, zero = 0.f;
  BRIE_BLAS(cublasSetStream(f->blas, s));
  const int64_t plane = d.n_cells * d.ld;
  for (int m = 0; m < d.n_models; ++m) {
    float* PM = scratch + f->off_PM + (size_t)m * plane;
    if (d.Kc > 0)
      BRIE_BLAS(cublasSgemm(f->blas, CUBLAS_OP_N, CUBLAS_OP_N, (int)d.ld, (int)d.n_cells, d.Kc, &one,
                            f->buf.Wc + (size_t)m * d.Kc * d.ld, (int)d.ld,
                            f->buf.Xc + (size_t)m * d.n_cells * d.Kc, d.Kc, &zero, PM, (int)d.ld));
    else
      BRIE_CUDA(cudaMemsetAsync(PM, 0, (size_t)plane * sizeof(float), s));
    if (d.Kg > 0)
      BRIE_BLAS(cublasSgemm(f->blas, CUBLAS_OP_T, CUBLAS_OP_N, (int)d.n_events, (int)d.n_cells, d.Kg, &one,
                            f->buf.Xg, d.Kg, f->buf.Wg + (size_t)m * d.n_cells * d.Kg, d.Kg, &one, PM, (int)d.ld));
  }
  f->launches += d.n_models * ((d.Kc > 0) + (d.Kg > 0));
  return BRIE_OK;
}

// Wide form, after the fused kernel: d loss / d Wc[m] = -Xc[m]^T R[m] (Kc x ld) and d loss / d Wg[m] = -R[m] Xg (Nc x Kg),
// the latter written into the per-cell gradient buffer G (M, Nc, Kg + 2 * cell_mode) the all-reduce and the per-cell
// Adam update read (SURVEY A.3).
int wide_gradients(brie_fit* f, cudaStream_t s) {
  const brie_fit_desc& d = f->d;
  float* scratch = (float*)f->buf.scratch;
  const float minus = -1.f, zero = 0.f;
  BRIE_BLAS(cublasSetStream(f->blas, s));
  const int64_t plane = d.n_cells * d.ld;
  for (int m = 0; m < d.n_models; ++m) {
    const float* R = scratch + f->off_R + (size_t)m * plane;
    if (d.Kc > 0)
      BRIE_BLAS(cublasSgemm(f->blas, CUBLAS_OP_N, CUBLAS_OP_T, (int)d.ld, d.Kc, (int)d.n_cells, &minus, R, (int)d.ld,
                            f->buf.Xc + (size_t)m * d.n_cells * d.Kc, d.Kc, &zero,
                            scratch + f->off_gWc + (size_t)m * d.Kc * d.ld, (int)d.ld));
    if (d.Kg > 0)
      BRIE_BLAS(cublasSgemm(f->blas, CUBLAS_OP_N, CUBLAS_OP_N, d.Kg, (int)d.n_cells, (int)d.n_events, &minus, f->buf.Xg,
                            d.Kg, R, (int)d.ld, &zero, scratch + f->off_G + (size_t)m * d.n_cells * f->ncell, f->ncell));
  }
  f->launches += d.n_models * ((d.Kc > 0) + (d.Kg > 0));
  return BRIE_OK;
}

// EXT: the wide form, whose kernels contract no covariates themselves (KC = KG = 0)
template <int KC, int KG, bool EXT = false>
cudaError_t dispatch_step2(const StepArgs& a, bool cell, bool loss, dim3 grid, cudaStream_t s) {
  if (cell)
    return loss ? launch_step_fmt<KC, KG, true, true, EXT>(a, grid, s) : launch_step_fmt<KC, KG, true, false, EXT>(a, grid, s);
  return loss ? launch_step_fmt<KC, KG, false, true, EXT>(a, grid, s) : launch_step_fmt<KC, KG, false, false, EXT>(a, grid, s);
}

template <int KC>
cudaError_t dispatch_step1(const StepArgs& a, int KG, bool cell, bool loss, dim3 grid, cudaStream_t s) {
  switch (KG) {
    case 0: return dispatch_step2<KC, 0>(a, cell, loss, grid, s);
    case 4: return dispatch_step2<KC, 4>(a, cell, loss, grid, s);
    case 8: return dispatch_step2<KC, 8>(a, cell, loss, grid, s);
  }
  return cudaErrorInvalidValue;
}

cudaError_t dispatch_step(const StepArgs& a, bool wide, int KC, int KG, bool cell, bool loss, dim3 grid,
                          cudaStream_t s) {
  if (wide) return dispatch_step2<0, 0, true>(a, cell, loss, grid, s);
  switch (KC) {
    case 0: return dispatch_step1<0>(a, KG, cell, loss, grid, s);
    case 1: return dispatch_step1<1>(a, KG, cell, loss, grid, s);
    case 2: return dispatch_step1<2>(a, KG, cell, loss, grid, s);
    case 4: return dispatch_step1<4>(a, KG, cell, loss, grid, s);
    case 8: return dispatch_step1<8>(a, KG, cell, loss, grid, s);
    case 16: return dispatch_step1<16>(a, KG, cell, loss, grid, s);   // 2 events per lane, 64-event tiles
  }
  return cudaErrorInvalidValue;
}

// bit m set iff model m still has an active event.  In shared-parameter fits
// (cell_mode or Kg > 0) the caller deactivates whole models; for per-event fits
// the kernels consult `active` per event and this mask stays all-ones.
uint32_t g_all_models(const brie_fit* f) {
  return f->d.n_models >= 32 ? 0xffffffffu : ((1u << f->d.n_models) - 1u);
}

// The fields that StepArgs, MarginArgs, EvalArgs and TermsArgs share under the same names; the rest are zero.
template <class A>
A fit_args(const brie_fit* f) {
  const brie_fit_desc& d = f->d;
  const brie_fit_buffers& b = f->buf;
  A a;
  memset(&a, 0, sizeof a);
  a.Nc = d.n_cells; a.Ng = d.n_events; a.ld = d.ld; a.event_offset = d.event_offset; a.seed = d.seed;
  a.c[0] = b.counts[0]; a.c[1] = b.counts[1]; a.c[2] = b.counts[2];
  a.eff = b.efflen3; a.Xc = b.Xc; a.Xg = b.Xg;
  a.Wc = b.Wc; a.b = b.intercept; a.tau = b.sigma_log; a.Wg = b.Wg;
  a.M = d.n_models;
  return a;
}

// Arguments of both per-cell kernels; n_tiles: the column tiles of per-cell partials that cell_reduce_kernel sums.
CellArgs cell_args(const brie_fit* f, int n_tiles) {
  const brie_fit_desc& d = f->d;
  float* scratch = (float*)f->buf.scratch;
  CellArgs c;
  memset(&c, 0, sizeof c);
  c.Nc = d.n_cells; c.M = d.n_models; c.KG = d.Kg; c.NCELL = f->ncell; c.n_tiles = n_tiles;
  c.cell_mode = d.cell_mode; c.train_b = d.train_intercept; c.train_tau = d.train_sigma;
  c.model_mask = g_all_models(f); c.alpha = f->alpha;
  c.part_cell = scratch + f->off_part_cell; c.G = scratch + f->off_G;
  c.Wg = f->buf.Wg; c.b = f->buf.intercept; c.tau = f->buf.sigma_log;
  c.mom = f->buf.adam_small + f->off_mom_cell;
  c.n_part = f->wide ? (d.cell_mode ? 2 : 0) : f->ncell;   // wide: d/dWg is already in G (wide_gradients)
  c.part_off = f->wide ? d.Kg : 0;
  return c;
}

// The launchers of one step, in stream order (brie_fit_step_phase).  Each launches only if its kernel has work.
// target marginLik: the prior-sampled objective reads counts only, no per-element state (brie_margin.cuh)
int launch_margin_step(brie_fit* f, int nev, int cell_tiles, cudaStream_t s) {
  const brie_fit_desc& d = f->d;
  float* scratch = (float*)f->buf.scratch;
  MarginArgs g = fit_args<MarginArgs>(f);
  g.active = f->buf.active;
  g.part_ev = scratch + f->off_part_ev; g.part_cell = scratch + f->off_part_cell;
  g.step = f->global_step; g.model_mask = g_all_models(f);
  g.S = d.mc_size; g.rows_per_cta = f->sz.rows_per_cta;
  g.KC = d.Kc; g.KG = d.Kg; g.cell_mode = d.cell_mode; g.NEV = nev; g.NCELL = f->ncell;
  for (int m = 0; m < d.n_models; ++m) g.model_id[m] = d.model_id[m];
  // the opt-in covers the widest per-event partials (Kc = BRIE_MAX_KC); the launch asks for this fit's
  BRIE_CUDA(opt_in_smem<margin_step_kernel>(kWarps * (BRIE_MAX_KC + 3) * kMarginTile * (int)sizeof(float)));
  const size_t smem = (size_t)kWarps * nev * kMarginTile * sizeof(float);
  margin_step_kernel<<<dim3(d.n_models, cell_tiles, f->sz.n_row_chunks), kThreads, smem, s>>>(g);
  BRIE_CUDA(cudaGetLastError());
  f->launches += 1;
  return BRIE_OK;
}

// target ELBO: the fused step kernel, between the wide form's prior-mean and gradient GEMMs.  The timing events
// (brie_fit_kernel_timing) bracket the fused kernel alone.
int launch_fused_step(brie_fit* f, bool loss, cudaStream_t s) {
  const brie_fit_desc& d = f->d;
  float* scratch = (float*)f->buf.scratch;
  StepArgs a = fit_args<StepArgs>(f);
  a.Zl = f->buf.Z_loc; a.Zs = f->buf.Z_std_log; a.aZ = f->buf.adam_Z;
  a.active = f->buf.active;
  a.part_ev = scratch + f->off_part_ev; a.part_cell = scratch + f->off_part_cell;
  a.alpha = f->alpha; a.inv_S = 1.0f / (float)d.mc_size;
  a.step = f->global_step; a.model_mask = g_all_models(f);
  a.S = d.mc_size; a.rows_per_cta = f->sz.rows_per_cta;
  for (int m = 0; m < d.n_models; ++m) a.model_id[m] = d.model_id[m];
  a.ev_ids = f->buf.event_ids; a.c_mstride = f->buf.counts_model_stride; a.eff_mstride = f->buf.efflen_model_stride;
  a.codes = f->codes; a.code_mstride = f->code_mstride; a.dict = f->code_dict;
  dim3 grid(d.n_models, f->sz.n_col_tiles, f->sz.n_row_chunks);
  if (f->blk_ids) {
    a.blk_ids = f->blk_ids; a.blk_stride = f->blk_stride;
    for (int m = 0; m < d.n_models; ++m) a.n_blk[m] = f->n_blk[m];
    grid.y = (unsigned)(f->blk_tiles > 0 ? f->blk_tiles : 1);
  }
  if (f->wide) {
    a.PM = scratch + f->off_PM; a.R = scratch + f->off_R;
    int rc = wide_prior_mean(f, s);
    if (rc) return rc;
  }
  const bool timed = f->ev_used < (int)f->ev0.size();
  if (timed) BRIE_CUDA(cudaEventRecord(f->ev0[f->ev_used], s));
  BRIE_CUDA(dispatch_step(a, f->wide, d.Kc, d.Kg, d.cell_mode != 0, loss, grid, s));
  if (timed) BRIE_CUDA(cudaEventRecord(f->ev1[f->ev_used++], s));
  f->launches += 1;
  return f->wide ? wide_gradients(f, s) : BRIE_OK;
}

// Per-event reduce of the row-chunk partials (nev rows, the loss last if loss_row), Adam on Wc and the per-event
// intercept / sigma_log, and the loss trace if trace_slot >= 0.  The wide form's d/dWc comes from wide_gradients.
int launch_event_update(brie_fit* f, int nev, bool loss_row, int32_t trace_slot, cudaStream_t s) {
  const brie_fit_desc& d = f->d;
  if (nev == 0 && !(f->wide && d.Kc > 0)) return BRIE_OK;
  float* scratch = (float*)f->buf.scratch;
  const int kc_kernel = f->wide ? 0 : d.Kc;
  EventArgs e;
  memset(&e, 0, sizeof e);
  e.ld = d.ld; e.Ng = d.n_events; e.M = d.n_models; e.KC = d.Kc; e.NEV = nev; e.n_chunks = f->sz.n_row_chunks;
  e.idx_gb = d.cell_mode ? -1 : kc_kernel; e.idx_gt = d.cell_mode ? -1 : kc_kernel + 1;
  e.idx_loss = loss_row ? kc_kernel + (d.cell_mode ? 0 : 2) : -1;
  e.wc_grad = f->wide ? scratch + f->off_gWc : nullptr;
  e.train_b = d.train_intercept; e.train_tau = d.train_sigma;
  e.trace_slot = trace_slot; e.trace_cap = d.trace_cap;
  e.alpha = f->alpha; e.part_ev = scratch + f->off_part_ev;
  e.Wc = f->buf.Wc; e.b = f->buf.intercept; e.tau = f->buf.sigma_log;
  e.mom = f->buf.adam_small; e.active = f->buf.active; e.trace = f->buf.loss_trace;
  for (int m = 0; m < d.n_models; ++m) { e.xc_mask[m] = d.xc_mask[m]; e.xc_width[m] = d.xc_width[m]; }
  event_update_kernel<<<dim3((unsigned)ceil_div(d.n_events, 32), d.n_models), 256, 0, s>>>(e);
  BRIE_CUDA(cudaGetLastError());
  f->launches += 1;
  return BRIE_OK;
}

// Per-cell sum of the column-tile partials into G, which the all-reduce and launch_cell_update read.
int launch_cell_reduce(brie_fit* f, int cell_tiles, cudaStream_t s) {
  const CellArgs c = cell_args(f, cell_tiles);
  if (c.n_part == 0) return BRIE_OK;
  cell_reduce_kernel<<<dim3((unsigned)ceil_div(f->d.n_cells * c.n_part, 256), f->d.n_models), 256, 0, s>>>(c);
  BRIE_CUDA(cudaGetLastError());
  f->launches += 1;
  return BRIE_OK;
}

// Adam on Wg and the per-cell intercept / sigma_log from G.
int launch_cell_update(brie_fit* f, cudaStream_t s) {
  if (f->ncell == 0) return BRIE_OK;
  cell_update_kernel<<<dim3((unsigned)ceil_div(f->d.n_cells, 256), f->d.n_models), 256, 0, s>>>(
      cell_args(f, f->sz.n_col_tiles));
  BRIE_CUDA(cudaGetLastError());
  f->launches += 1;
  return BRIE_OK;
}

}  // namespace

extern "C" {

int brie_abi_version(void) { return BRIE_ABI_VERSION; }

const char* brie_last_error(void) { return g_err.c_str(); }

int brie_fit_create(const brie_fit_desc* desc, brie_fit** out) {
  if (!desc || !out) return fail(BRIE_ERR_ARG, "null argument");
  const brie_fit_desc& d = *desc;
  if (d.n_cells <= 0 || d.n_events <= 0) return fail(BRIE_ERR_ARG, "n_cells and n_events must be positive");
  if (d.ld < d.n_events || d.ld % 4 != 0)
    return fail(BRIE_ERR_ARG, "ld must be a multiple of 4 and >= n_events");
  if (d.n_cells >= ((int64_t)1 << 32) || d.event_offset < 0 || d.event_offset + d.ld >= ((int64_t)1 << 32))
    return fail(BRIE_ERR_ARG, "cell / event index exceeds the 32-bit RNG counter words");
  if (d.n_models < 1 || d.n_models > BRIE_MAX_MODELS) return fail(BRIE_ERR_ARG, "n_models out of range");
  if (d.Kc < 0 || d.Kg < 0 || d.Kc > BRIE_MAX_K_WIDE || d.Kg > BRIE_MAX_K_WIDE)
    return fail(BRIE_ERR_ARG, "Kc and Kg must be in [0, %d]", BRIE_MAX_K_WIDE);
  const bool wide = d.Kc > BRIE_MAX_KC || d.Kg > BRIE_MAX_KG;
  if (!wide && !kc_supported(d.Kc))
    return fail(BRIE_ERR_UNSUPPORTED, "Kc must be one of 0,1,2,4,8,16 (pad Xc with zero columns) or above 16 (wide form)");
  if (!wide && !kg_supported(d.Kg))
    return fail(BRIE_ERR_UNSUPPORTED, "Kg must be one of 0,4,8 (pad Xg with zero columns) or above 8 (wide form)");
  if (wide && d.target != BRIE_TARGET_ELBO)
    return fail(BRIE_ERR_UNSUPPORTED, "target marginLik is limited to Kc <= %d and Kg <= %d", BRIE_MAX_KC, BRIE_MAX_KG);
  if (d.mc_size < 1 || d.mc_size > 4096) return fail(BRIE_ERR_ARG, "mc_size out of range");
  if (d.n_layers != 2 && d.n_layers != 3) return fail(BRIE_ERR_ARG, "n_layers must be 2 or 3");
  if (d.trace_cap < 0) return fail(BRIE_ERR_ARG, "trace_cap must be >= 0");
  if (d.rows_per_cta < 0 || d.rows_per_cta > 65536) return fail(BRIE_ERR_ARG, "rows_per_cta out of range");
  if (d.target != BRIE_TARGET_ELBO && d.target != BRIE_TARGET_MARGINLIK)
    return fail(BRIE_ERR_ARG, "target must be BRIE_TARGET_ELBO or BRIE_TARGET_MARGINLIK");
  for (int m = 0; m < d.n_models; ++m) {
    if (d.model_id[m] < 0 || d.model_id[m] >= 4096) return fail(BRIE_ERR_ARG, "model_id must be in [0, 4096)");
    if (!wide && (d.xc_mask[m] >> d.Kc) != 0) return fail(BRIE_ERR_ARG, "xc_mask has bits beyond Kc");
    if (wide && (d.xc_width[m] < 0 || d.xc_width[m] > d.Kc)) return fail(BRIE_ERR_ARG, "xc_width out of range");
  }
  brie_fit* f = new (std::nothrow) brie_fit();
  if (!f) return fail(BRIE_ERR_ARG, "out of host memory");
  f->d = d;
  f->wide = wide;
  memset(&f->buf, 0, sizeof f->buf);
  const int n_tiles = (int)ceil_div(d.ld, step_tile_cols(wide ? 0 : d.Kc, wide ? 0 : d.Kg));   // 128 events per tile, 64 when Kc = 16
  // rows per CTA: up to 256 (fewer row-chunk partials for event_update_kernel) while keeping
  // >= ~10 waves of 2 CTAs/SM (tail effect); small problems go down to one row per warp
  int rows = 256;
  const char* env = getenv("BRIE_ROWS_PER_CTA");
  if (d.rows_per_cta > 0) {
    rows = d.rows_per_cta;
  } else if (env && atoi(env) > 0) {
    rows = atoi(env);
  } else {
    const int64_t target = 148 * 2 * 10;
    while (rows > 8 && (int64_t)d.n_models * n_tiles * ceil_div(d.n_cells, rows) < target) rows >>= 1;
  }
  // the step kernel addresses a CTA's elements with 32-bit offsets (local row) * ld + column
  while (d.rows_per_cta == 0 && rows > 8 && (int64_t)rows * d.ld >= ((int64_t)1 << 31)) rows >>= 1;
  if ((int64_t)rows * d.ld >= ((int64_t)1 << 31)) {
    delete f;
    return fail(BRIE_ERR_UNSUPPORTED, "rows_per_cta * ld = %lld exceeds the 31-bit element offset of a CTA",
                (long long)rows * (long long)d.ld);
  }
  const int64_t n_chunks = ceil_div(d.n_cells, rows);
  if (n_chunks > 65535 || n_tiles > 65535) {
    delete f;
    return fail(BRIE_ERR_UNSUPPORTED, "grid too large (%lld row chunks, %d column tiles)", (long long)n_chunks,
                n_tiles);
  }
  f->nev_max = (wide ? 0 : d.Kc) + 2 + 1;
  f->ncell = d.Kg + (d.cell_mode ? 2 : 0);
  const int ncell_part = wide ? (d.cell_mode ? 2 : 0) : f->ncell;   // what the fused kernel leaves per cell and tile
  f->sz.rows_per_cta = rows;
  f->sz.n_row_chunks = (int)n_chunks;
  f->sz.n_col_tiles = n_tiles;
  f->sz.reserved = 0;
  size_t off = 0;
  f->off_part_ev = off;
  off += (size_t)n_chunks * d.n_models * f->nev_max * d.ld;
  f->off_part_cell = off;
  off += (size_t)n_tiles * d.n_models * d.n_cells * ncell_part;
  f->off_G = off;
  off += (size_t)d.n_models * d.n_cells * f->ncell;
  off = (off + 3) / 4 * 4;                     // 16-byte alignment of what follows
  if (wide) {
    f->off_PM = off;
    off += (size_t)d.n_models * d.n_cells * d.ld;
    f->off_R = off;
    off += (size_t)d.n_models * d.n_cells * d.ld;
    f->off_gWc = off;
    off += (size_t)d.n_models * (d.Kc > 0 ? d.Kc : 1) * d.ld;
  }
  f->sz.scratch_bytes = (off + 4) * sizeof(float);
  f->off_mom_cell = (size_t)2 * d.n_models * (d.Kc + 2) * d.ld;
  f->sz.adam_small_floats = f->off_mom_cell + (size_t)2 * d.n_models * d.n_cells * (d.Kg + 2);
  *out = f;
  return BRIE_OK;
}

int brie_fit_destroy(brie_fit* fit) {
  if (fit && fit->blas) cublasDestroy(fit->blas);
  if (fit) {
    for (cudaEvent_t e : fit->ev0) cudaEventDestroy(e);
    for (cudaEvent_t e : fit->ev1) cudaEventDestroy(e);
  }
  delete fit;
  return BRIE_OK;
}

int brie_fit_kernel_timing(brie_fit* f, int32_t capacity) {
  if (!f || capacity < 0) return fail(BRIE_ERR_ARG, "bad argument");
  for (cudaEvent_t e : f->ev0) cudaEventDestroy(e);
  for (cudaEvent_t e : f->ev1) cudaEventDestroy(e);
  f->ev0.assign(capacity, nullptr);
  f->ev1.assign(capacity, nullptr);
  f->ev_used = 0;
  for (int i = 0; i < capacity; ++i) {
    BRIE_CUDA(cudaEventCreate(&f->ev0[i]));
    BRIE_CUDA(cudaEventCreate(&f->ev1[i]));
  }
  return BRIE_OK;
}

int brie_fit_kernel_time_ms(brie_fit* f, double* total_ms, int32_t* n_launches) {
  if (!f || !total_ms || !n_launches) return fail(BRIE_ERR_ARG, "null argument");
  double sum = 0.0;
  for (int i = 0; i < f->ev_used; ++i) {
    BRIE_CUDA(cudaEventSynchronize(f->ev1[i]));
    float ms = 0.f;
    BRIE_CUDA(cudaEventElapsedTime(&ms, f->ev0[i], f->ev1[i]));
    sum += ms;
  }
  *total_ms = sum;
  *n_launches = f->ev_used;
  f->ev_used = 0;
  return BRIE_OK;
}

int brie_fit_get_sizes(const brie_fit* fit, brie_fit_sizes* out) {
  if (!fit || !out) return fail(BRIE_ERR_ARG, "null argument");
  *out = fit->sz;
  return BRIE_OK;
}

int brie_fit_bind(brie_fit* fit, const brie_fit_buffers* b) {
  if (!fit || !b) return fail(BRIE_ERR_ARG, "null argument");
  const brie_fit_desc& d = fit->d;
  const bool subfit = b->event_ids || b->counts_model_stride != 0 || b->efflen_model_stride != 0;
  // a gathered sub-fit may step on packed codes alone (brie_fit_set_count_codes) and bind no count tiles
  const bool no_counts = subfit && !b->counts[0] && !b->counts[1] && !b->counts[2];
  if (!no_counts && (!b->counts[0] || !b->counts[1])) return fail(BRIE_ERR_ARG, "counts[0], counts[1] required");
  if (!no_counts && (d.n_layers == 3) != (b->counts[2] != nullptr))
    return fail(BRIE_ERR_ARG, "counts[2] must be given iff n_layers == 3");
  if ((d.has_efflen != 0) != (b->efflen3 != nullptr))
    return fail(BRIE_ERR_ARG, "efflen3 must be given iff has_efflen");
  if (d.Kc > 0 && (!b->Xc || !b->Wc)) return fail(BRIE_ERR_ARG, "Xc and Wc required when Kc > 0");
  if (d.Kg > 0 && (!b->Xg || !b->Wg)) return fail(BRIE_ERR_ARG, "Xg and Wg required when Kg > 0");
  if (!b->Z_loc || !b->Z_std_log || !b->adam_Z || !b->intercept || !b->sigma_log || !b->adam_small ||
      !b->active || !b->scratch)
    return fail(BRIE_ERR_ARG, "missing state buffer");
  if (d.trace_cap > 0 && !b->loss_trace) return fail(BRIE_ERR_ARG, "loss_trace required when trace_cap > 0");
  const void* aligned[] = {b->counts[0], b->counts[1], b->counts[2], b->efflen3, b->Z_loc, b->Z_std_log,
                           b->adam_Z,    b->Wc,        b->intercept, b->sigma_log, b->active, b->scratch};
  for (const void* p : aligned)
    if (((uintptr_t)p & 15u) != 0) return fail(BRIE_ERR_ARG, "device buffers must be 16-byte aligned");
  if (subfit) {
    if (fit->ncell > 0 || d.target != BRIE_TARGET_ELBO)
      return fail(BRIE_ERR_UNSUPPORTED, "a gathered sub-fit needs per-event parameters only (Kg = 0, gene intercept) and target ELBO");
    if (b->counts_model_stride < 0 || b->counts_model_stride % 4 != 0 || b->efflen_model_stride < 0)
      return fail(BRIE_ERR_ARG, "model strides must be >= 0 (counts: a multiple of 4 floats)");
    if (fit->wide) return fail(BRIE_ERR_UNSUPPORTED, "gathered sub-fits are limited to Kc <= %d", BRIE_MAX_KC);
  }
  fit->buf = *b;
  fit->subfit = subfit;
  fit->bound = true;
  if (fit->wide) {   // residuals of never-active (padding) columns must be finite for the gradient GEMMs
    float* scratch = (float*)b->scratch;
    const size_t plane = (size_t)d.n_models * d.n_cells * d.ld;
    BRIE_CUDA(cudaMemset(scratch + fit->off_PM, 0, plane * sizeof(float)));
    BRIE_CUDA(cudaMemset(scratch + fit->off_R, 0, plane * sizeof(float)));
    if (!fit->blas) {
      cublasStatus_t st = cublasCreate(&fit->blas);
      if (st != CUBLAS_STATUS_SUCCESS) return fail(BRIE_ERR_CUDA, "cublasCreate failed: %s", blas_status(st));
      // fp32 in, fp32 accumulate: the default math mode never down-converts to TF32 on its own, and these skinny
      // (K x Nc x Ng) products want cuBLAS's split-K heuristics (pedantic mode ran them 2-3x slower)
      cublasSetMathMode(fit->blas, CUBLAS_DEFAULT_MATH);
    }
  }
  return BRIE_OK;
}

int brie_fit_init_params(brie_fit* f, float intercept_const, float sigma_const, void* stream) {
  if (!f || !f->bound) return fail(BRIE_ERR_ARG, "fit not bound");
  if (!(sigma_const > 0.f)) return fail(BRIE_ERR_ARG, "sigma must be positive");
  cudaStream_t s = (cudaStream_t)stream;
  const brie_fit_desc& d = f->d;
  const int64_t plane = d.n_cells * d.ld;
  const int64_t nsmall = d.cell_mode ? d.n_cells : d.ld;
  for (int m = 0; m < d.n_models; ++m) {
    const uint32_t mid = (uint32_t)d.model_id[m];
    normals_kernel<<<grid_1d(plane, 256), 256, 0, s>>>(d.seed, BRIE_PHASE_INIT, mid, BRIE_INIT_Z_LOC, 1,
                                                      d.n_cells, d.ld, d.event_offset, 0, d.ld,
                                                      f->buf.Z_loc + m * plane);
    normals_kernel<<<grid_1d(plane, 256), 256, 0, s>>>(d.seed, BRIE_PHASE_INIT, mid, BRIE_INIT_Z_STD_LOG, 1,
                                                      d.n_cells, d.ld, d.event_offset, 0, d.ld,
                                                      f->buf.Z_std_log + m * plane);
    f->launches += 2;
    // Wc: one row per column the model uses (the refits delete / append the tested column,
    // model_wrap.py:161, 167); rows of padded columns stay 0.
    int kk = 0;
    for (int k = 0; k < d.Kc; ++k) {
      float* dst = f->buf.Wc + ((int64_t)m * d.Kc + k) * d.ld;
      if (f->wide ? k < d.xc_width[m] : ((d.xc_mask[m] >> k) & 1u) != 0) {
        normals_kernel<<<grid_1d(d.ld, 256), 256, 0, s>>>(d.seed, BRIE_PHASE_INIT, mid, BRIE_INIT_WC, 1, 1, d.ld,
                                                         d.event_offset, kk, d.ld, dst);
        ++kk;
      } else {
        fill_kernel<<<grid_1d(d.ld, 256), 256, 0, s>>>(dst, d.ld, 0.f);
      }
      f->launches += 1;
    }
    if (d.Kg > 0) {
      normals_kernel<<<grid_1d(d.n_cells * d.Kg, 256), 256, 0, s>>>(d.seed, BRIE_PHASE_INIT, mid, BRIE_INIT_WG, 1,
                                                                    d.n_cells, d.Kg, 0, 0, d.Kg,
                                                                    f->buf.Wg + (int64_t)m * d.n_cells * d.Kg);
      f->launches += 1;
    }
    float* bdst = f->buf.intercept + (int64_t)m * nsmall;
    if (d.train_intercept) {
      if (d.cell_mode)
        normals_kernel<<<grid_1d(d.n_cells, 256), 256, 0, s>>>(d.seed, BRIE_PHASE_INIT, mid, BRIE_INIT_INTERCEPT, 1,
                                                              d.n_cells, 1, 0, 0, 1, bdst);
      else
        normals_kernel<<<grid_1d(d.ld, 256), 256, 0, s>>>(d.seed, BRIE_PHASE_INIT, mid, BRIE_INIT_INTERCEPT, 1, 1,
                                                         d.ld, d.event_offset, 0, d.ld, bdst);
    } else {
      fill_kernel<<<grid_1d(nsmall, 256), 256, 0, s>>>(bdst, nsmall, intercept_const);
    }
    fill_kernel<<<grid_1d(nsmall, 256), 256, 0, s>>>(f->buf.sigma_log + (int64_t)m * nsmall, nsmall,
                                                    logf(sigma_const));
    f->launches += 2;
  }
  BRIE_CUDA(cudaGetLastError());
  return BRIE_OK;
}

int brie_fit_begin_stage(brie_fit* f, float lr, void* stream) {
  if (!f || !f->bound) return fail(BRIE_ERR_ARG, "fit not bound");
  if (f->step_open) return fail(BRIE_ERR_ARG, "a split step is still open");
  cudaStream_t s = (cudaStream_t)stream;
  const brie_fit_desc& d = f->d;
  BRIE_CUDA(cudaMemsetAsync(f->buf.adam_Z, 0, (size_t)4 * d.n_models * d.n_cells * d.ld * sizeof(float), s));
  BRIE_CUDA(cudaMemsetAsync(f->buf.adam_small, 0, f->sz.adam_small_floats * sizeof(float), s));
  f->stage_open = true;
  f->lr = lr;
  f->t = 0;
  return BRIE_OK;
}

int brie_fit_resume_stage(brie_fit* f, float lr, int64_t adam_t, uint32_t global_step) {
  if (!f || !f->bound) return fail(BRIE_ERR_ARG, "fit not bound");
  if (f->step_open) return fail(BRIE_ERR_ARG, "a split step is still open");
  if (adam_t < 0) return fail(BRIE_ERR_ARG, "adam_t must be >= 0");
  f->stage_open = true;
  f->lr = lr;
  f->t = adam_t;
  f->global_step = global_step;
  return BRIE_OK;
}

int brie_fit_get_step(const brie_fit* f, int64_t* adam_t, uint32_t* global_step) {
  if (!f || !adam_t || !global_step) return fail(BRIE_ERR_ARG, "null argument");
  *adam_t = f->t;
  *global_step = f->global_step;
  return BRIE_OK;
}

int brie_fit_step_phase(brie_fit* f, int32_t phase, int32_t trace_slot, void* stream) {
  if (!f || !f->bound) return fail(BRIE_ERR_ARG, "fit not bound");
  cudaStream_t s = (cudaStream_t)stream;
  const brie_fit_desc& d = f->d;
  const bool loss = trace_slot >= 0;
  if (loss && trace_slot >= d.trace_cap) return fail(BRIE_ERR_ARG, "trace_slot %d >= trace_cap %d", trace_slot, d.trace_cap);
  if (phase == 0) {
    const bool margin = d.target == BRIE_TARGET_MARGINLIK;
    if (f->step_open) return fail(BRIE_ERR_ARG, "phase 0 called twice");
    if (!f->stage_open) return fail(BRIE_ERR_ARG, "brie_fit_begin_stage must be called before the first step");
    if (!f->codes && !f->buf.counts[0]) return fail(BRIE_ERR_ARG, "neither count tiles nor count codes bound");
    // checked: a refused call leaves the Adam step as it was
    f->t += 1;
    const double t = (double)f->t;
    f->alpha = (float)((double)f->lr * sqrt(1.0 - pow(0.999, t)) / (1.0 - pow(0.9, t)));
    // per-event partials: the covariates the step kernel contracts itself, intercept and sigma (gene mode), then the
    // loss, which the marginLik kernel always sums; marginLik tiles its columns its own way
    const bool loss_row = loss || margin;
    const int nev = (f->wide ? 0 : d.Kc) + (d.cell_mode ? 0 : 2) + (loss_row ? 1 : 0);
    const int cell_tiles = margin ? (int)ceil_div(d.ld, kMarginTile) : f->sz.n_col_tiles;
    int rc = margin ? launch_margin_step(f, nev, cell_tiles, s) : launch_fused_step(f, loss, s);
    if (!rc) rc = launch_event_update(f, nev, loss_row, trace_slot, s);
    if (!rc) rc = launch_cell_reduce(f, cell_tiles, s);
    if (rc) return rc;
    f->step_open = true;
    return BRIE_OK;
  }
  if (phase == 1) {
    if (!f->step_open) return fail(BRIE_ERR_ARG, "phase 1 without phase 0");
    int rc = launch_cell_update(f, s);
    if (rc) return rc;
    f->global_step += 1;
    f->step_open = false;
    return BRIE_OK;
  }
  return fail(BRIE_ERR_ARG, "phase must be 0 or 1");
}

int brie_fit_run_steps(brie_fit* f, int32_t n_steps, int32_t trace_slot0, void* stream) {
  if (!f || !f->bound) return fail(BRIE_ERR_ARG, "fit not bound");
  if (n_steps < 0) return fail(BRIE_ERR_ARG, "n_steps must be >= 0");
  const int64_t n_G = (int64_t)f->d.n_models * f->d.n_cells * f->ncell;
  for (int i = 0; i < n_steps; ++i) {
    const int slot = trace_slot0 >= 0 ? trace_slot0 + i : -1;
    int rc = brie_fit_step_phase(f, 0, slot, stream);
    if (rc) return rc;
    if (f->comm && n_G > 0) {   // the path's one exchange step, in stream order between the two halves
      rc = comm_allreduce_sum_f32(f->comm, (float*)f->buf.scratch + f->off_G, n_G, (cudaStream_t)stream);
      if (rc) return rc;
    }
    rc = brie_fit_step_phase(f, 1, slot, stream);
    if (rc) return rc;
  }
  return BRIE_OK;
}

int brie_fit_set_comm(brie_fit* f, brie_comm* comm) {
  if (!f) return fail(BRIE_ERR_ARG, "null argument");
  if (f->step_open) return fail(BRIE_ERR_ARG, "a split step is still open");
  f->comm = comm;
  return BRIE_OK;
}

int brie_fit_set_active_blocks(brie_fit* f, const int32_t* blk_ids, int64_t blk_stride, const int32_t* n_blk_host) {
  if (!f || !f->bound) return fail(BRIE_ERR_ARG, "fit not bound");
  if (f->step_open) return fail(BRIE_ERR_ARG, "a split step is still open");
  if (!blk_ids) {
    f->blk_ids = nullptr;
    f->blk_stride = 0;
    f->blk_tiles = 0;
    return BRIE_OK;
  }
  const brie_fit_desc& d = f->d;
  if (f->ncell > 0 || d.target != BRIE_TARGET_ELBO)
    return fail(BRIE_ERR_UNSUPPORTED, "column compaction needs per-event parameters only (Kg = 0, gene intercept) and target ELBO");
  if (d.ld % 8 != 0) return fail(BRIE_ERR_ARG, "column compaction needs ld %% 8 == 0");
  if (!n_blk_host || blk_stride < 1) return fail(BRIE_ERR_ARG, "n_blk_host and blk_stride required");
  const int bpt = step_tile_cols(f->wide ? 0 : d.Kc, f->wide ? 0 : d.Kg) / kBlkCols;
  int tiles = 0;
  for (int m = 0; m < d.n_models; ++m) {
    if (n_blk_host[m] < 0 || n_blk_host[m] > blk_stride || (int64_t)n_blk_host[m] * kBlkCols > d.ld)
      return fail(BRIE_ERR_ARG, "n_blk_host[%d] = %d out of range", m, n_blk_host[m]);
    f->n_blk[m] = n_blk_host[m];
    const int t = (int)ceil_div(n_blk_host[m], bpt);
    if (t > tiles) tiles = t;
  }
  f->blk_ids = blk_ids;
  f->blk_stride = blk_stride;
  f->blk_tiles = tiles;
  return BRIE_OK;
}

int brie_fit_set_count_codes(brie_fit* f, const uint32_t* codes, int64_t codes_model_stride, const float* dict) {
  if (!f) return fail(BRIE_ERR_ARG, "null argument");
  if (f->step_open) return fail(BRIE_ERR_ARG, "a split step is still open");
  if (codes) {
    if (!dict) return fail(BRIE_ERR_ARG, "dict required with codes");
    if ((((uintptr_t)codes) & 15u) != 0) return fail(BRIE_ERR_ARG, "codes must be 16-byte aligned");
    if (codes_model_stride < 0 || codes_model_stride % 4 != 0)
      return fail(BRIE_ERR_ARG, "codes_model_stride must be >= 0 and a multiple of 4");
  } else if (f->bound && !f->buf.counts[0]) {
    return fail(BRIE_ERR_ARG, "this fit has no count tiles to fall back to");
  }
  f->codes = codes;
  f->code_mstride = codes ? codes_model_stride : 0;
  f->code_dict = codes ? dict : nullptr;
  return BRIE_OK;
}

int brie_fit_cell_grad(brie_fit* f, float** ptr, int64_t* n_floats) {
  if (!f || !f->bound || !ptr || !n_floats) return fail(BRIE_ERR_ARG, "null argument or fit not bound");
  *ptr = (float*)f->buf.scratch + f->off_G;
  *n_floats = (int64_t)f->d.n_models * f->d.n_cells * f->ncell;
  return BRIE_OK;
}

int brie_fit_eval_loss_gene(brie_fit* f, int32_t n_eval, int32_t mc_size, float* loss_gene, void* stream) {
  if (!f || !f->bound || !loss_gene) return fail(BRIE_ERR_ARG, "null argument or fit not bound");
  if (n_eval < 1) return fail(BRIE_ERR_ARG, "n_eval must be >= 1");
  if (f->subfit) return fail(BRIE_ERR_UNSUPPORTED, "loss_gene is evaluated on the parent fit, not on a gathered sub-fit");
  if (mc_size < 1 || mc_size > 4096) return fail(BRIE_ERR_ARG, "mc_size out of range");
  cudaStream_t s = (cudaStream_t)stream;
  const brie_fit_desc& d = f->d;
  float* scratch = (float*)f->buf.scratch;
  EvalArgs a = fit_args<EvalArgs>(f);
  a.Zl = f->buf.Z_loc; a.Zs = f->buf.Z_std_log;
  a.part_ev = scratch + f->off_part_ev;
  a.S = mc_size; a.n_eval = n_eval; a.rows_per_cta = f->sz.rows_per_cta;
  a.KC = d.Kc; a.KG = d.Kg; a.cell_mode = d.cell_mode;
  a.margin = d.target == BRIE_TARGET_MARGINLIK;
  for (int m = 0; m < d.n_models; ++m) a.model_id[m] = d.model_id[m];
  const dim3 grid(d.n_models, (unsigned)ceil_div(d.ld, kTileCols), f->sz.n_row_chunks);
  eval_loss_kernel<<<grid, kThreads, 0, s>>>(a);
  BRIE_CUDA(cudaGetLastError());
  const dim3 g2((unsigned)ceil_div(d.ld, 256), d.n_models);
  eval_reduce_kernel<<<g2, 256, 0, s>>>(a.part_ev, f->sz.n_row_chunks, d.n_models, d.ld, d.n_events, loss_gene);
  BRIE_CUDA(cudaGetLastError());
  f->launches += 2;
  return BRIE_OK;
}

int brie_fit_posterior(brie_fit* f, int32_t model, float* Psi, float* Psi95CI, float* Z_std, void* stream) {
  if (!f || !f->bound) return fail(BRIE_ERR_ARG, "fit not bound");
  if (model < 0 || model >= f->d.n_models) return fail(BRIE_ERR_ARG, "model index out of range");
  const int64_t plane = f->d.n_cells * f->d.ld;
  posterior_kernel<<<grid_1d(plane, 256), 256, 0, (cudaStream_t)stream>>>(
      f->buf.Z_loc + model * plane, f->buf.Z_std_log + model * plane, plane, Psi, Psi95CI, Z_std);
  BRIE_CUDA(cudaGetLastError());
  f->launches += 1;
  return BRIE_OK;
}

int brie_fit_element_terms(brie_fit* f, int32_t model, const float* c1, const float* c2, const float* c3,
                           int32_t mc_size, uint32_t noise_step, int32_t margin, float* loglik, float* kl,
                           float* prior_mean, void* stream) {
  if (!f || !f->bound) return fail(BRIE_ERR_ARG, "fit not bound");
  if (model < 0 || model >= f->d.n_models) return fail(BRIE_ERR_ARG, "model index out of range");
  if (loglik && (!c1 || !c2)) return fail(BRIE_ERR_ARG, "count tiles required for loglik");
  if (loglik && (mc_size < 1 || mc_size > 4096)) return fail(BRIE_ERR_ARG, "mc_size out of range");
  if (f->subfit) return fail(BRIE_ERR_UNSUPPORTED, "element terms are evaluated on the parent fit");
  const brie_fit_desc& d = f->d;
  TermsArgs a = fit_args<TermsArgs>(f);
  a.c[0] = c1; a.c[1] = c2; a.c[2] = c3;   // the caller's count tiles, not the fitted ones
  a.Zl = f->buf.Z_loc; a.Zs = f->buf.Z_std_log;
  a.loglik = loglik; a.kl = kl; a.prior_mean = prior_mean;
  a.m = model; a.S = mc_size; a.KC = d.Kc; a.KG = d.Kg; a.cell_mode = d.cell_mode;
  a.margin = margin != 0; a.model_id = d.model_id[model]; a.noise_step = noise_step;
  element_terms_kernel<<<grid_1d(d.n_cells * d.ld, 256), 256, 0, (cudaStream_t)stream>>>(a);
  BRIE_CUDA(cudaGetLastError());
  f->launches += 1;
  return BRIE_OK;
}

}  // extern "C"

namespace {

// Geometry of the Wald information pass of model m (brie_wald.cuh): x~ width, pair block, row chunks.
struct WaldPlan {
  int width, has_b, kt, n_pairs, pb, n_pblk, n_tiles, n_chunks;
  int64_t rows_per_chunk;
  size_t scratch_bytes;
};

int wald_plan(const brie_fit* f, int32_t model, WaldPlan* w) {
  if (!f || !f->bound) return fail(BRIE_ERR_ARG, "fit not bound");
  const brie_fit_desc& d = f->d;
  if (model < 0 || model >= d.n_models) return fail(BRIE_ERR_ARG, "model index out of range");
  if (d.target != BRIE_TARGET_ELBO)
    return fail(BRIE_ERR_UNSUPPORTED, "Wald information needs a trained posterior (target ELBO)");
  if (f->subfit) return fail(BRIE_ERR_UNSUPPORTED, "Wald information is computed on the parent fit, not on a gathered sub-fit");
  w->width = f->wide ? d.xc_width[model] : __builtin_popcount(d.xc_mask[model]);
  w->has_b = (!d.cell_mode && d.train_intercept) ? 1 : 0;
  w->kt = w->width + w->has_b;
  w->n_pairs = w->kt * (w->kt + 1) / 2;
  w->pb = w->n_pairs <= 4 ? 4 : (w->n_pairs <= 12 ? 12 : kWaldMaxPairs);
  w->n_pblk = (int)ceil_div(w->n_pairs, w->pb);
  w->n_tiles = (int)ceil_div(d.n_events, kWaldCols);
  // Row chunks of >= kWaldMinRows cells, at most kWaldMaxChunks of them: a function of n_cells alone, so the float64
  // sums over cells associate the same way whatever the event count -- an event chunk or shard of a fit gets the
  // same bits as the whole -- and the scratch stays within kWaldMaxChunks partials per output.
  const int64_t blocks = (int64_t)w->n_tiles * w->n_pblk;
  const int64_t n_chunks = std::min<int64_t>(ceil_div(d.n_cells, kWaldMinRows), kWaldMaxChunks);
  w->rows_per_chunk = ceil_div(ceil_div(d.n_cells, n_chunks), kWaldBatch) * kWaldBatch;
  w->n_chunks = (int)ceil_div(d.n_cells, w->rows_per_chunk);
  if (blocks > 0x7fffffffLL) return fail(BRIE_ERR_UNSUPPORTED, "too many event tiles x pair blocks");
  w->scratch_bytes = (size_t)w->n_chunks * w->n_pairs * d.ld * sizeof(double);
  return BRIE_OK;
}

template <int PB>
cudaError_t launch_wald(const WaldArgs& a, dim3 grid, cudaStream_t s) {
  wald_info_kernel<PB><<<grid, kWaldCols * kWaldRowGroups, 0, s>>>(a);
  return cudaGetLastError();
}

}  // namespace

extern "C" {

int brie_fit_wald_sizes(const brie_fit* f, int32_t model, size_t* scratch_bytes, int32_t* k_tilde) {
  if (!scratch_bytes || !k_tilde) return fail(BRIE_ERR_ARG, "null argument");
  WaldPlan w;
  int rc = wald_plan(f, model, &w);
  if (rc) return rc;
  *scratch_bytes = w.scratch_bytes;
  *k_tilde = w.kt;
  return BRIE_OK;
}

int brie_fit_wald_info(brie_fit* f, int32_t model, double* info, void* scratch, void* stream) {
  WaldPlan w;
  int rc = wald_plan(f, model, &w);
  if (rc) return rc;
  if (w.n_pairs == 0) return BRIE_OK;
  if (!info || !scratch) return fail(BRIE_ERR_ARG, "info and scratch required");
  if ((((uintptr_t)info) & 7u) != 0 || (((uintptr_t)scratch) & 7u) != 0)
    return fail(BRIE_ERR_ARG, "info and scratch must be 8-byte aligned");
  const brie_fit_desc& d = f->d;
  cudaStream_t s = (cudaStream_t)stream;
  const int64_t plane = d.n_cells * d.ld;
  WaldArgs a;
  memset(&a, 0, sizeof a);
  a.Nc = d.n_cells; a.Ng = d.n_events; a.ld = d.ld;
  a.Zs = f->buf.Z_std_log + model * plane;
  a.tau = f->buf.sigma_log + (int64_t)model * (d.cell_mode ? d.n_cells : d.ld);
  a.xc_stride = d.Kc > 0 ? d.Kc : 1;
  a.Xc = f->buf.Xc ? f->buf.Xc + (int64_t)model * d.n_cells * a.xc_stride : nullptr;
  a.width = w.width; a.xc_mask = d.xc_mask[model]; a.wide = f->wide ? 1 : 0; a.has_b = w.has_b;
  a.n_pairs = w.n_pairs; a.cell_tau = d.cell_mode; a.rows_per_chunk = w.rows_per_chunk; a.n_tiles = w.n_tiles;
  a.part = (double*)scratch;
  if (w.width > 0 && !a.Xc) return fail(BRIE_ERR_ARG, "Xc required");
  const dim3 grid((unsigned)((int64_t)w.n_tiles * w.n_pblk), (unsigned)w.n_chunks);
  switch (w.pb) {
    case 4: BRIE_CUDA(launch_wald<4>(a, grid, s)); break;
    case 12: BRIE_CUDA(launch_wald<12>(a, grid, s)); break;
    default: BRIE_CUDA(launch_wald<kWaldMaxPairs>(a, grid, s)); break;
  }
  const int64_t n_out = d.n_events * w.n_pairs;
  wald_reduce_kernel<<<(unsigned)ceil_div(n_out, 256), 256, 0, s>>>(a.part, w.n_chunks, w.n_pairs, d.ld, d.n_events, info);
  BRIE_CUDA(cudaGetLastError());
  f->launches += 2;
  return BRIE_OK;
}

int brie_resample_counts(uint64_t seed, int64_t n_cells, int64_t n_events, int64_t ld, int64_t event_offset,
                         const float* total, const float* psi, const float* efflen3, float* c1, float* c2, float* c3,
                         void* stream) {
  if (n_cells <= 0 || n_events <= 0 || ld < n_events) return fail(BRIE_ERR_ARG, "bad shape");
  if (!total || !psi || !c1 || !c2) return fail(BRIE_ERR_ARG, "null argument");
  resample_counts_kernel<<<grid_1d(n_cells * ld, 256), 256, 0, (cudaStream_t)stream>>>(
      seed, n_cells, n_events, ld, event_offset, total, psi, efflen3, c1, c2, c3);
  BRIE_CUDA(cudaGetLastError());
  return BRIE_OK;
}

int brie_fit_group_trace(brie_fit* f, int32_t n_slots, int64_t group_size, int64_t n_groups, double* out,
                         void* stream) {
  if (!f || !f->bound || !out) return fail(BRIE_ERR_ARG, "null argument or fit not bound");
  const brie_fit_desc& d = f->d;
  if (n_slots < 1 || n_slots > d.trace_cap) return fail(BRIE_ERR_ARG, "n_slots out of range");
  if (group_size < 1 || n_groups < 1) return fail(BRIE_ERR_ARG, "bad group geometry");
  if (f->subfit) return fail(BRIE_ERR_UNSUPPORTED, "scatter the trace of a gathered sub-fit back to its parent first");
  const int64_t first_group = d.event_offset / group_size;
  const dim3 grid(n_slots, d.n_models);
  group_trace_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(f->buf.loss_trace, d.trace_cap, d.ld, d.n_events,
                                                           d.event_offset, group_size, first_group, n_groups,
                                                           n_slots, out);
  BRIE_CUDA(cudaGetLastError());
  f->launches += 1;
  return BRIE_OK;
}

int64_t brie_fit_launch_count(const brie_fit* f) { return f ? f->launches : -1; }

int brie_philox_normals_host(uint64_t seed, uint32_t phase, uint32_t model, uint32_t step, int32_t n_samples,
                             int64_t n_rows, int64_t n_cols, int64_t col_offset, float* out) {
  if (!out || n_samples < 1 || n_rows < 0 || n_cols < 0) return fail(BRIE_ERR_ARG, "bad argument");
  for (int64_t r = 0; r < n_rows; ++r)
    for (int64_t c = 0; c < n_cols; ++c)
      for (int s0 = 0; s0 < n_samples; s0 += 4) {
        float e[4];
        brie_normals4((uint32_t)(col_offset + c), (uint32_t)r, step, brie_stream_word(phase, model, (uint32_t)(s0 >> 2)),
                      seed, e);
        for (int q = 0; q < 4 && s0 + q < n_samples; ++q) out[((int64_t)(s0 + q) * n_rows + r) * n_cols + c] = e[q];
      }
  return BRIE_OK;
}

int brie_philox_normals_device(uint64_t seed, uint32_t phase, uint32_t model, uint32_t step, int32_t n_samples,
                               int64_t n_rows, int64_t n_cols, int64_t col_offset, float* out, void* stream) {
  if (!out || n_samples < 1 || n_rows < 0 || n_cols < 0) return fail(BRIE_ERR_ARG, "bad argument");
  normals_kernel<<<grid_1d(n_rows * n_cols, 256), 256, 0, (cudaStream_t)stream>>>(
      seed, phase, model, step, n_samples, n_rows, n_cols, col_offset, 0, n_cols, out);
  BRIE_CUDA(cudaGetLastError());
  return BRIE_OK;
}

int brie_simulate_counts(uint64_t seed, int64_t n_cells, int64_t n_events, int64_t ld, int64_t event_offset,
                         const float* logit_mean, const float* logit_sd, const float* Xc, const float* Wc,
                         int32_t Kc, const float* efflen3, const float* lam, const float* cdr, float pseudo_count,
                         float* c1, float* c2, float* c3, void* stream) {
  if (n_cells <= 0 || n_events <= 0 || ld < n_events) return fail(BRIE_ERR_ARG, "bad shape");
  if (!logit_mean || !logit_sd || !lam || !cdr || !c1 || !c2) return fail(BRIE_ERR_ARG, "null argument");
  if (Kc < 0 || (Kc > 0 && (!Xc || !Wc))) return fail(BRIE_ERR_ARG, "Xc and Wc required when Kc > 0");
  simulate_counts_kernel<<<grid_1d(n_cells * ld, 256), 256, 0, (cudaStream_t)stream>>>(
      seed, n_cells, n_events, ld, event_offset, logit_mean, logit_sd, Xc, Wc, Kc, efflen3, lam, cdr, pseudo_count,
      c1, c2, c3);
  BRIE_CUDA(cudaGetLastError());
  return BRIE_OK;
}

}  // extern "C"
