// Count ingest in front of the fit (SURVEY f1): sparse layers -> the dense padded
// (cells, ld) float32 tiles the step kernel streams, without a dense host copy.
//
// The reference densifies every sparse layer on the host
// (brie/models/model_wrap.py:108-111, brie/models/model_TFProb.py:135-137), applies the
// pseudo-count with boolean-mask indexing (model_wrap.py:113-117) and builds two dense
// float64 (cells, genes) matrices for the gene filter (brie/utils/preprocessing.py:39-45).
// Here the CSC/CSR triplets cross PCIe (8 B per stored count instead of 4 B per matrix
// element and layer) and the scatter, pseudo-count and per-gene filter statistics run on
// the device.
#include <stdint.h>

#include "brie_host.h"

namespace brie {

// One warp per event column of a CSC slab; lanes stride over the column's stored counts.
// atomicAdd so that duplicate (row, col) entries sum, as scipy's toarray() does.
__global__ void __launch_bounds__(256) ingest_csc_kernel(const int64_t* __restrict__ colptr,
                                                         const int32_t* __restrict__ rows,
                                                         const float* __restrict__ vals, int64_t n_events,
                                                         int64_t n_cells, int64_t ld, float* out) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; g < n_events; g += warps) {
    const int64_t lo = colptr[g], hi = colptr[g + 1];
    for (int64_t e = lo + lane; e < hi; e += 32) {
      const int64_t r = rows[e];
      if (r >= 0 && r < n_cells) atomicAdd(out + r * ld + g, vals[e]);
    }
  }
}

// One warp per cell row of a CSR matrix; keeps the columns of [event_begin, event_begin + n_events).
__global__ void __launch_bounds__(256) ingest_csr_kernel(const int64_t* __restrict__ rowptr,
                                                         const int32_t* __restrict__ cols,
                                                         const float* __restrict__ vals, int64_t n_cells,
                                                         int64_t event_begin, int64_t n_events, int64_t ld,
                                                         float* out) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n_cells; r += warps) {
    const int64_t lo = rowptr[r], hi = rowptr[r + 1];
    for (int64_t e = lo + lane; e < hi; e += 32) {
      const int64_t g = (int64_t)cols[e] - event_begin;
      if (g >= 0 && g < n_events) atomicAdd(out + r * ld + g, vals[e]);
    }
  }
}

// model_wrap.py:113-117: idx = c1 + c2 > 0; c1[idx] += pseudo; c2[idx] += pseudo   (float32)
__global__ void __launch_bounds__(256) pseudo_count_kernel(float4* c1, float4* c2, int64_t n4, float pseudo) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    float4 a = c1[i], b = c2[i];
    bool any = false;
    if (a.x + b.x > 0.f) { a.x += pseudo; b.x += pseudo; any = true; }
    if (a.y + b.y > 0.f) { a.y += pseudo; b.y += pseudo; any = true; }
    if (a.z + b.z > 0.f) { a.z += pseudo; b.z += pseudo; any = true; }
    if (a.w + b.w > 0.f) { a.w += pseudo; b.w += pseudo; any = true; }
    if (any) { c1[i] = a; c2[i] = b; }
  }
}

// Per-event filter statistics over a dense tile (preprocessing.py:38-61): column sums of each
// layer and the number of cells with unique (c1 + c2 > 0) / any (c1 + c2 + c3 > 0) counts.
// Stage 1: one thread per event, a CTA covers 128 events x one row chunk (coalesced 512-byte
// row segments); stage 2 adds the chunk partials in fixed order -> deterministic.
constexpr int kStatFields = 5;

__global__ void __launch_bounds__(128) gene_stats_partial_kernel(const float* __restrict__ c1,
                                                                 const float* __restrict__ c2,
                                                                 const float* __restrict__ c3, int64_t n_cells,
                                                                 int64_t ld, int64_t rows_per_chunk,
                                                                 double* part /* (chunks, 5, ld) */) {
  const int64_t g = (int64_t)blockIdx.x * 128 + threadIdx.x;
  if (g >= ld) return;
  const int64_t r0 = (int64_t)blockIdx.y * rows_per_chunk;
  const int64_t r1 = min(r0 + rows_per_chunk, n_cells);
  double s1 = 0.0, s2 = 0.0, s3 = 0.0;
  int64_t nu = 0, nt = 0;
  for (int64_t r = r0; r < r1; ++r) {
    const float a = c1[r * ld + g], b = c2[r * ld + g], c = c3 ? c3[r * ld + g] : 0.f;
    s1 += (double)a; s2 += (double)b; s3 += (double)c;
    const double u = (double)a + (double)b;    // the reference accumulates the layers in float64
    nu += u > 0.0;
    nt += (u + (double)c) > 0.0;
  }
  double* p = part + (int64_t)blockIdx.y * kStatFields * ld + g;
  p[0] = s1; p[ld] = s2; p[2 * ld] = s3; p[3 * ld] = (double)nu; p[4 * ld] = (double)nt;
}

__global__ void __launch_bounds__(256) gene_stats_reduce_kernel(const double* __restrict__ part, int n_chunks,
                                                                int64_t ld, double* out /* (5, ld) */) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;   // over 5 * ld
  if (i >= kStatFields * ld) return;
  double s = 0.0;
  for (int c = 0; c < n_chunks; ++c) s += part[(int64_t)c * kStatFields * ld + i];
  out[i] = s;
}

// keep[j] -> column gather of a dense tile (events that pass the filter), so the kept counts
// never go back to the host: out[r, j] = in[r, src[j]].
__global__ void __launch_bounds__(256) gather_columns_kernel(const float* __restrict__ in, int64_t ld_in,
                                                             const int64_t* __restrict__ src, int64_t n_cells,
                                                             int64_t n_out, int64_t ld_out, float* out) {
  const int64_t total = n_cells * ld_out;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / ld_out, j = i % ld_out;
    out[i] = j < n_out ? in[r * ld_in + src[j]] : 0.f;
  }
}

// inverse of the gather: out[r, dst[j]] = in[r, j]; columns not listed keep their contents
__global__ void __launch_bounds__(256) scatter_columns_kernel(const float* __restrict__ in, int64_t ld_in,
                                                              const int64_t* __restrict__ dst, int64_t n_cells,
                                                              int64_t n_in, int64_t ld_out, float* out) {
  const int64_t total = n_cells * n_in;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / n_in, j = i % n_in;
    out[r * ld_out + dst[j]] = in[r * ld_in + j];
  }
}

// ---- dictionary coding of the count tiles (brie_encode_counts) -------------------------------------------------
// Per layer, a 1024-slot open-addressing set of the non-zero values' bit patterns (0 = empty slot): a layer that
// can be coded holds at most 255 of them, so the set stays at most a quarter full.  Probes are bounded by the
// table size, so the passes end whatever the data.
constexpr int kCodeHash = 1024;
constexpr int kCodeMax = 255;                  // non-zero values per layer a code byte can index
constexpr int32_t kCodeOverflow = 1 << 30;     // n_values[l] once layer l cannot be coded

__device__ __forceinline__ uint32_t code_hash(uint32_t bits) { return (bits * 0x9E3779B1u) >> 22; }

// Inserts `bits` into a set; returns 1 if it was new, 0 if present, -1 if the set is full.
__device__ __forceinline__ int code_set_insert(uint32_t* keys, uint32_t bits) {
  uint32_t h = code_hash(bits);
  for (int i = 0; i < kCodeHash; ++i, h = (h + 1) & (kCodeHash - 1)) {
    const uint32_t k = *(volatile uint32_t*)&keys[h];
    if (k == bits) return 0;
    if (k == 0u) {
      const uint32_t old = atomicCAS(&keys[h], 0u, bits);
      if (old == 0u) return 1;
      if (old == bits) return 0;
    }
  }
  return -1;
}

// Pass 1: every CTA collects the values of its part of the tiles in shared memory, then merges its sets into the
// global ones (keys (3, kCodeHash)), counting the distinct values of each layer in n_values.
__global__ void __launch_bounds__(256) code_collect_kernel(const float* __restrict__ c1, const float* __restrict__ c2,
                                                           const float* __restrict__ c3, int64_t n4, uint32_t* keys,
                                                           int32_t* n_values) {
  __shared__ uint32_t s_keys[3][kCodeHash];
  __shared__ int s_n[3];
  for (int i = threadIdx.x; i < 3 * kCodeHash; i += blockDim.x) (&s_keys[0][0])[i] = 0u;
  if (threadIdx.x < 3) s_n[threadIdx.x] = 0;
  __syncthreads();
  const float* cs[3] = {c1, c2, c3};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
#pragma unroll
    for (int l = 0; l < 3; ++l) {
      if (!cs[l]) continue;
      const uint4 v = reinterpret_cast<const uint4*>(cs[l])[i];
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if ((w[j] & 0x7fffffffu) == 0u) continue;                      // +0 / -0: code 0
        if ((w[j] >> 31) != 0u || (w[j] & 0x7fffffffu) > 0x7f800000u) {  // negative or NaN: not codable
          atomicMax(&s_n[l], kCodeOverflow);
          continue;
        }
        if (*(volatile int*)&s_n[l] > kCodeMax) continue;
        const int r = code_set_insert(s_keys[l], w[j]);
        if (r > 0) atomicAdd(&s_n[l], 1);
        if (r < 0) atomicMax(&s_n[l], kCodeOverflow);
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 3 * kCodeHash; i += blockDim.x) {
    const int l = i / kCodeHash;
    if (s_n[l] > kCodeMax) {
      if (i % kCodeHash == 0) atomicMax(&n_values[l], kCodeOverflow);
      continue;
    }
    const uint32_t k = (&s_keys[0][0])[i];
    if (k == 0u || *(volatile int32_t*)&n_values[l] > kCodeMax) continue;
    const int r = code_set_insert(keys + l * kCodeHash, k);
    if (r > 0) atomicAdd(&n_values[l], 1);
    if (r < 0) atomicMax(&n_values[l], kCodeOverflow);
  }
}

// Pass 2 (one CTA per layer): code of a value = 1 + its rank among the layer's values (ascending: for non-negative
// floats the bit patterns order as the values), into slot_code (3, kCodeHash) and the dictionary.
__global__ void __launch_bounds__(kCodeHash) code_dict_kernel(const uint32_t* __restrict__ keys,
                                                              const int32_t* __restrict__ n_values,
                                                              uint8_t* slot_code, float* dict) {
  const int l = blockIdx.x;
  __shared__ uint32_t s_k[kCodeHash];
  const uint32_t k = keys[l * kCodeHash + threadIdx.x];
  s_k[threadIdx.x] = k;
  __syncthreads();
  if (n_values[l] > kCodeMax || k == 0u) return;
  int rank = 0;
  for (int i = 0; i < kCodeHash; ++i) rank += (s_k[i] != 0u && s_k[i] < k) ? 1 : 0;
  slot_code[l * kCodeHash + threadIdx.x] = (uint8_t)(rank + 1);
  dict[l * 256 + rank + 1] = __uint_as_float(k);
}

__device__ __forceinline__ uint32_t code_lookup(const uint32_t* keys, const uint8_t* codes, uint32_t bits) {
  if ((bits & 0x7fffffffu) == 0u) return 0u;
  uint32_t h = code_hash(bits);
  for (int i = 0; i < kCodeHash; ++i, h = (h + 1) & (kCodeHash - 1))
    if (keys[h] == bits) return codes[h];
  return 0u;   // not reached: pass 1 saw every value
}

// Pass 3: code words, four elements per thread.
__global__ void __launch_bounds__(256) code_write_kernel(const float* __restrict__ c1, const float* __restrict__ c2,
                                                         const float* __restrict__ c3, int64_t n4,
                                                         const uint32_t* __restrict__ keys,
                                                         const uint8_t* __restrict__ slot_code,
                                                         const int32_t* __restrict__ n_values, uint4* out) {
  if (n_values[0] > kCodeMax || n_values[1] > kCodeMax || n_values[2] > kCodeMax) return;
  __shared__ uint32_t s_keys[3 * kCodeHash];
  __shared__ uint8_t s_code[3 * kCodeHash];
  for (int i = threadIdx.x; i < 3 * kCodeHash; i += blockDim.x) {
    s_keys[i] = keys[i];
    s_code[i] = slot_code[i];
  }
  __syncthreads();
  const float* cs[3] = {c1, c2, c3};
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int l = 0; l < 3; ++l) {
      if (!cs[l]) continue;
      const uint4 v = reinterpret_cast<const uint4*>(cs[l])[i];
      const uint32_t b[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int j = 0; j < 4; ++j)
        w[j] |= code_lookup(s_keys + l * kCodeHash, s_code + l * kCodeHash, b[j]) << (8 * l);
    }
    out[i] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

namespace {
int stats_chunks(int64_t n_cells, int64_t ld, int64_t* rows_per_chunk) {
  const int64_t tiles = ceil_div(ld, 128);
  int64_t chunks = ceil_div((int64_t)148 * 16, tiles);
  if (chunks > n_cells) chunks = n_cells;
  if (chunks > 4096) chunks = 4096;
  if (chunks < 1) chunks = 1;
  *rows_per_chunk = ceil_div(n_cells, chunks);
  return (int)ceil_div(n_cells, *rows_per_chunk);
}
}  // namespace

}  // namespace brie

using namespace brie;

extern "C" {

int brie_ingest_csc(int64_t n_cells, int64_t n_events, int64_t ld, const int64_t* colptr, const int32_t* rows,
                    const float* vals, float* out, void* stream) {
  if (n_cells <= 0 || n_events <= 0 || ld < n_events) return fail(BRIE_ERR_ARG, "bad shape");
  if (!colptr || !out) return fail(BRIE_ERR_ARG, "null argument");
  cudaStream_t s = (cudaStream_t)stream;
  BRIE_CUDA(cudaMemsetAsync(out, 0, (size_t)n_cells * ld * sizeof(float), s));
  if (rows && vals) {
    ingest_csc_kernel<<<grid_1d(n_events * 32, 256), 256, 0, s>>>(colptr, rows, vals, n_events, n_cells, ld, out);
    BRIE_CUDA(cudaGetLastError());
  }
  return BRIE_OK;
}

int brie_ingest_csr(int64_t n_cells, int64_t event_begin, int64_t n_events, int64_t ld, const int64_t* rowptr,
                    const int32_t* cols, const float* vals, float* out, void* stream) {
  if (n_cells <= 0 || n_events <= 0 || ld < n_events || event_begin < 0) return fail(BRIE_ERR_ARG, "bad shape");
  if (!rowptr || !out) return fail(BRIE_ERR_ARG, "null argument");
  cudaStream_t s = (cudaStream_t)stream;
  BRIE_CUDA(cudaMemsetAsync(out, 0, (size_t)n_cells * ld * sizeof(float), s));
  if (cols && vals) {
    ingest_csr_kernel<<<grid_1d(n_cells * 32, 256), 256, 0, s>>>(rowptr, cols, vals, n_cells, event_begin, n_events,
                                                                ld, out);
    BRIE_CUDA(cudaGetLastError());
  }
  return BRIE_OK;
}

int brie_add_pseudo_count(int64_t n_cells, int64_t ld, float pseudo_count, float* c1, float* c2, void* stream) {
  if (n_cells <= 0 || ld <= 0 || ld % 4 != 0) return fail(BRIE_ERR_ARG, "bad shape (ld must be a multiple of 4)");
  if (!c1 || !c2) return fail(BRIE_ERR_ARG, "null argument");
  if ((((uintptr_t)c1) | ((uintptr_t)c2)) & 15u) return fail(BRIE_ERR_ARG, "buffers must be 16-byte aligned");
  const int64_t n4 = n_cells * ld / 4;
  pseudo_count_kernel<<<grid_1d(n4, 256), 256, 0, (cudaStream_t)stream>>>((float4*)c1, (float4*)c2, n4, pseudo_count);
  BRIE_CUDA(cudaGetLastError());
  return BRIE_OK;
}

size_t brie_gene_stats_scratch_bytes(int64_t n_cells, int64_t ld) {
  if (n_cells <= 0 || ld <= 0) return 0;
  int64_t rows;
  const int chunks = stats_chunks(n_cells, ld, &rows);
  return (size_t)chunks * kStatFields * ld * sizeof(double);
}

int brie_gene_stats(int64_t n_cells, int64_t ld, const float* c1, const float* c2, const float* c3, double* stats,
                    void* scratch, void* stream) {
  if (n_cells <= 0 || ld <= 0) return fail(BRIE_ERR_ARG, "bad shape");
  if (!c1 || !c2 || !stats || !scratch) return fail(BRIE_ERR_ARG, "null argument");
  cudaStream_t s = (cudaStream_t)stream;
  int64_t rows;
  const int chunks = stats_chunks(n_cells, ld, &rows);
  const dim3 grid((unsigned)ceil_div(ld, 128), (unsigned)chunks);
  gene_stats_partial_kernel<<<grid, 128, 0, s>>>(c1, c2, c3, n_cells, ld, rows, (double*)scratch);
  BRIE_CUDA(cudaGetLastError());
  gene_stats_reduce_kernel<<<(unsigned)ceil_div(kStatFields * ld, 256), 256, 0, s>>>((const double*)scratch, chunks,
                                                                                      ld, stats);
  BRIE_CUDA(cudaGetLastError());
  return BRIE_OK;
}

size_t brie_encode_counts_scratch_bytes(void) { return (size_t)3 * kCodeHash * (sizeof(uint32_t) + sizeof(uint8_t)); }

int brie_encode_counts(int64_t n_cells, int64_t ld, const float* c1, const float* c2, const float* c3,
                       uint32_t* codes, float* dict, int32_t* n_values, void* scratch, void* stream) {
  if (n_cells <= 0 || ld <= 0 || ld % 4 != 0) return fail(BRIE_ERR_ARG, "bad shape (ld must be a multiple of 4)");
  if (!c1 || !c2 || !codes || !dict || !n_values || !scratch) return fail(BRIE_ERR_ARG, "null argument");
  if ((((uintptr_t)c1) | ((uintptr_t)c2) | ((uintptr_t)c3) | ((uintptr_t)codes)) & 15u)
    return fail(BRIE_ERR_ARG, "tiles and codes must be 16-byte aligned");
  cudaStream_t s = (cudaStream_t)stream;
  uint32_t* keys = (uint32_t*)scratch;
  uint8_t* slot_code = (uint8_t*)(keys + 3 * kCodeHash);
  BRIE_CUDA(cudaMemsetAsync(scratch, 0, brie_encode_counts_scratch_bytes(), s));
  BRIE_CUDA(cudaMemsetAsync(n_values, 0, 3 * sizeof(int32_t), s));
  BRIE_CUDA(cudaMemsetAsync(dict, 0, 3 * 256 * sizeof(float), s));
  const int64_t n4 = n_cells * ld / 4;
  const int64_t blocks = ceil_div(n4, 256) < 148 * 8 ? ceil_div(n4, 256) : 148 * 8;
  code_collect_kernel<<<(unsigned)blocks, 256, 0, s>>>(c1, c2, c3, n4, keys, n_values);
  BRIE_CUDA(cudaGetLastError());
  code_dict_kernel<<<3, kCodeHash, 0, s>>>(keys, n_values, slot_code, dict);
  BRIE_CUDA(cudaGetLastError());
  code_write_kernel<<<(unsigned)blocks, 256, 0, s>>>(c1, c2, c3, n4, keys, slot_code, n_values, (uint4*)codes);
  BRIE_CUDA(cudaGetLastError());
  return BRIE_OK;
}

int brie_gather_events(int64_t n_cells, int64_t ld_in, const float* in, const int64_t* src, int64_t n_out,
                       int64_t ld_out, float* out, void* stream) {
  if (n_cells <= 0 || ld_in <= 0 || n_out < 0 || ld_out < n_out || ld_out <= 0) return fail(BRIE_ERR_ARG, "bad shape");
  if (!in || !out || (n_out > 0 && !src)) return fail(BRIE_ERR_ARG, "null argument");
  gather_columns_kernel<<<grid_1d(n_cells * ld_out, 256), 256, 0, (cudaStream_t)stream>>>(in, ld_in, src, n_cells,
                                                                                         n_out, ld_out, out);
  BRIE_CUDA(cudaGetLastError());
  return BRIE_OK;
}

int brie_scatter_events(int64_t n_cells, int64_t ld_in, const float* in, const int64_t* dst, int64_t n_in,
                        int64_t ld_out, float* out, void* stream) {
  if (n_cells <= 0 || ld_in <= 0 || n_in < 0 || ld_in < n_in || ld_out <= 0) return fail(BRIE_ERR_ARG, "bad shape");
  if (!in || !out || (n_in > 0 && !dst)) return fail(BRIE_ERR_ARG, "null argument");
  if (n_in == 0) return BRIE_OK;
  scatter_columns_kernel<<<grid_1d(n_cells * n_in, 256), 256, 0, (cudaStream_t)stream>>>(in, ld_in, dst, n_cells,
                                                                                        n_in, ld_out, out);
  BRIE_CUDA(cudaGetLastError());
  return BRIE_OK;
}

}  // extern "C"
