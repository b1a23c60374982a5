// range_search.cuh — kernels of the exact range search (fx_search_range): every row with distance <= radius.
//
// Tensor-core path: the filter kernels of tc_filter.cuh run in preset-threshold mode with the threshold taken from the
// radius (range_prep_kernel), then
//   range_count_kernel    candidates per query (its lists' entry counts): the size of its segment of the hit buffer
//   range_finish_kernel   exact fp64 rerank of every candidate (rerank8, the library's one summation order), keeps
//                         d <= radius as (distance, row) keys in the query's segment
// Scan path (overflowed candidate lists, shards the tensor-core path does not take, FX_PREC_EXACT_SCAN): the exact scan's
// distance column for a batch of queries, then
//   range_col_count_kernel / range_col_compact_kernel   rows with mask and d <= radius -> keys in the query's segment
// Both feed one emit stage: a segmented sort of the keys (CUB), then
//   range_gather_kernel   sorted keys -> (row_base + row, distance) at the query's output offset
#pragma once
#include "common.cuh"
#include "tc_filter.cuh"

namespace fx {

// Candidate count of every query (one warp each): the sum of its lists' entry counts, or -1 when a list overflowed
// (the filter flagged the query) or its threshold is ORD_SCAN (the filter's scores are not bounded): the scan settles it.
__global__ void __launch_bounds__(256)
range_count_kernel(FinishParams p, int64_t* __restrict__ cand) {
  const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (q >= p.n_q) return;
  const int qt = q / TC_BM, w = q - qt * TC_BM;
  const int r = (w % 4) * 32 + w / 4;
  const int n_lists = (p.rq ? 1 : TC_SPLIT) * p.n_slices;
  int64_t s = 0;
  for (int l = lane; l < n_lists; l += 32) { int count; fin_list(p, qt, r, l, count); s += count; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) cand[q] = (p.flags[q] != 0 || p.tau_g[q] == ORD_SCAN) ? int64_t(-1) : s;
}

// One CTA per query: every candidate of its lists is reranked exactly (8 lanes per candidate, as the k-NN finish kernel)
// and kept when its distance is <= radius. keys[seg[q] ...]: the hits in no particular order; hits[q]: their number.
// Queries the count kernel sent to the scan are skipped.
__global__ void __launch_bounds__(256)
range_finish_kernel(FinishParams p, float radius, const int64_t* __restrict__ seg, uint64_t* __restrict__ keys,
                    int* __restrict__ hits) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* qs = reinterpret_cast<float*>(smem_raw);   // [pitch]
  __shared__ int s_hits;
  __shared__ double s_qq;
  const int q = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, n_warps = blockDim.x >> 5;
  if (p.flags[q] != 0 || p.tau_g[q] == ORD_SCAN) {
    if (tid == 0) hits[q] = 0;
    return;
  }
  const int qt = q / TC_BM, w = q - qt * TC_BM;
  const int r = (w % 4) * 32 + w / 4;
  const size_t q_row = size_t(qt) * TC_BM + r;
  const int n_lists = (p.rq ? 1 : TC_SPLIT) * p.n_slices;
  for (int d = tid; d < p.pitch; d += blockDim.x) qs[d] = p.Qp[q_row * p.pitch + d];
  if (tid == 0) s_hits = 0;
  __syncthreads();
  if (warp == 0) {
    double s = 0.0;
    for (int d = lane; d < p.pitch; d += 32) s = fma(double(qs[d]), double(qs[d]), s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) s_qq = s;
  }
  __syncthreads();
  const double qq = s_qq;
  uint64_t* out = keys + seg[q];
  const int sub = lane & 7, grp = lane >> 3;
  for (int l = warp; l < n_lists; l += n_warps) {
    int count; const uint2* b = fin_list(p, qt, r, l, count);
    for (int c0 = 0; c0 < count; c0 += 4) {
      const int c = c0 + grp;
      const bool live = c < count;
      const uint32_t row = live ? b[c].y : 0u;
      double xx, qx;
      rerank8(p.X, p.pitch, row, live, qs, sub, xx, qx);
      if (sub == 0 && live) {
        const float d = finish_distance(p.metric, qq, xx, qx);
        if (d <= radius) out[atomicAdd(&s_hits, 1)] = make_key(d, row);
      }
    }
  }
  __syncthreads();
  if (tid == 0) hits[q] = s_hits;
}

// Rows of a batch of distance columns (col[slot][n_rows], the exact scan's column mode) that are unmasked and within the
// radius: counted per slot (cnt zeroed by the caller) ...
__global__ void __launch_bounds__(256)
range_col_count_kernel(const float* __restrict__ col, int64_t n_rows, const uint8_t* __restrict__ mask, float radius,
                       int* __restrict__ cnt) {
  const int slot = blockIdx.y;
  const float* d = col + size_t(slot) * n_rows;
  int c = 0;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n_rows; i += int64_t(gridDim.x) * blockDim.x)
    c += (d[i] <= radius && (mask == nullptr || mask[i] != 0)) ? 1 : 0;
  c = __reduce_add_sync(0xffffffffu, c);
  if ((threadIdx.x & 31) == 0 && c) atomicAdd(cnt + slot, c);
}

// ... and written as (distance, row) keys into the slot's segment keys[seg[slot] ...] (fill zeroed by the caller).
__global__ void __launch_bounds__(256)
range_col_compact_kernel(const float* __restrict__ col, int64_t n_rows, const uint8_t* __restrict__ mask, float radius,
                         const int64_t* __restrict__ seg, int* __restrict__ fill, uint64_t* __restrict__ keys) {
  const int slot = blockIdx.y, lane = threadIdx.x & 31;
  const float* d = col + size_t(slot) * n_rows;
  uint64_t* out = keys + seg[slot];
  const int64_t step = int64_t(gridDim.x) * blockDim.x;
  for (int64_t i0 = int64_t(blockIdx.x) * blockDim.x; i0 < n_rows; i0 += step) {
    const int64_t i = i0 + threadIdx.x;
    const float v = i < n_rows ? d[i] : 0.f;
    const bool hit = i < n_rows && v <= radius && (mask == nullptr || mask[i] != 0);
    const uint32_t ballot = __ballot_sync(0xffffffffu, hit);
    if (ballot == 0u) continue;
    int base = 0;
    if (lane == 0) base = atomicAdd(fill + slot, __popc(ballot));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (hit) out[base + __popc(ballot & ((1u << lane) - 1u))] = make_key(v, uint32_t(i));
  }
}

// One CTA per query: its sorted keys keys[seg[q] ...] -> rows (global) and distances at [off[q], off[q + 1]).
__global__ void __launch_bounds__(256)
range_gather_kernel(const uint64_t* __restrict__ keys, const int64_t* __restrict__ seg, const int64_t* __restrict__ off,
                    int64_t row_base, int64_t* __restrict__ rows, float* __restrict__ dist) {
  const int q = blockIdx.x;
  const int64_t o = off[q], n = off[q + 1] - o;
  const uint64_t* src = keys + seg[q];
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    const uint64_t key = src[i];
    rows[o + i] = row_base + int64_t(key & 0xffffffffull);
    dist[o + i] = ord2f(uint32_t(key >> 32));
  }
}

}  // namespace fx
