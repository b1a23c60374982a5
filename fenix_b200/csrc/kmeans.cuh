// kmeans.cuh — mini-batch k-means steps of IVF codebook training (fx_train_codebooks; DESIGN.md §4.11).
//
// One step trains every codebook j on its own sample of `batch` rows with three launches:
//   km_assign_kernel  nearest codeword of every sample row: fp64 sums of fp32 products, summed over d in ascending order,
//                     the reference-convention distance rounded once to fp32 (finish_distance), then the smallest
//                     (distance bits, codeword) key. Codeword ranges split over blocks meet in an atomicMin on the key,
//                     which is order-independent, so the result does not depend on scheduling.
//   km_bucket_kernel  counting sort of the sample by codeword, stable: each codeword's rows stay in sample order.
//   km_update_kernel  per codeword: fp64 sum of the old codeword, then its rows in sample order, one fp64 division by
//                     1 + count, one rounding to fp32. Cosine: the old codeword and the rows are normalised in fp64
//                     first and the mean is normalised in fp64 before the rounding.
// Every sum has a fixed order, so two runs on the same input give the same bits.
#pragma once
#include <cub/block/block_reduce.cuh>
#include <cub/block/block_scan.cuh>

#include "common.cuh"

namespace fx {

constexpr int KM_TR = 64;        // sample rows per assignment block
constexpr int KM_TC = 64;        // codewords per shared-memory tile
constexpr int KM_DK = 32;        // coordinates per tile
constexpr int KM_THREADS = 256;  // 16 x 16 threads, 4 x 4 (row, codeword) pairs each
constexpr int KM_BUCKET_THREADS = 256;
constexpr int KM_UPDATE_THREADS = 128;

struct KmParams {
  const float* X;          // sample rows: X + idx[i] * pitch
  int64_t pitch;
  const int64_t* idx;      // [n_books * batch] rows of this step, codebook j's at [j * batch, (j + 1) * batch)
  float* books;            // [n_books][k][dim]
  int dim, k, batch, metric;
  int cw_per_block;        // codewords per assignment block (a multiple of KM_TC)
  unsigned long long* keys;  // [n_books * batch] (distance, codeword) keys, KEY_PAD between steps
  double* xx;              // [n_books * batch] squared norms of the sample rows
  int* off;                // [n_books][k + 1] start of every codeword's slice of `order`
  int* cur;                // [n_books][k] fill cursors
  int* order;              // [n_books][batch] sample positions grouped by codeword, sample order within a codeword
};

__global__ void __launch_bounds__(KM_THREADS) km_assign_kernel(KmParams p) {
  __shared__ double As[KM_DK][KM_TR + 1];   // sample rows, transposed
  __shared__ double Bs[KM_DK][KM_TC + 1];   // codewords, transposed
  __shared__ double xs[KM_TR], cs[KM_TC];
  const int j = blockIdx.z, r0 = blockIdx.x * KM_TR;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int sd = tid & 31, sr = tid >> 5;   // staging: coordinate sd of tile rows sr + 8 i
  const int64_t* idx = p.idx + int64_t(j) * p.batch;
  const float* book = p.books + int64_t(j) * p.k * p.dim;
  const float* rowp[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = r0 + sr + 8 * i;
    rowp[i] = r < p.batch ? p.X + idx[r] * p.pitch : nullptr;
  }
  unsigned long long best[4] = {KEY_PAD, KEY_PAD, KEY_PAD, KEY_PAD};
  const int c_begin = blockIdx.y * p.cw_per_block, c_end = min(p.k, c_begin + p.cw_per_block);
  for (int c0 = c_begin; c0 < c_end; c0 += KM_TC) {
    double acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int t = 0; t < 4; ++t) acc[i][t] = 0.0;
    double nacc = 0.0;   // tid < 64: squared norm of row tid (first tile only); 64 <= tid < 128: of codeword tid - 64
    for (int d0 = 0; d0 < p.dim; d0 += KM_DK) {
      const int d = d0 + sd, nd = min(KM_DK, p.dim - d0);
      __syncthreads();
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int c = c0 + sr + 8 * i;
        As[sd][sr + 8 * i] = (rowp[i] && d < p.dim) ? double(rowp[i][d]) : 0.0;
        Bs[sd][sr + 8 * i] = (c < c_end && d < p.dim) ? double(book[int64_t(c) * p.dim + d]) : 0.0;
      }
      __syncthreads();
      if (tid < KM_TR) {
        if (c0 == c_begin)
          for (int e = 0; e < nd; ++e) nacc = fma(As[e][tid], As[e][tid], nacc);
      } else if (tid < KM_TR + KM_TC) {
        for (int e = 0; e < nd; ++e) nacc = fma(Bs[e][tid - KM_TR], Bs[e][tid - KM_TR], nacc);
      }
      for (int e = 0; e < nd; ++e) {
        double a[4], b[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = As[e][ty + 16 * i];
#pragma unroll
        for (int t = 0; t < 4; ++t) b[t] = Bs[e][tx + 16 * t];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int t = 0; t < 4; ++t) acc[i][t] = fma(a[i], b[t], acc[i][t]);
      }
    }
    if (tid < KM_TR) {
      if (c0 == c_begin) xs[tid] = nacc;
    } else if (tid < KM_TR + KM_TC) {
      cs[tid - KM_TR] = nacc;
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int c = c0 + tx + 16 * t;
        if (c < c_end) {
          const unsigned long long key = make_key(finish_distance(p.metric, xs[ty + 16 * i], cs[tx + 16 * t], acc[i][t]),
                                                  uint32_t(c));
          best[i] = key < best[i] ? key : best[i];
        }
      }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
      const unsigned long long other = __shfl_xor_sync(0xffffffffu, best[i], o);
      best[i] = other < best[i] ? other : best[i];
    }
    const int r = r0 + ty + 16 * i;
    if (tx == 0 && r < p.batch) atomicMin(&p.keys[int64_t(j) * p.batch + r], best[i]);
  }
  if (blockIdx.y == 0 && tid < KM_TR && r0 + tid < p.batch) p.xx[int64_t(j) * p.batch + r0 + tid] = xs[tid];
}

// One block per codebook: counts per codeword, their exclusive scan, then a stable scatter by one warp (rows in sample
// order, __match_any_sync ranks the lanes that share a codeword). Resets the keys for the next step.
__global__ void __launch_bounds__(KM_BUCKET_THREADS) km_bucket_kernel(KmParams p) {
  using Scan = cub::BlockScan<int, KM_BUCKET_THREADS>;
  __shared__ typename Scan::TempStorage scan_tmp;
  __shared__ int carry;
  const int j = blockIdx.x, tid = threadIdx.x;
  unsigned long long* keys = p.keys + int64_t(j) * p.batch;
  int* off = p.off + int64_t(j) * (p.k + 1);
  int* cur = p.cur + int64_t(j) * p.k;
  int* order = p.order + int64_t(j) * p.batch;
  for (int c = tid; c <= p.k; c += KM_BUCKET_THREADS) off[c] = 0;
  if (tid == 0) carry = 0;
  __syncthreads();
  for (int r = tid; r < p.batch; r += KM_BUCKET_THREADS) atomicAdd(&off[int(keys[r] & 0xffffffffu) + 1], 1);
  __syncthreads();
  for (int c0 = 0; c0 < p.k; c0 += KM_BUCKET_THREADS) {
    const int c = c0 + tid;
    int v = c < p.k ? off[c + 1] : 0, total;
    Scan(scan_tmp).InclusiveSum(v, v, total);
    if (c < p.k) off[c + 1] = v + carry;
    __syncthreads();
    if (tid == 0) carry += total;
    __syncthreads();
  }
  for (int c = tid; c < p.k; c += KM_BUCKET_THREADS) cur[c] = off[c];
  __syncthreads();
  if (tid >= 32) return;
  for (int r0 = 0; r0 < p.batch; r0 += 32) {
    const int r = r0 + tid;
    const bool ok = r < p.batch;
    const int c = ok ? int(keys[r] & 0xffffffffu) : -1;
    const unsigned peers = __match_any_sync(0xffffffffu, c);
    const int rank = __popc(peers & ((1u << tid) - 1u));
    if (ok) {
      order[cur[c] + rank] = r;
      keys[r] = KEY_PAD;
    }
    __syncwarp();
    if (ok && rank == 0) cur[c] += __popc(peers);
    __syncwarp();
  }
}

__device__ __forceinline__ double km_block_sum(double v, double* red) {
  using Reduce = cub::BlockReduce<double, KM_UPDATE_THREADS>;
  auto& tmp = *reinterpret_cast<typename Reduce::TempStorage*>(red);
  const double s = Reduce(tmp).Sum(v);
  __syncthreads();
  if (threadIdx.x == 0) red[0] = s;
  __syncthreads();
  const double out = red[0];
  __syncthreads();
  return out;
}

// One block per (codeword, codebook). Dynamic shared memory: dim doubles (the new codeword before rounding).
__global__ void __launch_bounds__(KM_UPDATE_THREADS) km_update_kernel(KmParams p) {
  extern __shared__ double m[];
  __shared__ __align__(16) double red[sizeof(typename cub::BlockReduce<double, KM_UPDATE_THREADS>::TempStorage) / 8 + 2];
  const int c = blockIdx.x, j = blockIdx.y, tid = threadIdx.x;
  const bool cosine = p.metric == 1;
  float* cw = p.books + (int64_t(j) * p.k + c) * p.dim;
  const int* off = p.off + int64_t(j) * (p.k + 1);
  const int* order = p.order + int64_t(j) * p.batch;
  const int64_t* idx = p.idx + int64_t(j) * p.batch;
  const int s0 = off[c], s1 = off[c + 1];
  double nc = 1.0;
  if (cosine) {
    double s = 0.0;
    for (int d = tid; d < p.dim; d += KM_UPDATE_THREADS) s = fma(double(cw[d]), double(cw[d]), s);
    nc = fmax(sqrt(km_block_sum(s, red)), 1e-12);
  }
  for (int d = tid; d < p.dim; d += KM_UPDATE_THREADS) m[d] = cosine ? double(cw[d]) / nc : double(cw[d]);
  for (int i = s0; i < s1; ++i) {
    const int r = order[i];
    const float* row = p.X + idx[r] * p.pitch;
    if (cosine) {
      const double nr = fmax(sqrt(p.xx[int64_t(j) * p.batch + r]), 1e-12);
      for (int d = tid; d < p.dim; d += KM_UPDATE_THREADS) m[d] += double(row[d]) / nr;
    } else {
      for (int d = tid; d < p.dim; d += KM_UPDATE_THREADS) m[d] += double(row[d]);
    }
  }
  const double div = 1.0 + double(s1 - s0);
  double s = 0.0;
  for (int d = tid; d < p.dim; d += KM_UPDATE_THREADS) {
    m[d] = m[d] / div;
    s = fma(m[d], m[d], s);
  }
  if (cosine) {
    const double nm = fmax(sqrt(km_block_sum(s, red)), 1e-12);
    for (int d = tid; d < p.dim; d += KM_UPDATE_THREADS) cw[d] = float(m[d] / nm);
  } else {
    for (int d = tid; d < p.dim; d += KM_UPDATE_THREADS) cw[d] = float(m[d]);
  }
}

// Rows of one shard into a dense staging buffer (multi-device training): out[i] = X[rows[i]], pitch floats each.
__global__ void km_gather_kernel(const float* X, int64_t pitch, const int64_t* rows, int64_t n, float* out) {
  for (int64_t i = blockIdx.x; i < n; i += gridDim.x) {
    const float* src = X + rows[i] * pitch;
    float* dst = out + i * pitch;
    for (int64_t d = threadIdx.x; d < pitch; d += blockDim.x) dst[d] = src[d];
  }
}

}  // namespace fx
