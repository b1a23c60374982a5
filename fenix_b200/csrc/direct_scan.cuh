// direct_scan.cuh — the latency path: ONE launch answers a handful of queries over a small shard, exactly.
//
// A single query against a 100k x 128 shard (BASELINE C1) is 51 MB of fp32 rows that live in L2: the tensor-core
// pipeline (prep, sample prepass, threshold pick, filter, finish: six launches, ~55 us of device time for ~12 us of
// filter) is all fixed cost there. This kernel reads the fp32 rows themselves once (coalesced, eight lanes per row,
// three row chunks in flight per lane), accumulates q.x and |x|^2 in fp64 from exact fp32 products - the arithmetic of
// the finish kernel's rerank, in the same summation order, so the distances are bit-identical to the tensor-core
// path's - and parks the raw sums of up to DS_CAP_STEPS * 64 rows in shared memory. A flush turns them into (distance,
// row) keys with every lane busy (one row per thread), and every warp folds its 32 keys into a sorted list of its 32 R
// best held in registers (shuffle bitonic networks: no atomics, no key buffers, no thresholds to maintain). A tree over
// the warps' lists gives the CTA's k best; the last CTA to finish joins the per-CTA lists the same way and writes the
// result. No shadow, no certificate, no second launch. A small query block (<= 896 floats) travels in the kernel
// parameters and the results may be written straight to mapped pinned host memory, so fx_search issues no copies.
// Measured dead ends (B200, C1): queries read from mapped host memory (every CTA fetches them over PCIe: ~30 us per
// query), block-wide shared-memory bitonic sorts (17 us), finishing each row inside the scan loop (a sqrt + append chain
// per step that four lanes of 32 execute: 11-15 us of scan).
// Replaces index.py:162-168 (distance column + select_k + take indices) like the rest of the library; HBM/L2-bound
// byte work, deliberately kept off the tensor cores.
#pragma once
#include "common.cuh"
#include "exact_scan.cuh"

namespace fx {

constexpr int DS_THREADS = 512;          // 16 warps: 64 rows per CTA and step, three steps in flight
constexpr int DS_MAX_Q = 8;              // queries per search (four per launch)
constexpr int DS_LAUNCH_Q = 4;
constexpr int DS_MAX_K = 128;
constexpr int DS_ROWS_PER_STEP = DS_THREADS / 8;         // 8 lanes per row, one row per lane group and step
constexpr int DS_CAP_STEPS = 16;         // steps whose raw sums are parked in shared memory between flushes (at most)
constexpr int DS_MAX_PROBES = 512;       // posting lists one query may probe (LISTS mode; prefix sums in shared memory)
constexpr int DS_INLINE_FLOATS = 896;    // query floats carried in the kernel parameters (3.5 KB of the 4 KB parameter space)

struct DirectParams {
  const float* X; int64_t n_rows; int pitch; int dim; int64_t row_base;
  const float* Q;            // [n_q][dim] in device memory, or null: the queries are q_inline
  int n_q; int metric; int k;
  const uint8_t* mask;       // [n_rows] or null
  uint64_t* partial;         // [gridDim.x][n_q][k] sorted keys of every CTA
  unsigned int* ticket;      // zero on entry; the last CTA leaves it zero again
  int cap_steps;             // steps between flushes (1 .. DS_CAP_STEPS; shared-memory budget)
  int64_t* out_rows; float* out_dist;   // [n_q][k]; device memory or mapped pinned host memory
  // LISTS mode (batched IVF, fx_search_cells): blockIdx.y = query; the query scans only the rows of the posting lists it
  // probes. inv_rows: local rows grouped by cell, cell_off[c .. c + 1): cell c's slice of it, probes[q][n_probe]: the
  // query's cells (-1: none); ticket then points at one counter per query and partial is [query][cta][k]
  const int* inv_rows; const long long* cell_off; const int* probes; int n_probe;
  unsigned long long* done;  // mapped pinned host words or null: [1] = kernel time (ns), then [0] = seq once the results are in host memory
  unsigned long long seq;
  unsigned long long* dbg;   // FENIX_DEBUG_DIRECT: globaltimer stamps ([0..7] phases of the last CTA, [8 + cta] end of each CTA's scan) or null
  float q_inline[DS_INLINE_FLOATS];
};

// ---- warp-level sorted lists: 32 * R keys per warp, key idx = r * 32 + lane held in v[r] of that lane ----
// One compare-exchange step of the bitonic network (partner idx ^ STRIDE, ascending where (idx & SIZE) == 0). Strides
// >= 32 pair registers of the same lane, smaller ones are shuffles; every loop bound is a compile-time constant, so the
// lists stay in registers.
template <int R, int SIZE, int STRIDE>
__device__ __forceinline__ void warp_cmpx(uint64_t (&v)[R], int lane) {
  if constexpr (STRIDE >= 32) {
    constexpr int RS = STRIDE / 32;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      if ((r & RS) == 0) {
        const bool up = ((r * 32) & SIZE) == 0;
        const uint64_t a = v[r], b = v[r | RS];
        const uint64_t lo = a < b ? a : b, hi = a < b ? b : a;
        v[r] = up ? lo : hi; v[r | RS] = up ? hi : lo;
      }
    }
  } else {
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const uint64_t o = __shfl_xor_sync(0xffffffffu, v[r], STRIDE);
      const bool up = ((r * 32 + lane) & SIZE) == 0;
      const bool keep_min = ((lane & STRIDE) == 0) == up;
      v[r] = (keep_min == (v[r] < o)) ? v[r] : o;
    }
  }
}
template <int R, int SIZE, int STRIDE>
__device__ __forceinline__ void warp_stage(uint64_t (&v)[R], int lane) {   // strides STRIDE, STRIDE / 2, ..., 1 of one stage
  warp_cmpx<R, SIZE, STRIDE>(v, lane);
  if constexpr (STRIDE > 1) warp_stage<R, SIZE, STRIDE / 2>(v, lane);
}
template <int R, int SIZE>
__device__ __forceinline__ void warp_sort_from(uint64_t (&v)[R], int lane) {   // stages SIZE, 2 SIZE, ..., 32 R
  warp_stage<R, SIZE, SIZE / 2>(v, lane);
  if constexpr (SIZE < 32 * R) warp_sort_from<R, SIZE * 2>(v, lane);
}
template <int R>
__device__ __forceinline__ void warp_sort(uint64_t (&v)[R], int lane) { warp_sort_from<R, 2>(v, lane); }
// best (sorted) <- the 32 R smallest of best U other (both sorted ascending): elementwise minimum against the reversed
// other list is bitonic, one merge stage sorts it
template <int R>
__device__ __forceinline__ void warp_merge_keep_low(uint64_t (&best)[R], const uint64_t (&other)[R], int lane) {
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const uint64_t o = __shfl_sync(0xffffffffu, other[R - 1 - r], 31 - lane);
    best[r] = best[r] < o ? best[r] : o;
  }
  warp_stage<R, 32 * R, 16 * R>(best, lane);
}

// Tree over the warps' sorted lists (wl[warp][32 R], shared memory): after log2(warps) rounds wl[0] holds the CTA's
// 32 R smallest keys, sorted. All threads of the CTA call it (barriers inside); it ends with a barrier.
template <int R>
__device__ __forceinline__ void cta_join_lists(uint64_t* wl) {
  constexpr int L = 32 * R;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
  for (int span = 1; span < n_warps; span <<= 1) {
    if ((warp & (2 * span - 1)) == 0 && warp + span < n_warps) {
      uint64_t best[R], v[R];
#pragma unroll
      for (int r = 0; r < R; ++r) { best[r] = wl[warp * L + r * 32 + lane]; v[r] = wl[(warp + span) * L + r * 32 + lane]; }
      warp_merge_keep_low<R>(best, v, lane);
#pragma unroll
      for (int r = 0; r < R; ++r) wl[warp * L + r * 32 + lane] = best[r];
    }
    __syncthreads();
  }
}

__device__ __forceinline__ unsigned long long ds_now() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}

// LISTS (batched IVF): one query per CTA column (blockIdx.y), rows come from the query's probed posting lists.
template <int NQ, int R, bool LISTS = false>
__global__ void __launch_bounds__(DS_THREADS, 1)
knn_direct_kernel(DirectParams p) {
  static_assert(!LISTS || NQ == 1, "LISTS mode scans one query per CTA");
  unsigned long long t_staged = 0, t_scanned = 0, t_published = 0;
  const unsigned long long t_start = ds_now();
  extern __shared__ __align__(16) unsigned char smem_raw[];
  // double qs[NQ][pitch_q] (rows zero-padded to whole 128-float chunks) | u64 wl[NQ][warps][32 R] (the warps' sorted
  // lists) | double sums[cap_rows][NQ + 1] (|x|^2, q.x per query) | int rowid[cap_rows] (-1: masked / past the end)
  constexpr int L = 32 * R;
  constexpr int NW = DS_THREADS / 32;
  const int pitch_q = (p.pitch + 127) & ~127;
  const int cap_rows = p.cap_steps * DS_ROWS_PER_STEP;
  double* qs = reinterpret_cast<double*>(smem_raw);
  uint64_t* wl = reinterpret_cast<uint64_t*>(qs + size_t(NQ) * pitch_q);
  double* sums = reinterpret_cast<double*>(wl + size_t(NQ) * NW * L);
  int* rowid = reinterpret_cast<int*>(sums + size_t(cap_rows) * (NQ + 1));
  __shared__ double s_qq[NQ];
  __shared__ unsigned int s_last;
  __shared__ int s_pre[LISTS ? DS_MAX_PROBES + 1 : 1];          // LISTS: rows before posting list t of this query
  __shared__ long long s_lst[LISTS ? DS_MAX_PROBES : 1];        // LISTS: where list t starts in inv_rows
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int qbase = LISTS ? int(blockIdx.y) : 0;                // first query of this CTA
  const int nq_here = LISTS ? 1 : p.n_q;
  // lane = grp + 4 * sub: row `grp` of the warp's four, float4 slot `sub` of eight. A quarter-warp (the unit a 128-bit
  // shared-memory load is served in) then reads TWO query addresses, 64 contiguous bytes, instead of eight 32 B apart
  // (sub-major lanes: 8 wavefronts per load, the query reads alone cost ~6 us per query on C1).
  const int grp = lane & 3, sub = lane >> 2;

  for (int q = 0; q < NQ; ++q) {
    for (int d = tid; d < pitch_q; d += DS_THREADS) {
      float v = 0.f;
      if (q < nq_here && d < p.dim) v = p.Q != nullptr ? p.Q[size_t(qbase + q) * p.dim + d] : p.q_inline[q * p.dim + d];
      qs[size_t(q) * pitch_q + d] = double(v);
    }
  }
  for (int i = tid; i < NQ * NW * L; i += DS_THREADS) wl[i] = KEY_PAD;
  if constexpr (LISTS) {
    for (int t = tid; t < p.n_probe; t += DS_THREADS) {
      const int cell = p.probes[size_t(qbase) * p.n_probe + t];
      const long long lo = cell >= 0 ? p.cell_off[cell] : 0, hi = cell >= 0 ? p.cell_off[cell + 1] : 0;
      s_lst[t] = lo; s_pre[t + 1] = int(hi - lo);
    }
    __syncthreads();
    if (tid == 0) { s_pre[0] = 0; for (int t = 0; t < p.n_probe; ++t) s_pre[t + 1] += s_pre[t]; }
  }
  __syncthreads();
  if (warp < NQ) {   // |q|^2, summed as the finish kernel sums it (lane-strided, xor tree)
    double s = 0.0;
    const double* qv = qs + size_t(warp) * pitch_q;
    for (int d = lane; d < p.pitch; d += 32) s = fma(qv[d], qv[d], s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) s_qq[warp] = s;
  }
  __syncthreads();
  if (p.dbg != nullptr) t_staged = ds_now();

  // The scan is a stream of work items (row of this lane group, chunk of 128 floats of that row): every lane holds four
  // float4 of the item, three items rotate through registers so that the loads of items t + 1 and t + 2 are in flight
  // while item t is multiplied. Summation order per accumulator = the finish kernel's: j = sub, sub + 8, ... then the xor
  // tree over the 8 lanes.
  const int n4 = p.pitch >> 2;
  const int C = (n4 + 31) >> 5;                       // chunks per row
  const int64_t n_items = LISTS ? int64_t(s_pre[p.n_probe]) : p.n_rows;   // rows this CTA column scans
  const int64_t n_steps = (n_items + DS_ROWS_PER_STEP - 1) / DS_ROWS_PER_STEP;
  const int my_steps = int64_t(blockIdx.x) < n_steps ? int((n_steps - 1 - blockIdx.x) / gridDim.x) + 1 : 0;
  const int total = my_steps * C;
  int parked = 0;                                     // steps parked in `sums` since the last flush
  // one accumulator per float4 component and sum (four independent fp64 chains each): the library's canonical order,
  // see the finish kernel's rerank (tc_filter.cuh)
  double xa[4] = {0.0, 0.0, 0.0, 0.0}, qa[NQ][4];
#pragma unroll
  for (int q = 0; q < NQ; ++q) { qa[q][0] = 0.0; qa[q][1] = 0.0; qa[q][2] = 0.0; qa[q][3] = 0.0; }

  auto item_of = [&](int st) { return (int64_t(blockIdx.x) + int64_t(st) * gridDim.x) * DS_ROWS_PER_STEP + warp * 4 + grp; };
  // the shard row behind an item: the item itself, or (LISTS) entry `item` of the query's concatenated posting lists
  auto row_of = [&](int st) -> int64_t {
    const int64_t item = item_of(st);
    if constexpr (!LISTS) return item;
    if (item >= n_items) return p.n_rows;   // (past the end: not live)
    int lo = 0, hi = p.n_probe;             // last list t with s_pre[t] <= item
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (int64_t(s_pre[mid]) <= item) lo = mid; else hi = mid; }
    return int64_t(p.inv_rows[s_lst[lo] + (item - s_pre[lo])]);
  };
  auto load = [&](float4 (&x)[4], bool& live, int& rowreg, int st, int ch) {
    const int64_t row = st < my_steps ? row_of(st) : p.n_rows;
    rowreg = int(row);
    live = st < my_steps && row < p.n_rows;
    if (live && p.mask != nullptr) live = p.mask[row] != 0;
    const float4* xp = reinterpret_cast<const float4*>(p.X + size_t(live ? row : 0) * p.pitch);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int j = ch * 32 + sub + 8 * u;
      x[u] = (live && j < n4) ? __ldg(xp + j) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  // parked sums -> keys (one row per thread, every lane busy), every warp folds its 32 R keys into its sorted list
  auto flush = [&](int n_parked_steps) {
    __syncthreads();
    const int n_slots = n_parked_steps * DS_ROWS_PER_STEP;
    for (int q = 0; q < nq_here; ++q) {
      uint64_t best[R];
      uint64_t* mine = wl + (size_t(q) * NW + warp) * L;
#pragma unroll
      for (int r = 0; r < R; ++r) best[r] = mine[r * 32 + lane];
      const double qq = s_qq[q];
      for (int base = warp * L; base < n_slots; base += NW * L) {
        uint64_t v[R];
        bool any = false;
        const uint64_t worst = __shfl_sync(0xffffffffu, best[R - 1], 31);   // the list's largest entry
#pragma unroll
        for (int r = 0; r < R; ++r) {
          // (no divergence around the distance arithmetic: dead slots compute on slot 0 and are discarded)
          const int slot = base + r * 32 + lane;
          const bool in = slot < n_slots;
          const int sl = in ? slot : 0;
          const int row = rowid[sl];
          const uint64_t key = make_key(finish_distance(p.metric, qq, sums[size_t(sl) * (NQ + 1)], sums[size_t(sl) * (NQ + 1) + 1 + q]), uint32_t(row));
          v[r] = (in && row >= 0) ? key : KEY_PAD;
          any = any || v[r] < worst;
        }
        __syncwarp();
        if (!__any_sync(0xffffffffu, any)) continue;
        warp_sort<R>(v, lane);
        warp_merge_keep_low<R>(best, v, lane);
      }
#pragma unroll
      for (int r = 0; r < R; ++r) mine[r * 32 + lane] = best[r];
    }
    __syncthreads();
  };
  auto compute = [&](const float4 (&x)[4], bool live, int rowreg, int ch) {
    if (__any_sync(0xffffffffu, live)) {
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = ch * 32 + sub + 8 * u;           // (j >= n4: x is zero, the query row is zero-padded to whole chunks)
        const double a0 = x[u].x, a1 = x[u].y, a2 = x[u].z, a3 = x[u].w;
        xa[0] = fma(a0, a0, xa[0]); xa[1] = fma(a1, a1, xa[1]); xa[2] = fma(a2, a2, xa[2]); xa[3] = fma(a3, a3, xa[3]);
#pragma unroll
        for (int q = 0; q < NQ; ++q) {
          const double2* qp = reinterpret_cast<const double2*>(qs + size_t(q) * pitch_q + 4 * j);
          const double2 v0 = qp[0], v1 = qp[1];
          qa[q][0] = fma(a0, v0.x, qa[q][0]); qa[q][1] = fma(a1, v0.y, qa[q][1]);
          qa[q][2] = fma(a2, v1.x, qa[q][2]); qa[q][3] = fma(a3, v1.y, qa[q][3]);
        }
      }
    }
    if (ch != C - 1) return;
    // the row is complete: reduce over the group's 8 lanes and park the raw sums (lane `sub` stores q.x of query `sub`)
    const int slot = parked * DS_ROWS_PER_STEP + warp * 4 + grp;
    if (__any_sync(0xffffffffu, live)) {
      double xx = (xa[0] + xa[1]) + (xa[2] + xa[3]), qx[NQ];
#pragma unroll
      for (int q = 0; q < NQ; ++q) qx[q] = (qa[q][0] + qa[q][1]) + (qa[q][2] + qa[q][3]);
#pragma unroll
      for (int o = 16; o > 2; o >>= 1) {   // sub ^ 4, sub ^ 2, sub ^ 1: the finish kernel's tree
        xx += __shfl_xor_sync(0xffffffffu, xx, o);
#pragma unroll
        for (int q = 0; q < NQ; ++q) qx[q] += __shfl_xor_sync(0xffffffffu, qx[q], o);
      }
      double dq = qx[0];
#pragma unroll
      for (int q = 1; q < NQ; ++q) { if (sub == q) dq = qx[q]; }
      if (sub < NQ) sums[size_t(slot) * (NQ + 1) + 1 + sub] = dq;
      if (sub == 0) sums[size_t(slot) * (NQ + 1)] = xx;
    }
    if (sub == 0) rowid[slot] = live ? rowreg : -1;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      xa[e] = 0.0;
#pragma unroll
      for (int q = 0; q < NQ; ++q) qa[q][e] = 0.0;
    }
    if (++parked == p.cap_steps) { flush(parked); parked = 0; }
  };
  {
    float4 x0[4], x1[4], x2[4];
    bool l0 = false, l1 = false, l2 = false;
    int r0 = 0, r1 = 0, r2 = 0;                         // shard row of the item in each buffer
    int ls = 0, lc = 0, cc = 0;                         // next item to load: (step, chunk); chunk of the next item to compute
    auto adv = [&](int& st, int& ch) { if (++ch == C) { ch = 0; ++st; } };
    auto advc = [&](int& ch) { if (++ch == C) ch = 0; };
    load(x0, l0, r0, ls, lc); adv(ls, lc);
    load(x1, l1, r1, ls, lc); adv(ls, lc);
    for (int t = 0; t < total; t += 3) {
      load(x2, l2, r2, ls, lc); adv(ls, lc);
      compute(x0, l0, r0, cc); advc(cc);
      if (t + 1 < total) {
        load(x0, l0, r0, ls, lc); adv(ls, lc);
        compute(x1, l1, r1, cc); advc(cc);
      }
      if (t + 2 < total) {
        load(x1, l1, r1, ls, lc); adv(ls, lc);
        compute(x2, l2, r2, cc); advc(cc);
      }
    }
  }
  if (p.dbg != nullptr) { t_scanned = ds_now(); if (tid == 0) p.dbg[8 + blockIdx.x] = t_scanned; }
  flush(parked);   // (barriers on both sides; also when nothing is parked)

  // ---- this CTA's k best per query, published ----
  // published lists: [cta][query][k]; LISTS: [query][cta][k]
  uint64_t* const part = LISTS ? p.partial + size_t(qbase) * gridDim.x * p.k : p.partial;
  const int part_nq = LISTS ? 1 : p.n_q;
  for (int q = 0; q < nq_here; ++q) {
    uint64_t* w0 = wl + size_t(q) * NW * L;
    cta_join_lists<R>(w0);
    for (int i = tid; i < p.k; i += DS_THREADS) part[(size_t(blockIdx.x) * part_nq + q) * p.k + i] = w0[i];
  }
  __threadfence();
  __syncthreads();
  if (p.dbg != nullptr) t_published = ds_now();
  unsigned int* const ticket = p.ticket + (LISTS ? qbase : 0);
  if (tid == 0) s_last = (atomicAdd(ticket, 1u) == gridDim.x - 1) ? 1u : 0u;
  __syncthreads();
  if (s_last == 0u) return;
  __threadfence();
  unsigned long long t_ticket = 0, t_joined = 0;
  if (p.dbg != nullptr) t_ticket = ds_now();

  // ---- the last CTA joins gridDim.x sorted lists of k keys per query: every warp folds chunks of 32 R keys (the next
  // chunk's loads in flight while one is sorted), then the same tree ----
  const int n_keys = int(gridDim.x) * p.k;
  const unsigned k_magic = p.k > 1 ? unsigned((0x100000000ull + unsigned(p.k) - 1u) / unsigned(p.k)) : 0u;   // i / k = umulhi(i, magic), i < 2^15
  for (int q = 0; q < nq_here; ++q) {
    auto get = [&](int i) {
      if (i >= n_keys) return KEY_PAD;
      const int cta = p.k > 1 ? int(__umulhi(unsigned(i), k_magic)) : i, e = i - cta * p.k;
      return __ldcg(part + (size_t(cta) * part_nq + q) * p.k + e);
    };
    uint64_t best[R], v[R], nv[R];
#pragma unroll
    for (int r = 0; r < R; ++r) { best[r] = KEY_PAD; v[r] = get(warp * L + r * 32 + lane); }
    for (int c0 = warp * L; c0 < n_keys; c0 += NW * L) {
#pragma unroll
      for (int r = 0; r < R; ++r) nv[r] = get(c0 + NW * L + r * 32 + lane);
      warp_sort<R>(v, lane);
      warp_merge_keep_low<R>(best, v, lane);
#pragma unroll
      for (int r = 0; r < R; ++r) v[r] = nv[r];
    }
    uint64_t* w0 = wl + size_t(q) * NW * L;
#pragma unroll
    for (int r = 0; r < R; ++r) w0[warp * L + r * 32 + lane] = best[r];
    __syncthreads();
    cta_join_lists<R>(w0);
    for (int i = tid; i < p.k; i += DS_THREADS) {
      const uint64_t key = w0[i];
      const bool pad = key == KEY_PAD;
      p.out_rows[size_t(qbase + q) * p.k + i] = pad ? int64_t(-1) : p.row_base + int64_t(key & 0xffffffffull);
      p.out_dist[size_t(qbase + q) * p.k + i] = pad ? __int_as_float(0x7f800000) : ord2f(uint32_t(key >> 32));
    }
  }
  if (p.dbg != nullptr) t_joined = ds_now();
  if (tid == 0) *ticket = 0u;
  if (p.done != nullptr) {
    // the host spins on done[0] instead of waiting for the stream (saves the driver's completion latency): results first,
    // system-wide fence, then the sequence number - writes of one GPU reach host memory in order
    if (tid == 0) { volatile unsigned long long* d = p.done; d[1] = ds_now() - t_start; }
    __threadfence_system();
    __syncthreads();
    if (tid == 0) { volatile unsigned long long* d = p.done; d[0] = p.seq; }
  }
  if (p.dbg != nullptr && tid == 0) {
    p.dbg[0] = t_start; p.dbg[1] = t_staged; p.dbg[2] = t_scanned; p.dbg[3] = t_published; p.dbg[4] = t_ticket; p.dbg[5] = t_joined;
    p.dbg[6] = ds_now(); p.dbg[7] = gridDim.x;
  }
}

// ---- host side ----
struct DirectPlan { bool ok = false; int nq_t = 0; int r = 0; int grid = 0; int cap_steps = 0; size_t smem = 0; size_t partial_bytes = 0; };

// Shapes the kernel takes: a handful of queries, k <= 128, queries + the warps' lists + at least one step of parked
// sums within shared memory.
inline DirectPlan direct_plan(int64_t n_rows, int pitch, int64_t n_q, int k, int sm_count) {
  DirectPlan pl;
  if (n_rows < 1 || n_rows > (int64_t(1) << 31) - 1 || n_q < 1 || n_q > DS_MAX_Q || k < 1 || k > DS_MAX_K) return pl;
  pl.nq_t = n_q <= 1 ? 1 : n_q <= 2 ? 2 : 4;     // more than four queries: two launches (the caller splits the batch)
  pl.r = k <= 32 ? 1 : k <= 64 ? 2 : 4;
  const int64_t n_steps = (n_rows + DS_ROWS_PER_STEP - 1) / DS_ROWS_PER_STEP;
  pl.grid = int(std::max<int64_t>(1, std::min<int64_t>(sm_count, n_steps)));
  const size_t fixed = size_t(pl.nq_t) * ((pitch + 127) & ~127) * 8 + size_t(pl.nq_t) * (DS_THREADS / 32) * 32 * pl.r * 8;
  const size_t per_step = size_t(DS_ROWS_PER_STEP) * ((pl.nq_t + 1) * 8 + 4);
  const size_t budget = size_t(200) * 1024;
  if (fixed + per_step > budget) return pl;
  const int64_t steps_per_cta = (n_steps + pl.grid - 1) / pl.grid;
  pl.cap_steps = int(std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(DS_CAP_STEPS, steps_per_cta), int64_t((budget - fixed) / per_step))));
  pl.smem = fixed + per_step * pl.cap_steps + 16;
  pl.partial_bytes = size_t(pl.grid) * n_q * k * 8;
  pl.ok = true;
  return pl;
}

// More than 48 KB of dynamic shared memory needs the opt-in attribute; it is set at the launch that needs it (wide rows,
// several queries with k > 64) rather than for all 12 instantiations at fx_init, which cost a second of module loading.
template <typename K>
inline void ds_launch(K kernel, dim3 grid, size_t smem, cudaStream_t stream, const DirectParams& p) {
  if (smem > size_t(48) * 1024) cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  kernel<<<grid, DS_THREADS, smem, stream>>>(p);
}

template <int NQ>
inline void direct_launch_q(const DirectPlan& pl, const DirectParams& p, cudaStream_t stream) {
  const dim3 grid(pl.grid);
  switch (pl.r) {
    case 1: ds_launch(knn_direct_kernel<NQ, 1>, grid, pl.smem, stream, p); break;
    case 2: ds_launch(knn_direct_kernel<NQ, 2>, grid, pl.smem, stream, p); break;
    default: ds_launch(knn_direct_kernel<NQ, 4>, grid, pl.smem, stream, p); break;
  }
}
inline cudaError_t direct_launch(const DirectPlan& pl, const DirectParams& p, cudaStream_t stream) {
  switch (pl.nq_t) {
    case 1: direct_launch_q<1>(pl, p, stream); break;
    case 2: direct_launch_q<2>(pl, p, stream); break;
    default: direct_launch_q<4>(pl, p, stream); break;
  }
  return cudaGetLastError();
}

// ---- LISTS mode (batched IVF): grid = (CTAs per query, queries) ----
struct CellsPlan { bool ok = false; int r = 0; int ctas = 0; int cap_steps = 0; size_t smem = 0; size_t partial_bytes = 0; };

// max_items: the longest concatenated posting list any query of the batch scans
inline CellsPlan cells_plan(int pitch, int64_t n_q, int k, int n_probe, int64_t max_items, int sm_count) {
  CellsPlan pl;
  if (n_q < 1 || n_q > 65535 || k < 1 || k > DS_MAX_K || n_probe < 1 || n_probe > DS_MAX_PROBES) return pl;
  pl.r = k <= 32 ? 1 : k <= 64 ? 2 : 4;
  const int64_t n_steps = std::max<int64_t>(1, (max_items + DS_ROWS_PER_STEP - 1) / DS_ROWS_PER_STEP);
  // enough CTAs to fill the GPU twice over, but at least four steps each (a CTA's fixed cost is ~3 us)
  pl.ctas = int(std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>((2 * int64_t(sm_count) + n_q - 1) / n_q, (n_steps + 3) / 4), sm_count)));
  const size_t fixed = size_t((pitch + 127) & ~127) * 8 + size_t(DS_THREADS / 32) * 32 * pl.r * 8;
  const size_t per_step = size_t(DS_ROWS_PER_STEP) * (2 * 8 + 4);
  const size_t budget = size_t(200) * 1024;
  if (fixed + per_step > budget) return pl;
  const int64_t steps_per_cta = (n_steps + pl.ctas - 1) / pl.ctas;
  pl.cap_steps = int(std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(DS_CAP_STEPS, steps_per_cta), int64_t((budget - fixed) / per_step))));
  pl.smem = fixed + per_step * pl.cap_steps + 16;
  pl.partial_bytes = size_t(n_q) * pl.ctas * k * 8;
  pl.ok = true;
  return pl;
}

template <int R>
inline void cells_launch_r(const CellsPlan& pl, const DirectParams& p, int n_q, cudaStream_t stream) {
  const dim3 grid(pl.ctas, n_q);
  ds_launch(knn_direct_kernel<1, R, true>, grid, pl.smem, stream, p);
}
inline cudaError_t cells_launch(const CellsPlan& pl, const DirectParams& p, int n_q, cudaStream_t stream) {
  switch (pl.r) {
    case 1: cells_launch_r<1>(pl, p, n_q, stream); break;
    case 2: cells_launch_r<2>(pl, p, n_q, stream); break;
    default: cells_launch_r<4>(pl, p, n_q, stream); break;
  }
  return cudaGetLastError();
}

}  // namespace fx
