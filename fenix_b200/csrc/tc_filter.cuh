// tc_filter.cuh - the tensor-core path: tcgen05/TMEM GEMM with a fused threshold-filter epilogue (no distance
// matrix ever reaches HBM), followed by an fp64 rerank + certificate. DESIGN.md section 4 is the narrative.
//
//   knn_prep_kernel        pads queries to whole tile pairs (fp32 and bf16 copies), resets per-query state
//   knn_tc_filter_kernel   streaming kernel (any row width): persistent, one CTA per SM
//                            warp 0     TMA producer  (cp.async.bulk.tensor, 128B swizzle, 4 stages of query + corpus blocks)
//                            warp 1     MMA issuer    (tcgen05.mma M=128 N=256, kind::f16 on the bf16 shadow or kind::tf32
//                                                      on the raw rows, fp32 accumulators in TMEM, double-buffered)
//                            warp 2     TMEM allocator
//                            warps 4-11 epilogue      (epi_tile / epi_tighten below)
//                          PAIR 1: CTA pairs (cta_group::2); PAIR 2: the same over the int8 shadow with the query tiles resident
//   knn_rq_filter_kernel   resident-query kernel (narrow rows, >= 2 query tiles): two query tiles stay in shared memory,
//                          128-row corpus blocks stream through a deep ring and feed two MMAs each (warps 1 and 3 issue)
//   MODE 2 of both + knn_tc_tau0_kernel   threshold prepass over a strided sample (narrow rows)
//   knn_tc_finish_kernel   one CTA per query: top-K' of the surviving candidates by approximate score, exact
//                          (fp64-accumulated) rerank, (distance,row) sort, certificate
//   refine_*_kernel        preset-threshold refinement of flagged queries
//
// Exactness argument (FX_PREC_FP32): every corpus row that is NOT a candidate has approximate score s^ <= T;
// |s^ - s| <= E (rigorous bf16 / TF32 rounding bound from |q|, max|x|, D); so its exact distance is >= f(T + E). If the
// k-th reranked distance is strictly below that bound the top-k is proven exact; otherwise the query is flagged and
// settled by the re-run / refinement tiers (fenix_knn.cu), in the last resort by the fp64 scan (exact_scan.cuh).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdlib>
#include <cstring>
#include <string>

#include "common.cuh"

namespace fx {

// ---------------------------------------------------------------------------------------------
// tile configuration
// ---------------------------------------------------------------------------------------------
constexpr int TC_BM = 128;                 // queries per CTA tile (UMMA M, TMEM lanes)
constexpr int TC_BN = 256;                 // corpus rows per accumulator (UMMA N)
constexpr int TC_BK = 32;                  // fp32 elements per k-block = 128 B = one swizzle row
constexpr int TC_UMMA_K = 8;               // kind::tf32: 32 bytes of K per instruction
constexpr int TC_STAGES = 4;
constexpr int TC_ACC_STAGES = 2;           // 2 x 256 TMEM columns = all 512
constexpr int TC_SPLIT = 2;                // two epilogue warps per TMEM lane quadrant, 128 accumulator columns each
constexpr int TC_EPI_UNROLL = 2;          // unroll factor of the epilogue's chunk-pair loop (1 = rolled, 2 = all four chunks)
constexpr int TC_EPI_WARPS = 4 * TC_SPLIT; // 4 warps cover the 128 TMEM lanes; TC_SPLIT groups split the columns
constexpr int TC_THREADS = 32 * (4 + TC_EPI_WARPS);
constexpr int TC_EPI_FIRST_WARP = 4;
constexpr int TC_HALF_COLS = TC_BN / TC_SPLIT;   // columns per epilogue warp group ("part")
constexpr int TC_SLOTS = TC_SPLIT * TC_BM;       // candidate buffers per unit
constexpr int TC_CW = 32;                  // accumulator columns per tcgen05.ld in the epilogue
constexpr uint32_t TC_A_BYTES = TC_BM * TC_BK * 4;   // 16 KB
constexpr uint32_t TC_B_BYTES = TC_BN * TC_BK * 4;   // 32 KB
constexpr uint32_t TC_STAGE_BYTES = TC_A_BYTES + TC_B_BYTES;
constexpr uint32_t TC_NORM_BYTES = TC_BN * 4;        // per accumulator stage
constexpr uint32_t TC_SMEM_BYTES = 1024 /*align slack*/ + TC_STAGES * TC_STAGE_BYTES +
                                   TC_ACC_STAGES * TC_NORM_BYTES + 512 /*barriers*/;
constexpr int TC2_STAGES = 6;               // CTA-pair kernel: stages of (query k-block, HALF a corpus k-block), 32 KB each
constexpr uint32_t TC2_B_BYTES = TC_B_BYTES / 2;
constexpr uint32_t TC2_STAGE_BYTES = TC_A_BYTES + TC2_B_BYTES;
constexpr uint32_t TC2_SMEM_BYTES = 1024 /*align slack*/ + TC2_STAGES * TC2_STAGE_BYTES +
                                    TC_ACC_STAGES * TC_NORM_BYTES + 512 /*barriers*/;
// Resident-query CTA-pair kernel (int8 shadow): each CTA keeps its whole query tile (n_kblocks blocks of 16 KB) for a
// unit, and the ring carries only corpus half blocks (16 KB); the ring gets whatever shared memory the query tile leaves.
constexpr int TC3_MAX_STAGES = 12;
constexpr uint32_t TC3_SMEM_MAX = 227 * 1024;
constexpr uint32_t TC3_FIXED_BYTES = 1024 /*align slack*/ + TC_ACC_STAGES * TC_NORM_BYTES + 512 /*barriers*/;
constexpr int TC3_MIN_STAGES = 4;
inline int tc3_stages(int n_kblocks) {
  const int s = (int(TC3_SMEM_MAX) - int(TC3_FIXED_BYTES) - n_kblocks * int(TC_A_BYTES)) / int(TC2_B_BYTES);
  return s < TC3_MAX_STAGES ? s : TC3_MAX_STAGES;
}
inline uint32_t tc3_smem_bytes(int n_kblocks) {
  return TC3_FIXED_BYTES + uint32_t(n_kblocks) * TC_A_BYTES + uint32_t(tc3_stages(n_kblocks)) * TC2_B_BYTES;
}
static_assert(TC3_FIXED_BYTES + 6 * TC_A_BYTES + 7 * TC2_B_BYTES <= TC3_SMEM_MAX, "D = 768 (6 int8 k-blocks): 7 corpus stages");
static_assert(TC3_FIXED_BYTES + 9 * TC_A_BYTES + TC3_MIN_STAGES * TC2_B_BYTES <= TC3_SMEM_MAX, "D <= 1152: 4 corpus stages");
constexpr size_t TC_HDR_BYTES = 256;        // scratch header (word 0: flagged-query counter of the last finish launch)
constexpr int TC_MAX_WAVES = 4;            // units per CTA at most (bounds the candidate-buffer scratch)
constexpr uint32_t ORD_NEG_INF = 0x007fffffu;  // f2ord(-inf)
// Preset threshold of a query the filter cannot settle (admission_threshold): below every ordered float (a NaN as a
// float, so the float epilogues admit nothing); the range search sends such queries to the exact scan.
constexpr uint32_t ORD_SCAN = 0u;

// Geometry of a bf16 shadow of a [n][dim] shard (see to_bf16_tiled_kernel). The four augmented columns - three terms
// of -|x|^2/2 and the row's error weight |x| - sit right after the data when the last 64-column k-block has room for
// them; otherwise (dim % 64 == 0 or > 60) they get one block per tile in a separate region behind the data blocks, so
// that searches that do not need them (inner product over rows of similar norm, cosine) stream exactly the data
// blocks, back to back.
constexpr int TC_AUG_COLS = 4;
struct ShadowGeom {
  int n_kb_data;     // 64-column k-blocks that hold data, per tile
  int aug_col;       // query / shadow column of the first augmented term (dim, or 64 * n_kb_data when separate)
  bool aug_separate;
  int pitch_q;       // elements per row of the bf16 query matrix (multiple of 64, covers the augmented columns)
};
inline ShadowGeom shadow_geom(int dim) {
  ShadowGeom g;
  g.n_kb_data = (dim + 63) / 64;
  const int used = dim - 64 * (g.n_kb_data - 1);      // columns of the last data block that hold data
  g.aug_separate = used + TC_AUG_COLS > 64;
  g.aug_col = g.aug_separate ? 64 * g.n_kb_data : dim;
  g.pitch_q = 64 * ((g.aug_col + TC_AUG_COLS + 63) / 64);   // whole 128-byte k-blocks: query tile rows stay 128 B aligned for TMA
  return g;
}

// The int8 normalised shadow (cosine, operand kind 2) and its quantised queries. ONE format, used by the shadow builder,
// the query quantiser, the filter epilogue and the certificate: a vector v (a corpus row or a query) is normalised in
// fp64, v^ = v / max(|v|, 1e-12) (the rerank's eps), and quantised with a scale S shared by its group (a 256-row tile of
// the shard, or the query alone), S = 127 / max |v^_i| over the group:  v~ = clamp(rint(S v^_i), -127, 127). With the
// residuals r_x = x^ - x~/S_t and r_q = q^ - q~/S_q, exactly
//     cos(q, x) = q~.x~ / (S_t S_q) + (q~/S_q).r_x + r_q.x^   <=   acc / (S_t S_q) + a_q E_t + e_q
// where acc = q~.x~ (exact in the int32 accumulator), E_t = max |r_x| over the tile's rows, a_q = |q~| / S_q and
// e_q = |r_q| (|x^| <= 1), all rounded up. So the filter score of a row is a certified UPPER bound of its exact cosine.
// Rows: 128 int8 columns per k-block (128 B, as a bf16 k-block), tiles of 256 rows; a tile's (S_t, E_t) is a float2.
constexpr int I8_KB = 128;                 // int8 columns per k-block
inline int i8_n_kb(int dim) { return (dim + I8_KB - 1) / I8_KB; }
__host__ __device__ __forceinline__ float i8_scale(double max_abs) { return max_abs > 0.0 ? float(127.0 / max_abs) : 1.f; }
__device__ __forceinline__ int i8_quant(double v, float scale) {
  return int(fmin(fmax(rint(v * double(scale)), -127.0), 127.0));
}
// acc -> the row's certified upper bound (ae = a_q E_t + e_q, padded for the rounding of this expression)
__device__ __forceinline__ float i8_upper(int acc, double inv_ss, double ae) { return __double2float_ru(fma(double(acc), inv_ss, ae)); }
// Integer admission threshold of one (query, tile): every acc whose upper bound can exceed tau is above it (the margin
// covers the fp32 rounding of the bound). Never below I8_FLOOR, so a masked row (row term I8_MASKED) can never pass.
constexpr int I8_FLOOR = -(1 << 29);       // below every unmasked acc: |acc| <= 127^2 D < 2^28 for D <= 16384
constexpr int I8_MASKED = -(1 << 30);
__device__ __forceinline__ int i8_threshold(float tau, double ss, double ae) {
  const double x = (double(tau) - ae) * ss - ss * 0x1p-21 - 2.0;
  return x >= 2147483647.0 ? 0x7fffffff : (x > double(I8_FLOOR) ? int(floor(x)) : I8_FLOOR);
}

// Tuning options. Read from the environment ONCE per context (fx_init) - the search path never calls getenv - and
// settable per context afterwards through fx_set_option, under the names of TC_KNOB_TABLE below.
struct TcKnobs {
  int kp = 0;              // force K' (candidates reranked per query)
  int no_rq = 0;           // never take the resident-query kernel
  int slices = 0;          // force the corpus slice count
  int pre = -1;            // 0: no sample prepass
  double pre_safety = 0.0; // sample prepass: rows the initial threshold passes, in units of K' (0: the planner's choice)
  double pre_m = 0.0;      // sample prepass: rank of the sample statistic (0: the planner's choice)
  int pair = -1;           // CTA-pair streaming kernel: 0 never, 1 whenever possible, -1 auto
  int resident = -1;       // int8 CTA-pair kernel with the query tiles resident in shared memory: -1 auto (wherever the CTA-pair
                           // kernel runs and the tile fits), 0 never, 1 whenever it fits
  int int8 = -1;           // exact cosine filters with int8 MMAs over the int8 normalised shadow: -1 auto (rows wider than 192
                           // columns, k <= 16), 0 never, 1 whenever the metric and precision allow
  int fp32_filter_tf32 = 0;// exact mode filters with TF32 over the fp32 rows even when a shadow exists
  int no_norm_shadow = 0;  // cosine keeps the plain shadow + multiplicative epilogue
  int debug_bf16 = 0;      // fx_debug_scores dumps the bf16 filter's scores
  int graph = 1;           // small searches (<= 64 queries, no mask) replay a captured CUDA graph from their second identical
                           // call on (0: always launch kernel by kernel)
  int direct = 1;          // 0: never take the single-launch direct scan (direct_scan.cuh: <= 8 queries, small shards)
  int direct_mb = 256;     // largest shard (MB of fp32 rows) the direct scan takes
  int debug_direct = 0;    // stderr timeline (globaltimer stamps) of every direct scan launched by fx_search. Kept although
                           // it is a debug aid: without its stamps ptxas (CUDA 12.9) spills in knn_direct_kernel<2, 4>
                           // (16 B) and gives two other instances 2 more registers
};
// Every option once: its name (the environment variable's) and the member it sets, an integer (atoi) or a real (atof).
using TcKnobInt = int TcKnobs::*;
using TcKnobReal = double TcKnobs::*;
struct TcKnobDef { const char* name; TcKnobInt i; TcKnobReal r; };
inline const TcKnobDef TC_KNOB_TABLE[] = {
    {"FENIX_TC_KP", &TcKnobs::kp, nullptr},
    {"FENIX_TC_NO_RQ", &TcKnobs::no_rq, nullptr},
    {"FENIX_TC_SLICES", &TcKnobs::slices, nullptr},
    {"FENIX_TC_PRE", &TcKnobs::pre, nullptr},
    {"FENIX_TC_PRE_SAFETY", nullptr, &TcKnobs::pre_safety},
    {"FENIX_TC_PRE_M", nullptr, &TcKnobs::pre_m},
    {"FENIX_TC_PAIR", &TcKnobs::pair, nullptr},
    {"FENIX_TC_RESIDENT", &TcKnobs::resident, nullptr},
    {"FENIX_INT8", &TcKnobs::int8, nullptr},
    {"FENIX_FP32_FILTER_TF32", &TcKnobs::fp32_filter_tf32, nullptr},
    {"FENIX_NO_NORM_SHADOW", &TcKnobs::no_norm_shadow, nullptr},
    {"FENIX_DEBUG_BF16", &TcKnobs::debug_bf16, nullptr},
    {"FENIX_GRAPH", &TcKnobs::graph, nullptr},
    {"FENIX_DIRECT", &TcKnobs::direct, nullptr},
    {"FENIX_DIRECT_MAX_MB", &TcKnobs::direct_mb, nullptr},
    {"FENIX_DEBUG_DIRECT", &TcKnobs::debug_direct, nullptr},
};
// value = the option's text, or null to restore the default. False: unknown name.
inline bool tc_set_knob(TcKnobs* k, const char* name, const char* value) {
  const TcKnobs d{};
  for (const TcKnobDef& o : TC_KNOB_TABLE) {
    if (!name || std::strcmp(name, o.name) != 0) continue;
    if (o.i) k->*o.i = value ? std::atoi(value) : d.*o.i;
    else k->*o.r = value ? std::atof(value) : d.*o.r;
    return true;
  }
  return false;
}
inline void tc_knobs_from_env(TcKnobs* k) {
  for (const TcKnobDef& o : TC_KNOB_TABLE)
    if (const char* v = std::getenv(o.name)) tc_set_knob(k, o.name, v);
}

struct TcState {
  int sm_count = 0;
  void* encode = nullptr;  // cuTensorMapEncodeTiled
  TcKnobs knobs;
};
struct TcCorpus {
  CUtensorMap map_x;       // [n_rows][pitch] fp32, box 32 x 256, 128B swizzle
  CUtensorMap map_xb;      // bf16 shadow, tiled [tile][k-block][256 rows][64], box 64 x 256 = one contiguous 32 KB block
  CUtensorMap map_xn;      // bf16 shadow of the NORMALISED rows x/|x| (cosine), same layout, built on first use
  CUtensorMap map_xb_h, map_xn_h;   // the same shadows seen through 128-row boxes (resident-query kernel)
  CUtensorMap map_x8, map_x8_h;     // int8 shadow of the normalised rows (cosine, kind 2), same tiling with 128 columns per k-block
  bool ok = false;
  bool ok_b = false;
  bool ok_n = false;
  bool ok_8 = false;
};
struct TcSearch {
  const float* X; const float* hx; const float* rx; int64_t n_rows; int dim; int pitch; int64_t row_base;
  float max_norm; const float* Q; int n_q; int metric; int k; bool certify;
  int64_t* out_rows; float* out_dist; cudaStream_t stream; cudaEvent_t ev_k0, ev_k1;
  unsigned ev_flags;       // cudaEventRecordExternal while the search is being captured into a CUDA graph, else 0
  float* dbg;              // optional [128][256] raw score dump (diagnostics)
  int kind;                // 0: TF32 filter over the fp32 rows, 1: bf16 filter over a bf16 shadow, 2: int8 filter over the int8
                           // normalised shadow (cosine; scores are certified upper bounds of the exact cosine)
  int pitch_b;             // elements per row of the bf16 (kind 2: int8) query matrix (whole 128-byte k-blocks)
  const float2* i8_tile;   // kind 2: (S_t, E_t) of every shard tile
  const uint32_t* tau_fixed; // refinement pass: preset per-query admission thresholds (ordered encoding) or null
  int epi;                   // epilogue form: 0 score = acc + hx[row], 1 score = acc * rx[row], 2 score = acc
  int shadow;                // kind 1: 0 = plain shadow (+ augmented columns), 1 = normalised shadow
  int aug;                   // kind 1: the query's augmented columns. 1 (L2): [1, 1, 1, u] pick up the shadow's -|x|^2/2 terms
                             // and the row's error weight; 2 (inner product, rows of very different norm): [0, 0, 0, u];
                             // u = c |q| rounded up, so that the filter score is a certified UPPER bound of the exact score
  double c_pair;             // aug != 0: the constant c of u = c |q| (product rounding + accumulation, see tc_c_err / tc_c_add)
  int sample_stride;         // > 1: threshold prepass over every sample_stride-th corpus tile (set by tc_search)
  int pre_m;                 // prepass: rank of the sample's block maximum that becomes the query's initial threshold
  int no_prepass;            // 1: adaptive thresholds only (re-run of queries the sample threshold failed)
  int seeded;                // set by tc_prepare: this main pass starts from the sample prepass's thresholds (list quotas >= k, see tc_plan)
  int full_lists;            // 1: every candidate list keeps K' entries (re-run of starved queries: when a query's neighbours sit in
                             // ONE list - clustered rows in row order - a list that keeps fewer than k can never supply them)
  int no_finish;             // 1: the filter only; the caller reads the candidate lists itself (range search, tc_finish_params)
};

// ---------------------------------------------------------------------------------------------
// PTX wrappers (sm_100a)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return uint32_t(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// Polling wait for the single-thread producer / MMA roles: between polls the thread sleeps, so its spin loop
// does not take issue slots from the epilogue warps that share its SM sub-partition (measured on C2: the two
// spin loops were 23 % of all executed instructions).
__device__ __forceinline__ void mbar_wait_backoff(uint64_t* bar, uint32_t parity, uint32_t ns) {
  uint32_t done;
  for (;;) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}" : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    if (done) break;
    if (ns) __nanosleep(ns);
  }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "elect.sync _|P1, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t"
      "}" : "=r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void bulk_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

// D[tmem] (+)= A[smem desc] * B[smem desc]^T, kind::tf32, issued by one thread.
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// Arrive on an mbarrier once every previously issued tcgen05.mma of this thread has completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- CTA pairs (cta_group::2): two CTAs of a cluster on one TPC share the B operand of a 256-row MMA ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same shared-memory location in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load into THIS CTA's shared memory whose completion bytes are counted on an mbarrier that may live in the peer
// CTA of the pair (the leader's "stage full" barrier)
__device__ __forceinline__ void tma_load_2d_pair(const CUtensorMap* map, uint32_t bar_cluster_addr, void* dst, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_cluster_addr), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem of both CTAs] (+)= A[128 rows from each CTA] * B[N/2 rows from each CTA]^T, issued by one thread of the leader
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_i8_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// Arrive (once the pair's previously issued MMAs have completed) on the mbarrier at this offset in BOTH CTAs.
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"(uint16_t(3)) : "memory");
}

// K-major, 128B-swizzled operand tile (rows of 128 B, 8-row groups 1024 B apart).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= uint64_t((smem_addr & 0x3ffffu) >> 4);        // start address        bits [0,14)
  d |= uint64_t(1) << 16;                            // leading byte offset  (ignored for swizzled K-major)
  d |= uint64_t(1024 >> 4) << 32;                    // stride byte offset   bits [32,46): 8 rows * 128 B
  d |= uint64_t(1) << 46;                            // descriptor version 1 (sm_100)
  d |= uint64_t(2) << 61;                            // layout: SWIZZLE_128B
  return d;
}
// kind::tf32, fp32 accumulate, both operands K-major.
__host__ __device__ constexpr uint32_t make_idesc_tf32(int m, int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (uint32_t(n >> 3) << 17) | (uint32_t(m >> 4) << 24);
}
// kind::f16 with bf16 operands, fp32 accumulate, both operands K-major.
__host__ __device__ constexpr uint32_t make_idesc_bf16(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(n >> 3) << 17) | (uint32_t(m >> 4) << 24);
}
// kind::i8 with signed 8-bit operands, s32 accumulate, both operands K-major: D format S32 = 2 in bits [4,6), A and B
// format signed = 1 in bits [7,10) and [10,13), no saturation (bit 3: the sums are far from the int32 range).
__host__ __device__ constexpr uint32_t make_idesc_i8(int m, int n) {
  return (2u << 4) | (1u << 7) | (1u << 10) | (uint32_t(n >> 3) << 17) | (uint32_t(m >> 4) << 24);
}

__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x4(uint32_t taddr, uint32_t (&v)[4]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// Same wait, with the loaded registers as in/out operands: the compiler cannot move a use of v[] above it.
__device__ __forceinline__ void tmem_ld_wait_dep(uint32_t (&v)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
                 "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]),
                 "+r"(v[16]), "+r"(v[17]), "+r"(v[18]), "+r"(v[19]), "+r"(v[20]), "+r"(v[21]), "+r"(v[22]), "+r"(v[23]),
                 "+r"(v[24]), "+r"(v[25]), "+r"(v[26]), "+r"(v[27]), "+r"(v[28]), "+r"(v[29]), "+r"(v[30]), "+r"(v[31])
               :: "memory");
}

__device__ __forceinline__ uint32_t ld_relaxed_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ float max4(const uint32_t (&v)[TC_CW], int g) {
  return fmaxf(fmaxf(__uint_as_float(v[4 * g + 0]), __uint_as_float(v[4 * g + 1])),
               fmaxf(__uint_as_float(v[4 * g + 2]), __uint_as_float(v[4 * g + 3])));
}

// ---------------------------------------------------------------------------------------------
// kernel parameters
// ---------------------------------------------------------------------------------------------
struct TcParams {
  int n_q;                // queries
  int n_qt;               // query tiles of 128
  int64_t n_rows;         // corpus rows in the shard
  int n_tiles;            // corpus tiles of 256 rows
  int n_slices;           // corpus slices (units = n_slices * n_qt)
  int tiles_per_slice;
  int n_vtiles;           // tiles the units iterate over: all of them, or every tile_stride-th one (threshold prepass)
  int tile_stride;
  float* pre_max;         // threshold prepass (PRE kernels): [query][record] maximum score of every 128-column block
  int pre_pitch;          // records per query
  int n_kblocks;          // k-blocks (128 B of K per row) loaded per tile: n_kb_data (+ 1 when a separate augmented block is used)
  int n_kb_data;          // data k-blocks per tile (the tile stride of the tiled shadow)
  int nk_last;            // MMA instructions (32 B of K each) of the last data block: only columns that hold data are multiplied
  int aug_line0;          // first 128-byte line of the separate augmented region of the shadow (one block per tile)
  int rq_stages;          // resident-query kernels (rq, CTA pair with resident query tiles): depth of the corpus-block ring
  uint32_t sleep_ns;      // producer / MMA polling loops sleep this long between polls (0: spin). Sleeping keeps their
                          // spin loops out of the epilogue warps' issue slots where the epilogue binds (narrow rows);
                          // where the tensor pipe binds (wide rows) a late wake-up costs ~2 % instead
  int kp;                 // K': candidates kept per (query, unit-half) selection
  int cap;                // candidate buffer capacity per epilogue thread (512 or 1024)
  const float* hx;        // [n_rows padded to 256] -0.5|x|^2
  const float* rx;        // [n_rows padded to 256] 1/max(|x|,eps)
  uint2* wbuf;            // [units][256][cap] candidate buffers (score bits, row), one per (unit, epilogue thread)
  int* wcnt;              // [units][256] entries left in each buffer when its unit finished
  uint32_t* tau_g;        // [n_q] shared per-query threshold, ordered-uint encoding
  int fixed;              // refinement pass: thresholds are preset in tau_g, no selection; buffer overflow sets flags[q]
  int* flags;             // [n_q]
  float* dbg;             // diagnostics: raw scores of (query tile 0) x (corpus tile 0), [128][256], or null
  const float2* i8_tile;  // kind 2: (S_t, E_t) per shard tile
  const float4* i8_q;     // kind 2: (S_q, a_q, e_q, 0) per query
};

// ---------------------------------------------------------------------------------------------
// warp-cooperative selection on one thread's candidate buffer
// ---------------------------------------------------------------------------------------------
// Keeps the kp best (largest score) of buf[0..cnt), compacted to the front; returns the kp-th best
// score in ordered-uint form (the new admission threshold: everything dropped is <= it).
template <int PER>
__device__ __noinline__ uint32_t warp_select_compact(uint2* buf, int cnt, int kp, int& new_cnt) {
  const uint32_t lane = lane_id();
  uint32_t s[PER];
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    int idx = i * 32 + int(lane);
    s[i] = (idx < cnt) ? f2ord(__uint_as_float(buf[idx].x)) : 0u;
  }
  // Radix descent for a value v with count(s >= v) >= kp. Bits above the highest bit in which the buffer's
  // minimum and maximum differ are common to all entries and skipped; the descent stops as soon as at most
  // kp + 16 entries remain at or above v (any such v is a valid threshold: everything dropped is <= v), and
  // only runs to bit 0 when many entries are (nearly) equal.
  uint32_t mx = 0u, mn = 0xffffffffu;
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    mx = max(mx, s[i]);
    if (i * 32 + int(lane) < cnt) mn = min(mn, s[i]);
  }
  mx = __reduce_max_sync(0xffffffffu, mx);
  mn = __reduce_min_sync(0xffffffffu, mn);
  uint32_t v = mn;
  if (mx != mn && cnt > kp) {
    const int top = 31 - __clz(mx ^ mn);
    v = (top == 31) ? 0u : (mx & ~((2u << top) - 1u));
    int c_v = cnt;
    for (int bit = top; bit >= 0 && c_v > kp + 16; --bit) {
      uint32_t cand = v | (1u << bit);
      int c = 0;
#pragma unroll
      for (int i = 0; i < PER; ++i) c += (s[i] >= cand) ? 1 : 0;
      c = __reduce_add_sync(0xffffffffu, c);
      if (c >= kp) { v = cand; c_v = c; }
    }
  }
  int n_gt = 0;
#pragma unroll
  for (int i = 0; i < PER; ++i) n_gt += (s[i] > v) ? 1 : 0;
  n_gt = __reduce_add_sync(0xffffffffu, n_gt);
  int ties_left = max(kp - n_gt, 0);
  int out = 0;
  const uint32_t lt_mask = (1u << lane) - 1u;
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    if (i * 32 < cnt) {   // warp-uniform
      int idx = i * 32 + int(lane);
      uint2 e = (idx < cnt) ? buf[idx] : make_uint2(0u, 0u);
      __syncwarp();
      bool gt = s[i] > v;
      bool tie = (idx < cnt) && (s[i] == v);
      uint32_t tie_ballot = __ballot_sync(0xffffffffu, tie);
      int tie_rank = __popc(tie_ballot & lt_mask);
      bool keep = gt || (tie && tie_rank < ties_left);
      ties_left -= min(ties_left, __popc(tie_ballot));
      uint32_t keep_ballot = __ballot_sync(0xffffffffu, keep);
      if (keep) buf[out + __popc(keep_ballot & lt_mask)] = e;
      out += __popc(keep_ballot);
      __syncwarp();
    }
  }
  new_cnt = out;
  return v;
}

// ---------------------------------------------------------------------------------------------
// epilogue building blocks shared by the two filter kernels
// ---------------------------------------------------------------------------------------------
// One call handles the TC_HALF_COLS (128) accumulator columns at TMEM address t_acc that belong to this thread's
// query: score, compare with the running threshold, append survivors at wp, hand the accumulator back (arrive on
// release_bar, one arrival per warp). ncols = valid columns (<= 0: nothing to look at, only the release).
//
// The hot code must be SMALL: with two epilogue warps per SM sub-partition nothing hides an instruction-cache miss
// or a branch (a build whose epilogue grew from 24 KB to 28 KB of SASS ran 28 % slower). So:
//  * scan: one chunk = 32 columns (one tcgen05.ld.x32, the next chunk's load already in flight), per-row terms
//    (METRIC 0 add / 1 multiply, from nrm in shared memory; METRIC 2: the score is the accumulator), eight quad
//    maxima, one warp vote. About 30 instructions per chunk, no per-element work.
//  * hits: appends are inherently frequent at large k / small N (a query admits ~K' ln(N/K') rows over the scan and
//    32 queries share a warp), yet a chunk rarely holds more than one or two. The warp ORs the lanes' 8-bit masks of
//    passing quads and, per quad in the union, re-reads those four columns from TMEM (tcgen05.ld.x4 takes a runtime
//    column address, registers cannot be indexed) and appends what passes: one compact loop instead of 32 unrolled
//    append sites per chunk. Columns past the shard's last row are rejected here, so the scan needs no tail handling.
// PAIR (CTA-pair kernel): the accumulator is handed back to the LEADER's MMA warp (release_leader: shared::cluster
// address of its barrier) and, separately, the norm buffer to this CTA's own producer (norm_release).
template <int METRIC, int MODE, int PAIR = 0>   // MODE 0: filter, 1: filter + raw score dump (diagnostics), 2: threshold prepass (block maximum only)
__device__ __forceinline__ void epi_tile(uint32_t t_acc, int ncols, const float* nrm, int col0, float tau, uint2* buf,
                                         uint32_t& wn, uint64_t* release_bar, uint32_t release_leader, uint64_t* norm_release,
                                         uint32_t lane, float* dbg_row, float* pre_out) {
  constexpr bool DBG = MODE == 1;
  float blk_max = -INFINITY;
  auto release = [&]() {
    tc_fence_before();
    __syncwarp();
    if (lane == 0) {
      if (PAIR) {
        mbar_arrive_cluster(release_leader);
        if (METRIC != 2) mbar_arrive(norm_release);
      } else {
        mbar_arrive(release_bar);
      }
    }
  };
  auto scan = [&](uint32_t (&v)[TC_CW], int c) {
    if (METRIC != 2) {
#pragma unroll
      for (int j = 0; j < TC_CW; j += 4) {
        const float4 n4 = *reinterpret_cast<const float4*>(nrm + c + j);
        float s0 = __uint_as_float(v[j + 0]), s1 = __uint_as_float(v[j + 1]);
        float s2 = __uint_as_float(v[j + 2]), s3 = __uint_as_float(v[j + 3]);
        if (METRIC == 0) { s0 += n4.x; s1 += n4.y; s2 += n4.z; s3 += n4.w; }
        if (METRIC == 1) { s0 *= n4.x; s1 *= n4.y; s2 *= n4.z; s3 *= n4.w; }
        v[j + 0] = __float_as_uint(s0); v[j + 1] = __float_as_uint(s1);
        v[j + 2] = __float_as_uint(s2); v[j + 3] = __float_as_uint(s3);
      }
    }
    if (DBG) {
      if (dbg_row != nullptr) {
#pragma unroll
        for (int j = 0; j < TC_CW; ++j) dbg_row[c + j] = __uint_as_float(v[j]);
      }
    }
    float qm[TC_CW / 4];
#pragma unroll
    for (int g = 0; g < TC_CW / 4; ++g) qm[g] = max4(v, g);
    float m = qm[0];
#pragma unroll
    for (int g = 1; g < TC_CW / 4; ++g) m = fmaxf(m, qm[g]);
    if (MODE == 2) { blk_max = fmaxf(blk_max, m); return; }
    if (__any_sync(0xffffffffu, m > tau)) {
      uint32_t mine = 0;
#pragma unroll
      for (int g = 0; g < TC_CW / 4; ++g) mine |= (qm[g] > tau) ? (1u << g) : 0u;
      uint32_t quads = __reduce_or_sync(0xffffffffu, mine);
      while (quads) {                       // warp-uniform
        const int g = __ffs(quads) - 1;
        quads &= quads - 1;
        const int cq = c + 4 * g;           // first column of the quad within these 128 columns
        uint32_t w[4];
        tmem_ld_32x32b_x4(t_acc + uint32_t(cq), w);
        tmem_ld_wait();
        float4 n4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (METRIC != 2) n4 = *reinterpret_cast<const float4*>(nrm + cq);
        const float nn[4] = {n4.x, n4.y, n4.z, n4.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float sc = __uint_as_float(w[j]);
          if (METRIC == 0) sc += nn[j];
          if (METRIC == 1) sc *= nn[j];
          if (sc > tau && cq + j < ncols) { buf[wn] = make_uint2(__float_as_uint(sc), uint32_t(col0 + cq + j)); ++wn; }
        }
      }
    }
  };
  if (ncols > 0) {
    // two register sets: the TMEM load of chunk i+1 is in flight while chunk i is scanned. The hit loop re-reads
    // the accumulator, so it goes back to the MMA warp only after the last chunk.
    static_assert(TC_HALF_COLS % (2 * TC_CW) == 0, "chunk pairs");
    uint32_t va[TC_CW], vb[TC_CW];
    tmem_ld_32x32b_x32(t_acc, va);
#pragma unroll TC_EPI_UNROLL
    for (int c = 0; c < TC_HALF_COLS; c += 2 * TC_CW) {
      tmem_ld_wait_dep(va);
      tmem_ld_32x32b_x32(t_acc + uint32_t(c + TC_CW), vb);
      scan(va, c);
      tmem_ld_wait_dep(vb);
      if (c + 2 * TC_CW < TC_HALF_COLS) tmem_ld_32x32b_x32(t_acc + uint32_t(c + 2 * TC_CW), va);
      scan(vb, c + TC_CW);
    }
  }
  release();
  // prepass: a block that reaches past the shard's last row is not recorded (its pad columns score 0, which can
  // exceed every real score, e.g. L2 scores q.x - |x|^2/2)
  if (MODE == 2) { if (pre_out != nullptr) *pre_out = ncols >= TC_HALF_COLS ? blk_max : -INFINITY; }
}

// The same tile for the int8 filter (kind 2): the accumulators are int32 and the scan stays in the integer domain -
// quad maxima and the compare against the (query, tile) threshold thr (i8_threshold) are one integer instruction per
// element, as in epi_tile. Only appended hits are converted, to the float upper bound (i8_upper), so candidate lists,
// tau_g and the finish kernel keep their float order encoding. METRIC 0 (masked searches): nrm holds an integer row
// term, 0 or I8_MASKED. MODE 2 records block maxima in upper-bound units, MODE 1 dumps upper bounds.
template <int METRIC, int MODE, int PAIR = 0>
__device__ __forceinline__ void epi_tile_i8(uint32_t t_acc, int ncols, const float* nrm, int col0, float tau, int thr,
                                            double inv_ss, double ae, uint2* buf, uint32_t& wn, uint64_t* release_bar,
                                            uint32_t release_leader, uint64_t* norm_release, uint32_t lane, float* dbg_row,
                                            float* pre_out) {
  int blk_max = I8_FLOOR;
  const int* term = reinterpret_cast<const int*>(nrm);
  auto release = [&]() {
    tc_fence_before();
    __syncwarp();
    if (lane == 0) {
      if (PAIR) {
        mbar_arrive_cluster(release_leader);
        if (METRIC != 2) mbar_arrive(norm_release);
      } else {
        mbar_arrive(release_bar);
      }
    }
  };
  auto scan = [&](uint32_t (&v)[TC_CW], int c) {
    if (METRIC == 0) {
#pragma unroll
      for (int j = 0; j < TC_CW; j += 4) {
        const int4 n4 = *reinterpret_cast<const int4*>(term + c + j);
        v[j + 0] += uint32_t(n4.x); v[j + 1] += uint32_t(n4.y); v[j + 2] += uint32_t(n4.z); v[j + 3] += uint32_t(n4.w);
      }
    }
    if (MODE == 1) {
      if (dbg_row != nullptr) {
#pragma unroll
        for (int j = 0; j < TC_CW; ++j) dbg_row[c + j] = i8_upper(int(v[j]), inv_ss, ae);
      }
    }
    int qm[TC_CW / 4];
#pragma unroll
    for (int g = 0; g < TC_CW / 4; ++g)
      qm[g] = max(max(int(v[4 * g + 0]), int(v[4 * g + 1])), max(int(v[4 * g + 2]), int(v[4 * g + 3])));
    int m = qm[0];
#pragma unroll
    for (int g = 1; g < TC_CW / 4; ++g) m = max(m, qm[g]);
    if (MODE == 2) { blk_max = max(blk_max, m); return; }
    if (__any_sync(0xffffffffu, m > thr)) {
      uint32_t mine = 0;
#pragma unroll
      for (int g = 0; g < TC_CW / 4; ++g) mine |= (qm[g] > thr) ? (1u << g) : 0u;
      uint32_t quads = __reduce_or_sync(0xffffffffu, mine);
      while (quads) {                       // warp-uniform
        const int g = __ffs(quads) - 1;
        quads &= quads - 1;
        const int cq = c + 4 * g;
        uint32_t w[4];
        tmem_ld_32x32b_x4(t_acc + uint32_t(cq), w);
        tmem_ld_wait();
        int4 n4 = make_int4(0, 0, 0, 0);
        if (METRIC == 0) n4 = *reinterpret_cast<const int4*>(term + cq);
        const int nn[4] = {n4.x, n4.y, n4.z, n4.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int a = int(w[j]);
          if (a + nn[j] > thr && cq + j < ncols) {
            const float sc = i8_upper(a, inv_ss, ae);
            if (sc > tau) { buf[wn] = make_uint2(__float_as_uint(sc), uint32_t(col0 + cq + j)); ++wn; }
          }
        }
      }
    }
  };
  if (ncols > 0) {
    uint32_t va[TC_CW], vb[TC_CW];
    tmem_ld_32x32b_x32(t_acc, va);
#pragma unroll TC_EPI_UNROLL
    for (int c = 0; c < TC_HALF_COLS; c += 2 * TC_CW) {
      tmem_ld_wait_dep(va);
      tmem_ld_32x32b_x32(t_acc + uint32_t(c + TC_CW), vb);
      scan(va, c);
      tmem_ld_wait_dep(vb);
      if (c + 2 * TC_CW < TC_HALF_COLS) tmem_ld_32x32b_x32(t_acc + uint32_t(c + 2 * TC_CW), va);
      scan(vb, c + TC_CW);
    }
  }
  release();
  if (MODE == 2) { if (pre_out != nullptr) *pre_out = ncols >= TC_HALF_COLS ? i8_upper(blk_max, inv_ss, ae) : -INFINITY; }
}

// Tighten thresholds after a tile. The common case costs one compare and one vote: every lane keeps the entry count
// at which it needs attention (wn_trig): K' while it has no threshold yet, cap - 127 (the next tile could overflow
// the buffer) afterwards. A lane that got there receives a warp-cooperative selection; its new threshold is shared
// through tau_g. In the refinement pass (preset thresholds) an overflowing lane flags its query instead.
__device__ __forceinline__ uint32_t epi_trigger(const TcParams& p, bool active, float tau) {
  if (!active) return 0xffffffffu;
  return (!p.fixed && tau == -INFINITY) ? uint32_t(p.kp) : uint32_t(p.cap - TC_HALF_COLS + 1);
}
__device__ __forceinline__ void epi_tighten(const TcParams& p, bool active, int q, uint2* buf, uint32_t& wn, uint32_t& wn_trig,
                                            float& tau, uint32_t lane) {
  if (!__any_sync(0xffffffffu, wn >= wn_trig)) return;
  wn_trig = epi_trigger(p, active, tau);   // a threshold may have arrived through tau_g since the trigger was set
  const bool hit = active && wn >= wn_trig;
  if (p.fixed) {
    if (hit) { p.flags[q] = 1; tau = INFINITY; wn_trig = 0xffffffffu; }   // more survivors than the buffer holds
    return;
  }
  uint32_t need_mask = __ballot_sync(0xffffffffu, hit);
  while (need_mask) {
    const int src = __ffs(need_mask) - 1;
    need_mask &= need_mask - 1;
    uint2* b = reinterpret_cast<uint2*>(__shfl_sync(0xffffffffu, reinterpret_cast<uint64_t>(buf), src));
    const int c_src = __shfl_sync(0xffffffffu, int(wn), src);
    int new_cnt;
    uint32_t v_ord = (p.cap == 1024) ? warp_select_compact<32>(b, c_src, p.kp, new_cnt)
                                     : warp_select_compact<16>(b, c_src, p.kp, new_cnt);
    if (int(lane) == src) {
      wn = uint32_t(new_cnt);
      tau = fmaxf(tau, ord2f(v_ord));
      atomicMax(p.tau_g + q, v_ord);
      wn_trig = epi_trigger(p, active, tau);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// the filter kernel
// ---------------------------------------------------------------------------------------------
// KIND 0: fp32 operands read as TF32 (k-block = 32 elements, UMMA K = 8)
// KIND 1: bf16 operands          (k-block = 64 elements, UMMA K = 16); both are 128 B rows / 32 B per MMA
// KIND 2: int8 operands          (k-block = 128 elements, UMMA K = 32, int32 accumulators; epilogue epi_tile_i8)
// PAIR 1: CTA pairs (cluster of 2, tcgen05 cta_group::2, bf16 or int8 shadow). The pair computes a 256-query x 256-row
//         tile per MMA: each CTA stages ITS query tile (A, 16 KB per k-block) and HALF of the corpus block (B, 128 of
//         the 256 rows, 16 KB); the tensor cores of both SMs read both halves. Per SM and k-block that is 32 KB of
//         L2 -> SM operand traffic instead of 48 KB, at the same tensor work (measured on C3, one CTA per tile:
//         742.8 GB per launch = 96 B/clk/SM at the full tensor rate, more than the fabric delivers once the power cap
//         lifts). The leader (cluster rank 0) issues every MMA; "stage full" lives in the leader (both CTAs' TMA
//         loads count their bytes there), "stage empty" / "accumulator full" are multicast to both CTAs by
//         tcgen05.commit, "accumulator empty" collects the epilogue warps of both CTAs in the leader.
//         Units: (query-tile pair) x (corpus slice); CTA r of the pair owns query tile 2*qp + r and keeps the
//         candidate lists of "CTA unit" slice * (2 n_qp) + 2 qp + r, the layout the finish kernel reads.
// PAIR 2: CTA pairs over the int8 shadow with the query tiles RESIDENT. An int8 query tile (n_kblocks x 16 KB, 96 KB at
//         D = 768) fits in shared memory next to a corpus ring, so each CTA loads ITS tile once per unit (a_full: both
//         CTAs' bytes counted in the leader; a_empty: committed to both CTAs by the leader after the unit's last MMA)
//         and the ring carries only corpus half blocks: per SM and k-block 16 KB of L2 -> SM operand traffic instead of
//         32 KB, and the ring (p.rq_stages deep, tc3_stages) looks further ahead. MMAs, commits, TMEM double buffer,
//         epilogue and the candidate-list layout are those of PAIR 1.
template <int METRIC, int KIND, int MODE, int PAIR>
__global__ void __launch_bounds__(TC_THREADS, 1)
knn_tc_filter_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_x, TcParams p) {
  static_assert(!PAIR || KIND >= 1, "CTA pairs stream a shadow");
  constexpr bool RES = PAIR == 2;
  static_assert(!RES || KIND == 2, "resident query tiles: int8 shadow");
  constexpr int STAGES = RES ? TC3_MAX_STAGES : (PAIR ? TC2_STAGES : TC_STAGES);   // (RES: barriers; p.rq_stages are used)
  constexpr uint32_t B_BYTES = PAIR ? TC2_B_BYTES : TC_B_BYTES;
  constexpr uint32_t STAGE_BYTES = (RES ? 0u : TC_A_BYTES) + B_BYTES;
  const int n_stages = RES ? p.rq_stages : STAGES;
  extern __shared__ unsigned char smem_raw[];
  // 1024-byte alignment for the 128B-swizzled operand tiles (the offset is the same in both CTAs of a pair:
  // the dynamic shared memory window starts at the same offset in every CTA of a kernel)
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* a_res = smem;                                                  // RES: [n_kblocks] query blocks
  unsigned char* tiles = RES ? smem + p.n_kblocks * TC_A_BYTES : smem;
  float* norm_smem = reinterpret_cast<float*>(tiles + n_stages * STAGE_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(tiles + n_stages * STAGE_BYTES + TC_ACC_STAGES * TC_NORM_BYTES);
  uint64_t* full_bar = bars;                         // [STAGES]      TMA -> MMA          (PAIR: the leader's is used)
  uint64_t* empty_bar = bars + STAGES;               // [STAGES]      MMA -> TMA          (PAIR: multicast to both CTAs)
  uint64_t* tmem_full = bars + 2 * STAGES;           // [2]           MMA -> epilogue     (PAIR: multicast to both CTAs)
  uint64_t* tmem_empty = tmem_full + TC_ACC_STAGES;  // [2]           epilogue -> MMA     (PAIR: both CTAs' warps, in the leader)
  uint64_t* norm_full = tmem_empty + TC_ACC_STAGES;  // [2]           TMA(norms) -> epilogue
  uint64_t* norm_empty = norm_full + TC_ACC_STAGES;  // [2]           epilogue -> TMA(norms) (PAIR only; otherwise tmem_empty serves)
  uint64_t* a_full = norm_empty + TC_ACC_STAGES;     // RES [1]       query tiles of the unit landed (the leader's is used)
  uint64_t* a_empty = a_full + 1;                    // RES [1]       the unit's last MMAs retired (multicast to both CTAs)
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(a_full + (RES ? 2 : 0));

  const int warp = threadIdx.x >> 5;
  const uint32_t lane = lane_id();
  const uint32_t rank = PAIR ? cluster_ctarank() : 0u;          // 0 = leader
  const int cid = PAIR ? int(blockIdx.x >> 1) : int(blockIdx.x);   // persistent worker index (cluster / CTA)
  const int n_workers = PAIR ? int(gridDim.x >> 1) : int(gridDim.x);

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&map_q);
    prefetch_tmap(&map_x);
    for (int i = 0; i < n_stages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < TC_ACC_STAGES; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], PAIR ? 2 * TC_EPI_WARPS : TC_EPI_WARPS);
      mbar_init(&norm_full[i], 1);
      mbar_init(&norm_empty[i], TC_EPI_WARPS);
    }
    if (RES) { mbar_init(a_full, 1); mbar_init(a_empty, 1); }
    fence_barrier_init();
  }
  if (warp == 2) { if (PAIR) tmem_alloc_pair(tmem_ptr, 512); else tmem_alloc(tmem_ptr, 512); }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();    // the peer's barriers are initialised before anything is signalled across the pair
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  const int n_qp = (p.n_qt + 1) >> 1;
  const int n_units = PAIR ? p.n_slices * n_qp : p.n_slices * p.n_qt;
  const int n_rows_i = int(p.n_rows);   // < 2^31 (tc_supported)
  // worker unit u -> (query tile of THIS CTA, corpus slice, index of this CTA's candidate-list block)
  auto decode = [&](int u, int& qt, int& slice, int& cu) {
    if (PAIR) { const int qp = u % n_qp; slice = u / n_qp; qt = 2 * qp + int(rank); cu = slice * (2 * n_qp) + qt; }
    else { slice = u / p.n_qt; qt = u - slice * p.n_qt; cu = u; }
  };

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      const uint32_t full_leader = PAIR ? mapa_u32(smem_u32(full_bar), 0) : 0u;   // the leader's full_bar[0]
      constexpr int kElemsPerBlock = KIND == 0 ? TC_BK : (KIND == 1 ? 2 * TC_BK : 4 * TC_BK);
      uint32_t a_phase = 0;
      for (int u = cid; u < n_units; u += n_workers) {
        int qt, slice, cu; decode(u, qt, slice, cu);
        const int t0 = slice * p.tiles_per_slice, t1 = min(p.n_vtiles, t0 + p.tiles_per_slice);
        if (RES) {
          // this CTA's query tile for the whole unit, once the previous unit's MMAs have retired. Deliberately simple: the
          // ring drains once per unit here (no corpus block of the next unit is issued before its query tile), one
          // ~2 us L2/HBM round trip per unit against ~2000 tiles of MMA work per unit at C3 (~5 ms), i.e. < 0.1 %
          mbar_wait_backoff(a_empty, a_phase ^ 1, p.sleep_ns);
          if (rank == 0) mbar_expect_tx(a_full, 2u * uint32_t(p.n_kblocks) * TC_A_BYTES);   // both CTAs' tiles
          const uint32_t a_bar = mapa_u32(smem_u32(a_full), 0);
          for (int kb = 0; kb < p.n_kblocks; ++kb)
            tma_load_2d_pair(&map_q, a_bar, a_res + kb * TC_A_BYTES, kb * kElemsPerBlock, qt * TC_BM);
          a_phase ^= 1;
        }
        for (int tv = t0; tv < t1; ++tv) {
          const int t = tv * p.tile_stride;
          if (METRIC != 2) {
            // per-column norm terms of this tile ride along, one buffer per accumulator stage
            mbar_wait_backoff(PAIR ? &norm_empty[acc] : &tmem_empty[acc], acc_phase ^ 1, p.sleep_ns);
            mbar_expect_tx(&norm_full[acc], TC_NORM_BYTES);
            const float* src = (METRIC == 0 ? p.hx : p.rx) + size_t(t) * TC_BN;
            bulk_load_1d(norm_smem + acc * TC_BN, src, TC_NORM_BYTES, &norm_full[acc]);
          }
          for (int kb = 0; kb < p.n_kblocks; ++kb) {
            mbar_wait_backoff(&empty_bar[stage], phase ^ 1, p.sleep_ns);
            unsigned char* a_dst = tiles + stage * STAGE_BYTES;
            // tiled shadow: one contiguous block of 256 (PAIR: this CTA's 128) rows x 128 B
            const int line = kb < p.n_kb_data ? (t * p.n_kb_data + kb) * TC_BN : p.aug_line0 + t * TC_BN;
            if (RES) {
              if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * STAGE_BYTES);    // both CTAs' corpus half blocks
              tma_load_2d_pair(&map_x, full_leader + uint32_t(stage) * 8u, a_dst, 0, line + int(rank) * (TC_BN / 2));
            } else if (PAIR) {
              if (rank == 0) mbar_expect_tx(&full_bar[stage], 2 * STAGE_BYTES);    // both CTAs' query + corpus blocks
              const uint32_t bar = full_leader + uint32_t(stage) * 8u;
              tma_load_2d_pair(&map_q, bar, a_dst, kb * kElemsPerBlock, qt * TC_BM);
              tma_load_2d_pair(&map_x, bar, a_dst + TC_A_BYTES, 0, line + int(rank) * (TC_BN / 2));
            } else {
              mbar_expect_tx(&full_bar[stage], STAGE_BYTES);
              tma_load_2d(&map_q, &full_bar[stage], a_dst, kb * kElemsPerBlock, qt * TC_BM);
              if (KIND == 0) tma_load_2d(&map_x, &full_bar[stage], a_dst + TC_A_BYTES, kb * kElemsPerBlock, t * TC_BN);
              else {
                tma_load_2d(&map_x, &full_bar[stage], a_dst + TC_A_BYTES, 0, line);
              }
            }
            if (++stage == n_stages) { stage = 0; phase ^= 1; }
          }
          if (++acc == TC_ACC_STAGES) { acc = 0; acc_phase ^= 1; }
        }
      }
    }
  } else if (warp == 1 && rank == 0) {
    // ===================== MMA issuer (PAIR: the leader CTA issues for both) =====================
    // The whole warp runs the loop (warp-uniform control flow keeps descriptors and addresses in uniform registers;
    // under `if (lane == 0)` the compiler wraps every MMA in a register-broadcast loop), one elected lane issues.
    {
      constexpr uint32_t idesc = KIND == 0 ? make_idesc_tf32(TC_BM, TC_BN)
                                           : KIND == 1 ? make_idesc_bf16(PAIR ? 2 * TC_BM : TC_BM, TC_BN)
                                                       : make_idesc_i8(PAIR ? 2 * TC_BM : TC_BM, TC_BN);
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint64_t desc0 = make_smem_desc(0);
      const uint32_t tiles_lo = smem_u32(tiles) >> 4;
      const uint32_t a_lo = smem_u32(a_res) >> 4;   // RES: query k-block kb at + kb * 1024
      const int n_kb = p.n_kblocks, n_kb_data = p.n_kb_data, nk_last = p.nk_last;
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      uint32_t a_phase = 0;
      for (int u = cid; u < n_units; u += n_workers) {
        int qt, slice, cu; decode(u, qt, slice, cu);
        const int t0 = slice * p.tiles_per_slice, t1 = min(p.n_vtiles, t0 + p.tiles_per_slice);
        if (RES) { mbar_wait(a_full, a_phase); a_phase ^= 1; }
        for (int t = t0; t < t1; ++t) {
          mbar_wait_backoff(&tmem_empty[acc], acc_phase ^ 1, p.sleep_ns >> 1);
          const uint32_t d_tmem = tmem_u + uint32_t(acc * TC_BN);
          for (int kb = 0; kb < n_kb; ++kb) {
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
            const uint64_t a_desc = RES ? desc0 | uint64_t(a_lo + uint32_t(kb) * (TC_A_BYTES >> 4))
                                        : desc0 | uint64_t(tiles_lo + uint32_t(stage) * (STAGE_BYTES >> 4));
            const uint64_t b_desc = RES ? desc0 | uint64_t(tiles_lo + uint32_t(stage) * (STAGE_BYTES >> 4))
                                        : a_desc + (TC_A_BYTES >> 4);
            const int nk = kb < n_kb_data - 1 ? TC_BK / TC_UMMA_K : (kb == n_kb_data - 1 ? nk_last : 1);
            if (elect_one()) {
              // advance 32 B along K inside the 128 B swizzle row: +2 in the (>>4) address field
              if (PAIR && KIND == 2) {
                umma_i8_pair(d_tmem, a_desc, b_desc, idesc, kb != 0 ? 1u : 0u);
                if (nk > 1) umma_i8_pair(d_tmem, a_desc + 2, b_desc + 2, idesc, 1u);
                if (nk > 2) umma_i8_pair(d_tmem, a_desc + 4, b_desc + 4, idesc, 1u);
                if (nk > 3) umma_i8_pair(d_tmem, a_desc + 6, b_desc + 6, idesc, 1u);
                umma_commit_pair(&empty_bar[stage]);
                if (kb == n_kb - 1) umma_commit_pair(&tmem_full[acc]);
              } else if (PAIR) {
                umma_bf16_pair(d_tmem, a_desc, b_desc, idesc, kb != 0 ? 1u : 0u);
                if (nk > 1) umma_bf16_pair(d_tmem, a_desc + 2, b_desc + 2, idesc, 1u);
                if (nk > 2) umma_bf16_pair(d_tmem, a_desc + 4, b_desc + 4, idesc, 1u);
                if (nk > 3) umma_bf16_pair(d_tmem, a_desc + 6, b_desc + 6, idesc, 1u);
                umma_commit_pair(&empty_bar[stage]);                       // frees the stage in BOTH CTAs
                if (kb == n_kb - 1) umma_commit_pair(&tmem_full[acc]);     // accumulators ready in both CTAs
              } else {
                if (KIND == 0) {
                  umma_tf32(d_tmem, a_desc, b_desc, idesc, kb != 0 ? 1u : 0u);
                  if (nk > 1) umma_tf32(d_tmem, a_desc + 2, b_desc + 2, idesc, 1u);
                  if (nk > 2) umma_tf32(d_tmem, a_desc + 4, b_desc + 4, idesc, 1u);
                  if (nk > 3) umma_tf32(d_tmem, a_desc + 6, b_desc + 6, idesc, 1u);
                } else if (KIND == 1) {
                  umma_bf16(d_tmem, a_desc, b_desc, idesc, kb != 0 ? 1u : 0u);
                  if (nk > 1) umma_bf16(d_tmem, a_desc + 2, b_desc + 2, idesc, 1u);
                  if (nk > 2) umma_bf16(d_tmem, a_desc + 4, b_desc + 4, idesc, 1u);
                  if (nk > 3) umma_bf16(d_tmem, a_desc + 6, b_desc + 6, idesc, 1u);
                } else {
                  umma_i8(d_tmem, a_desc, b_desc, idesc, kb != 0 ? 1u : 0u);
                  if (nk > 1) umma_i8(d_tmem, a_desc + 2, b_desc + 2, idesc, 1u);
                  if (nk > 2) umma_i8(d_tmem, a_desc + 4, b_desc + 4, idesc, 1u);
                  if (nk > 3) umma_i8(d_tmem, a_desc + 6, b_desc + 6, idesc, 1u);
                }
                umma_commit(&empty_bar[stage]);                       // frees the smem stage once these MMAs retire
                if (kb == n_kb - 1) umma_commit(&tmem_full[acc]);     // accumulator ready for the epilogue
              }
            }
            __syncwarp();
            if (++stage == n_stages) { stage = 0; phase ^= 1; }
          }
          if (++acc == TC_ACC_STAGES) { acc = 0; acc_phase ^= 1; }
        }
        // RES: both CTAs may replace their query tiles once everything issued so far has retired (not after the
        // worker's last unit: no reload waits for it, and no signal may reach a CTA that is leaving)
        if (RES && u + n_workers < n_units) {
          if (elect_one()) umma_commit_pair(a_empty);
          __syncwarp();
        }
      }
    }
  } else if (warp >= TC_EPI_FIRST_WARP) {
    // ===================== epilogue: score, threshold filter, candidate buffers =====================
    const int e = warp - TC_EPI_FIRST_WARP;
    const int lane_grp = warp & 3;               // TMEM lanes this warp may touch: 32*lane_grp ..
    const int half = e >> 2;                     // which 128 columns of the accumulator
    const int row_in_tile = lane_grp * 32 + int(lane);
    const int slot = half * TC_BM + row_in_tile; // candidate buffer of this thread
    const uint32_t t_lane = tmem_base + (uint32_t(lane_grp * 32) << 16) + uint32_t(half * TC_HALF_COLS);
    // PAIR: the accumulator goes back to the leader's MMA warp (arrive in the leader), the norm buffer to this CTA's producer
    const uint32_t tmem_empty_leader = PAIR ? mapa_u32(smem_u32(tmem_empty), 0) : 0u;
    int acc = 0; uint32_t acc_phase = 0;

    for (int u = cid; u < n_units; u += n_workers) {
      int qt, slice, cu; decode(u, qt, slice, cu);
      const int t0 = slice * p.tiles_per_slice, t1 = min(p.n_vtiles, t0 + p.tiles_per_slice);
      // tile row j = lane_grp*32 + lane holds query qt*128 + lane*4 + lane_grp (see knn_prep_kernel): a small
      // batch is spread over all four lane groups, i.e. over all epilogue warps and SM sub-partitions
      const int q = qt * TC_BM + int(lane) * 4 + lane_grp;
      const bool active = q < p.n_q;
      const bool any_active = __any_sync(0xffffffffu, active);
      uint2* buf = p.wbuf + (size_t(cu) * TC_SLOTS + slot) * p.cap;
      uint32_t wn = 0;   // entries in the buffer
      float tau = active ? -INFINITY : INFINITY;   // lanes past the last query never admit anything
      if (p.fixed && active) tau = ord2f(p.tau_g[q]);
      uint32_t wn_trig = epi_trigger(p, active, tau);
      // the shared threshold is re-read once per tile; the load is issued a tile ahead so its L2 latency
      // (hundreds of cycles) never sits on the critical path of the first compare
      const bool poll = active && !p.fixed;
      uint32_t tg_next = poll ? ld_relaxed_u32(p.tau_g + q) : ORD_NEG_INF;
      float4 qs = make_float4(1.f, 0.f, 0.f, 0.f);   // kind 2: (S_q, a_q, e_q) of this lane's query
      if (KIND == 2) { if (active) qs = p.i8_q[q]; }

      for (int tv = t0; tv < t1; ++tv) {
        const int t = tv * p.tile_stride;
        if (poll) {
          tau = fmaxf(tau, ord2f(tg_next));
          tg_next = ld_relaxed_u32(p.tau_g + q);
        }
        float2 ts = make_float2(1.f, 0.f);            // kind 2: (S_t, E_t) of this tile
        if (KIND == 2) ts = __ldg(p.i8_tile + t);
        mbar_wait(&tmem_full[acc], acc_phase);
        if (METRIC != 2) mbar_wait(&norm_full[acc], acc_phase);
        tc_fence_after();
        const int col0 = t * TC_BN + half * TC_HALF_COLS;                  // global row of column 0 of this half
        const int ncols = min(TC_HALF_COLS, n_rows_i - col0);                 // valid columns (<=0: none)
        const float* nrm = norm_smem + acc * TC_BN + half * TC_HALF_COLS;
        float* dbg_row = nullptr;
        if (MODE == 1) { if (u == 0 && tv == t0) dbg_row = p.dbg + (int(lane) * 4 + lane_grp) * TC_BN + half * TC_HALF_COLS; }
        float* pre_out = nullptr;
        if (MODE == 2) { if (active) pre_out = p.pre_max + size_t(q) * p.pre_pitch + (tv * TC_SPLIT + half); }
        if (KIND == 2) {
          const double ss = double(ts.x) * double(qs.x);
          const double ae = fma(double(qs.y), double(ts.y), double(qs.z)) + 0x1p-48;   // a_q E_t + e_q (+ rounding pad)
          epi_tile_i8<METRIC, MODE, (PAIR != 0)>(t_lane + uint32_t(acc * TC_BN), any_active ? ncols : 0, nrm, col0, tau,
                                                    i8_threshold(tau, ss, ae), 1.0 / ss, ae, buf, wn, &tmem_empty[acc],
                                                    tmem_empty_leader + uint32_t(acc) * 8u, &norm_empty[acc], lane, dbg_row, pre_out);
        } else {
          epi_tile<METRIC, MODE, (PAIR != 0)>(t_lane + uint32_t(acc * TC_BN), any_active ? ncols : 0, nrm, col0, tau, buf, wn,
                                                 &tmem_empty[acc], tmem_empty_leader + uint32_t(acc) * 8u, &norm_empty[acc], lane, dbg_row, pre_out);
        }
        if (++acc == TC_ACC_STAGES) { acc = 0; acc_phase ^= 1; }
        if (MODE != 2) epi_tighten(p, active, q, buf, wn, wn_trig, tau, lane);
      }

      // end of unit: the finish kernel reads the buffer in place
      if (MODE != 2) p.wcnt[size_t(cu) * TC_SLOTS + slot] = active ? int(wn) : 0;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();   // neither CTA leaves (or frees TMEM) while the pair's MMAs / barrier signals may still touch it
  if (warp == 2) {
    tc_fence_after();
    if (PAIR) tmem_dealloc_pair(tmem_base, 512); else tmem_dealloc(tmem_base, 512);
  }
}

// ---------------------------------------------------------------------------------------------
// the resident-query filter kernel (narrow rows: D + 3 <= 192 bf16 columns, at least two query tiles)
// ---------------------------------------------------------------------------------------------
// At small D the streaming kernel above is bound by L2 -> SM operand traffic, not by the tensor pipe: every
// 128 x 256 tile re-reads its query block and a corpus block that serves only 128 queries (C2: 9.6 TB/s of
// operand traffic at 0.40 of the bf16 peak). Here one CTA keeps TWO query tiles (256 queries) resident in shared
// memory for a whole unit and streams only corpus blocks of 128 rows; each block feeds two MMAs (one per query
// tile), so operand bytes per flop drop 3-4.5x:
//   smem   A: 2 query tiles x n_kb x 16 KB (loaded once per unit)      B: ring of RQ_STAGES x 16 KB (128 rows x 128 B)
//   TMEM   4 accumulators of 128 columns: (stage 0/1) x (query tile 0/1)
//   warps  0 TMA producer, 1 and 3 MMA issuers (one per query tile), 2 TMEM allocator, 4-7 epilogue of query tile 0,
//          8-11 of query tile 1;
//          every epilogue warp owns 32 queries and scans all 128 columns of its accumulator.
// Units: (query pair) x (corpus slice of 128-row tiles), slice-major like the streaming kernel; candidate lists:
// one per (unit, query).
constexpr int RQ_BN = 128;                       // corpus rows per accumulator
constexpr int RQ_MAX_KB = 3;                     // k-blocks (64 bf16 columns) per row at most
constexpr int RQ_MAX_STAGES = 12;               // ring depth is chosen at launch: whatever shared memory the query tiles leave
constexpr uint32_t RQ_BLOCK_BYTES = 128 * 128;   // 128 rows x 128 B: one k-block of a query tile or of a corpus tile
constexpr uint32_t RQ_NORM_BYTES = RQ_BN * 4;
constexpr uint32_t RQ_SMEM_MAX = 227 * 1024;
constexpr uint32_t RQ_FIXED_BYTES = 1024 /*align slack*/ + 2 * RQ_NORM_BYTES + 512 /*barriers*/;
inline int rq_stages(int n_kblocks) {
  const int s = int((RQ_SMEM_MAX - RQ_FIXED_BYTES - 2u * uint32_t(n_kblocks) * RQ_BLOCK_BYTES) / RQ_BLOCK_BYTES);
  return s < RQ_MAX_STAGES ? s : RQ_MAX_STAGES;
}
inline uint32_t rq_smem_bytes(int n_kblocks) {
  return RQ_FIXED_BYTES + uint32_t(2 * n_kblocks + rq_stages(n_kblocks)) * RQ_BLOCK_BYTES;
}

template <int METRIC, int MODE>   // METRIC 0: score = acc + hx[row] (masked searches), 2: score = acc; MODE 0 filter, 2 prepass
__global__ void __launch_bounds__(TC_THREADS, 1)
knn_rq_filter_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_x, TcParams p) {
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int n_stages = p.rq_stages;
  unsigned char* a_tiles = smem;                                      // [2][n_kblocks] blocks
  unsigned char* b_ring = smem + 2 * p.n_kblocks * RQ_BLOCK_BYTES;    // [n_stages] blocks
  float* norm_smem = reinterpret_cast<float*>(b_ring + n_stages * RQ_BLOCK_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<unsigned char*>(norm_smem) + 2 * RQ_NORM_BYTES);
  uint64_t* full_bar = bars;                      // [RQ_MAX_STAGES] TMA -> MMA
  uint64_t* empty_bar = full_bar + RQ_MAX_STAGES; // [RQ_MAX_STAGES] MMA -> TMA
  uint64_t* a_full = empty_bar + RQ_MAX_STAGES;   // [1]  query tiles of the unit have landed
  uint64_t* a_empty = a_full + 1;                 // [1]  the unit's last MMAs (both issuers) have retired
  uint64_t* tmem_full = a_empty + 1;              // [2][2] per (stage, query tile)
  uint64_t* tmem_empty = tmem_full + 4;           // [2][2] per (stage, query tile), 4 warps each
  uint64_t* norm_full = tmem_empty + 4;           // [2]
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(norm_full + 2);

  const int warp = threadIdx.x >> 5;
  const uint32_t lane = lane_id();
  if (warp == 0 && lane == 0) {
    prefetch_tmap(&map_q);
    prefetch_tmap(&map_x);
    for (int i = 0; i < n_stages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 2); }   // two MMA issuers free a stage
    mbar_init(a_full, 1); mbar_init(a_empty, 2);
    for (int i = 0; i < 2; ++i) mbar_init(&norm_full[i], 1);
    for (int i = 0; i < 4; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], 4); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(tmem_ptr, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  const int n_qp = (p.n_qt + 1) >> 1;
  const int n_units = p.n_slices * n_qp;
  const int n_t128 = p.n_vtiles;   // 128-row tiles the units iterate over
  const int n_rows_i = int(p.n_rows);   // < 2^31 (tc_supported)

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      uint32_t a_phase = 0;
      for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
        const int qp = u % n_qp, slice = u / n_qp;
        const int t0 = slice * p.tiles_per_slice, t1 = min(n_t128, t0 + p.tiles_per_slice);
        // the unit's two query tiles (the previous unit's MMAs must have retired first)
        mbar_wait_backoff(a_empty, a_phase ^ 1, p.sleep_ns);
        mbar_expect_tx(a_full, uint32_t(2 * p.n_kblocks) * RQ_BLOCK_BYTES);
        for (int qt = 0; qt < 2; ++qt)
          for (int kb = 0; kb < p.n_kblocks; ++kb)
            tma_load_2d(&map_q, a_full, a_tiles + (qt * p.n_kblocks + kb) * RQ_BLOCK_BYTES, kb * 64, (qp * 2 + qt) * TC_BM);
        a_phase ^= 1;
        for (int tv = t0; tv < t1; ++tv) {
          const int t = tv * p.tile_stride;
          if (METRIC != 2) {
            // per-row terms of this tile, one buffer per accumulator stage; both query-tile groups must have left it
            mbar_wait_backoff(&tmem_empty[acc * 2 + 0], acc_phase ^ 1, p.sleep_ns);
            mbar_wait_backoff(&tmem_empty[acc * 2 + 1], acc_phase ^ 1, p.sleep_ns);
            mbar_expect_tx(&norm_full[acc], RQ_NORM_BYTES);
            bulk_load_1d(norm_smem + acc * RQ_BN, p.hx + size_t(t) * RQ_BN, RQ_NORM_BYTES, &norm_full[acc]);
          }
          // corpus tile t = rows [128 t, 128 t + 128) = half (t & 1) of the shadow's 256-row block t >> 1
          const int blk = t >> 1, hrow = (t & 1) * RQ_BN;
          for (int kb = 0; kb < p.n_kblocks; ++kb) {
            mbar_wait_backoff(&empty_bar[stage], phase ^ 1, p.sleep_ns);
            mbar_expect_tx(&full_bar[stage], RQ_BLOCK_BYTES);
            const int line = (kb < p.n_kb_data ? (blk * p.n_kb_data + kb) * TC_BN : p.aug_line0 + blk * TC_BN) + hrow;
            tma_load_2d(&map_x, &full_bar[stage], b_ring + stage * RQ_BLOCK_BYTES, 0, line);
            if (++stage == n_stages) { stage = 0; phase ^= 1; }
          }
          if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
      }
    }
  } else if (warp == 1 || warp == 3) {
    // ===================== MMA issuers: warp 1 feeds query tile 0, warp 3 query tile 1 =====================
    // One thread issuing every tcgen05.mma of the CTA was the bottleneck of this kernel (about 18 scalar instructions
    // per MMA, 80 % busy): the two query tiles are independent GEMMs over the same corpus block, so each gets its
    // own issuer and accumulator barriers. The whole warp runs the loop (warp-uniform control flow keeps descriptors
    // and addresses in uniform registers; under `if (lane == 0)` the compiler wraps every MMA in a broadcast loop);
    // one elected lane issues.
    {
      constexpr uint32_t idesc = make_idesc_bf16(TC_BM, RQ_BN);
      const int qt = warp >> 1;
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint64_t desc0 = make_smem_desc(0);
      const uint32_t a_lo = (smem_u32(a_tiles) + uint32_t(qt * p.n_kblocks) * RQ_BLOCK_BYTES) >> 4;   // k-block kb: + kb * 1024
      const uint32_t b_lo = smem_u32(b_ring) >> 4;                                                    // stage s:    + s * 1024
      const int n_kb = p.n_kblocks, n_kb_data = p.n_kb_data, nk_last = p.nk_last;
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      uint32_t a_phase = 0;
      for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
        const int slice = u / n_qp;
        const int t0 = slice * p.tiles_per_slice, t1 = min(n_t128, t0 + p.tiles_per_slice);
        mbar_wait(a_full, a_phase);
        a_phase ^= 1;
        for (int t = t0; t < t1; ++t) {
          mbar_wait_backoff(&tmem_empty[acc * 2 + qt], acc_phase ^ 1, p.sleep_ns >> 1);
          const uint32_t d_tmem = tmem_u + uint32_t((acc * 2 + qt) * RQ_BN);
          for (int kb = 0; kb < n_kb; ++kb) {
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
            const uint64_t a_desc = desc0 | uint64_t(a_lo + uint32_t(kb) * (RQ_BLOCK_BYTES >> 4));
            const uint64_t b_desc = desc0 | uint64_t(b_lo + uint32_t(stage) * (RQ_BLOCK_BYTES >> 4));
            const int nk = kb < n_kb_data - 1 ? 4 : (kb == n_kb_data - 1 ? nk_last : 1);
            if (elect_one()) {
              umma_bf16(d_tmem, a_desc, b_desc, idesc, kb != 0 ? 1u : 0u);
              if (nk > 1) umma_bf16(d_tmem, a_desc + 2, b_desc + 2, idesc, 1u);
              if (nk > 2) umma_bf16(d_tmem, a_desc + 4, b_desc + 4, idesc, 1u);
              if (nk > 3) umma_bf16(d_tmem, a_desc + 6, b_desc + 6, idesc, 1u);
              umma_commit(&empty_bar[stage]);
              if (kb == n_kb - 1) umma_commit(&tmem_full[acc * 2 + qt]);
            }
            __syncwarp();
            if (++stage == n_stages) { stage = 0; phase ^= 1; }
          }
          if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
        if (elect_one()) umma_commit(a_empty);   // the resident query tiles may be replaced once everything issued so far has retired
        __syncwarp();
      }
    }
  } else if (warp >= TC_EPI_FIRST_WARP) {
    // ===================== epilogue =====================
    const int e = warp - TC_EPI_FIRST_WARP;
    const int lane_grp = warp & 3;
    const int qt_l = e >> 2;                      // which of the unit's two query tiles
    const int slot = qt_l * TC_BM + lane_grp * 32 + int(lane);
    const uint32_t t_lane = tmem_base + (uint32_t(lane_grp * 32) << 16) + uint32_t(qt_l * RQ_BN);
    int acc = 0; uint32_t acc_phase = 0;
    for (int u = blockIdx.x; u < n_units; u += gridDim.x) {
      const int qp = u % n_qp, slice = u / n_qp;
      const int t0 = slice * p.tiles_per_slice, t1 = min(n_t128, t0 + p.tiles_per_slice);
      const int q = (qp * 2 + qt_l) * TC_BM + int(lane) * 4 + lane_grp;
      const bool active = q < p.n_q;
      uint2* buf = p.wbuf + (size_t(u) * TC_SLOTS + slot) * p.cap;
      uint32_t wn = 0;
      float tau = active ? -INFINITY : INFINITY;
      if (p.fixed && active) tau = ord2f(p.tau_g[q]);
      uint32_t wn_trig = epi_trigger(p, active, tau);
      const bool any_active = __any_sync(0xffffffffu, active);
      const bool poll = active && !p.fixed;
      uint32_t tg_next = poll ? ld_relaxed_u32(p.tau_g + q) : ORD_NEG_INF;
      for (int tv = t0; tv < t1; ++tv) {
        const int t = tv * p.tile_stride;
        if (poll) {
          tau = fmaxf(tau, ord2f(tg_next));
          tg_next = ld_relaxed_u32(p.tau_g + q);
        }
        mbar_wait(&tmem_full[acc * 2 + qt_l], acc_phase);
        if (METRIC != 2) mbar_wait(&norm_full[acc], acc_phase);
        tc_fence_after();
        const int col0 = t * RQ_BN;
        const int ncols = min(RQ_BN, n_rows_i - col0);
        float* pre_out = nullptr;
        if (MODE == 2) { if (active) pre_out = p.pre_max + size_t(q) * p.pre_pitch + tv; }
        epi_tile<METRIC, MODE>(t_lane + uint32_t(acc * 2 * RQ_BN), any_active ? ncols : 0,
                               norm_smem + acc * RQ_BN, col0, tau, buf, wn, &tmem_empty[acc * 2 + qt_l], 0u, nullptr, lane, nullptr, pre_out);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        if (MODE != 2) epi_tighten(p, active, q, buf, wn, wn_trig, tau, lane);
      }
      if (MODE != 2) p.wcnt[size_t(u) * TC_SLOTS + slot] = active ? int(wn) : 0;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---------------------------------------------------------------------------------------------
// query preparation: pad to the TMA pitch, reset per-query state
// ---------------------------------------------------------------------------------------------
// Error weight of every query for the certified upper-bound scores: qerr[q] = c |q| (fp64 norm, rounded up to fp32 with
// a 2^-10 relative margin that also covers the bf16 round-up of the two factors being applied AFTER this product bound).
__global__ void __launch_bounds__(128)
knn_qerr_kernel(const float* __restrict__ Q, int n_q, int dim, double c, float* __restrict__ qerr) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n_q) return;
  double s = 0.0;
  for (int d = lane; d < dim; d += 32) { const double v = double(Q[size_t(warp) * dim + d]); s = fma(v, v, s); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) qerr[warp] = __double2float_ru(c * sqrt(s) * (1.0 + 1.0 / 1024.0));
}

__global__ void knn_prep_kernel(const float* __restrict__ Q, int n_q, int n_rows_p, int dim, int pitch, float* __restrict__ Qp,
                                uint32_t* __restrict__ tau_g, int* __restrict__ flags,
                                __nv_bfloat16* __restrict__ Qb, int pitch_b,
                                const uint32_t* __restrict__ tau_fixed, int aug_col, int* __restrict__ n_flagged,
                                int aug_mode, const float* __restrict__ qerr) {
  if (blockIdx.x == 0 && threadIdx.x == 0) *n_flagged = 0;
  // Rows are written in TILE order: row qt*128 + j holds query qt*128 + (j % 32) * 4 + j / 32 (zeros past the last
  // query), so that consecutive queries land in different TMEM lane groups.
  // n_rows_p: rows of the padded query matrices (whole tile pairs)
  const int64_t total = int64_t(n_rows_p) * pitch;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
    int row = int(i / pitch), d = int(i - int64_t(row) * pitch);
    int j = row % TC_BM;
    int q = row - j + (j % 32) * 4 + j / 32;
    Qp[i] = (d < dim && q < n_q) ? Q[size_t(q) * dim + d] : 0.f;
  }
  if (Qb != nullptr) {
    const int64_t total_b = int64_t(n_rows_p) * pitch_b;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total_b; i += int64_t(gridDim.x) * blockDim.x) {
      int row = int(i / pitch_b), d = int(i - int64_t(row) * pitch_b);
      int j = row % TC_BM;
      int q = row - j + (j % 32) * 4 + j / 32;
      float v = (d < dim && q < n_q) ? Q[size_t(q) * dim + d] : 0.f;
      if (aug_col > 0 && q < n_q && d >= aug_col && d < aug_col + 3 && aug_mode == 1) v = 1.f;   // picks up the shadow's three -|x|^2/2 columns
      if (aug_col > 0 && q < n_q && d == aug_col + 3) {
        Qb[i] = __float2bfloat16_ru(qerr[q]);            // u = c |q|, rounded UP (times the row's |x|, also rounded up)
        continue;
      }
      Qb[i] = __float2bfloat16_rn(v);
    }
  }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_q; i += gridDim.x * blockDim.x) {
    tau_g[i] = tau_fixed ? tau_fixed[i] : ORD_NEG_INF;
    flags[i] = 0;
  }
}

// Quantised queries of the int8 filter (kind 2, format above i8_scale): one warp per row of the padded int8 query matrix
// (tile order, as knn_prep_kernel; pitch8 bytes per row, zeros past the data and in pad rows), and (S_q, a_q, e_q) per
// query. A zero query quantises to zeros with a_q = e_q = 0.
__global__ void __launch_bounds__(256)
knn_qprep_i8_kernel(const float* __restrict__ Q, int n_q, int n_rows_p, int dim, int pitch8, int8_t* __restrict__ Q8,
                    float4* __restrict__ qstat) {
  const int row = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (row >= n_rows_p) return;
  const int j = row % TC_BM;
  const int q = row - j + (j % 32) * 4 + j / 32;
  int8_t* out = Q8 + size_t(row) * pitch8;
  if (q >= n_q) {
    for (int d = lane; d < pitch8; d += 32) out[d] = 0;
    return;
  }
  const float* qv = Q + size_t(q) * dim;
  double s = 0.0; float mx = 0.f;
  for (int d = lane; d < dim; d += 32) { const float v = qv[d]; s = fma(double(v), double(v), s); mx = fmaxf(mx, fabsf(v)); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o)); }
  const double nq = sqrt(s), inv = 1.0 / (nq > 1e-12 ? nq : 1e-12);
  const float scale = i8_scale(double(mx) * inv);
  const double inv_s = 1.0 / double(scale);
  double rr = 0.0, qq = 0.0;   // |q^ - q~/S|^2, |q~|^2
  for (int d = lane; d < pitch8; d += 32) {
    int v = 0;
    if (d < dim) {
      const double h = double(qv[d]) * inv;
      v = i8_quant(h, scale);
      const double r = h - double(v) * inv_s;
      rr = fma(r, r, rr); qq += double(v * v);
    }
    out[d] = int8_t(v);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { rr += __shfl_xor_sync(0xffffffffu, rr, o); qq += __shfl_xor_sync(0xffffffffu, qq, o); }
  if (lane == 0) {
    const double pad = 1.0 + 0x1p-40;   // the fp64 sums' rounding
    qstat[q] = make_float4(scale, __double2float_ru(sqrt(qq) * inv_s * pad), __double2float_ru(sqrt(rr) * pad), 0.f);
  }
}

// ---------------------------------------------------------------------------------------------
// finish: select K' by approximate score, exact rerank, sort, certificate
// ---------------------------------------------------------------------------------------------
constexpr int FIN_POOL = 2048;   // candidates the finish kernel can hold in shared memory

struct FinishParams {
  const float* X; int pitch; int dim; int64_t row_base;
  const float* Qp; int n_q; int n_qt; int n_slices; int cap; int metric; int k; int kp; int sort2;  // sort2: pow2 >= kp
  const uint32_t* tau_g; const uint2* wbuf; const int* wcnt; int rq; int n_qp;
  int* flags; int certify; float max_norm; double c_err; double c_add; double c_abs;
  int64_t* out_rows; float* out_dist;
  int* n_flagged;   // counts the queries this launch flags (read back by the host together with the results)
  int unit_q;       // 1: scores are cosine upper bounds of the NORMALISED query (int8 filter), not scaled by |q|
};

// Candidate list l of query tile qt, tile row r (the query's slot) - the layout every filter kernel writes: with the
// resident-query kernel one list per slice (its unit holds two query tiles), else list l = (slice, half), the buffer of
// thread slot half*128 + r of unit slice*n_qt + qt. count: its entries.
__device__ __forceinline__ const uint2* fin_list(const FinishParams& p, int qt, int r, int l, int& count) {
  size_t unit_slot;
  if (p.rq) {
    unit_slot = (size_t(l) * p.n_qp + (qt >> 1)) * TC_SLOTS + (qt & 1) * TC_BM + r;
  } else {
    const int slice = l / TC_SPLIT, half = l % TC_SPLIT;
    unit_slot = size_t(slice * p.n_qt + qt) * TC_SLOTS + half * TC_BM + r;
  }
  count = p.wcnt[unit_slot];
  return p.wbuf + unit_slot * p.cap;
}

// THE summation order of every exact distance this library reports from 8-lane groups (the finish kernels here and
// direct_scan.cuh, bit for bit): per lane one accumulator per float4 component over j = sub, sub + 8, ...; lane
// total = (x + y) + (z + w); then the xor tree over the 8 lanes. Four independent chains per sum: the fp64 pipe's
// latency, not its rate, bounded the single-chain form. Every lane of the warp calls it (the shuffles); xx = |x|^2 and
// qx = <q, x> of the group's row come back in every lane of the group.
__device__ __forceinline__ void rerank8(const float* X, int pitch, uint32_t row, bool live, const float* qs, int sub,
                                        double& xx, double& qx) {
  const float4* xp = reinterpret_cast<const float4*>(X + size_t(row) * pitch);
  const int n4 = pitch >> 2;
  double xa[4] = {0.0, 0.0, 0.0, 0.0}, qa[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll 4
  for (int j = sub; j < n4; j += 8) {
    const float4 xv = live ? __ldg(xp + j) : make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 qv = *reinterpret_cast<const float4*>(qs + 4 * j);
    xa[0] = fma(double(xv.x), double(xv.x), xa[0]); qa[0] = fma(double(xv.x), double(qv.x), qa[0]);
    xa[1] = fma(double(xv.y), double(xv.y), xa[1]); qa[1] = fma(double(xv.y), double(qv.y), qa[1]);
    xa[2] = fma(double(xv.z), double(xv.z), xa[2]); qa[2] = fma(double(xv.z), double(qv.z), qa[2]);
    xa[3] = fma(double(xv.w), double(xv.w), xa[3]); qa[3] = fma(double(xv.w), double(qv.w), qa[3]);
  }
  xx = (xa[0] + xa[1]) + (xa[2] + xa[3]); qx = (qa[0] + qa[1]) + (qa[2] + qa[3]);
#pragma unroll
  for (int o = 4; o > 0; o >>= 1) {
    xx += __shfl_xor_sync(0xffffffffu, xx, o);
    qx += __shfl_xor_sync(0xffffffffu, qx, o);
  }
}

// Error bound E of a query's filter scores (score units; nq = |q|, or 1 with unit_q; xm = the shard's max |x|), shared by
// the certificate and the preset thresholds. c_err / c_add: the relative bounds (0 where the score already is an upper
// bound); c_abs: products and partial sums below FLT_MIN, which the tensor cores may lose (tc_c_abs), multiplied for
// cosine by the epilogue's row factor 1/max(|x|, 1e-12) <= 1e12. NaN when a product or partial sum of the filter could
// overflow fp32 (|q| |x| + |x|^2/2 near FLT_MAX): its score may then be +-inf or NaN, which no threshold bounds.
__device__ __forceinline__ double score_error(int metric, double nq, double xm, double c_err, double c_add, double c_abs,
                                              int unit_q) {
  double e_abs, span;
  if (metric == 0) {
    e_abs = c_err * nq * xm + c_add * (0.5 * xm * xm + nq * xm) + c_abs;
    span = nq * xm + 0.5 * xm * xm;
  } else if (metric == 1) {
    e_abs = nq * (c_err + 1e-6) + c_abs * 1e12;
    span = nq * fmax(xm, 1.0);
  } else {
    e_abs = c_err * nq * xm + c_abs;
    span = nq * xm;
  }
  return (unit_q || span < 0x1p126) ? e_abs : __longlong_as_double(0x7ff8000000000000ll);
}

// One CTA per query. The query's candidates live in 2 * n_slices buffers (one per unit-half).
//  1. block-wide radix select (4 passes of 8 bits over the ordered score bits) finds the K'-th best
//     approximate score among the entries above the final shared threshold;
//  2. the <= K' winners are re-ranked exactly (fp64 accumulation, one warp per candidate);
//  3. bitonic sort by (distance, row), write top-k, evaluate the certificate.
__global__ void __launch_bounds__(1024)
knn_tc_finish_kernel(FinishParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint64_t* keys2 = reinterpret_cast<uint64_t*>(smem_raw);                 // [sort2] (distance,row) keys
  uint32_t* cand = reinterpret_cast<uint32_t*>(keys2 + p.sort2);           // [sort2] candidate rows
  float* qs = reinterpret_cast<float*>(cand + p.sort2);                    // [pitch]
  uint2* pool = reinterpret_cast<uint2*>(qs + p.pitch);                    // [FIN_POOL] gathered candidates (pitch is a multiple of 4 floats)
  __shared__ int hist[256];
  __shared__ int s_n_gt, s_n_tie, s_total;
  __shared__ uint32_t s_prefix;
  __shared__ int s_remaining;
  __shared__ double s_qq;
  const int q = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int n_warps = blockDim.x >> 5;
  const int qt = q / TC_BM, w = q - qt * TC_BM;
  const int r = (w % 4) * 32 + w / 4;               // tile row / candidate-buffer slot of this query
  const size_t q_row = size_t(qt) * TC_BM + r;      // its row in the (tile-ordered) padded query matrix
  const int n_lists = (p.rq ? 1 : TC_SPLIT) * p.n_slices;

  for (int d = tid; d < p.pitch; d += blockDim.x) qs[d] = p.Qp[q_row * p.pitch + d];
  if (tid == 0) { s_n_gt = 0; s_n_tie = 0; s_prefix = 0; s_remaining = p.kp; }
  __syncthreads();
  if (warp == 0) {
    double s = 0.0;
    for (int d = lane; d < p.pitch; d += 32) s = fma(double(qs[d]), double(qs[d]), s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) s_qq = s;
  }
  const uint32_t tg = p.tau_g[q];
  const bool overflowed = p.flags[q] != 0;   // set by the filter kernel in refinement mode

  auto list_ptr = [&](int l, int& count) -> const uint2* { return fin_list(p, qt, r, l, count); };

  // ---- 0. gather: one pass over the query's lists copies every entry at or above the final threshold into a
  // shared-memory pool, so the selection passes below never touch global memory again (with hundreds of short
  // lists per query - the small-batch regime - five dependent sweeps over them dominated the search latency).
  // If the pool overflows (thresholds still loose) the selection falls back to sweeping the lists.
  __shared__ int s_pool_n;
  if (tid == 0) s_pool_n = 0;
  __syncthreads();
  for (int l = warp; l < n_lists; l += n_warps) {
    int count; const uint2* b = list_ptr(l, count);
    for (int i0 = 0; i0 < count; i0 += 128) {
      // four independent loads per lane in flight, then four warp-aggregated appends
      uint2 ent[4]; bool ok[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int i = i0 + j * 32 + lane;
        ent[j] = (i < count) ? b[i] : make_uint2(0u, 0u);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int i = i0 + j * 32 + lane;
        ok[j] = (i < count) && f2ord(__uint_as_float(ent[j].x)) >= tg;
        const uint32_t ballot = __ballot_sync(0xffffffffu, ok[j]);
        if (ballot == 0u) continue;
        int base = 0;
        if (lane == 0) base = atomicAdd(&s_pool_n, __popc(ballot));
        base = __shfl_sync(0xffffffffu, base, 0);
        const int pos = base + __popc(ballot & ((1u << lane) - 1u));
        if (ok[j] && pos < FIN_POOL) pool[pos] = ent[j];
      }
    }
  }
  __syncthreads();
  const int pool_n = s_pool_n;
  const bool pooled = pool_n <= FIN_POOL;
  // visit every candidate entry (o = ordered score, row): from the pool, or from the lists when it overflowed
  auto for_each = [&](auto&& fn) {
    if (pooled) {
      for (int i = tid; i < pool_n; i += blockDim.x) fn(f2ord(__uint_as_float(pool[i].x)), pool[i].y);
    } else {
      for (int l = warp; l < n_lists; l += n_warps) {
        int count; const uint2* b = list_ptr(l, count);
        for (int i = lane; i < count; i += 32) {
          const uint2 ent = b[i];
          const uint32_t o = f2ord(__uint_as_float(ent.x));
          if (o >= tg) fn(o, ent.y);
        }
      }
    }
  };

  // ---- 1. radix select of the kp-th largest ordered score among entries >= tg ----
  uint32_t prefix = 0, mask = 0;
  bool keep_all = false;
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    for (int i = tid; i < 256; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    for_each([&](uint32_t o, uint32_t) {
      if ((o & mask) == prefix) atomicAdd(&hist[(o >> shift) & 0xffu], 1);
    });
    __syncthreads();
    if (warp == 0) {
      // find the highest bin b with sum(hist[b..255]) >= remaining: each lane owns 8 bins, suffix sums across lanes
      const int remaining = s_remaining;
      int h[8], lane_sum = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) { h[j] = hist[8 * lane + j]; lane_sum += h[j]; }
      int suffix = lane_sum;                                   // inclusive sum over lanes >= this one
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int up = __shfl_down_sync(0xffffffffu, suffix, o);
        if (lane + o < 32) suffix += up;
      }
      const int total = __shfl_sync(0xffffffffu, suffix, 0);
      if (pass == 0 && lane == 0) s_total = total;
      if (pass == 0 && total <= p.kp) {
        if (lane == 0) s_remaining = -1;                       // keep everything above tg
      } else {
        const uint32_t reach = __ballot_sync(0xffffffffu, suffix >= remaining);
        const int owner = reach ? 31 - __clz(reach) : 0;       // highest lane whose suffix reaches `remaining`
        if (lane == owner) {
          int cum = suffix - lane_sum, b = 8 * lane + 7;       // cum: everything in higher lanes
          for (int j = 7; j >= 0; --j, --b) {
            if (cum + h[j] >= remaining || b == 0) break;
            cum += h[j];
          }
          s_prefix = prefix | (uint32_t(b) << shift);
          s_remaining = remaining - cum;
        }
      }
    }
    __syncthreads();
    if (s_remaining < 0) { keep_all = true; break; }
    prefix = s_prefix;
    mask |= 0xffu << shift;
  }
  const uint32_t pivot = keep_all ? tg : prefix;          // kp-th best ordered score (or the threshold)
  const int ties_wanted = keep_all ? 0 : s_remaining;      // entries == pivot still admitted

  // ---- collect winners: score > pivot, plus `ties_wanted` entries equal to the pivot ----
  for_each([&](uint32_t o, uint32_t row) {
    if (o > pivot || (keep_all && o == pivot)) {
      int pos = atomicAdd(&s_n_gt, 1);
      if (pos < p.sort2) cand[pos] = row;
    } else if (!keep_all && o == pivot) {
      int t = atomicAdd(&s_n_tie, 1);
      if (t < ties_wanted) cand[p.kp - 1 - t] = row;    // ties fill the tail of the kp slots
    }
  });
  __syncthreads();
  // winners occupy cand[0, n_gt) and (when a pivot exists) cand[kp - n_tie_kept, kp)
  const int n_gt = min(s_n_gt, p.sort2);
  const int n_tie_kept = keep_all ? 0 : min(s_n_tie, ties_wanted);
  const int n_cand = n_gt + n_tie_kept;

  // ---- 2. exact rerank: one warp per candidate, fp64 accumulation of exact fp32 products ----
  // Eight lanes per candidate, four candidates per warp and step: the four row loads are independent (one memory
  // round trip per four candidates; the rows are scattered over the shard) and the fp64 reduction is three shuffle
  // rounds instead of five (the kernel is instruction-bound: 70 % issue utilisation on C2, half of it here).
  const double qq = s_qq;
  {
    const int sub = lane & 7, grp = lane >> 3;
    for (int c0 = warp * 4; c0 < p.sort2; c0 += n_warps * 4) {
      const int c = c0 + grp;
      const bool live = c < n_gt || (!keep_all && c >= p.kp - n_tie_kept && c < p.kp);
      const uint32_t row = live ? cand[c] : 0u;
      double xx, qx;
      rerank8(p.X, p.pitch, row, live, qs, sub, xx, qx);
      if (sub == 0 && c < p.sort2) keys2[c] = live ? make_key(finish_distance(p.metric, qq, xx, qx), row) : KEY_PAD;
    }
  }
  __syncthreads();
  // ---- 3. sort by (distance, row), output, certificate ----
  for (int size = 2; size <= p.sort2; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = tid; i < (p.sort2 >> 1); i += blockDim.x) {
        int pos = 2 * i - (i & (stride - 1));
        int j = pos + stride;
        bool up = (pos & size) == 0;
        uint64_t a = keys2[pos], b = keys2[j];
        if ((a > b) == up) { keys2[pos] = b; keys2[j] = a; }
      }
      __syncthreads();
    }
  }
  for (int i = tid; i < p.k; i += blockDim.x) {
    uint64_t key = (i < p.sort2) ? keys2[i] : KEY_PAD;
    bool pad = key == KEY_PAD;
    p.out_rows[size_t(q) * p.k + i] = pad ? int64_t(-1) : p.row_base + int64_t(key & 0xffffffffull);
    p.out_dist[size_t(q) * p.k + i] = pad ? __int_as_float(0x7f800000) : ord2f(uint32_t(key >> 32));
  }
  if (tid == 0) {
    int flag = 0;
    if (p.certify) {
      // every row that is not a candidate has approximate score <= T
      const float t_score = ord2f(pivot);
      const double nq = p.unit_q ? 1.0 : sqrt(qq);
      const double e_abs = score_error(p.metric, nq, double(p.max_norm), p.c_err, p.c_add, p.c_abs, p.unit_q);
      double lb;
      if (p.metric == 0) {
        double d2 = qq - 2.0 * (double(t_score) + e_abs);
        lb = sqrt(d2 > 0.0 ? d2 : 0.0);   // (a NaN bound clamps to 0: no distance is below it)
      } else if (p.metric == 1) {
        lb = 0.5 - 0.5 * (double(t_score) + e_abs) / (nq > 1e-12 ? nq : 1e-12);
      } else {
        lb = -(double(t_score) + e_abs);
      }
      lb = lb - 1e-6 * fabs(lb) - 1e-37;
      bool ok = false;
      if (n_cand >= p.k && s_n_gt <= p.sort2 && !overflowed) {
        float dk = ord2f(uint32_t(keys2[p.k - 1] >> 32));
        ok = double(dk) < lb;   // NaN compares false -> flagged
      }
      flag = ok ? 0 : (n_cand < p.k ? 2 : 1);   // 2: fewer than k candidates at all (no k-th distance to refine from)
    }
    p.flags[q] = flag;
    if (flag) atomicAdd(p.n_flagged, 1);
  }
}

// Threshold prepass, second half: a group of T threads per query (T = 32 ... 256, 16 records per thread) picks the
// m-th largest of the query's n_rec (<= 4096) block maxima - held in registers, bisection on the order-preserving
// uint encoding - and makes it the query's initial threshold. The m-th largest block maximum is never above the
// m-th largest sample score, so it errs on the loose (safe, cheap) side.
constexpr int TAU0_PER = 16;
template <int T>
__global__ void __launch_bounds__(256)
knn_tc_tau0_kernel(const float* __restrict__ pre_max, int n_q, int n_rec, int m, uint32_t* __restrict__ tau_g) {
  constexpr int W = T / 32;                   // warps per query
  __shared__ int s_cnt[2][8];
  const int tid = threadIdx.x, sub = tid % T, grp = tid / T;
  const int q = blockIdx.x * (256 / T) + grp;
  const bool live = q < n_q;
  const float* rec = pre_max + size_t(live ? q : 0) * n_rec;
  uint32_t o[TAU0_PER];
#pragma unroll
  for (int i = 0; i < TAU0_PER; ++i) {
    const int idx = i * T + sub;
    o[i] = (live && idx < n_rec) ? f2ord(rec[idx]) : 0u;
  }
  uint32_t v = 0;   // largest value with count(x >= v) >= m
  for (int bit = 31; bit >= 0; --bit) {
    const uint32_t cand = v | (1u << bit);
    int c = 0;
#pragma unroll
    for (int i = 0; i < TAU0_PER; ++i) c += o[i] >= cand ? 1 : 0;
    c = __reduce_add_sync(0xffffffffu, c);
    if (W > 1) {
      int* cnt = s_cnt[bit & 1];
      if ((tid & 31) == 0) cnt[tid >> 5] = c;
      __syncthreads();
      c = 0;
#pragma unroll
      for (int w = 0; w < W; ++w) c += cnt[grp * W + w];
    }
    if (c >= m) v = cand;
  }
  if (live && sub == 0) tau_g[q] = v > ORD_NEG_INF ? v : ORD_NEG_INF;
}

// Preset admission threshold (ordered encoding) for the rows at distance <= dk of a query with |q|^2 = qq: every such
// row has exact score >= s(dk), hence filter score >= s(dk) - E (E: score_error of the operand in use; unit_q: see
// FinishParams). dk = +inf admits everything; ORD_SCAN when E is undefined (the filter's sums could overflow).
__device__ __forceinline__ uint32_t admission_threshold(int metric, double qq, double dk, float max_norm, double c_err,
                                                        double c_add, double c_abs, int unit_q) {
  const double nq = unit_q ? 1.0 : sqrt(qq);
  const double e_abs = score_error(metric, nq, double(max_norm), c_err, c_add, c_abs, unit_q);
  dk = dk + 1e-6 * fabs(dk) + 1e-37;            // a row at distance <= dk (after fp32 rounding) must survive
  double score;
  if (metric == 0) score = 0.5 * (qq - dk * dk);
  else if (metric == 1) score = (1.0 - 2.0 * dk) * (nq > 1e-12 ? nq : 1e-12);
  else score = -dk;
  double t = score - e_abs;
  t = t - 1e-6 * fabs(t) - 1e-30;
  float tf = __double2float_rd(t);
  return t != t ? ORD_SCAN : (dk < 1e300 ? f2ord(tf) : ORD_NEG_INF);
}

// Refinement of flagged queries. One block per flagged query i (original index qlist[i]): gathers the query
// into Qr[i] and derives the preset admission threshold from the k-th distance d_k of the first pass:
// every row that can still beat d_k has exact score > s(d_k), hence filter score > s(d_k) - E.
__global__ void __launch_bounds__(128)
refine_prep_kernel(const float* __restrict__ Q, const int* __restrict__ qlist, int dim, int metric, int k,
                   const float* __restrict__ dist, float max_norm, double c_err, double c_add, double c_abs,
                   float* __restrict__ Qr, uint32_t* __restrict__ tau_fixed, int unit_q) {
  __shared__ double part[4];
  const int i = blockIdx.x, q = qlist[i];
  double s = 0.0;
  for (int d = threadIdx.x; d < dim; d += blockDim.x) {
    float v = Q[size_t(q) * dim + d];
    Qr[size_t(i) * dim + d] = v;
    s = fma(double(v), double(v), s);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    const double qq = part[0] + part[1] + part[2] + part[3];
    tau_fixed[i] = admission_threshold(metric, qq, double(dist[size_t(q) * k + (k - 1)]), max_norm, c_err, c_add, c_abs, unit_q);
  }
}

// Preset thresholds of a range search (fx_search_range): the same derivation from the radius, for every query.
// One warp per query; the queries stay where they are.
__global__ void __launch_bounds__(128)
range_prep_kernel(const float* __restrict__ Q, int n_q, int dim, int metric, float radius, float max_norm, double c_err,
                  double c_add, double c_abs, int unit_q, uint32_t* __restrict__ tau_fixed) {
  const int q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (q >= n_q) return;
  double s = 0.0;
  for (int d = lane; d < dim; d += 32) { const double v = double(Q[size_t(q) * dim + d]); s = fma(v, v, s); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) tau_fixed[q] = admission_threshold(metric, s, double(radius), max_norm, c_err, c_add, c_abs, unit_q);
}

// Copy refined results of the queries whose certificate now holds back to their slots.
__global__ void refine_scatter_kernel(const int* __restrict__ qlist, const int* __restrict__ flags2, int n_f, int k,
                                      const int64_t* __restrict__ rows2, const float* __restrict__ dist2,
                                      int64_t* __restrict__ out_rows, float* __restrict__ out_dist) {
  const int64_t total = int64_t(n_f) * k;
  for (int64_t t = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; t < total; t += int64_t(gridDim.x) * blockDim.x) {
    const int i = int(t / k), j = int(t - int64_t(i) * k);
    if (flags2 == nullptr || flags2[i] == 0) {
      out_rows[size_t(qlist[i]) * k + j] = rows2[t];
      out_dist[size_t(qlist[i]) * k + j] = dist2[t];
    }
  }
}

// Masked search (reference: `data.filter(expr)` before the distance column, index.py:161): fold the row mask
// into the per-row epilogue term so masked rows can never pass the threshold test:
//   additive term (L2: -0.5|x|^2, IP: 0) -> -inf;  multiplicative term (cosine 1/|x|) -> NaN (NaN > tau is false);
//   the int8 filter's integer row term (mode 3): 0 -> I8_MASKED, below every integer threshold (i8_threshold)
__global__ void masked_norms_kernel(const uint8_t* __restrict__ mask, const float* __restrict__ base, int64_t n_rows,
                                    int64_t n_alloc, int mode /*0 add-from-base, 1 mul-from-base, 2 add-zero, 3 int8 term*/,
                                    float* __restrict__ out) {
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n_alloc; i += int64_t(gridDim.x) * blockDim.x) {
    float v;
    if (i >= n_rows) v = 0.f;
    else if (mode == 3) v = __int_as_float(mask[i] ? 0 : I8_MASKED);
    else if (mask[i]) v = mode == 2 ? 0.f : base[i];
    else v = mode == 1 ? __int_as_float(0x7fc00000) : -INFINITY;
    out[i] = v;
  }
}

// fp32 rows -> bf16 shadow (round to nearest even) in the filter's streaming layout: for every corpus tile of
// 256 rows and every k-block of 64 elements, the 256 x 64 sub-block is stored contiguously (32 KB), i.e.
//   element (r, d) lives at ((tile * KB + kb) * 256 + r % 256) * 64 + d % 64,  tile = r / 256, kb = d / 64.
// One TMA box of the filter kernel is then a single contiguous 32 KB read. Pad rows / columns are zero.
//   mode 0 (plain + augmented): columns [0, dim) = x, columns dim..dim+2 = -|x|^2/2 split into three bf16 terms
//          (hi + mid + lo reproduce the fp32 value exactly), so that an L2 query [q, 1, 1, 1] gets
//          q.x - |x|^2/2 straight out of the MMA and the epilogue needs no per-row term; an inner-product query
//          (zeros there) ignores them.
//   mode 1 (normalised): columns [0, dim) = x / max(|x|, eps): cosine scores straight out of the MMA.
__global__ void to_bf16_tiled_kernel(const float* __restrict__ X, int64_t n_rows, int pitch, int dim,
                                     const float* __restrict__ hx, const float* __restrict__ rx, int mode,
                                     __nv_bfloat16* __restrict__ Xb, int n_kb, int64_t n_tiles, int aug_col, int aug_blocks,
                                     float h_scale) {
  const int64_t total = n_tiles * (n_kb + aug_blocks) * int64_t(TC_BN) * 32;   // bf16 pairs
  const int64_t main_pairs = n_tiles * n_kb * int64_t(TC_BN) * 32;
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
    const int dd = int(i & 31) * 2;
    int64_t line = i >> 5;                            // (tile * KB + kb) * 256 + rr, or past the data: tile * 256 + rr
    const bool in_aug = i >= main_pairs;
    if (in_aug) line -= main_pairs >> 5;
    const int rr = int(line % TC_BN);
    const int64_t blk = line / TC_BN;
    const int kb = in_aug ? n_kb : int(blk % n_kb);
    const int64_t r = (in_aug ? blk : blk / n_kb) * TC_BN + rr;
    const int d = kb * 64 + dd;
    float ab[2] = {0.f, 0.f};
    bool up[2] = {false, false};
    if (r < n_rows) {
      const float scale = mode == 1 ? rx[r] : 1.f;
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int de = d + e;
        if (de < dim) ab[e] = X[size_t(r) * pitch + de] * scale;
        else if (mode == 0 && de >= aug_col && de < aug_col + 3) {
          // -|x|^2/2, shrunk by the accumulation-rounding allowance (h_scale = 1 - c_add: the score errs upwards),
          // as three bf16 terms that reproduce the fp32 value exactly
          const float h = hx[r] * h_scale;
          const float hi = __bfloat162float(__float2bfloat16_rn(h));
          const float mid = __bfloat162float(__float2bfloat16_rn(h - hi));
          ab[e] = de == aug_col ? hi : (de == aug_col + 1 ? mid : (h - hi) - mid);
        } else if (mode == 0 && de == aug_col + 3) {
          // the row's error weight |x|, rounded up (hx = -|x|^2/2 is an fp32 rounding of the fp64 sum)
          const float nx = sqrtf(-2.f * hx[r]) * (1.f + 1.f / 4096.f);
          reinterpret_cast<__nv_bfloat16*>(Xb)[2 * i + e] = __float2bfloat16_ru(nx);
          up[e] = true;
        }
      }
    }
    if (!up[0] && !up[1]) reinterpret_cast<__nv_bfloat162*>(Xb)[i] = __floats2bfloat162_rn(ab[0], ab[1]);
    else {
      if (!up[0]) Xb[2 * i] = __float2bfloat16_rn(ab[0]);
      if (!up[1]) Xb[2 * i + 1] = __float2bfloat16_rn(ab[1]);
    }
  }
}

// fp32 rows -> int8 normalised shadow (format above i8_scale) in the bf16 shadows' streaming layout with 128 columns per
// k-block: element (r, d) at ((tile * n_kb + kb) * 256 + r % 256) * 128 + d % 128. One CTA (8 warps, 32 rows each) per
// tile: pass 1 finds the tile's largest |x^_i| (fp64 row norms, the rerank's definition of x^), pass 2 quantises and takes
// the largest residual norm. Pad rows and columns are zero. tile[t] = (S_t, E_t).
__global__ void __launch_bounds__(256)
to_i8_tiled_kernel(const float* __restrict__ X, int64_t n_rows, int pitch, int dim, int n_kb, int64_t n_tiles,
                   int8_t* __restrict__ X8, float2* __restrict__ tile) {
  __shared__ double s_inv[TC_BN];
  __shared__ double s_max[8], s_err[8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int64_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
    double wmax = 0.0;
    for (int rr = warp * 32; rr < warp * 32 + 32; ++rr) {
      const int64_t r = t * TC_BN + rr;
      double s = 0.0; float mx = 0.f;
      if (r < n_rows) {
        const float4* xp = reinterpret_cast<const float4*>(X + size_t(r) * pitch);
        for (int j = lane; j < (pitch >> 2); j += 32) {
          const float4 v = __ldg(xp + j);
          s = fma(double(v.x), double(v.x), s); s = fma(double(v.y), double(v.y), s);
          s = fma(double(v.z), double(v.z), s); s = fma(double(v.w), double(v.w), s);
          mx = fmaxf(fmaxf(mx, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o)); }
      const double n = sqrt(s), inv = 1.0 / (n > 1e-12 ? n : 1e-12);
      if (lane == 0) s_inv[rr] = inv;
      wmax = fmax(wmax, double(mx) * inv);
    }
    if (lane == 0) s_max[warp] = wmax;
    __syncthreads();
    double tmax = 0.0;
    for (int w = 0; w < 8; ++w) tmax = fmax(tmax, s_max[w]);
    const float scale = i8_scale(tmax);
    double werr = 0.0;
    for (int rr = warp * 32; rr < warp * 32 + 32; ++rr) {
      const int64_t r = t * TC_BN + rr;
      const bool live = r < n_rows;
      const double inv = s_inv[rr], inv_s = 1.0 / double(scale);
      double e2 = 0.0;
      for (int kb = 0; kb < n_kb; ++kb) {
        const int d0 = kb * I8_KB + 4 * lane;   // four columns per lane: one 128-byte line per warp and k-block
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (live && d0 < pitch) v = __ldg(reinterpret_cast<const float4*>(X + size_t(r) * pitch + d0));
        const float f[4] = {v.x, v.y, v.z, v.w};
        char4 o;
        int qv[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const double h = double(f[e]) * inv;
          qv[e] = (d0 + e < dim) ? i8_quant(h, scale) : 0;
          const double res = h - double(qv[e]) * inv_s;
          e2 = fma(res, res, e2);
        }
        o.x = char(qv[0]); o.y = char(qv[1]); o.z = char(qv[2]); o.w = char(qv[3]);
        reinterpret_cast<char4*>(X8 + ((size_t(t) * n_kb + kb) * TC_BN + rr) * I8_KB)[lane] = o;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) e2 += __shfl_xor_sync(0xffffffffu, e2, o);
      werr = fmax(werr, e2);
    }
    if (lane == 0) s_err[warp] = werr;
    __syncthreads();
    if (threadIdx.x == 0) {
      double e2 = 0.0;
      for (int w = 0; w < 8; ++w) e2 = fmax(e2, s_err[w]);
      tile[t] = make_float2(scale, __double2float_ru(sqrt(e2) * (1.0 + 0x1p-40)));
    }
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------
// host glue
// ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline bool tc_encode_2d(const TcState* st, CUtensorMap* map, const void* base, uint64_t inner, uint64_t outer,
                         uint64_t pitch_elems, uint32_t box_inner, uint32_t box_outer, std::string* err, int esize = 4) {
  // esize: bytes per element - 4 fp32, 2 bf16, 1 int8 (moved as raw bytes)
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {pitch_elems * uint64_t(esize)};
  const CUtensorMapDataType dt = esize == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                 : (esize == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_UINT8);
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = reinterpret_cast<EncodeTiledFn>(st->encode)(
      map, dt, 2, const_cast<void*>(base), dims, strides, box, estr,
      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    *err = "cuTensorMapEncodeTiled failed with CUresult " + std::to_string(int(r));
    return false;
  }
  return true;
}

inline bool tc_init(TcState* st, int sm_count, std::string* err) {
  st->sm_count = sm_count;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
    *err = std::string("cuTensorMapEncodeTiled entry point unavailable: ") + cudaGetErrorString(e);
    return false;
  }
  st->encode = fn;
  tc_knobs_from_env(&st->knobs);
  cudaError_t a = cudaSuccess;
  auto attr = [&](auto kernel, uint32_t bytes) {
    if (a == cudaSuccess) a = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(bytes));
  };
  attr(knn_tc_filter_kernel<0, 0, 0, 0>, TC_SMEM_BYTES); attr(knn_tc_filter_kernel<1, 0, 0, 0>, TC_SMEM_BYTES);
  attr(knn_tc_filter_kernel<2, 0, 0, 0>, TC_SMEM_BYTES); attr(knn_tc_filter_kernel<0, 1, 0, 0>, TC_SMEM_BYTES);
  attr(knn_tc_filter_kernel<1, 1, 0, 0>, TC_SMEM_BYTES); attr(knn_tc_filter_kernel<2, 1, 0, 0>, TC_SMEM_BYTES);
  attr(knn_tc_filter_kernel<0, 1, 2, 0>, TC_SMEM_BYTES); attr(knn_tc_filter_kernel<1, 1, 2, 0>, TC_SMEM_BYTES);
  attr(knn_tc_filter_kernel<2, 1, 2, 0>, TC_SMEM_BYTES);
  attr(knn_tc_filter_kernel<0, 1, 0, 1>, TC2_SMEM_BYTES); attr(knn_tc_filter_kernel<1, 1, 0, 1>, TC2_SMEM_BYTES);
  attr(knn_tc_filter_kernel<2, 1, 0, 1>, TC2_SMEM_BYTES);
  attr(knn_tc_filter_kernel<0, 1, 2, 1>, TC2_SMEM_BYTES); attr(knn_tc_filter_kernel<1, 1, 2, 1>, TC2_SMEM_BYTES);
  attr(knn_tc_filter_kernel<2, 1, 2, 1>, TC2_SMEM_BYTES);
  attr(knn_tc_filter_kernel<0, 2, 0, 0>, TC_SMEM_BYTES); attr(knn_tc_filter_kernel<2, 2, 0, 0>, TC_SMEM_BYTES);
  attr(knn_tc_filter_kernel<2, 2, 2, 0>, TC_SMEM_BYTES);
  attr(knn_tc_filter_kernel<0, 2, 0, 1>, TC2_SMEM_BYTES); attr(knn_tc_filter_kernel<2, 2, 0, 1>, TC2_SMEM_BYTES);
  attr(knn_tc_filter_kernel<2, 2, 2, 1>, TC2_SMEM_BYTES);
  attr(knn_tc_filter_kernel<0, 2, 0, 2>, TC3_SMEM_MAX); attr(knn_tc_filter_kernel<2, 2, 0, 2>, TC3_SMEM_MAX);
  attr(knn_tc_filter_kernel<2, 2, 2, 2>, TC3_SMEM_MAX);
  if (a == cudaSuccess) a = cudaFuncSetAttribute(knn_rq_filter_kernel<0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, RQ_SMEM_MAX);
  if (a == cudaSuccess) a = cudaFuncSetAttribute(knn_rq_filter_kernel<0, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, RQ_SMEM_MAX);
  if (a == cudaSuccess) a = cudaFuncSetAttribute(knn_rq_filter_kernel<2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, RQ_SMEM_MAX);
  if (a == cudaSuccess) a = cudaFuncSetAttribute(knn_rq_filter_kernel<2, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, RQ_SMEM_MAX);
  if (a == cudaSuccess) a = cudaFuncSetAttribute(knn_tc_finish_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
  if (a != cudaSuccess) { *err = std::string("cudaFuncSetAttribute(tc kernels) failed: ") + cudaGetErrorString(a); return false; }
  return true;
}

// tiled shadow: a flat list of 128-byte lines, 256 lines per (tile, k-block); esize: 2 bf16, 1 int8
inline bool tc_bind_shadow(const TcState* st, CUtensorMap* map, CUtensorMap* map_half, const void* Xb, int64_t n_rows,
                           int blocks_per_tile, std::string* err, int esize = 2) {
  const uint64_t lines = uint64_t((n_rows + TC_BN - 1) / TC_BN) * uint64_t(blocks_per_tile) * TC_BN;
  if (lines >= (uint64_t(1) << 31)) { *err = "shard too large for a tiled shadow (32-bit TMA coordinates)"; return false; }
  const uint32_t line = 128 / esize;   // elements per 128-byte line
  if (!tc_encode_2d(st, map_half, Xb, line, lines, line, line, TC_BN / 2, err, esize)) return false;
  return tc_encode_2d(st, map, Xb, line, lines, line, line, TC_BN, err, esize);
}

inline bool tc_bind_corpus(TcState* st, TcCorpus* tc, const float* X, int64_t n_rows, int dim, int pitch,
                           const void* Xb, int blocks_per_tile, std::string* err) {
  (void)dim;
  tc->ok = false; tc->ok_b = false;
  if (n_rows < 1) return true;
  if (!tc_encode_2d(st, &tc->map_x, X, uint64_t(pitch), uint64_t(n_rows), uint64_t(pitch), TC_BK, TC_BN, err)) return false;
  tc->ok = true;
  if (Xb != nullptr) {
    if (!tc_bind_shadow(st, &tc->map_xb, &tc->map_xb_h, Xb, n_rows, blocks_per_tile, err)) return false;
    tc->ok_b = true;
  }
  return true;
}

// K' (candidates kept by each selection) and the buffer capacity that goes with it
constexpr int TC_KP_I8 = 256;   // int8 filter, k <= 16: rows above the k-th exact cosine that the bound lets through (K' sweep)
inline int tc_kp(int k, bool certify, int kind = 0) {
  // slack so that the certificate holds for (nearly) every query in one pass: the bf16 bound is ~3.5x looser than
  // the TF32 one (2^-7 against 1.25 2^-9 per product; K' was measured on C3 when the bf16 constant was half its present,
  // correct value: K' = 32 flagged 25 of 4096 queries per batch with bf16, K' = 64 none); the int8 bound
  // (~0.02 in cosine units at D = 768) needs a few hundred rows, see TC_KP_I8
  if (kind == 2) return certify ? std::max(TC_KP_I8, (k + k / 2 + 31) & ~31) : ((k + 31) & ~31);
  int kp = certify ? k + std::max(kind == 1 ? 48 : 16, k / 2) : k;
  return (kp + 31) & ~31;
}
inline int tc_cap(int kp) { return kp <= 128 ? 512 : 1024; }

inline bool tc_supported(const TcState* st, const TcCorpus* tc, int64_t n_rows, int dim, int k, int n_q) {
  (void)n_q;
  if (!st->encode || !tc->ok) return false;
  if (dim > 8192) return false;                   // finish kernel stages the query in shared memory
  if (k > 320) return false;                      // K' <= 512 so that a 1024-entry buffer keeps room to append
  if (n_rows < 4096 || n_rows < 8 * int64_t(k)) return false;  // tiny shards: the scan is already instant
  if (n_rows > int64_t(0x7fffff00)) return false; // 32-bit tile arithmetic
  return true;
}

struct TcPlan {
  int n_qt, n_tiles, n_slices, tiles_per_slice, grid, units, kp, cap, n_kblocks, n_kb_data, nk_last, aug_line0, aug_col;
  int n_vtiles, tile_stride;
  int rq;        // 1: resident-query kernel (units = query pairs x slices of 128-row tiles, one list per unit and query)
  int pair;      // 1: CTA-pair streaming kernel (units = query pairs x slices; candidate lists per CTA as in the one-CTA kernel)
  int resident;  // 1: the CTA-pair kernel with resident query tiles (int8 shadow; same units and candidate lists as pair)
  int n_qt_lists;// query tiles the candidate-list layout is indexed with (2 n_qp for the pair kernel, else n_qt)
  int n_qp;      // query pairs
  int kp_list;   // candidates each (query, list) keeps at a selection (<= kp)
  int kb_bf16;   // the row width in bf16 k-blocks (64 columns; the plain shadow's augmented block counted), whatever the
                 // operand kind: what the CTA-pair and sample-prepass rules were measured against
  size_t off_qp, off_qb, off_tau, off_flags, off_qerr, off_wcnt, off_wbuf, off_pre, total;
  int n_rec, pre_pitch;   // threshold prepass: block-maximum records per query (= row pitch of the record matrix)
};

inline TcPlan tc_plan(const TcState* st, const TcSearch& s) {
  TcPlan pl{};
  pl.n_qt = (s.n_q + TC_BM - 1) / TC_BM;
  pl.n_tiles = int((s.n_rows + TC_BN - 1) / TC_BN);
  pl.kp = s.tau_fixed ? 1024 : tc_kp(s.k, s.certify, s.kind);   // refinement reranks every survivor (up to 1024)
  const bool pre = s.sample_stride > 1;                          // threshold prepass over a strided sample
  if (pre) pl.kp = 32;   // unused by the prepass kernels (no candidate lists); keeps the slice heuristics below sane
  const TcKnobs& kn = st->knobs;
  if (!s.tau_fixed && s.certify && !pre && kn.kp >= s.k && kn.kp <= 512) pl.kp = (kn.kp + 31) & ~31;
  pl.cap = tc_cap(pl.kp);
  // MMA instructions per tile: 32 B of K each (8 fp32 / 16 bf16 elements); only columns that hold data
  pl.aug_line0 = 0; pl.aug_col = 0;
  if (s.kind == 0) {
    pl.n_kb_data = (s.pitch + TC_BK - 1) / TC_BK;
    pl.nk_last = (s.pitch - TC_BK * (pl.n_kb_data - 1) + TC_UMMA_K - 1) / TC_UMMA_K;
    pl.n_kblocks = pl.n_kb_data;
  } else if (s.kind == 2) {
    pl.n_kb_data = i8_n_kb(s.dim);
    pl.nk_last = (s.dim - I8_KB * (pl.n_kb_data - 1) + 31) / 32;
    pl.n_kblocks = pl.n_kb_data;
  } else {
    const ShadowGeom g = shadow_geom(s.dim);
    pl.n_kb_data = g.n_kb_data;
    const int used = s.dim - 64 * (g.n_kb_data - 1) + ((s.aug && !g.aug_separate) ? TC_AUG_COLS : 0);
    pl.nk_last = (used + 15) / 16;
    pl.n_kblocks = g.n_kb_data + ((s.aug && g.aug_separate) ? 1 : 0);
    pl.aug_line0 = pl.n_tiles * g.n_kb_data * TC_BN;
    pl.aug_col = g.aug_col;
  }
  pl.kb_bf16 = s.kind == 2 ? (s.dim + 63) / 64 : pl.n_kblocks;
  // narrow rows and at least two query tiles: the resident-query kernel (operand traffic, not the tensor pipe, binds
  // the streaming kernel there); its tiles are 128 corpus rows, its units pair two query tiles
  pl.rq = (s.kind == 1 && pl.n_kblocks <= RQ_MAX_KB && pl.n_qt >= 2 && s.epi != 1 && s.dbg == nullptr && !kn.no_rq) ? 1 : 0;
  pl.n_qp = (pl.n_qt + 1) / 2;
  // wider rows and at least two query tiles: CTA pairs (cta_group::2) over the bf16 shadow - each SM stages half of
  // every corpus block, two thirds of the one-CTA kernel's L2 -> SM operand traffic at the same tensor work
  // (auto: from 7 k-blocks per row on. A tile of D = 384 is 24 MMAs and the pair's cluster-wide hand-offs cost more than
  // the halved B traffic saves - 1452 vs 1541 TFLOP/s at uncapped clocks; from D = 512 the pair wins, 1645 vs 1519 TFLOP/s at
  // D = 768: scripts/ubench/width_sweep.py, profiles/r02_sweep_row_width.txt)
  const bool pair_ok = !pl.rq && s.kind >= 1 && pl.n_qt >= 2 && s.dbg == nullptr;
  pl.pair = (pair_ok && (kn.pair == 1 || (kn.pair < 0 && pl.kb_bf16 >= 7))) ? 1 : 0;
  // int8 shadow: the query tile (16 KB per k-block) stays in shared memory for the whole unit when it leaves room for
  // TC3_MIN_STAGES corpus stages (D <= 1152). Auto: where the CTA-pair kernel runs over a shard of >= 4M rows. Measured
  // (4096 queries, D = 512 / 768 / 1024, profiles/r04_int8_widths.txt): 10M rows 7.7 / 6.6 / -0.3 % less filter time than
  // the streaming pair, 5M rows 1.4 / 7.9 / 4.4 % (4.4 % at D = 768 with the sample prepass off), but 2.5M and 1M rows
  // 2 - 25 % MORE, with or without the prepass
  constexpr int64_t TC3_MIN_ROWS = int64_t(1) << 22;
  const bool res_fits = s.kind == 2 && tc3_stages(pl.n_kblocks) >= TC3_MIN_STAGES;
  pl.resident = (pair_ok && res_fits && (kn.resident == 1 || (kn.resident < 0 && pl.pair && s.n_rows >= TC3_MIN_ROWS))) ? 1 : 0;
  if (pl.resident) pl.pair = 1;
  pl.n_qt_lists = pl.pair ? 2 * pl.n_qp : pl.n_qt;
  const int n_tiles_full = pl.rq ? int((s.n_rows + RQ_BN - 1) / RQ_BN) : pl.n_tiles;   // tiles in the kernel's own unit
  pl.tile_stride = pre ? s.sample_stride : 1;
  const int n_tiles_u = (n_tiles_full + pl.tile_stride - 1) / pl.tile_stride;          // tiles the units iterate over
  pl.n_vtiles = n_tiles_u;
  const int n_qu = (pl.rq || pl.pair) ? pl.n_qp : pl.n_qt;                          // query blocks per slice
  // Slices: units = n_qt * n_slices, slice major (all query tiles of a slice adjacent; query-tile-major order, which
  // runs all slices of a query tile at the same time, was measured slower on C3 - 112 vs 94 ms, profiles/r01_c3_sweep.txt -
  // and removed), are dealt round-robin to min(units, #SM) persistent CTAs.
  // Maximise SM utilisation units / (G * ceil(units / G)); few slices are preferred (longer units give
  // tighter thresholds and fewer candidate lists), and every unit should span enough tiles for its
  // threshold to become selective.
  const int sms = pl.pair ? st->sm_count / 2 : st->sm_count;   // persistent workers: CTAs, or CTA pairs
  const int min_tiles = pre ? 4 : std::max(4, (8 * pl.kp + TC_BN - 1) / TC_BN) * (pl.rq ? 2 : 1);
  const int s_cap = std::max(1, (TC_MAX_WAVES * sms) / n_qu);
  const int s_max = std::max(1, std::min(n_tiles_u / min_tiles, s_cap));
  double best = -1.0; int best_s = 1;
  for (int sl = 1; sl <= s_max; ++sl) {
    int tps = (n_tiles_u + sl - 1) / sl;
    int eff_s = (n_tiles_u + tps - 1) / tps;
    if (eff_s != sl) continue;
    long units = long(sl) * n_qu;
    long g = std::min<long>(units, sms);
    double eff = double(units) / double(sms * ((units + g - 1) / g));
    if (eff > best + 0.02) { best = eff; best_s = sl; }
  }
  if (kn.slices > 0) {   // tuning knob: force the slice count
    int forced = kn.slices;
    if (forced >= 1 && forced <= s_max) {
      int tps = (n_tiles_u + forced - 1) / forced;
      best_s = (n_tiles_u + tps - 1) / tps;
    }
  }
  pl.n_slices = best_s;
  pl.tiles_per_slice = (n_tiles_u + best_s - 1) / best_s;
  pl.units = pl.n_slices * n_qu;
  // Each query's candidates are spread over L = TC_SPLIT * n_slices lists. A list does not need to keep K'
  // entries: the global top-k lands ~k/L per list, so keeping 2k/L + 16 (>= 32) per list gives much tighter
  // local thresholds (fewer appends and selections). If a query's neighbours are concentrated in few lists
  // the certificate fails and the refinement pass settles it.
  {
    const int lists = (pl.rq ? 1 : TC_SPLIT) * pl.n_slices;
    int m = std::max(32, (2 * s.k + lists - 1) / lists + 16);
    m = (m + 31) & ~31;
    pl.kp_list = (s.tau_fixed || pre || s.full_lists) ? pl.kp : std::min(pl.kp, m);   // prepass: every list keeps the m best it sees
    // A pass seeded by the sample prepass selects only when a list overflows, so a quota below k buys nothing there -
    // and it is what starves queries whose neighbours sit in ONE list (a list that publishes its m-th best score as the
    // query's global threshold vouches for m candidates only): with quotas of k rounded up the reference tests' clustered
    // rows at C2 scale lose their 800 starved queries per batch (4.5 -> 3.3 ms per step; Gaussian rows unchanged).
    if (s.seeded && !pre && !s.full_lists && !s.tau_fixed) pl.kp_list = std::min(pl.kp, std::max(pl.kp_list, (s.k + 31) & ~31));
    pl.cap = (s.tau_fixed || pre) ? pl.cap : tc_cap(pl.kp_list);
  }
  pl.grid = int(std::min<long>(pl.units, sms)) * (pl.pair ? 2 : 1);
  const size_t list_units = size_t(pl.n_slices) * size_t(pl.pair ? 2 * pl.n_qp : n_qu);   // blocks of TC_SLOTS candidate lists
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = (off + bytes + 255) & ~size_t(255); return o; };
  take(TC_HDR_BYTES);   // header: word 0 counts the queries the finish kernel flagged (read back with the results)
  const size_t q_rows_p = size_t(pl.n_qp) * 2 * TC_BM;   // queries are stored in whole tile pairs
  pl.off_qp = take(q_rows_p * s.pitch * 4);
  pl.off_qb = take(s.kind == 1 ? q_rows_p * s.pitch_b * 2 : (s.kind == 2 ? q_rows_p * s.pitch_b : 0));
  pl.off_tau = take(size_t(s.n_q) * 4);
  pl.off_flags = take(size_t(s.n_q) * 4);
  pl.off_qerr = take(size_t(s.n_q) * 16);   // per query: the error weight (augmented queries), or (S_q, a_q, e_q) (kind 2)
  pl.n_rec = pl.n_vtiles * (pl.rq ? 1 : TC_SPLIT);
  pl.pre_pitch = pl.n_rec;
  if (pre) {
    pl.off_wcnt = pl.off_wbuf = off;
    pl.off_pre = take(size_t(s.n_q) * pl.pre_pitch * 4);
  } else {
    pl.off_wcnt = take(list_units * TC_SLOTS * 4);
    pl.off_wbuf = take(list_units * TC_SLOTS * pl.cap * 8);
    pl.off_pre = off;
  }
  pl.total = off;
  return pl;
}

inline bool tc_prepass_config(const TcState* st, const TcSearch& s, const TcPlan& main_pl, TcSearch* pre);
// Everything one search needs to know before it launches, computed ONCE per search: the plan of the main pass, whether
// a sample prepass runs first (and its plan), and the scratch both need.
struct TcLaunch {
  TcPlan pl;
  bool with_pre = false;
  TcSearch pre;
  TcPlan ppl;
  size_t scratch_bytes = 0;
};
inline TcLaunch tc_prepare(const TcState* st, const TcSearch& s) {
  TcLaunch L;
  L.pl = tc_plan(st, s);
  L.scratch_bytes = L.pl.total;
  L.with_pre = tc_prepass_config(st, s, L.pl, &L.pre);
  if (L.with_pre) {
    TcSearch seeded = s;
    seeded.seeded = 1;
    L.pl = tc_plan(st, seeded);          // (same kernel, units and slices; the list quotas - hence the scratch layout - differ)
    L.scratch_bytes = L.pl.total;
    L.ppl = tc_plan(st, L.pre);
    L.scratch_bytes = std::max(L.scratch_bytes, L.ppl.total);
  }
  return L;
}
inline const int* tc_flags(const TcLaunch& L, void* scratch) {
  return reinterpret_cast<const int*>(static_cast<char*>(scratch) + L.pl.off_flags);
}
inline const int* tc_flag_count(void* scratch) { return static_cast<const int*>(scratch); }   // header word 0
// rigorous bound constant of the TF32 dot product: |acc - <q,x>| <= c * |q| * |x|
// (operands truncated to 10 mantissa bits: 2^-10 each -> 2^-9 on the product, 25% margin;
//  fp32 accumulation of D terms: D * 2^-21)
// bf16 operands are rounded to nearest: 8 significant bits, so up to 2^-8 relative each -> 2^-7 on the product, 10%
// margin (tests/test_gpu_exactness_edges.py plants rows that reach 0.9 of it).
// L2 only: rounding of the -|x|^2/2 term and of its addition, relative to |x|^2/2 + |q||x|. When the term rides
// through the MMA (augmented shadow) every one of the tile's accumulation steps may round it again.
inline double tc_c_add(int dim, bool aug) { return 4.8e-7 + (aug ? double((dim + TC_AUG_COLS + 15) / 16) * 1.2e-7 : 0.0); }
inline double tc_c_err(int dim, int kind = 0) {
  const double prod = kind == 0 ? 1.25 * std::ldexp(1.0, -9) : 1.10 * std::ldexp(1.0, -7);
  return prod + double(dim) * std::ldexp(1.0, -21);
}

// Error constants the certificate and the refinement thresholds use. With augmented queries (TcSearch::aug) the filter
// score already carries c |q| |x| per row plus the folded |x|^2/2 allowance - it IS an upper bound of the exact score -
// so nothing is added on top and the certificate no longer depends on the largest norm of the shard: one 100x-norm
// outlier (or clustered rows far from the origin) inflates only its own row's score.
// Absolute term of the TF32 / bf16 bounds: every product and every partial sum of the MMA (data and augmented columns)
// that falls below FLT_MIN loses less than 2^-126, whether the tensor cores keep subnormals or flush them, and the
// relative terms above do not cover that loss on rows of tiny magnitude (tests/test_gpu_exactness_edges.py).
inline double tc_c_abs(int dim) { return 2.0 * double(dim + TC_AUG_COLS + 4) * std::ldexp(1.0, -126); }
// The int8 filter's scores are exact integer sums, converted once and rounded up: no absolute term.
inline void tc_cert_consts(const TcSearch& s, double* c_err, double* c_add, double* c_abs) {
  *c_abs = s.kind == 2 ? 0.0 : tc_c_abs(s.dim);
  if ((s.kind == 1 && s.aug != 0) || s.kind == 2) { *c_err = 0.0; *c_add = 0.0; return; }
  *c_err = tc_c_err(s.dim, s.kind);
  *c_add = tc_c_add(s.dim, false);
}
// c of the query's error weight u = c |q| (augmented queries): product rounding + fp32 accumulation over the data and
// augmented columns, plus (L2) the |q||x| share of the accumulation-rounding allowance
inline double tc_c_pair(int dim, int aug) {
  return tc_c_err(dim + TC_AUG_COLS + 4, 1) + (aug == 1 ? tc_c_add(dim, true) : 0.0);
}

// Threshold prepass (narrow rows, where the epilogue - not the tensor pipe - binds): the same filter kernel runs over
// every stride-th corpus tile, and the m-th best sample score of a query becomes its initial threshold for the main
// pass. With S sampled rows the threshold passes ~ m N / S rows of the shard; stride and m are chosen so that this is
// `safety` x K' with m ~ 10 (relative spread ~ 1/sqrt(m); a threshold that turns out too tight only costs the query
// a refinement pass, one that is too loose more appends - exactness never depends on the sample).
inline bool tc_prepass_config(const TcState* st, const TcSearch& s, const TcPlan& main_pl, TcSearch* pre) {
  const TcKnobs& kn = st->knobs;
  if (s.tau_fixed || s.no_prepass || s.sample_stride > 1 || s.kind == 0 || s.dbg != nullptr) return false;
  // Wide rows: small batches are HBM-bound with a lightly loaded tensor pipe, and there the epilogue's hit path and the
  // finish kernel's candidate volume show (C5 batch 64 +18 %, batch 8 +6 %). Large batches are tensor-bound and the
  // sample costs 1/stride of the scan (3 %); on a whole 10M x 768 shard it pays that back and no more (round 1: neutral),
  // but units get SHORT when the corpus is sharded (1.25M rows per GPU: 132 tiles per unit) and per-list thresholds - each
  // list keeps its own 32 best, ~2400 admitted rows per query over 74 lists - stay loose for most of a unit: measured on
  // one 8-GPU shard of C3 the filter kernel takes 6.35 ms without and 5.09 ms with the sample's GLOBAL thresholds
  // (0.76 -> 0.95 of the burst bf16 peak, profiles/r02_sweep_prepass.txt).
  const bool wide = main_pl.kb_bf16 > 4;
  if (s.epi != 2) return false;                            // a row mask (predicate / IVF cells) of unknown selectivity: the
                                                           // sample says nothing about how many LIVE rows pass a threshold
  if (kn.pre == 0) return false;
  // the threshold passes ~ safety x K' rows of the shard. Tensor-bound searches (wide rows, large batches) have epilogue
  // time to spare for a few more hits, so they take a thinner sample: safety 8 -> every ~85th tile, 1.2 % of the scan
  // instead of 3 % (profiles/r02_sweep_prepass.txt)
  double safety = (wide && main_pl.n_qt > 3) ? 8.0 : 3.0;
  if (kn.pre_safety >= 1.0 && kn.pre_safety <= 64.0) safety = kn.pre_safety;
  const int tile_rows = main_pl.rq ? RQ_BN : TC_BN;
  // rank m of the sample statistic: P(threshold too tight for k rows) = P(Gamma(m) < m k / (safety K')). Wide rows pay
  // for every sampled tile, so they take the thinner sample when k is small against K' (k = 10: m = 6, P ~ 1e-6)
  double target_m = (wide && double(s.k) <= 0.06 * safety * double(main_pl.kp)) ? 6.0 : 16.0;
  if (kn.pre_m >= 2.0 && kn.pre_m <= 256.0) target_m = kn.pre_m;
  int stride = int(double(main_pl.kp) * safety / target_m);         // S = N / stride, m = safety K' S / N
  const int64_t n_tiles_full = (s.n_rows + tile_rows - 1) / tile_rows;
  if (stride < 4 || n_tiles_full / stride < 32) return false;       // shard too small for a sample to pay off
  const int rec_per_tile = main_pl.rq ? 1 : TC_SPLIT;
  // at most 4096 records per query (they are held in registers by the tau0 kernel) and 256 MB of records in all
  const int64_t max_rec = std::min<int64_t>(4096, std::max<int64_t>(64, (int64_t(1) << 26) / std::max(s.n_q, 1)));
  stride = int(std::max<int64_t>(stride, (n_tiles_full * rec_per_tile + max_rec - 1) / max_rec));
  const int64_t sample_rows = ((n_tiles_full + stride - 1) / stride) * tile_rows;
  *pre = s;
  pre->sample_stride = stride;
  const double m_exact = safety * double(main_pl.kp) * double(sample_rows) / double(s.n_rows);
  if (m_exact < 4.0) return false;   // the sample the memory cap allows is too thin for a trustworthy rank statistic
  pre->pre_m = int(m_exact + 0.5);
  pre->certify = false;
  pre->ev_k0 = nullptr; pre->ev_k1 = nullptr;
  return true;
}

// Where a pass over the plan `pl` left its padded queries, thresholds, flags and candidate lists in `scratch`, and what
// the finish kernel does with them.
inline FinishParams tc_finish_params(const TcSearch& s, const TcPlan& pl, void* scratch) {
  char* base = static_cast<char*>(scratch);
  FinishParams f{};
  f.X = s.X; f.pitch = s.pitch; f.dim = s.dim; f.row_base = s.row_base; f.Qp = reinterpret_cast<float*>(base + pl.off_qp);
  f.n_q = s.n_q; f.n_qt = pl.n_qt_lists;
  f.n_flagged = reinterpret_cast<int*>(base);
  f.n_slices = pl.n_slices; f.cap = pl.cap; f.metric = s.metric; f.k = s.k; f.kp = pl.kp;
  int sort2 = 2; while (sort2 < pl.kp) sort2 <<= 1;
  f.sort2 = sort2; f.tau_g = reinterpret_cast<uint32_t*>(base + pl.off_tau); f.wbuf = reinterpret_cast<uint2*>(base + pl.off_wbuf);
  f.wcnt = reinterpret_cast<int*>(base + pl.off_wcnt); f.rq = pl.rq; f.n_qp = pl.n_qp;
  f.flags = reinterpret_cast<int*>(base + pl.off_flags); f.certify = s.certify ? 1 : 0;
  f.max_norm = s.max_norm; tc_cert_consts(s, &f.c_err, &f.c_add, &f.c_abs); f.out_rows = s.out_rows; f.out_dist = s.out_dist;
  f.unit_q = s.kind == 2 ? 1 : 0;
  return f;
}

// One filter launch (+ finish) over the plan of `s`; queries / state have been prepared in `scratch` already.
inline bool tc_run_pass(TcCorpus* tc, const TcSearch& s, const TcPlan& pl, void* scratch, const CUtensorMap& map_q,
                        std::string* err) {
  char* base = static_cast<char*>(scratch);
  uint32_t* tau_g = reinterpret_cast<uint32_t*>(base + pl.off_tau);
  int* flags = reinterpret_cast<int*>(base + pl.off_flags);
  int* wcnt = reinterpret_cast<int*>(base + pl.off_wcnt);
  uint2* wbuf = reinterpret_cast<uint2*>(base + pl.off_wbuf);
  const bool pre = s.sample_stride > 1;   // threshold prepass: block maxima of a strided sample, then tau0

  TcParams p{};
  p.pre_max = reinterpret_cast<float*>(base + pl.off_pre); p.pre_pitch = pl.pre_pitch;
  p.n_q = s.n_q; p.n_qt = pl.n_qt; p.n_rows = s.n_rows; p.n_tiles = pl.n_tiles; p.n_slices = pl.n_slices;
  p.tiles_per_slice = pl.tiles_per_slice; p.n_vtiles = pl.n_vtiles; p.tile_stride = pl.tile_stride;
  p.n_kblocks = pl.n_kblocks; p.n_kb_data = pl.n_kb_data; p.nk_last = pl.nk_last;
  p.aug_line0 = pl.aug_line0;
  p.i8_tile = s.i8_tile; p.i8_q = reinterpret_cast<const float4*>(base + pl.off_qerr);
  p.kp = pl.kp_list; p.cap = pl.cap;
  p.sleep_ns = pl.n_kblocks >= 6 ? 0u : 64u;
  p.hx = s.hx; p.rx = s.rx; p.dbg = s.dbg; p.wbuf = wbuf; p.wcnt = wcnt; p.tau_g = tau_g;
  p.fixed = s.tau_fixed ? 1 : 0; p.flags = flags;
  if (s.ev_k0) cudaEventRecordWithFlags(s.ev_k0, s.stream, s.ev_flags);
  const int epi = s.epi;   // epilogue form: 0 add, 1 multiply, 2 none
  // dispatch on (epilogue form, operand kind, mode: filter / diagnostics dump / prepass, CTA pairs)
  cudaError_t le = cudaSuccess;
  auto launch = [&](auto kernel, const CUtensorMap& map_b, uint32_t smem, int cluster) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(unsigned(pl.grid)); cfg.blockDim = dim3(TC_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = s.stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = unsigned(cluster); at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = cluster > 1 ? 1 : 0;
    le = cudaLaunchKernelEx(&cfg, kernel, map_q, map_b, p);
  };
  const bool dbg = s.dbg != nullptr;
  if (pl.rq) {
    const CUtensorMap& map_h = s.shadow == 1 ? tc->map_xn_h : tc->map_xb_h;
    p.rq_stages = rq_stages(pl.n_kblocks);
    const uint32_t rq_smem = rq_smem_bytes(pl.n_kblocks);
    if (pre) {
      if (epi == 0) launch(knn_rq_filter_kernel<0, 2>, map_h, rq_smem, 1);
      else launch(knn_rq_filter_kernel<2, 2>, map_h, rq_smem, 1);
    } else {
      if (epi == 0) launch(knn_rq_filter_kernel<0, 0>, map_h, rq_smem, 1);
      else launch(knn_rq_filter_kernel<2, 0>, map_h, rq_smem, 1);
    }
  } else if (pl.resident) {
    p.rq_stages = tc3_stages(pl.n_kblocks);
    const uint32_t smem = tc3_smem_bytes(pl.n_kblocks);
    if (epi == 0) launch(knn_tc_filter_kernel<0, 2, 0, 2>, tc->map_x8_h, smem, 2);   // (masked: no prepass)
    else if (pre) launch(knn_tc_filter_kernel<2, 2, 2, 2>, tc->map_x8_h, smem, 2);
    else launch(knn_tc_filter_kernel<2, 2, 0, 2>, tc->map_x8_h, smem, 2);
  } else if (pl.pair && s.kind == 2) {
    if (epi == 0) launch(knn_tc_filter_kernel<0, 2, 0, 1>, tc->map_x8_h, TC2_SMEM_BYTES, 2);   // (masked: no prepass)
    else if (pre) launch(knn_tc_filter_kernel<2, 2, 2, 1>, tc->map_x8_h, TC2_SMEM_BYTES, 2);
    else launch(knn_tc_filter_kernel<2, 2, 0, 1>, tc->map_x8_h, TC2_SMEM_BYTES, 2);
  } else if (s.kind == 2) {
    if (dbg) {
      cudaFuncSetAttribute(knn_tc_filter_kernel<2, 2, 1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_BYTES);
      launch(knn_tc_filter_kernel<2, 2, 1, 0>, tc->map_x8, TC_SMEM_BYTES, 1);
    } else if (epi == 0) launch(knn_tc_filter_kernel<0, 2, 0, 0>, tc->map_x8, TC_SMEM_BYTES, 1);
    else if (pre) launch(knn_tc_filter_kernel<2, 2, 2, 0>, tc->map_x8, TC_SMEM_BYTES, 1);
    else launch(knn_tc_filter_kernel<2, 2, 0, 0>, tc->map_x8, TC_SMEM_BYTES, 1);
  } else if (pl.pair) {
    // CTA pairs: each CTA loads 128-row half blocks of the tiled shadow
    const CUtensorMap& map_h = s.shadow == 1 ? tc->map_xn_h : tc->map_xb_h;
#define FX_TC2_CASE(E)                                                              \
  if (epi == E) {                                                                   \
    if (pre) launch(knn_tc_filter_kernel<E, 1, 2, 1>, map_h, TC2_SMEM_BYTES, 2);    \
    else launch(knn_tc_filter_kernel<E, 1, 0, 1>, map_h, TC2_SMEM_BYTES, 2);        \
  }
    FX_TC2_CASE(0) FX_TC2_CASE(1) FX_TC2_CASE(2)
#undef FX_TC2_CASE
  } else {
#define FX_TC_CASE(E, K, MAP)                                                       \
  if (epi == E && s.kind == K) {                                                    \
    if (dbg) {                                                                      \
      cudaFuncSetAttribute(knn_tc_filter_kernel<E, K, 1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_BYTES); \
      launch(knn_tc_filter_kernel<E, K, 1, 0>, MAP, TC_SMEM_BYTES, 1);              \
    } else if (pre && K == 1) {                                                     \
      launch(knn_tc_filter_kernel<E, 1, 2, 0>, MAP, TC_SMEM_BYTES, 1);              \
    } else {                                                                        \
      launch(knn_tc_filter_kernel<E, K, 0, 0>, MAP, TC_SMEM_BYTES, 1);              \
    }                                                                               \
  }
  FX_TC_CASE(0, 0, tc->map_x) FX_TC_CASE(1, 0, tc->map_x) FX_TC_CASE(2, 0, tc->map_x)
  const CUtensorMap& map_s = s.shadow == 1 ? tc->map_xn : tc->map_xb;
  FX_TC_CASE(0, 1, map_s) FX_TC_CASE(1, 1, map_s) FX_TC_CASE(2, 1, map_s)
#undef FX_TC_CASE
  }
  if (le != cudaSuccess) { *err = std::string("filter kernel launch failed: ") + cudaGetErrorString(le); return false; }
  if (s.ev_k1) cudaEventRecordWithFlags(s.ev_k1, s.stream, s.ev_flags);
  if (pre) {
    if (pl.n_rec <= 32 * TAU0_PER) knn_tc_tau0_kernel<32><<<(s.n_q + 7) / 8, 256, 0, s.stream>>>(p.pre_max, s.n_q, pl.n_rec, s.pre_m, tau_g);
    else if (pl.n_rec <= 64 * TAU0_PER) knn_tc_tau0_kernel<64><<<(s.n_q + 3) / 4, 256, 0, s.stream>>>(p.pre_max, s.n_q, pl.n_rec, s.pre_m, tau_g);
    else if (pl.n_rec <= 128 * TAU0_PER) knn_tc_tau0_kernel<128><<<(s.n_q + 1) / 2, 256, 0, s.stream>>>(p.pre_max, s.n_q, pl.n_rec, s.pre_m, tau_g);
    else knn_tc_tau0_kernel<256><<<s.n_q, 256, 0, s.stream>>>(p.pre_max, s.n_q, pl.n_rec, s.pre_m, tau_g);
    cudaError_t e0 = cudaGetLastError();
    if (e0 != cudaSuccess) { *err = std::string("threshold prepass launch failed: ") + cudaGetErrorString(e0); return false; }
    return true;
  }

  if (s.no_finish) return true;
  const FinishParams f = tc_finish_params(s, pl, scratch);
  const int sort2 = f.sort2;
  const size_t fin_smem = size_t(sort2) * 12 + size_t(s.pitch) * 4 + size_t(FIN_POOL) * 8 + 16;
  // many short lists per query (small batches split over all SMs): more warps sweep them in parallel
  // few lists, many candidates to rerank (K' >= 128: k = 100): 128-thread CTAs - more of them per SM cover the scattered
  // exact-row reads better (C2: 2.87 -> 2.78 ms per step; 512 threads: 3.04)
  const int fin_threads = (pl.rq ? 1 : TC_SPLIT) * pl.n_slices > 32 ? 1024 : (pl.kp >= 128 && pl.kp <= 512 ? 128 : 256);   // (refinement passes rerank up to 1024 survivors: 256)
  knn_tc_finish_kernel<<<s.n_q, fin_threads, fin_smem, s.stream>>>(f);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { *err = std::string("tensor-core path launch failed: ") + cudaGetErrorString(e); return false; }
  return true;
}

inline bool tc_search(TcState* st, TcCorpus* tc, const TcSearch& s, const TcLaunch& L, void* scratch, int* launched,
                      std::string* err, int* variant = nullptr) {
  const TcPlan& pl = L.pl;
  char* base = static_cast<char*>(scratch);
  float* qp = reinterpret_cast<float*>(base + pl.off_qp);
  uint32_t* tau_g = reinterpret_cast<uint32_t*>(base + pl.off_tau);
  int* flags = reinterpret_cast<int*>(base + pl.off_flags);

  __nv_bfloat16* qb = s.kind == 1 ? reinterpret_cast<__nv_bfloat16*>(base + pl.off_qb) : nullptr;
  CUtensorMap map_q;
  if (s.kind == 0) {
    if (!tc_encode_2d(st, &map_q, qp, uint64_t(s.pitch), uint64_t(pl.n_qp) * 2 * TC_BM, uint64_t(s.pitch), TC_BK, TC_BM, err)) return false;
  } else if (s.kind == 2) {
    if (!tc->ok_8) { *err = "int8 filter requested but the shard has no int8 shadow"; return false; }
    if (!tc_encode_2d(st, &map_q, base + pl.off_qb, uint64_t(s.pitch_b), uint64_t(pl.n_qp) * 2 * TC_BM, uint64_t(s.pitch_b), I8_KB, TC_BM, err, 1)) return false;
  } else {
    if (s.shadow == 1 ? !tc->ok_n : !tc->ok_b) { *err = "bf16 filter requested but the shard has no bf16 shadow"; return false; }
    if (!tc_encode_2d(st, &map_q, qb, uint64_t(s.pitch_b), uint64_t(pl.n_qp) * 2 * TC_BM, uint64_t(s.pitch_b), 2 * TC_BK, TC_BM, err, 2)) return false;
  }

  const int n_rows_p = pl.n_qp * 2 * TC_BM;
  const int prep_blocks = int(std::min<int64_t>((int64_t(n_rows_p) * s.pitch + 255) / 256, 4 * 148));
  float* qerr = reinterpret_cast<float*>(base + pl.off_qerr);
  const bool aug = s.kind == 1 && s.aug != 0;
  *launched = 3;
  if (aug) {
    knn_qerr_kernel<<<(s.n_q + 3) / 4, 128, 0, s.stream>>>(s.Q, s.n_q, s.dim, s.c_pair, qerr);
    *launched += 1;
  }
  knn_prep_kernel<<<std::max(prep_blocks, 1), 256, 0, s.stream>>>(s.Q, s.n_q, n_rows_p, s.dim, s.pitch, qp, tau_g, flags, qb, s.pitch_b, s.tau_fixed,
                                                                  aug ? pl.aug_col : 0, reinterpret_cast<int*>(base), s.aug, qerr);
  if (s.kind == 2) {
    knn_qprep_i8_kernel<<<(n_rows_p + 7) / 8, 256, 0, s.stream>>>(s.Q, s.n_q, n_rows_p, s.dim, s.pitch_b,
                                                                 reinterpret_cast<int8_t*>(base + pl.off_qb), reinterpret_cast<float4*>(qerr));
    *launched += 1;
  }
  // threshold prepass over a strided sample (the padded queries and tau_g sit at the same scratch offsets in both plans)
  if (variant) *variant = (pl.rq ? 1 : 0) | (L.with_pre ? 2 : 0) | (pl.pair ? 4 : 0) | (pl.resident ? 8 : 0);
  if (L.with_pre) {
    if (!tc_run_pass(tc, L.pre, L.ppl, scratch, map_q, err)) return false;
    *launched += 2;
  }
  return tc_run_pass(tc, s, pl, scratch, map_q, err);
}

}  // namespace fx
