/* fenix_knn.h — C ABI of libfenix_knn.so: exact k-NN search over device-resident corpus shards.
 *
 * This is the drop-in boundary for the one hot path of nrlugg/fenix that this repository
 * replaces: exact brute-force search = distance(query, every corpus row) + top-k.
 * Reference seam (citations relative to the reference tree):
 *   src/fenix/io/index/index.py:133-168   UDF `dist` + select_k_unstable + take   (replaced)
 *   src/fenix/io/coder/coder.py:38-50     distance(): l2 / cosine / dot            (replaced)
 *   src/fenix/io/torch/torch.py:6-10      from_arrow(): Arrow values buffer view   (replaced by
 *                                         fx_corpus_append: host buffer -> pinned ring -> HBM)
 *
 * Conventions
 *   - every function returns 0 on success, a negative FX_E* code on failure; the message
 *     is available (thread-local) from fx_last_error().
 *   - plain pointers and sizes only; no torch / Arrow types cross this boundary.
 *   - "row" always means the position of a vector in the corpus in append order
 *     (the reference has no id column of its own: Arrow `take` indices are row positions,
 *     index.py:166-167).
 *   - distances use the reference's conventions (coder.py:38-50): smaller is better;
 *       FX_METRIC_L2     Euclidean distance WITH sqrt              (torch.cdist, coder.py:40)
 *       FX_METRIC_COSINE 0.5 - 0.5 * cos(q, x), eps 1e-12 on norms (coder.py:43-45)
 *       FX_METRIC_IP     -<q, x>                                   (coder.py:48)
 *   - results are ordered by (distance ascending, row ascending); lists shorter than k are
 *     padded with (row = -1, distance = +inf).
 *   - there is no CPU fallback: every entry point that computes needs a CUDA device.
 */
#ifndef FENIX_KNN_H_
#define FENIX_KNN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FX_ABI_VERSION 6

/* error codes */
#define FX_OK 0
#define FX_EINVAL (-1)   /* bad argument (NULL, negative size, unknown metric, k < 1 ...) */
#define FX_ECUDA (-2)    /* a CUDA runtime / driver call failed */
#define FX_ENOMEM (-3)   /* host or device allocation failed */
#define FX_ESTATE (-4)   /* call not valid in this state (append after finalize, search before) */
#define FX_EUNSUP (-5)   /* valid request this build does not support (dtype, huge dim) */
#define FX_ETRUNC (-6)   /* output capacity too small: out_offsets holds the sizes needed (fx_search_range) */

/* metrics: the five reference names map to three arithmetic forms (coder.py:39,42,47) */
#define FX_METRIC_L2 0     /* "l2", "euclidean" */
#define FX_METRIC_COSINE 1 /* "cosine" */
#define FX_METRIC_IP 2     /* "dot", "inner_product" */

/* precision modes of fx_search
 *   FP32: exact. A tensor-core pass (tcgen05) filters candidates under a rigorous error bound, survivors are
 *         re-ranked with fp64-accumulated arithmetic, the result is certified; queries whose certificate fails are
 *         settled by a re-run / preset-threshold refinement pass, in the last resort by the exact scan kernel.
 *         The filter runs on a bf16 shadow copy of the shard (built at finalize when HBM allows; FENIX_BF16_SHADOW=0
 *         disables it) or, without one, on the fp32 rows read as TF32.
 *   TF32 / BF16: the same tensor-core pass (TF32 over the fp32 rows / bf16 over the shadow) without
 *         slack or certificate; distances of the returned rows are still exact, membership is
 *         approximate (recall reported by bench.py). BF16 needs the shadow (FX_ESTATE otherwise).
 *         A handful of queries (<= 8, k <= 128) over a small shard (fp32 rows <= FENIX_DIRECT_MAX_MB, default 256 MB)
 *         skip all of that: ONE launch computes the fp64-accumulated distance of every row and selects (the latency
 *         path; same distances bit for bit, FENIX_DIRECT=0 disables it).
 *   EXACT_SCAN: forces the fp64-accumulating CUDA-core scan kernel (checker / fallback path).
 */
#define FX_PREC_FP32 0
#define FX_PREC_TF32 1
#define FX_PREC_BF16 2
#define FX_PREC_EXACT_SCAN 3

/* dtype of corpus rows */
#define FX_DTYPE_F32 0

typedef struct fx_ctx fx_ctx;       /* one CUDA device + its streams and scratch */
typedef struct fx_corpus fx_corpus; /* one device-resident, row-major corpus shard */
typedef struct fx_comm fx_comm;     /* this rank's membership in a group of row shards (one NCCL communicator) */
typedef struct fx_group fx_group;   /* ONE process owning several devices: contexts + communicators + a worker thread each */

typedef struct fx_stats {
  int64_t n_rows;            /* rows resident in the shard */
  int32_t dim;               /* vector width D */
  int32_t pitch;             /* floats per stored row (D rounded up to a multiple of 4) */
  int64_t device_bytes;      /* HBM held by this shard (rows + norms) */
  int64_t searches;          /* fx_search* calls completed */
  int64_t queries;           /* queries answered */
  int64_t fallback_queries;  /* queries recomputed by the exact scan (certificate failed twice) */
  int64_t refined_queries;   /* queries whose certificate failed once and were settled by the refinement pass */
  int64_t kernel_launches;   /* kernels of this library launched so far */
  double last_search_ms;     /* device time of the last search (CUDA events) */
  double last_main_kernel_ms;/* device time of the dominant kernel of the last search */
  int32_t last_path;         /* 0 = exact scan, 1 = tcgen05 TF32 filter + rerank, 2 = tcgen05 shadow filter (bf16 or int8) + rerank,
                              * 3 = direct scan: one launch, fp64 distances of every row (<= 8 queries over a small shard) */
  int32_t last_variant;      /* tcgen05 paths: bit 0 = resident-query kernel (narrow rows; else the streaming kernel),
                              * bit 1 = thresholds seeded by the sample prepass, bit 2 = CTA-pair (cta_group::2) streaming kernel */
  double last_exchange_ms;   /* sharded searches: device time of all-gather + merge of the last search (CUDA events) */
  int32_t last_operand;      /* operand of the last search's filter: 0 = fp32 / TF32 (or no filter), 1 = bf16 shadow,
                              * 2 = int8 normalised shadow (exact cosine at small k) */
  int32_t last_resident_queries; /* 1 = the last search's filter was the int8 CTA-pair kernel with its query tiles resident in
                              * shared memory (last_variant bit 2 is set too), else 0 */
} fx_stats;

/* ---- lifetime -------------------------------------------------------------------------- */

/* Bind a context to CUDA device `device`. Replaces nothing in the reference (it never
 * touches a device); one context per process-visible GPU. */
int fx_init(int device, fx_ctx** out);
/* Destroy every corpus created on `ctx` (fx_corpus_destroy) BEFORE shutting the context down: a corpus handle that
 * outlives its context points at freed state. */
int fx_shutdown(fx_ctx* ctx);

/* Create an empty shard able to hold `capacity_rows` vectors of width `dim`.
 * `row_base` is the global row position of local row 0 (multi-GPU row sharding: the value is
 * added to every row this shard reports). Replaces the per-call mmap view of
 * table.py:12-21 / arrow.py:6-8 with a resident copy owned by the library. */
int fx_corpus_create(fx_ctx* ctx, int64_t capacity_rows, int32_t dim, int32_t dtype,
                     int64_t row_base, fx_corpus** out);

/* Append `n_rows` row-major vectors (tightly packed, `dim` floats each) from HOST memory.
 * Called once per Arrow record-batch values buffer (the buffer torch.py:8-10 would have
 * wrapped). Pageable memory is fine: rows are staged through an internal pinned ring and
 * copied asynchronously. */
int fx_corpus_append(fx_corpus* c, const void* host_rows, int64_t n_rows);

/* Same, source already in DEVICE memory of the context's device. */
int fx_corpus_append_device(fx_corpus* c, const void* device_rows, int64_t n_rows);

/* Seal the shard: waits for uploads, computes and caches per-row squared norms (the work
 * cdist / F.normalize redo on every call in the reference, coder.py:40,44). */
int fx_corpus_finalize(fx_corpus* c);

/* Frees the shard (rows, norms, bf16 shadows). Must precede fx_shutdown of its context. Safe against concurrent use:
 * the handle is retired first (later calls on it fail with FX_EINVAL instead of touching freed memory) and the call
 * waits for searches already running on the shard. */
int fx_corpus_destroy(fx_corpus* c);

/* Tuning knob of the context, by the name of the environment variable that provides its default (FENIX_TC_PRE,
 * FENIX_TC_NO_RQ, FENIX_TC_PAIR, ...; every name is listed once, in TC_KNOB_TABLE of fenix_b200/csrc/tc_filter.cuh).
 * The environment is read ONCE, at fx_init; the search path never calls getenv. value = NULL restores the built-in
 * default; an unknown name fails with FX_EINVAL. */
int fx_set_option(fx_ctx* ctx, const char* name, const char* value);

/* ---- search ---------------------------------------------------------------------------- */

/* k-NN of `n_q` queries (HOST, row-major n_q x dim floats) against the shard.
 * `row_mask` (HOST, one byte per shard row, non-zero = row participates) or NULL; it is the
 * device form of index.py:161 `data.filter(expr)`.
 * out_rows [n_q*k] global row positions (row_base + local), out_dist [n_q*k] distances.
 * Replaces index.py:162 (distance column) + index.py:165-168 (select_k + take indices). */
int fx_search(fx_corpus* c, const float* queries, int64_t n_q, int32_t metric, int32_t k,
              int32_t precision, const uint8_t* row_mask, int64_t* out_rows, float* out_dist);
/* k is unbounded (the reference's select_k_unstable takes any maxval): k <= 320 on shards of >= 4096 rows takes the
 * tensor-core path, larger k the fp64 scan - above 2048 in passes of 2048 neighbours, each pass admitting only keys
 * above the last (distance, row) of the previous one. */

/* Same with every pointer in DEVICE memory; enqueued on the context's stream and
 * synchronised before return. Used by the multi-GPU path so the shard-local top-k stays
 * in HBM for the NCCL all-gather. */
int fx_search_device(fx_corpus* c, const float* d_queries, int64_t n_q, int32_t metric,
                     int32_t k, int32_t precision, const uint8_t* d_row_mask,
                     int64_t* d_out_rows, float* d_out_dist);

/* ---- batched IVF: every query scans only the rows of the cells it probes -------------------------------------------
 * The reference builds `__CODED_ID__ isin(probe codes)` per query and filters the table before the distance step
 * (index.py:113-126, 161); a batch of Q queries is Q such filters. Here the shard keeps an inverted index - its rows
 * grouped by cell - and ONE launch answers the whole batch: query q reads the posting lists of probes[q][*] (exact fp64
 * distances, the direct scan's arithmetic), so the bytes read are the probed rows, not Q passes over the shard.
 *   fx_corpus_set_cells: inv_rows [n_inv] LOCAL row positions grouped by cell (HOST), cell_off [n_cells + 1] offsets of
 *                        every cell's slice (HOST). Replaces the shard's previous cell structure.
 *   fx_search_cells:     probes [n_q * n_probe] cell numbers per query, -1 = unused slot, no cell twice in one query
 *                        (HOST); row_mask as in fx_search (ANDed: index.py:119-126). k <= 128, n_probe <= 512, else
 *                        FX_EUNSUP (the caller runs one masked fx_search per query instead). Lists shorter than k are
 *                        padded with (-1, +inf). */
int fx_corpus_set_cells(fx_corpus* c, const int32_t* inv_rows, int64_t n_inv, const int64_t* cell_off, int64_t n_cells);
int fx_search_cells(fx_corpus* c, const float* queries, int64_t n_q, int32_t metric, int32_t k, const int32_t* probes,
                    int32_t n_probe, const uint8_t* row_mask, int64_t* out_rows, float* out_dist);

/* Full distance column of ONE query against every shard row (HOST in / HOST out,
 * out_dist[n_rows]). This is the `maxval is None or len(data) <= maxval` branch of
 * index.py:162-165, where the reference returns all rows with __DISTANCE__ attached. */
int fx_distances(fx_corpus* c, const float* query, int32_t metric, float* out_dist);

/* Range search: every shard row r (after row_mask) with distance d(q, r) <= radius, for each of `n_q` queries (HOST,
 * row-major n_q x dim floats). d is the distance fx_distances reports for the row; the comparison is inclusive; a
 * query's hits are ordered by (distance, row), rows global (row_base + local). radius: one float per call, NaN is
 * FX_EINVAL, negative values are valid (inner-product distances can be negative), +inf admits every unmasked row.
 * Output in CSR form (HOST): query q's hits are out_rows / out_dist [out_offsets[q], out_offsets[q + 1]).
 * out_offsets [n_q + 1] is always written; when out_offsets[n_q] > capacity the call returns FX_ETRUNC and leaves
 * out_rows / out_dist untouched, so the caller can size its buffers and call again (a second search).
 * precision: FX_PREC_FP32 (the tensor-core filter with thresholds preset from the radius, every candidate reranked in
 * fp64; queries whose candidate lists overflow, and shards the tensor-core path does not take, run on the exact scan) or
 * FX_PREC_EXACT_SCAN; TF32 / BF16 are FX_EUNSUP. fx_stats: last_path / last_operand name the filter that ran,
 * fallback_queries counts the queries whose candidate lists overflowed and the scan settled, last_search_ms is the
 * device time of the search. */
int fx_search_range(fx_corpus* c, const float* queries, int64_t n_q, int32_t metric, float radius, int32_t precision,
                    const uint8_t* row_mask, int64_t capacity, int64_t* out_offsets, int64_t* out_rows, float* out_dist);

/* ---- IVF codebook training ------------------------------------------------------------------------------------------
 * One epoch of mini-batch k-means over the rows of `n_shards` contiguous row shards (shard i's rows start at its
 * row_base; all shards share dim). books [n_books][k][dim] HOST, in: current codewords, out: trained.
 * positions [n_steps][n_books * batch] HOST, global row positions, ascending within a step; step s trains codebook j
 * on positions[s][j*batch .. (j+1)*batch). metric as fx_search. Runs on shard 0's device; rows of other shards are
 * gathered on their devices and copied there in bounded chunks. n_steps = 0 leaves `books` untouched.
 * Per step and codebook: every sample row takes the codeword with the smallest fp32 distance (fx_search's distance,
 * fp64 sums in ascending coordinate order; ties to the lowest codeword), then every codeword becomes
 * (old + sum of its rows) / (1 + count), summed in fp64 in sample order and rounded once to fp32. Cosine: the old
 * codeword and the rows are normalised (x / max(|x|, 1e-12), fp64) before the sum and the mean after it. The result
 * is deterministic: the same call gives the same bits. */
int fx_train_codebooks(fx_corpus* const* shards, int32_t n_shards, int32_t metric, int32_t n_books, int32_t k,
                       int32_t batch, const int64_t* positions, int64_t n_steps, float* books);

/* Merge `n_lists` per-shard results (DEVICE, each [n_q*k], laid out list-major:
 * rows[l*n_q*k + q*k + j]) into the global top-k ordered by (distance, row).
 * The step after the all-gather of the k*world candidates (fx_search_sharded does both itself). Any lists * k. */
int fx_merge_topk(fx_ctx* ctx, const int64_t* d_rows, const float* d_dist, int32_t n_lists,
                  int64_t n_q, int32_t k, int64_t* d_out_rows, float* d_out_dist);

/* ---- multi-GPU: row shards, one exchange step ------------------------------------------------
 * Rank r of W owns the contiguous rows [r*ceil(N/W), ...) (fx_corpus_create's row_base), answers every query on its
 * shard, and the k*W candidates per query are all-gathered (NCCL over NVLink / NVSwitch) and merged by (distance,
 * row). Everything - query all-gather, shard search, candidate all-gather, merge, result copy - is enqueued on the
 * context's stream with ONE host synchronisation at the end; a per-rank "flagged queries" word travels with the
 * candidates, so that the rare certificate failure is settled collectively (second exchange) without a host round
 * trip on the common path. The reference has no counterpart (SURVEY.md section 2.1: no parallelism at all).
 *
 * Two deployments share the per-rank code:
 *   - one process per GPU (torchrun): fx_comm_unique_id on rank 0, broadcast the 128 bytes by any means,
 *     fx_comm_init_rank everywhere, then fx_search_sharded / fx_search_sharded_device collectively;
 *   - one process owning all devices (the Flight server): fx_group_create, corpora on fx_group_ctx(g, i), then
 *     fx_group_search from any thread (searches on a group serialise).
 * NCCL is taken from the process (libnccl.so.2, dlopen; FENIX_NCCL_LIB overrides the name): nothing links against it. */
#define FX_COMM_ID_BYTES 128
int fx_comm_unique_id(void* out_id /* FX_COMM_ID_BYTES */);
int fx_comm_init_rank(fx_ctx* ctx, const void* id, int32_t world, int32_t rank, fx_comm** out);
int fx_comm_destroy(fx_comm* comm);

/* Collective. `queries`: the WHOLE batch in HOST memory on every rank (each rank uploads only its 1/W slice and the
 * slices are all-gathered over NVLink). `row_mask`: this shard's rows (HOST) or NULL. out_rows / out_dist: HOST
 * [n_q*k], or both NULL on ranks that do not need the merged result (they skip merge and copy). */
int fx_search_sharded(fx_corpus* c, fx_comm* comm, const float* queries, int64_t n_q, int32_t metric, int32_t k,
                      int32_t precision, const uint8_t* row_mask, int64_t* out_rows, float* out_dist);
/* Collective, everything in DEVICE memory: d_queries = the whole batch on every rank; d_out_* may be NULL. */
int fx_search_sharded_device(fx_corpus* c, fx_comm* comm, const float* d_queries, int64_t n_q, int32_t metric,
                             int32_t k, int32_t precision, const uint8_t* d_row_mask, int64_t* d_out_rows,
                             float* d_out_dist);

/* One process, n devices: contexts, an NCCL communicator per device (ncclCommInitAll) and one worker thread per
 * device. fx_group_ctx(g, i) is the context shard i must be created on. */
int fx_group_create(const int32_t* devices, int32_t n_devices, fx_group** out);
int fx_group_size(fx_group* g);
fx_ctx* fx_group_ctx(fx_group* g, int32_t i);
/* shards[i] lives on fx_group_ctx(g, i) and holds the i-th contiguous row range. queries / out_* HOST; row_mask:
 * HOST, one byte per row of the WHOLE corpus (shard i reads its range) or NULL. Replaces, for a corpus spread over
 * the GPUs of one box, what fx_search replaces for one GPU (index.py:162-168). */
int fx_group_search(fx_group* g, fx_corpus* const* shards, const float* queries, int64_t n_q, int32_t metric,
                    int32_t k, int32_t precision, const uint8_t* row_mask, int64_t* out_rows, float* out_dist);
/* Destroys the workers, communicators and contexts (destroy the shards first). */
int fx_group_destroy(fx_group* g);

/* ---- introspection --------------------------------------------------------------------- */

int fx_get_stats(fx_corpus* c, fx_stats* out);

/* Diagnostics: raw tensor-core filter scores of the first min(n_q,128) queries (HOST) against the
 * first 256 shard rows, out_scores[128*256] row-major (query, row). Scores are the filter's ranking
 * quantity: l2  <q,x> - 0.5|x|^2, cosine  <q,x>/max(|x|,eps), ip  <q,x>. Used by the tests to check the
 * TF32 error bound the exactness certificate relies on. */
int fx_debug_scores(fx_corpus* c, const float* queries, int64_t n_q, int32_t metric, float* out_scores);
const char* fx_last_error(void);
int fx_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* FENIX_KNN_H_ */
