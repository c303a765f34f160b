/*
 * voitta_b200.h — C ABI of libvoitta_b200.so, the B200 (sm_100a) backend for voitta-rag's
 * retrieval hot path.
 *
 * The reference has no FFI: its boundary is the Python class
 * voitta.services.vector_store.VectorStoreService, which forwards every arithmetic step to
 * Qdrant through qdrant_client.  Each entry point below replaces one of those qdrant_client
 * calls (file:line into /root/reference/src/voitta/services/vector_store.py) and is what the
 * Python host layer (voitta-rag_b200/engine.py, ctypes) binds.  INTEGRATION.md shows the
 * binding a voitta maintainer adds.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; vb_last_error() returns a
 *     thread-local message for the last failure on the calling thread;
 *   - plain pointers and sizes only; "host" pointers are caller-owned host memory, "dev"
 *     pointers are caller-owned device memory on the index's device;
 *   - rows are numbered in insertion order, starting at `row_base` (vb_create); a row id is
 *     the only handle the library returns — payloads and point ids stay in the host layer;
 *   - a missing timestamp is VB_TS_MISSING (a `must` range on a missing field fails);
 *   - thread-safety: every entry point takes the index's (recursive) mutex for its whole duration, so the
 *     one-call functions (vb_search, vb_upsert, vb_delete_rows, ...) may be called from any number of
 *     threads.  The staged form (vb_stage ... vb_fetch) is a multi-call protocol over per-index slots and must
 *     be driven by one thread at a time per index; a batch staged before a write is refused by vb_run_local.
 *   - no CPU fallback: every compute entry point fails if no sm_100 device is present.
 */
#ifndef VOITTA_B200_H
#define VOITTA_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VB_ABI_VERSION 4
#define VB_TS_MISSING INT64_MIN
#define VB_MAX_KPRIME 1024          /* limit*3 <= 1024 */
#define VB_MAX_QUERY_TERMS 256      /* non-zeros per sparse query */

typedef struct vb_index vb_index;   /* opaque */

/* fusion of the dense and sparse branch lists */
enum vb_fusion {
    VB_FUSE_DENSE_ONLY = 0, /* vector_store.py:611-619  dense-only query_points(limit)            */
    VB_FUSE_WEIGHTED   = 1, /* vector_store.py:659-697  min-max normalised weighted sum (voitta)  */
    VB_FUSE_RRF        = 2  /* qdrant Fusion.RRF: sum 1/(2+rank) (BASELINE.json configs 2-5)      */
};

enum vb_ts_field { VB_TS_NONE = 0, VB_TS_CREATED = 1, VB_TS_MODIFIED = 2 };

/* One evaluated filter (vector_store.py:462-530 _build_filter).  The host layer folds the
 * folder_path / index_folder string clauses into a bitset over scope ids (one scope id per
 * distinct (folder_path, index_folder) pair of unrestricted rows, and one per distinct
 * (folder_path, index_folder, allowed_users set) of rows that carry an ACL): bit s set <=> rows
 * of scope s pass
 *   must folder_path == folder_filter, must folder_path IN include_folders,
 *   must_not folder_path == e (each), must_not index_folder == f (each),
 *   and, for a caller with principals P, allowed_users absent or sharing an entry with P.
 * scope_bits == NULL means "no folder clause".  The range is inclusive on both sides
 * (gte / lte); use INT64_MIN+1 / INT64_MAX for an absent bound. */
typedef struct vb_filter {
    const uint32_t* scope_bits;   /* host, scope_words words, or NULL */
    uint32_t        scope_words;
    int32_t         ts_field;     /* enum vb_ts_field */
    int64_t         ts_lo, ts_hi;
} vb_filter;

/* A batch of B hybrid queries.  voitta itself always issues B = 1 (mcp_server.py:474). */
typedef struct vb_query_batch {
    uint32_t        n_queries;    /* B */
    const float*    dense;        /* host [B][dim] fp32, any norm (normalised inside)         */
    const int64_t*  sp_indptr;    /* host [B+1] or NULL (no sparse branch for any query)      */
    const uint32_t* sp_term;      /* host [nnz] hashed term ids (sparse_embedding.py:29-39)   */
    const double*   sp_weight;    /* host [nnz] query values (IDF applied iff !apply_idf)     */
    int32_t         apply_idf;    /* 1: multiply by ln(1+(N-df+.5)/(df+.5)) using this index  */
    uint32_t        n_filters;    /* filters passed, any number; one per query is fine        */
    const vb_filter* filters;     /* host [n_filters]; ones no query uses are ignored, ones of
                                     equal content (same ts_field, same range if it has one,
                                     same scope words up to trailing zeros) are merged          */
    const int32_t*  filter_of;    /* host [B] index into filters, -1 = unfiltered; NULL = all -1 */
    uint32_t        limit;        /* results per query                                        */
    uint32_t        kprime;       /* per-branch over-fetch, voitta: 3*limit (vector_store.py:636) */
    int32_t         fusion;       /* enum vb_fusion, applied to queries that have sparse terms */
    double          sparse_weight;/* w; dense weight is 1-w (vector_store.py:634)             */
} vb_query_batch;

/* Result buffers (host).  Any of the branch pointers may be NULL. */
typedef struct vb_result {
    uint64_t* rows;        /* [B][limit] fused result rows, rank order                        */
    double*   scores;      /* [B][limit] fused score (dense-only: the cosine, as float)       */
    int32_t*  counts;      /* [B]                                                             */
    uint64_t* dense_rows;  /* [B][kprime] dense branch, rank order (query_points :640-645)    */
    float*    dense_scores;
    int32_t*  dense_counts;
    uint64_t* sparse_rows; /* [B][kprime] sparse branch (query_points :647-656)               */
    float*    sparse_scores;
    int32_t*  sparse_counts;
} vb_result;

typedef struct vb_stats {
    uint64_t n_rows, n_live, nnz, n_terms;
    uint64_t searches, queries, overflow_reruns;
    double   last_search_ms;      /* device time of the last vb_search (CUDA events)          */
    double   last_dense_ms, last_sparse_ms, last_select_ms, last_mask_ms, last_fuse_ms;
    uint32_t last_dense_path;     /* 1 = GEMV scan (K1), 2 = tcgen05 GEMM (K2 / K2T), 3 = single-pass GEMV scan (K1F) */
    uint32_t last_launches;       /* kernels launched by the last vb_search                   */
    uint64_t device_bytes;
    uint64_t last_h2d_bytes, last_d2h_bytes;   /* host<->device copies of the last staged search */
    uint64_t last_dense_passes;                /* passes over the shard's dense rows (K1: B, K2: sub-batches) */
    uint64_t last_big_rows;                    /* rows of the largest (last) segment of the last search */
    double   last_dense_big_ms, last_sparse_big_ms;  /* profile: dense / sparse kernel time of that segment */
    uint64_t dim, row_base;                    /* geometry of the index (what vb_load restored)            */
    uint64_t index_builds;                     /* full builds of the inverted index so far (sort of every posting) */
    uint64_t delta_rows;                       /* rows appended since the last build (scored from the forward index) */
    uint32_t last_overflow_lists;              /* candidate lists that overflowed in the last fetched search (0 = none)  */
    uint32_t last_overflow_first;              /* the first of them: list q = dense list of query q, B + q = its sparse list */
    uint32_t last_sel_rows;                    /* K2T row selection: rows of the largest segment that pass the batch-wide filter (0 = not run) */
    uint32_t last_sel_used;                    /* 1 = the tensor-core kernel walked the compacted copy of those rows        */
} vb_stats;

int         vb_abi_version(void);
const char* vb_last_error(void);

/* Replaces QdrantClient(...) + create_collection (vector_store.py:66-115): cosine dense
 * vectors of `dim` floats stored as bf16 + fp32 inverse norm, sparse "bm25" with IDF.
 * `row_base` is added to every row id this index returns (shard offset, SURVEY §8e). */
int  vb_create(int32_t dim, int32_t device, uint64_t capacity_hint, uint64_t row_base, vb_index** out);
void vb_destroy(vb_index* h);

/* Replaces client.upsert (vector_store.py:311-313).  Appends n rows; returns the id of the
 * first in *first_row.  sp_indptr == NULL: rows carry no sparse vector.  Sparse indices must be
 * strictly ascending inside a row (the host layer sorts, as qdrant does at upsert). */
int vb_upsert(vb_index* h, uint64_t n, const float* dense,
              const int64_t* sp_indptr, const uint32_t* sp_term, const float* sp_val,
              const uint32_t* scope_id, const int64_t* created, const int64_t* modified,
              uint64_t* first_row);

/* Bulk variant of vb_upsert whose inputs already live on the device (bench / replay loaders;
 * rows_bf16 is [n][dim] bf16).  Any of sp_*, scope_id, created, modified may be NULL. */
int vb_upsert_dev(vb_index* h, uint64_t n, const void* rows_bf16,
                  const int64_t* sp_indptr, const uint32_t* sp_term, const float* sp_val,
                  const uint32_t* scope_id, const int64_t* created, const int64_t* modified,
                  uint64_t* first_row);

/* Replaces client.delete(FilterSelector) (vector_store.py:340,378,419): the host layer
 * resolves the payload predicate to rows; the library tombstones them (and they stop
 * counting towards N and df of the IDF, as in qdrant). */
int vb_delete_rows(vb_index* h, uint64_t n, const uint64_t* rows);

/* Replaces client.set_payload (vector_store.py:216-231) for the one payload field the device filters on:
 * scope_id[rows[i]] = scope_id[i] for rows that already exist.  The host layer calls it when a file's
 * allowed_users change, which moves its rows to another (folder, index folder, ACL) scope.  Rows are global
 * ids (row_base included), as in vb_delete_rows; deleted rows are accepted.  A NULL pointer, a row out of
 * range or a row given twice is an error that names the row, and then nothing is written.  Like every
 * write it refuses a batch staged before it and drops the kept row selection; N, df and the inverted index
 * do not change.  Synchronous: the new ids are in place when it returns. */
int vb_set_scope(vb_index* h, uint64_t n, const uint64_t* rows, const uint32_t* scope_id);

/* Index maintenance.  The reference interleaves store_chunks batches of 100 (indexing.py:434,560) and
 * deletes (indexing.py:284, watcher.py:149-171) with searches, so writes do not invalidate the sorted
 * inverted index: appended rows form a delta that is scored from the forward index, deletes only clear
 * alive bits, and N / df follow both exactly.  vb_upsert merges the delta once it passes a threshold
 * (max(16384, indexed rows / 32); option "delta_max"); a bulk load that jumps far past it is merged by the
 * next search or by vb_optimize, which forces the merge now (bulk loaders call it when they are done). */
int vb_optimize(vb_index* h);

/* N (live points) and the document frequency of each term over live rows: the two inputs of
 * qdrant's IDF modifier.  Used by the multi-GPU host layer to sum df across shards. */
int vb_term_stats(vb_index* h, uint32_t n_terms, const uint32_t* terms, uint64_t* df, uint64_t* n_live);

/* Replaces the two query_points calls and the fusion of vector_store.py:593-697 for a batch.
 * Host buffers in, host buffers out (copies inside).  */
int vb_search(vb_index* h, const vb_query_batch* q, vb_result* out);

/* Multi-GPU building blocks (one process per GPU, SURVEY §8e).
 * vb_search_local: branch top-k' of this shard, left on the device as ONE candidate block of
 *   VB_CAND_BLOCK_WORDS(B, kprime) u64 words: cand[2][B][kprime] (0 = empty slot; branch 0 dense,
 *   1 sparse) followed by one flag word (shard overflowed), ready for an all-gather.  Query
 *   weights must already carry the GLOBAL idf (apply_idf = 0).
 * vb_merge_fuse: merge `n_shards` gathered candidate blocks (device, contiguous) into the
 *   global branch lists, fuse, and write host results like vb_search. */
#define VB_CAND_BLOCK_WORDS(B, kprime) (2ull * (B) * (kprime) + 1ull)
int vb_search_local(vb_index* h, const vb_query_batch* q, uint64_t* cand_dev);
int vb_merge_fuse(vb_index* h, const vb_query_batch* q, uint32_t n_shards,
                  const uint64_t* gathered_dev, vb_result* out);

/* Staged form of the same work, for callers that overlap or time the phases themselves
 * (bench.py, the multi-GPU host layer).  vb_search == vb_stage + vb_run_local + vb_run_fuse + vb_fetch.
 *   vb_stage     validate, resolve terms/IDF, upload the batch (the only H2D copy); need_corpus = 0
 *                when only a merge of gathered candidates will follow.
 *   vb_run_local K0 + K1/K2 + K3 + select over this shard, asynchronously on the index's stream;
 *                cand_dev (optional) receives the packed branch candidates [2][B][kprime].
 *   vb_run_fuse  gathered_dev != NULL: merge n_shards candidate blocks first; then K4.  Asynchronous.
 *   vb_fetch     D2H of the results, stream sync, decode; *overflowed = 1 asks for a safe-mode re-run
 *                (vb_set_option "safe_mode"). */
int vb_stage(vb_index* h, const vb_query_batch* q, int32_t want_branches, int32_t need_corpus);
int vb_run_local(vb_index* h, uint64_t* cand_dev);
int vb_run_fuse(vb_index* h, uint32_t n_shards, const uint64_t* gathered_dev);
int vb_fetch(vb_index* h, vb_result* out, int32_t* overflowed);

/* Device-resident queries (SURVEY §8 f-4): the embedding forward (embedding.py:76-86 — `model.encode` then
 * `.tolist()`) can leave its output on the GPU and skip the list[float] -> H2D hop.  Same as vb_stage / vb_search, but
 * the dense rows are read from `dense_dev` (fp32 [B][dim] on this index's device; q->dense is ignored, may be NULL).
 * `producer_stream` is the cudaStream_t the producer wrote them on (NULL = the legacy default stream): the library
 * orders its device-to-device copy after that stream's work, without a host synchronisation.  The buffer may be
 * reused when vb_search_dev returns / after the vb_fetch of the staged batch.  A NaN or inf in a query is found on
 * the device and reported by vb_fetch / vb_search(_dev) as an error (qdrant-client local mode asserts on NaN). */
int vb_stage_dev(vb_index* h, const vb_query_batch* q, const float* dense_dev, void* producer_stream,
                 int32_t want_branches, int32_t need_corpus);
int vb_search_dev(vb_index* h, const vb_query_batch* q, const float* dense_dev, void* producer_stream, vb_result* out);

/* Tuning knobs (tests exercise every path with them): key = "dense_path" (0 auto, 1 K1, 2 K2),
 * "seg_first", "seg_ratio", "safe_mode", "profile" (per-phase CUDA-event times in vb_stats),
 * "stream" (a cudaStream_t to run on instead of the index's own stream; 0 restores it),
 * "dense_compact" (row selection for the tensor-core kernels under a batch-wide filter: -1 auto, 0 off,
 * 1..100 = walk the compacted copy when at most that % of a segment passes), "dense_compact_min_rows",
 * "sel_reuse" (1, the default: keep that copy across batches while the filter, the index and the plan stay the same;
 * 0: copy it every batch).
 * The full list with defaults is vb_set_option in csrc/vb_api.cu; unknown keys are an error.  Options belong to one
 * index, and every index starts at the defaults: the process environment does not change them. */
int vb_set_option(vb_index* h, const char* key, int64_t value);

int vb_get_stats(vb_index* h, vb_stats* out);
/* With option "profile" = 1: the timed regions of the last fetched search as (phase | 8 if largest launch, start ms,
 * end ms) triples relative to the start of the search, in launch order — phases 0 mask, 1 dense, 2 sparse, 3 select,
 * 4 fuse.  Start / end come from CUDA events on the stream each region ran on, so the overlap of the dense and the
 * sparse chain (two streams) can be read off.  *n = regions available; at most `cap` are written. */
int vb_get_timeline(vb_index* h, double* out, uint32_t cap, uint32_t* n);
int vb_sync(vb_index* h);

/* Snapshot of everything the shard holds on the device: bf16 rows, inverse norms, filter columns,
 * tombstones and the forward sparse CSR (the inverted index is derived data and is rebuilt on the
 * first search after vb_load).  Stands in for Qdrant's on-disk storage (/qdrant/storage,
 * docker-compose.yml:8-9): the host side (ids, payloads) is saved next to it by the Python layer.
 * vb_load creates a new index on `device` with the snapshot's dimension and row_base. */
int vb_save(vb_index* h, const char* path);
int vb_load(const char* path, int32_t device, vb_index** out);

#ifdef __cplusplus
}
#endif
#endif /* VOITTA_B200_H */
