// libvoitta_b200.so — host side of the C ABI declared in include/voitta_b200.h.
// Owns device memory, streams and the launch schedule; all arithmetic is in the kernels
// (mask.cuh K0/K5, dense_scan.cuh K1, dense_gemm.cuh K2, sparse.cuh K3, topk.cuh select + K4).
#include "../../include/voitta_b200.h"
#include "common.cuh"
#include "mask.cuh"
#include "dense_scan.cuh"
#include "dense_gemm.cuh"
#include "dense_compact.cuh"
#include "sparse.cuh"
#include "sparse_ms.cuh"
#include "sparse_mh.cuh"
#include "sparse_delta.cuh"
#include "topk.cuh"

#include <unistd.h>

#include <algorithm>
#include <array>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_err;

static int vb_fail(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return 1;
}

#define CK(call)                                                                          \
    do {                                                                                  \
        cudaError_t e__ = (call);                                                         \
        if (e__ != cudaSuccess)                                                           \
            return vb_fail("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)
#define CKK(what)                                                                         \
    do {                                                                                  \
        cudaError_t e__ = cudaGetLastError();                                             \
        if (e__ != cudaSuccess)                                                           \
            return vb_fail("launch %s failed: %s (%s:%d)", what, cudaGetErrorString(e__), __FILE__, __LINE__); \
    } while (0)
#define TRY(expr)                  \
    do {                           \
        int rc__ = (expr);         \
        if (rc__) return rc__;     \
    } while (0)

// ------------------------------------------------------------------------------------------------
// buffers
// ------------------------------------------------------------------------------------------------
struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

struct HostBuf {
    void* p = nullptr;
    size_t cap = 0;
    template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

struct Batch {
    uint32_t B = 0, k = 0, limit = 0, n_lists = 0, n_qterms = 0, nt_max = 1, n_filters = 0, mask_words = 0, n_blocks = 0;
    bool any_sparse = false, use_mask = false, any_heavy = false;
    bool any_ms = false, any_old = false, any_mh = false;   // some sparse query goes to K3M / stays on K3 / goes to K3H
    uint32_t n_old = 0;                        // sparse queries that stay on K3 in every segment
    uint32_t n_dir = 0;                        // sparse queries K3 scores in the direct segment when K3M runs in stages (K3 + K3H ones)
    uint32_t n_rows = 0;                       // rows of the index when the batch was staged
    uint64_t gen = 0;                          // write generation of the index when the batch was staged
    uint32_t seg_ratio = 32;                   // growth factor of the segment schedule for this batch
    std::vector<int32_t> mode, mask_of_host;
    std::vector<uint64_t> sel_filter;          // every query on one filter: its content as the mask kernel sees it (else empty)
    // device pointers into h->args
    const float* d_q = nullptr;
    const int64_t* d_qindptr = nullptr;
    const double* d_qweight = nullptr;
    const double* d_qub = nullptr;
    const uint32_t* d_qterm = nullptr;
    const int32_t* d_qhidx = nullptr;
    const uint8_t* d_qrelaxed = nullptr;
    const uint32_t* d_qlo = nullptr;
    const uint32_t* d_qhi = nullptr;
    const uint32_t* d_qplo = nullptr;          // full posting ranges (frequent terms included): MaxScore kernel
    const uint32_t* d_qphi = nullptr;
    const uint32_t* d_slotq = nullptr;         // query of every term slot
    const uint8_t* d_qms = nullptr;            // [B] 1 = scored by the MaxScore kernel outside the direct segment
    const uint32_t* d_oldq = nullptr;          // [n_old] the sparse queries neither K3M nor K3H takes
    const uint32_t* d_dirq = nullptr;          // [n_dir] those plus the K3H queries (first, direct segment)
    const uint32_t* d_qtab = nullptr;          // [n_qterms] bucket table offset of the term (VB_MS_NO_TAB = none)
    const uint8_t* d_qshift = nullptr;         // [n_qterms] bucket shift
    // the query batch inverted by term, for the delta rows (K3D)
    const uint32_t* d_ut = nullptr;            // [n_uterms] distinct terms, ascending
    const uint32_t* d_up = nullptr;            // [n_uterms + 1]
    const uint32_t* d_uq = nullptr;            // [n_qterms] query
    const double* d_uw = nullptr;              // [n_qterms] weight
    uint32_t n_uterms = 0;
    uint32_t base_rows = 0;                    // rows covered by the inverted index when the batch was staged
    uint64_t ms_max_post = 0;                  // most postings any K3M query's terms hold (how many stages a search needs)
    const int32_t* d_maskof = nullptr;
    VbFilterTiles ft_k2, ft_k2t;               // mask mode 3 (> 31 filters): filter tables per K2 sub-batch / per K2T query tile
    const int32_t* d_mode = nullptr;
    const VbFilterDev* d_filters = nullptr;
    uint32_t need_created = 0, need_modified = 0, need_scope = 0;
    // lists
    float* tau = nullptr;
    uint32_t* cnt = nullptr;
    uint32_t* overflow = nullptr;
    uint32_t* gtau = nullptr;                  // [n_lists] K1F: threshold shared by the CTAs of one pass (ordered score, 0 = none)
    uint32_t* done = nullptr;                  // [n_lists] K1F: CTAs that have appended their part (the last one merges)
    // fusion / output
    double w_sparse = 0.0;
    bool want_branches = false, valid = false, need_corpus = true;
    size_t o_rows = 0, o_sc = 0, o_cnt = 0, o_keys = 0, o_lcnt = 0, o_ovf = 0, o_bad = 0, out_bytes = 0;
    size_t h2d_bytes = 0;
};

struct vb_index {
    int32_t dim = 0, d_pad = 0, device = 0;
    uint64_t row_base = 0;
    uint64_t n_rows = 0, n_live = 0, cap_rows = 0;
    uint64_t nnz = 0, cap_nnz = 0;
    cudaStream_t stream = nullptr, own_stream = nullptr, aux_stream = nullptr, sel_stream = nullptr;
    cudaEvent_t ev_sel_fork = nullptr, ev_sel[8] = {};
    cudaEvent_t ev0s[2] = {nullptr, nullptr}, ev1s[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    int cur = 0;                               // current slot: two batches can be in flight (pipelined callers)
    std::recursive_mutex mu;               // one-call entry points hold it for the whole call; staged calls re-enter
    int sm_count = 148;
    uint64_t device_bytes = 0;

    // corpus (device)
    DevBuf rows, inv_norm, scope_id, created, modified, alive;
    DevBuf sp_indptr, sp_term, sp_val;     // row-major CSR as appended
    std::vector<uint32_t> alive_host;      // mirror of the alive bitmap
    bool any_ts_created = false, any_ts_modified = false;

    // inverted index (device) + host copy of the term directory
    bool sparse_dirty = true;
    uint64_t write_gen = 0;                // bumped by every upsert / delete: a staged batch must not outlive it
    DevBuf post_row, post_val;
    uint64_t nnz_live = 0;
    std::vector<uint32_t> terms_sorted;
    std::vector<uint64_t> term_ptr;
    std::vector<float> term_maxval;        // largest posting value per term (MaxScore upper bounds)
    std::vector<int32_t> heavy_of_slot;    // term slot -> dense column, -1 = none
    std::vector<uint32_t> tab_off_of_slot; // term slot -> first entry of its bucket table in term_tab (VB_MS_NO_TAB = none)
    std::vector<uint8_t> tab_shift_of_slot;
    DevBuf term_tab;                       // bucket tables: first posting with row >= b << shift, per term (K3M lookups)
    uint64_t base_rows = 0;                // rows the inverted index was built over; rows past it are the DELTA (K3D)
    std::unordered_map<uint32_t, int64_t> df_adj;   // term -> change of its live df since the build (delta rows +, deletes -)
    uint64_t dead_since_build = 0;         // rows tombstoned since the build (their postings are still in the index)
    DevBuf heavy_vals;                     // [n_heavy][heavy_stride] fp32, NaN = term absent from the row
    uint32_t n_heavy = 0, heavy_stride = 0;
    bool sparse_nonneg = false;            // no negative posting value in the shard

    // per-search scratch
    DevBuf args, mask, cand, lists, offs, plan, out, q_hat, q_bf16, q_scale, tmp;
    DevBuf sel_rows, sel_inv, sel_ids, sel_meta;   // K2T row selection (dense_compact.cuh): compacted copy, its inverse norms / row ids, {count, decision, block sums}
    bool sel_no_memory = false;               // the scratch matrix did not fit once: do not try again
    // What the row-selection scratch holds (run_branches): the copy depends only on the batch-wide filter's content, the
    // rows / inverse norms / filter columns / alive bits (versioned by write_gen) and the plan, never on the queries.  A
    // batch whose key equals it skips the copy of every segment listed in sel_segs.  Empty sel_key = nothing valid.
    std::vector<uint64_t> sel_key;
    std::vector<std::array<uint64_t, 5>> sel_segs;   // {r0, r1, row_off, meta_off, cap_rows} of every valid segment
    DevBuf ms_rec, ms_q, ms_units, ms_counters, mh_units;  // K3M / K3H: plan output, work-unit prefixes, counters
    HostBuf h_args_s[2], h_out_s[2], h_stage, h_sel[2];
    bool sel_ran[2] = {false, false};         // the row selection ran for the batch staged in this slot
    uint32_t cand_cap = 0;

    // options
    int64_t opt_dense_path = 0, opt_seg_first = 2048, opt_seg_ratio = 0 /* 0 = auto */, opt_safe_mode = 0, opt_profile = 0, opt_k2_precision = 0, opt_overlap = 1, opt_k2_tiled = 1, opt_sparse_prune = 20, opt_sparse_prune_force = 0, opt_sparse_dense = 1;
    int64_t opt_sparse_ms = 1;             // 1: posting-driven MaxScore kernel (K3M) outside the direct segment; 0: K3 everywhere
    int64_t opt_ms_budget = 100;           // K3M: non-essential ub budget in % of tau (100 = full MaxScore partition)
    int64_t opt_ms_chunk = 0;              // K3M: postings per work unit (0 = auto)
    int64_t opt_mh_budget = 50;            // K3H: non-essential ub budget in % of tau (see sparse_mh.cuh: 100 % leaves every touched row to be finished by lookups)
    int64_t opt_sparse_mh = 0;             // 1: long queries go to K3H (hash-accumulate MaxScore); 0 (default): they stay on K3 —
                                           // measured on the cfg5 shard: K3 190 ms, K3H 346-715 ms depending on the budget (sparse_mh.cuh)
    int64_t opt_k1f = 1;                   // single-pass dense scan (K1F) for batches of at most VB_K1F_MAX_B queries
    int64_t opt_ms_staged = 1;             // K3M: 1 = posting stages over the whole index, 0 = once per row segment
    int64_t opt_delta_max = 0;             // rows the delta may hold before vb_upsert merges it into the index (0 = auto)
    int64_t opt_dense_compact_min_rows = 1 << 18;   // ... on segments of at least this many rows (tests lower it)
    int64_t opt_sel_reuse = 1;             // row selection: 1 = keep the copy across batches while its key holds, 0 = copy every batch
    int64_t opt_dense_compact = -1;        // K2 / K2T: walk a compacted copy of the passing rows when a batch-wide filter passes at most this % of a
                                           // segment (0 = never, -1 = auto: where the copy costs less than the passes over the dropped rows)
    int64_t opt_ms_max_terms = VB_MS_MAX_TERMS;         // K3M scores queries of at most this many terms; longer ones accumulate (K3)

    const float* q_dev = nullptr;          // vb_stage_dev / vb_search_dev: dense queries of the batch being staged live on this device
    cudaStream_t q_dev_stream = nullptr;   //   ... written on this stream
    cudaEvent_t ev_q = nullptr;

    vb_stats stats{};
    Batch staged_s[2];
    bool staged_safe = false;
    std::vector<cudaEvent_t> prof_events;
    std::vector<int> prof_phase;
    std::vector<double> timeline;          // profile: (phase, start ms, end ms) of every timed region of the last search
};

static int dev_reserve(vb_index* h, DevBuf& b, size_t bytes, bool keep, size_t used_bytes = 0) {
    if (bytes <= b.cap) return 0;
    size_t ncap = keep ? std::max(bytes, b.cap + b.cap / 2) : bytes;
    ncap = align_up(ncap, 256);
    void* np = nullptr;
    CK(cudaMalloc(&np, ncap));
    if (keep && b.p && used_bytes) {
        CK(cudaMemcpyAsync(np, b.p, used_bytes, cudaMemcpyDeviceToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    if (b.p) { CK(cudaFree(b.p)); h->device_bytes -= b.cap; }
    b.p = np;
    b.cap = ncap;
    h->device_bytes += ncap;
    return 0;
}

static int host_reserve(HostBuf& b, size_t bytes) {
    if (bytes <= b.cap) return 0;
    if (b.p) CK(cudaFreeHost(b.p));
    b.p = nullptr;
    b.cap = 0;
    size_t ncap = align_up(bytes + bytes / 4, 4096);
    CK(cudaMallocHost(&b.p, ncap));
    b.cap = ncap;
    return 0;
}

static void dev_free(vb_index* h, DevBuf& b) {
    if (b.p) { cudaFree(b.p); h->device_bytes -= b.cap; }
    b.p = nullptr;
    b.cap = 0;
}

// ------------------------------------------------------------------------------------------------
// tiny utility kernels
// ------------------------------------------------------------------------------------------------
__global__ void vb_fill_i64_kernel(int64_t* p, uint64_t n, int64_t v) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) p[i] = v;
}
__global__ void vb_fill_u32_kernel(uint32_t* p, uint64_t n, uint32_t v) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) p[i] = v;
}
__global__ void vb_offset_i64_kernel(const int64_t* src, int64_t* dst, uint64_t n, int64_t add) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) dst[i] = src[i] + add;
}
__global__ void vb_set_alive_kernel(uint32_t* alive, uint64_t first, uint64_t n) {
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t r = first + i;
        atomicOr(&alive[r >> 5], 1u << (r & 31u));
    }
}
__global__ void vb_find_tail_kernel(const uint64_t* keys, uint64_t n, uint64_t* out) {
    uint64_t lo = 0, hi = n;
    while (lo < hi) { const uint64_t mid = (lo + hi) >> 1; if (keys[mid] != ~0ull) lo = mid + 1; else hi = mid; }
    *out = lo;
}

static int g_delta_smem_max = 48 * 1024;

// K3M queries of more than VB_MS_LONG_TERMS terms are planned with a non-essential budget of VB_MS_BUDGET_LONG % of tau
// instead of the full MaxScore partition (cfg5 shard, 2..65-term queries: 561 ms per batch at 100 %, 154 at 92,
// 153-156 at 85, 160 at 70, 188 at 40)
#define VB_MS_LONG_TERMS 16u
#define VB_MS_BUDGET_LONG 85u

#define VB_K1F_MAX_B 8u
// CTAs per query of the single-pass scan: ONE wave of resident CTAs (the register file holds 5 x 256 threads per SM;
// round 2 launched 8 per SM = 1.6 waves, so the kernel lasted two CTA lifetimes: 52 us for 77 MB at cfg1); fewer for
// large k' so that the merge of G * k' keys stays short
static uint32_t vb_k1f_resident(int d_pad) {
    static int resident[5] = {0, 0, 0, 0, 0};
    const int nch = std::min(4, std::max(1, (d_pad / 8 + 31) / 32));
    if (!resident[nch]) {
        int v = 0;
        cudaError_t e = cudaErrorUnknown;
        switch (nch) {
            case 1: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, vb_dense_scan1_kernel<1>, VB_K1F_THREADS, 0); break;
            case 2: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, vb_dense_scan1_kernel<2>, VB_K1F_THREADS, 0); break;
            case 3: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, vb_dense_scan1_kernel<3>, VB_K1F_THREADS, 0); break;
            default: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, vb_dense_scan1_kernel<4>, VB_K1F_THREADS, 0); break;
        }
        resident[nch] = (e == cudaSuccess && v > 0) ? std::min(v, 8) : 2;
    }
    return (uint32_t)resident[nch];
}
static uint32_t vb_k1f_grid(int sm_count, uint32_t k, uint32_t B, int d_pad) {
    const uint32_t per_sm = std::min<uint32_t>(vb_k1f_resident(d_pad), k <= 64u ? 8u : (k <= 256u ? 4u : 2u));
    return std::max<uint32_t>(1u, (uint32_t)sm_count * per_sm / std::max<uint32_t>(B, 1u));
}

static unsigned grid_for(uint64_t n, unsigned block, unsigned max_blocks = 148u * 16u) {
    uint64_t g = (n + block - 1) / block;
    if (g < 1) g = 1;
    return (unsigned)std::min<uint64_t>(g, max_blocks);
}

// ------------------------------------------------------------------------------------------------
// lifecycle
// ------------------------------------------------------------------------------------------------
extern "C" int vb_abi_version(void) { return VB_ABI_VERSION; }
extern "C" const char* vb_last_error(void) { return g_err.c_str(); }

extern "C" int vb_create(int32_t dim, int32_t device, uint64_t capacity_hint, uint64_t row_base, vb_index** out) {
    if (!out) return vb_fail("vb_create: out is NULL");
    *out = nullptr;
    if (dim <= 0 || dim > 4096) return vb_fail("vb_create: dim %d out of range (1..4096)", dim);
    int n_dev = 0;
    cudaError_t e = cudaGetDeviceCount(&n_dev);
    if (e != cudaSuccess || n_dev == 0)
        return vb_fail("vb_create: no CUDA device (%s); this backend has no CPU fallback",
                       e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    if (device < 0 || device >= n_dev) return vb_fail("vb_create: device %d not in [0,%d)", device, n_dev);
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return vb_fail("vb_create: device %d is sm_%d%d; libvoitta_b200 is built for sm_100a only", device, prop.major, prop.minor);
    vb_index* h = new vb_index();
    h->dim = dim;
    h->d_pad = (int32_t)align_up((size_t)dim, 64);
    h->device = device;
    h->row_base = row_base;
    h->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&h->aux_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreate(&h->ev0s[0]) != cudaSuccess || cudaEventCreate(&h->ev1s[0]) != cudaSuccess ||
        cudaEventCreate(&h->ev0s[1]) != cudaSuccess || cudaEventCreate(&h->ev1s[1]) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_done[0], cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->ev_done[1], cudaEventDisableTiming) != cudaSuccess) {
        delete h;
        return vb_fail("vb_create: stream/event creation failed");
    }
    h->stream = h->own_stream;
    if (vb_gemm_configure() != 0) { delete h; return vb_fail("vb_create: tensor-core kernel configuration failed: %s", vb_gemm_last_error()); }
    if (cudaFuncSetAttribute(vb_mh_score_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)vb_mh_smem_bytes(VB_MS_MAX_TERMS)) != cudaSuccess) {
        delete h;
        return vb_fail("vb_create: cannot reserve shared memory for the long-query sparse kernel");
    }
    {
        const int want = std::min<int>((int)prop.sharedMemPerBlockOptin, 200 * 1024);
        if (cudaFuncSetAttribute(vb_sparse_delta_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, want) == cudaSuccess) g_delta_smem_max = want;
    }
    (void)capacity_hint;
    *out = h;
    return 0;
}

extern "C" void vb_destroy(vb_index* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    for (DevBuf* b : {&h->rows, &h->inv_norm, &h->scope_id, &h->created, &h->modified, &h->alive, &h->sp_indptr,
                      &h->sp_term, &h->sp_val, &h->post_row, &h->post_val, &h->heavy_vals, &h->args, &h->mask, &h->cand, &h->lists,
                      &h->offs, &h->plan, &h->out, &h->q_hat, &h->q_bf16, &h->q_scale, &h->tmp,
                      &h->ms_rec, &h->ms_q, &h->ms_units, &h->ms_counters, &h->mh_units, &h->term_tab,
                      &h->sel_rows, &h->sel_inv, &h->sel_ids, &h->sel_meta})
        dev_free(h, *b);
    for (HostBuf* b : {&h->h_args_s[0], &h->h_args_s[1], &h->h_out_s[0], &h->h_out_s[1], &h->h_stage, &h->h_sel[0], &h->h_sel[1]}) if (b->p) cudaFreeHost(b->p);
    for (auto ev : h->prof_events) cudaEventDestroy(ev);
    for (int i = 0; i < 2; ++i) { cudaEventDestroy(h->ev0s[i]); cudaEventDestroy(h->ev1s[i]); cudaEventDestroy(h->ev_done[i]); }
    if (h->ev_q) cudaEventDestroy(h->ev_q);
    cudaEventDestroy(h->ev_fork);
    cudaEventDestroy(h->ev_join);
    cudaStreamDestroy(h->aux_stream);
    if (h->sel_stream) { cudaStreamDestroy(h->sel_stream); cudaEventDestroy(h->ev_sel_fork); for (auto e : h->ev_sel) cudaEventDestroy(e); }
    cudaStreamDestroy(h->own_stream);
    delete h;
}

// Every option changes this index only; an index starts at the defaults in vb_index.
extern "C" int vb_set_option(vb_index* h, const char* key, int64_t value) {
    if (!h || !key) return vb_fail("vb_set_option: NULL argument");
    std::lock_guard<std::recursive_mutex> lk(h->mu);
    std::string k(key);
    if (k == "dense_path") h->opt_dense_path = value;
    else if (k == "seg_first") h->opt_seg_first = std::max<int64_t>(VB_ROWS_PER_BLOCK, (int64_t)align_up((size_t)value, VB_ROWS_PER_BLOCK));
    else if (k == "seg_ratio") h->opt_seg_ratio = value <= 0 ? 0 : std::max<int64_t>(2, value);   // 0 = auto
    else if (k == "safe_mode") h->opt_safe_mode = value;
    else if (k == "profile") h->opt_profile = value;
    else if (k == "slot") h->cur = value ? 1 : 0;                   // which of the two in-flight batches the staged calls address
    else if (k == "overlap") h->opt_overlap = value;               // 1: dense and sparse chains on two streams
    else if (k == "sparse_dense") { h->opt_sparse_dense = value; h->sparse_dirty = true; }   // 0: no dense columns for frequent terms
    else if (k == "sparse_ms") h->opt_sparse_ms = value;           // 0: K3 in every segment (no MaxScore kernel)
    else if (k == "ms_budget") h->opt_ms_budget = value;           // K3M non-essential budget in % of tau
    else if (k == "ms_chunk") h->opt_ms_chunk = value;             // K3M postings per work unit (0 auto)
    else if (k == "mh_budget") h->opt_mh_budget = value;           // K3H non-essential budget in % of tau
    else if (k == "sparse_mh") h->opt_sparse_mh = value;           // 0: long queries stay on K3
    else if (k == "k1f") h->opt_k1f = value;                       // 0: K1 in row segments even for single queries
    else if (k == "ms_staged") h->opt_ms_staged = value;           // K3M: posting stages (1) or row segments (0)
    else if (k == "delta_max") h->opt_delta_max = value;           // delta rows that trigger a merge (0 = max(16384, base/32))
    else if (k == "dense_compact_min_rows") h->opt_dense_compact_min_rows = value;
    else if (k == "dense_compact") h->opt_dense_compact = value;   // row selection threshold in % of the segment's rows (0 = off, -1 = auto)
    else if (k == "sel_reuse") h->opt_sel_reuse = value;           // 0: copy the passing rows every batch (A/B runs, tests)
    else if (k == "ms_max_terms") h->opt_ms_max_terms = value;     // K3M only for queries of at most this many terms
    else if (k == "sparse_prune_force") h->opt_sparse_prune_force = value;   // 1: prune in every non-direct segment (tests)
    else if (k == "sparse_prune") h->opt_sparse_prune = value;     // MaxScore budget in % of tau (0: score every term's postings)
    else if (k == "k2_tiled") h->opt_k2_tiled = value;             // 0: never use the query-tiled kernel (multi-pass resident kernel instead)
    else if (k == "k2_precision") h->opt_k2_precision = value;   // 0 auto, 1 bf16 query, 2 bf16x2 (hi+lo) query
    else if (k == "stream") {   // run on the caller's stream (e.g. torch's current stream); 0 = own stream
        h->stream = value ? reinterpret_cast<cudaStream_t>(static_cast<uintptr_t>(value)) : h->own_stream;
        h->sel_key.clear();     // a kept row selection is ordered on the old stream only: copy again on the new one
    }
    else return vb_fail("vb_set_option: unknown key '%s'", key);
    return 0;
}

extern "C" int vb_get_stats(vb_index* h, vb_stats* out) {
    if (!h || !out) return vb_fail("vb_get_stats: NULL argument");
    std::lock_guard<std::recursive_mutex> lk(h->mu);
    h->stats.n_rows = h->n_rows;
    h->stats.n_live = h->n_live;
    h->stats.nnz = h->nnz;
    h->stats.n_terms = h->terms_sorted.size();
    h->stats.device_bytes = h->device_bytes;
    h->stats.dim = (uint64_t)h->dim;
    h->stats.row_base = h->row_base;
    h->stats.delta_rows = h->sparse_dirty ? h->n_rows : h->n_rows - h->base_rows;
    *out = h->stats;
    return 0;
}

extern "C" int vb_get_timeline(vb_index* h, double* out, uint32_t cap, uint32_t* n) {
    if (!h || !n) return vb_fail("vb_get_timeline: NULL argument");
    std::lock_guard<std::recursive_mutex> lk(h->mu);
    const uint32_t have = (uint32_t)(h->timeline.size() / 3);
    *n = have;
    for (uint32_t i = 0; i < std::min(have, cap) && out; ++i)
        for (int j = 0; j < 3; ++j) out[3 * i + j] = h->timeline[3 * (size_t)i + j];
    return 0;
}

extern "C" int vb_sync(vb_index* h) {
    if (!h) return vb_fail("vb_sync: NULL index");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// incremental index maintenance (SURVEY §8 f-1).  The sorted inverted index ("base") is immutable between
// builds.  Upserts append to the forward CSR and become the DELTA, scored by K3D (sparse_delta.cuh); deletes
// clear alive bits.  Both adjust df_adj so that the IDF keeps using the exact live document frequencies
// (qdrant updates its df table on every upsert/delete).  The delta is merged (full rebuild) by vb_upsert once
// it passes delta_max rows — off the search path — or lazily by the next search after a bulk load.
// ------------------------------------------------------------------------------------------------
static uint64_t delta_max(const vb_index* h) {
    if (h->opt_delta_max > 0) return (uint64_t)h->opt_delta_max;
    return std::max<uint64_t>(16384, h->base_rows / 32);
}

static uint64_t live_df(const vb_index* h, uint32_t term, int64_t slot) {
    int64_t d = slot >= 0 ? (int64_t)(h->term_ptr[slot + 1] - h->term_ptr[slot]) : 0;
    if (!h->df_adj.empty()) {
        auto it = h->df_adj.find(term);
        if (it != h->df_adj.end()) d += it->second;
    }
    return d < 0 ? 0 : (uint64_t)d;
}

__global__ void vb_row_ranges_kernel(const int64_t* __restrict__ indptr, const uint32_t* __restrict__ rows, uint32_t n, int64_t* __restrict__ se) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { se[2 * i] = indptr[rows[i]]; se[2 * i + 1] = indptr[rows[i] + 1]; }
}
__global__ void vb_gather_terms_kernel(const uint32_t* __restrict__ sp_term, const int64_t* __restrict__ se, const int64_t* __restrict__ dst0,
                                       uint32_t n, uint32_t* __restrict__ out) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += warps)
        for (int64_t p = se[2 * i] + lane; p < se[2 * i + 1]; p += 32) out[dst0[i] + (p - se[2 * i])] = sp_term[p];
}

static int ensure_sparse_index(vb_index* h);

// after an append of rows [first, first + n): keep the index incremental if the delta stays small
static int after_append(vb_index* h, const uint32_t* host_terms, uint64_t n_terms) {
    const uint64_t delta = h->n_rows - h->base_rows;
    if (h->sparse_dirty || delta > 2 * delta_max(h)) { h->sparse_dirty = true; return 0; }   // bulk load: rebuild lazily
    for (uint64_t p = 0; p < n_terms; ++p) ++h->df_adj[host_terms[p]];
    if (delta >= delta_max(h)) { h->sparse_dirty = true; TRY(ensure_sparse_index(h)); }       // merge, off the search path
    return 0;
}

// ------------------------------------------------------------------------------------------------
// ingest
// ------------------------------------------------------------------------------------------------
static int reserve_rows(vb_index* h, uint64_t n_total, uint64_t nnz_total) {
    if (n_total + h->row_base > 0xffffffffull) return vb_fail("row ids exceed 32 bits");
    if (n_total > h->cap_rows) {
        uint64_t ncap = std::max<uint64_t>(n_total, h->cap_rows + h->cap_rows / 2);
        ncap = align_up(ncap, 1024);
        const uint64_t old = h->n_rows;
        TRY(dev_reserve(h, h->rows, ncap * h->d_pad * 2, true, old * h->d_pad * 2));
        TRY(dev_reserve(h, h->inv_norm, ncap * 4, true, old * 4));
        TRY(dev_reserve(h, h->scope_id, ncap * 4, true, old * 4));
        TRY(dev_reserve(h, h->created, ncap * 8, true, old * 8));
        TRY(dev_reserve(h, h->modified, ncap * 8, true, old * 8));
        const uint64_t old_words = (h->cap_rows + 31) / 32, new_words = (ncap + 31) / 32;
        TRY(dev_reserve(h, h->alive, new_words * 4, true, old_words * 4));
        CK(cudaMemsetAsync(h->alive.as<uint32_t>() + old_words, 0, (new_words - old_words) * 4, h->stream));
        TRY(dev_reserve(h, h->sp_indptr, (ncap + 1) * 8, true, h->sp_indptr.p ? (old + 1) * 8 : 0));
        if (old == 0) CK(cudaMemsetAsync(h->sp_indptr.p, 0, 8, h->stream));
        h->alive_host.resize(new_words, 0u);
        h->cap_rows = ncap;
    }
    if (nnz_total > h->cap_nnz) {
        uint64_t ncap = std::max<uint64_t>(nnz_total, h->cap_nnz + h->cap_nnz / 2);
        ncap = align_up(ncap, 4096);
        TRY(dev_reserve(h, h->sp_term, ncap * 4, true, h->nnz * 4));
        TRY(dev_reserve(h, h->sp_val, ncap * 4, true, h->nnz * 4));
        h->cap_nnz = ncap;
    }
    return 0;
}

static void mark_alive_host(vb_index* h, uint64_t first, uint64_t n) {
    for (uint64_t r = first; r < first + n; ++r) h->alive_host[r >> 5] |= 1u << (r & 31u);
}

extern "C" int vb_upsert(vb_index* h, uint64_t n, const float* dense, const int64_t* sp_indptr,
                         const uint32_t* sp_term, const float* sp_val, const uint32_t* scope_id,
                         const int64_t* created, const int64_t* modified, uint64_t* first_row) {
    if (!h) return vb_fail("vb_upsert: NULL index");
    if (n == 0) { if (first_row) *first_row = h->row_base + h->n_rows; return 0; }
    if (!dense) return vb_fail("vb_upsert: dense is NULL");
    std::lock_guard<std::recursive_mutex> lk(h->mu);
    CK(cudaSetDevice(h->device));
    const uint64_t add_nnz = sp_indptr ? (uint64_t)(sp_indptr[n] - sp_indptr[0]) : 0;
    if (sp_indptr) {
        if (!sp_term || !sp_val) return vb_fail("vb_upsert: sparse arrays missing");
        for (uint64_t r = 0; r < n; ++r) {
            if (sp_indptr[r + 1] < sp_indptr[r]) return vb_fail("vb_upsert: sp_indptr not monotone at row %llu", (unsigned long long)r);
            for (int64_t p = sp_indptr[r] + 1; p < sp_indptr[r + 1]; ++p)
                if (sp_term[p] <= sp_term[p - 1])
                    return vb_fail("vb_upsert: sparse indices of row %llu are not strictly ascending", (unsigned long long)r);
        }
    }
    TRY(reserve_rows(h, h->n_rows + n, h->nnz + add_nnz));
    const uint64_t first = h->n_rows;
    // dense rows: staged through pinned memory in chunks, converted on the device
    const uint64_t chunk_rows = std::max<uint64_t>(1, (32ull << 20) / ((uint64_t)h->dim * 4));
    TRY(host_reserve(h->h_stage, std::min<uint64_t>(n, chunk_rows) * h->dim * 4));
    TRY(dev_reserve(h, h->tmp, std::min<uint64_t>(n, chunk_rows) * h->dim * 4, false));
    for (uint64_t r0 = 0; r0 < n; r0 += chunk_rows) {
        const uint64_t m = std::min<uint64_t>(chunk_rows, n - r0);
        memcpy(h->h_stage.p, dense + r0 * h->dim, m * h->dim * 4);
        CK(cudaMemcpyAsync(h->tmp.p, h->h_stage.p, m * h->dim * 4, cudaMemcpyHostToDevice, h->stream));
        vb_ingest_f32_kernel<<<grid_for(m * 32, 256), 256, 0, h->stream>>>(
            h->tmp.as<float>(), (uint32_t)m, (uint32_t)h->dim, (uint32_t)h->d_pad,
            h->rows.as<__nv_bfloat16>() + (first + r0) * h->d_pad, h->inv_norm.as<float>() + first + r0);
        CKK("vb_ingest_f32_kernel");
        CK(cudaStreamSynchronize(h->stream));
    }
    // columns
    if (scope_id) CK(cudaMemcpyAsync(h->scope_id.as<uint32_t>() + first, scope_id, n * 4, cudaMemcpyHostToDevice, h->stream));
    else CK(cudaMemsetAsync(h->scope_id.as<uint32_t>() + first, 0, n * 4, h->stream));
    if (created) { CK(cudaMemcpyAsync(h->created.as<int64_t>() + first, created, n * 8, cudaMemcpyHostToDevice, h->stream)); h->any_ts_created = true; }
    else { vb_fill_i64_kernel<<<grid_for(n, 256), 256, 0, h->stream>>>(h->created.as<int64_t>() + first, n, INT64_MIN); CKK("fill"); }
    if (modified) { CK(cudaMemcpyAsync(h->modified.as<int64_t>() + first, modified, n * 8, cudaMemcpyHostToDevice, h->stream)); h->any_ts_modified = true; }
    else { vb_fill_i64_kernel<<<grid_for(n, 256), 256, 0, h->stream>>>(h->modified.as<int64_t>() + first, n, INT64_MIN); CKK("fill"); }
    // CSR append
    {
        std::vector<int64_t> ip(n);
        for (uint64_t r = 0; r < n; ++r)
            ip[r] = (int64_t)h->nnz + (sp_indptr ? (sp_indptr[r + 1] - sp_indptr[0]) : 0);
        CK(cudaMemcpyAsync(h->sp_indptr.as<int64_t>() + first + 1, ip.data(), n * 8, cudaMemcpyHostToDevice, h->stream));
        if (add_nnz) {
            CK(cudaMemcpyAsync(h->sp_term.as<uint32_t>() + h->nnz, sp_term + sp_indptr[0], add_nnz * 4, cudaMemcpyHostToDevice, h->stream));
            CK(cudaMemcpyAsync(h->sp_val.as<float>() + h->nnz, sp_val + sp_indptr[0], add_nnz * 4, cudaMemcpyHostToDevice, h->stream));
        }
        CK(cudaStreamSynchronize(h->stream));
    }
    mark_alive_host(h, first, n);
    vb_set_alive_kernel<<<grid_for(n, 256), 256, 0, h->stream>>>(h->alive.as<uint32_t>(), first, n);
    CKK("vb_set_alive_kernel");
    CK(cudaStreamSynchronize(h->stream));
    h->n_rows += n;
    h->n_live += n;
    h->nnz += add_nnz;
    ++h->write_gen;
    if (first_row) *first_row = h->row_base + first;
    TRY(after_append(h, sp_indptr ? sp_term + sp_indptr[0] : nullptr, add_nnz));
    return 0;
}

extern "C" int vb_upsert_dev(vb_index* h, uint64_t n, const void* rows_bf16, const int64_t* sp_indptr,
                             const uint32_t* sp_term, const float* sp_val, const uint32_t* scope_id,
                             const int64_t* created, const int64_t* modified, uint64_t* first_row) {
    if (!h) return vb_fail("vb_upsert_dev: NULL index");
    if (n == 0) { if (first_row) *first_row = h->row_base + h->n_rows; return 0; }
    if (!rows_bf16) return vb_fail("vb_upsert_dev: rows is NULL");
    std::lock_guard<std::recursive_mutex> lk(h->mu);
    CK(cudaSetDevice(h->device));
    uint64_t add_nnz = 0;
    int64_t ip0 = 0;
    if (sp_indptr) {
        int64_t ends[2];
        CK(cudaMemcpy(&ends[0], sp_indptr, 8, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(&ends[1], sp_indptr + n, 8, cudaMemcpyDeviceToHost));
        ip0 = ends[0];
        add_nnz = (uint64_t)(ends[1] - ends[0]);
    }
    TRY(reserve_rows(h, h->n_rows + n, h->nnz + add_nnz));
    const uint64_t first = h->n_rows;
    vb_ingest_bf16_kernel<<<grid_for(n * 32, 256), 256, 0, h->stream>>>(
        reinterpret_cast<const __nv_bfloat16*>(rows_bf16), (uint32_t)n, (uint32_t)h->dim, (uint32_t)h->d_pad,
        h->rows.as<__nv_bfloat16>() + first * h->d_pad, h->inv_norm.as<float>() + first);
    CKK("vb_ingest_bf16_kernel");
    if (scope_id) CK(cudaMemcpyAsync(h->scope_id.as<uint32_t>() + first, scope_id, n * 4, cudaMemcpyDeviceToDevice, h->stream));
    else CK(cudaMemsetAsync(h->scope_id.as<uint32_t>() + first, 0, n * 4, h->stream));
    if (created) { CK(cudaMemcpyAsync(h->created.as<int64_t>() + first, created, n * 8, cudaMemcpyDeviceToDevice, h->stream)); h->any_ts_created = true; }
    else { vb_fill_i64_kernel<<<grid_for(n, 256), 256, 0, h->stream>>>(h->created.as<int64_t>() + first, n, INT64_MIN); CKK("fill"); }
    if (modified) { CK(cudaMemcpyAsync(h->modified.as<int64_t>() + first, modified, n * 8, cudaMemcpyDeviceToDevice, h->stream)); h->any_ts_modified = true; }
    else { vb_fill_i64_kernel<<<grid_for(n, 256), 256, 0, h->stream>>>(h->modified.as<int64_t>() + first, n, INT64_MIN); CKK("fill"); }
    if (sp_indptr) {
        vb_offset_i64_kernel<<<grid_for(n, 256), 256, 0, h->stream>>>(sp_indptr + 1, h->sp_indptr.as<int64_t>() + first + 1, n, (int64_t)h->nnz - ip0);
        CKK("vb_offset_i64_kernel");
        if (add_nnz) {
            CK(cudaMemcpyAsync(h->sp_term.as<uint32_t>() + h->nnz, sp_term + ip0, add_nnz * 4, cudaMemcpyDeviceToDevice, h->stream));
            CK(cudaMemcpyAsync(h->sp_val.as<float>() + h->nnz, sp_val + ip0, add_nnz * 4, cudaMemcpyDeviceToDevice, h->stream));
        }
    } else {
        vb_fill_i64_kernel<<<grid_for(n, 256), 256, 0, h->stream>>>(h->sp_indptr.as<int64_t>() + first + 1, n, (int64_t)h->nnz);
        CKK("fill");
    }
    mark_alive_host(h, first, n);
    vb_set_alive_kernel<<<grid_for(n, 256), 256, 0, h->stream>>>(h->alive.as<uint32_t>(), first, n);
    CKK("vb_set_alive_kernel");
    CK(cudaStreamSynchronize(h->stream));
    h->n_rows += n;
    h->n_live += n;
    h->nnz += add_nnz;
    ++h->write_gen;
    if (first_row) *first_row = h->row_base + first;
    if (!h->sparse_dirty && h->n_rows - h->base_rows <= 2 * delta_max(h)) {
        std::vector<uint32_t> terms(add_nnz);                   // small append: its terms feed the df table
        if (add_nnz) CK(cudaMemcpy(terms.data(), h->sp_term.as<uint32_t>() + (h->nnz - add_nnz), add_nnz * 4, cudaMemcpyDeviceToHost));
        TRY(after_append(h, terms.data(), add_nnz));
    } else {
        h->sparse_dirty = true;
    }
    return 0;
}

extern "C" int vb_delete_rows(vb_index* h, uint64_t n, const uint64_t* rows) {
    if (!h) return vb_fail("vb_delete_rows: NULL index");
    if (n == 0) return 0;
    if (!rows) return vb_fail("vb_delete_rows: rows is NULL");
    std::lock_guard<std::recursive_mutex> lk(h->mu);
    CK(cudaSetDevice(h->device));
    uint64_t killed = 0;
    std::vector<uint32_t> touched, dead;
    for (uint64_t i = 0; i < n; ++i) {
        if (rows[i] < h->row_base || rows[i] - h->row_base >= h->n_rows)
            return vb_fail("vb_delete_rows: row %llu out of range", (unsigned long long)rows[i]);
        const uint64_t r = rows[i] - h->row_base;
        uint32_t& w = h->alive_host[r >> 5];
        if (w & (1u << (r & 31u))) { w &= ~(1u << (r & 31u)); ++killed; touched.push_back((uint32_t)(r >> 5)); dead.push_back((uint32_t)r); }
    }
    if (!killed) return 0;
    ++h->write_gen;                        // before the upload: a failed one must not leave a kept row selection valid
    // one ranged upload of the touched bitmap words (a folder delete touches tens of thousands of them)
    const uint32_t w_lo = *std::min_element(touched.begin(), touched.end()), w_hi = *std::max_element(touched.begin(), touched.end());
    CK(cudaMemcpyAsync(h->alive.as<uint32_t>() + w_lo, &h->alive_host[w_lo], (size_t)(w_hi - w_lo + 1) * 4, cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    h->n_live -= killed;
    if (h->sparse_dirty) return 0;
    // Incremental path: the postings of the dead rows stay in the index (the alive bits mask them); only the live
    // document frequencies change.  Large deletes, or too many dead postings, fall back to a rebuild.
    h->dead_since_build += killed;
    if (killed > std::max<uint64_t>(4096, h->n_live / 16) || h->dead_since_build * 4 > std::max<uint64_t>(h->base_rows, 1)) {
        h->sparse_dirty = true;
        return 0;
    }
    if (h->nnz == 0) return 0;
    {
        const uint32_t m = (uint32_t)dead.size();
        DevBuf d_rows, d_se, d_dst, d_out;
        auto cleanup = [&]() { dev_free(h, d_rows); dev_free(h, d_se); dev_free(h, d_dst); dev_free(h, d_out); };
        int rc = dev_reserve(h, d_rows, (size_t)m * 4, false);
        if (!rc) rc = dev_reserve(h, d_se, (size_t)m * 16, false);
        if (!rc) rc = dev_reserve(h, d_dst, (size_t)m * 8, false);
        if (rc) { cleanup(); return rc; }
        std::vector<int64_t> se(2 * (size_t)m), dst(m);
        cudaError_t e = cudaMemcpyAsync(d_rows.p, dead.data(), (size_t)m * 4, cudaMemcpyHostToDevice, h->stream);
        if (e == cudaSuccess) {
            vb_row_ranges_kernel<<<(m + 255) / 256, 256, 0, h->stream>>>(h->sp_indptr.as<int64_t>(), d_rows.as<uint32_t>(), m, d_se.as<int64_t>());
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaMemcpyAsync(se.data(), d_se.p, (size_t)m * 16, cudaMemcpyDeviceToHost, h->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
        int64_t total = 0;
        for (uint32_t i = 0; i < m; ++i) { dst[i] = total; total += se[2 * i + 1] - se[2 * i]; }
        std::vector<uint32_t> terms((size_t)total);
        if (e == cudaSuccess && total > 0) {
            rc = dev_reserve(h, d_out, (size_t)total * 4, false);
            if (rc) { cleanup(); return rc; }
            e = cudaMemcpyAsync(d_dst.p, dst.data(), (size_t)m * 8, cudaMemcpyHostToDevice, h->stream);
            if (e == cudaSuccess) {
                vb_gather_terms_kernel<<<grid_for((uint64_t)m * 32, 256), 256, 0, h->stream>>>(
                    h->sp_term.as<uint32_t>(), d_se.as<int64_t>(), d_dst.as<int64_t>(), m, d_out.as<uint32_t>());
                e = cudaGetLastError();
            }
            if (e == cudaSuccess) e = cudaMemcpyAsync(terms.data(), d_out.p, (size_t)total * 4, cudaMemcpyDeviceToHost, h->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
        }
        cleanup();
        if (e != cudaSuccess) { h->sparse_dirty = true; return vb_fail("vb_delete_rows: df update failed: %s", cudaGetErrorString(e)); }
        for (uint32_t t : terms) --h->df_adj[t];
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------
// inverted index build (device; CUB radix sort of (term,row) keys)
// ------------------------------------------------------------------------------------------------
static int ensure_sparse_index(vb_index* h) {
    if (!h->sparse_dirty) return 0;
    h->terms_sorted.clear();
    h->term_ptr.assign(1, 0);
    h->term_maxval.clear();
    h->heavy_of_slot.clear();
    h->tab_off_of_slot.clear();
    h->tab_shift_of_slot.clear();
    h->n_heavy = 0;
    h->sparse_nonneg = false;
    h->nnz_live = 0;
    h->df_adj.clear();
    h->dead_since_build = 0;
    if (h->nnz == 0) { h->base_rows = h->n_rows; h->sparse_dirty = false; return 0; }
    const uint64_t nnz = h->nnz;
    if (nnz >= (1ull << 31)) return vb_fail("sparse index: %llu postings exceed the 2^31 limit of one shard", (unsigned long long)nnz);
    DevBuf keys_in, keys_out, vals_out, cub_tmp, misc;
    int rc = 0;
    auto cleanup = [&]() { dev_free(h, keys_in); dev_free(h, keys_out); dev_free(h, vals_out); dev_free(h, cub_tmp); dev_free(h, misc); };
#define TRYC(expr) do { rc = (expr); if (rc) { cleanup(); return rc; } } while (0)
#define CKC(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) { cleanup(); return vb_fail("%s failed: %s", #call, cudaGetErrorString(e__)); } } while (0)
    TRYC(dev_reserve(h, keys_in, nnz * 8, false));
    TRYC(dev_reserve(h, keys_out, nnz * 8, false));
    TRYC(dev_reserve(h, vals_out, nnz * 4, false));
    TRYC(dev_reserve(h, misc, 64, false));
    vb_posting_keys_kernel<<<grid_for(h->n_rows * 32, 256), 256, 0, h->stream>>>(
        h->sp_indptr.as<int64_t>(), h->sp_term.as<uint32_t>(), h->alive.as<uint32_t>(), (uint32_t)h->n_rows, keys_in.as<uint64_t>());
    CKC(cudaGetLastError());
    size_t tmp_bytes = 0;
    CKC(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, keys_in.as<uint64_t>(), keys_out.as<uint64_t>(),
                                        h->sp_val.as<float>(), vals_out.as<float>(), (int)nnz, 0, 64, h->stream));
    TRYC(dev_reserve(h, cub_tmp, tmp_bytes, false));
    CKC(cub::DeviceRadixSort::SortPairs(cub_tmp.p, tmp_bytes, keys_in.as<uint64_t>(), keys_out.as<uint64_t>(),
                                        h->sp_val.as<float>(), vals_out.as<float>(), (int)nnz, 0, 64, h->stream));
    vb_find_tail_kernel<<<1, 1, 0, h->stream>>>(keys_out.as<uint64_t>(), nnz, misc.as<uint64_t>());
    CKC(cudaGetLastError());
    uint64_t live = 0;
    CKC(cudaMemcpyAsync(&live, misc.p, 8, cudaMemcpyDeviceToHost, h->stream));
    CKC(cudaStreamSynchronize(h->stream));
    h->nnz_live = live;
    if (live == 0) { cleanup(); h->base_rows = h->n_rows; h->sparse_dirty = false; return 0; }
    TRYC(dev_reserve(h, h->post_row, live * 4, false));
    TRYC(dev_reserve(h, h->post_val, live * 4, false));
    // keys_in is free now: reuse it for post_term (u32), unique terms (u32), run lengths (u32)
    uint32_t* post_term = keys_in.as<uint32_t>();
    vb_posting_split_kernel<<<grid_for(live, 256), 256, 0, h->stream>>>(keys_out.as<uint64_t>(), live, h->post_row.as<uint32_t>(), post_term);
    CKC(cudaGetLastError());
    CKC(cudaMemcpyAsync(h->post_val.p, vals_out.p, live * 4, cudaMemcpyDeviceToDevice, h->stream));
    // run-length encode the sorted terms -> distinct terms + df
    DevBuf uniq, runs, ptrs;
    auto cleanup2 = [&]() { dev_free(h, uniq); dev_free(h, runs); dev_free(h, ptrs); cleanup(); };
#define CKC2(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) { cleanup2(); return vb_fail("%s failed: %s", #call, cudaGetErrorString(e__)); } } while (0)
    rc = dev_reserve(h, uniq, live * 4, false); if (rc) { cleanup2(); return rc; }
    rc = dev_reserve(h, runs, live * 8, false); if (rc) { cleanup2(); return rc; }
    size_t tb = 0;
    CKC2(cub::DeviceRunLengthEncode::Encode(nullptr, tb, post_term, uniq.as<uint32_t>(), runs.as<uint64_t>(), misc.as<uint32_t>() + 4, (int)live, h->stream));
    rc = dev_reserve(h, cub_tmp, tb, false); if (rc) { cleanup2(); return rc; }
    CKC2(cub::DeviceRunLengthEncode::Encode(cub_tmp.p, tb, post_term, uniq.as<uint32_t>(), runs.as<uint64_t>(), misc.as<uint32_t>() + 4, (int)live, h->stream));
    uint32_t T = 0;
    CKC2(cudaMemcpyAsync(&T, misc.as<uint32_t>() + 4, 4, cudaMemcpyDeviceToHost, h->stream));
    CKC2(cudaStreamSynchronize(h->stream));
    rc = dev_reserve(h, ptrs, ((size_t)T + 1) * 8, false); if (rc) { cleanup2(); return rc; }
    tb = 0;
    CKC2(cub::DeviceScan::ExclusiveSum(nullptr, tb, runs.as<uint64_t>(), ptrs.as<uint64_t>(), (int)T, h->stream));
    rc = dev_reserve(h, cub_tmp, tb, false); if (rc) { cleanup2(); return rc; }
    CKC2(cub::DeviceScan::ExclusiveSum(cub_tmp.p, tb, runs.as<uint64_t>(), ptrs.as<uint64_t>(), (int)T, h->stream));
    h->terms_sorted.resize(T);
    h->term_ptr.resize((size_t)T + 1);
    h->term_maxval.resize(T);
    // per-term largest posting value (segmented max over the sorted postings); `runs` is free now
    CKC2(cudaMemcpyAsync(ptrs.as<uint64_t>() + T, &live, 8, cudaMemcpyHostToDevice, h->stream));
    tb = 0;
    CKC2(cub::DeviceSegmentedReduce::Max(nullptr, tb, h->post_val.as<float>(), runs.as<float>(), (int)T,
                                         ptrs.as<uint64_t>(), ptrs.as<uint64_t>() + 1, h->stream));
    rc = dev_reserve(h, cub_tmp, tb, false); if (rc) { cleanup2(); return rc; }
    CKC2(cub::DeviceSegmentedReduce::Max(cub_tmp.p, tb, h->post_val.as<float>(), runs.as<float>(), (int)T,
                                         ptrs.as<uint64_t>(), ptrs.as<uint64_t>() + 1, h->stream));
    CKC2(cudaMemcpyAsync(h->term_maxval.data(), runs.p, (size_t)T * 4, cudaMemcpyDeviceToHost, h->stream));
    CKC2(cudaMemcpyAsync(h->terms_sorted.data(), uniq.p, (size_t)T * 4, cudaMemcpyDeviceToHost, h->stream));
    CKC2(cudaMemcpyAsync(h->term_ptr.data(), ptrs.p, (size_t)T * 8, cudaMemcpyDeviceToHost, h->stream));
    CKC2(cudaStreamSynchronize(h->stream));
    h->term_ptr[T] = live;
    // smallest posting value: the dense-column path below and its error bound need products >= 0
    {
        tb = 0;
        CKC2(cub::DeviceReduce::Min(nullptr, tb, h->post_val.as<float>(), runs.as<float>(), (int)live, h->stream));
        rc = dev_reserve(h, cub_tmp, tb, false); if (rc) { cleanup2(); return rc; }
        CKC2(cub::DeviceReduce::Min(cub_tmp.p, tb, h->post_val.as<float>(), runs.as<float>(), (int)live, h->stream));
        float mn = -1.0f;
        CKC2(cudaMemcpyAsync(&mn, runs.p, 4, cudaMemcpyDeviceToHost, h->stream));
        CKC2(cudaStreamSynchronize(h->stream));
        h->sparse_nonneg = mn >= 0.0f;
    }
    // Dense columns for the most frequent terms (df >= 1/8 of the live rows, at most 64 of them): such a
    // term's postings touch most rows of every block, so the scoring kernel reads its value per row from a
    // column (coalesced, no shared-memory scatter) instead of walking its posting list once per query.
    h->heavy_of_slot.assign(T, -1);
    if (h->opt_sparse_dense && h->sparse_nonneg && h->n_live >= 4096) {
        std::vector<std::pair<uint64_t, uint32_t>> cand;
        for (uint32_t sl = 0; sl < T; ++sl) {
            const uint64_t df = h->term_ptr[sl + 1] - h->term_ptr[sl];
            if (df * 8 >= h->n_live) cand.emplace_back(df, sl);
        }
        std::sort(cand.begin(), cand.end(), [](const auto& x, const auto& y) { return x.first > y.first; });
        if (cand.size() > 64) cand.resize(64);
        h->n_heavy = (uint32_t)cand.size();
        h->heavy_stride = (uint32_t)align_up((size_t)h->n_rows + 2, 64);
        if (h->n_heavy) {
            rc = dev_reserve(h, h->heavy_vals, (size_t)h->n_heavy * h->heavy_stride * 4, false); if (rc) { cleanup2(); return rc; }
            CKC2(cudaMemsetAsync(h->heavy_vals.p, 0xff, (size_t)h->n_heavy * h->heavy_stride * 4, h->stream));   // all NaN
            for (uint32_t k = 0; k < h->n_heavy; ++k) {
                const uint32_t sl = cand[k].second;
                h->heavy_of_slot[sl] = (int32_t)k;
                vb_heavy_fill_kernel<<<grid_for(cand[k].first, 256), 256, 0, h->stream>>>(
                    h->post_row.as<uint32_t>(), h->post_val.as<float>(), h->term_ptr[sl], h->term_ptr[sl + 1],
                    h->heavy_vals.as<float>() + (size_t)k * h->heavy_stride);
                CKC2(cudaGetLastError());
            }
            CKC2(cudaStreamSynchronize(h->stream));
        }
    }
    // Bucket tables for K3M's term lookups: per term with >= 32 postings, tab[b] = first posting whose row >=
    // b << shift, buckets sized for ~4 postings (frequent terms: 4096-row buckets, used only to find segment
    // bounds — their lookups read the dense column).  ~1 byte per posting on top of the 8-byte postings.
    h->tab_off_of_slot.assign(T, VB_MS_NO_TAB);
    h->tab_shift_of_slot.assign(T, 0);
    {
        std::vector<VbTabTerm> tt;
        uint64_t total = 0;
        const uint64_t nr = h->n_rows;
        for (uint32_t sl = 0; sl < T; ++sl) {
            const uint64_t df = h->term_ptr[sl + 1] - h->term_ptr[sl];
            if (df < 32) continue;
            uint32_t shift = 0;
            while (shift < 31u && (df << (shift + 1)) <= nr * 4) ++shift;       // 2^shift ~ 4 * rows / df
            if (h->heavy_of_slot[sl] >= 0) shift = std::max(shift, 12u);
            const uint64_t nb = (nr >> shift) + 2;
            if (total + nb >= 0xffffffffull) break;                              // table offsets are 32-bit: the rest stay without
            h->tab_off_of_slot[sl] = (uint32_t)total;
            h->tab_shift_of_slot[sl] = (uint8_t)shift;
            tt.push_back(VbTabTerm{(uint32_t)h->term_ptr[sl], (uint32_t)h->term_ptr[sl + 1], (uint32_t)total, shift});
            total += nb;
        }
        if (!tt.empty()) {
            DevBuf d_tt;
            rc = dev_reserve(h, h->term_tab, total * 4, false); if (rc) { cleanup2(); return rc; }
            rc = dev_reserve(h, d_tt, tt.size() * sizeof(VbTabTerm), false); if (rc) { cleanup2(); return rc; }
            cudaError_t e = cudaMemcpyAsync(d_tt.p, tt.data(), tt.size() * sizeof(VbTabTerm), cudaMemcpyHostToDevice, h->stream);
            if (e == cudaSuccess) {
                vb_ms_tab_fill_kernel<<<grid_for(total, 256, 148u * 32u), 256, 0, h->stream>>>(
                    h->post_row.as<uint32_t>(), d_tt.as<VbTabTerm>(), (uint32_t)tt.size(), total, h->term_tab.as<uint32_t>());
                e = cudaGetLastError();
            }
            if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
            dev_free(h, d_tt);
            if (e != cudaSuccess) { cleanup2(); return vb_fail("bucket table build failed: %s", cudaGetErrorString(e)); }
        }
    }
    cleanup2();
    h->base_rows = h->n_rows;
    ++h->stats.index_builds;
    h->sparse_dirty = false;
    return 0;
#undef TRYC
#undef CKC
#undef CKC2
}

// slot of a term in the directory, or -1
static int64_t term_slot(const vb_index* h, uint32_t term) {
    auto it = std::lower_bound(h->terms_sorted.begin(), h->terms_sorted.end(), term);
    if (it == h->terms_sorted.end() || *it != term) return -1;
    return it - h->terms_sorted.begin();
}

extern "C" int vb_optimize(vb_index* h) {
    if (!h) return vb_fail("vb_optimize: NULL index");
    std::lock_guard<std::recursive_mutex> lk(h->mu);
    CK(cudaSetDevice(h->device));
    if (h->n_rows != h->base_rows || h->dead_since_build) h->sparse_dirty = true;
    return ensure_sparse_index(h);
}

extern "C" int vb_term_stats(vb_index* h, uint32_t n_terms, const uint32_t* terms, uint64_t* df, uint64_t* n_live) {
    if (!h) return vb_fail("vb_term_stats: NULL index");
    std::lock_guard<std::recursive_mutex> lk(h->mu);
    CK(cudaSetDevice(h->device));
    TRY(ensure_sparse_index(h));
    for (uint32_t i = 0; i < n_terms; ++i) {
        df[i] = live_df(h, terms[i], term_slot(h, terms[i]));
    }
    if (n_live) *n_live = h->n_live;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// search
// ------------------------------------------------------------------------------------------------
struct Arena {
    size_t off = 0;
    size_t take(size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return o; }
};


enum { PH_MASK = 0, PH_DENSE = 1, PH_SPARSE = 2, PH_SELECT = 3, PH_FUSE = 4, PH_N = 5, PH_BIG = 8 /* flag: largest segment */ };

static int prof_begin(vb_index* h, int phase, cudaStream_t st = nullptr) {
    if (!h->opt_profile) return -1;
    const size_t i = h->prof_phase.size();
    while (h->prof_events.size() < 2 * (i + 1)) {
        cudaEvent_t e;
        cudaEventCreate(&e);
        h->prof_events.push_back(e);
    }
    h->prof_phase.push_back(phase);
    cudaEventRecord(h->prof_events[2 * i], st ? st : h->stream);
    return (int)i;
}
static void prof_end(vb_index* h, int idx = -2, cudaStream_t st = nullptr) {
    if (!h->opt_profile) return;
    if (idx == -2) idx = (int)h->prof_phase.size() - 1;
    if (idx < 0) return;
    cudaEventRecord(h->prof_events[2 * (size_t)idx + 1], st ? st : h->stream);
}
// call after the stream has been synchronised
static void prof_collect(vb_index* h) {
    double acc[PH_N] = {0, 0, 0, 0, 0};
    h->stats.last_dense_big_ms = h->stats.last_sparse_big_ms = 0.0;
    h->timeline.clear();
    for (size_t i = 0; i < h->prof_phase.size(); ++i) {
        float ms = 0.f, t0 = 0.f;
        cudaEventElapsedTime(&ms, h->prof_events[2 * i], h->prof_events[2 * i + 1]);
        if (cudaEventElapsedTime(&t0, h->ev0s[h->cur], h->prof_events[2 * i]) == cudaSuccess) {
            h->timeline.push_back((double)h->prof_phase[i]);
            h->timeline.push_back((double)t0);
            h->timeline.push_back((double)t0 + ms);
        }
        const int ph = h->prof_phase[i] & 7;
        acc[ph] += ms;
        if (h->prof_phase[i] & PH_BIG) (ph == PH_DENSE ? h->stats.last_dense_big_ms : h->stats.last_sparse_big_ms) = ms;
    }
    h->prof_phase.clear();
    h->stats.last_mask_ms = acc[PH_MASK];
    h->stats.last_dense_ms = acc[PH_DENSE];
    h->stats.last_sparse_ms = acc[PH_SPARSE];
    h->stats.last_select_ms = acc[PH_SELECT];
    h->stats.last_fuse_ms = acc[PH_FUSE];
}

static int validate_batch(const vb_index* h, const vb_query_batch* q) {
    if (!q) return vb_fail("query batch is NULL");
    if (q->n_queries == 0) return vb_fail("empty query batch");
    if (!q->dense && !h->q_dev) return vb_fail("dense queries are NULL");
    if (q->limit == 0) return vb_fail("limit must be > 0");
    if (q->kprime < q->limit) return vb_fail("kprime (%u) < limit (%u)", q->kprime, q->limit);
    if (q->kprime > VB_MAX_KPRIME) return vb_fail("kprime %u exceeds VB_MAX_KPRIME (%d)", q->kprime, VB_MAX_KPRIME);
    if (q->fusion < 0 || q->fusion > 2) return vb_fail("unknown fusion mode %d", q->fusion);
    if (q->n_filters && !q->filters) return vb_fail("filters is NULL");
    if (q->filter_of)
        for (uint32_t i = 0; i < q->n_queries; ++i)
            if (q->filter_of[i] >= (int32_t)q->n_filters) return vb_fail("filter_of[%u] out of range", i);
    (void)h;
    return 0;
}

// Filter content as the mask kernel sees it: scope words past scope_words read as 0, the range only counts with a field.
struct FilterKey {
    const vb_filter* f;
    uint32_t words;            // scope words up to the last non-zero one
};
struct FilterKeyHash {
    size_t operator()(const FilterKey& k) const {
        uint64_t x = 0x9E3779B97F4A7C15ull ^ (uint64_t)(k.f->scope_bits != nullptr) ^ ((uint64_t)(uint32_t)k.f->ts_field << 1);
        auto mix = [&](uint64_t v) { x = (x ^ v) * 0xBF58476D1CE4E5B9ull; x ^= x >> 31; };
        if (k.f->ts_field != VB_TS_NONE) { mix((uint64_t)k.f->ts_lo); mix((uint64_t)k.f->ts_hi); }
        for (uint32_t w = 0; w < k.words; ++w) mix(k.f->scope_bits[w]);
        return (size_t)x;
    }
};
struct FilterKeyEq {
    bool operator()(const FilterKey& a, const FilterKey& b) const {
        const vb_filter &x = *a.f, &y = *b.f;
        if (x.ts_field != y.ts_field || (x.scope_bits == nullptr) != (y.scope_bits == nullptr) || a.words != b.words) return false;
        if (x.ts_field != VB_TS_NONE && (x.ts_lo != y.ts_lo || x.ts_hi != y.ts_hi)) return false;
        return a.words == 0 || memcmp(x.scope_bits, y.scope_bits, (size_t)a.words * 4) == 0;
    }
};
static FilterKey filter_key(const vb_filter* f) {
    uint32_t w = f->scope_bits ? f->scope_words : 0u;
    while (w > 0 && f->scope_bits[w - 1] == 0u) --w;
    return FilterKey{f, w};
}

// Mask mode 3 tables for query tiles of `tile` queries: the distinct filters each tile uses (<= tile <= 256) and each
// query's index into its tile's list.  The tiles of one launch (`group` queries) share the launch's list when it holds
// at most 256 filters (VB_FTAB_SHARED).  Laid out at `off` of the staged argument block (host hp, device dp).
static size_t filter_tiles_bytes(uint32_t B, uint32_t tile) {
    const size_t tiles = (B + tile - 1) / tile;
    return (size_t)B * 4 + align_up(tiles * 4, 16) + tiles * VB_GEMM_MAX_FILTERS * 4;
}
static VbFilterTiles build_filter_tiles(const std::vector<int32_t>& mask_of, uint32_t n_filters, uint32_t tile, uint32_t group,
                                        unsigned char* hp, const unsigned char* dp, size_t off) {
    const uint32_t B = (uint32_t)mask_of.size(), tiles = (B + tile - 1) / tile;
    int32_t* loc = reinterpret_cast<int32_t*>(hp + off);
    uint32_t* cnt = reinterpret_cast<uint32_t*>(hp + off + (size_t)B * 4);
    int32_t* ids = reinterpret_cast<int32_t*>(hp + off + (size_t)B * 4 + align_up((size_t)tiles * 4, 16));
    std::vector<int32_t> local(n_filters, -1);                 // batch-wide id -> index in the current list
    std::vector<int32_t> list;
    // queries [q0, q1) on one list: tiles [t0, t1) get it (flag set: the tiles of a launch share it)
    auto make_list = [&](uint32_t q0, uint32_t q1) {
        list.clear();
        for (uint32_t i = q0; i < q1; ++i) {
            const int32_t f = mask_of[i];
            if (f >= 0 && local[f] < 0) { local[f] = (int32_t)list.size(); list.push_back(f); }
            loc[i] = f >= 0 ? local[f] : -1;
        }
        for (int32_t f : list) local[f] = -1;
    };
    for (uint32_t g0 = 0; g0 < B; g0 += group) {
        const uint32_t g1 = std::min(B, g0 + group);
        make_list(g0, g1);
        const bool shared = list.size() <= VB_GEMM_MAX_FILTERS;
        for (uint32_t t = g0 / tile; t < (g1 + tile - 1) / tile; ++t) {
            if (!shared) make_list(t * tile, std::min(B, (t + 1) * tile));
            std::copy(list.begin(), list.end(), ids + (size_t)t * VB_GEMM_MAX_FILTERS);
            cnt[t] = (uint32_t)list.size() | (shared ? VB_FTAB_SHARED : 0u);
        }
    }
    VbFilterTiles ft;
    ft.loc = reinterpret_cast<const int32_t*>(dp + off);
    ft.n = reinterpret_cast<const uint32_t*>(dp + off + (size_t)B * 4);
    ft.ids = reinterpret_cast<const int32_t*>(dp + off + (size_t)B * 4 + align_up((size_t)tiles * 4, 16));
    ft.tile = tile;
    return ft;
}

// Upload the batch, evaluate the filters, initialise the candidate lists.
static int prepare_batch(vb_index* h, const vb_query_batch* q, Batch& b, bool need_corpus) {
    b = Batch();
    b.need_corpus = need_corpus;
    b.w_sparse = q->sparse_weight;
    b.B = q->n_queries;
    b.k = q->kprime;
    b.limit = q->limit;
    b.n_lists = 2 * b.B;
    b.mode.assign(b.B, 0);
    const bool sparse_enabled = q->fusion != VB_FUSE_DENSE_ONLY && q->sp_indptr != nullptr;

    // ---- sparse queries: sort by term id, resolve posting ranges, apply IDF ----
    std::vector<int64_t> indptr(b.B + 1, 0);
    std::vector<double> weight, qub;
    std::vector<uint32_t> qlo, qhi, qterm, qplo, qphi, slotq, oldq, dirq;
    std::vector<int32_t> qhidx;
    std::vector<uint8_t> qrelaxed(b.B, 0), qms(b.B, 0), qshift;
    std::vector<uint32_t> qtab;
    if (sparse_enabled) {
        if (need_corpus) TRY(ensure_sparse_index(h));
        std::vector<std::pair<uint32_t, double>> tw;
        for (uint32_t i = 0; i < b.B; ++i) {
            const int64_t lo = q->sp_indptr[i], hi = q->sp_indptr[i + 1];
            if (hi < lo) return vb_fail("sp_indptr not monotone at query %u", i);
            if (hi - lo > VB_MAX_QUERY_TERMS) return vb_fail("query %u has %lld terms (max %d)", i, (long long)(hi - lo), VB_MAX_QUERY_TERMS);
            tw.clear();
            for (int64_t p = lo; p < hi; ++p) tw.emplace_back(q->sp_term[p], q->sp_weight[p]);
            std::sort(tw.begin(), tw.end(), [](const auto& x, const auto& y) { return x.first < y.first; });
            for (size_t t = 1; t < tw.size(); ++t)
                if (tw[t].first == tw[t - 1].first) return vb_fail("query %u repeats sparse index %u", i, tw[t].first);
            const size_t q_first = weight.size();
            bool all_pos = true;                                // dense columns need every product >= 0 (error bound)
            for (auto& pr : tw) {
                uint64_t plo = 0, phi = 0;
                int64_t slot = -1;
                if (need_corpus) {
                    slot = term_slot(h, pr.first);
                    if (slot >= 0) { plo = h->term_ptr[slot]; phi = h->term_ptr[slot + 1]; }
                }
                double w = pr.second;
                if (q->apply_idf) {
                    const double df = (double)(need_corpus ? live_df(h, pr.first, slot) : 0);
                    // local_collection.py _compute_idf: log((N - df + 0.5) / (df + 0.5) + 1)
                    w = w * std::log(((double)h->n_live - df + 0.5) / (df + 0.5) + 1.0);
                }
                all_pos = all_pos && w > 0.0 && w < INFINITY;
                qhidx.push_back((need_corpus && slot >= 0 && h->n_heavy) ? h->heavy_of_slot[slot] : -1);
                // MaxScore upper bound of this term's contribution to any row of the shard; +inf = "always
                // essential" (non-positive or non-finite weights are never pruned)
                double ub = INFINITY;
                if (w > 0.0 && w < INFINITY) ub = (slot >= 0 && h->term_maxval[slot] > 0.0f) ? w * (double)h->term_maxval[slot] : 0.0;
                weight.push_back(w);
                qub.push_back(ub);
                qterm.push_back(pr.first);
                qlo.push_back((uint32_t)plo);
                qhi.push_back((uint32_t)phi);
                qplo.push_back((uint32_t)plo);
                qphi.push_back((uint32_t)phi);
                slotq.push_back(i);
                qtab.push_back((need_corpus && slot >= 0 && !h->tab_off_of_slot.empty()) ? h->tab_off_of_slot[slot] : VB_MS_NO_TAB);
                qshift.push_back((need_corpus && slot >= 0 && !h->tab_shift_of_slot.empty()) ? h->tab_shift_of_slot[slot] : 0);
            }
            // terms routed to their dense column are not walked as postings (empty slice)
            // relaxed mode (order-free sums, dense columns) needs every product >= 0 for its error bound
            const bool relax = all_pos && need_corpus && h->sparse_nonneg && h->opt_sparse_dense;
            qrelaxed[i] = relax ? 1 : 0;
            // MaxScore kernel: bounds and the order-free sum need every product >= 0 as well
            // Every query length comes this way (up to VB_MS_MAX_TERMS terms).  Until the kernel tested the score
            // bound BEFORE the ownership lookups, a long query paid ~pe lookups per surviving posting and K3's
            // accumulate-everything beat it (hence the ms_max_terms option, then 16); now K3M with an 85 % budget for
            // long queries runs the 2..65-term MCP replay in 155 ms per 4096-query batch against 214 with K3.
            const bool bounded = all_pos && need_corpus && h->sparse_nonneg && h->opt_sparse_ms && hi > lo;
            const bool ms = bounded && hi - lo <= h->opt_ms_max_terms;
            const bool mh = bounded && !ms && h->opt_sparse_mh;         // long query: hash-accumulate MaxScore (K3H)
            qms[i] = ms ? 1 : (mh ? 2 : 0);
            if (ms) {
                b.any_ms = true;
                uint64_t tot = 0;
                for (size_t t = q_first; t < weight.size(); ++t) tot += qphi[t] - qplo[t];
                b.ms_max_post = std::max(b.ms_max_post, tot);
            }
            else if (hi > lo) {
                dirq.push_back(i);
                if (mh) b.any_mh = true;
                else { b.any_old = true; oldq.push_back(i); }
            }
            for (size_t t = q_first; t < weight.size(); ++t) {
                if (!relax) qhidx[t] = -1;
                if (qhidx[t] >= 0) { qlo[t] = qhi[t] = 0; b.any_heavy = true; }
            }
            indptr[i + 1] = (int64_t)weight.size();
            b.nt_max = std::max<uint32_t>(b.nt_max, (uint32_t)(indptr[i + 1] - indptr[i]));
            if (hi > lo) { b.mode[i] = q->fusion; b.any_sparse = true; }
        }
    }
    b.n_qterms = (uint32_t)weight.size();

    // ---- filters: the ones no query uses are dropped, the ones with equal content merged, so that every consumer
    // (mask kernel, mask mode, row selection) sees distinct, used filters: at most B + 1 of them ----
    const bool tombstones = h->n_live < h->n_rows;
    std::vector<int32_t> mask_of(b.B, -1);
    std::vector<vb_filter> flt;
    std::vector<int32_t> merged_as(q->n_filters, -2);          // caller's filter -> index in flt (-1: no clause, -2: not seen)
    std::unordered_map<FilterKey, int32_t, FilterKeyHash, FilterKeyEq> by_content;
    const vb_filter alive_only{nullptr, 0, VB_TS_NONE, 0, 0};
    auto merge = [&](const vb_filter* x) -> int32_t {
        auto it = by_content.emplace(filter_key(x), (int32_t)flt.size());
        if (it.second) flt.push_back(*x);
        return it.first->second;
    };
    bool any_filter = false;
    for (uint32_t i = 0; i < b.B; ++i) {
        int32_t f = q->filter_of ? q->filter_of[i] : -1;
        if (f >= 0) {
            if (merged_as[f] == -2) {
                const vb_filter& x = q->filters[f];
                merged_as[f] = (x.scope_bits == nullptr && x.ts_field == VB_TS_NONE && !tombstones) ? -1 : merge(&x);   // no clause
            }
            f = merged_as[f];
        }
        mask_of[i] = f;
        any_filter |= f >= 0;
    }
    if (tombstones) {   // unfiltered queries still need the alive bits
        int32_t alive_id = -1;
        for (uint32_t i = 0; i < b.B; ++i)
            if (mask_of[i] < 0) {
                if (alive_id < 0) alive_id = merge(&alive_only);
                mask_of[i] = alive_id;
            }
        any_filter = true;
    }
    b.use_mask = any_filter && need_corpus;
    b.mask_of_host = mask_of;
    if (b.use_mask && mask_of[0] >= 0 && std::all_of(mask_of.begin(), mask_of.end(), [&](int32_t f) { return f == mask_of[0]; })) {
        // the row selection's cache key: equal for content-equal filters (the normalisation of filter_key)
        const FilterKey fk = filter_key(&flt[mask_of[0]]);
        const vb_filter& x = *fk.f;
        const bool ts = x.ts_field != VB_TS_NONE;
        b.sel_filter = {x.scope_bits != nullptr, (uint64_t)(uint32_t)x.ts_field, ts ? (uint64_t)x.ts_lo : 0u, ts ? (uint64_t)x.ts_hi : 0u};
        b.sel_filter.insert(b.sel_filter.end(), x.scope_bits, x.scope_bits + fk.words);
    }
    b.n_filters = b.use_mask ? (uint32_t)flt.size() : 0;
    b.mask_words = (uint32_t)((h->n_rows + 31) / 32);
    b.n_blocks = (uint32_t)((h->base_rows + VB_ROWS_PER_BLOCK - 1) / VB_ROWS_PER_BLOCK);   // row blocks of the inverted index

    // ---- pack everything into one pinned block, one H2D copy ----
    Arena ar;
    const size_t o_q = ar.take((size_t)b.B * h->dim * 4);
    const size_t o_ip = ar.take((b.B + 1) * 8);
    const size_t o_w = ar.take((size_t)b.n_qterms * 8 + 8);
    const size_t o_ub = ar.take((size_t)b.n_qterms * 8 + 8);
    const size_t o_tid = ar.take((size_t)b.n_qterms * 4 + 8);
    const size_t o_hx = ar.take((size_t)b.n_qterms * 4 + 8);
    const size_t o_rx = ar.take((size_t)b.B + 8);
    const size_t o_lo = ar.take((size_t)b.n_qterms * 4 + 8);
    const size_t o_hi = ar.take((size_t)b.n_qterms * 4 + 8);
    const size_t o_plo = ar.take((size_t)b.n_qterms * 4 + 8);
    const size_t o_phi = ar.take((size_t)b.n_qterms * 4 + 8);
    const size_t o_sq = ar.take((size_t)b.n_qterms * 4 + 8);
    const size_t o_ms = ar.take((size_t)b.B + 8);
    const size_t o_oq = ar.take((size_t)oldq.size() * 4 + 8);
    const size_t o_dq = ar.take((size_t)dirq.size() * 4 + 8);
    const size_t o_tab = ar.take((size_t)b.n_qterms * 4 + 8);
    const size_t o_tsh = ar.take((size_t)b.n_qterms + 8);
    // delta rows present: the batch inverted by term (term -> queries, weights) for K3D
    std::vector<uint32_t> ut, up, uq;
    std::vector<double> uw;
    if (need_corpus && b.any_sparse && h->n_rows > h->base_rows) {
        std::vector<uint32_t> order(b.n_qterms);
        for (uint32_t t = 0; t < b.n_qterms; ++t) order[t] = t;
        std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return qterm[x] < qterm[y]; });   // (term, query)
        for (uint32_t t : order) {
            if (ut.empty() || ut.back() != qterm[t]) { ut.push_back(qterm[t]); up.push_back((uint32_t)uq.size()); }
            uq.push_back(slotq[t]);
            uw.push_back(weight[t]);
        }
        up.push_back((uint32_t)uq.size());
        b.n_uterms = (uint32_t)ut.size();
    }
    const size_t o_ut = ar.take(ut.size() * 4 + 8);
    const size_t o_up = ar.take(up.size() * 4 + 8);
    const size_t o_uq = ar.take(uq.size() * 4 + 8);
    const size_t o_uw = ar.take(uw.size() * 8 + 8);
    const size_t o_mo = ar.take((size_t)b.B * 4);
    const size_t o_md = ar.take((size_t)b.B * 4);
    const size_t o_fl = ar.take((size_t)std::max<uint32_t>(1, b.n_filters) * sizeof(VbFilterDev));
    std::vector<size_t> o_bits(b.n_filters, 0);
    for (uint32_t f = 0; f < b.n_filters; ++f)
        if (flt[f].scope_bits) o_bits[f] = ar.take((size_t)flt[f].scope_words * 4);
    // mask mode 3 tables: K2T tiles of VB_TILE_N queries, resident-K2 sub-batches as vb_gemm_plan cuts them
    const bool ftabs = b.n_filters > 31u && vb_gemm_supported(h->d_pad, b.B);
    const uint32_t k2_sub = ftabs ? vb_gemm_plan((uint32_t)h->d_pad, b.B, (int)h->opt_k2_precision).sub : 0u;
    const size_t o_ft2t = ftabs ? ar.take(filter_tiles_bytes(b.B, VB_TILE_N)) : 0;
    const size_t o_ft2 = ftabs ? ar.take(filter_tiles_bytes(b.B, k2_sub)) : 0;
    TRY(host_reserve(h->h_args_s[h->cur], ar.off));
    TRY(dev_reserve(h, h->args, ar.off, false));
    unsigned char* hp = h->h_args_s[h->cur].as<unsigned char>();
    unsigned char* dp = h->args.as<unsigned char>();
    if (!h->q_dev) {
        if (!q->dense) return vb_fail("dense queries are NULL");   // validate_batch ran before the lock
        memcpy(hp + o_q, q->dense, (size_t)b.B * h->dim * 4);
    }
    memcpy(hp + o_ip, indptr.data(), (b.B + 1) * 8);
    if (b.n_qterms) {
        memcpy(hp + o_w, weight.data(), (size_t)b.n_qterms * 8);
        memcpy(hp + o_ub, qub.data(), (size_t)b.n_qterms * 8);
        memcpy(hp + o_tid, qterm.data(), (size_t)b.n_qterms * 4);
        memcpy(hp + o_hx, qhidx.data(), (size_t)b.n_qterms * 4);
        memcpy(hp + o_rx, qrelaxed.data(), (size_t)b.B);
        memcpy(hp + o_lo, qlo.data(), (size_t)b.n_qterms * 4);
        memcpy(hp + o_hi, qhi.data(), (size_t)b.n_qterms * 4);
        memcpy(hp + o_plo, qplo.data(), (size_t)b.n_qterms * 4);
        memcpy(hp + o_phi, qphi.data(), (size_t)b.n_qterms * 4);
        memcpy(hp + o_sq, slotq.data(), (size_t)b.n_qterms * 4);
        memcpy(hp + o_ms, qms.data(), (size_t)b.B);
        if (!oldq.empty()) memcpy(hp + o_oq, oldq.data(), oldq.size() * 4);
        if (!dirq.empty()) memcpy(hp + o_dq, dirq.data(), dirq.size() * 4);
        memcpy(hp + o_tab, qtab.data(), (size_t)b.n_qterms * 4);
        memcpy(hp + o_tsh, qshift.data(), (size_t)b.n_qterms);
    }
    if (b.n_uterms) {
        memcpy(hp + o_ut, ut.data(), ut.size() * 4);
        memcpy(hp + o_up, up.data(), up.size() * 4);
        memcpy(hp + o_uq, uq.data(), uq.size() * 4);
        memcpy(hp + o_uw, uw.data(), uw.size() * 8);
    }
    b.n_old = (uint32_t)oldq.size();
    b.n_dir = (uint32_t)dirq.size();
    b.n_rows = (uint32_t)h->n_rows;
    b.base_rows = (uint32_t)h->base_rows;
    b.gen = h->write_gen;
    memcpy(hp + o_mo, mask_of.data(), (size_t)b.B * 4);
    if (ftabs) {
        b.ft_k2t = build_filter_tiles(mask_of, b.n_filters, VB_TILE_N, VB_TILED_MAX_Q, hp, dp, o_ft2t);
        b.ft_k2 = build_filter_tiles(mask_of, b.n_filters, k2_sub, k2_sub, hp, dp, o_ft2);
    }
    memcpy(hp + o_md, b.mode.data(), (size_t)b.B * 4);
    VbFilterDev* hf = reinterpret_cast<VbFilterDev*>(hp + o_fl);
    for (uint32_t f = 0; f < b.n_filters; ++f) {
        hf[f].scope_bits = flt[f].scope_bits ? reinterpret_cast<const uint32_t*>(dp + o_bits[f]) : nullptr;
        hf[f].scope_words = flt[f].scope_words;
        hf[f].ts_field = flt[f].ts_field;
        hf[f].ts_lo = flt[f].ts_lo;
        hf[f].ts_hi = flt[f].ts_hi;
        if (flt[f].scope_bits) { memcpy(hp + o_bits[f], flt[f].scope_bits, (size_t)flt[f].scope_words * 4); b.need_scope = 1; }
        if (flt[f].ts_field == VB_TS_CREATED) b.need_created = 1;
        if (flt[f].ts_field == VB_TS_MODIFIED) b.need_modified = 1;
    }
    // device hand-off (SURVEY §8 f-4): the query rows never visit the host — the H2D copy starts after their slot and a
    // D2D copy, ordered after the producer's stream, fills it
    const size_t h2d_skip = h->q_dev ? o_ip : 0;
    CK(cudaMemcpyAsync(dp + h2d_skip, hp + h2d_skip, ar.off - h2d_skip, cudaMemcpyHostToDevice, h->stream));
    if (h->q_dev) {
        if (!h->ev_q) CK(cudaEventCreateWithFlags(&h->ev_q, cudaEventDisableTiming));
        CK(cudaEventRecord(h->ev_q, h->q_dev_stream));
        CK(cudaStreamWaitEvent(h->stream, h->ev_q, 0));
        CK(cudaMemcpyAsync(dp + o_q, h->q_dev, (size_t)b.B * h->dim * 4, cudaMemcpyDeviceToDevice, h->stream));
    }
    b.d_q = reinterpret_cast<const float*>(dp + o_q);
    b.d_qindptr = reinterpret_cast<const int64_t*>(dp + o_ip);
    b.d_qweight = reinterpret_cast<const double*>(dp + o_w);
    b.d_qub = reinterpret_cast<const double*>(dp + o_ub);
    b.d_qterm = reinterpret_cast<const uint32_t*>(dp + o_tid);
    b.d_qhidx = reinterpret_cast<const int32_t*>(dp + o_hx);
    b.d_qrelaxed = reinterpret_cast<const uint8_t*>(dp + o_rx);
    b.d_qlo = reinterpret_cast<const uint32_t*>(dp + o_lo);
    b.d_qhi = reinterpret_cast<const uint32_t*>(dp + o_hi);
    b.d_qplo = reinterpret_cast<const uint32_t*>(dp + o_plo);
    b.d_qphi = reinterpret_cast<const uint32_t*>(dp + o_phi);
    b.d_slotq = reinterpret_cast<const uint32_t*>(dp + o_sq);
    b.d_qms = reinterpret_cast<const uint8_t*>(dp + o_ms);
    b.d_oldq = reinterpret_cast<const uint32_t*>(dp + o_oq);
    b.d_dirq = reinterpret_cast<const uint32_t*>(dp + o_dq);
    b.d_qtab = reinterpret_cast<const uint32_t*>(dp + o_tab);
    b.d_qshift = reinterpret_cast<const uint8_t*>(dp + o_tsh);
    b.d_ut = reinterpret_cast<const uint32_t*>(dp + o_ut);
    b.d_up = reinterpret_cast<const uint32_t*>(dp + o_up);
    b.d_uq = reinterpret_cast<const uint32_t*>(dp + o_uq);
    b.d_uw = reinterpret_cast<const double*>(dp + o_uw);
    b.d_maskof = reinterpret_cast<const int32_t*>(dp + o_mo);
    b.d_mode = reinterpret_cast<const int32_t*>(dp + o_md);
    b.d_filters = reinterpret_cast<const VbFilterDev*>(dp + o_fl);

    // ---- candidate lists ----
    // segment growth: each segment appends ~ratio * k' candidates per list before the next compaction.  Batches
    // keep 32 (list memory and compaction time scale with B); single queries are launch-latency bound and take
    // 128 (one segment fewer on 100k..10M rows; measured +7..25 % q/s at B = 1).
    // (round 2: 8 instead of 32 for batches — the appends of a segment cost more than the extra launch + compaction:
    //  cfg4 dense 18.0 -> 15.8 ms)
    b.seg_ratio = h->opt_seg_ratio > 0 ? (uint32_t)h->opt_seg_ratio : (b.B <= 4 ? 128u : 8u);
    uint32_t need_cap = std::max<uint32_t>(16384u, (uint32_t)align_up((size_t)2 * (size_t)std::max<uint32_t>(b.seg_ratio, 32u) * b.k, 4096));
    // roomier lists (up to 256 MB in all) let K3M take larger posting stages: fewer launches on small corpora
    need_cap = std::max<uint32_t>(need_cap, (uint32_t)std::min<uint64_t>(align_up((size_t)16 * 128 * b.k, 4096), (256ull << 20) / ((uint64_t)b.n_lists * 8u) / 4096u * 4096u));
    // K1F (single-pass scan for tiny batches) leaves one local top-k' per CTA in the list before the merge
    if (b.B <= VB_K1F_MAX_B) need_cap = std::max<uint32_t>(need_cap, (uint32_t)align_up((size_t)vb_k1f_grid(h->sm_count, b.k, b.B, h->d_pad) * b.k, 4096));
    // tiny batches are launch-latency bound: roomy lists (a few MB) let K3M take 1024x larger posting stages
    if (b.B <= VB_K1F_MAX_B) need_cap = std::max<uint32_t>(need_cap, 262144u);
    h->cand_cap = need_cap;
    TRY(dev_reserve(h, h->cand, (size_t)b.n_lists * need_cap * 8, false));
    TRY(dev_reserve(h, h->lists, (size_t)b.n_lists * (16 + 4 * VB_SUB), false));
    b.tau = h->lists.as<float>();
    b.overflow = h->lists.as<uint32_t>() + b.n_lists;
    b.cnt = h->lists.as<uint32_t>() + 2 * (size_t)b.n_lists;      // [n_lists][VB_SUB]
    b.gtau = h->lists.as<uint32_t>() + (2 + (size_t)VB_SUB) * b.n_lists;
    b.done = h->lists.as<uint32_t>() + (3 + (size_t)VB_SUB) * b.n_lists;
    b.h2d_bytes = ar.off - h2d_skip;
    h->stats.last_h2d_bytes = ar.off - h2d_skip;
    // output block layout
    Arena ao;
    b.o_rows = ao.take((size_t)b.B * b.limit * 4);
    b.o_sc = ao.take((size_t)b.B * b.limit * 8);
    b.o_cnt = ao.take((size_t)b.B * 4);
    b.o_lcnt = ao.take((size_t)b.n_lists * 4);
    b.o_ovf = ao.take((size_t)b.n_lists * 4);
    b.o_bad = ao.take((size_t)b.B * 4);
    b.o_keys = ao.take((size_t)b.n_lists * b.k * 8);
    b.out_bytes = ao.off;
    TRY(dev_reserve(h, h->out, b.out_bytes, false));
    TRY(host_reserve(h->h_out_s[h->cur], b.out_bytes));
    h->sel_ran[h->cur] = false;
    b.valid = true;
    return 0;
}

// direct_rows > 0: the first segment stores its keys at fixed slots [0, direct_rows) of every
// list (no atomics); slots nobody writes (masked rows, rows without postings) must read as empty.
static int init_lists(vb_index* h, const Batch& b, uint32_t direct_rows) {
    if (direct_rows)
        CK(cudaMemset2DAsync(h->cand.p, (size_t)h->cand_cap * 8, 0, (size_t)direct_rows * 8, b.n_lists, h->stream));
    return 0;
}
// empty lists for the paths that score nothing (empty index, merge of gathered shard lists)
__global__ void vb_init_lists_kernel(const VbListInit li) {
    vb_init_list(li, blockIdx.x * blockDim.x + threadIdx.x);
}
static int empty_lists(vb_index* h, const Batch& b) {
    VbListInit li{};
    li.tau = b.tau; li.cnt = b.cnt; li.overflow = b.overflow; li.gtau = b.gtau; li.n = b.n_lists; li.cnt0 = 0;
    li.no_direct = nullptr; li.n_queries = b.B; li.dense_direct = 1u;
    vb_init_lists_kernel<<<(b.n_lists + 255) / 256, 256, 0, h->stream>>>(li);
    CKK("vb_init_lists_kernel");
    ++h->stats.last_launches;
    return 0;
}

static VbLists make_lists(const vb_index* h, const Batch& b, bool safe) {
    VbLists L;
    L.cand = h->cand.as<uint64_t>();
    L.cnt = b.cnt;
    L.n_lists = b.n_lists;
    L.cap = h->cand_cap;
    const uint32_t nsub = safe ? 1u : VB_SUB;          // safe mode: one range, segments that cannot overflow it
    L.sub_cap = h->cand_cap / nsub;
    L.sub_mask = nsub - 1u;
    return L;
}

static int launch_scan(vb_index* h, const Batch& b, const VbLists& L, uint32_t row_begin, uint32_t row_end, uint32_t direct, cudaStream_t st) {
    VbScanArgs a{};
    a.rows = h->rows.as<uint4>();
    a.inv_norm = h->inv_norm.as<float>();
    a.mask = b.use_mask ? h->mask.as<uint32_t>() : nullptr;
    a.mask_of = b.use_mask ? b.d_maskof : nullptr;
    a.q_hat = h->q_hat.as<float>();
    a.tau = b.tau;
    a.lists = L;
    a.mask_words = b.mask_words;
    a.chunks = (uint32_t)h->d_pad / 8;
    a.row_begin = row_begin;
    a.row_end = row_end;
    a.row_base = (uint32_t)h->row_base;
    a.q_begin = 0;
    a.direct = direct;
    const uint32_t groups = (row_end - row_begin + 31) / 32;
    const uint32_t per_q = std::max<uint32_t>(1, (uint32_t)(h->sm_count * 8) / std::min<uint32_t>(b.B, 8));
    dim3 grid(std::min<uint32_t>((groups + 7) / 8, per_q), b.B);
    const int nch = (int)((a.chunks + 31) / 32);
    switch (nch) {
        case 1: vb_dense_scan_kernel<1><<<grid, 256, 0, st>>>(a); break;
        case 2: vb_dense_scan_kernel<2><<<grid, 256, 0, st>>>(a); break;
        case 3: vb_dense_scan_kernel<3><<<grid, 256, 0, st>>>(a); break;
        case 4: vb_dense_scan_kernel<4><<<grid, 256, 0, st>>>(a); break;
        default: vb_dense_scan_generic_kernel<<<grid, 256, 0, st>>>(a); break;
    }
    CKK("vb_dense_scan_kernel");
    ++h->stats.last_launches;
    return 0;
}

// Score both branches of this shard and leave the exact, sorted top-k' of every list in
// cand[list][0..cnt).  `safe`: fixed small segments that can never overflow a list.
static int run_branches(vb_index* h, const Batch& b, bool safe) {
    const uint32_t n = (uint32_t)h->n_rows;
    // segment schedule (boundaries are multiples of VB_ROWS_PER_BLOCK)
    std::vector<uint32_t> bounds{0};
    if (safe || h->opt_safe_mode) {
        const uint32_t step = (uint32_t)std::max<size_t>(VB_ROWS_PER_BLOCK, (h->cand_cap - b.k) / VB_ROWS_PER_BLOCK * VB_ROWS_PER_BLOCK);
        for (uint64_t r = step; r < n; r += step) bounds.push_back((uint32_t)r);
    } else {
        for (uint64_t r = (uint64_t)h->opt_seg_first; r < n; r *= (uint64_t)b.seg_ratio) bounds.push_back((uint32_t)r);
    }
    bounds.push_back(n);
    const bool safe_mode = safe || h->opt_safe_mode;
    const VbLists L = make_lists(h, b, safe_mode);
    // dense path choice
    int path = (int)h->opt_dense_path;
    if (path == 0) path = vb_gemm_supported(h->d_pad, b.B) && b.B >= 2 ? 2 : 1;
    if (path == 2 && !vb_gemm_supported(h->d_pad, b.B)) return vb_fail("dense_path=2 requested but unsupported for d_pad=%d B=%u", h->d_pad, b.B);
    h->stats.last_dense_path = (uint32_t)path;
    VbGemmPlan plan{1u, 0u};
    if (path == 2) plan = vb_gemm_plan((uint32_t)h->d_pad, b.B, (int)h->opt_k2_precision);
    // batches too large to sit resident in shared memory go to the query-tiled, tensor-bound kernel
    // (one corpus pass per 1024 queries)
    const bool tiled = path == 2 && b.B > plan.sub && !plan.split && h->opt_k2_tiled && vb_gemm_tiled_supported(h->d_pad);
    h->stats.last_dense_passes = path == 2 ? (tiled ? (b.B + VB_TILED_MAX_Q - 1) / VB_TILED_MAX_Q : (b.B + plan.sub - 1) / plan.sub) : b.B;
    // sparse work: the inverted index covers rows [0, nb); rows appended since (the delta) are scored by K3D
    const uint32_t nb = (uint32_t)std::min<uint64_t>(h->base_rows, n);
    const bool do_sparse = b.any_sparse && h->nnz_live > 0 && b.n_qterms > 0 && nb > 0;
    const bool do_delta = b.any_sparse && b.n_uterms > 0 && nb < n;
    // Which sparse kernel scores which query.  Queries whose products are all >= 0 and that are not too long go to
    // K3M, the posting-driven MaxScore kernel; the others (and everything when K3M is off) stay on K3 (block x query
    // CTAs over the row segments, first segment direct).
    //   normal mode: K3M runs in STAGES over the whole index (sparse_ms.cuh): stage 0 scores the first ms_p0
    //                postings of every query in descending-ub order with no threshold, each later stage 32x more;
    //   safe mode:   K3M runs once per (small) row segment, like K3, so that no list can overflow.
    const bool ms_on = do_sparse && b.any_ms && h->opt_sparse_ms;
    const bool ms_staged = ms_on && !safe_mode && h->opt_ms_staged;
    const bool mh_on = do_sparse && b.any_mh;                   // long queries: K3 direct segment, then K3H per segment
    // K1F: one pass over all rows for tiny batches (no segments, no direct slots)
    // (on large corpora the segmented K1 streams faster — no per-stretch barriers — and its launches are noise there:
    //  cfg3 10M rows, B = 1: K1 1.65 ms, K1F 1.83 ms; cfg1 100k rows: K1 59 us + 3 selects, K1F 48 us + 1 merge)
    const bool k1f = path == 1 && !safe_mode && h->opt_k1f && (h->opt_k1f > 1 || n <= (2u << 20)) && b.B <= VB_K1F_MAX_B && (h->d_pad / 8 + 31) / 32 <= 4 &&
                     b.k <= VB_K1F_CAP / 2u && (uint64_t)vb_k1f_grid(h->sm_count, b.k, b.B, h->d_pad) * b.k <= h->cand_cap;
    // the first segment writes its keys to fixed slots at the front of the list (no atomics) — unless nobody runs
    // a first segment: K1F scans in one pass, K3M in posting stages
    const bool k3_direct = do_sparse && (!ms_staged || b.n_dir > 0);
    const uint32_t direct_rows = (bounds[1] <= h->cand_cap && (!k1f || k3_direct)) ? bounds[1] : 0u;
    TRY(init_lists(h, b, direct_rows));
    // list set-up + query prep (fp32 unit queries for K1, packed bf16 operand for K2) in ONE launch
    TRY(dev_reserve(h, h->q_hat, (size_t)b.B * h->d_pad * 4, false));
    TRY(dev_reserve(h, h->q_bf16, (size_t)(2 * ((size_t)b.B + 256)) * h->d_pad * 2, false));
    TRY(dev_reserve(h, h->q_scale, (size_t)b.B * 4, false));
    VbListInit li{};
    li.tau = b.tau; li.cnt = b.cnt; li.overflow = b.overflow; li.gtau = b.gtau; li.n = b.n_lists; li.cnt0 = direct_rows;
    li.no_direct = ms_staged ? b.d_qms : nullptr; li.n_queries = b.B; li.dense_direct = k1f ? 0u : 1u;
    vb_prep_query_kernel<<<b.B, 128, 0, h->stream>>>(b.d_q, (uint32_t)h->dim, (uint32_t)h->d_pad, b.B, plan.sub, plan.split,
                                                     h->q_hat.as<float>(), h->q_bf16.as<__nv_bfloat16>(), h->q_scale.as<float>(),
                                                     reinterpret_cast<uint32_t*>(h->out.as<unsigned char>() + b.o_bad), li);
    CKK("vb_prep_query_kernel");
    ++h->stats.last_launches;
    // K0 filter masks
    if (b.use_mask) {
        prof_begin(h, PH_MASK);
        const size_t mask_bytes = (size_t)b.n_filters * b.mask_words * 4;
        if (dev_reserve(h, h->mask, mask_bytes, false) != 0) {
            cudaGetLastError();
            return vb_fail("filter masks of %u distinct filters over %u rows need %zu bytes of device memory: %s",
                           b.n_filters, n, mask_bytes, g_err.c_str());
        }
        vb_mask_kernel<<<grid_for((uint64_t)b.mask_words * 32, 256, h->sm_count * 8), 256, 0, h->stream>>>(
            h->scope_id.as<uint32_t>(), h->created.as<int64_t>(), h->modified.as<int64_t>(), h->alive.as<uint32_t>(), n,
            b.d_filters, b.n_filters, b.mask_words, b.need_created, b.need_modified, b.need_scope, h->mask.as<uint32_t>());
        CKK("vb_mask_kernel");
        ++h->stats.last_launches;
        prof_end(h);
    }
    // The dense chain (K1/K2 + select of the dense lists) and the sparse chain (slice table, K3 +
    // select of the sparse lists) are independent until the fusion, so they run on two streams:
    // the small kernels of one chain (selects, first segments, slice table) hide behind the big
    // kernels of the other.
    const bool two_streams = (do_sparse || do_delta) && h->opt_overlap;
    cudaStream_t sd = h->stream, ss = two_streams ? h->aux_stream : h->stream;
    if (two_streams) {
        CK(cudaEventRecord(h->ev_fork, sd));
        CK(cudaStreamWaitEvent(ss, h->ev_fork, 0));
    }
    // ---- K2T row selection plan (dense_compact.cuh): the tensor-bound kernel, ONE filter for the whole batch, every
    // segment of at least dense_compact_min_rows rows.  Count, list and copy run on a side stream right after the mask
    // kernel: the copy of segment s + 1 (HBM-bound) hides behind the GEMM of segment s (tensor-bound).  With the chains
    // serialised (overlap = 0: per-phase timing) they run inline on the dense stream and are charged to the dense phase.
    // The copy is kept across batches (h->sel_key): a segment whose key matches the scratch is not copied again, and
    // the tensor-core kernel reads the scratch and its device-side {count, decision} as they are.
    struct SelSeg { bool on = false, kept = false; uint32_t cap_rows = 0, n_blocks = 0, ev = 0; size_t row_off = 0, meta_off = 0; };
    std::vector<SelSeg> selseg(bounds.size() - 1);
    bool sel_any = false, sel_copy = false;
    std::vector<uint64_t> sel_key;
    const bool sel_side = h->opt_overlap != 0;
    // auto threshold: the copy costs ~0.49 ns per passing row (read + write of 2 * d_pad bytes at HBM speed, d_pad = 768);
    // one pass of the tensor-core kernel over a row costs max(0.245 ns (HBM), 1.08 ns * queries / 1024 (tensor pipe)) — both
    // scale with d_pad alike.  Copying pays when (1 - p) * passes' time > p * copy time.
    uint32_t sel_pct = (uint32_t)std::max<int64_t>(0, std::min<int64_t>(100, h->opt_dense_compact));
    if (h->opt_dense_compact < 0 && path == 2) {
        double T = 0.0;
        if (tiled) for (uint32_t q0 = 0; q0 < b.B; q0 += VB_TILED_MAX_Q) T += std::max(0.245, 1.08 * std::min(VB_TILED_MAX_Q, b.B - q0) / 1024.0);
        else T = 0.245 * ((b.B + plan.sub - 1) / plan.sub);
        sel_pct = (uint32_t)(95.0 * T / (T + 0.49));
    }
    if (path == 2 && !k1f && b.use_mask && sel_pct > 0 && !h->sel_no_memory && h->d_pad <= 1024) {
        bool uniform = b.mask_of_host[0] >= 0;
        for (uint32_t i = 1; uniform && i < b.B; ++i) uniform = b.mask_of_host[i] == b.mask_of_host[0];
        size_t rows_total = 0, meta_total = 0;
        uint32_t n_on = 0;
        for (size_t si = (direct_rows ? 1 : 0); uniform && si + 1 < bounds.size() && n_on < 8u; ++si) {
            const uint32_t r0 = bounds[si], r1 = bounds[si + 1];
            if ((r0 % 128u) != 0u || (int64_t)(r1 - r0) < h->opt_dense_compact_min_rows) continue;
            SelSeg& z = selseg[si];
            z.on = true; z.cap_rows = (uint32_t)align_up(r1 - r0, 128); z.n_blocks = ((r1 - r0 + 31u) / 32u + VB_SEL_WORDS - 1u) / VB_SEL_WORDS;
            z.row_off = rows_total; z.meta_off = meta_total; z.ev = n_on++;
            rows_total += z.cap_rows; meta_total += align_up((size_t)4 + z.n_blocks, 4);
        }
        const size_t scratch = rows_total * h->d_pad * 2;
        if (n_on && scratch > h->sel_rows.cap) {
            size_t free_b = 0, total_b = 0;
            if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess || free_b + h->sel_rows.cap < scratch + (4ull << 30)) {
                cudaGetLastError();
                h->sel_no_memory = true;                         // the scratch matrix does not fit beside the shard: stay in place
                h->sel_key.clear();
                n_on = 0;
            }
        }
        if (n_on) {
            const void* before[4] = {h->sel_rows.p, h->sel_inv.p, h->sel_ids.p, h->sel_meta.p};
            // Invalid from here until this batch has enqueued all of its work (end of run_branches): an error return
            // in between (a failed reserve, a copy enqueued in part) leaves the next batch to copy again.
            std::vector<uint64_t> cached_key;
            cached_key.swap(h->sel_key);
            TRY(dev_reserve(h, h->sel_rows, scratch, false));
            TRY(dev_reserve(h, h->sel_inv, rows_total * 4, false));
            TRY(dev_reserve(h, h->sel_ids, rows_total * 4, false));
            TRY(dev_reserve(h, h->sel_meta, meta_total * 4, false));
            const bool moved = before[0] != h->sel_rows.p || before[1] != h->sel_inv.p || before[2] != h->sel_ids.p || before[3] != h->sel_meta.p;
            sel_any = true;
            // the key: filter content, index version, and every input of the plan above
            sel_key = b.sel_filter;
            sel_key.insert(sel_key.end(), {h->write_gen, (uint64_t)n, (uint64_t)h->d_pad, sel_pct, (uint64_t)h->opt_dense_compact_min_rows,
                                           (uint64_t)path, (uint64_t)tiled, direct_rows});
            const bool key_holds = h->opt_sel_reuse && !moved && sel_key == cached_key;
            for (size_t si = 0; si < selseg.size(); ++si) {
                SelSeg& z = selseg[si];
                if (!z.on) continue;
                const std::array<uint64_t, 5> zk{bounds[si], bounds[si + 1], z.row_off, z.meta_off, z.cap_rows};
                z.kept = key_holds && std::find(h->sel_segs.begin(), h->sel_segs.end(), zk) != h->sel_segs.end();
                sel_copy |= !z.kept;
            }
        } else for (auto& z : selseg) z.on = false;
    }
    auto sel_launch = [&](size_t si, cudaStream_t st) -> int {
        const SelSeg& z = selseg[si];
        const uint32_t r0 = bounds[si], r1 = bounds[si + 1];
        VbRowSelArgs sa{};
        sa.mask = h->mask.as<uint32_t>() + (size_t)b.mask_of_host[0] * b.mask_words;
        sa.word_begin = r0 / 32u; sa.word_end = (r1 + 31u) / 32u; sa.row_end = r1;
        sa.sel = h->sel_meta.as<uint32_t>() + z.meta_off; sa.block_sums = sa.sel + 4; sa.ids = h->sel_ids.as<uint32_t>() + z.row_off;
        sa.pct = sel_pct; sa.pad_row = r0; sa.cap_rows = z.cap_rows;
        vb_rowsel_count_kernel<<<z.n_blocks, VB_SEL_THREADS, 0, st>>>(sa);
        CKK("vb_rowsel_count_kernel");
        vb_rowsel_scatter_kernel<<<z.n_blocks, VB_SEL_THREADS, 0, st>>>(sa);
        CKK("vb_rowsel_scatter_kernel");
        vb_rowsel_gather_kernel<<<h->sm_count * 4, 256, 0, st>>>(h->rows.as<uint4>(), h->inv_norm.as<float>(), sa.ids, sa.sel,
                                                                h->sel_rows.as<uint4>() + z.row_off * (h->d_pad / 8), h->sel_inv.as<float>() + z.row_off,
                                                                (uint32_t)h->d_pad / 8u);
        CKK("vb_rowsel_gather_kernel");
        h->stats.last_launches += 3;
        return 0;
    };
    // Ordering of the scratch (two batches can be in flight).  A kept segment is only read, by kernels on the dense
    // stream.  A copy waits for ev_sel_fork, recorded on the dense stream after this batch's mask kernel and therefore
    // after every kernel an earlier batch enqueued there, so it cannot overwrite the scratch while an earlier batch's
    // tensor-core kernel still reads it — whether that batch copied or kept.  A batch that keeps a copy made by an earlier
    // one reads it after that batch's dense kernels, which waited for the copy's events: the copy has finished.
    if (sel_copy && sel_side) {
        if (!h->sel_stream) {
            CK(cudaStreamCreateWithFlags(&h->sel_stream, cudaStreamNonBlocking));
            CK(cudaEventCreateWithFlags(&h->ev_sel_fork, cudaEventDisableTiming));
            for (auto& e : h->ev_sel) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        }
        CK(cudaEventRecord(h->ev_sel_fork, sd));                 // after the mask kernel (and after the previous batch's dense chain)
        CK(cudaStreamWaitEvent(h->sel_stream, h->ev_sel_fork, 0));
        for (size_t si = 0; si < selseg.size(); ++si)
            if (selseg[si].on && !selseg[si].kept) {
                TRY(sel_launch(si, h->sel_stream));
                CK(cudaEventRecord(h->ev_sel[selseg[si].ev], h->sel_stream));
            }
    }
    auto dense_single_pass = [&]() -> int {
        const int pi = prof_begin(h, PH_DENSE | PH_BIG, sd);
        VbScan1Args a{};
        a.rows = h->rows.as<uint4>(); a.inv_norm = h->inv_norm.as<float>();
        a.mask = b.use_mask ? h->mask.as<uint32_t>() : nullptr; a.mask_of = b.use_mask ? b.d_maskof : nullptr;
        a.q_hat = h->q_hat.as<float>(); a.gtau = b.gtau; a.cand = h->cand.as<uint64_t>(); a.cnt = b.cnt;
        a.cap = h->cand_cap; a.k = b.k; a.mask_words = b.mask_words; a.chunks = (uint32_t)h->d_pad / 8; a.n_rows = n;
        a.row_base = (uint32_t)h->row_base;
        a.done = b.done; a.tau = b.tau;
        const dim3 grid(vb_k1f_grid(h->sm_count, b.k, b.B, h->d_pad), b.B);
        // small corpora: fewer 32-row groups than warps — give each warp a half / quarter / eighth of a group
        const uint32_t n_groups = (n + 31u) / 32u, n_warps = grid.x * (VB_K1F_THREADS / 32u);
        a.split_shift = 0;
        while (a.split_shift < 3u && (n_groups << (a.split_shift + 1u)) <= n_warps) ++a.split_shift;
        // large corpora: units of 2..32 groups (one coalesced filter-word load per unit, row batches filled across its
        // groups), as long as every warp still gets >= 4 units (static interleaved assignment: +-1 unit of imbalance)
        a.unit_shift = 0;
        if (!a.split_shift)
            while (a.unit_shift < 5u && (n_groups >> (a.unit_shift + 1u)) >= 4u * n_warps) ++a.unit_shift;
        switch ((a.chunks + 31) / 32) {
            case 1: vb_dense_scan1_kernel<1><<<grid, VB_K1F_THREADS, 0, sd>>>(a); break;
            case 2: vb_dense_scan1_kernel<2><<<grid, VB_K1F_THREADS, 0, sd>>>(a); break;
            case 3: vb_dense_scan1_kernel<3><<<grid, VB_K1F_THREADS, 0, sd>>>(a); break;
            default: vb_dense_scan1_kernel<4><<<grid, VB_K1F_THREADS, 0, sd>>>(a); break;
        }
        CKK("vb_dense_scan1_kernel");
        ++h->stats.last_launches;
        prof_end(h, pi, sd);                                    // (the merge of the per-CTA lists happens inside: last CTA)
        h->stats.last_big_rows = n;
        h->stats.last_dense_path = 3u;                          // K1F
        return 0;
    };
    auto dense_segment = [&](uint32_t r0, uint32_t r1, uint32_t direct, bool big) -> int {
        if (k1f) return 0;                                      // the single pass covers every segment
        // Row selection (planned before the segment loop): nothing to do when the scratch kept this segment's copy;
        // otherwise wait for its copy (side stream), or run the selection here (chains serialised: its own timed region
        // of the dense phase, so that the PH_BIG region stays the tensor-core kernel alone)
        const SelSeg* zsel = nullptr;
        if (path == 2)
            for (size_t si = 0; si + 1 < bounds.size(); ++si)
                if (bounds[si] == r0 && selseg[si].on) {
                    zsel = &selseg[si];
                    if (!zsel->kept && sel_side) CK(cudaStreamWaitEvent(sd, h->ev_sel[zsel->ev], 0));
                    else if (!zsel->kept) {
                        const int pz = prof_begin(h, PH_DENSE, sd);
                        TRY(sel_launch(si, sd));
                        prof_end(h, pz, sd);
                    }
                    if (big) {                                   // {rows, decision} of the roofline's segment for vb_stats
                        TRY(host_reserve(h->h_sel[h->cur], 16));
                        CK(cudaMemcpyAsync(h->h_sel[h->cur].p, h->sel_meta.as<uint32_t>() + zsel->meta_off, 8, cudaMemcpyDeviceToHost, sd));
                        h->sel_ran[h->cur] = true;
                    }
                }
        const int pi = prof_begin(h, PH_DENSE | (big ? PH_BIG : 0), sd);
        if (path == 2) {
            VbGemmLaunch g{};
            g.rows = h->rows.p; g.inv_norm = h->inv_norm.as<float>(); g.q_bf16 = h->q_bf16.p;
            g.mask = b.use_mask ? h->mask.as<uint32_t>() : nullptr; g.mask_of = b.use_mask ? b.d_maskof : nullptr;
            g.mask_words = b.mask_words; g.n_filters = b.n_filters; g.tau = b.tau; g.q_scale = h->q_scale.as<float>(); g.lists = L;
            g.n_rows_total = n; g.row_begin = r0; g.row_end = r1; g.row_base = (uint32_t)h->row_base;
            g.d_pad = (uint32_t)h->d_pad; g.n_queries = b.B; g.sm_count = h->sm_count; g.stream = sd;
            g.direct = direct; g.plan = plan; g.mask_of_host = b.mask_of_host.data();
            g.ftab = tiled ? b.ft_k2t : b.ft_k2;
            if (zsel) {                                          // K2T walks the compacted copy when the device-side decision says so
                g.sel = h->sel_meta.as<uint32_t>() + zsel->meta_off; g.sel_ids = h->sel_ids.as<uint32_t>() + zsel->row_off;
                g.sel_inv_norm = h->sel_inv.as<float>() + zsel->row_off;
                g.sel_rows = h->sel_rows.as<unsigned char>() + zsel->row_off * h->d_pad * 2; g.sel_cap_rows = zsel->cap_rows;
            }
            int launches = 0;
            if ((tiled ? vb_gemm_tiled_launch(g, &launches) : vb_gemm_launch(g, &launches)) != 0)
                return vb_fail("tensor-core dense kernel: %s", vb_gemm_last_error());
            h->stats.last_launches += (uint32_t)launches;
        } else {
            TRY(launch_scan(h, b, L, r0, r1, direct, sd));
        }
        prof_end(h, pi, sd);
        const int ps = prof_begin(h, PH_SELECT, sd);
        vb_compact_kernel<<<b.B, VB_COMPACT_THREADS, 0, sd>>>(L, b.tau, b.overflow, b.k, 0u, direct ? std::max(direct_rows, L.sub_cap) : L.sub_cap);
        CKK("vb_compact_kernel");
        ++h->stats.last_launches;
        prof_end(h, ps, sd);
        return 0;
    };
    const uint32_t ms_chunk = h->opt_ms_chunk > 0 ? (uint32_t)align_up((size_t)h->opt_ms_chunk, VB_MS_U * VB_MS_THREADS)
                                                   : 512u;
    // classes: bit 0 = plan + score the K3M queries, bit 1 = the K3H (long) queries
    auto ms_launch = [&](uint32_t r0, uint32_t r1, uint64_t stage_lo, uint64_t stage_hi, uint32_t classes) -> int {
        VbMsPlanArgs pa{};
        pa.classes = classes; pa.hunit_prefix = h->mh_units.as<uint32_t>();
        pa.post_row = h->post_row.as<uint32_t>(); pa.term_tab = h->term_tab.as<uint32_t>(); pa.q_tab = b.d_qtab; pa.q_shift = b.d_qshift;
        pa.n_rows = (uint32_t)h->base_rows; pa.q_indptr = b.d_qindptr; pa.q_weight = b.d_qweight; pa.q_ub = b.d_qub;
        pa.q_hidx = b.any_heavy ? b.d_qhidx : nullptr; pa.q_plo = b.d_qplo; pa.q_phi = b.d_qphi; pa.q_ms = b.d_qms; pa.tau = b.tau;
        pa.rec = h->ms_rec.as<VbMsRec>(); pa.qinfo = h->ms_q.as<VbMsQuery>(); pa.unit_prefix = h->ms_units.as<uint32_t>();
        pa.counters = h->ms_counters.as<uint32_t>(); pa.n_queries = b.B; pa.n_qterms = b.n_qterms;
        pa.seg_row0 = r0; pa.seg_row1 = r1; pa.stage_lo = stage_lo; pa.stage_hi = stage_hi;
        pa.chunk = ms_chunk; pa.budget_pct = (uint32_t)std::max<int64_t>(0, h->opt_ms_budget);
        pa.budget_pct_long = (uint32_t)std::max<int64_t>(0, h->opt_mh_budget);
        pa.long_terms = VB_MS_LONG_TERMS; pa.budget_pct_mslong = VB_MS_BUDGET_LONG;
        vb_ms_plan_kernel<<<b.B, 256, 0, ss>>>(pa);
        CKK("vb_ms_plan_kernel");
        ++h->stats.last_launches;
        if (classes & 2u) {
            VbMhArgs m{};
            m.post_row = h->post_row.as<uint32_t>(); m.post_val = h->post_val.as<float>();
            m.heavy_vals = h->heavy_vals.as<float>(); m.heavy_stride = h->heavy_stride; m.term_tab = h->term_tab.as<uint32_t>();
            m.sp_indptr = h->sp_indptr.as<int64_t>(); m.sp_term = h->sp_term.as<uint32_t>(); m.sp_val = h->sp_val.as<float>();
            m.q_indptr = b.d_qindptr; m.q_term = b.d_qterm; m.q_weight = b.d_qweight;
            m.rec = h->ms_rec.as<VbMsRec>(); m.qinfo = h->ms_q.as<VbMsQuery>(); m.hunit_prefix = h->mh_units.as<uint32_t>();
            m.counters = h->ms_counters.as<uint32_t>();
            m.mask = b.use_mask ? h->mask.as<uint32_t>() : nullptr; m.mask_of = b.use_mask ? b.d_maskof : nullptr;
            m.tau = b.tau; m.lists = L; m.mask_words = b.mask_words; m.n_queries = b.B; m.n_rows = (uint32_t)h->base_rows;
            m.row_base = (uint32_t)h->row_base; m.nt_max = b.nt_max; m.seg_row0 = r0; m.seg_row1 = r1;
            const uint64_t max_units = std::max<uint64_t>(1, (uint64_t)h->nnz_live / 256 + b.B);
            const uint32_t grid = (uint32_t)std::min<uint64_t>((uint64_t)h->sm_count * 4u, max_units);
            vb_mh_score_kernel<<<grid, VB_MH_THREADS, vb_mh_smem_bytes(b.nt_max), ss>>>(m);
            CKK("vb_mh_score_kernel");
            ++h->stats.last_launches;
        }
        if (!(classes & 1u)) return 0;
        VbMsArgs a{};
        a.post_row = h->post_row.as<uint32_t>(); a.post_val = h->post_val.as<float>();
        a.heavy_vals = h->heavy_vals.as<float>(); a.heavy_stride = h->heavy_stride;
        a.sp_indptr = h->sp_indptr.as<int64_t>(); a.sp_term = h->sp_term.as<uint32_t>(); a.sp_val = h->sp_val.as<float>();
        a.q_indptr = b.d_qindptr; a.q_term = b.d_qterm; a.q_weight = b.d_qweight; a.slot_q = b.d_slotq;
        a.rec = h->ms_rec.as<VbMsRec>(); a.qinfo = h->ms_q.as<VbMsQuery>(); a.unit_prefix = h->ms_units.as<uint32_t>();
        a.counters = h->ms_counters.as<uint32_t>(); a.term_tab = h->term_tab.as<uint32_t>();
        a.mask = b.use_mask ? h->mask.as<uint32_t>() : nullptr; a.mask_of = b.use_mask ? b.d_maskof : nullptr;
        a.tau = b.tau; a.lists = L; a.mask_words = b.mask_words; a.n_qterms = b.n_qterms; a.n_queries = b.B;
        a.row_base = (uint32_t)h->row_base; a.chunk = ms_chunk; a.nt_max = b.nt_max;
        // persistent grid: enough CTAs to fill the machine (16 per SM: every register of the SM), never more than the
        // largest possible unit count
        const uint64_t span = std::min<uint64_t>(r1 - r0, stage_hi - stage_lo);
        const uint64_t max_units = std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)h->nnz_live / ms_chunk + b.n_qterms, (uint64_t)b.n_qterms * (span / ms_chunk + 1)));
        const uint32_t grid = (uint32_t)std::min<uint64_t>((uint64_t)h->sm_count * 16u, max_units);
        vb_ms_score_kernel<<<grid, VB_MS_THREADS, vb_ms_smem_bytes(b.nt_max), ss>>>(a);
        CKK("vb_ms_score_kernel");
        ++h->stats.last_launches;
        return 0;
    };
    auto sparse_compact = [&](uint32_t lim0) -> int {
        const int ps = prof_begin(h, PH_SELECT, ss);
        vb_compact_kernel<<<b.B, VB_COMPACT_THREADS, 0, ss>>>(L, b.tau, b.overflow, b.k, b.B, lim0);
        CKK("vb_compact_kernel");
        ++h->stats.last_launches;
        prof_end(h, ps, ss);
        return 0;
    };
    // K3 scores: every sparse query if K3M is off; else the queries K3M does not take (b.d_oldq) — plus, in the
    // segment flow, everybody in the direct segment
    auto sparse_segment = [&](uint32_t r0, uint32_t r1_all, uint32_t direct, bool big) -> int {
        const uint32_t r1 = std::min(r1_all, nb);               // the index stops at nb
        const bool rows_here = do_sparse && r0 < r1;
        const bool ms_here = rows_here && ms_on && !ms_staged && !direct;      // K3M once per segment (safe mode / ms_staged = 0)
        const bool mh_here = rows_here && mh_on && !direct;                    // K3H for the long queries
        // K3's queries here: everybody (no K3M / K3H at all, or the direct segment of the per-segment flow); in the
        // direct segment of the staged flow the K3 + K3H queries; otherwise only the ones nobody else takes
        const uint32_t* k3_list = nullptr;
        uint32_t k3_n = b.B;
        if (ms_on || mh_on) {
            if (!direct) { k3_list = b.d_oldq; k3_n = b.n_old; }
            else if (ms_staged) { k3_list = b.d_dirq; k3_n = b.n_dir; }
        }
        const bool k3_here = rows_here && k3_n > 0;
        if (!direct && !ms_here && !mh_here && !k3_here) return 0;             // nothing scored, nothing to compact
        if (ms_here || mh_here || k3_here) {
            const int pi = prof_begin(h, PH_SPARSE | (big ? PH_BIG : 0), ss);
            if (ms_here || mh_here) TRY(ms_launch(r0, r1, 0ull, ~0ull, (ms_here ? 1u : 0u) | (mh_here ? 2u : 0u)));
            if (k3_here) {
                // which terms are essential under the thresholds this segment starts with
                double* d_ubne = h->plan.as<double>();
                uint8_t* d_ess = reinterpret_cast<uint8_t*>(d_ubne + b.B);
                // Pruning pays on long segments (measured: -10..-22 % sparse time from 2M rows per segment up, a loss
                // on cfg2's 1M-row corpus where the per-survivor re-scoring outweighs the skipped postings).
                const uint32_t nblk_seg = (r1 - r0 + VB_ROWS_PER_BLOCK - 1) / VB_ROWS_PER_BLOCK;
                const uint32_t budget = (!direct && (h->opt_sparse_prune_force || nblk_seg >= 1000u)) ? (uint32_t)h->opt_sparse_prune : 0u;
                if (budget) {                                       // no budget: every term is essential, no plan needed
                    vb_sparse_plan_kernel<<<b.B, 256, 0, ss>>>(b.d_qindptr, b.d_qub, b.tau, b.B, budget, d_ess, d_ubne);
                    CKK("vb_sparse_plan_kernel");
                    ++h->stats.last_launches;
                }
                VbSparseArgs a{};
                a.post_row = h->post_row.as<uint32_t>(); a.post_val = h->post_val.as<float>(); a.off = h->offs.as<uint32_t>();
                a.q_indptr = b.d_qindptr; a.q_weight = b.d_qweight; a.q_term = b.d_qterm; a.ess = budget ? d_ess : nullptr; a.ubne = d_ubne;
                a.sp_indptr = h->sp_indptr.as<int64_t>(); a.sp_term = h->sp_term.as<uint32_t>(); a.sp_val = h->sp_val.as<float>();
                a.q_hidx = b.any_heavy ? b.d_qhidx : nullptr; a.q_relaxed = b.d_qrelaxed; a.heavy_vals = h->heavy_vals.as<float>(); a.heavy_stride = h->heavy_stride;
                a.mask = b.use_mask ? h->mask.as<uint32_t>() : nullptr; a.mask_of = b.use_mask ? b.d_maskof : nullptr;
                a.tau = b.tau; a.lists = L; a.mask_words = b.mask_words;
                a.n_qterms = b.n_qterms; a.nt_max = b.nt_max; a.blk_begin = r0 / VB_ROWS_PER_BLOCK; a.n_queries = b.B; a.n_rows = nb;
                a.row_base = (uint32_t)h->row_base; a.direct = direct;
                const uint32_t n_q = k3_n;
                if (k3_list != nullptr) { a.q_sel = k3_list; a.n_sel = k3_n; }          // K3M / K3H have the rest
                const uint32_t nblk = (r1 - r0 + VB_ROWS_PER_BLOCK - 1) / VB_ROWS_PER_BLOCK;
                vb_sparse_kernel<<<nblk * n_q, VB_SPARSE_THREADS, vb_sparse_smem_bytes(b.nt_max), ss>>>(a);
                CKK("vb_sparse_kernel");
                ++h->stats.last_launches;
            }
            prof_end(h, pi, ss);
        }
        // the sparse lists are compacted even without postings (first-segment slots -> empty lists)
        return sparse_compact(direct ? std::max(direct_rows, L.sub_cap) : L.sub_cap);
    };
    // fine (2048-row) slice table rows K3 will read
    const bool k3_all_segments = do_sparse && ((!ms_on && !mh_on) || b.any_old);
    const uint32_t fine_blocks = k3_all_segments ? b.n_blocks
                                 : (k3_direct ? std::min<uint32_t>(b.n_blocks, (direct_rows + VB_ROWS_PER_BLOCK - 1) / VB_ROWS_PER_BLOCK) : 0u);
    if (do_sparse) {
        const uint64_t total = (uint64_t)b.n_qterms * (fine_blocks + 1);
        TRY(dev_reserve(h, h->offs, std::max<uint64_t>(total, 1) * 4, false));
        TRY(dev_reserve(h, h->plan, (size_t)b.B * 8 + b.n_qterms + 64, false));
        if (ms_on || mh_on) {
            TRY(dev_reserve(h, h->mh_units, ((size_t)b.B + 1) * 4, false));
            TRY(dev_reserve(h, h->ms_rec, (size_t)b.n_qterms * sizeof(VbMsRec), false));
            TRY(dev_reserve(h, h->ms_q, (size_t)b.B * sizeof(VbMsQuery), false));
            TRY(dev_reserve(h, h->ms_units, ((size_t)b.n_qterms + 1) * 4, false));
            TRY(dev_reserve(h, h->ms_counters, 64, false));
        }
    }
    if (do_sparse) {                                            // sparse slice tables (sparse chain)
        const int pi = prof_begin(h, PH_SPARSE, ss);
        const uint64_t total = (uint64_t)b.n_qterms * (fine_blocks + 1);
        if (fine_blocks) {
            vb_slice_kernel<<<grid_for(total, 256), 256, 0, ss>>>(h->post_row.as<uint32_t>(), b.d_qlo, b.d_qhi, b.n_qterms, fine_blocks, h->offs.as<uint32_t>());
            CKK("vb_slice_kernel");
            ++h->stats.last_launches;
        }
        if (ms_on || mh_on) CK(cudaMemsetAsync(h->ms_counters.p, 0, 64, ss));
        prof_end(h, pi, ss);
    }
    // K3M stages (normal mode)
    auto ms_stages = [&]() -> int {
        // stage 0 scores its postings with no threshold (every lookup of every posting): just enough of them to fill a
        // list twice over after filters and ownership
        const uint64_t p0 = std::max<uint64_t>(ms_chunk, std::min<uint64_t>(align_up((size_t)8 * b.k, ms_chunk), h->cand_cap / 4));
        uint64_t lo = 0, hi = p0;
        while (lo < b.ms_max_post) {
            const bool last = hi >= b.ms_max_post;
            const int pi = prof_begin(h, PH_SPARSE | (last ? PH_BIG : 0), ss);
            TRY(ms_launch(0u, nb, lo, last ? ~0ull : hi, 1u));
            prof_end(h, pi, ss);
            TRY(sparse_compact(L.sub_cap));
            lo = hi;
            // a stage appends ~ratio * k' candidates per list at worst (rows are visited best-first, usually far fewer)
            const uint64_t ratio = std::min<uint64_t>(1024, std::max<uint64_t>(32, h->cand_cap / (16ull * b.k)));
            hi = hi * ratio;
        }
        return 0;
    };
    // enqueue the two chains interleaved so that neither stream starves on the host side
    const size_t n_seg = bounds.size() - 1;
    size_t big_seg = 0;
    for (size_t s = 1; s < n_seg; ++s) if (bounds[s + 1] - bounds[s] > bounds[big_seg + 1] - bounds[big_seg]) big_seg = s;
    // Order on the sparse stream: K3's direct first segment (fixed slots, counted by the list set-up) and its
    // compaction come BEFORE the K3M stages — a stage's compaction runs over every sparse list and would turn a
    // still-unwritten direct block into an empty list.
    if (k1f) TRY(dense_single_pass());
    for (size_t s = 0; s < n_seg; ++s) {
        const uint32_t direct = (s == 0 && direct_rows) ? 1u : 0u;
        const bool big = s == big_seg;                          // the segment with the most rows: the roofline's launch
        if (big && !k1f) h->stats.last_big_rows = bounds[s + 1] - bounds[s];
        TRY(dense_segment(bounds[s], bounds[s + 1], direct, big));
        TRY(sparse_segment(bounds[s], bounds[s + 1], direct, big));
        if (s == 0 && ms_staged) TRY(ms_stages());
    }
    if (do_delta) {
        // K3D: the rows appended since the index was built, straight from the forward CSR.  One launch (a few
        // thousand rows against thresholds the indexed rows have already established); the safe mode cuts it into
        // pieces a list cannot overflow on.
        const uint32_t piece = safe_mode ? (uint32_t)std::max<size_t>(VB_ROWS_PER_BLOCK, h->cand_cap - b.k) : n - nb;
        for (uint32_t r0 = nb; r0 < n; r0 += piece) {
            const uint32_t r1 = (uint32_t)std::min<uint64_t>(n, (uint64_t)r0 + piece);
            const int pi = prof_begin(h, PH_SPARSE, ss);
            VbDeltaArgs a{};
            a.sp_indptr = h->sp_indptr.as<int64_t>(); a.sp_term = h->sp_term.as<uint32_t>(); a.sp_val = h->sp_val.as<float>();
            a.qt_term = b.d_ut; a.qt_ptr = b.d_up; a.qt_query = b.d_uq; a.qt_weight = b.d_uw;
            a.mask = b.use_mask ? h->mask.as<uint32_t>() : nullptr; a.mask_of = b.use_mask ? b.d_maskof : nullptr;
            a.tau = b.tau; a.lists = L; a.mask_words = b.mask_words; a.n_uterms = b.n_uterms; a.n_queries = b.B;
            a.row_begin = r0; a.row_end = r1; a.row_base = (uint32_t)h->row_base;
            const uint32_t warps = vb_delta_warps(b.B);
            const size_t smem = (size_t)warps * b.B * 8;
            if (smem > (size_t)g_delta_smem_max) return vb_fail("batch of %u queries is too large for the delta rows (%zu bytes of shared memory)", b.B, smem);
            const uint32_t grid = std::min<uint32_t>((r1 - r0 + warps - 1) / warps, (uint32_t)h->sm_count * 8u);
            vb_sparse_delta_kernel<<<grid, warps * 32, smem, ss>>>(a);
            CKK("vb_sparse_delta_kernel");
            ++h->stats.last_launches;
            prof_end(h, pi, ss);
            const int ps = prof_begin(h, PH_SELECT, ss);
            vb_compact_kernel<<<b.B, VB_COMPACT_THREADS, 0, ss>>>(L, b.tau, b.overflow, b.k, b.B, L.sub_cap);
            CKK("vb_compact_kernel");
            ++h->stats.last_launches;
            prof_end(h, ps, ss);
        }
    }
    if (two_streams) {
        CK(cudaEventRecord(h->ev_join, ss));
        CK(cudaStreamWaitEvent(sd, h->ev_join, 0));
    }
    if (sel_any) {                                              // every selected segment is in the scratch now
        h->sel_segs.clear();
        for (size_t si = 0; si < selseg.size(); ++si)
            if (selseg[si].on) h->sel_segs.push_back({bounds[si], bounds[si + 1], selseg[si].row_off, selseg[si].meta_off, selseg[si].cap_rows});
        h->sel_key = std::move(sel_key);
    }
    return 0;
}

// K4 on the (already exact, sorted) branch lists; results stay in h->out on the device.
static int fuse_stage(vb_index* h, const Batch& b) {
    unsigned char* dp = h->out.as<unsigned char>();
    prof_begin(h, PH_FUSE);
    VbFuseArgs f{};
    f.cand = h->cand.as<uint64_t>(); f.cnt = b.cnt; f.mode = b.d_mode; f.cap = h->cand_cap; f.n_queries = b.B;
    f.k = b.k; f.limit = b.limit; f.w_sparse = b.w_sparse; f.w_dense = 1.0 - b.w_sparse;
    f.out_rows = reinterpret_cast<uint32_t*>(dp + b.o_rows); f.out_scores = reinterpret_cast<double*>(dp + b.o_sc);
    f.out_cnt = reinterpret_cast<int32_t*>(dp + b.o_cnt);
    f.overflow = b.overflow; f.out_lcnt = reinterpret_cast<uint32_t*>(dp + b.o_lcnt); f.out_ovf = reinterpret_cast<uint32_t*>(dp + b.o_ovf);
    vb_fuse_kernel<<<b.B, VB_FUSE_THREADS, vb_fuse_smem_bytes(b.k), h->stream>>>(f);
    CKK("vb_fuse_kernel");
    ++h->stats.last_launches;
    if (b.want_branches) {
        vb_export_kernel<<<b.n_lists, 128, 0, h->stream>>>(h->cand.as<uint64_t>(), b.cnt, h->cand_cap, b.k, reinterpret_cast<uint64_t*>(dp + b.o_keys), nullptr, b.n_lists);
        CKK("vb_export_kernel");
        ++h->stats.last_launches;
    }
    prof_end(h);
    CK(cudaEventRecord(h->ev1s[h->cur], h->stream));
    // results go to this slot's pinned buffer right away, so a pipelined caller's fetch does not
    // queue behind the next batch's kernels
    const size_t bytes = b.want_branches ? b.out_bytes : b.o_keys;
    h->stats.last_d2h_bytes = bytes;
    CK(cudaMemcpyAsync(h->h_out_s[h->cur].p, dp, bytes, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaEventRecord(h->ev_done[h->cur], h->stream));
    return 0;
}

// D2H of the result block, sync, decode into the caller's arrays.
// *overflowed = 1 if any list overflowed during scoring (caller re-runs in safe mode).
static int fetch_stage(vb_index* h, const Batch& b, vb_result* out, int* overflowed) {
    unsigned char* hp = h->h_out_s[h->cur].as<unsigned char>();
    CK(cudaEventSynchronize(h->ev_done[h->cur]));
    const uint32_t* ovf = reinterpret_cast<const uint32_t*>(hp + b.o_ovf);
    *overflowed = 0;
    h->stats.last_overflow_lists = 0;
    h->stats.last_overflow_first = 0xffffffffu;
    for (uint32_t i = 0; i < b.n_lists; ++i)
        if (ovf[i]) {
            *overflowed = 1;
            if (h->stats.last_overflow_lists++ == 0) h->stats.last_overflow_first = i;
        }
    if (b.need_corpus) {                                       // flags of the query-prep kernel (a device-resident query is only seen there)
        const uint32_t* bad = reinterpret_cast<const uint32_t*>(hp + b.o_bad);
        for (uint32_t i = 0; i < b.B; ++i)
            if (bad[i]) return vb_fail("Query vector must not contain NaN or inf (query %u of the batch)", i);
    }
    if (*overflowed || !out) return 0;
    const uint32_t* rows = reinterpret_cast<const uint32_t*>(hp + b.o_rows);
    const double* sc = reinterpret_cast<const double*>(hp + b.o_sc);
    const int32_t* cn = reinterpret_cast<const int32_t*>(hp + b.o_cnt);
    for (uint32_t i = 0; i < b.B; ++i) {
        if (out->counts) out->counts[i] = cn[i];
        for (int32_t j = 0; j < cn[i]; ++j) {
            if (out->rows) out->rows[(size_t)i * b.limit + j] = rows[(size_t)i * b.limit + j];
            if (out->scores) out->scores[(size_t)i * b.limit + j] = sc[(size_t)i * b.limit + j];
        }
    }
    if (b.want_branches) {
        const uint64_t* keys = reinterpret_cast<const uint64_t*>(hp + b.o_keys);
        const uint32_t* lc = reinterpret_cast<const uint32_t*>(hp + b.o_lcnt);
        for (uint32_t br = 0; br < 2; ++br) {
            uint64_t* orow = br ? out->sparse_rows : out->dense_rows;
            float* osc = br ? out->sparse_scores : out->dense_scores;
            int32_t* ocn = br ? out->sparse_counts : out->dense_counts;
            for (uint32_t i = 0; i < b.B; ++i) {
                const uint32_t list = br * b.B + i;
                const uint32_t c = std::min(lc[list], b.k);
                if (ocn) ocn[i] = (int32_t)c;
                for (uint32_t j = 0; j < c; ++j) {
                    const uint64_t key = keys[(size_t)list * b.k + j];
                    if (orow) orow[(size_t)i * b.k + j] = vb_key_row(key);
                    if (osc) {
                        const uint32_t bits = vb_ordered_f32((uint32_t)(key >> 32));
                        float sv;
                        memcpy(&sv, &bits, 4);
                        osc[(size_t)i * b.k + j] = sv;
                    }
                }
            }
        }
    }
    return 0;
}

static void finish_stats(vb_index* h, const Batch& b) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, h->ev0s[h->cur], h->ev1s[h->cur]);
    h->stats.last_search_ms = ms;
    h->stats.last_sel_rows = h->sel_ran[h->cur] ? h->h_sel[h->cur].as<uint32_t>()[0] : 0u;
    h->stats.last_sel_used = h->sel_ran[h->cur] ? h->h_sel[h->cur].as<uint32_t>()[1] : 0u;
    h->stats.searches += 1;
    h->stats.queries += b.B;
    if (h->opt_profile) prof_collect(h);
}

static void zero_result(const vb_query_batch* q, vb_result* out) {
    for (uint32_t i = 0; i < q->n_queries; ++i) {
        if (out->counts) out->counts[i] = 0;
        if (out->dense_counts) out->dense_counts[i] = 0;
        if (out->sparse_counts) out->sparse_counts[i] = 0;
    }
}

static bool wants_branches(const vb_result* out) {
    return out && (out->dense_rows || out->dense_scores || out->dense_counts || out->sparse_rows || out->sparse_scores || out->sparse_counts);
}

// ---- staged API: upload once, run the device work asynchronously, fetch ---------------------------
extern "C" int vb_stage(vb_index* h, const vb_query_batch* q, int32_t want_branches, int32_t need_corpus) {
    if (!h) return vb_fail("vb_stage: NULL index");
    TRY(validate_batch(h, q));
    std::lock_guard<std::recursive_mutex> lk(h->mu);
    CK(cudaSetDevice(h->device));
    h->staged_s[h->cur].valid = false;
    TRY(prepare_batch(h, q, h->staged_s[h->cur], need_corpus != 0));
    h->staged_s[h->cur].want_branches = want_branches != 0;
    return 0;
}

extern "C" int vb_run_local(vb_index* h, uint64_t* cand_dev) {
    if (!h) return vb_fail("vb_run_local: NULL index");
    std::lock_guard<std::recursive_mutex> lk(h->mu);
    if (!h->staged_s[h->cur].valid) return vb_fail("vb_run_local: no staged batch");
    if (h->staged_s[h->cur].need_corpus && (h->staged_s[h->cur].n_rows != (uint32_t)h->n_rows || h->staged_s[h->cur].gen != h->write_gen))
        return vb_fail("vb_run_local: the index changed since vb_stage; stage the batch again");
    CK(cudaSetDevice(h->device));
    h->stats.last_launches = 0;
    CK(cudaEventRecord(h->ev0s[h->cur], h->stream));
    if (h->n_rows == 0) {
        TRY(empty_lists(h, h->staged_s[h->cur]));
    } else {
        TRY(run_branches(h, h->staged_s[h->cur], h->staged_safe));
    }
    if (cand_dev) {
        vb_export_kernel<<<h->staged_s[h->cur].n_lists, 128, 0, h->stream>>>(h->cand.as<uint64_t>(), h->staged_s[h->cur].cnt, h->cand_cap, h->staged_s[h->cur].k, cand_dev, h->staged_s[h->cur].overflow, h->staged_s[h->cur].n_lists);
        CKK("vb_export_kernel");
        ++h->stats.last_launches;
    }
    return 0;
}

extern "C" int vb_run_fuse(vb_index* h, uint32_t n_shards, const uint64_t* gathered_dev) {
    if (!h) return vb_fail("vb_run_fuse: NULL index");
    std::lock_guard<std::recursive_mutex> lk(h->mu);
    Batch& b = h->staged_s[h->cur];
    if (!b.valid) return vb_fail("vb_run_fuse: no staged batch");
    CK(cudaSetDevice(h->device));
    if (gathered_dev) {
        if (n_shards == 0 || (uint64_t)n_shards * b.k > h->cand_cap) return vb_fail("vb_run_fuse: n_shards*kprime out of range");
        prof_begin(h, PH_SELECT);
        vb_import_kernel<<<b.n_lists, 256, 0, h->stream>>>(gathered_dev, n_shards, b.n_lists, b.k, h->cand_cap, h->cand.as<uint64_t>(), b.cnt, b.overflow);
        CKK("vb_import_kernel");
        vb_compact_kernel<<<b.n_lists, VB_COMPACT_THREADS, 0, h->stream>>>(make_lists(h, b, true), b.tau, b.overflow, b.k, 0u, h->cand_cap);
        CKK("vb_compact_kernel");
        h->stats.last_launches += 2;
        prof_end(h);
    }
    TRY(fuse_stage(h, b));
    return 0;
}

extern "C" int vb_fetch(vb_index* h, vb_result* out, int32_t* overflowed) {
    if (!h) return vb_fail("vb_fetch: NULL index");
    std::lock_guard<std::recursive_mutex> lk(h->mu);
    if (!h->staged_s[h->cur].valid) return vb_fail("vb_fetch: no staged batch");
    CK(cudaSetDevice(h->device));
    int ovf = 0;
    TRY(fetch_stage(h, h->staged_s[h->cur], out, &ovf));
    finish_stats(h, h->staged_s[h->cur]);
    if (overflowed) *overflowed = ovf;
    return 0;
}

// ---- one-call API ------------------------------------------------------------------------------------
extern "C" int vb_search(vb_index* h, const vb_query_batch* q, vb_result* out) {
    if (!h || !out) return vb_fail("vb_search: NULL argument");
    TRY(validate_batch(h, q));
    std::lock_guard<std::recursive_mutex> lk(h->mu);      // stage + run + fuse + fetch are one critical section
    if (h->n_rows == 0) { zero_result(q, out); return 0; }
    for (int attempt = 0; attempt < 2; ++attempt) {
        TRY(vb_stage(h, q, wants_branches(out), 1));
        h->staged_safe = attempt == 1;
        int rc = vb_run_local(h, nullptr);
        h->staged_safe = false;
        TRY(rc);
        TRY(vb_run_fuse(h, 0, nullptr));
        int32_t overflowed = 0;
        TRY(vb_fetch(h, out, &overflowed));
        if (!overflowed) return 0;
        if (attempt == 1) return vb_fail("vb_search: candidate list overflow even in safe mode (internal error)");
        ++h->stats.overflow_reruns;
    }
    return 0;
}

// ---- device-resident queries (SURVEY §8 f-4) ------------------------------------------------------------
// The embedding model's output (embedding.py:76-86) stays on the GPU: same calls, but the dense rows come from
// `dense_dev` (fp32 [B][dim] on this index's device; q->dense is ignored and may be NULL).  The library orders its
// copy after the work queued on `producer_stream` (a cudaStream_t; NULL = the legacy default stream) — no host sync.
struct QDevScope {
    vb_index* h;
    QDevScope(vb_index* h_, const float* p, void* s) : h(h_) { h->q_dev = p; h->q_dev_stream = (cudaStream_t)s; }
    ~QDevScope() { h->q_dev = nullptr; h->q_dev_stream = nullptr; }
};

static int check_dev_queries(vb_index* h, const float* dense_dev) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, dense_dev) != cudaSuccess || (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged)) {
        cudaGetLastError();
        return vb_fail("dense_dev is not a device pointer");
    }
    if (at.type == cudaMemoryTypeDevice && at.device != h->device) return vb_fail("dense_dev lives on device %d, the index on device %d", at.device, h->device);
    return 0;
}

extern "C" int vb_stage_dev(vb_index* h, const vb_query_batch* q, const float* dense_dev, void* producer_stream, int32_t want_branches, int32_t need_corpus) {
    if (!h || !dense_dev) return vb_fail("vb_stage_dev: NULL argument");
    std::lock_guard<std::recursive_mutex> lk(h->mu);
    CK(cudaSetDevice(h->device));
    TRY(check_dev_queries(h, dense_dev));
    QDevScope scope(h, dense_dev, producer_stream);
    return vb_stage(h, q, want_branches, need_corpus);
}

extern "C" int vb_search_dev(vb_index* h, const vb_query_batch* q, const float* dense_dev, void* producer_stream, vb_result* out) {
    if (!h || !dense_dev || !out) return vb_fail("vb_search_dev: NULL argument");
    std::lock_guard<std::recursive_mutex> lk(h->mu);
    CK(cudaSetDevice(h->device));
    TRY(check_dev_queries(h, dense_dev));
    QDevScope scope(h, dense_dev, producer_stream);
    return vb_search(h, q, out);
}

extern "C" int vb_search_local(vb_index* h, const vb_query_batch* q, uint64_t* cand_dev) {
    if (!h || !cand_dev) return vb_fail("vb_search_local: NULL argument");
    TRY(validate_batch(h, q));
    if (q->apply_idf) return vb_fail("vb_search_local: weights must carry the global IDF (apply_idf = 0)");
    std::lock_guard<std::recursive_mutex> lk(h->mu);
    for (int attempt = 0; attempt < 2; ++attempt) {
        TRY(vb_stage(h, q, 0, 1));
        h->staged_safe = attempt == 1;
        int rc = vb_run_local(h, cand_dev);
        h->staged_safe = false;
        TRY(rc);
        // overflow flags
        TRY(host_reserve(h->h_stage, (size_t)h->staged_s[h->cur].n_lists * 4));
        CK(cudaMemcpyAsync(h->h_stage.p, h->staged_s[h->cur].overflow, (size_t)h->staged_s[h->cur].n_lists * 4, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaEventRecord(h->ev1s[h->cur], h->stream));
        CK(cudaStreamSynchronize(h->stream));
        finish_stats(h, h->staged_s[h->cur]);
        bool ovf = false;
        for (uint32_t i = 0; i < h->staged_s[h->cur].n_lists; ++i) ovf |= h->h_stage.as<uint32_t>()[i] != 0;
        if (!ovf) return 0;
        if (attempt == 1) return vb_fail("vb_search_local: candidate list overflow even in safe mode (internal error)");
        ++h->stats.overflow_reruns;
    }
    return 0;
}

extern "C" int vb_merge_fuse(vb_index* h, const vb_query_batch* q, uint32_t n_shards, const uint64_t* gathered_dev, vb_result* out) {
    if (!h || !gathered_dev || !out) return vb_fail("vb_merge_fuse: NULL argument");
    TRY(validate_batch(h, q));
    std::lock_guard<std::recursive_mutex> lk(h->mu);
    TRY(vb_stage(h, q, wants_branches(out), 0));
    CK(cudaEventRecord(h->ev0s[h->cur], h->stream));
    h->stats.last_launches = 0;
    TRY(empty_lists(h, h->staged_s[h->cur]));
    TRY(vb_run_fuse(h, n_shards, gathered_dev));
    int32_t overflowed = 0;
    TRY(vb_fetch(h, out, &overflowed));
    if (overflowed) return vb_fail("vb_merge_fuse: unexpected overflow");
    return 0;
}

// ------------------------------------------------------------------------------------------------
// snapshot (replaces Qdrant's on-disk storage for this path)
// ------------------------------------------------------------------------------------------------
struct VbSnapHeader {
    char magic[8];                 // "VB200SNP"
    uint32_t version, dim, d_pad, flags;     // flags: bit0 any_ts_created, bit1 any_ts_modified
    uint64_t row_base, n_rows, n_live, nnz;
};

static int snap_write_dev(vb_index* h, FILE* f, const void* dev, size_t bytes) {
    const size_t chunk = 32u << 20;
    TRY(host_reserve(h->h_stage, std::min(bytes, chunk)));
    for (size_t o = 0; o < bytes; o += chunk) {
        const size_t m = std::min(chunk, bytes - o);
        CK(cudaMemcpyAsync(h->h_stage.p, static_cast<const char*>(dev) + o, m, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        if (fwrite(h->h_stage.p, 1, m, f) != m) return vb_fail("vb_save: short write");
    }
    return 0;
}
template <class Check>
static int snap_read_dev(vb_index* h, FILE* f, void* dev, size_t bytes, Check check) {
    const size_t chunk = 32u << 20;
    TRY(host_reserve(h->h_stage, std::min(bytes, chunk)));
    for (size_t o = 0; o < bytes; o += chunk) {
        const size_t m = std::min(chunk, bytes - o);
        if (fread(h->h_stage.p, 1, m, f) != m) return vb_fail("vb_load: snapshot truncated");
        check(h->h_stage.p, m);
        CK(cudaMemcpyAsync(static_cast<char*>(dev) + o, h->h_stage.p, m, cudaMemcpyHostToDevice, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    return 0;
}

static int snap_read_dev(vb_index* h, FILE* f, void* dev, size_t bytes) {
    return snap_read_dev(h, f, dev, bytes, [](const void*, size_t) {});
}

extern "C" int vb_save(vb_index* h, const char* path) {
    if (!h || !path) return vb_fail("vb_save: NULL argument");
    std::lock_guard<std::recursive_mutex> lk(h->mu);
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    FILE* f = fopen(path, "wb");
    if (!f) return vb_fail("vb_save: cannot open '%s' for writing", path);
    VbSnapHeader hd{};
    memcpy(hd.magic, "VB200SNP", 8);
    hd.version = 1; hd.dim = (uint32_t)h->dim; hd.d_pad = (uint32_t)h->d_pad;
    hd.flags = (h->any_ts_created ? 1u : 0u) | (h->any_ts_modified ? 2u : 0u);
    hd.row_base = h->row_base; hd.n_rows = h->n_rows; hd.n_live = h->n_live; hd.nnz = h->nnz;
    int rc = fwrite(&hd, sizeof hd, 1, f) == 1 ? 0 : vb_fail("vb_save: short write");
    const uint64_t n = h->n_rows, words = (n + 31) / 32;
    if (!rc && n) {
        rc = snap_write_dev(h, f, h->rows.p, n * h->d_pad * 2);
        if (!rc) rc = snap_write_dev(h, f, h->inv_norm.p, n * 4);
        if (!rc) rc = snap_write_dev(h, f, h->scope_id.p, n * 4);
        if (!rc) rc = snap_write_dev(h, f, h->created.p, n * 8);
        if (!rc) rc = snap_write_dev(h, f, h->modified.p, n * 8);
        if (!rc && fwrite(h->alive_host.data(), 4, words, f) != words) rc = vb_fail("vb_save: short write");
        if (!rc) rc = snap_write_dev(h, f, h->sp_indptr.p, (n + 1) * 8);
        if (!rc && h->nnz) rc = snap_write_dev(h, f, h->sp_term.p, h->nnz * 4);
        if (!rc && h->nnz) rc = snap_write_dev(h, f, h->sp_val.p, h->nnz * 4);
    }
    // the caller renames the file into place afterwards: the data must be on disk first
    if (!rc && (fflush(f) != 0 || fsync(fileno(f)) != 0)) rc = vb_fail("vb_save: flush/fsync failed");
    if (fclose(f) != 0 && !rc) rc = vb_fail("vb_save: close failed");
    return rc;
}

extern "C" int vb_load(const char* path, int32_t device, vb_index** out) {
    if (!path || !out) return vb_fail("vb_load: NULL argument");
    *out = nullptr;
    FILE* f = fopen(path, "rb");
    if (!f) return vb_fail("vb_load: cannot open '%s'", path);
    VbSnapHeader hd{};
    if (fread(&hd, sizeof hd, 1, f) != 1 || memcmp(hd.magic, "VB200SNP", 8) != 0 || hd.version != 1) {
        fclose(f);
        return vb_fail("vb_load: '%s' is not a version-1 snapshot", path);
    }
    // the header must describe exactly this file: nothing below trusts a count it has not checked
    {
        const uint64_t n = hd.n_rows, words = (n + 31) / 32;
        if (hd.dim == 0 || hd.dim > 4096 || hd.d_pad != (hd.dim + 63) / 64 * 64 || hd.n_live > n || hd.nnz >= (1ull << 40) ||
            n + hd.row_base > 0xffffffffull) {
            fclose(f);
            return vb_fail("vb_load: '%s' has an implausible header", path);
        }
        uint64_t want = sizeof hd;
        if (n) want += n * hd.d_pad * 2 + n * 4 + n * 4 + n * 8 + n * 8 + words * 4 + (n + 1) * 8 + hd.nnz * 8;
        if (fseek(f, 0, SEEK_END) != 0) { fclose(f); return vb_fail("vb_load: cannot seek in '%s'", path); }
        const long long have = ftell(f);
        if (have < 0 || (uint64_t)have != want) {
            fclose(f);
            return vb_fail("vb_load: '%s' is %lld bytes, its header describes %llu", path, have, (unsigned long long)want);
        }
        if (fseek(f, (long)sizeof hd, SEEK_SET) != 0) { fclose(f); return vb_fail("vb_load: cannot seek in '%s'", path); }
    }
    vb_index* h = nullptr;
    int rc = vb_create((int32_t)hd.dim, device, hd.n_rows, hd.row_base, &h);
    if (rc) { fclose(f); return rc; }
    auto body = [&]() -> int {
        if ((uint32_t)h->d_pad != hd.d_pad) return vb_fail("vb_load: snapshot row pitch %u != %d", hd.d_pad, h->d_pad);
        const uint64_t n = hd.n_rows, words = (n + 31) / 32;
        if (n == 0) return 0;
        std::lock_guard<std::recursive_mutex> lk(h->mu);
        TRY(reserve_rows(h, n, hd.nnz));
        TRY(snap_read_dev(h, f, h->rows.p, n * h->d_pad * 2));
        TRY(snap_read_dev(h, f, h->inv_norm.p, n * 4));
        TRY(snap_read_dev(h, f, h->scope_id.p, n * 4));
        TRY(snap_read_dev(h, f, h->created.p, n * 8));
        TRY(snap_read_dev(h, f, h->modified.p, n * 8));
        if (fread(h->alive_host.data(), 4, words, f) != words) return vb_fail("vb_load: snapshot truncated");
        // bits past n_rows never count; n_live is recomputed from the bitmap, not taken from the header
        if (n & 31u) h->alive_host[words - 1] &= (1u << (n & 31u)) - 1u;
        uint64_t live = 0;
        for (uint64_t w = 0; w < words; ++w) live += (uint64_t)__builtin_popcount(h->alive_host[w]);
        if (live != hd.n_live) return vb_fail("vb_load: header says %llu live rows, the bitmap holds %llu", (unsigned long long)hd.n_live, (unsigned long long)live);
        CK(cudaMemcpyAsync(h->alive.p, h->alive_host.data(), words * 4, cudaMemcpyHostToDevice, h->stream));
        {   // forward index offsets: monotone, starting at 0, ending at nnz (checked on their way through the staging buffer)
            int64_t prev = 0;
            bool first = true, ok = true;
            TRY(snap_read_dev(h, f, h->sp_indptr.p, (n + 1) * 8, [&](const void* p, size_t bytes) {
                const int64_t* v = static_cast<const int64_t*>(p);
                for (size_t i = 0; i < bytes / 8; ++i) {
                    if (first) { ok = ok && v[i] == 0; first = false; }
                    ok = ok && v[i] >= prev;
                    prev = v[i];
                }
            }));
            if (!ok || prev != (int64_t)hd.nnz) return vb_fail("vb_load: corrupt sparse offsets (not monotone from 0 to nnz)");
        }
        if (hd.nnz) { TRY(snap_read_dev(h, f, h->sp_term.p, hd.nnz * 4)); TRY(snap_read_dev(h, f, h->sp_val.p, hd.nnz * 4)); }
        CK(cudaStreamSynchronize(h->stream));
        h->n_rows = n; h->n_live = hd.n_live; h->nnz = hd.nnz;
        h->any_ts_created = hd.flags & 1u; h->any_ts_modified = (hd.flags & 2u) != 0;
        h->sparse_dirty = true;
        return 0;
    };
    rc = body();
    fclose(f);
    if (rc) { vb_destroy(h); return rc; }
    *out = h;
    return 0;
}
