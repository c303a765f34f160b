// K3 — sparse (BM25-style) scoring over an inverted index staged through shared memory.
// Replaces qdrant's sparse dot product with the IDF modifier for
// query_points(query=SparseVector, using="bm25", limit=k', query_filter)
// (vector_store.py:647-656; sparse_distances.py sparse_dot_product in local mode).
//
// Index layout (built on the device from the row-major CSR the upserts append):
//   postings sorted by (term, row):  post_row[nnz] u32, post_val[nnz] f32
//   terms_sorted[T] u32 (distinct hashed term ids), term_ptr[T+1] u64
// Rows are cut into blocks of VB_ROWS_PER_BLOCK rows.  For a batch, vb_slice_kernel finds,
// for every query term and every row block, the slice of that term's postings that falls in
// the block (binary search on post_row).  vb_sparse_kernel then gives one CTA a (row block,
// query) pair: fp64 accumulators for the block's rows live in shared memory, the query's terms
// are walked in ascending term-id order and each slice is streamed with coalesced loads.
// Inside one term a row occurs at most once, so no atomics are needed and the summation
// order (ascending term id, explicit mul then add in fp64, one final rounding to fp32) is
// exactly the order of the reference's two-pointer merge: sparse scores are bit-identical to
// np.float32(sum of python floats).  Rows never touched keep a sentinel: "no shared index"
// rows are excluded, as in the reference.
// Roofline: HBM (L2 for slices shared by queries of the batch).
// Algorithmic bytes = sum over queries, terms: df_shard(term) * 8.
#pragma once
#include "common.cuh"
#include <cub/cub.cuh>

#define VB_ACC_SENTINEL 0x8000000000000000ull   // -0.0: no sum can produce it (see vb_sparse_kernel)

// ---- index build ------------------------------------------------------------------------------
// key = term << 32 | row for live rows, ~0 for tombstoned rows (sorted to the tail, then cut).
__global__ void __launch_bounds__(256)
vb_posting_keys_kernel(const int64_t* __restrict__ indptr, const uint32_t* __restrict__ term,
                       const uint32_t* __restrict__ alive, uint32_t n_rows, uint64_t* __restrict__ keys)
{
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n_rows; r += warps) {
        const int64_t lo = indptr[r], hi = indptr[r + 1];
        const bool live = (alive[r >> 5] >> (r & 31u)) & 1u;
        for (int64_t p = lo + lane; p < hi; p += 32)
            keys[p] = live ? (((uint64_t)term[p] << 32) | r) : ~0ull;
    }
}

// After the sort: split keys into post_row, flag term starts.
__global__ void __launch_bounds__(256)
vb_posting_split_kernel(const uint64_t* __restrict__ keys, uint64_t nnz, uint32_t* __restrict__ post_row,
                        uint32_t* __restrict__ post_term)
{
    for (uint64_t p = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; p < nnz; p += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t k = keys[p];
        post_row[p] = (uint32_t)k;
        post_term[p] = (uint32_t)(k >> 32);
    }
}

// Dense column of a frequent term: out[row] = the term's value in that row (out is pre-filled with NaN).
__global__ void __launch_bounds__(256)
vb_heavy_fill_kernel(const uint32_t* __restrict__ post_row, const float* __restrict__ post_val, uint64_t lo, uint64_t hi,
                     float* __restrict__ out)
{
    for (uint64_t p = lo + blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; p < hi; p += (uint64_t)gridDim.x * blockDim.x)
        out[post_row[p]] = post_val[p];
}

// ---- per-batch slice table ----------------------------------------------------------------------
// off[b][j] = first posting of query-term j whose row >= b*VB_ROWS_PER_BLOCK  (b = 0..n_blocks),
// block-major so that the CTA of (row block, query) reads its terms' bounds as two contiguous runs.
// Posting offsets fit 32 bits (a shard holds < 2^31 postings).
__global__ void __launch_bounds__(256)
vb_slice_kernel(const uint32_t* __restrict__ post_row, const uint32_t* __restrict__ qt_lo,
                const uint32_t* __restrict__ qt_hi, uint32_t n_qterms, uint32_t n_blocks,
                uint32_t* __restrict__ off)
{
    const uint64_t total = (uint64_t)n_qterms * (n_blocks + 1u);
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t b = (uint32_t)(i / n_qterms);
        const uint32_t j = (uint32_t)(i % n_qterms);
        uint32_t lo = qt_lo[j], hi = qt_hi[j];
        const uint64_t target = (uint64_t)b * VB_ROWS_PER_BLOCK;
        while (lo < hi) {
            const uint32_t mid = lo + ((hi - lo) >> 1);
            if ((uint64_t)post_row[mid] < target) lo = mid + 1; else hi = mid;
        }
        off[i] = lo;
    }
}

struct VbSparseArgs {
    const uint32_t* post_row;
    const float* post_val;
    const uint32_t* off;        // [n_blocks+1][n_qterms]
    const int64_t* q_indptr;    // [B+1] into the sorted query-term arrays
    const double* q_weight;     // [n_qterms] idf-scaled query values, ascending term id per query
    const uint32_t* q_term;     // [n_qterms] term ids (ascending per query)
    const uint8_t* ess;         // [n_qterms] 1 = essential term for the current thresholds; nullptr = all
    const double* ubne;         // [B] sum of the upper bounds of the query's non-essential terms
    const int32_t* q_hidx;      // [n_qterms] dense-column index of the term for this query, -1 = scored from postings
    const uint8_t* q_relaxed;   // [B] 1 = all products of this query are >= 0: order-free accumulation + verification allowed
    const float* heavy_vals;    // [n_heavy][heavy_stride] value of the term in each row, NaN = absent
    uint32_t heavy_stride;
    const int64_t* sp_indptr;   // forward index (row-major CSR as appended), for exact re-scoring
    const uint32_t* sp_term;
    const float* sp_val;
    const uint32_t* mask;       // [n_filters][mask_words] or nullptr
    const int32_t* mask_of;     // [B] or nullptr
    const float* tau;
    VbLists lists;
    uint32_t mask_words;
    uint32_t n_qterms;          // query terms of the whole batch (row length of `off`)
    uint32_t nt_max;            // most terms of any query of the batch (sizes the shared term table)
    uint32_t blk_begin;         // first row block of this segment
    uint32_t n_queries;
    uint32_t n_rows;
    uint32_t row_base;
    uint32_t direct;            // 1: first segment — store keys at slot (row - segment begin), no atomics
    const uint32_t* q_sel;      // [n_sel] queries this launch scores (the rest go to K3M, sparse_ms.cuh); nullptr = all
    uint32_t n_sel;
};

// ---- MaxScore plan: which query terms are essential under the current thresholds --------------------
// ub[j] >= the largest contribution term j can make to any row of this shard (weight x the term's
// largest posting value; +inf = "always essential").  Sorting a query's terms by ub, the longest
// prefix whose ub sum stays below a fixed share of tau is NON-essential: a row that contains only such terms cannot
// beat tau, so the scoring kernel scatters only the essential terms' postings, drops every row
// whose partial score + (sum of non-essential ubs) is still below tau, and re-scores the few
// survivors exactly.  One CTA per query, launched before every sparse segment (tau moves).
// The 1e-9 relative margins dwarf the fp64 rounding of the sums involved (<= 256 terms, ~3e-14).
__global__ void __launch_bounds__(256)
vb_sparse_plan_kernel(const int64_t* __restrict__ q_indptr, const double* __restrict__ q_ub, const float* __restrict__ tau,
                      uint32_t n_queries, uint32_t budget_pct, uint8_t* __restrict__ ess, double* __restrict__ ubne)
{
    __shared__ double s_ub[256];
    __shared__ double s_red[8];
    const uint32_t q = blockIdx.x, j = threadIdx.x;
    const uint32_t t_lo = (uint32_t)q_indptr[q];
    const uint32_t nt = (uint32_t)q_indptr[q + 1] - t_lo;
    const double tau_d = (double)tau[n_queries + q];
    const double ub = j < nt ? q_ub[t_lo + j] : INFINITY;
    s_ub[j] = ub;
    __syncthreads();
    double cum = 0.0;                                           // ub sum of the sorted prefix that ends with term j
    for (uint32_t i = 0; i < nt; ++i) {
        const double u = s_ub[i];
        if (u < ub || (u == ub && i <= j)) cum += u;
    }
    // budget: the non-essential ubs may sum to at most budget_pct % of tau.  A small budget already
    // covers the most frequent (lowest-idf, longest) posting lists while keeping the survivor test
    // partial >= tau - sum(ub) selective, so that few rows need exact re-scoring.
    const bool ok = budget_pct != 0u && tau_d > 0.0 && tau_d < INFINITY;
    const bool ne = ok && j < nt && ub < INFINITY && cum < tau_d * (0.01 * (double)min(budget_pct, 100u)) * (1.0 - 2e-9);
    if (j < nt) ess[t_lo + j] = ne ? 0 : 1;
    double m = ne ? cum : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((j & 31u) == 0) s_red[j >> 5] = m;
    __syncthreads();
    if (j == 0) {
        for (uint32_t w = 1; w < 8; ++w) m = fmax(m, s_red[w]);
        ubne[q] = m;
    }
}

#define VB_SPARSE_THREADS 128
#define VB_SPARSE_U 2u                                          // postings per thread per batch
#define VB_SPARSE_BATCH (VB_SPARSE_U * VB_SPARSE_THREADS)       // 512 postings per batch
#define VB_SPARSE_PAD 32u                                       // dummy accumulators for padding lanes

static size_t vb_sparse_smem_bytes(uint32_t nt_max) {
    return (size_t)(VB_ROWS_PER_BLOCK + VB_SPARSE_PAD) * 8u + (size_t)VB_ROWS_PER_BLOCK * 2u + (size_t)nt_max * 27u + 48u;
}

// grid.x = (#blocks in segment) * B ; CTA (blk, q) with q fastest so that concurrently running
// CTAs share a row block (and the posting slices of common terms hit L2).
//
// One CTA's work is small (a few thousand postings in ~6 non-empty slices, 2048 fp64
// accumulators); the kernel is bound by memory latency and instruction issue, not bandwidth:
//   * the slice bounds of all the query's terms for this block arrive in one parallel step
//     (block-major slice table) and only the non-empty terms are kept, in ascending term id;
//   * postings are fetched in batches of 512 (4 per thread, all loads issued back to back), and the
//     batch after the current one — the rest of the slice or the head of the NEXT term's slice —
//     is already in flight while the current one is accumulated, so the L2/HBM latency is paid
//     about once per CTA instead of once per term;
//   * padding lanes accumulate into private dummy slots, so the accumulate code is branch-free;
//   * terms are applied in ascending term id with one barrier between terms (within a term a row
//     occurs once: no atomics).  That is the summation order of the reference's two-pointer
//     merge, and the arithmetic is explicit fp64 mul, add.
//   accumulators start at -0.0 and every product is canonicalised with "+ 0.0", so
//   acc = acc + (w*v + 0.0) reproduces Python's `result = 0.0; result += w*v` bit for bit (the only
//   differences would involve -0.0, which both sides turn into +0.0) while an untouched row is
//   still recognisable (-0.0 can never be a sum).
__global__ void __launch_bounds__(VB_SPARSE_THREADS, 9)
vb_sparse_kernel(const VbSparseArgs a)
{
    extern __shared__ __align__(16) unsigned char vb_sp_smem[];
    double* acc = reinterpret_cast<double*>(vb_sp_smem);                    // [VB_ROWS_PER_BLOCK + VB_SPARSE_PAD]
    double* s_w = acc + VB_ROWS_PER_BLOCK + VB_SPARSE_PAD;                  // [nt_max]
    uint32_t* s_lo = reinterpret_cast<uint32_t*>(s_w + a.nt_max);           // [nt_max]
    uint32_t* s_hi = s_lo + a.nt_max;                                       // [nt_max]
    uint16_t* s_surv = reinterpret_cast<uint16_t*>(s_hi + a.nt_max);        // [VB_ROWS_PER_BLOCK] rows to re-score
    uint16_t* s_nz = s_surv + VB_ROWS_PER_BLOCK;                            // [nt_max] non-empty ESSENTIAL terms, ascending
    uint16_t* s_all = s_nz + a.nt_max;                                      // [nt_max] all non-empty terms, ascending
    uint16_t* s_hv = s_all + a.nt_max;                                      // [nt_max] terms scored from their dense column
    uint32_t* s_cum = reinterpret_cast<uint32_t*>(s_hv + a.nt_max + (a.nt_max & 1u));   // [nt_max + 1] posting prefix sums over s_nz
    uint8_t* s_flag = reinterpret_cast<uint8_t*>(s_cum + a.nt_max + 1u);                // [nt_max] bit0 postings here, bit1 essential, bit2 dense column
    __shared__ uint32_t s_nsurv;

    const uint32_t tid = threadIdx.x;
    const uint32_t n_q = a.q_sel != nullptr ? a.n_sel : a.n_queries;
    const uint32_t q = a.q_sel != nullptr ? __ldg(a.q_sel + blockIdx.x % n_q) : blockIdx.x % n_q;
    const uint32_t blk_rel = blockIdx.x / n_q;
    const uint32_t blk = a.blk_begin + blk_rel;
    const uint32_t t_lo = (uint32_t)__ldg(a.q_indptr + q);
    const uint32_t nt = (uint32_t)__ldg(a.q_indptr + q + 1) - t_lo;
    VB_CHECK(q < a.n_queries && nt <= a.nt_max && (size_t)(blk + 1u) * VB_ROWS_PER_BLOCK <= (size_t)a.n_rows + VB_ROWS_PER_BLOCK);
    if (nt == 0) return;                                        // dense-only query

    // Term table: every warp builds it by itself (lane = term, 32 terms per step) and all warps store the
    // same values, so the four warps never wait for one of them and a single barrier (after the accumulator
    // initialisation below) publishes everything.
    const uint32_t lane = tid & 31u;
    auto load_term = [&](uint32_t j, uint32_t& lo, uint32_t& hi, uint32_t& fl, double& w) {
        lo = hi = fl = 0u; w = 0.0;
        if (j < nt) {
            lo = __ldg(a.off + (size_t)blk * a.n_qterms + t_lo + j);
            hi = __ldg(a.off + (size_t)(blk + 1u) * a.n_qterms + t_lo + j);
            w = __ldg(a.q_weight + t_lo + j);
            const bool es = a.ess == nullptr || __ldg(a.ess + t_lo + j) != 0;
            const bool hv = a.q_hidx != nullptr && __ldg(a.q_hidx + t_lo + j) >= 0;
            fl = (es ? 2u : 0u) | (hv ? 4u : 0u);
        }
    };
    uint32_t lo_c, hi_c, fl_c;
    double w_c;
    load_term(lane, lo_c, hi_c, fl_c, w_c);                     // first 32 terms: in flight during the initialisation
    const uint32_t list = a.n_queries + q;                      // sparse lists follow the dense ones
    const float tau = a.tau[list];
    const uint32_t* mask = nullptr;
    if (a.mask != nullptr && a.mask_of != nullptr) {
        const int32_t f = __ldg(a.mask_of + q);
        if (f >= 0) mask = a.mask + (size_t)f * a.mask_words;
    }
    const double neg_zero = __longlong_as_double((long long)VB_ACC_SENTINEL);
#pragma unroll
    for (uint32_t r = 2u * tid; r < VB_ROWS_PER_BLOCK + VB_SPARSE_PAD; r += 2u * VB_SPARSE_THREADS)
        *reinterpret_cast<double2*>(&acc[r]) = make_double2(neg_zero, neg_zero);
    uint32_t nnz = 0, n_all = 0, nh = 0;                        // essential terms with postings here / terms that can touch
    {                                                           // this block / essential terms read from a dense column
        uint32_t cum_base = 0;
        if (lane == 0) { s_cum[0] = 0u; if (tid == 0) s_nsurv = 0u; }
        for (uint32_t j0 = 0; j0 < nt; j0 += 32u) {
            const uint32_t j = j0 + lane;
            if (j0 != 0u) load_term(j, lo_c, hi_c, fl_c, w_c);
            if (j < nt) { s_lo[j] = lo_c; s_hi[j] = hi_c; s_w[j] = w_c; }
            const bool ne = hi_c > lo_c;                                             // postings in this block
            const bool es = ne && (fl_c & 2u);                                       // ... of an essential term
            const bool hv = (fl_c & 6u) == 6u;                                       // essential term with a dense column
            n_all += __popc(__ballot_sync(0xffffffffu, ne)) + __popc(__ballot_sync(0xffffffffu, (fl_c & 6u) == 4u));
            const uint32_t bal = __ballot_sync(0xffffffffu, es);
            const uint32_t bal_hv = __ballot_sync(0xffffffffu, hv);
            uint32_t incl = es ? hi_c - lo_c : 0u;                                   // running posting count over s_nz
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= (uint32_t)o) incl += t;
            }
            if (es) {
                const uint32_t k = nnz + __popc(bal & ((1u << lane) - 1u));
                s_nz[k] = (uint16_t)j;
                s_cum[k + 1u] = cum_base + incl;
            }
            cum_base += __shfl_sync(0xffffffffu, incl, 31);
            if (hv) s_hv[nh + __popc(bal_hv & ((1u << lane) - 1u))] = (uint16_t)j;
            nnz += __popc(bal);
            nh += __popc(bal_hv);
        }
    }
    __syncthreads();
    if (nnz == 0 && nh == 0) return;

    const uint32_t row0 = blk * VB_ROWS_PER_BLOCK;
    const uint32_t dummy = VB_ROWS_PER_BLOCK + (tid & 31u);     // this lane's private padding slot
    const uint32_t* __restrict__ prow = a.post_row;
    const float* __restrict__ pval = a.post_val;

    // fetch: postings p0 + tid + 128*u (u < 4) of a slice ending at hi; padding lanes get the dummy slot
    auto fetch = [&](uint32_t p0, uint32_t hi, uint32_t (&fr)[VB_SPARSE_U], float (&fv)[VB_SPARSE_U]) {
#pragma unroll
        for (uint32_t u = 0; u < VB_SPARSE_U; ++u) {
            const uint32_t p = p0 + tid + u * VB_SPARSE_THREADS;
            const bool ok = p < hi;
            fr[u] = ok ? __ldg(prow + p) : row0 + dummy;
            fv[u] = ok ? __ldg(pval + p) : 0.0f;
        }
    };
    // accumulate one batch; u-groups past the end of the slice are skipped (uniform per warp)
    auto rmw = [&](uint32_t p0, uint32_t hi, double w, const uint32_t (&fr)[VB_SPARSE_U], const float (&fv)[VB_SPARSE_U]) {
        const uint32_t wbase = p0 + (tid & ~31u);
#pragma unroll
        for (uint32_t u = 0; u < VB_SPARSE_U; ++u) {
            if (wbase + u * VB_SPARSE_THREADS < hi) {
                const uint32_t r = fr[u] - row0;
                acc[r] = __dadd_rn(acc[r], __dadd_rn(__dmul_rn(w, (double)fv[u]), 0.0));
            }
        }
    };

    const bool relaxed = a.q_relaxed != nullptr && __ldg(a.q_relaxed + q) != 0;
    if (nnz != 0u && relaxed) {
        // Order-free accumulation (verified afterwards, see below): all essential slices of this block form one
        // index space walked 128 postings at a time; a row may be hit by several terms at once, so the adds are
        // shared-memory atomics (a CAS loop for fp64 — affordable: frequent terms never come this way).
        const uint32_t P = s_cum[nnz];
        uint32_t k = 0;
        for (uint32_t pos = tid; pos < P; pos += VB_SPARSE_THREADS) {
            while (s_cum[k + 1u] <= pos) ++k;
            const uint32_t j = s_nz[k];
            const uint32_t pp = s_lo[j] + (pos - s_cum[k]);
            const uint32_t r = __ldg(prow + pp) - row0;
            const float v = __ldg(pval + pp);
            atomicAdd(&acc[r], __dadd_rn(__dmul_rn(s_w[j], (double)v), 0.0));
        }
        __syncthreads();
    } else if (nnz != 0u) {
        uint32_t rA[VB_SPARSE_U], rB[VB_SPARSE_U];
        float vA[VB_SPARSE_U], vB[VB_SPARSE_U];
        uint32_t ti = 0, term = s_nz[0], p0 = s_lo[term], hi = s_hi[term];
        fetch(p0, hi, rA, vA);
        for (;;) {
            // ---- A holds (term ti, p0); find the batch after it and put it in flight into B ----
            uint32_t n_ti = ti, n_p0 = p0 + VB_SPARSE_BATCH, n_hi = hi;
            if (n_p0 >= hi) { n_ti = ti + 1u; if (n_ti < nnz) { const uint32_t t2 = s_nz[n_ti]; n_p0 = s_lo[t2]; n_hi = s_hi[t2]; } }
            const bool more = n_ti < nnz;
            if (more) fetch(n_p0, n_hi, rB, vB);
            rmw(p0, hi, s_w[term], rA, vA);
            if (n_ti != ti) __syncthreads();                    // the next term may hit the same rows
            if (!more) break;
            ti = n_ti; p0 = n_p0; hi = n_hi; term = s_nz[ti];
            // ---- B holds (term ti, p0); same step with the roles swapped ----
            n_ti = ti; n_p0 = p0 + VB_SPARSE_BATCH; n_hi = hi;
            if (n_p0 >= hi) { n_ti = ti + 1u; if (n_ti < nnz) { const uint32_t t2 = s_nz[n_ti]; n_p0 = s_lo[t2]; n_hi = s_hi[t2]; } }
            const bool more2 = n_ti < nnz;
            if (more2) fetch(n_p0, n_hi, rA, vA);
            rmw(p0, hi, s_w[term], rB, vB);
            if (n_ti != ti) __syncthreads();
            if (!more2) break;
            ti = n_ti; p0 = n_p0; hi = n_hi; term = s_nz[ti];
        }
    }

    const uint32_t seg_row0 = a.blk_begin * VB_ROWS_PER_BLOCK;
    const uint32_t sub = blk_rel & a.lists.sub_mask;            // append counter of this row block
    const double tau_d = (double)tau;
    if (n_all == nnz && nh == 0u && !relaxed) {
        // Every term with postings here was accumulated in term order: the accumulators hold the exact scores.
        // Scan two per thread per step.  Cheap exact prefilter in fp64: rounding to fp32 is monotone, so
        // cur < (double)tau implies float(cur) <= tau — such rows (the vast majority once tau is
        // established, and every untouched -0.0 row when tau >= 0) are dropped with one compare.
#pragma unroll 4
        for (uint32_t r = 2u * tid; r < VB_ROWS_PER_BLOCK; r += 2u * VB_SPARSE_THREADS) {
            const double2 c2 = *reinterpret_cast<const double2*>(&acc[r]);
            const double cv[2] = {c2.x, c2.y};
            if (!a.direct && c2.x < tau_d && c2.y < tau_d) continue;
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const double cur = cv[e];
                const uint32_t row = row0 + r + e;
                bool pass = (unsigned long long)__double_as_longlong(cur) != VB_ACC_SENTINEL && row < a.n_rows;
                if (pass && mask) pass = (mask[row >> 5] >> (row & 31u)) & 1u;
                float s = 0.0f;
                if (pass) { s = __double2float_rn(cur); pass = s > tau; }
                if (a.direct) {
                    if (row < a.n_rows) a.lists.cand[(size_t)list * a.lists.cap + (row - seg_row0)] = pass ? vb_pack_key(s, a.row_base + row) : 0ull;
                } else if (pass) {
                    vb_push_sub(a.lists, list, sub, s, a.row_base + row);
                }
            }
        }
        return;
    }
    // Otherwise the accumulators hold PARTIAL sums (essential terms scattered from postings, in term order):
    //  * terms with a dense column (frequent terms) are added here, row by row, straight from the column
    //    (coalesced loads, no shared-memory traffic);
    //  * non-essential terms were skipped: partial + sum(ub) bounds the score from above.
    // The sum S computed this way adds the same fp64 products as the reference but in another order, so
    // |S - S_ref| <= delta * S with delta = 4 * nt * 2^-53 (all products >= 0 on this path).  If
    // float(S (1-delta)) == float(S (1+delta)) the fp32 score is PROVABLY the reference's and is used as is;
    // otherwise (~1e-7 of the rows) — and for every row that survives a bound test with skipped terms — the
    // row is re-scored exactly from the forward index (all shared terms in ascending term id).
    const bool pruned = n_all != nnz;
    const bool verify_only = relaxed && !pruned;                // fp32 score provable from the order-free sum
    const double ubne = pruned ? a.ubne[q] : 0.0;
    const double delta = (double)(4u * nt) * 1.1102230246251565e-16;
    const double tau_lo = a.direct ? -INFINITY : (tau_d > 0.0 ? tau_d * (1.0 - 1e-9) : tau_d * (1.0 + 1e-9));
    const bool has_acc = nnz != 0u;
    const float fnan = __int_as_float(0x7fc00000);
    // Fast variant (the large segments): with tau > 0 an untouched row (sum 0) can never pass, so presence
    // needs no tracking — per row and dense column one max(v, 0) (NaN = absent -> 0), one convert, one fma —
    // and a single compare against thr = tau (1 - 1e-9) - sum(ub of skipped terms) drops almost every row.
    const double thr = tau_lo - ubne;
    if (!a.direct && tau_d > 0.0 && thr > 0.0) {
        // Pass 1, fp32: the same sums in single precision with every input rounded UP (accumulators, weights;
        // column values are exact floats), against a threshold lowered by more than the fp32 summation error
        // (~nt * 6e-8 relative, all terms >= 0) — so a row with S >= thr always has s32 >= thr32.  Each thread
        // owns 16 rows (4 groups of 4 consecutive rows); per dense column: four 128-bit loads, then one max and
        // one fma per row on the full-rate fp32 pipe.  Pass 2 redoes only the groups that may hold a candidate
        // in fp64 and runs the candidate logic.
        const float thr32 = __double2float_rd(thr * (1.0 - 1e-6 - (double)nt * 2e-7));
        float s32[4][4];
        bool in[4];
#pragma unroll
        for (uint32_t g = 0; g < 4u; ++g) {
            const uint32_t r = 4u * tid + g * 4u * VB_SPARSE_THREADS;
            in[g] = row0 + r < a.n_rows;
            s32[g][0] = s32[g][1] = s32[g][2] = s32[g][3] = 0.0f;
            if (has_acc) {
                const double2 c01 = *reinterpret_cast<const double2*>(&acc[r]), c23 = *reinterpret_cast<const double2*>(&acc[r + 2u]);
                s32[g][0] = __double2float_ru(c01.x); s32[g][1] = __double2float_ru(c01.y);
                s32[g][2] = __double2float_ru(c23.x); s32[g][3] = __double2float_ru(c23.y);
            }
        }
        for (uint32_t k = 0; k < nh; ++k) {
            const uint32_t j = s_hv[k];
            const float* col = a.heavy_vals + (size_t)__ldg(a.q_hidx + t_lo + j) * a.heavy_stride + row0 + 4u * tid;
            const float w = __double2float_ru(s_w[j]);
            float4 h[4];
#pragma unroll
            for (uint32_t g = 0; g < 4u; ++g)
                h[g] = in[g] ? __ldg(reinterpret_cast<const float4*>(col + g * 4u * VB_SPARSE_THREADS)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (uint32_t g = 0; g < 4u; ++g) {
                s32[g][0] = fmaf(w, fmaxf(h[g].x, 0.0f), s32[g][0]);
                s32[g][1] = fmaf(w, fmaxf(h[g].y, 0.0f), s32[g][1]);
                s32[g][2] = fmaf(w, fmaxf(h[g].z, 0.0f), s32[g][2]);
                s32[g][3] = fmaf(w, fmaxf(h[g].w, 0.0f), s32[g][3]);
            }
        }
#pragma unroll
        for (uint32_t g = 0; g < 4u; ++g) {
            if (s32[g][0] < thr32 && s32[g][1] < thr32 && s32[g][2] < thr32 && s32[g][3] < thr32) continue;
            // ---- pass 2 for this group: exact-order-free fp64 sums, verification, candidates ----
            const uint32_t r = 4u * tid + g * 4u * VB_SPARSE_THREADS;
            double sv[4] = {0.0, 0.0, 0.0, 0.0};
            if (has_acc) {
                const double2 c01 = *reinterpret_cast<const double2*>(&acc[r]), c23 = *reinterpret_cast<const double2*>(&acc[r + 2u]);
                sv[0] = c01.x; sv[1] = c01.y; sv[2] = c23.x; sv[3] = c23.y;
            }
            if (in[g]) {
                for (uint32_t k = 0; k < nh; ++k) {
                    const uint32_t j = s_hv[k];
                    const float4 hq = __ldg(reinterpret_cast<const float4*>(a.heavy_vals + (size_t)__ldg(a.q_hidx + t_lo + j) * a.heavy_stride + row0 + r));
                    const double w = s_w[j];
                    sv[0] = fma(w, (double)fmaxf(hq.x, 0.0f), sv[0]);
                    sv[1] = fma(w, (double)fmaxf(hq.y, 0.0f), sv[1]);
                    sv[2] = fma(w, (double)fmaxf(hq.z, 0.0f), sv[2]);
                    sv[3] = fma(w, (double)fmaxf(hq.w, 0.0f), sv[3]);
                }
            }
#pragma unroll
            for (uint32_t e = 0; e < 4u; ++e) {
                const uint32_t row = row0 + r + e;
                const double S = sv[e];
                if (S < thr || row >= a.n_rows) continue;
                if (mask && !((mask[row >> 5] >> (row & 31u)) & 1u)) continue;
                const float f_lo = __double2float_rn(S * (1.0 - delta)), f_hi = __double2float_rn(S * (1.0 + delta));
                if (!verify_only || f_lo != f_hi) { s_surv[atomicAdd(&s_nsurv, 1u)] = (uint16_t)(r + e); continue; }
                if (f_lo > tau) vb_push_sub(a.lists, list, sub, f_lo, a.row_base + row);
            }
        }
    } else
    // General variant (first segments, thresholds <= 0): tracks which rows have a shared term at all.
    // each thread owns 4 groups of 4 consecutive rows; the column loads of two groups x two terms (four
    // 128-bit loads) are issued together before any of them is used
    for (uint32_t g0 = 0; g0 < 4u; g0 += 2u) {
        double sv[2][4];
        uint32_t tch[2] = {0u, 0u};                             // bit e: row e of the group has a shared term
#pragma unroll
        for (uint32_t g = 0; g < 2u; ++g) {
            const uint32_t r = 4u * tid + (g0 + g) * 4u * VB_SPARSE_THREADS;
            double2 c01 = make_double2(neg_zero, neg_zero), c23 = c01;
            if (has_acc) { c01 = *reinterpret_cast<const double2*>(&acc[r]); c23 = *reinterpret_cast<const double2*>(&acc[r + 2u]); }
            sv[g][0] = c01.x; sv[g][1] = c01.y; sv[g][2] = c23.x; sv[g][3] = c23.y;
#pragma unroll
            for (uint32_t e = 0; e < 4u; ++e)
                tch[g] |= ((unsigned long long)__double_as_longlong(sv[g][e]) != VB_ACC_SENTINEL ? 1u : 0u) << e;
        }
        for (uint32_t k0 = 0; k0 < nh; k0 += 2u) {
            const bool two = k0 + 1u < nh;
            const uint32_t j0 = s_hv[k0], j1 = two ? s_hv[k0 + 1u] : j0;
            const float* col0 = a.heavy_vals + (size_t)__ldg(a.q_hidx + t_lo + j0) * a.heavy_stride + row0;
            const float* col1 = a.heavy_vals + (size_t)__ldg(a.q_hidx + t_lo + j1) * a.heavy_stride + row0;
            const double w0 = s_w[j0], w1 = s_w[j1];
            float4 h[2][2];
#pragma unroll
            for (uint32_t g = 0; g < 2u; ++g) {
                const uint32_t r = 4u * tid + (g0 + g) * 4u * VB_SPARSE_THREADS;
                const bool in = row0 + r < a.n_rows;            // (columns are padded to a multiple of 64 rows with NaN)
                h[g][0] = in ? __ldg(reinterpret_cast<const float4*>(col0 + r)) : make_float4(fnan, fnan, fnan, fnan);
                h[g][1] = (in && two) ? __ldg(reinterpret_cast<const float4*>(col1 + r)) : make_float4(fnan, fnan, fnan, fnan);
            }
#pragma unroll
            for (uint32_t g = 0; g < 2u; ++g) {
#pragma unroll
                for (uint32_t t = 0; t < 2u; ++t) {
                    const float hv[4] = {h[g][t].x, h[g][t].y, h[g][t].z, h[g][t].w};
                    const double w = t ? w1 : w0;
#pragma unroll
                    for (uint32_t e = 0; e < 4u; ++e) {
                        if (hv[e] == hv[e]) {
                            const double pr = __dmul_rn(w, (double)hv[e]);
                            sv[g][e] = ((tch[g] >> e) & 1u) ? __dadd_rn(sv[g][e], pr) : __dadd_rn(pr, 0.0);
                            tch[g] |= 1u << e;
                        }
                    }
                }
            }
        }
#pragma unroll
        for (uint32_t g = 0; g < 2u; ++g) {
            const uint32_t r = 4u * tid + (g0 + g) * 4u * VB_SPARSE_THREADS;
#pragma unroll
            for (uint32_t e = 0; e < 4u; ++e) {
                const uint32_t row = row0 + r + e;
                if (!((tch[g] >> e) & 1u) || row >= a.n_rows) continue;
                const double S = sv[g][e];
                if ((S + ubne) * (1.0 + delta) < tau_lo) continue;                   // cannot beat tau
                if (mask && !((mask[row >> 5] >> (row & 31u)) & 1u)) continue;
                const float f_lo = __double2float_rn(S * (1.0 - delta)), f_hi = __double2float_rn(S * (1.0 + delta));
                if (!verify_only || f_lo != f_hi) { s_surv[atomicAdd(&s_nsurv, 1u)] = (uint16_t)(r + e); continue; }
                if (a.direct) a.lists.cand[(size_t)list * a.lists.cap + (row - seg_row0)] = vb_pack_key(f_lo, a.row_base + row);
                else if (f_lo > tau) vb_push_sub(a.lists, list, sub, f_lo, a.row_base + row);
            }
        }
    }
    __syncthreads();
    const uint32_t nsurv = s_nsurv;
    for (uint32_t i = tid >> 5; i < nsurv; i += VB_SPARSE_THREADS / 32u) {      // one warp per survivor
        const uint32_t row = row0 + s_surv[i];                                   // (in range, passes the mask)
        const int64_t ip0 = __ldg(a.sp_indptr + row), ip1 = __ldg(a.sp_indptr + row + 1);
        double sc = 0.0;
        for (uint32_t j = 0; j < nt; ++j) {                                      // every query term, ascending id
            const uint32_t term = __ldg(a.q_term + t_lo + j);
            for (int64_t c0 = ip0; c0 < ip1; c0 += 32) {
                const int64_t p = c0 + lane;
                const bool hit = p < ip1 && __ldg(a.sp_term + p) == term;
                const uint32_t bal = __ballot_sync(0xffffffffu, hit);
                if (bal) {
                    float v = hit ? __ldg(a.sp_val + p) : 0.0f;
                    v = __shfl_sync(0xffffffffu, v, __ffs(bal) - 1);
                    sc = __dadd_rn(sc, __dmul_rn(s_w[j], (double)v));
                    break;
                }
            }
        }
        if (lane == 0) {
            const float sf = __double2float_rn(sc);
            if (a.direct) a.lists.cand[(size_t)list * a.lists.cap + (row - seg_row0)] = vb_pack_key(sf, a.row_base + row);
            else if (sf > tau) vb_push_sub(a.lists, list, sub, sf, a.row_base + row);
        }
    }
}
