// Exact top-k' selection over a candidate list, and the K4 fusion merge kernel.
//
// vb_compact_kernel replaces the argsort + walk qdrant's local mode does after scoring
// (local_collection.py search(): `order = np.argsort(scores)[::-1]`, skip masked, stop at
// limit).  The scoring kernels append every row whose score beats the list's threshold tau
// (a lower bound on the k'-th best seen so far); this kernel reduces a list to its exact top-k'
// under the total order (score desc, row asc), sorted, and raises tau.  Because keys are
// unique, the result does not depend on the order in which candidates were appended.
//
// vb_fuse_kernel replaces voitta's own fusion (vector_store.py:659-697, min-max weighted sum)
// and adds Qdrant's RRF (qdrant_client/hybrid/fusion.py).  All arithmetic is fp64 with explicit
// round-to-nearest mul/add/div (no FMA contraction) so it reproduces the Python floats bit for bit.
#pragma once
#include "common.cuh"

#define VB_SORT_MAX 2048u
#define VB_COMPACT_THREADS 256

// descending bitonic sort of P (power of two <= VB_SORT_MAX) keys in shared memory
__device__ __forceinline__ void vb_bitonic_desc(uint64_t* s, uint32_t P) {
    for (uint32_t size = 2; size <= P; size <<= 1) {
        for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (uint32_t t = threadIdx.x; t < (P >> 1); t += blockDim.x) {
                const uint32_t i = 2u * t - (t & (stride - 1u));
                const uint32_t j = i + stride;
                const bool up = (i & size) == 0u;
                const uint64_t x = s[i], y = s[j];
                if ((x < y) == up) { s[i] = y; s[j] = x; }
            }
        }
    }
    __syncthreads();
}

// One CTA per list.  Afterwards: cand[list][0..cnt) = top-min(k, #valid) keys sorted descending,
// cnt[list] = that count, tau[list] = score of the k-th (or -inf if fewer than k).
//
// Selection, not sorting: a list holds a few thousand unsorted keys of which only k' (tens)
// survive, and this kernel sits on the critical path between two scoring segments.
//   1. the list (the used prefixes of its sub-ranges) is L2-resident and re-read in each pass;
//   2. block min/max of the active keys give their common bit prefix; ONE 2048-bin histogram
//      over the 11 bits below the highest differing bit and a block suffix scan find the pivot
//      bin (the bin holding the k'-th largest key);
//   3. every key >= the pivot bin's lower bound is gathered (k' + a few) and only those are
//      sorted.  If that would exceed VB_SORT_MAX keys, step 2 repeats inside the pivot bin.
#define VB_BINS 2048u

template <bool IS_MAX>
__device__ __forceinline__ uint64_t vb_block_reduce_u64(uint64_t v, uint64_t* s_red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const uint64_t t = __shfl_xor_sync(0xffffffffu, v, o);
        v = IS_MAX ? (t > v ? t : v) : (t < v ? t : v);
    }
    __syncthreads();                                   // s_red may still be read from a previous call
    if ((threadIdx.x & 31u) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    uint64_t r = s_red[0];
#pragma unroll
    for (uint32_t w = 1; w < VB_COMPACT_THREADS / 32; ++w) {
        const uint64_t t = s_red[w];
        r = IS_MAX ? (t > r ? t : r) : (t < r ? t : r);
    }
    return r;
}

// The general path: selection by histogram over the used prefixes of the sub-ranges (s_E[sub] keys each), which are
// L2-resident and re-read in each pass.  Deliberately compact code (run-time loops, no register image of the list, one
// instantiation): the first version unrolled every pass over the 8 sub-ranges and kept a second, register-resident
// variant — 9.5 k instructions (150 KB) for a kernel that runs after every segment / stage of both branches, ~10 times
// per search, with 8 CTAs per SM in different phases: instruction fetch, not the few thousand keys, set its duration.
__device__ __noinline__ void vb_compact_select(uint64_t* __restrict__ gkeys, const uint32_t* s_E, uint32_t sub_cap,
                                               uint32_t k, uint32_t* __restrict__ cnt_out, float* __restrict__ tau_out,
                                               uint64_t* s_sel, uint32_t* s_hist, uint64_t* s_red,
                                               uint32_t* s_scan, uint32_t* s_misc)
{
    // visit every key of the list
    auto for_each = [&](auto&& f) {
#pragma unroll 1
        for (uint32_t sub = 0; sub < VB_SUB; ++sub) {
            const uint32_t e = s_E[sub];
            const uint64_t* g = gkeys + (size_t)sub * sub_cap;
#pragma unroll 1
            for (uint32_t i = threadIdx.x; i < e; i += VB_COMPACT_THREADS) f(g[i]);
        }
    };

    uint32_t need = k;                                 // rank of the k-th largest among the active keys
    uint64_t pmask = 0ull, pval = 0ull;                // active: key != 0 && (key & pmask) == pval
    uint64_t bound = 1ull;                             // gather every key >= bound
#pragma unroll 1
    for (;;) {
        uint64_t kmax = 0ull, kmin = ~0ull;
        uint32_t n_act = 0;
        for_each([&](uint64_t key) {
            if (key != 0ull && (key & pmask) == pval) { ++n_act; kmax = key > kmax ? key : kmax; kmin = key < kmin ? key : kmin; }
        });
        kmax = vb_block_reduce_u64<true>(kmax, s_red);
        kmin = vb_block_reduce_u64<false>(kmin, s_red);
        __syncthreads();
        if (threadIdx.x == 0) s_misc[0] = 0u;
        __syncthreads();
        if (n_act) atomicAdd(&s_misc[0], n_act);
        __syncthreads();
        const uint32_t total_act = s_misc[0];
        if (total_act <= need || kmax == kmin) {       // everything active is kept
            bound = total_act ? kmin : 1ull;
            if (pmask != 0ull && total_act == 0) bound = pval ? pval : 1ull;
            break;
        }
        const int top = 63 - __clzll((long long)(kmax ^ kmin));   // highest differing bit
        const int shift = top >= 10 ? top - 10 : 0;                // digit = bits [shift, shift+11)
#pragma unroll 1
        for (uint32_t i = threadIdx.x; i < VB_BINS; i += VB_COMPACT_THREADS) s_hist[i] = 0u;
        __syncthreads();
        for_each([&](uint64_t key) {
            if (key != 0ull && (key & pmask) == pval) atomicAdd(&s_hist[(uint32_t)(key >> shift) & (VB_BINS - 1u)], 1u);
        });
        __syncthreads();
        // suffix scan over the bins: thread t owns bins [hi_bin - PER + 1, hi_bin], thread 0 the top ones
        constexpr uint32_t PER = VB_BINS / VB_COMPACT_THREADS;
        const uint32_t hi_bin = VB_BINS - 1u - threadIdx.x * PER;
        uint32_t mine = 0;
#pragma unroll 1
        for (uint32_t j = 0; j < PER; ++j) mine += s_hist[hi_bin - j];
        uint32_t incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
            if ((threadIdx.x & 31u) >= (uint32_t)o) incl += t;
        }
        if ((threadIdx.x & 31u) == 31u) s_scan[threadIdx.x >> 5] = incl;
        __syncthreads();
        uint32_t before = 0;
#pragma unroll 1
        for (uint32_t w = 0; w < (threadIdx.x >> 5); ++w) before += s_scan[w];
        const uint32_t above_me = before + incl - mine;           // active keys in bins above mine
        if (above_me < need && above_me + mine >= need) {         // the pivot bin is one of mine
            uint32_t above = above_me;
#pragma unroll 1
            for (uint32_t j = 0; j < PER; ++j) {
                const uint32_t c = s_hist[hi_bin - j];
                if (above < need && above + c >= need) { s_misc[1] = hi_bin - j; s_misc[2] = above; }
                above += c;
            }
        }
        __syncthreads();
        const uint32_t pivot = s_misc[1], above = s_misc[2], in_pivot = s_hist[pivot];
        const uint64_t low_mask = (1ull << shift) - 1ull;         // bits below the digit
        const uint64_t high_bits = (shift + 11 >= 64) ? 0ull : (kmax >> (shift + 11)) << (shift + 11);
        const uint64_t pivot_lo = high_bits | ((uint64_t)pivot << shift);     // smallest key value of the pivot bin
        if ((k - need) + above + in_pivot <= VB_SORT_MAX || shift == 0) { bound = pivot_lo; break; }
        need -= above;                                            // crowded pivot bin: refine inside it
        pmask = ~low_mask;
        pval = pivot_lo;
        __syncthreads();
    }
    __syncthreads();
    if (threadIdx.x == 0) s_misc[0] = 0u;
    __syncthreads();
    for_each([&](uint64_t key) {
        if (key != 0ull && key >= bound) {
            const uint32_t slot = atomicAdd(&s_misc[0], 1u);
            if (slot < VB_SORT_MAX) s_sel[slot] = key;
        }
    });
    __syncthreads();
}

__global__ void __launch_bounds__(VB_COMPACT_THREADS)
vb_compact_kernel(VbLists L, float* __restrict__ tau, uint32_t* __restrict__ overflow, uint32_t k, uint32_t list_begin,
                  uint32_t lim0 /* slots sub-range 0 may hold: sub_cap, or the first segment's direct block */)
{
    __shared__ uint64_t s_sel[VB_SORT_MAX];
    __shared__ uint32_t s_hist[VB_BINS];
    __shared__ uint64_t s_red[VB_COMPACT_THREADS / 32];
    __shared__ uint32_t s_scan[VB_COMPACT_THREADS / 32];
    __shared__ uint32_t s_misc[4];
    __shared__ uint32_t s_E[VB_SUB];
    const uint32_t list = list_begin + blockIdx.x;
    uint64_t* gkeys = L.cand + (size_t)list * L.cap;
    VB_CHECK(list < L.n_lists && lim0 <= L.cap);
    if (threadIdx.x < VB_SUB) {
        const uint32_t sub = threadIdx.x;
        const uint32_t raw = L.cnt[list * VB_SUB + sub];
        const uint32_t lim = sub == 0 ? lim0 : L.sub_cap;
        if (raw > lim || (sub > L.sub_mask && raw != 0u)) overflow[list] = 1u;
        s_E[sub] = raw < lim ? raw : lim;
    }
    if (threadIdx.x == 0) s_misc[0] = 0u;
    __syncthreads();                                   // everyone sees the counters before they are rewritten
    // Small lists (the common case once thresholds exist, and every list of a single-query search): no selection
    // needed — gather the non-empty keys of the used prefixes into shared memory, sort them, write back.  Empty slots
    // (a direct first segment under a selective filter is mostly empty) are dropped before the sort.
    uint32_t total = 0;
#pragma unroll 1
    for (uint32_t sub = 0; sub < VB_SUB; ++sub) total += s_E[sub];
    bool selected = false;
    if (total <= 4u * VB_SORT_MAX) {
#pragma unroll 1
        for (uint32_t sub = 0; sub < VB_SUB; ++sub) {
            const uint32_t e = s_E[sub];
            const uint64_t* g = gkeys + (size_t)sub * L.sub_cap;
#pragma unroll 1
            for (uint32_t i = threadIdx.x; i < e; i += VB_COMPACT_THREADS) {
                const uint64_t key = g[i];
                if (key != 0ull) {
                    const uint32_t slot = atomicAdd(&s_misc[0], 1u);
                    if (slot < VB_SORT_MAX) s_sel[slot] = key;
                }
            }
        }
        __syncthreads();
        selected = s_misc[0] <= VB_SORT_MAX;
        __syncthreads();                                // (s_misc[0] is reset by the general path)
    }
    if (!selected)                                      // too many live keys: select those that can be in the top k' first
        vb_compact_select(gkeys, s_E, L.sub_cap, k, L.cnt + (size_t)list * VB_SUB, tau + list, s_sel, s_hist, s_red, s_scan, s_misc);
    const uint32_t nsel = s_misc[0] < VB_SORT_MAX ? s_misc[0] : VB_SORT_MAX;
    uint32_t P = 2;
    while (P < nsel) P <<= 1;
    for (uint32_t i = nsel + threadIdx.x; i < P; i += VB_COMPACT_THREADS) s_sel[i] = 0ull;
    vb_bitonic_desc(s_sel, P);                          // (every stage starts with a barrier; ends with one)
    const uint32_t keep = nsel < k ? nsel : k;
    for (uint32_t i = threadIdx.x; i < keep; i += VB_COMPACT_THREADS) gkeys[i] = s_sel[i];
    if (threadIdx.x < VB_SUB) L.cnt[(size_t)list * VB_SUB + threadIdx.x] = threadIdx.x == 0 ? keep : 0u;   // the list now lives in sub-range 0
    if (threadIdx.x == 0) {
        // never below the threshold the segment ran with: a threshold is only ever raised (DESIGN §3), so a list
        // that holds fewer than k' entries keeps the one it has
        tau[list] = fmaxf(tau[list], (keep >= k) ? vb_key_score(s_sel[k - 1]) : -INFINITY);
    }
}

// Pack the first k keys of every list into out[list][k] (0-padded): the all-gather payload.
// If `overflow` is given, one extra word out[n_lists*k] carries "some list of this shard
// overflowed", so every rank learns it from the same all-gather and re-runs consistently.
__global__ void vb_export_kernel(const uint64_t* __restrict__ cand, const uint32_t* __restrict__ cnt,
                                 uint32_t cap, uint32_t k, uint64_t* __restrict__ out,
                                 const uint32_t* __restrict__ overflow, uint32_t n_lists)
{
    const uint32_t list = blockIdx.x;
    const uint32_t c = cnt[list * VB_SUB] < k ? cnt[list * VB_SUB] : k;
    for (uint32_t i = threadIdx.x; i < k; i += blockDim.x)
        out[(size_t)list * k + i] = i < c ? cand[(size_t)list * cap + i] : 0ull;
    if (overflow != nullptr && blockIdx.x == 0) {
        int any = 0;
        for (uint32_t i = threadIdx.x; i < n_lists; i += blockDim.x) any |= overflow[i] != 0u;
        any = __syncthreads_or(any);
        if (threadIdx.x == 0) out[(size_t)n_lists * k] = any ? 1ull : 0ull;
    }
}

// Scatter gathered[shard][list][k] (+1 flag word per shard) into cand[list][shard*k + i] and set
// cnt = n_shards*k (empty slots are 0 keys, which the compaction ignores).
__global__ void vb_import_kernel(const uint64_t* __restrict__ gathered, uint32_t n_shards, uint32_t n_lists,
                                 uint32_t k, uint32_t cap, uint64_t* __restrict__ cand, uint32_t* __restrict__ cnt,
                                 uint32_t* __restrict__ overflow)
{
    const uint32_t list = blockIdx.x;
    const size_t stride = (size_t)n_lists * k + 1;
    for (uint32_t i = threadIdx.x; i < n_shards * k; i += blockDim.x) {
        const uint32_t sh = i / k, j = i % k;
        cand[(size_t)list * cap + i] = gathered[sh * stride + (size_t)list * k + j];
    }
    if (threadIdx.x < VB_SUB) cnt[list * VB_SUB + threadIdx.x] = threadIdx.x == 0 ? n_shards * k : 0u;
    if (threadIdx.x == 0) {
        if (list == 0)
            for (uint32_t sh = 0; sh < n_shards; ++sh)
                if (gathered[sh * stride + (size_t)n_lists * k] != 0ull) overflow[0] = 1u;
    }
}

// ---------------------------------------------------------------------------------------------
// K4 fusion.  One CTA per query.  Dense list = list q, sparse list = list B+q, both already
// sorted (score desc).  Output: rows + fp64 scores in rank order, count.
//   mode 0: dense only (vector_store.py:611-619): first `limit` dense hits, score = cosine
//   mode 1: weighted   (vector_store.py:659-697)
//   mode 2: rrf        (qdrant hybrid/fusion.py, ranking constant 2)
// Ties of the fused score keep first-seen order (dense list, then sparse-only ids).
// ---------------------------------------------------------------------------------------------
struct VbFuseArgs {
    const uint64_t* cand;
    const uint32_t* cnt;
    const int32_t* mode;      // [B]
    uint32_t cap, n_queries, k, limit;
    double w_sparse, w_dense;
    uint32_t* out_rows;       // [B][limit]
    double* out_scores;       // [B][limit]
    int32_t* out_cnt;         // [B]
    // list bookkeeping for the host, written here instead of by two more copies after the kernel
    const uint32_t* overflow; // [2B]
    uint32_t* out_lcnt;       // [2B] entries of every list
    uint32_t* out_ovf;        // [2B] overflow flags
};

#define VB_FUSE_THREADS 256
static size_t vb_fuse_smem_bytes(uint32_t k) { return (size_t)2 * k * (8 + 4 + 4 + 1) + 16; }
__global__ void __launch_bounds__(VB_FUSE_THREADS)
vb_fuse_kernel(const VbFuseArgs a)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const uint32_t k = a.k;
    double* fin = reinterpret_cast<double*>(smem_raw);          // [2k] fused score
    uint32_t* row = reinterpret_cast<uint32_t*>(fin + 2 * k);   // [2k]
    uint32_t* lrow = row + 2 * k;                               // [2k] row ids of the two lists (dense [0,k), sparse [k,2k))
    uint8_t* valid = reinterpret_cast<uint8_t*>(lrow + 2 * k);  // [2k]

    const uint32_t q = blockIdx.x, B = a.n_queries;
    if (threadIdx.x < 2u && a.out_lcnt != nullptr) {
        const uint32_t l = threadIdx.x * B + q;
        a.out_lcnt[l] = a.cnt[l * VB_SUB];
        a.out_ovf[l] = a.overflow[l];
    }
    const uint64_t* dk = a.cand + (size_t)q * a.cap;
    const uint64_t* sk = a.cand + (size_t)(B + q) * a.cap;
    const uint32_t nd = a.cnt[q * VB_SUB] < k ? a.cnt[q * VB_SUB] : k;
    const int32_t mode = a.mode[q];

    if (mode == 0) {
        const uint32_t n = nd < a.limit ? nd : a.limit;
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
            a.out_rows[(size_t)q * a.limit + i] = vb_key_row(dk[i]);
            a.out_scores[(size_t)q * a.limit + i] = (double)vb_key_score(dk[i]);
        }
        if (threadIdx.x == 0) a.out_cnt[q] = (int32_t)n;
        return;
    }
    const uint32_t ns = a.cnt[(B + q) * VB_SUB] < k ? a.cnt[(B + q) * VB_SUB] : k;

    double dmin = 0.0, dspread = 0.0, smin = 0.0, sspread = 0.0;
    if (nd) { dmin = (double)vb_key_score(dk[nd - 1]); dspread = __dsub_rn((double)vb_key_score(dk[0]), dmin); }
    if (ns) { smin = (double)vb_key_score(sk[ns - 1]); sspread = __dsub_rn((double)vb_key_score(sk[0]), smin); }

    for (uint32_t i = threadIdx.x; i < 2 * k; i += blockDim.x) valid[i] = 0;
    // the membership tests below read every row id of the other list: from shared memory, not k' x k' global loads
    for (uint32_t i = threadIdx.x; i < nd; i += blockDim.x) lrow[i] = vb_key_row(dk[i]);
    for (uint32_t j = threadIdx.x; j < ns; j += blockDim.x) lrow[k + j] = vb_key_row(sk[j]);
    __syncthreads();

    // dense candidates: slot i
    for (uint32_t i = threadIdx.x; i < nd; i += blockDim.x) {
        const uint32_t r = lrow[i];
        int j = -1;
        for (uint32_t t = 0; t < ns; ++t) if (lrow[k + t] == r) { j = (int)t; break; }
        double f;
        if (mode == 1) {
            const double dn = dspread > 0.0 ? __ddiv_rn(__dsub_rn((double)vb_key_score(dk[i]), dmin), dspread) : 1.0;
            const double sn = j < 0 ? 0.0
                              : (sspread > 0.0 ? __ddiv_rn(__dsub_rn((double)vb_key_score(sk[j]), smin), sspread) : 1.0);
            f = __dadd_rn(__dmul_rn(a.w_dense, dn), __dmul_rn(a.w_sparse, sn));
        } else {
            f = __ddiv_rn(1.0, (double)(2u + i));
            if (j >= 0) f = __dadd_rn(f, __ddiv_rn(1.0, (double)(2u + (uint32_t)j)));
        }
        fin[i] = f; row[i] = r; valid[i] = 1;
    }
    // sparse-only candidates: slot k + j
    for (uint32_t j = threadIdx.x; j < ns; j += blockDim.x) {
        const uint32_t r = lrow[k + j];
        bool in_dense = false;
        for (uint32_t t = 0; t < nd; ++t) if (lrow[t] == r) { in_dense = true; break; }
        if (in_dense) continue;
        double f;
        if (mode == 1) {
            const double sn = sspread > 0.0 ? __ddiv_rn(__dsub_rn((double)vb_key_score(sk[j]), smin), sspread) : 1.0;
            f = __dadd_rn(__dmul_rn(a.w_dense, 0.0), __dmul_rn(a.w_sparse, sn));
        } else {
            f = __ddiv_rn(1.0, (double)(2u + j));
        }
        fin[k + j] = f; row[k + j] = r; valid[k + j] = 1;
    }
    __syncthreads();

    // rank by counting: better(c', c) = f' > f or (f' == f and slot' < slot)
    uint32_t total = 0;
    for (uint32_t c = threadIdx.x; c < 2 * k; c += blockDim.x) {
        if (!valid[c]) continue;
        const double f = fin[c];
        uint32_t rank = 0;
        for (uint32_t o = 0; o < 2 * k; ++o) {
            if (!valid[o]) continue;
            const double g = fin[o];
            rank += (g > f || (g == f && o < c)) ? 1u : 0u;
        }
        if (rank < a.limit) {
            a.out_rows[(size_t)q * a.limit + rank] = row[c];
            a.out_scores[(size_t)q * a.limit + rank] = f;
        }
        ++total;
    }
    // total candidates = nd + sparse-only; count via block reduction
    __shared__ uint32_t s_total;
    if (threadIdx.x == 0) s_total = 0;
    __syncthreads();
    atomicAdd(&s_total, total);
    __syncthreads();
    if (threadIdx.x == 0) a.out_cnt[q] = (int32_t)(s_total < a.limit ? s_total : a.limit);
}
