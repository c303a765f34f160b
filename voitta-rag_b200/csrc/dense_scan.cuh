// K1 — single-query / small-batch dense scoring: a bandwidth-bound GEMV over the bf16 corpus
// with the filter bitmask and the top-k' threshold fused into the row loop.
// Replaces qdrant's cosine scoring for query_points(query=vec, limit=k', query_filter)
// (vector_store.py:612-617, :640-645; distances.py cosine_similarity in local mode).
//
//   - one warp owns a 32-row group (= one mask word); masked rows are never loaded, so at 1 %
//     selectivity only 1 % of the row bytes move;
//   - a row is read with coalesced 128-bit streaming loads (lane l reads 16-byte chunks
//     l, l+32, ...), 4 rows in flight per warp for memory-level parallelism;
//   - the query (fp32, unit norm) lives in registers; fp32 FMA accumulate, xor-butterfly reduce;
//   - score = dot * inv_norm[row]; rows beating the list's threshold tau are appended to the
//     candidate list (vb_push); the exact top-k' is selected by vb_compact_kernel.
// Roofline: HBM.  Algorithmic bytes per launch = P*(d_pad*2 + 4) + groups*4 (mask words),
// P = rows that pass the mask.
#pragma once
#include "common.cuh"

struct VbScanArgs {
    const uint4* rows;          // [n][d_pad] bf16 as 16-byte chunks
    const float* inv_norm;      // [n]
    const uint32_t* mask;       // [n_filters][mask_words] or nullptr
    const int32_t* mask_of;     // [B] filter index per query, -1 = no mask; nullptr = none
    const float* q_hat;         // [B][d_pad] fp32 unit-norm queries
    const float* tau;           // [n_lists]
    VbLists lists;
    uint32_t mask_words;
    uint32_t chunks;            // d_pad / 8
    uint32_t row_begin, row_end;// segment (row_begin % 32 == 0)
    uint32_t row_base;          // added to the row in the candidate key (shard offset)
    uint32_t q_begin;           // first query handled by blockIdx.y == 0
    uint32_t direct;            // 1: first segment — store the key at slot (row - row_begin), no atomics
};

__device__ __forceinline__ float vb_dot8(const uint4 v, const float* q, float acc) {
    acc = fmaf(__uint_as_float(v.x << 16), q[0], acc);
    acc = fmaf(__uint_as_float(v.x & 0xffff0000u), q[1], acc);
    acc = fmaf(__uint_as_float(v.y << 16), q[2], acc);
    acc = fmaf(__uint_as_float(v.y & 0xffff0000u), q[3], acc);
    acc = fmaf(__uint_as_float(v.z << 16), q[4], acc);
    acc = fmaf(__uint_as_float(v.z & 0xffff0000u), q[5], acc);
    acc = fmaf(__uint_as_float(v.w << 16), q[6], acc);
    acc = fmaf(__uint_as_float(v.w & 0xffff0000u), q[7], acc);
    return acc;
}

// NCH = ceil(chunks / 32) register-resident query chunks per lane (d_pad <= NCH*256).
template <int NCH>
__global__ void __launch_bounds__(256)
vb_dense_scan_kernel(const VbScanArgs a)
{
    constexpr int ROWS = 4;
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t q_idx = a.q_begin + blockIdx.y;
    const uint32_t list = q_idx;  // dense lists come first
    const float tau = a.tau[list];
    const uint32_t* mask = nullptr;
    if (a.mask != nullptr && a.mask_of != nullptr) {
        const int32_t f = a.mask_of[q_idx];
        if (f >= 0) mask = a.mask + (size_t)f * a.mask_words;
    }

    float q[NCH][8];
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
        const uint32_t ch = lane + 32u * c;
        float4 lo = make_float4(0.f, 0.f, 0.f, 0.f), hi = lo;
        if (ch < a.chunks) {
            const float4* qp = reinterpret_cast<const float4*>(a.q_hat + (size_t)q_idx * a.chunks * 8u + ch * 8u);
            lo = __ldg(qp); hi = __ldg(qp + 1);
        }
        q[c][0] = lo.x; q[c][1] = lo.y; q[c][2] = lo.z; q[c][3] = lo.w;
        q[c][4] = hi.x; q[c][5] = hi.y; q[c][6] = hi.z; q[c][7] = hi.w;
    }

    const uint32_t warps = gridDim.x * (blockDim.x >> 5);
    const uint32_t g_begin = a.row_begin >> 5, g_end = (a.row_end + 31u) >> 5;
    for (uint32_t g = g_begin + blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); g < g_end; g += warps) {
        uint32_t bits = mask ? mask[g] : 0xffffffffu;
        const uint32_t row0 = g << 5;
        if (row0 + 32u > a.row_end) bits &= (1u << (a.row_end - row0)) - 1u;
        if (bits == 0u) continue;
        const float invn = (row0 + lane < a.row_end) ? a.inv_norm[row0 + lane] : 0.0f;
        while (bits) {
            int r[ROWS];
#pragma unroll
            for (int k = 0; k < ROWS; ++k) {
                r[k] = bits ? (__ffs(bits) - 1) : -1;
                bits &= bits - 1u;
            }
            uint4 v[ROWS][NCH];
#pragma unroll
            for (int k = 0; k < ROWS; ++k) {
#pragma unroll
                for (int c = 0; c < NCH; ++c) {
                    const uint32_t ch = lane + 32u * c;
                    v[k][c] = (r[k] >= 0 && ch < a.chunks)
                                  ? vb_ldg_stream(a.rows + (size_t)(row0 + r[k]) * a.chunks + ch)
                                  : make_uint4(0u, 0u, 0u, 0u);
                }
            }
#pragma unroll
            for (int k = 0; k < ROWS; ++k) {
#pragma unroll
                for (int c = 0; c < NCH; ++c) vb_keep_loaded(v[k][c]);
            }
            float acc[ROWS];
#pragma unroll
            for (int k = 0; k < ROWS; ++k) {
                acc[k] = 0.0f;
#pragma unroll
                for (int c = 0; c < NCH; ++c) acc[k] = vb_dot8(v[k][c], q[c], acc[k]);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
                for (int k = 0; k < ROWS; ++k) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
            }
            // lane k finishes row r[k]
            float mine = acc[0];
            int myr = r[0];
#pragma unroll
            for (int k = 1; k < ROWS; ++k) {
                if (lane == (uint32_t)k) { mine = acc[k]; myr = r[k]; }
            }
            const float inv_r = __shfl_sync(0xffffffffu, invn, myr < 0 ? 0 : myr);
            if (lane < (uint32_t)ROWS && myr >= 0) {
                const float s = mine * inv_r;
                const uint32_t row = row0 + (uint32_t)myr;
                if (a.direct) a.lists.cand[(size_t)list * a.lists.cap + (row - a.row_begin)] = s > tau ? vb_pack_key(s, a.row_base + row) : 0ull;
                else if (s > tau) vb_push(a.lists, list, s, a.row_base + row);
            }
        }
    }
}

// Generic variant for d_pad > 1024: the query is re-read through L1 per chunk.
__global__ void __launch_bounds__(256)
vb_dense_scan_generic_kernel(const VbScanArgs a)
{
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t q_idx = a.q_begin + blockIdx.y;
    const uint32_t list = q_idx;
    const float tau = a.tau[list];
    const uint32_t* mask = nullptr;
    if (a.mask != nullptr && a.mask_of != nullptr) {
        const int32_t f = a.mask_of[q_idx];
        if (f >= 0) mask = a.mask + (size_t)f * a.mask_words;
    }
    const float* qv = a.q_hat + (size_t)q_idx * a.chunks * 8u;
    const uint32_t warps = gridDim.x * (blockDim.x >> 5);
    const uint32_t g_begin = a.row_begin >> 5, g_end = (a.row_end + 31u) >> 5;
    for (uint32_t g = g_begin + blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); g < g_end; g += warps) {
        uint32_t bits = mask ? mask[g] : 0xffffffffu;
        const uint32_t row0 = g << 5;
        if (row0 + 32u > a.row_end) bits &= (1u << (a.row_end - row0)) - 1u;
        while (bits) {
            const uint32_t r = __ffs(bits) - 1;
            bits &= bits - 1u;
            float acc = 0.0f;
            for (uint32_t ch = lane; ch < a.chunks; ch += 32u) {
                const uint4 v = vb_ldg_stream(a.rows + (size_t)(row0 + r) * a.chunks + ch);
                float qq[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) qq[e] = __ldg(qv + ch * 8u + e);
                acc = vb_dot8(v, qq, acc);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
            if (lane == 0) {
                const float s = acc * a.inv_norm[row0 + r];
                const uint32_t row = row0 + r;
                if (a.direct) a.lists.cand[(size_t)list * a.lists.cap + (row - a.row_begin)] = s > tau ? vb_pack_key(s, a.row_base + row) : 0ull;
                else if (s > tau) vb_push(a.lists, list, s, a.row_base + row);
            }
        }
    }
}

// ---- K1F — single-pass form of K1 for the batch sizes voitta actually issues (B = 1, mcp_server.py:474) -----
// K1 above walks the rows in segments (2048, x128, ...) with a select kernel after each one, so that a global
// threshold exists before the bulk of the rows is scanned: 2-3 scan launches + 2-3 selects + list set-up per
// search, ~100 us of launch latency around ~15 us of HBM time at 100k rows.  K1F makes ONE pass: every CTA
// keeps its own candidate buffer in shared memory and its own threshold (the score of its current k'-th best),
// re-selecting whenever the buffer could overflow; CTAs publish their thresholds through one global word per
// list (atomicMax on the order-preserving score encoding) — any CTA's k'-th best is a lower bound of the
// global k'-th best — so late CTAs prune with the best threshold known anywhere.  At the end each CTA appends
// the part of its exact local top-k' that still reaches that threshold to the list (one atomic per CTA);
// vb_compact_kernel merges the few hundred keys (the same kernel that merges per-shard lists).  Rows are dealt to CTAs in an interleaved order, so every CTA sees a
// uniform sample of the corpus and its threshold converges after a few hundred rows.
// Exactness: pruning keeps every row with score >= threshold (ties stay, rows arrive out of row order); the
// final order (score desc, row asc) comes from the keys, which are unique.  Same arithmetic as K1.
#define VB_K1F_THREADS 256
#define VB_K1F_CAP 2048u           // candidate slots per CTA (16 KB of shared memory: 8 CTAs per SM, full occupancy —
                                   // the first version had 32 KB buffers, 2 CTAs per SM, and ran at half of K1's bandwidth)
#define VB_K1F_CHECK 4u            // iterations between buffer checks: 8 warps x (8 batches x 4 rows) x 4 = 1024 appends at most

struct VbScan1Args {
    const uint4* rows;
    const float* inv_norm;
    const uint32_t* mask;
    const int32_t* mask_of;
    const float* q_hat;
    uint32_t* gtau;             // [n_lists] shared threshold: vb_f32_ordered(score), 0 = none yet
    uint64_t* cand;
    uint32_t* cnt;
    uint32_t cap, k, mask_words, chunks, n_rows, row_base;
    uint32_t split_shift;       // a warp takes 32 >> split_shift rows of a group (tiny corpora: more warps than groups)
    uint32_t unit_shift;        // otherwise a warp's unit is 2^unit_shift consecutive groups (0..5)
    uint32_t* done;             // [n_lists] CTAs of the list that have appended their part (0 before the launch, 0 again after)
    float* tau;                 // [n_lists] list threshold, raised by the in-kernel merge like vb_compact_kernel does
};

// descending bitonic sort of P keys (power of two <= VB_K1F_CAP) by all threads of the CTA.  One out-of-line copy
// serves the scan loop and the final merge: a single-CTA tail is bound by instruction fetch, not by arithmetic.
__device__ __noinline__ void vb_k1f_sort(uint64_t* s, uint32_t P) {
    for (uint32_t size = 2; size <= P; size <<= 1)
        for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (uint32_t t = threadIdx.x; t < (P >> 1); t += VB_K1F_THREADS) {
                const uint32_t i = 2u * t - (t & (stride - 1u)), j = i + stride;
                const bool up = (i & size) == 0u;
                const uint64_t x = s[i], y = s[j];
                if ((x < y) == up) { s[i] = y; s[j] = x; }
            }
        }
    __syncthreads();
}

// No minimum-CTAs bound: an explicit 1 lets ptxas take 89-138 registers instead of 62-79, and 5 / 6 / 8 (fewer
// registers, spills) measured slower (DESIGN §K1F)
template <int NCH>
__global__ void __launch_bounds__(VB_K1F_THREADS)
vb_dense_scan1_kernel(const VbScan1Args a)
{
    constexpr int ROWS = 4;
    __shared__ uint64_t s_keys[VB_K1F_CAP];
    __shared__ uint32_t s_cnt;
    __shared__ float s_tau;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t q_idx = blockIdx.y, list = q_idx;
    const uint32_t* mask = nullptr;
    if (a.mask != nullptr && a.mask_of != nullptr) {
        const int32_t f = a.mask_of[q_idx];
        if (f >= 0) mask = a.mask + (size_t)f * a.mask_words;
    }
    float q[NCH][8];
#pragma unroll
    for (int c = 0; c < NCH; ++c) {
        const uint32_t ch = lane + 32u * c;
        float4 lo = make_float4(0.f, 0.f, 0.f, 0.f), hi = lo;
        if (ch < a.chunks) {
            const float4* qp = reinterpret_cast<const float4*>(a.q_hat + (size_t)q_idx * a.chunks * 8u + ch * 8u);
            lo = __ldg(qp); hi = __ldg(qp + 1);
        }
        q[c][0] = lo.x; q[c][1] = lo.y; q[c][2] = lo.z; q[c][3] = lo.w;
        q[c][4] = hi.x; q[c][5] = hi.y; q[c][6] = hi.z; q[c][7] = hi.w;
    }
    if (threadIdx.x == 0) { s_cnt = 0u; s_tau = -INFINITY; }
    __syncthreads();
    float tau = -INFINITY;
    // Work units.  A warp takes UNITS of 2^unit_shift consecutive 32-row groups (lane l holds the filter word of group
    // g0 + l: one coalesced load per unit, and the NEXT unit's words are already in flight while this one is scored), or,
    // on tiny corpora (split_shift > 0), a half / quarter / eighth of one group.  Rows are scored four at a time, and a
    // batch of four is filled ACROSS the groups of a unit (and across units): under a selective filter (1 % of the rows:
    // one passing row in three groups) every warp still keeps four rows of loads in flight.  (The first version
    // walked one group at a time: a dependent filter-word load, then 0..1 rows, per iteration.)
    const uint32_t n_groups = (a.n_rows + 31u) >> 5;
    const uint32_t U = 1u << a.unit_shift;
    const uint32_t n_units = a.split_shift ? (n_groups << a.split_shift) : ((n_groups + U - 1u) >> a.unit_shift);
    const uint32_t part_rows = 32u >> a.split_shift;
    const uint32_t stride = gridDim.x * (VB_K1F_THREADS / 32u);
    constexpr uint32_t NONE = 0xffffffffu;
    auto load_unit = [&](uint32_t u) -> uint32_t {                      // this lane's filter word of unit u (0 past the end)
        if (u >= n_units) return 0u;
        uint32_t g, bits;
        if (a.split_shift) {
            if (lane != 0u) return 0u;
            g = u >> a.split_shift;
            bits = mask ? mask[g] : 0xffffffffu;
            const uint32_t part = u & ((1u << a.split_shift) - 1u);
            bits &= ((1u << part_rows) - 1u) << (part * part_rows);
        } else {
            g = (u << a.unit_shift) + lane;
            if (lane >= U || g >= n_groups) return 0u;
            bits = mask ? mask[g] : 0xffffffffu;
        }
        if ((g << 5) + 32u > a.n_rows) bits &= (1u << (a.n_rows - (g << 5))) - 1u;
        return bits;
    };
    auto unit_g0 = [&](uint32_t u) -> uint32_t { return a.split_shift ? (u >> a.split_shift) : (u << a.unit_shift); };
    uint32_t u_cur = blockIdx.x * (VB_K1F_THREADS / 32u) + warp;
    uint32_t bits = load_unit(u_cur), g0 = unit_g0(u_cur);
    uint32_t u_nxt = u_cur + stride;
    uint32_t bits_nxt = load_unit(u_nxt);
    uint32_t nz = __ballot_sync(0xffffffffu, bits != 0u);               // lanes (groups) of the current unit with rows left
    bool more = true;                                                   // CTA-uniform: some warp still has rows
    for (uint32_t it = 0; more; ++it) {
        // up to 8 batches of 4 rows per warp and iteration: at most 8 x 32 = 256 appends per CTA and iteration
        for (uint32_t bt = 0; bt < 8u; ++bt) {
            uint32_t r[ROWS];
#pragma unroll
            for (int k = 0; k < ROWS; ++k) {
                while (nz == 0u && u_cur < n_units) {                   // unit exhausted: the prefetched one becomes current
                    u_cur = u_nxt; bits = bits_nxt; g0 = unit_g0(u_cur);
                    u_nxt += stride; bits_nxt = load_unit(u_nxt);
                    nz = __ballot_sync(0xffffffffu, bits != 0u);
                }
                if (nz) {
                    const uint32_t j = __ffs(nz) - 1u;
                    uint32_t bj = __shfl_sync(0xffffffffu, bits, j);
                    r[k] = ((g0 + j) << 5) + (__ffs(bj) - 1u);
                    bj &= bj - 1u;
                    if (lane == j) bits = bj;
                    if (bj == 0u) nz &= nz - 1u;
                } else r[k] = NONE;
            }
            if (r[0] == NONE) break;                                    // warp-uniform: nothing left for this warp
            uint32_t myr = r[0];
#pragma unroll
            for (int k = 1; k < ROWS; ++k)
                if (lane == (uint32_t)k) myr = r[k];
            const float inv_r = (lane < (uint32_t)ROWS && myr != NONE) ? a.inv_norm[myr] : 0.0f;
            uint4 v[ROWS][NCH];
#pragma unroll
            for (int k = 0; k < ROWS; ++k)
#pragma unroll
                for (int c = 0; c < NCH; ++c) {
                    const uint32_t ch = lane + 32u * c;
                    v[k][c] = (r[k] != NONE && ch < a.chunks) ? vb_ldg_stream(a.rows + (size_t)r[k] * a.chunks + ch)
                                                              : make_uint4(0u, 0u, 0u, 0u);
                }
#pragma unroll
            for (int k = 0; k < ROWS; ++k)
#pragma unroll
                for (int c = 0; c < NCH; ++c) vb_keep_loaded(v[k][c]);
            float acc[ROWS];
#pragma unroll
            for (int k = 0; k < ROWS; ++k) {
                acc[k] = 0.0f;
#pragma unroll
                for (int c = 0; c < NCH; ++c) acc[k] = vb_dot8(v[k][c], q[c], acc[k]);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1)
#pragma unroll
                for (int k = 0; k < ROWS; ++k) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
            float mine = acc[0];
#pragma unroll
            for (int k = 1; k < ROWS; ++k)
                if (lane == (uint32_t)k) mine = acc[k];
            if (lane < (uint32_t)ROWS && myr != NONE) {
                const float s = mine * inv_r;
                if (s >= tau) {                                         // ties stay: rows do not arrive in row order
                    const uint32_t slot = atomicAdd(&s_cnt, 1u);
                    if (slot < VB_K1F_CAP) s_keys[slot] = vb_pack_key(s, a.row_base + myr);
                }
            }
        }
        // every VB_K1F_CHECK iterations: is anybody still working?  re-select if the next stretch could overflow
        if ((it + 1u) % VB_K1F_CHECK == 0u) {
            more = __syncthreads_or((nz != 0u || u_cur < n_units) ? 1 : 0) != 0;
            const bool last = !more;
            const uint32_t c = s_cnt;                                   // <= CAP: a stretch appends at most CAP/2, a selection leaves <= k <= CAP/2
            VB_CHECK(c <= VB_K1F_CAP);
            if (last || c > VB_K1F_CAP - VB_K1F_CHECK * VB_K1F_THREADS) {
                uint32_t P = 2;
                while (P < c) P <<= 1;
                for (uint32_t i = c + threadIdx.x; i < P; i += VB_K1F_THREADS) s_keys[i] = 0ull;
                vb_k1f_sort(s_keys, P);
                const uint32_t keep = c < a.k ? c : a.k;
                if (threadIdx.x == 0) {
                    s_cnt = keep;
                    if (keep >= a.k) {
                        const uint32_t o = (uint32_t)(s_keys[a.k - 1u] >> 32);      // ordered encoding of the k'-th score
                        atomicMax(a.gtau + list, o);
                    }
                }
            }
            if (!last) {
                if (threadIdx.x == 0) {                                 // best threshold known anywhere
                    const uint32_t o = *reinterpret_cast<volatile uint32_t*>(a.gtau + list);
                    s_tau = o ? __uint_as_float(vb_ordered_f32(o)) : -INFINITY;
                }
                __syncthreads();
                tau = s_tau;
            }
        }
    }
    __syncthreads();
    // local top-k' -> the list.  Only entries at or above the best threshold known anywhere can be in the global
    // top-k' (the local list is sorted: they are a prefix); the CTA reserves that many slots with ONE atomic on the
    // list's counter (pre-set to 0 by the list set-up; at most G * k' <= cap in total) and the merge sees a few hundred
    // keys instead of G * k'.
    const uint32_t keep = s_cnt;
    VB_CHECK(keep <= a.k && keep <= VB_K1F_CAP);
    __shared__ uint32_t s_take, s_base;
    if (threadIdx.x == 0) {
        const uint32_t o = *reinterpret_cast<volatile uint32_t*>(a.gtau + list);
        uint32_t lo = 0, hi = keep;                              // first index whose ordered score is below the threshold
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if ((uint32_t)(s_keys[mid] >> 32) >= o) lo = mid + 1u; else hi = mid;
        }
        s_take = lo;
        s_base = lo ? atomicAdd(a.cnt + (size_t)list * VB_SUB, lo) : 0u;
    }
    __syncthreads();
    uint64_t* out = a.cand + (size_t)list * a.cap + s_base;
    VB_CHECK(s_base + s_take <= a.cap);
    for (uint32_t i = threadIdx.x; i < s_take; i += VB_K1F_THREADS) out[i] = s_keys[i];
    // ---- merge, by the last CTA of the list to get here (what a vb_compact_kernel launch did before: ~25 us of
    // launch + cold instruction fetch for a few hundred keys).  Every CTA publishes its keys (fence), then takes a
    // ticket; the CTA with the last ticket sees every other CTA's keys.
    __shared__ uint32_t s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(a.done + list, 1u) == gridDim.x - 1u ? 1u : 0u;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    uint64_t* in = a.cand + (size_t)list * a.cap;
    const uint32_t total = min(*reinterpret_cast<volatile uint32_t*>(a.cnt + (size_t)list * VB_SUB), a.cap);
    uint32_t kept = 0;
    // Every CTA has published by now: gtau is the best k'-th score any CTA holds, and that CTA's k' keys at or above it
    // were all appended (a CTA appends what reaches the threshold it sees, which is never above the final one).  Keys
    // below it cannot be in the global top-k': keep only the others — a few dozen instead of a few hundred to sort.
    {
        const uint32_t o_fin = *reinterpret_cast<volatile uint32_t*>(a.gtau + list);
        if (threadIdx.x == 0) s_cnt = 0u;
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < total; i += VB_K1F_THREADS) {
            const uint64_t key = __ldcg(in + i);
            if ((uint32_t)(key >> 32) >= o_fin) {
                const uint32_t slot = atomicAdd(&s_cnt, 1u);
                if (slot < VB_K1F_CAP) s_keys[slot] = key;
            }
        }
        __syncthreads();
        const uint32_t c = s_cnt;
        if (c <= VB_K1F_CAP) {
            uint32_t P = 2;
            while (P < c) P <<= 1;
            for (uint32_t i = c + threadIdx.x; i < P; i += VB_K1F_THREADS) s_keys[i] = 0ull;
            vb_k1f_sort(s_keys, P);
            kept = c < a.k ? c : a.k;
            for (uint32_t i = threadIdx.x; i < kept; i += VB_K1F_THREADS) in[i] = s_keys[i];
            if (threadIdx.x == 0) {
                a.cnt[(size_t)list * VB_SUB] = kept;
                a.tau[list] = fmaxf(a.tau[list], kept >= a.k ? vb_key_score(s_keys[a.k - 1u]) : -INFINITY);
                a.done[list] = 0u;
            }
            return;
        }
        __syncthreads();                                              // more survivors than slots (no threshold yet): the chunked merge below
    }
    for (uint32_t pos = 0; pos < total;) {                            // 2048 slots: (kept so far) + the next stretch of keys
        const uint32_t take = min(VB_K1F_CAP - kept, total - pos);
        for (uint32_t i = threadIdx.x; i < take; i += VB_K1F_THREADS) s_keys[kept + i] = __ldcg(in + pos + i);
        pos += take;
        const uint32_t c = kept + take;
        uint32_t P = 2;
        while (P < c) P <<= 1;
        for (uint32_t i = c + threadIdx.x; i < P; i += VB_K1F_THREADS) s_keys[i] = 0ull;
        vb_k1f_sort(s_keys, P);
        kept = c < a.k ? c : a.k;
    }
    for (uint32_t i = threadIdx.x; i < kept; i += VB_K1F_THREADS) in[i] = s_keys[i];
    if (threadIdx.x == 0) {
        a.cnt[(size_t)list * VB_SUB] = kept;                          // sub-ranges 1.. were never used by this pass
        a.tau[list] = fmaxf(a.tau[list], kept >= a.k ? vb_key_score(s_keys[a.k - 1u]) : -INFINITY);
        a.done[list] = 0u;
    }
}
