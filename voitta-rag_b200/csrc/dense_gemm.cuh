// K2 — batched dense scoring on the 5th-gen tensor cores (tcgen05 + TMEM, TMA-fed) with the
// filter bitmask and the top-k' threshold fused into the epilogue: the B x N score matrix is
// never written to memory.
// Replaces qdrant's cosine scoring for a BATCH of query_points(query=vec, limit=k', filter)
// calls (vector_store.py:640-645).  voitta issues B = 1; batches come from search_batch().
//
// Shape: D[128 rows, BN queries] = A[128 x d] (corpus tile, bf16, K-major) * Q[BN x d]^T
//   - persistent kernel, one CTA per SM, tiles of 128 corpus rows, round-robin over CTAs;
//   - warp 0: TMA producer — corpus tiles stream through an S-stage ring of 128x64 bf16 boxes
//     (16 KB, 128B swizzle), the query matrix is loaded once and stays resident in smem;
//   - warp 1: allocates TMEM (512 columns) and issues tcgen05.mma (M=128, N=BN, K=16) from one
//     elected lane; accumulators are double buffered in TMEM (2 x 256 columns);
//   - warps 2-5: epilogue — tcgen05.ld the accumulator (lane = corpus row, column = query),
//     score = acc * inv_norm[row], test the filter bit and the per-query threshold tau, and
//     append survivors to the query's candidate list (warp-ballot skips the common no-survivor
//     case).  vb_compact_kernel then selects the exact top-k'.
// Roofline: HBM for BN <~ 250 (one pass over the bf16 corpus per sub-batch), tensor pipe above.
// Algorithmic bytes per launch = rows*(d_pad*2 + 4) + mask words; flops = 2*rows*BN*d_pad.
#pragma once
#include "common.cuh"
#include <cuda.h>
#include <string>
#include <algorithm>

#define VB_GEMM_THREADS 320          // warp 0 TMA, warp 1 MMA, warps 2-9 epilogue (two per TMEM lane quadrant)
#define VB_TILE_M 128u
#define VB_BLOCK_K 64u
#define VB_STAGE_BYTES (VB_TILE_M * VB_BLOCK_K * 2u)   // 16 KB
#define VB_GEMM_MAX_FILTERS 256u       // mask words the epilogue caches per warp: one per filter of a query tile (<= 256 queries)

// Mask mode 3 (more than 31 distinct filters in the batch): the filters each query tile uses, so that the epilogue's
// per-warp mask-word cache is indexed by a tile-local id.  A tile holds at most 256 queries, hence at most 256 filters,
// whatever the batch holds in all.  Built on the host with the batch (vb_api.cu prepare_batch), one set per tile size.
// When all tiles of one launch use at most 256 filters between them, they share one list (n[t] carries
// VB_FTAB_SHARED): K2T then loads the mask words once per corpus tile instead of once per (corpus tile, query tile).
#define VB_FTAB_SHARED 0x80000000u
struct VbFilterTiles {
    const int32_t* loc = nullptr;    // [B] index of the query's filter in its tile's list, -1 = unfiltered
    const uint32_t* n = nullptr;     // [tiles] filters listed per tile (| VB_FTAB_SHARED: the launch's tiles share the list)
    const int32_t* ids = nullptr;    // [tiles][VB_GEMM_MAX_FILTERS] batch-wide filter id of each listed filter
    uint32_t tile = 0;               // queries per tile (0: no tables)
};

// mode 3: this warp's mask word (32 rows) of every listed filter, lane l loading entries l, l + 32, ...
__device__ __forceinline__ void vb_cache_mask_words(uint32_t* mw, const uint32_t* mask, const int32_t* tab, uint32_t nf,
                                                    uint32_t mask_words, uint32_t word, uint32_t lane) {
    for (uint32_t l = lane; l < nf; l += 32u)
        mw[l] = word < mask_words ? mask[(size_t)tab[l] * mask_words + word] : 0u;
}

static std::string g_gemm_err;
static const char* vb_gemm_last_error() { return g_gemm_err.c_str(); }

// ---- PTX wrappers -------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t vb_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void vb_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void vb_mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred P1;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void vb_mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void vb_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void vb_tma_load_2d(uint32_t dst, const CUtensorMap* map, int32_t c0, int32_t c1, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void vb_tma_load_3d(uint32_t dst, const CUtensorMap* map, int32_t c0, int32_t c1, int32_t c2, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ void vb_tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void vb_tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void vb_tcgen05_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void vb_tcgen05_mma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// 32 lanes x 16 consecutive columns, one fp32 per (lane, column)
__device__ __forceinline__ void vb_tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void vb_tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ float4 vb_lds_f4(uint32_t addr) {
    float4 r;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(addr));
    return r;
}
__device__ __forceinline__ int4 vb_lds_i4(uint32_t addr) {
    int4 r;
    asm volatile("ld.shared.v4.s32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr));
    return r;
}
__device__ __forceinline__ uint32_t vb_lds_u32(uint32_t addr) {
    uint32_t r;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(r) : "r"(addr));
    return r;
}

// UMMA shared-memory descriptor: K-major operand, 128-byte swizzle, 8-row groups 1024 B apart
// (bits: [0,14) addr>>4, [16,30) LBO>>4 = 0, [32,46) SBO>>4 = 64, [46,48) version = 1,
//  [61,64) layout = 2 (SWIZZLE_128B)).
__device__ __forceinline__ uint64_t vb_umma_desc(uint32_t smem_addr) {
    return (uint64_t)((smem_addr & 0x3ffffu) >> 4) | ((uint64_t)(1024u >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// UMMA instruction descriptor, kind::f16: D = f32, A = B = bf16, both K-major, M = 128, N = bn
__host__ __device__ __forceinline__ uint32_t vb_umma_idesc(uint32_t bn) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((bn >> 3) << 17) | ((VB_TILE_M >> 4) << 24);
}

// Plain-bf16 query precision: rounding the unit query to bf16 changes its length by up to ~2e-3, which
// would scale every score of that query.  The epilogue therefore multiplies by q_scale = 1/|bf16(q)|
// (exact cosine against the rounded query; only the direction error, ~2e-4, remains).  The hot loop
// compares the unscaled value against a pre-threshold tau/q_scale lowered by a safety margin; the
// rare survivor path applies the scale and repeats the comparison exactly.
__device__ __forceinline__ float vb_pre_threshold(float tau, float qs) {
    const float t = tau / qs;
    return t > 0.0f ? t * (1.0f - 1e-6f) : t * (1.0f + 1e-6f);
}

struct VbGemmArgs {
    const float* inv_norm;
    const uint32_t* mask;      // [n_filters][mask_words] or nullptr
    const int32_t* mask_of;    // [B_total] or nullptr; mask_mode 3: the tile-local ids (VbFilterTiles::loc)
    const uint32_t* ftab_n;    // mask_mode 3: [1] filters listed for this sub-batch
    const int32_t* ftab;       // mask_mode 3: [ftab_n[0]] their batch-wide ids
    const float* tau;          // [n_lists]
    const float* q_scale;      // [B_total] 1/|bf16(q)| (1 for the bf16x2 query)
    VbLists lists;
    uint32_t mask_words, n_filters;
    uint32_t tile_begin, tile_end;   // 128-row tiles of this segment
    uint32_t row_end;                // rows >= row_end are not part of the segment
    uint32_t row_base;
    uint32_t k_blocks;               // d_pad / 64
    uint32_t bn;                     // padded sub-batch (multiple of 16, <= 256)
    uint32_t n_q;                    // real queries in this sub-batch
    uint32_t q_begin;                // first query (list index) of the sub-batch
    uint32_t stages;
    uint32_t direct;                 // 1: first segment — write every key to slot (row - row_begin), no atomics
    uint32_t mask_mode;              // 0 none, 1 one filter for the whole sub-batch, 2 <= 31 filters, 3 general
    int32_t  uniform_filter;         // mask_mode 1: the filter index
    uint32_t split;                  // 1: columns [0,bn/2) hold q_hi, [bn/2,bn) hold q_lo (bf16x2 query precision)
    uint32_t kbox;                   // K-blocks (of 64) per TMA box / pipeline stage
    // SEL (dense_compact.cuh): sel[1] != 0 -> walk the compacted copy of the rows that pass the shared filter instead
    const uint32_t* sel;             // [0] rows of the copy, [1] decision (taken on the device)
    const uint32_t* sel_ids;         // [rows of the copy] shard row id of each copied row
    const float* sel_inv_norm;       // [rows of the copy]
};

// MODE: per-column mask handling (0 = none / one filter folded into the row scale, 2 = <= 31
// filters via a per-row bit set, 3 = general); SPLIT: bf16x2 query; DIRECT: first-segment stores.
// They are template parameters so that the per-column epilogue code is branch-free.
template <int MODE, bool SPLIT, bool DIRECT, bool SEL>
__global__ void __launch_bounds__(VB_GEMM_THREADS, 1)
vb_dense_gemm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_q,
                     const __grid_constant__ CUtensorMap tmap_c, const VbGemmArgs a)
{
    extern __shared__ unsigned char vb_gemm_smem_raw[];
    // 1024-byte alignment for the 128B-swizzle atoms
    unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)vb_gemm_smem_raw + 1023u) & ~(uintptr_t)1023u);
    const uint32_t q_bytes = a.bn * a.k_blocks * 128u;                       // resident query matrix
    unsigned char* smem_q = smem;
    unsigned char* smem_a = smem + q_bytes;                                   // stages * 16 KB (q_bytes % 1024 == 0)
    const uint32_t stage_bytes = a.kbox * VB_STAGE_BYTES;
    unsigned char* tail = smem_a + a.stages * stage_bytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(tail);                       // full[S], empty[S], tfull[2], tempty[2], qfull
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tail + 8u * (2u * 16u + 5u));
    float* tau_s = reinterpret_cast<float*>(tail + 320u);                         // [256], 16-byte aligned
    int32_t* mof_s = reinterpret_cast<int32_t*>(tau_s + 256);                     // [256]
    float* tex_s = reinterpret_cast<float*>(mof_s + 256);                         // [256] exact thresholds
    float* qs_s = tex_s + 256;                                                    // [256] query scales
    uint32_t* mw_s = reinterpret_cast<uint32_t*>(qs_s + 256);                     // [8 epilogue warps][VB_GEMM_MAX_FILTERS]

    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t S = a.stages;
    const uint32_t bar_full = vb_smem_u32(bars), bar_empty = bar_full + 8u * 16u;
    const uint32_t bar_tfull = bar_full + 8u * 32u, bar_tempty = bar_tfull + 16u, bar_q = bar_tfull + 32u;

    if (warp == 1) {
        if (lane == 0) {
            for (uint32_t s = 0; s < S; ++s) { vb_mbar_init(bar_full + 8u * s, 1); vb_mbar_init(bar_empty + 8u * s, 1); }
            for (uint32_t s = 0; s < 2; ++s) { vb_mbar_init(bar_tfull + 8u * s, 1); vb_mbar_init(bar_tempty + 8u * s, 8); }
            vb_mbar_init(bar_q, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(vb_smem_u32(tmem_ptr)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    for (uint32_t c = threadIdx.x; c < 256u; c += blockDim.x) {
        const bool live = c < a.n_q;
        const float t = live ? a.tau[a.q_begin + c] : INFINITY;
        const float qs = live ? a.q_scale[a.q_begin + c] : 1.0f;
        tex_s[c] = t;
        qs_s[c] = qs;
        tau_s[c] = SPLIT ? t : vb_pre_threshold(t, qs);        // bf16x2 query: no scale, the hot compare is exact
        mof_s[c] = (live && a.mask_of) ? a.mask_of[a.q_begin + c] : -1;
        VB_CHECK(MODE != 3 || mof_s[c] < (int32_t)(a.ftab_n[0] & ~VB_FTAB_SHARED));
    }
    vb_tcgen05_fence_before();
    __syncthreads();
    vb_tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    // SEL: the row-selection kernels decided (on the device) whether this launch walks the compacted copy
    const bool cmp = SEL && a.sel[1] != 0u;
    const uint32_t tile_begin = cmp ? 0u : a.tile_begin;
    const uint32_t row_end = cmp ? a.sel[0] : a.row_end;
    const uint32_t n_tiles = cmp ? (a.sel[0] + VB_TILE_M - 1u) / VB_TILE_M : a.tile_end - a.tile_begin;
    const uint32_t n_tab = MODE == 3 ? a.ftab_n[0] & ~VB_FTAB_SHARED : 0u;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            const CUtensorMap* tmap_rows = cmp ? &tmap_c : &tmap_a;
            vb_mbar_expect_tx(bar_q, q_bytes);
            for (uint32_t kb = 0; kb < a.k_blocks; ++kb)
                vb_tma_load_2d(vb_smem_u32(smem_q + kb * a.bn * 128u), &tmap_q, (int32_t)(kb * VB_BLOCK_K), 0, bar_q);
            uint32_t stage = 0, phase = 0;
            for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
                const int32_t row0 = (int32_t)((tile_begin + t) * VB_TILE_M);
                for (uint32_t kb = 0; kb < a.k_blocks; kb += a.kbox) {
                    vb_mbar_wait(bar_empty + 8u * stage, phase ^ 1u);
                    vb_mbar_expect_tx(bar_full + 8u * stage, stage_bytes);
                    // one box = 128 rows x kbox K-blocks: [kb][row][64] in smem, i.e. kbox UMMA slabs
                    vb_tma_load_3d(vb_smem_u32(smem_a + stage * stage_bytes), tmap_rows, 0, row0, (int32_t)kb, bar_full + 8u * stage);
                    if (++stage == S) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (one elected lane) =====
        if (lane == 0) {
            const uint32_t idesc = vb_umma_idesc(a.bn);
            vb_mbar_wait(bar_q, 0);
            uint32_t stage = 0, phase = 0, it = 0;
            for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x, ++it) {
                const uint32_t acc = it & 1u;
                vb_mbar_wait(bar_tempty + 8u * acc, ((it >> 1) & 1u) ^ 1u);
                vb_tcgen05_fence_after();
                const uint32_t tmem_d = tmem_base + acc * 256u;
                for (uint32_t kb0 = 0; kb0 < a.k_blocks; kb0 += a.kbox) {
                    vb_mbar_wait(bar_full + 8u * stage, phase);
                    vb_tcgen05_fence_after();
                    const uint32_t nkb = min(a.kbox, a.k_blocks - kb0);
                    for (uint32_t kk = 0; kk < nkb; ++kk) {
                        const uint32_t kb = kb0 + kk;
                        const uint32_t a_addr = vb_smem_u32(smem_a + stage * stage_bytes + kk * VB_STAGE_BYTES);
                        const uint32_t q_addr = vb_smem_u32(smem_q + kb * a.bn * 128u);
#pragma unroll
                        for (uint32_t k = 0; k < VB_BLOCK_K / 16u; ++k)
                            vb_tcgen05_mma_bf16(tmem_d, vb_umma_desc(a_addr + k * 32u), vb_umma_desc(q_addr + k * 32u), idesc, (kb | k) != 0u);
                    }
                    vb_tcgen05_commit(bar_empty + 8u * stage);     // smem stage free once these MMAs retire
                    if (++stage == S) { stage = 0; phase ^= 1u; }
                }
                vb_tcgen05_commit(bar_tfull + 8u * acc);           // accumulator ready for the epilogue
            }
        }
    } else {
        // ===== epilogue warps 2..9; TMEM lane quadrant = warp % 4, two warps per quadrant that
        //       split the 16-column chunks between them (even / odd) =====
        // Branch-free per column: 16 columns are compared against their thresholds into a bit
        // mask, ONE warp vote per 16-column chunk decides whether the (rare) append path runs.
        const uint32_t quad = warp & 3u;
        const uint32_t half = (warp - 2u) >> 2;            // 0: even chunks, 1: odd chunks
        const uint32_t tau_addr = vb_smem_u32(tau_s), mof_addr = vb_smem_u32(mof_s), qs_addr = vb_smem_u32(qs_s), tex_addr = vb_smem_u32(tex_s);
        const uint32_t mw_addr = vb_smem_u32(mw_s + (warp - 2u) * VB_GEMM_MAX_FILTERS);
        uint32_t* mw = mw_s + (warp - 2u) * VB_GEMM_MAX_FILTERS;   // private: the two warps of a quadrant may be one tile apart
        constexpr uint32_t mode = (uint32_t)MODE;
        constexpr bool split = SPLIT;
        const uint32_t ncol = split ? a.bn >> 1 : a.bn;       // query columns handled by the epilogue
        const float qnan = __int_as_float(0x7fc00000);
        uint32_t it = 0;
        for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x, ++it) {
            const uint32_t acc = it & 1u;
            const uint32_t tile = tile_begin + t;
            const uint32_t pos = tile * VB_TILE_M + quad * 32u + lane;       // row of the matrix this launch walks
            const bool row_ok = pos < row_end;
            // the shard row behind it: itself, or (compacted copy) the id the selection recorded
            const uint32_t row = cmp ? (row_ok ? a.sel_ids[pos] : 0u) : pos;
            VB_CHECK(row < a.row_end || !row_ok);
            // global loads are issued before blocking on the accumulator.
            // A row that is out of range or (modes 0/1) masked gets a NaN scale: every compare fails.
            float invn = row_ok ? (cmp ? a.sel_inv_norm[pos] : a.inv_norm[pos]) : qnan;
            const uint32_t word = tile * 4u + quad;
            uint32_t fbits = 0x80000000u;                 // mode 2: bit f = row passes filter f; bit 31 = unfiltered
            if (MODE == 0 && a.mask_mode == 1u && !cmp) { // (every row of the compacted copy passes the shared filter)
                const uint32_t w = word < a.mask_words ? a.mask[(size_t)a.uniform_filter * a.mask_words + word] : 0u;
                if (!((w >> lane) & 1u)) invn = qnan;
            } else if (mode == 2u) {
                const uint32_t w = (lane < a.n_filters && word < a.mask_words) ? a.mask[(size_t)lane * a.mask_words + word] : 0u;
                for (uint32_t f = 0; f < a.n_filters; ++f)
                    fbits |= ((__shfl_sync(0xffffffffu, w, f) >> lane) & 1u) << f;
            } else if (mode == 3u) {
                __syncwarp();
                vb_cache_mask_words(mw, a.mask, a.ftab, n_tab, a.mask_words, word, lane);
                __syncwarp();
            }
            vb_mbar_wait(bar_tfull + 8u * acc, (it >> 1) & 1u);
            vb_tcgen05_fence_after();
            const uint32_t taddr = tmem_base + ((quad * 32u) << 16) + acc * 256u;
            const uint32_t slot = row - a.tile_begin * VB_TILE_M;      // direct mode: position inside the segment
            // one 16-column chunk: compare, then (rarely) append — or, in direct mode, store all
            auto process = [&](const uint32_t (&v)[16], const uint32_t (&w)[16], uint32_t c0) {
                uint32_t m = 0;
#pragma unroll
                for (uint32_t j4 = 0; j4 < 4u; ++j4) {
                    const float4 tq = vb_lds_f4(tau_addr + (c0 + 4u * j4) * 4u);
                    const float tv[4] = {tq.x, tq.y, tq.z, tq.w};
                    int fv[4] = {-1, -1, -1, -1};
                    if (mode >= 2u) {
                        const int4 fq = vb_lds_i4(mof_addr + (c0 + 4u * j4) * 4u);
                        fv[0] = fq.x; fv[1] = fq.y; fv[2] = fq.z; fv[3] = fq.w;
                    }
#pragma unroll
                    for (uint32_t e = 0; e < 4u; ++e) {
                        const uint32_t j = 4u * j4 + e;
                        const float sc = (split ? __uint_as_float(v[j]) + __uint_as_float(w[j]) : __uint_as_float(v[j])) * invn;
                        uint32_t p = sc > tv[e] ? 1u : 0u;                    // tau = +inf for padded columns
                        if (mode == 2u) p &= fbits >> ((uint32_t)fv[e] & 31u);
                        else if (mode == 3u) p &= fv[e] < 0 ? 1u : (vb_lds_u32(mw_addr + (uint32_t)fv[e] * 4u) >> lane);
                        m |= (p & 1u) << j;
                    }
                }
                // final score of column c0 + j (query scale applied) and the exact comparison
                auto final_score = [&](uint32_t j) -> float {
                    if (split) return (__uint_as_float(v[j]) + __uint_as_float(w[j])) * invn;
                    return __uint_as_float(v[j]) * invn * qs_s[c0 + j];
                };
                if (DIRECT) {
                    if (row_ok) {
#pragma unroll
                        for (uint32_t j = 0; j < 16u; ++j) {
                            const uint32_t col = c0 + j;
                            if (col < a.n_q) {
                                const float fs = final_score(j);
                                a.lists.cand[(size_t)(a.q_begin + col) * a.lists.cap + slot] =
                                    (((m >> j) & 1u) && (split || fs > tex_s[col])) ? vb_pack_key(fs, a.row_base + row) : 0ull;
                            }
                        }
                    }
                } else {
                    // rare path: mm has a bit for every column in which some row of the warp survived the
                    // pre-threshold (warp-uniform) — a COMPACT loop over those columns (vb_append_flagged)
                    const uint32_t mm = __reduce_or_sync(0xffffffffu, m);
                    if (mm != 0u)
                        vb_append_flagged(a.lists, a.q_begin + c0, blockIdx.x & a.lists.sub_mask, mm, m, lane, (1u << lane) - 1u, a.row_base + row,
                                          [&](uint32_t j) -> float {
                                              if (split) return (__uint_as_float(vb_sel16(v, j)) + __uint_as_float(vb_sel16(w, j))) * invn;
                                              return __uint_as_float(vb_sel16(v, j)) * invn * __uint_as_float(vb_lds_u32(qs_addr + (c0 + j) * 4u));
                                          },
                                          [&](uint32_t j, float fs) -> bool { return split || fs > __uint_as_float(vb_lds_u32(tex_addr + (c0 + j) * 4u)); });
                }
            };
            uint32_t va[16], vb[16], wa[16], wb[16];
            auto load = [&](uint32_t (&v)[16], uint32_t (&w)[16], uint32_t c0) {
                vb_tmem_ld16(taddr + c0, v);
                if (split) vb_tmem_ld16(taddr + ncol + c0, w);
            };
            // this warp's chunks: 16*(2i + half); the next one is in flight while one is processed
            const uint32_t first = 16u * half;
            if (first < ncol) load(va, wa, first);
            for (uint32_t c0 = first; c0 < ncol; c0 += 64u) {
                vb_tmem_ld_wait();
                const bool second = c0 + 32u < ncol;
                if (second) load(vb, wb, c0 + 32u);
                process(va, wa, c0);
                if (second) {
                    vb_tmem_ld_wait();
                    if (c0 + 64u < ncol) load(va, wa, c0 + 64u);
                    process(vb, wb, c0 + 32u);
                }
            }
            vb_tcgen05_fence_before();
            __syncwarp();
            if (lane == 0) vb_mbar_arrive(bar_tempty + 8u * acc);
        }
    }
    vb_tcgen05_fence_before();
    __syncthreads();
    if (warp == 1) {
        vb_tcgen05_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    }
}

// ---- K2T: tensor-bound variant for large batches ------------------------------------------------------
// For B above what fits resident in shared memory the kernel above needs one pass over the corpus
// per sub-batch (HBM-bound: ~96 queries per pass at d = 768).  This variant tiles the QUERY dimension
// instead: D[128 rows x 256 queries] tiles, both operands streamed through the TMA ring (16 KB corpus
// box + 32 KB query box per 64-wide K block), accumulators double-buffered in TMEM (2 x 256
// columns).  A CTA walks all query tiles of a corpus tile back to back, so the corpus tile comes from
// HBM once and from L2 afterwards, and the query tiles (shared by all CTAs) stay L2-resident:
// HBM traffic is ONE pass over the corpus per <= 1024 queries and the tensor pipe is the roofline
// (flops = 2 * rows * B * d_pad).  Epilogue as above (threshold + mask + append, no score matrix).
#define VB_TILE_N 256u
#define VB_TILED_MAX_Q 1024u
#define VB_TILED_STAGE_BYTES (VB_STAGE_BYTES + VB_TILE_N * VB_BLOCK_K * 2u)     // 48 KB

struct VbGemmTiledArgs {
    const float* inv_norm;
    const uint32_t* mask;      // [n_filters][mask_words] or nullptr
    const int32_t* mask_of;    // [B_total] or nullptr; mask_mode 3: the tile-local ids (VbFilterTiles::loc)
    const uint32_t* ftab_n;    // mask_mode 3: [query tiles of this launch] filters listed per tile
    const int32_t* ftab;       // mask_mode 3: [query tiles of this launch][VB_GEMM_MAX_FILTERS] their batch-wide ids
    const float* tau;          // [n_lists]
    const float* q_scale;      // [B_total] 1/|bf16(q)|
    VbLists lists;
    uint32_t mask_words, n_filters;
    uint32_t tile_begin, tile_end;   // 128-row tiles of this segment
    uint32_t row_end;                // rows >= row_end are not part of the segment
    uint32_t row_base;
    uint32_t k_blocks;               // d_pad / 64
    uint32_t n_q;                    // queries of this launch (<= VB_TILED_MAX_Q)
    uint32_t q_begin;                // first query (list index) of this launch
    uint32_t stages;
    uint32_t mask_mode;              // 0 none, 1 one filter for all queries, 2 <= 31 filters, 3 general
    int32_t  uniform_filter;
    // SEL (dense_compact.cuh): sel[1] != 0 -> walk the compacted copy of the rows that pass the shared filter instead
    const uint32_t* sel;             // [0] rows of the copy, [1] decision (taken on the device)
    const uint32_t* sel_ids;         // [rows of the copy] shard row id of each copied row
    const float* sel_inv_norm;       // [rows of the copy]
};

template <int MODE, bool DIRECT, bool SEL>
__global__ void __launch_bounds__(VB_GEMM_THREADS, 1)
vb_dense_gemm_tiled_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_q,
                           const __grid_constant__ CUtensorMap tmap_c, const VbGemmTiledArgs a)
{
    extern __shared__ unsigned char vb_gemm_smem_raw[];
    unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)vb_gemm_smem_raw + 1023u) & ~(uintptr_t)1023u);
    unsigned char* tail = smem + a.stages * VB_TILED_STAGE_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(tail);                       // full[16], empty[16], tfull[2], tempty[2]
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tail + 8u * (2u * 16u + 4u));
    float* tau_s = reinterpret_cast<float*>(tail + 320u);                     // [VB_TILED_MAX_Q]
    int32_t* mof_s = reinterpret_cast<int32_t*>(tau_s + VB_TILED_MAX_Q);      // [VB_TILED_MAX_Q]
    float* tex_s = reinterpret_cast<float*>(mof_s + VB_TILED_MAX_Q);          // [VB_TILED_MAX_Q] exact thresholds
    float* qs_s = tex_s + VB_TILED_MAX_Q;                                     // [VB_TILED_MAX_Q] query scales
    uint32_t* mw_s = reinterpret_cast<uint32_t*>(qs_s + VB_TILED_MAX_Q);      // [8 epilogue warps][VB_GEMM_MAX_FILTERS]
    uint64_t* pk_s = reinterpret_cast<uint64_t*>(mw_s + 8u * VB_GEMM_MAX_FILTERS);   // [8 epilogue warps][VB_PEND] parked keys
    uint32_t* pl_s = reinterpret_cast<uint32_t*>(pk_s + 8u * VB_PEND);               // [8 epilogue warps][VB_PEND] their lists

    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
    const uint32_t S = a.stages;
    const uint32_t bar_full = vb_smem_u32(bars), bar_empty = bar_full + 8u * 16u;
    const uint32_t bar_tfull = bar_full + 8u * 32u, bar_tempty = bar_tfull + 16u;

    if (warp == 1) {
        if (lane == 0) {
            for (uint32_t s = 0; s < S; ++s) { vb_mbar_init(bar_full + 8u * s, 1); vb_mbar_init(bar_empty + 8u * s, 1); }
            for (uint32_t s = 0; s < 2; ++s) { vb_mbar_init(bar_tfull + 8u * s, 1); vb_mbar_init(bar_tempty + 8u * s, 8); }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(vb_smem_u32(tmem_ptr)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    for (uint32_t c = threadIdx.x; c < VB_TILED_MAX_Q; c += blockDim.x) {
        const bool live = c < a.n_q;
        const float t = live ? a.tau[a.q_begin + c] : INFINITY;
        const float qs = live ? a.q_scale[a.q_begin + c] : 1.0f;
        tex_s[c] = t;
        qs_s[c] = qs;
        tau_s[c] = vb_pre_threshold(t, qs);
        mof_s[c] = (live && a.mask_of) ? a.mask_of[a.q_begin + c] : -1;
        VB_CHECK(MODE != 3 || !live || mof_s[c] < (int32_t)(a.ftab_n[c / VB_TILE_N] & ~VB_FTAB_SHARED));
    }
    vb_tcgen05_fence_before();
    __syncthreads();
    vb_tcgen05_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    // SEL: the row-selection kernels decided (on the device) whether this launch walks the compacted copy
    const bool cmp = SEL && a.sel[1] != 0u;
    const uint32_t tile_begin = cmp ? 0u : a.tile_begin;
    const uint32_t row_end = cmp ? a.sel[0] : a.row_end;
    const uint32_t n_tiles = cmp ? (a.sel[0] + VB_TILE_M - 1u) / VB_TILE_M : a.tile_end - a.tile_begin;
    const uint32_t n_ntiles = (a.n_q + VB_TILE_N - 1u) / VB_TILE_N;
    const bool tab_once = MODE == 3 && (a.ftab_n[0] & VB_FTAB_SHARED) != 0u;    // one list for all query tiles

    if (warp == 0) {
        // ===== TMA producer: per (corpus tile, query tile, K block) one corpus box + one query box =====
        if (lane == 0) {
            const CUtensorMap* tmap_rows = cmp ? &tmap_c : &tmap_a;
            uint32_t stage = 0, phase = 0;
            for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
                const int32_t row0 = (int32_t)((tile_begin + t) * VB_TILE_M);
                for (uint32_t j = 0; j < n_ntiles; ++j) {
                    for (uint32_t kb = 0; kb < a.k_blocks; ++kb) {
                        vb_mbar_wait(bar_empty + 8u * stage, phase ^ 1u);
                        vb_mbar_expect_tx(bar_full + 8u * stage, VB_TILED_STAGE_BYTES);
                        const uint32_t dst = vb_smem_u32(smem + stage * VB_TILED_STAGE_BYTES);
                        vb_tma_load_2d(dst, tmap_rows, (int32_t)(kb * VB_BLOCK_K), row0, bar_full + 8u * stage);
                        vb_tma_load_2d(dst + VB_STAGE_BYTES, &tmap_q, (int32_t)(kb * VB_BLOCK_K), (int32_t)(j * VB_TILE_N), bar_full + 8u * stage);
                        if (++stage == S) { stage = 0; phase ^= 1u; }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (one elected lane) =====
        if (lane == 0) {
            uint32_t stage = 0, phase = 0, it = 0;
            for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
                for (uint32_t j = 0; j < n_ntiles; ++j, ++it) {
                    const uint32_t ncol = min(VB_TILE_N, (a.n_q - j * VB_TILE_N + 15u) & ~15u);
                    const uint32_t idesc = vb_umma_idesc(ncol);
                    const uint32_t acc = it & 1u;
                    vb_mbar_wait(bar_tempty + 8u * acc, ((it >> 1) & 1u) ^ 1u);
                    vb_tcgen05_fence_after();
                    const uint32_t tmem_d = tmem_base + acc * VB_TILE_N;
                    for (uint32_t kb = 0; kb < a.k_blocks; ++kb) {
                        vb_mbar_wait(bar_full + 8u * stage, phase);
                        vb_tcgen05_fence_after();
                        const uint32_t a_addr = vb_smem_u32(smem + stage * VB_TILED_STAGE_BYTES);
                        const uint32_t q_addr = a_addr + VB_STAGE_BYTES;
#pragma unroll
                        for (uint32_t k = 0; k < VB_BLOCK_K / 16u; ++k)
                            vb_tcgen05_mma_bf16(tmem_d, vb_umma_desc(a_addr + k * 32u), vb_umma_desc(q_addr + k * 32u), idesc, (kb | k) != 0u);
                        vb_tcgen05_commit(bar_empty + 8u * stage);     // smem stage free once these MMAs retire
                        if (++stage == S) { stage = 0; phase ^= 1u; }
                    }
                    vb_tcgen05_commit(bar_tfull + 8u * acc);           // accumulator ready for the epilogue
                }
            }
        }
    } else {
        // ===== epilogue warps 2..9: TMEM lane quadrant = warp % 4, two warps per quadrant split the
        //       16-column chunks (even / odd); branch-free compare, one vote per chunk =====
        const uint32_t quad = warp & 3u;
        const uint32_t half = (warp - 2u) >> 2;
        const uint32_t tau_addr = vb_smem_u32(tau_s), mof_addr = vb_smem_u32(mof_s), qs_addr = vb_smem_u32(qs_s), tex_addr = vb_smem_u32(tex_s);
        const uint32_t mw_addr = vb_smem_u32(mw_s + (warp - 2u) * VB_GEMM_MAX_FILTERS);
        uint32_t* mw = mw_s + (warp - 2u) * VB_GEMM_MAX_FILTERS;   // private: the two warps of a quadrant may be one tile apart
        constexpr uint32_t mode = (uint32_t)MODE;
        const float qnan = __int_as_float(0x7fc00000);
        const uint32_t sub = blockIdx.x & a.lists.sub_mask;
        const uint32_t lane_lt = (1u << lane) - 1u;
        const uint32_t pk_addr = vb_smem_u32(pk_s + (warp - 2u) * VB_PEND), pl_addr = vb_smem_u32(pl_s + (warp - 2u) * VB_PEND);
        uint32_t pn = 0u;                                     // parked candidates of this warp (warp-uniform)
        uint32_t it = 0;
        for (uint32_t t = blockIdx.x; t < n_tiles; t += gridDim.x) {
            const uint32_t tile = tile_begin + t;
            const uint32_t pos = tile * VB_TILE_M + quad * 32u + lane;       // row of the matrix this launch walks
            const bool row_ok = pos < row_end;
            // the shard row behind it: itself, or (compacted copy) the id the selection recorded
            const uint32_t row = cmp ? (row_ok ? a.sel_ids[pos] : 0u) : pos;
            VB_CHECK(row < a.row_end || !row_ok);
            // a row that is out of range or (modes 0/1) masked gets a NaN scale: every compare fails
            float invn = row_ok ? (cmp ? a.sel_inv_norm[pos] : a.inv_norm[pos]) : qnan;
            const uint32_t word = tile * 4u + quad;
            uint32_t fbits = 0x80000000u;                 // mode 2: bit f = row passes filter f; bit 31 = unfiltered
            if (MODE == 0 && a.mask_mode == 1u && !cmp) { // (every row of the compacted copy passes the shared filter)
                const uint32_t w = word < a.mask_words ? a.mask[(size_t)a.uniform_filter * a.mask_words + word] : 0u;
                if (!((w >> lane) & 1u)) invn = qnan;
            } else if (mode == 2u) {
                const uint32_t w = (lane < a.n_filters && word < a.mask_words) ? a.mask[(size_t)lane * a.mask_words + word] : 0u;
                for (uint32_t f = 0; f < a.n_filters; ++f)
                    fbits |= ((__shfl_sync(0xffffffffu, w, f) >> lane) & 1u) << f;
            } else if (mode == 3u && tab_once) {
                __syncwarp();
                vb_cache_mask_words(mw, a.mask, a.ftab, a.ftab_n[0] & ~VB_FTAB_SHARED, a.mask_words, word, lane);
                __syncwarp();
            }
            for (uint32_t j = 0; j < n_ntiles; ++j, ++it) {
                const uint32_t acc = it & 1u;
                const uint32_t qoff = j * VB_TILE_N;
                const uint32_t ncol = min(VB_TILE_N, (a.n_q - qoff + 15u) & ~15u);
                if (mode == 3u && !tab_once) {
                    // this query tile's own list (loads issued before blocking on the accumulator); the warp's previous
                    // tile has been fully read from mw (the __syncwarp that ends it)
                    vb_cache_mask_words(mw, a.mask, a.ftab + (size_t)j * VB_GEMM_MAX_FILTERS, a.ftab_n[j], a.mask_words, word, lane);
                    __syncwarp();
                }
                vb_mbar_wait(bar_tfull + 8u * acc, (it >> 1) & 1u);
                vb_tcgen05_fence_after();
                const uint32_t taddr = tmem_base + ((quad * 32u) << 16) + acc * VB_TILE_N;
                auto process = [&](const uint32_t (&v)[16], uint32_t c0) {
                    uint32_t m = 0;
#pragma unroll
                    for (uint32_t j4 = 0; j4 < 4u; ++j4) {
                        const float4 tq = vb_lds_f4(tau_addr + (qoff + c0 + 4u * j4) * 4u);
                        const float tv[4] = {tq.x, tq.y, tq.z, tq.w};
                        int fv[4] = {-1, -1, -1, -1};
                        if (mode >= 2u) {
                            const int4 fq = vb_lds_i4(mof_addr + (qoff + c0 + 4u * j4) * 4u);
                            fv[0] = fq.x; fv[1] = fq.y; fv[2] = fq.z; fv[3] = fq.w;
                        }
#pragma unroll
                        for (uint32_t e = 0; e < 4u; ++e) {
                            const uint32_t jj = 4u * j4 + e;
                            const float sc = __uint_as_float(v[jj]) * invn;
                            uint32_t p = sc > tv[e] ? 1u : 0u;                    // tau = +inf for padded columns
                            if (mode == 2u) p &= fbits >> ((uint32_t)fv[e] & 31u);
                            else if (mode == 3u) p &= fv[e] < 0 ? 1u : (vb_lds_u32(mw_addr + (uint32_t)fv[e] * 4u) >> lane);
                            m |= (p & 1u) << jj;
                        }
                    }
                    if (DIRECT) {
                        // first segment: every key goes to its fixed slot (row - segment begin), no atomics
                        if (row_ok) {
                            const uint32_t dslot = row - a.tile_begin * VB_TILE_M;
#pragma unroll
                            for (uint32_t jj = 0; jj < 16u; ++jj) {
                                const uint32_t col = qoff + c0 + jj;
                                if (col < a.n_q) {
                                    const float fs = __uint_as_float(v[jj]) * invn * qs_s[col];
                                    a.lists.cand[(size_t)(a.q_begin + col) * a.lists.cap + dslot] =
                                        (((m >> jj) & 1u) && fs > tex_s[col]) ? vb_pack_key(fs, a.row_base + row) : 0ull;
                                }
                            }
                        }
                    } else {
                        // rare path (see the resident kernel): a COMPACT loop over the flagged columns
                        const uint32_t mm = __reduce_or_sync(0xffffffffu, m);
                        if (mm != 0u)
                            pn = vb_park_flagged(a.lists, a.q_begin + qoff + c0, sub, mm, m, lane_lt, a.row_base + row, pk_addr, pl_addr, pn, lane,
                                              [&](uint32_t jj) -> float { return __uint_as_float(vb_sel16(v, jj)) * invn * __uint_as_float(vb_lds_u32(qs_addr + (qoff + c0 + jj) * 4u)); },
                                              [&](uint32_t jj, float fs) -> bool { return fs > __uint_as_float(vb_lds_u32(tex_addr + (qoff + c0 + jj) * 4u)); });
                    }
                };
                uint32_t va[16], vb[16];
                const uint32_t first = 16u * half;
                if (first < ncol) vb_tmem_ld16(taddr + first, va);
                for (uint32_t c0 = first; c0 < ncol; c0 += 64u) {
                    vb_tmem_ld_wait();
                    const bool second = c0 + 32u < ncol;
                    if (second) vb_tmem_ld16(taddr + c0 + 32u, vb);
                    process(va, c0);
                    if (second) {
                        vb_tmem_ld_wait();
                        if (c0 + 64u < ncol) vb_tmem_ld16(taddr + c0 + 64u, va);
                        process(vb, c0 + 32u);
                    }
                }
                vb_tcgen05_fence_before();
                __syncwarp();
                if (lane == 0) vb_mbar_arrive(bar_tempty + 8u * acc);
            }
        }
        if (pn != 0u) vb_flush_pending(a.lists.cand, a.lists.cnt, a.lists.cap, a.lists.sub_cap, sub, pk_addr, pl_addr, pn, lane);
    }
    vb_tcgen05_fence_before();
    __syncthreads();
    if (warp == 1) {
        vb_tcgen05_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
    }
}

// ---- host side ----------------------------------------------------------------------------------
typedef CUresult (*VbEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static VbEncodeTiledFn g_encode_tiled = nullptr;
static int g_gemm_smem_max = 0;

typedef void (*VbGemmKernel)(const CUtensorMap, const CUtensorMap, const CUtensorMap, const VbGemmArgs);
// variant index = modeIdx*4 + split*2 + direct, modeIdx: 0 -> MODE 0, 1 -> MODE 2, 2 -> MODE 3; 12 / 13: row selection (MODE 0, not direct), split 0 / 1
static VbGemmKernel vb_gemm_variant(int i) {
    static const VbGemmKernel table[14] = {
        vb_dense_gemm_kernel<0, false, false, false>, vb_dense_gemm_kernel<0, false, true, false>,
        vb_dense_gemm_kernel<0, true, false, false>,  vb_dense_gemm_kernel<0, true, true, false>,
        vb_dense_gemm_kernel<2, false, false, false>, vb_dense_gemm_kernel<2, false, true, false>,
        vb_dense_gemm_kernel<2, true, false, false>,  vb_dense_gemm_kernel<2, true, true, false>,
        vb_dense_gemm_kernel<3, false, false, false>, vb_dense_gemm_kernel<3, false, true, false>,
        vb_dense_gemm_kernel<3, true, false, false>,  vb_dense_gemm_kernel<3, true, true, false>,
        vb_dense_gemm_kernel<0, false, false, true>, vb_dense_gemm_kernel<0, true, false, true>,
    };
    return table[i];
}

static int vb_gemm_configure() {
    if (g_encode_tiled) return 0;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || fn == nullptr || qres != cudaDriverEntryPointSuccess) {
        g_gemm_err = "cuTensorMapEncodeTiled not available from the driver";
        return 1;
    }
    int dev = 0, smem = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    for (int i = 0; i < 14; ++i) {
        e = cudaFuncSetAttribute(vb_gemm_variant(i), cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) { g_gemm_err = std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e); return 1; }
    }
    e = cudaFuncSetAttribute(vb_dense_gemm_tiled_kernel<0, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(vb_dense_gemm_tiled_kernel<2, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(vb_dense_gemm_tiled_kernel<3, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(vb_dense_gemm_tiled_kernel<0, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(vb_dense_gemm_tiled_kernel<2, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(vb_dense_gemm_tiled_kernel<3, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(vb_dense_gemm_tiled_kernel<0, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) { g_gemm_err = std::string("cudaFuncSetAttribute(tiled): ") + cudaGetErrorString(e); return 1; }
    g_gemm_smem_max = smem;
    g_encode_tiled = reinterpret_cast<VbEncodeTiledFn>(fn);
    return 0;
}

static const uint32_t VB_GEMM_TAIL_BYTES = 320u + 4u * 256u * 4u + 8u * VB_GEMM_MAX_FILTERS * 4u;
static const uint32_t VB_K2_KBOX = 3u;         // K-blocks per TMA box of the resident kernel (pipeline stage granularity)
static const uint32_t VB_K2_MAX_STAGES = 12u;  // ring depth cap of the resident kernel
static const uint32_t VB_K2T_STAGES = 4u;      // ring depth of K2T (3 measured no faster, DESIGN §Scheduling)

// K-blocks per TMA box (pipeline stage granularity)
static uint32_t vb_gemm_kbox(uint32_t d_pad) {
    const uint32_t k_blocks = d_pad / VB_BLOCK_K;
    return VB_K2_KBOX > k_blocks ? k_blocks : VB_K2_KBOX;
}
// largest padded sub-batch whose resident query matrix leaves room for >= 4 stages
static uint32_t vb_gemm_max_bn(uint32_t d_pad) {
    const uint32_t reserve = std::max(4u, 2u * vb_gemm_kbox(d_pad)) * VB_STAGE_BYTES;   // room for the A ring
    const uint32_t avail = (uint32_t)g_gemm_smem_max - 1024u - VB_GEMM_TAIL_BYTES - reserve;
    uint32_t bn = avail / (d_pad * 2u);
    bn = bn / 16u * 16u;
    return bn > 256u ? 256u : bn;
}

// Sub-batch geometry shared by the query-packing kernel and the launcher: queries are cut into
// sub-batches of `sub` queries; sub-batch s occupies rows [s*sub*mult, ...) of the packed bf16
// operand: bn_q rows of q_hi followed (split) by bn_q rows of q_lo, bn_q = round_up(n_q, 16).
struct VbGemmPlan { uint32_t sub; uint32_t split; };
static VbGemmPlan vb_gemm_plan(uint32_t d_pad, uint32_t B, int precision /*0 auto, 1 bf16, 2 bf16x2*/) {
    const uint32_t bn_max = vb_gemm_max_bn(d_pad);
    const uint32_t half = (bn_max / 2u) / 16u * 16u;
    VbGemmPlan p;
    p.split = precision == 2 ? 1u : (precision == 1 ? 0u : (B <= half ? 1u : 0u));
    if (p.split && half < 16u) p.split = 0u;
    p.sub = p.split ? half : bn_max;
    return p;
}

static bool vb_gemm_supported(int d_pad, uint32_t B) {
    (void)B;
    return g_encode_tiled != nullptr && d_pad % 64 == 0 && vb_gemm_max_bn((uint32_t)d_pad) >= 16u;
}

struct VbGemmLaunch {
    const void* rows;          // [n_rows_total][d_pad] bf16
    const float* inv_norm;
    const void* q_bf16;        // [>= round_up(B,16)][d_pad] bf16
    const uint32_t* mask;
    const int32_t* mask_of;
    uint32_t mask_words, n_filters;
    const float* tau;
    const float* q_scale;      // [B]
    VbLists lists;
    uint32_t n_rows_total, row_begin, row_end, row_base, d_pad, n_queries;
    int sm_count;
    cudaStream_t stream;
    uint32_t direct;
    VbGemmPlan plan;
    const int32_t* mask_of_host;   // host copy of mask_of (to pick the epilogue's mask mode)
    VbFilterTiles ftab;            // mask mode 3: filter tables for this launcher's query tiles (K2: plan.sub, K2T: VB_TILE_N)
    // K2T over the compacted copy of the rows passing the batch's shared filter (dense_compact.cuh); sel == nullptr: off
    const uint32_t* sel = nullptr;
    const uint32_t* sel_ids = nullptr;
    const float* sel_inv_norm = nullptr;
    const void* sel_rows = nullptr;    // [sel_cap_rows][d_pad] bf16
    uint32_t sel_cap_rows = 0;
};

static int vb_encode_2d(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows) {
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {cols * 2};
    cuuint32_t box[2] = {VB_BLOCK_K, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = g_encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { g_gemm_err = "cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ")"; return 1; }
    return 0;
}

// A operand as a 3-D tensor [k_block][row][64]: one TMA box brings `kbox` K-blocks of 128 rows,
// landing as kbox consecutive [128 rows x 128 B] swizzled slabs (what the UMMA descriptors expect).
static int vb_encode_a3d(CUtensorMap* map, const void* base, uint64_t rows, uint64_t d_pad, uint32_t kbox) {
    cuuint64_t dims[3] = {VB_BLOCK_K, rows, d_pad / VB_BLOCK_K};
    cuuint64_t strides[2] = {d_pad * 2, VB_BLOCK_K * 2};
    cuuint32_t box[3] = {VB_BLOCK_K, VB_TILE_M, kbox};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = g_encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { g_gemm_err = "cuTensorMapEncodeTiled(3d) failed (" + std::to_string((int)r) + ")"; return 1; }
    return 0;
}

static int vb_gemm_launch(const VbGemmLaunch& g, int* launches) {
    if (!g_encode_tiled) { g_gemm_err = "tensor-core path not configured"; return 1; }
    const uint32_t sub = g.plan.sub, mult = g.plan.split ? 2u : 1u;
    if (g.mask && g.n_filters > 31u && g.ftab.tile != sub) { g_gemm_err = "filter tables were built for another sub-batch size"; return 1; }
    const uint32_t k_blocks = g.d_pad / VB_BLOCK_K;
    const uint32_t kbox = vb_gemm_kbox(g.d_pad);
    (void)k_blocks;
    CUtensorMap tmap_a;
    if (vb_encode_a3d(&tmap_a, g.rows, g.n_rows_total, g.d_pad, kbox)) return 1;
    CUtensorMap tmap_c = tmap_a;
    if (g.sel && vb_encode_a3d(&tmap_c, g.sel_rows, g.sel_cap_rows, g.d_pad, kbox)) return 1;
    for (uint32_t q0 = 0; q0 < g.n_queries; q0 += sub) {
        const uint32_t n_q = std::min(sub, g.n_queries - q0);
        const uint32_t bn = (n_q + 15u) / 16u * 16u * mult;
        CUtensorMap tmap_q;
        if (vb_encode_2d(&tmap_q, reinterpret_cast<const unsigned char*>(g.q_bf16) + (size_t)q0 * mult * g.d_pad * 2, bn, g.d_pad, bn)) return 1;
        VbGemmArgs a{};
        a.inv_norm = g.inv_norm; a.mask = g.mask; a.mask_of = g.mask_of; a.tau = g.tau; a.q_scale = g.q_scale; a.lists = g.lists;
        a.mask_words = g.mask_words; a.n_filters = g.n_filters;
        a.tile_begin = g.row_begin / VB_TILE_M; a.tile_end = (g.row_end + VB_TILE_M - 1) / VB_TILE_M;
        a.row_end = g.row_end; a.row_base = g.row_base; a.k_blocks = g.d_pad / VB_BLOCK_K;
        a.bn = bn; a.n_q = n_q; a.q_begin = q0;
        a.direct = g.direct;
        a.split = g.plan.split;
        a.mask_mode = 0; a.uniform_filter = -1;
        if (g.mask != nullptr) {
            bool uniform = true;
            for (uint32_t i = 1; i < n_q; ++i) uniform = uniform && g.mask_of_host[q0 + i] == g.mask_of_host[q0];
            if (uniform && g.mask_of_host[q0] < 0) { a.mask = nullptr; a.mask_of = nullptr; }
            else if (uniform) { a.mask_mode = 1; a.uniform_filter = g.mask_of_host[q0]; }
            else a.mask_mode = g.n_filters <= 31u ? 2 : 3;
            if (a.mask_mode == 3u) {                // sub-batch s is tile s of the tables
                a.mask_of = g.ftab.loc; a.ftab_n = g.ftab.n + q0 / sub; a.ftab = g.ftab.ids + (size_t)(q0 / sub) * VB_GEMM_MAX_FILTERS;
            }
        }
        const uint32_t q_bytes = bn * g.d_pad * 2u;
        a.kbox = kbox;
        const uint32_t stages = ((uint32_t)g_gemm_smem_max - 1024u - VB_GEMM_TAIL_BYTES - q_bytes) / (kbox * VB_STAGE_BYTES);
        a.stages = stages > VB_K2_MAX_STAGES ? VB_K2_MAX_STAGES : stages;
        if (a.stages < 2u) { g_gemm_err = "not enough shared memory for a 2-stage pipeline"; return 1; }
        const size_t smem = 1024u + q_bytes + a.stages * kbox * VB_STAGE_BYTES + VB_GEMM_TAIL_BYTES;
        const uint32_t tiles = a.tile_end - a.tile_begin;
        const uint32_t grid = std::min<uint32_t>(tiles, (uint32_t)g.sm_count);
        int variant = (a.mask_mode >= 2u ? (int)a.mask_mode - 1 : 0) * 4 + (a.split ? 2 : 0) + (a.direct ? 1 : 0);
        if (g.sel != nullptr && a.mask_mode == 1u && !a.direct) {
            a.sel = g.sel; a.sel_ids = g.sel_ids; a.sel_inv_norm = g.sel_inv_norm;
            variant = 12 + (a.split ? 1 : 0);
        }
        vb_gemm_variant(variant)<<<grid, VB_GEMM_THREADS, smem, g.stream>>>(tmap_a, tmap_q, tmap_c, a);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) { g_gemm_err = std::string("launch failed: ") + cudaGetErrorString(e); return 1; }
        ++*launches;
    }
    return 0;
}

// ---- K2T launcher -------------------------------------------------------------------------------------
static const uint32_t VB_TILED_TAIL_BYTES = 320u + VB_TILED_MAX_Q * 16u + 8u * VB_GEMM_MAX_FILTERS * 4u + 8u * VB_PEND * 12u;

static uint32_t vb_gemm_tiled_stages() {
    const uint32_t avail = (uint32_t)g_gemm_smem_max - 1024u - VB_TILED_TAIL_BYTES;
    const uint32_t st = avail / VB_TILED_STAGE_BYTES;
    return st > VB_K2T_STAGES ? VB_K2T_STAGES : st;
}
static bool vb_gemm_tiled_supported(int d_pad) {
    return g_encode_tiled != nullptr && d_pad % 64 == 0 && vb_gemm_tiled_stages() >= 2u;
}

// g.q_bf16 must hold the queries unsplit, row i = query i (vb_gemm_plan with split = 0).
static int vb_gemm_tiled_launch(const VbGemmLaunch& g, int* launches) {
    if (!g_encode_tiled) { g_gemm_err = "tensor-core path not configured"; return 1; }
    if (g.mask && g.n_filters > 31u && g.ftab.tile != VB_TILE_N) { g_gemm_err = "filter tables were built for another query tile"; return 1; }
    if (g.plan.split) { g_gemm_err = "tiled kernel needs the unsplit query layout"; return 1; }
    CUtensorMap tmap_a;
    if (vb_encode_2d(&tmap_a, g.rows, g.n_rows_total, g.d_pad, VB_TILE_M)) return 1;
    CUtensorMap tmap_c = tmap_a;
    if (g.sel && vb_encode_2d(&tmap_c, g.sel_rows, g.sel_cap_rows, g.d_pad, VB_TILE_M)) return 1;
    const uint32_t stages = vb_gemm_tiled_stages();
    for (uint32_t q0 = 0; q0 < g.n_queries; q0 += VB_TILED_MAX_Q) {
        const uint32_t n_q = std::min(VB_TILED_MAX_Q, g.n_queries - q0);
        CUtensorMap tmap_q;
        if (vb_encode_2d(&tmap_q, reinterpret_cast<const unsigned char*>(g.q_bf16) + (size_t)q0 * g.d_pad * 2,
                         (n_q + 15u) / 16u * 16u, g.d_pad, VB_TILE_N)) return 1;
        VbGemmTiledArgs a{};
        a.inv_norm = g.inv_norm; a.mask = g.mask; a.mask_of = g.mask_of; a.tau = g.tau; a.q_scale = g.q_scale; a.lists = g.lists;
        a.mask_words = g.mask_words; a.n_filters = g.n_filters;
        a.tile_begin = g.row_begin / VB_TILE_M; a.tile_end = (g.row_end + VB_TILE_M - 1) / VB_TILE_M;
        a.row_end = g.row_end; a.row_base = g.row_base; a.k_blocks = g.d_pad / VB_BLOCK_K;
        a.n_q = n_q; a.q_begin = q0; a.stages = stages;
        a.mask_mode = 0; a.uniform_filter = -1;
        if (g.mask != nullptr) {
            bool uniform = true;
            for (uint32_t i = 1; i < n_q; ++i) uniform = uniform && g.mask_of_host[q0 + i] == g.mask_of_host[q0];
            if (uniform && g.mask_of_host[q0] < 0) { a.mask = nullptr; a.mask_of = nullptr; }
            else if (uniform) { a.mask_mode = 1; a.uniform_filter = g.mask_of_host[q0]; }
            else a.mask_mode = g.n_filters <= 31u ? 2 : 3;
            if (a.mask_mode == 3u) {                // q0 is a multiple of VB_TILED_MAX_Q: this launch holds tiles q0 / VB_TILE_N ...
                a.mask_of = g.ftab.loc; a.ftab_n = g.ftab.n + q0 / VB_TILE_N; a.ftab = g.ftab.ids + (size_t)(q0 / VB_TILE_N) * VB_GEMM_MAX_FILTERS;
            }
        }
        const bool use_sel = g.sel != nullptr && a.mask_mode == 1u && !g.direct;
        const size_t smem = 1024u + (size_t)stages * VB_TILED_STAGE_BYTES + VB_TILED_TAIL_BYTES;
        const uint32_t tiles = a.tile_end - a.tile_begin;
        const uint32_t grid = std::min<uint32_t>(tiles, (uint32_t)g.sm_count);
        if (g.direct) {
            if (a.mask_mode == 2u) vb_dense_gemm_tiled_kernel<2, true, false><<<grid, VB_GEMM_THREADS, smem, g.stream>>>(tmap_a, tmap_q, tmap_a, a);
            else if (a.mask_mode == 3u) vb_dense_gemm_tiled_kernel<3, true, false><<<grid, VB_GEMM_THREADS, smem, g.stream>>>(tmap_a, tmap_q, tmap_a, a);
            else vb_dense_gemm_tiled_kernel<0, true, false><<<grid, VB_GEMM_THREADS, smem, g.stream>>>(tmap_a, tmap_q, tmap_a, a);
        } else {
            if (a.mask_mode == 2u) vb_dense_gemm_tiled_kernel<2, false, false><<<grid, VB_GEMM_THREADS, smem, g.stream>>>(tmap_a, tmap_q, tmap_a, a);
            else if (a.mask_mode == 3u) vb_dense_gemm_tiled_kernel<3, false, false><<<grid, VB_GEMM_THREADS, smem, g.stream>>>(tmap_a, tmap_q, tmap_a, a);
            else if (use_sel) {
                a.sel = g.sel; a.sel_ids = g.sel_ids; a.sel_inv_norm = g.sel_inv_norm;
                vb_dense_gemm_tiled_kernel<0, false, true><<<grid, VB_GEMM_THREADS, smem, g.stream>>>(tmap_a, tmap_q, tmap_c, a);
            } else vb_dense_gemm_tiled_kernel<0, false, false><<<grid, VB_GEMM_THREADS, smem, g.stream>>>(tmap_a, tmap_q, tmap_a, a);
        }
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) { g_gemm_err = std::string("tiled launch failed: ") + cudaGetErrorString(e); return 1; }
        ++*launches;
    }
    return 0;
}
