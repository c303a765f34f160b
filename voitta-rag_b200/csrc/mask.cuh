// K0 — filter evaluation.  Replaces the payload-filter evaluation qdrant performs for
// query_filter (vector_store.py:462-530 builds it; :612-617/:640-656 pass it).
//
// One pass over the per-row columns (scope id u32, one or two i64 timestamps, alive bits)
// produces, for every distinct filter of the batch, a packed bitmask (bit r%32 of word r/32).
// The scoring kernels K1/K2/K3 then apply the filter as a bitmask inside their loops.
// HBM-bound: algorithmic bytes = n*(4 [+8 per timestamp column used]) + n/8 read,
// n_filters*n/8 written.
#pragma once
#include "common.cuh"

#define VB_MASK_WORDS_PER_STEP 4u   // mask words (x32 rows) a warp has in flight: 4 scope + 4 timestamp loads per thread

__global__ void __launch_bounds__(256)
vb_mask_kernel(const uint32_t* __restrict__ scope_id, const int64_t* __restrict__ created,
               const int64_t* __restrict__ modified, const uint32_t* __restrict__ alive,
               uint32_t n_rows, const VbFilterDev* __restrict__ filters, uint32_t n_filters,
               uint32_t words, uint32_t need_created, uint32_t need_modified, uint32_t need_scope,
               uint32_t* __restrict__ out)
{
    constexpr uint32_t U = VB_MASK_WORDS_PER_STEP;
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t w0 = ((blockIdx.x * blockDim.x + threadIdx.x) >> 5) * U; w0 < words; w0 += warps * U) {
        // all column loads of the step are issued before any filter is evaluated (one word per step left the
        // kernel at 43 % of the HBM peak: a single 4 + 8 byte load pair in flight per thread)
        uint32_t sid[U], alive_w[U];
        int64_t tc[U], tm[U];
#pragma unroll
        for (uint32_t u = 0; u < U; ++u) {
            const uint32_t w = w0 + u;
            const uint32_t row = w * 32u + lane;
            const bool valid = w < words && row < n_rows;
            alive_w[u] = w < words ? alive[w] : 0u;
            sid[u] = (valid && need_scope) ? scope_id[row] : 0u;
            tc[u] = (valid && need_created) ? created[row] : INT64_MIN;
            tm[u] = (valid && need_modified) ? modified[row] : INT64_MIN;
        }
        for (uint32_t f = 0; f < n_filters; ++f) {
            const VbFilterDev flt = filters[f];
#pragma unroll
            for (uint32_t u = 0; u < U; ++u) {
                const uint32_t w = w0 + u;
                if (w >= words) break;                           // warp-uniform
                const uint32_t row = w * 32u + lane;
                bool pass = row < n_rows && ((alive_w[u] >> lane) & 1u);
                if (flt.scope_bits != nullptr) {
                    const uint32_t sw = sid[u] >> 5;
                    pass = pass && sw < flt.scope_words && ((flt.scope_bits[sw] >> (sid[u] & 31u)) & 1u);
                }
                if (flt.ts_field != 0) {
                    const int64_t t = (flt.ts_field == 1) ? tc[u] : tm[u];
                    // a must-range on a missing field fails (payload_filters semantics)
                    pass = pass && t != INT64_MIN && t >= flt.ts_lo && t <= flt.ts_hi;
                }
                const uint32_t bits = __ballot_sync(0xffffffffu, pass);
                if (lane == 0) out[(size_t)f * words + w] = bits;
            }
        }
    }
}

// vb_set_scope: scope_id[rows[i]] = ids[i].  The host checked that the rows are in range and distinct, so the
// scatter has no write conflicts.
__global__ void __launch_bounds__(256)
vb_scatter_scope_kernel(uint32_t* __restrict__ scope_id, const uint32_t* __restrict__ rows,
                        const uint32_t* __restrict__ ids, uint32_t n)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        scope_id[rows[i]] = ids[i];
}

// Ingest (K5): fp32 -> bf16 rows (zero padded to d_pad) + fp32 inverse norm of the ROUNDED row,
// so that score = dot(bf16 row, q_hat) * inv_norm is the cosine against the stored point.
// Replaces the normalise-at-upsert step of qdrant's COSINE distance (vector_store.py:93, :313).
__global__ void __launch_bounds__(256)
vb_ingest_f32_kernel(const float* __restrict__ src, uint32_t n, uint32_t dim, uint32_t d_pad,
                     __nv_bfloat16* __restrict__ dst, float* __restrict__ inv_norm)
{
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n; r += warps) {
        double ss = 0.0;
        for (uint32_t c = lane; c < d_pad; c += 32u) {
            __nv_bfloat16 b = __float2bfloat16_rn(c < dim ? src[(size_t)r * dim + c] : 0.0f);
            dst[(size_t)r * d_pad + c] = b;
            const double v = (double)__bfloat162float(b);
            ss += v * v;
        }
        for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
        if (lane == 0) inv_norm[r] = ss > 0.0 ? (float)(1.0 / sqrt(ss)) : 0.0f;
    }
}

// Same for rows that are already bf16 on the device (bulk loader): copy/pad + inverse norm.
__global__ void __launch_bounds__(256)
vb_ingest_bf16_kernel(const __nv_bfloat16* __restrict__ src, uint32_t n, uint32_t dim, uint32_t d_pad,
                      __nv_bfloat16* __restrict__ dst, float* __restrict__ inv_norm)
{
    const uint32_t lane = threadIdx.x & 31u;
    const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
    for (uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n; r += warps) {
        double ss = 0.0;
        for (uint32_t c = lane; c < d_pad; c += 32u) {
            __nv_bfloat16 b = c < dim ? src[(size_t)r * dim + c] : __float2bfloat16_rn(0.0f);
            dst[(size_t)r * d_pad + c] = b;
            const double v = (double)__bfloat162float(b);
            ss += v * v;
        }
        for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
        if (lane == 0) inv_norm[r] = ss > 0.0 ? (float)(1.0 / sqrt(ss)) : 0.0f;
    }
}

// Query preparation: q_hat = q/||q|| in fp32 (zero vector stays zero), zero padded to d_pad
// (distances.py cosine_similarity normalises the query the same way); also packed as the bf16
// B-operand of the tensor-core path: sub-batches of `sub` queries, each bn_q = round_up(n_q,16)
// rows of q_hi = bf16(q_hat) followed, if `split`, by bn_q rows of q_lo = bf16(q_hat - q_hi), so
// that q_hi + q_lo carries ~16 mantissa bits and the MMA result matches the fp32 dot to ~1e-5.
__global__ void __launch_bounds__(128)
vb_prep_query_kernel(const float* __restrict__ q, uint32_t dim, uint32_t d_pad, uint32_t n_queries,
                     uint32_t sub, uint32_t split, float* __restrict__ q_hat, __nv_bfloat16* __restrict__ q_bf16,
                     float* __restrict__ q_scale, uint32_t* __restrict__ q_bad, const VbListInit li)
{
    __shared__ double red[4];
    const uint32_t b = blockIdx.x;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < li.n; i += gridDim.x * blockDim.x) vb_init_list(li, i);
    double ss = 0.0;
    for (uint32_t c = threadIdx.x; c < dim; c += blockDim.x) {
        const double v = (double)q[(size_t)b * dim + c];
        ss += v * v;
    }
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    if ((threadIdx.x & 31u) == 0) red[threadIdx.x >> 5] = ss;
    __syncthreads();
    ss = red[0] + red[1] + red[2] + red[3];
    __syncthreads();
    if (threadIdx.x == 0) q_bad[b] = ss <= 1.0e300 ? 0u : 1u;  // NaN or inf anywhere in the query (qdrant asserts; reported at vb_fetch)
    const float inv = ss > 0.0 ? (float)(1.0 / sqrt(ss)) : 0.0f;
    const uint32_t s_idx = b / sub, j = b % sub;
    const uint32_t n_q = min(sub, n_queries - s_idx * sub);
    const uint32_t bn_q = (n_q + 15u) / 16u * 16u;
    const size_t base = (size_t)s_idx * sub * (split ? 2u : 1u);
    double rr = 0.0;                                            // squared length of the rounded unit query
    for (uint32_t c = threadIdx.x; c < d_pad; c += blockDim.x) {
        const float v = c < dim ? q[(size_t)b * dim + c] * inv : 0.0f;
        q_hat[(size_t)b * d_pad + c] = v;
        const __nv_bfloat16 hi = __float2bfloat16_rn(v);
        q_bf16[(base + j) * d_pad + c] = hi;
        if (split) q_bf16[(base + bn_q + j) * d_pad + c] = __float2bfloat16_rn(v - __bfloat162float(hi));
        const double hv = (double)__bfloat162float(hi);
        rr += hv * hv;
    }
    for (int o = 16; o > 0; o >>= 1) rr += __shfl_xor_sync(0xffffffffu, rr, o);
    if ((threadIdx.x & 31u) == 0) red[threadIdx.x >> 5] = rr;
    __syncthreads();
    rr = red[0] + red[1] + red[2] + red[3];
    // plain bf16 query: rescale scores by 1/|bf16(q)| (see vb_pre_threshold); the bf16x2 query keeps ~16 bits
    if (threadIdx.x == 0) q_scale[b] = (!split && rr > 0.0) ? (float)(1.0 / sqrt(rr)) : 1.0f;
}
