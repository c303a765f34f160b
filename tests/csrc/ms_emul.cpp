// CPU emulation of K3M (voitta-rag_b200/csrc/sparse_ms.cuh) — TEST INFRASTRUCTURE ONLY.
// The development container has no GPU, so the host/device functions that carry the MaxScore logic
// (plan phases, per-posting scoring, lookups, re-score) are compiled here with g++ and driven the way
// the two kernels drive them: plan phases as loops over the terms, then every work unit, every posting.
// tests/test_ms_emul.py checks the candidates against the oracle.  Nothing in the product links this.
#include "../../voitta-rag_b200/csrc/sparse_ms.cuh"
#include <vector>
#include <algorithm>

extern "C" int ms_emul_segment(
    const uint32_t* post_row, const float* post_val, const float* heavy_vals, uint32_t heavy_stride,
    const uint32_t* term_tab, const uint32_t* q_tab, const uint8_t* q_shift,
    const int64_t* sp_indptr, const uint32_t* sp_term, const float* sp_val,
    uint32_t nt, const uint32_t* q_term, const double* q_weight, const double* q_ub, const int32_t* q_hidx,
    const uint32_t* q_plo, const uint32_t* q_phi, const uint32_t* mask, float tau,
    uint32_t seg_row0, uint32_t seg_row1, uint32_t n_rows, uint32_t chunk, uint32_t budget_pct, uint64_t stage_lo, uint64_t stage_hi,
    uint32_t* out_rows, float* out_scores, uint32_t max_out, uint64_t* stats /* [4]: essential postings, units, n_ess, lookups-unused */)
{
    if (nt == 0 || nt > VB_MS_MAX_TERMS) return -1;
    tau = vb_ms_exact_tau(tau);                                 // K3M runs under the next float below the list's tau
    // ---- plan (vb_ms_plan_kernel) ----
    VbMsPlanShared s;
    for (uint32_t j = 0; j < nt; ++j)
        vb_ms_plan_load(s, j, post_row, term_tab, q_plo[j], q_phi[j], q_tab[j], q_shift[j], n_rows, seg_row0, seg_row1, q_ub[j]);
    // the table-assisted segment bounds must equal plain lower bounds
    for (uint32_t j = 0; j < nt; ++j) {
        const uint32_t lo = vb_ms_lower_bound(post_row, q_plo[j], q_phi[j], seg_row0);
        const uint32_t hi = seg_row1 >= n_rows ? q_phi[j] : vb_ms_lower_bound(post_row, q_plo[j], q_phi[j], seg_row1);
        if (s.slo[j] != lo || s.shi[j] != hi) return -4;
    }
    for (uint32_t j = 0; j < nt; ++j) vb_ms_plan_position(s, j, nt);
    { std::vector<uint32_t> p(s.term_at, s.term_at + nt); std::sort(p.begin(), p.end()); for (uint32_t i = 0; i < nt; ++i) if (p[i] != i) return -2; }
    std::vector<VbMsRec> rec(nt);
    std::vector<uint32_t> units(nt + 1, 0);
    uint32_t n_ess = 0;
    bool seen_ne = false;
    for (uint32_t i = 0; i < nt; ++i) {
        const VbMsPos ps = vb_ms_plan_pos(s, i, nt, (double)tau, budget_pct, stage_lo, stage_hi);
        if (ps.essential) { if (seen_ne) return -5; ++n_ess; } else seen_ne = true;      // NE must be a suffix
        const uint32_t t = s.term_at[i];
        VbMsRec r;
        r.slo = s.slo[t] + ps.w0; r.shi = s.slo[t] + ps.w1; r.w = q_weight[t]; r.suf = ps.suf;
        r.hidx = q_hidx ? q_hidx[t] : -1; r.tab = q_tab[t]; r.shift = q_shift[t]; r.plo = q_plo[t]; r.phi = q_phi[t]; r.pad = 0;
        rec[i] = r;
        units[i] = (ps.w1 - ps.w0 + chunk - 1u) / chunk;
    }
    { uint32_t run = 0; for (uint32_t i = 0; i <= nt; ++i) { const uint32_t c = i < nt ? units[i] : 0u; units[i] = run; run += c; } }
    const uint32_t total = units[nt];
    // ---- score (vb_ms_score_kernel) ----
    std::vector<double> w(nt), suf(nt);
    std::vector<int32_t> hidx(nt);
    std::vector<uint32_t> tab(nt), shift(nt), plo(nt), phi(nt);
    uint32_t n_out = 0;
    uint64_t ess_post = 0;
    for (uint32_t u = 0; u < total; ++u) {
        uint32_t lo = 0, hi = nt;
        while (hi - lo > 1u) { const uint32_t mid = lo + ((hi - lo) >> 1); if (units[mid] <= u) lo = mid; else hi = mid; }
        const uint32_t pe = lo;
        const VbMsRec e = rec[pe];
        const uint32_t p0 = e.slo + (u - units[pe]) * chunk;
        const uint32_t p1 = std::min(e.shi, p0 + chunk);
        if (p0 >= p1) return -3;
        for (uint32_t i = 0; i < nt; ++i) {
            const VbMsRec r = rec[i];
            w[i] = r.w; suf[i] = r.suf; hidx[i] = r.hidx; tab[i] = r.tab; shift[i] = r.shift; plo[i] = r.plo; phi[i] = r.phi;
        }
        VbMsCtx c;
        c.post_row = post_row; c.post_val = post_val; c.heavy_vals = heavy_vals; c.heavy_stride = heavy_stride; c.term_tab = term_tab;
        c.sp_indptr = sp_indptr; c.sp_term = sp_term; c.sp_val = sp_val; c.q_term = q_term; c.q_weight = q_weight;
        c.mask = mask; c.w = w.data(); c.suf = suf.data(); c.hidx = hidx.data(); c.tab = tab.data(); c.shift = shift.data(); c.plo = plo.data(); c.phi = phi.data();
        c.nt = nt; c.n_ess = n_ess; c.tau_lo = vb_ms_tau_lo((double)tau); c.delta = (double)(4u * nt) * 1.1102230246251565e-16; c.tau = tau;
        for (uint32_t p = p0; p < p1; ++p) {
            ++ess_post;
            float score;
            if (vb_ms_score_posting(c, pe, post_row[p], post_val[p], score)) {
                if (n_out < max_out) { out_rows[n_out] = post_row[p]; out_scores[n_out] = score; }
                ++n_out;
            }
        }
    }
    if (stats) { stats[0] = ess_post; stats[1] = total; stats[2] = n_ess; stats[3] = 0; }
    return (int)n_out;
}

// K3H (csrc/sparse_mh.cuh): the plan as above, then per row range of the query the essential postings are summed per
// row (what the shared-memory hash table does) and every touched row goes through vb_ms_finish_row.
#include <map>
extern "C" int mh_emul_segment(
    const uint32_t* post_row, const float* post_val, const float* heavy_vals, uint32_t heavy_stride,
    const uint32_t* term_tab, const uint32_t* q_tab, const uint8_t* q_shift,
    const int64_t* sp_indptr, const uint32_t* sp_term, const float* sp_val,
    uint32_t nt, const uint32_t* q_term, const double* q_weight, const double* q_ub, const int32_t* q_hidx,
    const uint32_t* q_plo, const uint32_t* q_phi, const uint32_t* mask, float tau,
    uint32_t seg_row0, uint32_t seg_row1, uint32_t n_rows, uint32_t budget_pct, uint32_t max_post,
    uint32_t* out_rows, float* out_scores, uint32_t max_out, uint64_t* stats /* [4]: essential postings, units, n_ess, halvings */)
{
    if (nt == 0 || nt > VB_MS_MAX_TERMS) return -1;
    VbMsPlanShared s;
    for (uint32_t j = 0; j < nt; ++j)
        vb_ms_plan_load(s, j, post_row, term_tab, q_plo[j], q_phi[j], q_tab[j], q_shift[j], n_rows, seg_row0, seg_row1, q_ub[j]);
    for (uint32_t j = 0; j < nt; ++j) vb_ms_plan_position(s, j, nt);
    std::vector<VbMsRec> rec(nt);
    uint32_t n_ess = 0;
    uint64_t ess_post = 0;
    for (uint32_t i = 0; i < nt; ++i) {
        const VbMsPos ps = vb_ms_plan_pos(s, i, nt, (double)tau, budget_pct, 0ull, ~0ull);
        if (ps.essential) ++n_ess;
        const uint32_t t = s.term_at[i];
        VbMsRec r;
        r.slo = s.slo[t] + ps.w0; r.shi = s.slo[t] + ps.w1; r.w = q_weight[t]; r.suf = ps.suf;
        r.hidx = q_hidx ? q_hidx[t] : -1; r.tab = q_tab[t]; r.shift = q_shift[t]; r.plo = q_plo[t]; r.phi = q_phi[t]; r.pad = 0;
        rec[i] = r;
        ess_post += ps.w1 - ps.w0;
    }
    uint32_t n_out = 0;
    uint64_t halvings = 0, units = 0;
    if (ess_post) {
        const uint32_t seg_rows = seg_row1 - seg_row0;
        const uint32_t shift = vb_mh_shift(ess_post, seg_rows);
        units = ((uint64_t)seg_rows + (1ull << shift) - 1ull) >> shift;
        std::vector<double> w(nt), suf(nt);
        std::vector<int32_t> hidx(nt);
        std::vector<uint32_t> tab(nt), shf(nt), plo(nt), phi(nt);
        for (uint32_t i = 0; i < nt; ++i) { w[i] = rec[i].w; suf[i] = rec[i].suf; hidx[i] = rec[i].hidx; tab[i] = rec[i].tab; shf[i] = rec[i].shift; plo[i] = rec[i].plo; phi[i] = rec[i].phi; }
        VbMsCtx c;
        c.post_row = post_row; c.post_val = post_val; c.heavy_vals = heavy_vals; c.heavy_stride = heavy_stride; c.term_tab = term_tab;
        c.sp_indptr = sp_indptr; c.sp_term = sp_term; c.sp_val = sp_val; c.q_term = q_term; c.q_weight = q_weight;
        c.mask = nullptr; c.w = w.data(); c.suf = suf.data(); c.hidx = hidx.data(); c.tab = tab.data(); c.shift = shf.data(); c.plo = plo.data(); c.phi = phi.data();
        c.nt = nt; c.n_ess = n_ess; c.tau_lo = vb_ms_tau_lo((double)tau); c.delta = (double)(4u * nt) * 1.1102230246251565e-16; c.tau = tau;
        for (uint64_t u = 0; u < units; ++u) {
            const uint32_t unit_row0 = seg_row0 + (uint32_t)(u << shift);
            const uint32_t unit_row1 = (uint32_t)std::min<uint64_t>(seg_row1, (uint64_t)unit_row0 + (1ull << shift));
            uint32_t width = unit_row1 - unit_row0, pos = unit_row0;
            while (pos < unit_row1) {
                const uint32_t r1 = (uint32_t)std::min<uint64_t>(unit_row1, (uint64_t)pos + width);
                std::vector<uint32_t> lo(n_ess), hi(n_ess);
                uint32_t T = 0;
                for (uint32_t i = 0; i < n_ess; ++i) {
                    lo[i] = vb_ms_seg_bound(post_row, term_tab, rec[i].slo, rec[i].shi, rec[i].tab, rec[i].shift, n_rows, pos);
                    hi[i] = vb_ms_seg_bound(post_row, term_tab, rec[i].slo, rec[i].shi, rec[i].tab, rec[i].shift, n_rows, r1);
                    if (hi[i] < lo[i]) return -6;
                    T += hi[i] - lo[i];
                }
                if (T > max_post && width > 1u) { width = (width + 1u) >> 1; ++halvings; continue; }
                std::map<uint32_t, double> acc;
                for (uint32_t i = 0; i < n_ess; ++i)
                    for (uint32_t p = lo[i]; p < hi[i]; ++p) {
                        if (post_row[p] < pos || post_row[p] >= r1) return -7;          // the slice must lie inside the row range
                        acc[post_row[p]] += rec[i].w * (double)post_val[p];
                    }
                for (const auto& kv : acc) {
                    const uint32_t row = kv.first;
                    if (mask != nullptr && !((mask[row >> 5] >> (row & 31u)) & 1u)) continue;
                    float score;
                    if (vb_ms_finish_row(c, n_ess, row, kv.second, score)) {
                        if (n_out < max_out) { out_rows[n_out] = row; out_scores[n_out] = score; }
                        ++n_out;
                    }
                }
                pos = r1;
            }
        }
    }
    if (stats) { stats[0] = ess_post; stats[1] = units; stats[2] = n_ess; stats[3] = halvings; }
    return (int)n_out;
}
