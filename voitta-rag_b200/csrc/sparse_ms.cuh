// K3M — posting-driven MaxScore sparse scoring (the batched / large-segment form of K3).
// Replaces, like sparse.cuh, qdrant's sparse dot product with the IDF modifier for
// query_points(query=SparseVector, using="bm25", limit=k', query_filter)
// (vector_store.py:647-656; sparse_distances.py sparse_dot_product in local mode) — same results,
// bit for bit, but the work is proportional to the postings that can still matter.
//
// Why: K3 (sparse.cuh) gives one CTA a (2048-row block, query) pair, initialises 2048 fp64
// accumulators and scans every row of the block against the query's frequent-term columns.  Once a
// list has a threshold tau (the score of its current k'-th best), almost all of that work is
// provably useless: with ub_t = weight_t * (largest posting value of term t), a row that contains
// only terms whose ub sum stays below tau cannot enter the list (MaxScore).  Measured on the
// benchmark corpora (tools/proto_maxscore.py) the ESSENTIAL postings are 2-4 % of the posting mass.
//
// Per launch, per query (vb_ms_plan_kernel, one CTA per query):
//   * terms ordered by DESCENDING ub = "position" order (independent of tau); suf[i] = sum of ub over the
//     positions after i; the lowest-ub suffix whose ub sum stays below tau is NON-essential (NE);
//   * the query's postings are numbered in position order, and a search runs in STAGES over the whole index:
//     stage 0 scores the first ~16 k' of them (the highest-ub terms' postings: the rows most likely to be the
//     best) with no threshold at all, every later stage 32x more under the threshold the stages before it
//     established (vb_compact_kernel between stages).  A row is scored exactly once, by the posting of its
//     earliest position ("owner"), in the stage that posting falls in.  (The safe mode runs the same kernels
//     per row segment instead.)
//   * every essential term's postings of the stage are cut into work units of `chunk` postings.
// vb_ms_score_kernel (persistent, dynamic unit counter): one thread per essential posting (e, row):
//   1. filter bit of the row;
//   2. w_e*v + suf[e] < tau  =>  drop (even with every later term present at its maximum the row
//      cannot reach tau; a frequent essential term's postings almost all end here: 8 bytes, one
//      fma, one compare);
//   3. the terms at LATER positions are looked up in position order, stopping as soon as partial + suf[i] < tau
//      (~2 lookups per posting that got here, and ~98 % of them stop);
//   4. ownership, for the rows whose sum reached tau: if a term at an EARLIER position also occurs in the row, that
//      term's posting owns the row (checked last: it answers "absent" 98 % of the time and costs pe lookups).
//      A lookup is one load from the term's dense column (frequent terms) or one 8-byte load from the
//      term's BUCKET TABLE — built with the index: tab[b] = first posting with row >= b << shift, buckets
//      sized for ~4 postings — which settles the common "absent" case at once and leaves <= 3 binary
//      search steps otherwise (the first version searched whole posting ranges: ncu showed the kernel
//      stalled on those dependent load chains, long_scoreboard 10 of 12 stall cycles per issue);
//   5. the surviving sum S adds the reference's fp64 products in another order:
//      |S - S_ref| <= delta*S, delta = 4*nt*2^-53 (all products >= 0).  If float(S(1-delta)) ==
//      float(S(1+delta)) the fp32 score is provably the reference's; otherwise the row is re-scored
//      from the forward index in ascending term id (the reference's two-pointer merge order).
// Only queries whose products are all >= 0 ("relaxed", always true for BM25 vectors) come this way;
// the others, and the first (direct) segment, stay on K3.
// Roofline: HBM/L2 gathers.  Algorithmic bytes per launch: 8 B per essential posting + 4..32 B per
// lookup; bench.py still quotes SURVEY §8(d)'s sum(df)*8 for comparability.
//
// The per-posting logic lives in host/device functions so that tests/csrc/ms_emul.cpp can run the
// very same code on the CPU against the oracle (no GPU in the development container).
#pragma once
#include <stdint.h>
#include <math.h>

#ifdef __CUDACC__
#define VB_HD __host__ __device__ __forceinline__
#else
#define VB_HD inline
#endif

#if defined(__CUDA_ARCH__)
#define VB_LD(p) __ldg(p)
#define VB_DMUL(a, b) __dmul_rn((a), (b))
#define VB_DADD(a, b) __dadd_rn((a), (b))
#define VB_D2F(a) __double2float_rn(a)
#else
#define VB_LD(p) (*(p))
#define VB_DMUL(a, b) ((a) * (b))      // host build uses -ffp-contract=off
#define VB_DADD(a, b) ((a) + (b))
#define VB_D2F(a) ((float)(a))
#endif

#define VB_MS_MAX_TERMS 256u

// One query term in POSITION order (descending ub; the non-essential terms are a suffix).
#define VB_MS_NO_TAB 0xffffffffu
struct VbMsRec {
    uint32_t slo, shi;      // the term's postings this launch scores: [slo, shi) of post_row / post_val (empty for NE terms)
    double w;               // idf-scaled query weight
    double suf;             // sum of ub over the positions after this one
    int32_t hidx;           // dense column of a frequent term, -1 = none
    uint32_t tab;           // offset of the term's bucket table in term_tab, VB_MS_NO_TAB = none (short list)
    uint32_t shift;         // rows per bucket = 1 << shift
    uint32_t plo, phi;      // the term's whole posting range (lookups of short lists search it directly)
    uint32_t pad;
};

struct VbMsQuery {          // per query, written by the plan kernel
    double tau_lo;          // tau lowered by 1e-9 relative (raised towards 0 for tau <= 0)
    uint32_t n_ess;         // essential terms (positions [0, n_ess))
    uint32_t active;        // 0 = not planned, 1 = K3M (posting units), 2 = K3H (row-range units)
    uint32_t shift;         // K3H: rows per work unit = 1 << shift
    uint32_t pad;
};

// ---- term presence lookups -------------------------------------------------------------------------
// lower bound of `row` in post_row[lo, hi)
VB_HD uint32_t vb_ms_lower_bound(const uint32_t* post_row, uint32_t lo, uint32_t hi, uint32_t row) {
    while (lo < hi) {
        const uint32_t mid = lo + ((hi - lo) >> 1);
        if (VB_LD(post_row + mid) < row) lo = mid + 1u; else hi = mid;
    }
    return lo;
}

// the postings of a term whose row falls in the bucket of `row`: [lo, hi) from the term's bucket table
VB_HD void vb_ms_bucket(const uint32_t* term_tab, uint32_t tab, uint32_t shift, uint32_t row, uint32_t& lo, uint32_t& hi) {
    const uint32_t* t = term_tab + (size_t)tab + (row >> shift);
    lo = VB_LD(t);
    hi = VB_LD(t + 1);
#if defined(__CUDA_ARCH__) && defined(VB_DEBUG_BOUNDS)
    assert(lo <= hi);
#endif
}

// value of a term in `row`: dense column (NaN = absent), bucket table + short search, or (short lists) a
// search of the whole list [lo0, hi0)
VB_HD bool vb_ms_lookup(const uint32_t* post_row, const float* post_val, const float* heavy_vals, uint32_t heavy_stride,
                        const uint32_t* term_tab, int32_t hidx, uint32_t tab, uint32_t shift, uint32_t lo0, uint32_t hi0,
                        uint32_t row, float& val) {
    if (hidx >= 0) {
        const float v = VB_LD(heavy_vals + (size_t)hidx * heavy_stride + row);
        val = v;
        return v == v;
    }
    uint32_t lo = lo0, hi = hi0;
    if (tab != VB_MS_NO_TAB) {
        vb_ms_bucket(term_tab, tab, shift, row, lo, hi);
        if (lo == hi) return false;
    }
    const uint32_t p = vb_ms_lower_bound(post_row, lo, hi, row);
    if (p < hi && VB_LD(post_row + p) == row) { val = VB_LD(post_val + p); return true; }
    return false;
}

// exact score of a row: the reference's two-pointer merge (ascending term id, fp64 mul then add, one
// rounding to fp32) over the forward index
VB_HD float vb_ms_rescore(const int64_t* sp_indptr, const uint32_t* sp_term, const float* sp_val, uint32_t row,
                          const uint32_t* q_term, const double* q_weight, uint32_t nt) {
    int64_t p = VB_LD(sp_indptr + row);
    const int64_t pe = VB_LD(sp_indptr + row + 1);
    double sc = 0.0;
    uint32_t j = 0;
    while (p < pe && j < nt) {
        const uint32_t t = VB_LD(sp_term + p), qt = VB_LD(q_term + j);
        if (t == qt) { sc = VB_DADD(sc, VB_DMUL(VB_LD(q_weight + j), (double)VB_LD(sp_val + p))); ++p; ++j; }
        else if (t < qt) ++p;
        else ++j;
    }
    return VB_D2F(sc);
}

// Everything one posting needs (pointers into the index + the query's position-ordered tables).
struct VbMsCtx {
    const uint32_t* post_row;
    const float* post_val;
    const float* heavy_vals;
    uint32_t heavy_stride;
    const uint32_t* term_tab;       // bucket tables of the index
    const int64_t* sp_indptr;       // forward index, for the exact re-score
    const uint32_t* sp_term;
    const float* sp_val;
    const uint32_t* q_term;         // this query's terms, ascending id  [nt]
    const double* q_weight;         // weights in the same order          [nt]
    const uint32_t* mask;           // filter bitmask of this query or nullptr
    // position-ordered tables of this query (shared memory on the device)
    const double* w;                // [nt]
    const double* suf;              // [nt]
    const int32_t* hidx;            // [nt]
    const uint32_t* tab;            // [nt] bucket table offset or VB_MS_NO_TAB
    const uint32_t* shift;          // [nt]
    const uint32_t* plo;            // [nt] whole posting range of the term
    const uint32_t* phi;
    uint32_t nt, n_ess;
    double tau_lo;                  // conservative threshold for the bound tests
    double delta;                   // 4 * nt * 2^-53
    float tau;                      // the list's threshold (exact compare)
};

// `partial` = the row's contributions from the positions before `first` that are ACCOUNTED FOR (present, or known
// absent); positions [0, own_before) are NOT accounted for yet: a term present there means another posting owns the
// row.  Looks up the remaining positions while the row can still reach tau, then — only for the few rows whose sum
// reaches tau — the ownership positions, then turns the order-free fp64 sum into the reference's fp32 score (verified,
// or re-scored from the forward index).
//   Order matters for cost, not for the result: the first version checked ownership FIRST (pe lookups per surviving
//   posting, ~4 on the benchmark queries, 98 % of them answering "absent") and pruned by score afterwards (~2 lookups,
//   98 % of the rows dropped).  Score first: the ownership lookups are paid by the ~1 % of rows that would be candidates.
VB_HD bool vb_ms_finish_row(const VbMsCtx& c, uint32_t first, uint32_t row, double partial, float& score, uint32_t own_before = 0u) {
    float lv;
    for (uint32_t i = first; i < c.nt; ++i) {
        if (partial + (i ? c.suf[i - 1u] : INFINITY) < c.tau_lo) return false;
        if (vb_ms_lookup(c.post_row, c.post_val, c.heavy_vals, c.heavy_stride, c.term_tab, c.hidx[i], c.tab[i], c.shift[i], c.plo[i], c.phi[i], row, lv))
            partial = VB_DADD(partial, VB_DMUL(c.w[i], (double)lv));
    }
    if (partial < c.tau_lo) return false;
    for (uint32_t i = 0; i < own_before; ++i)                   // ownership: an earlier essential term in the row owns it
        if (vb_ms_lookup(c.post_row, c.post_val, c.heavy_vals, c.heavy_stride, c.term_tab, c.hidx[i], c.tab[i], c.shift[i], c.plo[i], c.phi[i], row, lv)) return false;
    const float f_lo = VB_D2F(partial * (1.0 - c.delta)), f_hi = VB_D2F(partial * (1.0 + c.delta));
    score = f_lo == f_hi ? f_lo : vb_ms_rescore(c.sp_indptr, c.sp_term, c.sp_val, row, c.q_term, c.q_weight, c.nt);
    return score > c.tau;
}

// Score the posting (position pe, row, v).  Returns true and sets `score` iff the row is a candidate
// owned by this posting (its fp32 score, identical to the reference's, beats tau).
VB_HD bool vb_ms_score_posting(const VbMsCtx& c, uint32_t pe, uint32_t row, float v, float& score) {
    if (c.mask != nullptr && !((VB_LD(c.mask + (row >> 5)) >> (row & 31u)) & 1u)) return false;
    const double partial = VB_DMUL(c.w[pe], (double)v);
    if (partial + c.suf[pe] < c.tau_lo) return false;          // cannot reach tau even with every later term at its maximum
    return vb_ms_finish_row(c, pe + 1u, row, partial, score, pe);
}

// ---- plan: one query, `nt` terms.  Thread j owns term j in phases 1-2 and POSITION j in phase 3; phases are
// separated by barriers on the device and by loops in the CPU emulation. ---------------------------------
// Position order = descending ub (ties: term index).  It does not depend on tau, so it is the same in every
// stage of a search, and the non-essential terms (the lowest-ub terms whose ub sum stays below tau) are always
// a SUFFIX of it.  That makes row ownership stable: the posting of the earliest position that contains a row
// owns it in every stage, whatever the thresholds were when the other stages ran.
struct VbMsPlanShared {
    double ub[VB_MS_MAX_TERMS];         // term order
    double ub_pos[VB_MS_MAX_TERMS];     // position order
    uint32_t len[VB_MS_MAX_TERMS];      // postings inside the row range, term order
    uint32_t len_pos[VB_MS_MAX_TERMS];  // position order
    uint32_t slo[VB_MS_MAX_TERMS], shi[VB_MS_MAX_TERMS];    // term order
    uint32_t term_at[VB_MS_MAX_TERMS];  // position -> term
    uint32_t n_ess;
};

// first posting of a term with row >= target: the bucket table leaves a handful of search steps
VB_HD uint32_t vb_ms_seg_bound(const uint32_t* post_row, const uint32_t* term_tab, uint32_t plo, uint32_t phi,
                               uint32_t tab, uint32_t shift, uint32_t n_rows, uint32_t target) {
    if (target >= n_rows) return phi;
    if (target == 0u) return plo;                              // (the staged flow plans the whole index: no loads at all)
    uint32_t lo = plo, hi = phi;
    if (tab != VB_MS_NO_TAB) vb_ms_bucket(term_tab, tab, shift, target, lo, hi);
    return vb_ms_lower_bound(post_row, lo, hi, target);
}

// phase 1: row-range slice and upper bound of term j
VB_HD void vb_ms_plan_load(VbMsPlanShared& s, uint32_t j, const uint32_t* post_row, const uint32_t* term_tab, uint32_t plo, uint32_t phi,
                           uint32_t tab, uint32_t shift, uint32_t n_rows, uint32_t seg_row0, uint32_t seg_row1, double ub) {
    const uint32_t lo = vb_ms_seg_bound(post_row, term_tab, plo, phi, tab, shift, n_rows, seg_row0);
    const uint32_t hi = vb_ms_seg_bound(post_row, term_tab, plo, phi, tab, shift, n_rows, seg_row1);
    s.slo[j] = lo; s.shi[j] = hi; s.len[j] = hi - lo; s.ub[j] = ub;
}

// phase 2: position of term j in descending-ub order
VB_HD void vb_ms_plan_position(VbMsPlanShared& s, uint32_t j, uint32_t nt) {
    uint32_t before = 0;
    for (uint32_t i = 0; i < nt; ++i) before += (s.ub[i] > s.ub[j] || (s.ub[i] == s.ub[j] && i < j)) ? 1u : 0u;
    s.ub_pos[before] = s.ub[j];
    s.len_pos[before] = s.len[j];
    s.term_at[before] = j;
}

// phase 3, position i: the ub sum after it (summed from the tail: small values first), whether it is essential
// under tau (the 2e-9 margin dwarfs the rounding of sums of <= 256 terms), and the part of its postings this
// STAGE scores: the query's postings are numbered in position order, a stage takes numbers [stage_lo, stage_hi).
struct VbMsPos { double suf; uint32_t w0, w1; bool essential; };
VB_HD VbMsPos vb_ms_plan_pos(const VbMsPlanShared& s, uint32_t i, uint32_t nt, double tau_d, uint32_t budget_pct,
                             uint64_t stage_lo, uint64_t stage_hi) {
    VbMsPos r;
    double acc = 0.0;
    for (uint32_t k = nt; k-- > i + 1u;) acc += s.ub_pos[k];
    r.suf = acc;
    const bool ok = budget_pct != 0u && tau_d > 0.0 && tau_d < INFINITY;
    const uint32_t pct = budget_pct < 100u ? budget_pct : 100u;
    r.essential = !(ok && acc + s.ub_pos[i] < tau_d * (0.01 * (double)pct) * (1.0 - 2e-9));
    uint64_t cum = 0;
    for (uint32_t k = 0; k < i; ++k) cum += s.len_pos[k];
    const uint64_t len = s.len_pos[i];
    const uint64_t lo = stage_lo > cum ? (stage_lo - cum < len ? stage_lo - cum : len) : 0;
    const uint64_t hi = stage_hi > cum ? (stage_hi - cum < len ? stage_hi - cum : len) : 0;
    r.w0 = (uint32_t)lo;
    r.w1 = r.essential ? (uint32_t)hi : (uint32_t)lo;
    return r;
}

// K3H (sparse_mh.cuh): width (as a shift) of a long query's row ranges — the largest power of two with
// essential postings * W / rows <= VB_MH_TARGET
#define VB_MH_TARGET 1024u
VB_HD uint32_t vb_mh_shift(uint64_t essential_postings, uint32_t seg_rows) {
    uint32_t shift = 31;
    while (shift > 6u && (essential_postings << shift) > (uint64_t)VB_MH_TARGET * (seg_rows ? seg_rows : 1u)) --shift;
    return shift;
}

VB_HD double vb_ms_tau_lo(double tau_d) { return tau_d > 0.0 ? tau_d * (1.0 - 1e-9) : tau_d * (1.0 + 1e-9); }

// K3M keeps a row whose score EQUALS the list's threshold: the stages visit rows in posting order (descending ub), not
// in row order, so a row that ties with the k'-th best can arrive after it and still win the tie on its lower row id;
// the compaction then picks by key.  So a K3M launch runs under the next float below the list's tau (the rule of
// vb_tau_import_kernel): the plan's partition, the bound tests (tau_lo) and the exact compare all derive from it —
// lowering the exact compare alone is not enough, the fp32 rounding of a tied row's score may lie above its fp64
// sum by more than tau_lo's margin.  Every row is still scored once; the cost is an append per tied row.
VB_HD float vb_ms_exact_tau(float tau) { return nextafterf(tau, -INFINITY); }

#ifdef __CUDACC__
#include "common.cuh"

// ---- bucket tables (index build): tab[off_e + b] = first posting of term e whose row >= b << shift_e -------
struct VbTabTerm { uint32_t start, end, off, shift; };     // posting range, first table entry, bucket shift

__global__ void __launch_bounds__(256)
vb_ms_tab_fill_kernel(const uint32_t* __restrict__ post_row, const VbTabTerm* __restrict__ terms, uint32_t n_terms,
                      uint64_t total, uint32_t* __restrict__ tab)
{
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t lo = 0, hi = n_terms;                       // last term whose table starts at or before entry i
        while (hi - lo > 1u) {
            const uint32_t mid = lo + ((hi - lo) >> 1);
            if ((uint64_t)terms[mid].off <= i) lo = mid; else hi = mid;
        }
        const VbTabTerm t = terms[lo];
        const uint64_t target = (i - t.off) << t.shift;
        tab[i] = target > 0xffffffffull ? t.end : vb_ms_lower_bound(post_row, t.start, t.end, (uint32_t)target);
    }
}

struct VbMsPlanArgs {
    const uint32_t* post_row;
    const uint32_t* term_tab;    // bucket tables of the index
    const uint32_t* q_tab;       // [n_qterms] table offset per query term (VB_MS_NO_TAB = none)
    const uint8_t* q_shift;      // [n_qterms]
    uint32_t n_rows;             // rows covered by the inverted index
    const int64_t* q_indptr;     // [B+1]
    const double* q_weight;      // [n_qterms] term order
    const double* q_ub;          // [n_qterms]
    const int32_t* q_hidx;       // [n_qterms] or nullptr
    const uint32_t* q_plo;       // [n_qterms] full posting range of the term (frequent terms included)
    const uint32_t* q_phi;
    const uint8_t* q_ms;         // [B] 0 = not ours, 1 = K3M (short queries), 2 = K3H (long queries, sparse_mh.cuh)
    uint32_t classes;            // bit 0: plan the K3M queries, bit 1: plan the K3H queries
    uint32_t* hunit_prefix;      // [B + 1] out: exclusive prefix of the K3H work units per query
    const float* tau;            // [n_lists]
    VbMsRec* rec;                // [n_qterms] out, position order
    VbMsQuery* qinfo;            // [B] out
    uint32_t* unit_prefix;       // [n_qterms + 1] out: exclusive prefix of the work units per (query, position)
    uint32_t* counters;          // [0] blocks done (self-resetting), [1] next work unit (reset here), [2] total units
    uint32_t n_queries, n_qterms;
    uint32_t seg_row0, seg_row1; // rows this launch covers
    uint64_t stage_lo, stage_hi; // the query's postings (numbered in position order) this launch scores
    uint32_t chunk;              // postings per work unit
    uint32_t budget_pct;         // MaxScore budget in % of tau (100 = the full MaxScore partition)
    uint32_t budget_pct_long;    // the same for the K3H (long) queries
    uint32_t long_terms;         // K3M queries of more terms than this plan with budget_pct_mslong:
    uint32_t budget_pct_mslong;  //   a long query's non-essential ub sum (the slack of the per-posting bound test) is better kept
                                 //   well below tau — more essential postings, but far fewer of them reach the lookups
};

__global__ void __launch_bounds__(256)
vb_ms_plan_kernel(const VbMsPlanArgs a)
{
    __shared__ VbMsPlanShared s;
    __shared__ uint32_t s_last;
    const uint32_t q = blockIdx.x, j = threadIdx.x;
    const uint32_t t_lo = (uint32_t)a.q_indptr[q];
    const uint32_t nt = (uint32_t)a.q_indptr[q + 1] - t_lo;
    const uint32_t cls = nt != 0u ? a.q_ms[q] : 0u;
    const bool active = cls != 0u && ((a.classes >> (cls - 1u)) & 1u);
    __shared__ unsigned long long s_ess_post;
    if (j == 0) s_ess_post = 0ull;
    const float tau_f = a.tau[a.n_queries + q];
    const double tau_d = (double)(cls == 1u ? vb_ms_exact_tau(tau_f) : tau_f);     // K3M: ties kept (vb_ms_exact_tau)
    if (active) {
        if (j < nt) vb_ms_plan_load(s, j, a.post_row, a.term_tab, a.q_plo[t_lo + j], a.q_phi[t_lo + j], a.q_tab[t_lo + j], a.q_shift[t_lo + j],
                                    a.n_rows, a.seg_row0, a.seg_row1, a.q_ub[t_lo + j]);
        if (j == 0) s.n_ess = 0u;
        __syncthreads();
        if (j < nt) vb_ms_plan_position(s, j, nt);
        __syncthreads();
        if (j < nt) {                                          // thread j now finishes POSITION j
            const VbMsPos ps = vb_ms_plan_pos(s, j, nt, tau_d, cls == 2u ? a.budget_pct_long : (nt > a.long_terms ? a.budget_pct_mslong : a.budget_pct), a.stage_lo, a.stage_hi);
            const uint32_t t = s.term_at[j];
            VbMsRec r;
            r.slo = s.slo[t] + ps.w0; r.shi = s.slo[t] + ps.w1; r.w = a.q_weight[t_lo + t];
            r.suf = ps.suf;
            r.hidx = a.q_hidx ? a.q_hidx[t_lo + t] : -1;
            r.tab = a.q_tab[t_lo + t]; r.shift = a.q_shift[t_lo + t];
            r.plo = a.q_plo[t_lo + t]; r.phi = a.q_phi[t_lo + t]; r.pad = 0u;
            a.rec[t_lo + j] = r;
            a.unit_prefix[t_lo + j] = cls == 1u ? (ps.w1 - ps.w0 + a.chunk - 1u) / a.chunk : 0u;   // counts; scanned below
            if (ps.essential) atomicAdd(&s.n_ess, 1u);
            if (cls == 2u && ps.w1 > ps.w0) atomicAdd(&s_ess_post, (unsigned long long)(ps.w1 - ps.w0));
        }
        __syncthreads();
        if (j == 0) {
            VbMsQuery qi;
            qi.tau_lo = vb_ms_tau_lo(tau_d); qi.n_ess = s.n_ess; qi.active = cls; qi.shift = 0u; qi.pad = 0u;
            uint32_t hunits = 0u;
            if (cls == 2u && s_ess_post != 0ull) {               // K3H: row ranges of ~VB_MH_TARGET essential postings
                const uint32_t seg_rows = a.seg_row1 - a.seg_row0;
                qi.shift = vb_mh_shift((uint64_t)s_ess_post, seg_rows);
                hunits = (uint32_t)(((uint64_t)seg_rows + (1ull << qi.shift) - 1ull) >> qi.shift);
            }
            a.qinfo[q] = qi;
            a.hunit_prefix[q] = hunits;
        }
    } else {
        for (uint32_t i = j; i < nt; i += blockDim.x) a.unit_prefix[t_lo + i] = 0u;
        if (j == 0) { VbMsQuery qi; qi.tau_lo = 0.0; qi.n_ess = 0u; qi.active = 0u; qi.shift = 0u; qi.pad = 0u; a.qinfo[q] = qi; a.hunit_prefix[q] = 0u; }
    }
    // the last CTA to finish turns the per-position unit counts into an exclusive prefix sum
    __threadfence();
    __syncthreads();
    if (j == 0) s_last = atomicAdd(&a.counters[0], 1u) == gridDim.x - 1u ? 1u : 0u;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    __shared__ uint32_t s_scan[256];
    const uint32_t n = a.n_qterms;
    const uint32_t per = (n + 255u) / 256u;
    const uint32_t b0 = j * per, b1 = min(n, b0 + per);
    uint32_t sum = 0;
    volatile uint32_t* up = a.unit_prefix;
    for (uint32_t i = b0; i < b1; ++i) sum += up[i];
    s_scan[j] = sum;
    __syncthreads();
    for (uint32_t o = 1; o < 256u; o <<= 1) {               // inclusive scan of the 256 partial sums
        const uint32_t v = j >= o ? s_scan[j - o] : 0u;
        __syncthreads();
        s_scan[j] += v;
        __syncthreads();
    }
    uint32_t run = j ? s_scan[j - 1u] : 0u;
    for (uint32_t i = b0; i < b1; ++i) { const uint32_t c = up[i]; up[i] = run; run += c; }
    if (j == 255u) { up[n] = s_scan[255]; a.counters[2] = s_scan[255]; a.counters[1] = 0u; a.counters[0] = 0u; }
    // same for the K3H units per query
    __syncthreads();
    {
        const uint32_t nq = a.n_queries;
        const uint32_t perq = (nq + 255u) / 256u;
        const uint32_t c0 = j * perq, c1 = min(nq, c0 + perq);
        volatile uint32_t* hp = a.hunit_prefix;
        uint32_t hs = 0;
        for (uint32_t i = c0; i < c1; ++i) hs += hp[i];
        s_scan[j] = hs;
        __syncthreads();
        for (uint32_t o = 1; o < 256u; o <<= 1) {
            const uint32_t v = j >= o ? s_scan[j - o] : 0u;
            __syncthreads();
            s_scan[j] += v;
            __syncthreads();
        }
        uint32_t hrun = j ? s_scan[j - 1u] : 0u;
        for (uint32_t i = c0; i < c1; ++i) { const uint32_t c = hp[i]; hp[i] = hrun; hrun += c; }
        if (j == 255u) { hp[nq] = s_scan[255]; a.counters[3] = 0u; }
    }
}

struct VbMsArgs {
    const uint32_t* post_row;
    const float* post_val;
    const float* heavy_vals;
    uint32_t heavy_stride;
    const int64_t* sp_indptr;
    const uint32_t* sp_term;
    const float* sp_val;
    const int64_t* q_indptr;
    const uint32_t* q_term;      // term order
    const double* q_weight;      // term order
    const uint32_t* slot_q;      // [n_qterms] query of every term slot
    const VbMsRec* rec;
    const VbMsQuery* qinfo;
    const uint32_t* unit_prefix; // [n_qterms + 1]
    uint32_t* counters;
    const uint32_t* term_tab;    // bucket tables of the index
    const uint32_t* mask;        // [n_filters][mask_words] or nullptr
    const int32_t* mask_of;      // [B] or nullptr
    const float* tau;
    VbLists lists;
    uint32_t mask_words, n_qterms, n_queries, row_base, chunk, nt_max;
};

#define VB_MS_THREADS 128
#define VB_MS_U 4u               // postings per thread in flight

static size_t vb_ms_smem_bytes(uint32_t nt_max) { return (size_t)nt_max * (8u + 8u + 4u * 5u) + 16u; }

__global__ void __launch_bounds__(VB_MS_THREADS)
vb_ms_score_kernel(const VbMsArgs a)
{
    extern __shared__ __align__(16) unsigned char vb_ms_smem[];
    double* s_w = reinterpret_cast<double*>(vb_ms_smem);                 // [nt_max]
    double* s_suf = s_w + a.nt_max;                                      // [nt_max]
    int32_t* s_hidx = reinterpret_cast<int32_t*>(s_suf + a.nt_max);      // [nt_max]
    uint32_t* s_tab = reinterpret_cast<uint32_t*>(s_hidx + a.nt_max);    // [nt_max]
    uint32_t* s_shift = s_tab + a.nt_max;                                // [nt_max]
    uint32_t* s_plo = s_shift + a.nt_max;                                // [nt_max]
    uint32_t* s_phi = s_plo + a.nt_max;                                  // [nt_max]
    __shared__ uint32_t s_unit;
    const uint32_t tid = threadIdx.x;
    const uint32_t total = a.unit_prefix[a.n_qterms];
    for (;;) {
        __syncthreads();                                                 // the previous unit's tables are no longer read
        if (tid == 0) s_unit = atomicAdd(&a.counters[1], 1u);
        __syncthreads();
        const uint32_t u = s_unit;
        if (u >= total) break;
        // slot = last index with unit_prefix[slot] <= u  (empty slots share their successor's prefix)
        uint32_t lo = 0, hi = a.n_qterms;
        while (hi - lo > 1u) {
            const uint32_t mid = lo + ((hi - lo) >> 1);
            if (__ldg(a.unit_prefix + mid) <= u) lo = mid; else hi = mid;
        }
        const uint32_t slot = lo;
        const uint32_t q = __ldg(a.slot_q + slot);
        const uint32_t t_lo = (uint32_t)__ldg(a.q_indptr + q);
        const uint32_t nt = (uint32_t)__ldg(a.q_indptr + q + 1) - t_lo;
        const uint32_t pe = slot - t_lo;
        const VbMsRec e = a.rec[slot];
        const uint32_t p0 = e.slo + (u - __ldg(a.unit_prefix + slot)) * a.chunk;
        const uint32_t p1 = min(e.shi, p0 + a.chunk);
        VB_CHECK(slot < a.n_qterms && q < a.n_queries && pe < nt && nt <= a.nt_max && p0 < p1 && e.plo <= e.slo && e.shi <= e.phi);
        for (uint32_t i = tid; i < nt; i += VB_MS_THREADS) {
            const VbMsRec r = a.rec[t_lo + i];
            s_w[i] = r.w; s_suf[i] = r.suf; s_hidx[i] = r.hidx;
            s_tab[i] = r.tab; s_shift[i] = r.shift; s_plo[i] = r.plo; s_phi[i] = r.phi;
        }
        const VbMsQuery qi = a.qinfo[q];
        const uint32_t list = a.n_queries + q;
        VbMsCtx c;
        c.post_row = a.post_row; c.post_val = a.post_val; c.heavy_vals = a.heavy_vals; c.heavy_stride = a.heavy_stride;
        c.term_tab = a.term_tab;
        c.sp_indptr = a.sp_indptr; c.sp_term = a.sp_term; c.sp_val = a.sp_val;
        c.q_term = a.q_term + t_lo; c.q_weight = a.q_weight + t_lo;
        c.mask = nullptr;
        if (a.mask != nullptr && a.mask_of != nullptr) {
            const int32_t f = __ldg(a.mask_of + q);
            if (f >= 0) c.mask = a.mask + (size_t)f * a.mask_words;
        }
        c.w = s_w; c.suf = s_suf; c.hidx = s_hidx; c.tab = s_tab; c.shift = s_shift; c.plo = s_plo; c.phi = s_phi;
        c.nt = nt; c.n_ess = qi.n_ess; c.tau_lo = qi.tau_lo;
        c.delta = (double)(4u * nt) * 1.1102230246251565e-16;
        c.tau = vb_ms_exact_tau(a.tau[list]);                           // (the plan derived tau_lo from the same value)
        __syncthreads();
        // U postings per thread per step: their (row, value) loads and filter words are issued together
        for (uint32_t pb = p0 + tid; pb < p1; pb += VB_MS_U * VB_MS_THREADS) {
            uint32_t row[VB_MS_U];
            float val[VB_MS_U];
            uint32_t mw[VB_MS_U];
#pragma unroll
            for (uint32_t k = 0; k < VB_MS_U; ++k) {
                const uint32_t p = pb + k * VB_MS_THREADS;
                const bool ok = p < p1;
                row[k] = ok ? __ldg(a.post_row + p) : 0xffffffffu;
                val[k] = ok ? __ldg(a.post_val + p) : 0.0f;
            }
#pragma unroll
            for (uint32_t k = 0; k < VB_MS_U; ++k)
                mw[k] = (c.mask != nullptr && row[k] != 0xffffffffu) ? __ldg(c.mask + (row[k] >> 5)) : 0xffffffffu;
            const uint32_t* keep_mask = c.mask;
            c.mask = nullptr;                                            // the filter bit is tested here, on the prefetched word
#pragma unroll
            for (uint32_t k = 0; k < VB_MS_U; ++k) {
                if (row[k] == 0xffffffffu || !((mw[k] >> (row[k] & 31u)) & 1u)) continue;
                float score;
                // the append counter is picked by a hash of the row: one query's candidates often come from one or
                // two work units (= CTAs), and must still spread over all sub-ranges of its list
                if (vb_ms_score_posting(c, pe, row[k], val[k], score))
                    vb_push_sub(a.lists, list, ((row[k] * 2654435761u) >> 20) & a.lists.sub_mask, score, a.row_base + row[k]);
            }
            c.mask = keep_mask;
        }
    }
}
#endif  // __CUDACC__
