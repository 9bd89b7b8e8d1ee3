// K3b: Ascores.  cpp/Ascore.cpp:212-254 (calculateAscores), :157-210 (calculateAmbiguity),
// cpp/ModifiedPeptide.cpp:259-320 (getSiteDeterminingIons).  The merges themselves (asc_merge_type) live in
// pa_kernels.cuh; this file holds how the work is cut and handed out.
#pragma once

// minimum of floats of either sign through integer atomics (the slot starts at +inf)
__device__ __forceinline__ void asc_atomic_min(float* slot, float v) {
    if (v >= 0.f) atomicMin((int*)slot, __float_as_int(v));
    else atomicMax((unsigned int*)slot, __float_as_uint(v));
}

// ---------------------------------------------------------------------------------------------------------------
// K3b scheduling: the unit of work is one (entry, tied competitor) pair, handed out 32 at a time from a global
// cursor to one resident wave of warps.  The pairs are numbered through an exclusive scan over the work-sorted
// entry list (stream class, then estimated merge length, longest first), so a kernel no longer lasts as long as
// its heaviest entry (config 5: entries with up to 9 tied competitors, 6-8 % of the warp slots busy) or its
// heaviest warp.  A pair runs the register / stream merges (asc_merge_type, pa_kernels.cuh) for every ion type
// and lowers the entry's Ascore with an atomic minimum; entries a merge cannot cover go, once, to k_ascore_generic.
// ---------------------------------------------------------------------------------------------------------------
struct PaAscItemArgs {
    int32_t* item_cnt;           // [n_entries + 1] tied competitors of the i-th entry of the sorted list (0 past the work)
    const int32_t* item_off;     // [n_entries + 1] exclusive scan of item_cnt
    unsigned long long* cursor;  // [4] next pair of each stream class (zeroed before the launch)
    int* gen_flag;               // [n_entries] entry already queued for the generic kernel (zeroed)
};

// pairs per entry of the sorted work list; Ascores of the entries with work start at +inf
__global__ void k_asc_item_count(PaAscArgs a, PaAscItemArgs it) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i > a.n_entries) return;
    const int64_t n_work = (int64_t)a.work_count[0] + a.work_count[1] + a.work_count[2] + a.work_count[3];
    int c = 0;
    if (i < n_work) {
        const int64_t t = a.work_sorted[i];
        c = __popcll(a.tie[t]);
        if (a.ascores) a.ascores[a.mod_lo + t] = __int_as_float(0x7f800000);
    }
    it.item_cnt[i] = c;
}

// Ambiguity of the best isoform of entry t against its comp-th tied competitor (cpp/Ascore.cpp:157-210).
// Returns false when a merge does not cover the shape (-> generic kernel).  DEEP: a scorer with n_top > 10, whose depth
// argmax goes on over depths 10 .. n_top-1 (scores from dp.T at the K2d counts dp.cnt).
template <int NQ, bool DEEP>
__device__ __forceinline__ bool asc_pair(const PaCfg& cfg, const PaBatchDev& b, const PaAscArgs& a, int64_t t, int comp,
                                         float& amb, const PaDeep& dp) {
    const int32_t p = a.mod_psm[t];
    const int j = (int)(a.mod_lo + t - a.mod_off[p]);
    const int S = a.psm_S[p], k = b.n_mod[p];
    const int64_t ib = a.iso_off[p];
    AscPep q;
    const int po = b.pep_off[p];
    q.pep = b.pep + po; q.L = b.pep_off[p + 1] - po; q.Z = b.max_charge[p];
    q.a0 = 0; q.a1 = 0; q.aux_pos = b.aux_pos; q.aux_mass = b.aux_mass; q.aux_lo = 0; q.aux_hi = 0;
    if (b.aux_off != nullptr) {
        q.a0 = b.aux_off[p]; q.a1 = b.aux_off[p + 1];
        for (int x = q.a0; x < q.a1; x++) {
            const uint32_t pos = q.aux_pos[x];
            const int idx = pos > 0 ? (int)pos - 1 : 0;
            if (idx < 64) q.aux_lo |= 1ull << idx; else if (idx < 128) q.aux_hi |= 1ull << (idx - 64);
        }
    }
    amb = 0.f;
    if ((q.L < 2) || (NQ <= 4 && (cfg.has_nl || q.Z > NQ))) return false;
    const int sp = b.psm_spec[p];
    AscPeaks pk;
    pk.pp = b.rpk + (b.spec_off[sp] - b.spec_base); pk.R = b.rcount[sp];
    pk.ctab = b.ctab + (size_t)sp * PA_NCELL;
    { const float2 chead = b.chead[sp]; pk.cbase = chead.x; pk.cinv = chead.y; }
    const uint32_t best = a.best_idx[p];
    const uint64_t best_bits = pa_unrank(cfg.binom, S, k, best);
    uint64_t rem = best_bits;
    for (int jj = 0; jj < j; jj++) rem &= rem - 1;
    const int site = __ffsll((long long)rem) - 1;
    uint64_t tt = a.tie[t];
    for (int c = 0; c < comp; c++) tt &= tt - 1;
    const int u = __ffsll((long long)tt) - 1;
    // residue masks of both isoforms: the competitor has the mod of `site` on site u instead
    uint64_t alo = 0, ahi = 0;
    int pos_site = 0, pos_u = 0;
    {
        int n = 0;
        for (int i = 0; i < q.L && n < 64; i++) {
            const int c = (int)q.pep[i] - 'A';
            const bool is = ((cfg.mod_letters >> c) & 1u) || (cfg.allow_n && i == 0) || (cfg.allow_c && i == q.L - 1);
            if (!is) continue;
            if ((best_bits >> n) & 1ull) { if (i < 64) alo |= 1ull << i; else ahi |= 1ull << (i - 64); }
            if (n == site) pos_site = i;
            if (n == u) pos_u = i;
            n++;
        }
    }
    uint64_t blo = alo, bhi = ahi;
    if (pos_site < 64) blo &= ~(1ull << pos_site); else bhi &= ~(1ull << (pos_site - 64));
    if (pos_u < 64) blo |= 1ull << pos_u; else bhi |= 1ull << (pos_u - 64);
    const uint32_t ci = pa_rank(cfg.binom, S, k, (best_bits & ~(1ull << site)) | (1ull << u));
    const float wA = a.iso.w[ib + best], wB = a.iso.w[ib + ci];
    if ((double)fabsf(__fsub_rn(wA, wB)) < 1e-6) return true;                 // cpp/Ascore.cpp:161-163: ambiguity 0
    // depth with the largest score difference (cpp/Ascore.cpp:165-175), first strict maximum
    int depth = 0;
    {
        const unsigned long long loA = a.iso.lo[ib + best], hiA = a.iso.hi[ib + best];
        const unsigned long long loB = a.iso.lo[ib + ci], hiB = a.iso.hi[ib + ci];
        const int nfA = (int)a.iso.nfrag[ib + best], nfB = (int)a.iso.nfrag[ib + ci];
        float max_diff = 0.f;
        for (int d = 0; d < PA_N_TOP; d++) {
            const float diff = __fsub_rn(__ldg(cfg.T + pa_tab_index(nfA, pa_cum_get(loA, hiA, d), d)),
                                         __ldg(cfg.T + pa_tab_index(nfB, pa_cum_get(loB, hiB, d), d)));
            if (diff > max_diff) { max_diff = diff; depth = d; }
        }
        if constexpr (DEEP) {
            const uint16_t* cA = dp.cnt + (size_t)(ib + best) * dp.nd;
            const uint16_t* cB = dp.cnt + (size_t)(ib + ci) * dp.nd;
            for (int dd = 0; dd < dp.nd; dd++) {
                const float diff = __fsub_rn(__ldg(dp.T + pa_tab_index_deep(nfA, cA[dd], dd, dp.nd)),
                                             __ldg(dp.T + pa_tab_index_deep(nfB, cB[dd], dd, dp.nd)));
                if (diff > max_diff) { max_diff = diff; depth = PA_N_TOP + dd; }
            }
        }
    }
    int hitsA = 0, hitsB = 0, trialsA = 0, trialsB = 0;
    for (int ti = 0; ti < cfg.n_types; ti++)
        if (!asc_merge_type<NQ>(cfg, q, pk, cfg.types[ti], alo, ahi, blo, bhi, depth, hitsA, trialsA, hitsB, trialsB))
            return false;
    if constexpr (DEEP) amb = __fsub_rn(pa_depth_score(cfg.T, dp, trialsA, hitsA, depth), pa_depth_score(cfg.T, dp, trialsB, hitsB, depth));
    else amb = __fsub_rn(__ldg(cfg.T + pa_tab_index(trialsA, hitsA, depth)), __ldg(cfg.T + pa_tab_index(trialsB, hitsB, depth)));
    return true;
}

#ifndef PA_ASC3_GRAB
#define PA_ASC3_GRAB 1           // rounds of 32 pairs a warp takes per visit to the cursor
#endif
template <int NQ, int CLS, bool DEEP>
__global__ void __launch_bounds__(128, (NQ <= 1 ? PA_ASC_MINBLOCKS : (NQ <= 2 ? PA_ASC2_MINBLOCKS : (NQ <= 4 ? PA_ASC4_MINBLOCKS : PA_ASC12_MINBLOCKS))))
k_ascore_pairs(PaCfg cfg, PaBatchDev b, PaAscArgs a, PaAscItemArgs it, PaDeep deep) {
    const int lane = threadIdx.x & 31;
    int64_t first = 0;                       // classes are contiguous in the sorted entry list, hence in the pair numbering
#pragma unroll
    for (int c = 0; c < CLS; c++) first += a.work_count[c];
    const int64_t last = first + a.work_count[CLS];
    const int64_t g0 = it.item_off[first], g1 = it.item_off[last];
    if (g1 <= g0) return;
    for (;;) {
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(it.cursor + CLS, 32ull * PA_ASC3_GRAB);
        base = __shfl_sync(PA_FULL, base, 0);
        if ((int64_t)base >= g1 - g0) break;
        for (int rr = 0; rr < PA_ASC3_GRAB; rr++) {
            const int64_t g = g0 + (int64_t)base + rr * 32 + lane;
            if (g >= g1) continue;
            // entry of pair g: last position of [first, last) whose first pair is <= g
            int64_t lo = first, hi = last;
            while (hi - lo > 1) { const int64_t mid = (lo + hi) >> 1; if ((int64_t)it.item_off[mid] <= g) lo = mid; else hi = mid; }
            const int64_t t = a.work_sorted[lo];
            float amb;
            // (`deep` is the last parameter, and the n_top = 10 form does not read it: its code stays that of the kernel
            // before the parameter existed)
            if (asc_pair<NQ, DEEP>(cfg, b, a, t, (int)(g - it.item_off[lo]), amb, DEEP ? deep : PaDeep())) {
                if (a.ascores) asc_atomic_min(a.ascores + a.mod_lo + t, amb);
            } else if (atomicExch(it.gen_flag + t, 1) == 0)
                a.generic_list[atomicAdd(a.generic_count, 1)] = (int32_t)t;
        }
    }
}
