// Kernels of libpyascore_b200 (sm_100a).  The unit of domain work decides who owns it:
//   K0  k_tail_table     one block per trial count n: float32-faithful binomial score table
//   K1  k_bin_rows       one warp per spectrum: top-n_top peaks per bin_size-Th bin (BinnedSpectra), row form for the
//                        spectra that are the rule (pa_bin_rows.cuh); k_bin_topn takes the ones it declines
//   P1  k_plan           one thread per PSM: validation, #sites, #isoforms, work units
//   K2  k_count_score    one warp per unit of <=1024 positional isoforms: fragments, matches, PepScore
//   K2d k_count_deep     n_top > 10 only: one warp per K2 unit, lane per isoform: cumulative counts of depths 10..n_top-1
//   K3a k_select_thread  one thread per PSM: reference-order best isoform, tied competitors per site,
//                        sort keys of the Ascore entries; k_select (one warp per PSM) for the PSMs it declines
//   K3b k_ascore_pairs   one thread per (PSM, modified site, tied competitor) pair, pairs handed out from a global
//                        cursor in work-sorted order (pa_ascore.cuh): site-determining-ion merges -> Ascore
//   K3c k_ascore_generic one warp per entry: list-materialising form for the shapes K3b declines
// Nothing here is a dense contraction: no tensor cores.  The work is integer / float32 / a little
// FP64 per fragment, bound by instruction issue and shared-memory latency (DESIGN.md).
#pragma once
#include "pa_device.cuh"

// ---------------------------------------------------------------------------------------------
// K0: score table  T[(n(n+1)/2 + k) * 10 + d] = | -10 * log10 P(X >= k) |,  X ~ Binomial(n, p_d)
// cpp/Util.cpp:28-83 + cpp/Ascore.cpp:23-36, :127-133, in the reference's float32 rounding order.
// logd[m] = log((double)m) and lps/lpf = logf(p_d), (float)log(1-p_d) are host constants from the
// platform libm (the reference gets them from the same place).  One thread per depth: depths 0..9 go to T, depths
// 10 .. n_top-1 of a scorer with n_top > 10 to T_deep (PaDeep).
// ---------------------------------------------------------------------------------------------
struct PaTailArgs {
    float* T;
    const double* logd;
    float lps[PA_MAX_N_TOP], lpf[PA_MAX_N_TOP];
    double log10e;
    float* T_deep;
    int n_top;
};

__device__ __forceinline__ float* pa_tail_cell(const PaTailArgs& a, int n, int k, int d) {
    return d < PA_N_TOP ? a.T + pa_tab_index(n, k, d) : a.T_deep + pa_tab_index_deep(n, k, d - PA_N_TOP, a.n_top - PA_N_TOP);
}

__global__ void __launch_bounds__(128) k_tail_table(PaTailArgs a, int n0, int n1) {
    extern __shared__ float s_lbc[];
    const int n = n0 + blockIdx.x;
    if (n > n1) return;
    for (int k = threadIdx.x; k <= n; k += blockDim.x) {
        int kk = (n - k < k) ? n - k : k;
        float c = 0.f;
        for (int m = n - kk + 1; m <= n; m++) c = __double2float_rn(__dadd_rn((double)c, a.logd[m]));
        for (int m = 2; m <= kk; m++) c = __double2float_rn(__dsub_rn((double)c, a.logd[m]));
        s_lbc[k] = c;
    }
    __syncthreads();
    if (threadIdx.x < a.n_top) {
        const int d = threadIdx.x;
        const float lps = a.lps[d], lpf = a.lpf[d];
        float tail = __int_as_float(0xff800000);   // -inf
        *pa_tail_cell(a, n, 0, d) = fabsf(__fmul_rn(-10.f, __double2float_rn(__dmul_rn(a.log10e, 0.0))));
        for (int k = n; k >= 1; k--) {
            float pmf = __fadd_rn(__fadd_rn(s_lbc[k], __fmul_rn((float)k, lps)), __fmul_rn((float)(n - k), lpf));
            tail = pa_log_sum(tail, pmf);
            float l10 = __double2float_rn(__dmul_rn(a.log10e, (double)tail));
            *pa_tail_cell(a, n, k, d) = fabsf(__fmul_rn(-10.f, l10));
        }
    }
}

// ---------------------------------------------------------------------------------------------
// K1: BinnedSpectra.  cpp/Spectra.cpp:43-68 (bounds + bin index), :24-41 (top n_top by intensity).
// Fast path: the spectrum fits the warp's shared-memory slot and is m/z-sorted, so a bin is a
// contiguous run and each lane ranks its peak by scanning outwards inside the run.
// General path (unsorted or oversized spectra): all-pairs ranking through global scratch.
// Output per spectrum: retained peaks as (float)mz ascending + rank, stored at the input offsets.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t pa_inten_key(double x) {
    uint64_t b = (uint64_t)__double_as_longlong(x);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

struct PaBinArgs {
    const int64_t* spec_off;
    const double* mz;
    const double* inten;     // intensities as float64 (the reference's dtype), or
    const float* inten32;    //   as float32 when the caller holds them in that precision (F32 instantiation)
    const float* mz32;       // optional (then mz is not read): m/z narrowed to float32 by the host for the spectra it proved
    const int32_t* esc_off;  //   safe (same bounds, same bin of every peak); per spectrum the offset of its exact float64
    const double* mz_esc;    //   copy in mz_esc, or -1
    int64_t peak_base;       // spec_off values are relative to this
    int64_t n_spec;
    float2* rpk;             // retained peaks {(float)mz, rank as int bits}, m/z ascending, at the input offsets
    float* rmz;              // probe outputs (null on the scoring path): the same as separate arrays
    uint8_t* rrank;
    int32_t* rcount;
    uint8_t* ctab;           // per spectrum PA_NCELL bytes (m/z cell index of the retained peaks)
    float2* chead;           // per spectrum {cell base, 1 / cell width}
    int32_t* g_bin;          // scratch, one per peak
    uint8_t* g_tmp;          // scratch, one per peak
    int32_t* rindex;         // probe outputs (null on the scoring path): index of each retained peak in
    int32_t* rbin;           //   its spectrum, its bin, and per spectrum {min_mz, max_mz, n_bins}
    float* bounds;
    float bin_size;
    int n_top;
    int cap;                 // peaks per warp slot in shared memory
    int32_t* list;           // k_bin_rows: the spectra it declines go here (count in *list_n); k_bin_topn: when non-null,
    unsigned int* list_n;    //   the spectra to process (those k_bin_rows declined) instead of 0..n_spec-1
};

#define PA_NBIN_SMEM 128     // bins whose [start,end) ranges are tabulated in shared memory

// Shared memory per warp slot (cap = peaks per slot, a multiple of 32 and >= PA_BIN_MINCAP):
//   [0, 16 cap)   staging: mz f64[cap] | intensity f64[cap]; the binning pass compacts it in place to
//                 mzf f32[cap] at 0 and ranking keys (float)intensity f32[cap] at 8 cap (entry i lands in
//                 the staging slot of entry i/2, which the pass has already consumed), after which
//                 tie masks u32[128] sit at 4 cap and ranks u8[cap] at 4 cap + 512
//   bin u8[cap] | bstart u16[128] | bend u16[128] | cell u8[256]
#define PA_BIN_MINCAP 192
#ifndef PA_K1_UNROLL
#define PA_K1_UNROLL 2       // interior groups of the rank walk per trip (bins hold ~5 groups: deeper unrolling only adds remainders)
#endif
#define PA_BIN_SLOT_BYTES(cap) ((size_t)(cap) * 17 + PA_NBIN_SMEM * 4 + PA_NCELL)

__device__ __forceinline__ uint32_t pa_inten_key32(float x) {
    const uint32_t b = (uint32_t)__float_as_int(x);
    return (b >> 31) ? ~b : (b | 0x80000000u);
}

__device__ __forceinline__ void pa_cp_async4(void* smem_dst, const void* gsrc) {
    unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(d), "l"(gsrc) : "memory");
}

// F32: intensities arrive as float32 (4 instead of 8 bytes per peak over the host link and out of HBM).  A float is
// its own ranking key and (double)float is exact and monotone, so the ranks are those the reference computes on the
// same values handed to it as float64.
template <bool F32>
__global__ void __launch_bounds__(256) k_bin_topn(PaBinArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const int cap = a.cap;
    unsigned char* slot = smem_raw + (size_t)wib * PA_BIN_SLOT_BYTES(cap);
    double* s_mz = (double*)slot;                                    // staging
    uint64_t* s_key = (uint64_t*)(slot + (size_t)cap * 8);           // staging (intensity bits)
    float* s_mzf = (float*)slot;                                     // compacted (float)m/z, later the retained m/z
    uint32_t* s_bmask = (uint32_t*)(slot + (size_t)cap * 4);         // per bin: ranks taken (bit r), bit 31 = tie seen
    uint8_t* s_cnt = slot + (size_t)cap * 4 + PA_NBIN_SMEM * 4;      // rank of each peak inside its bin (255 = dropped)
    float* s_hi = (float*)(slot + (size_t)cap * 8);                  // (float)intensity: the ranking key
    uint8_t* s_bin = slot + (size_t)cap * 16;
    uint16_t* s_bstart = (uint16_t*)(slot + (size_t)cap * 17);
    uint16_t* s_bend = s_bstart + PA_NBIN_SMEM;
    uint8_t* s_cell = (uint8_t*)(s_bend + PA_NBIN_SMEM);
    const int64_t gw = (int64_t)blockIdx.x * wpb + wib, nw = (int64_t)gridDim.x * wpb;
    const int n_top = a.n_top;
    const double INF = __longlong_as_double(0x7ff0000000000000ll);

    const int64_t n_items = a.list ? (int64_t)*a.list_n : a.n_spec;
    for (int64_t item = gw; item < n_items; item += nw) {
        const int64_t s = a.list ? (int64_t)a.list[item] : item;
        const int64_t off = a.spec_off[s] - a.peak_base;
        const int P = (int)(a.spec_off[s + 1] - a.spec_off[s]);
        if (P <= 0) { if (lane == 0) { a.rcount[s] = 0; a.chead[s] = make_float2(0.f, 0.f); } continue; }
        const bool fits = P <= cap;
        double mn, mx;
        // m/z of peak i: float64 as given; or, when the host narrowed the batch (pa_narrow_mz), the float32 value widened
        // again -- proven on the host to give the same bounds and bins -- unless this spectrum kept an exact copy
        const double* em = a.mz;
        if (a.mz32 != nullptr) em = (a.esc_off[s] >= 0) ? a.mz_esc + a.esc_off[s] - off : nullptr;
        auto MZ = [&](int i) -> double { return em ? em[off + i] : (double)a.mz32[off + i]; };
        if (fits) {
            // stage the whole spectrum with asynchronous 8-byte copies: every load of the warp is
            // in flight at once (the arrays are only 8-byte aligned at a CSR offset)
            for (int i = lane; i < P; i += 32) {
                if (em) pa_cp_async8(&s_mz[i], em + off + i);
                else s_mz[i] = (double)a.mz32[off + i];
                if (F32) pa_cp_async4(&s_hi[i], a.inten32 + off + i);      // (lands where the ranking key of peak i will live)
                else pa_cp_async8(&s_key[i], a.inten + off + i);
            }
            asm volatile("cp.async.commit_group;\n" ::: "memory");
            asm volatile("cp.async.wait_group 0;\n" ::: "memory");
            __syncwarp();
            // optimistic: an m/z-sorted spectrum has its extremes at the ends (verified below)
            mn = s_mz[0]; mx = s_mz[P - 1];
        }
        float min_mz = 0.f, max_mz = 0.f;
        long long n_bins = 1;
        double dmin = 0., dbs = (double)a.bin_size;
        auto bounds = [&]() {
            // cpp/Spectra.cpp:46-48: the 100 is a literal there, independent of bin_size
            min_mz = __double2float_rn(__dmul_rn(floor(__ddiv_rn(mn, 100.)), 100.));
            max_mz = __double2float_rn(__dmul_rn(ceil(__ddiv_rn(mx, 100.)), 100.));
            n_bins = (long long)ceilf(__fdiv_rn(__fsub_rn(max_mz, min_mz), a.bin_size));
            if (n_bins < 1) n_bins = 1;     // degenerate spectrum: undefined in the reference
            dmin = (double)min_mz;
        };
        bool fast = false;
        if (fits) {
            bounds();
            fast = n_bins <= PA_NBIN_SMEM;
        }
        // The binning and output passes give every lane two neighbouring peaks (i0 = base + 2 lane,
        // i1 = i0 + 1): one 16-byte shared-memory access serves both and the per-round overhead is halved.
        if (fast) {
            // bins, float m/z and ranking keys; a sorted spectrum makes every bin one contiguous
            // run [bstart, bend).  Sortedness is checked on what the fast path relies on:
            // non-decreasing bins and non-decreasing (float)m/z.
            bool sorted = true;
            const double inv_bs = __ddiv_rn(1.0, dbs);
            int carry_bin = -1;
            float carry_mz = -INFINITY;
            auto bin_of = [&](double m) {
                const double x = __dsub_rn(m, dmin);
                // floor(x / bin_size) as the reference computes it; the reciprocal product decides
                // unless it lands within 1e-9 of an integer, where the IEEE quotient is taken
                double t = __dmul_rn(x, inv_bs);
                double q = floor(t);
                const double fr = __dsub_rn(t, q);
                if (!(fr > 1e-9 && fr < 1. - 1e-9)) q = floor(__ddiv_rn(x, dbs));
                long long b64 = (long long)q;
                if (b64 > n_bins - 1) b64 = n_bins - 1;
                if (b64 < 0) b64 = 0;               // only reachable for unsorted input (general path follows)
                return (int)b64;
            };
            for (int base = 0; base < P; base += 64) {
                const int i0 = base + 2 * lane, i1 = i0 + 1;
                const bool v0 = i0 < P, v1 = i1 < P;
                int bq0 = 0x7fffffff, bq1 = 0x7fffffff;
                float mz0 = INFINITY, mz1 = INFINITY, k0 = 0.f, k1 = 0.f;
                if (v0) {
                    // (the second element of the pair may lie past the spectrum: still inside the slot)
                    const double2 m2 = *(const double2*)&s_mz[i0];
                    double2 t2 = make_double2(0., 0.);
                    float2 t2f = make_float2(0.f, 0.f);
                    if (F32) t2f = *(const float2*)&s_hi[i0]; else t2 = *(const double2*)&s_key[i0];
                    if (m2.x < mn || m2.x > mx) sorted = false;      // the ends must be the true extremes
                    bq0 = bin_of(m2.x);
                    mz0 = __double2float_rn(m2.x);
                    // ranking key: the intensity rounded to float.  The rounding is monotone, so two peaks
                    // with different keys are ordered as their doubles are, and peaks of one bin that
                    // share a key (ties, +-0, NaN) are caught below and ranked on the doubles instead
                    k0 = F32 ? t2f.x : __double2float_rn(t2.x);
                    if (v1) {
                        if (m2.y < mn || m2.y > mx) sorted = false;
                        bq1 = bin_of(m2.y);
                        mz1 = __double2float_rn(m2.y);
                        k1 = F32 ? t2f.y : __double2float_rn(t2.y);
                        if (bq1 < bq0 || mz1 < mz0) sorted = false;
                    }
                }
                __syncwarp();                       // every lane has read its staging slots
                if (v0) {
                    *(float2*)&s_mzf[i0] = make_float2(mz0, mz1);
                    *(float2*)&s_hi[i0] = make_float2(k0, k1);
                    *(uchar2*)&s_bin[i0] = make_uchar2((unsigned char)bq0, (unsigned char)bq1);
                }
                // bin and m/z of the preceding peak: the last valid peak of the lane below
                int bprev = __shfl_up_sync(PA_FULL, v1 ? bq1 : bq0, 1);
                float mprev = __shfl_up_sync(PA_FULL, v1 ? mz1 : mz0, 1);
                if (lane == 0) { bprev = carry_bin; mprev = carry_mz; }
                if (v0) {
                    if (bq0 < bprev || mz0 < mprev) sorted = false;
                    if (bq0 != bprev) { s_bstart[bq0] = (uint16_t)i0; if (i0 > 0 && bprev >= 0 && bprev < PA_NBIN_SMEM) s_bend[bprev] = (uint16_t)i0; }
                    if (v1 && bq1 != bq0) { s_bstart[bq1] = (uint16_t)i1; s_bend[bq0] = (uint16_t)i1; }
                    if (i0 == P - 1) s_bend[bq0] = (uint16_t)P;
                    if (i1 == P - 1) s_bend[bq1] = (uint16_t)P;
                }
                carry_bin = __shfl_sync(PA_FULL, bq1, 31);
                carry_mz = __shfl_sync(PA_FULL, mz1, 31);
            }
            fast = __all_sync(PA_FULL, sorted);
            __syncwarp();
        }

        if (fast) {
            // exact rank of peak i inside [b0, b1) from the full 64-bit intensity keys (read back from
            // global memory: only needed when two peaks of a bin share a float key, or n_top > 31);
            // an equal intensity wins only from an earlier index
            auto exact_rank = [&](int i, int b0, int b1) {
                const uint64_t ki = F32 ? (uint64_t)pa_inten_key32(a.inten32[off + i]) : pa_inten_key(a.inten[off + i]);
                int c = 0;
                for (int j = b0; j < b1; j++) {
                    const uint64_t kj = F32 ? (uint64_t)pa_inten_key32(a.inten32[off + j]) : pa_inten_key(a.inten[off + j]);
                    c += (kj > ki) || (kj == ki && j < i);
                }
                return c;
            };
            const bool exact_all = n_top > 31;
            ((uint4*)s_bmask)[lane] = make_uint4(0u, 0u, 0u, 0u);
            __syncwarp();
            // rank = peaks of the same bin that beat this one, counted on the float keys, four per
            // shared-memory load; the first and last group of a bin are masked to [b0, b1).
            // Two peaks of a bin with the same key get the same count: every kept peak marks its
            // count in the bin's mask, and a mark found already set flags the bin for exact ranking.
            const float4* h4 = (const float4*)s_hi;
            constexpr int kRankUnroll = PA_K1_UNROLL;
            const float NINF = __int_as_float(0xff800000);
            auto mark = [&](int bq, int cnt) {
                if (cnt < n_top) {
                    const uint32_t bit = 1u << cnt;
                    if (atomicOr(&s_bmask[bq], bit) & bit) atomicOr(&s_bmask[bq], 0x80000000u);
                }
            };
            // (one peak per lane here: the lanes of a round walk their bins in lock step, so a second
            // peak per lane would only double the work of every trip)
            for (int base = 0; base < P; base += 32) {
                const int i = base + lane;
                if (i < P) {
                    const int bq = s_bin[i];
                    const int b0 = s_bstart[bq], b1 = s_bend[bq];
                    int cnt;
                    if (exact_all) cnt = exact_rank(i, b0, b1);
                    else {
                        const float hi = s_hi[i];
                        const unsigned n = (unsigned)(b1 - b0);
                        const int g0 = b0 >> 2, gl = (b1 - 1) >> 2;
                        float4 v = h4[g0];
                        int r = (g0 << 2) - b0;
                        v.x = (unsigned)r < n ? v.x : NINF; v.y = (unsigned)(r + 1) < n ? v.y : NINF;
                        v.z = (unsigned)(r + 2) < n ? v.z : NINF; v.w = (unsigned)(r + 3) < n ? v.w : NINF;
                        // one compare-to-1.0f and one add per peak; the sums are small integers, exact in float
                        float c = (v.x > hi ? 1.f : 0.f) + (v.y > hi ? 1.f : 0.f) + (v.z > hi ? 1.f : 0.f) + (v.w > hi ? 1.f : 0.f);
#pragma unroll kRankUnroll
                        for (int g = g0 + 1; g < gl; g++) {
                            v = h4[g];
                            c += (v.x > hi ? 1.f : 0.f) + (v.y > hi ? 1.f : 0.f) + (v.z > hi ? 1.f : 0.f) + (v.w > hi ? 1.f : 0.f);
                        }
                        if (gl > g0) {
                            v = h4[gl];
                            r = (gl << 2) - b0;
                            v.x = (unsigned)r < n ? v.x : NINF; v.y = (unsigned)(r + 1) < n ? v.y : NINF;
                            v.z = (unsigned)(r + 2) < n ? v.z : NINF; v.w = (unsigned)(r + 3) < n ? v.w : NINF;
                            c += (v.x > hi ? 1.f : 0.f) + (v.y > hi ? 1.f : 0.f) + (v.z > hi ? 1.f : 0.f) + (v.w > hi ? 1.f : 0.f);
                        }
                        cnt = (int)c;
                        mark(bq, cnt);
                    }
                    s_cnt[i] = (uint8_t)(cnt < n_top ? cnt : 255);
                }
            }
            __syncwarp();
            int out = 0;
            for (int base = 0; base < P; base += 64) {
                const int i0 = base + 2 * lane, i1 = i0 + 1;
                int cnt0 = 255, cnt1 = 255, bq0 = 0, bq1 = 0;
                float mz0 = 0.f, mz1 = 0.f;
                if (i0 < P) {
                    const float2 mm = *(const float2*)&s_mzf[i0];
                    const uchar2 bb = *(const uchar2*)&s_bin[i0];
                    const uchar2 cc = *(const uchar2*)&s_cnt[i0];
                    mz0 = mm.x; mz1 = mm.y; bq0 = bb.x; bq1 = bb.y; cnt0 = cc.x;
                    if (!exact_all && (s_bmask[bq0] >> 31)) cnt0 = exact_rank(i0, s_bstart[bq0], s_bend[bq0]);
                    if (i1 < P) {
                        cnt1 = cc.y;
                        if (!exact_all && (s_bmask[bq1] >> 31)) cnt1 = exact_rank(i1, s_bstart[bq1], s_bend[bq1]);
                    }
                }
                const bool keep0 = cnt0 < n_top, keep1 = cnt1 < n_top;
                const unsigned bal0 = __ballot_sync(PA_FULL, keep0), bal1 = __ballot_sync(PA_FULL, keep1);
                const unsigned below = (1u << lane) - 1u;       // every lane has read its own entries by now
                int pos = out + __popc(bal0 & below) + __popc(bal1 & below);
                if (keep0) {
                    a.rpk[off + pos] = make_float2(mz0, __int_as_float(cnt0));
                    if (a.rmz) { a.rmz[off + pos] = mz0; a.rrank[off + pos] = (uint8_t)cnt0; }
                    if (a.rindex) { a.rindex[off + pos] = i0; a.rbin[off + pos] = bq0; }
                    s_mzf[pos] = mz0;               // pos <= i0: only entries this or earlier rounds own
                    pos++;
                }
                if (keep1) {
                    a.rpk[off + pos] = make_float2(mz1, __int_as_float(cnt1));
                    if (a.rmz) { a.rmz[off + pos] = mz1; a.rrank[off + pos] = (uint8_t)cnt1; }
                    if (a.rindex) { a.rindex[off + pos] = i1; a.rbin[off + pos] = bq1; }
                    s_mzf[pos] = mz1;
                }
                out += __popc(bal0) + __popc(bal1);
                __syncwarp();
            }
            const float* s_out = s_mzf;
            if (lane == 0) {
                a.rcount[s] = out;
                if (a.bounds) { a.bounds[3 * s] = min_mz; a.bounds[3 * s + 1] = max_mz; a.bounds[3 * s + 2] = (float)n_bins; }
            }
            // m/z cell index over the retained peaks (consumers: pa_match_rank)
            if (out <= PA_RCAP && out > 0) {
                __syncwarp();
                const float cbase = s_out[0];
                const float cinv = pa_cell_inv(cbase, s_out[out - 1]);
                // cell[c] = first retained peak whose cell is >= c.  Mark the first peak of every
                // occupied cell (empty = `out`), then take the suffix minimum over the 256 cells:
                // 8 cells per lane locally, a shuffle scan across lanes.
                ((unsigned long long*)s_cell)[lane] = 0x0101010101010101ull * (unsigned long long)out;
                __syncwarp();
                for (int j = lane; j < out; j += 32) {
                    const int cj = pa_cell(s_out[j], cbase, cinv);
                    const int cp = j > 0 ? pa_cell(s_out[j - 1], cbase, cinv) : -1;
                    if (cj != cp) s_cell[cj] = (uint8_t)j;
                }
                __syncwarp();
                unsigned long long v = ((const unsigned long long*)s_cell)[lane];
                unsigned bb[8];
#pragma unroll
                for (int t = 0; t < 8; t++) bb[t] = (unsigned)(v >> (8 * t)) & 0xffu;
#pragma unroll
                for (int t = 6; t >= 0; t--) bb[t] = min(bb[t], bb[t + 1]);
                unsigned x = bb[0];                      // suffix minimum over this and the higher lanes
                for (int o = 1; o < 32; o <<= 1) {
                    const unsigned y = __shfl_down_sync(PA_FULL, x, o);
                    if (lane + o < 32) x = min(x, y);
                }
                unsigned carry = __shfl_down_sync(PA_FULL, x, 1);
                if (lane == 31) carry = (unsigned)out;
                v = 0;
#pragma unroll
                for (int t = 0; t < 8; t++) v |= (unsigned long long)min(bb[t], carry) << (8 * t);
                ((unsigned long long*)(a.ctab + (size_t)s * PA_NCELL))[lane] = v;
                if (lane == 0) a.chead[s] = make_float2(cbase, cinv);
            } else if (lane == 0) a.chead[s] = make_float2(0.f, 0.f);
        } else {
            // general path through global scratch (unsorted or oversized spectra)
            mn = INF; mx = -INF;
            for (int i = lane; i < P; i += 32) {
                const double m = MZ(i);
                mn = m < mn ? m : mn;
                mx = m > mx ? m : mx;
            }
            for (int o = 16; o > 0; o >>= 1) {
                double t = __shfl_xor_sync(PA_FULL, mn, o); mn = t < mn ? t : mn;
                t = __shfl_xor_sync(PA_FULL, mx, o); mx = t > mx ? t : mx;
            }
            bounds();
            for (int i = lane; i < P; i += 32) {
                double q = floor(__ddiv_rn(__dsub_rn(MZ(i), dmin), dbs));
                long long bq = (long long)q;
                if (bq > n_bins - 1) bq = n_bins - 1;
                a.g_bin[off + i] = (int32_t)bq;
            }
            __syncwarp();
            for (int i = lane; i < P; i += 32) {
                const int bq = a.g_bin[off + i];
                const uint64_t ki = F32 ? (uint64_t)pa_inten_key32(a.inten32[off + i]) : pa_inten_key(a.inten[off + i]);
                int cnt = 0;
                for (int j = 0; j < P && cnt < n_top; j++) {
                    if (a.g_bin[off + j] != bq || j == i) continue;
                    uint64_t kj = F32 ? (uint64_t)pa_inten_key32(a.inten32[off + j]) : pa_inten_key(a.inten[off + j]);
                    cnt += (kj > ki) || (kj == ki && j < i);
                }
                a.g_tmp[off + i] = (uint8_t)(cnt < n_top ? cnt : 255);
            }
            __syncwarp();
            int total = 0;
            for (int base = 0; base < P; base += 32) {
                int i = base + lane;
                bool keep = (i < P) && a.g_tmp[off + i] != 255;
                if (keep) {
                    const float fi = __double2float_rn(MZ(i));
                    int pos = 0;
                    for (int j = 0; j < P; j++) {
                        if (a.g_tmp[off + j] == 255 || j == i) continue;
                        float fj = __double2float_rn(MZ(j));
                        pos += (fj < fi) || (fj == fi && j < i);
                    }
                    a.rpk[off + pos] = make_float2(fi, __int_as_float((int)a.g_tmp[off + i]));
                    if (a.rmz) { a.rmz[off + pos] = fi; a.rrank[off + pos] = a.g_tmp[off + i]; }
                    if (a.rindex) { a.rindex[off + pos] = i; a.rbin[off + pos] = a.g_bin[off + i]; }
                }
                total += __popc(__ballot_sync(PA_FULL, keep));
            }
            if (lane == 0) {
                a.rcount[s] = total; a.chead[s] = make_float2(0.f, 0.f);
                if (a.bounds) { a.bounds[3 * s] = min_mz; a.bounds[3 * s + 1] = max_mz; a.bounds[3 * s + 2] = (float)n_bins; }
            }
        }
        __syncwarp();
    }
}

#include "pa_bin_rows.cuh"

__global__ void k_max_peaks(const int64_t* spec_off, int64_t n_spec, int* out) {
    int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int v = 0;
    if (q < n_spec) { int64_t d = spec_off[q + 1] - spec_off[q]; v = d > (1 << 20) ? (1 << 20) : (int)d; }
    for (int o = 16; o > 0; o >>= 1) { int t = __shfl_xor_sync(PA_FULL, v, o); v = t > v ? t : v; }
    if ((threadIdx.x & 31) == 0 && v > 0) atomicMax(out, v);
}

// ---------------------------------------------------------------------------------------------
// P1: per-PSM planning (validation, sites, isoform count, K2 work units)
// ---------------------------------------------------------------------------------------------
struct PaPlanOut {
    int32_t* psm_S;
    int32_t* psm_status;
    int64_t* psm_I;          // [n_psm+1], last = 0 (input of the exclusive scan)
    int32_t* psm_units;      // [n_psm+1], last = 0
    unsigned long long* combo_bits;  // [64]: bit k of row S set when (S,k) occurs with > 1 isoform
    int* max_frag;           // max fragments per isoform (all types/charges) over the chunk
    int* max_list;           // max fragments per (isoform, type) over the chunk (K3 list size)
    int* max_len;            // longest scored peptide of the chunk
};

// Status k_plan gives a PSM of a typed batch (pa_score_typed) that belongs to another type than the pass's: no
// isoforms, no units, and k_select_thread<true> writes none of its results.  It never reaches the caller.
#define PA_PSM_OTHER_TYPE 0x100

// psm_type (typed batches, chunk-relative; null: every PSM is of the pass's type): PSMs of another type get
// PA_PSM_OTHER_TYPE; the pass of type 0 reports a type >= n_types as PA_PSM_BAD_INDEX.
__global__ void __launch_bounds__(256) k_plan(PaCfg cfg, PaBatchDev b, int64_t n_psm, PaPlanOut o,
                                              const uint8_t* psm_type, int type, int n_types) {
    // chunk-wide maxima and the (S,k) combinations seen are collected per block in shared memory and
    // flushed once: a global atomic per PSM and field would queue up on four addresses
    __shared__ unsigned long long s_combo[64];
    __shared__ int s_max[3];
    if (threadIdx.x < 64) s_combo[threadIdx.x] = 0ull;
    if (threadIdx.x < 3) s_max[threadIdx.x] = 0;
    __syncthreads();
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n_psm) {
        const int off = b.pep_off[p];
        const int L = b.pep_off[p + 1] - off;
        const int k = b.n_mod[p], Z = b.max_charge[p];
        const int sp = b.psm_spec[p];
        int status = PA_PSM_OK, S = 0;
        const int t = psm_type != nullptr ? (int)psm_type[p] : type;
        if (t != type) status = (type == 0 && t >= n_types) ? PA_PSM_BAD_INDEX : PA_PSM_OTHER_TYPE;
        else if (sp < 0 || sp >= b.n_spec || k < 0 || Z < 1 || L < 1) status = PA_PSM_BAD_INDEX;  // Z == 0 crashes the reference
        else if (L > PA_MAX_PEPTIDE) status = PA_PSM_TOO_LONG;
        else {
            for (int i = 0; i < L; i++) {
                const int c = (int)b.pep[off + i] - 'A';
                if (c < 0 || c >= 26 || !((cfg.known_letters >> c) & 1u)) { status = PA_PSM_BAD_RESIDUE; break; }
                const bool site = ((cfg.mod_letters >> c) & 1u) || (cfg.allow_n && i == 0) || (cfg.allow_c && i == L - 1);
                S += site;
            }
            if (status == PA_PSM_OK && b.aux_off != nullptr)
                for (int a = b.aux_off[p]; a < b.aux_off[p + 1]; a++)
                    if (b.aux_pos[a] > (uint32_t)L) status = PA_PSM_BAD_AUX;
            if (status == PA_PSM_OK && S > PA_MAX_SITES) status = PA_PSM_TOO_MANY_SITES;
            if (status == PA_PSM_OK && b.rcount[sp] <= 0) status = PA_PSM_EMPTY_SPECTRUM;
        }
        int64_t I = 0;
        if (status == PA_PSM_OK) {
            // Upper bound of the fragments one isoform emits (all ion types, charges, neutral-loss variants).
            // Without neutral losses it is exact.  With them, every residue is taken to push every loss it could
            // carry in either state: the variant count only grows with the stack, so walking this superset bounds
            // every real isoform (tighter than "worst state at every step", which rejected long high-charge peptides).
            const int steps = L > 1 ? L - 1 : 1;
            long long nf = (long long)steps * Z * cfg.n_types;
            if (cfg.has_nl) {
                long long tot[2] = {0, 0};
                for (int dir = 0; dir < 2; dir++) {
                    int st = 0;
                    for (int step = 0; step < steps; step++) {
                        const int c = (int)b.pep[off + (dir ? L - 1 - step : step)] - 'A';
                        if (cfg.nl_upper[c]) st = pa_nl_bump(st, cfg.nl_upper[c]);
                        if (cfg.nl_lower[c]) st = pa_nl_bump(st, cfg.nl_lower[c]);
                        tot[dir] += cfg.nl_nvar[st];
                    }
                }
                nf = 0;
                for (int t = 0; t < cfg.n_types; t++) nf += tot[(cfg.types[t] == 'b' || cfg.types[t] == 'c') ? 0 : 1] * Z;
            }
            if (nf > PA_MAX_FRAGMENTS) status = PA_PSM_TOO_MANY_FRAGMENTS;
            else {
                uint32_t c = (k <= S) ? cfg.binom[S * 64 + k] : 0u;
                if ((long long)c > PA_MAX_ISOFORMS) status = PA_PSM_TOO_MANY_ISOFORMS;
                else {
                    I = c;
                    atomicMax(&s_max[0], (int)nf);
                    atomicMax(&s_max[1], steps * cfg.nvar_cap * Z);      // the list kernels size their arenas by this looser bound
                    atomicMax(&s_max[2], L);
                    if (I > 1) atomicOr(&s_combo[S], 1ull << k);
                }
            }
        }
        o.psm_S[p] = S;
        o.psm_status[p] = status;
        o.psm_I[p] = I;
        o.psm_units[p] = (int32_t)((I + PA_UNIT - 1) / PA_UNIT);
    }
    __syncthreads();
    if (threadIdx.x < 64 && s_combo[threadIdx.x]) atomicOr(&o.combo_bits[threadIdx.x], s_combo[threadIdx.x]);
    if (threadIdx.x == 64 && s_max[0] > 0) atomicMax(o.max_frag, s_max[0]);
    if (threadIdx.x == 65 && s_max[1] > 0) atomicMax(o.max_list, s_max[1]);
    if (threadIdx.x == 66 && s_max[2] > 0) atomicMax(o.max_len, s_max[2]);
}

__global__ void k_expand_units(int64_t n_psm, const int32_t* unit_off, int32_t* unit_psm) {
    int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_psm) return;
    for (int u = unit_off[p]; u < unit_off[p + 1]; u++) unit_psm[u] = (int32_t)p;
}

// ---------------------------------------------------------------------------------------------
// K2: per-isoform fragment generation, peak matching, per-depth counts and PepScore.
// cpp/ModifiedPeptide.cpp:379-408, :500-524, :570-591 (fragments), :126-150 (matching),
// cpp/Ascore.cpp:53-121 (counts), :123-139 (scores).  One lane owns one isoform at a time and
// performs the reference's sequential float32 running sum for it, so every fragment m/z has the
// reference's bits.
// ---------------------------------------------------------------------------------------------
struct PaIso {                 // per-isoform records of a chunk (SoA), indexed iso_off[p] + idx
    unsigned long long* lo;    // cumulative counts depth 0..4, 12 bits each
    unsigned long long* hi;    // cumulative counts depth 5..9
    uint32_t* nfrag;           // total_fragments
    float* w;                  // weighted PepScore
};

struct PaCountArgs {
    int64_t n_units;
    const int32_t* unit_psm;
    const int32_t* unit_off;
    const int64_t* iso_off;
    const int32_t* psm_S;
    const int32_t* psm_status;
    PaIso iso;
    unsigned long long* n_lookups;   // counter
    unsigned long long* next_unit;   // work cursor (zeroed before the launch): warps take `grab` units at a time
    int grab;                        // 1 .. PA_K2_GRAB units per grab; negative: do not reserve the next grab ahead
};

#ifndef PA_K2_MINBLOCKS
#define PA_K2_MINBLOCKS 4
#endif
#ifndef PA_K2_UNROLL
#define PA_K2_UNROLL 1
#endif
#ifndef PA_K2_GRAB
#define PA_K2_GRAB 4
#endif
// One fragment position: every neutral-loss variant and charge of running sum `run`, matched
// against the staged peaks; hands the rank of each fragment's match (255: none) to `hit` and
// returns the number of fragments emitted.
template <bool HAS_NL, bool EGH, class Hit>
__device__ __forceinline__ int pa_emit_ranks(const PaCfg& cfg, const PsmInfo& info, const float* s_nl, float run,
                                             int nls, double a1, double a2, double zm1, double zm2, Hit& hit) {
    const int Z = info.Z;
    int nv = 1;
    if (HAS_NL) nv = ((const uint8_t*)(s_nl + 256 * 16))[nls];       // variant counts sit behind the sums in shared memory
    // L == 1: the walk starts on the last residue and the reference's end test lets all but
    // the last neutral-loss variant through (cpp/ModifiedPeptide.cpp:516-524)
    if (info.L == 1) nv -= 1;
    for (int v = 0; v < nv; v++) {
        float base = run;
        if (HAS_NL) base = __fsub_rn(run, s_nl[nls * 16 + v]);
        const double d = __dsub_rn(__dadd_rn((double)base, a1), a2);
        // charge z: (d + z * 1.007825) / z  (cpp/ModifiedPeptide.cpp:585-587); 1 and 2 are unrolled
        hit(pa_match_rank<EGH>(info, __double2float_rn(__dadd_rn(d, zm1)), cfg.err, cfg.err_gt_half));
        if (Z >= 2) hit(pa_match_rank<EGH>(info, __double2float_rn(__dmul_rn(__dadd_rn(d, zm2), 0.5)), cfg.err, cfg.err_gt_half));
        for (int z = 3; z <= Z; z++) hit(pa_match_rank<EGH>(info, pa_charge_mz(d, z), cfg.err, cfg.err_gt_half));
    }
    return nv * Z;
}

// Walk ion type `type` of the isoform with residue mask (mlo,mhi) from step `f` on, where the
// float32 running sum / neutral-loss state before step f are (run, nls): the reference's
// sequential adds are replayed for steps [f, s0) and fragments are emitted and matched for
// steps [s0, s1), each match's rank handed to `hit`.  Returns the number of fragments emitted.
template <bool HAS_NL, bool EGH, class Hit>
__device__ __forceinline__ uint32_t pa_walk_ranks(const PaCfg& cfg, const PsmSmem* sm, const PsmInfo& info,
                                                  const float* s_nl, uint64_t mlo, uint64_t mhi, char type, int f,
                                                  float run, int nls, int s0, int s1, Hit& hit) {
    const int L = info.L;
    uint32_t nfrag = 0;
    const bool fwd = (type == 'b' || type == 'c');
    double a1, a2;
    pa_type_consts(type, a1, a2);
    const double zm1 = c_zmass[1], zm2 = c_zmass[2];
    // replay: the lanes of a split walk have different s0, but this loop is cheap; the matching
    // loop below then runs in lock step over all lanes of the warp
    for (int step = f; step < s0; step++) {
        const int i = fwd ? step : L - 1 - step;
        const int st = (int)(((i < 64) ? (mlo >> i) : (mhi >> (i - 64))) & 1ull);
        run = __fadd_rn(sm->res[i][st], run);          // r + 0.f == r: the first step needs no special case
        if (HAS_NL) {
            int idx = sm->nlidx[i][st];
            if (idx) nls = pa_nl_bump(nls, idx);
        }
    }
    constexpr int kUnroll = PA_K2_UNROLL;
#pragma unroll kUnroll
    for (int step = s0; step < s1; step++) {
        const int i = fwd ? step : L - 1 - step;
        const int st = (int)(((i < 64) ? (mlo >> i) : (mhi >> (i - 64))) & 1ull);
        run = __fadd_rn(sm->res[i][st], run);
        if (HAS_NL) {
            int idx = sm->nlidx[i][st];
            if (idx) nls = pa_nl_bump(nls, idx);
        }
        nfrag += pa_emit_ranks<HAS_NL, EGH>(cfg, info, s_nl, run, nls, a1, a2, zm1, zm2, hit);
    }
    return nfrag;
}

// The same with packed non-cumulative per-rank counts of depths 0..9 (`lut[r]`, lut[10] = 0 for "no match" and for
// the ranks >= 10).
template <bool HAS_NL, bool EGH>
__device__ __forceinline__ void pa_walk_isoform(const PaCfg& cfg, const PsmSmem* sm, const PsmInfo& info,
                                                const float* s_nl, uint64_t mlo, uint64_t mhi, char type, int f,
                                                float run, int nls, int s0, int s1, const ulonglong2* lut,
                                                unsigned long long& clo, unsigned long long& chi, uint32_t& nfrag) {
    clo = 0; chi = 0;
    auto add = [&](int rk) {
        const ulonglong2 inc = lut[rk < 10 ? rk : 10];
        clo += inc.x; chi += inc.y;
    };
    nfrag = pa_walk_ranks<HAS_NL, EGH>(cfg, sm, info, s_nl, mlo, mhi, type, f, run, nls, s0, s1, add);
}

// ---- the walk of the common case: staged peaks with a cell index, 2 <= L <= 64 ------------------------------
// Same arithmetic as pa_walk_isoform / pa_emit_ranks / pa_match_rank, fewer instructions per step: the residue states of
// the walk come off a 64-bit word one bit per step (reversed up front for the y-side walks) instead of a variable shift of
// a 128-bit mask, the residue table is followed by a running shared-memory address, the peaks need no "are they staged"
// test per lookup, and the increment table is read through a 32-bit shared address.
struct PaFastCtx {
    uint32_t res_a, nli_a, pk_a, cell_a, lut_a, nl_a;     // shared-window addresses: res[][2], nlidx[][2], pk[], cell[], lut[], s_nl
    float cbase, cinv, err;
    int Z, L;
};

__device__ __forceinline__ float pa_lds_f32(uint32_t a) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint32_t pa_lds_u8(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ float2 pa_lds_f32x2(uint32_t a) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ ulonglong2 pa_lds_u64x2(uint32_t a) {
    ulonglong2 v;
    asm volatile("ld.shared.v2.u64 {%0, %1}, [%2];" : "=l"(v.x), "=l"(v.y) : "r"(a));
    return v;
}

// rank of the best retained peak matching fragment f (pa_match_rank, staged form), added into the packed counters
template <bool EGH>
__device__ __forceinline__ void pa_fast_lookup(const PaFastCtx& c, float f, int egh_rt, unsigned long long& clo,
                                               unsigned long long& chi) {
    const bool err_gt_half = EGH && egh_rt;
    const float lo = __fsub_rn(f, c.err), hi = __fadd_rn(f, c.err);
    int best = 10;                                   // lut[10] = no increment
    uint32_t pa = c.pk_a + 8u * pa_lds_u8(c.cell_a + (uint32_t)pa_cell(lo, c.cbase, c.cinv));
    float2 e = pa_lds_f32x2(pa), e_next = pa_lds_f32x2(pa + 8);
    for (;;) {
        if (!(e.x < hi)) break;
        if (e.x > lo && !(err_gt_half && !((double)f >= (double)e.x - .5))) {
            const int r = __float_as_int(e.y);
            best = r < best ? r : best;
        }
        pa += 8;
        e = e_next;
        if (!(e.x < hi)) break;
        e_next = pa_lds_f32x2(pa + 8);
    }
    const ulonglong2 inc = pa_lds_u64x2(c.lut_a + 16u * (uint32_t)best);
    clo += inc.x; chi += inc.y;
}

template <bool HAS_NL, bool EGH>
__device__ __forceinline__ void pa_walk_fast(const PaCfg& cfg, const PaFastCtx& c0, uint64_t mlo, char type, int s0, int s1,
                                             unsigned long long& clo, unsigned long long& chi, uint32_t& nfrag) {
    PaFastCtx c = c0;
    // (see below: kept in registers instead of being rebuilt per lookup; measured to pay only in the neutral-loss form)
    if (HAS_NL) { asm volatile("" : "+r"(c.lut_a)); asm volatile("" : "+r"(c.nl_a)); }
    clo = 0; chi = 0; nfrag = 0;
    const bool fwd = (type == 'b' || type == 'c');
    double a1, a2;
    pa_type_consts(type, a1, a2);
    const double zm1 = c_zmass[1], zm2 = c_zmass[2];
    // bit t of `w` = state of the residue visited at step t
    uint64_t w = fwd ? mlo : (__brevll(mlo) >> (64 - c.L));
    uint32_t ra = fwd ? c.res_a : c.res_a + 8u * (uint32_t)(c.L - 1);
    uint32_t na = fwd ? c.nli_a : c.nli_a + 2u * (uint32_t)(c.L - 1);
    int dr = fwd ? 8 : -8, dn = fwd ? 2 : -2;
    // (values derived from the lane are otherwise recomputed at every trip under this register budget -- ~20 instructions
    // per step: an empty asm makes them opaque, so they stay in their registers)
    asm volatile("" : "+r"(dr));
    if (HAS_NL) asm volatile("" : "+r"(dn));
    float run = 0.f;
    int nls = 0;
    // replay of the running sum up to the lane's segment (the adds must stay sequential: the reference's rounding)
    // (both loops count down: a bound derived from the lane would be recomputed at every trip under this register budget)
    for (int n = s0; n > 0; n--) {
        const uint32_t st = (uint32_t)w & 1u;
        w >>= 1;
        run = __fadd_rn(pa_lds_f32(ra + 4u * st), run);
        if (HAS_NL) {
            const int idx = (int)pa_lds_u8(na + st);
            if (idx) nls = pa_nl_bump(nls, idx);
            na += dn;
        }
        ra += dr;
    }
    const int Z = c.Z;
    for (int n = s1 - s0; n > 0; n--) {
        const uint32_t st = (uint32_t)w & 1u;
        w >>= 1;
        run = __fadd_rn(pa_lds_f32(ra + 4u * st), run);
        ra += dr;
        int nv = 1;
        if (HAS_NL) {
            const int idx = (int)pa_lds_u8(na + st);
            if (idx) nls = pa_nl_bump(nls, idx);
            na += dn;
            nv = (int)pa_lds_u8(c.nl_a + 256 * 16 * 4 + (uint32_t)nls);
        }
        for (int v = 0; v < nv; v++) {
            float base = run;
            if (HAS_NL) base = __fsub_rn(run, pa_lds_f32(c.nl_a + 4u * (uint32_t)(nls * 16 + v)));
            const double d = __dsub_rn(__dadd_rn((double)base, a1), a2);
            // charge z: (d + z * 1.007825) / z  (cpp/ModifiedPeptide.cpp:585-587); 1 and 2 are unrolled
            pa_fast_lookup<EGH>(c, __double2float_rn(__dadd_rn(d, zm1)), cfg.err_gt_half, clo, chi);
            if (Z >= 2) pa_fast_lookup<EGH>(c, __double2float_rn(__dmul_rn(__dadd_rn(d, zm2), 0.5)), cfg.err_gt_half, clo, chi);
            for (int z = 3; z <= Z; z++) pa_fast_lookup<EGH>(c, pa_charge_mz(d, z), cfg.err_gt_half, clo, chi);
        }
        nfrag += (uint32_t)(nv * Z);
    }
}

// packed per-rank counts -> packed cumulative counts (cpp/Ascore.cpp:113-117)
__device__ __forceinline__ void pa_cumulate(unsigned long long& lo, unsigned long long& hi) {
    // prefix sums of 12-bit fields; totals stay < 4096 (PA_MAX_FRAGMENTS)
    lo += lo << 12; lo += lo << 24; lo += lo << 48;        // fields 0..4 (60 bits): inclusive scan
    unsigned long long top = (lo >> 48) & 0xfffull;        // cumulative count of ranks 0..4
    hi += hi << 12; hi += hi << 24; hi += hi << 48;
    hi += top * 0x001001001001001ull;
    lo &= 0x0fffffffffffffffull; hi &= 0x0fffffffffffffffull;
}

__device__ __forceinline__ int pa_cum_get(unsigned long long lo, unsigned long long hi, int d) {
    return (int)(((d < 5) ? (lo >> (12 * d)) : (hi >> (12 * (d - 5)))) & 0xfffull);
}

// cpp/Ascore.cpp:123-139
__device__ __forceinline__ float pa_weighted(const PaCfg& cfg, unsigned long long lo, unsigned long long hi, int n) {
    double acc = 0.;
#pragma unroll
    for (int d = 0; d < PA_N_TOP; d++) {
        float sc = __ldg(cfg.T + pa_tab_index(n, pa_cum_get(lo, hi, d), d));
        acc = __dadd_rn(acc, (double)__fmul_rn(cfg.weights[d], sc));
    }
    return __double2float_rn(acc);
}

__device__ __forceinline__ void pa_sites_to_mask(const PsmSmem* sm, uint64_t bits, uint64_t& mlo, uint64_t& mhi) {
    mlo = 0; mhi = 0;
    while (bits) {
        int j = __ffsll((long long)bits) - 1;
        bits &= bits - 1;
        int pos = sm->site_pos[j];
        if (pos < 64) mlo |= 1ull << pos; else mhi |= 1ull << (pos - 64);
    }
}

// Lane mapping inside a unit: isoform x ion type x segment.  PAIR (exactly two ion types, the
// default "by") gives each type of an isoform its own lane; when the unit has few isoforms each
// walk is further split into H segments of consecutive steps (a lane replays the cheap running sum
// up to its segment and matches only its own fragments), so that small PSMs still fill the warp.
// The lanes of one isoform are contiguous and add their packed counts with xor-shuffles.
template <bool HAS_NL, bool PAIR, bool EGH>
__global__ void __launch_bounds__(256, PA_K2_MINBLOCKS) k_count_score(PaCfg cfg, PaBatchDev b, PaCountArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ ulonglong2 s_lut[16];
    __shared__ float s_nl[HAS_NL ? 256 * 16 + 64 : 1];   // neutral-loss variant sums [256][16] + variant counts u8[256]
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    if (threadIdx.x < 16) {
        const int r = threadIdx.x;
        s_lut[r] = make_ulonglong2(r < 5 ? 1ull << (12 * r) : 0ull, (r >= 5 && r < 10) ? 1ull << (12 * (r - 5)) : 0ull);
    }
    if (HAS_NL) {
        for (int i = threadIdx.x; i < 256 * 16; i += blockDim.x) s_nl[i] = cfg.nl_sums[i];
        if (threadIdx.x < 256) ((uint8_t*)(s_nl + 256 * 16))[threadIdx.x] = cfg.nl_nvar[threadIdx.x];
    }
    __syncthreads();
    PsmSmem* sm = (PsmSmem*)smem_raw + wib;
    const int64_t gw = (int64_t)blockIdx.x * wpb + wib, nw = (int64_t)gridDim.x * wpb;
    int64_t cur = -1;
    PsmInfo info;
    PaFastCtx fc;
    bool fast = false;
    fc.res_a = (uint32_t)__cvta_generic_to_shared(&sm->res[0][0]);
    fc.nli_a = (uint32_t)__cvta_generic_to_shared(&sm->nlidx[0][0]);
    fc.pk_a = (uint32_t)__cvta_generic_to_shared(&sm->pk[0]);
    fc.cell_a = (uint32_t)__cvta_generic_to_shared(&sm->cell[0]);
    fc.lut_a = (uint32_t)__cvta_generic_to_shared(&s_lut[0]);
    fc.nl_a = (uint32_t)__cvta_generic_to_shared(&s_nl[0]);
    fc.err = cfg.err; fc.cbase = 0.f; fc.cinv = 0.f; fc.Z = 0; fc.L = 0;
    unsigned long long lookups = 0;
    const int T = PAIR ? 2 : 1;
    // Units differ in cost by two orders of magnitude (1 .. 1024 isoforms), so they are handed out
    // dynamically: a warp takes `grab` consecutive units from a global cursor and asks for its next
    // grab before it starts on the current one (the atomic's round trip hides behind the work).
    (void)gw; (void)nw;
    unsigned long long pend = 0;
    const int grab = a.grab < 0 ? -a.grab : a.grab;
    if (lane == 0) pend = atomicAdd(a.next_unit, (unsigned long long)grab);
    int64_t base = (int64_t)__shfl_sync(PA_FULL, pend, 0);
    // (with few units per warp -- grab < 0 -- the next grab is only taken when this one is done: a unit held
    // in reserve by a busy warp would wait while other warps sit idle)
    const bool ahead = a.grab > 0;
    while (base < a.n_units) {
      if (ahead && lane == 0) pend = atomicAdd(a.next_unit, (unsigned long long)grab);
      const int64_t u_end = base + grab < a.n_units ? base + grab : a.n_units;
      for (int64_t u = base; u < u_end; u++) {
        const int64_t p = a.unit_psm[u];
        const int64_t I = a.iso_off[p + 1] - a.iso_off[p];
        if (p != cur) {
            pa_setup_psm(cfg, b, p, sm, info, true);
            cur = p;
            // the common case takes the leaner walk (pa_walk_fast): peaks staged with their cell index, 2 <= L <= 64
            fast = info.cell != nullptr && info.L >= 2 && info.L <= 64;
            fc.cbase = info.cell_base; fc.cinv = info.cell_inv; fc.Z = info.Z; fc.L = info.L;
        }
        const int S = a.psm_S[p], k = info.k;
        const int64_t first = (int64_t)(u - a.unit_off[p]) * PA_UNIT;
        const int cnt = (int)((I - first < PA_UNIT) ? I - first : PA_UNIT);
        const int steps = (info.L == 1) ? 1 : info.L - 1;
        int hs = 0;                                  // log2 of the segments per walk
        while (hs < 3 && (cnt * T << (hs + 1)) <= 32 && (2 << hs) <= steps) hs++;
        const int H = 1 << hs, gs = hs + (PAIR ? 1 : 0), G = 1 << gs;      // G lanes per isoform
        const int items = cnt << gs;
        for (int q0 = 0; q0 < items; q0 += 32) {
            const int q = q0 + lane;
            const bool active = q < items;
            const uint32_t idx = (uint32_t)(first + (q >> gs));
            const int sub = q & (G - 1), h = sub & (H - 1);
            unsigned long long clo = 0, chi = 0; uint32_t nf = 0;
            if (active) {
                const uint64_t bits = pa_unrank(cfg.binom, S, k, idx);
                uint64_t mlo, mhi;
                pa_sites_to_mask(sm, bits, mlo, mhi);
                const int s0 = (steps * h) >> hs, s1 = (steps * (h + 1)) >> hs;
                if (fast) {
                    if (PAIR) {
                        pa_walk_fast<HAS_NL, EGH>(cfg, fc, mlo, cfg.types[sub >> hs], s0, s1, clo, chi, nf);
                    } else {
                        for (int t = 0; t < cfg.n_types; t++) {
                            unsigned long long xlo, xhi; uint32_t xn;
                            pa_walk_fast<HAS_NL, EGH>(cfg, fc, mlo, cfg.types[t], s0, s1, xlo, xhi, xn);
                            clo += xlo; chi += xhi; nf += xn;
                        }
                    }
                } else if (PAIR) {
                    pa_walk_isoform<HAS_NL, EGH>(cfg, sm, info, s_nl, mlo, mhi, cfg.types[sub >> hs], 0, 0.f, 0, s0, s1, s_lut, clo, chi, nf);
                } else {
                    for (int t = 0; t < cfg.n_types; t++) {
                        unsigned long long xlo, xhi; uint32_t xn;
                        pa_walk_isoform<HAS_NL, EGH>(cfg, sm, info, s_nl, mlo, mhi, cfg.types[t], 0, 0.f, 0, s0, s1, s_lut, xlo, xhi, xn);
                        clo += xlo; chi += xhi; nf += xn;
                    }
                }
                lookups += nf;
            }
            for (int o = 1; o < G; o <<= 1) {
                clo += __shfl_xor_sync(PA_FULL, clo, o);
                chi += __shfl_xor_sync(PA_FULL, chi, o);
                nf += __shfl_xor_sync(PA_FULL, nf, o);
            }
            if (active && sub == 0) {
                pa_cumulate(clo, chi);
                const int64_t g = a.iso_off[p] + idx;
                a.iso.lo[g] = clo; a.iso.hi[g] = chi; a.iso.nfrag[g] = nf;
                a.iso.w[g] = pa_weighted(cfg, clo, chi, (int)nf);
            }
        }
      }
      if (!ahead && lane == 0) pend = atomicAdd(a.next_unit, (unsigned long long)grab);
      base = (int64_t)__shfl_sync(PA_FULL, pend, 0);
    }
    for (int o = 16; o > 0; o >>= 1) lookups += __shfl_xor_sync(PA_FULL, lookups, o);
    if (lane == 0 && lookups) atomicAdd(a.n_lookups, lookups);
}

// ---------------------------------------------------------------------------------------------
// K2d (n_top > 10 only, after K2): cumulative counts of depths 10 .. n_top-1 for every isoform of the chunk,
// cnt_d = cnt_9 + sum of the ranks 10..d, with cnt_9 from K2.  One warp per K2 unit, one lane per isoform walking
// every ion type with the reference's arithmetic (pa_walk_ranks); the ranks >= 10 go to the lane's own histogram in
// shared memory.  K2 sees these ranks as "no match" (lut[10]), so its depth 0-9 counts and PepScores stand.
// ---------------------------------------------------------------------------------------------
struct PaDeepCountArgs {
    int64_t n_units;
    const int32_t* unit_psm;
    const int32_t* unit_off;
    const int64_t* iso_off;
    const int32_t* psm_S;
    const unsigned long long* iso_hi;   // K2's packed cumulative counts of depths 5..9
    uint16_t* cnt;                      // [total isoforms * nd]
    int nd;                             // n_top - 10
};

template <bool HAS_NL>
__global__ void __launch_bounds__(128) k_count_deep(PaCfg cfg, PaBatchDev b, PaDeepCountArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ float s_nl[HAS_NL ? 256 * 16 + 64 : 1];   // as in k_count_score
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    if (HAS_NL) {
        for (int i = threadIdx.x; i < 256 * 16; i += blockDim.x) s_nl[i] = cfg.nl_sums[i];
        for (int i = threadIdx.x; i < 256; i += blockDim.x) ((uint8_t*)(s_nl + 256 * 16))[i] = cfg.nl_nvar[i];
    }
    __syncthreads();
    const int nd = a.nd;
    PsmSmem* sm = (PsmSmem*)smem_raw + wib;
    uint16_t* hist = (uint16_t*)((PsmSmem*)smem_raw + wpb) + (size_t)(wib * 32 + lane) * nd;
    auto add = [&](int rk) { if (rk >= PA_N_TOP && rk < PA_N_TOP + nd) hist[rk - PA_N_TOP]++; };
    int64_t cur = -1;
    PsmInfo info;
    for (int64_t u = (int64_t)blockIdx.x * wpb + wib; u < a.n_units; u += (int64_t)gridDim.x * wpb) {
        const int64_t p = a.unit_psm[u];
        if (p != cur) { pa_setup_psm(cfg, b, p, sm, info, true); cur = p; }
        const int64_t I = a.iso_off[p + 1] - a.iso_off[p];
        const int S = a.psm_S[p];
        const int64_t first = (int64_t)(u - a.unit_off[p]) * PA_UNIT;
        const int cnt = (int)((I - first < PA_UNIT) ? I - first : PA_UNIT);
        const int steps = (info.L == 1) ? 1 : info.L - 1;
        for (int q = lane; q < cnt; q += 32) {
            for (int d = 0; d < nd; d++) hist[d] = 0;
            uint64_t mlo, mhi;
            pa_sites_to_mask(sm, pa_unrank(cfg.binom, S, info.k, (uint32_t)(first + q)), mlo, mhi);
            for (int t = 0; t < cfg.n_types; t++)
                pa_walk_ranks<HAS_NL, true>(cfg, sm, info, s_nl, mlo, mhi, cfg.types[t], 0, 0.f, 0, 0, steps, add);
            const int64_t g = a.iso_off[p] + first + q;
            int c = (int)((a.iso_hi[g] >> 48) & 0xfffull);       // cumulative count of depth 9
            for (int d = 0; d < nd; d++) { c += hist[d]; a.cnt[g * nd + d] = (uint16_t)c; }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// K3: best isoform in the reference's order, Ascores and alternative sites.
// cpp/Ascore.cpp:38-51 (unambiguous), :141-146 (std::sort), :212-254 (calculateAscores),
// :157-210 (calculateAmbiguity), cpp/ModifiedPeptide.cpp:259-320 (site-determining ions).
// ---------------------------------------------------------------------------------------------
#define PA_LCAP 256      // fragments per (isoform, ion type) list staged in shared memory (power of two)
#define PA_SORTCAP 256   // isoforms sortable in shared memory (aliases the list area)

struct SelSmem {
    PsmSmem psm;
    float run[2][PA_LMAX];          // running float sums of the two isoforms
    uint8_t nls[2][PA_LMAX];        // neutral-loss state after each step
    uint16_t foff[2][PA_LMAX + 4];  // fragment offset of each step (in units of one charge)
    alignas(8) float raw[2][PA_LCAP];  // unsorted fragment lists A, B (also the std::sort arena)
    float srt[2][PA_LCAP];          // sorted
};

struct PaSelArgs {
    int64_t n_psm;
    const int64_t* iso_off;
    const int32_t* psm_S;
    const int32_t* psm_status;
    PaIso iso;
    const int64_t* perm_off;     // [64*64] offset into perm_pool of the hash-order list of (S,k), -1 = none
    const uint32_t* perm_pool;   // isoform index (lexicographic rank) at each hash-iteration position
    const int64_t* mod_off;
    // outputs (device)
    uint64_t* best_sig;
    float* best_score;
    int64_t* n_iso;
    int32_t* n_sites;
    float* ascores;
    uint64_t* alt_sites;
    int32_t* psm_status_out;
    // scratch
    unsigned long long* g_sort;  // per isoform (iso_off), for std::sort emulation beyond PA_SORTCAP
    uint32_t* g_lr;              // partition stop lists of the warp replay: iso_off[p] + 2 p, n/2 + 1 entries per side
    int64_t mod_lo;              // absolute index of the chunk's first mod entry
    uint32_t* best_idx;          // [n_psm] best isoform (lexicographic rank), 0xffffffff = none
    int32_t* mod_psm;            // [entries] chunk-relative PSM of each mod entry, -1 = no Ascore to compute
    unsigned long long* tie;     // [entries] tied best competitors of each mod entry
    uint16_t* work_key;          // [entries] sort key of each mod entry: stream class << 10 | (1023 - estimated merge
    int32_t* work_val;           // [entries]   trips), PA_WORK_NONE = no site-determining-ion comparison needed; identity
    int* work_count;             // [4] entries per stream class (k_ascore)
    unsigned long long* next_psm;    // k_select's cursor into rest_list (zeroed before the launch)
    int32_t* rest_list;              // PSMs k_select_thread declines, for k_select (large isoform sets, tied top scores)
    int* rest_count;                 // their number (zeroed before the launch)
};
#define PA_WORK_BITS 13
#ifndef PA_WORK_SHIFT
#define PA_WORK_SHIFT 5      // low bits of the trip estimate dropped from the key (coarser classes keep more input order)
#endif
#define PA_WORK_NONE 0x1fffu

// --- libstdc++ std::sort (introsort + final insertion sort), comparator a.w > b.w ------------
// bits/stl_algo.h of GCC 13, as in SURVEY.md appendix A.2: the steps that decide its first element.
// Elements are (float w, uint32 id) packed in 64 bits: w in the high word.  The heap sort is run by ONE lane.
__device__ __forceinline__ float srt_w(unsigned long long e) { return __int_as_float((int)(e >> 32)); }
#define SRT_CMP(x, y) (srt_w(x) > srt_w(y))

__device__ void srt_adjust_heap(unsigned long long* a, long hole, long len, unsigned long long v) {
    const long top = hole;
    long child = hole;
    while (child < (len - 1) / 2) {
        child = 2 * (child + 1);
        if (SRT_CMP(a[child], a[child - 1])) child--;
        a[hole] = a[child]; hole = child;
    }
    if ((len & 1) == 0 && child == (len - 2) / 2) {
        child = 2 * (child + 1);
        a[hole] = a[child - 1]; hole = child - 1;
    }
    long parent = (hole - 1) / 2;
    while (hole > top && SRT_CMP(a[parent], v)) { a[hole] = a[parent]; hole = parent; parent = (hole - 1) / 2; }
    a[hole] = v;
}

__device__ void srt_heap_sort(unsigned long long* a, long n) {
    if (n < 2) return;
    for (long parent = (n - 2) / 2;; parent--) {
        srt_adjust_heap(a, parent, n, a[parent]);
        if (parent == 0) break;
    }
    for (long last = n; last > 1;) {
        --last;
        unsigned long long v = a[last];
        a[last] = a[0];
        srt_adjust_heap(a, 0, last, v);
    }
}

// Only the element std::sort would leave at index 0 is needed on the device (the full listing
// order is produced on the host by pa_fetch_pep_scores).  Introsort never moves an element from
// the right part of a partition into the left part afterwards, and the closing insertion sort moves
// an element left only past strictly smaller scores, so position 0 is decided by the chain of
// LEFTMOST partitions alone: replay those partitions (O(n) instead of O(n log n)), then take the
// first maximal element of the final left segment (the insertion sort is stable there).
__device__ uint32_t pa_gcc_sort_front(unsigned long long* a, long n) {
    if (n < 1) return 0xffffffffu;
    long lg = 0;
    for (long t = n; t > 1; t >>= 1) lg++;
    long last = n, depth = 2 * lg;
    const long first = 0;
    while (last - first > 16) {
        if (depth == 0) { srt_heap_sort(a, last); return (uint32_t)(a[0] & 0xffffffffull); }
        --depth;
        long mid = first + (last - first) / 2;
        long x = first + 1, y = mid, z = last - 1, pick;
        if (SRT_CMP(a[x], a[y])) { if (SRT_CMP(a[y], a[z])) pick = y; else if (SRT_CMP(a[x], a[z])) pick = z; else pick = x; }
        else if (SRT_CMP(a[x], a[z])) pick = x; else if (SRT_CMP(a[y], a[z])) pick = z; else pick = y;
        { unsigned long long t = a[first]; a[first] = a[pick]; a[pick] = t; }
        long f = first + 1, l = last;
        const unsigned long long pv = a[first];
        for (;;) {
            while (SRT_CMP(a[f], pv)) f++;
            --l;
            while (SRT_CMP(pv, a[l])) l--;
            if (!(f < l)) break;
            { unsigned long long t = a[f]; a[f] = a[l]; a[l] = t; }
            f++;
        }
        last = f;
    }
    long bi = 0;
    for (long i = 1; i < last; i++) if (SRT_CMP(a[i], a[bi])) bi = i;
    return (uint32_t)(a[bi] & 0xffffffffull);
}

// The same replay run by a whole WARP, for isoform sets too large for one lane's shared-memory arena (`a` lives in
// global memory; a single lane walking it pays an L2 round trip per element: 5.8 ms on the 15 504-isoform stress
// config).  One partition of std::__unguarded_partition is a function of the ORIGINAL arrangement: with
//   L_0 < L_1 < ...  the positions in [1, last) whose element does not beat the pivot   (where `first` stops),
//   R_0 > R_1 > ...  the positions the pivot does not beat, from the right               (where `last` stops),
// the sequential loop swaps the pairs (L_t, R_t) while L_t < R_t -- the elements between two stops are never
// touched, and a position a swap has filled stops the opposite cursor exactly where the next original stop or the
// swapped position comes first -- and returns cut = min(L_m, R_{m-1}) for the first m with L_m >= R_m.  Both stop
// lists are stream compactions (ballot + popc), the swaps are independent, so a partition costs two coalesced
// passes.  Only the first n/2 + 1 stops of each side can pair; `lst` holds 2 * (n/2 + 1) indices.
__device__ uint32_t pa_gcc_sort_front_warp(unsigned long long* a, long n, uint32_t* lst) {
    const int lane = threadIdx.x & 31;
    if (n < 1) return 0xffffffffu;
    long lg = 0;
    for (long t = n; t > 1; t >>= 1) lg++;
    long last = n, depth = 2 * lg;
    const long cap = n / 2 + 1;
    uint32_t* Ls = lst;
    uint32_t* Rs = lst + cap;
    const unsigned below = (1u << lane) - 1u;
    while (last > 16) {
        if (depth == 0) {                    // introsort's heap-sort fallback: sequential, as rare as in the reference
            unsigned long long r = 0;
            if (lane == 0) { srt_heap_sort(a, last); r = a[0]; }
            r = __shfl_sync(PA_FULL, r, 0);
            return (uint32_t)(r & 0xffffffffull);
        }
        --depth;
        if (lane == 0) {                     // median of a[1], a[mid], a[last-1] to the front (std::__move_median_to_first)
            const long mid = last / 2;
            const long x = 1, y = mid, z = last - 1;
            long pick;
            if (SRT_CMP(a[x], a[y])) { if (SRT_CMP(a[y], a[z])) pick = y; else if (SRT_CMP(a[x], a[z])) pick = z; else pick = x; }
            else if (SRT_CMP(a[x], a[z])) pick = x; else if (SRT_CMP(a[y], a[z])) pick = z; else pick = y;
            const unsigned long long t = a[0]; a[0] = a[pick]; a[pick] = t;
        }
        __syncwarp();
        const unsigned long long pv = a[0];
        long nL = 0, nR = 0;
        for (long base = 1; base < last; base += 32) {
            const long i = base + lane, j = last - base - lane;          // i ascends from 1, j descends from last - 1
            const bool okL = i < last && !SRT_CMP(a[i], pv);
            const bool okR = j >= 1 && !SRT_CMP(pv, a[j]);
            const unsigned bl = __ballot_sync(PA_FULL, okL), br = __ballot_sync(PA_FULL, okR);
            const long pl = nL + __popc(bl & below), pr = nR + __popc(br & below);
            if (okL && pl < cap) Ls[pl] = (uint32_t)i;
            if (okR && pr < cap) Rs[pr] = (uint32_t)j;
            nL += __popc(bl); nR += __popc(br);
        }
        __syncwarp();
        long lim = nL < nR ? nL : nR;
        lim = lim < cap ? lim : cap;
        // proper pairs: a prefix of t (L ascends, R descends)
        long m = 0;
        for (long t0 = 0; t0 < lim; t0 += 32) {
            const long t = t0 + lane;
            const unsigned ok = __ballot_sync(PA_FULL, t < lim && Ls[t] < Rs[t]);
            m += __popc(ok);
            if (ok != PA_FULL) break;
        }
        for (long t = lane; t < m; t += 32) {
            const uint32_t l = Ls[t], r = Rs[t];
            const unsigned long long tmp = a[l]; a[l] = a[r]; a[r] = tmp;
        }
        long cut = last;                     // (a stop always exists: the median-of-three leaves one on either side)
        if (m < nL && m < cap) cut = Ls[m];
        if (m > 0 && (long)Rs[m - 1] < cut) cut = Rs[m - 1];
        __syncwarp();
        last = cut;
    }
    // the closing insertion sort is stable on the left-most segment: its first maximal element comes to the front
    unsigned long long e = lane < last ? a[lane] : 0ull;
    float w = lane < last ? srt_w(e) : -INFINITY;
    float wm = w;
    for (int o = 16; o > 0; o >>= 1) { const float t = __shfl_xor_sync(PA_FULL, wm, o); wm = t > wm ? t : wm; }
    const unsigned is = __ballot_sync(PA_FULL, lane < last && w == wm);
    e = __shfl_sync(PA_FULL, e, __ffs(is) - 1);
    return (uint32_t)(e & 0xffffffffull);
}

// --- site-determining ions of isoforms A (slot 0) and B (slot 1) for one ion type ------------
// Returns via hits/trials accumulators (lane-uniform).  `la`,`lb`: list pointers (smem or global).
__device__ __forceinline__ void pa_sdi_type(const PaCfg& cfg, SelSmem* sm, const PsmInfo& info, char type,
                                            uint64_t maskA_lo, uint64_t maskA_hi, uint64_t maskB_lo,
                                            uint64_t maskB_hi, float* raw0, float* raw1, float* srt0,
                                            float* srt1, int depth, int& hitsA, int& trialsA, int& hitsB,
                                            int& trialsB) {
    const int lane = threadIdx.x & 31;
    const int L = info.L, Z = info.Z;
    const bool fwd = (type == 'b' || type == 'c');
    const int steps = (L == 1) ? 1 : L - 1;     // see pa_walk_isoform for the one-residue rule
    // 1. sequential running sums (lane 0: A, lane 1: B)
    if (lane < 2) {
        const uint64_t mlo = lane ? maskB_lo : maskA_lo, mhi = lane ? maskB_hi : maskA_hi;
        float run = 0.f;
        int nls = 0, off = 0;
        for (int step = 0; step < steps; step++) {
            const int i = fwd ? step : L - 1 - step;
            const int st = (int)(((i < 64) ? (mlo >> i) : (mhi >> (i - 64))) & 1ull);
            const float r = sm->psm.res[i][st];
            run = (step == 0) ? r : __fadd_rn(r, run);
            int nv = 1;
            if (cfg.has_nl) {
                int idx = sm->psm.nlidx[i][st];
                if (idx) nls = pa_nl_bump(nls, idx);
                nv = cfg.nl_nvar[nls];
            }
            if (L == 1) nv -= 1;
            sm->run[lane][step] = run;
            sm->nls[lane][step] = (uint8_t)nls;
            sm->foff[lane][step] = (uint16_t)off;
            off += nv;
        }
        sm->foff[lane][steps] = (uint16_t)off;
    }
    __syncwarp();
    const int nA = sm->foff[0][steps] * Z, nB = sm->foff[1][steps] * Z;
    // 2. all fragments (charges 1..Z) straight into the sort arrays, padded with +inf to a power of two
    const float PINF = __int_as_float(0x7f800000);
    int NA = 32, NB = 32;
    while (NA < nA) NA <<= 1;
    while (NB < nB) NB <<= 1;
    double a1, a2;
    pa_type_consts(type, a1, a2);
    for (int w = 0; w < 2; w++) {
        float* dst = w ? srt1 : srt0;
        const int n = w ? nB : nA, N = w ? NB : NA;
        for (int e = n + lane; e < N; e += 32) dst[e] = PINF;
        for (int step = lane; step < steps; step += 32) {
            const float run = sm->run[w][step];
            const int nls = sm->nls[w][step];
            const int nv = sm->foff[w][step + 1] - sm->foff[w][step];
            const int o = sm->foff[w][step] * Z;
            for (int v = 0; v < nv; v++) {
                float base = cfg.has_nl ? __fsub_rn(run, __ldg(cfg.nl_sums + nls * 16 + v)) : run;
                const double d = __dsub_rn(__dadd_rn((double)base, a1), a2);
                for (int z = 1; z <= Z; z++) dst[o + v * Z + (z - 1)] = pa_charge_mz(d, z);
            }
        }
    }
    __syncwarp();
    // 3. sort both lists ascending: warp-wide bitonic network over shared (or global) memory.
    //    Only the sorted VALUES matter downstream, so any correct sort reproduces std::sort here.
    for (int w = 0; w < 2; w++) {
        float* arr = w ? srt1 : srt0;
        const int N = w ? NB : NA;
        for (int kk = 2; kk <= N; kk <<= 1) {
            for (int j = kk >> 1; j > 0; j >>= 1) {
                for (int t = lane; t < (N >> 1); t += 32) {
                    const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                    const int l = i | j;
                    const bool asc = (i & kk) == 0;
                    const float x = arr[i], y = arr[l];
                    if ((x > y) == asc) { arr[i] = y; arr[l] = x; }
                }
                __syncwarp();
            }
        }
    }
    // 4. greedy tolerance merge (cpp/ModifiedPeptide.cpp:288-316): sequential by nature, run by
    //    lane 0 until one list is exhausted; the tail of the other list survives wholesale.
    //    Survivors are compacted at the front of raw0 / raw1.
    int cA = 0, cB = 0, ti = 0, tj = 0;
    if (lane == 0) {
        int i = 0, j = 0;
        const float err = cfg.err;
        float x = nA > 0 ? srt0[0] : PINF, y = nB > 0 ? srt1[0] : PINF;
        while (i < nA && j < nB) {
            if (fabsf(__fsub_rn(x, y)) < err) {
                i++; j++;
                x = i < nA ? srt0[i] : PINF;
                y = j < nB ? srt1[j] : PINF;
            } else if (x < y) {
                raw0[cA++] = x; i++;
                x = i < nA ? srt0[i] : PINF;
            } else {
                raw1[cB++] = y; j++;
                y = j < nB ? srt1[j] : PINF;
            }
        }
        ti = i; tj = j;
    }
    cA = __shfl_sync(PA_FULL, cA, 0);
    cB = __shfl_sync(PA_FULL, cB, 0);
    ti = __shfl_sync(PA_FULL, ti, 0);
    tj = __shfl_sync(PA_FULL, tj, 0);
    for (int e = ti + lane; e < nA; e += 32) raw0[cA + (e - ti)] = srt0[e];
    for (int e = tj + lane; e < nB; e += 32) raw1[cB + (e - tj)] = srt1[e];
    cA += nA - ti;
    cB += nB - tj;
    __syncwarp();
    // 5. hits: survivors whose matched rank <= depth
    int hA = 0, hB = 0;
    for (int e = lane; e < cA; e += 32)
        hA += pa_match_rank(info, raw0[e], cfg.err, cfg.err_gt_half) <= depth;
    for (int e = lane; e < cB; e += 32)
        hB += pa_match_rank(info, raw1[e], cfg.err, cfg.err_gt_half) <= depth;
    for (int o = 16; o > 0; o >>= 1) { hA += __shfl_xor_sync(PA_FULL, hA, o); hB += __shfl_xor_sync(PA_FULL, hB, o); }
    hitsA += hA; hitsB += hB; trialsA += cA; trialsB += cB;
    __syncwarp();
}

// cpp/Ascore.cpp:157-210.  scA/scB: the depth scores of the two isoforms (lane-uniform arrays): ten, or with DEEP
// (a scorer with n_top > 10) 10 + dp.nd, the argmax running over all of them and the final scores of a depth >= 10
// coming from dp.T.
template <bool DEEP>
__device__ __forceinline__ float pa_ambiguity(const PaCfg& cfg, SelSmem* sm, const PsmInfo& info, uint64_t bitsA,
                                              const float* scA, float wA, uint64_t bitsB, const float* scB,
                                              float wB, float* raw0, float* raw1, float* srt0, float* srt1,
                                              const PaDeep& dp) {
    if ((double)fabsf(__fsub_rn(wA, wB)) < 1e-6) return 0.f;
    float max_diff = 0.f;
    int depth = 0;
#pragma unroll
    for (int d = 0; d < PA_N_TOP; d++) {
        float diff = __fsub_rn(scA[d], scB[d]);
        if (diff > max_diff) { max_diff = diff; depth = d; }
    }
    if (DEEP)
        for (int d = PA_N_TOP; d < PA_N_TOP + dp.nd; d++) {
            float diff = __fsub_rn(scA[d], scB[d]);
            if (diff > max_diff) { max_diff = diff; depth = d; }
        }
    uint64_t alo, ahi, blo, bhi;
    pa_sites_to_mask(&sm->psm, bitsA, alo, ahi);
    pa_sites_to_mask(&sm->psm, bitsB, blo, bhi);
    int hitsA = 0, hitsB = 0, trialsA = 0, trialsB = 0;
    for (int t = 0; t < cfg.n_types; t++)
        pa_sdi_type(cfg, sm, info, cfg.types[t], alo, ahi, blo, bhi, raw0, raw1, srt0, srt1, depth, hitsA,
                    trialsA, hitsB, trialsB);
    if (DEEP) return __fsub_rn(pa_depth_score(cfg.T, dp, trialsA, hitsA, depth), pa_depth_score(cfg.T, dp, trialsB, hitsB, depth));
    const float sA = __ldg(cfg.T + pa_tab_index(trialsA, hitsA, depth));
    const float sB = __ldg(cfg.T + pa_tab_index(trialsB, hitsB, depth));
    return __fsub_rn(sA, sB);
}

__device__ __forceinline__ void pa_depth_scores(const PaCfg& cfg, unsigned long long lo, unsigned long long hi,
                                                int n, float* sc) {
#pragma unroll
    for (int d = 0; d < PA_N_TOP; d++) sc[d] = __ldg(cfg.T + pa_tab_index(n, pa_cum_get(lo, hi, d), d));
}

// depths 10 .. n_top-1 of isoform g (K2d counts), into sc[10 ..]
__device__ __forceinline__ void pa_deep_scores(const PaDeep& dp, int64_t g, int n, float* sc) {
    for (int dd = 0; dd < dp.nd; dd++)
        sc[PA_N_TOP + dd] = __ldg(dp.T + pa_tab_index_deep(n, dp.cnt[(size_t)g * dp.nd + dd], dd, dp.nd));
}

// position of the n-th set bit (n counted from 0) of a 128-bit mask
__device__ __forceinline__ int pa_nth_set(uint64_t lo, uint64_t hi, int n) {
    const int c = __popcll(lo);
    uint64_t x = lo;
    int base = 0;
    if (n >= c) { x = hi; n -= c; base = 64; }
    for (int i = 0; i < n; i++) x &= x - 1;
    return base + __ffsll((long long)x) - 1;
}

// K3a, the Ascore-0 shortcut: every tied competitor has exactly the score m; within 1e-6 of the best score wb the
// ambiguity is 0 without looking at any ion (cpp/Ascore.cpp:161-163), so the Ascore (the minimum over the tie set)
// is 0.
__device__ __forceinline__ bool pa_asc_zero(float wb, float m) { return (double)fabsf(__fsub_rn(wb, m)) < 1e-6; }

// K3a, the sort key of an Ascore entry that goes to k_ascore: stream class `cls` (so that the lanes of a k_ascore
// warp run the same code), then the estimated number of merge trips, longest first -- per tied competitor one trip
// per residue plus three per residue between the two sites, times the charges -- and the host sorts the entries by
// it, so that the lanes of a warp also finish together.  pos(s) is the residue index of site s.
template <class Pos>
__device__ __forceinline__ uint32_t pa_work_key(const PaCfg& cfg, int Z, int L, int site, uint64_t tie, Pos pos,
                                                int& cls) {
    cls = cfg.has_nl ? 3 : (Z == 1 ? 0 : (Z == 2 ? 1 : (Z <= 4 ? 2 : 3)));
    int work = 0;
    const int ps = pos(site);
    for (uint64_t tt = tie; tt; tt &= tt - 1) {
        const int pu = pos(__ffsll((long long)tt) - 1);
        work += (L - 1) + 3 * (pu > ps ? pu - ps : ps - pu);
    }
    work *= Z < 8 ? Z : 8;
    return ((uint32_t)cls << 10) | (((uint32_t)(1023 - (work > 1023 ? 1023 : work)) >> PA_WORK_SHIFT) << PA_WORK_SHIFT);
}

// K3a, common case: one THREAD per PSM.  A PSM of config-2 size has a dozen isoforms and a handful of
// sites: a warp per PSM spends its instructions on reductions over mostly empty lanes.  A thread walks
// the same steps serially (best isoform, per modified site the tied best competitors, Ascore-0 shortcut,
// sort key of every Ascore entry).  PSMs whose best score is tied among more than 16 isoforms (the
// reference's std::sort order decides, which takes the warp kernel's sort replay) or that have more than
// PA_SEL_THREAD_MAX isoforms are left, untouched, to k_select through rest_list.  TYPED (a pass of a typed batch):
// a PSM of another type (PA_PSM_OTHER_TYPE) gets only the scratch entries that keep its Ascore entries out of K3b /
// K3c, and none of the results, which belong to its own type's pass.  (k_select needs no gate: such a PSM is never
// declined to it.)
#define PA_SEL_THREAD_MAX 512
template <bool TYPED>
__global__ void __launch_bounds__(128) k_select_thread(PaCfg cfg, PaBatchDev b, PaSelArgs a) {
    __shared__ int s_cls[4];
    if (threadIdx.x < 4) s_cls[threadIdx.x] = 0;
    __syncthreads();
    const float INF = __int_as_float(0x7f800000);
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < a.n_psm) {
        const int status = a.psm_status[p];
        const int k = b.n_mod[p];
        const int64_t mo = a.mod_off[p];
        const int S = a.psm_S[p];
        const int64_t ib = a.iso_off[p];
        const int64_t I = a.iso_off[p + 1] - ib;
        bool rest = false;
        float wmax = -INF;
        uint32_t best = 0xffffffffu;
        const bool none = status != PA_PSM_OK || I == 0 || k >= S;
        if (!none) {
            if (I > PA_SEL_THREAD_MAX) rest = true;
            else {
                int ties = 0;
                for (int64_t q = 0; q < I; q++) {
                    const float w = a.iso.w[ib + q];
                    if (w > wmax) { wmax = w; ties = 1; best = (uint32_t)q; }
                    else if (w == wmax) { if (ties == 0) best = (uint32_t)q; ties++; }
                }
                if (ties > 1) {
                    if (I > 16) rest = true;
                    else {
                        // std::sort on <= 16 elements is a stable insertion sort: the first maximal element
                        // in hash-iteration order stays in front
                        const uint32_t* perm = a.perm_pool + a.perm_off[S * 64 + k];
                        for (int t = 0; t < (int)I; t++) {
                            const uint32_t id = perm[t];
                            if (a.iso.w[ib + id] == wmax) { best = id; break; }
                        }
                    }
                }
            }
        }
        const bool own = !TYPED || status != PA_PSM_OTHER_TYPE;
        if (rest) {
            a.rest_list[atomicAdd(a.rest_count, 1)] = (int32_t)p;
        } else {
            if (own) {
                if (a.psm_status_out) a.psm_status_out[p] = status;
                if (a.n_iso) a.n_iso[p] = I;
                if (a.n_sites) a.n_sites[p] = S;
            }
            if (none) {
                // no isoform: best_sequence "" / best_score -1 (cpp/Ascore.cpp:273-295); k >= #sites is
                // "unambiguous" (cpp/Ascore.cpp:38-51: ascores inf, no alternatives); errors report NaN
                const bool ok = status == PA_PSM_OK;
                const float fill = ok ? INF : __int_as_float(0x7fc00000);
                uint64_t sig = 0; float sc = ok ? -1.f : fill;
                if (ok && I > 0) { sig = (S >= 64) ? ~0ull : ((1ull << S) - 1ull); sc = a.iso.w[ib]; }
                if (own) {
                    if (a.best_sig) a.best_sig[p] = sig;
                    if (a.best_score) a.best_score[p] = sc;
                }
                a.best_idx[p] = (ok && I > 0) ? 0u : 0xffffffffu;
                for (int j = 0; j < k; j++) {
                    if (own) {
                        if (a.ascores) a.ascores[mo + j] = fill;
                        if (a.alt_sites) a.alt_sites[mo + j] = 0;
                    }
                    a.mod_psm[mo + j - a.mod_lo] = -1;
                    a.work_key[mo + j - a.mod_lo] = (uint16_t)PA_WORK_NONE;
                    a.work_val[mo + j - a.mod_lo] = (int32_t)(mo + j - a.mod_lo);
                }
            } else {
                const uint64_t best_bits = pa_unrank(cfg.binom, S, k, best);
                const float wb = a.iso.w[ib + best];
                if (a.best_sig) a.best_sig[p] = best_bits;
                if (a.best_score) a.best_score[p] = wb;
                a.best_idx[p] = best;
                // residues that are sites, for the merge-length estimate (see pa_work_key)
                const int pep0 = b.pep_off[p], L = b.pep_off[p + 1] - pep0;
                uint64_t slo = 0, shi = 0;
                if (a.ascores)
                    for (int i = 0; i < L; i++) {
                        const int c = (int)b.pep[pep0 + i] - 'A';
                        const bool is = ((c >= 0 && c < 26) && ((cfg.mod_letters >> c) & 1u)) || (cfg.allow_n && i == 0) || (cfg.allow_c && i == L - 1);
                        if (is) { if (i < 64) slo |= 1ull << i; else shi |= 1ull << (i - 64); }
                    }
                const uint64_t all = (S >= 64) ? ~0ull : ((1ull << S) - 1ull);
                const uint64_t free_sites = all & ~best_bits;
                uint64_t rem = best_bits;
                for (int j = 0; j < k; j++) {
                    const int site = __ffsll((long long)rem) - 1;
                    rem &= rem - 1;
                    // tied best competitors of this site (cpp/Ascore.cpp:212-254)
                    float m = -INF;
                    uint64_t tie = 0;
                    for (uint64_t f = free_sites; f; f &= f - 1) {
                        const int u = __ffsll((long long)f) - 1;
                        const float w = a.iso.w[ib + pa_rank(cfg.binom, S, k, (best_bits & ~(1ull << site)) | (1ull << u))];
                        if (w > m) { m = w; tie = 1ull << u; }
                        else if (w == m) tie |= 1ull << u;
                    }
                    if (a.alt_sites) a.alt_sites[mo + j] = tie;
                    a.tie[mo + j - a.mod_lo] = tie;
                    a.mod_psm[mo + j - a.mod_lo] = (int32_t)p;
                    if (a.ascores) {
                        uint32_t key = PA_WORK_NONE;
                        if (pa_asc_zero(wb, m)) a.ascores[mo + j] = 0.f;
                        else {
                            int cls;
                            key = pa_work_key(cfg, b.max_charge[p], L, site, tie,
                                              [&](int s) { return pa_nth_set(slo, shi, s); }, cls);
                            atomicAdd(&s_cls[cls], 1);
                        }
                        a.work_key[mo + j - a.mod_lo] = (uint16_t)key;
                        a.work_val[mo + j - a.mod_lo] = (int32_t)(mo + j - a.mod_lo);
                    }
                }
            }
        }
    }
    __syncthreads();
    if (threadIdx.x < 4 && s_cls[threadIdx.x]) atomicAdd(a.work_count + threadIdx.x, s_cls[threadIdx.x]);
}

// K3a for the PSMs k_select_thread declines: one WARP per PSM, taken from rest_list.  Every PSM here has status
// OK, I > 0 and k < S, and either more than PA_SEL_THREAD_MAX isoforms or a top score tied among more than 16
// isoforms (where the reference's std::sort order decides).  Best isoform in the reference's order + per modified
// site the set of tied best competitors (= alternative sites).  The thread kernel writes nothing for these PSMs, so
// their status, n_iso and n_sites are written here too.
__global__ void __launch_bounds__(256) k_select(PaCfg cfg, PaBatchDev b, PaSelArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    unsigned long long* s_sort = (unsigned long long*)smem_raw + (size_t)wib * PA_SORTCAP;
    __shared__ uint8_t s_pos_all[8][64];              // per warp: residue index of each site of the current PSM
    uint8_t* s_pos = s_pos_all[wib];
    int qn0 = 0, qn1 = 0, qn2 = 0, qn3 = 0;           // Ascore entries found per stream class (lane-uniform)
    const float INF = __int_as_float(0x7f800000);

    // Warps take one PSM at a time from a global cursor (the cost per PSM grows with its isoform count, so a
    // static split leaves warps idle).
    const int64_t n = *a.rest_count;
    for (;;) {
        unsigned long long pi = 0;
        if (lane == 0) pi = atomicAdd(a.next_psm, 1ull);
        pi = __shfl_sync(PA_FULL, pi, 0);
        if ((int64_t)pi >= n) break;
        const int64_t p = a.rest_list[pi];
        const int k = b.n_mod[p];
        const int64_t mo = a.mod_off[p];
        const int S = a.psm_S[p];
        const int64_t I = a.iso_off[p + 1] - a.iso_off[p];
        const int64_t ib = a.iso_off[p];
        if (lane == 0) {
            if (a.psm_status_out) a.psm_status_out[p] = a.psm_status[p];
            if (a.n_iso) a.n_iso[p] = I;
            if (a.n_sites) a.n_sites[p] = S;
        }
        // residue positions of the sites: the distance between two sites is what an Ascore merge costs
        const int pep0 = b.pep_off[p], L = b.pep_off[p + 1] - pep0;
        if (a.ascores) {
            int ns = 0;
            __syncwarp();
            for (int base = 0; base < L; base += 32) {
                const int i = base + lane;
                bool is = false;
                if (i < L) {
                    const int c = (int)b.pep[pep0 + i] - 'A';
                    is = ((c >= 0 && c < 26) && ((cfg.mod_letters >> c) & 1u)) || (cfg.allow_n && i == 0) || (cfg.allow_c && i == L - 1);
                }
                const unsigned bal = __ballot_sync(PA_FULL, is);
                if (is) { const int j = ns + __popc(bal & ((1u << lane) - 1u)); if (j < 64) s_pos[j] = (uint8_t)i; }
                ns += __popc(bal);
            }
            __syncwarp();
        }
        // ---- best isoform ---------------------------------------------------------------
        float wmax = -INF;
        for (int64_t q = lane; q < I; q += 32) { float w = a.iso.w[ib + q]; wmax = w > wmax ? w : wmax; }
        for (int o = 16; o > 0; o >>= 1) { float t = __shfl_xor_sync(PA_FULL, wmax, o); wmax = t > wmax ? t : wmax; }
        int ties = 0;
        uint32_t first_tie = 0xffffffffu;
        for (int64_t q = lane; q < I; q += 32)
            if (a.iso.w[ib + q] == wmax) { ties++; if (first_tie == 0xffffffffu) first_tie = (uint32_t)q; }
        for (int o = 16; o > 0; o >>= 1) {
            ties += __shfl_xor_sync(PA_FULL, ties, o);
            uint32_t t = __shfl_xor_sync(PA_FULL, first_tie, o); first_tie = t < first_tie ? t : first_tie;
        }
        uint32_t best = first_tie;
        if (ties > 1) {
            // a tie among more than 16 isoforms: replay std::sort's partitions over the hash-iteration order
            const uint32_t* perm = a.perm_pool + a.perm_off[S * 64 + k];
            unsigned long long* arr = (I <= PA_SORTCAP) ? s_sort : a.g_sort + ib;
            __syncwarp();
            for (int64_t q = lane; q < I; q += 32) {
                uint32_t id = perm[q];
                arr[q] = ((unsigned long long)(uint32_t)__float_as_int(a.iso.w[ib + id]) << 32) | id;
            }
            __syncwarp();
            if (I <= PA_SORTCAP) {           // shared-memory arena: one lane replays the partitions
                if (lane == 0) best = pa_gcc_sort_front(arr, (long)I);
                best = __shfl_sync(PA_FULL, best, 0);
            } else best = pa_gcc_sort_front_warp(arr, (long)I, a.g_lr + ib + 2 * p);
            __syncwarp();
        }
        const uint64_t best_bits = pa_unrank(cfg.binom, S, k, best);
        const float wb = a.iso.w[ib + best];
        if (lane == 0) {
            if (a.best_sig) a.best_sig[p] = best_bits;
            if (a.best_score) a.best_score[p] = wb;
            a.best_idx[p] = best;
        }
        // ---- tied best competitors per modified site (cpp/Ascore.cpp:212-254) ---------------
        const uint64_t all = (S >= 64) ? ~0ull : ((1ull << S) - 1ull);
        const uint64_t free_sites = all & ~best_bits;
        uint64_t rem = best_bits;
        for (int j = 0; j < k; j++) {
            const int site = __ffsll((long long)rem) - 1;
            rem &= rem - 1;
            float w0 = -INF, w1 = -INF;      // competitor scores of free sites lane, lane+32
            if (lane < S && ((free_sites >> lane) & 1ull))
                w0 = a.iso.w[ib + pa_rank(cfg.binom, S, k, (best_bits & ~(1ull << site)) | (1ull << lane))];
            if (lane + 32 < S && ((free_sites >> (lane + 32)) & 1ull))
                w1 = a.iso.w[ib + pa_rank(cfg.binom, S, k, (best_bits & ~(1ull << site)) | (1ull << (lane + 32)))];
            float m = w0 > w1 ? w0 : w1;
            for (int o = 16; o > 0; o >>= 1) { float t = __shfl_xor_sync(PA_FULL, m, o); m = t > m ? t : m; }
            const bool f0 = lane < S && ((free_sites >> lane) & 1ull) && w0 == m;
            const bool f1 = lane + 32 < S && ((free_sites >> (lane + 32)) & 1ull) && w1 == m;
            const uint64_t tie = (uint64_t)__ballot_sync(PA_FULL, f0) | ((uint64_t)__ballot_sync(PA_FULL, f1) << 32);
            if (lane == 0) {
                if (a.alt_sites) a.alt_sites[mo + j] = tie;
                a.tie[mo + j - a.mod_lo] = tie;
                a.mod_psm[mo + j - a.mod_lo] = (int32_t)p;
            }
            if (a.ascores) {
                const bool zero = pa_asc_zero(wb, m);
                uint32_t key = PA_WORK_NONE;
                if (!zero) {
                    int cls;
                    key = pa_work_key(cfg, b.max_charge[p], L, site, tie, [&](int s) { return (int)s_pos[s]; }, cls);
                    int& qn = cls == 0 ? qn0 : (cls == 1 ? qn1 : (cls == 2 ? qn2 : qn3));
                    qn++;
                }
                if (lane == 0) {
                    if (zero) a.ascores[mo + j] = 0.f;
                    a.work_key[mo + j - a.mod_lo] = (uint16_t)key;
                    a.work_val[mo + j - a.mod_lo] = (int32_t)(mo + j - a.mod_lo);
                }
            }
        }
        __syncwarp();
    }
    if (a.ascores && lane == 0) {
        if (qn0) atomicAdd(a.work_count + 0, qn0);
        if (qn1) atomicAdd(a.work_count + 1, qn1);
        if (qn2) atomicAdd(a.work_count + 2, qn2);
        if (qn3) atomicAdd(a.work_count + 3, qn3);
    }
}

// ---------------------------------------------------------------------------------------------
// K3b: one THREAD per (PSM, modified site) entry.  For every tied competitor: the site-determining
// ion comparison of cpp/Ascore.cpp:157-210 + cpp/ModifiedPeptide.cpp:259-320, computed without
// materialising or sorting the fragment lists: each (charge, neutral-loss variant) is a stream that
// is already ascending along the peptide, so "sort, then tolerance-merge" becomes a k-way streaming
// merge whose element VALUES are exactly those of the reference's sorted lists.  If a stream is
// ever found non-ascending (non-positive residue mass), or the shape is out of range (too many
// streams, one-residue peptide), the entry is queued for k_ascore_generic instead.
// ---------------------------------------------------------------------------------------------
#define PA_MAXSTREAM 12

struct PaAscArgs {
    int64_t n_entries;           // mod entries of this chunk
    int64_t mod_lo;              // absolute index of the chunk's first entry
    const int32_t* mod_psm;      // [n_entries] chunk-relative PSM, -1 = nothing to do
    const unsigned long long* tie;   // [n_entries] tied competitor sites
    const uint32_t* best_idx;    // [n_psm]
    const int64_t* mod_off;      // [n_psm+1] absolute
    const int64_t* iso_off;
    const int32_t* psm_S;
    PaIso iso;
    float* ascores;              // absolute-indexed output (may be null)
    const int32_t* work_sorted;  // mod entries sorted by K3a's key: class 0 first, longest merges first
    const int* work_count;       // [4] entries per stream class
    int32_t* generic_list;       // entries that need the generic kernel
    int* generic_count;
};

struct AscPep {                  // what a thread needs to know about its peptide
    const uint8_t* pep;
    int L, Z, a0, a1;
    const uint32_t* aux_pos;
    const float* aux_mass;
    uint64_t aux_lo, aux_hi;     // residues that carry a fixed mod
};

// residue mass / neutral-loss index of residue i in modification state st
// (cpp/ModifiedPeptide.cpp:24-79 evaluated on the fly instead of tabulated)
__device__ __forceinline__ float asc_res(const PaCfg& cfg, const AscPep& q, int i, int st, int& nlidx) {
    const int c = (int)q.pep[i] - 'A';
    float m = __ldg(cfg.res_tab + c);
    if (st) m = __fadd_rn(m, cfg.mod_mass);
    nlidx = 0;
    if (cfg.has_nl) nlidx = st ? __ldg(cfg.nl_lo_tab + c) : __ldg(cfg.nl_up_tab + c);
    if (((i < 64) ? (q.aux_lo >> i) : (q.aux_hi >> (i - 64))) & 1ull) {
        for (int a = q.a0; a < q.a1; a++) {
            const uint32_t pos = q.aux_pos[a];
            const int idx = pos > 0 ? (int)pos - 1 : 0;
            if (idx == i) {
                m = __fadd_rn(m, q.aux_mass[a]);
                if (cfg.has_nl && __ldg(cfg.nl_lo_tab + c)) nlidx = __ldg(cfg.nl_lo_tab + c);
            }
        }
    }
    return m;
}

__device__ __forceinline__ int asc_match(const float2* pp, int R, const uint8_t* ctab, float cbase,
                                         float cinv, float f, float err, int err_gt_half) {
    const float lo = __fsub_rn(f, err), hi = __fadd_rn(f, err);
    int a;
    if (cinv != 0.f) {
        a = __ldg(ctab + pa_cell(lo, cbase, cinv));
    } else {
        a = 0;
        int n = R;
        while (n > 0) {
            int h = n >> 1;
            if (!(__ldg(pp + a + h).x > lo)) { a += h + 1; n -= h + 1; } else n = h;
        }
    }
    int best = 255;
    if (a < R) {
        // {mz, rank bits}: one load per candidate, the first two in flight together (most scans end on the second)
        float2 e = __ldg(pp + a);
        float2 e_next = __ldg(pp + (a + 1 < R ? a + 1 : R - 1));
        for (;;) {
            if (!(e.x < hi)) break;
            if (e.x > lo && !(err_gt_half && !((double)f >= (double)e.x - .5))) {
                const int r = __float_as_int(e.y);
                best = r < best ? r : best;
            }
            if (++a >= R) break;
            e = e_next;
            if (!(e.x < hi)) break;
            e_next = __ldg(pp + (a + 1 < R ? a + 1 : R - 1));
        }
    }
    return best;
}

struct AscPeaks {
    const float2* pp; int R; const uint8_t* ctab; float cbase, cinv;
};

#define ASC_BLOCK 128

// a survivor of the merge: one trial of its list, a hit when its matched peak is ranked within `depth`
__device__ __forceinline__ void asc_survivor(const PaCfg& cfg, const AscPeaks& pk, int depth, float v, bool from_a,
                                             int& hitsA, int& trialsA, int& hitsB, int& trialsB) {
    const int hit = asc_match(pk.pp, pk.R, pk.ctab, pk.cbase, pk.cinv, v, cfg.err, cfg.err_gt_half) <= depth;
    if (from_a) { trialsA++; hitsA += hit; } else { trialsB++; hitsB += hit; }
}

// ---- general stream form (neutral losses and/or more than four charges) ---------------------
// Per thread up to PA_MAXSTREAM streams per list, one per (neutral-loss sum, charge); their state
// lives in shared memory ([field][list][stream][thread]: conflict-free) so that a stream can be
// addressed by a run-time index without spilling to local memory.
struct AscSm {
    float run[2][PA_MAXSTREAM][ASC_BLOCK];     // float32 running sum at the stream's current step
    float val[2][PA_MAXSTREAM][ASC_BLOCK];     // pending fragment m/z (+inf: exhausted)
    float sig[2][PA_MAXSTREAM][ASC_BLOCK];     // neutral-loss sum of the stream
    int stz[2][PA_MAXSTREAM][ASC_BLOCK];       // current step | charge << 16
};

// Streams of list w (mask mlo/mhi).  Returns the stream count, or -1 when the shape is not supported.
__device__ __forceinline__ int asc_streams_init(const PaCfg& cfg, const AscPep& q, AscSm* sm, int w, uint64_t mlo,
                                                uint64_t mhi, bool fwd, double a1, double a2, int& left) {
    const int tid = threadIdx.x;
    const int L = q.L, Z = q.Z, steps = L - 1;
    int V = 1;
    if (!cfg.has_nl) {
        if (Z > PA_MAXSTREAM) return -1;
        const int i = fwd ? 0 : L - 1;
        int idx;
        sm->sig[w][0][tid] = 0.f; sm->stz[w][0][tid] = 0;
        sm->run[w][0][tid] = asc_res(cfg, q, i, (int)(((i < 64) ? (mlo >> i) : (mhi >> (i - 64))) & 1ull), idx);
    } else {
        // pass 1: the final neutral-loss state says which sums will ever exist
        int nls = 0;
        for (int step = 0; step < steps; step++) {
            const int i = fwd ? step : L - 1 - step;
            int idx;
            (void)asc_res(cfg, q, i, (int)(((i < 64) ? (mlo >> i) : (mhi >> (i - 64))) & 1ull), idx);
            if (idx) nls = pa_nl_bump(nls, idx);
        }
        V = cfg.nl_nvar[nls];
        if (V * Z > PA_MAXSTREAM) return -1;
        for (int v = 0; v < V; v++) { sm->sig[w][v][tid] = __ldg(cfg.nl_sums + nls * 16 + v); sm->stz[w][v][tid] = -1; sm->run[w][v][tid] = 0.f; }
        // pass 2: the step at which each sum first becomes available (the stack only grows, so it
        // stays available afterwards) and the running sum there
        int started = 0;
        float run = 0.f;
        nls = 0;
        for (int step = 0; step < steps && started < V; step++) {
            const int i = fwd ? step : L - 1 - step;
            int idx;
            run = __fadd_rn(asc_res(cfg, q, i, (int)(((i < 64) ? (mlo >> i) : (mhi >> (i - 64))) & 1ull), idx), run);
            const int before = nls;
            if (idx) nls = pa_nl_bump(nls, idx);
            if (step == 0 || nls != before) {
                const int nv = cfg.nl_nvar[nls];
                for (int v = 0; v < V; v++) {
                    if (sm->stz[w][v][tid] >= 0) continue;
                    const float sg = sm->sig[w][v][tid];
                    bool in = false;
                    for (int u = 0; u < nv; u++) in |= (__ldg(cfg.nl_sums + nls * 16 + u) == sg);
                    if (in) { sm->stz[w][v][tid] = step; sm->run[w][v][tid] = run; started++; }
                }
            }
        }
    }
    // expand variant v into its Z charge streams v*Z .. v*Z+Z-1, back to front (slot v is read
    // before a lower-numbered variant's stream can overwrite it)
    left = 0;
    for (int qi = V * Z - 1; qi >= 0; qi--) {
        const int v = qi / Z, z = qi - v * Z + 1;
        const float run = sm->run[w][v][tid], sg = sm->sig[w][v][tid];
        const int start = sm->stz[w][v][tid] & 0xffff;
        sm->run[w][qi][tid] = run; sm->sig[w][qi][tid] = sg; sm->stz[w][qi][tid] = start | (z << 16);
        sm->val[w][qi][tid] = pa_charge_mz(__dsub_rn(__dadd_rn((double)__fsub_rn(run, sg), a1), a2), z);
        left += steps - start;
    }
    return V * Z;
}

__device__ __forceinline__ bool asc_merge_streams(const PaCfg& cfg, const AscPep& q, const AscPeaks& pk, bool fwd,
                                                  double a1, double a2, uint64_t alo, uint64_t ahi, uint64_t blo,
                                                  uint64_t bhi, int depth, int& hitsA, int& trialsA,
                                                  int& hitsB, int& trialsB) {
    extern __shared__ __align__(16) unsigned char asc_smem_raw[];
    AscSm* sm = (AscSm*)asc_smem_raw;
    const int tid = threadIdx.x;
    const int L = q.L, steps = L - 1;
    const float PINF = __int_as_float(0x7f800000);
    int leftA, leftB;
    const int nqA = asc_streams_init(cfg, q, sm, 0, alo, ahi, fwd, a1, a2, leftA);
    const int nqB = asc_streams_init(cfg, q, sm, 1, blo, bhi, fwd, a1, a2, leftB);
    if (nqA < 0 || nqB < 0) return false;
    bool mono = true;
    float x = 0.f, y = 0.f;
    bool hx = false, hy = false;
    for (;;) {
        const bool needA = !hx && leftA > 0, needB = !hy && leftB > 0;
        if (needA || needB) {
            const int w = needA ? 0 : 1;
            const int nq = w ? nqB : nqA;
            int bq = 0;
            float xm = sm->val[w][0][tid];
            for (int i = 1; i < nq; i++) { const float v = sm->val[w][i][tid]; if (v < xm) { xm = v; bq = i; } }
            const int stz = sm->stz[w][bq][tid];
            const int step = (stz & 0xffff) + 1, z = stz >> 16;
            float nv = PINF;
            if (step < steps) {
                const int i = fwd ? step : L - 1 - step;
                const uint64_t mlo = w ? blo : alo, mhi = w ? bhi : ahi;
                int idx;
                const float run = __fadd_rn(asc_res(cfg, q, i, (int)(((i < 64) ? (mlo >> i) : (mhi >> (i - 64))) & 1ull), idx),
                                            sm->run[w][bq][tid]);
                sm->run[w][bq][tid] = run;
                nv = pa_charge_mz(__dsub_rn(__dadd_rn((double)__fsub_rn(run, sm->sig[w][bq][tid]), a1), a2), z);
                if (nv < xm) mono = false;
            }
            sm->stz[w][bq][tid] = step | (z << 16);
            sm->val[w][bq][tid] = nv;
            if (w) { y = xm; hy = true; leftB--; } else { x = xm; hx = true; leftA--; }
        }
        if ((hx || leftA == 0) && (hy || leftB == 0)) {
            if (!hx && !hy) break;
            int takeA;                       // 1: A survives, 0: B survives, -1: both dropped
            if (!hy) takeA = 1;
            else if (!hx) takeA = 0;
            else if (fabsf(__fsub_rn(x, y)) < cfg.err) takeA = -1;
            else takeA = x < y;
            if (takeA < 0) { hx = false; hy = false; }
            else {
                asc_survivor(cfg, pk, depth, takeA ? x : y, takeA != 0, hitsA, trialsA, hitsB, trialsB);
                if (takeA) hx = false; else hy = false;
            }
        }
    }
    return mono;
}

// greedy tolerance merge of cpp/ModifiedPeptide.cpp:288-316 over the streams of the best isoform
// (mask a) and one competitor (mask b) for one ion type; false = needs the generic kernel.
//
// Two exact shortcuts keep the merge short:
//  * Common prefix.  Up to the first residue at which the two isoforms differ (step d of the walk)
//    both lists hold the same fragments.  With T = the smallest fragment of step d over both lists and
//    all charges, every fragment below T stems from a common step, so the sorted lists start with the
//    same values and the greedy merge drops them pairwise (|x - y| = 0 < mz_error).  The streams are
//    therefore started at their first fragment >= T; the steps before cost one float add each.
//  * One trip settles both heads.  A trip pops a head for whichever list lacks one (both, after a
//    pairwise drop) and then takes the one decision the reference takes on two settled heads.
template <int NQ>
__device__ __forceinline__ bool asc_merge_type(const PaCfg& cfg, const AscPep& q, const AscPeaks& pk, char type,
                                               uint64_t alo, uint64_t ahi, uint64_t blo, uint64_t bhi, int depth,
                                               int& hitsA, int& trialsA, int& hitsB, int& trialsB) {
    const bool fwd = (type == 'b' || type == 'c');
    double a1, a2;
    pa_type_consts(type, a1, a2);
    bool mono = true;
    float x = 0.f, y = 0.f;
    bool hx = false, hy = false;         // a popped element is pending
    if (NQ <= 4) {
        // no neutral loss: stream z-1 holds charge z; everything in registers
        const int L = q.L, Z = q.Z, steps = L - 1;
        const float PINF = __int_as_float(0x7f800000);
        float runA[NQ], valA[NQ], runB[NQ], valB[NQ];
        int stepA[NQ], stepB[NQ];
        auto res_at = [&](int step, uint64_t mlo, uint64_t mhi) {
            const int i = fwd ? step : L - 1 - step;
            int idx;
            return asc_res(cfg, q, i, (int)(((i < 64) ? (mlo >> i) : (mhi >> (i - 64))) & 1ull), idx);
        };
        auto frag = [&](float run, int z) { return pa_charge_mz(__dsub_rn(__dadd_rn((double)run, a1), a2), z); };
        // d = first step whose residue differs between the two isoforms
        int d;
        {
            const uint64_t xlo = alo ^ blo, xhi = ahi ^ bhi;
            const int p_first = xlo ? __ffsll((long long)xlo) - 1 : (xhi ? 63 + __ffsll((long long)xhi) : 128);
            const int p_last = xhi ? 127 - __clzll((long long)xhi) : (xlo ? 63 - __clzll((long long)xlo) : -1);
            d = fwd ? p_first : L - 1 - p_last;
            if (!(cfg.err > 0.f)) d = 0;                 // nothing is ever dropped: no shortcut
            d = d < 0 ? 0 : (d > steps ? steps : d);
        }
        // float32 running sum over the common steps [0, d)
        float runc = 0.f;
        for (int s = 0; s < d; s++) {
            const float r = res_at(s, alo, ahi);
            const float nr = (s == 0) ? r : __fadd_rn(r, runc);
            if (s > 0 && nr < runc) mono = false;
            runc = nr;
        }
        if (d >= steps) return mono;                     // every walked residue is common: all fragments drop
        float runAd = res_at(d, alo, ahi), runBd = res_at(d, blo, bhi);
        if (d > 0) {
            runAd = __fadd_rn(runAd, runc); runBd = __fadd_rn(runBd, runc);
            if (runAd < runc || runBd < runc) mono = false;
        }
        float T = PINF;
#pragma unroll
        for (int z = 0; z < NQ; z++)
            if (z < Z) { const float va = frag(runAd, z + 1), vb = frag(runBd, z + 1); T = fminf(T, fminf(va, vb)); }
#pragma unroll
        for (int z = 0; z < NQ; z++) {
            runA[z] = runAd; runB[z] = runBd; stepA[z] = d; stepB[z] = d;
            valA[z] = (z < Z) ? frag(runAd, z + 1) : PINF;
            valB[z] = (z < Z) ? frag(runBd, z + 1) : PINF;
        }
        if (NQ > 1 && d > 0 && Z > 1) {
            // a lower charge reaches T at an earlier (common) step: start its streams there
            unsigned open = (1u << Z) - 1u;              // streams not yet started
            float run = 0.f;
            for (int s = 0; s < d && open; s++) {
                const float r = res_at(s, alo, ahi);
                run = (s == 0) ? r : __fadd_rn(r, run);
#pragma unroll
                for (int z = 0; z < NQ; z++) {
                    if ((open >> z) & 1u) {
                        const float v = frag(run, z + 1);
                        if (v >= T) {
                            runA[z] = run; runB[z] = run; stepA[z] = s; stepB[z] = s; valA[z] = v; valB[z] = v;
                            open &= ~(1u << z);
                        }
                    }
                }
            }
        }
        int leftA = 0;
#pragma unroll
        for (int z = 0; z < NQ; z++) if (z < Z) leftA += steps - stepA[z];
        int leftB = leftA;
        for (;;) {
            if (!hx && leftA > 0) {
                int bq = 0;
                float xm = valA[0], runb = runA[0];
                int stepb = stepA[0];
#pragma unroll
                for (int i = 1; i < NQ; i++)
                    if (valA[i] < xm) { xm = valA[i]; bq = i; runb = runA[i]; stepb = stepA[i]; }
                const int step = stepb + 1;
                float nv = PINF, run = runb;
                if (step < steps) {
                    run = __fadd_rn(res_at(step, alo, ahi), runb);
                    nv = frag(run, bq + 1);
                    if (nv < xm) mono = false;
                }
#pragma unroll
                for (int i = 0; i < NQ; i++)
                    if (i == bq) { runA[i] = run; stepA[i] = step; valA[i] = nv; }
                x = xm; hx = true; leftA--;
            }
            if (!hy && leftB > 0) {
                int bq = 0;
                float xm = valB[0], runb = runB[0];
                int stepb = stepB[0];
#pragma unroll
                for (int i = 1; i < NQ; i++)
                    if (valB[i] < xm) { xm = valB[i]; bq = i; runb = runB[i]; stepb = stepB[i]; }
                const int step = stepb + 1;
                float nv = PINF, run = runb;
                if (step < steps) {
                    run = __fadd_rn(res_at(step, blo, bhi), runb);
                    nv = frag(run, bq + 1);
                    if (nv < xm) mono = false;
                }
#pragma unroll
                for (int i = 0; i < NQ; i++)
                    if (i == bq) { runB[i] = run; stepB[i] = step; valB[i] = nv; }
                y = xm; hy = true; leftB--;
            }
            if (!hx && !hy) break;
            int takeA;                       // 1: A survives, 0: B survives, -1: both dropped
            if (!hy) takeA = 1;
            else if (!hx) takeA = 0;
            else if (fabsf(__fsub_rn(x, y)) < cfg.err) takeA = -1;
            else takeA = x < y;
            if (takeA < 0) { hx = false; hy = false; }
            else {
                asc_survivor(cfg, pk, depth, takeA ? x : y, takeA != 0, hitsA, trialsA, hitsB, trialsB);
                if (takeA) hx = false; else hy = false;
            }
        }
        return mono;
    } else {
        return asc_merge_streams(cfg, q, pk, fwd, a1, a2, alo, ahi, blo, bhi, depth, hitsA, trialsA, hitsB, trialsB);
    }
}

// residue index of modifiable site `u` (sites count the modifiable residues N->C)
__device__ __forceinline__ int asc_site_pos(const PaCfg& cfg, const AscPep& q, int u) {
    int n = 0;
    for (int i = 0; i < q.L; i++) {
        const int c = (int)q.pep[i] - 'A';
        const bool is = ((cfg.mod_letters >> c) & 1u) || (cfg.allow_n && i == 0) || (cfg.allow_c && i == q.L - 1);
        if (is) { if (n == u) return i; n++; }
    }
    return 0;
}

// One launch per stream class (0: one charge, 1: two, 2: up to four, 3: neutral losses or more
// charges), so that each instantiation gets its own register budget and occupancy.
#ifndef PA_ASC_MINBLOCKS
#define PA_ASC_MINBLOCKS 8
#endif
#ifndef PA_ASC2_MINBLOCKS
#define PA_ASC2_MINBLOCKS 8
#endif
#ifndef PA_ASC4_MINBLOCKS
#define PA_ASC4_MINBLOCKS 4
#endif
#ifndef PA_ASC12_MINBLOCKS
#define PA_ASC12_MINBLOCKS 4
#endif
#include "pa_ascore.cuh"

// K3c: generic (warp-cooperative, list-materialising) Ascore for the entries k_ascore queued.  DEEP: n_top > 10 (see
// asc_pair); `deep` comes last so that the parameters of the n_top = 10 form keep their offsets.
template <bool DEEP>
__global__ void __launch_bounds__(256) k_ascore_generic(PaCfg cfg, PaBatchDev b, PaAscArgs a, float* g_lists,
                                                         int64_t list_stride, PaDeep deep) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    SelSmem* sm = (SelSmem*)smem_raw + wib;
    const int64_t gw = (int64_t)blockIdx.x * wpb + wib, nw = (int64_t)gridDim.x * wpb;
    const int n = *a.generic_count;
    for (int64_t e = gw; e < n; e += nw) {
        const int64_t t = a.generic_list[e];
        const int32_t p = a.mod_psm[t];
        const int j = (int)(a.mod_lo + t - a.mod_off[p]);
        const int S = a.psm_S[p], k = b.n_mod[p];
        const int64_t ib = a.iso_off[p];
        PsmInfo info;
        pa_setup_psm(cfg, b, p, &sm->psm, info, true);
        const uint32_t best = a.best_idx[p];
        const uint64_t best_bits = pa_unrank(cfg.binom, S, k, best);
        uint64_t rem = best_bits;
        for (int jj = 0; jj < j; jj++) rem &= rem - 1;
        const int site = __ffsll((long long)rem) - 1;
        float scBest[DEEP ? PA_MAX_N_TOP : PA_N_TOP];
        pa_depth_scores(cfg, a.iso.lo[ib + best], a.iso.hi[ib + best], (int)a.iso.nfrag[ib + best], scBest);
        if (DEEP) pa_deep_scores(deep, ib + best, (int)a.iso.nfrag[ib + best], scBest);
        const float wbest = a.iso.w[ib + best];
        float* raw0 = sm->raw[0]; float* raw1 = sm->raw[1]; float* srt0 = sm->srt[0]; float* srt1 = sm->srt[1];
        long long per_type = (long long)(info.L > 1 ? info.L - 1 : 1) * cfg.nvar_cap * info.Z;
        if (per_type > PA_LCAP) {     // list_stride = power of two >= the chunk's longest list
            float* g = g_lists + (size_t)gw * 4 * list_stride;
            raw0 = g; raw1 = g + list_stride; srt0 = g + 2 * list_stride; srt1 = g + 3 * list_stride;
        }
        float asc = __int_as_float(0x7f800000);
        for (uint64_t tt = a.tie[t]; tt; tt &= tt - 1) {
            const int u = __ffsll((long long)tt) - 1;
            const uint64_t cb = (best_bits & ~(1ull << site)) | (1ull << u);
            const uint32_t ci = pa_rank(cfg.binom, S, k, cb);
            float scC[DEEP ? PA_MAX_N_TOP : PA_N_TOP];
            pa_depth_scores(cfg, a.iso.lo[ib + ci], a.iso.hi[ib + ci], (int)a.iso.nfrag[ib + ci], scC);
            if (DEEP) pa_deep_scores(deep, ib + ci, (int)a.iso.nfrag[ib + ci], scC);
            const float amb = pa_ambiguity<DEEP>(cfg, sm, info, best_bits, scBest, wbest, cb, scC, a.iso.w[ib + ci],
                                                 raw0, raw1, srt0, srt1, deep);
            asc = amb < asc ? amb : asc;
        }
        if (lane == 0 && a.ascores) a.ascores[a.mod_lo + t] = asc;
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------------
// export of one PSM's per-isoform table (pep_scores) and a stand-alone ambiguity call
// ---------------------------------------------------------------------------------------------
// counts / scores rows are n_top = 10 + dp.nd wide
__global__ void k_export_psm(PaCfg cfg, int64_t ib, int64_t I, int S, int k, PaIso iso, uint64_t* sig,
                             int32_t* counts, float* scores, float* weighted, int32_t* total, PaDeep dp) {
    int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= I) return;
    unsigned long long lo = iso.lo[ib + q], hi = iso.hi[ib + q];
    int n = (int)iso.nfrag[ib + q];
    const int w = PA_N_TOP + dp.nd;
    sig[q] = pa_unrank(cfg.binom, S, k, (uint32_t)q);
    for (int d = 0; d < w; d++) {
        int c = d < PA_N_TOP ? pa_cum_get(lo, hi, d) : dp.cnt[(size_t)(ib + q) * dp.nd + (d - PA_N_TOP)];
        counts[q * w + d] = c;
        scores[q * w + d] = pa_depth_score(cfg.T, dp, n, c, d);
    }
    weighted[q] = iso.w[ib + q];
    total[q] = n;
}

struct PaAmbArgs {
    int64_t psm;
    uint64_t sigA, sigB;
    float scA[PA_MAX_N_TOP], scB[PA_MAX_N_TOP];   // n_top entries
    float wA, wB;
    float* out;
    float* g_lists;
    int64_t list_stride;
    PaDeep deep;                                   // nd = 0 for n_top = 10
};

__global__ void __launch_bounds__(32) k_ambiguity(PaCfg cfg, PaBatchDev b, PaAmbArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SelSmem* sm = (SelSmem*)smem_raw;
    PsmInfo info;
    pa_setup_psm(cfg, b, a.psm, &sm->psm, info, true);
    float* raw0 = sm->raw[0]; float* raw1 = sm->raw[1]; float* srt0 = sm->srt[0]; float* srt1 = sm->srt[1];
    long long per_type = (long long)(info.L > 1 ? info.L - 1 : 1) * cfg.nvar_cap * info.Z;
    if (per_type > PA_LCAP) {
        float* g = a.g_lists;
        raw0 = g; raw1 = g + a.list_stride; srt0 = g + 2 * a.list_stride; srt1 = g + 3 * a.list_stride;
    }
    float r = pa_ambiguity<true>(cfg, sm, info, a.sigA, a.scA, a.wA, a.sigB, a.scB, a.wB, raw0, raw1, srt0, srt1, a.deep);
    if ((threadIdx.x & 31) == 0) *a.out = r;
}
