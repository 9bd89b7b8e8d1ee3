// Device-side building blocks shared by the kernels of libpyascore_b200.
//
// Everything here follows the bit-exact semantic spec in SURVEY.md section 7.3: float32 operations are
// written with explicit round-to-nearest intrinsics (and the library is compiled with
// -fmad=false), double is used exactly where the reference promotes to double.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pyascore_b200.h"

#define PA_LMAX 128          // smem rows per peptide (PA_MAX_PEPTIDE + 2)
#define PA_RCAP 255          // retained peaks staged in shared memory per PSM (else read from global)
#define PA_NCELL 256         // m/z cells of the per-PSM peak index (first peak at or after each cell)
#define PA_UNIT 1024         // isoforms per K2 work unit
#define PA_FULL 0xffffffffu

struct PaCfg {
    float bin_size, mod_mass, err;
    int n_top;
    uint32_t mod_letters;            // bit (c-'A') set: residue c takes the variable mod
    int allow_n, allow_c;            // 'n' / 'c' in mod_group (cpp/ModifiedPeptide.cpp:44-46)
    int n_types;
    char types[8];                   // fragment_types, in the caller's order
    int has_nl;                      // any neutral loss configured
    uint8_t nl_upper[26], nl_lower[26];  // 0 = none, else 1-based index of the distinct loss mass
    float res_mass[26];              // cpp/Types.h:7-30; NaN = unknown letter
    uint32_t known_letters;          // bit (c-'A') set: res_mass[c] is a number (register test instead of a gather)
    float weights[PA_N_TOP];         // cpp/Ascore.cpp:15-19
    int err_gt_half;                 // mz_error > 0.5: the lower_bound(mz - .5) clause can bind
    int nvar_cap;                    // max neutral-loss variants per residue for this scorer
    // device tables
    const float* T;                  // score table [(n(n+1)/2 + k) * 10 + d]
    int table_n;                     // rows 0..table_n available
    const uint32_t* binom;           // saturating C(n,k), [64*64]
    const float* nl_sums;            // [256][16] sorted distinct <=2-subset sums per capped-count state
    const uint8_t* nl_nvar;          // [256]
    const float* res_tab;            // global copies of res_mass / nl_upper / nl_lower for per-lane gathers
    const uint8_t* nl_up_tab;        // (kernel parameters sit in the constant bank: divergent indices serialise)
    const uint8_t* nl_lo_tab;
};

// ---------------------------------------------------------------------------------------------
// glibc 2.39 expf / logf, restated.  The reference's log_sum (cpp/Util.cpp:16-26) calls libm's
// float exp/log, which are not correctly rounded; to get the same float32 tail table as the
// CPU reference the GPU evaluates glibc's algorithm itself: double-precision table + cubic,
// sysdeps/ieee754/flt-32/e_expf.c and e_logf.c (ARM optimized-routines), in the FMA-contracted
// form x86-64 libm selects on FMA hardware.  Checked against libm for every float in
// [-104.5, 89] (expf) and every positive normal float (logf): 0 mismatches (DESIGN.md).
// The constants are glibc's __exp2f_data / __logf_data tables.
// ---------------------------------------------------------------------------------------------
__constant__ uint64_t c_exp2f_tab[32] = {
    0x3ff0000000000000ull, 0x3fefd9b0d3158574ull, 0x3fefb5586cf9890full, 0x3fef9301d0125b51ull,
    0x3fef72b83c7d517bull, 0x3fef54873168b9aaull, 0x3fef387a6e756238ull, 0x3fef1e9df51fdee1ull,
    0x3fef06fe0a31b715ull, 0x3feef1a7373aa9cbull, 0x3feedea64c123422ull, 0x3feece086061892dull,
    0x3feebfdad5362a27ull, 0x3feeb42b569d4f82ull, 0x3feeab07dd485429ull, 0x3feea47eb03a5585ull,
    0x3feea09e667f3bcdull, 0x3fee9f75e8ec5f74ull, 0x3feea11473eb0187ull, 0x3feea589994cce13ull,
    0x3feeace5422aa0dbull, 0x3feeb737b0cdc5e5ull, 0x3feec49182a3f090ull, 0x3feed503b23e255dull,
    0x3feee89f995ad3adull, 0x3feeff76f2fb5e47ull, 0x3fef199bdd85529cull, 0x3fef3720dcef9069ull,
    0x3fef5818dcfba487ull, 0x3fef7c97337b9b5full, 0x3fefa4afa2a490daull, 0x3fefd0765b6e4540ull};

__constant__ double c_logf_tab[16][2] = {
    {0x1.661ec79f8f3bep+0, -0x1.57bf7808caadep-2}, {0x1.571ed4aaf883dp+0, -0x1.2bef0a7c06ddbp-2},
    {0x1.49539f0f010bp+0, -0x1.01eae7f513a67p-2},  {0x1.3c995b0b80385p+0, -0x1.b31d8a68224e9p-3},
    {0x1.30d190c8864a5p+0, -0x1.6574f0ac07758p-3}, {0x1.25e227b0b8eap+0, -0x1.1aa2bc79c81p-3},
    {0x1.1bb4a4a1a343fp+0, -0x1.a4e76ce8c0e5ep-4}, {0x1.12358f08ae5bap+0, -0x1.1973c5a611cccp-4},
    {0x1.0953f419900a7p+0, -0x1.252f438e10c1ep-5}, {0x1p+0, 0x0p+0},
    {0x1.e608cfd9a47acp-1, 0x1.aa5aa5df25984p-5},  {0x1.ca4b31f026aap-1, 0x1.c5e53aa362eb4p-4},
    {0x1.b2036576afce6p-1, 0x1.526e57720db08p-3},  {0x1.9c2d163a1aa2dp-1, 0x1.bc2860d22477p-3},
    {0x1.886e6037841edp-1, 0x1.1058bc8a07ee1p-2},  {0x1.767dcf5534862p-1, 0x1.4043057b6ee09p-2}};

__device__ __forceinline__ float pa_expf(float x) {
    if (x < -0x1.9fe368p6f) return 0.0f;                 // __math_uflowf
    if (x > 0x1.62e42ep6f) return __int_as_float(0x7f800000);
    const double InvLn2N = 0x1.71547652b82fep+5, Shift = 0x1.8p+52;
    const double C0 = 0x1.c6af84b912394p-20, C1 = 0x1.ebfce50fac4f3p-13, C2 = 0x1.62e42ff0c52d6p-6;
    double xd = (double)x;
    double kd = fma(InvLn2N, xd, Shift);
    uint64_t ki = (uint64_t)__double_as_longlong(kd);
    kd = __dsub_rn(kd, Shift);
    double r = fma(InvLn2N, xd, -kd);
    uint64_t t = c_exp2f_tab[ki & 31];
    t += ki << (52 - 5);
    double s = __longlong_as_double((long long)t);
    double p = fma(C0, r, C1);
    double r2 = __dmul_rn(r, r);
    double y = fma(C2, r, 1.0);
    y = fma(p, r2, y);
    y = __dmul_rn(y, s);
    return __double2float_rn(y);
}

__device__ __forceinline__ float pa_logf(float x) {      // x positive, normal
    uint32_t ix = (uint32_t)__float_as_int(x);
    if (ix == 0x3f800000u) return 0.f;
    const double Ln2 = 0x1.62e42fefa39efp-1;
    const double A0 = -0x1.00ea348b88334p-2, A1 = 0x1.5575b0be00b6ap-2, A2 = -0x1.ffffef20a4123p-2;
    uint32_t tmp = ix - 0x3f330000u;
    int i = (tmp >> 19) & 15;
    int k = (int32_t)tmp >> 23;
    uint32_t iz = ix - (tmp & 0xff800000u);
    double invc = c_logf_tab[i][0], logc = c_logf_tab[i][1];
    double z = (double)__int_as_float((int)iz);
    double r = fma(z, invc, -1.0);
    double y0 = fma((double)k, Ln2, logc);
    double r2 = __dmul_rn(r, r);
    double y = fma(A1, r, A2);
    y = fma(A0, r2, y);
    y = fma(y, r2, __dadd_rn(y0, r));
    return __double2float_rn(y);
}

// cpp/Util.cpp:16-26
__device__ __forceinline__ float pa_log_sum(float a, float b) {
    if (isinf(a)) return b;
    if (isinf(b)) return a;
    float m = (a < b) ? b : a;
    float t = pa_logf(__fadd_rn(pa_expf(__fsub_rn(a, m)), pa_expf(__fsub_rn(b, m))));
    return __fadd_rn(m, t);
}

// ---------------------------------------------------------------------------------------------
// combinatorics: lexicographic k-subsets of S sites (site 0 = most N-terminal)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pa_binom(const uint32_t* __restrict__ tab, int n, int k) {
    if (k < 0 || n < 0 || k > n) return 0u;
    return __ldg(tab + n * 64 + k);
}

// idx-th subset in lexicographic order -> bit mask (bit j = site j)
__device__ __forceinline__ uint64_t pa_unrank(const uint32_t* __restrict__ tab, int S, int k, uint32_t idx) {
    uint64_t bits = 0;
    int c = 0;
    uint32_t r = idx;
    for (int i = 0; i < k; i++) {
        for (;;) {
            uint32_t cnt = pa_binom(tab, S - 1 - c, k - 1 - i);
            if (r < cnt) break;
            r -= cnt;
            c++;
        }
        bits |= 1ull << c;
        c++;
    }
    return bits;
}

// lexicographic rank of a k-subset.  The subsets that precede `bits` and first differ at its
// i-th element c_i are those whose i-th element lies in (c_{i-1}, c_i): by the hockey-stick
// identity their number is C(S-1-c_{i-1}, k-i) - C(S-c_i, k-i).
__device__ __forceinline__ uint32_t pa_rank(const uint32_t* __restrict__ tab, int S, int k, uint64_t bits) {
    uint32_t r = 0;
    int prev = -1, i = 0;
    while (bits) {
        int c = __ffsll((long long)bits) - 1;
        bits &= bits - 1;
        r += pa_binom(tab, S - 1 - prev, k - i) - pa_binom(tab, S - c, k - i);
        prev = c;
        i++;
    }
    return r;
}

// ---------------------------------------------------------------------------------------------
// per-PSM tables in shared memory (one slot per warp)
// ---------------------------------------------------------------------------------------------
struct PsmSmem {
    float res[PA_LMAX][2];        // residue mass: [i][0] plain, [i][1] with the variable mod
    uint8_t nlidx[PA_LMAX][2];    // neutral-loss index per state (0 = none)
    uint8_t site_pos[64];         // residue index of site j
    float2 pk[PA_RCAP + 2];       // retained peaks {(float)mz ascending, rank as int bits}; pk[R] = {+inf, 255}, pk[R + 1] readable
    alignas(8) uint8_t cell[PA_NCELL];  // cell[c] = index of the first peak whose cell is >= c
};

struct PsmInfo {
    int L, k, Z, S, R;
    int status;
    const float2* gp;             // global peaks {mz, rank bits} (used when they are not staged: cell == nullptr)
    const float2* pk;             // staged peaks in shared memory (cell != nullptr)
    const uint8_t* cell;          // -> smem cell index, or nullptr (binary search over global peaks)
    float cell_base, cell_inv;    // cell(x) = clamp(floor((x - base) * inv), 0, PA_NCELL-1)
};

// cell width = power of two such that [first peak, last peak] spans fewer than PA_NCELL cells
__device__ __forceinline__ float pa_cell_inv(float first, float last) {
    const float range = __fsub_rn(last, first);
    int e = 0;
    if (range > 0.f) e = ilogbf(__fmul_rn(range, 1.0f / PA_NCELL)) + 1;
    e = e < -20 ? -20 : (e > 60 ? 60 : e);
    return ldexpf(1.0f, -e);
}

__device__ __forceinline__ int pa_cell(float x, float base, float inv) {
    // (round-down conversion, saturating, NaN -> 0: the same cell as floorf + float clamps for every input, one instruction less)
    const int c = __float2int_rd(__fmul_rn(__fsub_rn(x, base), inv));
    return min(max(c, 0), PA_NCELL - 1);
}

struct PaBatchDev {               // device views of one chunk
    const int64_t* spec_off;
    const int32_t* psm_spec;
    const int32_t* pep_off;
    const uint8_t* pep;
    const int32_t* n_mod;
    const int32_t* max_charge;
    const int32_t* aux_off;       // may be null
    const uint32_t* aux_pos;
    const float* aux_mass;
    const float2* rpk;            // K1 output, indexed with spec_off: retained peaks {(float)mz ascending, rank as int bits}
    const int32_t* rcount;
    const uint8_t* ctab;          // per spectrum PA_NCELL bytes: first retained peak at or after each m/z cell
    const float2* chead;          // per spectrum {cell base, 1/cell width}; width 0 = no table (binary search)
    int64_t spec_base;            // spec_off values are relative to this peak index
    int64_t n_spec;
};

__device__ __forceinline__ void pa_cp_async8(void* smem_dst, const void* gsrc) {
    unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(d), "l"(gsrc) : "memory");
}

// Build the residue / neutral-loss / site tables of PSM p and stage its retained peaks.
// cpp/ModifiedPeptide.cpp:24-57 (initializeResidues), :59-79 (applyAuxMods).
// Must be called by all 32 lanes of a warp.
__device__ __forceinline__ void pa_setup_psm(const PaCfg& cfg, const PaBatchDev& b, int64_t p, PsmSmem* sm,
                                             PsmInfo& info, bool want_peaks) {
    const int lane = threadIdx.x & 31;
    const int o = b.pep_off[p];
    const int L = b.pep_off[p + 1] - o;
    info.L = L;
    info.k = b.n_mod[p];
    info.Z = b.max_charge[p];
    int S = 0;
    __syncwarp();
    // the retained peaks and the spectrum's m/z cell index travel global -> shared asynchronously while
    // the residue tables are built (K1 stores the peaks in the staged {mz, rank} form)
    bool staged = false;
    if (want_peaks) {
        const int sp = b.psm_spec[p];
        const int64_t off = b.spec_off[sp] - b.spec_base;
        const int R = b.rcount[sp];
        const float2 head = b.chead[sp];
        info.R = R;
        info.gp = b.rpk + off;
        info.cell_base = head.x;
        info.cell_inv = head.y;
        staged = R <= PA_RCAP && head.y != 0.f;
        if (staged) {
            for (int i = lane; i < R; i += 32) pa_cp_async8(&sm->pk[i], b.rpk + off + i);
            // (pa_cell is monotone in x, so every peak before cell[pa_cell(lo)] is <= lo)
            pa_cp_async8((unsigned long long*)sm->cell + lane, (const unsigned long long*)(b.ctab + (size_t)sp * PA_NCELL) + lane);
            asm volatile("cp.async.commit_group;\n" ::: "memory");
            if (lane == 0) sm->pk[R] = make_float2(__int_as_float(0x7f800000), __int_as_float(255));   // sentinel
        }
    }
    for (int base = 0; base < L; base += 32) {
        int i = base + lane;
        bool site = false;
        if (i < L) {
            int c = (int)b.pep[o + i] - 'A';
            float m0 = (c >= 0 && c < 26) ? __ldg(cfg.res_tab + c) : __int_as_float(0x7fc00000);
            bool lett = (c >= 0 && c < 26) && ((cfg.mod_letters >> c) & 1u);
            site = lett || (cfg.allow_n && i == 0) || (cfg.allow_c && i == L - 1);
            sm->res[i][0] = m0;
            sm->res[i][1] = site ? __fadd_rn(m0, cfg.mod_mass) : 0.f;
            uint8_t n0 = 0, n1 = 0;
            if (cfg.has_nl && c >= 0 && c < 26) { n0 = __ldg(cfg.nl_up_tab + c); n1 = site ? __ldg(cfg.nl_lo_tab + c) : 0; }
            sm->nlidx[i][0] = n0;
            sm->nlidx[i][1] = n1;
        }
        unsigned bal = __ballot_sync(PA_FULL, site);
        if (site) {
            int j = S + __popc(bal & ((1u << lane) - 1u));
            if (j < 64) sm->site_pos[j] = (uint8_t)i;
        }
        S += __popc(bal);
    }
    info.S = S;
    __syncwarp();
    // fixed mods, applied in the caller's order (float adds do not commute bit-exactly)
    if (b.aux_off != nullptr && lane == 0) {
        int a0 = b.aux_off[p], a1 = b.aux_off[p + 1];
        for (int a = a0; a < a1; a++) {
            uint32_t pos = b.aux_pos[a];
            int idx = pos > 0 ? (int)pos - 1 : 0;
            if (idx >= L) continue;                       // flagged PA_PSM_BAD_AUX by the planner
            float am = b.aux_mass[a];
            // both states take the fixed mod (state 1 only exists for modifiable residues)
            int c = (int)b.pep[o + idx] - 'A';
            bool lett = (c >= 0 && c < 26) && ((cfg.mod_letters >> c) & 1u);
            bool site = lett || (cfg.allow_n && idx == 0) || (cfg.allow_c && idx == L - 1);
            sm->res[idx][0] = __fadd_rn(sm->res[idx][0], am);
            if (site) sm->res[idx][1] = __fadd_rn(sm->res[idx][1], am);
            if (cfg.has_nl && c >= 0 && c < 26 && cfg.nl_lower[c]) {
                // cpp/ModifiedPeptide.cpp:73-77: the residue's loss list becomes [lower-case loss];
                // the reference then reads out of bounds for state 1 -- we give it the same loss
                sm->nlidx[idx][0] = cfg.nl_lower[c];
                sm->nlidx[idx][1] = cfg.nl_lower[c];
            }
        }
    }
    __syncwarp();
    if (want_peaks) {
        if (staged) {
            asm volatile("cp.async.wait_group 0;\n" ::: "memory");
            info.pk = sm->pk;
            info.cell = sm->cell;
        } else {
            info.pk = nullptr;
            info.cell = nullptr;
            info.cell_base = 0.f;
            info.cell_inv = 0.f;
        }
        __syncwarp();
    }
}

// rank of the best (most intense) retained peak matching theoretical fragment f, or 255.
// cpp/ModifiedPeptide.cpp:126-142 seen from the fragment's side (SURVEY.md section 7.3 "Matching").
template <bool EGH = true>
__device__ __forceinline__ int pa_match_rank(const PsmInfo& info, float f, float err, int err_gt_half_rt) {
    const bool err_gt_half = EGH && err_gt_half_rt;      // EGH = false: mz_error <= 0.5, the clause cannot bind
    const float lo = __fsub_rn(f, err), hi = __fadd_rn(f, err);
    int best = 255;
    if (info.cell != nullptr) {
        // staged peaks: every peak before cell[pa_cell(lo)] is <= lo; peaks <= lo inside the cell
        // are passed over by the same loop (they are < hi), and the +inf sentinel at pk[R] ends it
        const float2* pk = info.pk + info.cell[pa_cell(lo, info.cell_base, info.cell_inv)];
        // the first two candidates are fetched together (most scans end on the second): pk[R + 1] is readable
        float2 e = pk[0], e_next = pk[1];
        for (;;) {
            if (!(e.x < hi)) break;
            if (e.x > lo && !(err_gt_half && !((double)f >= (double)e.x - .5))) {
                const int r = __float_as_int(e.y);
                best = r < best ? r : best;
            }
            pk++;
            e = e_next;
            if (!(e.x < hi)) break;      // (tested before the next fetch: the entry after the +inf sentinel is never read)
            e_next = pk[1];
        }
        return best;
    }
    const float2* gp = info.gp;
    const int R = info.R;
    int a = 0;
    int n = R;                          // first index with mz > lo
    while (n > 0) {
        int h = n >> 1;
        if (!(gp[a + h].x > lo)) { a += h + 1; n -= h + 1; } else n = h;
    }
    for (; a < R; a++) {
        const float2 e = gp[a];
        if (!(e.x < hi)) break;
        if (err_gt_half && !((double)f >= (double)e.x - .5)) continue;
        const int r = __float_as_int(e.y);
        best = r < best ? r : best;
    }
    return best;
}

// cpp/ModifiedPeptide.cpp:570-591
__device__ __forceinline__ double pa_type_adjust(double d, char type) {
    if (type == 'y') d = __dadd_rn(d, 18.010565);
    else if (type == 'z') { d = __dadd_rn(d, 18.010565); d = __dsub_rn(d, 17.026549); }
    else if (type == 'Z') { d = __dadd_rn(d, 18.010565); d = __dsub_rn(d, 16.018724); }
    else if (type == 'c') d = __dadd_rn(d, 17.026549);
    return d;
}

// z * 1.007825 for z < 16, filled by the host in IEEE double (the product the reference forms)
__constant__ double c_zmass[16];

__device__ __forceinline__ float pa_charge_mz(double d, int z) {
    // (d + z * 1.007825) / z  (cpp/ModifiedPeptide.cpp:585-587).  Dividing by 1, 2 or 4 is exact
    // scaling, so the IEEE division routine is only needed for the other charges.
    if (z > 0) {
        const double t = __dadd_rn(d, z < 16 ? c_zmass[z] : __dmul_rn((double)z, 1.007825));
        if (z == 1) d = t;
        else if (z == 2) d = __dmul_rn(t, 0.5);
        else if (z == 4) d = __dmul_rn(t, 0.25);
        else d = __ddiv_rn(t, (double)z);
    }
    return __double2float_rn(d);
}

// branch-free form of pa_type_adjust: d + A1 - A2 with A = 0 where the reference does nothing
// (x + 0.0 and x - 0.0 are exact, so the bits are those of the branched form)
__device__ __forceinline__ void pa_type_consts(char type, double& a1, double& a2) {
    a1 = 0.; a2 = 0.;
    if (type == 'y') a1 = 18.010565;
    else if (type == 'z') { a1 = 18.010565; a2 = 17.026549; }
    else if (type == 'Z') { a1 = 18.010565; a2 = 16.018724; }
    else if (type == 'c') a1 = 17.026549;
}

__device__ __forceinline__ int pa_nl_bump(int state, int idx) {   // idx 1-based
    int sh = 2 * (idx - 1);
    int f = (state >> sh) & 3;
    return state + ((f < 2) << sh);
}

__device__ __forceinline__ size_t pa_tab_index(int n, int k, int d) {
    return ((size_t)n * (size_t)(n + 1) / 2 + (size_t)k) * PA_N_TOP + (size_t)d;
}

// Depths 10 .. n_top-1 of a scorer with n_top > 10.  The score table of those depths is a second table beside T, with
// the same rows: T_deep[(n(n+1)/2 + k) * nd + (d - 10)], nd = n_top - 10.  Per isoform of a chunk, K2d stores the
// cumulative counts of those depths: cnt[(iso_off[p] + idx) * nd + (d - 10)].  nd = 0: a scorer of n_top = 10.
struct PaDeep {
    const float* T;
    const uint16_t* cnt;
    int nd;
};

__device__ __forceinline__ size_t pa_tab_index_deep(int n, int k, int dd, int nd) {
    return ((size_t)n * (size_t)(n + 1) / 2 + (size_t)k) * (size_t)nd + (size_t)dd;
}

// score of depth d (0 .. n_top-1) at n trials and k hits
__device__ __forceinline__ float pa_depth_score(const float* T, const PaDeep& dp, int n, int k, int d) {
    return d < PA_N_TOP ? __ldg(T + pa_tab_index(n, k, d)) : __ldg(dp.T + pa_tab_index_deep(n, k, d - PA_N_TOP, dp.nd));
}
