/* TEST INFRASTRUCTURE ONLY -- CPU restatement ("oracle") of pyAscore's PTM-localisation
 * scoring path.  Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline /
 * --impl reference legs may load this; the product (pyascore_b200/) never does.
 *
 * This is NOT a copy of the reference: it is a deliberately naive re-derivation -- one
 * brute-force walk per positional isoform, no fragment graph, no hash maps of fragments --
 * written from the bit-exact semantic spec in SURVEY.md section 7.3.  Every function cites the
 * reference lines whose *results* it must reproduce (paths relative to
 * /root/reference/pyascore/ptm_scoring/).
 *
 * Parity status: PINNED.  tests/test_oracle_vs_ref.py (runs where oracle/_ref exists) and
 * tests/test_oracle_golden.py (committed vectors in tests/golden/, generated from the
 * compiled reference by tests/golden/make_golden.py) check this file against the
 * UNMODIFIED reference C++ bit for bit.
 *
 * Platform dependence reproduced on purpose (see SURVEY.md 0.4-0.6):
 *   - float32 arithmetic order, glibc expf/logf/log (we call the same libm),
 *   - libstdc++-13 unordered_map<long,...> iteration order (modelled in hash_order()),
 *   - libstdc++ std::sort = introsort + final insertion sort (ported in gcc_sort()).
 */
#include <ctype.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#define ORC_MAX_TOP 64
#define ORC_WEIGHTS 10

/* ------------------------------------------------------------------ residue masses */
/* cpp/Types.h:7-30 (values are narrowed to float there) */
static float residue_mass(char c, int *ok) {
    *ok = 1;
    switch (c) {
        case 'G': return 57.02146f;  case 'A': return 71.03711f;  case 'S': return 87.03203f;
        case 'P': return 97.05276f;  case 'V': return 99.06841f;  case 'T': return 101.04768f;
        case 'C': return 103.00919f; case 'L': return 113.08406f; case 'I': return 113.08406f;
        case 'N': return 114.04293f; case 'D': return 115.02694f; case 'Q': return 128.05858f;
        case 'K': return 128.09496f; case 'E': return 129.04259f; case 'M': return 131.04049f;
        case 'H': return 137.05891f; case 'F': return 147.06841f; case 'U': return 150.95364f;
        case 'R': return 156.10111f; case 'Y': return 163.06333f; case 'W': return 186.07931f;
        case 'O': return 237.14773f;
    }
    *ok = 0;
    return 0.f;
}

/* ------------------------------------------------------------------ binomial maths */
/* cpp/Util.cpp:16-26 */
static float f_log_sum(float a, float b) {
    if (isinf(a)) return b;
    if (isinf(b)) return a;
    float m = (a < b) ? b : a;
    float t = logf(expf(a - m) + expf(b - m));
    return m + t;
}

/* cpp/Util.cpp:28-41 */
static float f_log_bin_coef(size_t k, size_t n) {
    float coef = 0;
    if (n - k < k) k = n - k;
    for (size_t m = n - k + 1; m <= n; m++) coef = (float)((double)coef + log((double)m));
    for (size_t m = 2; m <= k; m++) coef = (float)((double)coef - log((double)m));
    return coef;
}

typedef struct {
    float lps, lpf;     /* cpp/Util.cpp:52-55 */
    float **rows;       /* rows[n][k] = log upper tail, k in 0..n+1; NULL until first use */
    size_t cap;
} orc_binom;

static void binom_init(orc_binom *b, float prob) {
    b->lps = logf(prob);
    b->lpf = (float)log(1. - (double)prob);
    b->rows = NULL;
    b->cap = 0;
}

static void binom_free(orc_binom *b) {
    for (size_t i = 0; i < b->cap; i++) free(b->rows[i]);
    free(b->rows);
    b->rows = NULL; b->cap = 0;
}

/* cpp/Util.cpp:57-59 */
static float binom_log_pmf(const orc_binom *b, size_t k, size_t n) {
    float r = f_log_bin_coef(k, n) + (float)k * b->lps;
    return r + (float)(n - k) * b->lpf;
}

/* cpp/Util.cpp:61-79.  The reference memoises (k,n) -> tail lazily from the top; every
 * entry is a pure function of (k,n), so filling the whole row at once is equivalent. */
static float binom_log_pvalue(orc_binom *b, size_t k, size_t n) {
    if (k == 0) return 0.f;
    if (n >= b->cap) {
        size_t nc = n + 64;
        b->rows = (float **)realloc(b->rows, nc * sizeof(float *));
        for (size_t i = b->cap; i < nc; i++) b->rows[i] = NULL;
        b->cap = nc;
    }
    if (!b->rows[n]) {
        float *r = (float *)malloc((n + 2) * sizeof(float));
        r[n + 1] = -INFINITY;
        for (size_t j = n; j >= 1; j--) r[j] = f_log_sum(r[j + 1], binom_log_pmf(b, j, n));
        r[0] = 0.f;
        b->rows[n] = r;
    }
    return b->rows[n][k];
}

/* cpp/Util.cpp:81-83 */
static float binom_log10_pvalue(orc_binom *b, size_t k, size_t n) {
    return (float)(log10(exp(1.0)) * (double)binom_log_pvalue(b, k, n));
}

/* |-10 * log10 p|, cpp/Ascore.cpp:127-133 and :202-206 */
static float binom_score(orc_binom *b, size_t k, size_t n) {
    return fabsf(-10.f * binom_log10_pvalue(b, k, n));
}

/* ------------------------------------------------------------------ the scorer object */
typedef struct {
    /* configuration: Ascore.pyx:64-73, cpp/ModifiedPeptide.cpp:15-20, :99-103 */
    float bin_size;
    int n_top;
    char mod_group[128];
    float mod_mass, mz_error;
    char frag_types[16];
    float nl_mass[256];
    unsigned char nl_has[256];
    orc_binom dist[ORC_MAX_TOP];
    int n_dist;
    float weights[ORC_WEIGHTS];

    /* retained peaks of the current spectrum */
    float *pk_mz;  double *pk_mz64, *pk_int; int *pk_rank, *pk_bin; int n_pk;
    float min_mz, max_mz; long n_bins;

    /* current peptide */
    char pep[1024]; int L; int k; int Z;
    float res[1024][2]; float nl[1024][2]; int modifiable[1024];
    int site_pos[1024]; int S;
    unsigned aux_pos[1024]; float aux_mass[1024]; int n_aux;

    /* results */
    long n_iso;
    uint64_t *key;       /* signature bits, N->C, first site = MSB (cpp/Ascore.cpp:91-94) */
    int32_t *counts;     /* n_iso x n_top cumulative */
    float *scores;       /* n_iso x n_top */
    float *weighted;
    int64_t *total;
    int n_asc; float asc[64]; int n_alt[64]; uint32_t alt[64][64];
} orc;

orc *orc_new(float bin_size, size_t n_top, const char *mod_group, float mod_mass, float mz_error,
             const char *fragment_types) {
    orc *o = (orc *)calloc(1, sizeof(orc));
    o->bin_size = bin_size;
    o->n_top = (int)n_top;
    strncpy(o->mod_group, mod_group, sizeof(o->mod_group) - 1);
    o->mod_mass = mod_mass;
    o->mz_error = mz_error;
    strncpy(o->frag_types, fragment_types, sizeof(o->frag_types) - 1);
    /* cpp/Ascore.cpp:15-19 */
    static const float w0[ORC_WEIGHTS] = {0.5f, 0.75f, 1.0f, 1.0f, 1.0f, 1.0f, 0.75f, 0.5f, 0.25f, 0.25f};
    double sum = 0.;
    for (int i = 0; i < ORC_WEIGHTS; i++) sum += w0[i];
    float fsum = (float)sum;
    for (int i = 0; i < ORC_WEIGHTS; i++) o->weights[i] = w0[i] / fsum;
    /* cpp/Ascore.cpp:23-36: p_d = 2 * err * d / 100. */
    o->n_dist = o->n_top < ORC_MAX_TOP ? o->n_top : ORC_MAX_TOP;
    for (int d = 1; d <= o->n_dist; d++) {
        float p = (float)((double)((2 * mz_error) * (float)d) / 100.);
        binom_init(&o->dist[d - 1], p);
    }
    return o;
}

static void free_results(orc *o) {
    free(o->key); free(o->counts); free(o->scores); free(o->weighted); free(o->total);
    o->key = NULL; o->counts = NULL; o->scores = NULL; o->weighted = NULL; o->total = NULL;
    o->n_iso = 0;
}

void orc_free(orc *o) {
    if (!o) return;
    for (int d = 0; d < o->n_dist; d++) binom_free(&o->dist[d]);
    free(o->pk_mz); free(o->pk_mz64); free(o->pk_int); free(o->pk_rank); free(o->pk_bin);
    free_results(o);
    free(o);
}

/* cpp/ModifiedPeptide.cpp:99-103 */
void orc_add_neutral_loss(orc *o, const char *group, float mass) {
    for (const char *c = group; *c; c++) { o->nl_mass[(unsigned char)*c] = mass; o->nl_has[(unsigned char)*c] = 1; }
}

/* ------------------------------------------------------------------ binning */
/* cpp/Spectra.cpp:43-68 (bounds, bin index) and :24-41 (top n_top per bin by intensity,
 * rank 0 = most intense).  Intensity ties are implementation-defined in the reference
 * (nth_element + unstable sort); here the earlier peak wins. */
void orc_consume_spectra(orc *o, const double *mz, const double *inten, size_t n) {
    free(o->pk_mz); free(o->pk_mz64); free(o->pk_int); free(o->pk_rank); free(o->pk_bin);
    o->pk_mz = (float *)malloc((n + 1) * sizeof(float));
    o->pk_mz64 = (double *)malloc((n + 1) * sizeof(double));
    o->pk_int = (double *)malloc((n + 1) * sizeof(double));
    o->pk_rank = (int *)malloc((n + 1) * sizeof(int));
    o->pk_bin = (int *)malloc((n + 1) * sizeof(int));
    o->n_pk = 0;
    if (n == 0) { o->n_bins = 0; return; }
    double lo = mz[0], hi = mz[0];
    for (size_t i = 1; i < n; i++) { if (mz[i] < lo) lo = mz[i]; if (mz[i] > hi) hi = mz[i]; }
    o->min_mz = (float)(floor(lo / 100.) * 100.);
    o->max_mz = (float)(ceil(hi / 100.) * 100.);
    o->n_bins = (long)ceilf((o->max_mz - o->min_mz) / o->bin_size);
    long nb = o->n_bins;
    long *bins = (long *)malloc(n * sizeof(long));
    for (size_t i = 0; i < n; i++) {
        double q = floor((mz[i] - (double)o->min_mz) / (double)o->bin_size);
        long b = (long)(size_t)q;
        if (b > nb - 1) b = nb - 1;
        bins[i] = b;
    }
    /* emit in (bin, rank) order like the reference's cursor walk (Ascore.pyx:142-150) */
    for (long b = 0; b < nb; b++) {
        for (int r = 0; r < o->n_top; r++) {
            /* r-th most intense of bin b: the peak with exactly r peaks ahead of it */
            long pick = -1;
            for (size_t i = 0; i < n && pick < 0; i++) {
                if (bins[i] != b) continue;
                int ahead = 0;
                for (size_t j = 0; j < n; j++) {
                    if (bins[j] != b || j == i) continue;
                    if (inten[j] > inten[i] || (inten[j] == inten[i] && j < i)) ahead++;
                }
                if (ahead == r) pick = (long)i;
            }
            if (pick < 0) break;
            o->pk_mz64[o->n_pk] = mz[pick];
            o->pk_mz[o->n_pk] = (float)mz[pick];
            o->pk_int[o->n_pk] = inten[pick];
            o->pk_rank[o->n_pk] = r;
            o->pk_bin[o->n_pk] = (int)b;
            o->n_pk++;
        }
    }
    free(bins);
}

/* faster variant used by the batch/timing entry: same result, per-bin selection sort */
static void consume_spectra_fast(orc *o, const double *mz, const double *inten, size_t n) {
    free(o->pk_mz); free(o->pk_mz64); free(o->pk_int); free(o->pk_rank); free(o->pk_bin);
    o->pk_mz = (float *)malloc((n + 1) * sizeof(float));
    o->pk_mz64 = (double *)malloc((n + 1) * sizeof(double));
    o->pk_int = (double *)malloc((n + 1) * sizeof(double));
    o->pk_rank = (int *)malloc((n + 1) * sizeof(int));
    o->pk_bin = (int *)malloc((n + 1) * sizeof(int));
    o->n_pk = 0;
    if (n == 0) { o->n_bins = 0; return; }
    double lo = mz[0], hi = mz[0];
    for (size_t i = 1; i < n; i++) { if (mz[i] < lo) lo = mz[i]; if (mz[i] > hi) hi = mz[i]; }
    o->min_mz = (float)(floor(lo / 100.) * 100.);
    o->max_mz = (float)(ceil(hi / 100.) * 100.);
    o->n_bins = (long)ceilf((o->max_mz - o->min_mz) / o->bin_size);
    long nb = o->n_bins;
    int T = o->n_top;
    long *top = (long *)malloc((size_t)nb * T * sizeof(long));   /* per bin: indices, best first */
    int *cnt = (int *)calloc((size_t)nb, sizeof(int));
    for (size_t i = 0; i < n; i++) {
        double q = floor((mz[i] - (double)o->min_mz) / (double)o->bin_size);
        long b = (long)(size_t)q;
        if (b > nb - 1) b = nb - 1;
        long *t = top + b * T;
        int c = cnt[b];
        /* insertion: strictly greater moves ahead; equal stays behind earlier index */
        int p = c;
        while (p > 0 && inten[i] > inten[t[p - 1]]) p--;
        if (p >= T) continue;
        int last = c < T ? c : T - 1;
        for (int q2 = last; q2 > p; q2--) t[q2] = t[q2 - 1];
        t[p] = (long)i;
        if (c < T) cnt[b] = c + 1;
    }
    for (long b = 0; b < nb; b++)
        for (int r = 0; r < cnt[b]; r++) {
            long pick = top[b * T + r];
            o->pk_mz64[o->n_pk] = mz[pick];
            o->pk_mz[o->n_pk] = (float)mz[pick];
            o->pk_int[o->n_pk] = inten[pick];
            o->pk_rank[o->n_pk] = r;
            o->pk_bin[o->n_pk] = (int)b;
            o->n_pk++;
        }
    free(top); free(cnt);
}

/* ------------------------------------------------------------------ peptide tables */
/* cpp/ModifiedPeptide.cpp:24-57 (residue / neutral-loss tables), :59-79 (fixed mods) */
int orc_consume_peptide(orc *o, const char *pep, size_t k, size_t Z, const unsigned *aux_pos,
                        const float *aux_mass, size_t n_aux) {
    int L = (int)strlen(pep);
    if (L <= 0 || L >= 1024) return -1;
    memcpy(o->pep, pep, L + 1);
    o->L = L; o->k = (int)k; o->Z = (int)Z;
    int has_n = strchr(o->mod_group, 'n') != NULL, has_c = strchr(o->mod_group, 'c') != NULL;
    o->S = 0;
    for (int i = 0; i < L; i++) {
        int ok;
        unsigned char c = (unsigned char)pep[i];
        o->res[i][0] = residue_mass(pep[i], &ok);
        if (!ok) return -2;
        o->nl[i][0] = o->nl_has[c] ? o->nl_mass[c] : 0.f;
        int m = (strchr(o->mod_group, pep[i]) != NULL) || (has_n && i == 0) || (has_c && i == L - 1);
        o->modifiable[i] = m;
        o->res[i][1] = 0.f; o->nl[i][1] = 0.f;
        if (m) {
            o->res[i][1] = o->res[i][0] + o->mod_mass;
            unsigned char lc = (unsigned char)tolower(c);
            o->nl[i][1] = o->nl_has[lc] ? o->nl_mass[lc] : 0.f;
            o->site_pos[o->S++] = i;
        }
    }
    o->n_aux = (int)n_aux;
    for (size_t a = 0; a < n_aux; a++) {
        o->aux_pos[a] = aux_pos[a]; o->aux_mass[a] = aux_mass[a];
        size_t idx = aux_pos[a];
        if (idx > 0) idx -= 1;
        if ((int)idx >= L) return -3;                 /* out of bounds in the reference */
        o->res[idx][0] += aux_mass[a];
        if (o->modifiable[idx]) o->res[idx][1] += aux_mass[a];
        unsigned char lc = (unsigned char)tolower((unsigned char)pep[idx]);
        if (o->nl_has[lc]) { o->nl[idx][0] = o->nl_mass[lc]; o->nl[idx][1] = o->nl_mass[lc]; /* [1] is UB there */ }
    }
    return 0;
}

/* ------------------------------------------------------------------ fragments of ONE isoform */
/* PowerSetSum(stack, 2): cpp/Util.cpp:99-123 -- subset sums of size <= 2 in the
 * reference's float evaluation order, sorted ascending, exact-equality de-duplicated. */
static int power_set_sums(const float *stack, int m, float *out /* cap >= 1+m+m(m-1)/2 */) {
    int n = 0;
    out[n++] = 0.f;
    for (int i = 0; i < m; i++) {
        float s1 = 0.f + stack[i];
        out[n++] = s1;
        if (m >= 2) for (int j = i + 1; j < m; j++) out[n++] = s1 + stack[j];
    }
    for (int i = 1; i < n; i++) {          /* insertion sort */
        float v = out[i]; int j = i;
        while (j > 0 && out[j - 1] > v) { out[j] = out[j - 1]; j--; }
        out[j] = v;
    }
    int u = 1;
    for (int i = 1; i < n; i++) if (out[i] != out[u - 1]) out[u++] = out[i];
    return u;
}

/* PowerSetSum::initializeSums for any max_depth (cpp/Util.cpp:99-107): children right after the
 * parent, each sum = parent + element; the test against max_depth - 1 is unsigned there, so a
 * max_depth of 0 (after clamping to the target size) lifts the limit. */
static void pss_rec(const float *v, size_t n, size_t start, size_t depth, size_t max_depth, float base,
                    float *out, long *cnt, long cap) {
    for (; start < n; start++) {
        float s = base + v[start];
        if (*cnt < cap) out[*cnt] = s;
        (*cnt)++;
        if (start < n - 1 && depth < max_depth - 1) pss_rec(v, n, start + 1, depth + 1, max_depth, s, out, cnt, cap);
    }
}

long orc_power_set_sum(const float *v, size_t n, size_t depth, float *out, long cap) {
    if (n > 20) return -1;
    long total = 1L << n, c = 0;
    float *tmp = (float *)malloc((size_t)(total + 1) * sizeof(float));
    if (n < depth) depth = n;
    tmp[c++] = 0.f;
    pss_rec(v, n, 0, 0, depth, 0.f, tmp, &c, total + 1);
    for (long i = 1; i < c; i++) { float x = tmp[i]; long j = i; while (j > 0 && tmp[j-1] > x) { tmp[j] = tmp[j-1]; j--; } tmp[j] = x; }
    long u = 1;
    for (long i = 1; i < c; i++) if (tmp[i] != tmp[u-1]) tmp[u++] = tmp[i];
    for (long i = 0; i < u && i < cap; i++) out[i] = tmp[i];
    free(tmp);
    return u;
}

/* cpp/ModifiedPeptide.cpp:570-591 */
static float fragment_mz(float run, float nlsum, char type, int z) {
    double d = (double)(run - nlsum);
    if (type == 'y') d += 18.010565;
    else if (type == 'z') { d += 18.010565; d -= 17.026549; }
    else if (type == 'Z') { d += 18.010565; d -= 16.018724; }
    else if (type == 'c') d += 17.026549;
    if (z > 0) d = (d + (double)z * 1.007825) / (double)z;
    return (float)d;
}

/* All fragments of the isoform whose per-residue mod state is `state[0..L)`, for one ion
 * type and charge, in emission order.  Restates FragmentGraph's walk
 * (cpp/ModifiedPeptide.cpp:379-408, :500-524): running float sum over residues in
 * traversal order, last residue never emitted, neutral-loss stack grows as residues with a
 * non-zero loss are passed, one fragment per distinct <=2-subset sum. */
static long isoform_fragments(const orc *o, const unsigned char *state, char type, int z, float *out, long cap) {
    int L = o->L;
    int fwd = (type == 'b' || type == 'c');
    float run = 0.f;
    float *stack = (float *)malloc((L + 1) * sizeof(float));
    float *sums = (float *)malloc((2 + L + (size_t)L * L) * sizeof(float));
    int m = 0, ns = 1;
    sums[0] = 0.f;
    long n = 0;
    /* A one-residue peptide is the one case where the walk starts ON the last residue: the
     * reference's end test (isFragmentEnd: last residue AND no neutral-loss variant left,
     * cpp/ModifiedPeptide.cpp:516-524) then lets every variant but the last one through. */
    int steps = (L == 1) ? 1 : L - 1;
    for (int step = 0; step < steps; step++) {
        int i = fwd ? step : L - 1 - step;
        int s = state[i];
        run = (step == 0) ? o->res[i][s] : (o->res[i][s] + run);
        if (o->nl[i][s] != 0.f) { stack[m++] = o->nl[i][s]; ns = power_set_sums(stack, m, sums); }
        int emit = (L == 1) ? ns - 1 : ns;
        for (int v = 0; v < emit; v++) {
            if (n < cap) out[n] = fragment_mz(run, sums[v], type, z);
            n++;
        }
    }
    free(stack); free(sums);
    return n;
}

/* ------------------------------------------------------------------ matching */
/* cpp/ModifiedPeptide.cpp:126-150 + the peak loop of Ascore.pyx:142-150: the rank a
 * theoretical fragment value f ends up with = min rank over retained peaks p=(float)mz with
 * (double)f >= (double)p - .5, p > f - err and p < f + err (float arithmetic). -1: none. */
static int match_rank(const orc *o, float f) {
    int best = -1;
    float lo = f - o->mz_error, hi = f + o->mz_error;
    for (int i = 0; i < o->n_pk; i++) {
        float p = o->pk_mz[i];
        if (!((double)f >= (double)p - .5)) continue;
        if (p > lo && p < hi) { if (best < 0 || o->pk_rank[i] < best) best = o->pk_rank[i]; }
    }
    return best;
}

/* ------------------------------------------------------------------ libstdc++ models */
/* unordered_map<long,...> iteration order after inserting distinct keys in the given
 * order (cpp/Ascore.cpp:54,96-108,113-120).  Model of GCC-13 _Hashtable with identity hash,
 * max load factor 1 and _Prime_rehash_policy; bucket-count chain measured on this image's
 * libstdc++ (13 -> 29 -> 59 -> ... next prime in __prime_list >= 2*n). */
static const uint64_t BKT_CHAIN[] = {13ull, 29ull, 59ull, 127ull, 257ull, 541ull, 1109ull, 2357ull, 5087ull, 10273ull, 20753ull,
    42043ull, 85229ull, 172933ull, 351061ull, 712697ull, 1447153ull, 2938679ull, 5967347ull, 12117689ull,
    24607243ull, 49969847ull, 101473717ull, 206062531ull, 418451333ull, 849749479ull, 1725587117ull};

static void hash_order(const uint64_t *keys, long n, long *order /* out: indices into keys */) {
    /* singly linked list through next[]; node n = the before-begin sentinel */
    long *next = (long *)malloc((n + 1) * sizeof(long));
    long BB = n;
    next[BB] = -1;
    uint64_t n_bkt = 1; int chain = -1; uint64_t next_resize = 0;
    long *bkt = (long *)malloc(sizeof(long));      /* bkt[b] = node BEFORE first node of bucket, -1 empty */
    bkt[0] = -1;
    for (long e = 0; e < n; e++) {
        if ((uint64_t)e + 1 > next_resize) {
            /* _M_need_rehash: first time min 11 buckets -> 13; afterwards next prime >= 2*n_bkt */
            uint64_t nb;
            if (next_resize == 0) nb = BKT_CHAIN[++chain];
            else nb = BKT_CHAIN[++chain];
            next_resize = nb;
            /* _M_rehash_aux (unique keys): relink every node front to back */
            long *nbk = (long *)malloc(nb * sizeof(long));
            for (uint64_t i = 0; i < nb; i++) nbk[i] = -1;
            long p = next[BB];
            next[BB] = -1;
            uint64_t bbegin_bkt = 0;
            while (p >= 0) {
                long nx = next[p];
                uint64_t b = (uint64_t)keys[p] % nb;
                if (nbk[b] < 0) {
                    next[p] = next[BB]; next[BB] = p; nbk[b] = BB;
                    if (next[p] >= 0) nbk[bbegin_bkt] = p;
                    bbegin_bkt = b;
                } else { next[p] = next[nbk[b]]; next[nbk[b]] = p; }
                p = nx;
            }
            free(bkt); bkt = nbk; n_bkt = nb;
        }
        /* _M_insert_bucket_begin */
        uint64_t b = (uint64_t)keys[e] % n_bkt;
        if (bkt[b] >= 0) { next[e] = next[bkt[b]]; next[bkt[b]] = e; }
        else {
            next[e] = next[BB]; next[BB] = e;
            if (next[e] >= 0) bkt[(uint64_t)keys[next[e]] % n_bkt] = e;
            bkt[b] = BB;
        }
    }
    long c = 0;
    for (long p = next[BB]; p >= 0; p = next[p]) order[c++] = p;
    free(next); free(bkt);
}

/* std::sort(first,last, a.weighted > b.weighted) of libstdc++ (bits/stl_algo.h, GCC 13:
 * __introsort_loop with _S_threshold 16, median-of-three to first, unguarded partition,
 * heap sort on depth exhaustion, then __final_insertion_sort).  cpp/Ascore.cpp:141-146.
 * Sorts an index array by w[] so the caller can permute whole records. */
typedef struct { float w; long id; } srt;
#define CMP(x, y) ((x).w > (y).w)

static void adjust_heap(srt *a, long hole, long len, srt v) {
    long top = hole, child = hole;
    while (child < (len - 1) / 2) {
        child = 2 * (child + 1);
        if (CMP(a[child], a[child - 1])) child--;
        a[hole] = a[child]; hole = child;
    }
    if ((len & 1) == 0 && child == (len - 2) / 2) {
        child = 2 * (child + 1);
        a[hole] = a[child - 1]; hole = child - 1;
    }
    long parent = (hole - 1) / 2;                  /* __push_heap */
    while (hole > top && CMP(a[parent], v)) { a[hole] = a[parent]; hole = parent; parent = (hole - 1) / 2; }
    a[hole] = v;
}

static void heap_sort(srt *a, long n) {            /* __partial_sort(first,last,last) */
    if (n < 2) return;
    for (long parent = (n - 2) / 2;; parent--) {    /* __make_heap */
        srt v = a[parent];
        adjust_heap(a, parent, n, v);
        if (parent == 0) break;
    }
    /* __heap_select's loop over [middle,last) is empty; __sort_heap: */
    for (long last = n; last > 1;) {
        --last;
        srt v = a[last]; a[last] = a[0];
        adjust_heap(a, 0, last, v);
    }
}

static void introsort_loop(srt *a, long first, long last, long depth) {
    while (last - first > 16) {
        if (depth == 0) { heap_sort(a + first, last - first); return; }
        --depth;
        long mid = first + (last - first) / 2;
        /* __move_median_to_first(first, first+1, mid, last-1) */
        long x = first + 1, y = mid, z = last - 1, r = first, pick;
        if (CMP(a[x], a[y])) { if (CMP(a[y], a[z])) pick = y; else if (CMP(a[x], a[z])) pick = z; else pick = x; }
        else if (CMP(a[x], a[z])) pick = x; else if (CMP(a[y], a[z])) pick = z; else pick = y;
        { srt t = a[r]; a[r] = a[pick]; a[pick] = t; }
        /* __unguarded_partition(first+1, last, first) */
        long f = first + 1, l = last;
        for (;;) {
            while (CMP(a[f], a[first])) f++;
            --l;
            while (CMP(a[first], a[l])) l--;
            if (!(f < l)) break;
            { srt t = a[f]; a[f] = a[l]; a[l] = t; }
            f++;
        }
        introsort_loop(a, f, last, depth);
        last = f;
    }
}

static void unguarded_linear_insert(srt *a, long i) {
    srt v = a[i];
    long j = i - 1;
    while (CMP(v, a[j])) { a[j + 1] = a[j]; j--; }
    a[j + 1] = v;
}

static void insertion_sort(srt *a, long first, long last) {
    if (first == last) return;
    for (long i = first + 1; i < last; i++) {
        if (CMP(a[i], a[first])) { srt v = a[i]; memmove(a + first + 1, a + first, (i - first) * sizeof(srt)); a[first] = v; }
        else unguarded_linear_insert(a, i);
    }
}

static void gcc_sort(srt *a, long n) {
    if (n == 0) return;
    long lg = 0; { long t = n; while (t > 1) { t >>= 1; lg++; } }
    introsort_loop(a, 0, n, 2 * lg);
    if (n > 16) { insertion_sort(a, 0, 16); for (long i = 16; i < n; i++) unguarded_linear_insert(a, i); }
    else insertion_sort(a, 0, n);
}

/* exposed for unit tests */
void orc_hash_order(const uint64_t *keys, long n, long *order) { hash_order(keys, n, order); }
long orc_bkt_chain(uint64_t *out, long cap) {
    long n = (long)(sizeof(BKT_CHAIN) / sizeof(BKT_CHAIN[0]));
    for (long i = 0; i < n && i < cap; i++) out[i] = BKT_CHAIN[i];
    return n;
}
void orc_gcc_sort(const float *w, long n, long *order_inout) {
    srt *a = (srt *)malloc((n + 1) * sizeof(srt));
    for (long i = 0; i < n; i++) { a[i].w = w[order_inout[i]]; a[i].id = order_inout[i]; }
    gcc_sort(a, n);
    for (long i = 0; i < n; i++) order_inout[i] = a[i].id;
    free(a);
}

/* ------------------------------------------------------------------ isoform enumeration */
static void key_to_state(const orc *o, uint64_t key, unsigned char *state) {
    memset(state, 0, o->L);
    for (int j = 0; j < o->S; j++) if ((key >> (o->S - 1 - j)) & 1ull) state[o->site_pos[j]] = 1;
}

/* k-combinations of S sites in lexicographic order of TRAVERSAL positions of the first
 * fragment type (cpp/ModifiedPeptide.cpp:410-472): N->C for b/c, C->N for y/z/Z. */
static long enumerate_keys(const orc *o, uint64_t **out) {
    int S = o->S, k = o->k;
    *out = NULL;
    if (k > S) return 0;
    /* count */
    double cnt = 1; for (int i = 0; i < k; i++) cnt = cnt * (S - i) / (i + 1);
    long n = (long)(cnt + 0.5);
    uint64_t *keys = (uint64_t *)malloc((n + 1) * sizeof(uint64_t));
    int fwd = (o->frag_types[0] == 'b' || o->frag_types[0] == 'c');
    int c[64];
    for (int i = 0; i < k; i++) c[i] = i;
    long m = 0;
    for (;;) {
        uint64_t key = 0;
        for (int i = 0; i < k; i++) {
            int site = fwd ? c[i] : S - 1 - c[i];     /* traversal index -> N->C site index */
            key |= 1ull << (S - 1 - site);
        }
        keys[m++] = key;
        int i = k - 1;
        while (i >= 0 && c[i] == S - k + i) i--;
        if (i < 0) break;
        c[i]++;
        for (int j = i + 1; j < k; j++) c[j] = c[j - 1] + 1;
    }
    *out = keys;
    return m;
}

/* ------------------------------------------------------------------ site-determining ions */
static int cmp_float(const void *a, const void *b) { float x = *(const float *)a, y = *(const float *)b; return (x > y) - (x < y); }

/* cpp/ModifiedPeptide.cpp:259-320 */
static void site_determining(const orc *o, uint64_t ka, uint64_t kb, char type, int Z,
                             float **oa, long *na, float **ob, long *nb) {
    unsigned char *sa = (unsigned char *)malloc(o->L), *sb = (unsigned char *)malloc(o->L);
    key_to_state(o, ka, sa); key_to_state(o, kb, sb);
    long cap = 0;
    for (int z = 1; z <= Z; z++) { long t = isoform_fragments(o, sa, type, z, NULL, 0); long u = isoform_fragments(o, sb, type, z, NULL, 0); cap += (t > u ? t : u); }
    float *A = (float *)malloc((cap + 1) * sizeof(float)), *B = (float *)malloc((cap + 1) * sizeof(float));
    long la = 0, lb = 0;
    for (int z = 1; z <= Z; z++) { la += isoform_fragments(o, sa, type, z, A + la, cap - la); lb += isoform_fragments(o, sb, type, z, B + lb, cap - lb); }
    qsort(A, la, sizeof(float), cmp_float); qsort(B, lb, sizeof(float), cmp_float);
    float *ra = (float *)malloc((la + 1) * sizeof(float)), *rb = (float *)malloc((lb + 1) * sizeof(float));
    long i = 0, j = 0, ca = 0, cb = 0;
    while (i < la || j < lb) {
        if (j == lb) ra[ca++] = A[i++];
        else if (i == la) rb[cb++] = B[j++];
        else if (fabsf(A[i] - B[j]) < o->mz_error) { i++; j++; }
        else if (A[i] < B[j]) ra[ca++] = A[i++];
        else rb[cb++] = B[j++];
    }
    free(A); free(B); free(sa); free(sb);
    *oa = ra; *na = ca; *ob = rb; *nb = cb;
}

long orc_site_determining(orc *o, size_t S, const int32_t *sig_a, const int32_t *sig_b, char type,
                          size_t max_charge, float *out_a, long *n_a, float *out_b, long *n_b, long cap) {
    uint64_t ka = 0, kb = 0;
    for (size_t i = 0; i < S; i++) { ka = (ka << 1) | (uint64_t)(sig_a[i] != 0); kb = (kb << 1) | (uint64_t)(sig_b[i] != 0); }
    float *a, *b;
    site_determining(o, ka, kb, type, (int)max_charge, &a, n_a, &b, n_b);
    for (long i = 0; i < *n_a && i < cap; i++) out_a[i] = a[i];
    for (long i = 0; i < *n_b && i < cap; i++) out_b[i] = b[i];
    free(a); free(b);
    return 0;
}

/* cpp/Ascore.cpp:157-210 */
static float ambiguity(orc *o, uint64_t ka, const float *sc_a, float w_a, uint64_t kb, const float *sc_b, float w_b) {
    if (fabsf(w_a - w_b) < 1e-6) return 0.f;
    float max_diff = 0.f; int depth = 0;
    for (int d = 0; d < o->n_top; d++) { float diff = sc_a[d] - sc_b[d]; if (diff > max_diff) { max_diff = diff; depth = d; } }
    size_t hits[2] = {0, 0}, trials[2] = {0, 0};
    for (const char *t = o->frag_types; *t; t++) {
        float *a, *b; long na, nb;
        site_determining(o, ka, kb, *t, o->Z, &a, &na, &b, &nb);
        trials[0] += na; trials[1] += nb;
        for (long i = 0; i < na; i++) { int r = match_rank(o, a[i]); if (r >= 0 && r <= depth) hits[0]++; }
        for (long i = 0; i < nb; i++) { int r = match_rank(o, b[i]); if (r >= 0 && r <= depth) hits[1]++; }
        free(a); free(b);
    }
    float s0 = binom_score(&o->dist[depth], hits[0], trials[0]);
    float s1 = binom_score(&o->dist[depth], hits[1], trials[1]);
    return s0 - s1;
}

/* ------------------------------------------------------------------ the scoring pipeline */
/* cpp/Ascore.cpp:256-271 (score), :53-121 (counts), :123-139 (scores), :38-51, :141-146, :212-254 */
int orc_score_current(orc *o) {
    free_results(o);
    o->n_asc = 0;
    int D = o->n_top, k = o->k, S = o->S, L = o->L;
    uint64_t *ins = NULL;
    long n = enumerate_keys(o, &ins);
    if (n > 0) {
        long *ord = (long *)malloc(n * sizeof(long));
        hash_order(ins, n, ord);
        o->n_iso = n;
        o->key = (uint64_t *)malloc(n * sizeof(uint64_t));
        o->counts = (int32_t *)calloc((size_t)n * D, sizeof(int32_t));
        o->scores = (float *)calloc((size_t)n * D, sizeof(float));
        o->weighted = (float *)calloc(n, sizeof(float));
        o->total = (int64_t *)calloc(n, sizeof(int64_t));
        unsigned char *state = (unsigned char *)malloc(L);
        long fcap = 0; float *fr = NULL;
        for (long q = 0; q < n; q++) {
            uint64_t key = ins[ord[q]];
            o->key[q] = key;
            key_to_state(o, key, state);
            int32_t *cnt = o->counts + q * D;
            for (const char *t = o->frag_types; *t; t++)
                for (int z = 1; z <= o->Z; z++) {
                    long nf = isoform_fragments(o, state, *t, z, NULL, 0);
                    if (nf > fcap) { fcap = nf; fr = (float *)realloc(fr, fcap * sizeof(float)); }
                    isoform_fragments(o, state, *t, z, fr, fcap);
                    for (long f = 0; f < nf; f++) { int r = match_rank(o, fr[f]); if (r >= 0) cnt[r]++; }
                    o->total[q] += nf;
                }
            for (int d = 1; d < D; d++) cnt[d] += cnt[d - 1];
            /* cpp/Ascore.cpp:123-139 */
            float *sc = o->scores + q * D;
            for (int d = 0; d < D; d++) sc[d] = binom_score(&o->dist[d], (size_t)cnt[d], (size_t)o->total[q]);
            double acc = 0.;
            for (int d = 0; d < ORC_WEIGHTS && d < D; d++) acc += (double)(o->weights[d] * sc[d]);
            o->weighted[q] = (float)acc;
        }
        free(state); free(fr); free(ord);
    }
    free(ins);

    if (k >= S) {                                     /* cpp/Ascore.cpp:38-51 */
        o->n_asc = k;
        for (int j = 0; j < k && j < 64; j++) { o->asc[j] = INFINITY; o->n_alt[j] = 0; }
        return 0;
    }
    /* sortScores */
    {
        srt *a = (srt *)malloc((n + 1) * sizeof(srt));
        for (long i = 0; i < n; i++) { a[i].w = o->weighted[i]; a[i].id = i; }
        gcc_sort(a, n);
        uint64_t *key2 = (uint64_t *)malloc(n * sizeof(uint64_t));
        int32_t *cnt2 = (int32_t *)malloc((size_t)n * D * sizeof(int32_t));
        float *sc2 = (float *)malloc((size_t)n * D * sizeof(float));
        float *w2 = (float *)malloc(n * sizeof(float));
        int64_t *t2 = (int64_t *)malloc(n * sizeof(int64_t));
        for (long i = 0; i < n; i++) {
            long s = a[i].id;
            key2[i] = o->key[s]; w2[i] = o->weighted[s]; t2[i] = o->total[s];
            memcpy(cnt2 + i * D, o->counts + s * D, D * sizeof(int32_t));
            memcpy(sc2 + i * D, o->scores + s * D, D * sizeof(float));
        }
        free(o->key); free(o->counts); free(o->scores); free(o->weighted); free(o->total); free(a);
        o->key = key2; o->counts = cnt2; o->scores = sc2; o->weighted = w2; o->total = t2;
    }
    /* calculateAscores: cpp/Ascore.cpp:212-254 */
    uint64_t best = o->key[0];
    int site_of[64], nmod = 0;                        /* findModifiedPos */
    for (int j = 0; j < S; j++) if ((best >> (S - 1 - j)) & 1ull) site_of[nmod++] = j;
    float last_pep[64]; int n_cand[64]; float min_asc[64];
    for (int j = 0; j < nmod; j++) { n_cand[j] = 0; o->n_alt[j] = 0; min_asc[j] = 0.f; last_pep[j] = 0.f; }
    for (long q = 0; q < n; q++) {
        uint64_t c = o->key[q];
        int common = __builtin_popcountll(best & c);
        if (k - common != 1) continue;
        uint64_t lost = best & ~c, gained = c & ~best;
        int lost_site = S - 1 - (63 - __builtin_clzll(lost));
        int gained_site = S - 1 - (63 - __builtin_clzll(gained));
        int aj = 0; for (int j = 0; j < nmod; j++) if (site_of[j] == lost_site) aj = j;
        if (n_cand[aj] == 0 || o->weighted[q] == last_pep[aj]) {
            float amb = ambiguity(o, best, o->scores, o->weighted[0], c, o->scores + q * D, o->weighted[q]);
            if (o->n_alt[aj] < 64) o->alt[aj][o->n_alt[aj]++] = (uint32_t)(o->site_pos[gained_site] + 1);
            last_pep[aj] = o->weighted[q];
            if (n_cand[aj] == 0 || amb < min_asc[aj]) min_asc[aj] = amb;
            n_cand[aj]++;
        }
    }
    o->n_asc = nmod;
    for (int j = 0; j < nmod; j++) {
        o->asc[j] = min_asc[j];
        /* getAlternativeSites sorts: cpp/Ascore.cpp:315-319 */
        for (int a = 1; a < o->n_alt[j]; a++) { uint32_t v = o->alt[j][a]; int b = a; while (b > 0 && o->alt[j][b-1] > v) { o->alt[j][b] = o->alt[j][b-1]; b--; } o->alt[j][b] = v; }
    }
    return 0;
}

/* Ascore.pyx:103-152 */
int orc_score(orc *o, const double *mz, const double *inten, size_t n_peaks, const char *pep, size_t k,
              size_t Z, const unsigned *aux_pos, const float *aux_mass, size_t n_aux) {
    consume_spectra_fast(o, mz, inten, n_peaks);
    int rc = orc_consume_peptide(o, pep, k, Z, aux_pos, aux_mass, (aux_pos && aux_mass) ? n_aux : 0);
    if (rc) return rc;
    return orc_score_current(o);
}

/* ------------------------------------------------------------------ result getters */
/* cpp/ModifiedPeptide.cpp:199-253 */
static int peptide_string(const orc *o, uint64_t key, int have_key, char *buf, int cap) {
    int L = o->L, S = o->S;
    float *mm = (float *)calloc(L + 2, sizeof(float));
    if (o->k > S) { if (strchr(o->mod_group, 'n')) mm[0] += o->mod_mass; else mm[L + 1] += o->mod_mass; }
    for (int j = 0; j < S; j++) {
        int on = have_key ? (int)((key >> (S - 1 - j)) & 1ull) : (j < (o->k < S ? o->k : S));
        if (!on) continue;
        int p = o->site_pos[j];
        if (strchr(o->mod_group, o->pep[p])) mm[p + 1] += o->mod_mass;
        else if (p == 0) mm[0] += o->mod_mass;
        else if (p + 1 == L) mm[L + 1] += o->mod_mass;
    }
    for (int a = 0; a < o->n_aux; a++) if ((int)o->aux_pos[a] < L + 2) mm[o->aux_pos[a]] += o->aux_mass[a];
    int start = (mm[0] == 0.f) ? 1 : 0, end = (mm[L + 1] == 0.f) ? L + 1 : L + 2, n = 0;
    for (int i = start; i < end; i++) {
        char c = (i == 0) ? 'n' : (i == L + 1) ? 'c' : o->pep[i - 1];
        if (n + 16 >= cap) { free(mm); return -1; }
        buf[n++] = c;
        if (mm[i] > 0.f) n += sprintf(buf + n, "[%d]", (int)roundf(mm[i]));
    }
    buf[n] = 0;
    free(mm);
    return n;
}

int orc_get_peptide(orc *o, size_t S, const int32_t *sig, char *buf, int cap) {
    /* an empty signature means "the first one" (cpp/ModifiedPeptide.cpp:201-204); entries beyond
     * the modifiable residues are ignored, missing ones count as 0, only the value 1 marks a mod */
    if (S == 0) return peptide_string(o, 0, 0, buf, cap);
    uint64_t key = 0;
    for (size_t i = 0; i < S && (int)i < o->S; i++) if (sig[i] == 1) key |= 1ull << (o->S - 1 - (int)i);
    return peptide_string(o, key, 1, buf, cap);
}

int orc_best_sequence(orc *o, char *buf, int cap) {
    if (o->n_iso == 0) { if (cap > 0) buf[0] = 0; return 0; }
    return peptide_string(o, o->key[0], 1, buf, cap);
}
float orc_best_score(orc *o) { return o->n_iso ? o->weighted[0] : -1.f; }
size_t orc_n_pep_scores(orc *o) { return (size_t)o->n_iso; }
size_t orc_sig_len(orc *o) { return o->n_iso ? (size_t)o->S : 0; }

void orc_pep_scores(orc *o, int32_t *signature, int32_t *counts, float *scores, float *weighted, int64_t *total) {
    int S = o->S, D = o->n_top;
    for (long i = 0; i < o->n_iso; i++) {
        for (int j = 0; j < S; j++) signature[i * S + j] = (int32_t)((o->key[i] >> (S - 1 - j)) & 1ull);
        memcpy(counts + i * D, o->counts + i * D, D * sizeof(int32_t));
        memcpy(scores + i * D, o->scores + i * D, D * sizeof(float));
        weighted[i] = o->weighted[i]; total[i] = o->total[i];
    }
}

long orc_sequences(orc *o, char *buf, long cap) {
    long need = 33; char tmp[8192];
    for (long i = 0; i < o->n_iso; i++) need += peptide_string(o, o->key[i], 1, tmp, sizeof(tmp)) + (i ? 1 : 0);
    if (need > cap) return need;
    long n = 0;
    for (long i = 0; i < o->n_iso; i++) { if (i) buf[n++] = '\n'; n += peptide_string(o, o->key[i], 1, buf + n, (int)(cap - n)); }
    buf[n] = 0;
    return need;
}

size_t orc_n_ascores(orc *o) { return (size_t)o->n_asc; }
void orc_ascores(orc *o, float *out) { for (int i = 0; i < o->n_asc; i++) out[i] = o->asc[i]; }
long orc_alt_sites(orc *o, size_t site, uint32_t *out, long cap) {
    if ((int)site >= o->n_asc) return 0;
    long n = (o->k >= o->S) ? 0 : o->n_alt[site];
    for (long i = 0; i < n && i < cap; i++) out[i] = o->alt[site][i];
    return n;
}

float orc_calculate_ambiguity(orc *o, size_t S, size_t D, const int32_t *sig_a, const int32_t *cnt_a,
                              const float *sc_a, float w_a, int64_t tot_a, const int32_t *sig_b,
                              const int32_t *cnt_b, const float *sc_b, float w_b, int64_t tot_b) {
    (void)cnt_a; (void)cnt_b; (void)tot_a; (void)tot_b; (void)D;
    uint64_t ka = 0, kb = 0;
    for (size_t i = 0; i < S; i++) { ka = (ka << 1) | (uint64_t)(sig_a[i] != 0); kb = (kb << 1) | (uint64_t)(sig_b[i] != 0); }
    return ambiguity(o, ka, sc_a, w_a, kb, sc_b, w_b);
}

/* ---- stage probes ---- */
long orc_binned(orc *o, int32_t *bin, int32_t *rank, double *mz, double *inten, long cap, float *min_mz,
                float *max_mz, int64_t *n_bins) {
    *min_mz = o->min_mz; *max_mz = o->max_mz; *n_bins = o->n_bins;
    for (long i = 0; i < o->n_pk && i < cap; i++) { bin[i] = o->pk_bin[i]; rank[i] = o->pk_rank[i]; mz[i] = o->pk_mz64[i]; inten[i] = o->pk_int[i]; }
    return o->n_pk;
}

void orc_consume_spectra_fast(orc *o, const double *mz, const double *inten, size_t n) { consume_spectra_fast(o, mz, inten, n); }

/* every isoform (in the first fragment type's enumeration order... here: order of `type`'s
 * own graph, like refshim_fragment_graph) with all its fragments */
long orc_fragment_graph(orc *o, char type, size_t charge, int32_t *sig_out, long sig_cap, int64_t *frag_off,
                        float *frag_out, long frag_cap, int64_t *n_frag_total) {
    char saved = o->frag_types[0];
    o->frag_types[0] = type;                       /* enumeration direction of this type */
    uint64_t *keys; long n = enumerate_keys(o, &keys);
    o->frag_types[0] = saved;
    unsigned char *state = (unsigned char *)malloc(o->L);
    int64_t nf = 0;
    for (long q = 0; q < n; q++) {
        key_to_state(o, keys[q], state);
        if (q < sig_cap) {
            for (int j = 0; j < o->S; j++) sig_out[q * o->S + j] = (int32_t)((keys[q] >> (o->S - 1 - j)) & 1ull);
            frag_off[q] = nf;
        }
        long c = isoform_fragments(o, state, type, (int)charge, frag_out ? frag_out + (nf < frag_cap ? nf : frag_cap) : NULL,
                                   frag_out && nf < frag_cap ? frag_cap - nf : 0);
        nf += c;
    }
    if (frag_off && n <= sig_cap) frag_off[n < sig_cap ? n : sig_cap] = nf;
    *n_frag_total = nf;
    free(keys); free(state);
    return n;
}

int orc_has_match(orc *o, float mz, float *peak_mz, int64_t *rank) {
    int r = match_rank(o, mz);
    if (r < 0) return 0;
    *rank = r; *peak_mz = 0.f;
    float lo = mz - o->mz_error, hi = mz + o->mz_error;
    /* the reference keeps the first peak (in bin,rank walk order) that achieved the min rank */
    for (int i = 0; i < o->n_pk; i++) {
        float p = o->pk_mz[i];
        if ((double)mz >= (double)p - .5 && p > lo && p < hi && o->pk_rank[i] == r) { *peak_mz = p; break; }
    }
    return 1;
}

float orc_log_sum(float a, float b) { return f_log_sum(a, b); }
float orc_log_bin_coef(size_t k, size_t n) { return f_log_bin_coef(k, n); }
void *orc_binom_new(float p) { orc_binom *b = (orc_binom *)malloc(sizeof(orc_binom)); binom_init(b, p); return b; }
void orc_binom_free(void *b) { binom_free((orc_binom *)b); free(b); }
float orc_binom_log_pmf(void *b, size_t k, size_t n) { return binom_log_pmf((orc_binom *)b, k, n); }
float orc_binom_log_pvalue(void *b, size_t k, size_t n) { return binom_log_pvalue((orc_binom *)b, k, n); }
float orc_binom_log10_pvalue(void *b, size_t k, size_t n) { return binom_log10_pvalue((orc_binom *)b, k, n); }
/* score table probe used to check the GPU tail table: |-10 log10 tail_d(k,n)| */
float orc_depth_score(orc *o, int depth /*0-based*/, size_t k, size_t n) { return binom_score(&o->dist[depth], k, n); }

/* ---- batched scoring over CSR arrays (CPU "port" baseline; serial) ---- */
void orc_score_batch(orc *o, int64_t n_psm, const int64_t *spec_off, const double *mz, const double *inten,
                     const int32_t *psm_spec, const int32_t *pep_off, const char *pep, const int32_t *n_mod,
                     const int32_t *max_charge, const int32_t *aux_off, const uint32_t *aux_pos,
                     const float *aux_mass, float *best_score, float *ascores, int32_t max_k) {
    char buf[1024];
    for (int64_t i = 0; i < n_psm; i++) {
        int64_t sp = psm_spec[i];
        int len = pep_off[i + 1] - pep_off[i];
        memcpy(buf, pep + pep_off[i], len); buf[len] = 0;
        int32_t na = aux_off ? aux_off[i + 1] - aux_off[i] : 0;
        orc_score(o, mz + spec_off[sp], inten + spec_off[sp], (size_t)(spec_off[sp + 1] - spec_off[sp]), buf,
                  (size_t)n_mod[i], (size_t)max_charge[i], na ? aux_pos + aux_off[i] : NULL,
                  na ? aux_mass + aux_off[i] : NULL, (size_t)na);
        best_score[i] = orc_best_score(o);
        if (ascores) for (int32_t j = 0; j < max_k; j++) ascores[i * max_k + j] = j < o->n_asc ? o->asc[j] : 0.f;
    }
}
