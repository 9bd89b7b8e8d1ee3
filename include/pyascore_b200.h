/* pyascore_b200 -- C ABI of the B200-native PTM-localisation scoring library.
 *
 * This is the drop-in boundary for ONE path of Villen-Lab/pyAscore: what the Cython class
 * `pyascore.PyAscore` (reference: pyascore/ptm_scoring/Ascore.pyx:12-288, bound to the C++
 * classes declared in Ascore.pxd:9-26, ModifiedPeptide.pxd:9-46, Spectra.pxd) does for
 * `score()` and its result properties.  Plain pointers and sizes only; no C++ or torch types.
 * The reference-side binding is shown in INTEGRATION.md; pyascore_b200/_lib.py is the ctypes
 * binding this repo ships.
 *
 * Conventions
 *   - every function returns PA_OK (0) or a negative pa_status; pa_last_error() gives text.
 *   - array arguments may point to HOST memory (pageable or pinned) or DEVICE memory of the
 *     scorer's GPU; the library detects which (cudaPointerGetAttributes) and copies as needed.
 *     All arrays of one call's `pa_batch` must live on the same side, likewise `pa_results`.
 *   - a scorer is bound to one GPU and is NOT thread-safe (like the reference object:
 *     SURVEY.md section 8b); use one scorer per (GPU, host thread).
 *   - no CPU fallback exists: without a usable CUDA device pa_create fails.
 */
#ifndef PYASCORE_B200_H
#define PYASCORE_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct pa_scorer pa_scorer;

typedef enum {
    PA_OK = 0,
    PA_ERR_CUDA = -1,        /* CUDA runtime / driver error (text in pa_last_error) */
    PA_ERR_ARG = -2,         /* invalid argument (NULL pointer, bad fragment type, inconsistent CSR arrays ...) */
    PA_ERR_UNSUPPORTED = -3, /* outside the supported envelope (see limits below) */
    PA_ERR_STATE = -4        /* call needs a kept batch (PA_KEEP_ISOFORMS) and there is none, or an asynchronous call is in flight */
} pa_status;

/* per-PSM status written to pa_results.psm_status (0 = scored) */
enum {
    PA_PSM_OK = 0,
    PA_PSM_BAD_RESIDUE = 1,    /* letter outside cpp/Types.h:7-30 (reference: std::out_of_range -> abort) */
    PA_PSM_TOO_LONG = 2,       /* peptide longer than PA_MAX_PEPTIDE */
    PA_PSM_TOO_MANY_SITES = 3, /* more than 63 modifiable residues (reference packs the signature in a long) */
    PA_PSM_TOO_MANY_ISOFORMS = 4,
    PA_PSM_EMPTY_SPECTRUM = 5, /* reference: undefined behaviour */
    PA_PSM_BAD_AUX = 6,        /* fixed-mod position beyond the last residue (reference: out of bounds) */
    PA_PSM_BAD_INDEX = 7,      /* psm_spec out of range / negative n_mod / max_charge < 1 */
    PA_PSM_TOO_MANY_FRAGMENTS = 8 /* theoretical fragments per isoform exceed PA_MAX_FRAGMENTS */
};

/* Peak depth of a scoring handle.  The reference's weight vector has 10 entries (cpp/Ascore.cpp:15-19): n_top < 10 reads
 * out of bounds there; for n_top > 10 the PepScores, the isoform order, best_sequence and the alternative sites are
 * those of n_top = 10, while deeper ranks add count / score columns for depths 10 .. n_top-1 and can move the depth
 * calculateAmbiguity picks (cpp/Ascore.cpp:165-175 -- shown on the compiled reference by tests/test_oracle_vs_ref.py::
 * test_reference_behaviour_for_n_top_above_10), so an Ascore may be computed at a depth >= 10.  pa_create takes
 * PA_N_TOP <= n_top <= PA_MAX_N_TOP and computes all of that as the reference does; n_top < 10 (out-of-bounds reads in
 * the reference) and n_top > 64 (beyond the tested envelope) are PA_ERR_UNSUPPORTED.  pyascore/__main__.py:69
 * hard-codes n_top = 10.  Per-depth arrays of the ABI (pa_fetch_pep_scores, pa_calculate_ambiguity, pa_tail_table)
 * are n_top wide. */
#define PA_N_TOP 10
#define PA_MAX_N_TOP 64
#define PA_MAX_PEPTIDE 126
#define PA_MAX_SITES 63
#define PA_MAX_ISOFORMS (1ll << 26)
#define PA_MAX_FRAGMENTS 4095     /* per isoform, all ion types/charges/neutral-loss variants */
#define PA_MAX_NL_MASSES 4        /* distinct neutral-loss masses over all add_neutral_loss calls */

/* Replaces PyAscore.__cinit__ (Ascore.pyx:64-73): BinnedSpectra(bin_size, n_top) +
 * ModifiedPeptide(mod_group, mod_mass, mz_error, fragment_types) + Ascore().
 * `device` is the CUDA ordinal.  n_top in PA_N_TOP .. PA_MAX_N_TOP (see PA_N_TOP). */
int pa_create(float bin_size, int n_top, const char* mod_group, float mod_mass, float mz_error,
              const char* fragment_types, int device, pa_scorer** out);

/* Replaces PyBinnedSpectra.__cinit__ (Spectra.pyx:47-48): a handle that only bins spectra
 * (pa_bin_spectra / pa_bin_spectra_ex); any n_top in 1..254.  pa_score_batch refuses it. */
int pa_create_binner(float bin_size, int n_top, int device, pa_scorer** out);

/* Replaces PyAscore.add_neutral_loss (Ascore.pyx:81-99 -> cpp/ModifiedPeptide.cpp:99-103). */
int pa_add_neutral_loss(pa_scorer* s, const char* group, float mass);

/* Replaces PyAscore.__dealloc__ (Ascore.pyx:75-79). */
void pa_destroy(pa_scorer* s);

/* Text of the last error on this scorer (or of the last failed pa_create when s == NULL). */
const char* pa_last_error(const pa_scorer* s);

/* Inputs of a batch: spectra in CSR form + PSMs referring to them.  Replaces the per-PSM
 * arguments of PyAscore.score (Ascore.pyx:103-108) and the loop of __main__.py:129-164. */
typedef struct {
    int64_t n_spec;
    const int64_t* spec_off;  /* [n_spec+1] peak range of spectrum s in mz/inten */
    const double* mz;         /* m/z (float64 like np.ndarray[double]) */
    const double* inten;      /* intensities */
    int64_t n_psm;
    const int32_t* psm_spec;  /* [n_psm] spectrum of each PSM */
    const int32_t* pep_off;   /* [n_psm+1] byte range of each peptide in pep */
    const uint8_t* pep;       /* upper-case residue letters, no terminator */
    const int32_t* n_mod;     /* [n_psm] n_of_mod */
    const int32_t* max_charge;/* [n_psm] max_fragment_charge */
    const int32_t* aux_off;   /* [n_psm+1] or NULL: range in aux_pos/aux_mass */
    const uint32_t* aux_pos;  /* aux_mod_pos: 0 = N-term, else 1-based residue */
    const float* aux_mass;    /* aux_mod_mass */
    const int64_t* mod_off;   /* [n_psm+1] exclusive prefix sum of n_mod: layout of ascores/alt_sites */
    const float* inten32;     /* optional: the intensities as float32 (then `inten` may be NULL).  For callers that hold
                               * them in that precision anyway -- mzML files store 32-bit intensity arrays -- it saves a
                               * quarter of the bytes the host link carries.  (double)float is exact and monotone, so the
                               * ranks are those the reference computes on the same values handed to it as float64 */
} pa_batch;

/* Outputs (caller-allocated; any pointer may be NULL to skip that result).
 * Site indices count the modifiable residues of the peptide N->C from 0. */
typedef struct {
    uint64_t* best_sig;   /* [n_psm] bit j set = site j carries a mod in the best isoform */
    float* best_score;    /* [n_psm] best PepScore (Ascore.pyx:236-238); -1 when no isoform exists */
    int64_t* n_iso;       /* [n_psm] number of positional isoforms scored */
    int32_t* n_sites;     /* [n_psm] number of modifiable residues */
    float* ascores;       /* [mod_off[n_psm]] Ascore of the j-th mod of PSM i at mod_off[i]+j (Ascore.pyx:254-264) */
    uint64_t* alt_sites;  /* [mod_off[n_psm]] bit u set = site u is an alternative position (Ascore.pyx:266-288) */
    int32_t* psm_status;  /* [n_psm] PA_PSM_* */
} pa_results;

#define PA_KEEP_ISOFORMS 1u /* keep the batch's per-isoform table on the GPU for pa_fetch_pep_scores / pa_calculate_ambiguity */

/* Replaces PyAscore.score for n_psm PSMs at once (Ascore.pyx:103-152 -> cpp/Spectra.cpp:43-68,
 * cpp/ModifiedPeptide.cpp:105-150, cpp/Ascore.cpp:256-271).  Synchronous: results are complete on return. */
int pa_score_batch(pa_scorer* s, const pa_batch* in, const pa_results* out, uint32_t flags);

/* The same for PSMs [psm_lo, psm_hi) of the batch only.  Results land at their ABSOLUTE positions in `out`
 * (best_sig[p], ascores[mod_off[p] + j], ...), so several scorers -- one per GPU -- can each take a range of one
 * batch and fill one set of result arrays without a gather step: the sharded form of the loop in
 * pyascore/__main__.py:129-164 (pyascore_b200/shard.py cuts the ranges on spectrum boundaries). */
int pa_score_range(pa_scorer* s, const pa_batch* in, const pa_results* out, int64_t psm_lo, int64_t psm_hi,
                   uint32_t flags);

/* Several modification types in one call: scores each PSM p of `in` under the scorer s[psm_type[p]] -- its mod_group,
 * mod_mass, neutral losses, mz_error and fragment_types.  The spectra are staged and binned ONCE for all types, so a run
 * that localises, say, phospho on STY and acetyl on K pays one host-link transfer and one binning pass for its spectra;
 * "the same spectrum scored for phospho and for acetyl" is two PSM rows of the batch.  Every scorer must be a scoring
 * handle (not a binner) on the same device with the same bin_size and n_top (PA_ERR_ARG otherwise, also for n_types
 * outside 1 .. 255); none may have an asynchronous call in flight (PA_ERR_STATE).  psm_type is on the same side (host /
 * device) as the batch's arrays; NULL means every PSM is type 0.  A PSM whose type is >= n_types gets PA_PSM_BAD_INDEX.
 * Results are written as by pa_score_batch: each PSM at its own position, ascores / alt_sites at mod_off; for the PSMs
 * of type t they are bit-identical to pa_score_batch(s[t], ...) on a batch of the type-t rows alone.  PA_KEEP_ISOFORMS
 * with n_types > 1 is PA_ERR_UNSUPPORTED.  pa_counters(s[0]) describes the call; pa_last_error(s[0]) has the text of
 * a failure (pa_last_error(NULL) when s or s[0] is NULL). */
int pa_score_typed(pa_scorer* const* s, int32_t n_types, const pa_batch* in, const uint8_t* psm_type,
                   const pa_results* out, uint32_t flags);

/* Asynchronous form of pa_score_range: returns once the work is handed to the scorer's own orchestration thread
 * (the path takes one host decision per chunk -- the plan totals size the isoform scratch -- so it cannot be a
 * pure stream enqueue).  `stream` (a cudaStream_t of the scorer's device, or NULL) is honoured as a dependency:
 * everything queued on it before this call completes before the inputs are read.  psm_hi < 0 means n_psm.
 * The arrays behind `in` / `out` must stay valid until pa_wait returns; the two structs themselves are copied.
 * At most one call may be in flight per scorer (other entry points return PA_ERR_STATE meanwhile). */
int pa_score_batch_async(pa_scorer* s, const pa_batch* in, const pa_results* out, int64_t psm_lo, int64_t psm_hi,
                         uint32_t flags, void* stream);

/* Blocks until the call started by pa_score_batch_async is complete and returns its status
 * (PA_OK at once when nothing is in flight).  Results and pa_counters are valid afterwards. */
int pa_wait(pa_scorer* s);

/* Cut points for sharding a HOST batch over `world` scorers (one per GPU): cuts[0] = 0 <= cuts[1] <= ... <=
 * cuts[world] = n_psm, rank r takes PSMs [cuts[r], cuts[r+1]).  psm_spec must be non-decreasing (scan-sorted PSMs,
 * as pyascore/__main__.py:38-44 sorts them); cuts never split the hits of one spectrum.  Ranges are balanced by
 * estimated cost: isoforms x fragments + peak_weight x peaks of the spectrum / its hits (peak_weight ~ 55 for host
 * inputs, where the host -> device copy of the peaks dominates; ~ 4 for kernel time alone).  `share` (NULL = equal) gives
 * rank r the fraction share[r] / sum(share) of the cost: when every GPU of a box copies at once they do not all get the
 * same host-link bandwidth (measured: 23 vs 35 GB/s on the two halves of an 8-GPU box).  Host arithmetic only. */
int pa_shard_ranges(const pa_scorer* s, const pa_batch* in, int32_t world, double peak_weight, const double* share,
                    int64_t* cuts);
/* The same without a scorer handle (no GPU needed): mod_group as given to pa_create, the number of ion types and
 * the largest neutral-loss variant count per residue (1 without neutral losses). */
int pa_shard_ranges_for(const char* mod_group, int32_t n_types, int32_t nl_variants, const pa_batch* in,
                        int32_t world, double peak_weight, const double* share, int64_t* cuts);

/* Replaces the pep_scores property (Ascore.pyx:240-252 -> cpp/Ascore.cpp:281-303) for PSM
 * `psm` of the last batch scored with PA_KEEP_ISOFORMS.  Rows come in the reference's order
 * (libstdc++ hash-iteration order + std::sort by descending weighted score).
 * sig: bit j = site j; counts/scores: [cap x n_top] row-major (the scorer's n_top).  Returns the number of isoforms
 * (>= 0; only min(cap, n) rows are written) or a negative pa_status. */
int64_t pa_fetch_pep_scores(pa_scorer* s, int64_t psm, int64_t cap, uint64_t* sig, int32_t* counts,
                            float* scores, float* weighted, int32_t* total_fragments);

/* Replaces PyAscore.calculate_ambiguity (Ascore.pyx:208-230 -> cpp/Ascore.cpp:157-210) against
 * the peptide/spectrum of PSM `psm` of the kept batch.  scores_a / scores_b: the n_top depth scores of the two
 * isoforms (a pep_scores row of the scorer's n_top). */
int pa_calculate_ambiguity(pa_scorer* s, int64_t psm, uint64_t sig_a, const float* scores_a, float weighted_a,
                           uint64_t sig_b, const float* scores_b, float weighted_b, float* out);

/* Host-side string helper: the bracketed sequence the reference prints for a signature
 * (cpp/ModifiedPeptide.cpp:199-253).  have_sig = 0 reproduces best_sequence for "no isoform" (""). */
int pa_format_sequence(const pa_scorer* s, const uint8_t* pep, int32_t len, int32_t n_mod,
                       const uint32_t* aux_pos, const float* aux_mass, int32_t n_aux, uint64_t sig,
                       char* buf, int32_t cap);

/* 1-based residue positions of the modifiable sites of a peptide (cpp/ModifiedPeptide.cpp:184-193, +1). */
int pa_site_positions(const pa_scorer* s, const uint8_t* pep, int32_t len, int32_t* pos, int32_t cap);

/* Stage probe (tests, profiling): BinnedSpectra alone (cpp/Spectra.cpp:43-68, :24-41).
 * out_mz/out_rank use the input offsets (spec_off); out_count[s] entries are valid per spectrum,
 * sorted by m/z.  out_mz holds (float)mz exactly as the reference hands it to consumePeak. */
int pa_bin_spectra(pa_scorer* s, int64_t n_spec, const int64_t* spec_off, const double* mz,
                   const double* inten, float* out_mz, uint8_t* out_rank, int32_t* out_count);

/* BinnedSpectra probe with the cursor data PyBinnedSpectra exposes (Spectra.pyx:74-125): for every
 * retained peak also its index inside the input spectrum and its bin; per spectrum
 * out_bounds[3*s+0..2] = {min_mz, max_mz, n_bins} (cpp/Spectra.cpp:46-52).  Extra outputs may be NULL. */
int pa_bin_spectra_ex(pa_scorer* s, int64_t n_spec, const int64_t* spec_off, const double* mz,
                      const double* inten, float* out_mz, uint8_t* out_rank, int32_t* out_count,
                      int32_t* out_index, int32_t* out_bin, float* out_bounds);

/* Stage probe behind PyFragmentGraph (ModifiedPeptide.pyx:160-329 -> cpp/ModifiedPeptide.cpp:379-408,
 * :570-591): for ONE positional isoform `sig` (bit j = site j, N->C) of `pep`, ion type `fragment_type`
 * and charge `charge` (0 = neutral), the m/z of every neutral-loss variant at every residue step of
 * the traversal (N->C for b/c, C->N for y/z/Z; the last residue included).
 * out_mz[step*16 + v], v < out_nvar[step]; both arrays hold `len` steps. */
int pa_fragment_table(pa_scorer* s, const uint8_t* pep, int32_t len, const uint32_t* aux_pos,
                      const float* aux_mass, int32_t n_aux, uint64_t sig, char fragment_type, int32_t charge,
                      float* out_mz, int32_t* out_nvar);

/* Replaces PyModifiedPeptide.get_site_determining_ions (ModifiedPeptide.pyx:117-157 ->
 * cpp/ModifiedPeptide.cpp:259-320): ions of isoform a not matched (within mz_error) in isoform b and
 * vice versa, ascending, charges 1..max_charge.  Writes min(count, cap) values; counts in n_a/n_b. */
int pa_site_determining_ions(pa_scorer* s, const uint8_t* pep, int32_t len, const uint32_t* aux_pos,
                             const float* aux_mass, int32_t n_aux, uint64_t sig_a, uint64_t sig_b,
                             char fragment_type, int32_t max_charge, float* out_a, int32_t* n_a,
                             float* out_b, int32_t* n_b, int32_t cap);

/* Replaces PyLogMath / PyBinomialDist (Util.pyx:6-98 -> cpp/Util.cpp:16-83), n values at once.
 * op 0: log_sum(x[i], y[i]);  1: log_bin_coef(k[i], tr[i]);  2: log_pmf;  3: log_pvalue;
 * 4: log10_pvalue of Binomial(tr[i], prob) at k[i] successes.  Unused inputs may be NULL. */
int pa_log_math(pa_scorer* s, int32_t op, int32_t n, const float* x, const float* y, const int32_t* k,
                const int32_t* tr, float prob, float* out);

/* Replaces PyPowerSetSum (Util.pyx:100-134 -> cpp/Util.cpp:89-160): sorted, de-duplicated float32
 * sums of the subsets of `target` with at most max_depth elements (0 first).  Host arithmetic -- it is
 * the routine that also builds the neutral-loss variant table of the kernels.  Returns the count. */
int64_t pa_power_set_sums(const float* target, int32_t n, int32_t max_depth, float* out, int64_t cap);

/* Stage probe: the score table |-10 log10 P(X >= k)| for depth d (0-based), n trials, k hits
 * (cpp/Util.cpp:47-83 + cpp/Ascore.cpp:127-133).  out[(n*(n+1)/2 + k)*n_top + d], n <= n_max, d < the scorer's n_top. */
int pa_tail_table(pa_scorer* s, int32_t n_max, float* out);

typedef struct {
    int64_t n_psm, n_spec, n_peaks, n_retained, n_isoforms, n_fragment_lookups;
    int64_t bytes_h2d, bytes_d2h;      /* copied by the library during the last pa_score_batch */
    int64_t kernel_launches;           /* kernels launched by the last pa_score_batch */
    float ms_bin, ms_plan, ms_count, ms_select, ms_total; /* CUDA-event times, summed over chunks */
    int64_t launches_bin, launches_count, launches_select, launches_ascore;
    float ms_ascore, ms_narrow_wait;    /* ms_select = best-isoform selection, ms_ascore = Ascore kernels; ms_narrow_wait = host
                                           time the call spent waiting for the m/z narrowing pass (pa_narrow_mz) of a chunk */
    int64_t n_chunks;                   /* chunks the batch was cut into: every stage launches once per chunk */
    int64_t n_spec_exact;               /* spectra whose m/z kept an exact float64 copy beside the narrowed batch (pa_narrow_mz) */
    int64_t launches_deep;              /* n_top > 10 only: launches of the depth 10 .. n_top-1 counting kernel (K2d), also in */
    float ms_deep;                      /*   kernel_launches, and its CUDA-event time; both 0 for n_top = 10 */
} pa_counters_t;

/* Counters of the last pa_score_batch (roofline arithmetic: SURVEY.md section 8d). */
int pa_counters(const pa_scorer* s, pa_counters_t* out);

/* Host-side helper behind the end-to-end path of host batches: out32[i] = (float)mz[i] for every peak of the CSR block and
 * exact_flag[s] = 1 for the spectra whose kernels' view would change if the float32 values were widened back -- different
 * bounds (cpp/Spectra.cpp:46-48) or a different bin for some peak (:58-60) -- which therefore keep their float64 values.
 * pa_score_batch applies it per chunk to host inputs (on the scorer's host threads -- PA_HOST_THREADS, default min(16,
 * the process's CPUs / (scorers alive in it x LOCAL_WORLD_SIZE)) -- while the previous chunk's bytes are on the wire) so that the link carries 4 instead of
 * 8 bytes of m/z per peak; results are bit-identical by construction and by test.  By default a scorer with at least 10
 * host threads decides by measurement: of its first large host batches (>= 2^20 peaks) the first two narrow, the third does
 * not, and the faster way (peaks per second of the whole call) is kept.  PA_NARROW=0 / 1 force it off / on;
 * pa_counters_t.ms_narrow_wait is the time a call waited for the pass.
 * Returns the number of flagged spectra.  Needs no GPU. */
int64_t pa_narrow_mz(const double* mz, const int64_t* spec_off, int64_t n_spec, float bin_size, float* out32,
                     uint8_t* exact_flag);

/* Pinned host memory for CSR batches, so H2D/D2H copies run asynchronously. */
void* pa_alloc_pinned(int64_t bytes);
void pa_free_pinned(void* p);

/* The same with placement flags.  PA_PINNED_PORTABLE: pinned for every CUDA context of the process (one batch read by
 * the scorers of several GPUs).  PA_PINNED_WRITE_COMBINED: write-combined pages -- faster for the device to read on
 * some hosts, very slow for the CPU to read back: only for arrays the host writes once (m/z, intensities). */
#define PA_PINNED_WRITE_COMBINED 1u
#define PA_PINNED_PORTABLE 2u
void* pa_alloc_pinned_ex(int64_t bytes, uint32_t flags);

/* ---- mzML spectra decoded on the GPU ----
 * pa_mzml_index (host, no GPU) reads the XML structure of an mzML file held in memory; pa_decode_arrays decodes the
 * binary arrays it lists (base64, zlib, dtype conversion) on the GPU, straight into CSR peak arrays.  Together they give
 * what the stdlib reader gives for SpectraParser(path, "mzML").to_csr() (reference: spec_parsers.py:49-110, :175-282). */
#define PA_MZML_F64 0          /* MS:1000523 */
#define PA_MZML_F32 1          /* MS:1000521 */
#define PA_MZML_I32 2          /* MS:1000519 */
#define PA_MZML_I64 3          /* MS:1000522 */
#define PA_MZML_ZLIB 1         /* pa_mzml_array.flags: MS:1000574 */
#define PA_MZML_INTENSITY 2    /* pa_mzml_array.flags: intensity array (else m/z) */

typedef struct {
    int64_t text_off;   /* byte offset of the <binary> element's text in the file */
    int64_t text_len;   /* its length in bytes */
    int64_t out_off;    /* first element of the array in the output: spec_off of its spectrum */
    int64_t count;      /* expected elements: arrayLength of the binaryDataArray, else defaultArrayLength of the spectrum */
    int64_t spec;       /* its spectrum: position in the sorted index */
    int32_t dtype;      /* PA_MZML_F64 .. PA_MZML_I64 */
    int32_t flags;      /* PA_MZML_ZLIB | PA_MZML_INTENSITY */
} pa_mzml_array;

typedef struct {
    int64_t n_spec;                  /* retained spectra (ms_level filter), stably sorted by scan */
    const int64_t* scan;             /* [n_spec] scan= number of the id attribute, -1 without one */
    const int32_t* ms_level;         /* [n_spec] */
    const double* precursor_mz;      /* [n_spec] NaN = missing */
    const int32_t* precursor_charge; /* [n_spec] 0 = missing */
    const int64_t* spec_off;         /* [n_spec+1] peak ranges laid out from the expected counts */
    int64_t n_arrays;                /* two per spectrum with both arrays (m/z then intensity, in spectrum order) */
    const pa_mzml_array* arrays;
} pa_mzml_index_t;

/* Replaces the XML half of MzMLExtractor (spec_parsers.py:49-110) and SpectraParser._get_spectra (:175-282) for the
 * `n` bytes of an mzML file at `bytes`: spectra of level ms_level (0 = all), referenceableParamGroup references resolved,
 * sorted by scan (ties in file order).  Payloads of spectra the filter drops are skipped, never decoded.  Returns PA_OK
 * and *out (free it with pa_mzml_index_free), or PA_ERR_ARG with the text in err[0, err_cap): for the files the stdlib
 * reader rejects with a ValueError (several precursors, numpress) the same text, otherwise why this path refuses the
 * file (markup inside <binary>, m/z and intensity counts that differ, a missing array length ...).  Needs no GPU. */
int pa_mzml_index(const uint8_t* bytes, int64_t n, int32_t ms_level, pa_mzml_index_t** out, char* err, int32_t err_cap);
void pa_mzml_index_free(pa_mzml_index_t* index);

/* Decodes the n_arrays binary arrays of `arrays` (host memory) on CUDA device `device`: file_dev holds the file bytes on
 * that device; array j goes to (PA_MZML_INTENSITY ? inten_out : mz_out)[out_off, out_off + count) as float64.
 * status_out[j] (device): 0 = decoded, 1 = base64 text b64decode rejects (or refused: non-ASCII, '&', data after padding),
 * 2 = a zlib stream zlib.decompress rejects, 3 = decoded length other than `count` elements.  *inexact_out (device) = 1
 * when some decoded intensity is not exactly a float32 value.  Synchronous.  Returns PA_OK or a negative pa_status (text
 * in err). */
int pa_decode_arrays(int device, const uint8_t* file_dev, const pa_mzml_array* arrays, int64_t n_arrays, double* mz_out,
                     double* inten_out, int32_t* status_out, int32_t* inexact_out, char* err, int32_t err_cap);

/* The inflate core of pa_decode_arrays built for the CPU: zlib.decompress(in) into out[0, cap).  Returns the output
 * length, -1 for a stream zlib rejects (header, blocks, truncation, Adler-32), -2 when the output exceeds cap. */
int64_t pa_inflate_host(const uint8_t* in, int64_t n_in, uint8_t* out, int64_t cap);

/* Library/ABI version. */
int pa_version(void);

#ifdef __cplusplus
}
#endif
#endif
