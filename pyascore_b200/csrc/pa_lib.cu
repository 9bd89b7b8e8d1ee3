// libpyascore_b200: host orchestration + C ABI (include/pyascore_b200.h).
//
// One scorer = one GPU.  A batch is cut into chunks of PSMs (and the spectra they reference);
// chunks alternate between two CUDA streams so that the H2D copy and binning of chunk c+1
// overlap the scoring of chunk c.  The only host<->device synchronisation inside a chunk is
// the read-back of the plan totals (number of isoforms / work units), which sizes the scratch.
#include <cub/cub.cuh>
#include <cuda_runtime.h>
#include <sched.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "pa_probes.cuh"

#define PA_VERSION 200
#define PA_CHUNK_PSM 131072
#define PA_CHUNK_MIN 16384
#define PA_CHUNK_PEAKS (96ll << 20)     // peaks per chunk (1.5 GB of float64 pairs)
#define PA_TABLE_MIN 512

static thread_local std::string g_create_error;

namespace {

template <cudaError_t (*Free)(void*)>
struct OwnedMem {            // a CUDA allocation freed with its owner
    void* p = nullptr;
    size_t cap = 0;
    OwnedMem() = default;
    OwnedMem(OwnedMem&& o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
    OwnedMem& operator=(OwnedMem&& o) noexcept { std::swap(p, o.p); std::swap(cap, o.cap); return *this; }
    ~OwnedMem() { if (p) Free(p); }
    template <class T> T* as() const { return (T*)p; }
};

struct DevBuf : OwnedMem<cudaFree> {
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) { cudaError_t e = cudaFree(p); p = nullptr; cap = 0; if (e != cudaSuccess) return e; }
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { e = cudaMalloc(&p, bytes); want = bytes; }
        if (e == cudaSuccess) cap = want;
        return e;
    }
};

struct PinnedBuf : OwnedMem<cudaFreeHost> {     // page-locked host memory
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) { cudaFreeHost(p); p = nullptr; cap = 0; }
        const size_t want = bytes + bytes / 2 + 4096;
        cudaError_t e = cudaMallocHost(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
};

struct PlanTotals {          // device -> host after planning a chunk
    unsigned long long combo_bits[64];
    int max_frag, max_list;
    long long total_iso;
    int total_units;
    int max_len;
};

struct Slot {                // per-stream working set
    cudaStream_t st = nullptr;
    // staged inputs
    DevBuf spec_off, mz, inten, inten32, psm_spec, pep_off, pep, n_mod, max_charge, aux_off, aux_pos, aux_mass, mod_off, psm_type;
    // K1
    DevBuf rpk, rcount, ctab, chead, g_bin, g_tmp;
    // plan
    DevBuf psm_S, psm_status, psm_I, psm_units, iso_off, unit_off, unit_psm, totals, cub_tmp;
    // K2/K3
    DevBuf iso_lo, iso_hi, iso_n, iso_w, iso_deep, g_sort, g_lr, g_lists, lookups, sched, best_idx, mod_psm, tie, generic_list, generic_count, work_key, work_key2, work_val, work_sorted, rest_list, item_cnt, item_off, gen_flag, asc_cursor;
    // staged outputs
    DevBuf o_sig, o_score, o_niso, o_nsites, o_asc, o_alt, o_status;
    PinnedBuf h_totals, h_lookups;       // PlanTotals, unsigned long long
    // small host batches (a single PyAscore.score call): every input array packed into one pinned block and copied
    // with one transfer, every result array read back with one; the user's (pageable) arrays are touched by memcpy only
    DevBuf d_pack, d_opack, mz32, esc, escoff, bin_list, bin_list_n;
    PinnedBuf h_pack, h_opack;
    cudaEvent_t ev_plan = nullptr;
};

struct ChunkView {           // device-side views of the chunk in flight (kept for fetch calls)
    PaBatchDev b;
    int64_t n_psm = 0, psm_lo = 0;
    const int64_t* iso_off = nullptr;
    const int32_t* psm_S = nullptr;
    const int32_t* psm_status = nullptr;
    PaIso iso;
    const uint16_t* iso_deep = nullptr;    // n_top > 10: K2d counts
    int max_list = 0;
    bool valid = false;
    int slot = 0;
};

}  // namespace

// ---- host-side narrowing of the m/z array -----------------------------------------------------------------
// The end-to-end rate of a host batch is the host link's: 16 bytes per peak at ~53 GB/s.  What the kernels need from
// the float64 m/z is little -- the spectrum's bounds (cpp/Spectra.cpp:46-48), the bin of every peak (:58-60) and
// (float)m/z (Ascore.pyx:146) -- so the host may send the float32 value instead whenever it can PROVE that the value
// widened back to double gives the same bounds and the same bins; (float)m/z is then the float32 itself.  The proof
// per spectrum: the two bounds formulas evaluated on the rounded extremes, and for every peak the position of
// (m/z - min) / bin_size between two integers -- further from both than float32 rounding can move it (one multiply,
// vectorised), or else the reference's own formula evaluated on both values.  A spectrum that fails keeps an exact
// float64 copy (a few per thousand on continuous data).  Runs on a small pool of host threads owned by the scorer while
// the previous chunk's bytes are on the wire; the narrowed bytes are what the timed end-to-end region then moves.
// Host threads of one scorer's narrowing pool when PA_HOST_THREADS does not say: the CPUs this process may run on, shared
// between the scorers alive in it (MultiScorer: one per GPU) and the processes of the job on this node (one rank per GPU
// under torchrun: LOCAL_WORLD_SIZE), at most 16.  Settled when the pool starts.
static std::atomic<int> g_live_scorers{0};
static int host_thread_budget(int cpus) {
    int procs = 1;
    if (const char* e = getenv("LOCAL_WORLD_SIZE")) procs = std::max(1, atoi(e));
    const int scorers = std::max(1, g_live_scorers.load());
    return std::max(1, std::min(16, cpus / (procs * scorers)));
}

// Measured on a 16-core box (config 2, one GPU, `profiles/r06b_narrowing_threads.txt`): with 16 threads the pass keeps
// ahead of the link (end to end 11.7 -> 13.7 M PSM/s), with 8 it does not (8.3 M), with 4: 8.0 M, with 2: 4.1 M.
#define PA_NARROW_MIN_THREADS 10

struct HostPool {
    std::vector<std::thread> th;
    std::mutex mu;
    std::condition_variable cv_job, cv_done;
    std::function<void(int)> fn;
    int n_tasks = 0, next = 0, left = 0;
    uint64_t gen = 0;
    bool quit = false;
    void start(int n) {
        for (int i = 0; i < n; i++)
            th.emplace_back([this]() {
                uint64_t seen = 0;
                std::unique_lock<std::mutex> lk(mu);
                for (;;) {
                    cv_job.wait(lk, [&] { return quit || (gen != seen && next < n_tasks); });
                    if (quit) return;
                    while (next < n_tasks) {
                        const int t = next++;
                        lk.unlock();
                        fn(t);
                        lk.lock();
                        if (--left == 0) cv_done.notify_all();
                    }
                    seen = gen;
                }
            });
    }
    void run_async(int tasks, std::function<void(int)> f) {    // the pool threads alone; wait() collects
        std::lock_guard<std::mutex> lk(mu);
        fn = std::move(f); n_tasks = tasks; next = 0; left = tasks; gen++;
        cv_job.notify_all();
    }
    void wait() {
        std::unique_lock<std::mutex> lk(mu);
        cv_done.wait(lk, [&] { return left == 0; });
    }
    void run(int tasks, std::function<void(int)> f) {          // the calling thread works too
        std::unique_lock<std::mutex> lk(mu);
        fn = std::move(f); n_tasks = tasks; next = 0; left = tasks; gen++;
        cv_job.notify_all();
        while (next < n_tasks) {
            const int t = next++;
            lk.unlock();
            fn(t);
            lk.lock();
            --left;
        }
        cv_done.wait(lk, [&] { return left == 0; });
    }
    void stop() {
        { std::lock_guard<std::mutex> lk(mu); quit = true; }
        cv_job.notify_all();
        for (auto& t : th) if (t.joinable()) t.join();
        th.clear();
    }
};

struct NarrowStage {          // one of three rotating staging sets of the narrowing pass (chunk c uses set c % 3)
    PinnedBuf h_mz32;                                      // float: narrowed m/z of the chunk,
    PinnedBuf h_esc;                                       //   double: exact copies of the spectra that need them,
    PinnedBuf h_escoff;                                    //   int32_t: their per-spectrum offsets (-1: none)
    std::vector<uint8_t> flags;
    cudaEvent_t ev = nullptr;                              // the copies out of this set are done
    bool busy = false;                                     // tasks in flight on the pool
    int64_t s0 = 0, ns = 0, peak_lo = 0, npk = 0, n_esc = 0, n_flag = 0;
    bool ok = false;
};

struct pa_scorer {
    int device = 0;
    int sm_count = 148;
    std::string mod_group, frag_types;
    float bin_size = 100.f, mod_mass = 0.f, err = 0.5f;
    int n_top = PA_N_TOP;
    int n_deep = 0;                        // scoring depths beyond 10: n_top - 10 (0 for a binner, whose n_top only bins)
    float nl_mass[256];
    bool nl_has[256];
    std::vector<float> nl_values;          // distinct non-zero loss masses, index+1 = device index
    bool nl_dirty = true;
    PaCfg cfg;
    DevBuf d_T, d_logd, d_binom, d_nl_sums, d_nl_nvar, d_perm_pool, d_perm_off, d_lut;
    DevBuf d_T_deep;                       // n_top > 10: score table of depths 10 .. n_top-1 (PaDeep), same rows as d_T
    int table_n = -1;
    float lps[PA_MAX_N_TOP], lpf[PA_MAX_N_TOP];
    std::vector<int64_t> perm_off;         // [64*64]
    std::vector<uint32_t> perm_pool;
    bool perm_dirty = true;
    Slot slot[2];
    ChunkView kept;
    pa_counters_t ctr;
    std::string error;
    std::vector<cudaEvent_t> ev_pool;
    size_t ev_used = 0;
    int attr_set = 0;
    bool binner_only = false;
    HostPool pool;                         // host threads of the m/z narrowing pass (started on first use)
    NarrowStage nstage[3];
    int host_threads = 1;                  // PA_HOST_THREADS; default: see host_thread_budget
    int host_cpus = 1;                     // CPUs this process may run on
    bool host_threads_fixed = false;
    int narrow_mode = -1;                  // PA_NARROW: 0 never, 1 always, default: host chunks of >= 2^19 peaks when the scorer
                                           // has PA_NARROW_MIN_THREADS (10) host threads and the pass keeps ahead of the copies
    int narrow_state = 0;                  // default mode: 0 first (cold) narrowed call, 1 timed with the pass, 2 timed without, 3 decided
    double narrow_rate_on = 0.;            //   peaks per second of the timed call with the pass
    bool narrow_keep = true;               //   the decision (see score_impl)
    bool bin_rows = true;                  // PA_K1=topn: k_bin_topn alone (the row form k_bin_rows off)
    // pa_score_batch_async: the scorer's own orchestration thread (started on first use, parked between calls: a
    // fresh thread per call would pay thread creation and the CUDA runtime's per-thread set-up every time)
    std::thread worker;
    std::mutex mu;
    std::condition_variable cv;
    bool busy = false;                     // a call is in flight (set by the caller, cleared by pa_wait)
    bool job_ready = false, job_done = false, quit = false;
    int async_rc = PA_OK;
    pa_batch async_in;
    pa_results async_out;
    int64_t async_lo = 0, async_hi = 0;
    uint32_t async_flags = 0;
};

// Blocks of `kernel` one SM keeps resident at this block size and dynamic shared memory: the
// persistent kernels launch exactly one such wave (sm_count * resident_blocks) and loop.
template <typename K>
static int resident_blocks(K kernel, int threads, size_t smem) {
    int n = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, threads, smem) != cudaSuccess || n < 1) {
        (void)cudaGetLastError();
        n = 1;
    }
    return n;
}

// Items a warp of a persistent kernel takes per visit to the work cursor: up to `most` when every warp
// has at least eight visits' worth; with fewer than four items per warp the sign is flipped, which
// tells the kernel not to reserve its next grab ahead of time.
static int grab_size(int64_t items, int64_t warps, int most) {
    const int64_t per_warp = items / std::max<int64_t>(warps, 1);
    const int g = (int)std::max<int64_t>(1, std::min<int64_t>(most, per_warp / 8));
    return per_warp < 4 ? -g : g;
}

// Launch shape of k_bin_topn for spectra of up to `max_peaks` peaks: slot capacity, warps per block
// (the count that keeps the most warps resident per SM -- the slots are what limits occupancy) and a
// grid of one resident wave.
static void bin_launch_shape(int sm_count, int64_t max_peaks, int64_t n_spec, int* cap_out, int* wpb_out,
                             size_t* smem_out, int* blocks_out) {
    int cap = (int)std::min<int64_t>(((std::max<int64_t>(max_peaks, PA_BIN_MINCAP) + 31) / 32) * 32, 4096);
    int best_wpb = 1, best_warps = 0, best_res = 1;
    for (int wpb = 8; wpb >= 1; wpb--) {
        const size_t smem = (size_t)wpb * PA_BIN_SLOT_BYTES(cap);
        if (smem > 200 * 1024) continue;
        const int res = resident_blocks(k_bin_topn<false>, wpb * 32, smem);
        if (res * wpb > best_warps) { best_warps = res * wpb; best_wpb = wpb; best_res = res; }
    }
    *cap_out = cap; *wpb_out = best_wpb; *smem_out = (size_t)best_wpb * PA_BIN_SLOT_BYTES(cap);
    *blocks_out = (int)std::max<int64_t>(1, std::min<int64_t>((n_spec + best_wpb - 1) / best_wpb, (int64_t)sm_count * best_res));
}

// Launch shape of k_bin_rows: slots of up to PA_ROWS_MAXCAP peaks (larger spectra are declined to k_bin_topn)
#define PA_ROWS_MIN_SPECTRA 256
typedef void (*bin_rows_fn)(PaBinArgs);
static bin_rows_fn bin_rows_kernel(bool f32, bool narrow) {
    return f32 ? (narrow ? k_bin_rows<true, true> : k_bin_rows<true, false>) : (narrow ? k_bin_rows<false, true> : k_bin_rows<false, false>);
}

static void bin_rows_launch_shape(int sm_count, int64_t max_peaks, int64_t n_spec, bin_rows_fn fn, int* cap_out, int* wpb_out,
                                  size_t* smem_out, int* blocks_out) {
    const int cap = (int)std::min<int64_t>(((std::max<int64_t>(max_peaks, 64) + 31) / 32) * 32, PA_ROWS_MAXCAP);
    int best_wpb = 1, best_warps = 0, best_res = 1;
    for (int wpb = 8; wpb >= 1; wpb--) {
        const size_t smem = (size_t)wpb * PA_ROWS_SLOT_BYTES(cap);
        const int res = resident_blocks(fn, wpb * 32, smem);
        if (res * wpb > best_warps) { best_warps = res * wpb; best_wpb = wpb; best_res = res; }
    }
    *cap_out = cap; *wpb_out = best_wpb; *smem_out = (size_t)best_wpb * PA_ROWS_SLOT_BYTES(cap);
    *blocks_out = (int)std::max<int64_t>(1, std::min<int64_t>((n_spec + best_wpb - 1) / best_wpb, (int64_t)sm_count * best_res));
}

static int fail(pa_scorer* s, int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (s) s->error = buf; else g_create_error = buf;
    return code;
}

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(s, PA_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

static bool is_device_ptr(const void* p) {
    if (!p) return false;
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

// cpp/Types.h:7-30
static float residue_mass_host(char c) {
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
    return NAN;
}

// ---- neutral-loss variant table -----------------------------------------------------------------
// cpp/Util.cpp:89-160 (PowerSetSum): float32 sums of the subsets of `target` with at most max_depth
// elements, generated in the reference's recursion order (each sum = parent + element), then sorted
// and de-duplicated by exact equality.  max_depth is clamped to the target size; 0 then means "no
// limit" because the reference compares against an unsigned max_depth - 1.
static void power_set_sums(const std::vector<float>& target, size_t max_depth, std::vector<float>& sums) {
    if (target.size() < max_depth) max_depth = target.size();
    sums.clear();
    sums.push_back(0.f);
    // iterative form of initializeSums(target, start, depth): children are visited right after
    // their parent is appended, exactly like the recursion
    std::vector<std::pair<size_t, size_t>> stack;       // (next start, depth), base kept alongside
    std::vector<float> bases;
    stack.push_back({0, 0}); bases.push_back(0.f);
    while (!stack.empty()) {
        size_t& start = stack.back().first;
        const size_t depth = stack.back().second;
        const float base = bases.back();
        if (start >= target.size()) { stack.pop_back(); bases.pop_back(); continue; }
        const size_t cur = start++;
        const float v = base + target[cur];
        sums.push_back(v);
        if (cur < target.size() - 1 && depth < max_depth - 1) { stack.push_back({cur + 1, depth + 1}); bases.push_back(v); }
    }
    std::sort(sums.begin(), sums.end());
    sums.erase(std::unique(sums.begin(), sums.end()), sums.end());
}

// State = capped multiplicity (0,1,2) of each distinct loss mass on the stack, 2 bits per mass.
// For every state: PowerSetSum(stack, 2) of the residues' loss stack.  Only the multiset of the stack
// matters (sums of <= 2 elements commute, and a third copy of a mass adds no new sum).
static void build_nl_tables(const std::vector<float>& vals, std::vector<float>& sums, std::vector<uint8_t>& nvar,
                            int& nvar_cap) {
    sums.assign(256 * 16, 0.f);
    nvar.assign(256, 1);
    nvar_cap = 1;
    int g = (int)vals.size();
    for (int st = 0; st < 256; st++) {
        int cnt[4];
        bool ok = true;
        for (int v = 0; v < 4; v++) { cnt[v] = (st >> (2 * v)) & 3; if (cnt[v] == 3 || (v >= g && cnt[v])) ok = false; }
        if (!ok) continue;
        std::vector<float> stack;
        for (int v = 0; v < g; v++) for (int c = 0; c < cnt[v]; c++) stack.push_back(vals[v]);
        std::vector<float> out;
        power_set_sums(stack, 2, out);
        if (out.size() > 16) out.resize(16);   // cannot happen for g <= 4 (1 + 4 + 10 = 15)
        nvar[st] = (uint8_t)out.size();
        for (size_t i = 0; i < out.size(); i++) sums[st * 16 + i] = out[i];
        nvar_cap = std::max(nvar_cap, (int)out.size());
    }
}

static int refresh_config(pa_scorer* s) {
    PaCfg& c = s->cfg;
    c.bin_size = s->bin_size; c.mod_mass = s->mod_mass; c.err = s->err; c.n_top = s->n_top;
    c.mod_letters = 0; c.allow_n = 0; c.allow_c = 0;
    for (char ch : s->mod_group) {
        if (ch >= 'A' && ch <= 'Z') c.mod_letters |= 1u << (ch - 'A');
        if (ch == 'n') c.allow_n = 1;
        if (ch == 'c') c.allow_c = 1;
    }
    c.n_types = (int)s->frag_types.size();
    memset(c.types, 0, sizeof(c.types));
    memcpy(c.types, s->frag_types.data(), s->frag_types.size());
    c.known_letters = 0;
    for (int i = 0; i < 26; i++) {
        c.res_mass[i] = residue_mass_host((char)('A' + i));
        if (!std::isnan(c.res_mass[i])) c.known_letters |= 1u << i;
    }
    // cpp/Ascore.cpp:15-19
    const float w0[PA_N_TOP] = {0.5f, 0.75f, 1.0f, 1.0f, 1.0f, 1.0f, 0.75f, 0.5f, 0.25f, 0.25f};
    double sum = 0.;
    for (float w : w0) sum += w;
    float fsum = (float)sum;
    for (int i = 0; i < PA_N_TOP; i++) c.weights[i] = w0[i] / fsum;
    c.err_gt_half = s->err > 0.5f;
    if (s->nl_dirty) {
        s->nl_values.clear();
        memset(c.nl_upper, 0, sizeof(c.nl_upper));
        memset(c.nl_lower, 0, sizeof(c.nl_lower));
        for (int ch = 0; ch < 256; ch++) {
            if (!s->nl_has[ch] || s->nl_mass[ch] == 0.f) continue;
            float m = s->nl_mass[ch];
            int idx = -1;
            for (size_t v = 0; v < s->nl_values.size(); v++) if (s->nl_values[v] == m) idx = (int)v;
            if (idx < 0) {
                if (s->nl_values.size() >= PA_MAX_NL_MASSES)
                    return fail(s, PA_ERR_UNSUPPORTED, "more than %d distinct neutral-loss masses", PA_MAX_NL_MASSES);
                s->nl_values.push_back(m);
                idx = (int)s->nl_values.size() - 1;
            }
            if (ch >= 'A' && ch <= 'Z') c.nl_upper[ch - 'A'] = (uint8_t)(idx + 1);
            if (ch >= 'a' && ch <= 'z') c.nl_lower[ch - 'a'] = (uint8_t)(idx + 1);
        }
        c.has_nl = !s->nl_values.empty();
        std::vector<float> sums; std::vector<uint8_t> nvar;
        build_nl_tables(s->nl_values, sums, nvar, c.nvar_cap);
        CK(s->d_nl_sums.ensure(sums.size() * sizeof(float)));
        CK(s->d_nl_nvar.ensure(nvar.size()));
        CK(cudaMemcpy(s->d_nl_sums.p, sums.data(), sums.size() * sizeof(float), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(s->d_nl_nvar.p, nvar.data(), nvar.size(), cudaMemcpyHostToDevice));
        s->nl_dirty = false;
    }
    {   // global copies of the small per-letter tables (gathered per lane in the kernels)
        unsigned char lut[26 * 4 + 52];
        memcpy(lut, c.res_mass, 26 * 4);
        memcpy(lut + 104, c.nl_upper, 26);
        memcpy(lut + 130, c.nl_lower, 26);
        CK(s->d_lut.ensure(sizeof(lut)));
        CK(cudaMemcpy(s->d_lut.p, lut, sizeof(lut), cudaMemcpyHostToDevice));
        c.res_tab = s->d_lut.as<float>();
        c.nl_up_tab = s->d_lut.as<uint8_t>() + 104;
        c.nl_lo_tab = s->d_lut.as<uint8_t>() + 130;
    }
    c.nl_sums = s->d_nl_sums.as<float>();
    c.nl_nvar = s->d_nl_nvar.as<uint8_t>();
    c.binom = s->d_binom.as<uint32_t>();
    c.T = s->d_T.as<float>();
    c.table_n = s->table_n;
    return PA_OK;
}

// Score table rows 0..n_max (grown geometrically).  cpp/Ascore.cpp:23-36: p_d = 2*err*d/100.
static int ensure_table(pa_scorer* s, int n_max) {
    if (n_max <= s->table_n) return PA_OK;
    int want = std::max(PA_TABLE_MIN, s->table_n);
    while (want < n_max) want *= 2;
    want = std::min(want, (int)PA_MAX_FRAGMENTS);
    if (want < n_max) return fail(s, PA_ERR_UNSUPPORTED, "score table beyond %d trials", PA_MAX_FRAGMENTS);
    CK(cudaDeviceSynchronize());
    size_t entries = ((size_t)want + 1) * ((size_t)want + 2) / 2;
    const int nd = s->n_deep;                    // depths of the second table (PaDeep); 0 for n_top = 10
    DevBuf nt, nt_deep;
    CK(nt.ensure(entries * PA_N_TOP * sizeof(float)));
    if (nd > 0) CK(nt_deep.ensure(entries * nd * sizeof(float)));
    std::vector<double> logd(want + 2);
    logd[0] = 0.;
    for (int m = 1; m <= want + 1; m++) logd[m] = std::log((double)m);
    CK(s->d_logd.ensure(logd.size() * sizeof(double)));
    CK(cudaMemcpy(s->d_logd.p, logd.data(), logd.size() * sizeof(double), cudaMemcpyHostToDevice));
    PaTailArgs a;
    a.T = nt.as<float>();
    a.logd = s->d_logd.as<double>();
    for (int d = 0; d < PA_N_TOP + nd; d++) { a.lps[d] = s->lps[d]; a.lpf[d] = s->lpf[d]; }
    a.T_deep = nt_deep.as<float>(); a.n_top = PA_N_TOP + nd;
    volatile double one = 1.0;
    a.log10e = std::log10(std::exp(one));      // cpp/Util.cpp:82
    int n0 = 0;
    if (s->table_n >= 0) {                     // keep the rows already built
        size_t old_entries = ((size_t)s->table_n + 1) * ((size_t)s->table_n + 2) / 2;
        CK(cudaMemcpy(nt.p, s->d_T.p, old_entries * PA_N_TOP * sizeof(float), cudaMemcpyDeviceToDevice));
        if (nd > 0) CK(cudaMemcpy(nt_deep.p, s->d_T_deep.p, old_entries * nd * sizeof(float), cudaMemcpyDeviceToDevice));
        n0 = s->table_n + 1;
    }
    int rows = want - n0 + 1;
    k_tail_table<<<rows, 128, (want + 2) * sizeof(float)>>>(a, n0, want);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    s->d_T = std::move(nt);                  // (nt takes the old table and frees it)
    s->d_T_deep = std::move(nt_deep);
    s->table_n = want;
    s->cfg.T = s->d_T.as<float>();
    s->cfg.table_n = want;
    return PA_OK;
}

// ---- reference tie order ----------------------------------------------------------------------
// cpp/Ascore.cpp:54,113-120: isoforms come out of a std::unordered_map<long, ScoreContainer> that
// was filled in the first fragment graph's enumeration order.  We run the very same container
// (same libstdc++) on the same keys and record, for each hash-iteration position, the isoform's
// lexicographic rank.  One list per (sites, mods); cached for the life of the scorer.
static int ensure_perm(pa_scorer* s, int S, int k) {
    if (s->perm_off[S * 64 + k] >= 0) return PA_OK;
    const bool fwd = (s->frag_types[0] == 'b' || s->frag_types[0] == 'c');
    std::vector<int> c(k);
    for (int i = 0; i < k; i++) c[i] = i;
    // binomials for ranking
    std::vector<std::vector<unsigned long long>> C(65, std::vector<unsigned long long>(65, 0));
    for (int n = 0; n <= 64; n++) { C[n][0] = 1; for (int j = 1; j <= n; j++) C[n][j] = std::min<unsigned long long>(C[n - 1][j - 1] + (j <= n - 1 ? C[n - 1][j] : 0), 1ull << 62); }
    std::unordered_map<long, uint32_t> m;
    for (;;) {
        long key = 0;
        unsigned long long bits = 0;
        for (int i = 0; i < k; i++) {
            int site = fwd ? c[i] : S - 1 - c[i];
            key |= 1l << (S - 1 - site);
            bits |= 1ull << site;
        }
        // lexicographic rank of the site set (N->C)
        unsigned long long r = 0;
        int prev = -1, i = 0;
        for (int site = 0; site < S; site++)
            if ((bits >> site) & 1ull) {
                for (int j = prev + 1; j < site; j++) r += C[S - 1 - j][k - 1 - i];
                prev = site; i++;
            }
        m[key] = (uint32_t)r;
        int q = k - 1;
        while (q >= 0 && c[q] == S - k + q) q--;
        if (q < 0) break;
        c[q]++;
        for (int j = q + 1; j < k; j++) c[j] = c[j - 1] + 1;
    }
    s->perm_off[S * 64 + k] = (int64_t)s->perm_pool.size();
    for (auto& kv : m) s->perm_pool.push_back(kv.second);
    s->perm_dirty = true;
    return PA_OK;
}

static int upload_perms(pa_scorer* s) {
    if (!s->perm_dirty) return PA_OK;
    CK(cudaDeviceSynchronize());
    CK(s->d_perm_pool.ensure(std::max<size_t>(s->perm_pool.size(), 1) * sizeof(uint32_t)));
    CK(s->d_perm_off.ensure(s->perm_off.size() * sizeof(int64_t)));
    if (!s->perm_pool.empty())
        CK(cudaMemcpy(s->d_perm_pool.p, s->perm_pool.data(), s->perm_pool.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(s->d_perm_off.p, s->perm_off.data(), s->perm_off.size() * sizeof(int64_t), cudaMemcpyHostToDevice));
    s->perm_dirty = false;
    return PA_OK;
}

static cudaEvent_t next_event(pa_scorer* s) {
    if (s->ev_used == s->ev_pool.size()) {
        cudaEvent_t e = nullptr;
        if (cudaEventCreate(&e) != cudaSuccess) { (void)cudaGetLastError(); return nullptr; }   // cudaEventRecord(nullptr) then reports the failure
        s->ev_pool.push_back(e);
    }
    return s->ev_pool[s->ev_used++];
}

// ---------------------------------------------------------------------------------------------
extern "C" int pa_version(void) { return PA_VERSION; }

extern "C" const char* pa_last_error(const pa_scorer* s) { return s ? s->error.c_str() : g_create_error.c_str(); }

extern "C" void* pa_alloc_pinned(int64_t bytes) {
    void* p = nullptr;
    if (cudaMallocHost(&p, (size_t)std::max<int64_t>(bytes, 1)) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}

extern "C" void* pa_alloc_pinned_ex(int64_t bytes, uint32_t flags) {
    void* p = nullptr;
    unsigned f = cudaHostAllocDefault;
    if (flags & PA_PINNED_WRITE_COMBINED) f |= cudaHostAllocWriteCombined;
    if (flags & PA_PINNED_PORTABLE) f |= cudaHostAllocPortable;
    if (cudaHostAlloc(&p, (size_t)std::max<int64_t>(bytes, 1), f) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}

extern "C" void pa_free_pinned(void* p) { if (p) cudaFreeHost(p); }

static int create_scorer(float bin_size, int n_top, const char* mod_group, float mod_mass, float mz_error,
                         const char* fragment_types, int device, bool binner_only, pa_scorer** out) {
    pa_scorer* s = nullptr;
    if (!out || !mod_group || !fragment_types) return fail(nullptr, PA_ERR_ARG, "NULL argument");
    *out = nullptr;
    if (binner_only ? (n_top < 1 || n_top > 254) : (n_top < PA_N_TOP || n_top > PA_MAX_N_TOP))
        return fail(nullptr, PA_ERR_UNSUPPORTED, "n_top must be in %d..%d: below %d the reference reads past the end of its "
                    "%d score weights; above %d is beyond what the oracle models and beyond the tested envelope",
                    PA_N_TOP, PA_MAX_N_TOP, PA_N_TOP, PA_N_TOP, PA_MAX_N_TOP);
    if (!(bin_size > 0.f)) return fail(nullptr, PA_ERR_ARG, "bin_size must be positive");
    size_t nt = strlen(fragment_types);
    if (nt == 0 || nt > 7) return fail(nullptr, PA_ERR_ARG, "fragment_types must hold 1..7 characters");
    for (size_t i = 0; i < nt; i++)
        if (!strchr("bcyzZ", fragment_types[i]))
            return fail(nullptr, PA_ERR_ARG, "fragment type '%c' not in \"bcyzZ\"", fragment_types[i]);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, PA_ERR_CUDA, "no CUDA device available (%s); this library has no CPU path",
                    cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(nullptr, PA_ERR_ARG, "device %d out of range (0..%d)", device, ndev - 1);
    e = cudaSetDevice(device);
    if (e != cudaSuccess) return fail(nullptr, PA_ERR_CUDA, "cudaSetDevice: %s", cudaGetErrorString(e));
    s = new pa_scorer();
    s->device = device;
    s->binner_only = binner_only;
    if (!binner_only) g_live_scorers++;
    {
        int cpus = (int)std::thread::hardware_concurrency();
        cpu_set_t set;
        if (sched_getaffinity(0, sizeof(set), &set) == 0) cpus = CPU_COUNT(&set);
        s->host_cpus = std::max(1, cpus);
        s->host_threads = std::max(1, std::min(16, cpus / std::max(ndev, 1)));       // (settled at the pool's start: host_thread_budget)
        if (const char* e = getenv("PA_HOST_THREADS")) { s->host_threads = std::max(1, std::min(64, atoi(e))); s->host_threads_fixed = true; }
        if (const char* e = getenv("PA_K1")) s->bin_rows = strcmp(e, "topn") != 0;
        if (const char* e = getenv("PA_NARROW")) s->narrow_mode = (e[0] == '0') ? 0 : (e[0] == '1' ? 1 : -1);
    }
    cudaDeviceGetAttribute(&s->sm_count, cudaDevAttrMultiProcessorCount, device);
    s->mod_group = mod_group; s->frag_types = fragment_types;
    s->bin_size = bin_size; s->mod_mass = mod_mass; s->err = mz_error; s->n_top = n_top;
    s->n_deep = binner_only ? 0 : n_top - PA_N_TOP;
    memset(s->nl_mass, 0, sizeof(s->nl_mass));
    memset(s->nl_has, 0, sizeof(s->nl_has));
    memset(&s->ctr, 0, sizeof(s->ctr));
    memset(&s->cfg, 0, sizeof(s->cfg));
    s->perm_off.assign(64 * 64, -1);
    // cpp/Ascore.cpp:23-36 + cpp/Util.cpp:52-55 (platform libm, like the reference)
    for (int d = 1; d <= PA_N_TOP + s->n_deep; d++) {
        float p = (float)((double)((2 * mz_error) * (float)d) / 100.);
        s->lps[d - 1] = logf(p);
        s->lpf[d - 1] = (float)log(1. - (double)p);
    }
    // saturating binomials
    std::vector<uint32_t> bin(64 * 64, 0);
    {
        std::vector<std::vector<unsigned long long>> C(64, std::vector<unsigned long long>(64, 0));
        for (int n = 0; n < 64; n++) {
            C[n][0] = 1;
            for (int k = 1; k <= n; k++) C[n][k] = std::min<unsigned long long>(C[n - 1][k - 1] + (k <= n - 1 ? C[n - 1][k] : 0), 0xffffffffull);
            for (int k = 0; k <= n; k++) bin[n * 64 + k] = (uint32_t)C[n][k];
        }
    }
    int rc = PA_OK;
    auto init = [&]() -> int {
        CK(s->d_binom.ensure(bin.size() * sizeof(uint32_t)));
        CK(cudaMemcpy(s->d_binom.p, bin.data(), bin.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
        {   // z * 1.007825 as the reference forms it (cpp/ModifiedPeptide.cpp:586), in IEEE double
            double zm[16];
            for (int z = 0; z < 16; z++) { volatile double zd = (double)z; zm[z] = zd * 1.007825; }
            CK(cudaMemcpyToSymbol(c_zmass, zm, sizeof(zm)));
        }
        CK(cudaEventCreateWithFlags(&s->nstage[2].ev, cudaEventDisableTiming));
        for (int i = 0; i < 2; i++) {
            CK(cudaStreamCreateWithFlags(&s->slot[i].st, cudaStreamNonBlocking));
            CK(s->slot[i].h_totals.ensure(sizeof(PlanTotals)));
            CK(s->slot[i].h_lookups.ensure(sizeof(unsigned long long)));
            CK(cudaEventCreateWithFlags(&s->slot[i].ev_plan, cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&s->nstage[i].ev, cudaEventDisableTiming));
        }
        CK(cudaFuncSetAttribute(k_ascore_generic<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        CK(cudaFuncSetAttribute(k_ascore_pairs<PA_MAXSTREAM, 3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(AscSm)));
        if (s->n_deep > 0) {
            CK(cudaFuncSetAttribute(k_ascore_generic<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
            CK(cudaFuncSetAttribute(k_ascore_pairs<PA_MAXSTREAM, 3, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(AscSm)));
            CK(cudaFuncSetAttribute(k_count_deep<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
            CK(cudaFuncSetAttribute(k_count_deep<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        }
        CK(cudaFuncSetAttribute(k_bin_topn<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        CK(cudaFuncSetAttribute(k_bin_topn<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        for (int v = 0; v < 4; v++)
            CK(cudaFuncSetAttribute(bin_rows_kernel((v & 1) != 0, (v & 2) != 0), cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        CK(cudaFuncSetAttribute(k_tail_table, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        CK(cudaFuncSetAttribute(k_ambiguity, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
        int r = refresh_config(s);
        if (r != PA_OK) return r;
        return ensure_table(s, PA_TABLE_MIN);
    };
    rc = init();
    if (rc != PA_OK) { g_create_error = s->error; pa_destroy(s); return rc; }
    *out = s;
    return PA_OK;
}

extern "C" int pa_create(float bin_size, int n_top, const char* mod_group, float mod_mass, float mz_error,
                         const char* fragment_types, int device, pa_scorer** out) {
    return create_scorer(bin_size, n_top, mod_group, mod_mass, mz_error, fragment_types, device, false, out);
}

extern "C" int pa_create_binner(float bin_size, int n_top, int device, pa_scorer** out) {
    return create_scorer(bin_size, n_top, "STY", 79.966331f, 0.5f, "by", device, true, out);
}

extern "C" int pa_add_neutral_loss(pa_scorer* s, const char* group, float mass) {
    if (!s || !group) return PA_ERR_ARG;
    CK(cudaSetDevice(s->device));
    float old_mass[256]; bool old_has[256];
    memcpy(old_mass, s->nl_mass, sizeof(old_mass)); memcpy(old_has, s->nl_has, sizeof(old_has));
    for (const char* c = group; *c; c++) { s->nl_mass[(unsigned char)*c] = mass; s->nl_has[(unsigned char)*c] = true; }
    s->nl_dirty = true;
    CK(cudaDeviceSynchronize());
    int rc = refresh_config(s);
    if (rc != PA_OK) { memcpy(s->nl_mass, old_mass, sizeof(old_mass)); memcpy(s->nl_has, old_has, sizeof(old_has)); s->nl_dirty = true; refresh_config(s); }
    s->kept.valid = false;
    return rc;
}

extern "C" void pa_destroy(pa_scorer* s) {
    if (!s) return;
    if (s->worker.joinable()) {
        if (s->busy) pa_wait(s);
        { std::lock_guard<std::mutex> lk(s->mu); s->quit = true; }
        s->cv.notify_all();
        s->worker.join();
    }
    cudaSetDevice(s->device);
    cudaDeviceSynchronize();
    s->pool.stop();
    for (NarrowStage& ns : s->nstage) if (ns.ev) cudaEventDestroy(ns.ev);
    for (Slot& sl : s->slot) {
        if (sl.ev_plan) cudaEventDestroy(sl.ev_plan);
        if (sl.st) cudaStreamDestroy(sl.st);
    }
    for (cudaEvent_t e : s->ev_pool) cudaEventDestroy(e);
    if (!s->binner_only) g_live_scorers--;
    delete s;                                          // frees every buffer
}

// ---- staging ------------------------------------------------------------------------------------
// One array of a chunk on its way to or from the device.  The device view it produces is indexed like the caller's
// array (absolute indices lo..lo+n-1); it is null when the caller passed no array.
struct ChunkArray {
    const void* arr = nullptr;       // the caller's array (host or device), or null
    int64_t lo = 0, n = 0;           // the chunk's elements [lo, lo + n)
    size_t elem = 0;                 // element size
    DevBuf* buf = nullptr;           // the slot's staging buffer (per-array transfers)
    void* view = nullptr;            // the T* (T: the element type) that receives the device view
    size_t off = 0;                  // packed transfers: offset in the block
    ChunkArray() = default;
    template <class T> ChunkArray(T* arr, int64_t lo, int64_t n, DevBuf& buf, T*& view)
        : arr(arr), lo(lo), n(n), elem(sizeof(T)), buf(&buf), view(&view) {}
    size_t bytes() const { return (size_t)std::max<int64_t>(n, 0) * elem; }
    void set_view(const unsigned char* base) const {        // base: where element `lo` is (null: no view)
        const unsigned char* v = base ? base - lo * (int64_t)elem : nullptr;
        memcpy(view, &v, sizeof(v));                        // (the view's pointer type is known to the caller only)
    }
};

// Per-array transfers.  An array on the device is used in place; a host array gets the slot's buffer, and with `h2d`
// given (inputs) its elements are copied there and counted.
static cudaError_t stage(const ChunkArray& a, bool on_dev, cudaStream_t st, int64_t* h2d) {
    if (!a.arr || on_dev) {
        a.set_view(a.arr ? (const unsigned char*)a.arr + a.lo * (int64_t)a.elem : nullptr);
        return cudaSuccess;
    }
    cudaError_t e = a.buf->ensure(std::max(a.bytes(), a.elem));
    if (e != cudaSuccess) return e;
    if (h2d && a.n > 0) {
        e = cudaMemcpyAsync(a.buf->p, (const unsigned char*)a.arr + a.lo * (int64_t)a.elem, a.bytes(), cudaMemcpyHostToDevice, st);
        if (e != cudaSuccess) return e;
        *h2d += (int64_t)a.bytes();
    }
    a.set_view(a.buf->as<unsigned char>());
    return cudaSuccess;
}

static cudaError_t copy_back(const ChunkArray& a, bool on_dev, cudaStream_t st, int64_t* d2h) {
    if (!a.arr || on_dev || a.n <= 0) return cudaSuccess;
    *d2h += (int64_t)a.bytes();
    return cudaMemcpyAsync((unsigned char*)a.arr + a.lo * (int64_t)a.elem, a.buf->p, a.bytes(), cudaMemcpyDeviceToHost, st);
}

#define PA_PACK_MAX (1 << 20)            // host batches up to this many input bytes travel as one packed block

// Packed transfers of a small host batch: the arrays the caller passed are laid out in one block from byte `used` on,
// each at a 16-byte aligned offset, with their device views in the block at `dev`.  Returns the block's size.
static size_t pack_layout(ChunkArray* list, size_t count, size_t used, unsigned char* dev) {
    for (size_t i = 0; i < count; i++) {
        ChunkArray& a = list[i];
        if (!a.arr) { a.set_view(nullptr); continue; }
        a.off = (used + 15) & ~(size_t)15;
        a.set_view(dev + a.off);
        used = a.off + a.bytes();
    }
    return used;
}

// (pa_host.cpp: vectorised with the host compiler's AVX2 when the CPU has it)
void pa_narrow_spectra(const double* mz, const int64_t* spec_off, int64_t sa, int64_t sb, int64_t peak_base,
                       float bin_size, float* out32, uint8_t* flag);

extern "C" int64_t pa_narrow_mz(const double* mz, const int64_t* spec_off, int64_t n_spec, float bin_size, float* out32,
                                uint8_t* exact_flag) {
    if (!mz || !spec_off || !out32 || !exact_flag || n_spec < 0 || !(bin_size > 0.f)) return PA_ERR_ARG;
    pa_narrow_spectra(mz, spec_off, 0, n_spec, spec_off[0], bin_size, out32, exact_flag);
    int64_t n = 0;
    for (int64_t s = 0; s < n_spec; s++) n += exact_flag[s];
    return n;
}

// ---- range ends of a device-resident batch --------------------------------------------------------
// A device-resident batch is scored as one chunk.  Measured on config 2 (1 M PSMs): 1 chunk 91.5 M PSM/s, 2 chunks
// 94.1 M, 4 chunks 84.0 M, 8 chunks 70.2 M -- the persistent kernels of two chunks cannot share an SM (registers /
// shared memory), so more chunks only add launches and tails.  One chunk keeps the per-kernel event times free of
// overlap, which the roofline arithmetic relies on.
struct DevBounds {
    int bad;                            // see k_check_batch
    int max_peaks;                      // largest spectrum of the batch
    int64_t n_aux;                      // fixed-mod entries of the range
    int64_t s0, s1;                     // first spectrum the range references, one past the last
    int64_t peak0, peak1;               // spec_off at s0 / s1
    int64_t pep0, pep1, mod0, mod1;     // pep_off / mod_off at p_lo / p_hi
};

// Range ends of the non-empty PSM range [p_lo, p_hi): one thread, so that the host needs one copy, not one per value.
__global__ void k_dev_bounds(const int64_t* spec_off, const int32_t* psm_spec, const int32_t* pep_off,
                             const int32_t* aux_off, const int64_t* mod_off, int64_t p_lo, int64_t p_hi, int64_t n_spec,
                             DevBounds* o) {
    int64_t s0 = psm_spec[p_lo], s1 = (int64_t)psm_spec[p_hi - 1] + 1;
    s0 = s0 < 0 ? 0 : (s0 > n_spec ? n_spec : s0);
    s1 = s1 < 0 ? 0 : (s1 > n_spec ? n_spec : s1);
    o->n_aux = aux_off ? (int64_t)aux_off[p_hi] - (int64_t)aux_off[p_lo] : 0;
    o->s0 = s0; o->s1 = s1;
    o->peak0 = spec_off[s0]; o->peak1 = spec_off[s1];
    o->pep0 = pep_off[p_lo]; o->pep1 = pep_off[p_hi];
    o->mod0 = mod_off[p_lo]; o->mod1 = mod_off[p_hi];
}

// Consistency of a device-resident batch (the host path checks the same things per chunk): `bad` bit 0 =
// psm_spec decreasing or out of range (the batch is then scored as one chunk over every spectrum),
// bit 1 = an offset array is not a non-decreasing CSR index or mod_off does not follow n_mod (PA_ERR_ARG).
__global__ void k_check_batch(const int32_t* psm_spec, const int32_t* pep_off, const int32_t* aux_off,
                              const int32_t* n_mod, const int64_t* mod_off, const int64_t* spec_off, int64_t p_lo,
                              int64_t p_hi, int64_t n_spec, int* bad) {
    int b = 0;
    for (int64_t p = p_lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < p_hi; p += (int64_t)gridDim.x * blockDim.x) {
        const int32_t v = psm_spec[p];
        if (v < 0 || v >= n_spec || (p > p_lo && v < psm_spec[p - 1])) b |= 1;
        if (pep_off[p + 1] < pep_off[p] || pep_off[p] < 0) b |= 2;
        if (aux_off && (aux_off[p + 1] < aux_off[p] || aux_off[p] < 0)) b |= 2;
        if (mod_off[p + 1] - mod_off[p] != (int64_t)(n_mod[p] > 0 ? n_mod[p] : 0) || mod_off[p] < 0) b |= 2;
    }
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n_spec; q += (int64_t)gridDim.x * blockDim.x)
        if (spec_off[q + 1] < spec_off[q] || spec_off[q] < 0) b |= 2;
    for (int o = 16; o > 0; o >>= 1) b |= __shfl_xor_sync(0xffffffffu, b, o);
    if (b && (threadIdx.x & 31) == 0) atomicOr(bad, b);
}

struct ChunkRange { int64_t p0, p1, s0, s1; };

struct PassEvents {               // one scoring pass of a chunk: one per type that has PSMs in it
    cudaEvent_t e_plan0, e_plan1, e_cnt0, e_cnt1, e_sel1, e_asc1;
    cudaEvent_t e_deep1 = nullptr;   // n_top > 10: end of K2d (which starts at e_cnt1)
};

struct ChunkState {              // what the back half of a chunk needs from the front half
    ChunkRange r;
    PaBatchDev b;
    int64_t mod_lo = 0, mod_hi = 0;
    const int64_t* mod_off_abs = nullptr;
    const uint8_t* psm_type = nullptr;   // typed batches: chunk-relative view of the PSMs' types
    std::vector<int> types;          // the types with PSMs in the chunk, in pass order (untyped: {0})
    cudaEvent_t e_bin0, e_bin1;
    std::vector<PassEvents> ev;      // [pass]
    uint64_t* o_sig; float* o_score; int64_t* o_niso; int32_t* o_nsites; float* o_asc; uint64_t* o_alt; int32_t* o_status;
    ChunkArray res[7];               // the result arrays (views: the o_* above)
    bool single_chunk = false;       // the call has one chunk
    bool packed = false;             // inputs travel as one block (small host batch)
    bool packed_res = false;         // ... and so do the results, in a block of this size:
    size_t packed_res_bytes = 0;
};

// Narrowing of the m/z of host chunk `r` into staging set `ns`: narrow_begin hands the per-spectrum work to the pool and
// returns; narrow_end waits for it and lays out the exact copies.  The pipeline runs it one chunk ahead of the copies.
static int narrow_begin(pa_scorer* s, NarrowStage& ns, const pa_batch* in, const ChunkRange& r) {
    ns.ok = false; ns.busy = false;
    ns.s0 = r.s0; ns.ns = r.s1 - r.s0;
    ns.peak_lo = in->spec_off[r.s0]; ns.npk = in->spec_off[r.s1] - ns.peak_lo;
    if (ns.ns <= 0 || !(s->narrow_mode == 1 || (s->narrow_mode < 0 && ns.npk >= (1 << 19)))) return PA_OK;
    // the pass runs a chunk ahead of that chunk's consistency check (prepare_host_chunk): it only touches a chunk whose
    // spectrum offsets ascend -- anything else goes unnarrowed and is refused by the check when its turn comes
    for (int64_t q = r.s0; q < r.s1; q++)
        if (in->spec_off[q + 1] < in->spec_off[q]) return PA_OK;
    CK(cudaEventSynchronize(ns.ev));                      // the chunk that used this set three chunks ago has left it
    CK(ns.h_mz32.ensure((size_t)ns.npk * 4));
    CK(ns.h_escoff.ensure((size_t)ns.ns * 4));
    ns.flags.resize((size_t)ns.ns);
    if (s->pool.th.empty()) s->pool.start(std::max(1, s->host_threads));
    const int tasks = (int)std::min<int64_t>(ns.ns, (int64_t)s->host_threads * 4);
    const double* mzh = in->mz; const int64_t* offh = in->spec_off;
    float* o32 = ns.h_mz32.as<float>(); uint8_t* fl = ns.flags.data() - r.s0;
    const float bsz = s->bin_size;
    const int64_t s0 = r.s0, nsp = ns.ns, peak_lo = ns.peak_lo, npk = ns.npk;
    s->pool.run_async(tasks, [=](int t) {
        // tasks of about equal peak counts: cut the chunk's peak range evenly, snap to spectrum starts
        const int64_t lo = peak_lo + npk * t / tasks, hi = peak_lo + npk * (t + 1) / tasks;
        const int64_t sa = std::lower_bound(offh + s0, offh + s0 + nsp, lo) - offh;
        const int64_t sb = (t + 1 == tasks) ? s0 + nsp : std::lower_bound(offh + s0, offh + s0 + nsp, hi) - offh;
        pa_narrow_spectra(mzh, offh, sa, sb, peak_lo, bsz, o32, fl);
    });
    ns.busy = true;
    return PA_OK;
}

static int narrow_end(pa_scorer* s, NarrowStage& ns, const pa_batch* in) {
    if (!ns.busy) return PA_OK;
    {
        const auto t0 = std::chrono::steady_clock::now();
        s->pool.wait();
        s->ctr.ms_narrow_wait += std::chrono::duration<float, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
    ns.busy = false;
    ns.n_esc = 0; ns.n_flag = 0;
    for (int64_t q = 0; q < ns.ns; q++)
        if (ns.flags[q]) { ns.n_esc += in->spec_off[ns.s0 + q + 1] - in->spec_off[ns.s0 + q]; ns.n_flag++; }
    if (ns.n_esc * 4 > ns.npk) return PA_OK;              // m/z that sit on bin boundaries wholesale: nothing to gain
    CK(ns.h_esc.ensure((size_t)std::max<int64_t>(ns.n_esc, 1) * 8));
    int32_t* escoff = ns.h_escoff.as<int32_t>();
    int64_t eo = 0;
    for (int64_t q = 0; q < ns.ns; q++) {
        escoff[q] = -1;
        if (!ns.flags[q]) continue;
        const int64_t o = in->spec_off[ns.s0 + q], P = in->spec_off[ns.s0 + q + 1] - o;
        escoff[q] = (int32_t)eo;
        memcpy(ns.h_esc.as<double>() + eo, in->mz + o, (size_t)P * 8);
        eo += P;
    }
    ns.ok = true;
    return PA_OK;
}

static int chunk_plan(pa_scorer* s, pa_scorer* ts, int si, ChunkState& cs, int pass, int n_types);

// Staging of a chunk, K1 and the plan of the chunk's first pass.  psm_type: the typed batch's types (null: untyped).
static int chunk_front(pa_scorer* s, pa_scorer* const* sc, int n_types, int si, const pa_batch* in, const uint8_t* psm_type,
                       bool in_dev, const ChunkRange& r, int64_t mod_lo, int64_t mod_hi, int max_peaks, ChunkState& cs,
                       const DevBounds* ends_dev, NarrowStage* nst = nullptr) {
    Slot& sl = s->slot[si];
    cudaStream_t st = sl.st;
    const int64_t np = r.p1 - r.p0, ns = r.s1 - r.s0;
    int64_t peak_lo, peak_hi, pep_lo, pep_hi, aux_lo = 0, aux_hi = 0;
    if (in_dev) {
        // offsets live on the device: score_impl fetched the range ends in one go
        peak_lo = ends_dev->peak0; peak_hi = ends_dev->peak1; pep_lo = ends_dev->pep0; pep_hi = ends_dev->pep1;
    } else {
        peak_lo = in->spec_off[r.s0]; peak_hi = in->spec_off[r.s1];
        pep_lo = in->pep_off[r.p0]; pep_hi = in->pep_off[r.p1];
        if (in->aux_off) { aux_lo = in->aux_off[r.p0]; aux_hi = in->aux_off[r.p1]; }
    }
    const int64_t npk = peak_hi - peak_lo;
    cs.r = r; cs.mod_lo = mod_lo; cs.mod_hi = mod_hi;
    int64_t* h2d = &s->ctr.bytes_h2d;
    PaBatchDev& b = cs.b;
    const double *v_mz = nullptr, *v_int = nullptr;
    const float* v_int32 = nullptr;
    ChunkArray ins[] = {
        {in->spec_off, r.s0, ns + 1, sl.spec_off, b.spec_off},
        {in->mz, peak_lo, npk, sl.mz, v_mz},
        in->inten32 ? ChunkArray(in->inten32, peak_lo, npk, sl.inten32, v_int32) : ChunkArray(in->inten, peak_lo, npk, sl.inten, v_int),
        {in->psm_spec, r.p0, np, sl.psm_spec, b.psm_spec},
        {in->pep_off, r.p0, np + 1, sl.pep_off, b.pep_off},
        {in->pep, pep_lo, pep_hi - pep_lo, sl.pep, b.pep},
        {in->n_mod, r.p0, np, sl.n_mod, b.n_mod},
        {in->max_charge, r.p0, np, sl.max_charge, b.max_charge},
        {in->aux_off, r.p0, np + 1, sl.aux_off, b.aux_off},
        {in->aux_off ? in->aux_pos : nullptr, aux_lo, aux_hi - aux_lo, sl.aux_pos, b.aux_pos},
        {in->aux_off ? in->aux_mass : nullptr, aux_lo, aux_hi - aux_lo, sl.aux_mass, b.aux_mass},
        {in->mod_off, r.p0, np + 1, sl.mod_off, cs.mod_off_abs},
        {psm_type, r.p0, psm_type ? np : 0, sl.psm_type, cs.psm_type},
    };
    const ChunkArray& mz_in = ins[1];
    // packed block bound: every array at full size, the absent ones too, and 16 bytes of alignment for each
    size_t pack_bytes = 16 * 16;
    for (const ChunkArray& a : ins) pack_bytes += (size_t)a.n * a.elem;
    bool narrowed = false;
    cs.packed = !in_dev && cs.single_chunk && pack_bytes <= PA_PACK_MAX && s->narrow_mode != 1 && !(nst != nullptr && nst->busy);
    if (cs.packed) {
        CK(sl.h_pack.ensure(pack_bytes));
        CK(sl.d_pack.ensure(pack_bytes));
        const size_t used = pack_layout(ins, sizeof(ins) / sizeof(ins[0]), 0, sl.d_pack.as<unsigned char>());
        for (const ChunkArray& a : ins)
            if (a.arr && a.n > 0) memcpy(sl.h_pack.as<unsigned char>() + a.off, (const unsigned char*)a.arr + a.lo * (int64_t)a.elem, a.bytes());
        CK(cudaMemcpyAsync(sl.d_pack.p, sl.h_pack.p, used, cudaMemcpyHostToDevice, st));
        *h2d += (int64_t)used;
    } else {
    for (const ChunkArray& a : ins)
        if (&a != &mz_in) CK(stage(a, in_dev, st, h2d));
    // host batches: the m/z array goes over the link as float32 wherever the host proved that nothing the kernels
    // derive from it changes (narrow_begin / narrow_end); spectra that failed the proof come with an exact copy.  It goes
    // last: the chunk's other arrays are on the wire while the pool finishes the chunk's narrowing.
    if (nst != nullptr && nst->busy) { const int nrc = narrow_end(s, *nst, in); if (nrc != PA_OK) return nrc; }
    if (nst != nullptr && nst->ok) {
        CK(sl.mz32.ensure((size_t)std::max<int64_t>(npk, 1) * 4));
        CK(sl.escoff.ensure((size_t)ns * 4));
        CK(sl.esc.ensure((size_t)std::max<int64_t>(nst->n_esc, 1) * 8));
        CK(cudaMemcpyAsync(sl.mz32.p, nst->h_mz32.p, (size_t)npk * 4, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(sl.escoff.p, nst->h_escoff.p, (size_t)ns * 4, cudaMemcpyHostToDevice, st));
        if (nst->n_esc > 0) CK(cudaMemcpyAsync(sl.esc.p, nst->h_esc.p, (size_t)nst->n_esc * 8, cudaMemcpyHostToDevice, st));
        CK(cudaEventRecord(nst->ev, st));
        *h2d += npk * 4 + ns * 4 + nst->n_esc * 8;
        s->ctr.n_spec_exact += nst->n_flag;
        narrowed = true;
    }
    if (!narrowed) CK(stage(mz_in, in_dev, st, h2d));
    }
    // PSM-indexed views become chunk-relative
    b.psm_spec += r.p0; b.pep_off += r.p0; b.n_mod += r.p0; b.max_charge += r.p0;
    if (b.aux_off) b.aux_off += r.p0;
    cs.mod_off_abs += r.p0;
    if (cs.psm_type) cs.psm_type += r.p0;
    b.spec_base = 0; b.n_spec = r.s1;   // spectrum indices stay absolute (views are pre-offset)

    // K1 buffers, indexed by absolute peak / spectrum index
    CK(sl.rpk.ensure((size_t)std::max<int64_t>(npk, 1) * sizeof(float2)));
    CK(sl.g_bin.ensure((size_t)std::max<int64_t>(npk, 1) * sizeof(int32_t)));
    CK(sl.g_tmp.ensure((size_t)std::max<int64_t>(npk, 1)));
    CK(sl.rcount.ensure((size_t)std::max<int64_t>(ns, 1) * sizeof(int32_t)));
    CK(sl.ctab.ensure((size_t)std::max<int64_t>(ns, 1) * PA_NCELL));
    CK(sl.chead.ensure((size_t)std::max<int64_t>(ns, 1) * sizeof(float2)));
    PaBinArgs ba;
    ba.spec_off = b.spec_off + r.s0;          // kernel indexes spectra 0..ns-1
    ba.mz = v_mz; ba.inten = v_int; ba.inten32 = v_int32; ba.peak_base = 0; ba.n_spec = ns;
    ba.mz32 = narrowed ? sl.mz32.as<float>() - peak_lo : nullptr;
    ba.esc_off = narrowed ? sl.escoff.as<int32_t>() : nullptr; ba.mz_esc = narrowed ? sl.esc.as<double>() : nullptr;
    ba.rpk = sl.rpk.as<float2>() - peak_lo; ba.rmz = nullptr; ba.rrank = nullptr;
    ba.g_bin = sl.g_bin.as<int32_t>() - peak_lo; ba.g_tmp = sl.g_tmp.as<uint8_t>() - peak_lo;
    ba.rcount = sl.rcount.as<int32_t>();
    ba.ctab = sl.ctab.as<uint8_t>(); ba.chead = sl.chead.as<float2>();
    ba.bin_size = s->bin_size; ba.n_top = s->n_top;
    ba.rindex = nullptr; ba.rbin = nullptr; ba.bounds = nullptr;
    // one resident wave: the grid-stride loop gives every warp the same number of spectra
    int cap, wpb, blocks;
    size_t smem;
    bin_launch_shape(s->sm_count, max_peaks, ns, &cap, &wpb, &smem, &blocks);
    ba.cap = cap;
    cs.e_bin0 = next_event(s); cs.e_bin1 = next_event(s);
    CK(cudaEventRecord(cs.e_bin0, st));
    ba.list = nullptr; ba.list_n = nullptr;
    if (ns >= PA_ROWS_MIN_SPECTRA && s->bin_rows && s->n_top <= 31) {     // (a handful of spectra: one launch instead of two)
        // the row form takes the spectra that are the rule and lists the rest, which k_bin_topn then takes from the list
        CK(sl.bin_list.ensure((size_t)ns * sizeof(int32_t)));
        CK(sl.bin_list_n.ensure(sizeof(unsigned int)));
        CK(cudaMemsetAsync(sl.bin_list_n.p, 0, sizeof(unsigned int), st));
        ba.list = sl.bin_list.as<int32_t>(); ba.list_n = sl.bin_list_n.as<unsigned int>();
        int rcap, rwpb, rblocks;
        size_t rsmem;
        const bin_rows_fn fn = bin_rows_kernel(ba.inten32 != nullptr, ba.mz32 != nullptr);
        bin_rows_launch_shape(s->sm_count, max_peaks, ns, fn, &rcap, &rwpb, &rsmem, &rblocks);
        ba.cap = rcap;
        fn<<<std::max(rblocks, 1), rwpb * 32, rsmem, st>>>(ba);
        CK(cudaGetLastError());
        s->ctr.kernel_launches++; s->ctr.launches_bin++;
        ba.cap = cap;
    }
    if (ns > 0) {
        if (ba.inten32) k_bin_topn<true><<<std::max(blocks, 1), wpb * 32, smem, st>>>(ba);
        else k_bin_topn<false><<<std::max(blocks, 1), wpb * 32, smem, st>>>(ba);
        CK(cudaGetLastError());
        s->ctr.kernel_launches++; s->ctr.launches_bin++;
    }
    CK(cudaEventRecord(cs.e_bin1, st));
    b.rpk = ba.rpk; b.rcount = sl.rcount.as<int32_t>() - r.s0;
    b.ctab = sl.ctab.as<uint8_t>() - (size_t)r.s0 * PA_NCELL; b.chead = sl.chead.as<float2>() - r.s0;
    cs.ev.assign(cs.types.size(), PassEvents());
    return chunk_plan(s, sc[cs.types[0]], si, cs, 0, n_types);
}

// Plan of pass `pass` of a chunk (the PSMs of type cs.types[pass], scored with ts's settings and tables), up to the
// read-back of its totals.  s owns the slots and the counters.
static int chunk_plan(pa_scorer* s, pa_scorer* ts, int si, ChunkState& cs, int pass, int n_types) {
    Slot& sl = s->slot[si];
    cudaStream_t st = sl.st;
    const int64_t np = cs.r.p1 - cs.r.p0;
    PassEvents& ev = cs.ev[pass];
    ev.e_plan0 = cs.e_bin1;
    if (pass > 0) { ev.e_plan0 = next_event(s); CK(cudaEventRecord(ev.e_plan0, st)); }
    ev.e_plan1 = next_event(s);
    CK(sl.psm_S.ensure((size_t)(np + 1) * sizeof(int32_t)));
    CK(sl.psm_status.ensure((size_t)(np + 1) * sizeof(int32_t)));
    CK(sl.psm_I.ensure((size_t)(np + 1) * sizeof(int64_t)));
    CK(sl.psm_units.ensure((size_t)(np + 1) * sizeof(int32_t)));
    CK(sl.iso_off.ensure((size_t)(np + 1) * sizeof(int64_t)));
    CK(sl.unit_off.ensure((size_t)(np + 1) * sizeof(int32_t)));
    CK(sl.totals.ensure(sizeof(PlanTotals)));
    CK(cudaMemsetAsync(sl.totals.p, 0, sizeof(PlanTotals), st));
    CK(cudaMemsetAsync(sl.psm_I.as<int64_t>() + np, 0, sizeof(int64_t), st));
    CK(cudaMemsetAsync(sl.psm_units.as<int32_t>() + np, 0, sizeof(int32_t), st));
    PaPlanOut po;
    po.psm_S = sl.psm_S.as<int32_t>(); po.psm_status = sl.psm_status.as<int32_t>();
    po.psm_I = sl.psm_I.as<int64_t>(); po.psm_units = sl.psm_units.as<int32_t>();
    PlanTotals* dt = sl.totals.as<PlanTotals>();
    po.combo_bits = dt->combo_bits; po.max_frag = &dt->max_frag; po.max_list = &dt->max_list; po.max_len = &dt->max_len;
    if (np > 0) {
        k_plan<<<(unsigned)((np + 255) / 256), 256, 0, st>>>(ts->cfg, cs.b, np, po, cs.psm_type, cs.types[pass], n_types);
        CK(cudaGetLastError());
        s->ctr.kernel_launches++;
    }
    size_t t1 = 0, t2 = 0;
    CK(cub::DeviceScan::ExclusiveSum(nullptr, t1, po.psm_I, sl.iso_off.as<int64_t>(), (int)(np + 1), st));
    CK(cub::DeviceScan::ExclusiveSum(nullptr, t2, po.psm_units, sl.unit_off.as<int32_t>(), (int)(np + 1), st));
    CK(sl.cub_tmp.ensure(std::max(t1, t2) + 256));
    size_t tb = sl.cub_tmp.cap;
    CK(cub::DeviceScan::ExclusiveSum(sl.cub_tmp.p, tb, po.psm_I, sl.iso_off.as<int64_t>(), (int)(np + 1), st));
    tb = sl.cub_tmp.cap;
    CK(cub::DeviceScan::ExclusiveSum(sl.cub_tmp.p, tb, po.psm_units, sl.unit_off.as<int32_t>(), (int)(np + 1), st));
    s->ctr.kernel_launches += 2;
    CK(cudaMemcpyAsync(&dt->total_iso, sl.iso_off.as<int64_t>() + np, sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(&dt->total_units, sl.unit_off.as<int32_t>() + np, sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
    CK(cudaMemcpyAsync(sl.h_totals.p, dt, sizeof(PlanTotals), cudaMemcpyDeviceToHost, st));
    CK(cudaEventRecord(ev.e_plan1, st));
    CK(cudaEventRecord(sl.ev_plan, st));
    return PA_OK;
}

// The result arrays of a chunk: device views that every pass of the chunk writes into, read back once after the last.
static int stage_results(pa_scorer* s, int si, const pa_results* out, bool out_dev, ChunkState& cs) {
    Slot& sl = s->slot[si];
    cudaStream_t st = sl.st;
    const ChunkRange& r = cs.r;
    const int64_t np = r.p1 - r.p0;
    const int64_t nm = cs.mod_hi - cs.mod_lo;
    ChunkArray* res = cs.res;
    res[0] = {out->best_sig, r.p0, np, sl.o_sig, cs.o_sig};
    res[1] = {out->best_score, r.p0, np, sl.o_score, cs.o_score};
    res[2] = {out->n_iso, r.p0, np, sl.o_niso, cs.o_niso};
    res[3] = {out->n_sites, r.p0, np, sl.o_nsites, cs.o_nsites};
    res[4] = {out->ascores, cs.mod_lo, nm, sl.o_asc, cs.o_asc};
    res[5] = {out->alt_sites, cs.mod_lo, nm, sl.o_alt, cs.o_alt};
    res[6] = {out->psm_status, r.p0, np, sl.o_status, cs.o_status};
    const size_t res_bound = (size_t)np * 32 + (size_t)nm * 12 + 8 * 16;
    cs.packed_res = cs.packed && !out_dev && res_bound <= PA_PACK_MAX;
    if (cs.packed_res) {
        CK(sl.d_opack.ensure(res_bound));
        CK(sl.h_opack.ensure(res_bound));
        // (the results start at byte 16 of the block: the read-back that bytes_d2h reports keeps its size)
        cs.packed_res_bytes = pack_layout(res, 7, 16, sl.d_opack.as<unsigned char>());
    } else {
        for (int i = 0; i < 7; i++) CK(stage(res[i], out_dev, st, nullptr));
    }
    return PA_OK;
}

// Pass `pass` of a chunk once its plan is on the host: K2, K2d, K3a, K3b / K3c for the PSMs of type cs.types[pass],
// with ts's settings and device tables; s owns the slots (scratch reused in stream order) and the counters.
static int chunk_pass(pa_scorer* s, pa_scorer* ts, int si, ChunkState& cs, int pass, bool keep) {
    Slot& sl = s->slot[si];
    cudaStream_t st = sl.st;
    const ChunkRange& r = cs.r;
    const int64_t np = r.p1 - r.p0;
    PassEvents& ev = cs.ev[pass];
    CK(cudaEventSynchronize(sl.ev_plan));
    PlanTotals T = *sl.h_totals.as<PlanTotals>();
    const int64_t total_iso = T.total_iso;
    const int n_units = T.total_units;
    // tables that depend on what the chunk contains (errors are reported on s, the handle of the call)
    int rc = ensure_table(ts, std::max(T.max_frag, 1));
    for (int S = 0; S < 64 && rc == PA_OK; S++)
        for (int k = 0; k < 64 && rc == PA_OK; k++)
            if ((T.combo_bits[S] >> k) & 1ull) rc = ensure_perm(ts, S, k);
    if (rc == PA_OK) rc = upload_perms(ts);
    if (rc != PA_OK) { if (ts != s) s->error = ts->error; return rc; }
    // scratch
    CK(sl.iso_lo.ensure((size_t)std::max<int64_t>(total_iso, 1) * 8));
    CK(sl.iso_hi.ensure((size_t)std::max<int64_t>(total_iso, 1) * 8));
    CK(sl.iso_n.ensure((size_t)std::max<int64_t>(total_iso, 1) * 4));
    CK(sl.iso_w.ensure((size_t)std::max<int64_t>(total_iso, 1) * 4));
    CK(sl.g_sort.ensure((size_t)std::max<int64_t>(total_iso, 1) * 8));
    CK(sl.g_lr.ensure((size_t)(std::max<int64_t>(total_iso, 1) + 2 * np + 2) * 4));
    CK(sl.unit_psm.ensure((size_t)std::max(n_units, 1) * 4));
    PaIso iso;
    iso.lo = sl.iso_lo.as<unsigned long long>(); iso.hi = sl.iso_hi.as<unsigned long long>();
    iso.nfrag = sl.iso_n.as<uint32_t>(); iso.w = sl.iso_w.as<float>();
    ev.e_cnt0 = next_event(s); ev.e_cnt1 = next_event(s); ev.e_sel1 = next_event(s);
    CK(sl.sched.ensure(16));                          // work cursors of k_count_score [0] and k_select [1]
    CK(cudaMemsetAsync(sl.sched.p, 0, 16, st));
    if (np > 0) {
        k_expand_units<<<(unsigned)((np + 255) / 256), 256, 0, st>>>(np, sl.unit_off.as<int32_t>(), sl.unit_psm.as<int32_t>());
        CK(cudaGetLastError());
        s->ctr.kernel_launches++;
    }
    CK(cudaEventRecord(ev.e_cnt0, st));
    if (n_units > 0) {
        PaCountArgs ca;
        ca.n_units = n_units; ca.unit_psm = sl.unit_psm.as<int32_t>(); ca.unit_off = sl.unit_off.as<int32_t>();
        ca.iso_off = sl.iso_off.as<int64_t>(); ca.psm_S = sl.psm_S.as<int32_t>(); ca.psm_status = sl.psm_status.as<int32_t>();
        ca.iso = iso; ca.n_lookups = sl.lookups.as<unsigned long long>();
        const int wpb = 8;
        const bool pair = ts->cfg.n_types == 2;
        size_t smem = wpb * sizeof(PsmSmem);
        ca.next_unit = sl.sched.as<unsigned long long>();
        const int64_t want = ((int64_t)n_units + wpb - 1) / wpb;
        // template switches: neutral losses configured, exactly two ion types, mz_error > 0.5.
        // One resident wave of blocks; the warps pull units from the cursor.
#define PA_K2_LAUNCH(NL, PR, EG) { \
            int blocks = (int)std::min<int64_t>(want, (int64_t)s->sm_count * resident_blocks(k_count_score<NL, PR, EG>, wpb * 32, smem)); \
            ca.grab = grab_size(n_units, (int64_t)blocks * wpb, PA_K2_GRAB); \
            k_count_score<NL, PR, EG><<<blocks, wpb * 32, smem, st>>>(ts->cfg, cs.b, ca); }
        const int variant = (ts->cfg.has_nl ? 4 : 0) | (pair ? 2 : 0) | (ts->cfg.err_gt_half ? 1 : 0);
        switch (variant) {
            case 0: PA_K2_LAUNCH(false, false, false) break;
            case 1: PA_K2_LAUNCH(false, false, true) break;
            case 2: PA_K2_LAUNCH(false, true, false) break;
            case 3: PA_K2_LAUNCH(false, true, true) break;
            case 4: PA_K2_LAUNCH(true, false, false) break;
            case 5: PA_K2_LAUNCH(true, false, true) break;
            case 6: PA_K2_LAUNCH(true, true, false) break;
            default: PA_K2_LAUNCH(true, true, true) break;
        }
#undef PA_K2_LAUNCH
        CK(cudaGetLastError());
        s->ctr.kernel_launches++; s->ctr.launches_count++;
    }
    CK(cudaEventRecord(ev.e_cnt1, st));
    // K2d: depths 10 .. n_top-1 (n_top > 10 only)
    PaDeep deep;
    deep.nd = ts->n_deep; deep.T = ts->d_T_deep.as<float>(); deep.cnt = nullptr;
    if (deep.nd > 0) {
        CK(sl.iso_deep.ensure((size_t)std::max<int64_t>(total_iso, 1) * deep.nd * sizeof(uint16_t)));
        deep.cnt = sl.iso_deep.as<uint16_t>();
        ev.e_deep1 = next_event(s);
        if (n_units > 0) {
            PaDeepCountArgs da;
            da.n_units = n_units; da.unit_psm = sl.unit_psm.as<int32_t>(); da.unit_off = sl.unit_off.as<int32_t>();
            da.iso_off = sl.iso_off.as<int64_t>(); da.psm_S = sl.psm_S.as<int32_t>(); da.iso_hi = iso.hi;
            da.cnt = sl.iso_deep.as<uint16_t>(); da.nd = deep.nd;
            const int wpb = 4;
            const size_t smem = wpb * (sizeof(PsmSmem) + 32 * deep.nd * sizeof(uint16_t));
            const int64_t want = ((int64_t)n_units + wpb - 1) / wpb;
            if (ts->cfg.has_nl) {
                const int blocks = (int)std::min<int64_t>(want, (int64_t)s->sm_count * resident_blocks(k_count_deep<true>, wpb * 32, smem));
                k_count_deep<true><<<blocks, wpb * 32, smem, st>>>(ts->cfg, cs.b, da);
            } else {
                const int blocks = (int)std::min<int64_t>(want, (int64_t)s->sm_count * resident_blocks(k_count_deep<false>, wpb * 32, smem));
                k_count_deep<false><<<blocks, wpb * 32, smem, st>>>(ts->cfg, cs.b, da);
            }
            CK(cudaGetLastError());
            s->ctr.kernel_launches++; s->ctr.launches_deep++;
        }
        CK(cudaEventRecord(ev.e_deep1, st));
    }
    // K3a .. K3c (the result views: stage_results)
    const int64_t nm = cs.mod_hi - cs.mod_lo;
    CK(sl.best_idx.ensure((size_t)std::max<int64_t>(np, 1) * 4));
    CK(sl.mod_psm.ensure((size_t)std::max<int64_t>(nm, 1) * 4));
    CK(sl.tie.ensure((size_t)std::max<int64_t>(nm, 1) * 8));
    CK(sl.generic_list.ensure((size_t)std::max<int64_t>(nm, 1) * 4));
    CK(sl.work_key.ensure((size_t)std::max<int64_t>(nm, 1) * 2)); CK(sl.work_key2.ensure((size_t)std::max<int64_t>(nm, 1) * 2));
    CK(sl.work_val.ensure((size_t)std::max<int64_t>(nm, 1) * 4)); CK(sl.work_sorted.ensure((size_t)std::max<int64_t>(nm, 1) * 4));
    CK(sl.generic_count.ensure(32));                 // [0] generic entries, [1..4] k_ascore work entries by class
    CK(cudaMemsetAsync(sl.generic_count.p, 0, 32, st));
    ev.e_asc1 = next_event(s);
    if (np > 0) {
        PaSelArgs sa;
        sa.n_psm = np; sa.iso_off = sl.iso_off.as<int64_t>(); sa.psm_S = sl.psm_S.as<int32_t>();
        sa.psm_status = sl.psm_status.as<int32_t>(); sa.iso = iso;
        sa.perm_off = ts->d_perm_off.as<int64_t>(); sa.perm_pool = ts->d_perm_pool.as<uint32_t>();
        sa.mod_off = cs.mod_off_abs;
        sa.best_sig = cs.o_sig ? cs.o_sig + r.p0 : nullptr;
        sa.best_score = cs.o_score ? cs.o_score + r.p0 : nullptr;
        sa.n_iso = cs.o_niso ? cs.o_niso + r.p0 : nullptr;
        sa.n_sites = cs.o_nsites ? cs.o_nsites + r.p0 : nullptr;
        sa.ascores = cs.o_asc; sa.alt_sites = cs.o_alt;            // indexed with absolute mod_off
        sa.psm_status_out = cs.o_status ? cs.o_status + r.p0 : nullptr;
        sa.g_sort = sl.g_sort.as<unsigned long long>(); sa.g_lr = sl.g_lr.as<uint32_t>();
        sa.mod_lo = cs.mod_lo; sa.best_idx = sl.best_idx.as<uint32_t>(); sa.mod_psm = sl.mod_psm.as<int32_t>();
        sa.tie = sl.tie.as<unsigned long long>();
        sa.work_key = sl.work_key.as<uint16_t>(); sa.work_val = sl.work_val.as<int32_t>();
        sa.work_count = sl.generic_count.as<int>() + 1;
        sa.next_psm = sl.sched.as<unsigned long long>() + 1;
        // thread per PSM for the common shapes; what it declines (generic_count[5] PSMs in rest_list) goes to
        // the warp-per-PSM kernel, whose visit count is therefore only known on the device
        CK(sl.rest_list.ensure((size_t)std::max<int64_t>(np, 1) * 4));
        sa.rest_list = sl.rest_list.as<int32_t>(); sa.rest_count = sl.generic_count.as<int>() + 5;
        if (cs.psm_type) k_select_thread<true><<<(unsigned)((np + 127) / 128), 128, 0, st>>>(ts->cfg, cs.b, sa);
        else k_select_thread<false><<<(unsigned)((np + 127) / 128), 128, 0, st>>>(ts->cfg, cs.b, sa);
        CK(cudaGetLastError());
        const int wpb = 8;
        const size_t sel_smem = wpb * PA_SORTCAP * sizeof(unsigned long long);
        int blocks = (int)std::min<int64_t>((np + wpb - 1) / wpb, (int64_t)s->sm_count * resident_blocks(k_select, wpb * 32, sel_smem));
        k_select<<<blocks, wpb * 32, sel_smem, st>>>(ts->cfg, cs.b, sa);
        CK(cudaGetLastError());
        s->ctr.kernel_launches += 2; s->ctr.launches_select += 2;
    }
    CK(cudaEventRecord(ev.e_sel1, st));
    if (np > 0 && nm > 0 && cs.o_asc != nullptr) {
        PaAscArgs aa;
        aa.n_entries = nm; aa.mod_lo = cs.mod_lo; aa.mod_psm = sl.mod_psm.as<int32_t>();
        aa.tie = sl.tie.as<unsigned long long>(); aa.best_idx = sl.best_idx.as<uint32_t>();
        aa.mod_off = cs.mod_off_abs; aa.iso_off = sl.iso_off.as<int64_t>(); aa.psm_S = sl.psm_S.as<int32_t>();
        aa.iso = iso; aa.ascores = cs.o_asc; aa.generic_list = sl.generic_list.as<int32_t>();
        aa.generic_count = sl.generic_count.as<int>();
        aa.work_sorted = sl.work_sorted.as<int32_t>(); aa.work_count = sl.generic_count.as<int>() + 1;
        // Ascore entries by stream class, longest merges first (keys written by K3a, pa_work_key)
        size_t tw = 0;
        CK(cub::DeviceRadixSort::SortPairs(nullptr, tw, sl.work_key.as<uint16_t>(), sl.work_key2.as<uint16_t>(),
                                           sl.work_val.as<int32_t>(), sl.work_sorted.as<int32_t>(), (int)nm, 0, PA_WORK_BITS, st));
        CK(sl.cub_tmp.ensure(tw + 256));
        tw = sl.cub_tmp.cap;
        CK(cub::DeviceRadixSort::SortPairs(sl.cub_tmp.p, tw, sl.work_key.as<uint16_t>(), sl.work_key2.as<uint16_t>(),
                                           sl.work_val.as<int32_t>(), sl.work_sorted.as<int32_t>(), (int)nm, 0, PA_WORK_BITS, st));
        s->ctr.kernel_launches += 3;
        const unsigned ab = (unsigned)((nm + 127) / 128);
        // pairs (entry, tied competitor) numbered by a scan over the sorted entry list, handed out from a cursor
        CK(sl.item_cnt.ensure((size_t)(nm + 1) * 4)); CK(sl.item_off.ensure((size_t)(nm + 1) * 4));
        CK(sl.gen_flag.ensure((size_t)nm * 4));
        CK(sl.asc_cursor.ensure(32));
        CK(cudaMemsetAsync(sl.gen_flag.p, 0, (size_t)nm * 4, st));
        CK(cudaMemsetAsync(sl.asc_cursor.p, 0, 32, st));
        PaAscItemArgs ia;
        ia.item_cnt = sl.item_cnt.as<int32_t>(); ia.item_off = sl.item_off.as<int32_t>();
        ia.cursor = sl.asc_cursor.as<unsigned long long>(); ia.gen_flag = sl.gen_flag.as<int>();
        k_asc_item_count<<<(unsigned)((nm + 1 + 255) / 256), 256, 0, st>>>(aa, ia);
        size_t tsz = 0;
        CK(cub::DeviceScan::ExclusiveSum(nullptr, tsz, ia.item_cnt, sl.item_off.as<int32_t>(), (int)(nm + 1), st));
        CK(sl.cub_tmp.ensure(tsz + 256));
        tsz = sl.cub_tmp.cap;
        CK(cub::DeviceScan::ExclusiveSum(sl.cub_tmp.p, tsz, ia.item_cnt, sl.item_off.as<int32_t>(), (int)(nm + 1), st));
        s->ctr.kernel_launches += 2;
        // (n_top > 10: the DEEP instantiations, whose depth argmax goes on over depths 10 .. n_top-1)
#define PA_PAIRS_LAUNCH(NQ, CLS, SMEM) { \
            if (deep.nd > 0) { \
                const int blocks = (int)std::min<int64_t>(ab, (int64_t)s->sm_count * resident_blocks(k_ascore_pairs<NQ, CLS, true>, 128, SMEM)); \
                k_ascore_pairs<NQ, CLS, true><<<blocks, 128, SMEM, st>>>(ts->cfg, cs.b, aa, ia, deep); \
            } else { \
                const int blocks = (int)std::min<int64_t>(ab, (int64_t)s->sm_count * resident_blocks(k_ascore_pairs<NQ, CLS, false>, 128, SMEM)); \
                k_ascore_pairs<NQ, CLS, false><<<blocks, 128, SMEM, st>>>(ts->cfg, cs.b, aa, ia, deep); \
            } }
        if (!ts->cfg.has_nl) {
            PA_PAIRS_LAUNCH(1, 0, 0) PA_PAIRS_LAUNCH(2, 1, 0) PA_PAIRS_LAUNCH(4, 2, 0)
            s->ctr.kernel_launches += 3;
        }
        PA_PAIRS_LAUNCH(PA_MAXSTREAM, 3, sizeof(AscSm))
#undef PA_PAIRS_LAUNCH
        CK(cudaGetLastError());
        const int wpb = 8;
        int blocks = s->sm_count * 2;
        int64_t stride = 32;
        while (stride < T.max_list) stride <<= 1;
        if (T.max_list > PA_LCAP) CK(sl.g_lists.ensure((size_t)blocks * wpb * 4 * stride * sizeof(float)));
        if (deep.nd > 0) k_ascore_generic<true><<<blocks, wpb * 32, wpb * sizeof(SelSmem), st>>>(ts->cfg, cs.b, aa, sl.g_lists.as<float>(), stride, deep);
        else k_ascore_generic<false><<<blocks, wpb * 32, wpb * sizeof(SelSmem), st>>>(ts->cfg, cs.b, aa, sl.g_lists.as<float>(), stride, deep);
        CK(cudaGetLastError());
        s->ctr.kernel_launches += 2; s->ctr.launches_ascore += 2;
    }
    CK(cudaEventRecord(ev.e_asc1, st));
    s->ctr.n_isoforms += total_iso;
    if (keep) {
        s->kept.b = cs.b; s->kept.n_psm = np; s->kept.psm_lo = r.p0;
        s->kept.iso_off = sl.iso_off.as<int64_t>(); s->kept.psm_S = sl.psm_S.as<int32_t>();
        s->kept.psm_status = sl.psm_status.as<int32_t>(); s->kept.iso = iso; s->kept.max_list = T.max_list;
        s->kept.iso_deep = deep.cnt;
        s->kept.valid = true; s->kept.slot = si;
    }
    return PA_OK;
}

static int chunk_back(pa_scorer* s, pa_scorer* const* sc, int n_types, int si, const pa_results* out, bool out_dev,
                      ChunkState& cs, bool keep) {
    Slot& sl = s->slot[si];
    cudaStream_t st = sl.st;
    int rc = stage_results(s, si, out, out_dev, cs);
    for (size_t pass = 0; pass < cs.types.size() && rc == PA_OK; pass++) {
        if (pass > 0) rc = chunk_plan(s, sc[cs.types[pass]], si, cs, (int)pass, n_types);
        if (rc == PA_OK) rc = chunk_pass(s, sc[cs.types[pass]], si, cs, (int)pass, keep);
    }
    if (rc != PA_OK) return rc;
    int64_t* d2h = &s->ctr.bytes_d2h;
    if (cs.packed_res) {         // (score_impl copies the block into the caller's arrays once the stream is done)
        CK(cudaMemcpyAsync(sl.h_opack.p, sl.d_opack.p, cs.packed_res_bytes, cudaMemcpyDeviceToHost, st));
        *d2h += (int64_t)cs.packed_res_bytes;
    } else {
        for (int i = 0; i < 7; i++) CK(copy_back(cs.res[i], out_dev, st, d2h));
    }
    return PA_OK;
}

// Host-side consistency check of PSMs [p0, p1) of a host batch and the spectra [s0, s1) they reference
// (the device-resident path runs k_check_batch instead).  Called per chunk, so that all but the first
// chunk's check overlaps the GPU work of the chunk before.
static const char* check_host_range(const pa_batch* in, int64_t p0, int64_t p1, int64_t s0, int64_t s1) {
    for (int64_t q = s0; q < s1; q++)
        if (in->spec_off[q + 1] < in->spec_off[q] || in->spec_off[q] < 0) return "spec_off is not a non-decreasing CSR index";
    for (int64_t p = p0; p < p1; p++) {
        if (in->pep_off[p + 1] < in->pep_off[p] || in->pep_off[p] < 0) return "pep_off is not a non-decreasing CSR index";
        if (in->aux_off && (in->aux_off[p + 1] < in->aux_off[p] || in->aux_off[p] < 0)) return "aux_off is not a non-decreasing CSR index";
        if (in->mod_off[p + 1] - in->mod_off[p] != (int64_t)std::max(in->n_mod[p], 0) || in->mod_off[p] < 0)
            return "mod_off is not the exclusive prefix sum of n_mod";
    }
    if (in->aux_off && in->aux_off[p1] > in->aux_off[p0] && (!in->aux_pos || !in->aux_mass)) return "aux_off is not empty but aux_pos / aux_mass is NULL";
    return nullptr;
}

// Types of PSMs [p_lo, p_hi) of a typed batch: count[t] PSMs of type t, a type >= n_types counted as type 0 (whose
// pass reports it).
__global__ void k_type_count(const uint8_t* psm_type, int64_t p_lo, int64_t p_hi, int n_types, unsigned int* count) {
    __shared__ unsigned int c[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) c[i] = 0;
    __syncthreads();
    for (int64_t p = p_lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < p_hi; p += (int64_t)gridDim.x * blockDim.x) {
        const int t = psm_type[p];
        atomicAdd(&c[t < n_types ? t : 0], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 256; i += blockDim.x) if (c[i]) atomicAdd(&count[i], c[i]);
}

// sc[0 .. n_types) (typed batches, pa_score_typed; null: s alone) score the PSMs of each type; s == sc[0] owns the
// slots, the counters and the error text.  psm_type: on the side of the batch's arrays, null = every PSM is type 0.
static int score_impl(pa_scorer* s, const pa_batch* in, const pa_results* out, int64_t p_lo, int64_t p_hi, uint32_t flags,
                      pa_scorer* const* sc = nullptr, int n_types = 1, const uint8_t* psm_type = nullptr) {
    if (!s) return PA_ERR_ARG;
    if (!sc) sc = &s;
    if (!in || !out) return fail(s, PA_ERR_ARG, "NULL batch or results");
    if (s->binner_only) return fail(s, PA_ERR_STATE, "this handle was made by pa_create_binner: it only bins spectra");
    if (in->n_psm < 0 || in->n_spec < 0) return fail(s, PA_ERR_ARG, "negative sizes");
    if (p_lo < 0 || p_hi > in->n_psm || p_lo > p_hi) return fail(s, PA_ERR_ARG, "PSM range [%lld, %lld) outside the batch of %lld", (long long)p_lo, (long long)p_hi, (long long)in->n_psm);
    if (in->n_psm > 0 && (!in->spec_off || !in->mz || (!in->inten && !in->inten32) || !in->psm_spec || !in->pep_off || !in->pep ||
                          !in->n_mod || !in->max_charge || !in->mod_off))
        return fail(s, PA_ERR_ARG, "NULL input array");
    CK(cudaSetDevice(s->device));
    int rc = PA_OK;         // (the device-side config is current: pa_create / pa_add_neutral_loss refresh it)
    const auto t_call = std::chrono::steady_clock::now();
    memset(&s->ctr, 0, sizeof(s->ctr));
    s->ev_used = 0;
    s->kept.valid = false;
    s->ctr.n_psm = p_hi - p_lo; s->ctr.n_spec = in->n_spec;
    if (p_hi == p_lo) return PA_OK;
    const bool in_dev = is_device_ptr(in->mz);
    const bool out_dev = is_device_ptr(out->best_score ? (void*)out->best_score
                                       : out->best_sig ? (void*)out->best_sig
                                       : out->ascores ? (void*)out->ascores : (void*)out->psm_status);
    const bool keep = (flags & PA_KEEP_ISOFORMS) != 0;
    const int64_t n_range = p_hi - p_lo;
    // ms_total spans the whole call on the device time line: the pre-pass over a device-resident batch included
    cudaEvent_t e_all0 = next_event(s), e_all1 = next_event(s);
    CK(cudaEventRecord(e_all0, s->slot[0].st));
    for (int i = 0; i < 2; i++) {
        CK(s->slot[i].lookups.ensure(8));
        CK(cudaMemsetAsync(s->slot[i].lookups.p, 0, 8, s->slot[i].st));
    }

    // ---- chunking ----
    std::vector<ChunkRange> chunks;
    std::vector<int> chunk_maxp;
    std::vector<int64_t> mod_lo, mod_hi;
    DevBounds hb;
    unsigned int dev_type_n[256];
    if (in_dev) {
        // Device-resident batch: one chunk (see DevBounds).  One small kernel gathers the range ends the host needs,
        // a second checks the CSR arrays (and that psm_spec is non-decreasing: the spectrum range relies on it), a
        // third finds the largest spectrum: one device -> host copy instead of one per value.
        DevBuf& tb = s->slot[0].totals;
        CK(tb.ensure(sizeof(PlanTotals) + sizeof(DevBounds) + 256 * sizeof(unsigned int)));
        DevBounds* d_b = (DevBounds*)tb.p;
        CK(cudaMemset(d_b, 0, sizeof(DevBounds)));
        k_dev_bounds<<<1, 1>>>(in->spec_off, in->psm_spec, in->pep_off, in->aux_off, in->mod_off, p_lo, p_hi, in->n_spec, d_b);
        k_check_batch<<<(unsigned)std::min<int64_t>((std::max(n_range, in->n_spec) + 255) / 256, 1184), 256>>>(
            in->psm_spec, in->pep_off, in->aux_off, in->n_mod, in->mod_off, in->spec_off, p_lo, p_hi, in->n_spec, &d_b->bad);
        k_max_peaks<<<(unsigned)((in->n_spec + 255) / 256), 256>>>(in->spec_off, in->n_spec, &d_b->max_peaks);
        CK(cudaGetLastError());
        s->ctr.kernel_launches += 3;
        CK(cudaMemcpy(&hb, d_b, sizeof(DevBounds), cudaMemcpyDeviceToHost));
        if (hb.bad & 2) return fail(s, PA_ERR_ARG, "inconsistent batch: an offset array is not a non-decreasing CSR index or mod_off does not follow n_mod");
        if (hb.n_aux > 0 && (!in->aux_pos || !in->aux_mass)) return fail(s, PA_ERR_ARG, "aux_off is not empty but aux_pos / aux_mass is NULL");
        if (hb.bad & 1) {                        // unordered PSM -> spectrum map: the chunk takes every spectrum
            hb.s0 = 0; hb.s1 = in->n_spec;
            CK(cudaMemcpy(&hb.peak0, in->spec_off, 8, cudaMemcpyDeviceToHost));
            CK(cudaMemcpy(&hb.peak1, in->spec_off + in->n_spec, 8, cudaMemcpyDeviceToHost));
        }
        chunks.push_back({p_lo, p_hi, hb.s0, hb.s1});
        if (psm_type) {          // the types present: one more small kernel and copy
            unsigned int* d_cnt = (unsigned int*)(d_b + 1);
            CK(cudaMemset(d_cnt, 0, 256 * sizeof(unsigned int)));
            k_type_count<<<(unsigned)std::min<int64_t>((n_range + 255) / 256, 1184), 256>>>(psm_type, p_lo, p_hi, n_types, d_cnt);
            CK(cudaGetLastError());
            s->ctr.kernel_launches++;
            CK(cudaMemcpy(dev_type_n, d_cnt, sizeof(dev_type_n), cudaMemcpyDeviceToHost));
        }
        mod_lo.push_back(hb.mod0); mod_hi.push_back(hb.mod1);
        chunk_maxp.push_back(hb.max_peaks);
        s->ctr.n_peaks += hb.peak1 - hb.peak0;
    } else {
        // one branch-free pass (the compiler vectorises it): PSMs in spectrum order, indices in range
        int bad = 0;
        {
            const int32_t* ps = in->psm_spec;
            const int32_t ns = (int32_t)std::min<int64_t>(in->n_spec, INT32_MAX);
            bad |= (ps[p_lo] < 0) | (ps[p_lo] >= ns);
            for (int64_t p = p_lo + 1; p < p_hi; p++) bad |= (ps[p] < ps[p - 1]) | (ps[p] >= ns);
        }
        const bool mono = bad == 0;
        if (!mono || keep) chunks.push_back({p_lo, p_hi, mono ? (int64_t)in->psm_spec[p_lo] : 0, mono ? (int64_t)in->psm_spec[p_hi - 1] + 1 : in->n_spec});
        else {
            // about eight chunks per call (copy of chunk c+1 under the kernels of chunk c), never beyond PA_CHUNK_PSM PSMs
            // or PA_CHUNK_PEAKS peaks; small ranges (one GPU's share of a sharded batch) get small chunks
            const int64_t per = std::min<int64_t>(PA_CHUNK_PSM, std::max<int64_t>(PA_CHUNK_MIN, ((n_range + 7) / 8 + 1023) / 1024 * 1024));
            int64_t p0 = p_lo;
            while (p0 < p_hi) {
                int64_t s0 = in->psm_spec[p0];
                // PSMs sharing the spectrum of p0 that were cut off by the previous chunk stay reachable:
                // chunk spectra start at the first spectrum referenced
                int64_t p1 = std::min<int64_t>(p0 + per, p_hi);
                while (p1 > p0 + 1 && in->spec_off[in->psm_spec[p1 - 1] + 1] - in->spec_off[s0] > PA_CHUNK_PEAKS) p1 = p0 + (p1 - p0) / 2;
                int64_t s1 = (int64_t)in->psm_spec[p1 - 1] + 1;
                chunks.push_back({p0, p1, s0, s1});
                p0 = p1;
            }
        }
        chunk_maxp.assign(chunks.size(), 0); mod_lo.assign(chunks.size(), 0); mod_hi.assign(chunks.size(), 0);
    }
    // per-chunk host work of a host batch, done right before the chunk is staged (so that all but the first chunk's
    // share overlaps the GPU): consistency of the CSR arrays, largest spectrum, range in the per-mod outputs
    auto prepare_host_chunk = [&](size_t c) -> const char* {
        const ChunkRange& r = chunks[c];
        const char* why = check_host_range(in, r.p0, r.p1, r.s0, r.s1);
        if (why) return why;
        int64_t m = 0;
        for (int64_t q = r.s0; q < r.s1; q++) m = std::max<int64_t>(m, in->spec_off[q + 1] - in->spec_off[q]);
        chunk_maxp[c] = (int)std::min<int64_t>(std::max<int64_t>(m, 0), 1 << 20);
        mod_lo[c] = in->mod_off[r.p0]; mod_hi[c] = in->mod_off[r.p1];
        s->ctr.n_peaks += in->spec_off[r.s1] - in->spec_off[r.s0];
        return nullptr;
    };
    if (!in_dev) {
        const char* why = prepare_host_chunk(0);
        if (why) return fail(s, PA_ERR_ARG, "inconsistent batch: %s", why);
    }
    const bool check_chunks = !in_dev && chunks.size() > 1;      // chunk 0 was prepared above

    // ---- two-slot software pipeline ----
    std::vector<ChunkState> cs(chunks.size());
    // the passes of each chunk: one per type with PSMs in it (a type >= n_types goes with type 0, whose pass reports it)
    for (size_t c = 0; c < chunks.size(); c++) {
        if (!psm_type) { cs[c].types = {0}; continue; }
        std::vector<int64_t> n(256, 0);
        if (in_dev) for (int t = 0; t < 256; t++) n[t] = dev_type_n[t];
        else for (int64_t p = chunks[c].p0; p < chunks[c].p1; p++) n[psm_type[p] < n_types ? psm_type[p] : 0]++;
        for (int t = 0; t < n_types; t++) if (n[t] > 0) cs[c].types.push_back(t);
    }
    s->ctr.n_chunks = (int64_t)chunks.size();
    cs[0].single_chunk = chunks.size() == 1;
    // The m/z narrowing of a host chunk (narrow_begin / narrow_end) runs on the pool one chunk AHEAD of the copies: the
    // set of chunk c+2 is being filled while chunk c+1 is on the wire and this thread waits for chunk c's plan, so the
    // copy engine never waits for a conversion.  Three staging sets rotate; a set is reused once its copies are done.
    // Default mode decides by measurement whether the pass pays on this box: the scorer's first large host batch narrows
    // (and pins the staging buffers, starts the threads), the second narrows and is timed, the third does not and is
    // timed, and the faster way (peaks per second of the whole call) is kept.  It needs PA_NARROW_MIN_THREADS to try.
    const int64_t call_peaks = in_dev || chunks.empty() ? 0 : in->spec_off[chunks.back().s1] - in->spec_off[chunks[0].s0];
    if (!s->host_threads_fixed && s->pool.th.empty()) s->host_threads = host_thread_budget(s->host_cpus);
    const bool narrow_trial = s->narrow_mode < 0 && !in_dev && call_peaks >= (1 << 20) && s->host_threads >= PA_NARROW_MIN_THREADS;
    const bool want_narrow = s->narrow_mode == 1 || (narrow_trial && (s->narrow_state <= 1 || (s->narrow_state == 3 && s->narrow_keep)));
    const bool may_narrow = !in_dev && want_narrow &&
                            !(chunks.size() == 1 && s->narrow_mode != 1 && in->spec_off[chunks[0].s1] - in->spec_off[chunks[0].s0] < (1 << 19));
    auto nstage = [&](size_t c) -> NarrowStage& { return s->nstage[c % 3]; };
    auto bail = [&](int code) { if (may_narrow) for (int i = 0; i < 3; i++) if (s->nstage[i].busy) { s->pool.wait(); s->nstage[i].busy = false; } cudaDeviceSynchronize(); return code; };
    if (may_narrow) {
        rc = narrow_begin(s, nstage(0), in, chunks[0]);           // (chunk_front waits for it, after the chunk's other copies)
        if (rc != PA_OK) return bail(rc);
    }
    rc = chunk_front(s, sc, n_types, 0, in, psm_type, in_dev, chunks[0], mod_lo[0], mod_hi[0], chunk_maxp[0], cs[0],
                     in_dev ? &hb : nullptr, may_narrow ? &nstage(0) : nullptr);
    if (rc != PA_OK) return bail(rc);
    if (may_narrow && chunks.size() > 1) { rc = narrow_begin(s, nstage(1), in, chunks[1]); if (rc != PA_OK) return bail(rc); }
    for (size_t c = 0; c < chunks.size(); c++) {
        if (c + 1 < chunks.size()) {
            if (check_chunks) {
                const char* why = prepare_host_chunk(c + 1);
                if (why) { bail(0); return fail(s, PA_ERR_ARG, "inconsistent batch: %s", why); }
            }
            // slot (c+1)&1 was last used by chunk c-1: its stream order keeps buffers safe
            rc = chunk_front(s, sc, n_types, (int)((c + 1) & 1), in, psm_type, in_dev, chunks[c + 1], mod_lo[c + 1],
                             mod_hi[c + 1], chunk_maxp[c + 1], cs[c + 1], in_dev ? &hb : nullptr,
                             may_narrow ? &nstage(c + 1) : nullptr);
            if (rc != PA_OK) return bail(rc);
            if (may_narrow && c + 2 < chunks.size()) { rc = narrow_begin(s, nstage(c + 2), in, chunks[c + 2]); if (rc != PA_OK) return bail(rc); }
        }
        rc = chunk_back(s, sc, n_types, (int)(c & 1), out, out_dev, cs[c], keep);
        if (rc != PA_OK) return bail(rc);
    }
    for (int i = 0; i < 2; i++)
        CK(cudaMemcpyAsync(s->slot[i].h_lookups.p, s->slot[i].lookups.p, 8, cudaMemcpyDeviceToHost, s->slot[i].st));
    CK(cudaStreamSynchronize(s->slot[0].st));
    CK(cudaStreamSynchronize(s->slot[1].st));
    CK(cudaEventRecord(e_all1, s->slot[0].st));
    CK(cudaEventSynchronize(e_all1));
    for (size_t c = 0; c < chunks.size(); c++)       // packed results: from the pinned block into the caller's arrays
        if (cs[c].packed_res)
            for (const ChunkArray& a : cs[c].res)
                if (a.arr && a.n > 0)
                    memcpy((unsigned char*)a.arr + a.lo * (int64_t)a.elem, s->slot[c & 1].h_opack.as<unsigned char>() + a.off, a.bytes());
    // counters
    for (size_t c = 0; c < chunks.size(); c++) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, cs[c].e_bin0, cs[c].e_bin1); s->ctr.ms_bin += ms;
        for (const PassEvents& ev : cs[c].ev) {
            cudaEventElapsedTime(&ms, ev.e_plan0, ev.e_plan1); s->ctr.ms_plan += ms;
            cudaEventElapsedTime(&ms, ev.e_cnt0, ev.e_cnt1); s->ctr.ms_count += ms;
            if (ev.e_deep1) { cudaEventElapsedTime(&ms, ev.e_cnt1, ev.e_deep1); s->ctr.ms_deep += ms; }
            cudaEventElapsedTime(&ms, ev.e_deep1 ? ev.e_deep1 : ev.e_cnt1, ev.e_sel1); s->ctr.ms_select += ms;
            cudaEventElapsedTime(&ms, ev.e_sel1, ev.e_asc1); s->ctr.ms_ascore += ms;
        }
    }
    cudaEventElapsedTime(&s->ctr.ms_total, e_all0, e_all1);
    s->ctr.n_fragment_lookups = (int64_t)*s->slot[0].h_lookups.as<unsigned long long>() + (int64_t)*s->slot[1].h_lookups.as<unsigned long long>();
    if (narrow_trial && s->narrow_state < 3) {
        const double rate = (double)call_peaks / std::chrono::duration<double>(std::chrono::steady_clock::now() - t_call).count();
        if (s->narrow_state == 1) s->narrow_rate_on = rate;
        else if (s->narrow_state == 2) s->narrow_keep = s->narrow_rate_on > 1.02 * rate;
        s->narrow_state++;
    }
    return PA_OK;
}

static int busy_error(pa_scorer* s) { return fail(s, PA_ERR_STATE, "an asynchronous pa_score_batch_async call is in flight: call pa_wait first"); }

extern "C" int pa_score_batch(pa_scorer* s, const pa_batch* in, const pa_results* out, uint32_t flags) {
    if (!s) return PA_ERR_ARG;
    if (s->busy) return busy_error(s);
    return score_impl(s, in, out, 0, in ? in->n_psm : 0, flags);
}

extern "C" int pa_score_range(pa_scorer* s, const pa_batch* in, const pa_results* out, int64_t psm_lo, int64_t psm_hi,
                              uint32_t flags) {
    if (!s) return PA_ERR_ARG;
    if (s->busy) return busy_error(s);
    return score_impl(s, in, out, psm_lo, psm_hi, flags);
}

extern "C" int pa_score_typed(pa_scorer* const* s, int32_t n_types, const pa_batch* in, const uint8_t* psm_type,
                              const pa_results* out, uint32_t flags) {
    if (!s || !s[0]) return fail(nullptr, PA_ERR_ARG, "pa_score_typed: NULL scorer list or NULL first handle");
    pa_scorer* s0 = s[0];
    if (n_types < 1 || n_types > 255) return fail(s0, PA_ERR_ARG, "pa_score_typed: n_types = %d outside 1 .. 255", (int)n_types);
    for (int t = 0; t < n_types; t++) {
        if (!s[t]) return fail(s0, PA_ERR_ARG, "pa_score_typed: handle of type %d is NULL", t);
        if (s[t]->binner_only) return fail(s0, PA_ERR_ARG, "pa_score_typed: handle of type %d was made by pa_create_binner: it only bins spectra", t);
        if (s[t]->device != s0->device) return fail(s0, PA_ERR_ARG, "pa_score_typed: handle of type %d is on device %d, type 0 on device %d", t, s[t]->device, s0->device);
        if (s[t]->bin_size != s0->bin_size || s[t]->n_top != s0->n_top)
            return fail(s0, PA_ERR_ARG, "pa_score_typed: handle of type %d bins with bin_size %g / n_top %d, type 0 with %g / %d: the "
                        "spectra are binned once for every type", t, (double)s[t]->bin_size, s[t]->n_top, (double)s0->bin_size, s0->n_top);
    }
    for (int t = 0; t < n_types; t++)
        if (s[t]->busy) return fail(s0, PA_ERR_STATE, "pa_score_typed: handle of type %d has an asynchronous call in flight: call pa_wait first", t);
    if ((flags & PA_KEEP_ISOFORMS) && n_types > 1)
        return fail(s0, PA_ERR_UNSUPPORTED, "pa_score_typed: PA_KEEP_ISOFORMS is not supported with more than one type");
    return score_impl(s0, in, out, 0, in ? in->n_psm : 0, flags, s, n_types, psm_type);
}

// The path has one host decision per chunk (the plan totals size the isoform scratch), so "asynchronous" means a
// host thread owned by the scorer runs the same orchestration while the caller goes on; the caller's stream
// (if any) is honoured as a dependency: work queued on it before this call completes before the inputs are read.
extern "C" int pa_score_batch_async(pa_scorer* s, const pa_batch* in, const pa_results* out, int64_t psm_lo,
                                    int64_t psm_hi, uint32_t flags, void* stream) {
    if (!s) return PA_ERR_ARG;
    if (!in || !out) return fail(s, PA_ERR_ARG, "NULL batch or results");
    if (s->busy) return busy_error(s);
    CK(cudaSetDevice(s->device));
    if (stream) {
        cudaEvent_t ev;
        CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        CK(cudaEventRecord(ev, (cudaStream_t)stream));
        for (int i = 0; i < 2; i++) CK(cudaStreamWaitEvent(s->slot[i].st, ev, 0));
        CK(cudaEventDestroy(ev));
    }
    if (psm_hi < 0) psm_hi = in->n_psm;
    if (!s->worker.joinable()) {
        try {
            s->worker = std::thread([s]() {
                std::unique_lock<std::mutex> lk(s->mu);
                for (;;) {
                    s->cv.wait(lk, [s] { return s->job_ready || s->quit; });
                    if (s->quit) return;
                    s->job_ready = false;
                    lk.unlock();
                    const int rc = score_impl(s, &s->async_in, &s->async_out, s->async_lo, s->async_hi, s->async_flags);
                    lk.lock();
                    s->async_rc = rc;
                    s->job_done = true;
                    s->cv.notify_all();
                }
            });
        } catch (...) {
            return fail(s, PA_ERR_STATE, "could not start the orchestration thread");
        }
    }
    {
        std::lock_guard<std::mutex> lk(s->mu);
        s->async_in = *in; s->async_out = *out;
        s->async_lo = psm_lo; s->async_hi = psm_hi; s->async_flags = flags;
        s->async_rc = PA_OK;
        s->job_done = false; s->job_ready = true;
        s->busy = true;
    }
    s->cv.notify_all();
    return PA_OK;
}

extern "C" int pa_wait(pa_scorer* s) {
    if (!s) return PA_ERR_ARG;
    if (!s->busy) return PA_OK;
    std::unique_lock<std::mutex> lk(s->mu);
    s->cv.wait(lk, [s] { return s->job_done; });
    s->busy = false;
    return s->async_rc;
}

// ---------------------------------------------------------------------------------------------
extern "C" int64_t pa_fetch_pep_scores(pa_scorer* s, int64_t psm, int64_t cap, uint64_t* sig, int32_t* counts,
                                       float* scores, float* weighted, int32_t* total_fragments) {
    if (!s) return PA_ERR_ARG;
    if (!s->kept.valid) return fail(s, PA_ERR_STATE, "no kept batch: score with PA_KEEP_ISOFORMS first");
    if (psm < s->kept.psm_lo || psm >= s->kept.psm_lo + s->kept.n_psm) return fail(s, PA_ERR_ARG, "psm index out of range");
    CK(cudaSetDevice(s->device));
    const int64_t q = psm - s->kept.psm_lo;
    int64_t off[2]; int32_t S, k, status;
    CK(cudaMemcpy(off, s->kept.iso_off + q, 16, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(&S, s->kept.psm_S + q, 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(&status, s->kept.psm_status + q, 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(&k, s->kept.b.n_mod + q, 4, cudaMemcpyDeviceToHost));
    const int64_t I = off[1] - off[0];
    if (I <= 0 || status != PA_PSM_OK) return 0;
    const int64_t D = PA_N_TOP + s->n_deep;   // row width of counts / scores: the scorer's n_top
    PaDeep deep;
    deep.nd = s->n_deep; deep.T = s->d_T_deep.as<float>(); deep.cnt = s->kept.iso_deep;
    DevBuf d_sig, d_cnt, d_sc, d_w, d_tot;
    CK(d_sig.ensure(I * 8)); CK(d_cnt.ensure(I * D * 4)); CK(d_sc.ensure(I * D * 4));
    CK(d_w.ensure(I * 4)); CK(d_tot.ensure(I * 4));
    k_export_psm<<<(unsigned)((I + 127) / 128), 128>>>(s->cfg, off[0], I, S, k, s->kept.iso, d_sig.as<uint64_t>(),
                                                        d_cnt.as<int32_t>(), d_sc.as<float>(), d_w.as<float>(), d_tot.as<int32_t>(), deep);
    CK(cudaGetLastError());
    std::vector<uint64_t> h_sig(I); std::vector<int32_t> h_cnt(I * D), h_tot(I);
    std::vector<float> h_sc(I * D), h_w(I);
    CK(cudaMemcpy(h_sig.data(), d_sig.p, I * 8, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(h_cnt.data(), d_cnt.p, I * D * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(h_sc.data(), d_sc.p, I * D * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(h_w.data(), d_w.p, I * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(h_tot.data(), d_tot.p, I * 4, cudaMemcpyDeviceToHost));
    // listing order: hash-iteration order, then std::sort by descending weighted score unless
    // the PSM is unambiguous (cpp/Ascore.cpp:263-269)
    std::vector<uint32_t> order(I);
    if (I > 1) {
        int rc = ensure_perm(s, S, k);
        if (rc != PA_OK) return rc;
        const uint32_t* perm = s->perm_pool.data() + s->perm_off[S * 64 + k];
        for (int64_t i = 0; i < I; i++) order[i] = perm[i];
        if (k < S) {
            const float* w = h_w.data();
            std::sort(order.begin(), order.end(), [w](uint32_t a, uint32_t b) { return w[a] > w[b]; });
        }
    } else order[0] = 0;
    for (int64_t i = 0; i < I && i < cap; i++) {
        uint32_t id = order[i];
        if (sig) sig[i] = h_sig[id];
        if (counts) memcpy(counts + i * D, &h_cnt[id * D], D * 4);
        if (scores) memcpy(scores + i * D, &h_sc[id * D], D * 4);
        if (weighted) weighted[i] = h_w[id];
        if (total_fragments) total_fragments[i] = h_tot[id];
    }
    return I;
}

extern "C" int pa_calculate_ambiguity(pa_scorer* s, int64_t psm, uint64_t sig_a, const float* scores_a, float weighted_a,
                                      uint64_t sig_b, const float* scores_b, float weighted_b, float* out) {
    if (!s || !scores_a || !scores_b || !out) return PA_ERR_ARG;
    if (!s->kept.valid) return fail(s, PA_ERR_STATE, "no kept batch: score with PA_KEEP_ISOFORMS first");
    if (psm < s->kept.psm_lo || psm >= s->kept.psm_lo + s->kept.n_psm) return fail(s, PA_ERR_ARG, "psm index out of range");
    CK(cudaSetDevice(s->device));
    PaAmbArgs a;
    a.psm = psm - s->kept.psm_lo; a.sigA = sig_a; a.sigB = sig_b; a.wA = weighted_a; a.wB = weighted_b;
    memcpy(a.scA, scores_a, (PA_N_TOP + s->n_deep) * sizeof(float)); memcpy(a.scB, scores_b, (PA_N_TOP + s->n_deep) * sizeof(float));
    a.deep.nd = s->n_deep; a.deep.T = s->d_T_deep.as<float>(); a.deep.cnt = s->kept.iso_deep;
    DevBuf d_out, d_lists;
    CK(d_out.ensure(4));
    a.list_stride = 32;
    while (a.list_stride < s->kept.max_list) a.list_stride <<= 1;
    if (s->kept.max_list > PA_LCAP) CK(d_lists.ensure((size_t)4 * a.list_stride * sizeof(float)));
    a.g_lists = d_lists.as<float>(); a.out = d_out.as<float>();
    k_ambiguity<<<1, 32, sizeof(SelSmem)>>>(s->cfg, s->kept.b, a);
    CK(cudaGetLastError());
    CK(cudaMemcpy(out, d_out.p, 4, cudaMemcpyDeviceToHost));
    return PA_OK;
}

// ---- sharding over the GPUs of one box (SURVEY.md section 8e) --------------------------------------
// PSMs are independent, so a batch shards with no collective: every GPU takes a contiguous PSM range cut where
// psm_spec changes (one spectrum is binned by exactly one GPU).  Ranges are balanced by estimated cost, not by
// count: isoforms x fragments per isoform for the scoring kernels plus `peak_weight` x the spectrum's peaks (shared
// between the hits of a spectrum) for binning and, with host inputs, the host -> device copy that dominates there.
// The estimate is taken on a strided sample (<= 8192 PSMs), so the call costs a fraction of a millisecond.  `share`
// (optional, one positive number per rank) gives rank r that fraction of the cost instead of 1 / world: the GPUs of a box
// do not all get the same host-link bandwidth when every one of them copies at once.
extern "C" int pa_shard_ranges_for(const char* mod_group_c, int32_t n_types_in, int32_t nvar_in, const pa_batch* in,
                                   int32_t world, double peak_weight, const double* share, int64_t* cuts) {
    if (!mod_group_c || !in || !cuts || world < 1) return PA_ERR_ARG;
    double share_sum = 0.;
    if (share) for (int r = 0; r < world; r++) { if (!(share[r] > 0.)) return PA_ERR_ARG; share_sum += share[r]; }
    const std::string mod_group(mod_group_c);
    const int64_t n = in->n_psm;
    for (int r = 0; r <= world; r++) cuts[r] = (r == world) ? n : 0;
    if (n <= 0 || world == 1) return PA_OK;
    if (!in->spec_off || !in->psm_spec || !in->pep_off || !in->pep || !in->n_mod || !in->max_charge) return PA_ERR_ARG;
    if (is_device_ptr(in->psm_spec)) return PA_ERR_ARG;          // host batches only
    bool is_site[256] = {false};
    for (char ch : mod_group) if (ch >= 'A' && ch <= 'Z') is_site[(unsigned char)ch] = true;
    const bool term_n = mod_group.find('n') != std::string::npos, term_c = mod_group.find('c') != std::string::npos;
    const int n_types = std::max<int>(1, n_types_in);
    const int nvar = std::max(1, nvar_in);
    const int64_t stride = std::max<int64_t>(1, n / 8192);
    const int64_t m = (n + stride - 1) / stride;
    std::vector<double> cum(m + 1, 0.);
    for (int64_t i = 0; i < m; i++) {
        const int64_t p = i * stride;
        const int32_t sp = in->psm_spec[p];
        if (sp < 0 || sp >= in->n_spec || (p > 0 && in->psm_spec[p] < in->psm_spec[p - stride])) return PA_ERR_ARG;   // needs scan-sorted PSMs
        const int a = in->pep_off[p], L = in->pep_off[p + 1] - a;
        int S = 0;
        for (int j = 0; j < L; j++) S += is_site[in->pep[a + j]] || (term_n && j == 0) || (term_c && j == L - 1);
        const int k = in->n_mod[p];
        double iso = 0.;
        if (k >= 0 && k <= S) { iso = 1.; for (int j = 0; j < std::min(k, S - k); j++) iso = iso * (S - j) / (j + 1); }
        const double frag = (double)n_types * std::max(L - 1, 1) * std::max(in->max_charge[p], 1) * (nvar > 1 ? 0.5 * (nvar + 1) : 1.);
        // hits of the spectrum: neighbours with the same spectrum index
        int hits = 1;
        for (int64_t q = p - 1; q >= 0 && in->psm_spec[q] == sp && hits < 64; q--) hits++;
        for (int64_t q = p + 1; q < n && in->psm_spec[q] == sp && hits < 64; q++) hits++;
        const double peaks = (double)(in->spec_off[sp + 1] - in->spec_off[sp]);
        cum[i + 1] = cum[i] + iso * frag + peak_weight * peaks / hits + 64.;
    }
    double share_acc = 0.;
    for (int r = 1; r < world; r++) {
        share_acc += share ? share[r - 1] : 0.;
        const double target = share ? cum[m] * share_acc / share_sum : cum[m] * r / world;
        int64_t i = std::lower_bound(cum.begin(), cum.end(), target) - cum.begin();
        int64_t p = std::min<int64_t>(std::max<int64_t>(i, 0) * stride, n);
        p = std::max(p, cuts[r - 1]);
        while (p > 0 && p < n && in->psm_spec[p] == in->psm_spec[p - 1]) p++;      // never split a spectrum
        cuts[r] = p;
    }
    return PA_OK;
}

extern "C" int pa_shard_ranges(const pa_scorer* s, const pa_batch* in, int32_t world, double peak_weight,
                               const double* share, int64_t* cuts) {
    if (!s) return PA_ERR_ARG;
    return pa_shard_ranges_for(s->mod_group.c_str(), (int32_t)s->frag_types.size(), s->cfg.nvar_cap, in, world, peak_weight, share, cuts);
}

// cpp/ModifiedPeptide.cpp:184-193
extern "C" int pa_site_positions(const pa_scorer* s, const uint8_t* pep, int32_t len, int32_t* pos, int32_t cap) {
    if (!s || !pep) return PA_ERR_ARG;
    bool has_n = s->mod_group.find('n') != std::string::npos, has_c = s->mod_group.find('c') != std::string::npos;
    int n = 0;
    for (int i = 0; i < len; i++) {
        bool site = s->mod_group.find((char)pep[i]) != std::string::npos || (has_n && i == 0) || (has_c && i == len - 1);
        if (site) { if (pos && n < cap) pos[n] = i + 1; n++; }
    }
    return n;
}

// cpp/ModifiedPeptide.cpp:199-253
extern "C" int pa_format_sequence(const pa_scorer* s, const uint8_t* pep, int32_t len, int32_t n_mod,
                                  const uint32_t* aux_pos, const float* aux_mass, int32_t n_aux, uint64_t sig,
                                  char* buf, int32_t cap) {
    if (!s || !pep || !buf || len < 0) return PA_ERR_ARG;
    std::vector<float> mm(len + 2, 0.f);
    std::vector<int> sites;
    bool has_n = s->mod_group.find('n') != std::string::npos, has_c = s->mod_group.find('c') != std::string::npos;
    for (int i = 0; i < len; i++)
        if (s->mod_group.find((char)pep[i]) != std::string::npos || (has_n && i == 0) || (has_c && i == len - 1)) sites.push_back(i);
    if (n_mod > (int)sites.size()) { if (has_n) mm.front() += s->mod_mass; else mm.back() += s->mod_mass; }
    for (size_t j = 0; j < sites.size() && j < 64; j++) {
        if (!((sig >> j) & 1ull)) continue;
        int p = sites[j];
        if (s->mod_group.find((char)pep[p]) != std::string::npos) mm[p + 1] += s->mod_mass;
        else if (p == 0) mm.front() += s->mod_mass;
        else if (p + 1 == len) mm.back() += s->mod_mass;
    }
    for (int a = 0; a < n_aux; a++) if (aux_pos[a] < mm.size()) mm[aux_pos[a]] += aux_mass[a];
    std::string o;
    size_t start = (mm.front() == 0.f) ? 1 : 0, end = (mm.back() == 0.f) ? mm.size() - 1 : mm.size();
    for (size_t i = start; i < end; i++) {
        o += (i == 0) ? 'n' : (i == (size_t)len + 1) ? 'c' : (char)pep[i - 1];
        if (mm[i] > 0.f) { char t[16]; snprintf(t, sizeof(t), "[%d]", (int)std::round(mm[i])); o += t; }
    }
    if ((int)o.size() + 1 > cap) return -(int)o.size() - 1;
    memcpy(buf, o.c_str(), o.size() + 1);
    return (int)o.size();
}

extern "C" int pa_bin_spectra_ex(pa_scorer* s, int64_t n_spec, const int64_t* spec_off, const double* mz,
                                 const double* inten, float* out_mz, uint8_t* out_rank, int32_t* out_count,
                                 int32_t* out_index, int32_t* out_bin, float* out_bounds) {
    if (!s || !spec_off || !mz || !inten || !out_mz || !out_rank || !out_count) return PA_ERR_ARG;
    CK(cudaSetDevice(s->device));
    if (n_spec <= 0) return PA_OK;
    if (is_device_ptr(mz)) return fail(s, PA_ERR_ARG, "pa_bin_spectra takes host arrays");
    Slot& sl = s->slot[0];
    cudaStream_t st = sl.st;
    const int64_t lo = spec_off[0], npk = spec_off[n_spec] - lo;
    const size_t npk1 = (size_t)std::max<int64_t>(npk, 1);
    PaBinArgs ba;
    int64_t h2d = 0;
    for (const ChunkArray& a : {ChunkArray(spec_off, 0, n_spec + 1, sl.spec_off, ba.spec_off), ChunkArray(mz, lo, npk, sl.mz, ba.mz),
                                ChunkArray(inten, lo, npk, sl.inten, ba.inten)})
        CK(stage(a, false, st, &h2d));
    DevBuf rmz, rrank;
    CK(sl.rpk.ensure(npk1 * sizeof(float2))); CK(rmz.ensure(npk1 * 4)); CK(rrank.ensure(npk1));
    CK(sl.g_bin.ensure(npk1 * 4)); CK(sl.g_tmp.ensure(npk1));
    CK(sl.rcount.ensure((size_t)n_spec * 4));
    CK(sl.ctab.ensure((size_t)n_spec * PA_NCELL)); CK(sl.chead.ensure((size_t)n_spec * sizeof(float2)));
    const bool extra = out_index || out_bin || out_bounds;
    DevBuf d_index, d_bin, d_bounds;
    if (extra) { CK(d_index.ensure(npk1 * 4)); CK(d_bin.ensure(npk1 * 4)); CK(d_bounds.ensure((size_t)n_spec * 12)); }
    int64_t m = 0;
    for (int64_t q = 0; q < n_spec; q++) m = std::max<int64_t>(m, spec_off[q + 1] - spec_off[q]);
    ba.inten32 = nullptr; ba.peak_base = 0; ba.n_spec = n_spec;
    ba.mz32 = nullptr; ba.esc_off = nullptr; ba.mz_esc = nullptr;
    ba.rpk = sl.rpk.as<float2>() - lo; ba.rmz = rmz.as<float>() - lo; ba.rrank = rrank.as<uint8_t>() - lo;
    ba.g_bin = sl.g_bin.as<int32_t>() - lo; ba.g_tmp = sl.g_tmp.as<uint8_t>() - lo;
    ba.rcount = sl.rcount.as<int32_t>(); ba.bin_size = s->bin_size; ba.n_top = s->n_top;
    ba.ctab = sl.ctab.as<uint8_t>(); ba.chead = sl.chead.as<float2>();
    ba.list = nullptr; ba.list_n = nullptr;
    ba.rindex = extra ? d_index.as<int32_t>() - lo : nullptr;
    ba.rbin = extra ? d_bin.as<int32_t>() - lo : nullptr;
    ba.bounds = extra ? d_bounds.as<float>() : nullptr;
    int cap, wpb, blocks;
    size_t smem;
    bin_launch_shape(s->sm_count, m, n_spec, &cap, &wpb, &smem, &blocks);
    ba.cap = cap;
    k_bin_topn<false><<<blocks, wpb * 32, smem, st>>>(ba);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out_mz + lo, rmz.p, (size_t)npk * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(out_rank + lo, rrank.p, (size_t)npk, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(out_count, sl.rcount.p, (size_t)n_spec * 4, cudaMemcpyDeviceToHost, st));
    if (out_index) CK(cudaMemcpyAsync(out_index + lo, d_index.p, (size_t)npk * 4, cudaMemcpyDeviceToHost, st));
    if (out_bin) CK(cudaMemcpyAsync(out_bin + lo, d_bin.p, (size_t)npk * 4, cudaMemcpyDeviceToHost, st));
    if (out_bounds) CK(cudaMemcpyAsync(out_bounds, d_bounds.p, (size_t)n_spec * 12, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return PA_OK;
}

extern "C" int pa_bin_spectra(pa_scorer* s, int64_t n_spec, const int64_t* spec_off, const double* mz,
                              const double* inten, float* out_mz, uint8_t* out_rank, int32_t* out_count) {
    return pa_bin_spectra_ex(s, n_spec, spec_off, mz, inten, out_mz, out_rank, out_count, nullptr, nullptr, nullptr);
}

// ---- single-peptide probes ------------------------------------------------------------------------
// One peptide (+ fixed mods) staged as a 1-PSM chunk without a spectrum, for the probe kernels.
struct ProbePsm {
    DevBuf buf;
    PaBatchDev b;
};

static int stage_probe_psm(pa_scorer* s, const uint8_t* pep, int32_t len, const uint32_t* aux_pos,
                           const float* aux_mass, int32_t n_aux, int32_t max_charge, ProbePsm& pp) {
    if (len < 1 || len > PA_MAX_PEPTIDE) return fail(s, PA_ERR_UNSUPPORTED, "peptide length must be 1..%d", PA_MAX_PEPTIDE);
    for (int i = 0; i < len; i++)
        if (pep[i] < 'A' || pep[i] > 'Z' || std::isnan(residue_mass_host((char)pep[i])))
            return fail(s, PA_ERR_ARG, "unknown residue letter '%c'", pep[i]);
    for (int a = 0; a < n_aux; a++)
        if (aux_pos[a] > (uint32_t)len) return fail(s, PA_ERR_ARG, "fixed-mod position %u beyond the peptide", aux_pos[a]);
    // layout: pep_off i32[2] | n_mod i32 | max_charge i32 | aux_off i32[2] | psm_spec i32 | pad | aux_pos | aux_mass | pep
    const size_t n_aux1 = (size_t)std::max(n_aux, 1);
    std::vector<unsigned char> h(32 + n_aux1 * 8 + (size_t)len + 8, 0);
    int32_t* hi = (int32_t*)h.data();
    hi[0] = 0; hi[1] = len; hi[2] = 0; hi[3] = max_charge; hi[4] = 0; hi[5] = n_aux; hi[6] = 0;
    if (n_aux > 0) { memcpy(h.data() + 32, aux_pos, (size_t)n_aux * 4); memcpy(h.data() + 32 + n_aux1 * 4, aux_mass, (size_t)n_aux * 4); }
    memcpy(h.data() + 32 + n_aux1 * 8, pep, (size_t)len);
    CK(pp.buf.ensure(h.size()));
    CK(cudaMemcpy(pp.buf.p, h.data(), h.size(), cudaMemcpyHostToDevice));
    unsigned char* d = pp.buf.as<unsigned char>();
    memset(&pp.b, 0, sizeof(pp.b));
    pp.b.pep_off = (const int32_t*)d; pp.b.n_mod = (const int32_t*)(d + 8); pp.b.max_charge = (const int32_t*)(d + 12);
    pp.b.aux_off = (const int32_t*)(d + 16); pp.b.psm_spec = (const int32_t*)(d + 24);
    pp.b.aux_pos = (const uint32_t*)(d + 32); pp.b.aux_mass = (const float*)(d + 32 + n_aux1 * 4);
    pp.b.pep = d + 32 + n_aux1 * 8;
    return PA_OK;
}

extern "C" int pa_fragment_table(pa_scorer* s, const uint8_t* pep, int32_t len, const uint32_t* aux_pos,
                                 const float* aux_mass, int32_t n_aux, uint64_t sig, char fragment_type,
                                 int32_t charge, float* out_mz, int32_t* out_nvar) {
    if (!s || !pep || !out_mz || !out_nvar || (n_aux > 0 && (!aux_pos || !aux_mass))) return PA_ERR_ARG;
    if (!strchr("bcyzZ", fragment_type) || fragment_type == 0) return fail(s, PA_ERR_ARG, "fragment type not in \"bcyzZ\"");
    if (charge < 0) return fail(s, PA_ERR_ARG, "negative charge");
    CK(cudaSetDevice(s->device));
    ProbePsm pp;
    int rc = stage_probe_psm(s, pep, len, aux_pos, aux_mass, n_aux, std::max(charge, 1), pp);
    if (rc != PA_OK) return rc;
    DevBuf d_mz, d_nv;
    CK(d_mz.ensure((size_t)len * 16 * 4)); CK(d_nv.ensure((size_t)len * 4));
    CK(cudaMemset(d_mz.p, 0, (size_t)len * 16 * 4));
    PaFragArgs a;
    a.sig = sig; a.type = fragment_type; a.charge = charge; a.out_mz = d_mz.as<float>(); a.out_nvar = d_nv.as<int32_t>();
    k_fragment_table<<<1, 32, sizeof(PsmSmem)>>>(s->cfg, pp.b, a);
    CK(cudaGetLastError());
    CK(cudaMemcpy(out_mz, d_mz.p, (size_t)len * 16 * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(out_nvar, d_nv.p, (size_t)len * 4, cudaMemcpyDeviceToHost));
    return PA_OK;
}

extern "C" int pa_site_determining_ions(pa_scorer* s, const uint8_t* pep, int32_t len, const uint32_t* aux_pos,
                                        const float* aux_mass, int32_t n_aux, uint64_t sig_a, uint64_t sig_b,
                                        char fragment_type, int32_t max_charge, float* out_a, int32_t* n_a,
                                        float* out_b, int32_t* n_b, int32_t cap) {
    if (!s || !pep || !out_a || !out_b || !n_a || !n_b || (n_aux > 0 && (!aux_pos || !aux_mass))) return PA_ERR_ARG;
    if (!strchr("bcyzZ", fragment_type) || fragment_type == 0) return fail(s, PA_ERR_ARG, "fragment type not in \"bcyzZ\"");
    if (max_charge < 1) return fail(s, PA_ERR_ARG, "max_charge must be >= 1");
    CK(cudaSetDevice(s->device));
    ProbePsm pp;
    int rc = stage_probe_psm(s, pep, len, aux_pos, aux_mass, n_aux, max_charge, pp);
    if (rc != PA_OK) return rc;
    const long long per_type = (long long)(len > 1 ? len - 1 : 1) * s->cfg.nvar_cap * max_charge;
    if (per_type > (1 << 20)) return fail(s, PA_ERR_UNSUPPORTED, "fragment list too long");
    PaSdiArgs a;
    a.sig_a = sig_a; a.sig_b = sig_b; a.type = fragment_type; a.max_charge = max_charge;
    a.list_stride = 32;
    while (a.list_stride < per_type) a.list_stride <<= 1;
    DevBuf d_a, d_b, d_cnt, d_lists;
    CK(d_a.ensure((size_t)a.list_stride * 4)); CK(d_b.ensure((size_t)a.list_stride * 4)); CK(d_cnt.ensure(8));
    if (per_type > PA_LCAP) CK(d_lists.ensure((size_t)4 * a.list_stride * sizeof(float)));
    a.out_a = d_a.as<float>(); a.out_b = d_b.as<float>(); a.counts = d_cnt.as<int32_t>(); a.g_lists = d_lists.as<float>();
    CK(cudaFuncSetAttribute(k_sdi_probe, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    k_sdi_probe<<<1, 32, sizeof(SelSmem)>>>(s->cfg, pp.b, a);
    CK(cudaGetLastError());
    int32_t cnt[2];
    CK(cudaMemcpy(cnt, d_cnt.p, 8, cudaMemcpyDeviceToHost));
    *n_a = cnt[0]; *n_b = cnt[1];
    if (std::min(cnt[0], cap) > 0) CK(cudaMemcpy(out_a, d_a.p, (size_t)std::min(cnt[0], cap) * 4, cudaMemcpyDeviceToHost));
    if (std::min(cnt[1], cap) > 0) CK(cudaMemcpy(out_b, d_b.p, (size_t)std::min(cnt[1], cap) * 4, cudaMemcpyDeviceToHost));
    return PA_OK;
}

extern "C" int pa_log_math(pa_scorer* s, int32_t op, int32_t n, const float* x, const float* y, const int32_t* k,
                           const int32_t* tr, float prob, float* out) {
    if (!s || !out || n < 0 || op < 0 || op > 4) return PA_ERR_ARG;
    if (op == 0 ? (!x || !y) : (!k || !tr)) return PA_ERR_ARG;
    if (n == 0) return PA_OK;
    CK(cudaSetDevice(s->device));
    int max_tr = 0;
    if (op > 0)
        for (int i = 0; i < n; i++) {
            if (k[i] < 0 || tr[i] < 0 || k[i] > tr[i]) return fail(s, PA_ERR_ARG, "successes %d / trials %d out of range", k[i], tr[i]);
            max_tr = std::max(max_tr, tr[i]);
        }
    if (max_tr > 65535) return fail(s, PA_ERR_UNSUPPORTED, "trials beyond 65535 (the reference packs (k, n) in 2 x 16 bits)");
    std::vector<double> logd(max_tr + 2);
    logd[0] = 0.;
    for (int m = 1; m <= max_tr + 1; m++) logd[m] = std::log((double)m);
    DevBuf d_in0, d_in1, d_logd, d_out;
    CK(d_in0.ensure((size_t)n * 4)); CK(d_in1.ensure((size_t)n * 4)); CK(d_out.ensure((size_t)n * 4));
    CK(d_logd.ensure(logd.size() * 8));
    CK(cudaMemcpy(d_in0.p, op == 0 ? (const void*)x : (const void*)k, (size_t)n * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_in1.p, op == 0 ? (const void*)y : (const void*)tr, (size_t)n * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_logd.p, logd.data(), logd.size() * 8, cudaMemcpyHostToDevice));
    PaMathArgs a;
    a.op = op; a.n = n; a.x = d_in0.as<float>(); a.y = d_in1.as<float>(); a.k = d_in0.as<int32_t>(); a.tr = d_in1.as<int32_t>();
    a.logd = d_logd.as<double>(); a.out = d_out.as<float>();
    // cpp/Util.cpp:52-55 with the platform libm, as the scorer itself does
    a.lps = logf(prob);
    a.lpf = (float)std::log(1. - (double)prob);
    volatile double one = 1.0;
    a.log10e = std::log10(std::exp(one));
    k_math_probe<<<(n + 127) / 128, 128>>>(a);
    CK(cudaGetLastError());
    CK(cudaMemcpy(out, d_out.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
    return PA_OK;
}

extern "C" int64_t pa_power_set_sums(const float* target, int32_t n, int32_t max_depth, float* out, int64_t cap) {
    if (n < 0 || max_depth < 0 || (n > 0 && !target)) return PA_ERR_ARG;
    if (n > 24) return PA_ERR_UNSUPPORTED;
    std::vector<float> t(target, target + n), sums;
    power_set_sums(t, (size_t)max_depth, sums);
    for (int64_t i = 0; i < (int64_t)sums.size() && i < cap; i++) out[i] = sums[i];
    return (int64_t)sums.size();
}

extern "C" int pa_tail_table(pa_scorer* s, int32_t n_max, float* out) {
    if (!s || !out || n_max < 0) return PA_ERR_ARG;
    CK(cudaSetDevice(s->device));
    int rc = ensure_table(s, n_max);
    if (rc != PA_OK) return rc;
    size_t entries = ((size_t)n_max + 1) * ((size_t)n_max + 2) / 2;
    const int nd = s->n_deep;
    if (nd == 0) {
        CK(cudaMemcpy(out, s->d_T.p, entries * PA_N_TOP * sizeof(float), cudaMemcpyDeviceToHost));
        return PA_OK;
    }
    // rows of n_top: depths 0..9 from T, 10 .. n_top-1 from T_deep (strided copies straight into the caller's rows)
    CK(cudaMemcpy2D(out, (size_t)(PA_N_TOP + nd) * sizeof(float), s->d_T.p, PA_N_TOP * sizeof(float), PA_N_TOP * sizeof(float),
                    entries, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy2D(out + PA_N_TOP, (size_t)(PA_N_TOP + nd) * sizeof(float), s->d_T_deep.p, nd * sizeof(float), nd * sizeof(float),
                    entries, cudaMemcpyDeviceToHost));
    return PA_OK;
}

extern "C" int pa_counters(const pa_scorer* s, pa_counters_t* out) {
    if (!s || !out) return PA_ERR_ARG;
    *out = s->ctr;
    return PA_OK;
}
