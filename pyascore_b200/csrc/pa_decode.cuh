// mzML binary arrays on the GPU: base64 -> (zlib inflate) -> float64 at the array's CSR offset.
//
// Stands in for the byte work of the stdlib reader's _decode_mzml_array (pyascore_b200/parsing/_xml.py, reference:
// MzMLExtractor, spec_parsers.py:49-110): base64.b64decode(text) with validate=False, zlib.decompress, then
// np.frombuffer(raw, dtype).astype(np.float64).
//
// Layout: k_decode_arrays runs 128-thread blocks, one warp per binary array (grid-stride over the array table).
//   - base64: the warp reads 32 characters per step; a ballot keeps the alphabet characters, their prefix rank packs
//     the 6-bit values into a per-warp shared buffer, and every complete quad becomes 3 bytes in the array's scratch.
//   - zlib: lane 0 runs pa_inflate (the __host__ __device__ core below; pa_inflate_host builds the same source for
//     the CPU tests) with its Huffman tables in the warp's shared memory.
//   - conversion: all lanes convert the raw elements to float64 and write them at the array's output offset.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define PA_HD __host__ __device__
#else
#define PA_HD
#endif

enum { PA_DEC_OK = 0, PA_DEC_BASE64 = 1, PA_DEC_ZLIB = 2, PA_DEC_LENGTH = 3 };

// ---------------------------------------------------------------------------------------------
// inflate (RFC 1950 zlib stream around RFC 1951 DEFLATE), canonical-code decoding one bit at a time
// ---------------------------------------------------------------------------------------------
#define PA_MAXBITS 15
#define PA_MAXLCODES 286
#define PA_MAXDCODES 30
#define PA_FIXLCODES 288

struct PaHuff {
    int16_t count[PA_MAXBITS + 1];   // codes of each length
    int16_t symbol[PA_FIXLCODES];    // symbols ordered by code
};

struct PaInflateTables {
    PaHuff len, dist;
    uint8_t lengths[PA_MAXLCODES + PA_MAXDCODES];
};

struct PaInflate {
    const uint8_t* in;
    int64_t n_in, pos;
    uint32_t bitbuf;
    int bitcnt;
    uint8_t* out;
    int64_t cap, n_out;
    int err;     // 0, or 1 = malformed / truncated stream, 2 = output beyond `cap`
};

PA_HD inline int pa_bits(PaInflate& s, int need) {
    uint32_t v = s.bitbuf;
    while (s.bitcnt < need) {
        if (s.pos >= s.n_in) { s.err = 1; return 0; }
        v |= (uint32_t)s.in[s.pos++] << s.bitcnt;
        s.bitcnt += 8;
    }
    s.bitbuf = v >> need;
    s.bitcnt -= need;
    return (int)(v & ((1u << need) - 1u));
}

PA_HD inline int pa_decode_sym(PaInflate& s, const PaHuff& h) {
    int code = 0, first = 0, index = 0;
    for (int len = 1; len <= PA_MAXBITS; len++) {
        code |= pa_bits(s, 1);
        if (s.err) return -1;
        const int count = h.count[len];
        if (code - count < first) return h.symbol[index + (code - first)];
        index += count;
        first += count;
        first <<= 1;
        code <<= 1;
    }
    return -1;      // no code of 15 bits or fewer matches
}

// < 0: over-subscribed; 0: complete (or no codes at all); > 0: incomplete
PA_HD inline int pa_construct(PaHuff& h, const uint8_t* length, int n) {
    for (int len = 0; len <= PA_MAXBITS; len++) h.count[len] = 0;
    for (int sym = 0; sym < n; sym++) h.count[length[sym]]++;
    if (h.count[0] == n) return 0;
    int left = 1;
    for (int len = 1; len <= PA_MAXBITS; len++) {
        left <<= 1;
        left -= h.count[len];
        if (left < 0) return left;
    }
    int16_t offs[PA_MAXBITS + 1];
    offs[1] = 0;
    for (int len = 1; len < PA_MAXBITS; len++) offs[len + 1] = offs[len] + h.count[len];
    for (int sym = 0; sym < n; sym++)
        if (length[sym] != 0) h.symbol[offs[length[sym]]++] = (int16_t)sym;
    return left;
}

PA_HD inline bool pa_codes(PaInflate& s, const PaHuff& lc, const PaHuff& dc) {
    for (;;) {
        int sym = pa_decode_sym(s, lc);
        if (sym < 0) { s.err = 1; return false; }
        if (sym < 256) {
            if (s.n_out >= s.cap) { s.err = 2; return false; }
            s.out[s.n_out++] = (uint8_t)sym;
        } else if (sym == 256) {
            return true;
        } else {
            const int i = sym - 257;
            if (i >= 29) { s.err = 1; return false; }
            int len;
            if (i < 8) len = 3 + i;
            else if (i == 28) len = 258;
            else { const int eb = (i - 4) >> 2; len = ((4 + (i & 3)) << eb) + 3 + pa_bits(s, eb); }
            const int d = pa_decode_sym(s, dc);
            if (d < 0 || d >= 30) { s.err = 1; return false; }
            int dist;
            if (d < 4) dist = 1 + d;
            else { const int eb = (d >> 1) - 1; dist = ((2 + (d & 1)) << eb) + 1 + pa_bits(s, eb); }
            if (s.err) return false;
            if ((int64_t)dist > s.n_out) { s.err = 1; return false; }
            if (s.n_out + len > s.cap) { s.err = 2; return false; }
            uint8_t* o = s.out + s.n_out;
            for (int k = 0; k < len; k++) o[k] = o[k - dist];
            s.n_out += len;
        }
    }
}

PA_HD inline bool pa_stored(PaInflate& s) {
    s.bitbuf = 0;               // the rest of the current byte
    s.bitcnt = 0;
    if (s.pos + 4 > s.n_in) { s.err = 1; return false; }
    const uint32_t len = s.in[s.pos] | ((uint32_t)s.in[s.pos + 1] << 8);
    const uint32_t nlen = s.in[s.pos + 2] | ((uint32_t)s.in[s.pos + 3] << 8);
    s.pos += 4;
    if (len != (~nlen & 0xffffu)) { s.err = 1; return false; }
    if (s.pos + len > s.n_in) { s.err = 1; return false; }
    if (s.n_out + len > s.cap) { s.err = 2; return false; }
    for (uint32_t k = 0; k < len; k++) s.out[s.n_out + k] = s.in[s.pos + k];
    s.pos += len;
    s.n_out += len;
    return true;
}

PA_HD inline bool pa_fixed(PaInflate& s, PaInflateTables& t) {
    for (int k = 0; k < 144; k++) t.lengths[k] = 8;
    for (int k = 144; k < 256; k++) t.lengths[k] = 9;
    for (int k = 256; k < 280; k++) t.lengths[k] = 7;
    for (int k = 280; k < PA_FIXLCODES; k++) t.lengths[k] = 8;
    pa_construct(t.len, t.lengths, PA_FIXLCODES);
    for (int k = 0; k < PA_MAXDCODES; k++) t.lengths[k] = 5;
    pa_construct(t.dist, t.lengths, PA_MAXDCODES);
    return pa_codes(s, t.len, t.dist);
}

PA_HD inline bool pa_dynamic(PaInflate& s, PaInflateTables& t) {
    const uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
    const int nlen = pa_bits(s, 5) + 257, ndist = pa_bits(s, 5) + 1, ncode = pa_bits(s, 4) + 4;
    if (s.err || nlen > PA_MAXLCODES || ndist > PA_MAXDCODES) { s.err = 1; return false; }
    int idx;
    for (idx = 0; idx < ncode; idx++) t.lengths[order[idx]] = (uint8_t)pa_bits(s, 3);
    for (; idx < 19; idx++) t.lengths[order[idx]] = 0;
    if (s.err || pa_construct(t.len, t.lengths, 19) != 0) { s.err = 1; return false; }   // complete code-length code
    idx = 0;
    while (idx < nlen + ndist) {
        int sym = pa_decode_sym(s, t.len);
        if (sym < 0) { s.err = 1; return false; }
        if (sym < 16) { t.lengths[idx++] = (uint8_t)sym; continue; }
        int len = 0, rep;
        if (sym == 16) {
            if (idx == 0) { s.err = 1; return false; }
            len = t.lengths[idx - 1];
            rep = 3 + pa_bits(s, 2);
        } else if (sym == 17) rep = 3 + pa_bits(s, 3);
        else rep = 11 + pa_bits(s, 7);
        if (s.err || idx + rep > nlen + ndist) { s.err = 1; return false; }
        while (rep--) t.lengths[idx++] = (uint8_t)len;
    }
    if (t.lengths[256] == 0) { s.err = 1; return false; }
    // incomplete codes are accepted only for a single code of one bit, as zlib does
    int err = pa_construct(t.len, t.lengths, nlen);
    if (err && (err < 0 || nlen != t.len.count[0] + t.len.count[1])) { s.err = 1; return false; }
    err = pa_construct(t.dist, t.lengths + nlen, ndist);
    if (err && (err < 0 || ndist != t.dist.count[0] + t.dist.count[1])) { s.err = 1; return false; }
    return pa_codes(s, t.len, t.dist);
}

// zlib.decompress(in) into out[0, cap): returns the output length, -1 for a stream zlib rejects (bad header, preset
// dictionary, bad block, truncated, Adler-32 mismatch), -2 when the output would exceed cap.  Bytes after the trailer are
// ignored, as zlib.decompress ignores them.
PA_HD inline int64_t pa_inflate(const uint8_t* in, int64_t n_in, uint8_t* out, int64_t cap, PaInflateTables& t) {
    if (n_in < 2) return -1;
    const int cmf = in[0], flg = in[1];
    if ((cmf & 15) != 8 || (cmf >> 4) > 7 || ((cmf << 8) | flg) % 31 != 0 || (flg & 0x20)) return -1;
    PaInflate s{in, n_in, 2, 0u, 0, out, cap, 0, 0};
    int last;
    do {
        last = pa_bits(s, 1);
        const int type = pa_bits(s, 2);
        if (s.err) return -1;
        bool ok;
        if (type == 0) ok = pa_stored(s);
        else if (type == 1) ok = pa_fixed(s, t);
        else if (type == 2) ok = pa_dynamic(s, t);
        else { s.err = 1; ok = false; }
        if (!ok) return s.err == 2 ? -2 : -1;
    } while (!last);
    if (s.pos + 4 > s.n_in) return -1;      // the trailer starts at the next byte boundary
    const uint32_t want = ((uint32_t)in[s.pos] << 24) | ((uint32_t)in[s.pos + 1] << 16) | ((uint32_t)in[s.pos + 2] << 8) |
                          in[s.pos + 3];
    uint32_t a = 1, b = 0;
    for (int64_t k = 0; k < s.n_out;) {
        const int64_t end = k + 5552 < s.n_out ? k + 5552 : s.n_out;
        for (; k < end; k++) { a += out[k]; b += a; }
        a %= 65521u;
        b %= 65521u;
    }
    if (((b << 16) | a) != want) return -1;
    return s.n_out;
}

#ifdef __CUDACC__
// ---------------------------------------------------------------------------------------------
// the kernel
// ---------------------------------------------------------------------------------------------
struct PaDecodeJob {                // one binary array: the public pa_mzml_array + its scratch ranges
    int64_t text_off, text_len, out_off, count;
    int64_t raw_off;                // base64 output (capacity 3 * (text_len / 4) + 3)
    int64_t inf_off;                // inflate output (capacity count * element size), zlib arrays only
    int32_t dtype, flags;
};

#define PA_DEC_WARPS 4
#define PA_DEC_ZLIB_FLAG 1
#define PA_DEC_INTEN_FLAG 2

__device__ __forceinline__ int pa_elem_size(int dtype) { return (dtype == 0 || dtype == 3) ? 8 : 4; }

// 0..63: alphabet value; 64: '='; 65: skipped by b64decode(validate=False); 66: refused (non-ASCII -- str.encode('ascii')
// fails -- or '&', the start of an entity whose decoded text the raw bytes do not show)
__device__ __forceinline__ int pa_b64_class(unsigned c) {
    if (c >= 'A' && c <= 'Z') return c - 'A';
    if (c >= 'a' && c <= 'z') return c - 'a' + 26;
    if (c >= '0' && c <= '9') return c - '0' + 52;
    if (c == '+') return 62;
    if (c == '/') return 63;
    if (c == '=') return 64;
    if (c >= 0x80 || c == '&') return 66;
    return 65;
}

__global__ void __launch_bounds__(32 * PA_DEC_WARPS) k_decode_arrays(
    const uint8_t* __restrict__ file, const PaDecodeJob* __restrict__ jobs, int64_t n_jobs, uint8_t* __restrict__ scratch,
    double* __restrict__ mz_out, double* __restrict__ inten_out, int32_t* __restrict__ status, int32_t* __restrict__ inexact) {
    __shared__ PaInflateTables tables[PA_DEC_WARPS];
    __shared__ uint8_t sext[PA_DEC_WARPS][40];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const unsigned lt_mask = (1u << lane) - 1u;
    const int64_t warps = (int64_t)gridDim.x * PA_DEC_WARPS;
    for (int64_t j = (int64_t)blockIdx.x * PA_DEC_WARPS + w; j < n_jobs; j += warps) {
        const PaDecodeJob a = jobs[j];
        const uint8_t* text = file + a.text_off;
        uint8_t* raw = scratch + a.raw_off;
        int st = PA_DEC_OK;
        // ---- base64 ----
        int carry = 0, pads = 0;
        bool pad_seen = false;
        int64_t nraw = 0;
        for (int64_t base = 0; base < a.text_len; base += 32) {
            const int64_t i = base + lane;
            const int v = i < a.text_len ? pa_b64_class(text[i]) : 65;
            const unsigned valid = __ballot_sync(~0u, v < 64), padm = __ballot_sync(~0u, v == 64),
                           bad = __ballot_sync(~0u, v == 66);
            // data after padding: b64decode stops at a complete pad or ignores a stray one; neither is followed here
            if (bad || (pad_seen && valid) || (padm && (valid >> (__ffs(padm) - 1)))) { st = PA_DEC_BASE64; break; }
            pad_seen |= padm != 0;
            pads += __popc(padm);
            if (v < 64) sext[w][carry + __popc(valid & lt_mask)] = (uint8_t)v;
            __syncwarp();
            const int tot = carry + __popc(valid), nq = tot >> 2;
            if (lane < nq) {
                const uint8_t* q = sext[w] + 4 * lane;
                uint8_t* o = raw + nraw + 3 * lane;
                o[0] = (uint8_t)((q[0] << 2) | (q[1] >> 4));
                o[1] = (uint8_t)((q[1] << 4) | (q[2] >> 2));
                o[2] = (uint8_t)((q[2] << 6) | q[3]);
            }
            nraw += 3 * nq;
            const int left = tot & 3;
            uint8_t keep = lane < left ? sext[w][4 * nq + lane] : 0;
            __syncwarp();
            if (lane < left) sext[w][lane] = keep;
            __syncwarp();
            carry = left;
        }
        if (st == PA_DEC_OK) {
            // 1 data character past a quad, or 2 / 3 without their padding: "Incorrect padding"
            if (carry == 1 || (carry == 2 && pads < 2) || (carry == 3 && pads < 1)) st = PA_DEC_BASE64;
            else if (carry >= 2 && lane == 0) {
                raw[nraw] = (uint8_t)((sext[w][0] << 2) | (sext[w][1] >> 4));
                if (carry == 3) raw[nraw + 1] = (uint8_t)((sext[w][1] << 4) | (sext[w][2] >> 2));
            }
            nraw += carry > 1 ? carry - 1 : 0;
        }
        __syncwarp();
        // ---- zlib ----
        const int esz = pa_elem_size(a.dtype);
        const uint8_t* elems = raw;
        int64_t nbytes = nraw;
        if (st == PA_DEC_OK && (a.flags & PA_DEC_ZLIB_FLAG) && nraw > 0) {
            int64_t r = 0;
            if (lane == 0) r = pa_inflate(raw, nraw, scratch + a.inf_off, a.count * esz, tables[w]);
            r = __shfl_sync(~0u, r, 0);
            if (r == -1) st = PA_DEC_ZLIB;
            else if (r == -2) st = PA_DEC_LENGTH;
            elems = scratch + a.inf_off;
            nbytes = r;
        }
        __syncwarp();
        // ---- length check and conversion ----
        if (st == PA_DEC_OK && (nbytes % esz != 0 || nbytes / esz != a.count)) st = PA_DEC_LENGTH;
        if (st == PA_DEC_OK) {
            const bool is_inten = (a.flags & PA_DEC_INTEN_FLAG) != 0;
            double* out = (is_inten ? inten_out : mz_out) + a.out_off;
            bool inexact_here = false;
            for (int64_t e = lane; e < a.count; e += 32) {
                double v;
                if (a.dtype == 0) v = ((const double*)elems)[e];
                else if (a.dtype == 1) v = (double)((const float*)elems)[e];
                else if (a.dtype == 2) v = (double)((const int32_t*)elems)[e];
                else v = (double)((const long long*)elems)[e];
                out[e] = v;
                inexact_here |= is_inten && !((double)(float)v == v);
            }
            if (__any_sync(~0u, inexact_here) && lane == 0) atomicOr(inexact, 1);
        }
        if (lane == 0) status[j] = st;
    }
}
#endif
