// C ABI of the mzML decoder (include/pyascore_b200.h): pa_decode_arrays launches k_decode_arrays (pa_decode.cuh) over the
// array table pa_mzml_index (pa_mzml.cpp) built; pa_inflate_host is the same inflate core on the CPU.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <vector>

#include "../../include/pyascore_b200.h"
#include "pa_decode.cuh"

namespace {

int fail_text(char* err, int32_t cap, int code, const char* what, cudaError_t e) {
    if (err && cap > 0) snprintf(err, (size_t)cap, "%s: %s", what, e == cudaSuccess ? "invalid argument" : cudaGetErrorString(e));
    return code;
}

struct DeviceMem {
    void* p = nullptr;
    ~DeviceMem() { if (p) cudaFree(p); }
};

}  // namespace

// spec_parsers.py:49-110 (the payload half of MzMLExtractor: b64decode, zlib.decompress, np.frombuffer(...).astype(f8))
extern "C" int pa_decode_arrays(int device, const uint8_t* file_dev, const pa_mzml_array* arrays, int64_t n_arrays,
                                double* mz_out, double* inten_out, int32_t* status_out, int32_t* inexact_out, char* err,
                                int32_t err_cap) {
    if (n_arrays < 0 || (n_arrays > 0 && (!file_dev || !arrays || !mz_out || !inten_out || !status_out)) || !inexact_out)
        return fail_text(err, err_cap, PA_ERR_ARG, "pa_decode_arrays: NULL or negative argument", cudaSuccess);
    int prev = 0;
    cudaError_t e = cudaGetDevice(&prev);
    if (e == cudaSuccess) e = cudaSetDevice(device);
    if (e != cudaSuccess) return fail_text(err, err_cap, PA_ERR_CUDA, "cudaSetDevice", e);
    struct Restore { int d; ~Restore() { cudaSetDevice(d); } } restore{prev};     // the caller's current device stays
    e = cudaMemsetAsync(inexact_out, 0, sizeof(int32_t), 0);
    if (e != cudaSuccess) return fail_text(err, err_cap, PA_ERR_CUDA, "cudaMemsetAsync", e);
    if (n_arrays == 0) {
        e = cudaStreamSynchronize(0);
        return e == cudaSuccess ? PA_OK : fail_text(err, err_cap, PA_ERR_CUDA, "cudaStreamSynchronize", e);
    }
    // scratch: every array's base64 output, then the inflate output of the zlib arrays (16-byte aligned ranges)
    std::vector<PaDecodeJob> jobs((size_t)n_arrays);
    int64_t off = 0;
    auto take = [&](int64_t bytes) { const int64_t o = off; off += (bytes + 15) & ~(int64_t)15; return o; };
    for (int64_t j = 0; j < n_arrays; j++) {
        const pa_mzml_array& a = arrays[j];
        if (a.dtype < PA_MZML_F64 || a.dtype > PA_MZML_I64 || a.count < 0 || a.text_len < 0 || a.text_off < 0)
            return fail_text(err, err_cap, PA_ERR_ARG, "pa_decode_arrays: bad array table entry", cudaSuccess);
        PaDecodeJob& jb = jobs[(size_t)j];
        jb.text_off = a.text_off;
        jb.text_len = a.text_len;
        jb.out_off = a.out_off;
        jb.count = a.count;
        jb.dtype = a.dtype;
        jb.flags = ((a.flags & PA_MZML_ZLIB) ? PA_DEC_ZLIB_FLAG : 0) | ((a.flags & PA_MZML_INTENSITY) ? PA_DEC_INTEN_FLAG : 0);
        jb.raw_off = take(3 * (a.text_len / 4) + 3);
    }
    for (auto& jb : jobs)
        jb.inf_off = (jb.flags & PA_DEC_ZLIB_FLAG) ? take(jb.count * ((jb.dtype == 0 || jb.dtype == 3) ? 8 : 4)) : 0;
    DeviceMem scratch, table;
    e = cudaMalloc(&scratch.p, (size_t)std::max<int64_t>(off, 16));
    if (e == cudaSuccess) e = cudaMalloc(&table.p, jobs.size() * sizeof(PaDecodeJob));
    if (e != cudaSuccess) return fail_text(err, err_cap, PA_ERR_CUDA, "cudaMalloc (decode scratch)", e);
    e = cudaMemcpyAsync(table.p, jobs.data(), jobs.size() * sizeof(PaDecodeJob), cudaMemcpyHostToDevice, 0);
    if (e != cudaSuccess) return fail_text(err, err_cap, PA_ERR_CUDA, "cudaMemcpyAsync (array table)", e);
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    const int64_t blocks = std::min<int64_t>((n_arrays + PA_DEC_WARPS - 1) / PA_DEC_WARPS, (int64_t)sms * 16);
    k_decode_arrays<<<(unsigned)blocks, 32 * PA_DEC_WARPS, 0, 0>>>(file_dev, (const PaDecodeJob*)table.p, n_arrays,
                                                                   (uint8_t*)scratch.p, mz_out, inten_out, status_out,
                                                                   inexact_out);
    e = cudaGetLastError();
    if (e != cudaSuccess) return fail_text(err, err_cap, PA_ERR_CUDA, "k_decode_arrays launch", e);
    e = cudaStreamSynchronize(0);
    if (e != cudaSuccess) return fail_text(err, err_cap, PA_ERR_CUDA, "k_decode_arrays", e);
    return PA_OK;
}

extern "C" int64_t pa_inflate_host(const uint8_t* in, int64_t n_in, uint8_t* out, int64_t cap) {
    if ((!in && n_in > 0) || (!out && cap > 0) || n_in < 0 || cap < 0) return -1;
    PaInflateTables t;
    return pa_inflate(in, n_in, out, cap, t);
}
