// A witness generator outside libhfb200, in the shape of upstream's GPU witgen: a compact per-job record (one 64-bit seed per
// data column, standing in for the preflight trace) is copied from pinned host memory into the context's scratch, expanded on
// the device into the active rows of every data column with a counter-based hash, and the blinding rows come from the
// library (hfb200_segment_data_blind).  The same expansion in numpy: tests/test_device_witness_seam.py `expand_columns`.
#include <cuda_runtime.h>
#include "hfb200.h"

static const uint64_t P_ = 2013265921ull;

typedef struct {
    const uint64_t* seeds;  // pinned host [jobs][w_data]: the record of job j starts at seeds + j * w_data
    uint32_t w_data;
    int calls;              // callbacks that returned 0 (atomic)
} witness_seam_input;

__device__ __forceinline__ uint64_t splitmix64(uint64_t z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// data[c][r] = splitmix64(seed[c] + r) mod p for r < rows; grid.y = column, consecutive threads on consecutive rows
__global__ void expand_kernel(uint32_t* data, const uint64_t* seeds, uint64_t n, uint64_t rows) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t c = blockIdx.y;
    if (r >= rows) return;
    data[(uint64_t)c * n + r] = (uint32_t)(splitmix64(seeds[c] + r) % P_);
}

extern "C" int seam_witgen(void* user, hfb200_ctx* ctx, const hfb200_witness_dev* w, size_t job) {
    witness_seam_input* in = (witness_seam_input*)user;
    if (!in || in->w_data != w->w_data) return 5;
    const size_t bytes = (size_t)w->w_data * sizeof(uint64_t);
    void* scratch = nullptr;
    const char* e = hfb200_segment_scratch(ctx, bytes, &scratch);
    if (e) { hfb200_free_error(e); return 3; }
    cudaStream_t st = (cudaStream_t)w->stream;
    if (cudaMemcpyAsync(scratch, in->seeds + job * w->w_data, bytes, cudaMemcpyHostToDevice, st) != cudaSuccess) return 2;
    const uint64_t n = 1ull << w->po2, rows = n - w->zk_rows;
    expand_kernel<<<dim3((unsigned)((rows + 255) / 256), w->w_data), 256, 0, st>>>(w->data, (const uint64_t*)scratch, n, rows);
    if (cudaGetLastError() != cudaSuccess) return 2;
    e = hfb200_segment_data_blind(ctx);
    if (e) { hfb200_free_error(e); return 4; }
    __atomic_fetch_add(&in->calls, 1, __ATOMIC_RELAXED);
    return 0;
}
