// The caller's step_accum of the stand-in circuit, outside libhfb200: terms data[chain_src(r)] + mix_r on the active rows,
// written by this file's kernel on the context's stream, then the library's scan and blinding rows.
#include <cuda_runtime.h>
#include "hfb200.h"

static const uint32_t P_ = 2013265921u;

__global__ void terms_kernel(uint32_t* accum, const uint32_t* data, const uint32_t* mix, uint32_t w_data, uint64_t n, uint64_t rows) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t r = blockIdx.y;
    if (i >= rows) return;
    uint32_t v = data[(uint64_t)((13 * r + 5) % w_data) * n + i] + mix[4 * r];
    if (v >= P_) v -= P_;
    accum[(uint64_t)(4 * r) * n + i] = v;
    for (int k = 1; k < 4; k++) accum[(uint64_t)(4 * r + k) * n + i] = mix[4 * r + k];
}

extern "C" int seam_accum(void* user, hfb200_ctx* ctx, const hfb200_segment_dev* seg, size_t job) {
    (void)job;
    const uint64_t n = 1ull << seg->po2, rows = n - seg->zk_rows;
    const uint32_t chains = seg->w_accum / 4;
    terms_kernel<<<dim3((unsigned)((rows + 255) / 256), chains), 256, 0, (cudaStream_t)seg->stream>>>(seg->accum, seg->data, seg->mix, seg->w_data, n, rows);
    if (cudaGetLastError() != cudaSuccess) return 2;
    const char* e = hfb200_segment_accum_scan(ctx, HFB200_SCAN_PRODUCT, 0, chains, rows);
    if (e) { hfb200_free_error(e); return 3; }
    e = hfb200_segment_accum_blind(ctx);
    if (e) { hfb200_free_error(e); return 4; }
    if (user) __atomic_fetch_add((int*)user, 1, __ATOMIC_RELAXED);
    return 0;
}
