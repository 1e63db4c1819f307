// reset.cu — per-channel state reset (dspb_reset_channels): zeroes the state rows of a list of channels in every state buffer
// of the graph with one launch.  A scattered channel list would otherwise take one cudaMemset2DAsync per (buffer, contiguous
// run of channels): thousands of API calls to reset every channel of a chain, against one launch here.
#include <cuda_runtime.h>

#include <algorithm>

#include "plan.h"

namespace dspb {

namespace {

constexpr int kClearThreads = 256;

// Zeroes p[0, n) with the CTA's threads: scalar stores up to the first 16-byte boundary, float4 stores, a scalar tail.
__device__ void clear_span(float* p, long long n) {
    const long long head = min(n, (long long)((16 - ((uintptr_t)p & 15)) & 15) / 4);
    if (threadIdx.x < head) p[threadIdx.x] = 0.0f;
    p += head;
    n -= head;
    float4* q = reinterpret_cast<float4*>(p);
    const long long n4 = n / 4;
    for (long long i = threadIdx.x; i < n4; i += kClearThreads) q[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    if (threadIdx.x < n - 4 * n4) p[4 * n4 + threadIdx.x] = 0.0f;
}

// CTA (x, y) clears row channels[x] of buffer descs[y]: slots (first + i) mod ring, i in [0, len), as at most two spans.
__global__ void __launch_bounds__(kClearThreads)
clear_rows_kernel(const ClearDesc* __restrict__ descs, const int* __restrict__ channels) {
    const ClearDesc d = descs[blockIdx.y];
    float* row = d.base + (long long)channels[blockIdx.x] * d.pitch;
    const long long a = min(d.len, d.ring - d.first);
    clear_span(row + d.first, a);
    if (d.len > a) clear_span(row, d.len - a);
}

}  // namespace

int launch_clear_rows(const ClearDesc* descs, int n_descs, const int* channels, int n_channels, void* stream) {
    if (n_descs <= 0 || n_channels <= 0) return 0;
    for (int d = 0; d < n_descs; d += 65535)  // gridDim.y limit
        clear_rows_kernel<<<dim3((unsigned)n_channels, (unsigned)std::min(65535, n_descs - d)), kClearThreads, 0,
                            (cudaStream_t)stream>>>(descs + d, channels);
    return (int)cudaGetLastError();
}

}  // namespace dspb
