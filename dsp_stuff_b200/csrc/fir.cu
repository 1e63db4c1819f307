// fir.cu — FIR node (nodes/fir.rs:179-225) on the device.
//
// Two paths behind launch_fir():
//   FIR_DIRECT  time domain, f64 products and f64 sequential accumulation in exactly the reference's
//               order (oldest sample first, no FMA) -> bit-identical to `zip(state, taps).sum::<f64>()`.
//               8192 f64 flop per sample at 4096 taps: the parity-grade / cross-check path.
//   FIR_FFT     overlap-save FFT convolution in shared memory (fir_fft.cu): the throughput path.
//   FIR_TOEPLITZ  Toeplitz-tiled tcgen05 GEMM on split bf16 operands (fir_toeplitz.cu): the tensor-core comparison path.
// Both honour the reference's warm-up quirk: until N-1 samples have been seen the oldest sample pairs
// with taps[0] (a running prefix sum of x[i]*taps[i]), not zero-padded convolution.
#include <cuda_runtime.h>

#include <atomic>

#include "plan.h"

namespace dspb {

int launch_fir_fft(const FirPlan& fp, const float* U, int64_t u_stride, float* Y, int64_t y_stride, int c_begin, int c_end,
                   int64_t T, cudaStream_t st, int* n_launches);

int launch_fir_upc(const FirPlan& fp, const float* U, int64_t u_stride, float* Y, int64_t y_stride, int c_begin, int c_end, int64_t T,
                   cudaStream_t st, int* n_launches);

int launch_fir_toeplitz(const FirPlan& fp, const float* U, int64_t u_stride, float* Y, int64_t y_stride, int c_begin, int c_end,
                        int64_t T, cudaStream_t st, int* n_launches);

namespace {

constexpr int kDirectTile = 256;

// One thread per output sample; the CTA's input window lives in shared memory.
// PC: per-channel impulse responses, channel ch reads the reversed taps of its set, taps + set_index[ch] * N.
template <bool PC>
__global__ void __launch_bounds__(kDirectTile)
fir_direct_kernel(const float* __restrict__ U, long long u_stride, int hist_pad, int u_ring, int u_pos, float* __restrict__ Y, long long y_stride,
                  const double* __restrict__ taps, int N, long long T, long long started, float divisor, float post_nf,
                  int c_begin, long long n_begin, long long n_end, const int* __restrict__ set_index) {
    extern __shared__ float xw[];  // [kDirectTile + N - 1]
    const int ch = c_begin + blockIdx.y;
    if constexpr (PC) taps += (long long)set_index[ch] * N;
    const long long tile0 = n_begin + (long long)blockIdx.x * kDirectTile;
    const long long w0 = tile0 - (N - 1);  // call-relative index of xw[0]; >= -hist_pad
    const float* row = U + (long long)ch * u_stride;  // a ring of u_ring samples, call sample n at slot (u_pos + n) mod u_ring
    const int W = kDirectTile + N - 1;
    for (int i = threadIdx.x; i < W; i += kDirectTile) {
        const long long n = w0 + i;
        xw[i] = (n < T && n >= -(long long)hist_pad) ? row[ring_slot(u_pos, (int)n, u_ring)] : 0.0f;
    }
    __syncthreads();
    const long long n = tile0 + threadIdx.x;
    if (n >= n_end || n >= T) return;
    const long long a = started + n;  // samples seen before this one since reset
    double acc = 0.0;
    if (a >= N - 1) {  // full history: sum_i hist[i]*taps[i], hist[0] = x[n-N+1]
        const float* x = xw + threadIdx.x;
        for (int i = 0; i < N; i++) acc = __dadd_rn(acc, __dmul_rn((double)x[i], taps[i]));
    } else {  // warm-up: hist = x_abs[0..a]  (fir.rs:193-216)
        const float* x = xw + (threadIdx.x + (N - 1) - (int)a);  // x_abs[0]
        for (int i = 0; i <= (int)a; i++) acc = __dadd_rn(acc, __dmul_rn((double)x[i], taps[i]));
    }
    float y = __fmul_rn((float)acc, divisor);
    if (post_nf != 0.0f) y = __fdiv_rn(__fadd_rn(0.0f, y), post_nf);  // fused sink fan-in average (node.rs:162-194)
    Y[(long long)ch * y_stride + n] = y;
}

}  // namespace

int launch_fir_direct(const FirPlan& fp, const float* U, int64_t u_stride, float* Y, int64_t y_stride, int c_begin, int c_end,
                      int64_t T, int64_t started, int64_t n_begin, int64_t n_end, cudaStream_t st) {
    const int N = fp.n_taps;
    const size_t smem = (size_t)(kDirectTile + N - 1) * 4;
    const bool pc = fp.set_index != nullptr;
    auto kernel = pc ? fir_direct_kernel<true> : fir_direct_kernel<false>;
    // per device and instantiation: the opt-in is a per-device function attribute
    static std::atomic<size_t> configured_dev[kMaxDevices][2];
    std::atomic<size_t>& configured = configured_dev[current_device_slot()][pc];
    if (smem > 48 * 1024 && smem > configured.load(std::memory_order_acquire)) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return (int)e;
        configured.store(smem, std::memory_order_release);
    }
    if (n_end <= n_begin) return 0;
    const int C = c_end - c_begin;
    const long long tiles = (n_end - n_begin + kDirectTile - 1) / kDirectTile;
    for (int c = 0; c < C; c += 65535) {  // gridDim.y limit
        dim3 grid((unsigned)tiles, (unsigned)std::min(65535, C - c));
        kernel<<<grid, kDirectTile, smem, st>>>(U, u_stride, fp.hist_pad, fp.u_ring, fp.u_pos, Y, y_stride, fp.taps, N, T, started,
                                               fp.divisor, fp.post_nf, c_begin + c, n_begin, n_end, fp.set_index);
    }
    return (int)cudaGetLastError();
}

int launch_fir(const FirPlan& fp, const float* U, int64_t u_stride, float* Y, int64_t y_stride, int c_begin, int c_end,
               int64_t T, int64_t started, void* stream, int* n_launches) {
    cudaStream_t st = (cudaStream_t)stream;
    if (fp.mode == FIR_DIRECT) {
        if (n_launches) *n_launches += 1;
        return launch_fir_direct(fp, U, u_stride, Y, y_stride, c_begin, c_end, T, started, 0, T, st);
    }
    if (fp.mode == FIR_TOEPLITZ && fp.set_index) return (int)cudaErrorInvalidValue;  // shared taps only
    int rc = fp.mode == FIR_TOEPLITZ ? launch_fir_toeplitz(fp, U, u_stride, Y, y_stride, c_begin, c_end, T, st, n_launches)
             : (fp.mode == FIR_FFT && fp.upc_fdl) ? launch_fir_upc(fp, U, u_stride, Y, y_stride, c_begin, c_end, T, st, n_launches)
                                                  : launch_fir_fft(fp, U, u_stride, Y, y_stride, c_begin, c_end, T, st, n_launches);
    if (rc) return rc;
    // Samples that still belong to the warm-up are recomputed exactly by the direct kernel.
    const int64_t warm_end = (int64_t)fp.n_taps - 1 - started;  // call-relative
    if (warm_end > 0) {
        if (n_launches) *n_launches += 1;
        rc = launch_fir_direct(fp, U, u_stride, Y, y_stride, c_begin, c_end, T, started, 0, std::min<int64_t>(warm_end, T), st);
    }
    return rc;
}

}  // namespace dspb
