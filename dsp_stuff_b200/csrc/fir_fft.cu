// fir_fft.cu — overlap-save FFT convolution for the Fir node (nodes/fir.rs:179-225), sm_100a.
//
// One 8192-point complex transform lives in (padded, bank-conflict-free) shared memory and carries TWO channels at
// once: z = xA + i*xB, Z = FFT(z), Y = Z .* H, y = IFFT(Y); because h is real, Re(y) = xA * h and Im(y) = xB * h.
// The transform is decimation-in-frequency with radices 8, 8, 8, 16 forward and the exact mirror (decimation-in-time,
// conjugate twiddles) backward, so the forward output order is irrelevant: H is produced ONCE per tap set by running the
// very same forward passes (in f64) on the zero-padded impulse response and is stored in that same order, pre-scaled.
// The last forward pass, the spectrum product and the first inverse pass happen in registers.  The first pass reads the
// input window straight from global memory and the last pass writes the valid outputs straight back.
//
// Segments.  An 8192-point window yields V13 = 8192 - (Ne-1) valid outputs -- half of it at 4096 taps; a 16384-point
// window yields V14 = 16384 - (Ne-1), three quarters.  segment_plan cuts a call into 16384-point ("double") segments,
// which fir_fft_wide_kernel runs, followed by 8192-point ("single") segments, which fir_fft_kernel runs.
//
// fir_fft_kernel is persistent (3 CTAs per SM, 256 threads): CTAs fetch work items (channel pair, segment) from an
// atomic counter in segment-major order within a pair, so the overlapping windows of neighbouring segments meet in L2.
// The input rows are rings (plan.h FirPlan::u_ring): a call's last N-1 samples are the next call's history in place.
//
// Accuracy: f32 butterflies, twiddles from an f64-computed table: ~2e-7 of the signal peak, inside the 1e-5 / -100 dBFS
// parity bar against the reference's f64 accumulation (tests/test_gpu_fir.py).
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <mutex>
#include <type_traits>
#include <utility>
#include <vector>

#include "plan.h"

namespace dspb {
namespace {

constexpr int kF = 8192;       // complex FFT size
constexpr int kLog2F = 13;
constexpr int kNT = 256;       // threads
constexpr int kPadded = kF + kF / 16;

template <typename T>
struct __align__(2 * sizeof(T)) C2 {
    T x, y;
};
__device__ __forceinline__ C2<double> operator+(C2<double> a, C2<double> b) { return {a.x + b.x, a.y + b.y}; }
__device__ __forceinline__ C2<double> operator-(C2<double> a, C2<double> b) { return {a.x - b.x, a.y - b.y}; }
// f32 complex add/sub.  Default: two scalar FADDs.  -DDSPB_FIR_FADD2 selects one packed add/sub.f32x2 instead (half the
// issue slots of two FADDs on paper): compiled both ways the kernel has 2320 (packed) vs 2368 (scalar) SASS
// instructions -- the packed form needs 256 MOVs to pair registers and blocks the mul+add -> FFMA contraction -- and
// the packed ops hold the FP32 pipe for two cycles each.  Measured on B200 (config 4, 4096 x 16384): 0.456 ms scalar
// vs 0.473 ms packed, so scalar is the default.
__device__ __forceinline__ unsigned long long pack2(C2<float> a) {
    return (unsigned long long)__float_as_uint(a.x) | ((unsigned long long)__float_as_uint(a.y) << 32);
}
__device__ __forceinline__ C2<float> unpack2(unsigned long long r) {
    return {__uint_as_float((unsigned)r), __uint_as_float((unsigned)(r >> 32))};
}
#ifdef DSPB_FIR_FADD2
__device__ __forceinline__ C2<float> operator+(C2<float> a, C2<float> b) {
    unsigned long long d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(pack2(a)), "l"(pack2(b)));
    return unpack2(d);
}
__device__ __forceinline__ C2<float> operator-(C2<float> a, C2<float> b) {
    unsigned long long d;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(pack2(a)), "l"(pack2(b)));
    return unpack2(d);
}
#else
__device__ __forceinline__ C2<float> operator+(C2<float> a, C2<float> b) { return {a.x + b.x, a.y + b.y}; }
__device__ __forceinline__ C2<float> operator-(C2<float> a, C2<float> b) { return {a.x - b.x, a.y - b.y}; }
#endif
template <typename T> __device__ __forceinline__ C2<T> cmul(C2<T> a, C2<T> w) { return {a.x * w.x - a.y * w.y, a.x * w.y + a.y * w.x}; }
template <typename T> __device__ __forceinline__ C2<T> cmulc(C2<T> a, C2<T> w) { return {a.x * w.x + a.y * w.y, a.y * w.x - a.x * w.y}; }  // a * conj(w)

template <int N, class Fn, int... I>
__device__ __forceinline__ void static_for_impl(Fn&& f, std::integer_sequence<int, I...>) {
    (f(std::integral_constant<int, I>{}), ...);
}
template <int N, class Fn>
__device__ __forceinline__ void static_for(Fn&& f) {
    static_for_impl<N>(static_cast<Fn&&>(f), std::make_integer_sequence<int, N>{});
}

// cos / sin of 2 pi m / 32 as compile-time constants
__host__ __device__ constexpr double cos32(int m) {
    constexpr double tab[9] = {1.0, 0.98078528040323044913, 0.92387953251128675613, 0.83146961230254523708, 0.70710678118654752440,
                               0.55557023301960222474, 0.38268343236508977173, 0.19509032201612826785, 0.0};
    m = ((m % 32) + 32) % 32;
    if (m > 16) m = 32 - m;
    return m > 8 ? -tab[16 - m] : tab[m];
}
__host__ __device__ constexpr double sin32(int m) { return cos32(m - 8); }

// a * w_SZ^I  (forward: w = exp(-2 pi i / SZ); INV: conjugate), I < SZ/2, SZ in {2,4,8,16,32}
template <int SZ, int I, bool INV, typename T>
__device__ __forceinline__ C2<T> tw(C2<T> a) {
    if constexpr (I == 0) {
        return a;
    } else if constexpr (4 * I == SZ) {
        if constexpr (INV) return {-a.y, a.x};
        else return {a.y, -a.x};
    } else if constexpr (8 * I == SZ) {
        const T h = T(0.70710678118654752440);
        if constexpr (INV) return {(a.x - a.y) * h, (a.x + a.y) * h};
        else return {(a.x + a.y) * h, (a.y - a.x) * h};
    } else if constexpr (8 * I == 3 * SZ) {
        const T h = T(0.70710678118654752440);
        if constexpr (INV) return {-(a.x + a.y) * h, (a.x - a.y) * h};
        else return {(a.y - a.x) * h, -(a.x + a.y) * h};
    } else {
        static_assert(SZ == 16 || SZ == 32, "generic twiddles are tabulated for SZ = 16 and 32");
        const T c = T(cos32(I * (32 / SZ))), s = T(sin32(I * (32 / SZ)));
        if constexpr (INV) return {a.x * c - a.y * s, a.y * c + a.x * s};
        else return {a.x * c + a.y * s, a.y * c - a.x * s};
    }
}

// in-register radix-2 decimation-in-frequency DFT of R points: natural in, bit-reversed out
template <int R, typename T>
__device__ __forceinline__ void fft_dif(C2<T> (&v)[R]) {
    static_for<5>([&](auto st) {
        constexpr int sz = R >> decltype(st)::value;
        if constexpr (sz >= 2) {
            constexpr int half = sz / 2;
            static_for<R / sz>([&](auto bk) {
                static_for<half>([&](auto ii) {
                    constexpr int i = decltype(ii)::value, o = decltype(bk)::value * sz;
                    const C2<T> a = v[o + i], b = v[o + i + half];
                    v[o + i] = a + b;
                    v[o + i + half] = tw<sz, i, false, T>(a - b);
                });
            });
        }
    });
}
// exact mirror: bit-reversed in, natural out, conjugate twiddles, unnormalised (gain R)
template <int R, typename T>
__device__ __forceinline__ void ifft_dit(C2<T> (&v)[R]) {
    static_for<5>([&](auto st) {
        constexpr int sz = 2 << decltype(st)::value;
        if constexpr (sz <= R) {
            constexpr int half = sz / 2;
            static_for<R / sz>([&](auto bk) {
                static_for<half>([&](auto ii) {
                    constexpr int i = decltype(ii)::value, o = decltype(bk)::value * sz;
                    const C2<T> a = v[o + i], b = tw<sz, i, true, T>(v[o + i + half]);
                    v[o + i] = a + b;
                    v[o + i + half] = a - b;
                });
            });
        }
    });
}

__host__ __device__ constexpr int bitrev3(int s) { return ((s & 1) << 2) | (s & 2) | ((s >> 2) & 1); }
__host__ __device__ constexpr int bitrev4(int s) { return ((s & 1) << 3) | ((s & 2) << 1) | ((s & 4) >> 1) | ((s >> 3) & 1); }
__host__ __device__ constexpr int bitrev5(int s) { return ((s & 1) << 4) | ((s & 2) << 2) | (s & 4) | ((s & 8) >> 2) | ((s >> 4) & 1); }
__device__ __forceinline__ int pad(int p) { return p + (p >> 4); }

// Twiddle source.  W16384^n = coarse[n >> 5] * fine[n & 31] with coarse[m] = exp(-2 pi i m / 512) (512 entries) and
// fine[b] = exp(-2 pi i b / 16384) (32 entries): 4.3 KB of shared memory instead of an L2-resident table.  The
// 8192-point passes index in units of W8192 = W16384^2: W8192^k = coarse[k >> 4] * fine[2 (k & 15)].
constexpr int kCoarse = kF / 16, kFine = 32, kT128 = 7 * 16;
constexpr int kTwEntries = kCoarse + kFine + kT128;
template <typename T>
struct Tw {
    const C2<T>* coarse;  // [512] exp(-2 pi i m / 512)
    const C2<T>* fine;    // [32]  exp(-2 pi i b / 16384)
    const C2<T>* t128;    // [7][16] W128^(j q), q = 1..7 major: the twiddles of the M = 128 pass, one conflict-free LDS.64
                          // per value (picked out of `coarse` their 16 addresses are 32 / 64 / 128 bytes apart: up to
                          // 16-way bank conflicts, 42 % excess wavefronts on that pass -- ncu, profiles/r02_*)
    __device__ __forceinline__ C2<T> at(int k) const {   // W8192^k
        k &= kF - 1;
        const C2<T> c = coarse[k >> 4];
        if ((k & 15) == 0) return c;
        return cmul(c, fine[2 * (k & 15)]);
    }
    __device__ __forceinline__ C2<T> at2(int n) const {  // W16384^n
        n &= 2 * kF - 1;
        const C2<T> c = coarse[n >> 5];
        if ((n & 31) == 0) return c;
        return cmul(c, fine[n & 31]);
    }
};
// twiddles w^q, q = 1..7, from three look-ups (w, w^2, w^4) and four products.  STEP = F/M: every index is
// a multiple of STEP, so look-ups whose index is a multiple of 16 need no fine factor.
template <int STEP, typename T>
__device__ __forceinline__ void twiddles8(const Tw<T>& W, int k1, C2<T> (&w)[8]) {
    if constexpr (STEP % 16 == 0) {
        w[1] = W.coarse[(k1 >> 4) & (kCoarse - 1)];
        w[2] = W.coarse[(k1 >> 3) & (kCoarse - 1)];
        w[4] = W.coarse[(k1 >> 2) & (kCoarse - 1)];
    } else if constexpr (STEP % 8 == 0) {
        w[1] = W.at(k1);
        w[2] = W.coarse[(k1 >> 3) & (kCoarse - 1)];
        w[4] = W.coarse[(k1 >> 2) & (kCoarse - 1)];
    } else {
        w[1] = W.at(k1);
        w[2] = W.at(2 * k1);
        w[4] = W.at(4 * k1);
    }
    w[3] = cmul(w[1], w[2]);
    w[5] = cmul(w[1], w[4]);
    w[6] = cmul(w[2], w[4]);
    w[7] = cmul(w[3], w[4]);
}
template <typename T, typename TG>
__device__ __forceinline__ Tw<T> load_tables(C2<T>* sm, const TG* __restrict__ Wg, int t) {
    // sm: [512 + 32]; Wg: the compact table in global memory, same layout
    for (int i = t; i < kCoarse + kFine; i += kNT) sm[i] = C2<T>{(T)Wg[i].x, (T)Wg[i].y};
    if (t < kT128) {  // W128^(j q) = W512^(4 j q): exact table entries
        const int q = t / 16 + 1, j = t % 16;
        const TG w = Wg[(4 * j * q) & (kCoarse - 1)];
        sm[kCoarse + kFine + t] = C2<T>{(T)w.x, (T)w.y};
    }
    return Tw<T>{sm, sm + kCoarse, sm + kCoarse + kFine};
}

// forward radix-8 pass on the shared array: sub-transform size M, L = M/8.  Butterfly u = t + 256 k of
// thread t has j = u % L; for L <= 256 that is the same for every k, so the twiddles are loop-invariant.
template <int M, typename T>
__device__ __forceinline__ void fwd_pass8(C2<T>* a, const Tw<T>& W, int t) {
    constexpr int L = M / 8;
    static_assert(L % 16 == 0, "constant padded stride needs L % 16 == 0");
    constexpr int LP = L + L / 16;  // pad(base + r*L) == pad(base) + r*LP
    constexpr bool kInvariant = (kNT % L) == 0;
    C2<T> w[8];
    if constexpr (M == 128) {
#pragma unroll
        for (int q = 1; q < 8; q++) w[q] = W.t128[(q - 1) * 16 + (t % L)];
    } else if constexpr (kInvariant) twiddles8<kF / M>(W, (t % L) * (kF / M), w);
#pragma unroll 1
    for (int k = 0; k < kF / 8 / kNT; k++) {
        const int u = t + kNT * k, b = u / L, j = u % L, base = b * M + j;
        C2<T>* p = a + pad(base);
        C2<T> v[8];
#pragma unroll
        for (int r = 0; r < 8; r++) v[r] = p[r * LP];
        if constexpr (!kInvariant) twiddles8<kF / M>(W, j * (kF / M), w);
        fft_dif<8>(v);
        p[0] = v[0];
#pragma unroll
        for (int s = 1; s < 8; s++) p[bitrev3(s) * LP] = cmul(v[s], w[bitrev3(s)]);
    }
}
template <int M, typename T>
__device__ __forceinline__ void inv_pass8(C2<T>* a, const Tw<T>& W, int t) {
    constexpr int L = M / 8;
    constexpr int LP = L + L / 16;
    constexpr bool kInvariant = (kNT % L) == 0;
    C2<T> w[8];
    if constexpr (M == 128) {
#pragma unroll
        for (int q = 1; q < 8; q++) w[q] = W.t128[(q - 1) * 16 + (t % L)];
    } else if constexpr (kInvariant) twiddles8<kF / M>(W, (t % L) * (kF / M), w);
#pragma unroll 1
    for (int k = 0; k < kF / 8 / kNT; k++) {
        const int u = t + kNT * k, b = u / L, j = u % L, base = b * M + j;
        C2<T>* p = a + pad(base);
        C2<T> v[8];
        if constexpr (!kInvariant) twiddles8<kF / M>(W, j * (kF / M), w);
        v[0] = p[0];
#pragma unroll
        for (int s = 1; s < 8; s++) v[s] = cmulc(p[bitrev3(s) * LP], w[bitrev3(s)]);
        ifft_dit<8>(v);
#pragma unroll
        for (int r = 0; r < 8; r++) p[r * LP] = v[r];
    }
}

// ---- the convolution kernel --------------------------------------------------------------------------
// hist = Ne - 1, Ne = effective tap count: N padded with zero taps so that hist is a multiple of 4.  Then every window
// start (s0 - hist, s0 a multiple of the valid length) and every output run is 16-byte aligned and the first / last pass
// move two consecutive samples per 64-bit access.
// post: optional epilogue "acc = 0.0 + y; acc /= post_nf" = the fan-in average of a sink fed only by this node
// (node.rs:162-194, nodes/output.rs:223), so no separate kernel has to touch the output again.
// (0.0 + y) / nf uses Markstein's three-instruction sequence (exact_math.cuh: correctly rounded except in the denormal /
// overflow fringes, where it is one ulp off -- far inside this path's 1e-5 tolerance, and this path is never bit-exact
// anyway: the warm-up samples that ARE bit-exact come from fir_direct_kernel, which divides with __fdiv_rn).
__device__ __forceinline__ float div_nf(float y, float nf, float rnf) {
    const float a = __fadd_rn(0.0f, y);
    const float q0 = __fmul_rn(a, rnf);
    return __fmaf_rn(__fmaf_rn(-q0, nf, a), rnf, q0);
}

struct FftArgs {
    const float* U;        // [C x u_stride] input rings
    long long u_stride;
    int u_ring, u_pos;     // call sample i lives at slot (u_pos + i) mod u_ring
    int hist;              // Ne - 1: window samples in front of a segment's first output (multiple of 4, <= 4096)
    float* Y;
    long long y_stride;
    const float2* H13;     // spectrum of h for an 8192-point segment, transform order, scaled 1/8192
    const float2* Wg;      // compact twiddle table [512 + 32]
    long long T;
    float divisor, post_nf;
    int c_begin, c_end;
    int n13;               // single segments per channel pair (V13 outputs each)
    long long single_base; // first output sample of the single segments (= the wide kernel's double segments * V14)
    int n_items;           // pairs * n13
    unsigned* work;        // [0] next item, [1] CTAs done  (slots 2 / 3 belong to the wide kernel on the same lane)
    // per-channel impulse responses only (template PC = true): a "pair" is an entry of the transform table, whose set k
    // reads its spectrum at H13 + k * h_stride
    const int4* xf;        // this launch's slice of the transform table {chA, chB or -1, set, 0}
    long long h_stride;    // float2 elements per set
};

// FAST (CTA-uniform): the whole window lies inside this call's samples and does not wrap around the ring, and
// hist == 4096, so no load is predicated and the valid outputs are exactly the butterfly outputs r >= 4.
template <bool FAST>
__device__ __forceinline__ void fwd_pass1(C2<float>* a, const Tw<float>& W, const float* __restrict__ rowA, const float* __restrict__ rowB,
                                          int wb, int R, int lim, int t) {
    constexpr int L = kF / 8, LP = L + L / 16;
    auto load2 = [&](int n, float2& xa, float2& xb) {
        if constexpr (FAST) {
            xa = __ldg(reinterpret_cast<const float2*>(rowA + wb + n));
            xb = __ldg(reinterpret_cast<const float2*>(rowB + wb + n));
        } else {
            xa = make_float2(0.f, 0.f);
            xb = make_float2(0.f, 0.f);
            if (n < lim) {  // lim and n are even: the pair is inside or outside together; n < lim <= R: one wrap at most
                int sl = wb + n;
                if (sl >= R) sl -= R;
                xa = __ldg(reinterpret_cast<const float2*>(rowA + sl));
                xb = __ldg(reinterpret_cast<const float2*>(rowB + sl));
            }
        }
    };
#pragma unroll 1
    for (int k = 0; k < kF / 8 / kNT / 2; k++) {
        const int j = 2 * (t + kNT * k);
        C2<float> v0[8], v1[8], w[8];
        static_for<8>([&](auto rr) {
            constexpr int r = decltype(rr)::value;
            float2 xa, xb;
            load2(j + r * L, xa, xb);
            v0[r] = C2<float>{xa.x, xb.x};
            v1[r] = C2<float>{xa.y, xb.y};
        });
        C2<float>* p = a + pad(j);  // j is even: j and j + 1 share the padding offset
        twiddles8<1>(W, j, w);
        fft_dif<8>(v0);
        p[0] = v0[0];
#pragma unroll
        for (int s = 1; s < 8; s++) p[bitrev3(s) * LP] = cmul(v0[s], w[bitrev3(s)]);
        twiddles8<1>(W, j + 1, w);
        fft_dif<8>(v1);
        p[1] = v1[0];
#pragma unroll
        for (int s = 1; s < 8; s++) p[1 + bitrev3(s) * LP] = cmul(v1[s], w[bitrev3(s)]);
    }
}

// forward pass 4 (radix 16, no twiddles) . spectrum product . inverse pass 4, all in registers
__device__ __forceinline__ void mid_pass16(C2<float>* a, const C2<float>* __restrict__ H, int t) {
#pragma unroll 1
    for (int k = 0; k < kF / 16 / kNT; k++) {
        const int u = t + kNT * k, base = 16 * u;
        C2<float> v[16];
        float4 h[8];
        // H is stored [k][s / 2][thread] (float4 = two consecutive bins): every request of a warp is one
        // contiguous 512-byte run.  (In natural order each thread owns a 128-byte line: 32 lines per request,
        // which alone kept the L1 data pipe 84 % busy -- ncu l1tex__data_pipe_lsu_wavefronts.)
        const float4* h4 = reinterpret_cast<const float4*>(H) + (k * 8) * kNT + t;
#pragma unroll
        for (int s = 0; s < 8; s++) h[s] = __ldg(h4 + s * kNT);
#pragma unroll
        for (int s = 0; s < 16; s++) v[s] = a[pad(base) + s];
        fft_dif<16>(v);
#pragma unroll
        for (int s = 0; s < 16; s += 2) {
            v[s] = cmul(v[s], C2<float>{h[s / 2].x, h[s / 2].y});
            v[s + 1] = cmul(v[s + 1], C2<float>{h[s / 2].z, h[s / 2].w});
        }
        ifft_dit<16>(v);
#pragma unroll
        for (int s = 0; s < 16; s++) a[pad(base) + s] = v[s];
    }
}

template <bool FAST>
__device__ __forceinline__ void inv_pass1(const C2<float>* a, const Tw<float>& W, float* __restrict__ outA, float* __restrict__ outB,
                                          bool hasB, int hist, int lim, float divisor, float post_nf, int t) {
    constexpr int L = kF / 8, LP = L + L / 16;
    // Epilogue: `* divisor` (fir.rs:187-190, 222) and the fused sink average `(0.0 + y) / nf` collapse into ONE multiplication by
    // divisor / nf (formed in f64 on the host side of this expression, rounded once).  Against the two separately rounded
    // operations that is at most two ulps (1.2e-7) on a path whose transform error is 2-3e-7 and whose bar is 1e-5; the
    // bit-exact samples of this node (warm-up, fir_mode = 1) come from fir_direct_kernel, which keeps the exact division.
    const float scale = post_nf != 0.0f ? (float)((double)divisor / (double)post_nf) : divisor;
    const bool unit = scale == 1.0f;
    auto fin = [&](float y) { return unit ? y : __fmul_rn(y, scale); };
    auto store2 = [&](int n, float a0, float a1, float b0, float b1) {  // samples n, n + 1 of both channels
        *reinterpret_cast<float2*>(outA + n) = make_float2(fin(a0), fin(a1));
        if (hasB) *reinterpret_cast<float2*>(outB + n) = make_float2(fin(b0), fin(b1));
    };
#pragma unroll 1
    for (int k = 0; k < kF / 8 / kNT / 2; k++) {
        const int j = 2 * (t + kNT * k);
        C2<float> v0[8], v1[8], w[8];
        const C2<float>* p = a + pad(j);
        twiddles8<1>(W, j, w);
        v0[0] = p[0];
#pragma unroll
        for (int s = 1; s < 8; s++) v0[s] = cmulc(p[bitrev3(s) * LP], w[bitrev3(s)]);
        ifft_dit<8>(v0);
        twiddles8<1>(W, j + 1, w);
        v1[0] = p[1];
#pragma unroll
        for (int s = 1; s < 8; s++) v1[s] = cmulc(p[1 + bitrev3(s) * LP], w[bitrev3(s)]);
        ifft_dit<8>(v1);
        static_for<8>([&](auto rr) {
            constexpr int r = decltype(rr)::value;
            const int n = j + r * L;
            if (FAST ? r >= 4 : (n >= hist && n < lim)) store2(n, v0[r].x, v1[r].x, v0[r].y, v1[r].y);
        });
    }
}

// PC: the spectrum of tap set `set` (per-channel impulse responses); otherwise `set` is unused
template <bool FAST, bool PC>
__device__ __forceinline__ void transform(C2<float>* a, const Tw<float>& W, const FftArgs& g, int set, const float* rowA,
                                          const float* rowB, float* outA, float* outB, bool hasB, int wb, int lim, int t) {
    fwd_pass1<FAST>(a, W, rowA, rowB, wb, g.u_ring, lim, t);
    __syncthreads();
    fwd_pass8<kF / 8>(a, W, t);
    __syncthreads();
    fwd_pass8<kF / 64>(a, W, t);
    __syncthreads();
    mid_pass16(a, reinterpret_cast<const C2<float>*>(PC ? g.H13 + set * g.h_stride : g.H13), t);
    __syncthreads();
    inv_pass8<kF / 64>(a, W, t);
    __syncthreads();
    inv_pass8<kF / 8>(a, W, t);
    __syncthreads();
    inv_pass1<FAST>(a, W, outA, outB, hasB, g.hist, lim, g.divisor, g.post_nf, t);
}

// PC: per-channel impulse responses (see FftArgs::xf); PC = false is the shared-taps kernel.
template <bool PC>
__global__ void __launch_bounds__(kNT, 3)
fir_fft_kernel(const __grid_constant__ FftArgs g) {
    extern __shared__ float2 smem_f2[];
    __shared__ int s_item;
    C2<float>* a = reinterpret_cast<C2<float>*>(smem_f2);
    const int t = threadIdx.x;
    const Tw<float> W = load_tables<float>(a + kPadded, g.Wg, t);
    const int V13 = kF - g.hist;
    for (;;) {
        __syncthreads();  // the previous item's last pass has read the shared array (and s_item); tables visible
        if (t == 0) s_item = (int)atomicAdd(g.work, 1u);
        __syncthreads();
        const int item = s_item;
        if (item >= g.n_items) break;
        const int pr = item / g.n13, sg = item - pr * g.n13;
        const int4 x = PC ? g.xf[pr] : int4{};   // per-channel taps: {chA, chB or -1, set} of transform pr
        const int chA = PC ? x.x : g.c_begin + 2 * pr, chB = PC ? x.y : chA + 1;
        const bool hasB = PC ? chB >= 0 : chB < g.c_end;
        const long long s0 = g.single_base + (long long)sg * V13;
        const long long w0 = s0 - g.hist;                      // call-relative index of window sample 0 (>= -hist)
        const long long lim_ll = g.T - w0;                     // window samples >= lim lie beyond this call's input: zeros
        const int lim = lim_ll > kF ? kF : (int)lim_ll;
        const int wb = ring_slot(g.u_pos, (int)w0, g.u_ring);  // ring slot of window sample 0
        const float* rowA = g.U + (long long)chA * g.u_stride;
        const float* rowB = g.U + (long long)(hasB ? chB : chA) * g.u_stride;  // odd channel count: B mirrors A, never stored
        float* outA = g.Y + (long long)chA * g.y_stride + w0;
        float* outB = g.Y + (long long)(hasB ? chB : chA) * g.y_stride + w0;
        if (g.hist == kF / 2 && lim == kF && wb + kF <= g.u_ring)
            transform<true, PC>(a, W, g, x.z, rowA, rowB, outA, outB, hasB, wb, lim, t);
        else
            transform<false, PC>(a, W, g, x.z, rowA, rowB, outA, outB, hasB, wb, lim, t);
    }
    // the last CTA out re-arms the work counter for the next launch on this lane (stream-ordered behind this one)
    if (t == 0) {
        __threadfence();
        if (atomicAdd(g.work + 1, 1u) == gridDim.x - 1) {
            g.work[0] = 0;
            g.work[1] = 0;
        }
    }
}

// ======================= 16384-point segments in one piece ("wide" kernel) =======================
// A double segment run as two 8192-point sub-transforms (after one radix-2 step) costs 2.9 single segments (measured):
// each sub-transform has all six shared-memory round trips of the pipeline above, which is what bounds it (ncu: l1tex
// data pipe 69 % busy, 79 % of it shared memory).  This kernel keeps a whole 16384-point transform of a channel pair in
// shared memory (139 KB, one 512-thread CTA per SM, 128 registers per thread) with radices 16 . 32 . 32: FOUR
// shared-memory round trips per transform instead of six, on 16384 points that yield 12288 outputs per channel instead of
// 8192 points that yield 4096.
//   pass 1   global -> radix 16 over stride 1024 -> twiddle W16384^(j k) -> shared
//   pass 2   radix 32 over stride 32 inside each 1024-block -> twiddle W1024^(j k) (table in shared memory) -> shared
//   middle   radix 32 over 32 contiguous points . spectrum product . inverse radix 32, in registers
//   pass 2', pass 1' mirror images; pass 1' writes the 12288 valid outputs of both channels to global memory
// Output position p = k1 * 1024 + k2 * 32 + s holds bin f = k1 + 16 k2 + 512 bitrev5(s); the spectrum table is computed
// directly in that order (fir_spectrum_wide_kernel).  Layout: p + 2 (p >> 5): every access pattern above is
// conflict-free (the middle pass moves two complex values per 128-bit access).  Persistent: one CTA per SM fetches
// (channel pair, segment) items from an atomic counter and prefetches the next item's window into L2 while it computes.
constexpr int kN2 = 2 * kF;                 // 16384
constexpr int kNTW = 512;                   // threads
constexpr int kPadW = kN2 + kN2 / 16;       // 17408 complex
constexpr int kT2 = 31 * 32;                // W1024^(j k), k = 1..31 major, j < 32
constexpr int kTwW = kCoarse + kFine + kT2; // table entries in shared memory
__device__ __forceinline__ int padw(int p) { return p + ((p >> 5) << 1); }

struct WideArgs {
    const float* U;
    long long u_stride;
    int u_ring, u_pos, hist;
    float* Y;
    long long y_stride;
    const float4* Hw;      // [16][8192] float4: (H[32 u + 2 q], H[32 u + 2 q + 1]) at [q * 512 ... ] per 512-thread round, see mid pass
    const float2* Wg;      // compact twiddle table [512 + 32] followed by the W1024 table [31 * 32]
    float divisor, post_nf;
    int c_begin, c_end;
    int n14;               // double segments per channel pair (all lie fully inside the call)
    int n_items;           // pairs * n14
    unsigned* work;        // [2] next item, [3] CTAs done  (slots 0 / 1 belong to fir_fft_kernel on the same lane)
    const int4* xf;        // PC = true: transform table slice, set k's table at Hw + k * h_stride / 2 (see FftArgs)
    long long h_stride;
};

template <bool PC>
__global__ void __launch_bounds__(kNTW, 1)
fir_fft_wide_kernel(const __grid_constant__ WideArgs g) {
    extern __shared__ float2 smem_f2[];
    __shared__ int s_item[2];
    C2<float>* a = reinterpret_cast<C2<float>*>(smem_f2);
    C2<float>* tabs = a + kPadW;
    const int t = threadIdx.x;
    for (int i = t; i < kTwW; i += kNTW) tabs[i] = C2<float>{g.Wg[i].x, g.Wg[i].y};
    const Tw<float> W{tabs, tabs + kCoarse, nullptr};
    const C2<float>* T2 = tabs + kCoarse + kFine;   // [(k - 1) * 32 + j]
    const int V14 = kN2 - g.hist;
    // one multiplication by divisor / nf instead of `* divisor` and the sink's `(0.0 + y) / nf` (see inv_pass1)
    const float scale = g.post_nf != 0.0f ? (float)((double)g.divisor / (double)g.post_nf) : g.divisor;
    const bool unit = scale == 1.0f;
    auto fin = [&](float y) { return unit ? y : __fmul_rn(y, scale); };
    if (t == 0) s_item[0] = (int)atomicAdd(g.work + 2, 1u);
    __syncthreads();
    for (int it = 0;; it++) {
        const int item = s_item[it & 1];
        if (item >= g.n_items) break;
        if (t == 0) s_item[(it + 1) & 1] = (int)atomicAdd(g.work + 2, 1u);  // the next item: known one item ahead (L2 prefetch)
        const int pr = item / g.n14, sg = item - pr * g.n14;
        const int4 x = PC ? g.xf[pr] : int4{};   // per-channel taps: {chA, chB or -1, set} of transform pr
        const int chA = PC ? x.x : g.c_begin + 2 * pr, chB = PC ? x.y : chA + 1;
        const bool hasB = PC ? chB >= 0 : chB < g.c_end;
        const long long w0 = (long long)sg * V14 - g.hist;          // call-relative index of window sample 0
        const int wb = ring_slot(g.u_pos, (int)w0, g.u_ring);       // its ring slot; the window holds kN2 <= u_ring samples
        const float* rowA = g.U + (long long)chA * g.u_stride;
        const float* rowB = g.U + (long long)(hasB ? chB : chA) * g.u_stride;
        const bool nowrap = wb + kN2 <= g.u_ring;

        // ---- pass 1: global -> radix 16 -> shared
#pragma unroll 1
        for (int k = 0; k < 2; k++) {
            const int j = t + kNTW * k;
            C2<float> v[16];
            if (nowrap) {
                const float* pa = rowA + wb + j;
                const float* pb = rowB + wb + j;
#pragma unroll
                for (int r = 0; r < 16; r++) v[r] = C2<float>{__ldg(pa + r * 1024), __ldg(pb + r * 1024)};
            } else {
#pragma unroll
                for (int r = 0; r < 16; r++) {
                    int sl = wb + j + r * 1024;
                    if (sl >= g.u_ring) sl -= g.u_ring;
                    v[r] = C2<float>{__ldg(rowA + sl), __ldg(rowB + sl)};
                }
            }
            fft_dif<16>(v);
            // twiddles W16384^(j q): w1, w2, w4, w8 from the table, the rest by products
            C2<float> w[16];
            w[1] = W.at2(j); w[2] = W.at2(2 * j); w[4] = W.at2(4 * j); w[8] = W.at2(8 * j);
            w[3] = cmul(w[1], w[2]); w[5] = cmul(w[1], w[4]); w[6] = cmul(w[2], w[4]); w[7] = cmul(w[3], w[4]);
#pragma unroll
            for (int q = 9; q < 16; q++) w[q] = cmul(w[q - 8], w[8]);
            C2<float>* p = a + padw(j);   // padw(j + 1024 q) = padw(j) + 1088 q
            p[0] = v[0];
#pragma unroll
            for (int s = 1; s < 16; s++) p[bitrev4(s) * 1088] = cmul(v[s], w[bitrev4(s)]);
        }
        __syncthreads();
        // L2 prefetch of the next item's window (the counter was fetched one item ahead)
        {
            const int nxt = s_item[(it + 1) & 1];
            if (nxt < g.n_items) {
                const int npr = nxt / g.n14, nsg = nxt - npr * g.n14;
                const int4 nx = PC ? g.xf[npr] : int4{};   // per-channel taps: the next item's table entry
                const int nA = PC ? nx.x : g.c_begin + 2 * npr;
                const int nwb = ring_slot(g.u_pos, (int)((long long)nsg * V14 - g.hist), g.u_ring);
                // 2 rows x 16384 floats = 1024 lines of 128 bytes: two per thread
                const int line = t & 511;
                int sl = nwb + line * 32;
                if (sl >= g.u_ring) sl -= g.u_ring;
                const float* q0 = g.U + (long long)nA * g.u_stride + sl;
                const float* q1 = g.U + (long long)(PC ? (nx.y >= 0 ? nx.y : nA) : (nA + 1 < g.c_end ? nA + 1 : nA)) * g.u_stride + sl;
                asm volatile("prefetch.global.L2 [%0];" ::"l"(q0));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(q1));
            }
        }
        // ---- pass 2: radix 32 over stride 32 inside each 1024-block
        {
            const int b = t >> 5, j = t & 31;
            C2<float>* p = a + padw(b * 1024 + j);   // padw(base + 32 r) = padw(base) + 34 r
            C2<float> v[32];
#pragma unroll
            for (int r = 0; r < 32; r++) v[r] = p[r * 34];
            fft_dif<32>(v);
            p[0] = v[0];
#pragma unroll
            for (int s = 1; s < 32; s++) p[bitrev5(s) * 34] = cmul(v[s], T2[(bitrev5(s) - 1) * 32 + j]);
        }
        // Pass 2, the middle pass and pass 2' of 1024-block b all run on warp b (threads 32 b .. 32 b + 31 own both the
        // butterflies b * 1024 + j + 32 r and the points 32 t .. 32 t + 31 of that block): warp-level synchronisation is
        // enough, so the 16 warps drift apart over three quarters of the item instead of marching in lockstep.
        __syncwarp();
        // ---- middle: radix 32 on contiguous points . spectrum . inverse radix 32
        {
            float4* p4 = reinterpret_cast<float4*>(a + padw(32 * t));   // 32 contiguous points, no pad inside, 16-byte aligned
            const float4* h4 = (PC ? g.Hw + x.z * (g.h_stride / 2) : g.Hw) + t;
            C2<float> v[32];
#pragma unroll
            for (int q = 0; q < 16; q++) {
                const float4 x = p4[q];
                v[2 * q] = C2<float>{x.x, x.y};
                v[2 * q + 1] = C2<float>{x.z, x.w};
            }
            fft_dif<32>(v);
#pragma unroll
            for (int q = 0; q < 16; q++) {
                const float4 h = __ldg(h4 + q * kNTW);
                v[2 * q] = cmul(v[2 * q], C2<float>{h.x, h.y});
                v[2 * q + 1] = cmul(v[2 * q + 1], C2<float>{h.z, h.w});
            }
            ifft_dit<32>(v);
#pragma unroll
            for (int q = 0; q < 16; q++) p4[q] = make_float4(v[2 * q].x, v[2 * q].y, v[2 * q + 1].x, v[2 * q + 1].y);
        }
        __syncwarp();
        // ---- pass 2': inverse radix 32 over stride 32
        {
            const int b = t >> 5, j = t & 31;
            C2<float>* p = a + padw(b * 1024 + j);
            C2<float> v[32];
            v[0] = p[0];
#pragma unroll
            for (int s = 1; s < 32; s++) v[s] = cmulc(p[bitrev5(s) * 34], T2[(bitrev5(s) - 1) * 32 + j]);
            ifft_dit<32>(v);
#pragma unroll
            for (int r = 0; r < 32; r++) p[r * 34] = v[r];
        }
        __syncthreads();
        // ---- pass 1': inverse radix 16 over stride 1024 -> the valid outputs (window index >= hist) to global memory
        {
            float* outA = g.Y + (long long)chA * g.y_stride + w0;
            float* outB = g.Y + (long long)(hasB ? chB : chA) * g.y_stride + w0;
#pragma unroll 1
            for (int k = 0; k < 2; k++) {
                const int j = t + kNTW * k;
                C2<float> w[16];
                w[1] = W.at2(j); w[2] = W.at2(2 * j); w[4] = W.at2(4 * j); w[8] = W.at2(8 * j);
                w[3] = cmul(w[1], w[2]); w[5] = cmul(w[1], w[4]); w[6] = cmul(w[2], w[4]); w[7] = cmul(w[3], w[4]);
#pragma unroll
                for (int q = 9; q < 16; q++) w[q] = cmul(w[q - 8], w[8]);
                const C2<float>* p = a + padw(j);
                C2<float> v[16];
                v[0] = p[0];
#pragma unroll
                for (int s = 1; s < 16; s++) v[s] = cmulc(p[bitrev4(s) * 1088], w[bitrev4(s)]);
                ifft_dit<16>(v);
#pragma unroll
                for (int r = 0; r < 16; r++) {
                    const int n = j + r * 1024;
                    if (n >= g.hist) {
                        outA[n] = fin(v[r].x);
                        if (hasB) outB[n] = fin(v[r].y);
                    }
                }
            }
        }
        __syncthreads();  // the shared array (and s_item[(it + 1) & 1]) are free / visible for the next item
    }
    if (t == 0) {
        __threadfence();
        if (atomicAdd(g.work + 3, 1u) == gridDim.x - 1) {
            g.work[2] = 0;
            g.work[3] = 0;
        }
    }
}

// Spectrum for the wide kernel: H16384[f] / 16384 by direct f64 summation (exact argument reduction), stored where the
// middle pass of thread u finds it: float4 [q * 512 + u] = (H[f(32 u + 2 q)], H[f(32 u + 2 q + 1)]),
// f(p) = k1 + 16 k2 + 512 bitrev5(s) for p = k1 * 1024 + k2 * 32 + s.
// blockIdx.y: tap set (taps_rev + set * N, Hout + set * stride), here and in the other spectrum kernels.
__global__ void fir_spectrum_wide_kernel(const double* __restrict__ taps_rev, int N, float2* __restrict__ Hout, long long stride) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= kN2) return;
    taps_rev += (long long)blockIdx.y * N;
    Hout += blockIdx.y * stride;
    const int k1 = p >> 10, k2 = (p >> 5) & 31, sreg = p & 31;
    const int f = k1 + 16 * k2 + 512 * bitrev5(sreg);
    double re = 0.0, im = 0.0;
    for (int n = 0; n < N; n++) {
        const int m = (int)(((long long)f * n) & (kN2 - 1));
        double sn, cs;
        sincospi(-2.0 * (double)m / (double)kN2, &sn, &cs);
        const double h = taps_rev[N - 1 - n];  // h[n] = taps[N-1-n] (fir.rs:163-168)
        re += h * cs;
        im += h * sn;
    }
    const int u = p >> 5, q = sreg >> 1;
    Hout[(size_t)(q * kNTW + u) * 2 + (sreg & 1)] = make_float2((float)(re / kN2), (float)(im / kN2));
}

// ======================= uniformly partitioned convolution for short calls ("UPC" kernel) =======================
// A call of 1024 samples still needs an 8192-point window with the kernels above (N - 1 = 4095 samples of history in front of
// 1024 new ones): four times the transform work per output.  For such calls the impulse response is cut into P = ceil(N / 1024)
// partitions of B = 1024 taps and the convolution runs block by block in the frequency domain (north_star's "uniformly
// partitioned FFT convolution in shared memory"):
//     X_b = FFT2048([block b-1, block b])                     one forward transform per new block, kept in a frequency-domain
//     Y_b = sum_p X_(b-p) . H_p,  H_p = FFT2048([h_p, 0])     delay line (FDL) of the last P spectra per channel pair
//     y_b = last 1024 samples of IFFT2048(Y_b)
// Two channels share a complex transform as everywhere else.  One 128-thread CTA per channel pair walks the call's blocks in
// order; 2048 points = radices 16 . 16 . 8, 19 KB of shared memory, so eight CTAs share an SM.  The FDL lives in global memory
// ([pair][slot = block mod P][2048], written and read back in the middle pass's own register order); when the previous call
// was not a UPC call the launch first recomputes the P-1 previous spectra from the time-domain ring ("prime" blocks).
// Position p = k1 * 128 + k2 * 8 + s holds bin f = k1 + 16 k2 + 256 bitrev3(s).
constexpr int kUB = 1024;                    // partition / block length
constexpr int kUF = 2 * kUB;                 // transform size
constexpr int kUNT = 128;                    // threads
constexpr int kUPad = kUF + kUF / 8 + 8 * (kUF / 128);   // 2432 complex
constexpr int kUT2 = 15 * 8;                 // W128^(j k), k = 1..15 major, j < 8
constexpr int kUTw = kCoarse + kFine + kUT2;
constexpr int kUMaxP = 4;
__device__ __forceinline__ int padu(int p) { return p + (p >> 3) + ((p >> 7) << 3); }

struct UpcArgs {
    const float* U;
    long long u_stride;
    int u_ring, u_pos;
    float* Y;
    long long y_stride;
    const float4* H;       // [P][2][4][128] float4: partition spectra in middle-pass order, scaled 1 / 2048
    float4* fdl;           // [pairs][P][2][4][128] float4
    const float2* Wg;      // compact twiddle table (coarse 512 | fine 32 | ...)
    float scale;           // divisor (and the fused sink average), one multiplication
    int c_begin, c_end;
    int P, n_blocks, prime;
    long long b0;          // running block counter of the call's first block (FDL slot = counter mod P)
    int pair0;             // first channel pair (PC: first transform of the slice) of this launch inside the FDL
    const int4* xf;        // PC = true: transform table slice, set k's partitions at H + k * h_stride / 2 (see FftArgs)
    long long h_stride;
};

template <bool PC>
__global__ void __launch_bounds__(kUNT, 8)
fir_upc_kernel(const __grid_constant__ UpcArgs g) {
    extern __shared__ float2 smem_f2[];
    C2<float>* a = reinterpret_cast<C2<float>*>(smem_f2);
    C2<float>* tabs = a + kUPad;
    const int t = threadIdx.x;
    for (int i = t; i < kCoarse + kFine; i += kUNT) tabs[i] = C2<float>{g.Wg[i].x, g.Wg[i].y};
    if (t < kUT2) {  // W128^(j k) = W512^(4 j k)
        const int k = t / 8 + 1, j = t % 8;
        const float2 w = g.Wg[(4 * j * k) & (kCoarse - 1)];
        tabs[kCoarse + kFine + t] = C2<float>{w.x, w.y};
    }
    const Tw<float> W{tabs, tabs + kCoarse, nullptr};
    const C2<float>* T2 = tabs + kCoarse + kFine;
    const int pr = blockIdx.x;
    const int4 x = PC ? g.xf[pr] : int4{};   // per-channel taps: {chA, chB or -1, set} of transform pr
    const int chA = PC ? x.x : g.c_begin + 2 * pr, chB = PC ? x.y : chA + 1;
    const bool hasB = PC ? chB >= 0 : chB < g.c_end;
    const float* rowA = g.U + (long long)chA * g.u_stride;
    const float* rowB = g.U + (long long)(hasB ? chB : chA) * g.u_stride;
    float4* fdl = g.fdl + (size_t)(g.pair0 + pr) * g.P * 1024;
    const bool unit = g.scale == 1.0f;
    __syncthreads();
    // twiddles of pass 1 / 1': W2048^(j q) = W16384^(8 j q), j = t; rebuilt in each of the two passes (84 instructions) rather
    // than held in 30 registers for the whole launch: the kernel waits on memory, and 64 registers mean 8 CTAs per SM, not 6
    auto twiddles1 = [&](C2<float> (&w1)[16]) {
        const int j = t;
        w1[1] = W.at2(8 * j); w1[2] = W.at2(16 * j); w1[4] = W.at2(32 * j); w1[8] = W.at2(64 * j);
        w1[3] = cmul(w1[1], w1[2]); w1[5] = cmul(w1[1], w1[4]); w1[6] = cmul(w1[2], w1[4]); w1[7] = cmul(w1[3], w1[4]);
#pragma unroll
        for (int q = 9; q < 16; q++) w1[q] = cmul(w1[q - 8], w1[8]);
    };
    for (int blk = -g.prime; blk < g.n_blocks; blk++) {
        const long long bidx = g.b0 + blk;
        const int slot = (int)(((bidx % g.P) + g.P) % g.P);
        const int wb = ring_slot(g.u_pos, (blk - 1) * kUB, g.u_ring);   // ring slot of window sample 0 (block blk - 1)
        // The middle pass reads the P-1 previous spectra (16 KB each) from the delay line with nothing but a complex multiply
        // between the loads (ncu: 68 % of the stall samples there, 80 % of them on the loads, L2 hit rate 9 %): pull them
        // into L2 now, two passes ahead -- one 128-byte line per thread and slot.
        if (blk >= 0)
            for (int pp = 1; pp < g.P; pp++) {
                const int sl2 = (int)((((bidx - pp) % g.P) + g.P) % g.P);
                asm volatile("prefetch.global.L2 [%0];" ::"l"(fdl + (size_t)sl2 * 1024 + t * 8));
            }
        // ---- pass 1: global -> radix 16 over stride 128 -> shared
        {
            const int j = t;
            C2<float> v[16];
#pragma unroll
            for (int r = 0; r < 16; r++) {
                int sl = wb + j + r * 128;
                if (sl >= g.u_ring) sl -= g.u_ring;
                v[r] = C2<float>{__ldg(rowA + sl), __ldg(rowB + sl)};
            }
            fft_dif<16>(v);
            C2<float> w1[16];
            twiddles1(w1);
            C2<float>* p = a + padu(j);   // padu(j + 128 q) = padu(j) + 152 q
            p[0] = v[0];
#pragma unroll
            for (int s = 1; s < 16; s++) p[bitrev4(s) * 152] = cmul(v[s], w1[bitrev4(s)]);
        }
        __syncthreads();
        // ---- pass 2: radix 16 over stride 8 inside each 128-block
        {
            const int b = t >> 3, j = t & 7;
            C2<float>* p = a + padu(b * 128 + j);   // padu(base + 8 r) = padu(base) + 9 r
            C2<float> v[16];
#pragma unroll
            for (int r = 0; r < 16; r++) v[r] = p[r * 9];
            fft_dif<16>(v);
            p[0] = v[0];
#pragma unroll
            for (int s = 1; s < 16; s++) p[bitrev4(s) * 9] = cmul(v[s], T2[(bitrev4(s) - 1) * 8 + j]);
        }
        __syncthreads();
        // ---- middle: radix 8 on contiguous points; spectrum into the FDL; partitioned product; inverse radix 8
#pragma unroll 1
        for (int q = 0; q < 2; q++) {
            const int u = t + kUNT * q;
            C2<float>* p = a + padu(8 * u);   // 8 contiguous points, no pad inside
            C2<float> v[8];
#pragma unroll
            for (int s = 0; s < 8; s++) v[s] = p[s];
            fft_dif<8>(v);
            float4* xs = fdl + ((size_t)(slot * 2 + q) * 4) * kUNT + t;
#pragma unroll
            for (int s2 = 0; s2 < 4; s2++) __stcg(xs + s2 * kUNT, make_float4(v[2 * s2].x, v[2 * s2].y, v[2 * s2 + 1].x, v[2 * s2 + 1].y));
            if (blk < 0) continue;   // prime block: only its spectrum is needed
            C2<float> acc[8];
            {
                const float4* h = (PC ? g.H + x.z * (g.h_stride / 2) : g.H) + ((size_t)(0 * 2 + q) * 4) * kUNT + t;
#pragma unroll
                for (int s2 = 0; s2 < 4; s2++) {
                    const float4 hh = __ldg(h + s2 * kUNT);
                    acc[2 * s2] = cmul(v[2 * s2], C2<float>{hh.x, hh.y});
                    acc[2 * s2 + 1] = cmul(v[2 * s2 + 1], C2<float>{hh.z, hh.w});
                }
            }
            for (int pp = 1; pp < g.P; pp++) {
                const int sl2 = (int)((((bidx - pp) % g.P) + g.P) % g.P);
                const float4* xo = fdl + ((size_t)(sl2 * 2 + q) * 4) * kUNT + t;
                const float4* h = (PC ? g.H + x.z * (g.h_stride / 2) : g.H) + ((size_t)(pp * 2 + q) * 4) * kUNT + t;
#pragma unroll
                for (int s2 = 0; s2 < 4; s2++) {
                    const float4 x = __ldcg(xo + s2 * kUNT);
                    const float4 hh = __ldg(h + s2 * kUNT);
                    const C2<float> m0 = cmul(C2<float>{x.x, x.y}, C2<float>{hh.x, hh.y});
                    const C2<float> m1 = cmul(C2<float>{x.z, x.w}, C2<float>{hh.z, hh.w});
                    acc[2 * s2] = acc[2 * s2] + m0;
                    acc[2 * s2 + 1] = acc[2 * s2 + 1] + m1;
                }
            }
            ifft_dit<8>(acc);
#pragma unroll
            for (int s = 0; s < 8; s++) p[s] = acc[s];
        }
        __syncthreads();
        if (blk < 0) continue;
        // ---- pass 2'
        {
            const int b = t >> 3, j = t & 7;
            C2<float>* p = a + padu(b * 128 + j);
            C2<float> v[16];
            v[0] = p[0];
#pragma unroll
            for (int s = 1; s < 16; s++) v[s] = cmulc(p[bitrev4(s) * 9], T2[(bitrev4(s) - 1) * 8 + j]);
            ifft_dit<16>(v);
#pragma unroll
            for (int r = 0; r < 16; r++) p[r * 9] = v[r];
        }
        __syncthreads();
        // ---- pass 1': the last 1024 samples of the 2048-point result are this block's outputs
        {
            const int j = t;
            const C2<float>* p = a + padu(j);
            C2<float> v[16], w1[16];
            twiddles1(w1);
            v[0] = p[0];
#pragma unroll
            for (int s = 1; s < 16; s++) v[s] = cmulc(p[bitrev4(s) * 152], w1[bitrev4(s)]);
            ifft_dit<16>(v);
            float* outA = g.Y + (long long)chA * g.y_stride + (long long)blk * kUB - kUB;
            float* outB = g.Y + (long long)(hasB ? chB : chA) * g.y_stride + (long long)blk * kUB - kUB;
#pragma unroll
            for (int r = 8; r < 16; r++) {
                const int n = j + r * 128;   // >= 1024
                outA[n] = unit ? v[r].x : __fmul_rn(v[r].x, g.scale);
                if (hasB) outB[n] = unit ? v[r].y : __fmul_rn(v[r].y, g.scale);
            }
        }
        __syncthreads();
    }
}

// Partition spectra for the UPC kernel, by direct f64 summation, in the middle pass's order:
// float4 [((p * 2 + q) * 4 + s2) * 128 + t] = (H_p[f(8 u + 2 s2)], H_p[f(8 u + 2 s2 + 1)]), u = t + 128 q.
__global__ void fir_spectrum_upc_kernel(const double* __restrict__ taps_rev, int N, int P, float2* __restrict__ Hout, long long stride) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= P * kUF) return;
    taps_rev += (long long)blockIdx.y * N;
    Hout += blockIdx.y * stride;
    const int p = idx / kUF, pos = idx % kUF;
    const int k1 = pos >> 7, k2 = (pos >> 3) & 15, sreg = pos & 7;
    const int f = k1 + 16 * k2 + 256 * bitrev3(sreg);
    double re = 0.0, im = 0.0;
    for (int n = 0; n < kUB; n++) {
        const int tap = p * kUB + n;
        if (tap >= N) break;
        const int m = (int)(((long long)f * n) & (kUF - 1));
        double sn, cs;
        sincospi(-2.0 * (double)m / (double)kUF, &sn, &cs);
        const double h = taps_rev[N - 1 - tap];
        re += h * cs;
        im += h * sn;
    }
    const int u = pos >> 3, q = u / kUNT, tt = u % kUNT, s2 = sreg >> 1;
    Hout[((size_t)((p * 2 + q) * 4 + s2) * kUNT + tt) * 2 + (sreg & 1)] = make_float2((float)(re / kUF), (float)(im / kUF));
}

// ======================= packed variant: two sub-transforms per register pair =======================
// One radix-2 decimation-in-frequency step turns the F = 8192 point transform of z into two INDEPENDENT
// 4096-point transforms (E[n] = z[n] + z[n+4096] -> even bins, O[n] = (z[n] - z[n+4096]) W_F^n -> odd bins)
// with identical structure and twiddles.  They are carried side by side in 64-bit register pairs
// (re = (E.re, O.re), im = (E.im, O.im)) through four radix-8 passes, the spectrum product and four inverse
// passes, so every butterfly add, twiddle multiply, shared-memory access and index computation is issued ONCE
// for both (add/mul/fma.rn.f32x2).  MEASURED OUTCOME (B200, profiles/r01s3_target_fir_fft_packed_kernel.txt): this
// kernel issues 16 % fewer warp-instructions than the scalar kernel above (266 M vs 315 M per launch) but runs
// 0.441 ms against 0.412 ms: the packed instructions occupy the FP32 pipe for two cycles each and have longer
// dependent-issue latency (tests/cuda/f32x2_microbench.cu: 2.0 packed vs 3.7 scalar FFMA per clock per SM), so
// with 24 warps per SM the kernel becomes latency-bound (issue-active 55 %, FP32 pipe 44 %) instead of
// issue-bound (70 %).  It therefore stays an opt-in (fir_mode = 3) and the scalar kernel is the default.
// Only the upper half of the circular convolution is valid with 4096 + 1 taps, and
// z[n + 4096] = E'[n] - W_F^-n O'[n] is exactly the half the last radix-2 step has to produce.
// Shared memory: 4096 float4 (E.re, O.re, E.im, O.im) with an XOR swizzle of the low three index bits (no
// padding), + the twiddle tables stored duplicated (wr, wr, wi, wi) so one LDS.128 yields packed operands.
typedef unsigned long long u64;
constexpr int kH2 = kF / 2;  // points of each sub-transform
constexpr int kFineP = 16;   // fine twiddle entries of this kernel (W8192^b, b < 16)
struct VF { u64 re, im; };   // packed complex pair: lo half = E, hi half = O
struct WF { u64 re, im; };   // one twiddle, duplicated into both halves
__device__ __forceinline__ u64 pk(float lo, float hi) { return (u64)__float_as_uint(lo) | ((u64)__float_as_uint(hi) << 32); }
__device__ __forceinline__ float lo32(u64 a) { return __uint_as_float((unsigned)a); }
__device__ __forceinline__ float hi32(u64 a) { return __uint_as_float((unsigned)(a >> 32)); }
__device__ __forceinline__ u64 add2(u64 a, u64 b) { u64 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 sub2(u64 a, u64 b) { u64 d; asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 mul2(u64 a, u64 b) { u64 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) { u64 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ u64 neg2(u64 a) { return a ^ 0x8000000080000000ull; }  // integer pipe: free next to the FP32 pipe
__device__ __forceinline__ VF operator+(VF a, VF b) { return {add2(a.re, b.re), add2(a.im, b.im)}; }
__device__ __forceinline__ VF operator-(VF a, VF b) { return {sub2(a.re, b.re), sub2(a.im, b.im)}; }
// a * w and a * conj(w); the factor may differ per half (spectrum product) or be duplicated (twiddles)
__device__ __forceinline__ VF vmul(VF a, u64 wre, u64 wim) { return {fma2(neg2(a.im), wim, mul2(a.re, wre)), fma2(a.re, wim, mul2(a.im, wre))}; }
__device__ __forceinline__ VF vmulc(VF a, u64 wre, u64 wim) { return {fma2(a.im, wim, mul2(a.re, wre)), fma2(neg2(a.re), wim, mul2(a.im, wre))}; }
__device__ __forceinline__ WF wmul(WF a, WF b) { const VF r = vmul(VF{a.re, a.im}, b.re, b.im); return {r.re, r.im}; }

// a * w_SZ^I for the rotations a radix-8 butterfly needs (SZ in {2, 4, 8})
template <int SZ, int I, bool INV>
__device__ __forceinline__ VF vtw(VF a) {
    if constexpr (I == 0) {
        return a;
    } else if constexpr (4 * I == SZ) {
        if constexpr (INV) return {neg2(a.im), a.re};
        else return {a.im, neg2(a.re)};
    } else {
        static_assert(SZ == 8 && (I == 1 || I == 3), "radix-8 rotations only");
        const u64 h = pk(0.70710678118654752440f, 0.70710678118654752440f), nh = neg2(h);
        if constexpr (I == 1) {
            if constexpr (INV) return {mul2(sub2(a.re, a.im), h), mul2(add2(a.re, a.im), h)};
            else return {mul2(add2(a.re, a.im), h), mul2(sub2(a.im, a.re), h)};
        } else {
            if constexpr (INV) return {mul2(add2(a.re, a.im), nh), mul2(sub2(a.re, a.im), h)};
            else return {mul2(sub2(a.im, a.re), h), mul2(add2(a.re, a.im), nh)};
        }
    }
}
// Radix-8 butterflies written out so that the +-i rotations fold into the choice of add / sub of the next stage
// (a negation of a packed pair would cost two LOP3).
// x + (-i) y and x - (-i) y;  x + (i) y and x - (i) y
__device__ __forceinline__ VF add_mi(VF x, VF y) { return {add2(x.re, y.im), sub2(x.im, y.re)}; }
__device__ __forceinline__ VF sub_mi(VF x, VF y) { return {sub2(x.re, y.im), add2(x.im, y.re)}; }
__device__ __forceinline__ void fft_dif8v(VF (&v)[8]) {  // natural in, bit-reversed out (v[s] = bin bitrev3(s))
    const VF a0 = v[0] + v[4], a1 = v[1] + v[5], a2 = v[2] + v[6], a3 = v[3] + v[7];
    const VF b0 = v[0] - v[4], b2 = v[2] - v[6];
    const VF b1 = vtw<8, 1, false>(v[1] - v[5]), b3 = vtw<8, 3, false>(v[3] - v[7]);
    const VF c0 = a0 + a2, c1 = a1 + a3, d0 = a0 - a2, d1 = a1 - a3;        // d1 still lacks its factor -i
    const VF e0 = add_mi(b0, b2), e1 = b1 + b3, f0 = sub_mi(b0, b2), f1 = b1 - b3;  // b2 (-i) folded; f1 lacks -i
    v[0] = c0 + c1; v[1] = c0 - c1;
    v[2] = add_mi(d0, d1); v[3] = sub_mi(d0, d1);
    v[4] = e0 + e1; v[5] = e0 - e1;
    v[6] = add_mi(f0, f1); v[7] = sub_mi(f0, f1);
}
__device__ __forceinline__ void ifft_dit8v(VF (&v)[8]) {  // exact mirror: bit-reversed in, natural out, conjugate rotations
    const VF c0 = v[0] + v[1], c1 = v[0] - v[1], d0 = v[2] + v[3], d1 = v[2] - v[3];  // d1 lacks its factor +i
    const VF e0 = v[4] + v[5], e1 = v[4] - v[5], f0 = v[6] + v[7], f1 = v[6] - v[7];  // f1 lacks +i
    const VF a0 = c0 + d0, a2 = c0 - d0, a1 = sub_mi(c1, d1), a3 = add_mi(c1, d1);   // x + i y = sub_mi(x, y)
    const VF b0 = e0 + f0, b2 = e0 - f0;                                             // b2 lacks +i
    const VF b1 = vtw<8, 1, true>(sub_mi(e1, f1)), b3 = vtw<8, 3, true>(add_mi(e1, f1));
    v[0] = a0 + b0; v[4] = a0 - b0;
    v[1] = a1 + b1; v[5] = a1 - b1;
    v[2] = sub_mi(a2, b2); v[6] = add_mi(a2, b2);
    v[3] = a3 + b3; v[7] = a3 - b3;
}
__device__ __forceinline__ int swz8(int p) { return p ^ ((p >> 3) & 7); }
// explicit 128-bit accesses straight into / out of the two 64-bit register pairs (left to itself the compiler splits
// the float4 into two LDS.64, which at a 16-byte lane stride are two-way bank conflicts)
__device__ __forceinline__ VF ld_vf(const float4* a, int p) {
    VF v;
    asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(v.re), "=l"(v.im) : "r"((unsigned)__cvta_generic_to_shared(a + swz8(p))));
    return v;
}
__device__ __forceinline__ void st_vf(float4* a, int p, VF v) {
    asm volatile("st.shared.v2.b64 [%0], {%1, %2};" ::"r"((unsigned)__cvta_generic_to_shared(a + swz8(p))), "l"(v.re), "l"(v.im) : "memory");
}

// duplicated twiddle tables in shared memory: W_F^k = coarse[k >> 4] * fine[k & 15]
struct TwP {
    const float4* coarse;  // [512]
    const float4* fine;    // [16]
    __device__ __forceinline__ WF c(int m) const {
        WF w;
        asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(w.re), "=l"(w.im) : "r"((unsigned)__cvta_generic_to_shared(coarse + (m & (kCoarse - 1)))));
        return w;
    }
    __device__ __forceinline__ WF at(int k) const {
        const float4 q = fine[k & 15];
        return wmul(c(k >> 4), WF{pk(q.x, q.y), pk(q.z, q.w)});
    }
    __device__ __forceinline__ C2<float> scalar(int k) const {  // W_F^k as one scalar complex
        const float4 a = coarse[(k >> 4) & (kCoarse - 1)], b = fine[k & 15];
        return cmul(C2<float>{a.x, a.z}, C2<float>{b.x, b.z});
    }
};
// w[q] = w1^q for q = 1..7 from w1, w2, w4
__device__ __forceinline__ void powers8(WF w1, WF w2, WF w4, WF (&w)[8]) {
    w[1] = w1; w[2] = w2; w[4] = w4;
    w[3] = wmul(w1, w2);
    w[5] = wmul(w1, w4);
    w[6] = wmul(w2, w4);
    w[7] = wmul(w[3], w4);
}
// forward / inverse radix-8 pass on the shared array, sub-transform size M in {512, 64}: both butterflies of a
// thread share j, so the twiddles are computed once
template <int M>
__device__ __forceinline__ void fwd_pass8v(float4* a, const TwP& W, int t) {
    constexpr int L = M / 8, CS = (kF / 16) / M;  // coarse-table step of W_M
    const int j = t % L;
    WF w[8];
    powers8(W.c(j * CS), W.c(2 * j * CS), W.c(4 * j * CS), w);
#pragma unroll 1
    for (int k = 0; k < kH2 / 8 / kNT; k++) {
        const int u = t + kNT * k, base = (u / L) * M + j;
        VF v[8];
#pragma unroll
        for (int r = 0; r < 8; r++) v[r] = ld_vf(a, base + r * L);
        fft_dif8v(v);
        st_vf(a, base, v[0]);
#pragma unroll
        for (int s = 1; s < 8; s++) st_vf(a, base + bitrev3(s) * L, vmul(v[s], w[bitrev3(s)].re, w[bitrev3(s)].im));
    }
}
template <int M>
__device__ __forceinline__ void inv_pass8v(float4* a, const TwP& W, int t) {
    constexpr int L = M / 8, CS = (kF / 16) / M;
    const int j = t % L;
    WF w[8];
    powers8(W.c(j * CS), W.c(2 * j * CS), W.c(4 * j * CS), w);
#pragma unroll 1
    for (int k = 0; k < kH2 / 8 / kNT; k++) {
        const int u = t + kNT * k, base = (u / L) * M + j;
        VF v[8];
        v[0] = ld_vf(a, base);
#pragma unroll
        for (int s = 1; s < 8; s++) v[s] = vmulc(ld_vf(a, base + bitrev3(s) * L), w[bitrev3(s)].re, w[bitrev3(s)].im);
        ifft_dit8v(v);
#pragma unroll
        for (int r = 0; r < 8; r++) st_vf(a, base + r * L, v[r]);
    }
}

// Window of segment s: call-relative samples [4096 (s - 1), 4096 (s + 1)); outputs [4096 s, 4096 (s + 1)).
// Requires n_taps <= 4097 (taps beyond the stored history multiply zeros: samples before -hist_pad read as 0).
__global__ void __launch_bounds__(kNT, 3)
fir_fft_packed_kernel(const float* __restrict__ U, long long u_stride, int hist_pad, int u_ring, int u_pos, float* __restrict__ Y, long long y_stride,
                      const float4* __restrict__ Hg, const float2* __restrict__ Wg, long long T, float divisor, float post_nf,
                      int c_begin, int c_end) {
    extern __shared__ float4 smem_f4[];
    float4* a = smem_f4;  // [4096]
    float4* tab = a + kH2;
    const int t = threadIdx.x;
    for (int i = t; i < kCoarse; i += kNT) { const float2 w = Wg[i]; tab[i] = make_float4(w.x, w.x, w.y, w.y); }
    if (t < kFineP) { const float2 w = Wg[kCoarse + 2 * t]; tab[kCoarse + t] = make_float4(w.x, w.x, w.y, w.y); }  // W8192^t = fine[2 t]
    const TwP W{tab, tab + kCoarse};
    const long long s0 = (long long)blockIdx.x * kH2;
    const int chA = c_begin + 2 * blockIdx.y, chB = chA + 1;
    const bool hasB = chB < c_end;
    const float* rowA = U + (long long)chA * u_stride;  // ring rows: window sample i at slot (wb + i) mod u_ring
    const float* rowB = U + (long long)(hasB ? chB : chA) * u_stride;
    // window samples below lo precede the stored history, samples >= lim lie beyond this call's input: zeros.
    // 0 <= lo <= 4096 < lim <= 8192 after clamping, so [lo, lim) is never empty and clamped indices are loadable.
    const long long lo_ll = -(long long)hist_pad - (s0 - kH2), lim_ll = T - (s0 - kH2);
    const int lo = lo_ll < 0 ? 0 : (int)lo_ll, lim = lim_ll > kF ? kF : (int)lim_ll;
    // ring slot of window sample `lo` (the first loadable one: lo - kH2 + s0 >= -hist_pad); loaded samples i lie in
    // [lo, lim), lim - lo <= hist_pad + T <= u_ring: one wrap at most
    const int wlo = ring_slot(u_pos, (int)(s0 - kH2 + lo), u_ring);
    auto slot = [&](int i) { int p = wlo + (i - lo); return p >= u_ring ? p - u_ring : p; };
    __syncthreads();

    // ---- forward pass 0: global -> radix-2 split -> radix-8 (M = 4096) -> shared
#pragma unroll 1
    for (int k = 0; k < kH2 / 8 / kNT; k++) {
        const int j = t + kNT * k;
        const C2<float> wj = W.scalar(j);
        VF v[8];
        static_for<8>([&](auto rr) {
            constexpr int r = decltype(rr)::value;
            const int n = j + r * (kH2 / 8);
            // branch-free (clamped index, select afterwards) so that all 32 loads of a butterfly are issued back to back
            const int i0 = min(max(n, lo), lim - 1), i1 = min(n + kH2, lim - 1);  // n + 4096 >= lo always
            const bool ok0 = n >= lo && n < lim, ok1 = n + kH2 < lim;
            const int p0 = slot(i0), p1 = slot(i1);
            float a0 = __ldg(rowA + p0), b0 = __ldg(rowB + p0), a1 = __ldg(rowA + p1), b1 = __ldg(rowB + p1);
            a0 = ok0 ? a0 : 0.f; b0 = (ok0 && hasB) ? b0 : 0.f; a1 = ok1 ? a1 : 0.f; b1 = (ok1 && hasB) ? b1 : 0.f;
            const C2<float> d = tw<16, r, false, float>(cmul(C2<float>{a0 - a1, b0 - b1}, wj));  // (z[n] - z[n+4096]) W_F^(j + 512 r)
            v[r] = VF{pk(a0 + a1, d.x), pk(b0 + b1, d.y)};
        });
        fft_dif8v(v);
        WF w[8];
        powers8(W.at(2 * j), W.at(4 * j), W.at(8 * j), w);
        st_vf(a, j, v[0]);
#pragma unroll
        for (int s = 1; s < 8; s++) st_vf(a, j + bitrev3(s) * (kH2 / 8), vmul(v[s], w[bitrev3(s)].re, w[bitrev3(s)].im));
    }
    __syncthreads();
    fwd_pass8v<kH2 / 8>(a, W, t);
    __syncthreads();
    fwd_pass8v<kH2 / 64>(a, W, t);
    __syncthreads();
    // ---- pass 3 (radix 8, no twiddles) . spectrum product . inverse pass 3, in registers
#pragma unroll 1
    for (int k = 0; k < kH2 / 8 / kNT; k++) {
        const int base = 8 * (t + kNT * k);
        const float4* h4 = Hg + (k * 8) * kNT + t;  // [k][s][thread]: (H_even.re, H_odd.re, H_even.im, H_odd.im)
        float4 h[8];
#pragma unroll
        for (int s = 0; s < 8; s++) h[s] = __ldg(h4 + s * kNT);
        VF v[8];
#pragma unroll
        for (int s = 0; s < 8; s++) v[s] = ld_vf(a, base + s);
        fft_dif8v(v);
#pragma unroll
        for (int s = 0; s < 8; s++) v[s] = vmul(v[s], pk(h[s].x, h[s].y), pk(h[s].z, h[s].w));
        ifft_dit8v(v);
#pragma unroll
        for (int s = 0; s < 8; s++) st_vf(a, base + s, v[s]);
    }
    __syncthreads();
    inv_pass8v<kH2 / 64>(a, W, t);
    __syncthreads();
    inv_pass8v<kH2 / 8>(a, W, t);
    __syncthreads();
    // ---- inverse pass 0: shared -> radix-8 -> last radix-2 step (upper half only) -> global
    {
        float* outA = Y + (long long)chA * y_stride + s0;
        float* outB = Y + (long long)chB * y_stride + s0;
        const bool post = post_nf != 0.0f;
        const float post_rnf = post ? __frcp_rn(post_nf) : 0.0f;
        const long long out_lim = T - s0;
#pragma unroll 1
        for (int k = 0; k < kH2 / 8 / kNT; k++) {
            const int j = t + kNT * k;
            WF w[8];
            powers8(W.at(2 * j), W.at(4 * j), W.at(8 * j), w);
            VF v[8];
            v[0] = ld_vf(a, j);
#pragma unroll
            for (int s = 1; s < 8; s++) v[s] = vmulc(ld_vf(a, j + bitrev3(s) * (kH2 / 8)), w[bitrev3(s)].re, w[bitrev3(s)].im);
            ifft_dit8v(v);
            const C2<float> wj = W.scalar(j);
            static_for<8>([&](auto rr) {
                constexpr int r = decltype(rr)::value;
                const int n = j + r * (kH2 / 8);
                const C2<float> o = tw<16, r, true, float>(cmulc(C2<float>{hi32(v[r].re), hi32(v[r].im)}, wj));  // O'[n] W_F^-(j + 512 r)
                float ya = __fmul_rn(lo32(v[r].re) - o.x, divisor), yb = __fmul_rn(lo32(v[r].im) - o.y, divisor);
                if (post) { ya = div_nf(ya, post_nf, post_rnf); yb = div_nf(yb, post_nf, post_rnf); }
                if (n < out_lim) {
                    outA[n] = ya;
                    if (hasB) outB[n] = yb;
                }
            });
        }
    }
}

// Spectrum for the packed kernel: bin f of the zero-padded impulse response by direct f64 summation (exact
// argument reduction: f n mod F is an integer), scaled by 1/F, stored where pass 3 of the packed kernel finds
// it: float4 [(k * 8 + s) * 256 + t] = (H[2 f'].re, H[2 f' + 1].re, H[2 f'].im, H[2 f' + 1].im) with
// f' = d3 + 8 d2 + 64 d1 + 512 d0, (d3, d2, d1) the base-8 digits of u = t + 256 k, d0 = bitrev3(s).
__global__ void fir_spectrum_packed_kernel(const double* __restrict__ taps_rev, int N, float4* __restrict__ Hout, long long stride4) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;  // [k][s][t]
    if (idx >= kH2) return;
    taps_rev += (long long)blockIdx.y * N;
    Hout += blockIdx.y * stride4;
    const int tt = idx % kNT, s = (idx / kNT) % 8, k = idx / (8 * kNT);
    const int u = tt + kNT * k;
    const int d3 = u / 64, d2 = (u / 8) % 8, d1 = u % 8, d0 = bitrev3(s);
    const int fp = d3 + 8 * d2 + 64 * d1 + 512 * d0;
    double acc[4] = {0, 0, 0, 0};
    for (int half = 0; half < 2; half++) {
        const int f = 2 * fp + half;
        double re = 0.0, im = 0.0;
        for (int n = 0; n < N; n++) {
            const int m = (int)(((long long)f * n) & (kF - 1));
            double sn, cs;
            sincospi(-2.0 * (double)m / (double)kF, &sn, &cs);
            const double h = taps_rev[N - 1 - n];  // h[n] = taps[N-1-n] (fir.rs:163-168)
            re += h * cs;
            im += h * sn;
        }
        acc[half] = re / kF;
        acc[2 + half] = im / kF;
    }
    Hout[idx] = make_float4((float)acc[0], (float)acc[1], (float)acc[2], (float)acc[3]);
}

// ---- spectrum of h in the transform's own output order (f64) -----------------------------------------------
// FFT8192(h) / 8192: the bins of an 8192-point segment, in the order mid_pass16 reads them.
__global__ void __launch_bounds__(kNT, 1)
fir_spectrum_kernel(const double* __restrict__ taps_rev, int N, const double2* __restrict__ Wd, float2* __restrict__ Hout, long long stride) {
    extern __shared__ double2 smem_d2[];
    taps_rev += (long long)blockIdx.y * N;
    Hout += blockIdx.y * stride;
    C2<double>* a = reinterpret_cast<C2<double>*>(smem_d2);
    const int t = threadIdx.x;
    const Tw<double> W = load_tables<double>(a + kPadded, Wd, t);
    for (int n = t; n < kF; n += kNT) {
        const double h = n < N ? taps_rev[N - 1 - n] : 0.0;  // h[n] = taps[N-1-n]
        a[pad(n)] = C2<double>{h, 0.0};
    }
    __syncthreads();
    fwd_pass8<kF>(a, W, t);
    __syncthreads();
    fwd_pass8<kF / 8>(a, W, t);
    __syncthreads();
    fwd_pass8<kF / 64>(a, W, t);
    __syncthreads();
    for (int k = 0; k < kF / 16 / kNT; k++) {
        const int u = t + kNT * k, base = 16 * u;
        C2<double> v[16];
#pragma unroll
        for (int s = 0; s < 16; s++) v[s] = a[pad(base) + s];
        fft_dif<16>(v);
#pragma unroll
        for (int s = 0; s < 16; s++)  // [k][s / 2][thread] float4 order, see mid_pass16
            Hout[((k * 8 + (s >> 1)) * kNT + t) * 2 + (s & 1)] = make_float2((float)(v[s].x / kF), (float)(v[s].y / kF));
    }
}

struct Tables {
    float2* Wf = nullptr;    // compact twiddle table [512 coarse + 32 fine] (see Tw)
    double2* Wd = nullptr;
    int n_sm = 0;
};
Tables g_tab_dev[kMaxDevices];  // device memory: one set per device, built once
std::mutex g_tab_mu;
#define g_tab g_tab_dev[current_device_slot()]

int ensure_tables() {
    std::lock_guard<std::mutex> lk(g_tab_mu);
    if (g_tab.Wf) return 0;
    constexpr int n = kTwW;  // coarse | fine | W1024^(j k) table of the wide kernel
    std::vector<float2> wf(n);
    std::vector<double2> wd(n);
    for (int k = 0; k < n; k++) {
        double ang;
        if (k < kCoarse) ang = -2.0 * M_PI * (double)k / (double)kCoarse;
        else if (k < kCoarse + kFine) ang = -2.0 * M_PI * (double)(k - kCoarse) / (2.0 * kF);
        else {
            const int e = k - kCoarse - kFine, q = e / 32 + 1, j = e % 32;
            ang = -2.0 * M_PI * (double)((j * q) & 1023) / 1024.0;
        }
        wd[k] = make_double2(std::cos(ang), std::sin(ang));
        wf[k] = make_float2((float)wd[k].x, (float)wd[k].y);
    }
    cudaError_t e;
    float2* f = nullptr;
    double2* d = nullptr;
    if ((e = cudaMalloc(&f, n * sizeof(float2))) != cudaSuccess) return (int)e;
    if ((e = cudaMalloc(&d, n * sizeof(double2))) != cudaSuccess) return (int)e;
    if ((e = cudaMemcpy(f, wf.data(), n * sizeof(float2), cudaMemcpyHostToDevice)) != cudaSuccess) return (int)e;
    if ((e = cudaMemcpy(d, wd.data(), n * sizeof(double2), cudaMemcpyHostToDevice)) != cudaSuccess) return (int)e;
    int dev = 0, n_sm = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    g_tab.n_sm = n_sm > 0 ? n_sm : 148;
    g_tab.Wd = d;
    g_tab.Wf = f;
    return 0;
}

}  // namespace

int fir_fft_max_taps() { return kF / 2 + 1; }
// H13 (F) | packed-kernel order (F) | wide (2 F) | UPC partitions (4 x 2048 = F)
size_t fir_fft_spectrum_bytes() { return (size_t)5 * kF * sizeof(float2); }
int fir_upc_partitions(int n_taps) { return n_taps <= kUMaxP * kUB ? (n_taps + kUB - 1) / kUB : 0; }
size_t fir_upc_fdl_bytes(int n_taps, int transforms) { return (size_t)transforms * fir_upc_partitions(n_taps) * kUF * sizeof(float2); }
// [0] next item, [1] CTAs done of fir_fft_kernel; [2], [3] the same for fir_fft_wide_kernel
size_t fir_fft_work_bytes() { return 4 * sizeof(unsigned); }
static int effective_taps(int n) { return (n - 1 + 3) / 4 * 4 + 1; }  // Ne - 1 multiple of 4

// Segment plan of one call: n14 double (16384-point) segments first, the wide kernel's items, then n13 single ones for
// fir_fft_kernel.  A double segment must lie fully inside the call, and it is used when it costs less per output than
// single segments at the cost rule kCost14 (one double segment = kCost14 single ones) the plan has used since c4abfd4.
static void segment_plan(int hist, int64_t T, int* n14, int* n13) {
    constexpr double kCost14 = 2.3;
    const int64_t V13 = kF - hist, V14 = 2 * kF - hist;
    const bool use14 = kCost14 / (double)V14 < 1.0 / (double)V13;
    int64_t a = use14 ? T / V14 : 0;
    // the rest: single segments, unless one more double segment would be cheaper -- it would not fit, so no
    const int64_t rem = T - a * V14;
    *n14 = (int)a;
    *n13 = (int)((rem + V13 - 1) / V13);
}

int launch_fir_fft(const FirPlan& fp, const float* U, int64_t u_stride, float* Y, int64_t y_stride, int c_begin, int c_end,
                   int64_t T, cudaStream_t st, int* n_launches) {
    if (fp.log2F != kLog2F || fp.n_taps > fir_fft_max_taps() || fp.n_taps < 1) return (int)cudaErrorInvalidValue;
    if (fp.u_ring <= 0 || (fp.u_ring & 127) || fp.hist_pad + T > fp.u_ring) return (int)cudaErrorInvalidValue;
    int rc = ensure_tables();
    if (rc) return rc;
    if (fp.mode == FIR_FFT_PACKED) {  // opt-in: measured 5 % slower than the scalar kernel (see the comment above VF)
        if (fp.xf) return (int)cudaErrorInvalidValue;  // shared taps only
        static std::atomic<bool> configured2_dev[kMaxDevices];
        std::atomic<bool>& configured2 = configured2_dev[current_device_slot()];
        const int smem2 = (kH2 + kCoarse + kFineP) * (int)sizeof(float4);
        if (!configured2.load(std::memory_order_acquire)) {
            cudaError_t e = cudaFuncSetAttribute(fir_fft_packed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem2);
            if (e != cudaSuccess) return (int)e;
            configured2.store(true, std::memory_order_release);
        }
        const long long n_seg2 = (T + kH2 - 1) / kH2;
        const int pairs2 = (c_end - c_begin + 1) / 2;
        const float4* Hp = reinterpret_cast<const float4*>(fp.H + kF);  // packed-order spectrum follows the H13 table
        for (int p0 = 0; p0 < pairs2; p0 += 65535) {
            dim3 grid((unsigned)n_seg2, (unsigned)std::min(65535, pairs2 - p0));
            fir_fft_packed_kernel<<<grid, kNT, smem2, st>>>(U, u_stride, fp.hist_pad, fp.u_ring, fp.u_pos, Y, y_stride, Hp, g_tab.Wf, T, fp.divisor,
                                                           fp.post_nf, c_begin + 2 * p0, c_end);
            if (n_launches) *n_launches += 1;
        }
        return (int)cudaGetLastError();
    }
    if (!fp.fft_work) return (int)cudaErrorInvalidValue;
    const bool pc = fp.xf != nullptr;
    auto narrow = pc ? fir_fft_kernel<true> : fir_fft_kernel<false>;
    static std::atomic<bool> configured_dev[kMaxDevices][2];
    std::atomic<bool>& configured = configured_dev[current_device_slot()][pc];
    const int smem = (kPadded + kTwEntries) * (int)sizeof(float2);
    if (!configured.load(std::memory_order_acquire)) {
        cudaError_t e = cudaFuncSetAttribute(narrow, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return (int)e;
        configured.store(true, std::memory_order_release);
    }
    FftArgs g;
    g.U = U;
    g.u_stride = u_stride;
    g.u_ring = fp.u_ring;
    g.u_pos = fp.u_pos;
    g.hist = effective_taps(fp.n_taps) - 1;
    g.Y = Y;
    g.y_stride = y_stride;
    g.H13 = fp.H;
    g.Wg = g_tab.Wf;
    g.T = T;
    g.divisor = fp.divisor;
    g.post_nf = fp.post_nf;
    g.c_begin = c_begin;
    g.c_end = c_end;
    g.xf = fp.xf;
    g.h_stride = fp.h_stride;
    int n14 = 0;
    segment_plan(g.hist, T, &n14, &g.n13);
    const long long pairs = pc ? fp.n_xf : (c_end - c_begin + 1) / 2;  // per-channel taps: the table slice's transforms
    g.single_base = (long long)n14 * (2 * kF - g.hist);
    g.work = reinterpret_cast<unsigned*>(fp.fft_work);
    if (n14 > 0) {
        auto wide = pc ? fir_fft_wide_kernel<true> : fir_fft_wide_kernel<false>;
        static std::atomic<bool> wconf_dev[kMaxDevices][2];
        std::atomic<bool>& wconf = wconf_dev[current_device_slot()][pc];
        const int wsmem = (kPadW + kTwW) * (int)sizeof(float2);
        if (!wconf.load(std::memory_order_acquire)) {
            cudaError_t e = cudaFuncSetAttribute(wide, cudaFuncAttributeMaxDynamicSharedMemorySize, wsmem);
            if (e != cudaSuccess) return (int)e;
            wconf.store(true, std::memory_order_release);
        }
        WideArgs w;
        w.U = U; w.u_stride = u_stride; w.u_ring = fp.u_ring; w.u_pos = fp.u_pos; w.hist = g.hist;
        w.Y = Y; w.y_stride = y_stride;
        w.Hw = reinterpret_cast<const float4*>(fp.H + 2 * kF);
        w.Wg = g_tab.Wf;
        w.divisor = fp.divisor; w.post_nf = fp.post_nf;
        w.c_begin = c_begin; w.c_end = c_end;
        w.n14 = n14;
        w.xf = fp.xf;
        w.h_stride = fp.h_stride;
        const long long wi = pairs * n14;
        if (wi > (1ll << 30)) return (int)cudaErrorInvalidValue;
        w.n_items = (int)wi;
        w.work = g.work;
        const int wgrid = (int)std::min<long long>(wi, g_tab.n_sm);
        wide<<<wgrid, kNTW, wsmem, st>>>(w);
        if (n_launches) *n_launches += 1;
    }
    if (g.n13 > 0) {
        const long long n_items = pairs * g.n13;
        if (n_items > (1ll << 30)) return (int)cudaErrorInvalidValue;
        g.n_items = (int)n_items;
        const int grid = (int)std::min<long long>(n_items, 3 * g_tab.n_sm);
        narrow<<<grid, kNT, smem, st>>>(g);
        if (n_launches) *n_launches += 1;
    }
    return (int)cudaGetLastError();
}

// Short calls: uniformly partitioned convolution (see fir_upc_kernel).  fp.upc_* describe the FDL and the block counter.
int launch_fir_upc(const FirPlan& fp, const float* U, int64_t u_stride, float* Y, int64_t y_stride, int c_begin, int c_end, int64_t T,
                   cudaStream_t st, int* n_launches) {
    const int P = fir_upc_partitions(fp.n_taps);
    if (!P || T % kUB || !fp.upc_fdl || fp.hist_pad < P * kUB || fp.hist_pad + T > fp.u_ring) return (int)cudaErrorInvalidValue;
    int rc = ensure_tables();
    if (rc) return rc;
    const bool pc = fp.xf != nullptr;
    auto kernel = pc ? fir_upc_kernel<true> : fir_upc_kernel<false>;
    static std::atomic<bool> conf_dev[kMaxDevices][2];
    std::atomic<bool>& conf = conf_dev[current_device_slot()][pc];
    const int smem = (kUPad + kUTw) * (int)sizeof(float2);
    if (!conf.load(std::memory_order_acquire)) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return (int)e;
        conf.store(true, std::memory_order_release);
    }
    UpcArgs g;
    g.U = U; g.u_stride = u_stride; g.u_ring = fp.u_ring; g.u_pos = fp.u_pos;
    g.Y = Y; g.y_stride = y_stride;
    g.H = reinterpret_cast<const float4*>(fp.H + 4 * kF);
    g.fdl = reinterpret_cast<float4*>(fp.upc_fdl);
    g.Wg = g_tab.Wf;
    g.scale = fp.post_nf != 0.0f ? (float)((double)fp.divisor / (double)fp.post_nf) : fp.divisor;
    g.c_begin = c_begin; g.c_end = c_end;
    g.P = P; g.n_blocks = (int)(T / kUB); g.prime = fp.upc_prime;
    g.b0 = fp.upc_block0;
    g.pair0 = pc ? fp.xf0 : c_begin / 2;   // per-channel taps: delay-line slot = transform index
    g.xf = fp.xf;
    g.h_stride = fp.h_stride;
    const int pairs = pc ? fp.n_xf : (c_end - c_begin + 1) / 2;
    if (pairs <= 0) return 0;
    kernel<<<pairs, kUNT, smem, st>>>(g);
    if (n_launches) *n_launches += 1;
    return (int)cudaGetLastError();
}

int fir_prepare_spectrum(int log2F, const double* taps_rev_dev, int n_taps, int n_sets, float2* H_dev, void* stream) {
    if (log2F != kLog2F || n_taps > fir_fft_max_taps() || n_sets < 1) return (int)cudaErrorInvalidValue;
    int rc = ensure_tables();
    if (rc) return rc;
    const int smem = (kPadded + kTwEntries) * (int)sizeof(double2);
    cudaError_t e = cudaFuncSetAttribute(fir_spectrum_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return (int)e;
    cudaStream_t st = (cudaStream_t)stream;
    const long long S = 5 * kF;   // float2 elements per set: fir_fft_spectrum_bytes()
    for (int k0 = 0; k0 < n_sets; k0 += 65535) {  // gridDim.y limit: one launch per table kind and 65535 sets
        const unsigned ns = (unsigned)std::min(65535, n_sets - k0);
        const double* tr = taps_rev_dev + (size_t)k0 * n_taps;
        float2* H = H_dev + k0 * S;
        fir_spectrum_kernel<<<dim3(1, ns), kNT, smem, st>>>(tr, n_taps, g_tab.Wd, H, S);
        fir_spectrum_packed_kernel<<<dim3(kH2 / 128, ns), 128, 0, st>>>(tr, n_taps, reinterpret_cast<float4*>(H + kF), S / 2);
        fir_spectrum_wide_kernel<<<dim3(kN2 / 128, ns), 128, 0, st>>>(tr, n_taps, H + 2 * kF, S);
        if (const int P = fir_upc_partitions(n_taps))
            fir_spectrum_upc_kernel<<<dim3((P * kUF + 127) / 128, ns), 128, 0, st>>>(tr, n_taps, P, H + 4 * kF, S);
    }
    return (int)cudaGetLastError();
}

}  // namespace dspb
