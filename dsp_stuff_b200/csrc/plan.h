// plan.h — the device-side "program" a fused segment executes, shared by the host scheduler
// (engine.cpp) and the kernels (fused_chain.cu, fir_fft.cu).
//
// One fused kernel runs a straight-line program over a tile of [G channels x S samples]
// (G*S = 4096, 512 threads, 8 consecutive samples of one channel per thread).  The program is an
// accumulator machine: `acc` is the thread's 8 samples in registers; other live values sit in
// thread-private shared-memory "vregs" or in global scratch.  Recurrences (biquad, one-pole,
// envelope) run lane = channel, strictly sequential in time, so they are bit-identical to the
// reference arithmetic (DESIGN.md "IIR exactness").
#pragma once
#include <cuda_runtime.h>

#include <cstdint>

namespace dspb {

// slot of sample (pos + i) in a ring of R samples; pos in [0, R), i in [-R, R)
__host__ __device__ inline int ring_slot(int pos, int i, int R) {
    int p = pos + i;
    if (p < 0) p += R;
    if (p >= R) p -= R;
    return p;
}

// Launch-time caches (cudaFuncSetAttribute opt-ins, SM counts, register counts, twiddle tables) are PER DEVICE:
// one process may hold engines on several GPUs (include/dspb200.h), and a function attribute set on device 0 says
// nothing about device 1.  Every such cache is an array indexed by the current device ordinal.
constexpr int kMaxDevices = 64;
inline int current_device_slot() {
    int d = 0;
    cudaGetDevice(&d);
    return (d < 0 || d >= kMaxDevices) ? 0 : d;
}

constexpr int kThreads = 512;       // elementwise threads per CTA
constexpr int kChunk = 8;           // consecutive samples per thread (8: twice the warps of 16 for latency hiding)
constexpr int kTile = kThreads * kChunk;  // 4096 samples per CTA tile
constexpr int kRefBlock = 128;      // node.rs:257 BUF_SIZE
constexpr int kMaxOps = 48;
constexpr int kMaxBufs = 12;
constexpr int kMaxRings = 6;
constexpr int kMaxStates = 12;
constexpr int kMaxPrefetch = 2;
constexpr int kMaxScan = 4;         // recurrences of one fused segment that may run as a time-parallel scan

enum OpCode : uint8_t {
    OP_END = 0,
    OP_NOP,        // only the fan-in prologue (pre) runs
    OP_ZERO,       // acc = 0
    OP_LOADG,      // acc = 0.0f + G[buf]           (first link of a fan-in sum, node.rs:181-183)
    OP_ADDG,       // acc = acc + G[buf]
    OP_LOADV,      // acc = 0.0f + V[vreg]
    OP_ADDV,       // acc = acc + V[vreg]
    OP_COPYV,      // acc = V[vreg]                 (plain reload, no +0)
    OP_COPYG,      // acc = G[buf]
    OP_DIVC,       // (lowering only: folded into the next op's `pre`) acc = acc / p0, node.rs:189-191
    OP_SAVEV,      // V[vreg] = acc
    OP_STOREG,     // G[buf] = acc
    OP_MODMAP,     // acc = p0 + (p1-p0)*clamp((acc+1)/2,0,1)   (lib.rs:138-146)
    OP_GAIN,       // acc = acc * P0
    OP_DISTORT,    // mode in `mode`; level P0      (nodes/distort.rs)
    OP_OVERDRIVE,  // boost P0, drive P1, level P2  (nodes/overdrive.rs:31-43)
    OP_CHEBY,      // p0 level_pos, p1 level_neg, p2 tanh(level_pos), p3 tanh(level_neg)
    OP_ADD,        // acc = acc + V[vreg]           (nodes/add.rs: a + b, acc = a)
    OP_MIX,        // acc = V[vreg]*r + acc*(1-r), r = P0 (nodes/mix.rs:45; acc = a, vreg = b)
    OP_COMB,       // acc = acc + ring*p0 ; ring = acc      (nodes/reverb.rs:87-103), ring index `aux`
    OP_BIQUAD,     // exact DF1, coefs p0..p3 = b0,b1,b2,a1 and Op::a2; state slot `aux`
    OP_LP1,        // y = x*p1 + p0*z ; z = y  (p0 = ratio, p1 = 1-ratio), state slot `aux`
    OP_HP1,        // z = x*p1 + p0*z ; y = x - z
    OP_ENVELOPE,   // p0 attack gain, p1 release gain, state slot `aux`
    OP_SIGGEN,     // mode; amplitude P0, frequency P1; p2 = sample rate; state slot `aux`
    OP_GATE,       // EXTENSION (no reference node): acc = acc >= p0 ? V[vreg] : 0   (acc = envelope, vreg = the signal)
};

// Parameter source flags: bit i set => parameter Pi is a per-sample tile read from vreg pv[i]
// (a connected `as_input` control port), else the scalar p[i].
// Time-parallel ("scan") evaluation of a linear recurrence y[n] = p[n] - a1 y[n-1] - a2 y[n-2] (opt-in, NOT bit-exact:
// dspb_config::iir_mode).  State s[n] = (y[n], y[n-1]) obeys s[n] = A s[n-1] + (p[n], 0), A = [[-a1, -a2], [1, 0]].
// A thread owns kChunk = 8 consecutive samples; P[i] = A^(8 * 2^i) (row-major 2x2, f64) are the strides of the Kogge-Stone
// scan over the lanes of a warp (i = 0..4) and over warps (i = 5: A^256).
struct ScanTab {
    double P[6][4];    // f64: the carried states are computed in double (plain DFMA, half the FP32 rate on B200), so the scan
                       // itself adds ~1e-7; what is left against the reference is the reference's own f32 rounding
    float a1, a2;
    float probe_err;   // measured at dspb_compile: max |scan - exact| / max |exact| on the probe signal
    float pad_;
};

struct Op {
    uint8_t code;
    uint8_t mode;     // DISTORT / SIGGEN: variant.  BIQUAD / LP1 / HP1: 0 = exact sequential evaluation, k > 0 = scan, table k - 1
    uint8_t pflags;
    uint8_t vreg;     // operand vreg for LOADV/ADDV/SAVEV/ADD/MIX
    uint8_t pv[3];    // vregs of tile-valued parameters
    uint8_t buf;      // global buffer index for LOADG/ADDG/STOREG, prefetch slot + 1 in `aux`
    uint16_t aux;     // ring / state slot, or prefetch slot (0 = none, k+1 = slot k)
    uint8_t pad;      // bits 0-1: DivTier of the op's own constant divisor p[0] (Distort level): p[1] = RN(1/p[0]) when
                      // DIV_MARKSTEIN, p[1], p[2] = zh, zl when DIV_MULFMA;
                      // bits 2-7: per-channel parameters, 1 + the column of this op's first value in Program::pc (0 = shared)
    uint8_t pre;      // fan-in prologue folded into this op: 1 = acc = 0.0 + acc; 2 = acc /= p[4]; bits 2-3: DivTier of
                      // that division (4: p[5] = RN(1/p[4]); 8: p[5], p[6] = zh, zl)
    float p[7];       // p[4], p[5], p[6]: fan-in divisor and its reciprocal or zh, zl when pre & 2
    float a2;         // biquad: a2 (p[0..3] = b0, b1, b2, a1)
};
// How a constant division runs (exact_math.cuh); the host picks the first tier whose exhaustive device check passes.
enum DivTier { DIV_IEEE = 0, DIV_MARKSTEIN = 1, DIV_MULFMA = 2 };
__host__ __device__ inline int op_div_tier(const Op& o) { return o.pad & 3; }
__host__ __device__ inline constexpr int pre_div_tier(int pre) { return (pre >> 2) & 3; }

// Per-channel parameters (dspb_node_set_f32_channels).  An op whose `pad >> 2` is k > 0 reads its parameters from row `ch`
// (the ABSOLUTE channel) of the step's table Program::pc, columns k-1 ... k-2+op_pc_cols(code), in this order: p[0], p[1],
// ... and, for the biquad, a2 last.  Everything else (fan-in divisor, sample rate, control-port tiles) stays in the Op.
constexpr int kMaxPcCols = 32;      // columns of one step's table (a segment that needs more is cut)
__host__ __device__ inline constexpr int op_pc_cols(int code) {
    return code == OP_BIQUAD ? 5 : code == OP_CHEBY ? 4 : code == OP_OVERDRIVE ? 3
         : (code == OP_LP1 || code == OP_HP1 || code == OP_ENVELOPE || code == OP_SIGGEN) ? 2
         : (code == OP_GAIN || code == OP_DISTORT || code == OP_MIX || code == OP_COMB || code == OP_GATE) ? 1 : 0;
}
__host__ __device__ inline int op_pc_col(const Op& o) { return (o.pad >> 2) - 1; }  // -1: shared parameters

// Does an op of this code read the shared-memory vreg named by Op::vreg?  (SAVEV writes it; parameter tiles are in pv[].)
inline constexpr bool op_reads_vreg_field(int code) {
    return code == OP_LOADV || code == OP_ADDV || code == OP_COPYV || code == OP_ADD || code == OP_MIX || code == OP_GATE;
}

struct BufDesc {       // a [C x n] f32 array in global memory
    float* base;       // element (channel 0, sample 0 of this call); ring_len != 0: element (channel 0, ring slot 0)
    int64_t row_stride;
    // ring_len != 0: every row is a ring of ring_len samples (a multiple of 128) and this call's sample m lives at
    // slot (ring_pos + m) mod ring_len.  Used for the FIR input U, so that a call's last N-1 samples are the next
    // call's history without any copy.  ring_pos is a multiple of 128: an aligned 8-sample chunk never wraps.
    int32_t ring_len;
    int32_t ring_pos;
};

struct RingDesc {      // Reverb ring, [C x D] f32
    float* base;
    int64_t D;         // delay length in samples (bit-exact index work)
    int64_t pos;       // slot of this call's sample 0
};

struct Program {
    int32_t n_ops;
    int32_t n_vregs;       // shared-memory vregs (16 KB each); vreg ids >= n_vregs do not exist
    int32_t n_prefetch;    // cp.async staging slots in use
    int32_t needs_tile;    // program has lane=channel recurrences (transposition tile in smem)
    Op ops[kMaxOps];
    BufDesc bufs[kMaxBufs];
    RingDesc rings[kMaxRings];
    float* states[kMaxStates];  // [C x 4] f32 per stateful op
    // prefetch slot k stages global buffer pf_buf[k] (>=0) or ring pf_ring[k] (>=0)
    int16_t pf_buf[kMaxPrefetch];
    int16_t pf_ring[kMaxPrefetch];
    int16_t st_buf;        // buffer of the first STOREG (its op has aux = 1): row pointer kept in a register, or -1
    int16_t n_scan;        // scan tables in use
    ScanTab scan[kMaxScan];
    const float* pc;       // per-channel parameter table [C x pc_stride] f32, row = absolute channel (null: none)
    int64_t pc_stride;
};
// passed by value as a kernel parameter (__grid_constant__): keep it well inside the 4 KB parameter space
static_assert(sizeof(Program) <= 4096, "Program must stay a kernel parameter");

// ---- launchers (defined in the .cu files) -----------------------------------------------------------
// Runs `prog` for channels [c_begin, c_end) and samples [0, T) of this call.  G in {1,2,4,8,16,32}.
int launch_fused(const Program& prog, int G, int c_begin, int c_end, int64_t T, void* stream);
int fused_smem_bytes(const Program& prog, int G);
// Enumerates all 2^32 dividends on the device; *mismatches == 0 proves div_const exact for divisor b.
int verify_const_div(float b, float r, unsigned long long* mismatches);
// The same for div_const2 with zh, zl (exact_math.cuh ConstDiv2) under its own acceptance rule.
int verify_const_div2(float b, float zh, float zl, unsigned long long* mismatches);
// Runs a one-recurrence probe program in exact and in scan mode on the device (noise + log sweep, 16384 samples) and
// returns max |scan - exact| / max |exact|: the measured error that gates scan mode for one coefficient set.
int measure_scan_error(const Op& exact_op, const ScanTab& tab, float* rel_err);

enum FirMode { FIR_FFT = 0, FIR_DIRECT = 1, FIR_TOEPLITZ = 2, FIR_FFT_PACKED = 3 };
struct FirPlan {
    int mode;             // FIR_FFT: overlap-save FFT (f32); FIR_DIRECT: time domain, f64, reference summation order;
                          // FIR_TOEPLITZ: Toeplitz-tiled tcgen05 GEMM, split bf16 (fir_toeplitz.cu);
                          // FIR_FFT_PACKED: the FFT path with two sub-transforms per f32x2 register pair (experiment)
    int log2F;            // FFT size F = 1 << log2F complex points, two channels per transform
    int n_taps;           // N
    int hist_pad;         // history samples kept in U before this call's sample 0 (>= N-1, multiple of 4)
    int u_ring;           // U rows are rings of u_ring samples (multiple of 128, >= hist_pad + T): sample i of this call
    int u_pos;            // (i in [-hist_pad, T)) lives at slot (u_pos + i) mod u_ring
    void* fft_work;       // FIR_FFT: this launch lane's work counters of the persistent kernels (fir_fft_work_bytes())
    // FIR_FFT, short calls: uniformly partitioned convolution (fir_fft.cu fir_upc_kernel)
    void* upc_fdl = nullptr;      // frequency-domain delay line [pairs][P][2048] float2, or null: not eligible
    int upc_prime = 0;            // previous blocks whose spectra must be recomputed from the ring first (0 .. P - 1)
    long long upc_block0 = 0;     // running block counter of this call's first block
    const float2* H;      // [2F] spectrum of h pre-scaled by 1/F: [0, F) in the scalar kernel's output order, then F/2 float4
                          // (even bin, odd bin) pairs in the packed kernel's order
    const double* taps;   // [N] reversed taps (f64) for the warm-up path
    float divisor;        // 1/N (Average) or 1 (Balanced), fir.rs:187-190
    float post_nf;        // != 0: epilogue y = (0.0 + y) / post_nf, the fan-in average of a sink fed only by this node
    // FIR_TOEPLITZ only: pre-built Toeplitz tiles of the tap set, scratch for the hi/lo bf16 split of U, and the
    // max_samples the scratch was sized for
    const void* toep_tiles = nullptr;
    void* toep_split = nullptr;
    int64_t toep_max_samples = 0;
    // Per-channel impulse responses (dspb_node_set_taps_channels), FIR_FFT and FIR_DIRECT only; all null / zero when the
    // taps are shared.  Set k's spectra start at H + k * h_stride and its reversed taps at taps + k * n_taps.
    const int* set_index = nullptr;  // [C] set of each (absolute) channel: the direct kernel
    const int4* xf = nullptr;        // this launch's slice of the transform table: {chA, chB or -1, set, 0} per transform
    int n_xf = 0;                    // transforms in the slice (channels [c_begin, c_end) are exactly theirs)
    int xf0 = 0;                     // index of the slice's first transform in the whole table (UPC delay-line slot)
    int64_t h_stride = 0;            // float2 elements per set in H (fir_fft_spectrum_bytes() / 8)
    // Channels reset by dspb_reset_channels that are still in their own warm-up while the node is past it at their position:
    // {channel, samples since that channel's reset}, ascending channels, all inside [c_begin, c_end).  The direct kernel
    // recomputes samples [0, min(T, N - 1 - started)) of each of them after the main launch; warm_len = the longest of those.
    const int2* warm = nullptr;
    int n_warm = 0;
    int warm_len = 0;
};
// U: [C x u_ring] input rings (see FirPlan::u_ring / u_pos), u_stride = row pitch; Y: [C x T] output.
// started = samples seen before this call.
int launch_fir(const FirPlan& fp, const float* U, int64_t u_stride, float* Y, int64_t y_stride, int c_begin, int c_end,
               int64_t T, int64_t started, void* stream, int* n_launches);
// Computes H from the (device-resident, reversed, f64) taps with the kernel's own forward passes in f64.  n_sets tap sets
// stored one after the other ([n_sets x n_taps]) give n_sets spectra, set k at H_dev + k * fir_fft_spectrum_bytes() / 8,
// in one launch per table kind.
int fir_prepare_spectrum(int log2F, const double* taps_rev_dev, int n_taps, int n_sets, float2* H_dev, void* stream);
int fir_fft_max_taps();
size_t fir_fft_spectrum_bytes();   // H buffer of one tap set (all spectrum tables of the FFT kernels)
size_t fir_fft_work_bytes();       // one launch lane's work area (the persistent kernels' work counters, zeroed once)
int fir_upc_partitions(int n_taps);                      // 1024-tap partitions of the UPC kernel, 0 = impulse response too long
size_t fir_upc_fdl_bytes(int n_taps, int transforms);     // delay line of `transforms` channel pairs (shared taps: ceil(C / 2))
constexpr int kUpcBlock = 1024;
// device-boundary format steps (boundary.cu): stereo fold a + b, mono -> stereo duplicate; flat [C * n] streams
int launch_fold_stereo(const float* interleaved, float* mono, long long total_mono, cudaStream_t st);
int launch_dup_stereo(const float* mono, float* interleaved, long long total_mono, cudaStream_t st);
// 48 kHz -> device-rate sinc converter + duplicate (boundary.cu): meta = int2 per output frame {frames pushed so far in this
// call, Sinc::idx}, w = 16 f64 window weights per output frame (left tap n, right tap n interleaved)
int launch_resample_dup(const float* mono, long long n_in, const float* hist_old, float* hist_new, const void* meta, const double* w,
                        float* interleaved, long long n_out, long long pushed, int channels, cudaStream_t st);
// Toeplitz tensor-core path (fir_toeplitz.cu): buffer sizes, tile construction for one tap set
int fir_toeplitz_max_taps();
size_t fir_toeplitz_tiles_bytes(int n_taps);
size_t fir_toeplitz_split_bytes(int n_taps, int channels, int64_t max_samples);
int fir_toeplitz_prepare(const double* taps_rev_dev, int n_taps, void* tiles_dev, void* stream);

// Per-channel state reset (reset.cu).  One state buffer of the graph: rows of `pitch` f32 from `base`; a listed channel's
// slots (first + i) mod ring, i in [0, len), are zeroed (a [C x 4] state row or a reverb ring: first 0, len = ring = row).
struct ClearDesc {
    float* base;
    int64_t pitch;
    int64_t first, len, ring;
};
// Zeroes those slots of every (channel, descriptor) pair in one launch; descs and channels are device arrays.
int launch_clear_rows(const ClearDesc* descs, int n_descs, const int* channels, int n_channels, void* stream);

}  // namespace dspb
