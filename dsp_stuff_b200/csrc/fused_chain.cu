// fused_chain.cu — the fused effect-segment kernel (sm_100a).
//
// One launch runs a whole fused segment of the node graph (every node except Fir) for a range of
// channels over all samples of the call.  Replaces, for those nodes, the reference's per-node task
// loop + SimpleNode::process bodies (dsp-stuff/src/node.rs:267-352, nodes/*.rs).
//
// Geometry: a CTA owns G channels for the whole call and walks time in tiles of S = 4096/G samples,
// so every sequential dependency (IIR state, comb ring, Fuzz 128-sample blocks) stays inside one
// CTA.  512 elementwise threads; thread (g, j) holds 8 consecutive samples of channel g in registers (`acc`).
// HBM traffic is 128-bit per thread; the next tile's input and ring chunks are prefetched one tile ahead
// straight into registers.  Three kernels share the op code below:
//   fused_kernel      any program (run-time interpreter or a compile-time chain), recurrences in place
//   fused_kernel_ws   one recurrence: warp-specialised pipeline (elementwise warps + one recurrence warp)
//   fused_kernel_ws2  two recurrences in series: two recurrence warps, three-phase pipeline
//
// Recurrences (biquad / one-pole / envelope) are bit-identical to the reference: everything that
// does not depend on the previous OUTPUT (the feed-forward taps) is computed time-parallel with the
// reference's operation order, then one warp runs the remaining 2-4 dependent f32 ops per sample
// lane = channel, strictly in time order, on a conflict-free transposed tile in shared memory.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "exact_math.cuh"
#include "plan.h"

namespace dspb {
namespace {

// distort.rs:53-61
__device__ __forceinline__ float clipf(float s) { return s < -1.0f ? -1.0f : (s > 1.0f ? 1.0f : s); }
// f32::signum: NaN -> NaN, else copysign(1, x)
__device__ __forceinline__ float signumf(float x) { return x != x ? x : copysignf(1.0f, x); }
__device__ __forceinline__ float clamp01(float x) { return x < 0.0f ? 0.0f : (x > 1.0f ? 1.0f : x); }

constexpr int kF4 = kChunk / 4;            // float4s per thread chunk
constexpr int kBlk = kRefBlock / kChunk;    // threads per 128-sample reference block
static_assert(kF4 == 2 || kF4 == 4, "swizzles below are written for 8 or 16 samples per thread");
// swizzle of a thread's float4 slots inside a transposed tile row (conflict-free for 8 consecutive lanes)
__device__ __forceinline__ int sw_of(int j) { return kF4 == 4 ? ((j >> 1) & 3) : ((j >> 2) & 1); }

enum DistortMode { HardClip, SoftClip, Tanh, RecipSoftClip, Fuzz, Sin, Atan, Square, Chebyshev4 };

// Per-sample level (control port connected): kept out of line so the rare path costs no registers.
__device__ __noinline__ float shape_generic(int mode, float x, float l) {
    if (l < 0.001f) return x;
    switch (mode) {
        case HardClip: return dv(clipf(mul(x, l)), l);
        case SoftClip: {
            float s = mul(x, l);
            if (s > 1.0f) s = 2.0f / 3.0f;
            else if (s >= -1.0f && s <= 1.0f) s = sub(s, dv(mul(mul(s, s), s), 3.0f));
            else s = -2.0f / 3.0f;
            return dv(clipf(s), l);
        }
        case Tanh: return tanhf(mul(x, l));
        case RecipSoftClip: return mul(signumf(x), sub(1.0f, dv(1.0f, add(mul(fabsf(x), l), 1.0f))));
        case Sin: return sinf(mul(x, l));
        case Atan: return atanf(mul(x, l));
        case Square: { float v = mul(x, l); return mul(mul(v, v), signumf(v)); }
        case Chebyshev4: {
            float v2 = mul(x, l);
            v2 = mul(v2, v2);
            return add(sub(mul(8.0f, mul(v2, v2)), mul(8.0f, v2)), 1.0f);
        }
    }
    return x;
}
__device__ __noinline__ float overdrive_generic(float x, float b, float dr, float l) {  // overdrive.rs:31-43
    if (l < 0.001f) return x;
    const float FRAC_PI_4 = 0.785398163397448309615660845819875721f;
    const float FRAC_2_PI = 0.636619772367581343075535053490057448f;
    float d = mul(FRAC_2_PI, atanf(mul(FRAC_PI_4, mul(x, b))));
    return mul(add(mul(dr, d), mul(sub(1.0f, dr), x)), l);
}

// max over the kBlk consecutive threads (= one 128-sample reference block) of |v| under
// f32::total_cmp: non-negative floats and NaNs order like their bit patterns.
__device__ __forceinline__ float block128_max_abs(const float (&v)[kChunk]) {
    unsigned m = 0;
#pragma unroll
    for (int i = 0; i < kChunk; i++) m = max(m, __float_as_uint(fabsf(v[i])));
#pragma unroll
    for (int d = 1; d < kBlk; d <<= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, d));
    return __uint_as_float(m);
}

__device__ __forceinline__ float4 ldg_stream(const float4* p) {
    float4 r;
    asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
    return r;
}
// Prefetch flavour: the "memory" clobber pins the load where it is written.  Without it the compiler sinks
// the load down to its first use in the NEXT tile iteration (measured: a full DRAM round trip per tile).
// The outputs ARE the prefetch registers: going through a temporary float4 makes the compiler emit MOVs
// right behind the load, which stall on it at once (measured: prefetching was slower than not prefetching).
__device__ __forceinline__ void ldg_prefetch(const float4* p, float& a, float& b, float& c, float& d) {
    asm volatile("ld.global.cg.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(a), "=f"(b), "=f"(c), "=f"(d) : "l"(p) : "memory");
}
__device__ __forceinline__ void stg_stream(float4* p, float4 v) {
    asm volatile("st.global.cg.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

// ---- sequential cores: only the ops that depend on the previous output ---------------------------------
struct DF1Core {  // y = (p - a1*y1) - a2*y2, p = b0*x + b1*x1 + b2*x2 precomputed (biquad 0.4.2 DirectForm1::run)
    float a1, a2, y1, y2;
    __device__ __forceinline__ void from_row(const float* r) { a1 = r[3]; a2 = r[4]; }  // per-channel table: b0 b1 b2 a1 a2
    __device__ __forceinline__ void load(const float4 s) { y1 = s.z; y2 = s.w; }
    __device__ __forceinline__ void save(float4& s) const { s.z = y1; s.w = y2; }
    __device__ __forceinline__ float step(float p) {
        float out = sub(sub(p, mul(a1, y1)), mul(a2, y2));
        y2 = y1; y1 = out;
        return out;
    }
};
struct OnePoleCore {  // z = xr + r*z, xr = x*(1-r) precomputed (nodes/low_pass.rs:37, high_pass.rs:37)
    float r, z;
    __device__ __forceinline__ void from_row(const float* row) { r = row[0]; }  // per-channel table: ratio, 1 - ratio
    __device__ __forceinline__ void load(const float4 s) { z = s.x; }
    __device__ __forceinline__ void save(float4& s) const { s.x = z; }
    __device__ __forceinline__ float step(float xr) { z = add(xr, mul(r, z)); return z; }
};
struct EnvCore {  // dasp_envelope 0.11.0 Detector<f32, Peak<FullWave>>::next, d = |x| precomputed
    float ga, gr, prev;
    __device__ __forceinline__ void from_row(const float* r) { ga = r[0]; gr = r[1]; }
    __device__ __forceinline__ void load(const float4 s) { prev = s.x; }
    __device__ __forceinline__ void save(float4& s) const { s.x = prev; }
    __device__ __forceinline__ float step(float d) {
        float g = prev < d ? ga : gr;
        prev = add(d, mul(sub(prev, d), g));
        return prev;
    }
};

// Swizzled float4 slot of logical float4 index m inside a tile row: thread j writes its four
// float4s to 4j + (k ^ ((j>>1)&3)), which makes both the time-parallel accesses (8 lanes, stride 64 B)
// and the lane = channel accesses (rows padded by 4 floats) bank-conflict free.
__device__ __forceinline__ int swz(int m) { return (m & ~(kF4 - 1)) | ((m & (kF4 - 1)) ^ sw_of(m / kF4)); }


// Sequential feedback loop over one tile row (lane = channel): `valid_f4` float4s at swizzled slots.  Loads run two
// float4s ahead of their use.  valid_f4 is a multiple of 32 (calls are multiples of 128 samples), so the row is walked in
// blocks of 16 float4s -- one period of the swizzle -- with compile-time slot offsets: the loop body is nothing but
// LDS.128, the dependent f32 chain and STS.128 (303 instructions per 64 samples, 256 of them the FMUL / FADD chain).
// The recurrence warps set the pace of the whole launch: every channel is in flight at once, one lane per channel, so a
// call cannot finish before n x (cycles per recurrence step), and next to the elementwise warps on its scheduler a
// recurrence warp gets an issue slot only every ~8 cycles (ncu r02: ~37 cycles per step against 14 alone; the elementwise
// warps wait at the DONE barrier).  Every instruction it does not issue counts: the generic index arithmetic and clamps
// were a quarter of its instructions (fused step 0.513 -> 0.464 ms at 4096 x 24576 without them).
__host__ __device__ constexpr int swz_c(int m) { return (m & ~(kF4 - 1)) | ((m & (kF4 - 1)) ^ (kF4 == 4 ? ((m / kF4 >> 1) & 3) : ((m / kF4 >> 2) & 1))); }
template <class Core>
__device__ __forceinline__ void recurrence_row(Core& core, float4* r, int valid_f4) {
    float4 a = r[swz_c(0)];
    float4 b = r[swz_c(1)];
#pragma unroll 1
    for (int q = 0; q < valid_f4; q += 16) {
        float4* rq = r + q;
        const bool more = q + 16 < valid_f4;
#pragma unroll
        for (int i = 0; i < 16; i++) {
            float4 nxt = b;
            if (i < 14) nxt = rq[swz_c(i + 2)];
            else if (more) nxt = rq[swz_c(i + 2)];   // 16 + swz_c(i - 14): the first slots of the next block
            float4 x = a;
            x.x = core.step(x.x);
            x.y = core.step(x.y);
            x.z = core.step(x.z);
            x.w = core.step(x.w);
            rq[swz_c(i)] = x;
            a = b;
            b = nxt;
        }
    }
}

template <int G>
struct Geo {
    static constexpr int S = kTile / G;        // samples per channel per tile
    static constexpr int TPC = kThreads / G;   // threads per channel
    static constexpr int ROW = S + 4;          // padded tile row (floats)
};

struct TileCtx {
    float* tile;
    int g, j, valid_f4, rec_warp;
};

// v (time-parallel, 16 per thread) -> tile; one warp runs `core` lane = channel; tile -> v.
// pcr != null: per-channel coefficients, the op's columns of table row 0; lane l takes row ch0 + l (ch0: the CTA's first channel).
template <int G, class Core>
__device__ __forceinline__ void run_recurrence(Core core, float (&v)[kChunk], const TileCtx& c, float4* st,
                                               const float* pcr = nullptr, long long pc_stride = 0, int ch0 = 0) {
    using Q = Geo<G>;
    float4* row = reinterpret_cast<float4*>(c.tile + c.g * Q::ROW);
#pragma unroll
    for (int k = 0; k < kF4; k++)
        row[kF4 * c.j + (k ^ sw_of(c.j))] = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    if ((threadIdx.x >> 5) == c.rec_warp && lane < G && c.valid_f4 > 0) {  // strictly sequential in time
        float4* r = reinterpret_cast<float4*>(c.tile + lane * Q::ROW);
        if (pcr) core.from_row(pcr + (long long)(ch0 + lane) * pc_stride);
        float4 s = st[lane];
        core.load(s);
        recurrence_row(core, r, c.valid_f4);
        core.save(s);
        st[lane] = s;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kF4; k++) {
        float4 q = row[kF4 * c.j + (k ^ sw_of(c.j))];
        v[4 * k] = q.x; v[4 * k + 1] = q.y; v[4 * k + 2] = q.z; v[4 * k + 3] = q.w;
    }
}

// Time-parallel evaluation of y[n] = p[n] - a1 y[n-1] - a2 y[n-2] over one tile (opt-in, dspb_config::iir_mode = 1; see
// plan.h ScanTab).  v holds this thread's 8 values of p on entry and of y on exit.  (1) every thread runs its chunk from a
// zero state: the chunk's end state e; (2) Kogge-Stone scan of the end states over the lanes of the channel with the
// strides A^(8 d), the state carried in from the previous tile (or from the warps in front) entering at lane 0;
// (3) every thread re-runs its chunk from its true start state.  Steps (1) and (2) run in f64, step (3) in f32 with FMA:
// the result is closer to exact filtering than the reference's own f32 evaluation, and it is NOT the reference's rounding.
// ONEPOLE: the state is the single value z, kept in .x like the exact path keeps it (a ratio change may flip a filter between
// the two evaluations without touching its state); else (y1, y2) in .z / .w.
template <int G, bool ONEPOLE>
__device__ __forceinline__ void scan_recurrence(const ScanTab& tab, float (&v)[kChunk], const TileCtx& tc, int j_last, float4* st,
                                                double2* wend) {
    constexpr int TPC = Geo<G>::TPC;
    constexpr int W = TPC < 32 ? TPC : 32;   // lanes of one channel inside a warp
    constexpr int NW = TPC / W;              // warps per channel
    const double a1 = tab.a1, a2 = tab.a2;
    const int li = tc.j % W, wi = tc.j / W;
    double e1 = 0.0, e2 = 0.0;
#pragma unroll
    for (int i = 0; i < kChunk; i++) {
        const double y = fma(-a1, e1, fma(-a2, e2, (double)v[i]));
        e2 = e1; e1 = y;
    }
    double c1 = ONEPOLE ? st[tc.g].x : st[tc.g].z, c2 = ONEPOLE ? 0.0f : st[tc.g].w;  // carried in from the previous tile
    auto scan = [&](double s1, double s2) {
#pragma unroll
        for (int i = 0, d = 1; d < W; i++, d <<= 1) {
            const double u1 = __shfl_up_sync(0xffffffffu, s1, d, W), u2 = __shfl_up_sync(0xffffffffu, s2, d, W);
            if (li >= d) {
                s1 = fma(tab.P[i][0], u1, fma(tab.P[i][1], u2, s1));
                s2 = fma(tab.P[i][2], u1, fma(tab.P[i][3], u2, s2));
            }
        }
        return make_double2(s1, s2);
    };
    if constexpr (NW > 1) {
        const double2 z = scan(e1, e2);                // zero carry-in: the warp's own contribution
        if (li == W - 1) wend[tc.g * NW + wi] = z;
        __syncthreads();
        for (int w = 0; w < wi; w++) {                 // carry into this warp: c <- E_w + A^256 c
            const double2 E = wend[tc.g * NW + w];
            const double n1 = fma(tab.P[5][0], c1, fma(tab.P[5][1], c2, E.x));
            const double n2 = fma(tab.P[5][2], c1, fma(tab.P[5][3], c2, E.y));
            c1 = n1; c2 = n2;
        }
    }
    double s1 = e1, s2 = e2;
    if (li == 0) {  // the carry enters at lane 0: its chunk end becomes e + A^8 c
        s1 = fma(tab.P[0][0], c1, fma(tab.P[0][1], c2, e1));
        s2 = fma(tab.P[0][2], c1, fma(tab.P[0][3], c2, e2));
    }
    const double2 S = scan(s1, s2);                    // true end state of every chunk
    double q1 = __shfl_up_sync(0xffffffffu, S.x, 1, W), q2 = __shfl_up_sync(0xffffffffu, S.y, 1, W);
    if (li == 0) { q1 = c1; q2 = c2; }
    float p1 = (float)q1, p2 = (float)q2;
    const float fa1 = tab.a1, fa2 = tab.a2;
#pragma unroll
    for (int i = 0; i < kChunk; i++) {
        const float y = fmaf(-fa1, p1, fmaf(-fa2, p2, v[i]));
        p2 = p1; p1 = y;
        v[i] = y;
    }
    // every thread of the channel has read st by now (NW > 1: the barrier above; else one warp: __syncwarp)
    if constexpr (NW == 1) __syncwarp();
    if (tc.j == j_last) {
        if constexpr (ONEPOLE) st[tc.g].x = (float)S.x;
        else { st[tc.g].z = (float)S.x; st[tc.g].w = (float)S.y; }
    }
    if constexpr (NW > 1) __syncthreads();  // wend is free again (the next scan op of this tile rewrites it)
}

__device__ __forceinline__ void load16(const float4* s, int stride, float (&v)[kChunk]) {
#pragma unroll
    for (int k = 0; k < kF4; k++) {
        float4 q = s[k * stride];
        v[4 * k] = q.x; v[4 * k + 1] = q.y; v[4 * k + 2] = q.z; v[4 * k + 3] = q.w;
    }
}
__device__ __forceinline__ void store16(float4* s, int stride, const float (&v)[kChunk]) {
#pragma unroll
    for (int k = 0; k < kF4; k++) s[k * stride] = make_float4(v[4 * k], v[4 * k + 1], v[4 * k + 2], v[4 * k + 3]);
}

// acc[i] = (add0 ? 0.0 + acc[i] : acc[i]) / b for a host-known divisor b, in the tier the host verified for it (plan.h
// DivTier; z1, z2 = r or zh, zl).  The fast forms are exact wherever their guard accepts the chunk; a chunk with zeros,
// denormal-range or huge values takes IEEE division.  div_const2 accepts only chunks without zeros, where 0.0 + a == a bit
// for bit, so the fan-in's zero-add is left to the fallback; the Markstein and IEEE tiers add first, as the reference does.
__device__ __forceinline__ void div_chunk(float (&acc)[kChunk], float b, float z1, float z2, int tier, bool add0) {
    if (tier == DIV_MULFMA) {
        float q[kChunk];
        float mn = kDiv2Hi, mx = 0.0f;
#pragma unroll
        for (int i = 0; i < kChunk; i++) q[i] = div_const2(acc[i], ConstDiv2{z1, z2}, mn, mx);
        if (div_const2_accept(mn, mx)) {
#pragma unroll
            for (int i = 0; i < kChunk; i++) acc[i] = q[i];
            return;
        }
    }
    if (add0) {
#pragma unroll
        for (int i = 0; i < kChunk; i++) acc[i] = add(0.0f, acc[i]);
    }
    if (tier == DIV_MARKSTEIN) {
        float q[kChunk];
        float mn = kDivHi, mx = 0.0f;
#pragma unroll
        for (int i = 0; i < kChunk; i++) q[i] = div_const(acc[i], ConstDiv{b, z1}, mn, mx);
        if (div_const_accept(mn, mx)) {
#pragma unroll
            for (int i = 0; i < kChunk; i++) acc[i] = q[i];
            return;
        }
    }
#pragma unroll
    for (int i = 0; i < kChunk; i++) acc[i] = dv(acc[i], b);
}
// The fan-in prologue folded into an op (plan.h Op::pre): acc = 0.0 + acc (pre & 1), acc /= p[4] (pre & 2).
__device__ __forceinline__ void fanin_prologue(float (&acc)[kChunk], int pre, const Op& op) {
    if (pre & 2) {
        div_chunk(acc, op.p[4], op.p[5], op.p[6], pre_div_tier(pre), pre & 1);
    } else if (pre & 1) {
#pragma unroll
        for (int i = 0; i < kChunk; i++) acc[i] = add(0.0f, acc[i]);
    }
}

// Per-CTA / per-tile context shared by every op.
template <int G>
struct Ctx {
    const Program* prog;
    float4* sm_state;
    float2* edge;
    double2* wend;  // [kThreads / 32] zero-carry end states of the warps (scan mode, channels wider than one warp)
    float4* stage;
    float4* vregs;
    TileCtx tc;
    int n0, tile_i, n_tiles, T;  // samples per call < 2^31 (checked by the launcher)
    int t, g, j, ch, j_last;
    bool ch_ok, active;
    // Loop-carried addressing of the three streams every tile touches (prefetched input, prefetched ring,
    // first stored output): row pointers are computed once per thread, the ring slot advances by S with a
    // compare-and-subtract.  Recomputing them from the tile index cost ~150 of the ~800 instructions a thread
    // spent per tile (64-bit multiplies and two 32-bit modulo sequences).
    const float* in_row;
    float* out_row;
    float* ring_row;
    int ring_D;
    int out_ring, out_pos;  // the first stored output is a ring-addressed FIR input (BufDesc::ring_len / ring_pos), or 0
    mutable int ring_slot;  // this thread's ring slot of the tile whose comb runs next

    template <class P>
    __device__ __forceinline__ void init_streams(const P& pr) {
        in_row = nullptr; out_row = nullptr; ring_row = nullptr; ring_D = 1; ring_slot = 0;
        if (pr.pf_buf[0] >= 0) { const BufDesc& b = pr.bufs[pr.pf_buf[0]]; in_row = b.base + (long long)ch * b.row_stride; }
        out_ring = 0; out_pos = 0;
        if (pr.st_buf >= 0) {
            const BufDesc& b = pr.bufs[pr.st_buf];
            out_row = b.base + (long long)ch * b.row_stride;
            out_ring = b.ring_len;
            out_pos = b.ring_pos;
        }
        if (pr.pf_ring[1] >= 0) {
            const RingDesc& r = pr.rings[pr.pf_ring[1]];
            ring_row = r.base + (long long)ch * r.D;
            ring_D = (int)r.D;
            ring_slot = (int)((r.pos + (long long)j * kChunk) % r.D);
        }
    }

    // Register prefetch, one tile ahead: right after a tile's input chunk (slot 0: the first streamed global
    // read) or ring chunk (slot 1: the first eligible comb ring) has been copied out of pf_*, the loads for
    // the next tile are issued straight into the same registers and stay in flight while this tile computes.
    // (An earlier version staged these through shared memory with cp.async; its 16 extra shared-memory
    // instructions per thread and tile clogged the SM-wide LSU queue the sequential R warp depends on.)
    // The destination must be a register array of the kernel itself (like `acc`), NOT a member of this struct:
    // the struct lives in local memory inside the interpreter loop, and a load whose result is stored to the
    // stack right away stalls on it immediately (measured: the "prefetch" then hides nothing).
    __device__ __forceinline__ void prefetch_in(int ti, float (&pf)[kChunk]) const {
        const int m0 = ti * Geo<G>::S + j * kChunk;
        if (ch_ok && m0 < T) {
            const float4* p = reinterpret_cast<const float4*>(in_row + m0);
#pragma unroll
            for (int k = 0; k < kF4; k++) ldg_prefetch(p + k, pf[4 * k], pf[4 * k + 1], pf[4 * k + 2], pf[4 * k + 3]);
        }
    }
    // ring chunk at `slot` for the tile whose first sample (of this thread) is m0
    __device__ __forceinline__ void prefetch_ring(int slot, int m0, float (&pf)[kChunk]) const {
        if (ch_ok && m0 < T) {
            const float4* p = reinterpret_cast<const float4*>(ring_row + slot);
#pragma unroll
            for (int k = 0; k < kF4; k++) ldg_prefetch(p + k, pf[4 * k], pf[4 * k + 1], pf[4 * k + 2], pf[4 * k + 3]);
        }
    }
};

// the two prefetch register sets of a thread (input chunk, ring chunk of the next tile)
struct Pf {
    float in[kChunk], ring[kChunk];
};

// One op of the segment program on this thread's 16 samples.  `code`, `mode` and `pre` are
// compile-time constants in the specialised kernels (the switch folds away) and run-time values in
// the generic interpreter.  pre & 1: acc = 0.0 + acc (first link of a fan-in sum, node.rs:181-183);
// pre & 2: acc /= nf (node.rs:189-191) with the divisor in p[4] and its tier's constants in p[5], p[6] (fanin_prologue).
// PC: the op may carry per-channel parameters (plan.h Program::pc); false in the compiled specialised chains, whose ops
// never do (chain_matches), so their code is the shared-parameter code only.
template <int G, bool PC = false>
__device__ __forceinline__ void exec_op(const int code, const int mode, const int pre, const int pfc, const Op& op,
                                        const Ctx<G>& c, float (&acc)[kChunk], Pf& pf) {
    const Program& prog = *c.prog;
    const int t = c.t;
    // scalar parameters: the op's own, or this thread's channel row of the per-channel table (resolved here, once: the code
    // below is the shared-parameter code run with per-thread values).  Table rows exist for every channel a CTA covers.
    // prm(i): p[i], prm(4): a2.  Without PC the op's fields are read where they are used, exactly as before.
    float pcv[5] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
    const float* pcr = nullptr;  // the op's first column in row 0 (the recurrence lanes pick their own rows)
    if constexpr (PC) {
        pcv[0] = op.p[0]; pcv[1] = op.p[1]; pcv[2] = op.p[2]; pcv[3] = op.p[3]; pcv[4] = op.a2;
        if (op_pc_col(op) >= 0) {
            pcr = prog.pc + op_pc_col(op);
            const float* r = pcr + (long long)c.ch * prog.pc_stride;
            const int n = op_pc_cols(code);
            for (int k = 0; k < n; k++) pcv[k] = r[k];
        }
    }
    auto prm = [&](int i) -> float {
        if constexpr (PC) return pcv[i];
        else return i < 4 ? op.p[i] : op.a2;
    };
    fanin_prologue(acc, pre, op);
    switch (code) {
        case OP_NOP: break;
        case OP_ZERO: {
#pragma unroll
            for (int i = 0; i < kChunk; i++) acc[i] = 0.0f;
        } break;
        case OP_LOADG:
        case OP_ADDG:
        case OP_COPYG: {
            float v[kChunk];
#pragma unroll
            for (int i = 0; i < kChunk; i++) v[i] = 0.0f;
            // pfc: is this op's operand register-prefetched?  0/1 = compile-time (specialised chains), -1 = look
            // at the op.  It has to be a compile-time fact where speed matters: with both variants in one
            // kernel ptxas gives the direct load and the prefetch load the same scoreboard, and the first use
            // of the direct load's registers then waits for the prefetch just issued (ncu: 2 x 11% of all
            // stall samples on that one instruction).
            if (pfc < 0 ? op.aux != 0 : pfc != 0) {  // prefetched one tile ago; request the next tile right away
                if (c.active) {
#pragma unroll
                    for (int i = 0; i < kChunk; i++) v[i] = pf.in[i];
                }
                c.prefetch_in(c.tile_i + 1, pf.in);
            } else if (c.active) {
                const BufDesc& b = prog.bufs[op.buf];
                const float4* p = reinterpret_cast<const float4*>(b.base + (long long)c.ch * b.row_stride + c.n0);
#pragma unroll
                for (int k = 0; k < kF4; k++) {
                    float4 q = ldg_stream(p + k);
                    v[4 * k] = q.x; v[4 * k + 1] = q.y; v[4 * k + 2] = q.z; v[4 * k + 3] = q.w;
                }
            }
#pragma unroll
            for (int i = 0; i < kChunk; i++)
                acc[i] = code == OP_COPYG ? v[i] : add(code == OP_LOADG ? 0.0f : acc[i], v[i]);
        } break;
        case OP_LOADV:
        case OP_ADDV:
        case OP_COPYV:
        case OP_ADD: {
            float v[kChunk];
            load16(c.vregs + (op.vreg * kF4) * kThreads + t, kThreads, v);
#pragma unroll
            for (int i = 0; i < kChunk; i++)
                acc[i] = code == OP_COPYV ? v[i] : add(code == OP_LOADV ? 0.0f : acc[i], v[i]);
        } break;
        case OP_SAVEV: {
            store16(c.vregs + (op.vreg * kF4) * kThreads + t, kThreads, acc);
        } break;
        case OP_STOREG: {
            if (c.active) {
                float4* p;
                if (pfc < 0 ? op.aux != 0 : pfc != 0) {
                    int m = c.n0;
                    if (c.out_ring) {  // FIR input ring (plan.h BufDesc): slot (ring_pos + m) mod ring_len, chunks never wrap
                        m += c.out_pos;
                        if (m >= c.out_ring) m -= c.out_ring;
                    }
                    p = reinterpret_cast<float4*>(c.out_row + m);
                } else {
                    const BufDesc& b = prog.bufs[op.buf];
                    int m = c.n0;
                    if (b.ring_len) {
                        m += b.ring_pos;
                        if (m >= b.ring_len) m -= b.ring_len;
                    }
                    p = reinterpret_cast<float4*>(b.base + (long long)c.ch * b.row_stride + m);
                }
#pragma unroll
                for (int k = 0; k < kF4; k++) stg_stream(p + k, make_float4(acc[4 * k], acc[4 * k + 1], acc[4 * k + 2], acc[4 * k + 3]));
            }
        } break;
        case OP_MODMAP: {  // lib.rs:138-146; (x + 1) / 2 == (x + 1) * 0.5 exactly
            const float lo = op.p[0], span = sub(op.p[1], op.p[0]);
#pragma unroll
            for (int i = 0; i < kChunk; i++) acc[i] = add(lo, mul(span, clamp01(mul(add(acc[i], 1.0f), 0.5f))));
        } break;
        case OP_GAIN: {
            if (op.pflags & 1) {
                float P[kChunk];
                load16(c.vregs + (op.pv[0] * kF4) * kThreads + t, kThreads, P);
#pragma unroll
                for (int i = 0; i < kChunk; i++) acc[i] = mul(acc[i], P[i]);
            } else {
                const float l = prm(0);
#pragma unroll
                for (int i = 0; i < kChunk; i++) acc[i] = mul(acc[i], l);
            }
        } break;
        case OP_DISTORT: {
            if (!(op.pflags & 1) && mode != Fuzz) {  // scalar level: the common case
                const float l = prm(0);       // per-channel: the host leaves the tier at DIV_IEEE, so the divisions below are dv
                if (l < 0.001f) break;  // every shaper returns the sample unchanged (distort.rs:64,...)
                const int tier = op_div_tier(op);
                switch (mode) {
                    case HardClip: {
#pragma unroll
                        for (int i = 0; i < kChunk; i++) acc[i] = clipf(mul(acc[i], l));
                        div_chunk(acc, l, op.p[1], op.p[2], tier, false);
                    } break;
                    case SoftClip: {
                        float c3[kChunk];
#pragma unroll
                        for (int i = 0; i < kChunk; i++) {
                            acc[i] = mul(acc[i], l);
                            c3[i] = mul(mul(acc[i], acc[i]), acc[i]);
                        }
                        // / 3: zh = RN(1/3), zl = RN(1/3 - zh); tests/test_gpu_const_div2.py enumerates all 2^32 dividends
                        div_chunk(c3, 3.0f, 0x1.555556p-2f, -0x1.555556p-27f, DIV_MULFMA, false);
#pragma unroll
                        for (int i = 0; i < kChunk; i++) {
                            float s = acc[i];
                            if (s > 1.0f) s = 2.0f / 3.0f;
                            else if (s >= -1.0f && s <= 1.0f) s = sub(s, c3[i]);
                            else s = -2.0f / 3.0f;
                            acc[i] = clipf(s);
                        }
                        div_chunk(acc, l, op.p[1], op.p[2], tier, false);
                    } break;
                    case Tanh: {
#pragma unroll
                        for (int i = 0; i < kChunk; i++) acc[i] = tanhf(mul(acc[i], l));
                    } break;
                    case RecipSoftClip: {
#pragma unroll
                        for (int i = 0; i < kChunk; i++)
                            acc[i] = mul(signumf(acc[i]), sub(1.0f, dv(1.0f, add(mul(fabsf(acc[i]), l), 1.0f))));
                    } break;
                    case Sin: {
#pragma unroll
                        for (int i = 0; i < kChunk; i++) acc[i] = sinf(mul(acc[i], l));
                    } break;
                    case Atan: {
#pragma unroll
                        for (int i = 0; i < kChunk; i++) acc[i] = atanf(mul(acc[i], l));
                    } break;
                    case Square: {
#pragma unroll
                        for (int i = 0; i < kChunk; i++) {
                            float v = mul(acc[i], l);
                            acc[i] = mul(mul(v, v), signumf(v));
                        }
                    } break;
                    case Chebyshev4: {
#pragma unroll
                        for (int i = 0; i < kChunk; i++) {
                            float v2 = mul(acc[i], l);
                            v2 = mul(v2, v2);
                            acc[i] = add(sub(mul(8.0f, mul(v2, v2)), mul(8.0f, v2)), 1.0f);
                        }
                    } break;
                }
                break;
            }
            float P[kChunk];
            if (op.pflags & 1) load16(c.vregs + (op.pv[0] * kF4) * kThreads + t, kThreads, P);
            else {
#pragma unroll
                for (int i = 0; i < kChunk; i++) P[i] = prm(0);
            }
            if (mode == Fuzz) {  // nodes/distort.rs:146-172, per 128-sample reference block
                const float mx = block128_max_abs(acc);
                float z[kChunk];
#pragma unroll
                for (int i = 0; i < kChunk; i++) {
                    float q = dv(clipf(mul(acc[i], P[i])), mx);
                    z[i] = copysignf(sub(1.0f, expf(copysignf(q, -1.0f))), -1.0f);
                }
                const float mz = block128_max_abs(z);
#pragma unroll
                for (int i = 0; i < kChunk; i++) z[i] = dv(clipf(mul(z[i], mx)), mz);
                const float my = block128_max_abs(z);
#pragma unroll
                for (int i = 0; i < kChunk; i++) acc[i] = dv(mul(z[i], mx), my);
            } else {  // per-sample level from a control port: generic path
#pragma unroll
                for (int i = 0; i < kChunk; i++) acc[i] = shape_generic(mode, acc[i], P[i]);
            }
        } break;
        case OP_OVERDRIVE: {
            if (op.pflags & 7) {
                float B[kChunk], D[kChunk], L[kChunk];
#pragma unroll
                for (int i = 0; i < kChunk; i++) { B[i] = prm(0); D[i] = prm(1); L[i] = prm(2); }
                if (op.pflags & 1) load16(c.vregs + (op.pv[0] * kF4) * kThreads + t, kThreads, B);
                if (op.pflags & 2) load16(c.vregs + (op.pv[1] * kF4) * kThreads + t, kThreads, D);
                if (op.pflags & 4) load16(c.vregs + (op.pv[2] * kF4) * kThreads + t, kThreads, L);
#pragma unroll
                for (int i = 0; i < kChunk; i++) acc[i] = overdrive_generic(acc[i], B[i], D[i], L[i]);
            } else {
                const float FRAC_PI_4 = 0.785398163397448309615660845819875721f;
                const float FRAC_2_PI = 0.636619772367581343075535053490057448f;
                const float b = prm(0), dr = prm(1), l = prm(2);
                if (l < 0.001f) break;
                const float omd = sub(1.0f, dr);
#pragma unroll
                for (int i = 0; i < kChunk; i++) {
                    const float x = acc[i];
                    float d = mul(FRAC_2_PI, atanf(mul(FRAC_PI_4, mul(x, b))));
                    acc[i] = mul(add(mul(dr, d), mul(omd, x)), l);
                }
            }
        } break;
        case OP_CHEBY: {
            const float lp = prm(0), ln = prm(1), tp = prm(2), tn = prm(3);
#pragma unroll
            for (int i = 0; i < kChunk; i++) {
                const float x = acc[i];
                if (x >= 0.0f) { if (!(lp < 0.001f)) acc[i] = dv(tanhf(mul(x, lp)), tp); }
                else { if (!(ln < 0.001f)) acc[i] = dv(tanhf(mul(x, ln)), tn); }
            }
        } break;
        case OP_MIX: {
            float b[kChunk];
            load16(c.vregs + (op.vreg * kF4) * kThreads + t, kThreads, b);
            if (op.pflags & 1) {
                float R[kChunk];
                load16(c.vregs + (op.pv[0] * kF4) * kThreads + t, kThreads, R);
#pragma unroll
                for (int i = 0; i < kChunk; i++) acc[i] = add(mul(b[i], R[i]), mul(acc[i], sub(1.0f, R[i])));
            } else {
                const float r = prm(0), omr = sub(1.0f, r);
#pragma unroll
                for (int i = 0; i < kChunk; i++) acc[i] = add(mul(b[i], r), mul(acc[i], omr));
            }
        } break;
        case OP_COMB: {
            const RingDesc& r = prog.rings[op.aux & 0xff];
            const float decay = prm(0);
            const int pslot = op.aux >> 8;  // 0 = not staged
            float* rrow = r.base + (long long)c.ch * r.D;
            const bool pfd = pfc < 0 ? pslot != 0 : pfc != 0;
            if (pfd || ((r.D & (kChunk - 1)) == 0 && (r.pos & (kChunk - 1)) == 0)) {
                long long slot;
                float old[kChunk];
#pragma unroll
                for (int i = 0; i < kChunk; i++) old[i] = 0.0f;
                if (pfd) {
                    if (c.active) {
#pragma unroll
                        for (int i = 0; i < kChunk; i++) old[i] = pf.ring[i];
                    }
                    slot = c.ring_slot;
                    int nxt = c.ring_slot + Geo<G>::S;
                    if (nxt >= c.ring_D) nxt -= c.ring_D;
                    c.ring_slot = nxt;
                    rrow = c.ring_row;
                    c.prefetch_ring(nxt, c.n0 + Geo<G>::S, pf.ring);
                } else {
                    slot = (r.pos + c.n0) % r.D;
                }
                if (!pfd && c.active) {
                    const float4* p = reinterpret_cast<const float4*>(rrow + slot);
#pragma unroll
                    for (int k = 0; k < kF4; k++) {
                        float4 q = ldg_stream(p + k);
                        old[4 * k] = q.x; old[4 * k + 1] = q.y; old[4 * k + 2] = q.z; old[4 * k + 3] = q.w;
                    }
                }
                if (c.active) {
#pragma unroll
                    for (int i = 0; i < kChunk; i++) acc[i] = add(acc[i], mul(old[i], decay));
                    float4* p = reinterpret_cast<float4*>(rrow + slot);
#pragma unroll
                    for (int k = 0; k < kF4; k++) stg_stream(p + k, make_float4(acc[4 * k], acc[4 * k + 1], acc[4 * k + 2], acc[4 * k + 3]));
                }
            } else if (c.active) {  // ring length not a multiple of 16: element-wise wrap
                long long slot = (r.pos + c.n0) % r.D;
#pragma unroll
                for (int i = 0; i < kChunk; i++) {
                    float o = __ldcg(rrow + slot);
                    acc[i] = add(acc[i], mul(o, decay));
                    __stcg(rrow + slot, acc[i]);
                    if (++slot == r.D) slot = 0;
                }
            }
        } break;
        case OP_BIQUAD: {
            // p[n] = b0*x[n] + b1*x[n-1] + b2*x[n-2] in the reference's order, time-parallel
            const float b0 = prm(0), b1 = prm(1), b2 = prm(2);
            float4* st = c.sm_state + op.aux * G;
            c.edge[t] = make_float2(acc[kChunk - 2], acc[kChunk - 1]);
            __syncthreads();
            float xm1, xm2;
            if (c.j == 0) { const float4 s = st[c.g]; xm1 = s.x; xm2 = s.y; }
            else { const float2 e = c.edge[t - 1]; xm2 = e.x; xm1 = e.y; }
            const float nx1 = acc[kChunk - 1], nx2 = acc[kChunk - 2];
            float pm1 = acc[0], pm2;
            acc[0] = add(add(mul(b0, acc[0]), mul(b1, xm1)), mul(b2, xm2));
            pm2 = pm1; pm1 = acc[1];
            acc[1] = add(add(mul(b0, acc[1]), mul(b1, pm2)), mul(b2, xm1));
#pragma unroll
            for (int i = 2; i < kChunk; i++) {
                const float xi = acc[i];
                acc[i] = add(add(mul(b0, xi), mul(b1, pm1)), mul(b2, pm2));
                pm2 = pm1; pm1 = xi;
            }
            if (mode != 0) {  // opt-in time-parallel evaluation (not bit-exact)
                scan_recurrence<G, false>(prog.scan[mode - 1], acc, c.tc, c.j_last, st, c.wend);
                // x1 / x2: read by the j == 0 thread of the channel right after the edge barrier above, i.e. before the
                // barrier / __syncwarp inside scan_recurrence that every thread of the channel has passed by now
                if (c.j == c.j_last) { st[c.g].x = nx1; st[c.g].y = nx2; }
                break;
            }
            DF1Core core;
            core.a1 = prm(3);
            core.a2 = prm(4);
            run_recurrence<G>(core, acc, c.tc, st, pcr, prog.pc_stride, c.ch - c.g);  // first barrier inside: every thread has read st / edge
            if (c.j == c.j_last) { st[c.g].x = nx1; st[c.g].y = nx2; }
        } break;
        case OP_LP1:
        case OP_HP1: {
            const float omr = prm(1);
            float v[kChunk];
#pragma unroll
            for (int i = 0; i < kChunk; i++) v[i] = mul(acc[i], omr);
            if (mode != 0) {  // z[n] = xr[n] + r z[n-1] as the scan with a1 = -r, a2 = 0; z lives in .z of the state (exact: .x)
                scan_recurrence<G, true>(prog.scan[mode - 1], v, c.tc, c.j_last, c.sm_state + op.aux * G, c.wend);
#pragma unroll
                for (int i = 0; i < kChunk; i++) acc[i] = code == OP_LP1 ? v[i] : sub(acc[i], v[i]);
                break;
            }
            OnePoleCore core;
            core.r = prm(0);
            run_recurrence<G>(core, v, c.tc, c.sm_state + op.aux * G, pcr, prog.pc_stride, c.ch - c.g);
#pragma unroll
            for (int i = 0; i < kChunk; i++) acc[i] = code == OP_LP1 ? v[i] : sub(acc[i], v[i]);
        } break;
        case OP_ENVELOPE: {
#pragma unroll
            for (int i = 0; i < kChunk; i++) acc[i] = fabsf(acc[i]);
            EnvCore core;
            core.ga = prm(0);
            core.gr = prm(1);
            run_recurrence<G>(core, acc, c.tc, c.sm_state + op.aux * G, pcr, prog.pc_stride, c.ch - c.g);
        } break;
        case OP_GATE: {  // extension: hard noise gate keyed by the envelope already in acc
            float x[kChunk];
            load16(c.vregs + (op.vreg * kF4) * kThreads + t, kThreads, x);
            const float thr = prm(0);
#pragma unroll
            for (int i = 0; i < kChunk; i++) acc[i] = acc[i] >= thr ? x[i] : 0.0f;
        } break;
        case OP_SIGGEN: {  // nodes/signal_gen.rs:55-130: phase accumulates per 128-sample reference block
            float A[kChunk];
            if (op.pflags & 1) load16(c.vregs + (op.pv[0] * kF4) * kThreads + t, kThreads, A);
            else {
#pragma unroll
                for (int i = 0; i < kChunk; i++) A[i] = prm(0);
            }
            if (mode == 3) {  // Constant: output = amplitude, clock untouched
#pragma unroll
                for (int i = 0; i < kChunk; i++) acc[i] = A[i];
                break;
            }
            using Q = Geo<G>;
            const float sr = op.p[2];
            const int pos = (c.j & (kBlk - 1)) * kChunk;  // first sample of this chunk inside its 128-block
            float tot[kChunk], total_end;
            if (op.pflags & 2) {  // frequency from a control port: sequential f32 sum of the block's steps
                __syncthreads();  // the seven other threads of the block wrote their frequency tiles
                const float4* fv = c.vregs + (op.pv[1] * kF4) * kThreads;
                float run = 0.0f;
                const int t0 = t - (c.j & (kBlk - 1));
                for (int th = 0; th < kBlk; th++) {
#pragma unroll
                    for (int k = 0; k < kF4; k++) {
                        const float4 q = fv[k * kThreads + t0 + th];
                        const float f4[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
                        for (int e = 0; e < 4; e++) {
                            run = add(run, dv(f4[e], sr));
                            if (th == (c.j & (kBlk - 1))) tot[4 * k + e] = run;
                        }
                    }
                }
                total_end = run;
            } else {
                const float step = dv(prm(1), sr);
                float run = 0.0f;
                for (int m = 0; m < pos; m++) run = add(run, step);
#pragma unroll
                for (int i = 0; i < kChunk; i++) { run = add(run, step); tot[i] = run; }
                for (int m = pos + kChunk; m < kRefBlock; m++) run = add(run, step);
                total_end = run;
            }
            // clock at the start of this thread's block: state, advanced once per earlier block of the tile.
            // With a modulated frequency every block has its own total: exchange them through edge[].
            float4* st = c.sm_state + op.aux * G;
            float clk = st[c.g].x;
            const int blk = c.j / kBlk;  // block index inside the tile
            __syncthreads();
            if ((c.j & (kBlk - 1)) == 0) c.edge[t / kBlk] = make_float2(total_end, 0.0f);
            __syncthreads();
            const int blk0 = (c.g * Q::TPC) / kBlk;
            for (int b = 0; b < blk; b++) clk = fmodf(add(clk, c.edge[blk0 + b].x), 1.0f);
            const float TAU = 6.28318530717958647692528676655900577f;
#pragma unroll
            for (int i = 0; i < kChunk; i++) {
                float v;
                if (mode == 0) v = sinf(mul(add(clk, tot[i]), TAU));
                else if (mode == 1) v = sub(mul(2.0f, fmodf(add(clk, tot[i]), 1.0f)), 1.0f);
                else v = tot[i] > 0.5f ? 1.0f : -1.0f;  // do_square ignores the clock (signal_gen.rs:93)
                acc[i] = mul(v, A[i]);
            }
            __syncthreads();
            if (c.j == 0) {  // one thread per channel advances the clock over the valid blocks of this tile
                float k2 = st[c.g].x;
                const int nblk = c.tc.valid_f4 / 32;
                for (int b = 0; b < nblk; b++) k2 = fmodf(add(k2, c.edge[blk0 + b].x), 1.0f);
                st[c.g].x = k2;
            }
        } break;
        default: break;
    }
}

// Compile-time op signatures of the BASELINE chains: same exec_op code, opcodes constant-folded.
// sig(i) packs code | mode << 8 | pre << 16; n = 0 selects the run-time interpreter.
struct ChainDynamic { static constexpr int n = 0; static constexpr int rec = 0; __host__ __device__ static constexpr int sig(int) { return 0; } __host__ __device__ static constexpr int pf_of(int) { return -1; } };
#define DSPB_SIG(code, mode, pre) ((code) | ((mode) << 8) | ((pre) << 16))
// The chains' fan-in prologues (every node of a chain has one link: acc /= 1.0001) are compiled for the mul-fma tier;
// a program whose divisor got another tier does not match a chain and runs in the interpreter.
constexpr int kPreDiv = 2 | (DIV_MULFMA << 2);   // acc /= p[4]
constexpr int kPreAddDiv = 1 | kPreDiv;          // acc = 0.0 + acc; acc /= p[4]
// PF (template argument of the chains): bit 0 = the input chunk (op 0) is register-prefetched, bit 1 = the
// comb ring chunk is; pf_of(i) is the compile-time pfc of op i.
template <int PF>
struct ChainGDBR {  // src -> gain -> distort(SoftClip) -> biquad -> reverb -> store   (config 3 / target front end)
    static constexpr int n = 6;
    static constexpr int rec = 3;
    __host__ __device__ static constexpr int pf_of(int i) { return i == 0 ? (PF & 1) : i == 4 ? ((PF >> 1) & 1) : i == n - 1 ? 1 : 0; }
    __host__ __device__ static constexpr int sig(int i) {
        return i == 0 ? DSPB_SIG(OP_LOADG, 0, 0) : i == 1 ? DSPB_SIG(OP_GAIN, 0, kPreDiv) : i == 2 ? DSPB_SIG(OP_DISTORT, SoftClip, kPreAddDiv)
             : i == 3 ? DSPB_SIG(OP_BIQUAD, 0, kPreAddDiv) : i == 4 ? DSPB_SIG(OP_COMB, 0, kPreAddDiv) : DSPB_SIG(OP_STOREG, 0, kPreAddDiv);
    }
};
template <int PF>
struct ChainGDBRScan {  // the same chain with the biquad in scan mode (dspb_config::iir_mode = 1, scan table 0)
    static constexpr int n = 6;
    [[maybe_unused]] static constexpr int rec = -1;
    __host__ __device__ static constexpr int pf_of(int i) { return ChainGDBR<PF>::pf_of(i); }
    __host__ __device__ static constexpr int sig(int i) { return i == 3 ? DSPB_SIG(OP_BIQUAD, 1, kPreAddDiv) : ChainGDBR<PF>::sig(i); }
};
template <int PF>
struct ChainGDR {  // src -> gain -> distort(SoftClip) -> reverb -> store   (config 1)
    static constexpr int n = 5;
    [[maybe_unused]] static constexpr int rec = -1;
    __host__ __device__ static constexpr int pf_of(int i) { return i == 0 ? (PF & 1) : i == 3 ? ((PF >> 1) & 1) : i == n - 1 ? 1 : 0; }
    __host__ __device__ static constexpr int sig(int i) {
        return i == 0 ? DSPB_SIG(OP_LOADG, 0, 0) : i == 1 ? DSPB_SIG(OP_GAIN, 0, kPreDiv) : i == 2 ? DSPB_SIG(OP_DISTORT, SoftClip, kPreAddDiv)
             : i == 3 ? DSPB_SIG(OP_COMB, 0, kPreAddDiv) : DSPB_SIG(OP_STOREG, 0, kPreAddDiv);
    }
};
template <int PF>
struct ChainBB {  // src -> biquad -> biquad -> store   (config 2)
    static constexpr int n = 4;
    [[maybe_unused]] static constexpr int rec = -1;
    __host__ __device__ static constexpr int pf_of(int i) { return i == 0 ? (PF & 1) : i == -1 ? ((PF >> 1) & 1) : i == n - 1 ? 1 : 0; }
    __host__ __device__ static constexpr int sig(int i) {
        return i == 0 ? DSPB_SIG(OP_LOADG, 0, 0) : i == 1 ? DSPB_SIG(OP_BIQUAD, 0, kPreDiv) : i == 2 ? DSPB_SIG(OP_BIQUAD, 0, kPreAddDiv) : DSPB_SIG(OP_STOREG, 0, kPreAddDiv);
    }
};
template <int PF>
struct ChainLH {  // src -> low_pass -> high_pass -> store   (config 2, one-pole variant)
    static constexpr int n = 4;
    [[maybe_unused]] static constexpr int rec = -1;
    __host__ __device__ static constexpr int pf_of(int i) { return i == 0 ? (PF & 1) : i == -1 ? ((PF >> 1) & 1) : i == n - 1 ? 1 : 0; }
    __host__ __device__ static constexpr int sig(int i) {
        return i == 0 ? DSPB_SIG(OP_LOADG, 0, 0) : i == 1 ? DSPB_SIG(OP_LP1, 0, kPreDiv) : i == 2 ? DSPB_SIG(OP_HP1, 0, kPreAddDiv) : DSPB_SIG(OP_STOREG, 0, kPreAddDiv);
    }
};
template <int PF>
struct ChainCopy {  // G -> (/nf) -> store   (the segment after a Fir node)
    static constexpr int n = 2;
    [[maybe_unused]] static constexpr int rec = -1;
    __host__ __device__ static constexpr int pf_of(int i) { return i == 0 ? (PF & 1) : i == -1 ? ((PF >> 1) & 1) : i == n - 1 ? 1 : 0; }
    __host__ __device__ static constexpr int sig(int i) { return i == 0 ? DSPB_SIG(OP_LOADG, 0, 0) : DSPB_SIG(OP_STOREG, 0, kPreDiv); }
};

template <int G, class Chain, int I>
__device__ __forceinline__ void run_static(const Program& prog, const Ctx<G>& c, float (&acc)[kChunk], Pf& pf) {
    if constexpr (I < Chain::n) {
        constexpr int s = Chain::sig(I);
        exec_op<G>(s & 0xff, (s >> 8) & 0xff, (s >> 16) & 0xff, Chain::pf_of(I), prog.ops[I], c, acc, pf);
        run_static<G, Chain, I + 1>(prog, c, acc, pf);
    }
}

template <int G, class Chain>
__global__ void __launch_bounds__(kThreads, 2)
fused_kernel(const __grid_constant__ Program prog, int c_begin, int c_end, long long T, int n_states, int n_sm) {
    using Q = Geo<G>;
    extern __shared__ float4 smem4[];
    Ctx<G> c;
    c.prog = &prog;
    c.t = threadIdx.x;
    c.g = c.t / Q::TPC;
    c.j = c.t % Q::TPC;
    c.ch = c_begin + blockIdx.x * G + c.g;
    c.ch_ok = c.ch < c_end;
    c.T = (int)T;
    c.init_streams(prog);
    const int t = c.t;

    // shared memory carve-up
    c.sm_state = smem4;                                                  // [kMaxStates][G]
    c.edge = reinterpret_cast<float2*>(c.sm_state + kMaxStates * G);     // [kThreads] chunk-edge samples
    c.wend = reinterpret_cast<double2*>(c.edge + kThreads);              // [kThreads / 32] warp end states (scan mode)
    float* tile = reinterpret_cast<float*>(c.wend + kThreads / 32);
    c.stage = reinterpret_cast<float4*>(tile + (prog.needs_tile ? G * Q::ROW : 0));  // (unused: prefetch lives in registers)
    c.vregs = c.stage;                                                               // [n_vregs][kF4][kThreads]

    for (int i = t; i < n_states * G; i += kThreads) {
        int s = i / G, cc = c_begin + blockIdx.x * G + (i % G);
        c.sm_state[s * G + (i % G)] = cc < c_end ? reinterpret_cast<const float4*>(prog.states[s])[cc] : make_float4(0, 0, 0, 0);
    }

    c.n_tiles = (int)((T + Q::S - 1) / Q::S);
    c.tc.tile = tile;
    c.tc.g = c.g;
    c.tc.j = c.j;
    // co-resident CTAs (bid, bid + n_sm, ...) put their sequential warp on different SM sub-partitions
    c.tc.rec_warp = 7 - (int)((blockIdx.x / (unsigned)n_sm) & 3u);

    Pf pf;
#pragma unroll
    for (int i = 0; i < kChunk; i++) pf.in[i] = pf.ring[i] = 0.0f;
    if (prog.pf_buf[0] >= 0) c.prefetch_in(0, pf.in);
    if (prog.pf_ring[1] >= 0) c.prefetch_ring(c.ring_slot, c.j * kChunk, pf.ring);
    __syncthreads();

    for (int tile_i = 0; tile_i < c.n_tiles; tile_i++) {
        c.tile_i = tile_i;
        c.n0 = tile_i * Q::S + c.j * kChunk;
        c.active = c.ch_ok && c.n0 < c.T;
        const int rem = c.T - tile_i * Q::S;
        c.tc.valid_f4 = (rem < Q::S ? rem : Q::S) / 4;
        c.j_last = c.tc.valid_f4 / kF4 - 1;  // thread holding the last valid chunk of each channel

        __syncthreads();  // ring / tile hazards across tiles

        float acc[kChunk];
#pragma unroll
        for (int i = 0; i < kChunk; i++) acc[i] = 0.0f;

        if constexpr (Chain::n > 0) {
            run_static<G, Chain, 0>(prog, c, acc, pf);
        } else {
            for (int ip = 0; ip < prog.n_ops; ip++) {
                const Op& op = prog.ops[ip];
                exec_op<G, true>(op.code, op.mode, op.pre, -1, op, c, acc, pf);
            }
        }
    }
    __syncthreads();
    for (int i = t; i < n_states * G; i += kThreads) {
        int s = i / G, cc = c_begin + blockIdx.x * G + (i % G);
        if (cc < c_end) reinterpret_cast<float4*>(prog.states[s])[cc] = c.sm_state[s * G + (i % G)];
    }
}


// ======================= warp-specialised variant: one recurrence, fully overlapped =======================
// For programs with exactly one recurrence op (biquad / low_pass / envelope) and no shared-memory vregs.
// 9 warps: warps 0-7 ("E") run the time-parallel ops, warp 8 ("R") runs nothing but the lane = channel
// feedback loop.  Tiles are double-buffered: in iteration i the E warps run the ops before the recurrence
// for tile i (and hand tile buffer i&1 to R), then the ops after it for tile i-1 (once R is done with it),
// so the sequential 12-cycle-per-sample chain is hidden behind elementwise work of neighbouring tiles.
// Hand-offs use named barriers (bar.arrive / bar.sync with the 288-thread count).
// The one R warp serves all channels of the CTA (lane = channel).  With many channels per SM it does not bound the
// kernel, the E warps do: measured, E never waits for DONE and R idles ~30 % of the time waiting for FULL, and a
// second R warp splitting the channels changed nothing.  When the recurrence chain does bound the kernel (few channels
// per SM), the XR layout below gives the R warp a sub-partition of its own.
constexpr int kWsLaunchThreads = kThreads + 32;
enum { BAR_FULL0 = 1, BAR_FULL1 = 2, BAR_DONE0 = 3, BAR_DONE1 = 4, BAR_EONLY = 5 };
__device__ __forceinline__ void bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void bar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }

// `lane` is the channel index inside the CTA (or >= G for idle lanes); `row` is its state row, read and written only
// when `ok`.  A biquad writes back y1, y2 (.z/.w) only: the elementwise warps own x1, x2.
template <int G, class Core>
__device__ __forceinline__ void ws_recurrence_warp(Core core, float* tiles, float4* row, int lane, bool ok, long long n_tiles,
                                                   long long T, int n_ws, bool biquad) {
    using Q = Geo<G>;
    float4 s = make_float4(0, 0, 0, 0);
    if (ok) s = *row;
    core.load(s);
    for (long long i = 0; i < n_tiles; i++) {
        const int b = (int)(i & 1);
        const long long rem = T - i * Q::S;
        const int valid_f4 = (int)((rem < Q::S ? rem : Q::S) / 4);
        bar_sync(BAR_FULL0 + b, n_ws);
        if (lane < G) {
            float4* r = reinterpret_cast<float4*>(tiles + b * (G * Q::ROW) + lane * Q::ROW);
            recurrence_row(core, r, valid_f4);
        }
        __threadfence_block();  // bar.arrive alone orders nothing: make the tile visible first
        __syncwarp();
        bar_arrive(BAR_DONE0 + b, n_ws);
    }
    if (ok) {
        core.save(s);
        float* f = reinterpret_cast<float*>(row);
        if (biquad) { f[2] = s.z; f[3] = s.w; }
        else *row = s;
    }
}

template <int G, class Chain, int I, int END>
__device__ __forceinline__ void run_static_range(const Program& prog, const Ctx<G>& c, float (&acc)[kChunk], Pf& pf) {
    if constexpr (I < END) {
        constexpr int s = Chain::sig(I);
        exec_op<G>(s & 0xff, (s >> 8) & 0xff, (s >> 16) & 0xff, Chain::pf_of(I), prog.ops[I], c, acc, pf);
        run_static_range<G, Chain, I + 1, END>(prog, c, acc, pf);
    }
}

// XR ("exclusive R"): the recurrence warp gets an SM sub-partition of its own.  Warp w of a CTA issues on
// sub-partition w % 4; measured (tests/cuda/rec_microbench.cu) the lane = channel feedback loop takes 14.2 cycles per
// sample alone or next to FP work on the OTHER sub-partitions, but 39.6 cycles as soon as two busy warps share its
// scheduler.  In the XR layout physical warp 3 is the R warp, warps 7, 11, ... exit at once and the elementwise
// threads are renumbered over the remaining warps; the CTA is launched with 24 warps (a multiple of 4 keeps the
// mapping aligned for a co-resident CTA).  The elementwise warps lose a quarter of the issue slots, so the
// launcher uses XR only when the recurrence chain, not the elementwise work, bounds the kernel (few channels per SM).
constexpr int kXrLaunchThreads = 768;
template <int G, class Chain, bool XR>
__global__ void __launch_bounds__(XR ? kXrLaunchThreads : kWsLaunchThreads, XR ? 1 : 2)
fused_kernel_ws(const __grid_constant__ Program prog, int c_begin, int c_end, long long T, int gc, int rec_index) {
    // gc <= G: channels this CTA really owns.  The launcher trims gc so that the grid is ONE balanced wave (every SM
    // gets the same number of channels); the CTA is launched with only gc * TPC elementwise threads + the R warp.
    const int n_e = gc * Geo<G>::TPC, n_ws = n_e + 32;
    using Q = Geo<G>;
    extern __shared__ float4 smem4[];
    int t = threadIdx.x;  // logical index; t < n_e: elementwise thread, else R-warp thread
    if constexpr (XR) {
        const int pw = t >> 5;
        if ((pw & 3) == 3) {
            if (pw != 3) return;
            t = n_e + (t & 31);
        } else {
            t = (pw - (pw >> 2)) * 32 + (t & 31);
            if (t >= n_e) return;
        }
    }
    // shared memory: [G] x-state (float2) | edge[256] | tiles[2][G*ROW] | stage
    float2* xstate = reinterpret_cast<float2*>(smem4);
    float2* edge = xstate + 64;  // xstate[2][32]: read parity i & 1, written parity (i + 1) & 1
    float* tiles = reinterpret_cast<float*>(edge + kThreads);
    const long long n_tiles = (T + Q::S - 1) / Q::S;
    const Op& rop = prog.ops[rec_index];
    const int rcode = Chain::n > 0 ? (Chain::sig(Chain::rec) & 0xff) : rop.code;
    // high_pass (y = x - z, nodes/high_pass.rs:36-41) needs x again after the recurrence: kept in a second pair of
    // tile buffers, same thread-private positions
    float* keep = tiles + 2 * G * Q::ROW;
    float4* stage = reinterpret_cast<float4*>(keep + (rcode == OP_HP1 ? 2 * G * Q::ROW : 0));
    float* stp = prog.states[rop.aux];
    // per-channel coefficients of the recurrence op (interpreter only: chain_matches keeps such ops out of the chains)
    constexpr bool PC = Chain::n == 0;
    const bool rpc = PC && op_pc_col(rop) >= 0;

    if (t >= n_e) {  // ---------------- R warp ----------------
        const int rl = t & 31;
        const int lane = rl < gc ? rl : G;  // channel inside the CTA; G = idle lane
        const int ch = c_begin + blockIdx.x * gc + lane;
        const bool ok = lane < G && ch < c_end;
        float4* row = reinterpret_cast<float4*>(stp) + (ok ? ch : 0);
        if (rcode == OP_BIQUAD) {
            DF1Core core; core.a1 = rop.p[3]; core.a2 = rop.a2;
            if (PC && rpc && ok) core.from_row(prog.pc + op_pc_col(rop) + (long long)ch * prog.pc_stride);
            ws_recurrence_warp<G>(core, tiles, row, lane, ok, n_tiles, T, n_ws, true);
        } else if (rcode == OP_LP1 || rcode == OP_HP1) {
            OnePoleCore core; core.r = rop.p[0];
            if (PC && rpc && ok) core.from_row(prog.pc + op_pc_col(rop) + (long long)ch * prog.pc_stride);
            ws_recurrence_warp<G>(core, tiles, row, lane, ok, n_tiles, T, n_ws, false);
        } else {
            EnvCore core; core.ga = rop.p[0]; core.gr = rop.p[1];
            if (PC && rpc && ok) core.from_row(prog.pc + op_pc_col(rop) + (long long)ch * prog.pc_stride);
            ws_recurrence_warp<G>(core, tiles, row, lane, ok, n_tiles, T, n_ws, false);
        }
        return;
    }

    // ---------------- E warps ----------------
    Ctx<G> c;
    c.prog = &prog;
    c.t = t;
    c.g = t / Q::TPC;
    c.j = t % Q::TPC;
    c.ch = c_begin + blockIdx.x * gc + c.g;
    c.ch_ok = c.ch < c_end;
    c.T = (int)T;
    c.init_streams(prog);
    c.sm_state = nullptr;
    c.wend = nullptr;
    c.edge = edge;
    c.stage = stage;
    c.vregs = stage;  // [n_vregs][kF4][kThreads]; none of them is live across the recurrence (ws_rec_index)
    c.n_tiles = (int)n_tiles;
    c.tc.tile = tiles;
    c.tc.g = c.g;
    c.tc.j = c.j;
    c.tc.rec_warp = 8;
    if (t < gc) {
        const int ch = c_begin + blockIdx.x * gc + t;
        xstate[t] = (rcode == OP_BIQUAD && ch < c_end) ? *reinterpret_cast<const float2*>(stp + 4 * (long long)ch) : make_float2(0.f, 0.f);
    }
    float cx1 = 0.0f, cx2 = 0.0f;  // biquad x1, x2 carried from tile to tile (TPC <= 32: every lane of the channel holds them)
    if (Q::TPC <= 32 && rcode == OP_BIQUAD && c.ch_ok) {
        const float2 s2 = *reinterpret_cast<const float2*>(stp + 4 * (long long)c.ch);
        cx1 = s2.x; cx2 = s2.y;
    }
    Pf pf;
#pragma unroll
    for (int i = 0; i < kChunk; i++) pf.in[i] = pf.ring[i] = 0.0f;
    if (prog.pf_buf[0] >= 0) c.prefetch_in(0, pf.in);
    if (prog.pf_ring[1] >= 0) c.prefetch_ring(c.ring_slot, c.j * kChunk, pf.ring);
    bar_sync(BAR_EONLY, n_e);

    auto set_tile = [&](int ti) {
        c.tile_i = ti;
        c.n0 = ti * Q::S + c.j * kChunk;
        c.active = c.ch_ok && c.n0 < c.T;
        const int rem = c.T - ti * Q::S;
        c.tc.valid_f4 = (rem < Q::S ? rem : Q::S) / 4;
        c.j_last = c.tc.valid_f4 / kF4 - 1;
    };

    const int nt = (int)n_tiles;
    for (int i = 0; i <= nt; i++) {
        // edge[] is rewritten below: from i = 2 on, the BAR_DONE sync of the previous iteration already orders
        // that behind every thread's reads (and the ring stores of tile i-2 before the loads of tile i-1)
        if (i <= 1) bar_sync(BAR_EONLY, n_e);
        float acc[kChunk];
        if (i < nt) {  // ---- ops before the recurrence, tile i ----
            set_tile(i);
#pragma unroll
            for (int k = 0; k < kChunk; k++) acc[k] = 0.0f;
            if constexpr (Chain::n > 0) run_static_range<G, Chain, 0, Chain::rec>(prog, c, acc, pf);
            else
                for (int ip = 0; ip < rec_index; ip++) exec_op<G, true>(prog.ops[ip].code, prog.ops[ip].mode, prog.ops[ip].pre, -1, prog.ops[ip], c, acc, pf);
            // the recurrence op's own prologue and feed-forward part
            fanin_prologue(acc, Chain::n > 0 ? ((Chain::sig(Chain::rec) >> 16) & 0xff) : rop.pre, rop);
            if (rcode == OP_BIQUAD) {
                float b0 = rop.p[0], b1 = rop.p[1], b2 = rop.p[2];
                if constexpr (PC) {
                    if (rpc) { const float* r = prog.pc + op_pc_col(rop) + (long long)c.ch * prog.pc_stride; b0 = r[0]; b1 = r[1]; b2 = r[2]; }
                }
                const float nx1 = acc[kChunk - 1], nx2 = acc[kChunk - 2];
                float xm1, xm2;
                if constexpr (Q::TPC <= 32) {
                    // a channel's threads sit in one warp: the two samples before this chunk come from the lane
                    // below by shuffle, the tile-to-tile carry (x1, x2 of the DF1 state) stays in registers --
                    // no shared-memory exchange and no CTA-wide barrier on the elementwise warps' path
                    xm1 = __shfl_up_sync(0xffffffffu, nx1, 1, Q::TPC);
                    xm2 = __shfl_up_sync(0xffffffffu, nx2, 1, Q::TPC);
                    if (c.j == 0) { xm1 = cx1; xm2 = cx2; }
                    cx1 = __shfl_sync(0xffffffffu, nx1, c.j_last, Q::TPC);
                    cx2 = __shfl_sync(0xffffffffu, nx2, c.j_last, Q::TPC);
                } else {
                    edge[t] = make_float2(acc[kChunk - 2], acc[kChunk - 1]);
                    bar_sync(BAR_EONLY, n_e);
                    if (c.j == 0) { const float2 s2 = xstate[(i & 1) * 32 + c.g]; xm1 = s2.x; xm2 = s2.y; }
                    else { const float2 e = edge[t - 1]; xm2 = e.x; xm1 = e.y; }
                }
                float pm1 = acc[0], pm2;
                acc[0] = add(add(mul(b0, acc[0]), mul(b1, xm1)), mul(b2, xm2));
                pm2 = pm1; pm1 = acc[1];
                acc[1] = add(add(mul(b0, acc[1]), mul(b1, pm2)), mul(b2, xm1));
#pragma unroll
                for (int k = 2; k < kChunk; k++) {
                    const float xi = acc[k];
                    acc[k] = add(add(mul(b0, xi), mul(b1, pm1)), mul(b2, pm2));
                    pm2 = pm1; pm1 = xi;
                }
                if constexpr (Q::TPC > 32) {
                    if (c.j == c.j_last) xstate[((i + 1) & 1) * 32 + c.g] = make_float2(nx1, nx2);
                }
            } else if (rcode == OP_LP1 || rcode == OP_HP1) {
                if (rcode == OP_HP1) {
                    float4* krow = reinterpret_cast<float4*>(keep + (int)(i & 1) * (G * Q::ROW) + c.g * Q::ROW);
#pragma unroll
                    for (int k = 0; k < kF4; k++)
                        krow[kF4 * c.j + (k ^ sw_of(c.j))] = make_float4(acc[4 * k], acc[4 * k + 1], acc[4 * k + 2], acc[4 * k + 3]);
                }
                float omr = rop.p[1];
                if constexpr (PC) {
                    if (rpc) omr = prog.pc[op_pc_col(rop) + 1 + (long long)c.ch * prog.pc_stride];
                }
#pragma unroll
                for (int k = 0; k < kChunk; k++) acc[k] = mul(acc[k], omr);
            } else {
#pragma unroll
                for (int k = 0; k < kChunk; k++) acc[k] = fabsf(acc[k]);
            }
            float4* row = reinterpret_cast<float4*>(tiles + (int)(i & 1) * (G * Q::ROW) + c.g * Q::ROW);
#pragma unroll
            for (int k = 0; k < kF4; k++)
                row[kF4 * c.j + (k ^ sw_of(c.j))] = make_float4(acc[4 * k], acc[4 * k + 1], acc[4 * k + 2], acc[4 * k + 3]);
            __threadfence_block();
            bar_arrive(BAR_FULL0 + (int)(i & 1), n_ws);
        }
        if (i >= 1) {  // ---- ops after the recurrence, tile i-1 ----
            const int b = (int)((i - 1) & 1);
            bar_sync(BAR_DONE0 + b, n_ws);
            set_tile(i - 1);
            const float4* row = reinterpret_cast<const float4*>(tiles + b * (G * Q::ROW) + c.g * Q::ROW);
#pragma unroll
            for (int k = 0; k < kF4; k++) {
                const float4 q = row[kF4 * c.j + (k ^ sw_of(c.j))];
                acc[4 * k] = q.x; acc[4 * k + 1] = q.y; acc[4 * k + 2] = q.z; acc[4 * k + 3] = q.w;
            }
            if (rcode == OP_HP1) {  // y = x - z
                const float4* krow = reinterpret_cast<const float4*>(keep + b * (G * Q::ROW) + c.g * Q::ROW);
#pragma unroll
                for (int k = 0; k < kF4; k++) {
                    const float4 x = krow[kF4 * c.j + (k ^ sw_of(c.j))];
                    acc[4 * k] = sub(x.x, acc[4 * k]); acc[4 * k + 1] = sub(x.y, acc[4 * k + 1]);
                    acc[4 * k + 2] = sub(x.z, acc[4 * k + 2]); acc[4 * k + 3] = sub(x.w, acc[4 * k + 3]);
                }
            }
            if constexpr (Chain::n > 0) run_static_range<G, Chain, Chain::rec + 1, Chain::n>(prog, c, acc, pf);
            else
                for (int ip = rec_index + 1; ip < prog.n_ops; ip++) exec_op<G, true>(prog.ops[ip].code, prog.ops[ip].mode, prog.ops[ip].pre, -1, prog.ops[ip], c, acc, pf);
        }
    }
    bar_sync(BAR_EONLY, n_e);
    if constexpr (Q::TPC <= 32) {
        if (rcode == OP_BIQUAD && c.j == 0 && c.ch_ok) *reinterpret_cast<float2*>(stp + 4 * (long long)c.ch) = make_float2(cx1, cx2);
    } else if (rcode == OP_BIQUAD && t < gc) {
        const int ch = c_begin + blockIdx.x * gc + t;
        if (ch < c_end) *reinterpret_cast<float2*>(stp + 4 * (long long)ch) = xstate[(nt & 1) * 32 + t];
    }
}


// ======================= two recurrences in series, pipelined over two recurrence warps =======================
// BASELINE config 2 (biquad low-pass -> biquad high-pass) is nothing but two sequential feedback chains: run back to
// back they cost ~2 x 15 cycles per sample.  Here recurrence warp R1 works on tile i while R2 works on tile i-1 and
// the elementwise warps feed both: iteration i runs the ops before recurrence 1 for tile i, the ops between the two
// for tile i-1 and the ops after recurrence 2 for tile i-2.  Same hand-off protocol as fused_kernel_ws (named
// barriers FULL / DONE per stage and tile parity), same XR layout (R1 = physical warp 3, R2 = warp 7: both on
// sub-partition 3, where two dependent chains interleave without slowing each other down).
enum { BAR2_FULL = 1, BAR2_DONE = 5, BAR2_EONLY = 9 };  // FULL/DONE: + 2 * stage + parity

template <int G>
struct Ws2Smem {
    static constexpr int kXstate = 2 * 2 * 32;                      // float2 [stage][parity][32]
    static constexpr int kEdge = 2 * kThreads;                      // float2 [stage][kThreads]
    static constexpr int kTiles = 2 * 2 * G * Geo<G>::ROW;          // float  [stage][parity][G * ROW]
    static constexpr int bytes = (kXstate + kEdge) * 8 + 2 * kTiles * 4;  // tiles + the high_pass keep buffers
};

template <int G, class Core>
__device__ __forceinline__ void ws2_rec_loop(Core core, float* tiles, float* stp, int lane, int ch, bool ok, int n_tiles, int T,
                                             int bar_full, int bar_done, int n_ws, bool biquad) {
    using Q = Geo<G>;
    float4 s = make_float4(0, 0, 0, 0);
    if (ok) s = *reinterpret_cast<const float4*>(stp + 4 * (long long)ch);
    core.load(s);
    for (int i = 0; i < n_tiles; i++) {
        const int b = i & 1;
        const int rem = T - i * Q::S;
        const int valid_f4 = (rem < Q::S ? rem : Q::S) / 4;
        bar_sync(bar_full + b, n_ws);
        if (lane < G) recurrence_row(core, reinterpret_cast<float4*>(tiles + b * (G * Q::ROW) + lane * Q::ROW), valid_f4);
        __threadfence_block();
        __syncwarp();
        bar_arrive(bar_done + b, n_ws);
    }
    if (ok) {
        core.save(s);
        float* f = stp + 4 * (long long)ch;
        if (biquad) { f[2] = s.z; f[3] = s.w; }  // y1, y2; the elementwise warps own x1, x2
        else *reinterpret_cast<float4*>(f) = s;
    }
}

template <int G>
__global__ void __launch_bounds__(kXrLaunchThreads, 1)
fused_kernel_ws2(const __grid_constant__ Program prog, int c_begin, int c_end, long long T64, int r1, int r2) {
    using Q = Geo<G>;
    constexpr int n_e = kThreads, n_ws = kThreads + 32;
    extern __shared__ float4 smem4[];
    float2* xstate = reinterpret_cast<float2*>(smem4);
    float2* edge = xstate + Ws2Smem<G>::kXstate;
    float* tiles = reinterpret_cast<float*>(edge + Ws2Smem<G>::kEdge);
    float* keep = tiles + Ws2Smem<G>::kTiles;  // x of a high_pass stage, [stage][parity][G * ROW]
    const int T = (int)T64;
    const int nt = (T + Q::S - 1) / Q::S;
    int t = threadIdx.x, role = 0;  // 0 = elementwise, 1 = R1, 2 = R2
    const int pw = t >> 5;
    if ((pw & 3) == 3) {
        if (pw > 7) return;
        role = pw == 3 ? 1 : 2;
    } else {
        t = (pw - (pw >> 2)) * 32 + (t & 31);
        if (t >= n_e) return;
    }
    const Op& rop1 = prog.ops[r1];
    const Op& rop2 = prog.ops[r2];

    if (role) {  // ---------------- recurrence warps ----------------
        const Op& rop = role == 1 ? rop1 : rop2;
        const int st = role - 1;
        const int rl = threadIdx.x & 31;
        const int lane = rl < G ? rl : G;
        const int ch = c_begin + blockIdx.x * G + lane;
        const bool ok = lane < G && ch < c_end;
        float* stp = prog.states[rop.aux];
        float* tl = tiles + st * (2 * G * Q::ROW);
        const int bf = BAR2_FULL + 2 * st, bd = BAR2_DONE + 2 * st;
        // per-channel coefficients: this lane's channel row (plan.h Program::pc)
        const float* pr = op_pc_col(rop) >= 0 && ok ? prog.pc + op_pc_col(rop) + (long long)ch * prog.pc_stride : nullptr;
        if (rop.code == OP_BIQUAD) {
            DF1Core core; core.a1 = rop.p[3]; core.a2 = rop.a2;
            if (pr) core.from_row(pr);
            ws2_rec_loop<G>(core, tl, stp, lane, ch, ok, nt, T, bf, bd, n_ws, true);
        } else if (rop.code == OP_LP1 || rop.code == OP_HP1) {
            OnePoleCore core; core.r = rop.p[0];
            if (pr) core.from_row(pr);
            ws2_rec_loop<G>(core, tl, stp, lane, ch, ok, nt, T, bf, bd, n_ws, false);
        } else {
            EnvCore core; core.ga = rop.p[0]; core.gr = rop.p[1];
            if (pr) core.from_row(pr);
            ws2_rec_loop<G>(core, tl, stp, lane, ch, ok, nt, T, bf, bd, n_ws, false);
        }
        return;
    }

    // ---------------- elementwise warps ----------------
    Ctx<G> c;
    c.prog = &prog;
    c.t = t;
    c.g = t / Q::TPC;
    c.j = t % Q::TPC;
    c.ch = c_begin + blockIdx.x * G + c.g;
    c.ch_ok = c.ch < c_end;
    c.T = T;
    c.init_streams(prog);
    c.sm_state = nullptr;
    c.wend = nullptr;
    c.edge = edge;
    c.stage = nullptr;
    c.vregs = nullptr;
    c.n_tiles = nt;
    c.tc.tile = tiles;
    c.tc.g = c.g;
    c.tc.j = c.j;
    c.tc.rec_warp = 0;
    // biquad x1, x2 of each stage, carried from tile to tile: registers (TPC <= 32) or xstate[stage][parity][g]
    float cx[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
    for (int st = 0; st < 2; st++) {
        const Op& rop = st == 0 ? rop1 : rop2;
        if (rop.code != OP_BIQUAD) continue;
        const float* stp = prog.states[rop.aux];
        if (Q::TPC <= 32) {
            if (c.ch_ok) { const float2 s2 = *reinterpret_cast<const float2*>(stp + 4 * (long long)c.ch); cx[st][0] = s2.x; cx[st][1] = s2.y; }
        } else if (t < G) {
            const int ch = c_begin + blockIdx.x * G + t;
            xstate[st * 64 + t] = ch < c_end ? *reinterpret_cast<const float2*>(stp + 4 * (long long)ch) : make_float2(0.f, 0.f);
        }
    }
    Pf pf;
#pragma unroll
    for (int i = 0; i < kChunk; i++) pf.in[i] = pf.ring[i] = 0.0f;
    if (prog.pf_buf[0] >= 0) c.prefetch_in(0, pf.in);
    if (prog.pf_ring[1] >= 0) c.prefetch_ring(c.ring_slot, c.j * kChunk, pf.ring);
    bar_sync(BAR2_EONLY, n_e);

    auto set_tile = [&](int ti) {
        c.tile_i = ti;
        c.n0 = ti * Q::S + c.j * kChunk;
        c.active = c.ch_ok && c.n0 < c.T;
        const int rem = c.T - ti * Q::S;
        c.tc.valid_f4 = (rem < Q::S ? rem : Q::S) / 4;
        c.j_last = c.tc.valid_f4 / kF4 - 1;
    };
    // prologue + time-parallel part of recurrence op `rop` (stage st) for the tile set by set_tile(ti), then the hand-off
    auto feed = [&](const Op& rop, int st, int ti, float (&acc)[kChunk]) {
        fanin_prologue(acc, rop.pre, rop);
        // per-channel parameters: this thread's channel row
        const float* pr = op_pc_col(rop) >= 0 ? prog.pc + op_pc_col(rop) + (long long)c.ch * prog.pc_stride : nullptr;
        if (rop.code == OP_BIQUAD) {
            float b0 = rop.p[0], b1 = rop.p[1], b2 = rop.p[2];
            if (pr) { b0 = pr[0]; b1 = pr[1]; b2 = pr[2]; }
            const float nx1 = acc[kChunk - 1], nx2 = acc[kChunk - 2];
            float xm1, xm2;
            if constexpr (Q::TPC <= 32) {
                xm1 = __shfl_up_sync(0xffffffffu, nx1, 1, Q::TPC);
                xm2 = __shfl_up_sync(0xffffffffu, nx2, 1, Q::TPC);
                if (c.j == 0) { xm1 = cx[st][0]; xm2 = cx[st][1]; }
                cx[st][0] = __shfl_sync(0xffffffffu, nx1, c.j_last, Q::TPC);
                cx[st][1] = __shfl_sync(0xffffffffu, nx2, c.j_last, Q::TPC);
            } else {
                float2* ed = edge + st * kThreads;
                float2* xs = xstate + st * 64;
                ed[t] = make_float2(nx2, nx1);
                bar_sync(BAR2_EONLY, n_e);
                if (c.j == 0) { const float2 s2 = xs[(ti & 1) * 32 + c.g]; xm1 = s2.x; xm2 = s2.y; }
                else { const float2 e = ed[t - 1]; xm2 = e.x; xm1 = e.y; }
                if (c.j == c.j_last) xs[((ti + 1) & 1) * 32 + c.g] = make_float2(nx1, nx2);
            }
            float pm1 = acc[0], pm2;
            acc[0] = add(add(mul(b0, acc[0]), mul(b1, xm1)), mul(b2, xm2));
            pm2 = pm1; pm1 = acc[1];
            acc[1] = add(add(mul(b0, acc[1]), mul(b1, pm2)), mul(b2, xm1));
#pragma unroll
            for (int k = 2; k < kChunk; k++) {
                const float xi = acc[k];
                acc[k] = add(add(mul(b0, xi), mul(b1, pm1)), mul(b2, pm2));
                pm2 = pm1; pm1 = xi;
            }
        } else if (rop.code == OP_LP1 || rop.code == OP_HP1) {
            if (rop.code == OP_HP1) {
                float4* krow = reinterpret_cast<float4*>(keep + (st * 2 + (ti & 1)) * (G * Q::ROW) + c.g * Q::ROW);
#pragma unroll
                for (int k = 0; k < kF4; k++)
                    krow[kF4 * c.j + (k ^ sw_of(c.j))] = make_float4(acc[4 * k], acc[4 * k + 1], acc[4 * k + 2], acc[4 * k + 3]);
            }
            const float omr = pr ? pr[1] : rop.p[1];
#pragma unroll
            for (int k = 0; k < kChunk; k++) acc[k] = mul(acc[k], omr);
        } else {
#pragma unroll
            for (int k = 0; k < kChunk; k++) acc[k] = fabsf(acc[k]);
        }
        float4* row = reinterpret_cast<float4*>(tiles + (st * 2 + (ti & 1)) * (G * Q::ROW) + c.g * Q::ROW);
#pragma unroll
        for (int k = 0; k < kF4; k++)
            row[kF4 * c.j + (k ^ sw_of(c.j))] = make_float4(acc[4 * k], acc[4 * k + 1], acc[4 * k + 2], acc[4 * k + 3]);
        __threadfence_block();
        bar_arrive(BAR2_FULL + 2 * st + (ti & 1), n_ws);
    };
    auto fetch = [&](int st, int ti, float (&acc)[kChunk]) {  // wait for recurrence `st` on tile ti and read it back
        bar_sync(BAR2_DONE + 2 * st + (ti & 1), n_ws);
        const float4* row = reinterpret_cast<const float4*>(tiles + (st * 2 + (ti & 1)) * (G * Q::ROW) + c.g * Q::ROW);
#pragma unroll
        for (int k = 0; k < kF4; k++) {
            const float4 q = row[kF4 * c.j + (k ^ sw_of(c.j))];
            acc[4 * k] = q.x; acc[4 * k + 1] = q.y; acc[4 * k + 2] = q.z; acc[4 * k + 3] = q.w;
        }
        if ((st == 0 ? rop1 : rop2).code == OP_HP1) {  // y = x - z (nodes/high_pass.rs:36-41)
            const float4* krow = reinterpret_cast<const float4*>(keep + (st * 2 + (ti & 1)) * (G * Q::ROW) + c.g * Q::ROW);
#pragma unroll
            for (int k = 0; k < kF4; k++) {
                const float4 x = krow[kF4 * c.j + (k ^ sw_of(c.j))];
                acc[4 * k] = sub(x.x, acc[4 * k]); acc[4 * k + 1] = sub(x.y, acc[4 * k + 1]);
                acc[4 * k + 2] = sub(x.z, acc[4 * k + 2]); acc[4 * k + 3] = sub(x.w, acc[4 * k + 3]);
            }
        }
    };

    // One interpreter call site (the phase loop is not unrolled): phase 0 = ops before recurrence 1 on tile i,
    // phase 1 = ops between the recurrences on tile i-1, phase 2 = ops after recurrence 2 on tile i-2.
    const int lo[3] = {0, r1 + 1, r2 + 1}, hi[3] = {r1, r2, prog.n_ops};
    bar_sync(BAR2_EONLY, n_e);
    for (int i = 0; i < nt + 2; i++) {
        // ring stores of a tile's post-ops become visible to the other threads' later ring loads through the DONE
        // syncs (CTA-scope barriers among all elementwise threads, at least one per iteration from i = 1 on)
        // (iteration 1 has no DONE sync before its first edge[] write yet: order it behind iteration 0's reads)
        if (i == 1) bar_sync(BAR2_EONLY, n_e);
#pragma unroll 1
        for (int ph = 0; ph < 3; ph++) {
            const int ti = i - ph;
            if (ti < 0 || ti >= nt) continue;
            float acc[kChunk];
            set_tile(ti);
            if (ph == 0) {
#pragma unroll
                for (int k = 0; k < kChunk; k++) acc[k] = 0.0f;
            } else {
                fetch(ph - 1, ti, acc);
            }
            for (int ip = lo[ph]; ip < hi[ph]; ip++) exec_op<G, true>(prog.ops[ip].code, prog.ops[ip].mode, prog.ops[ip].pre, -1, prog.ops[ip], c, acc, pf);
            if (ph < 2) feed(ph == 0 ? rop1 : rop2, ph, ti, acc);
        }
    }
    bar_sync(BAR2_EONLY, n_e);
    for (int st = 0; st < 2; st++) {
        const Op& rop = st == 0 ? rop1 : rop2;
        if (rop.code != OP_BIQUAD) continue;
        float* stp = prog.states[rop.aux];
        if (Q::TPC <= 32) {
            if (c.j == 0 && c.ch_ok) *reinterpret_cast<float2*>(stp + 4 * (long long)c.ch) = make_float2(cx[st][0], cx[st][1]);
        } else if (t < G) {
            const int ch = c_begin + blockIdx.x * G + t;
            if (ch < c_end) *reinterpret_cast<float2*>(stp + 4 * (long long)ch) = xstate[st * 64 + (nt & 1) * 32 + t];
        }
    }
}

// indices of the two recurrence ops if the program qualifies for fused_kernel_ws2
bool ws2_rec_indices(const Program& p, int* r1, int* r2) {
    if (p.n_vregs != 0) return false;
    int n = 0, idx[2] = {-1, -1};
    for (int i = 0; i < p.n_ops; i++) {
        const int c = p.ops[i].code;
        if (c == OP_BIQUAD || c == OP_LP1 || c == OP_HP1 || c == OP_ENVELOPE) {
            if (n == 2) return false;
            if (p.ops[i].pflags) return false;
            idx[n++] = i;
        }
        if (c == OP_SIGGEN) return false;
    }
    if (n != 2) return false;
    *r1 = idx[0];
    *r2 = idx[1];
    return true;
}

template <int G>
int launch_ws2(const Program& prog, int c_begin, int c_end, int64_t T, int r1, int r2, cudaStream_t st) {
    const int smem = Ws2Smem<G>::bytes;
    static std::atomic<bool> configured_dev[kMaxDevices];
    std::atomic<bool>& configured = configured_dev[current_device_slot()];
    if (!configured.load(std::memory_order_acquire)) {
        cudaError_t e = cudaFuncSetAttribute(fused_kernel_ws2<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return (int)e;
        configured.store(true, std::memory_order_release);
    }
    const int n_cta = (c_end - c_begin + G - 1) / G;
    fused_kernel_ws2<G><<<n_cta, kXrLaunchThreads, smem, st>>>(prog, c_begin, c_end, (long long)T, r1, r2);
    return (int)cudaGetLastError();
}
int ws_smem_bytes(const Program& prog, int G) {
    const int S = kTile / G;
    bool hp = false;
    for (int i = 0; i < prog.n_ops; i++) hp = hp || prog.ops[i].code == OP_HP1;
    return 64 * 8 + kThreads * 8 + (hp ? 4 : 2) * G * (S + 4) * 4 + prog.n_vregs * kTile * 4;
}
// does op read / write shared-memory vreg v?
bool op_reads_vreg(const Op& op, int v) {
    if (op_reads_vreg_field(op.code) && op.vreg == v) return true;
    for (int i = 0; i < 3; i++)
        if ((op.pflags & (1 << i)) && op.pv[i] == v) return true;
    return false;
}
// index of the single recurrence op if the program qualifies for the warp-specialised kernel, else -1.
// Shared-memory vregs are fine as long as none is live ACROSS the recurrence: the elementwise warps run the ops
// before it for tile i and the ops after it for tile i-1 in the same iteration, so a value saved before and read
// after would be overwritten by the next tile in between.
int ws_rec_index(const Program& p) {
    int idx = -1;
    for (int i = 0; i < p.n_ops; i++) {
        const int c = p.ops[i].code;
        if (c == OP_BIQUAD || c == OP_LP1 || c == OP_HP1 || c == OP_ENVELOPE) {
            if (idx >= 0) return -1;
            idx = i;
        }
        if (c == OP_SIGGEN) return -1;
    }
    if (idx < 0) return -1;
    for (int v = 0; v < p.n_vregs; v++) {
        bool before = false, after = false;
        for (int i = 0; i < p.n_ops; i++) {
            const bool touches = op_reads_vreg(p.ops[i], v) || (p.ops[i].code == OP_SAVEV && p.ops[i].vreg == v);
            if (touches && i < idx) before = true;
            if (touches && i > idx) after = true;
        }
        if (op_reads_vreg(p.ops[idx], v)) return -1;  // a control-port tile feeding the recurrence op itself
        if (before && after) return -1;
    }
    return idx;
}

template <int G, class Chain, bool XR>
int launch_ws(const Program& prog, int c_begin, int c_end, int64_t T, int rec_index, cudaStream_t st) {
    const int smem = ws_smem_bytes(prog, G);
    struct DevCfg { std::mutex mu; int configured = -1; int regs = 0; };
    static DevCfg cfg_dev[kMaxDevices];
    DevCfg& dc = cfg_dev[current_device_slot()];
    int regs;
    {
        std::lock_guard<std::mutex> lk(dc.mu);
        if (smem > dc.configured) {
            cudaError_t e = cudaFuncSetAttribute(fused_kernel_ws<G, Chain, XR>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
            if (e != cudaSuccess) return (int)e;
            dc.configured = smem;
            cudaFuncAttributes fa;
            if (cudaFuncGetAttributes(&fa, fused_kernel_ws<G, Chain, XR>) == cudaSuccess) dc.regs = fa.numRegs;
        }
        regs = dc.regs;
    }
    if (XR) {
        const int n_cta = (c_end - c_begin + G - 1) / G;
        fused_kernel_ws<G, Chain, true><<<n_cta, kXrLaunchThreads, smem, st>>>(prog, c_begin, c_end, (long long)T, G, rec_index);
        return (int)cudaGetLastError();
    }
    // Channels per CTA: G, or a smaller power of two when a channel is one warp (TPC == 32): smaller CTAs (8 channels
    // = 9 warps, 4 resident per SM) balance better and measured 0.344 ms against 0.368 ms for the config-3 chain at
    // 4096 channels.  The grid has to stay ONE wave, and the capacity that counts is not n_sm x CTAs-per-SM:
    // measured on B200 (a sweep over gc, profiles/r01s3_fused_gc_sweep.txt), CTAs are dealt evenly to the 8 GPCs
    // and the smallest GPC has 16 SMs, so a grid runs in one wave only while n_cta / 8 <= 16 x CTAs-per-SM.
    // 293 CTAs of 14 channels (a "perfectly balanced" 2 per SM on paper) took 2.1x as long: the CTAs that did not
    // fit their GPC started when the first ones had finished (ncu: sm__cycles_active min 437 K / max 1506 K).
    int gc = G;
    if (Geo<G>::TPC == 32 && regs > 0) {
        const int n = c_end - c_begin;
        for (int g = G / 2; g >= 8; g >>= 1) {
            const int warps = g + 1;  // one elementwise warp per channel, and the R warp
            const int cps = std::min(65536 / (regs * 32 * warps), (227 * 1024) / (smem + 1024));
            const int n_cta = (n + g - 1) / g;
            if (cps >= 1 && (n_cta + 7) / 8 <= 16 * cps) gc = g;
        }
    }
    const int n_cta = (c_end - c_begin + gc - 1) / gc;
    fused_kernel_ws<G, Chain, false><<<n_cta, gc * Geo<G>::TPC + 32, smem, st>>>(prog, c_begin, c_end, (long long)T, gc, rec_index);
    return (int)cudaGetLastError();
}

template <class Chain>
bool chain_matches(const Program& p) {
    if (Chain::n == 0 || p.n_ops != Chain::n) return false;
    for (int i = 0; i < Chain::n; i++) {
        const int s = Chain::sig(i);
        const Op& o = p.ops[i];
        if (o.code != (s & 0xff) || o.pre != ((s >> 16) & 0xff) || o.pflags != 0) return false;
        if (op_pc_col(o) >= 0) return false;  // per-channel parameters: the interpreter (ChainDynamic) runs them
        if (o.code == OP_DISTORT && o.mode != ((s >> 8) & 0xff)) return false;
        if ((o.code == OP_BIQUAD || o.code == OP_LP1 || o.code == OP_HP1) && o.mode != ((s >> 8) & 0xff)) return false;  // exact vs scan
        const bool is_src = o.code == OP_LOADG || o.code == OP_ADDG || o.code == OP_COPYG || o.code == OP_STOREG;
        const int has = is_src ? (o.aux != 0) : o.code == OP_COMB ? ((o.aux >> 8) != 0) : 0;
        if (has != Chain::pf_of(i)) return false;
    }
    return true;
}

template <int G, class Chain>
int launch_gc(const Program& prog, int c_begin, int c_end, int64_t T, int n_states, cudaStream_t st) {
    const int smem = fused_smem_bytes(prog, G);
    struct DevCfg { std::mutex mu; int configured = -1; int n_sm = 0; };
    static DevCfg cfg_dev[kMaxDevices];
    DevCfg& dc = cfg_dev[current_device_slot()];
    int n_sm;
    {
        std::lock_guard<std::mutex> lk(dc.mu);
        if (smem > dc.configured) {
            cudaError_t e = cudaFuncSetAttribute(fused_kernel<G, Chain>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
            if (e != cudaSuccess) return (int)e;
            dc.configured = smem;
        }
        if (!dc.n_sm) {
            int dev = 0;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&dc.n_sm, cudaDevAttrMultiProcessorCount, dev);
            if (dc.n_sm <= 0) dc.n_sm = 148;
        }
        n_sm = dc.n_sm;
    }
    const int n_cta = (c_end - c_begin + G - 1) / G;
    fused_kernel<G, Chain><<<n_cta, kThreads, smem, st>>>(prog, c_begin, c_end, (long long)T, n_states, n_sm);
    return (int)cudaGetLastError();
}

template <int G>
int launch_g(const Program& prog, int c_begin, int c_end, int64_t T, int n_states, cudaStream_t st) {
    // a recurrence in scan mode has no sequential part to hide: such programs take the plain kernel
    const bool no_ws = prog.n_scan > 0;
    {   // two recurrences in series: pipelined over two recurrence warps
        int r1 = -1, r2 = -1;
        if (!no_ws && G <= 16 && ws2_rec_indices(prog, &r1, &r2) && Ws2Smem<G>::bytes <= 200 * 1024) {
            // only the chain-bound regime (one CTA per SM, one wave) has a variant: with many channels per SM the
            // elementwise work dominates and the plain kernel below is as good
            if ((c_end - c_begin + G - 1) / G <= 128) return launch_ws2<G>(prog, c_begin, c_end, T, r1, r2, st);
        }
    }
    const int rec = (G <= 32 && !no_ws) ? ws_rec_index(prog) : -1;
    if (rec >= 0 && ws_smem_bytes(prog, G) <= 200 * 1024) {
        // chain-bound launches (at most one CTA per SM and one wave: n_cta <= 8 GPCs x 16 SMs) give the recurrence
        // warp a sub-partition of its own
        const bool xr = (c_end - c_begin + G - 1) / G <= 128 && prog.n_vregs == 0 && prog.n_ops <= 8;
        if (xr) {
            if (chain_matches<ChainGDBR<3>>(prog)) return launch_ws<G, ChainGDBR<3>, true>(prog, c_begin, c_end, T, rec, st);
            return launch_ws<G, ChainDynamic, true>(prog, c_begin, c_end, T, rec, st);
        }
        if (chain_matches<ChainGDBR<3>>(prog)) return launch_ws<G, ChainGDBR<3>, false>(prog, c_begin, c_end, T, rec, st);
        if (chain_matches<ChainGDBR<1>>(prog)) return launch_ws<G, ChainGDBR<1>, false>(prog, c_begin, c_end, T, rec, st);
        return launch_ws<G, ChainDynamic, false>(prog, c_begin, c_end, T, rec, st);
    }
    if (chain_matches<ChainGDBR<3>>(prog)) return launch_gc<G, ChainGDBR<3>>(prog, c_begin, c_end, T, n_states, st);
    if (chain_matches<ChainGDBRScan<3>>(prog)) return launch_gc<G, ChainGDBRScan<3>>(prog, c_begin, c_end, T, n_states, st);
    if (chain_matches<ChainGDR<3>>(prog)) return launch_gc<G, ChainGDR<3>>(prog, c_begin, c_end, T, n_states, st);
    if (chain_matches<ChainGDR<1>>(prog)) return launch_gc<G, ChainGDR<1>>(prog, c_begin, c_end, T, n_states, st);
    if (chain_matches<ChainBB<1>>(prog)) return launch_gc<G, ChainBB<1>>(prog, c_begin, c_end, T, n_states, st);
    if (chain_matches<ChainLH<1>>(prog)) return launch_gc<G, ChainLH<1>>(prog, c_begin, c_end, T, n_states, st);
    if (chain_matches<ChainCopy<1>>(prog)) return launch_gc<G, ChainCopy<1>>(prog, c_begin, c_end, T, n_states, st);
    return launch_gc<G, ChainDynamic>(prog, c_begin, c_end, T, n_states, st);
}

}  // namespace
// Exhaustive device-side proof that div_const(a, {b, r}) == a / b (IEEE) for ALL 2^32 dividends a that
// it does not flag: the engine enables the 3-instruction division for a divisor only after this passed.
namespace {
__global__ void div_verify_kernel(float b, float r, unsigned long long* mism) {
    const unsigned long long base = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) * 256ull;
    unsigned long long m = 0;
    for (int k = 0; k < 256; k++) {
        const float a = __uint_as_float((unsigned)(base + k));
        float mn = kDivHi, mx = 0.0f;
        const float q = div_const(a, ConstDiv{b, r}, mn, mx);
        const float ref = __fdiv_rn(a, b);
        if (div_const_accept(mn, mx) && __float_as_uint(q) != __float_as_uint(ref) && !(q != q && ref != ref)) m++;
    }
    if (m) atomicAdd(mism, m);
}
// The same proof for div_const2 (zh, zl) under its own acceptance rule: the engine's first tier.
__global__ void div2_verify_kernel(float b, float zh, float zl, unsigned long long* mism) {
    const unsigned long long base = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) * 256ull;
    unsigned long long m = 0;
    for (int k = 0; k < 256; k++) {
        const float a = __uint_as_float((unsigned)(base + k));
        float mn = kDiv2Hi, mx = 0.0f;
        const float q = div_const2(a, ConstDiv2{zh, zl}, mn, mx);
        const float ref = __fdiv_rn(a, b);
        if (div_const2_accept(mn, mx) && __float_as_uint(q) != __float_as_uint(ref) && !(q != q && ref != ref)) m++;
    }
    if (m) atomicAdd(mism, m);
}
template <class Launch>
int count_mismatches(Launch launch, unsigned long long* mismatches) {
    unsigned long long* d = nullptr;
    cudaError_t e = cudaMalloc(&d, 8);
    if (e != cudaSuccess) return (int)e;
    cudaMemset(d, 0, 8);
    launch(d);
    e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpy(mismatches, d, 8, cudaMemcpyDeviceToHost);
    cudaFree(d);
    return (int)e;
}
}  // namespace

int verify_const_div(float b, float r, unsigned long long* mismatches) {
    return count_mismatches([&](unsigned long long* d) { div_verify_kernel<<<65536, 256>>>(b, r, d); }, mismatches);
}
int verify_const_div2(float b, float zh, float zl, unsigned long long* mismatches) {
    return count_mismatches([&](unsigned long long* d) { div2_verify_kernel<<<65536, 256>>>(b, zh, zl, d); }, mismatches);
}

// Probe for one recurrence: the same op in exact and in scan mode over 8 channels x 16384 samples (four of uniform noise,
// four log sweeps 20 Hz - 20 kHz, amplitude 0.5), zero initial state; the result gates scan mode for this coefficient set.
int measure_scan_error(const Op& exact_op, const ScanTab& tab, float* rel_err) {
    constexpr int C = 8, G = 4;
    constexpr int64_t T = 16384;
    std::vector<float> x((size_t)C * T);
    unsigned long long lcg = 0x9E3779B97F4A7C15ull;
    for (int c = 0; c < C; c++)
        for (int64_t n = 0; n < T; n++) {
            float v;
            if (c < 4) {
                lcg = lcg * 6364136223846793005ull + 1442695040888963407ull;
                v = ((float)(int)((lcg >> 40) & 0xFFFFFF) - 8388608.0f) * (1.0f / 8388608.0f) * 0.5f;
            } else {
                const double t = (double)n / 48000.0, Ts = (double)T / 48000.0, k = std::log(1000.0);
                v = (float)(0.5 * std::sin(2.0 * M_PI * 20.0 * Ts / k * (std::exp(t / Ts * k) - 1.0) + 0.7 * c));
            }
            x[(size_t)c * T + n] = v;
        }
    float *dx = nullptr, *dy = nullptr, *ds = nullptr;
    cudaError_t e;
    if ((e = cudaMalloc(&dx, x.size() * 4)) != cudaSuccess) return (int)e;
    if ((e = cudaMalloc(&dy, 2 * x.size() * 4)) != cudaSuccess) { cudaFree(dx); return (int)e; }
    if ((e = cudaMalloc(&ds, 2 * C * 16)) != cudaSuccess) { cudaFree(dx); cudaFree(dy); return (int)e; }
    cudaMemcpy(dx, x.data(), x.size() * 4, cudaMemcpyHostToDevice);
    cudaMemset(ds, 0, 2 * C * 16);
    int rc = 0;
    for (int m = 0; m < 2 && rc == 0; m++) {
        Program P;
        memset(&P, 0, sizeof P);
        P.n_ops = 3;
        P.ops[0].code = OP_LOADG; P.ops[0].buf = 0;
        P.ops[1] = exact_op;
        P.ops[1].pre = 0; P.ops[1].pflags = 0; P.ops[1].aux = 0; P.ops[1].mode = (uint8_t)m;
        P.ops[2].code = OP_STOREG; P.ops[2].buf = 1;
        P.needs_tile = m == 0;
        P.n_scan = (int16_t)m;
        P.scan[0] = tab;
        P.bufs[0] = BufDesc{dx, T, 0, 0};
        P.bufs[1] = BufDesc{dy + (size_t)m * C * T, T, 0, 0};
        P.states[0] = ds + (size_t)m * C * 4;
        for (int k = 0; k < kMaxPrefetch; k++) P.pf_buf[k] = P.pf_ring[k] = -1;
        P.st_buf = -1;
        rc = launch_fused(P, G, 0, C, T, nullptr);
    }
    std::vector<float> y(2 * x.size());
    if (rc == 0) rc = (int)cudaMemcpy(y.data(), dy, y.size() * 4, cudaMemcpyDeviceToHost);
    cudaFree(dx); cudaFree(dy); cudaFree(ds);
    if (rc) return rc;
    double peak = 0.0, err = 0.0;
    bool finite = true;
    for (size_t i = 0; i < x.size(); i++) {
        const double a = y[i], b = y[x.size() + i];
        finite = finite && std::isfinite(a) && std::isfinite(b);
        peak = std::max(peak, std::fabs(a));
        err = std::max(err, std::fabs(a - b));
    }
    *rel_err = (finite && peak > 0.0) ? (float)(err / peak) : 1.0f;  // an unstable filter never qualifies
    return 0;
}

int fused_smem_bytes(const Program& prog, int G) {
    const int S = kTile / G;
    size_t b = (size_t)kMaxStates * G * 16 + (size_t)kThreads * 8 + (size_t)(kThreads / 32) * 16;
    if (prog.needs_tile) b += (size_t)G * (S + 4) * 4;
    b += (size_t)prog.n_vregs * kTile * 4;
    return (int)b;
}

int launch_fused(const Program& prog, int G, int c_begin, int c_end, int64_t T, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (T <= 0 || T > (1ll << 30)) return (int)cudaErrorInvalidValue;  // the kernels index samples of one call with int
    for (int k = 0; k < kMaxPrefetch; k++)
        if (prog.pf_ring[k] >= 0 && prog.rings[prog.pf_ring[k]].D > (1ll << 30)) return (int)cudaErrorInvalidValue;
    int n_states = 0;
    for (int i = 0; i < kMaxStates; i++)
        if (prog.states[i]) n_states = i + 1;
    switch (G) {
        case 1: return launch_g<1>(prog, c_begin, c_end, T, n_states, st);
        case 2: return launch_g<2>(prog, c_begin, c_end, T, n_states, st);
        case 4: return launch_g<4>(prog, c_begin, c_end, T, n_states, st);
        case 8: return launch_g<8>(prog, c_begin, c_end, T, n_states, st);
        case 16: return launch_g<16>(prog, c_begin, c_end, T, n_states, st);
        case 32: return launch_g<32>(prog, c_begin, c_end, T, n_states, st);
    }
    return (int)cudaErrorInvalidValue;
}

}  // namespace dspb
