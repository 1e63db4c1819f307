// exact_math.cuh — f32 arithmetic that must round exactly like the reference's (rustc: IEEE, no FMA
// contraction, no reassociation).  The *_rn intrinsics are never contracted by nvcc.
#pragma once
#include <cuda_runtime.h>

namespace dspb {

__device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float dv(float a, float b) { return __fdiv_rn(a, b); }

// Correctly rounded a / b for a divisor known on the host (b > 0, r = RN(1/b) in IEEE f32).
// Markstein's sequence: q0 = RN(a*r); rem = a - q0*b (one FMA); q1 = RN(q0 + rem*r).  Measured on the
// device over all 2^32 dividends (tests/cuda/div_explore.cu): q1 == RN(a/b) for EVERY dividend whose
// biased exponent lies in [30, 220]; the only failures are in the underflow fringe (rem loses bits),
// the overflow fringe, +-inf and -0.  So the caller keeps the running min of |q1| and max of |a| over
// its chunk and accepts the fast results only if min|q1| >= 2^-90 and max|a| <= 2^90 (a chunk with
// zeros, denormal tails or infinities is redone with __fdiv_rn, which is always right).  The engine
// additionally enables this path per divisor only after verify_const_div() enumerated all 2^32
// dividends under exactly this acceptance rule with zero mismatches.
struct ConstDiv {
    float b, r;
};
constexpr float kDivLo = 8.0779357e-28f;  // 2^-90
constexpr float kDivHi = 1.2379400e27f;   // 2^90
__device__ __forceinline__ float div_const(float a, const ConstDiv d, float& mn_q, float& mx_a) {
    const float q0 = __fmul_rn(a, d.r);
    const float rem = __fmaf_rn(-q0, d.b, a);
    const float q1 = __fmaf_rn(rem, d.r, q0);
    mn_q = fminf(mn_q, fabsf(q1));
    mx_a = fmaxf(mx_a, fabsf(a));
    return q1;
}
__device__ __forceinline__ bool div_const_accept(float mn_q, float mx_a) { return mn_q >= kDivLo && mx_a <= kDivHi; }

// Correctly rounded a / b in two instructions (Brisebarre, Muller, Raina, "Accelerating correctly rounded floating-point
// division when the divisor is known in advance", IEEE TC 53(8), 2004): zh = RN(1/b), zl = RN(1/b - zh) (formed in double
// on the host), q = RN(a*zh + RN(a*zl)) with one FMUL and one FFMA.  Like div_const it is exact for many divisors but not
// all, and it goes wrong where a*zl underflows or q leaves the normal range.  The host enables it only for divisors in
// [2^-20, 2^20], so a bound on |a| alone bounds |q|: the caller keeps the running min and max of |a| over its chunk and
// accepts the fast results only if min|a| >= 2^-96 and max|a| <= 2^96 (a chunk with zeros, denormals, huge values or
// infinities is redone with __fdiv_rn).  Inside an accepted chunk a != 0, so a fan-in prologue's `0.0 + a` is a and can be
// left to the fallback.  The engine enables this form per divisor only after verify_const_div2() enumerated all 2^32
// dividends under exactly this acceptance rule with zero mismatches.
struct ConstDiv2 {
    float zh, zl;
};
constexpr float kDiv2Lo = 0x1p-96f;
constexpr float kDiv2Hi = 0x1p96f;
__device__ __forceinline__ float div_const2(float a, const ConstDiv2 d, float& mn_a, float& mx_a) {
    mn_a = fminf(mn_a, fabsf(a));
    mx_a = fmaxf(mx_a, fabsf(a));
    return __fmaf_rn(a, d.zh, __fmul_rn(a, d.zl));
}
__device__ __forceinline__ bool div_const2_accept(float mn_a, float mx_a) { return mn_a >= kDiv2Lo && mx_a <= kDiv2Hi; }

}  // namespace dspb
