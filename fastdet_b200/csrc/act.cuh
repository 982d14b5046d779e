// act.cuh — Mish, x * tanh(softplus(x)), for the convolution epilogues (fp32 in, fp32 out).
//
// One special-function instruction per element: e = exp(x) by ex2.approx, then tanh(log1p(e)) = n / (n + 2) with
// n = e (e + 2) = (1 + e)^2 - 1, exact algebra.  The reciprocal of d = n + 2 >= 2 is an integer first guess (relative
// error < 1/8) refined by three Newton steps on the FMA pipe, so the MUFU pipe (16 ops / clock / SM, a quarter of the
// FMA rate) issues the ex2 only.  For x > 20, tanh(softplus(x)) rounds to 1 in fp32 and mish(x) = x (this also keeps n
// from overflowing).  Error against the exact Mish of the fp32 input: the rounding of x * log2(e) is a relative change of
// x by 2^-24 (counted with the accumulation's roundings, tests/mish_compare.py); the rest stays within 6 * 2^-23 of |mish|:
// ex2.approx <= 2, n <= 1, n + 2 <= 1/2, the reciprocal <= 3/2, the two products <= 1 (units of 2^-23, relative).
#pragma once
#include <stdint.h>

namespace fd {

__device__ __forceinline__ float mish_f32(float x) {
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 1.44269504088896341f));
    const float n = e * (e + 2.f);
    const float d = n + 2.f;
    float r = __int_as_float(0x7EF311C3 - __float_as_int(d));
#pragma unroll
    for (int i = 0; i < 3; ++i) r = fmaf(r, fmaf(-d, r, 1.f), r);
    const float y = x * (n * r);
    return x > 20.f ? x : y;
}

// bias + Mish on two accumulator columns
__device__ __forceinline__ float2 bias_mish2(uint32_t a0, uint32_t a1, float b0, float b1) {
    const float2 x = __fadd2_rn(make_float2(__uint_as_float(a0), __uint_as_float(a1)), make_float2(b0, b1));
    return make_float2(mish_f32(x.x), mish_f32(x.y));
}

}  // namespace fd
