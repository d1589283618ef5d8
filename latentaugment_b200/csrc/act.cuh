// Activation backward from a SAVED output, shared by every kernel that needs it: the tap-GEMM backward and linear
// epilogues, the two gradient-seed passes, the FIR passes with an activation backward and the discriminator's
// minibatch-stddev backward.
//
// The forward stores y = clamp(lrelu(z) * gain, -c, c) as bf16 (the hi plane), in split mode plus the bf16 residual
// (the lo plane, lo = bf16_rn(y - hi)).  A unit clamped to c is therefore stored as bf16_rn(c) (+ the residual of c),
// which can lie BELOW c: c = 256 sqrt(1/2) = 181.019 is stored as 181.0, c = 0.7 as 0.69921875.  Compared with c itself
// such a unit reads as unclamped and passes its gradient where the reference's (fp32 output, bias_act.cu) is 0.  So the
// clamped test compares with the clamp AS THE SAVED TENSOR STORES IT.  (An unclamped unit within one bf16 step below c
// then reads as clamped: the error moves from a point mass of clamped units to a thin window of unclamped ones.)
#pragma once

#include <cuda_bf16.h>

// The threshold of the clamped test: |saved| >= it  <=>  the unit was clamped.  with_lo: the reader adds the lo plane to
// the hi plane in fp32 (this sum is rounded the same way).  c < 0: no clamp.  For c = 256 the threshold is c.
__device__ __forceinline__ float act_saved_clamp(float c, bool with_lo) {
    if (!(c >= 0.f)) return __int_as_float(0x7f800000);
    const float hi = __bfloat162float(__float2bfloat16_rn(c));
    return with_lo ? hi + __bfloat162float(__float2bfloat16_rn(c - hi)) : hi;
}

// Gradient g (activation gain already applied) through lrelu + clamp, decided by the saved output s:
// g * (s > 0 ? 1 : slope), and 0 where the unit was clamped (thr from act_saved_clamp).
__device__ __forceinline__ float act_grad(float g, float s, float slope, float thr) {
    return fabsf(s) < thr ? g * (s > 0.f ? 1.f : slope) : 0.f;
}
