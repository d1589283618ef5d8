// Forward half of torchvision's VGG16 `features` on the tap-GEMM, shared by the perceptual term (lpips.cu) and the
// VGG16 detector (detector.cu): weight preparation and the 2x2 max-pool.  Each 3x3 convolution + bias + ReLU is a plain
// layer of plan.cuh (plan_layer, then fwd_epilogue with gain 1, no clamp and slope 0).  Activations are NHWC bf16 (hi, plus
// the lo plane in split precision).  Implemented in lpips.cu.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include "common.cuh"

namespace la {

constexpr int kNConv = 13;
constexpr int kCout[kNConv] = {64, 64, 128, 128, 256, 256, 256, 512, 512, 512, 512, 512, 512};
constexpr int kCin[kNConv] = {3, 64, 64, 128, 128, 256, 256, 256, 512, 512, 512, 512, 512};
constexpr int kShift[kNConv] = {0, 0, 1, 1, 2, 2, 2, 3, 3, 3, 4, 4, 4};       // resolution = input >> shift
constexpr int kPoolConv[5] = {1, 3, 6, 9, 12};                                 // convs followed by a max-pool

// w [cout, cin, 3, 3] fp32 -> wf [9][cout][cin_pad] (forward operand) and, unless wb is null, wb [9][cin_pad][cout]
// (data-gradient operand); zero padded, residual planes behind the main ones when split.
int vgg_prep_weights(const float* w, int cout, int cin, int cin_pad, int split, __nv_bfloat16* wf, __nv_bfloat16* wb, cudaStream_t s);
// 2x2 max-pool x [n, R, R, C] -> out [n, R/2, R/2, C].
int vgg_pool_fwd(const Pl& x, int n, int R, int C, const Pl& out, cudaStream_t s);

}  // namespace la
