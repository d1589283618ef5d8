// StyleGAN2 'resnet' discriminator of the realism term (reference calc_loss_disc,
// augments/utils/util_latent_aug.py:363-371): forward, loss and the gradient back to the image.
// Plain (unmodulated) layers on the same tap-GEMM kernel as the generator; see disc.cu.
#pragma once
#include <cuda_runtime.h>

#include "../../include/latentaugment_b200.h"

struct la_disc;

namespace la {

int disc_workspace_bytes(const la_disc_desc& d, int batch, int split, size_t* bytes);
// split = 1: split-bf16 (hi/lo) operands like the engine's fp32_parity precision
int disc_create(const la_disc_desc& d, int batch, int split, int num_sms, void* ws, size_t bytes, cudaStream_t s, la_disc** out);
void disc_destroy(la_disc* D);

// img: float4 per pixel [B, R, R] (channel k in .x / .y / .z).  Leaves the logits in disc_logits().
int disc_forward(la_disc* D, const float4* img, cudaStream_t s, long long* launches);
// loss = w_disc * mean softplus(-logit) -> d_loss[0];  g_img[pix] (+)= d loss / d img  (after disc_forward)
int disc_backward(la_disc* D, float w_disc, float4* g_img, int accumulate, float* d_loss, cudaStream_t s, long long* launches);
const float* disc_logits(const la_disc* D);
int disc_batch(const la_disc* D);
int disc_resolution(const la_disc* D);
int disc_channels(const la_disc* D);

// NCHW fp32 <-> float4-per-pixel image converters (stand-alone entry points)
int nchw_to_f4(const float* src, int batch, int C, int res, float4* dst, cudaStream_t s);
int f4_to_nchw(const float4* src, int batch, int C, int res, float* dst, cudaStream_t s);

}  // namespace la
