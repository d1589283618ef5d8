// Perceptual (LPIPS) term of the LatentAugment loop: VGG16 feature extractor + LPIPS distance to the bank of real
// features, forward and gradient back to the image (reference calc_loss_lpips_torchscript / calc_loss_lpips_tr,
// augments/utils/util_latent_aug.py:387-424; augments/criteria/lpips/{lpips,networks,utils}.py).
// Plain 3x3 convolutions on the same tap-GEMM kernel as the generator; see lpips.cu.
#pragma once
#include <cuda_runtime.h>

#include "../../include/latentaugment_b200.h"

struct la_lpips;

namespace la {

int lpips_workspace_bytes(const la_vgg_desc& d, int batch, int img_channels, int split, size_t* bytes);
int lpips_create(const la_vgg_desc& d, int batch, int img_channels, int img_resolution, int split, int num_sms, void* ws, size_t bytes,
                 cudaStream_t s, la_lpips** out);
void lpips_destroy(la_lpips* L);

// Bank of real crops [M, img_channels, crop, crop] fp32 in [-1, 1] (already cropped by the caller, one random window
// per image like util_latent_aug.py:564-579): only the bank MOMENTS of the normalised activations are kept.
int lpips_set_bank(la_lpips* L, const float* d_crops, int M, cudaStream_t s, long long* launches);
int lpips_has_bank(const la_lpips* L);

// Per-call constants (device-resident so a captured graph serves every call): crop window origin inside the image
// (absolute pixel coordinates), term weight, pair normaliser (0: mean over (sample, bank) pairs -- the lpips_script
// form; 1: sum over samples of the bank mean -- the forward_tr form).  Asynchronous on s.
int lpips_set_call(la_lpips* L, int crop_x, int crop_y, float w_lpips, int norm_mode, cudaStream_t s);

// img: float4 per pixel [B, R, R].  Crops, z-scores and runs VGG16 up to the last tap.  targets != 0: the window is the whole
// image (crop origin 0, 0), area-pooled 2x2 when the image is twice the crop (per-sample-target mode).
int lpips_forward(la_lpips* L, const float4* img, int targets, cudaStream_t s, long long* launches);
// (after lpips_forward) loss value = w_lpips * mean over modalities of the pair-normalised LPIPS distance -> d_loss[0];
// g_img[pix] (+)= d(-loss)/d img  (the term enters the objective with a minus sign, util_latent_aug.py:270).
// targets != 0 (projection): d_loss[b] = sum over modalities and taps of sample b's distance to its own target,
// g_img (+)= d (sum_b d_loss[b]) / d img  (minimised, so no sign flip and no w_lpips / pair normaliser).
int lpips_backward(la_lpips* L, float4* g_img, int accumulate, float* d_loss, int targets, cudaStream_t s, long long* launches);

// Per-sample targets of the projection: img float4 [B, R, R] -> normalised activations per (sample, modality, tap), fp32.
// Needs la_vgg_desc.per_sample_targets (the storage is planned in the workspace).  Sets the call constants to the whole window.
int lpips_set_targets(la_lpips* L, const float4* img, cudaStream_t s, long long* launches);
int lpips_has_targets(const la_lpips* L);

// Test hook: normalised activations of tap k of the crops computed by the last lpips_forward -> fp32 [n_crops, h, w, C] (NHWC).
int lpips_copy_tap(la_lpips* L, int k, float* d_out, size_t* count, cudaStream_t s);
int lpips_num_taps(const la_lpips* L);

}  // namespace la
