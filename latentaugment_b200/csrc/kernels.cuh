// Small SIMT kernels around the tap-GEMM: weight preparation, style / demodulation
// coefficients, toRGB + skip pyramid (forward and backward), criteria, style gradients,
// the fused Adam step on w, the mapping network and bank statistics.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace la {

constexpr int kMaxLayers = 24;    // conv layers (<= 2*log2(res)-3) ; rgb layers (<= log2(res)-1)

// All "cat" arrays are layer-blocked: element (layer, n, i) lives at batch*off_l + n*dim_l + i.
struct ConvDesc {
    const float* w2;     // [cout][cin]  sum_k w^2
    const float* w2t;    // [cin][cout]
    int cin, cout;
    int soff;            // style block offset (rows of A_cat)
    int doff;            // demod block offset
    int ws_idx;          // which row of ws feeds the affine
};
struct RgbDesc {
    const float* wt;     // [img_c][cin]
    int cin, img_c;
    int soff;            // style block offset
    int roff;            // offset (in float4 / float columns) of this layer's rgbw / red_rgb block
    int ws_idx;
};
struct LayerTable {
    ConvDesc conv[kMaxLayers];
    RgbDesc rgb[kMaxLayers];
    int nconv, nrgb;
};

// ---- one-time preparation
int prep_conv_weights(const float* w, int cout, int cin, int up, const float* fir4x4, int split, void* wf, void* wb,
                      float* w2, float* w2t, cudaStream_t s);
int prep_affine(const float* aw, const float* ab, int cin, int w_dim, float wscale, float bscale, float* a_cat_rows,
                float* b_cat_rows, cudaStream_t s);
int prep_scale(const float* src, float scale, float* dst, long long n, cudaStream_t s);
int prep_axpy(const float* x, float a, float* y, long long n, cudaStream_t s);      // y += a x
int prep_const(const float* cst /*[C,4,4]*/, int C, int hw, float* c_f32 /*[hw][C]*/, void* hi, void* lo, cudaStream_t s);

// ---- x2 up-sampling conv, split form: transposed-conv GEMM -> T [(2H+1) x (2W+1)] -> 4x4 FIR (pad 1, gain 4)
// (reference conv2d_resample.py:112-129 + upfirdn2d.py:167-211), fused with the layer epilogue.
struct UpFirParams {
    const void* t_hi; const void* t_lo;      // bf16 T / g_T  [B, TH, TWp, C]  (TH = 2H+1 rows, TWp = pitch >= 2W+1)
    int B, OH, OW, C, TH, TWp, split;
    float fk[16];                            // fk[jy*4+jx] = F[3-jy][3-jx] * 4   (true convolution, gain up^2)
    float fy[4], fx[4]; int separable;       // fk = fy (x) fx when the filter is rank 1 (setup_filter([1,3,3,1]) is)
    // forward epilogue (same meaning as TapGemmParams)
    const float* demod; const float* bias; const float* noise; long long noise_stride_n; float noise_scale;
    const float* s_next;
    void* x_hi; void* x_lo; void* xs_hi; void* xs_lo;
    float act_gain, act_clamp, act_slope;
    // forward, activation-backward variant (discriminator: gradient through blur + lrelu): when act_saved is set the
    // epilogue is  y = FIR(T) * act_gain * (saved > 0 ? 1 : act_slope), 0 where saved is clamped (act.cuh)  -> x_hi
    const void* act_saved;                   // bf16 [B, OH, OW, C] saved activation output, or null
    const void* act_saved_lo;                // its residual plane (split mode, sliding-window kernel), or null
    // backward: g_y [B, OH, OW, C] -> g_T
    const void* gy_hi; const void* gy_lo;
    void* gt_hi; void* gt_lo;
    // TMA-pipelined variant (bf16 mode, separable filter, OW >= 32, C % 64 == 0): tensor maps over
    // [C, width, height, B] with boxes [64, 35, 1, 1] (loads, no swizzle) and [64, 8, 1, 1] (stores).
    int use_tma;
    alignas(64) CUtensorMap fwd_in, fwd_out_x, fwd_out_xs;     // T -> x, x * s_next
    alignas(64) CUtensorMap bwd_in, bwd_out;                   // g_y -> g_T
};
int upfir_forward(const UpFirParams& p, cudaStream_t s);
int upfir_backward(const UpFirParams& p, cudaStream_t s);

// ---- per step
int styles_forward(const LayerTable& T, const float* ws, long long ws_stride_n, long long ws_stride_idx, const float* a_cat,
                   const float* b_cat, int w_dim, int batch, float* s_cat, cudaStream_t s);
int demod_rgbw_forward(const LayerTable& T, int batch, const float* s_cat, float* d_cat, float4* rgbw, cudaStream_t s);
int const_modulate(const float* c_f32, const float* s0 /*[B,C]*/, int batch, int hw, int C, int split, void* xs_hi, void* xs_lo,
                   cudaStream_t s);
int rgb_combine(const float4* parts, int nparts, const float* bias, int img_c, float clamp, const float4* img_low, int batch,
                int res, float4* img, float* out_nchw /*or null*/, cudaStream_t s);
int rgb_backward(const float4* g_img, const float4* parts, int nparts, const float* bias, int img_c, float clamp, int batch,
                 int res, float4* g_rgb, float4* g_img_low /*or null*/, cudaStream_t s);
int pix_loss(const float4* img, const float4* bank_mean, const float* bank_m2 /*[4]*/, int batch, int res, int img_c,
             int crop_off, int crop_size, float w_pix, float4* g_img, float* loss_parts, int* nparts_out, cudaStream_t s);
int style_grad(const LayerTable& T, int batch, const float* s_cat, const float* d_cat, const float* red_s, const float* red_d,
               const float* red_rgb, float* g_s, cudaStream_t s);
int gw_partial(const float* g_s, const float* a_cat, const int* chunk_soff, const int* chunk_cin, int nchunks, int batch,
               int w_dim, float* partial, cudaStream_t s);

struct AdamConsts {      // device-resident so one captured graph serves every option set
    float lr, beta1, beta2, eps;
    float w_latent, w_pix;
    int num_ws, has_bank;
};
int adam_step(const float* partial, int nchunks, int use_partial, const float* w_sum_bank, const float* lat_m2, const AdamConsts* consts, int* step_counter,
              float* w, float* m, float* v, int batch, int w_dim, const float* pix_parts, int n_pix_parts, const float* bank_m2,
              int img_c, int crop_size, float* loss_log, int max_steps, const float* disc_loss /*or null*/, const float* lpips_loss /*or null*/,
              cudaStream_t s);
// Projection (la_project): the per-step schedule, device-resident so one captured graph serves every call.
struct ProjConsts {
    const float* lr;          // [num_steps]
    const float* sigma;       // [num_steps] absolute w-noise scale
    const float* noise;       // [num_steps, batch, w_dim] unit normal, or null
    int num_steps;
};
// Adam step with lr = lr[t] (t = *step_counter), then w_pert = w + sigma[t+1] * noise[t+1] (the code the next step's style
// GEMMs read; the gradient wrt the perturbed code is the gradient wrt w), then ++*step_counter.
int adam_scheduled(const float* partial, int nchunks, const ProjConsts* pc, int* step_counter, float* w, float* m, float* v,
                   float* w_pert, int batch, int w_dim, cudaStream_t s);
// w_pert = w + sigma[0] * noise[0]  (the code of step 0)
int perturb_first(const float* w, const ProjConsts* pc, float* w_pert, int batch, int w_dim, cudaStream_t s);
// out[0] = sum of x[0..n)
int sum_floats(const float* x, int n, float* out, cudaStream_t s);
constexpr int kLossCols = 5;      // loss-log row: latent, pixel, total, discriminator, perceptual (== LA_LOSS_COLS)
int finalize_w(const float* w_opt, const float* w0, float alpha, int soft, int batch, int w_dim, float* w_aug, cudaStream_t s);

// ---- banks
int latent_bank_stats(const float* W, int M, int num_ws, int w_dim, float* w_sum /*[w_dim]*/, float* m2 /*[1]*/, cudaStream_t s);
int image_bank_stats(const float* X /*[M,C,res,res]*/, int M, int C, int res, int crop_off, int crop_size, float4* mean,
                     float* m2 /*[4]*/, cudaStream_t s);

// ---- mapping network
int mapping_normalize(const float* z, int batch, int z_dim, float* out, cudaStream_t s);
int mapping_fc(const float* x, const float* w, const float* b, int batch, int n_in, int n_out, float w_gain, float b_gain,
               int lrelu, float* y, cudaStream_t s);
int mapping_truncate(const float* w, const float* w_avg, float psi, int batch, int w_dim, float* out, cudaStream_t s);

}  // namespace la
