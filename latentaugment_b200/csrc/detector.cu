// VGG16 detector of precision / recall (DESIGN.md §13): torchvision vgg16 up to fc7 on the tap-GEMM, for any image size.
//
//   image [n, C, res, res] in [-1, 1] -> channel `modality` quantised to 0..255 (StyleGAN3's saved-image rule) -> replicated
//   to 3 channels -> area-resized to 224^2 -> (v - mean) / std -> 13 x (3x3 conv + ReLU), 5 max-pools (vgg.cuh, shared with
//   the perceptual term) -> NCHW flatten -> fc6 + ReLU -> fc7 + ReLU -> [n, 4096] fp32.
//
// The convolutions ping-pong between two NHWC activation buffers (the largest, 224^2 x 64, sets their size).  fc6 and fc7
// are one-tap dense layers whose M rows are images (plan.cuh LayerTaps::kDense, as the discriminator's dense layers): fc6
// contracts K = 25088 over the NHWC view [n, 1, 1, 7 * 7 * 512] of the pool5 output, with its weights permuted from
// torchvision's NCHW flatten order at preparation time.  fc7 stores raw fp32 accumulators and a small kernel adds the bias
// and applies the ReLU, so the embedding is never rounded to bf16.
#include <cuda_bf16.h>

#include "../../include/latentaugment_b200.h"
#include "common.cuh"
#include "kernels.cuh"
#include "plan.cuh"
#include "tapgemm.cuh"
#include "vgg.cuh"

using namespace la;

namespace {

constexpr char kModule[] = "detector";
typedef __nv_bfloat16 bf16;

constexpr int kIn = 224;                  // detector input resolution
constexpr int kPool5 = 7 * 7 * 512;       // fc6 fan-in
constexpr int kFc = 4096;

struct Norm { float mean[3], std[3]; };

// StyleGAN3's saved-image value of a generator output: clamp(x * 127.5 + 128, 0, 255) truncated (two roundings, no FMA,
// as the eager torch expression computes it).
__device__ __forceinline__ float quantise(float x) {
    const float u = __fadd_rn(__fmul_rn(x, 127.5f), 128.f);
    return truncf(fminf(fmaxf(u, 0.f), 255.f));
}

// Thread per pixel of the [n, 224, 224, 64] operand: channels 0..2 = (area mean of the quantised window - mean_k) / std_k,
// 3..63 = 0.  Window [floor(i * res / 224), ceil((i + 1) * res / 224)) per axis, summed row-major and divided by its height
// then its width (adaptive_avg_pool2d, i.e. F.interpolate(mode='area')).
__global__ void detector_input_kernel(const float* __restrict__ img, int n, int C, int res, int modality, Norm z, bf16* x_hi, bf16* x_lo) {
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (idx >= static_cast<long long>(n) * kIn * kIn) return;
    const int ox = static_cast<int>(idx % kIn), oy = static_cast<int>((idx / kIn) % kIn);
    const long long b = idx / (kIn * kIn);
    const int y0 = oy * res / kIn, y1 = ((oy + 1) * res + kIn - 1) / kIn;
    const int x0 = ox * res / kIn, x1 = ((ox + 1) * res + kIn - 1) / kIn;
    const float* src = img + (b * C + modality) * res * res;
    float sum = 0.f;
    for (int y = y0; y < y1; ++y)
        for (int x = x0; x < x1; ++x) sum += quantise(__ldg(src + static_cast<long long>(y) * res + x));
    const float v = sum / static_cast<float>(y1 - y0) / static_cast<float>(x1 - x0);
    float ch[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) ch[k] = (v - z.mean[k]) / z.std[k];
    const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
    uint4* dh = reinterpret_cast<uint4*>(x_hi + idx * 64);
    dh[0] = make_uint4(pack2(ch[0], ch[1]), pack2(ch[2], 0.f), 0u, 0u);
#pragma unroll
    for (int j = 1; j < 8; ++j) dh[j] = zero;
    if (x_lo) {
        uint4* dl = reinterpret_cast<uint4*>(x_lo + idx * 64);
        dl[0] = make_uint4(pack2(ch[0] - rnd(ch[0]), ch[1] - rnd(ch[1])), pack2(ch[2] - rnd(ch[2]), 0.f), 0u, 0u);
#pragma unroll
        for (int j = 1; j < 8; ++j) dl[j] = zero;
    }
}

// dense w [rows, K] fp32 -> K-major bf16 [rows][K] (+ residual plane behind it when split).  nchw_c > 0: the input index of w
// is torchvision's NCHW flatten c * hw + p of a [nchw_c, hw] map and the operand's column k = p * nchw_c + c is NHWC.
__global__ void prep_dense_kernel(const float* __restrict__ w, int rows, int K, int nchw_c, int split, bf16* out) {
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    const long long total = static_cast<long long>(rows) * K;
    if (idx >= total) return;
    const int k = static_cast<int>(idx % K);
    const long long o = idx / K;
    const int src = nchw_c ? (k % nchw_c) * (K / nchw_c) + k / nchw_c : k;
    const float v = w[o * K + src];
    const bf16 h = __float2bfloat16_rn(v);
    out[idx] = h;
    if (split) out[total + idx] = __float2bfloat16_rn(v - __bfloat162float(h));
}

__global__ void bias_relu_kernel(const float* __restrict__ raw, const float* __restrict__ bias, long long total, int N, float* out) {
    const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (i < total) out[i] = fmaxf(raw[i] + __ldg(bias + i % N), 0.f);
}

}  // namespace

struct la_detector {
    la_detector_desc d;
    int batch, split, num_sms;
    Pl buf[2];                  // ping-pong activations [batch, <= 224^2 x 64]; buf[1] takes the input operand
    Pl h6;                      // fc6 output [batch, 4096]
    bf16* wconv[kNConv];
    bf16 *w6, *w7;
    float *ones, *raw7;
    int* err_flag;
    int pool5;                  // which buffer holds the pool5 output
    TapGemmParams conv[kNConv], fc6, fc7;
};

namespace {

int validate(const la_detector_desc* d, int batch, int precision) {
    if (!d || batch < 1) return fail(-2, "detector: bad arguments");
    if (precision != LA_PRECISION_BF16 && precision != LA_PRECISION_FP32_PARITY) return fail(-2, "detector: unknown precision %d", precision);
    for (int i = 0; i < kNConv; ++i)
        if (!d->d_conv_weight[i] || !d->d_conv_bias[i]) return fail(-2, "detector: missing parameters of conv %d", i);
    if (!d->d_fc6_weight || !d->d_fc6_bias || !d->d_fc7_weight || !d->d_fc7_bias) return fail(-2, "detector: missing fc6 / fc7 parameters");
    for (int k = 0; k < 3; ++k)
        if (!(d->std[k] > 0.f)) return fail(-2, "detector: std[%d] must be positive", k);
    return 0;
}

size_t plan_detector(la_detector* D, char* ws) {
    Bump bp;
    bp.base = ws;
    const size_t B = D->batch, wm = D->split ? 2 : 1;
    for (int k = 0; k < 2; ++k) D->buf[k] = bp.take_pl(B * kIn * kIn * 64, D->split);
    D->h6 = bp.take_pl(B * kFc, D->split);
    for (int i = 0; i < kNConv; ++i) D->wconv[i] = bp.take<bf16>(wm * 9 * kCout[i] * ((kCin[i] + 63) / 64 * 64));
    D->w6 = bp.take<bf16>(wm * kFc * kPool5);
    D->w7 = bp.take<bf16>(wm * kFc * kFc);
    D->ones = bp.take<float>(B * kFc);
    D->raw7 = bp.take<float>(B * kFc);
    D->err_flag = bp.take<int>(1);
    bp.take<char>(1024);
    return bp.off;
}

int build_detector(la_detector* D) {
    const int B = D->batch, split = D->split;
    int cur = 1;
    for (int i = 0; i < kNConv; ++i) {
        const int R = kIn >> kShift[i];
        LA(plan_layer(D->conv[i], LayerTaps::k3x3, D->buf[cur], B, R, (kCin[i] + 63) / 64 * 64, kCout[i], D->wconv[i], split, D->err_flag));
        fwd_epilogue(D->conv[i], D->ones, D->d.d_conv_bias[i], 1.f, -1.f, 0.f, D->buf[cur ^ 1]);          // ReLU
        cur ^= 1;
        for (int k = 0; k < 5; ++k) if (kPoolConv[k] == i) cur ^= 1;
    }
    D->pool5 = cur;
    // fc6 + ReLU -> h6 (bf16, the A operand of fc7)
    LA(plan_layer(D->fc6, LayerTaps::kDense, D->buf[cur], B, 1, kPool5, kFc, D->w6, split, D->err_flag));
    fwd_epilogue(D->fc6, D->ones, D->d.d_fc6_bias, 1.f, -1.f, 0.f, D->h6);
    // fc7 -> raw fp32 accumulators (bias + ReLU follow); the activation constants are a linear layer's
    LA(plan_layer(D->fc7, LayerTaps::kDense, D->h6, B, 1, kFc, kFc, D->w7, split, D->err_flag));
    linear_epilogue(D->fc7, 0.f);
    D->fc7.epilogue = kEpiRawF32;
    D->fc7.raw_out = D->raw7;
    return 0;
}

int prepare_detector(la_detector* D, cudaStream_t s) {
    for (int i = 0; i < kNConv; ++i)
        LA(vgg_prep_weights(D->d.d_conv_weight[i], kCout[i], kCin[i], (kCin[i] + 63) / 64 * 64, D->split, D->wconv[i], nullptr, s));
    prep_dense_kernel<<<cdiv(static_cast<long long>(kFc) * kPool5, 256), 256, 0, s>>>(D->d.d_fc6_weight, kFc, kPool5, 512, D->split, D->w6);
    CU(cudaGetLastError());
    prep_dense_kernel<<<cdiv(static_cast<long long>(kFc) * kFc, 256), 256, 0, s>>>(D->d.d_fc7_weight, kFc, kFc, 0, D->split, D->w7);
    CU(cudaGetLastError());
    const long long n_ones = static_cast<long long>(D->batch) * kFc;
    LA(fill(D->ones, 1.f, n_ones, s));
    CU(cudaMemsetAsync(D->err_flag, 0, sizeof(int), s));
    CU(cudaStreamSynchronize(s));
    return 0;
}

}  // namespace

#define LA_API __attribute__((visibility("default")))
extern "C" {

LA_API int la_detector_workspace_bytes(const la_detector_desc* d, int batch, int precision, size_t* bytes) {
    if (!bytes) return fail(-2, "detector: bad arguments");
    if (int r = validate(d, batch, precision)) return r;
    la_detector* tmp = new la_detector{};
    tmp->batch = batch; tmp->split = precision == LA_PRECISION_FP32_PARITY;
    *bytes = plan_detector(tmp, nullptr);
    delete tmp;
    return 0;
}

LA_API int la_detector_create(const la_detector_desc* d, int batch, int precision, void* d_workspace, size_t workspace_bytes, la_stream stream,
                              la_detector** out) {
    if (!out || !d_workspace) return fail(-2, "detector: bad arguments");
    if (int r = validate(d, batch, precision)) return r;
    la_detector* D = new la_detector{};
    D->d = *d; D->batch = batch; D->split = precision == LA_PRECISION_FP32_PARITY;
    const size_t need = plan_detector(D, static_cast<char*>(d_workspace));
    if (int r = check_workspace(kModule, need, workspace_bytes, d_workspace)) { delete D; return r; }
    int dev = 0;
    int r = static_cast<int>(cudaGetDevice(&dev));
    if (!r) r = static_cast<int>(cudaDeviceGetAttribute(&D->num_sms, cudaDevAttrMultiProcessorCount, dev));
    if (r) { delete D; return fail(r, "detector: %s", cudaGetErrorString(static_cast<cudaError_t>(r))); }
    r = build_detector(D);
    if (!r) r = prepare_detector(D, static_cast<cudaStream_t>(stream));
    if (r) { delete D; return r; }
    *out = D;
    return 0;
}

LA_API void la_detector_destroy(la_detector* det) { delete det; }

LA_API int la_detector_features(la_detector* D, const float* d_img, int n, int C, int res, int modality, float* d_out, la_stream stream) {
    if (!D || !d_img || !d_out) return fail(-2, "detector: bad arguments");
    if (n < 1 || n > D->batch) return fail(-2, "detector: n = %d outside 1..%d (the planned batch)", n, D->batch);
    if (C < 1 || modality < 0 || modality >= C) return fail(-2, "detector: modality %d outside 0..%d", modality, C - 1);
    if (res < 16 || res > 1024) return fail(-2, "detector: resolution %d outside 16..1024", res);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    Norm z;
    for (int k = 0; k < 3; ++k) { z.mean[k] = D->d.mean[k]; z.std[k] = D->d.std[k]; }
    const long long npx = static_cast<long long>(n) * kIn * kIn;
    detector_input_kernel<<<cdiv(npx, 256), 256, 0, s>>>(d_img, n, C, res, modality, z, D->buf[1].hi, D->buf[1].lo);
    CU(cudaGetLastError());
    int cur = 1;
    for (int i = 0; i < kNConv; ++i) {
        LA(launch_tapgemm(D->conv[i], D->num_sms, s));
        cur ^= 1;
        for (int k = 0; k < 5; ++k)
            if (kPoolConv[k] == i) {
                LA(vgg_pool_fwd(D->buf[cur], n, kIn >> kShift[i], kCout[i], D->buf[cur ^ 1], s));
                cur ^= 1;
            }
    }
    LA(launch_tapgemm(D->fc6, D->num_sms, s));
    LA(launch_tapgemm(D->fc7, D->num_sms, s));
    const long long total = static_cast<long long>(n) * kFc;
    bias_relu_kernel<<<cdiv(total, 256), 256, 0, s>>>(D->raw7, D->d.d_fc7_bias, total, kFc, d_out);
    CU(cudaGetLastError());
    return 0;
}

}  // extern "C"
