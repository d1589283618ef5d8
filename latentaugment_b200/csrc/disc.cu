// StyleGAN2 'resnet' discriminator for the realism term of the LatentAugment loop
// (reference calc_loss_disc, augments/utils/util_latent_aug.py:363-371; parameter contract
// models/stylegan3/legacy.py:220-289; layer ops conv2d_resample.py:94-97,106-109 + bias_act.py).
//
// Block at resolution R (channels C -> Cn):   y = skip(x) + conv1(conv0(x))
//   conv0 : 3x3, lrelu*sqrt2, clamp                               -> tap-GEMM, forward epilogue (demod = 1)
//   conv1 : blur (4x4 FIR, pad 2) -> 3x3 stride 2, gain sqrt(.5)  -> FIR pass + tap-GEMM over 4 phase views
//   skip  : blur + decimate (pad 1) -> 1x1, gain sqrt(.5)         -> decimating FIR + 1-tap GEMM (kEpiLinear adds y1)
// Epilogue at 4x4: minibatch-stddev channel, 3x3 conv, dense 16C -> C (a 16-tap GEMM whose M rows are samples),
// dense C -> 1.  The backward pass needs data gradients only (D's weights are fixed): every GEMM above has its
// transposed twin; activation gradients are taken from the saved outputs (bias_act.cu:48,72,141 semantics).
// Operands are bf16 with fp32 accumulation in both engine precisions (DESIGN.md §3.6).
#include "disc.cuh"

#include <cuda_bf16.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <string>
#include <vector>

#include "act.cuh"
#include "kernels.cuh"
#include "plan.cuh"
#include "tapgemm.cuh"

using namespace la;

namespace {

typedef __nv_bfloat16 bf16;
thread_local std::string g_derr;

int dfail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_derr = buf;
    return code ? code : -1;
}
#define DCU(x)                                                                                               \
    do {                                                                                                     \
        cudaError_t e_ = (x);                                                                                \
        if (e_ != cudaSuccess) return dfail(static_cast<int>(e_), "%s: %s (%s:%d)", #x, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)
#define DLA(x)                                                                                               \
    do {                                                                                                     \
        int r_ = (x);                                                                                        \
        if (r_) return dfail(r_, "%s failed (%d) (%s:%d)", #x, r_, __FILE__, __LINE__);                      \
    } while (0)

inline int cdiv(long long a, long long b) { return static_cast<int>((a + b - 1) / b); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ unsigned pack2(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<unsigned*>(&v);
}
__device__ __forceinline__ float lo_f(unsigned u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float hi_f(unsigned u) { return __uint_as_float(u & 0xffff0000u); }
// value of element i of a (hi [, lo]) bf16 pair / pair store
__device__ __forceinline__ float ld_sp(const bf16* hi, const bf16* lo, long long i) {
    float v = __bfloat162float(hi[i]);
    if (lo) v += __bfloat162float(lo[i]);
    return v;
}
__device__ __forceinline__ void st_sp(bf16* hi, bf16* lo, long long i, float v) {
    const bf16 h = __float2bfloat16_rn(v);
    hi[i] = h;
    if (lo) lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
}
__device__ __forceinline__ void st_sp2(unsigned* hi, unsigned* lo, long long i, float a, float b) {
    hi[i] = pack2(a, b);
    if (lo) lo[i] = pack2(a - __bfloat162float(__float2bfloat16_rn(a)), b - __bfloat162float(__float2bfloat16_rn(b)));
}
__device__ __forceinline__ float act_fwd(float z, float gain, float slope, float clamp) {
    z = (z > 0.f ? z : z * slope) * gain;
    return clamp >= 0.f ? fminf(fmaxf(z, -clamp), clamp) : z;
}

// ------------------------------------------------------------------------- weight preparation
// w [cout, cin, k, k] fp32 -> wf [k*k][cout][cin_pad] and wb [k*k][cin_pad][cout], both * scale, zero padded;
// with split the bf16 residual planes follow as a second stack of k*k matrices
__global__ void prep_plain_weights_kernel(const float* __restrict__ w, int cout, int cin, int k2, float scale, int cin_pad, int split,
                                          bf16* wf, bf16* wb) {
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    const long long total = static_cast<long long>(k2) * cout * cin_pad;
    if (idx >= total) return;
    const int i = static_cast<int>(idx % cin_pad);
    const int o = static_cast<int>((idx / cin_pad) % cout);
    const int t = static_cast<int>(idx / (static_cast<long long>(cin_pad) * cout));
    const float v = i < cin ? w[(static_cast<long long>(o) * cin + i) * k2 + t] * scale : 0.f;
    const long long bidx = (static_cast<long long>(t) * cin_pad + i) * cout + o;
    st_sp(wf, split ? wf + total : nullptr, idx, v);
    st_sp(wb, split ? wb + total : nullptr, bidx, v);
}
// dense [C, 16*C] over the NCHW flatten (index c*16 + hw) -> wf [16][C(o)][C(c)], wb [16*C (hw, c)][C(o)]
__global__ void prep_fc_weights_kernel(const float* __restrict__ w, int C, float scale, int split, bf16* wf, bf16* wb) {
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    const long long total = 16LL * C * C;
    if (idx >= total) return;
    const int c = static_cast<int>(idx % C);
    const int o = static_cast<int>((idx / C) % C);
    const int hw = static_cast<int>(idx / (static_cast<long long>(C) * C));
    const float v = w[static_cast<long long>(o) * 16 * C + c * 16 + hw] * scale;
    st_sp(wf, split ? wf + total : nullptr, idx, v);
    st_sp(wb, split ? wb + total : nullptr, (static_cast<long long>(hw) * C + c) * C + o, v);
}
__global__ void prep_rgb_w4_kernel(const float* __restrict__ w, int C, int imgc, float wg, float* w4) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    w4[4 * c + 0] = w[c * imgc] * wg;
    w4[4 * c + 1] = imgc > 1 ? w[c * imgc + 1] * wg : 0.f;
    w4[4 * c + 2] = imgc > 2 ? w[c * imgc + 2] * wg : 0.f;
    w4[4 * c + 3] = 0.f;
}
__global__ void fill_kernel(float* p, float v, long long n) {
    const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (i < n) p[i] = v;
}

// ------------------------------------------------------------------------- image layout
__global__ void nchw_to_f4_kernel(const float* __restrict__ src, int C, int hw, long long total, float4* dst) {
    const long long p = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (p >= total) return;
    const long long n = p / hw, q = p - n * hw;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    v.x = src[(n * C + 0) * hw + q];
    if (C > 1) v.y = src[(n * C + 1) * hw + q];
    if (C > 2) v.z = src[(n * C + 2) * hw + q];
    dst[p] = v;
}
__global__ void f4_to_nchw_kernel(const float4* __restrict__ src, int C, int hw, long long total, float* dst) {
    const long long p = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (p >= total) return;
    const long long n = p / hw, q = p - n * hw;
    const float4 v = src[p];
    dst[(n * C + 0) * hw + q] = v.x;
    if (C > 1) dst[(n * C + 1) * hw + q] = v.y;
    if (C > 2) dst[(n * C + 2) * hw + q] = v.z;
}

// ------------------------------------------------------------------------- fromrgb (1x1 conv from the image)
// x[p][c] = act(sum_k img[p].k * w[c][k] * wg + b[c]).  A thread owns one channel pair (weights in registers) and
// walks a run of pixels; a warp writes 128 contiguous bytes per pixel.
constexpr int kRgbPixels = 128;
__global__ void fromrgb_fwd_kernel(const float4* __restrict__ img, const float* __restrict__ w, const float* __restrict__ b, long long npix,
                                   int C, int imgc, float wg, float gain, float slope, float clamp, unsigned* x, unsigned* x_lo) {
    const int hc = C >> 1;
    const int cpb = hc < 256 ? hc : 256, lanes = 256 / cpb;
    const int cp = blockIdx.y * cpb + threadIdx.x % cpb, lane = threadIdx.x / cpb;
    float wr[2][3], br[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
        const int c = 2 * cp + u;
        wr[u][0] = w[c * imgc] * wg;
        wr[u][1] = imgc > 1 ? w[c * imgc + 1] * wg : 0.f;
        wr[u][2] = imgc > 2 ? w[c * imgc + 2] * wg : 0.f;
        br[u] = b[c];
    }
    const long long p0 = static_cast<long long>(blockIdx.x) * kRgbPixels;
    for (int i = lane; i < kRgbPixels; i += lanes) {
        const long long p = p0 + i;
        if (p >= npix) break;
        const float4 v = __ldg(img + p);
        const float z0 = act_fwd(fmaf(v.x, wr[0][0], fmaf(v.y, wr[0][1], v.z * wr[0][2])) + br[0], gain, slope, clamp);
        const float z1 = act_fwd(fmaf(v.x, wr[1][0], fmaf(v.y, wr[1][1], v.z * wr[1][2])) + br[1], gain, slope, clamp);
        st_sp2(x, x_lo, p * hc + cp, z0, z1);
    }
}
// ------------------------------------------------------------------------- decimating FIR of the skip branch
// upfirdn2d(x, f, down=2, padding=1) (conv2d_resample.py:94-97):  ys[m, n] = sum_j fk[jy][jx] * x[2m + jy - 1, 2n + jx - 1]
// (fk = flipped filter: true convolution, upfirdn2d.py:196-199).  Thread per (output pixel, channel pair).
struct Fir16 { float k[16]; };
__global__ void firdown_fwd_kernel(const unsigned* __restrict__ x, const unsigned* __restrict__ x_lo, int B, int R, int C, Fir16 f, unsigned* ys,
                                   unsigned* ys_lo) {
    const int hc = C >> 1, Ro = R >> 1;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;       // (n, channel pair) of output row m = blockIdx.y, sample blockIdx.z
    if (e >= Ro * hc) return;
    const int cp = e % hc, n = e / hc, m = blockIdx.y, b = blockIdx.z;
    // all 16 (x 2 planes) loads are issued before the first FMA: out-of-range taps read a clamped address with weight 0
    // (a `continue` per tap kept the loads from being batched and left the kernel latency-bound)
    unsigned u[16], l[16];
    float wgt[16];
#pragma unroll
    for (int jy = 0; jy < 4; ++jy) {
        const int y = 2 * m + jy - 1;
        const bool oky = y >= 0 && y < R;
        const long long roff = (static_cast<long long>(b) * R + (oky ? y : 0)) * R * hc + cp;
#pragma unroll
        for (int jx = 0; jx < 4; ++jx) {
            const int xx = 2 * n + jx - 1;
            const bool ok = oky && xx >= 0 && xx < R;
            const long long off = roff + static_cast<long long>(ok ? xx : 0) * hc;
            u[jy * 4 + jx] = __ldg(x + off);
            l[jy * 4 + jx] = x_lo ? __ldg(x_lo + off) : 0u;
            wgt[jy * 4 + jx] = ok ? f.k[jy * 4 + jx] : 0.f;
        }
    }
    float a0 = 0.f, a1 = 0.f;
#pragma unroll
    for (int t = 0; t < 16; ++t) {
        const float v0 = lo_f(u[t]) + lo_f(l[t]), v1 = hi_f(u[t]) + hi_f(l[t]);
        a0 = fmaf(wgt[t], v0, a0);
        a1 = fmaf(wgt[t], v1, a1);
    }
    st_sp2(ys, ys_lo, ((static_cast<long long>(b) * Ro + m) * Ro) * hc + e, a0, a1);
}

// ------------------------------------------------------------------------- minibatch standard deviation (4x4 epilogue)
// x [B,4,4,C] bf16; groups of G samples {m, m + M, ...} (M = B / G);  feat[m] = mean_{c,hw} sqrt(var_g + 1e-8)
__global__ void mbstd_stat_kernel(const bf16* __restrict__ x, const bf16* __restrict__ x_lo, int B, int G, int C, float* feat) {
    const int M = B / G, m = blockIdx.x;
    const int E = 16 * C;
    float acc = 0.f;
    for (int e = threadIdx.x; e < E; e += blockDim.x) {
        float mean = 0.f;
        for (int g = 0; g < G; ++g) mean += ld_sp(x, x_lo, static_cast<long long>(g * M + m) * E + e);
        mean /= G;
        float var = 0.f;
        for (int g = 0; g < G; ++g) {
            const float d = ld_sp(x, x_lo, static_cast<long long>(g * M + m) * E + e) - mean;
            var = fmaf(d, d, var);
        }
        acc += sqrtf(var / G + 1e-8f);
    }
    __shared__ float sm[32];
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        float v = threadIdx.x < (blockDim.x >> 5) ? sm[threadIdx.x] : 0.f;
        v = warp_sum(v);
        if (threadIdx.x == 0) feat[m] = v / E;
    }
}
// x4p [B,4,4,Cp]: channels [0,C) = x, channel C = feat[n % M], the rest zero
__global__ void mbstd_concat_kernel(const bf16* __restrict__ x, const bf16* __restrict__ x_lo, const float* __restrict__ feat, int B, int M, int C,
                                    int Cp, bf16* x4p, bf16* x4p_lo) {
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (idx >= static_cast<long long>(B) * 16 * Cp) return;
    const int c = static_cast<int>(idx % Cp);
    const long long p = idx / Cp;           // n*16 + hw
    const int n = static_cast<int>(p / 16);
    float v = 0.f;
    if (c < C) v = ld_sp(x, x_lo, p * C + c);
    else if (c == C) v = feat[n % M];
    st_sp(x4p, x4p_lo, idx, v);
}
// gfeat[m] = sum over the group's samples and positions of the gradient of the stddev channel
__global__ void mbstd_gfeat_kernel(const bf16* __restrict__ gx4p, const bf16* __restrict__ gx4p_lo, int B, int M, int C, int Cp, float* gfeat) {
    const int m = blockIdx.x;
    float acc = 0.f;
    for (int e = threadIdx.x; e < (B / M) * 16; e += blockDim.x) {
        const int g = e / 16, hw = e % 16;
        acc += ld_sp(gx4p, gx4p_lo, (static_cast<long long>(g * M + m) * 16 + hw) * Cp + C);
    }
    __shared__ float sm[32];
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        float v = threadIdx.x < (blockDim.x >> 5) ? sm[threadIdx.x] : 0.f;
        v = warp_sum(v);
        if (threadIdx.x == 0) gfeat[m] = v;
    }
}
// g_y[n][e] = gx4p[n][e] + gfeat[m] * (x - mean_g) / (G * 16C * sd);   g_z1 = g_y * act'(y1)
__global__ void mbstd_bwd_kernel(const bf16* __restrict__ x, const bf16* __restrict__ x_lo, const bf16* __restrict__ gx4p,
                                 const bf16* __restrict__ gx4p_lo, const float* __restrict__ gfeat, const bf16* __restrict__ y1, const bf16* __restrict__ y1_lo, int B, int G, int C,
                                 int Cp, float gain, float slope, float clamp, bf16* g_y, bf16* g_y_lo, bf16* g_z1, bf16* g_z1_lo) {
    const int M = B / G, E = 16 * C;
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (idx >= static_cast<long long>(M) * E) return;
    const int e = static_cast<int>(idx % E), m = static_cast<int>(idx / E);
    float xv[8];
    float mean = 0.f;
    for (int g = 0; g < G; ++g) { xv[g] = ld_sp(x, x_lo, static_cast<long long>(g * M + m) * E + e); mean += xv[g]; }
    mean /= G;
    float var = 0.f;
    for (int g = 0; g < G; ++g) var = fmaf(xv[g] - mean, xv[g] - mean, var);
    const float sd = sqrtf(var / G + 1e-8f);
    const float k = gfeat[m] / (static_cast<float>(G) * E * sd);
    const int hw = e / C, c = e % C;
    const float thr = act_saved_clamp(clamp, y1_lo != nullptr);
    for (int g = 0; g < G; ++g) {
        const long long n = g * M + m;
        const float gv = ld_sp(gx4p, gx4p_lo, (n * 16 + hw) * Cp + c) + k * (xv[g] - mean);
        st_sp(g_y, g_y_lo, n * E + e, gv);
        st_sp(g_z1, g_z1_lo, n * E + e, act_grad(gv * gain, ld_sp(y1, y1_lo, n * E + e), slope, thr));
    }
}

// ------------------------------------------------------------------------- output layer, loss, gradient seed
// logits[n] = sum_c x6[n][c] * w[c] * wg + b;  warp per sample
__global__ void out_fwd_kernel(const bf16* __restrict__ x6, const bf16* __restrict__ x6_lo, const float* __restrict__ w, const float* __restrict__ b,
                               int B, int C, float wg, float* logits) {
    const int n = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (n >= B) return;
    float a = 0.f;
    for (int c = lane; c < C; c += 32) a = fmaf(ld_sp(x6, x6_lo, static_cast<long long>(n) * C + c), w[c], a);
    a = warp_sum(a);
    if (lane == 0) logits[n] = a * wg + b[0];
}
// loss = w_disc * mean softplus(-logit);  gl[n] = -w_disc / B * sigmoid(-logit[n])   (one block)
__global__ void disc_loss_kernel(const float* __restrict__ logits, int B, float w_disc, float* loss, float* gl) {
    float acc = 0.f;
    for (int n = threadIdx.x; n < B; n += blockDim.x) {
        const float l = logits[n];
        acc += l > 0.f ? log1pf(expf(-l)) : (-l + log1pf(expf(l)));     // softplus(-l), stable
        gl[n] = -w_disc / B / (1.f + expf(l));
    }
    __shared__ float sm[32];
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float v = 0.f;
        for (int i = 0; i < (blockDim.x >> 5); ++i) v += sm[i];
        loss[0] = w_disc * v / B;
    }
}
// gz6[n][c] = gl[n] * w[c] * wg * act'(x6[n][c])
__global__ void out_bwd_kernel(const float* __restrict__ gl, const float* __restrict__ w, const bf16* __restrict__ x6, int B, int C, float wg,
                               float gain, float slope, bf16* gz6, bf16* gz6_lo) {
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (idx >= static_cast<long long>(B) * C) return;
    const int c = static_cast<int>(idx % C), n = static_cast<int>(idx / C);
    st_sp(gz6, gz6_lo, idx, act_grad(gl[n] * w[c] * wg * gain, __bfloat162float(x6[idx]), slope, act_saved_clamp(-1.f, false)));
}

struct Bump {
    char* base = nullptr;
    size_t off = 0;
    template <class T>
    T* take(size_t count) {
        off = (off + 1023) & ~size_t(1023);
        T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
        off += count * sizeof(T);
        return p;
    }
};

struct Pl {                 // a bf16 tensor as (hi [, lo]) planes; lo only in split (fp32_parity) precision
    bf16* hi = nullptr;
    bf16* lo = nullptr;
};

struct Block {
    int R, C, Cn;
    la_disc_block_params p;
    bf16 *w0f, *w0b, *w1f, *w1b, *wsf, *wsb;
    Pl x_in, x0, y1, y;                       // saved activations (y is the next block's x_in)
    Pl g_y, g_z1;                             // gradient wrt y and through conv1's activation
    TapGemmParams F0, F1, FS, BS, B1, B0;
    UpFirParams blur;
};

constexpr float kSqrt2 = 1.41421356237309515f, kSqrtHalf = 0.70710678118654752f;

}  // namespace

struct la_disc {
    la_disc_desc d;
    int batch, num_sms, split;
    std::vector<Block> blk;
    float fir[16];                            // flipped, normalised 4x4 filter (true convolution)
    // shared scratch (sized for the top block)
    Pl yb, ys, g_ys, g_yb, g_z0;
    float* ones;                              // demod = 1 for the plain layers
    float* rgb_w4;                            // [C_top][4]: fromrgb weights * weight gain, for the fused fromrgb backward
    // epilogue
    int C4, Cp;
    Pl x4p, x5, x6, gz6, gz5, gx4p;
    bf16 *wef, *web, *wff, *wfb;
    float *feat, *gfeat, *logits, *gl;
    TapGemmParams FE, FF, BF, BE;
    int* err_flag;
};

namespace {

void fwd_epi(TapGemmParams& P, const la_disc* D, const float* bias, const Pl& out, float gain, float clamp, int n_total, int bn, int res) {
    P.epilogue = kEpiFwd;
    P.n_total = n_total; P.n_blocks = n_total / bn;
    P.OH = P.OW = res; P.osy = P.osx = 1; P.split = D->split;
    P.act_gain = gain; P.act_clamp = clamp; P.act_slope = 0.2f;
    P.demod = D->ones; P.bias = bias; P.noise = nullptr; P.s_next = nullptr; P.rgbw = nullptr;
    P.x_hi = out.hi; P.x_lo = out.lo;
    P.staged = P.nb == 1 && !D->split && !getenv("LA_NO_STAGED");
}
void lin_epi(TapGemmParams& P, const la_disc* D, int n_total, int bn, int oh, int ow) {
    P.epilogue = kEpiLinear;
    P.n_total = n_total; P.n_blocks = n_total / bn;
    P.OH = oh; P.OW = ow; P.osy = P.osx = 1; P.split = D->split;
    P.act_gain = 1.f; P.act_clamp = -1.f; P.act_slope = 0.2f;
}
int choose_bn(int n, long long m_tiles) { return n % 128 ? 64 : pick_bn(n, m_tiles); }

// A map(s) of a dense NHWC tensor [B, H, W, C]: map `slot` = hi plane, `slot + lo_slot` = lo plane
int dense_maps(const la_disc* D, TapGemmParams& P, int slot, int lo_slot, const Pl& t, int C, int W, int H, int tw, int th, int nb) {
    const long long sW = C, sH = static_cast<long long>(W) * C, sN = sH * H;
    if (make_a_map(&P.a_map[slot], t.hi, C, W, H, D->batch, sW, sH, sN, tw, th, nb)) return -1;
    if (D->split && make_a_map(&P.a_map[slot + lo_slot], t.lo, C, W, H, D->batch, sW, sH, sN, tw, th, nb)) return -1;
    return 0;
}

int plan_disc(la_disc* D, char* ws, size_t* bytes_out) {
    const la_disc_desc& d = D->d;
    const int B = D->batch, split = D->split;
    if (d.num_blocks < 1 || d.num_blocks + 1 > LA_MAX_BLOCKS || (8 << (d.num_blocks - 1)) != d.img_resolution)
        return dfail(-2, "discriminator: img_resolution %d does not match num_blocks %d", d.img_resolution, d.num_blocks);
    if (d.img_channels < 1 || d.img_channels > 3) return dfail(-2, "discriminator: img_channels must be 1..3");
    if (d.mbstd_group_size < 1 || d.mbstd_group_size > 8) return dfail(-2, "discriminator: mbstd_group_size must be 1..8");
    for (int b = 0; b <= d.num_blocks; ++b)
        if (d.channels[b] % 64 || d.channels[b] < 64 || d.channels[b] > 1024) return dfail(-2, "discriminator: channels[%d]=%d unsupported", b, d.channels[b]);
    Bump bp;
    bp.base = ws;
    auto take_pl = [&](size_t n) { Pl t; t.hi = bp.take<bf16>(n); t.lo = split ? bp.take<bf16>(n) : nullptr; return t; };
    const size_t wm = split ? 2 : 1;            // weight stacks carry the residual planes behind the main ones
    D->blk.assign(d.num_blocks, Block{});
    size_t max_full = 0, max_half = 0, max_t = 0;
    int cmax = 0;
    for (int b = 0; b < d.num_blocks; ++b) {
        Block& k = D->blk[b];
        k.R = d.img_resolution >> b; k.C = d.channels[b]; k.Cn = d.channels[b + 1]; k.p = d.block[b];
        const size_t C = k.C, Cn = k.Cn, R = k.R;
        k.w0f = bp.take<bf16>(wm * 9 * C * C); k.w0b = bp.take<bf16>(wm * 9 * C * C);
        k.w1f = bp.take<bf16>(wm * 9 * Cn * C); k.w1b = bp.take<bf16>(wm * 9 * Cn * C);
        k.wsf = bp.take<bf16>(wm * Cn * C); k.wsb = bp.take<bf16>(wm * Cn * C);
        const size_t full = B * R * R * C, half = B * (R / 2) * (R / 2) * Cn;
        k.x_in = b == 0 ? take_pl(full) : D->blk[b - 1].y;
        k.x0 = take_pl(full);
        k.y1 = take_pl(half);
        k.y = take_pl(half);
        k.g_y = take_pl(half);
        k.g_z1 = take_pl(half);
        max_full = full > max_full ? full : max_full;
        const size_t hs = B * (R / 2) * (R / 2) * C;
        max_half = hs > max_half ? hs : max_half;
        const size_t t = B * (R + 1) * (R + 2) * C;
        max_t = t > max_t ? t : max_t;
        cmax = k.C > cmax ? k.C : cmax;
        cmax = k.Cn > cmax ? k.Cn : cmax;
    }
    D->yb = take_pl(max_t); D->g_yb = take_pl(max_t);
    D->ys = take_pl(max_half); D->g_ys = take_pl(max_half);
    D->g_z0 = take_pl(max_full);
    const int C4 = d.channels[d.num_blocks], Cp = C4 + 64;
    D->C4 = C4; D->Cp = Cp;
    cmax = 16 * C4 > cmax ? 16 * C4 : cmax;
    D->ones = bp.take<float>(static_cast<size_t>(B) * cmax);
    D->rgb_w4 = bp.take<float>(4 * static_cast<size_t>(d.channels[0]));
    D->x4p = take_pl(static_cast<size_t>(B) * 16 * Cp); D->gx4p = take_pl(static_cast<size_t>(B) * 16 * Cp);
    D->x5 = take_pl(static_cast<size_t>(B) * 16 * C4); D->gz5 = take_pl(static_cast<size_t>(B) * 16 * C4);
    D->x6 = take_pl(static_cast<size_t>(B) * C4); D->gz6 = take_pl(static_cast<size_t>(B) * C4);
    D->wef = bp.take<bf16>(wm * 9 * C4 * Cp); D->web = bp.take<bf16>(wm * 9 * C4 * Cp);
    D->wff = bp.take<bf16>(wm * 16 * C4 * C4); D->wfb = bp.take<bf16>(wm * 16 * C4 * C4);
    D->feat = bp.take<float>(B); D->gfeat = bp.take<float>(B); D->logits = bp.take<float>(B); D->gl = bp.take<float>(B);
    D->err_flag = bp.take<int>(1);
    bp.take<char>(1024);
    *bytes_out = bp.off;
    return 0;
}

// 3x3 taps over map 0 (lo map 1)
int conv_taps(const la_disc* D, TapGemmParams& P, bool flipped) {
    int nt = 0;
    P.prob[0].tap_begin = 0;
    for (int t = 0; t < 9; ++t) {
        const int dy = t / 3 - 1, dx = t % 3 - 1;
        add_tap(P, nt, flipped ? -dy : dy, flipped ? -dx : dx, t, 0, 1, 9, D->split);
    }
    P.prob[0].ntaps = nt;
    return tapgemm_finalize(P);
}
int one_tap(const la_disc* D, TapGemmParams& P) {
    int nt = 0;
    add_tap(P, nt, 0, 0, 0, 0, 1, 1, D->split);
    P.prob[0].tap_begin = 0; P.prob[0].ntaps = nt;
    return tapgemm_finalize(P);
}

int build_disc(la_disc* D) {
    const la_disc_desc& d = D->d;
    const int B = D->batch, split = D->split;
    const int wm = split ? 2 : 1;
    const float clamp = d.conv_clamp;
    for (int b = 0; b < d.num_blocks; ++b) {
        Block& k = D->blk[b];
        const int R = k.R, C = k.C, Cn = k.Cn, Ro = R / 2, TH = R + 1, TWp = R + 2;
        // ---- conv0 forward: x_in -> x0
        {
            TapGemmParams& P = k.F0;
            memset(&P, 0, sizeof P);
            set_grid(P, R, B, 1);
            DLA(dense_maps(D, P, 0, 1, k.x_in, C, R, R, P.tw, P.th + P.halo, P.nb));
            const int bn = choose_bn(C, P.m_tiles);
            DLA(make_b_map(P, k.w0f, C, C, 9 * wm, bn));
            P.kchunks = C / 64;
            fwd_epi(P, D, k.p.d_conv0_bias, k.x0, kSqrt2, clamp, C, bn, R);
            P.err_flag = D->err_flag;
            DLA(conv_taps(D, P, false));
        }
        // ---- blur (pad 2): x0 -> yb, and its adjoint fused with conv0's activation gradient: g_yb -> g_z0
        {
            UpFirParams& U = k.blur;
            memset(&U, 0, sizeof U);
            U.B = B; U.OH = U.OW = R; U.C = C; U.TH = TH; U.TWp = TWp; U.split = split;
            // kernel forms: forward out[o] = sum_j fk[j] in[o + j - 1], backward out[u] = sum_j fk[j] in[u - j + 1]; the blur
            // yb[u] = sum_j c[j] x0[u + j - 2] (c = flipped filter) and its adjoint both need fk = the unflipped filter
            for (int i = 0; i < 16; ++i) U.fk[i] = D->fir[15 - i];
            {
                int bi = 0;
                for (int i = 1; i < 16; ++i) if (fabsf(U.fk[i]) > fabsf(U.fk[bi])) bi = i;
                const int by = bi / 4, bx = bi % 4;
                U.separable = U.fk[bi] != 0.f;
                for (int i = 0; i < 4 && U.separable; ++i) { U.fy[i] = U.fk[i * 4 + bx] / U.fk[bi]; U.fx[i] = U.fk[by * 4 + i]; }
                for (int i = 0; i < 16 && U.separable; ++i)
                    if (fabsf(U.fy[i / 4] * U.fx[i % 4] - U.fk[i]) > 1e-6f * fabsf(U.fk[bi])) U.separable = 0;
            }
            U.gy_hi = k.x0.hi; U.gy_lo = k.x0.lo; U.gt_hi = D->yb.hi; U.gt_lo = D->yb.lo;      // "backward" FIR direction = the blur
            U.t_hi = D->g_yb.hi; U.t_lo = D->g_yb.lo; U.x_hi = D->g_z0.hi; U.x_lo = D->g_z0.lo; U.act_saved = k.x0.hi; U.act_saved_lo = k.x0.lo;
            U.act_gain = kSqrt2; U.act_clamp = clamp; U.act_slope = 0.2f;
            if (!split && U.separable && R >= 32 && !getenv("LA_NO_FIR_TMA")) {
                const uint64_t Cc = C, Rr = R;
                const uint64_t tdims[4] = {Cc, Rr + 1, Rr + 1, static_cast<uint64_t>(B)};
                const uint64_t tstr[3] = {Cc * 2, static_cast<uint64_t>(TWp) * Cc * 2, static_cast<uint64_t>(TH) * TWp * Cc * 2};
                const uint64_t ydims[4] = {Cc, Rr, Rr, static_cast<uint64_t>(B)};
                const uint64_t ystr[3] = {Cc * 2, Rr * Cc * 2, Rr * Rr * Cc * 2};
                const uint32_t lbox[4] = {64, 35, 1, 1}, sbox[4] = {64, 8, 1, 1};
                int r = encode_tmap_bf16(&U.fwd_in, D->g_yb.hi, 4, tdims, tstr, lbox, 0);
                r |= encode_tmap_bf16(&U.fwd_out_x, D->g_z0.hi, 4, ydims, ystr, sbox, 0);
                r |= encode_tmap_bf16(&U.bwd_in, k.x0.hi, 4, ydims, ystr, lbox, 0);
                r |= encode_tmap_bf16(&U.bwd_out, D->yb.hi, 4, tdims, tstr, sbox, 0);
                if (r) return dfail(-5, "tensor map encoding failed (discriminator blur)");
                U.use_tma = 1;
            }
        }
        // ---- conv1 forward: 3x3 stride 2 over the four phase views of yb -> y1
        {
            TapGemmParams& P = k.F1;
            memset(&P, 0, sizeof P);
            set_grid(P, Ro, B, 1);
            const long long gW = 2LL * C, gH = 2LL * TWp * C, gN = static_cast<long long>(TH) * TWp * C;
            for (int ph = 0; ph < 4; ++ph) {
                const int py = ph / 2, px = ph % 2;
                const int ph_h = Ro + (py == 0), ph_w = Ro + (px == 0);
                const long long off = (static_cast<long long>(py) * TWp + px) * C;
                DLA(make_a_map(&P.a_map[ph], D->yb.hi + off, C, ph_w, ph_h, B, gW, gH, gN, P.tw, P.th + P.halo, P.nb));
                if (split) DLA(make_a_map(&P.a_map[4 + ph], D->yb.lo + off, C, ph_w, ph_h, B, gW, gH, gN, P.tw, P.th + P.halo, P.nb));
            }
            int nt = 0;
            for (int a = 0; a < 3; ++a)
                for (int bb = 0; bb < 3; ++bb) {
                    const int ph = (a & 1) * 2 + (bb & 1);
                    add_tap(P, nt, a >> 1, bb >> 1, a * 3 + bb, ph, 4 + ph, 9, split);
                }
            P.prob[0].tap_begin = 0; P.prob[0].ntaps = nt;
            const int bn = choose_bn(Cn, P.m_tiles);
            DLA(make_b_map(P, k.w1f, C, Cn, 9 * wm, bn));
            P.kchunks = C / 64;
            fwd_epi(P, D, k.p.d_conv1_bias, k.y1, kSqrt2 * kSqrtHalf, clamp >= 0.f ? clamp * kSqrtHalf : clamp, Cn, bn, Ro);
            P.err_flag = D->err_flag;
            DLA(tapgemm_finalize(P));
        }
        // ---- skip forward: 1x1 on the decimated blur, + y1 -> y
        {
            TapGemmParams& P = k.FS;
            memset(&P, 0, sizeof P);
            set_grid(P, Ro, B, 1);
            DLA(dense_maps(D, P, 0, 1, D->ys, C, Ro, Ro, P.tw, P.th + P.halo, P.nb));
            const int bn = choose_bn(Cn, P.m_tiles);
            DLA(make_b_map(P, k.wsf, C, Cn, wm, bn));
            P.kchunks = C / 64;
            lin_epi(P, D, Cn, bn, Ro, Ro);
            P.lin_add = k.y1.hi; P.lin_add_lo = k.y1.lo; P.lin_out = k.y.hi; P.lin_out_lo = k.y.lo;
            P.err_flag = D->err_flag;
            DLA(one_tap(D, P));
        }
        // ---- skip backward: g_ys = Ws^T g_y
        {
            TapGemmParams& P = k.BS;
            memset(&P, 0, sizeof P);
            set_grid(P, Ro, B, 1);
            DLA(dense_maps(D, P, 0, 1, k.g_y, Cn, Ro, Ro, P.tw, P.th + P.halo, P.nb));
            const int bn = choose_bn(C, P.m_tiles);
            DLA(make_b_map(P, k.wsb, Cn, C, wm, bn));
            P.kchunks = Cn / 64;
            lin_epi(P, D, C, bn, Ro, Ro);
            P.lin_out = D->g_ys.hi; P.lin_out_lo = D->g_ys.lo;
            P.err_flag = D->err_flag;
            DLA(one_tap(D, P));
        }
        // ---- conv1 backward: transposed stride-2 convolution, g_z1 -> g_yb (four output phases)
        {
            TapGemmParams& P = k.B1;
            memset(&P, 0, sizeof P);
            const int gh[4] = {Ro + 1, Ro + 1, Ro, Ro}, gw[4] = {Ro + 1, Ro, Ro + 1, Ro};
            set_grid(P, Ro, B, 4, gh, gw);
            DLA(dense_maps(D, P, 0, 1, k.g_z1, Cn, Ro, Ro, P.tw, P.th + P.halo, P.nb));
            int nt = 0;
            for (int ph = 0; ph < 4; ++ph) {
                P.prob[ph].tap_begin = nt;
                for (int ay = ph / 2; ay < 3; ay += 2)
                    for (int ax = ph % 2; ax < 3; ax += 2) add_tap(P, nt, -(ay >> 1), -(ax >> 1), ay * 3 + ax, 0, 1, 9, split);
                P.prob[ph].ntaps = nt - P.prob[ph].tap_begin;
                P.prob[ph].oy0 = ph / 2; P.prob[ph].ox0 = ph % 2;
            }
            const int bn = choose_bn(C, P.m_tiles);
            DLA(make_b_map(P, k.w1b, Cn, C, 9 * wm, bn));
            P.kchunks = Cn / 64; P.n_total = C; P.n_blocks = C / bn;
            P.epilogue = kEpiStoreBf16; P.OH = TH; P.OW = TWp; P.osy = P.osx = 2; P.split = split;
            P.x_hi = D->g_yb.hi; P.x_lo = D->g_yb.lo;
            P.staged = P.nb == 1 && !split && !getenv("LA_NO_STAGED");
            P.err_flag = D->err_flag;
            DLA(tapgemm_finalize(P));
        }
        // ---- conv0 backward: g_z0 -> (+ skip-branch gradient) -> gradient wrt the block input, raw and through the producer's activation
        {
            TapGemmParams& P = k.B0;
            memset(&P, 0, sizeof P);
            set_grid(P, R, B, 1);
            DLA(dense_maps(D, P, 0, 1, D->g_z0, C, R, R, P.tw, P.th + P.halo, P.nb));
            const int bn = choose_bn(C, P.m_tiles);
            DLA(make_b_map(P, k.w0b, C, C, 9 * wm, bn));
            P.kchunks = C / 64;
            lin_epi(P, D, C, bn, R, R);
            P.lin_add_down = D->g_ys.hi; P.lin_add_down_lo = D->g_ys.lo;      // FIRdown^T(g_ys) is evaluated inside the epilogue
            for (int i = 0; i < 16; ++i) P.lin_fir[i] = D->fir[i];
            if (b == 0) {                     // the producer is fromrgb (lrelu*sqrt2, clamp): its backward is fused (atomics into g_img)
                P.lin_saved = k.x_in.hi; P.lin_saved_lo = k.x_in.lo; P.lin_rgb_w = D->rgb_w4;       // lin_rgb_g is set per call
                P.act_gain = kSqrt2; P.act_clamp = clamp;
            } else {                          // the producer is conv1 of the block above (gain sqrt2*sqrt(.5), clamp*sqrt(.5))
                Block& up = D->blk[b - 1];
                P.lin_out = up.g_y.hi; P.lin_out_lo = up.g_y.lo; P.lin_saved = up.y1.hi; P.lin_saved_lo = up.y1.lo; P.lin_gz = up.g_z1.hi; P.lin_gz_lo = up.g_z1.lo;
                P.act_gain = kSqrt2 * kSqrtHalf; P.act_clamp = clamp >= 0.f ? clamp * kSqrtHalf : clamp;
            }
            P.err_flag = D->err_flag;
            DLA(conv_taps(D, P, true));
        }
    }
    // ------------------------------------------------------------------ 4x4 epilogue
    const int C4 = D->C4, Cp = D->Cp;
    {   // 3x3 conv on [x | stddev] : x4p -> x5
        TapGemmParams& P = D->FE;
        memset(&P, 0, sizeof P);
        set_grid(P, 4, B, 1);
        DLA(dense_maps(D, P, 0, 1, D->x4p, Cp, 4, 4, P.tw, P.th + P.halo, P.nb));
        const int bn = choose_bn(C4, P.m_tiles);
        DLA(make_b_map(P, D->wef, Cp, C4, 9 * wm, bn));
        P.kchunks = Cp / 64;
        fwd_epi(P, D, d.d_b4_conv_bias, D->x5, kSqrt2, d.conv_clamp, C4, bn, 4);
        P.err_flag = D->err_flag;
        DLA(conv_taps(D, P, false));
    }
    auto sample_rows = [&](TapGemmParams& P) {        // M rows = samples: 128 samples x one pixel per tile
        P.th = 1; P.tw = 1; P.nb = 128; P.halo = 0;
        P.tiles_n = (B + 127) / 128; P.batch = B; P.nprob = 1;
        P.prob[0].vh = P.prob[0].vw = 1; P.prob[0].tiles_h = P.prob[0].tiles_w = 1; P.prob[0].tile_begin = 0;
        P.m_tiles = P.tiles_n;
    };
    {   // dense 16*C4 -> C4 as 16 taps over the 4x4 positions of x5
        TapGemmParams& P = D->FF;
        memset(&P, 0, sizeof P);
        sample_rows(P);
        DLA(dense_maps(D, P, 0, 1, D->x5, C4, 4, 4, 1, 1, 128));
        int nt = 0;
        for (int hw = 0; hw < 16; ++hw) add_tap(P, nt, hw / 4, hw % 4, hw, 0, 1, 16, split);
        P.prob[0].tap_begin = 0; P.prob[0].ntaps = nt;
        const int bn = 64;
        DLA(make_b_map(P, D->wff, C4, C4, 16 * wm, bn));
        P.kchunks = C4 / 64;
        fwd_epi(P, D, d.d_b4_fc_bias, D->x6, kSqrt2, -1.f, C4, bn, 1);
        P.staged = 0;
        P.err_flag = D->err_flag;
        DLA(tapgemm_finalize(P));
    }
    {   // dense backward: gz6 [B, C4] -> gradient wrt x5 (all 16 positions as columns), through conv's activation -> gz5
        TapGemmParams& P = D->BF;
        memset(&P, 0, sizeof P);
        sample_rows(P);
        DLA(dense_maps(D, P, 0, 1, D->gz6, C4, 1, 1, 1, 1, 128));
        const int bn = 64;
        DLA(make_b_map(P, D->wfb, C4, 16 * C4, wm, bn));
        P.kchunks = C4 / 64;
        lin_epi(P, D, 16 * C4, bn, 1, 1);
        P.lin_saved = D->x5.hi; P.lin_saved_lo = D->x5.lo; P.lin_gz = D->gz5.hi; P.lin_gz_lo = D->gz5.lo;
        P.act_gain = kSqrt2; P.act_clamp = d.conv_clamp;
        P.err_flag = D->err_flag;
        DLA(one_tap(D, P));
    }
    {   // 3x3 conv backward: gz5 -> gradient wrt [x | stddev]
        TapGemmParams& P = D->BE;
        memset(&P, 0, sizeof P);
        set_grid(P, 4, B, 1);
        DLA(dense_maps(D, P, 0, 1, D->gz5, C4, 4, 4, P.tw, P.th + P.halo, P.nb));
        const int bn = 64;
        DLA(make_b_map(P, D->web, C4, Cp, 9 * wm, bn));
        P.kchunks = C4 / 64;
        lin_epi(P, D, Cp, bn, 4, 4);
        P.lin_out = D->gx4p.hi; P.lin_out_lo = D->gx4p.lo;
        P.err_flag = D->err_flag;
        DLA(conv_taps(D, P, true));
    }
    return 0;
}

int prepare_disc(la_disc* D, cudaStream_t s) {
    const la_disc_desc& d = D->d;
    const int split = D->split;
    auto prep = [&](const float* w, int cout, int cin, int k2, float scale, int cin_pad, bf16* wf, bf16* wb) -> int {
        const long long total = static_cast<long long>(k2) * cout * cin_pad;
        prep_plain_weights_kernel<<<cdiv(total, 256), 256, 0, s>>>(w, cout, cin, k2, scale, cin_pad, split, wf, wb);
        return static_cast<int>(cudaGetLastError());
    };
    for (Block& k : D->blk) {
        if (!k.p.d_conv0_weight || !k.p.d_conv0_bias || !k.p.d_conv1_weight || !k.p.d_conv1_bias || !k.p.d_skip_weight)
            return dfail(-2, "discriminator: missing block parameters at resolution %d", k.R);
        DLA(prep(k.p.d_conv0_weight, k.C, k.C, 9, 1.f / sqrtf(9.f * k.C), k.C, k.w0f, k.w0b));
        DLA(prep(k.p.d_conv1_weight, k.Cn, k.C, 9, 1.f / sqrtf(9.f * k.C), k.C, k.w1f, k.w1b));
        DLA(prep(k.p.d_skip_weight, k.Cn, k.C, 1, kSqrtHalf / sqrtf(static_cast<float>(k.C)), k.C, k.wsf, k.wsb));
    }
    if (!D->blk[0].p.d_fromrgb_weight || !D->blk[0].p.d_fromrgb_bias) return dfail(-2, "discriminator: missing fromrgb parameters");
    if (!d.d_b4_conv_weight || !d.d_b4_conv_bias || !d.d_b4_fc_weight || !d.d_b4_fc_bias || !d.d_b4_out_weight || !d.d_b4_out_bias)
        return dfail(-2, "discriminator: missing epilogue parameters");
    prep_rgb_w4_kernel<<<cdiv(D->blk[0].C, 128), 128, 0, s>>>(D->blk[0].p.d_fromrgb_weight, D->blk[0].C, d.img_channels,
                                                             1.f / sqrtf(static_cast<float>(d.img_channels)), D->rgb_w4);
    DCU(cudaGetLastError());
    const int C4 = D->C4, Cp = D->Cp;
    DLA(prep(d.d_b4_conv_weight, C4, C4 + 1, 9, 1.f / sqrtf(9.f * (C4 + 1)), Cp, D->wef, D->web));
    prep_fc_weights_kernel<<<cdiv(16LL * C4 * C4, 256), 256, 0, s>>>(d.d_b4_fc_weight, C4, 1.f / sqrtf(16.f * C4), split, D->wff, D->wfb);
    DCU(cudaGetLastError());
    size_t cmax = 16 * static_cast<size_t>(C4);
    for (const Block& k : D->blk) { cmax = k.C > static_cast<int>(cmax) ? k.C : cmax; cmax = k.Cn > static_cast<int>(cmax) ? k.Cn : cmax; }
    const long long n_ones = static_cast<long long>(D->batch) * cmax;
    fill_kernel<<<cdiv(n_ones, 256), 256, 0, s>>>(D->ones, 1.f, n_ones);
    DCU(cudaGetLastError());
    DCU(cudaMemsetAsync(D->err_flag, 0, sizeof(int), s));
    DCU(cudaStreamSynchronize(s));
    return 0;
}

int gemm(la_disc* D, const TapGemmParams& P, cudaStream_t s, long long* launches) {
    if (launches) ++*launches;
    return launch_tapgemm(P, D->num_sms, s);
}
inline unsigned* U32(bf16* p) { return reinterpret_cast<unsigned*>(p); }
inline const unsigned* CU32(const bf16* p) { return reinterpret_cast<const unsigned*>(p); }

}  // namespace

namespace la {

const char* disc_last_error() { return g_derr.c_str(); }
const float* disc_logits(const la_disc* D) { return D->logits; }
int disc_batch(const la_disc* D) { return D->batch; }
int disc_resolution(const la_disc* D) { return D->d.img_resolution; }
int disc_channels(const la_disc* D) { return D->d.img_channels; }

int nchw_to_f4(const float* src, int batch, int C, int res, float4* dst, cudaStream_t s) {
    const long long total = static_cast<long long>(batch) * res * res;
    nchw_to_f4_kernel<<<cdiv(total, 256), 256, 0, s>>>(src, C, res * res, total, dst);
    return static_cast<int>(cudaGetLastError());
}
int f4_to_nchw(const float4* src, int batch, int C, int res, float* dst, cudaStream_t s) {
    const long long total = static_cast<long long>(batch) * res * res;
    f4_to_nchw_kernel<<<cdiv(total, 256), 256, 0, s>>>(src, C, res * res, total, dst);
    return static_cast<int>(cudaGetLastError());
}

int disc_workspace_bytes(const la_disc_desc& d, int batch, int split, size_t* bytes) {
    la_disc tmp{};
    tmp.d = d; tmp.batch = batch; tmp.split = split;
    return plan_disc(&tmp, nullptr, bytes);
}

int disc_create(const la_disc_desc& d, int batch, int split, int num_sms, void* ws, size_t bytes, cudaStream_t s, la_disc** out) {
    la_disc* D = new la_disc{};
    D->d = d; D->batch = batch; D->num_sms = num_sms; D->split = split;
    size_t need = 0;
    int r = plan_disc(D, static_cast<char*>(ws), &need);
    if (!r && need > bytes) r = dfail(-2, "discriminator workspace too small: %zu < %zu", bytes, need);
    if (!r && (reinterpret_cast<uintptr_t>(ws) & 1023)) r = dfail(-2, "discriminator workspace must be 1024-byte aligned");
    if (!r) {
        float f[16];
        cudaError_t ce = cudaMemcpyAsync(f, d.d_resample_filter, sizeof f, cudaMemcpyDeviceToHost, s);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(s);
        if (ce != cudaSuccess) r = dfail(static_cast<int>(ce), "reading the resample filter: %s", cudaGetErrorString(ce));
        for (int jy = 0; jy < 4; ++jy)
            for (int jx = 0; jx < 4; ++jx) D->fir[jy * 4 + jx] = f[(3 - jy) * 4 + (3 - jx)];      // true convolution, gain 1
    }
    if (!r) r = build_disc(D);
    if (!r) r = prepare_disc(D, s);
    if (r) { delete D; return r; }
    *out = D;
    return 0;
}

void disc_destroy(la_disc* D) { delete D; }

int disc_forward(la_disc* D, const float4* img, cudaStream_t s, long long* launches) {
    const la_disc_desc& d = D->d;
    const int B = D->batch;
    Fir16 f;
    for (int i = 0; i < 16; ++i) f.k[i] = D->fir[i];
    {
        Block& k = D->blk[0];
        const long long npix = static_cast<long long>(B) * k.R * k.R;
        const int hc = k.C / 2, cpb = hc < 256 ? hc : 256;
        fromrgb_fwd_kernel<<<dim3(cdiv(npix, kRgbPixels), hc / cpb), 256, 0, s>>>(img, k.p.d_fromrgb_weight, k.p.d_fromrgb_bias, npix, k.C, d.img_channels,
                                                                                1.f / sqrtf(static_cast<float>(d.img_channels)), kSqrt2, 0.2f, d.conv_clamp,
                                                                                U32(k.x_in.hi), U32(k.x_in.lo));
        DCU(cudaGetLastError());
        if (launches) ++*launches;
    }
    for (Block& k : D->blk) {
        DLA(gemm(D, k.F0, s, launches));
        DLA(upfir_backward(k.blur, s));                               // blur: x0 -> yb
        DLA(gemm(D, k.F1, s, launches));
        firdown_fwd_kernel<<<dim3(cdiv((k.R / 2) * (k.C / 2), 256), k.R / 2, B), 256, 0, s>>>(CU32(k.x_in.hi), CU32(k.x_in.lo), B, k.R, k.C, f,
                                                                                           U32(D->ys.hi), U32(D->ys.lo));
        DCU(cudaGetLastError());
        DLA(gemm(D, k.FS, s, launches));
        if (launches) *launches += 2;
    }
    const Block& last = D->blk.back();
    const int G = d.mbstd_group_size < B ? d.mbstd_group_size : B;
    if (B % G) return dfail(-2, "discriminator: batch %d is not a multiple of the minibatch-stddev group %d", B, G);
    const int M = B / G;
    mbstd_stat_kernel<<<M, 256, 0, s>>>(last.y.hi, last.y.lo, B, G, D->C4, D->feat);
    mbstd_concat_kernel<<<cdiv(static_cast<long long>(B) * 16 * D->Cp, 256), 256, 0, s>>>(last.y.hi, last.y.lo, D->feat, B, M, D->C4, D->Cp, D->x4p.hi,
                                                                                      D->x4p.lo);
    DCU(cudaGetLastError());
    DLA(gemm(D, D->FE, s, launches));
    DLA(gemm(D, D->FF, s, launches));
    out_fwd_kernel<<<cdiv(B, 8), 256, 0, s>>>(D->x6.hi, D->x6.lo, d.d_b4_out_weight, d.d_b4_out_bias, B, D->C4, 1.f / sqrtf(static_cast<float>(D->C4)),
                                              D->logits);
    DCU(cudaGetLastError());
    if (launches) *launches += 3;
    return 0;
}

int disc_backward(la_disc* D, float w_disc, float4* g_img, int accumulate, float* d_loss, cudaStream_t s, long long* launches) {
    const la_disc_desc& d = D->d;
    const int B = D->batch, C4 = D->C4, Cp = D->Cp;
    const int G = d.mbstd_group_size < B ? d.mbstd_group_size : B;
    const int M = B / G;
    Block& last = D->blk.back();
    disc_loss_kernel<<<1, 256, 0, s>>>(D->logits, B, w_disc, d_loss, D->gl);
    out_bwd_kernel<<<cdiv(static_cast<long long>(B) * C4, 256), 256, 0, s>>>(D->gl, d.d_b4_out_weight, D->x6.hi, B, C4, 1.f / sqrtf(static_cast<float>(C4)),
                                                                         kSqrt2, 0.2f, D->gz6.hi, D->gz6.lo);
    DCU(cudaGetLastError());
    DLA(gemm(D, D->BF, s, launches));
    DLA(gemm(D, D->BE, s, launches));
    mbstd_gfeat_kernel<<<M, 128, 0, s>>>(D->gx4p.hi, D->gx4p.lo, B, M, C4, Cp, D->gfeat);
    mbstd_bwd_kernel<<<cdiv(static_cast<long long>(M) * 16 * C4, 256), 256, 0, s>>>(
        last.y.hi, last.y.lo, D->gx4p.hi, D->gx4p.lo, D->gfeat, last.y1.hi, last.y1.lo, B, G, C4, Cp, kSqrt2 * kSqrtHalf, 0.2f,
        d.conv_clamp >= 0.f ? d.conv_clamp * kSqrtHalf : d.conv_clamp, last.g_y.hi, last.g_y.lo, last.g_z1.hi, last.g_z1.lo);
    DCU(cudaGetLastError());
    if (launches) *launches += 4;
    for (int b = d.num_blocks - 1; b >= 0; --b) {
        Block& k = D->blk[b];
        DLA(gemm(D, k.BS, s, launches));                              // g_ys = Ws^T g_y
        DLA(gemm(D, k.B1, s, launches));                              // g_yb = conv1^T g_z1
        DLA(upfir_forward(k.blur, s));                                // g_z0 = blur^T(g_yb) * act0'(x0)
        if (b == 0) {                                                 // + fused fromrgb backward: atomics into g_img
            if (!accumulate) DCU(cudaMemsetAsync(g_img, 0, sizeof(float4) * static_cast<size_t>(B) * k.R * k.R, s));
            TapGemmParams P = k.B0;
            P.lin_rgb_g = g_img;
            DLA(gemm(D, P, s, launches));
        } else {
            DLA(gemm(D, k.B0, s, launches));                          // conv0^T + FIRdown^T(g_ys) -> block input gradient
        }
        if (launches) *launches += 1;
    }
    return 0;
}

}  // namespace la
