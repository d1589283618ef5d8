// Perceptual (LPIPS) term of the LatentAugment loop (reference calc_loss_lpips_torchscript / calc_loss_lpips_tr,
// augments/utils/util_latent_aug.py:387-424; augments/criteria/lpips/networks.py:36-97, lpips.py:44-68, utils.py:6-8;
// crop pipeline augments/utils/util_dataset.py:284-332).
//
//   per modality c of the synthetic image:  64x64 crop -> replicate to 3 channels -> z-score -> VGG16 (13 plain 3x3
//   convs + ReLU, 2x2 max-pools) -> taps relu{1_2, 2_2, 3_3, 4_3, 5_3} (the used subset) -> channel-normalised
//   activations n^ -> distance to every bank image  d_ij = sum_taps mean_hw sum_ch w_ch (n^_i - n^_j)^2.
//
// The loss is a pair mean / pair sum of d_ij, so like the other bank criteria (SURVEY.md App. B) it depends on the bank
// only through its moments: b_bar = mean_j n^_j (per modality, tap, position, channel) and M2 = mean_j sum w n^_j^2 / hw.
// Every convolution and its data gradient is a tap-GEMM launch (forward epilogue with demod = 1, ReLU as lrelu with
// slope 0; kEpiLinear for the transposed convolutions with the producer's ReLU mask fused); pools, taps and the crop are
// small SIMT kernels.  Runs in the engine's precision (bf16, or split-bf16 planes in fp32_parity).
#include "lpips.cuh"

#include <cuda_bf16.h>
#include <math.h>
#include <string.h>

#include "common.cuh"
#include "kernels.cuh"
#include "plan.cuh"
#include "tapgemm.cuh"
#include "vgg.cuh"

using namespace la;

namespace {

constexpr char kModule[] = "lpips";
typedef __nv_bfloat16 bf16;

static_assert(kNConv == LA_VGG_CONVS, "VGG16 has 13 convolutions");
const int kTapConv[LA_VGG_TAPS] = {1, 3, 6, 9, 12};                        // conv whose ReLU output is tap t (a pool follows 1, 3, 6, 9)

// per-call constants, device resident (one captured graph serves every call)
struct CallConsts {
    int crop_x, crop_y;      // absolute origin of the crop window in the image
    float w_lpips;
    float norm;              // pair normaliser: 1 / n (lpips_script form) or 1 (forward_tr form)
};

// ------------------------------------------------------------------------- crop (+ replicate + z-score) and its adjoint
// x_in [crop = b*imgc + c][y][x][64]: channels 0..2 = (img[b, cy+y, cx+x].c - mean_k) / std_k, 3..63 = 0.
// src_nchw != null: bank path, crops come as fp32 [n, imgc, cs, cs] (n_valid crops, the rest of the chunk is zero).
struct ZScore { float mean[3], inv_std[3]; };
// f > 0: whole-image window of a per-sample-target call (origin 0, 0; res = f * cs), area-downsampled f x f (the mean of each
// f x f block).  f == 0: the crop window at the call's origin (bank mode).
__global__ void lpips_crop_kernel(const float4* __restrict__ img, const float* __restrict__ src_nchw, int n_valid, const CallConsts* cc, int res,
                                  int imgc, int cs, int ncrops, ZScore z, int f, bf16* x_hi, bf16* x_lo) {
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (idx >= static_cast<long long>(ncrops) * cs * cs) return;
    const int x = static_cast<int>(idx % cs), y = static_cast<int>((idx / cs) % cs), crop = static_cast<int>(idx / (static_cast<long long>(cs) * cs));
    const int b = crop / imgc, c = crop - b * imgc;
    float v = 0.f;
    bool valid = true;
    if (src_nchw) {
        valid = b < n_valid;
        if (valid) v = __ldg(src_nchw + (static_cast<long long>(crop) * cs + y) * cs + x);
    } else {
        const int oy = f ? 0 : cc->crop_y, ox = f ? 0 : cc->crop_x, k = f ? f : 1;
        for (int dy = 0; dy < k; ++dy)
            for (int dx = 0; dx < k; ++dx) {
                const float4 p = __ldg(img + (static_cast<long long>(b) * res + oy + k * y + dy) * res + ox + k * x + dx);
                v += c == 0 ? p.x : (c == 1 ? p.y : p.z);
            }
        if (k > 1) v *= 1.f / static_cast<float>(k * k);
    }
    float ch[4] = {0.f, 0.f, 0.f, 0.f};
    if (valid) {
#pragma unroll
        for (int k = 0; k < 3; ++k) ch[k] = (v - z.mean[k]) * z.inv_std[k];
    }
    uint4* dh = reinterpret_cast<uint4*>(x_hi + idx * 64);
    uint4 first = make_uint4(pack2(ch[0], ch[1]), pack2(ch[2], 0.f), 0u, 0u);
    const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
    dh[0] = first;
#pragma unroll
    for (int j = 1; j < 8; ++j) dh[j] = zero;
    if (x_lo) {
        uint4* dl = reinterpret_cast<uint4*>(x_lo + idx * 64);
        dl[0] = make_uint4(pack2(ch[0] - rnd(ch[0]), ch[1] - rnd(ch[1])), pack2(ch[2] - rnd(ch[2]), 0.f), 0u, 0u);
#pragma unroll
        for (int j = 1; j < 8; ++j) dl[j] = zero;
    }
}
// g_img[b, cy+y, cx+x].c += sum_k g_in[crop, y, x, k] / std_k   (f as in lpips_crop_kernel; f > 1: / f^2 to each pixel of the
// f x f block, the pool's adjoint)
__global__ void lpips_crop_bwd_kernel(const bf16* __restrict__ g_hi, const bf16* __restrict__ g_lo, const CallConsts* cc, int res, int imgc, int cs,
                                      int ncrops, ZScore z, int f, float4* g_img) {
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (idx >= static_cast<long long>(ncrops) * cs * cs) return;
    const int x = static_cast<int>(idx % cs), y = static_cast<int>((idx / cs) % cs), crop = static_cast<int>(idx / (static_cast<long long>(cs) * cs));
    const int b = crop / imgc, c = crop - b * imgc;
    float g = 0.f;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        float v = __bfloat162float(g_hi[idx * 64 + k]);
        if (g_lo) v += __bfloat162float(g_lo[idx * 64 + k]);
        g = fmaf(v, z.inv_std[k], g);
    }
    const int oy = f ? 0 : cc->crop_y, ox = f ? 0 : cc->crop_x, k = f ? f : 1;
    if (k > 1) g *= 1.f / static_cast<float>(k * k);
    for (int dy = 0; dy < k; ++dy)
        for (int dx = 0; dx < k; ++dx) {
            float* dst = reinterpret_cast<float*>(g_img + (static_cast<long long>(b) * res + oy + k * y + dy) * res + ox + k * x + dx) + c;
            *dst += g;
        }
}

// ------------------------------------------------------------------------- 2x2 max-pool and its adjoint (+ tap gradient + ReLU mask)
// thread per (coarse pixel, channel pair)
__global__ void pool_fwd_kernel(const unsigned* __restrict__ x_hi, const unsigned* __restrict__ x_lo, int n, int R, int C, unsigned* p_hi,
                                unsigned* p_lo) {
    const int hc = C >> 1, Ro = R >> 1;
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (idx >= static_cast<long long>(n) * Ro * Ro * hc) return;
    const int cp = static_cast<int>(idx % hc);
    const long long pix = idx / hc;
    const int ox = static_cast<int>(pix % Ro), oy = static_cast<int>((pix / Ro) % Ro);
    const long long b = pix / (static_cast<long long>(Ro) * Ro);
    float m0 = -__int_as_float(0x7f800000), m1 = m0;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int dx = 0; dx < 2; ++dx) {
            const float2 v = ld_sp2(x_hi, x_lo, ((b * R + 2 * oy + dy) * R + 2 * ox + dx) * hc + cp);
            m0 = fmaxf(m0, v.x);
            m1 = fmaxf(m1, v.y);
        }
    st_sp2(p_hi, p_lo, idx, m0, m1);
}
// g_z[fine] = (route(g_pool) + tap gradient) * (x > 0);  route: the first maximum of the window in row-major order takes
// the coarse gradient (torch max_pool2d backward); x is a ReLU output, so the mask is its own activation gradient.
__global__ void pool_bwd_kernel(const unsigned* __restrict__ gp_hi, const unsigned* __restrict__ gp_lo, const unsigned* __restrict__ x_hi,
                                const unsigned* __restrict__ x_lo, const unsigned* __restrict__ tg_hi, const unsigned* __restrict__ tg_lo, int n, int R,
                                int C, unsigned* gz_hi, unsigned* gz_lo) {
    const int hc = C >> 1, Ro = R >> 1;
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (idx >= static_cast<long long>(n) * Ro * Ro * hc) return;
    const int cp = static_cast<int>(idx % hc);
    const long long pix = idx / hc;
    const int ox = static_cast<int>(pix % Ro), oy = static_cast<int>((pix / Ro) % Ro);
    const long long b = pix / (static_cast<long long>(Ro) * Ro);
    const float2 g = ld_sp2(gp_hi, gp_lo, idx);
    float2 v[4];
    long long off[4];
    int a0 = 0, a1 = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        off[k] = ((b * R + 2 * oy + (k >> 1)) * R + 2 * ox + (k & 1)) * hc + cp;
        v[k] = ld_sp2(x_hi, x_lo, off[k]);
        if (k > 0) {
            if (v[k].x > v[a0].x) a0 = k;
            if (v[k].y > v[a1].y) a1 = k;
        }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        float o0 = k == a0 ? g.x : 0.f, o1 = k == a1 ? g.y : 0.f;
        if (tg_hi) { const float2 t = ld_sp2(tg_hi, tg_lo, off[k]); o0 += t.x; o1 += t.y; }
        o0 = v[k].x > 0.f ? o0 : 0.f;
        o1 = v[k].y > 0.f ? o1 : 0.f;
        st_sp2(gz_hi, gz_lo, off[k], o0, o1);
    }
}

// ------------------------------------------------------------------------- taps
// Warp per pixel of one tap tensor x [ncrops, R, R, C] (C = 64 .. 512: each lane owns C / 64 channel pairs).
//   n^ = x / (|x| + 1e-10)                                        (utils.py:6-8)
//   mode 0 (loss + gradient):  S += sum_ch w (n^2 - 2 n^ b_bar) / P;   g_n = coef * w * (n^ - b_bar),
//        coef = -(w_lpips / imgc) * norm * 2 / P;   g_x = g_n / (r + eps) - x <g_n, x> / (r (r + eps)^2)
//        -> out (masked by x > 0 when `mask`: the tap is the last layer, its ReLU gradient is applied here)
//   mode 1 (bank):  b_bar += n^ / M,  M2 += sum_ch w n^2 / (P M)   for the valid crops
//   mode 2 (test hook):  n^ -> fp32 out
// TGT (per-sample targets; bank_mean is then [crop][P][C], one target per crop):
//   mode 1 stores n^ of the target crop;  mode 0:  S[sample] += sum_ch w (n^ - t)^2 / P,  g_n = (2 / P) w (n^ - t)
//   (the projection minimises the distance, so the sign is the opposite of the bank term's)
template <int MODE, bool TGT = false>
__global__ void __launch_bounds__(256) lpips_tap_kernel(const unsigned* __restrict__ x_hi, const unsigned* __restrict__ x_lo, int ncrops, int imgc, int P,
                                                        int C, const float* __restrict__ lin_w, float* bank_mean, const CallConsts* cc, int n_valid_crops,
                                                        float inv_m, double* S, float* m2, int mask, unsigned* out_hi, unsigned* out_lo, float* out_f32) {
    const int warps = blockDim.x >> 5, lane = threadIdx.x & 31;
    const long long total_px = static_cast<long long>(ncrops) * P;
    float s_block = 0.f;             // this warp's loss partial over all its pixels (grid-stride walk: few, long-lived blocks, so
                                     // the loss needs one double atomic per block instead of one per 8 pixels)
    extern __shared__ float s_part[];      // TGT mode 0: this block's loss partial per sample [batch] (dynamic shared memory)
    if (MODE == 0 && TGT) {
        for (int i = threadIdx.x; i < ncrops / imgc; i += blockDim.x) s_part[i] = 0.f;
        __syncthreads();
    }
    for (long long pix = blockIdx.x * static_cast<long long>(warps) + (threadIdx.x >> 5); pix < total_px;
         pix += static_cast<long long>(gridDim.x) * warps) {
    float s_acc = 0.f;
    {
        const int crop = static_cast<int>(pix / P), p = static_cast<int>(pix - static_cast<long long>(crop) * P);
        const int mod = crop % imgc;
        const int hc = C >> 1, npair = C >> 6;           // pairs per lane
        float2 x[8];
        float r2 = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j)
            if (j < npair) {
                x[j] = ld_sp2(x_hi, x_lo, pix * hc + j * 32 + lane);
                r2 = fmaf(x[j].x, x[j].x, fmaf(x[j].y, x[j].y, r2));
            }
        r2 = warp_sum(r2);
        const float r = sqrtf(r2);
        const float inv = 1.f / (r + 1e-10f);
        if (MODE == 2) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (j < npair) reinterpret_cast<float2*>(out_f32)[pix * hc + j * 32 + lane] = make_float2(x[j].x * inv, x[j].y * inv);
        } else if (MODE == 1 && TGT) {
            float* bm = bank_mean + (static_cast<long long>(crop) * P + p) * C;
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (j < npair) reinterpret_cast<float2*>(bm)[j * 32 + lane] = make_float2(__fmul_rn(x[j].x, inv), __fmul_rn(x[j].y, inv));
        } else if (MODE == 1) {
            if (crop < n_valid_crops) {
                float* bm = bank_mean + (static_cast<long long>(mod) * P + p) * C;
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    if (j < npair) {
                        const int ch = 2 * (j * 32 + lane);
                        const float2 w = __ldg(reinterpret_cast<const float2*>(lin_w + ch));
                        const float n0 = x[j].x * inv, n1 = x[j].y * inv;
                        atomicAdd(bm + ch, n0 * inv_m);
                        atomicAdd(bm + ch + 1, n1 * inv_m);
                        s_acc = fmaf(w.x * n0, n0, fmaf(w.y * n1, n1, s_acc));
                    }
                s_acc = warp_sum(s_acc);
                if (lane == 0) atomicAdd(m2 + mod, s_acc * inv_m / P);
            }
        } else {
            const float* bm = bank_mean + (static_cast<long long>(TGT ? crop : mod) * P + p) * C;
            const float coef = TGT ? 2.f / P : -(cc->w_lpips / imgc) * cc->norm * 2.f / P;
            float2 g[8];
            float dot = 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (j < npair) {
                    const int ch = 2 * (j * 32 + lane);
                    const float2 w = __ldg(reinterpret_cast<const float2*>(lin_w + ch));
                    const float2 b = __ldg(reinterpret_cast<const float2*>(bm + ch));
                    // TGT: n^ rounded exactly as the target pass stored it (no FMA contraction into n^ - t), so an image
                    // equal to its target gives exactly zero loss and gradient
                    const float n0 = TGT ? __fmul_rn(x[j].x, inv) : x[j].x * inv, n1 = TGT ? __fmul_rn(x[j].y, inv) : x[j].y * inv;
                    if (TGT) s_acc = fmaf(w.x * (n0 - b.x), n0 - b.x, fmaf(w.y * (n1 - b.y), n1 - b.y, s_acc));
                    else s_acc = fmaf(w.x * n0, n0 - 2.f * b.x, fmaf(w.y * n1, n1 - 2.f * b.y, s_acc));
                    g[j].x = coef * w.x * (n0 - b.x);
                    g[j].y = coef * w.y * (n1 - b.y);
                    dot = fmaf(g[j].x, x[j].x, fmaf(g[j].y, x[j].y, dot));
                }
            dot = warp_sum(dot);
            const float k2 = r > 0.f ? dot * inv * inv / r : 0.f;
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (j < npair) {
                    float o0 = g[j].x * inv - x[j].x * k2, o1 = g[j].y * inv - x[j].y * k2;
                    if (mask) { o0 = x[j].x > 0.f ? o0 : 0.f; o1 = x[j].y > 0.f ? o1 : 0.f; }
                    st_sp2(out_hi, out_lo, pix * hc + j * 32 + lane, o0, o1);
                }
            s_acc = warp_sum(s_acc) / P;
            if (TGT) {
                if (lane == 0) atomicAdd(s_part + crop / imgc, s_acc);
            } else {
                s_block += s_acc;
            }
        }
    }
    }
    if (MODE == 0 && TGT) {       // one double atomic per (block, sample it touched)
        __syncthreads();
        for (int i = threadIdx.x; i < ncrops / imgc; i += blockDim.x)
            if (s_part[i] != 0.f) atomicAdd(S + i, static_cast<double>(s_part[i]));
    } else if (MODE == 0) {       // one double atomic per block
        __shared__ float sm[8];
        if (lane == 0) sm[threadIdx.x >> 5] = s_block;
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int i = 0; i < warps; ++i) t += sm[i];
            atomicAdd(S, t);
        }
    }
}
// loss = (w_lpips / imgc) * norm * (S + n * sum_mod M2_mod)
__global__ void lpips_loss_kernel(const double* S, const float* m2, int imgc, int batch, const CallConsts* cc, float* loss) {
    double m = 0.0;
    for (int c = 0; c < imgc; ++c) m += m2[c];
    loss[0] = static_cast<float>((cc->w_lpips / imgc) * cc->norm * (S[0] + batch * m));
}
// per-sample targets: loss[b] = sum over modalities and taps of the distance of sample b to its own target
__global__ void lpips_target_loss_kernel(const double* S, int batch, float* loss) {
    for (int b = threadIdx.x; b < batch; b += blockDim.x) loss[b] = static_cast<float>(S[b]);
}

struct Conv {
    int R, cin, cin_pad, cout;
    bf16 *wf, *wb;
    Pl x;                       // ReLU output, saved for backward
    TapGemmParams F, B;
};
struct TapL {
    int used, conv, C, R;
    const float* lin_w;
    float* bank_mean;           // [imgc][R*R][C]
    float* target;              // [ncrops][R*R][C] normalised activations of the per-sample targets (when planned)
    Pl tg;                      // gradient wrt the tap tensor (before its ReLU mask); unused for the last tap
};

}  // namespace

struct la_lpips {
    la_vgg_desc d;
    int batch, imgc, res, split, num_sms, ncrops, cs, last_conv, ntaps_used, has_bank;
    int has_targets, pool_f;    // per-sample targets set; area-pool factor res / crop of the whole-image window
    Conv conv[kNConv];
    TapL tap[LA_VGG_TAPS];
    Pl x_in, g_in, pool[4], gp, gz[2];
    float* ones;
    float* m2;                  // [4] per-modality bank constant
    double* S;                  // [batch] (loss partials; one per sample in target mode)
    CallConsts* cc;
    int* err_flag;
    ZScore z;
    float norm_n;
};

namespace {

// blocks of 8 warps, a warp per pixel, grid-stride: at most 8 resident blocks per SM
inline int tap_grid(long long pixels, int num_sms) {
    const long long want = (pixels + 7) / 8, cap = static_cast<long long>(num_sms > 0 ? num_sms : 148) * 8;
    return static_cast<int>(want < cap ? want : cap);
}

int plan_lpips(la_lpips* L, char* ws, size_t* bytes_out) {
    const la_vgg_desc& d = L->d;
    const int cs = d.crop_size, split = L->split;
    if (cs < 64 || (cs & (cs - 1))) return fail(-2, "lpips: crop_size %d unsupported (power of two >= 64)", cs);
    if (L->imgc < 1 || L->imgc > 3) return fail(-2, "lpips: img_channels must be 1..3");
    if (cs > L->res) return fail(-2, "lpips: crop %d larger than the image %d", cs, L->res);
    L->cs = cs;
    L->ncrops = L->batch * L->imgc;
    L->last_conv = -1; L->ntaps_used = 0;
    for (int t = 0; t < LA_VGG_TAPS; ++t) {
        TapL& T = L->tap[t];
        T.used = d.d_lin_weight[t] != nullptr;
        T.conv = kTapConv[t]; T.C = kCout[T.conv]; T.R = cs >> kShift[T.conv]; T.lin_w = d.d_lin_weight[t];
        if (T.used) { L->last_conv = T.conv; ++L->ntaps_used; }
    }
    if (L->last_conv < 0) return fail(-2, "lpips: no tap has a lin weight");
    Bump bp;
    bp.base = ws;
    const size_t n = L->ncrops, wm = split ? 2 : 1;
    L->x_in = bp.take_pl(n * cs * cs * 64, split);
    L->g_in = bp.take_pl(n * cs * cs * 64, split);
    size_t max_x = 0, max_p = 0;
    for (int i = 0; i <= L->last_conv; ++i) {
        Conv& c = L->conv[i];
        c.R = cs >> kShift[i]; c.cin = kCin[i]; c.cin_pad = (kCin[i] + 63) / 64 * 64; c.cout = kCout[i];
        c.wf = bp.take<bf16>(wm * 9 * c.cout * c.cin_pad);
        c.wb = bp.take<bf16>(wm * 9 * c.cout * c.cin_pad);
        const size_t xs = n * c.R * c.R * c.cout;
        c.x = bp.take_pl(xs, split);
        max_x = xs > max_x ? xs : max_x;
    }
    for (int k = 0; k < 4; ++k) {
        const int ci = kTapConv[k];
        if (ci + 1 > L->last_conv) break;
        const size_t ps = n * (L->conv[ci].R / 2) * (L->conv[ci].R / 2) * L->conv[ci].cout;
        L->pool[k] = bp.take_pl(ps, split);
        max_p = ps > max_p ? ps : max_p;
    }
    L->gp = bp.take_pl(max_p ? max_p : 64, split);
    L->gz[0] = bp.take_pl(max_x, split);
    L->gz[1] = bp.take_pl(max_x, split);
    for (int t = 0; t < LA_VGG_TAPS; ++t) {
        TapL& T = L->tap[t];
        if (!T.used) continue;
        T.bank_mean = bp.take<float>(static_cast<size_t>(L->imgc) * T.R * T.R * T.C);
        if (T.conv != L->last_conv) T.tg = bp.take_pl(n * T.R * T.R * T.C, split);
        T.target = d.per_sample_targets ? bp.take<float>(n * T.R * T.R * T.C) : nullptr;    // fp32, ~32 MB per crop at a 256 window
    }
    L->ones = bp.take<float>(n * 512);
    L->m2 = bp.take<float>(4);
    L->S = bp.take<double>(L->batch);
    L->cc = bp.take<CallConsts>(1);
    L->err_flag = bp.take<int>(1);
    bp.take<char>(1024);
    *bytes_out = bp.off;
    return 0;
}

int build_lpips(la_lpips* L) {
    const int split = L->split;
    for (int i = 0; i <= L->last_conv; ++i) {
        Conv& c = L->conv[i];
        bool pooled_in = false;
        int pk = -1;
        for (int k = 0; k < 4; ++k) if (kTapConv[k] + 1 == i) { pooled_in = true; pk = k; }
        const Pl& in = i == 0 ? L->x_in : (pooled_in ? L->pool[pk] : L->conv[i - 1].x);
        LA(plan_layer(c.F, LayerTaps::k3x3, in, L->ncrops, c.R, c.cin_pad, c.cout, c.wf, split, L->err_flag));
        fwd_epilogue(c.F, L->ones, L->d.d_conv_bias[i], 1.f, -1.f, 0.f, c.x);                  // ReLU
        // data gradient: g_z (wrt this conv's pre-activation) -> gradient wrt its input
        TapGemmParams& P = c.B;
        LA(plan_layer(P, LayerTaps::k3x3Flipped, L->gz[i & 1], L->ncrops, c.R, c.cout, c.cin_pad, c.wb, split, L->err_flag));
        linear_epilogue(P, 0.f);
        if (i == 0) { P.lin_out = L->g_in.hi; P.lin_out_lo = L->g_in.lo; }
        else if (pooled_in) { P.lin_out = L->gp.hi; P.lin_out_lo = L->gp.lo; }
        else { P.lin_saved = L->conv[i - 1].x.hi; P.lin_gz = L->gz[(i - 1) & 1].hi; P.lin_gz_lo = L->gz[(i - 1) & 1].lo; }
    }
    return 0;
}

int prepare_lpips(la_lpips* L, cudaStream_t s) {
    for (int i = 0; i <= L->last_conv; ++i) {
        Conv& c = L->conv[i];
        if (!L->d.d_conv_weight[i] || !L->d.d_conv_bias[i]) return fail(-2, "lpips: missing parameters of conv %d", i);
        LA(vgg_prep_weights(L->d.d_conv_weight[i], c.cout, c.cin, c.cin_pad, L->split, c.wf, c.wb, s));
    }
    const long long n_ones = static_cast<long long>(L->ncrops) * 512;
    LA(fill(L->ones, 1.f, n_ones, s));
    CU(cudaMemsetAsync(L->err_flag, 0, sizeof(int), s));
    CU(cudaMemsetAsync(L->m2, 0, 4 * sizeof(float), s));
    CU(cudaMemsetAsync(L->S, 0, sizeof(double) * L->batch, s));
    CU(cudaMemsetAsync(L->cc, 0, sizeof(CallConsts), s));
    CU(cudaStreamSynchronize(s));
    return 0;
}

// convs + pools from x_in up to the last used tap
int run_network(la_lpips* L, cudaStream_t s, long long* launches) {
    for (int i = 0; i <= L->last_conv; ++i) {
        Conv& c = L->conv[i];
        LA(launch_tapgemm(c.F, L->num_sms, s));
        if (launches) ++*launches;
        for (int k = 0; k < 4; ++k)
            if (kTapConv[k] == i && i + 1 <= L->last_conv) {
                LA(vgg_pool_fwd(c.x, L->ncrops, c.R, c.cout, L->pool[k], s));
                if (launches) ++*launches;
            }
    }
    return 0;
}

}  // namespace

namespace la {

int vgg_prep_weights(const float* w, int cout, int cin, int cin_pad, int split, bf16* wf, bf16* wb, cudaStream_t s) {
    return prep_plain_weights(w, cout, cin, 9, 1.f, cin_pad, split, wf, wb, s);
}

int vgg_pool_fwd(const Pl& x, int n, int R, int C, const Pl& out, cudaStream_t s) {
    const long long total = static_cast<long long>(n) * (R / 2) * (R / 2) * (C / 2);
    pool_fwd_kernel<<<cdiv(total, 256), 256, 0, s>>>(CU32(x.hi), CU32(x.lo), n, R, C, U32(out.hi), U32(out.lo));
    CU(cudaGetLastError());
    return 0;
}
int lpips_has_bank(const la_lpips* L) { return L->has_bank; }
int lpips_num_taps(const la_lpips* L) { return L->ntaps_used; }

int lpips_workspace_bytes(const la_vgg_desc& d, int batch, int img_channels, int split, size_t* bytes) {
    la_lpips* tmp = new la_lpips{};
    tmp->d = d; tmp->batch = batch; tmp->imgc = img_channels; tmp->split = split; tmp->res = 1 << 20;
    const int r = plan_lpips(tmp, nullptr, bytes);
    delete tmp;
    return r;
}

int lpips_create(const la_vgg_desc& d, int batch, int img_channels, int img_resolution, int split, int num_sms, void* ws, size_t bytes,
                 cudaStream_t s, la_lpips** out) {
    la_lpips* L = new la_lpips{};
    L->d = d; L->batch = batch; L->imgc = img_channels; L->res = img_resolution; L->split = split; L->num_sms = num_sms;
    for (int k = 0; k < 3; ++k) {
        if (!(d.std[k] > 0.f)) { delete L; return fail(-2, "lpips: std[%d] must be positive", k); }
        L->z.mean[k] = d.mean[k]; L->z.inv_std[k] = 1.f / d.std[k];
    }
    L->pool_f = 1;
    if (d.per_sample_targets) {       // whole-image window: crop == res, or res / 2 with a 2x2 area pool (512 -> 256)
        if (img_resolution > 512 || (d.crop_size != img_resolution && 2 * d.crop_size != img_resolution) ||
            d.crop_size != (img_resolution < 256 ? img_resolution : 256)) {
            delete L;
            return fail(-2, "lpips: per-sample targets need crop_size == min(res, 256) and res <= 512 (crop %d, res %d)", d.crop_size, img_resolution);
        }
        L->pool_f = img_resolution / d.crop_size;
    }
    size_t need = 0;
    int r = plan_lpips(L, static_cast<char*>(ws), &need);
    if (!r) r = check_workspace(kModule, need, bytes, ws);
    if (!r) r = build_lpips(L);
    if (!r) r = prepare_lpips(L, s);
    if (r) { delete L; return r; }
    *out = L;
    return 0;
}

void lpips_destroy(la_lpips* L) { delete L; }

int lpips_set_call(la_lpips* L, int crop_x, int crop_y, float w_lpips, int norm_mode, cudaStream_t s) {
    if (crop_x < 0 || crop_y < 0 || crop_x + L->cs > L->res || crop_y + L->cs > L->res)
        return fail(-2, "lpips: crop window (%d, %d) + %d leaves the %d x %d image", crop_x, crop_y, L->cs, L->res, L->res);
    // (staged through pageable host memory: the copy is complete when the call returns, so the stack value may die)
    const CallConsts h{crop_x, crop_y, w_lpips, norm_mode ? 1.f : 1.f / static_cast<float>(L->batch)};
    CU(cudaMemcpyAsync(L->cc, &h, sizeof h, cudaMemcpyHostToDevice, s));
    return 0;
}

int lpips_set_bank(la_lpips* L, const float* d_crops, int M, cudaStream_t s, long long* launches) {
    if (M < 1) return fail(-2, "lpips: empty bank");
    for (int t = 0; t < LA_VGG_TAPS; ++t)
        if (L->tap[t].used)
            CU(cudaMemsetAsync(L->tap[t].bank_mean, 0, sizeof(float) * static_cast<size_t>(L->imgc) * L->tap[t].R * L->tap[t].R * L->tap[t].C, s));
    CU(cudaMemsetAsync(L->m2, 0, 4 * sizeof(float), s));
    const long long npx = static_cast<long long>(L->ncrops) * L->cs * L->cs;
    for (int m0 = 0; m0 < M; m0 += L->batch) {
        const int nv = M - m0 < L->batch ? M - m0 : L->batch;
        lpips_crop_kernel<<<cdiv(npx, 256), 256, 0, s>>>(nullptr, d_crops + static_cast<long long>(m0) * L->imgc * L->cs * L->cs, nv, L->cc, L->res,
                                                        L->imgc, L->cs, L->ncrops, L->z, 0, L->x_in.hi, L->x_in.lo);
        CU(cudaGetLastError());
        LA(run_network(L, s, launches));
        for (int t = 0; t < LA_VGG_TAPS; ++t) {
            TapL& T = L->tap[t];
            if (!T.used) continue;
            const Conv& c = L->conv[T.conv];
            const long long pixels = static_cast<long long>(L->ncrops) * T.R * T.R;
            lpips_tap_kernel<1><<<tap_grid(pixels, L->num_sms), 256, 0, s>>>(CU32(c.x.hi), CU32(c.x.lo), L->ncrops, L->imgc, T.R * T.R, T.C, T.lin_w, T.bank_mean, L->cc,
                                                              nv * L->imgc, 1.f / M, nullptr, L->m2, 0, nullptr, nullptr, nullptr);
            CU(cudaGetLastError());
        }
    }
    L->has_bank = 1;
    return 0;
}

int lpips_forward(la_lpips* L, const float4* img, int targets, cudaStream_t s, long long* launches) {
    const long long npx = static_cast<long long>(L->ncrops) * L->cs * L->cs;
    lpips_crop_kernel<<<cdiv(npx, 256), 256, 0, s>>>(img, nullptr, L->batch, L->cc, L->res, L->imgc, L->cs, L->ncrops, L->z, targets ? L->pool_f : 0,
                                                    L->x_in.hi, L->x_in.lo);
    CU(cudaGetLastError());
    if (launches) ++*launches;
    return run_network(L, s, launches);
}

int lpips_has_targets(const la_lpips* L) { return L->has_targets; }

int lpips_set_targets(la_lpips* L, const float4* img, cudaStream_t s, long long* launches) {
    bool planned = false;
    for (int t = 0; t < LA_VGG_TAPS; ++t) planned = planned || L->tap[t].target;
    if (!planned) return fail(-2, "lpips: per-sample targets were not planned (la_vgg_desc.per_sample_targets = 0)");
    LA(lpips_set_call(L, 0, 0, 1.f, 1, s));
    LA(lpips_forward(L, img, 1, s, launches));
    for (int t = 0; t < LA_VGG_TAPS; ++t) {
        TapL& T = L->tap[t];
        if (!T.used) continue;
        const Conv& c = L->conv[T.conv];
        const long long pixels = static_cast<long long>(L->ncrops) * T.R * T.R;
        lpips_tap_kernel<1, true><<<tap_grid(pixels, L->num_sms), 256, 0, s>>>(CU32(c.x.hi), CU32(c.x.lo), L->ncrops, L->imgc, T.R * T.R, T.C, T.lin_w,
                                                                          T.target, L->cc, L->ncrops, 0.f, nullptr, nullptr, 0, nullptr, nullptr, nullptr);
        CU(cudaGetLastError());
        if (launches) ++*launches;
    }
    L->has_targets = 1;
    return 0;
}

int lpips_backward(la_lpips* L, float4* g_img, int accumulate, float* d_loss, int targets, cudaStream_t s, long long* launches) {
    if (targets && !L->has_targets) return fail(-2, "lpips: no per-sample targets (la_set_projection_targets)");
    if (!targets && !L->has_bank) return fail(-2, "lpips: no feature bank (la_set_feature_bank)");
    CU(cudaMemsetAsync(L->S, 0, sizeof(double) * (targets ? L->batch : 1), s));
    if (!accumulate) CU(cudaMemsetAsync(g_img, 0, sizeof(float4) * static_cast<size_t>(L->batch) * L->res * L->res, s));
    for (int t = 0; t < LA_VGG_TAPS; ++t) {
        TapL& T = L->tap[t];
        if (!T.used) continue;
        const Conv& c = L->conv[T.conv];
        const bool last = T.conv == L->last_conv;
        const Pl& out = last ? L->gz[T.conv & 1] : T.tg;
        const long long pixels = static_cast<long long>(L->ncrops) * T.R * T.R;
        if (targets)
            lpips_tap_kernel<0, true><<<tap_grid(pixels, L->num_sms), 256, sizeof(float) * L->batch, s>>>(CU32(c.x.hi), CU32(c.x.lo), L->ncrops, L->imgc, T.R * T.R, T.C, T.lin_w, T.target,
                                                                              L->cc, L->ncrops, 0.f, L->S, nullptr, last ? 1 : 0, U32(out.hi), U32(out.lo), nullptr);
        else
            lpips_tap_kernel<0><<<tap_grid(pixels, L->num_sms), 256, 0, s>>>(CU32(c.x.hi), CU32(c.x.lo), L->ncrops, L->imgc, T.R * T.R, T.C, T.lin_w, T.bank_mean, L->cc,
                                                              L->ncrops, 0.f, L->S, nullptr, last ? 1 : 0, U32(out.hi), U32(out.lo), nullptr);
        CU(cudaGetLastError());
        if (launches) ++*launches;
    }
    for (int i = L->last_conv; i >= 0; --i) {
        Conv& c = L->conv[i];
        LA(launch_tapgemm(c.B, L->num_sms, s));
        if (launches) ++*launches;
        if (i == 0) break;
        int pk = -1;
        for (int k = 0; k < 4; ++k) if (kTapConv[k] + 1 == i) pk = k;
        if (pk >= 0) {          // gradient wrt the pooled tensor -> through the pool, + the tap's own gradient, through the ReLU
            const Conv& pc = L->conv[i - 1];
            const TapL& T = L->tap[pk];
            const long long total = static_cast<long long>(L->ncrops) * (pc.R / 2) * (pc.R / 2) * (pc.cout / 2);
            pool_bwd_kernel<<<cdiv(total, 256), 256, 0, s>>>(CU32(L->gp.hi), CU32(L->gp.lo), CU32(pc.x.hi), CU32(pc.x.lo), T.used ? CU32(T.tg.hi) : nullptr,
                                                            T.used ? CU32(T.tg.lo) : nullptr, L->ncrops, pc.R, pc.cout, U32(L->gz[(i - 1) & 1].hi),
                                                            U32(L->gz[(i - 1) & 1].lo));
            CU(cudaGetLastError());
            if (launches) ++*launches;
        }
    }
    const long long npx = static_cast<long long>(L->ncrops) * L->cs * L->cs;
    lpips_crop_bwd_kernel<<<cdiv(npx, 256), 256, 0, s>>>(L->g_in.hi, L->g_in.lo, L->cc, L->res, L->imgc, L->cs, L->ncrops, L->z,
                                                        targets ? L->pool_f : 0, g_img);
    CU(cudaGetLastError());
    if (targets) lpips_target_loss_kernel<<<1, 128, 0, s>>>(L->S, L->batch, d_loss);
    else lpips_loss_kernel<<<1, 1, 0, s>>>(L->S, L->m2, L->imgc, L->batch, L->cc, d_loss);
    CU(cudaGetLastError());
    if (launches) *launches += 2;
    return 0;
}

int lpips_copy_tap(la_lpips* L, int k, float* d_out, size_t* count, cudaStream_t s) {
    int seen = 0;
    for (int t = 0; t < LA_VGG_TAPS; ++t) {
        TapL& T = L->tap[t];
        if (!T.used) continue;
        if (seen++ != k) continue;
        const size_t n = static_cast<size_t>(L->ncrops) * T.R * T.R * T.C;
        if (count) *count = n;
        if (!d_out) return 0;
        const Conv& c = L->conv[T.conv];
        const long long pixels = static_cast<long long>(L->ncrops) * T.R * T.R;
        lpips_tap_kernel<2><<<tap_grid(pixels, L->num_sms), 256, 0, s>>>(CU32(c.x.hi), CU32(c.x.lo), L->ncrops, L->imgc, T.R * T.R, T.C, T.lin_w, nullptr, L->cc, 0, 0.f,
                                                          nullptr, nullptr, 0, nullptr, nullptr, d_out);
        CU(cudaGetLastError());
        return 0;
    }
    return fail(-2, "lpips: tap %d does not exist", k);
}

}  // namespace la
