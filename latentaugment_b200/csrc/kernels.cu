// Small SIMT kernels around the tap-GEMM (see kernels.cuh).  All fp32 arithmetic.
#include "kernels.cuh"

#include <cuda_bf16.h>

#include "act.cuh"
#include "sm100.cuh"

namespace la {

namespace {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ void split_store(__nv_bfloat16* hi, __nv_bfloat16* lo, long long i, float v) {
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    hi[i] = h;
    if (lo) lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
}
inline int cdiv(long long a, long long b) { return static_cast<int>((a + b - 1) / b); }
inline int last_err() { return static_cast<int>(cudaGetLastError()); }

// ------------------------------------------------------------------------- weight preparation
// One thread per (o, i).  Normal conv: matrix t = ay*3+ax holds w[o,i,ay,ax] (forward tap
// offset (ay-1, ax-1)).  Up-sampling conv (conv_transpose2d stride 2, then 4x4 FIR with
// pad 1 and gain 4 -- reference conv2d_resample.py:112-129, upfirdn2d.py:167-211) folded
// into per-output-phase 3x3 weights: matrix ph*9 + (dy+1)*3 + (dx+1),
//   Wc = sum_{ay,ax} F[3-jy][3-jx] * gain * w[o,i,ay,ax],  j = a + 1 - phase + 2*delta in [0,3].
__global__ void prep_conv_weights_kernel(const float* __restrict__ w, int cout, int cin, int up,
                                         const float* __restrict__ fir, int split, __nv_bfloat16* wf, __nv_bfloat16* wb,
                                         float* w2, float* w2t) {
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (idx >= static_cast<long long>(cout) * cin) return;
    const int o = static_cast<int>(idx / cin), i = static_cast<int>(idx % cin);
    float k[3][3];
    float sq = 0.f;
    for (int a = 0; a < 9; ++a) {
        k[a / 3][a % 3] = w[idx * 9 + a];
        sq += k[a / 3][a % 3] * k[a / 3][a % 3];
    }
    w2[idx] = sq;
    w2t[static_cast<long long>(i) * cout + o] = sq;
    const int nmat = up == 2 ? 36 : 9;
    const long long msz = static_cast<long long>(cout) * cin;
    __nv_bfloat16* wf_lo = split ? wf + nmat * msz : nullptr;
    __nv_bfloat16* wb_lo = split ? wb + nmat * msz : nullptr;
    if (up == 1) {
        for (int a = 0; a < 9; ++a) {
            const float v = k[a / 3][a % 3];
            split_store(wf, wf_lo, a * msz + static_cast<long long>(o) * cin + i, v);
            split_store(wb, wb_lo, a * msz + static_cast<long long>(i) * cout + o, v);
        }
    } else {
        for (int py = 0; py < 2; ++py)
            for (int px = 0; px < 2; ++px)
                for (int dy = -1; dy <= 1; ++dy)
                    for (int dx = -1; dx <= 1; ++dx) {
                        float v = 0.f;
                        for (int ay = 0; ay < 3; ++ay) {
                            const int jy = ay + 1 - py + 2 * dy;
                            if (jy < 0 || jy > 3) continue;
                            for (int ax = 0; ax < 3; ++ax) {
                                const int jx = ax + 1 - px + 2 * dx;
                                if (jx < 0 || jx > 3) continue;
                                v += fir[(3 - jy) * 4 + (3 - jx)] * 4.f * k[ay][ax];
                            }
                        }
                        const int m = (py * 2 + px) * 9 + (dy + 1) * 3 + (dx + 1);
                        split_store(wf, wf_lo, m * msz + static_cast<long long>(o) * cin + i, v);
                        split_store(wb, wb_lo, m * msz + static_cast<long long>(i) * cout + o, v);
                    }
    }
}

__global__ void prep_affine_kernel(const float* __restrict__ aw, const float* __restrict__ ab, int cin, int w_dim,
                                   float wscale, float bscale, float* a_rows, float* b_rows) {
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (idx < static_cast<long long>(cin) * w_dim) a_rows[idx] = aw[idx] * wscale;
    if (idx < cin) b_rows[idx] = ab[idx] * bscale;
}

__global__ void prep_scale_kernel(const float* __restrict__ src, float scale, float* dst, long long n) {
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (idx < n) dst[idx] = src[idx] * scale;
}

__global__ void prep_const_kernel(const float* __restrict__ cst, int C, int hw, float* c_f32, __nv_bfloat16* hi,
                                  __nv_bfloat16* lo) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= C * hw) return;
    const int p = idx / C, c = idx % C;
    const float v = cst[c * hw + p];
    c_f32[idx] = v;
    split_store(hi, lo, idx, v);
}

constexpr int kMaxRowRegs = 32;   // mapping network: a weight row of up to 1024 floats stays in a warp's registers

// ------------------------------------------------------------------------- style GEMMs
// The three per-step style products are small GEMMs  out[n, j] = epi( sum_k X[n, k] * M[j, k] )  over the batch:
//   styles      : X = w (per layer row of ws),        M = affine rows A_cat,  epi = + bias
//   demodulation: X = s^2,                            M = W2  [cout][cin],    epi = rsqrt(. + 1e-8)
//   style grad  : X = red_d * d^2,                    M = W2t [cin][cout],    epi = red_s - s * .
// One block = 32 rows j x 32 samples, K walked in 32-wide slabs staged k-major in shared memory (the next slab is
// fetched into registers while the current one computes); a thread owns a 2 x 4 register tile.  (The earlier warp-per-row kernels re-read every sample vector
// once per row: 0.45 ms per Adam step for 0.5 GFLOP.)
constexpr int kSgRows = 32, kSgK = 32, kSgSamples = 32;
enum { kSgStyles = 0, kSgDemod = 1, kSgGrad = 2 };
struct StyleGemmArgs {
    const float* ws; long long sn, sidx; const float* a_cat; const float* b_cat; int w_dim;     // styles
    const float* s_cat; const float* d_cat; const float* red_s; const float* red_d;           // demod / grad
    float* out;
};
template <int MODE>
__global__ void __launch_bounds__(128) style_gemm_kernel(LayerTable T, int batch, StyleGemmArgs A) {
    __shared__ __align__(16) float Ms[kSgK][kSgRows + 4];
    __shared__ __align__(16) float Xs[kSgK][kSgSamples + 4];
    const int L = blockIdx.y;
    int J, K;
    const float* M;
    long long xbase = 0, obase = 0;       // sample stride of out is J
    long long xs_n = 0;
    int soff = 0;
    if (MODE == kSgStyles) {
        int widx;
        if (L < T.nconv) { J = T.conv[L].cin; soff = T.conv[L].soff; widx = T.conv[L].ws_idx; }
        else { J = T.rgb[L - T.nconv].cin; soff = T.rgb[L - T.nconv].soff; widx = T.rgb[L - T.nconv].ws_idx; }
        K = A.w_dim;
        M = A.a_cat + static_cast<long long>(soff) * K;
        xbase = widx * A.sidx; xs_n = A.sn;
        obase = static_cast<long long>(batch) * soff;
    } else {
        const ConvDesc D = T.conv[L];
        if (MODE == kSgDemod) { J = D.cout; K = D.cin; M = D.w2; xbase = static_cast<long long>(batch) * D.soff; obase = static_cast<long long>(batch) * D.doff; }
        else { J = D.cin; K = D.cout; M = D.w2t; xbase = static_cast<long long>(batch) * D.doff; obase = static_cast<long long>(batch) * D.soff; }
        xs_n = K;
    }
    const int j0 = blockIdx.x * kSgRows;
    if (j0 >= J) return;
    const int n0 = blockIdx.z * kSgSamples;
    const int t = threadIdx.x;
    const int rg = t >> 3, sg = t & 7;          // rows 2*rg.., samples 4*sg..
    const int lk = t & 31, lr = t >> 5;         // loader: k within the slab, first row / sample
    float acc[2][4];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
    float mreg[kSgRows / 4], xreg[kSgSamples / 4];
    auto fetch = [&](int k0) {               // the next slab travels in registers while this one computes
        const int k = k0 + lk;
        const bool kok = k < K;
#pragma unroll
        for (int i = 0; i < kSgRows / 4; ++i) {
            const int r = lr + 4 * i;
            mreg[i] = (kok && j0 + r < J) ? __ldg(M + static_cast<long long>(j0 + r) * K + k) : 0.f;
        }
#pragma unroll
        for (int i = 0; i < kSgSamples / 4; ++i) {
            const int n = lr + 4 * i;
            float v = 0.f;
            if (kok && n0 + n < batch) {
                const long long e = xbase + static_cast<long long>(n0 + n) * xs_n + k;
                if (MODE == kSgStyles) v = __ldg(A.ws + e);
                else if (MODE == kSgDemod) { v = __ldg(A.s_cat + e); v = v * v; }
                else { const float d = __ldg(A.d_cat + e); v = __ldg(A.red_d + e) * d * d; }
            }
            xreg[i] = v;
        }
    };
    fetch(0);
    for (int k0 = 0; k0 < K; k0 += kSgK) {
#pragma unroll
        for (int i = 0; i < kSgRows / 4; ++i) Ms[lk][lr + 4 * i] = mreg[i];
#pragma unroll
        for (int i = 0; i < kSgSamples / 4; ++i) Xs[lk][lr + 4 * i] = xreg[i];
        __syncthreads();
        if (k0 + kSgK < K) fetch(k0 + kSgK);
#pragma unroll 8
        for (int kk = 0; kk < kSgK; ++kk) {
            const float2 m = *reinterpret_cast<const float2*>(&Ms[kk][2 * rg]);
            const float4 x = *reinterpret_cast<const float4*>(&Xs[kk][4 * sg]);
            const float xv[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
            for (int b = 0; b < 4; ++b) { acc[0][b] = fmaf(m.x, xv[b], acc[0][b]); acc[1][b] = fmaf(m.y, xv[b], acc[1][b]); }
        }
        __syncthreads();
    }
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        const int n = n0 + 4 * sg + b;
        if (n >= batch) continue;
#pragma unroll
        for (int a = 0; a < 2; ++a) {
            const int j = j0 + 2 * rg + a;
            if (j >= J) continue;
            const long long o = obase + static_cast<long long>(n) * J + j;
            if (MODE == kSgStyles) A.out[o] = acc[a][b] + __ldg(A.b_cat + soff + j);
            else if (MODE == kSgDemod) A.out[o] = rsqrtf(acc[a][b] + 1e-8f);
            else A.out[o] = __ldg(A.red_s + o) - __ldg(A.s_cat + o) * acc[a][b];
        }
    }
}

__global__ void rgbw_kernel(LayerTable T, int batch, const float* __restrict__ s_cat, float4* rgbw) {
    const RgbDesc D = T.rgb[blockIdx.y];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = blockIdx.z;
    if (i >= D.cin) return;
    const float s = s_cat[static_cast<long long>(batch) * D.soff + static_cast<long long>(n) * D.cin + i];
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    v.x = D.wt[i] * s;
    if (D.img_c > 1) v.y = D.wt[D.cin + i] * s;
    if (D.img_c > 2) v.z = D.wt[2 * D.cin + i] * s;
    rgbw[static_cast<long long>(batch) * D.roff + static_cast<long long>(n) * D.cin + i] = v;
}

__global__ void const_modulate_kernel(const float* __restrict__ c_f32, const float* __restrict__ s0, int batch, int hw, int C,
                                      __nv_bfloat16* hi, __nv_bfloat16* lo) {
    const long long idx = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (idx >= static_cast<long long>(batch) * hw * C) return;
    const int c = static_cast<int>(idx % C);
    const int p = static_cast<int>((idx / C) % hw);
    const int n = static_cast<int>(idx / (static_cast<long long>(C) * hw));
    split_store(hi, lo, idx, c_f32[p * C + c] * s0[static_cast<long long>(n) * C + c]);
}

// ------------------------------------------------------------------------- x2 up-sampling FIR passes
__device__ __forceinline__ unsigned pack2(float a, float b) {
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<unsigned*>(&v);
}
__device__ __forceinline__ void st_bf16x2(unsigned* hi, unsigned* lo, long long i, float a, float b) {
    hi[i] = pack2(a, b);
    if (lo) lo[i] = pack2(a - __bfloat162float(__float2bfloat16_rn(a)), b - __bfloat162float(__float2bfloat16_rn(b)));
}

// Sliding-window 4x4 FIR.  A block = (256 / cpb) consecutive output rows x cpb channel pairs; every thread
// walks 32 output pixels along x keeping the 4x4 source window of its channel pair in registers, so each
// step loads one new window column (4 coalesced 128-byte rows per warp) instead of 16 values; the 4-row
// vertical overlap of neighbouring rows is served by L1.
//   forward : Y[y,x]   = sum_j fk[jy][jx] * T[y+jy-1, x+jx-1]   then  z = Y*d + noise + b; x = clamp(lrelu(z)*gain); x, x*s_next
//   backward: g_T[u]   = sum_j fk[jy][jx] * g_Y[u_y-jy+1, u_x-jx+1]                                  (adjoint)
constexpr int kFirSeg = 32;
template <bool FWD, bool SPLIT, bool SEP>
__global__ void __launch_bounds__(256, SEP ? 3 : 2) upfir_slide_kernel(const __grid_constant__ UpFirParams P, int cpb, int chan_blocks) {
    const int hc = P.C >> 1;
    const int rows_per_block = 256 / cpb;
    const int cb = blockIdx.z % chan_blocks, n = blockIdx.z / chan_blocks;
    const int cp = cb * cpb + threadIdx.x % cpb;
    const int r = blockIdx.y * rows_per_block + threadIdx.x / cpb;
    const int x0 = blockIdx.x * kFirSeg;
    const int TW = P.OW + 1;
    const int out_h = FWD ? P.OH : P.TH, out_w = FWD ? P.OW : TW, out_pitch = FWD ? P.OW : P.TWp;
    const int src_h = FWD ? P.TH : P.OH, src_w = FWD ? TW : P.OW, src_pitch = FWD ? P.TWp : P.OW;
    if (r >= out_h) return;
    const int org = FWD ? -1 : -2;                 // window origin relative to the output pixel
    const unsigned* sh = reinterpret_cast<const unsigned*>(FWD ? P.t_hi : P.gy_hi);
    const unsigned* sl = reinterpret_cast<const unsigned*>(FWD ? P.t_lo : P.gy_lo);
    float wk[16], wy[4], wx[4];                    // SEP: fk[jy][jx] = fy[jy] * fx[jx]
#pragma unroll
    for (int k = 0; k < 16; ++k) wk[k] = FWD ? P.fk[k] : P.fk[15 - k];
#pragma unroll
    for (int k = 0; k < 4; ++k) { wy[k] = FWD ? P.fy[k] : P.fy[3 - k]; wx[k] = FWD ? P.fx[k] : P.fx[3 - k]; }
    // the 4 window rows: element offsets (channel-pair units) of column 0; invalid rows are clamped and masked
    long long rowoff[4];
    float rowmask[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int sr = r + org + k;
        const bool ok = sr >= 0 && sr < src_h;
        rowoff[k] = ((static_cast<long long>(n) * src_h + (ok ? sr : 0)) * src_pitch) * hc + cp;
        rowmask[k] = ok ? 1.f : 0.f;
    }
    float2 win[SEP ? 1 : 4][7];                    // [window row][column]; 3 carried + 4 new columns per group
                                                   // (SEP: one row of vertically filtered column sums)
    auto load_col = [&](int slot, int sc) {        // unconditional (clamped) loads, masked afterwards: no branches
        const bool cok = sc >= 0 && sc < src_w;
        const long long coff = static_cast<long long>(cok ? sc : 0) * hc;
        unsigned u[4], l[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            u[k] = __ldg(sh + rowoff[k] + coff);
            if (SPLIT) l[k] = __ldg(sl + rowoff[k] + coff);
        }
        float2 colsum = make_float2(0.f, 0.f);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float2 v = make_float2(__uint_as_float(u[k] << 16), __uint_as_float(u[k] & 0xffff0000u));
            if (SPLIT) { v.x += __uint_as_float(l[k] << 16); v.y += __uint_as_float(l[k] & 0xffff0000u); }
            if (SEP) {
                const float m = wy[k] * rowmask[k];
                colsum.x = fmaf(m, v.x, colsum.x);
                colsum.y = fmaf(m, v.y, colsum.y);
            } else {
                const float m = cok ? rowmask[k] : 0.f;
                win[k][slot] = make_float2(v.x * m, v.y * m);
            }
        }
        if (SEP) win[0][slot] = cok ? colsum : make_float2(0.f, 0.f);
    };
#pragma unroll
    for (int k = 0; k < 3; ++k) load_col(k, x0 + org + k);

    float2 dm = make_float2(0.f, 0.f), bs = dm, sn = dm;
    const float* nrow = nullptr;
    if (FWD && !P.act_saved) {
        const int c = 2 * cp;
        dm = __ldg(reinterpret_cast<const float2*>(P.demod + static_cast<long long>(n) * P.C + c));
        bs = __ldg(reinterpret_cast<const float2*>(P.bias + c));
        if (P.s_next) sn = __ldg(reinterpret_cast<const float2*>(P.s_next + static_cast<long long>(n) * P.C + c));
        if (P.noise) nrow = P.noise + n * P.noise_stride_n + static_cast<long long>(r) * P.OW;
    }
    unsigned* oh = reinterpret_cast<unsigned*>(FWD ? P.x_hi : P.gt_hi);
    unsigned* ol = SPLIT ? reinterpret_cast<unsigned*>(FWD ? P.x_lo : P.gt_lo) : nullptr;
    unsigned* xsh = reinterpret_cast<unsigned*>(P.xs_hi);
    unsigned* xsl = SPLIT ? reinterpret_cast<unsigned*>(P.xs_lo) : nullptr;
    const long long obase = ((static_cast<long long>(n) * out_h + r) * out_pitch) * hc + cp;

#pragma unroll 1
    for (int xb = 0; xb < kFirSeg; xb += 4) {
        if (x0 + xb >= out_w) break;
#pragma unroll
        for (int u = 0; u < 4; ++u) load_col(3 + u, x0 + xb + org + 3 + u);      // 16 (32) independent loads in flight
        float nzv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) nzv[u] = (FWD && nrow && x0 + xb + u < out_w) ? __ldg(nrow + x0 + xb + u) * P.noise_scale : 0.f;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int x = x0 + xb + u;
            if (x >= out_w) continue;
            float a0 = 0.f, a1 = 0.f;
            if (SEP) {
#pragma unroll
                for (int kx = 0; kx < 4; ++kx) {
                    a0 = fmaf(wx[kx], win[0][u + kx].x, a0);
                    a1 = fmaf(wx[kx], win[0][u + kx].y, a1);
                }
            } else {
#pragma unroll
                for (int ky = 0; ky < 4; ++ky)
#pragma unroll
                    for (int kx = 0; kx < 4; ++kx) {
                        const float2 v = win[ky][u + kx];
                        a0 = fmaf(wk[ky * 4 + kx], v.x, a0);
                        a1 = fmaf(wk[ky * 4 + kx], v.y, a1);
                    }
            }
            const long long o = obase + static_cast<long long>(x) * hc;
            if (FWD && P.act_saved) {
                const unsigned sv = __ldg(reinterpret_cast<const unsigned*>(P.act_saved) + o);
                const unsigned svl = P.act_saved_lo ? __ldg(reinterpret_cast<const unsigned*>(P.act_saved_lo) + o) : 0u;
                const float s0 = __uint_as_float(sv << 16) + __uint_as_float(svl << 16);
                const float s1 = __uint_as_float(sv & 0xffff0000u) + __uint_as_float(svl & 0xffff0000u);
                const float thr = act_saved_clamp(P.act_clamp, P.act_saved_lo != nullptr);
                const float g0 = act_grad(a0 * P.act_gain, s0, P.act_slope, thr), g1 = act_grad(a1 * P.act_gain, s1, P.act_slope, thr);
                st_bf16x2(oh, ol, o, g0, g1);
            } else if (FWD) {
                float z0 = fmaf(a0, dm.x, nzv[u]) + bs.x, z1 = fmaf(a1, dm.y, nzv[u]) + bs.y;
                z0 = (z0 > 0.f ? z0 : z0 * P.act_slope) * P.act_gain;
                z1 = (z1 > 0.f ? z1 : z1 * P.act_slope) * P.act_gain;
                if (P.act_clamp >= 0.f) {
                    z0 = fminf(fmaxf(z0, -P.act_clamp), P.act_clamp);
                    z1 = fminf(fmaxf(z1, -P.act_clamp), P.act_clamp);
                }
                st_bf16x2(oh, ol, o, z0, z1);
                if (P.s_next) st_bf16x2(xsh, xsl, o, z0 * sn.x, z1 * sn.y);
            } else {
                st_bf16x2(oh, ol, o, a0, a1);
            }
        }
#pragma unroll
        for (int ky = 0; ky < (SEP ? 1 : 4); ++ky)
#pragma unroll
            for (int k = 0; k < 3; ++k) win[ky][k] = win[ky][4 + k];
    }
}

// TMA-pipelined 4x4 separable FIR (the same two operators as upfir_slide_kernel).  A CTA owns a strip of
// 32 output columns x 64 channels of one sample and walks down a run of output rows; a producer warp
// streams the source rows (35 pixels x 128 B, zero-filled outside the tensor) into a ring of kFirRing
// slots, four consumer warps (8 output pixels each, lane = channel pair) keep the vertical window in
// the ring, and each warp writes its pixels through a double-buffered staging tile with tensor stores.
// Every source element is read from global memory once (+ the 3-pixel strip halo).
constexpr int kFirRing = 8, kFirStrip = 32, kFirSlotBytes = 4608, kFirInPx = 35;
template <bool FWD>
__global__ void __launch_bounds__(160) upfir_tma_kernel(const __grid_constant__ UpFirParams P, int rows_per_cta, int nslabs) {
    extern __shared__ __align__(128) uint8_t fsm[];
    uint8_t* ring = fsm;                                         // kFirRing x 4608
    uint8_t* stage = fsm + kFirRing * kFirSlotBytes;             // 4 warps x 2 buffers x 2 tensors x 1 KB
    uint64_t* full = reinterpret_cast<uint64_t*>(stage + 4 * 2 * 2 * 1024);
    uint64_t* empty = full + kFirRing;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slab = blockIdx.y % nslabs, rblk = blockIdx.y / nslabs;
    const int n = blockIdx.z;
    const int x0 = blockIdx.x * kFirStrip;
    const int out_h = FWD ? P.OH : P.TH;
    const int r0 = rblk * rows_per_cta, r1 = min(r0 + rows_per_cta, out_h);
    const int org = FWD ? -1 : -2;
    const int c0 = slab * 64;
    const CUtensorMap* in_map = FWD ? &P.fwd_in : &P.bwd_in;
    if (threadIdx.x == 0) {
        for (int s = 0; s < kFirRing; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 4); }
        fence_barrier_init();
        prefetch_tmap(in_map);
    }
    __syncthreads();
    const int nrows_in = (r1 - r0) + 3;
    if (warp == 4) {
        if (lane == 0) {
            for (int j = 0; j < nrows_in; ++j) {
                const int s = j % kFirRing;
                mbar_wait(&empty[s], ((j / kFirRing) & 1) ^ 1, nullptr, 0);
                mbar_expect_tx(&full[s], kFirInPx * 128);
                tma_load_4d(ring + s * kFirSlotBytes, in_map, &full[s], c0, x0 + org, r0 + org + j, n);
            }
        }
        return;
    }
    float wy[4], wx[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) { wy[k] = FWD ? P.fy[k] : P.fy[3 - k]; wx[k] = FWD ? P.fx[k] : P.fx[3 - k]; }
    float2 dm = make_float2(0.f, 0.f), bs = dm, sn = dm;
    const int c = c0 + 2 * lane;
    if (FWD && !P.act_saved) {
        dm = __ldg(reinterpret_cast<const float2*>(P.demod + static_cast<long long>(n) * P.C + c));
        bs = __ldg(reinterpret_cast<const float2*>(P.bias + c));
        if (P.s_next) sn = __ldg(reinterpret_cast<const float2*>(P.s_next + static_cast<long long>(n) * P.C + c));
    }
    const float clampv = P.act_clamp >= 0.f ? P.act_clamp : __int_as_float(0x7f800000);
    const float saved_thr = act_saved_clamp(P.act_clamp, false);         // act_saved: hi plane only (bf16 mode)
    const int px0 = warp * 8;                                    // this warp's first output pixel inside the strip
    uint8_t* my_stage = stage + warp * 4096;
    if constexpr (!FWD) {
        // Separable FIR, horizontal pass first: every input row is read from the ring ONCE, turned into 8 horizontally
        // filtered pixels (x 2 channels) and released; the vertical pass combines the last four such rows, which roll
        // through four register sets (the row loop is unrolled by four so the rotation is a renaming).
        float2 ha[8], hb[8], hc[8], hd[8];
        auto hpass = [&](int j, float2 (&h)[8]) {
            mbar_wait(&full[j % kFirRing], (j / kFirRing) & 1, nullptr, 0);
            const unsigned* row = reinterpret_cast<const unsigned*>(ring + (j % kFirRing) * kFirSlotBytes) + px0 * 32 + lane;
            float2 in[11];
#pragma unroll
            for (int q = 0; q < 11; ++q) {
                const unsigned u = row[q * 32];
                in[q] = make_float2(__uint_as_float(u << 16), __uint_as_float(u & 0xffff0000u));
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[j % kFirRing]);         // the row lives in registers now
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                float a0 = wx[0] * in[i].x, a1 = wx[0] * in[i].y;
#pragma unroll
                for (int k = 1; k < 4; ++k) { a0 = fmaf(wx[k], in[i + k].x, a0); a1 = fmaf(wx[k], in[i + k].y, a1); }
                h[i] = make_float2(a0, a1);
            }
        };
        auto out_row = [&](int r, const float2 (&h0)[8], const float2 (&h1)[8], const float2 (&h2)[8], float2 (&h3)[8]) {
            const int j0 = r - r0;
            hpass(j0 + 3, h3);
            float nzv[8];
            unsigned svv[8];
            if (FWD && P.act_saved) {
                const unsigned* sp = reinterpret_cast<const unsigned*>(P.act_saved) +
                                     ((static_cast<long long>(n) * P.OH + r) * P.OW) * (P.C >> 1) + (c0 >> 1) + lane;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int x = x0 + px0 + i;
                    svv[i] = x < P.OW ? __ldg(sp + static_cast<long long>(x) * (P.C >> 1)) : 0u;
                }
            }
            if (FWD && P.noise && !P.act_saved) {
                const float4* np = reinterpret_cast<const float4*>(P.noise + n * P.noise_stride_n + static_cast<long long>(r) * P.OW + x0 + px0);
                const bool in = x0 + px0 + 8 <= P.OW;
                const float4 a = in ? __ldg(np) : make_float4(0.f, 0.f, 0.f, 0.f), b = in ? __ldg(np + 1) : a;
                nzv[0] = a.x; nzv[1] = a.y; nzv[2] = a.z; nzv[3] = a.w; nzv[4] = b.x; nzv[5] = b.y; nzv[6] = b.z; nzv[7] = b.w;
#pragma unroll
                for (int i = 0; i < 8; ++i) nzv[i] *= P.noise_scale;
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) nzv[i] = 0.f;
            }
            uint8_t* sx = my_stage + (j0 & 1) * 2048;                // [x | xs] x 1 KB, double-buffered by row parity
            if (lane == 0) bulk_wait_read<1>();                       // the stores of two rows ago have read this buffer
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float a0 = fmaf(wy[3], h3[i].x, fmaf(wy[2], h2[i].x, fmaf(wy[1], h1[i].x, wy[0] * h0[i].x)));
                const float a1 = fmaf(wy[3], h3[i].y, fmaf(wy[2], h2[i].y, fmaf(wy[1], h1[i].y, wy[0] * h0[i].y)));
                if (FWD && P.act_saved) {
                    const float s0 = __uint_as_float(svv[i] << 16), s1 = __uint_as_float(svv[i] & 0xffff0000u);
                    const float g0 = act_grad(a0 * P.act_gain, s0, P.act_slope, saved_thr);
                    const float g1 = act_grad(a1 * P.act_gain, s1, P.act_slope, saved_thr);
                    reinterpret_cast<unsigned*>(sx)[i * 32 + lane] = pack2(g0, g1);
                } else if (FWD) {
                    float z0 = fmaf(a0, dm.x, nzv[i]) + bs.x, z1 = fmaf(a1, dm.y, nzv[i]) + bs.y;
                    z0 = (z0 > 0.f ? z0 : z0 * P.act_slope) * P.act_gain;
                    z1 = (z1 > 0.f ? z1 : z1 * P.act_slope) * P.act_gain;
                    z0 = fminf(fmaxf(z0, -clampv), clampv);
                    z1 = fminf(fmaxf(z1, -clampv), clampv);
                    reinterpret_cast<unsigned*>(sx)[i * 32 + lane] = pack2(z0, z1);
                    reinterpret_cast<unsigned*>(sx + 1024)[i * 32 + lane] = pack2(z0 * sn.x, z1 * sn.y);
                } else {
                    reinterpret_cast<unsigned*>(sx)[i * 32 + lane] = pack2(a0, a1);
                }
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                if (FWD) {
                    tma_store_4d(&P.fwd_out_x, sx, c0, x0 + px0, r, n);
                    if (P.s_next && !P.act_saved) tma_store_4d(&P.fwd_out_xs, sx + 1024, c0, x0 + px0, r, n);
                } else {
                    tma_store_4d(&P.bwd_out, sx, c0, x0 + px0, r, n);
                }
                bulk_commit();
            }
        };
        if (r0 < r1) { hpass(0, ha); hpass(1, hb); hpass(2, hc); }
        for (int r = r0; r < r1; r += 4) {
            out_row(r, ha, hb, hc, hd);
            if (r + 1 < r1) out_row(r + 1, hb, hc, hd, ha);
            if (r + 2 < r1) out_row(r + 2, hc, hd, ha, hb);
            if (r + 3 < r1) out_row(r + 3, hd, ha, hb, hc);
        }
    } else {
        // (the forward pass keeps the vertical-first order: with the epilogue state the rolling window needs 136 registers,
        // which costs a resident CTA -- measured slower than the extra arithmetic)
        for (int j = 0; j < 3; ++j) mbar_wait(&full[j % kFirRing], (j / kFirRing) & 1, nullptr, 0);
        for (int r = r0; r < r1; ++r) {
            const int j0 = r - r0;
            mbar_wait(&full[(j0 + 3) % kFirRing], ((j0 + 3) / kFirRing) & 1, nullptr, 0);
            // vertical pass: 11 window columns, 2 channels each
            float2 cs[11];
#pragma unroll
            for (int q = 0; q < 11; ++q) cs[q] = make_float2(0.f, 0.f);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const unsigned* row = reinterpret_cast<const unsigned*>(ring + ((j0 + k) % kFirRing) * kFirSlotBytes) + px0 * 32 + lane;
#pragma unroll
                for (int q = 0; q < 11; ++q) {
                    const unsigned u = row[q * 32];
                    cs[q].x = fmaf(wy[k], __uint_as_float(u << 16), cs[q].x);
                    cs[q].y = fmaf(wy[k], __uint_as_float(u & 0xffff0000u), cs[q].y);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[j0 % kFirRing]);       // the oldest row of the window is done
            float nzv[8];
            unsigned svv[8];
            if (FWD && P.act_saved) {
                const unsigned* sp = reinterpret_cast<const unsigned*>(P.act_saved) +
                                     ((static_cast<long long>(n) * P.OH + r) * P.OW) * (P.C >> 1) + (c0 >> 1) + lane;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int x = x0 + px0 + i;
                    svv[i] = x < P.OW ? __ldg(sp + static_cast<long long>(x) * (P.C >> 1)) : 0u;
                }
            }
            if (FWD && P.noise && !P.act_saved) {
                const float4* np = reinterpret_cast<const float4*>(P.noise + n * P.noise_stride_n + static_cast<long long>(r) * P.OW + x0 + px0);
                const bool in = x0 + px0 + 8 <= P.OW;
                const float4 a = in ? __ldg(np) : make_float4(0.f, 0.f, 0.f, 0.f), b = in ? __ldg(np + 1) : a;
                nzv[0] = a.x; nzv[1] = a.y; nzv[2] = a.z; nzv[3] = a.w; nzv[4] = b.x; nzv[5] = b.y; nzv[6] = b.z; nzv[7] = b.w;
#pragma unroll
                for (int i = 0; i < 8; ++i) nzv[i] *= P.noise_scale;
            } else {
#pragma unroll
                for (int i = 0; i < 8; ++i) nzv[i] = 0.f;
            }
            uint8_t* sx = my_stage + (j0 & 1) * 2048;                // [x | xs] x 1 KB, double-buffered by row parity
            if (lane == 0) bulk_wait_read<1>();                       // the stores of two rows ago have read this buffer
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                float a0 = 0.f, a1 = 0.f;
#pragma unroll
                for (int k = 0; k < 4; ++k) { a0 = fmaf(wx[k], cs[i + k].x, a0); a1 = fmaf(wx[k], cs[i + k].y, a1); }
                if (FWD && P.act_saved) {
                    const float s0 = __uint_as_float(svv[i] << 16), s1 = __uint_as_float(svv[i] & 0xffff0000u);
                    const float g0 = act_grad(a0 * P.act_gain, s0, P.act_slope, saved_thr);
                    const float g1 = act_grad(a1 * P.act_gain, s1, P.act_slope, saved_thr);
                    reinterpret_cast<unsigned*>(sx)[i * 32 + lane] = pack2(g0, g1);
                } else if (FWD) {
                    float z0 = fmaf(a0, dm.x, nzv[i]) + bs.x, z1 = fmaf(a1, dm.y, nzv[i]) + bs.y;
                    z0 = (z0 > 0.f ? z0 : z0 * P.act_slope) * P.act_gain;
                    z1 = (z1 > 0.f ? z1 : z1 * P.act_slope) * P.act_gain;
                    z0 = fminf(fmaxf(z0, -clampv), clampv);
                    z1 = fminf(fmaxf(z1, -clampv), clampv);
                    reinterpret_cast<unsigned*>(sx)[i * 32 + lane] = pack2(z0, z1);
                    reinterpret_cast<unsigned*>(sx + 1024)[i * 32 + lane] = pack2(z0 * sn.x, z1 * sn.y);
                } else {
                    reinterpret_cast<unsigned*>(sx)[i * 32 + lane] = pack2(a0, a1);
                }
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
                if (FWD) {
                    tma_store_4d(&P.fwd_out_x, sx, c0, x0 + px0, r, n);
                    if (P.s_next && !P.act_saved) tma_store_4d(&P.fwd_out_xs, sx + 1024, c0, x0 + px0, r, n);
                } else {
                    tma_store_4d(&P.bwd_out, sx, c0, x0 + px0, r, n);
                }
                bulk_commit();
            }
        }
        // the last three window rows were never released: nobody waits for them
    }
    if (lane == 0) bulk_wait_read<0>();
}

// ------------------------------------------------------------------------- toRGB + skip pyramid
// upsample2d (upfirdn2d.py:313-348: zero-insert x2, pad [2,1,2,1], 4x4 FIR, gain 4) of the
// default [1,3,3,1] filter is the separable 2-tap interpolation out[2m] = (x[m-1]+3x[m])/4,
// out[2m+1] = (3x[m]+x[m+1])/4 with zero padding.
__device__ __forceinline__ void up_taps(int v, int lowres, int& i0, int& i1, float& c0, float& c1) {
    const int m = v >> 1;
    if (v & 1) { i0 = m; i1 = m + 1; c0 = 0.75f; c1 = 0.25f; }
    else { i0 = m - 1; i1 = m; c0 = 0.25f; c1 = 0.75f; }
    if (i0 < 0) { c0 = 0.f; i0 = 0; }
    if (i1 >= lowres) { c1 = 0.f; i1 = lowres - 1; }
}

__device__ __forceinline__ float4 f4_fma(float c, float4 a, float4 acc) {
    return make_float4(fmaf(c, a.x, acc.x), fmaf(c, a.y, acc.y), fmaf(c, a.z, acc.z), fmaf(c, a.w, acc.w));
}

__device__ __forceinline__ float4 rgb_preclamp(const float4* __restrict__ parts, int nparts, long long stride, long long pix,
                                               const float* __restrict__ bias, int img_c) {
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int b = 0; b < nparts; ++b) {
        const float4 p = parts[b * stride + pix];
        t.x += p.x; t.y += p.y; t.z += p.z;
    }
    t.x += bias[0];
    if (img_c > 1) t.y += bias[1];
    if (img_c > 2) t.z += bias[2];
    return t;
}

__global__ void rgb_combine_kernel(const float4* __restrict__ parts, int nparts, const float* __restrict__ bias, int img_c,
                                   float clamp, const float4* __restrict__ img_low, int batch, int res, float4* img,
                                   float* out_nchw) {
    const long long pix = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    const long long total = static_cast<long long>(batch) * res * res;
    if (pix >= total) return;
    float4 t = rgb_preclamp(parts, nparts, total, pix, bias, img_c);
    if (clamp >= 0.f) {
        t.x = fminf(fmaxf(t.x, -clamp), clamp);
        t.y = fminf(fmaxf(t.y, -clamp), clamp);
        t.z = fminf(fmaxf(t.z, -clamp), clamp);
    }
    const int w = static_cast<int>(pix % res), h = static_cast<int>((pix / res) % res);
    const int n = static_cast<int>(pix / (static_cast<long long>(res) * res));
    if (img_low) {
        const int lr = res >> 1;
        int y0, y1, x0, x1;
        float cy0, cy1, cx0, cx1;
        up_taps(h, lr, y0, y1, cy0, cy1);
        up_taps(w, lr, x0, x1, cx0, cx1);
        const float4* base = img_low + static_cast<long long>(n) * lr * lr;
        float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
        // same association as the reference's depthwise conv is not reproducible bit-for-bit
        // (it sums 16 taps, 12 of them zeros); fp32 2x2 accumulation here.
        u = f4_fma(cy0 * cx0, base[y0 * lr + x0], u);
        u = f4_fma(cy0 * cx1, base[y0 * lr + x1], u);
        u = f4_fma(cy1 * cx0, base[y1 * lr + x0], u);
        u = f4_fma(cy1 * cx1, base[y1 * lr + x1], u);
        t.x += u.x; t.y += u.y; t.z += u.z;
    }
    img[pix] = t;
    if (out_nchw) {
        const long long plane = static_cast<long long>(res) * res;
        float* o = out_nchw + static_cast<long long>(n) * img_c * plane + static_cast<long long>(h) * res + w;
        o[0] = t.x;
        if (img_c > 1) o[plane] = t.y;
        if (img_c > 2) o[2 * plane] = t.z;
    }
}

// g_rgb = g_img * [|pre-clamp| < clamp]; g_img_low = upsample2d^T(g_img).
__global__ void rgb_backward_kernel(const float4* __restrict__ g_img, const float4* __restrict__ parts, int nparts,
                                    const float* __restrict__ bias, int img_c, float clamp, int batch, int res, float4* g_rgb,
                                    float4* g_img_low) {
    const long long pix = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    const long long total = static_cast<long long>(batch) * res * res;
    if (pix >= total) return;
    const float4 g = g_img[pix];
    const float4 t = rgb_preclamp(parts, nparts, total, pix, bias, img_c);
    float4 r = g;
    if (clamp >= 0.f) {
        if (!(fabsf(t.x) <= clamp)) r.x = 0.f;     // torch.clamp passes the gradient on the closed interval
        if (!(fabsf(t.y) <= clamp)) r.y = 0.f;
        if (!(fabsf(t.z) <= clamp)) r.z = 0.f;
    }
    r.w = 0.f;
    g_rgb[pix] = r;
    if (g_img_low) {
        const int w = static_cast<int>(pix % res), h = static_cast<int>((pix / res) % res);
        if ((w | h) & 1) return;
        const int n = static_cast<int>(pix / (static_cast<long long>(res) * res));
        const int my = h >> 1, mx = w >> 1, lr = res >> 1;
        // low-res pixel m feeds out[2m-1] (1/4), out[2m] (3/4), out[2m+1] (3/4), out[2m+2] (1/4)
        const float cf[4] = {0.25f, 0.75f, 0.75f, 0.25f};
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        const float4* base = g_img + static_cast<long long>(n) * res * res;
        for (int a = 0; a < 4; ++a) {
            const int yy = 2 * my - 1 + a;
            if (yy < 0 || yy >= res) continue;
            for (int b = 0; b < 4; ++b) {
                const int xx = 2 * mx - 1 + b;
                if (xx < 0 || xx >= res) continue;
                acc = f4_fma(cf[a] * cf[b], base[static_cast<long long>(yy) * res + xx], acc);
            }
        }
        g_img_low[(static_cast<long long>(n) * lr + my) * lr + mx] = acc;
    }
}

// ------------------------------------------------------------------------- pixel criterion
// Reference calc_loss_pix (util_latent_aug.py:373-385) = per-modality mean over all
// (sample, bank image) pairs of the squared L2 between centre crops, / (h*w), * w_pix,
// averaged over modalities.  The pair mean only needs the bank mean image and the mean bank
// energy (SURVEY.md App. B):  mean_ij |x_i - y_j|^2 = mean_i |x_i|^2 - 2 <mean_i x_i, ybar> + mean_j |y_j|^2.
// Gradient (loss enters the objective with a minus sign, :270):
//   g_img = -(w_pix/C) * 2/(n*h*w) * (x - ybar) inside the crop, 0 outside.
__global__ void pix_loss_kernel(const float4* __restrict__ img, const float4* __restrict__ bank_mean, int batch, int res,
                                int img_c, int crop_off, int crop_size, float w_pix, float4* g_img, float* loss_parts) {
    const long long total = static_cast<long long>(batch) * res * res;
    const float gs = -(w_pix / img_c) * 2.f / (static_cast<float>(batch) * crop_size * crop_size);
    float acc = 0.f;
    for (long long pix = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; pix < total;
         pix += static_cast<long long>(gridDim.x) * blockDim.x) {
        const int w = static_cast<int>(pix % res), h = static_cast<int>((pix / res) % res);
        float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
        if (h >= crop_off && h < crop_off + crop_size && w >= crop_off && w < crop_off + crop_size) {
            const float4 x = img[pix];
            const float4 y = bank_mean[h * res + w];
            g.x = gs * (x.x - y.x);
            acc += x.x * x.x - 2.f * x.x * y.x;
            if (img_c > 1) { g.y = gs * (x.y - y.y); acc += x.y * x.y - 2.f * x.y * y.y; }
            if (img_c > 2) { g.z = gs * (x.z - y.z); acc += x.z * x.z - 2.f * x.z * y.z; }
        }
        g_img[pix] = g;
    }
    __shared__ float sm[32];
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        float v = threadIdx.x < (blockDim.x >> 5) ? sm[threadIdx.x] : 0.f;
        v = warp_sum(v);
        if (threadIdx.x == 0) loss_parts[blockIdx.x] = v;
    }
}

// ------------------------------------------------------------------------- style gradients
// conv layer:  g_s[n,i] = red_s[n,i] - s[n,i] * sum_o red_d[n,o] * d[n,o]^2 * W2[o,i]      (SURVEY.md App. A.4): style_gemm_kernel<kSgGrad>
// toRGB layer:  g_s[n,i] = sum_c W_rgb[c,i] * red_rgb[c][n,i]
__global__ void style_grad_rgb_kernel(LayerTable T, int batch, const float* __restrict__ red_rgb, float* g_s) {
    const RgbDesc D = T.rgb[blockIdx.y];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = blockIdx.z;
    if (i >= D.cin) return;
    const float* rr = red_rgb + 3LL * batch * D.roff;
    const long long e = static_cast<long long>(n) * D.cin + i;
    const long long plane = static_cast<long long>(batch) * D.cin;
    float g = D.wt[i] * rr[e];
    if (D.img_c > 1) g += D.wt[D.cin + i] * rr[plane + e];
    if (D.img_c > 2) g += D.wt[2 * D.cin + i] * rr[2 * plane + e];
    g_s[static_cast<long long>(batch) * D.soff + e] = g;
}

// partial[c][n][k] = sum_{r in 64-row chunk c} g_s[n, r] * A_cat[r, k]   (deterministic two-stage reduction)
constexpr int kGwRows = 64, kGwSamples = 4;
__global__ void gw_partial_kernel(const float* __restrict__ g_s, const float* __restrict__ a_cat, const int* __restrict__ chunk_soff,
                                  const int* __restrict__ chunk_cin, int batch, int w_dim, float* partial) {
    const int c = blockIdx.x;
    const int n0 = blockIdx.y * kGwSamples;
    const int soff = chunk_soff[c], cin = chunk_cin[c];
    const int row0 = c * kGwRows;                // global affine row of this chunk
    __shared__ float sg[kGwSamples][kGwRows];
    for (int e = threadIdx.x; e < kGwSamples * kGwRows; e += blockDim.x) {
        const int j = e / kGwRows, r = e % kGwRows;
        const int n = n0 + j;
        sg[j][r] = n < batch ? g_s[static_cast<long long>(batch) * soff + static_cast<long long>(n) * cin + (row0 - soff) + r] : 0.f;
    }
    __syncthreads();
    for (int k = threadIdx.x; k < w_dim; k += blockDim.x) {
        float acc[kGwSamples] = {0.f, 0.f, 0.f, 0.f};
        for (int r = 0; r < kGwRows; ++r) {
            const float a = a_cat[static_cast<long long>(row0 + r) * w_dim + k];
#pragma unroll
            for (int j = 0; j < kGwSamples; ++j) acc[j] = fmaf(sg[j][r], a, acc[j]);
        }
#pragma unroll
        for (int j = 0; j < kGwSamples; ++j)
            if (n0 + j < batch) partial[(static_cast<long long>(c) * batch + n0 + j) * w_dim + k] = acc[j];
    }
}

// ------------------------------------------------------------------------- loss values + Adam
// Loss values (logging only; reference util_latent_aug.py:233-271).  One block.
__global__ void loss_value_kernel(const float* __restrict__ w, const float* __restrict__ w_sum_bank, const float* __restrict__ lat_m2, const AdamConsts* C,
                                  const int* step_counter, int batch, int w_dim, const float* __restrict__ pix_parts,
                                  int n_pix_parts, const float* __restrict__ bank_m2, int img_c, int crop_size, float* loss_log,
                                  int max_steps, const float* __restrict__ disc_loss, const float* __restrict__ lpips_loss) {
    double sq = 0.0, dot = 0.0, px = 0.0;
    for (int e = threadIdx.x; e < batch * w_dim; e += blockDim.x) {
        const double v = w[e];
        sq += v * v;
        if (C->has_bank) dot += v * w_sum_bank[e % w_dim];
    }
    for (int e = threadIdx.x; e < n_pix_parts; e += blockDim.x) px += pix_parts[e];
    __shared__ double sm[3][32];
    sq = warp_sum_d(sq); dot = warp_sum_d(dot); px = warp_sum_d(px);
    if ((threadIdx.x & 31) == 0) { sm[0][threadIdx.x >> 5] = sq; sm[1][threadIdx.x >> 5] = dot; sm[2][threadIdx.x >> 5] = px; }
    __syncthreads();
    if (threadIdx.x == 0) {
        sq = dot = px = 0.0;
        for (int i = 0; i < (blockDim.x >> 5); ++i) { sq += sm[0][i]; dot += sm[1][i]; px += sm[2][i]; }
        const int t = *step_counter;
        if (t < max_steps) {
            double l_lat = 0.0, l_pix = 0.0;
            if (C->w_latent > 0.f && C->has_bank)
                l_lat = C->w_latent * ((C->num_ws * sq - 2.0 * dot) / batch + lat_m2[0]) / (static_cast<double>(C->num_ws) * w_dim);
            if (C->w_pix > 0.f) {
                double m2 = 0.0;
                for (int c = 0; c < img_c && c < 3; ++c) m2 += bank_m2[c];
                const double hw = static_cast<double>(crop_size) * crop_size;
                l_pix = C->w_pix * (px / (batch * hw) + m2 / hw) / img_c;
            }
            loss_log[kLossCols * t + 0] = static_cast<float>(l_lat);
            loss_log[kLossCols * t + 1] = static_cast<float>(l_pix);
            const double l_disc = disc_loss ? disc_loss[0] : 0.0;
            const double l_lpips = lpips_loss ? lpips_loss[0] : 0.0;
            loss_log[kLossCols * t + 2] = static_cast<float>(-l_lat - l_pix - l_lpips + l_disc);      // util_latent_aug.py:270
            loss_log[kLossCols * t + 3] = static_cast<float>(l_disc);
            loss_log[kLossCols * t + 4] = static_cast<float>(l_lpips);
        }
    }
}

// torch.optim.Adam semantics (betas, eps, no weight decay / amsgrad), state restarts per call
// (util_latent_aug.py:213).  Gradient = sum of the style-path partials (pixel criterion through
// the generator) + the latent criterion's closed form  -w_latent * 2/(n*w_dim*num_ws) * (num_ws*w - sum_j Wbar_j).
__global__ void adam_kernel(const float* __restrict__ partial, int nchunks, int use_partial, const float* __restrict__ w_sum_bank,
                            const AdamConsts* C, const int* step_counter, float* w, float* m, float* v, int batch, int w_dim) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= batch * w_dim) return;
    float g = 0.f;
    if (use_partial)
        for (int c = 0; c < nchunks; ++c) g += partial[static_cast<long long>(c) * batch * w_dim + e];
    const float wv = w[e];
    if (C->w_latent > 0.f && C->has_bank)
        g -= C->w_latent * 2.f / (static_cast<float>(batch) * C->num_ws * w_dim) * (C->num_ws * wv - w_sum_bank[e % w_dim]);
    const int t = *step_counter + 1;
    const float mm = C->beta1 * m[e] + (1.f - C->beta1) * g;
    const float vv = C->beta2 * v[e] + (1.f - C->beta2) * g * g;
    m[e] = mm;
    v[e] = vv;
    const float bc1 = 1.f - powf(C->beta1, static_cast<float>(t));
    const float bc2 = 1.f - powf(C->beta2, static_cast<float>(t));
    const float step_size = C->lr / bc1;
    const float denom = sqrtf(vv) / sqrtf(bc2) + C->eps;
    w[e] = wv - step_size * (mm / denom);
}
__global__ void step_inc_kernel(int* step_counter) { *step_counter += 1; }

// projection: the same update with the learning rate of step t from the schedule table (projector.py::project)
__global__ void adam_sched_kernel(const float* __restrict__ partial, int nchunks, const ProjConsts* pc, const int* step_counter, float* w, float* m,
                                  float* v, float* w_pert, int batch, int w_dim) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = batch * w_dim;
    if (e >= n) return;
    float g = 0.f;
    for (int c = 0; c < nchunks; ++c) g += partial[static_cast<long long>(c) * n + e];
    const int t = *step_counter;
    const float b1 = 0.9f, b2 = 0.999f;
    const float mm = b1 * m[e] + (1.f - b1) * g;
    const float vv = b2 * v[e] + (1.f - b2) * g * g;
    m[e] = mm;
    v[e] = vv;
    const float bc1 = 1.f - powf(b1, static_cast<float>(t + 1));
    const float bc2 = 1.f - powf(b2, static_cast<float>(t + 1));
    const float denom = sqrtf(vv) / sqrtf(bc2) + 1e-8f;
    const float wn = w[e] - (pc->lr[t] / bc1) * (mm / denom);
    w[e] = wn;
    const int next = t + 1;
    w_pert[e] = (pc->noise && next < pc->num_steps) ? fmaf(pc->sigma[next], pc->noise[static_cast<long long>(next) * n + e], wn) : wn;
}
__global__ void perturb_first_kernel(const float* __restrict__ w, const ProjConsts* pc, float* w_pert, int n) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    w_pert[e] = (pc->noise && pc->num_steps > 0) ? fmaf(pc->sigma[0], pc->noise[e], w[e]) : w[e];
}
__global__ void sum_floats_kernel(const float* __restrict__ x, int n, float* out) {
    double acc = 0.0;
    for (int i = threadIdx.x; i < n; i += 32) acc += x[i];
    acc = warp_sum_d(acc);
    if (threadIdx.x == 0) out[0] = static_cast<float>(acc);
}

__global__ void finalize_w_kernel(const float* __restrict__ w_opt, const float* __restrict__ w0, float alpha, int soft, int n,
                                  float* w_aug) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    w_aug[e] = soft ? alpha * w_opt[e] + (1.f - alpha) * w0[e] : w_opt[e];
}

// ------------------------------------------------------------------------- bank statistics
constexpr int kBankBlocks = 256;
__global__ void latent_bank_partial_kernel(const float* __restrict__ W, int M, int num_ws, int w_dim, double* psum, double* pm2) {
    const int m0 = static_cast<int>(static_cast<long long>(blockIdx.x) * M / gridDim.x);
    const int m1 = static_cast<int>(static_cast<long long>(blockIdx.x + 1) * M / gridDim.x);
    double sq = 0.0;
    for (int k = threadIdx.x; k < w_dim; k += blockDim.x) {
        double acc = 0.0;
        for (int m = m0; m < m1; ++m)
            for (int j = 0; j < num_ws; ++j) {
                const double v = W[(static_cast<long long>(m) * num_ws + j) * w_dim + k];
                acc += v;
                sq += v * v;
            }
        psum[static_cast<long long>(blockIdx.x) * w_dim + k] = acc;
    }
    __shared__ double sm[32];
    sq = warp_sum_d(sq);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = sq;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < (blockDim.x >> 5); ++i) t += sm[i];
        pm2[blockIdx.x] = t;
    }
}
__global__ void latent_bank_final_kernel(const double* __restrict__ psum, const double* __restrict__ pm2, int nblocks, int M,
                                         int w_dim, float* w_sum, float* m2) {
    for (int k = threadIdx.x; k < w_dim; k += blockDim.x) {
        double acc = 0.0;
        for (int b = 0; b < nblocks; ++b) acc += psum[static_cast<long long>(b) * w_dim + k];
        w_sum[k] = static_cast<float>(acc / M);
    }
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int b = 0; b < nblocks; ++b) t += pm2[b];
        m2[0] = static_cast<float>(t / M);
    }
}

__global__ void image_bank_mean_kernel(const float* __restrict__ X, int M, int C, int res, float4* mean) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= res * res) return;
    float acc[3] = {0.f, 0.f, 0.f};
    const long long plane = static_cast<long long>(res) * res;
    for (int m = 0; m < M; ++m)
        for (int c = 0; c < C && c < 3; ++c) acc[c] += X[(static_cast<long long>(m) * C + c) * plane + p];
    mean[p] = make_float4(acc[0] / M, acc[1] / M, acc[2] / M, 0.f);
}
// one block per channel: mean_j sum_{p in crop} Y_j,c[p]^2
__global__ void image_bank_m2_kernel(const float* __restrict__ X, int M, int C, int res, int crop_off, int crop_size, float* m2) {
    const int c = blockIdx.x;
    const long long plane = static_cast<long long>(res) * res;
    const long long per = static_cast<long long>(crop_size) * crop_size;
    double acc = 0.0;
    for (long long e = threadIdx.x; e < per * M; e += blockDim.x) {
        const int m = static_cast<int>(e / per);
        const int q = static_cast<int>(e % per);
        const int h = crop_off + q / crop_size, w = crop_off + q % crop_size;
        const double v = X[(static_cast<long long>(m) * C + c) * plane + static_cast<long long>(h) * res + w];
        acc += v * v;
    }
    __shared__ double sm[32];
    acc = warp_sum_d(acc);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < (blockDim.x >> 5); ++i) t += sm[i];
        m2[c] = static_cast<float>(t / M);
    }
}

// ------------------------------------------------------------------------- mapping network
__global__ void mapping_normalize_kernel(const float* __restrict__ z, int z_dim, float* out) {
    const int n = blockIdx.x;
    float acc = 0.f;
    for (int k = threadIdx.x; k < z_dim; k += blockDim.x) { const float v = z[static_cast<long long>(n) * z_dim + k]; acc += v * v; }
    __shared__ float sm[32];
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = acc;
    __syncthreads();
    float t = 0.f;
    for (int i = 0; i < (blockDim.x >> 5); ++i) t += sm[i];
    const float r = rsqrtf(t / z_dim + 1e-8f);
    for (int k = threadIdx.x; k < z_dim; k += blockDim.x) out[static_cast<long long>(n) * z_dim + k] = z[static_cast<long long>(n) * z_dim + k] * r;
}

__global__ void mapping_fc_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ b, int batch,
                                  int n_in, int n_out, float w_gain, float b_gain, int lrelu, float* y) {
    const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (j >= n_out) return;
    float a[kMaxRowRegs];
#pragma unroll
    for (int r = 0; r < kMaxRowRegs; ++r) a[r] = (lane + 32 * r < n_in) ? w[static_cast<long long>(j) * n_in + lane + 32 * r] * w_gain : 0.f;
    const float bj = b[j] * b_gain;
    for (int n = 0; n < batch; ++n) {
        float acc = 0.f;
#pragma unroll
        for (int r = 0; r < kMaxRowRegs; ++r)
            if (lane + 32 * r < n_in) acc = fmaf(a[r], x[static_cast<long long>(n) * n_in + lane + 32 * r], acc);
        acc = warp_sum(acc);
        if (lane == 0) {
            float v = acc + bj;
            if (lrelu) v = (v > 0.f ? v : 0.2f * v) * 1.41421356237309515f;
            y[static_cast<long long>(n) * n_out + j] = v;
        }
    }
}

__global__ void mapping_truncate_kernel(const float* __restrict__ w, const float* __restrict__ w_avg, float psi, int n, int w_dim,
                                        float* out) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const float a = w_avg[e % w_dim];
    out[e] = a + psi * (w[e] - a);          // w_avg.lerp(w, psi)
}

}  // namespace

// ===================================================================================== launchers
int prep_conv_weights(const float* w, int cout, int cin, int up, const float* fir4x4, int split, void* wf, void* wb, float* w2,
                      float* w2t, cudaStream_t s) {
    const long long n = static_cast<long long>(cout) * cin;
    prep_conv_weights_kernel<<<cdiv(n, 128), 128, 0, s>>>(w, cout, cin, up, fir4x4, split, static_cast<__nv_bfloat16*>(wf),
                                                          static_cast<__nv_bfloat16*>(wb), w2, w2t);
    return last_err();
}
int prep_affine(const float* aw, const float* ab, int cin, int w_dim, float wscale, float bscale, float* a_rows, float* b_rows,
                cudaStream_t s) {
    prep_affine_kernel<<<cdiv(static_cast<long long>(cin) * w_dim, 256), 256, 0, s>>>(aw, ab, cin, w_dim, wscale, bscale, a_rows, b_rows);
    return last_err();
}
__global__ void prep_axpy_kernel(const float* __restrict__ x, float a, float* y, long long n) {
    const long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (i < n) y[i] = fmaf(a, x[i], y[i]);
}
int prep_axpy(const float* x, float a, float* y, long long n, cudaStream_t s) {
    prep_axpy_kernel<<<cdiv(n, 256), 256, 0, s>>>(x, a, y, n);
    return last_err();
}
int prep_scale(const float* src, float scale, float* dst, long long n, cudaStream_t s) {
    prep_scale_kernel<<<cdiv(n, 256), 256, 0, s>>>(src, scale, dst, n);
    return last_err();
}
int prep_const(const float* cst, int C, int hw, float* c_f32, void* hi, void* lo, cudaStream_t s) {
    prep_const_kernel<<<cdiv(C * hw, 256), 256, 0, s>>>(cst, C, hw, c_f32, static_cast<__nv_bfloat16*>(hi), static_cast<__nv_bfloat16*>(lo));
    return last_err();
}

static int max_cin(const LayerTable& T, bool conv, bool rgb) {
    int m = 0;
    if (conv) for (int i = 0; i < T.nconv; ++i) m = T.conv[i].cin > m ? T.conv[i].cin : m;
    if (rgb) for (int i = 0; i < T.nrgb; ++i) m = T.rgb[i].cin > m ? T.rgb[i].cin : m;
    return m;
}

static int upfir_launch(const UpFirParams& p, bool fwd, cudaStream_t s) {
    if (p.use_tma) {
        const int smem = kFirRing * kFirSlotBytes + 4 * 2 * 2 * 1024 + 2 * kFirRing * 8;
        const int out_h = fwd ? p.OH : p.TH, out_w = fwd ? p.OW : p.OW + 1;
        const int nslabs = p.C / 64;
        const int strips = cdiv(out_w, kFirStrip);
        // enough CTAs for ~4 per SM, but runs of at least 32 rows (3 halo rows are re-read per run)
        int rblocks = 1;
        while (static_cast<long long>(strips) * nslabs * p.B * rblocks < 148 * 6 && out_h / (rblocks * 2) >= 32) rblocks *= 2;
        const int rows_per_cta = cdiv(out_h, rblocks);
        dim3 grid(strips, nslabs * cdiv(out_h, rows_per_cta), p.B);
        if (fwd) {
            static bool a[kMaxDevices] = {};
            const int dev = current_device_slot();
            if (!a[dev]) { cudaFuncSetAttribute(upfir_tma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); a[dev] = true; }
            upfir_tma_kernel<true><<<grid, 160, smem, s>>>(p, rows_per_cta, nslabs);
        } else {
            static bool a[kMaxDevices] = {};
            const int dev = current_device_slot();
            if (!a[dev]) { cudaFuncSetAttribute(upfir_tma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem); a[dev] = true; }
            upfir_tma_kernel<false><<<grid, 160, smem, s>>>(p, rows_per_cta, nslabs);
        }
        return last_err();
    }
    const int hc = p.C / 2;
    int cpb = hc < 256 ? hc : 256;
    if (256 % cpb || hc % cpb) return static_cast<int>(cudaErrorInvalidValue);   // channel counts are 64 * 2^k
    const int chan_blocks = hc / cpb, rows_per_block = 256 / cpb;
    const int out_h = fwd ? p.OH : p.TH, out_w = fwd ? p.OW : p.OW + 1;
    dim3 grid(cdiv(out_w, kFirSeg), cdiv(out_h, rows_per_block), p.B * chan_blocks);
#define LA_FIR(F, S, Q) upfir_slide_kernel<F, S, Q><<<grid, 256, 0, s>>>(p, cpb, chan_blocks)
    const int sel = (fwd ? 4 : 0) | (p.split ? 2 : 0) | (p.separable ? 1 : 0);
    switch (sel) {
        case 0: LA_FIR(false, false, false); break;
        case 1: LA_FIR(false, false, true); break;
        case 2: LA_FIR(false, true, false); break;
        case 3: LA_FIR(false, true, true); break;
        case 4: LA_FIR(true, false, false); break;
        case 5: LA_FIR(true, false, true); break;
        case 6: LA_FIR(true, true, false); break;
        default: LA_FIR(true, true, true); break;
    }
#undef LA_FIR
    return last_err();
}
int upfir_forward(const UpFirParams& p, cudaStream_t s) { return upfir_launch(p, true, s); }
int upfir_backward(const UpFirParams& p, cudaStream_t s) { return upfir_launch(p, false, s); }

int styles_forward(const LayerTable& T, const float* ws, long long sn, long long sidx, const float* a_cat, const float* b_cat,
                   int w_dim, int batch, float* s_cat, cudaStream_t s) {
    StyleGemmArgs A{};
    A.ws = ws; A.sn = sn; A.sidx = sidx; A.a_cat = a_cat; A.b_cat = b_cat; A.w_dim = w_dim; A.out = s_cat;
    dim3 grid(cdiv(max_cin(T, true, true), kSgRows), T.nconv + T.nrgb, cdiv(batch, kSgSamples));
    style_gemm_kernel<kSgStyles><<<grid, 128, 0, s>>>(T, batch, A);
    return last_err();
}
int demod_rgbw_forward(const LayerTable& T, int batch, const float* s_cat, float* d_cat, float4* rgbw, cudaStream_t s) {
    int mco = 0;
    for (int i = 0; i < T.nconv; ++i) mco = T.conv[i].cout > mco ? T.conv[i].cout : mco;
    StyleGemmArgs A{};
    A.s_cat = s_cat; A.out = d_cat;
    style_gemm_kernel<kSgDemod><<<dim3(cdiv(mco, kSgRows), T.nconv, cdiv(batch, kSgSamples)), 128, 0, s>>>(T, batch, A);
    int e = last_err();
    if (e) return e;
    rgbw_kernel<<<dim3(cdiv(max_cin(T, false, true), 128), T.nrgb, batch), 128, 0, s>>>(T, batch, s_cat, rgbw);
    return last_err();
}
int const_modulate(const float* c_f32, const float* s0, int batch, int hw, int C, int split, void* xs_hi, void* xs_lo, cudaStream_t s) {
    const long long n = static_cast<long long>(batch) * hw * C;
    const_modulate_kernel<<<cdiv(n, 256), 256, 0, s>>>(c_f32, s0, batch, hw, C, static_cast<__nv_bfloat16*>(xs_hi),
                                                        split ? static_cast<__nv_bfloat16*>(xs_lo) : nullptr);
    return last_err();
}
int rgb_combine(const float4* parts, int nparts, const float* bias, int img_c, float clamp, const float4* img_low, int batch, int res,
                float4* img, float* out_nchw, cudaStream_t s) {
    const long long n = static_cast<long long>(batch) * res * res;
    rgb_combine_kernel<<<cdiv(n, 256), 256, 0, s>>>(parts, nparts, bias, img_c, clamp, img_low, batch, res, img, out_nchw);
    return last_err();
}
int rgb_backward(const float4* g_img, const float4* parts, int nparts, const float* bias, int img_c, float clamp, int batch, int res,
                 float4* g_rgb, float4* g_img_low, cudaStream_t s) {
    const long long n = static_cast<long long>(batch) * res * res;
    rgb_backward_kernel<<<cdiv(n, 256), 256, 0, s>>>(g_img, parts, nparts, bias, img_c, clamp, batch, res, g_rgb, g_img_low);
    return last_err();
}
int pix_loss(const float4* img, const float4* bank_mean, const float* /*bank_m2*/, int batch, int res, int img_c, int crop_off,
             int crop_size, float w_pix, float4* g_img, float* loss_parts, int* nparts_out, cudaStream_t s) {
    const long long n = static_cast<long long>(batch) * res * res;
    int grid = cdiv(n, 256);
    if (grid > 1024) grid = 1024;
    pix_loss_kernel<<<grid, 256, 0, s>>>(img, bank_mean, batch, res, img_c, crop_off, crop_size, w_pix, g_img, loss_parts);
    *nparts_out = grid;
    return last_err();
}
int style_grad(const LayerTable& T, int batch, const float* s_cat, const float* d_cat, const float* red_s, const float* red_d,
               const float* red_rgb, float* g_s, cudaStream_t s) {
    int mco = 0;
    for (int i = 0; i < T.nconv; ++i) mco = T.conv[i].cout > mco ? T.conv[i].cout : mco;
    (void)mco;
    StyleGemmArgs A{};
    A.s_cat = s_cat; A.d_cat = d_cat; A.red_s = red_s; A.red_d = red_d; A.out = g_s;
    style_gemm_kernel<kSgGrad><<<dim3(cdiv(max_cin(T, true, false), kSgRows), T.nconv, cdiv(batch, kSgSamples)), 128, 0, s>>>(T, batch, A);
    int e = last_err();
    if (e) return e;
    style_grad_rgb_kernel<<<dim3(cdiv(max_cin(T, false, true), 128), T.nrgb, batch), 128, 0, s>>>(T, batch, red_rgb, g_s);
    return last_err();
}
int gw_partial(const float* g_s, const float* a_cat, const int* chunk_soff, const int* chunk_cin, int nchunks, int batch, int w_dim,
               float* partial, cudaStream_t s) {
    gw_partial_kernel<<<dim3(nchunks, cdiv(batch, kGwSamples)), 256, 0, s>>>(g_s, a_cat, chunk_soff, chunk_cin, batch, w_dim, partial);
    return last_err();
}
int adam_step(const float* partial, int nchunks, int use_partial, const float* w_sum_bank, const float* lat_m2, const AdamConsts* consts, int* step_counter,
              float* w, float* m, float* v, int batch, int w_dim, const float* pix_parts, int n_pix_parts, const float* bank_m2,
              int img_c, int crop_size, float* loss_log, int max_steps, const float* disc_loss, const float* lpips_loss, cudaStream_t s) {
    loss_value_kernel<<<1, 512, 0, s>>>(w, w_sum_bank, lat_m2, consts, step_counter, batch, w_dim, pix_parts, n_pix_parts, bank_m2, img_c,
                                        crop_size, loss_log, max_steps, disc_loss, lpips_loss);
    adam_kernel<<<cdiv(batch * w_dim, 256), 256, 0, s>>>(partial, nchunks, use_partial, w_sum_bank, consts, step_counter, w, m, v, batch, w_dim);
    step_inc_kernel<<<1, 1, 0, s>>>(step_counter);
    return last_err();
}
int adam_scheduled(const float* partial, int nchunks, const ProjConsts* pc, int* step_counter, float* w, float* m, float* v,
                   float* w_pert, int batch, int w_dim, cudaStream_t s) {
    adam_sched_kernel<<<cdiv(batch * w_dim, 256), 256, 0, s>>>(partial, nchunks, pc, step_counter, w, m, v, w_pert, batch, w_dim);
    step_inc_kernel<<<1, 1, 0, s>>>(step_counter);
    return last_err();
}
int perturb_first(const float* w, const ProjConsts* pc, float* w_pert, int batch, int w_dim, cudaStream_t s) {
    perturb_first_kernel<<<cdiv(batch * w_dim, 256), 256, 0, s>>>(w, pc, w_pert, batch * w_dim);
    return last_err();
}
int sum_floats(const float* x, int n, float* out, cudaStream_t s) {
    sum_floats_kernel<<<1, 32, 0, s>>>(x, n, out);
    return last_err();
}
int finalize_w(const float* w_opt, const float* w0, float alpha, int soft, int batch, int w_dim, float* w_aug, cudaStream_t s) {
    finalize_w_kernel<<<cdiv(batch * w_dim, 256), 256, 0, s>>>(w_opt, w0, alpha, soft, batch * w_dim, w_aug);
    return last_err();
}

int latent_bank_stats(const float* W, int M, int num_ws, int w_dim, float* w_sum, float* m2, cudaStream_t s) {
    double* scratch = nullptr;
    const int nb = M < kBankBlocks ? M : kBankBlocks;
    cudaError_t e = cudaMallocAsync(&scratch, sizeof(double) * (static_cast<size_t>(nb) * w_dim + nb), s);
    if (e != cudaSuccess) return static_cast<int>(e);
    latent_bank_partial_kernel<<<nb, 256, 0, s>>>(W, M, num_ws, w_dim, scratch, scratch + static_cast<size_t>(nb) * w_dim);
    latent_bank_final_kernel<<<1, 256, 0, s>>>(scratch, scratch + static_cast<size_t>(nb) * w_dim, nb, M, w_dim, w_sum, m2);
    int r = last_err();
    cudaFreeAsync(scratch, s);
    return r;
}
int image_bank_stats(const float* X, int M, int C, int res, int crop_off, int crop_size, float4* mean, float* m2, cudaStream_t s) {
    image_bank_mean_kernel<<<cdiv(res * res, 256), 256, 0, s>>>(X, M, C, res, mean);
    image_bank_m2_kernel<<<C < 3 ? C : 3, 1024, 0, s>>>(X, M, C, res, crop_off, crop_size, m2);
    return last_err();
}

int mapping_normalize(const float* z, int batch, int z_dim, float* out, cudaStream_t s) {
    mapping_normalize_kernel<<<batch, 256, 0, s>>>(z, z_dim, out);
    return last_err();
}
int mapping_fc(const float* x, const float* w, const float* b, int batch, int n_in, int n_out, float w_gain, float b_gain, int lrelu,
               float* y, cudaStream_t s) {
    if (n_in > 32 * kMaxRowRegs) return static_cast<int>(cudaErrorInvalidValue);
    mapping_fc_kernel<<<cdiv(n_out, 4), 128, 0, s>>>(x, w, b, batch, n_in, n_out, w_gain, b_gain, lrelu, y);
    return last_err();
}
int mapping_truncate(const float* w, const float* w_avg, float psi, int batch, int w_dim, float* out, cudaStream_t s) {
    mapping_truncate_kernel<<<cdiv(batch * w_dim, 256), 256, 0, s>>>(w, w_avg, psi, batch * w_dim, w_dim, out);
    return last_err();
}

}  // namespace la
