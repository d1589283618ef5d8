// Tap-GEMM: the one tensor-core kernel of the synthesis path (forward and backward-to-w).
//
//   acc[pixel, col] = sum_{t in taps} sum_{k < K}  A_{src_t}[pixel + (dy_t, dx_t), k] * Wstack[widx_t][col][k]
//
// A_* are NHWC bf16 activation tensors (each described by one 4-D TMA tensor map), Wstack a
// stack of K-major [N x K] bf16 matrices.  Every 3x3 modulated convolution of the generator,
// its data gradient, the four sub-pixel phases of the x2 up-sampling convolution (transposed
// conv + 4x4 FIR folded into per-phase 3x3 weights) and the gradient of that layer are
// instances of this contraction; split-bf16 ("fp32-parity") precision is three taps per
// geometric tap: (A_hi,W_hi) + (A_lo,W_hi) + (A_hi,W_lo).   See DESIGN.md §3.
//
// M tile = nb images x th rows x tw cols (<= 128 pixels); zero padding is TMA out-of-bounds
// fill.  Taps that share (source map, dx) and differ only in dy form a GROUP: with `halo` = 2
// (tw == 8, nb == 1) one TMA box of th + 2 rows per (group, 64-channel chunk) feeds all of
// them -- a row of 8 pixels is one 1024-byte swizzle atom, so the tap (dy) is just a start
// offset of the UMMA descriptor -- and two consecutive M tiles share every weight tile
// (operand traffic from L2 is the bound of this kernel: DESIGN.md §3.1).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace la {

constexpr int kMaxTaps = 108;     // 36 geometric taps x 3 split-precision passes
constexpr int kMaxProblems = 4;   // 4 sub-pixel phases
constexpr int kMaxAMaps = 8;      // 4 phase planes x {hi, lo}

struct Tap {
    int8_t dy, dx;       // spatial offset added to the tile origin
    uint8_t widx;        // which [N x K] matrix of the weight stack
    uint8_t src;         // which A tensor map
};

struct TapGroup {
    int8_t dx, dy0;      // box origin offset of the group (dy0 = smallest dy of its taps)
    uint8_t src;         // A tensor map
    uint8_t ntaps;
    uint16_t tap_begin;  // first entry of gdyrel / gwidx
    uint16_t pad;
};

struct TapProblem {
    int tap_begin, ntaps;
    int grp_begin, ngroups;
    int oy0, ox0;                  // output pixel = (h*osy + oy0, w*osx + ox0)
    int tile_begin;                // first M-tile index of this problem
    int tiles_h, tiles_w;          // tile grid of this problem (x tiles_n images)
    int vh, vw;                    // valid extent (rows, cols); tile overhang is masked
};

enum TapEpilogue : int {
    kEpiRawF32 = 0,    // store accumulators as fp32 [pixel][n_total]                  (tests)
    kEpiFwd = 1,       // demod + noise + bias + lrelu*gain + clamp -> x, x*s_next, toRGB partials
    kEpiBwd = 2,       // style-gradient reductions + activation backward of the producer layer -> g_y
    kEpiTopK = 3,      // rows = queries, columns = bank codes: the 2 smallest |y|^2 - 2<x,y> per row and 32-code chunk
    kEpiStoreBf16 = 4, // store accumulators as bf16 (hi [+ lo]) into x_hi / x_lo [pixel][n_total]
    kEpiLinear = 5,    // plain (unmodulated) layers of the discriminator: r = acc (+ lin_add) -> lin_out;
                       // r * act'(lin_saved) -> lin_gz   (bf16 [pixel][n_total] tensors, each optional)
};

struct TapGemmParams {
    alignas(64) CUtensorMap a_map[kMaxAMaps];
    alignas(64) CUtensorMap b_map;
    int staged;                      // 1 (bf16 mode, nb == 1): the row-owner epilogues stage their bf16 outputs through shared
                                     //    memory (whole 64-byte row segments per store) and, in the forward epilogue, read the
                                     //    per-column coefficients from a shared-memory table
    Tap taps[kMaxTaps];              // flat tap list (host bookkeeping + the SIMT twin)
    TapGroup groups[kMaxTaps];       // the same taps grouped for the tensor-core kernel (tapgemm_finalize)
    uint8_t gdyrel[kMaxTaps];        // per grouped tap: dy - dy0 of its group (0..halo)
    uint8_t gwidx[kMaxTaps];         // per grouped tap: weight matrix
    int halo;                        // extra rows of the A box (0 or 2); 2 needs tw == 8 and nb == 1
    int no_pair;                     // 1: never pair M tiles (tuning switch)
    int cost_fixed;                  // set by the launcher: fixed (epilogue) share of a tile's cost in K steps, for the range balance
    int no_quad;                     // set by the launcher (pair launches): one M tile per CTA, never four-tile work items
    int cta2;                        // 1: CTA pairs (clusters of 2, cta_group::2 MMAs with M = 256): the b_map box holds HALF a column block
    int interleave;                  // 1: all problems share one tile grid (tiles_h/w equal, vh/vw mask) and are walked
                                     //    [column block][pair of spatial tiles][problem][tile of the pair], so that every
                                     //    CTA gets the same mix of cheap and expensive problems
    int dbg_skip_epi;                // 1: epilogues only drain the accumulators (timing experiment: wrong results)
    TapProblem prob[kMaxProblems];
    int nprob;
    int th, tw, nb;        // M-tile box: nb images x th rows x tw cols (nb*th*tw <= 128)
    int tiles_n;           // ceil(batch / nb)
    int batch;             // images
    int kchunks;           // K / 64 per tap
    int n_total;           // N (columns = output channels of this GEMM)
    int n_blocks;          // N / BN
    int m_tiles;           // sum of M tiles over problems
    int epilogue;          // TapEpilogue
    int OH, OW, osy, osx;  // output tensor spatial dims and the pixel stride of the tile grid in it
    int split;             // 1: *_lo planes are written / read (split-bf16 precision)
    float act_gain, act_clamp, act_slope;

    float* raw_out;                    // kEpiRawF32: [batch, OH, OW, n_total]

    // ---- kEpiFwd: this GEMM is layer l, columns = its output channels
    const float* demod;                // [batch, N]
    const float* bias;                 // [N]
    const float* noise;                // [*, OH, OW] unit noise, or null
    long long noise_stride_n;          // 0 = shared across the batch, OH*OW = per sample
    float noise_scale;                 // noise_strength
    const float* s_next;               // [batch, N] style of the consumer conv, or null
    void* x_hi; void* x_lo;            // bf16 [batch, OH, OW, N]  activation (saved for backward)
    void* xs_hi; void* xs_lo;          // bf16 [batch, OH, OW, N]  x * s_next (A operand of the consumer)
    const float4* rgbw;                // [batch, N] (W_rgb[c][col] * s_rgb[n][col], c = x,y,z) or null
    float4* rgb_part;                  // [2*n_blocks][batch, OH, OW] toRGB partial sums per (column block, epilogue group)

    // ---- kEpiBwd: this GEMM is the data gradient of layer l; columns = channels of x_{l-1}
    const float* s_cur;                // [batch, N] style of layer l
    const void* xp_hi; const void* xp_lo;   // bf16 x_{l-1} [batch(or 1), OH, OW, N]
    long long xp_stride_n;             // must be OH*OW*N (the learned constant is replicated per sample)
    const float4* g_rgb;               // [batch, OH, OW] gradient wrt the toRGB output fed by x_{l-1}, or null
    const float4* rgbw_prev;           // [batch, N]
    const float* demod_prev;           // [batch, N]   (layer l-1)
    const float* bias_prev;            // [N]
    const float* noise_prev;           // [*, OH, OW] or null
    long long noise_prev_stride_n;
    float noise_prev_scale;
    void* gy_hi; void* gy_lo;          // bf16 [batch, OH, OW, N]  g_y of layer l-1 (A operand of its dgrad)
    float* red_s;                      // [batch, N]      += sum_px acc * x_{l-1}
    float* red_d;                      // [batch, N]      += sum_px g_z * (z - noise - bias)
    float* red_rgb;                    // [3][batch, N]   += sum_px x_{l-1} * g_rgb[c]
    int bwd_last;                      // 1: x_{l-1} is the constant input: only red_s is produced

    // ---- kEpiLinear
    const void* lin_add;               // bf16 addend (residual branch / second gradient path) or null
    const void* lin_add_down;          // bf16 [batch, OH/2, OW/2, N] or null: adds the ADJOINT of the decimating 4x4 FIR
                                       // (upfirdn2d down=2, pad 1) of this tensor: sum_{2m+j-1=v} lin_fir[j] * t[m]
    float lin_fir[16];                 // flipped 4x4 filter of lin_add_down
    void* lin_out;                     // bf16 r or null
    const void* lin_saved;             // bf16 saved activation output deciding the activation gradient, or null
    void* lin_gz;                      // bf16 r * act_gain * (saved > 0 ? 1 : act_slope), 0 where saved is clamped (act.cuh), or null
    const void* lin_add_lo; const void* lin_add_down_lo; void* lin_out_lo; void* lin_gz_lo;   // residual planes when split
    const void* lin_saved_lo;          // residual plane of lin_saved (split), or null: the clamp decision reads hi + lo
    const float* lin_rgb_w;            // [N][4] or null: fused 1x1 "fromrgb" backward -- the activation-gradient row (the lin_gz
    float4* lin_rgb_g;                 // value) is contracted with these weights and atomically added to lin_rgb_g[pixel].xyz

    // ---- kEpiTopK: acc[query, code] = <x, y>
    const float* code_sqnorm;          // [n_codes] |y_j|^2
    int n_codes, n_queries, topk;      // topk = 2
    float* cand_score;                 // [n_queries][n_blocks * BN / 32][2]  ascending per 32-code chunk
    int* cand_idx;                     // [n_queries][n_blocks * BN / 32][2]  (-1 = empty)

    int* err_flag;
    unsigned long long* dbg_clock;     // optional [64]: CTA 0 cycles, nanoseconds and MMA-thread timeline stamps (LA_DBG_CLK experiments)
};

// Groups the flat taps of every problem (call after taps / prob[].tap_begin / ntaps are set).  Returns 0 on success.
int tapgemm_finalize(TapGemmParams& p);

// Column block width the kernel is instantiated for: 64, 128 or 256.
inline int tapgemm_bn(const TapGemmParams& p) { return p.n_total / p.n_blocks; }

// tcgen05 path.  Returns cudaError_t as int.
int launch_tapgemm(const TapGemmParams& p, int num_sms, cudaStream_t stream);

// Seed of the backward chain: the kEpiBwd epilogue with a zero accumulator (no GEMM).
int launch_tapgemm_seed(const TapGemmParams& p, int num_sms, cudaStream_t stream);

// SIMT evaluation of the same contraction with the SAME epilogue code: the debug cross-check
// of the tensor-core path in tests.  `a_ptrs[i]` / `a_dims` describe what a_map[i] maps
// (dims = {C, W, H, N}, strides in elements {sW, sH, sN}); `w` is the weight stack.
struct TapSimtOperands {
    const void* a_ptrs[kMaxAMaps];
    long long a_sw, a_sh, a_sn;
    int a_ws[kMaxAMaps], a_hs[kMaxAMaps];    // spatial extent of each map
    const void* w;
};
int launch_tapgemm_simt(const TapGemmParams& p, const TapSimtOperands& ops, cudaStream_t stream);

// Host helper: encode a bf16 tiled tensor map with 128B swizzle.  dims/box are innermost
// first; strides (bytes) has rank-1 entries.  Returns 0 on success.
int encode_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides,
                     const uint32_t* box, int swizzle_bytes = 128);

}  // namespace la
