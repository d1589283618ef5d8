// Host-side planning helpers shared by the clients of the tap-GEMM (engine, discriminator, VGG16 in lpips.cu / detector.cu):
// tile geometry, column-block choice, TMA tensor maps and tap lists of one tap-GEMM launch, and the planners of the plain
// layers, of the four-phase transposed stride-2 convolution and of the stride-2 convolution over its phase views.
#pragma once
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "tapgemm.cuh"

namespace la {

// M tile of a grid of resolution g: 16 rows x 8 pixels with a 2-row halo (the three vertical taps share
// one TMA box) from 9^2 up (below 16^2 and at sizes that are not multiples of the tile the overhang is masked,
// e.g. the 14^2 conv5 stage of a 224^2 VGG16); whole small images below that.
inline void tile_geometry(int g, int& th, int& tw, int& nb, int& halo) {
    if (g >= 9) { th = 16; tw = 8; nb = 1; halo = 2; }
    else if (g == 8) { th = 8; tw = 8; nb = 2; halo = 0; }
    else { th = g; tw = g; nb = 128 / (g * g); halo = 0; }
}
inline long long grid_m_tiles(int g, int batch) {
    int th, tw, nb, halo;
    tile_geometry(g, th, tw, nb, halo);
    return static_cast<long long>((batch + nb - 1) / nb) * ((g + th - 1) / th) * ((g + tw - 1) / tw);
}
// Column block: 256 where the channel count allows (N = 256 MMAs run at the full tensor rate, N = 128 ones at
// about 80 % of it), 128 with two M tiles sharing each weight tile otherwise, 64 when the layer has 64 channels
// or the grid is too small to occupy the SMs with wider blocks.
inline int pick_bn(int n, long long m_tiles = 1 << 30) {
    if (n % 64) return 0;
    if (n == 64) return 64;
    if (n % 128) return 0;
    static const int force = getenv("LA_BN") ? atoi(getenv("LA_BN")) : 0;      // tuning switch
    if (force && n % force == 0) return force;
    if (m_tiles * (n / 128) <= 74) return 64;
    return n % 256 == 0 ? 256 : 128;
}
// Column block of a plain layer, whose channel count may be an odd multiple of 64
inline int choose_bn(int n, long long m_tiles) { return n % 128 ? 64 : pick_bn(n, m_tiles); }

inline int make_a_map(CUtensorMap* m, const void* base, int C, int W, int H, int N, long long sW, long long sH, long long sN, int tw, int th,
               int nb) {
    uint64_t dims[4] = {static_cast<uint64_t>(C), static_cast<uint64_t>(W), static_cast<uint64_t>(H), static_cast<uint64_t>(N)};
    uint64_t strides[3] = {static_cast<uint64_t>(sW) * 2, static_cast<uint64_t>(sH) * 2, static_cast<uint64_t>(sN) * 2};
    uint32_t box[4] = {64, static_cast<uint32_t>(tw), static_cast<uint32_t>(th), static_cast<uint32_t>(nb)};
    return encode_tmap_bf16(m, base, 4, dims, strides, box);
}
// A maps of a dense NHWC tensor [n, H, W, C] with box tw x th x nb: a_map[0] = hi plane, a_map[1] = lo plane (split)
inline int dense_maps(TapGemmParams& P, const Pl& t, int n, int C, int W, int H, int tw, int th, int nb, int split) {
    const long long sW = C, sH = static_cast<long long>(W) * C, sN = sH * H;
    if (make_a_map(&P.a_map[0], t.hi, C, W, H, n, sW, sH, sN, tw, th, nb)) return -1;
    if (split && make_a_map(&P.a_map[1], t.lo, C, W, H, n, sW, sH, sN, tw, th, nb)) return -1;
    return 0;
}
// CTA pairs (cta_group::2, M = 256 MMAs over two SMs, each SM reading half the weight tile): measured on the C2
// layers 8-12 % faster at BN = 256 / 64.  At BN = 128 a pair works on four M tiles (two per CTA); that wins for
// the plain forward convolutions (-13 %), and loses or ties for the data-gradient and up-sampling launches, whose
// epilogues set the pace -- those stay on the single-CTA kernel (callers say which with pair128).
// LA_CTA2=0: never, LA_CTA2=2: always (tuning / A-B switch).
inline int pair_mode() {
    static const int v = getenv("LA_CTA2") ? atoi(getenv("LA_CTA2")) : 1;
    return v;
}
// LA_NO_STAGED: the row-owner epilogues store bf16 outputs per element instead of staging them (A-B switch).
inline bool no_staged() {
    static const bool v = getenv("LA_NO_STAGED") != nullptr;
    return v;
}
// Weight tensor map of a launch [K, rows, nmat]; decides the CTA-pair mode of the launch: a pair's CTAs load
// half a column block each.
inline int make_b_map(TapGemmParams& P, const void* base, int K, int rows, int nmat, int bn, int pair128 = 0) {
    P.cta2 = (pair_mode() == 2 || (pair_mode() == 1 && (bn != 128 || pair128))) ? 1 : 0;
    uint64_t dims[3] = {static_cast<uint64_t>(K), static_cast<uint64_t>(rows), static_cast<uint64_t>(nmat)};
    uint64_t strides[2] = {static_cast<uint64_t>(K) * 2, static_cast<uint64_t>(K) * rows * 2};
    uint32_t box[3] = {64, static_cast<uint32_t>(P.cta2 ? bn / 2 : bn), 1};
    return encode_tmap_bf16(&P.b_map, base, 3, dims, strides, box);
}

inline void set_ops_dims(TapSimtOperands& o, int w, int h) {
    for (int i = 0; i < kMaxAMaps; ++i) { o.a_ws[i] = w; o.a_hs[i] = h; }
}

inline void add_tap(TapGemmParams& P, int& nt, int dy, int dx, int widx, int src_hi, int src_lo, int nmat, int split) {
    P.taps[nt++] = Tap{static_cast<int8_t>(dy), static_cast<int8_t>(dx), static_cast<uint8_t>(widx), static_cast<uint8_t>(src_hi)};
    if (split) {
        P.taps[nt++] = Tap{static_cast<int8_t>(dy), static_cast<int8_t>(dx), static_cast<uint8_t>(widx), static_cast<uint8_t>(src_lo)};
        P.taps[nt++] = Tap{static_cast<int8_t>(dy), static_cast<int8_t>(dx), static_cast<uint8_t>(nmat + widx), static_cast<uint8_t>(src_hi)};
    }
}

// Tile box from the grid resolution g; problem i covers a gh[i] x gw[i] grid (all = g unless given).
inline void set_grid(TapGemmParams& P, int g, int batch, int nprob, const int* gh = nullptr, const int* gw = nullptr) {
    tile_geometry(g, P.th, P.tw, P.nb, P.halo);
    P.tiles_n = (batch + P.nb - 1) / P.nb;
    P.batch = batch;
    P.nprob = nprob;
    P.m_tiles = 0;
    for (int i = 0; i < nprob; ++i) {
        TapProblem& pr = P.prob[i];
        pr.vh = gh ? gh[i] : g;
        pr.vw = gw ? gw[i] : g;
        pr.tiles_h = (pr.vh + P.th - 1) / P.th;
        pr.tiles_w = (pr.vw + P.tw - 1) / P.tw;
        pr.tile_begin = P.m_tiles;
        P.m_tiles += P.tiles_n * pr.tiles_h * pr.tiles_w;
    }
}

// Interleaved walk of a multi-problem launch: one common tile grid (the largest), problems masked by vh / vw.
inline void set_interleaved(TapGemmParams& P) {
    int th = 0, tw = 0;
    for (int i = 0; i < P.nprob; ++i) { th = P.prob[i].tiles_h > th ? P.prob[i].tiles_h : th; tw = P.prob[i].tiles_w > tw ? P.prob[i].tiles_w : tw; }
    for (int i = 0; i < P.nprob; ++i) { P.prob[i].tiles_h = th; P.prob[i].tiles_w = tw; P.prob[i].tile_begin = 0; }
    const int spatial = P.tiles_n * th * tw;
    P.m_tiles = 2 * P.nprob * ((spatial + 1) / 2);
    P.interleave = 1;
}

// ------------------------------------------------------------------------- plain layers
// Every planner below returns 0 or the failing call's code; the caller reports it under its own module name.

// Weights w [nmat][N][K] (residual planes behind them when split) of a launch whose grid is set: N columns in blocks of bn
// (0: choose_bn), K / 64 chunks per tap.
inline int plan_columns(TapGemmParams& P, const __nv_bfloat16* w, int K, int N, int nmat, int split, int bn = 0) {
    if (!bn) bn = choose_bn(N, P.m_tiles);
    if (int r = make_b_map(P, w, K, N, nmat * (split ? 2 : 1), bn)) return r;
    P.kchunks = K / 64; P.n_total = N; P.n_blocks = N / bn; P.split = split;
    return 0;
}

enum class LayerTaps {
    k3x3,          // 3x3 convolution, pad 1: out[y, x] += in[y + dy, x + dx] W[(dy + 1) * 3 + dx + 1]
    k3x3Flipped,   // its data gradient (offsets negated)
    k1x1,
    kDense,        // fully connected over the whole R x R x K input: one tap per input position, a 1 x 1 output, so
                   // the M rows are samples (128 per tile, tile_geometry of a 1 x 1 grid)
};

// P <- a launch over the dense NHWC input in [n, R, R, K] (hi, plus lo when split) with N output columns and weights w
// [taps][N][K]: everything but the epilogue, which fwd_epilogue / linear_epilogue (or the caller) sets.  bn = 0: choose_bn.
inline int plan_layer(TapGemmParams& P, LayerTaps taps, const Pl& in, int n, int R, int K, int N, const __nv_bfloat16* w, int split,
                      int* err_flag, int bn = 0) {
    const bool dense = taps == LayerTaps::kDense;
    const int g = dense ? 1 : R;
    const int nmat = dense ? R * R : taps == LayerTaps::k1x1 ? 1 : 9;
    memset(&P, 0, sizeof P);
    set_grid(P, g, n, 1);
    if (int r = dense_maps(P, in, n, K, R, R, P.tw, P.th + P.halo, P.nb, split)) return r;
    if (int r = plan_columns(P, w, K, N, nmat, split, bn)) return r;
    P.OH = P.OW = g; P.osy = P.osx = 1;
    P.err_flag = err_flag;
    int nt = 0;
    for (int t = 0; t < nmat; ++t) {
        int dy = 0, dx = 0;
        if (dense) { dy = t / R; dx = t % R; }
        else if (nmat == 9) { dy = t / 3 - 1; dx = t % 3 - 1; }
        if (taps == LayerTaps::k3x3Flipped) { dy = -dy; dx = -dx; }
        add_tap(P, nt, dy, dx, t, 0, 1, nmat, split);
    }
    P.prob[0].ntaps = nt;
    return tapgemm_finalize(P);
}

// Unmodulated forward epilogue: out = act(acc + bias) (act.cuh: gain, clamp, slope), demod = ones (>= batch * N 1.0f).
inline void fwd_epilogue(TapGemmParams& P, const float* ones, const float* bias, float gain, float clamp, float slope, const Pl& out) {
    P.epilogue = kEpiFwd;
    P.act_gain = gain; P.act_clamp = clamp; P.act_slope = slope;
    P.demod = ones; P.bias = bias;
    P.x_hi = out.hi; P.x_lo = out.lo;
    P.staged = P.nb == 1 && !P.split && !no_staged();
}
// kEpiLinear with gain 1 and no clamp; slope is the producer activation's (its gradient, when lin_gz is set).
inline void linear_epilogue(TapGemmParams& P, float slope) {
    P.epilogue = kEpiLinear;
    P.act_gain = 1.f; P.act_clamp = -1.f; P.act_slope = slope;
}

// ------------------------------------------------------------------------- stride-2 convolutions through T
// T [n, 2R + 1, 2R + 2, C] (rows, row pitch) holds a transposed stride-2 3x3 convolution of an R x R input before its FIR pass
// (the x2 up-sampling of the generator, the gradient of the discriminator's stride-2 conv1).

// P <- the transposed stride-2 3x3 convolution of the dense NHWC input in [n, R, R, K] into T = t with N channels (weights w
// [9][N][K]): T[2i + a] += in[i] W[a], so output phase (py, px) = (T[2i + py], T[2j + px]) is problem py * 2 + px of the launch
// with the taps whose a = phase (mod 2); the even phases have one more row / column.  kEpiStoreBf16.  Does not clear P: fields
// the caller set before stay.  interleave: walk the phases interleaved (set_interleaved).
inline int plan_upconv(TapGemmParams& P, const Pl& in, int n, int R, int K, int N, const __nv_bfloat16* w, int split, const Pl& t,
                       bool interleave = false) {
    const int gh[4] = {R + 1, R + 1, R, R}, gw[4] = {R + 1, R, R + 1, R};
    set_grid(P, R, n, 4, gh, gw);
    if (interleave) set_interleaved(P);
    if (int r = dense_maps(P, in, n, K, R, R, P.tw, P.th + P.halo, P.nb, split)) return r;
    if (int r = plan_columns(P, w, K, N, 9, split)) return r;
    int nt = 0;
    for (int ph = 0; ph < 4; ++ph) {
        P.prob[ph].tap_begin = nt;
        for (int ay = ph / 2; ay < 3; ay += 2)
            for (int ax = ph % 2; ax < 3; ax += 2) add_tap(P, nt, -(ay >> 1), -(ax >> 1), ay * 3 + ax, 0, 1, 9, split);
        P.prob[ph].ntaps = nt - P.prob[ph].tap_begin;
        P.prob[ph].oy0 = ph / 2; P.prob[ph].ox0 = ph % 2;
    }
    P.epilogue = kEpiStoreBf16;
    P.OH = 2 * R + 1; P.OW = 2 * R + 2; P.osy = P.osx = 2;
    P.x_hi = t.hi; P.x_lo = t.lo;
    P.staged = P.nb == 1 && !split && !no_staged();
    return tapgemm_finalize(P);
}

// A maps and taps of the stride-2 3x3 convolution over T = t [n, R + 1, R + 2, K] (plan_upconv's output for an R / 2 input),
// read as its four phase views (py, px) = T[2i + py, 2j + px]: hi maps 0-3, lo maps 4-7, tap W[a] reads view a (mod 2) at
// offset a >> 1.  P's grid (R / 2) must be set; the taps are appended at nt (as add_tap does) and the caller finalizes.  ops,
// when given, gets the same views for the SIMT twin.
inline int phase_view_taps(TapGemmParams& P, int& nt, const Pl& t, int n, int R, int K, int split, TapSimtOperands* ops = nullptr) {
    const int TH = R + 1, TWp = R + 2, Ro = R / 2;
    const long long gW = 2LL * K, gH = 2LL * TWp * K, gN = static_cast<long long>(TH) * TWp * K;
    if (ops) { ops->a_sw = gW; ops->a_sh = gH; ops->a_sn = gN; }
    for (int ph = 0; ph < 4; ++ph) {
        const int py = ph / 2, px = ph % 2;
        const int ph_h = Ro + (py == 0), ph_w = Ro + (px == 0);
        const long long off = (static_cast<long long>(py) * TWp + px) * K;
        for (int plane = 0; plane <= split; ++plane) {
            const int m = ph + 4 * plane;
            const __nv_bfloat16* base = (plane ? t.lo : t.hi) + off;
            if (int r = make_a_map(&P.a_map[m], base, K, ph_w, ph_h, n, gW, gH, gN, P.tw, P.th + P.halo, P.nb)) return r;
            if (ops) { ops->a_ptrs[m] = base; ops->a_ws[m] = ph_w; ops->a_hs[m] = ph_h; }
        }
    }
    for (int ay = 0; ay < 3; ++ay)
        for (int ax = 0; ax < 3; ++ax) {
            const int ph = (ay & 1) * 2 + (ax & 1);
            add_tap(P, nt, ay >> 1, ax >> 1, ay * 3 + ax, ph, 4 + ph, 9, split);
        }
    return 0;
}

}  // namespace la
