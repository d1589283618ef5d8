// Host-side planning helpers shared by the clients of the tap-GEMM (engine, discriminator, VGG16 in lpips.cu / detector.cu):
// tile geometry, column-block choice, TMA tensor maps and tap lists of one tap-GEMM launch.
#pragma once
#include <stdlib.h>

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


}  // namespace la
