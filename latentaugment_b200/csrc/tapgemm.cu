// Tap-GEMM kernel for sm_100a: TMA-fed, tcgen05.mma with TMEM accumulators, warp-specialised,
// persistent.  See tapgemm.cuh for the contraction and DESIGN.md §3 for the tiling.
#include "tapgemm.cuh"

#include <cuda_bf16.h>
#include <stdio.h>

#include <type_traits>

#include "act.cuh"
#include "sm100.cuh"

namespace la {

namespace {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;                       // 64 bf16 = one 128-byte swizzle row
constexpr int kASubBytes = 18 * 1024;             // A box of one M tile: (16 + 2 halo) rows x 8 pixels x 128 B (16 KB without halo)
constexpr int kThreads = 384;                     // warp0 TMA, warp1 MMA, warp2 TMEM alloc, warp3 idle, warps4-11 epilogue
constexpr int kEpiThreads = 256;                  // 8 epilogue warps; warp e owns TMEM lanes 32*(e%4)..+31
constexpr unsigned kRowMasked = 0xffffffffu;
constexpr int kTransStride = 36;                  // floats per row of a warp's 32x32 transpose tile (144 B: conflict-free both ways)
constexpr int kRegsProducer = 56, kRegsEpilogue = 224;   // setmaxnreg: 128*56 + 256*224 = 64512 <= 65536

// Per-warp scratch of the backward epilogue.
struct WarpSmem {                     // (row data is double-buffered: the next tile's rows are staged while this one computes)
    float trans[32 * kTransStride];   // accumulator chunk, row-owner write -> column-owner read
    float4 grgb[2][32];               // per row: gradient wrt the toRGB output
    float nz[2][32];                  // per row: noise * strength of the producer layer
    unsigned off[2][32];              // per row: pixel index * N/2 (offset of the row in bf16x2 units), kRowMasked = masked
};

template <int BN, int EPI, bool kPair = false>
struct Cfg {
    static constexpr int kMtMax = BN == 256 ? 1 : 2;             // M tiles per unit (they share every weight tile)
    static constexpr int kASlotBytes = kMtMax * kASubBytes;
    static constexpr int kBBytes = BN * kBlockK * 2;
    static constexpr int kAStages = (BN == 256 && EPI == kEpiBwd) ? 4 : 3;
    static constexpr int kBStages = EPI == kEpiBwd ? (BN == 256 ? 3 : (BN == 128 ? 4 : 6)) : (BN == 256 ? 4 : (BN == 128 ? (EPI == kEpiFwd ? 5 : 6) : 8));
    static constexpr int kTmemCols = 2 * kMtMax * BN;            // two accumulator stages
    // row-owner epilogues: a 2 KB staging tile per warp (32 rows x 32 channels bf16) for coalesced stores and,
    // for the forward epilogue, one table of per-column coefficients per warp group:
    // [demod | s_next | rgbw.x | rgbw.y | rgbw.z | bias] x BN floats of the (sample, column block) being processed
    static constexpr int kStageTensors = (EPI == kEpiFwd || EPI == kEpiStoreBf16) ? 1 : 0;
    static constexpr int kCoefBytes = EPI == kEpiFwd ? 2 * 6 * BN * 4 : 0;
    static constexpr int kEpiSmemBytes = EPI == kEpiBwd ? 8 * static_cast<int>(sizeof(WarpSmem)) : 8 * 2048 * kStageTensors + kCoefBytes;
    static constexpr int kABytes = kAStages * kASlotBytes;       // unpaired launches cut this region into kASubBytes slots
    // CTA pairs: each CTA holds half a weight tile per stage, so the same bytes give a ring twice as deep
    static constexpr int kBSlotBytes = kPair ? kBBytes / 2 : kBBytes;
    static constexpr int kBRing = kPair ? 2 * kBStages : kBStages;
    static constexpr int kSmemBytes = kABytes + kBStages * kBBytes + kEpiSmemBytes + 512 /*barriers*/ + 1024 /*align slack*/;
    static constexpr int kBwdSteps = BN == 64 ? 2 : 4;           // 32-column steps one warp walks per tile (all of BN, or half of it)
};

struct TileCoord {
    int prob, nblk, n0, h0, w0;
    bool empty;          // interleaved walk only: the tile lies outside its problem's valid extent
};

__device__ __forceinline__ TileCoord decode_tile(const TapGemmParams& P, int t) {
    TileCoord c;
    c.nblk = t / P.m_tiles;                  // M fastest: a CTA's contiguous chunk shares the weight tile
    int m = t - c.nblk * P.m_tiles;
    int local;
    if (P.interleave) {
        const int per = 2 * P.nprob;
        const int grp = m / per, r = m - grp * per;
        c.prob = r >> 1;
        local = grp * 2 + (r & 1);
    } else {
        int p = 0;
#pragma unroll
        for (int i = 1; i < kMaxProblems; ++i)
            if (i < P.nprob && m >= P.prob[i].tile_begin) p = i;
        c.prob = p;
        local = m - P.prob[p].tile_begin;
    }
    const TapProblem& pr = P.prob[c.prob];
    int tx = local % pr.tiles_w;
    int ty = (local / pr.tiles_w) % pr.tiles_h;
    int tn = local / (pr.tiles_w * pr.tiles_h);
    c.n0 = tn * P.nb;
    c.h0 = ty * P.th;
    c.w0 = tx * P.tw;
    c.empty = P.interleave && (tn >= P.tiles_n || c.h0 >= pr.vh || c.w0 >= pr.vw);
    return c;
}

// A unit = one or two consecutive M tiles of the same (column block, problem); mt == 0: nothing to do.
struct Unit {
    TileCoord tc0, tc1;      // (no array: a dynamic index would put the struct in local memory)
    int mt, adv;
    __device__ __forceinline__ const TileCoord& tile(int s) const { return s ? tc1 : tc0; }
};
template <int MTMAX>
__device__ __forceinline__ Unit get_unit(const TapGemmParams& P, int t, int t_end) {
    Unit u;
    u.tc0 = decode_tile(P, t);
    u.tc1 = u.tc0;
    u.mt = 1;
    if (P.interleave) {      // ranges are aligned to whole groups: t is the first tile of a (pair, problem)
        u.adv = 2;
        const TileCoord c = decode_tile(P, t + 1);
        if (u.tc0.empty) { u.tc0 = c; u.tc1 = c; u.mt = c.empty ? 0 : 1; }
        else if (!c.empty) {
            if (MTMAX == 2 && !P.no_pair) { u.tc1 = c; u.mt = 2; }
            else u.adv = 1;  // unpaired kernels take the two tiles one after the other
        }
        return u;
    }
    if (MTMAX == 2 && t + 1 < t_end && !P.no_pair) {
        const TileCoord c = decode_tile(P, t + 1);
        if (c.nblk == u.tc0.nblk && c.prob == u.tc0.prob) { u.tc1 = c; u.mt = 2; }
    }
    u.adv = u.mt;
    return u;
}

// CTA-pair launches (cta_group::2): the two M tiles of a unit go to the two CTAs of the cluster.  A CTA without a
// tile of its own (odd tile at a range or problem boundary) loads tile 0 again and runs its epilogue with every
// row masked, so both CTAs walk the same barrier sequence.
__device__ __forceinline__ TileCoord pair_tile(const Unit& u, uint32_t rank) {
    TileCoord tc = (rank == 1u && u.mt == 2) ? u.tc1 : u.tc0;
    if (static_cast<int>(rank) >= u.mt) tc.empty = true;
    return tc;
}

// Work item of a CTA pair: unit a (its tiles go to the leader / the peer) and, where two M tiles fit a CTA (BN <= 128),
// the next unit b of the same (column block, problem) as second sub-tile -- four M tiles share every weight tile.
struct PairWork {
    Unit a, b;
    int nsub, adv;
};
template <int MTMAX>
__device__ __forceinline__ PairWork get_pair_work(const TapGemmParams& P, int t, int t_end) {
    PairWork w;
    w.a = get_unit<2>(P, t, t_end);
    w.b = w.a;
    w.nsub = 1;
    w.adv = w.a.adv;
    if (MTMAX == 2 && !P.no_quad && w.a.mt == 2 && t + 2 < t_end) {
        const Unit n = get_unit<2>(P, t + 2, t_end);
        if (n.tc0.nblk == w.a.tc0.nblk && n.tc0.prob == w.a.tc0.prob) { w.b = n; w.nsub = 2; w.adv += n.adv; }
    }
    return w;
}

// Contiguous, COST-balanced tile range of this CTA.  The phases of the transposed convolution have 4 / 2 / 2 / 1
// taps; a tile costs (taps x K chunks) MMA steps plus a fixed epilogue share worth about four steps (measured:
// with taps alone the CTAs that own the one-tap phase finish 35 % after the others).  Tiles are ordered
// [nblk][problem][tile].
__device__ __forceinline__ long long tile_cost(const TapGemmParams& P, const TapProblem& pr) {
    return pr.ntaps > 0 ? static_cast<long long>(pr.ntaps) * P.kchunks + P.cost_fixed : 1;
}
__device__ __forceinline__ long long tiles_before(const TapGemmParams& P, long long cost_per_nblk, long long x) {
    long long nb_full = x / cost_per_nblk;
    if (nb_full >= P.n_blocks) return static_cast<long long>(P.n_blocks) * P.m_tiles;
    long long rem = x - nb_full * cost_per_nblk, count = nb_full * P.m_tiles;
    for (int p = 0; p < P.nprob; ++p) {
        const TapProblem& pr = P.prob[p];
        const long long c = tile_cost(P, pr);
        const long long tiles = static_cast<long long>(pr.tiles_h) * pr.tiles_w * P.tiles_n;
        if (rem >= tiles * c) { count += tiles; rem -= tiles * c; }
        else { count += (rem + c - 1) / c; break; }
    }
    return count;
}
__device__ __forceinline__ void tile_range(const TapGemmParams& P, int& begin, int& end, int worker, int nworkers) {
    if (P.interleave) {      // every group of 2 * nprob tiles costs the same: split the groups evenly
        const int per = 2 * P.nprob;
        const long long groups = static_cast<long long>(P.n_blocks) * (P.m_tiles / per);
        begin = static_cast<int>(groups * worker / nworkers) * per;
        end = static_cast<int>(groups * (worker + 1) / nworkers) * per;
        return;
    }
    long long cost = 0;
    for (int p = 0; p < P.nprob; ++p)
        cost += static_cast<long long>(P.prob[p].tiles_h) * P.prob[p].tiles_w * P.tiles_n * tile_cost(P, P.prob[p]);
    const long long total = cost * P.n_blocks;
    begin = static_cast<int>(tiles_before(P, cost, total * worker / nworkers));
    end = static_cast<int>(tiles_before(P, cost, total * (worker + 1) / nworkers));
}
__device__ __forceinline__ void tile_range(const TapGemmParams& P, int& begin, int& end) {
    tile_range(P, begin, end, static_cast<int>(blockIdx.x), static_cast<int>(gridDim.x));
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ void st_global_if(unsigned* p, unsigned v, bool ok) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.b32 q, %2, 0;\n\t@q st.global.b32 [%0], %1;\n\t}" ::"l"(p), "r"(v), "r"(static_cast<int>(ok)));
}
__device__ __forceinline__ float bf16_round(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }
__device__ __forceinline__ float bf16lo_f(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16hi_f(uint32_t u) { return __uint_as_float(u & 0xffff0000u); }

// store 32 consecutive values as bf16 (hi plane) and, if lo != null, the bf16 residual (lo plane)
__device__ __forceinline__ void store_bf16x32(void* hi, void* lo, long long off, const float (&v)[32]) {
    uint4* dh = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(hi) + off);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        uint4 o;
        o.x = pack_bf16(v[8 * j + 0], v[8 * j + 1]);
        o.y = pack_bf16(v[8 * j + 2], v[8 * j + 3]);
        o.z = pack_bf16(v[8 * j + 4], v[8 * j + 5]);
        o.w = pack_bf16(v[8 * j + 6], v[8 * j + 7]);
        dh[j] = o;
    }
    if (lo) {
        uint4* dl = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(lo) + off);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float r[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) r[i] = v[8 * j + i] - bf16_round(v[8 * j + i]);
            uint4 o;
            o.x = pack_bf16(r[0], r[1]);
            o.y = pack_bf16(r[2], r[3]);
            o.z = pack_bf16(r[4], r[5]);
            o.w = pack_bf16(r[6], r[7]);
            dl[j] = o;
        }
    }
}

__device__ __forceinline__ void load_bf16x32(const void* p, long long off, float (&v)[32]) {
    const uint4* s = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p) + off);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint4 a = __ldg(s + j);
        v[8 * j + 0] = bf16lo_f(a.x); v[8 * j + 1] = bf16hi_f(a.x);
        v[8 * j + 2] = bf16lo_f(a.y); v[8 * j + 3] = bf16hi_f(a.y);
        v[8 * j + 4] = bf16lo_f(a.z); v[8 * j + 5] = bf16hi_f(a.z);
        v[8 * j + 6] = bf16lo_f(a.w); v[8 * j + 7] = bf16hi_f(a.w);
    }
}

__device__ __forceinline__ void load_f32x32(const float* p, float (&v)[32]) {
    const float4* s = reinterpret_cast<const float4*>(p);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        float4 a = __ldg(s + j);
        v[4 * j] = a.x; v[4 * j + 1] = a.y; v[4 * j + 2] = a.z; v[4 * j + 3] = a.w;
    }
}

// ------------------------------------------------------------------------------------
// Epilogues shared by the tensor-core kernel, its SIMT twin and the seed kernel.  They are written
// per WARP: epilogue warp e (0..7) owns accumulator rows 32*(e & 3)..+31 (its TMEM lane quarter) of
// one M tile and a range of 32-column chunks; no barrier wider than a warp is ever taken.

struct RowCtx {
    bool valid;
    int n;
    long long pix;       // output pixel index (n*OH + oh)*OW + ow
    long long px_in_img; // oh*OW + ow
};

__device__ __forceinline__ RowCtx make_row(const TapGemmParams& P, const TileCoord& tc, int row) {
    RowCtx r;
    const int box_px = P.th * P.tw;
    const int ni = row / box_px;
    const int rem = row - ni * box_px;
    const int hi = rem / P.tw;
    const int wi = rem - hi * P.tw;
    const int n = tc.n0 + ni, h = tc.h0 + hi, w = tc.w0 + wi;
    const TapProblem& pr = P.prob[tc.prob];
    r.valid = !tc.empty && (ni < P.nb) && (n < P.batch) && (h < pr.vh) && (w < pr.vw);
    r.n = n;
    const int oh = h * P.osy + pr.oy0, ow = w * P.osx + pr.ox0;
    r.px_in_img = static_cast<long long>(oh) * P.OW + ow;
    r.pix = static_cast<long long>(n) * P.OH * P.OW + r.px_in_img;
    return r;
}

// Stage one 32-value row chunk as bf16 into the warp's [32 rows x 64 B] SWIZZLE_64B staging tile.
__device__ __forceinline__ void stage_bf16x32(uint8_t* stg, int lane, const float (&v)[32]) {
    uint8_t* rowp = stg + lane * 64;
    const int sw = (lane >> 1) & 3;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        uint4 o;
        o.x = pack_bf16(v[8 * j + 0], v[8 * j + 1]);
        o.y = pack_bf16(v[8 * j + 2], v[8 * j + 3]);
        o.z = pack_bf16(v[8 * j + 4], v[8 * j + 5]);
        o.w = pack_bf16(v[8 * j + 6], v[8 * j + 7]);
        *reinterpret_cast<uint4*>(rowp + ((j ^ sw) << 4)) = o;
    }
}

// ---- row-owner epilogues: raw store, bf16 store, forward activation, top-k.
// The lane owns row 32*q + lane and walks chunks [ch_begin, ch_end); `part` selects the per-column-block
// slot (0 / 1) of the per-row outputs (toRGB partial, top-k candidates); with `fill_other` the other slot is
// written as empty (the warp covered the whole column block).  With kStaged (one sample per tile) the bf16
// outputs go through the warp's 2 KB shared-memory staging tile `stg` and are re-read so that every store
// instruction writes whole 64-byte row segments instead of 32 scattered 16-byte pieces, and the forward
// epilogue reads its per-column coefficients from the warp group's table `ctab` instead of global memory.
template <int BN, int EPI, bool kStaged, class LoadChunk>
__device__ __forceinline__ void rowowner_warp_tile(const TapGemmParams& P, const TileCoord& tc, int q, int lane, int ch_begin, int ch_end,
                                                   int part, bool fill_other, uint8_t* stg, const float* ctab, LoadChunk&& load_chunk) {
    const RowCtx rc = make_row(P, tc, q * 32 + lane);
    float nz = 0.f;
    if (EPI == kEpiFwd && rc.valid && P.noise) nz = __ldg(P.noise + rc.n * P.noise_stride_n + rc.px_in_img) * P.noise_scale;
    float rgb0 = 0.f, rgb1 = 0.f, rgb2 = 0.f;
    const bool tk_valid = rc.valid && rc.pix < P.n_queries;
    const float clampv = P.act_clamp >= 0.f ? P.act_clamp : __int_as_float(0x7f800000);
    const float saved_thr = act_saved_clamp(P.act_clamp, P.split && P.lin_saved_lo);
    // staged stores: the lane re-reads 16-byte piece (lane & 3) of rows 8j + (lane >> 2), j = 0..3, so that
    // every store instruction writes whole 64-byte row segments (row-owner stores write 32 scattered pieces)
    long long srow[4];
    bool sok[4];
    if (kStaged) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const RowCtx r = make_row(P, tc, q * 32 + 8 * j + (lane >> 2));
            srow[j] = r.pix * P.n_total + (lane & 3) * 8;
            sok[j] = r.valid;
        }
    }
    auto flush_stage = [&](const uint8_t* tile, void* dst_base, int col0) {
        __syncwarp();
        __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(dst_base) + col0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int rr = 8 * j + (lane >> 2);
            const uint4 v = *reinterpret_cast<const uint4*>(tile + rr * 64 + ((((lane & 3) ^ (rr >> 1)) & 3) << 4));
            if (sok[j]) *reinterpret_cast<uint4*>(dst + srow[j]) = v;
        }
        __syncwarp();
    };

#pragma unroll 1
    for (int ch = ch_begin; ch < ch_end; ++ch) {
        float acc[32];
        load_chunk(ch, acc);
        if (P.dbg_skip_epi == 1) continue;
        const int col0 = tc.nblk * BN + ch * 32;
        const long long eoff = rc.pix * P.n_total + col0;             // element offset in [pixel][N] tensors
        const long long coff = static_cast<long long>(rc.n) * P.n_total + col0;   // offset in [batch][N] tensors
        if constexpr (EPI == kEpiRawF32) {
            if (rc.valid) {
                float4* dst = reinterpret_cast<float4*>(P.raw_out + eoff);
#pragma unroll
                for (int j = 0; j < 8; ++j) dst[j] = make_float4(acc[4 * j], acc[4 * j + 1], acc[4 * j + 2], acc[4 * j + 3]);
            }
        } else if constexpr (EPI == kEpiStoreBf16) {
            if (kStaged) {
                stage_bf16x32(stg, lane, acc);
                flush_stage(stg, P.x_hi, col0);
            } else if (rc.valid) {
                store_bf16x32(P.x_hi, P.split ? P.x_lo : nullptr, eoff, acc);
            }
        } else if constexpr (EPI == kEpiLinear) {
            if (rc.valid) {
                float t[32];
                if (P.lin_add) {
                    load_bf16x32(P.lin_add, eoff, t);
#pragma unroll
                    for (int j = 0; j < 32; ++j) acc[j] += t[j];
                    if (P.split) {
                        load_bf16x32(P.lin_add_lo, eoff, t);
#pragma unroll
                        for (int j = 0; j < 32; ++j) acc[j] += t[j];
                    }
                }
                if (P.lin_add_down) {       // gradient of the skip branch: 2 x 2 coarse pixels reach this fine pixel
                    const int vy = static_cast<int>(rc.px_in_img / P.OW), vx = static_cast<int>(rc.px_in_img - static_cast<long long>(vy) * P.OW);
                    const int Ho = P.OH >> 1, Wo = P.OW >> 1;
#pragma unroll
                    for (int ty = 0; ty < 2; ++ty) {
                        const int jy = ((vy + 1) & 1) + 2 * ty, my = vy + 1 - jy;
                        if (my < 0 || (my >> 1) >= Ho) continue;
#pragma unroll
                        for (int tx = 0; tx < 2; ++tx) {
                            const int jx = ((vx + 1) & 1) + 2 * tx, mx = vx + 1 - jx;
                            if (mx < 0 || (mx >> 1) >= Wo) continue;
                            const float wgt = P.lin_fir[jy * 4 + jx];
                            const long long doff = ((static_cast<long long>(rc.n) * Ho + (my >> 1)) * Wo + (mx >> 1)) * P.n_total + col0;
                            load_bf16x32(P.lin_add_down, doff, t);
#pragma unroll
                            for (int j = 0; j < 32; ++j) acc[j] = fmaf(wgt, t[j], acc[j]);
                            if (P.split) {
                                load_bf16x32(P.lin_add_down_lo, doff, t);
#pragma unroll
                                for (int j = 0; j < 32; ++j) acc[j] = fmaf(wgt, t[j], acc[j]);
                            }
                        }
                    }
                }
                if (P.lin_out) store_bf16x32(P.lin_out, P.split ? P.lin_out_lo : nullptr, eoff, acc);
                if (P.lin_gz || P.lin_rgb_w) {
                    load_bf16x32(P.lin_saved, eoff, t);
                    if (P.split && P.lin_saved_lo) {      // hi + lo, eight values at a time (no second 32-register row)
                        const uint4* s = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(P.lin_saved_lo) + eoff);
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const uint4 a = __ldg(s + q);
                            t[8 * q + 0] += bf16lo_f(a.x); t[8 * q + 1] += bf16hi_f(a.x);
                            t[8 * q + 2] += bf16lo_f(a.y); t[8 * q + 3] += bf16hi_f(a.y);
                            t[8 * q + 4] += bf16lo_f(a.z); t[8 * q + 5] += bf16hi_f(a.z);
                            t[8 * q + 6] += bf16lo_f(a.w); t[8 * q + 7] += bf16hi_f(a.w);
                        }
                    }
#pragma unroll
                    for (int j = 0; j < 32; ++j) acc[j] = act_grad(acc[j] * P.act_gain, t[j], P.act_slope, saved_thr);
                    if (P.lin_gz) store_bf16x32(P.lin_gz, P.split ? P.lin_gz_lo : nullptr, eoff, acc);
                    if (P.lin_rgb_w) {
                        const float4* w4 = reinterpret_cast<const float4*>(P.lin_rgb_w) + col0;
#pragma unroll
                        for (int j = 0; j < 32; ++j) {
                            const float4 w = __ldg(w4 + j);
                            rgb0 = fmaf(acc[j], w.x, rgb0);
                            rgb1 = fmaf(acc[j], w.y, rgb1);
                            rgb2 = fmaf(acc[j], w.z, rgb2);
                        }
                    }
                }
            }
        } else if constexpr (EPI == kEpiTopK) {
            // the two smallest scores of this row within the 32-code chunk, branch-free (a per-lane sorted insertion into a
            // deeper list diverges on almost every column and made this epilogue four times longer than the MMAs of its
            // tile); ties keep the lower code.  The exact re-rank rescans any chunk whose list may be incomplete.
            if (tk_valid) {
                const float INF = __int_as_float(0x7f800000);
                float m1 = INF, m2 = INF;
                int i1 = -1, i2 = -1;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const int code = col0 + j;
                    const float sc = code < P.n_codes ? fmaf(-2.f, acc[j], __ldg(P.code_sqnorm + code)) : INF;
                    const bool lt1 = sc < m1, lt2 = sc < m2;
                    m2 = lt1 ? m1 : (lt2 ? sc : m2);
                    i2 = lt1 ? i1 : (lt2 ? code : i2);
                    m1 = lt1 ? sc : m1;
                    i1 = lt1 ? code : i1;
                }
                const long long base = (rc.pix * (static_cast<long long>(P.n_blocks) * (BN / 32)) + tc.nblk * (BN / 32) + ch) * 2;
                *reinterpret_cast<float2*>(P.cand_score + base) = make_float2(m1, m2);
                *reinterpret_cast<int2*>(P.cand_idx + base) = make_int2(i1, i2);
            }
        } else if constexpr (EPI == kEpiMember) {
            // d = s^ - (T_j - |x|^2) with s^ = |y|^2 - 2<x,y>: d <= -margin is a definite hit, |d| <= margin ambiguous (the
            // exact recheck decides), anything else a definite miss.  T_j = +inf gives d = -inf: a hit.
            if (tk_valid) {
                const float xi = __ldg(P.query_sqnorm + rc.pix);
                const float ymax = __ldg(P.code_sqnorm + P.n_codes);
                const float eps = P.member_eps * sqrtf(xi) * sqrtf(ymax) + 6e-7f * (xi + ymax);
                bool hit = false;
                unsigned amb = 0u;
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const int code = col0 + j;
                    if (code < P.n_codes) {
                        const float4 t = __ldg(P.member_tab + code);
                        const float d = fmaf(-2.f, acc[j], t.x) - (t.y - xi);
                        const float mg = eps + t.z;
                        hit |= d <= -mg;
                        amb |= (d <= mg ? 1u : 0u) << j;
                    }
                }
                if (hit) {
                    P.member_hit[rc.pix] = 1;
                } else if (amb) {
                    int slot = atomicAdd(P.member_cnt + rc.pix, __popc(amb));
                    int* lst = P.member_list + rc.pix * P.member_cap;
                    while (amb && slot < P.member_cap) {
                        lst[slot++] = col0 + __ffs(amb) - 1;
                        amb &= amb - 1;
                    }
                }
            }
        } else if constexpr (EPI == kEpiFwd) {
            if (kStaged) {
                // staged path (one sample per tile): coefficients come from the warp group's shared-memory table
                const float4* t_dm = reinterpret_cast<const float4*>(ctab + ch * 32);
                const float4* t_bs = reinterpret_cast<const float4*>(ctab + 5 * BN + ch * 32);
#pragma unroll
                for (int j4 = 0; j4 < 8; ++j4) {
                    const float4 d4 = t_dm[j4], b4 = t_bs[j4];
                    const float dd[4] = {d4.x, d4.y, d4.z, d4.w}, bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        float z = fmaf(acc[4 * j4 + k], dd[k], nz) + bb[k];
                        z = fmaxf(z, z * P.act_slope) * P.act_gain;          // lrelu (slope < 1)
                        acc[4 * j4 + k] = fminf(fmaxf(z, -clampv), clampv);
                    }
                }
                stage_bf16x32(stg, lane, acc);
                flush_stage(stg, P.x_hi, col0);
                if (P.rgbw) {
                    const float4* t0 = reinterpret_cast<const float4*>(ctab + 2 * BN + ch * 32);
                    const float4* t1 = reinterpret_cast<const float4*>(ctab + 3 * BN + ch * 32);
                    const float4* t2 = reinterpret_cast<const float4*>(ctab + 4 * BN + ch * 32);
#pragma unroll
                    for (int j4 = 0; j4 < 8; ++j4) {
                        const float4 a4 = t0[j4], b4 = t1[j4], c4 = t2[j4];
                        rgb0 = fmaf(acc[4 * j4], a4.x, fmaf(acc[4 * j4 + 1], a4.y, fmaf(acc[4 * j4 + 2], a4.z, fmaf(acc[4 * j4 + 3], a4.w, rgb0))));
                        rgb1 = fmaf(acc[4 * j4], b4.x, fmaf(acc[4 * j4 + 1], b4.y, fmaf(acc[4 * j4 + 2], b4.z, fmaf(acc[4 * j4 + 3], b4.w, rgb1))));
                        rgb2 = fmaf(acc[4 * j4], c4.x, fmaf(acc[4 * j4 + 1], c4.y, fmaf(acc[4 * j4 + 2], c4.z, fmaf(acc[4 * j4 + 3], c4.w, rgb2))));
                    }
                }
                if (P.s_next) {
                    const float4* t_sn = reinterpret_cast<const float4*>(ctab + BN + ch * 32);
#pragma unroll
                    for (int j4 = 0; j4 < 8; ++j4) {
                        const float4 s4 = t_sn[j4];
                        acc[4 * j4] *= s4.x; acc[4 * j4 + 1] *= s4.y; acc[4 * j4 + 2] *= s4.z; acc[4 * j4 + 3] *= s4.w;
                    }
                    stage_bf16x32(stg, lane, acc);
                    flush_stage(stg, P.xs_hi, col0);
                }
            } else if (rc.valid) {
                float dm[32], bs[32];
                load_f32x32(P.demod + coff, dm);
                load_f32x32(P.bias + col0, bs);
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    float z = fmaf(acc[j], dm[j], nz) + bs[j];
                    z = fmaxf(z, z * P.act_slope) * P.act_gain;
                    acc[j] = fminf(fmaxf(z, -clampv), clampv);
                }
                store_bf16x32(P.x_hi, P.split ? P.x_lo : nullptr, eoff, acc);
                if (P.rgbw) {
                    const float4* rw = P.rgbw + coff;
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float4 w4 = __ldg(rw + j);
                        rgb0 = fmaf(acc[j], w4.x, rgb0);
                        rgb1 = fmaf(acc[j], w4.y, rgb1);
                        rgb2 = fmaf(acc[j], w4.z, rgb2);
                    }
                }
                if (P.s_next) {
                    load_f32x32(P.s_next + coff, dm);
#pragma unroll
                    for (int j = 0; j < 32; ++j) acc[j] *= dm[j];
                    store_bf16x32(P.xs_hi, P.split ? P.xs_lo : nullptr, eoff, acc);
                }
            }
        }
    }
    if (EPI == kEpiLinear && P.lin_rgb_w && rc.valid) {
        float* g = reinterpret_cast<float*>(P.lin_rgb_g + rc.pix);
        atomicAdd(g, rgb0); atomicAdd(g + 1, rgb1); atomicAdd(g + 2, rgb2);
    }
    if (EPI == kEpiFwd && P.rgbw && rc.valid) {   // one partial per (column block, slot): summed in fixed order later
        const long long plane = static_cast<long long>(P.batch) * P.OH * P.OW;
        P.rgb_part[(tc.nblk * 2 + part) * plane + rc.pix] = make_float4(rgb0, rgb1, rgb2, 0.f);
        if (fill_other) P.rgb_part[(tc.nblk * 2 + (part ^ 1)) * plane + rc.pix] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

// ---- column-owner backward epilogue, per warp.
// Per 32-column step: the lane (= row) moves its accumulator chunk TMEM -> registers -> the warp's
// 32x32 transpose tile; then lane (half = lane >> 4, cp = lane & 15) owns columns 2cp, 2cp+1 of the
// step and rows 16*half..+15, so the per-column coefficients sit in registers, global accesses are
// 64-byte row segments and the style-gradient column sums are plain per-thread accumulations that
// survive across tiles until the (sample, column block) key changes.  x_{l-1} of the NEXT step is
// prefetched into registers before the current step is computed.
template <int NSTEP>
struct BwdState {
    float racc[NSTEP][10];        // (red_s, red_d, red_rgb0..2) x 2 columns, per step slot
    int key;                      // ((sample * n_blocks + column block) * 8 + first step) of the accumulators, -1 = empty
    int nsteps;
};

template <int NSTEP>
__device__ __forceinline__ void bwd_state_init(BwdState<NSTEP>& st) {
#pragma unroll
    for (int c = 0; c < NSTEP; ++c)
#pragma unroll
        for (int k = 0; k < 10; ++k) st.racc[c][k] = 0.f;
    st.key = -1;
    st.nsteps = 0;
}

__device__ __forceinline__ float* red_base(const TapGemmParams& P, int kind) {
    return kind == 0 ? P.red_s : (kind == 1 ? P.red_d : P.red_rgb + static_cast<long long>(kind - 2) * P.batch * P.n_total);
}

template <int BN, int NSTEP>
__device__ __forceinline__ void bwd_flush(const TapGemmParams& P, BwdState<NSTEP>& st, int lane) {
    if (st.key >= 0) {
        const int cp = lane & 15;
        const int kinds = P.bwd_last ? 1 : (P.g_rgb ? 5 : 2);
        const int step0 = st.key & 7, nn = st.key >> 3;
        const int n = nn / P.n_blocks, nblk = nn - n * P.n_blocks;
#pragma unroll
        for (int c = 0; c < NSTEP; ++c)
#pragma unroll
            for (int k = 0; k < 10; ++k) {
                if (c < st.nsteps && (k >> 1) < kinds)
                    atomicAdd(red_base(P, k >> 1) + static_cast<long long>(n) * P.n_total + nblk * BN + (step0 + c) * 32 + 2 * cp + (k & 1),
                              st.racc[c][k]);
                st.racc[c][k] = 0.f;
            }
    }
    st.key = -1;
}

// One warp's share of one M tile in the backward epilogue.
struct BwdTile {
    TileCoord tc;
    int step0, nsteps;      // 32-column steps [step0, step0 + nsteps) of the column block
    int sub_tile;           // which M tile of its unit
};
struct BwdRowRegs {          // lane = row: what phase 0 loads for it
    unsigned off;
    float nz;
    float4 g;
};
__device__ __forceinline__ BwdRowRegs bwd_row_load(const TapGemmParams& P, const BwdTile& t, int q, int lane) {
    const RowCtx rc = make_row(P, t.tc, q * 32 + lane);
    BwdRowRegs r;
    r.off = rc.valid ? static_cast<unsigned>(rc.pix) * static_cast<unsigned>(P.n_total >> 1) : kRowMasked;
    r.nz = (rc.valid && P.noise_prev && !P.bwd_last)
               ? __ldg(P.noise_prev + rc.n * P.noise_prev_stride_n + rc.px_in_img) * P.noise_prev_scale : 0.f;
    r.g = (rc.valid && P.g_rgb) ? __ldg(P.g_rgb + rc.pix) : make_float4(0.f, 0.f, 0.f, 0.f);
    return r;
}
__device__ __forceinline__ void bwd_row_store(WarpSmem* ws, int buf, int lane, const BwdRowRegs& r) {
    ws->off[buf][lane] = r.off;
    ws->nz[buf][lane] = r.nz;
    ws->grgb[buf][lane] = r.g;
}
// x_{l-1} of one 32-column step: 16 rows of this half-warp, one bf16 pair per lane
template <int BN>
__device__ __forceinline__ void bwd_prefetch_x(const TapGemmParams& P, const WarpSmem* ws, int buf, const BwdTile& t, int slot, int lane,
                                               unsigned (&xu)[16]) {
    const unsigned* xph = reinterpret_cast<const unsigned*>(P.xp_hi) + ((t.tc.nblk * BN + (t.step0 + slot) * 32) >> 1) + (lane & 15);
    const unsigned* soff = ws->off[buf] + (lane >> 4) * 16;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const unsigned o = soff[i];
        xu[i] = __ldg(xph + (o == kRowMasked ? 0u : o));
        if (o == kRowMasked) xu[i] = 0u;
    }
}

// `xa` holds x_{l-1} of the tile's first step on entry (prefetched while the previous tile was computed) and
// that of `next`'s first step on exit; the row data of `next` goes to ws buffer buf ^ 1.
template <int BN, int NSTEP, bool kSplit, class LoadChunk, class Release>
__device__ __forceinline__ void bwd_warp_tile(const TapGemmParams& P, const BwdTile& cur, const BwdTile* next, int q, int lane, WarpSmem* ws,
                                              int buf, BwdState<NSTEP>& st, unsigned (&xa)[16], LoadChunk&& load_chunk, Release&& release_acc) {
    const TileCoord& tc = cur.tc;
    const int step0 = cur.step0, nsteps = cur.nsteps;
    const int half = lane >> 4, cp = lane & 15;
    // loads of the NEXT tile's row data are issued now and parked in registers until the last step
    BwdRowRegs nrow;
    if (next) nrow = bwd_row_load(P, *next, q, lane);
    const bool row_valid = ws->off[buf][lane] != kRowMasked;
    const bool any_invalid = __any_sync(0xffffffffu, !row_valid);
    // sample of this half-warp's 16 rows (a half never straddles two samples: box_px is 16, 64 or 128)
    const int box_px = P.th * P.tw;
    const int ni_h = (q * 32 + half * 16) / box_px;
    const int n_h = tc.n0 + ni_h;
    const bool n_ok = ni_h < P.nb && n_h < P.batch;
    const int new_key = n_ok ? ((n_h * P.n_blocks + tc.nblk) * 8 + step0) : -1;
    if (new_key != st.key) {
        bwd_flush<BN, NSTEP>(P, st, lane);
        st.key = new_key;
        st.nsteps = 0;
    }
    // the accumulators of a key live across tiles whose step counts differ (a two-tile unit gives the warp all steps of its
    // tile, a single-tile unit -- the odd tile at the end of a CTA's range -- only half of them): flush the widest seen
    if (n_ok && nsteps > st.nsteps) st.nsteps = nsteps;

    const float inv_gain = 1.f / P.act_gain, inv_gain_slope = 1.f / (P.act_gain * P.act_slope);
    const float saved_thr = act_saved_clamp(P.act_clamp, kSplit);
    const bool last = P.bwd_last != 0;        // x_{l-1} is the constant input: only red_s is wanted (coefficients stay 0, no store)
    const unsigned* soff = ws->off[buf] + half * 16;
    const float* snz = ws->nz[buf] + half * 16;
    const float4* sgr = ws->grgb[buf] + half * 16;
    const float* strans = ws->trans + half * 16 * kTransStride + 2 * cp;
    const int colp0 = ((tc.nblk * BN + step0 * 32) >> 1) + cp;      // column pair of step slot 0

    // One 32-column step, branch-free over its 16 rows (masked rows carry a == x == g_rgb == 0 and only
    // their store is predicated off), so the compiler interleaves the rows.
    auto step_body = [&](auto rgb_tag, int c, float (&r)[10]) {
        constexpr bool kRgb = decltype(rgb_tag)::value;
        const int col = tc.nblk * BN + (step0 + c) * 32 + 2 * cp;
        const long long coff = static_cast<long long>(n_h) * P.n_total + col;
        float2 sc = make_float2(0.f, 0.f), dm = sc, bs = sc;
        float4 rw0 = make_float4(0.f, 0.f, 0.f, 0.f), rw1 = rw0;
        if (!last && n_ok) {
            sc = __ldg(reinterpret_cast<const float2*>(P.s_cur + coff));
            dm = __ldg(reinterpret_cast<const float2*>(P.demod_prev + coff));
            bs = __ldg(reinterpret_cast<const float2*>(P.bias_prev + col));
            sc.x *= P.act_gain; sc.y *= P.act_gain;               // activation gain folded into the coefficients
            if (kRgb) {
                rw0 = __ldg(P.rgbw_prev + coff); rw1 = __ldg(P.rgbw_prev + coff + 1);
                rw0.x *= P.act_gain; rw0.y *= P.act_gain; rw0.z *= P.act_gain;
                rw1.x *= P.act_gain; rw1.y *= P.act_gain; rw1.z *= P.act_gain;
            }
        }
        unsigned* gy_step = reinterpret_cast<unsigned*>(P.gy_hi) + (colp0 + c * 16);
        unsigned* gyl_step = kSplit ? reinterpret_cast<unsigned*>(P.gy_lo) + (colp0 + c * 16) : nullptr;
        unsigned xl[16];
        if (kSplit) {
            const unsigned* xpl = reinterpret_cast<const unsigned*>(P.xp_lo) + (colp0 + c * 16);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const unsigned o = soff[i];
                xl[i] = __ldg(xpl + (o == kRowMasked ? 0u : o));
                if (o == kRowMasked) xl[i] = 0u;
            }
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const unsigned o = soff[i];
            const float2 a = *reinterpret_cast<const float2*>(strans + i * kTransStride);
            float x0 = bf16lo_f(xa[i]), x1 = bf16hi_f(xa[i]);
            if (kSplit) { x0 += bf16lo_f(xl[i]); x1 += bf16hi_f(xl[i]); }
            r[0] = fmaf(a.x, x0, r[0]);
            r[1] = fmaf(a.y, x1, r[1]);
            float g0 = a.x * sc.x, g1 = a.y * sc.y;
            if (kRgb) {
                const float4 g = sgr[i];
                g0 = fmaf(g.x, rw0.x, fmaf(g.y, rw0.y, fmaf(g.z, rw0.z, g0)));
                g1 = fmaf(g.x, rw1.x, fmaf(g.y, rw1.y, fmaf(g.z, rw1.z, g1)));
                r[4] = fmaf(x0, g.x, r[4]); r[5] = fmaf(x1, g.x, r[5]);
                r[6] = fmaf(x0, g.y, r[6]); r[7] = fmaf(x1, g.y, r[7]);
                r[8] = fmaf(x0, g.z, r[8]); r[9] = fmaf(x1, g.z, r[9]);
            }
            const float nz = snz[i];
            // activation backward of layer l-1 decided by its saved output; y recovered from it
            const bool p0 = x0 > 0.f, p1 = x1 > 0.f;
            const float gz0 = act_grad(g0, x0, P.act_slope, saved_thr), gz1 = act_grad(g1, x1, P.act_slope, saved_thr);
            const float z0 = x0 * (p0 ? inv_gain : inv_gain_slope), z1 = x1 * (p1 ? inv_gain : inv_gain_slope);
            r[2] = fmaf(gz0, z0 - (nz + bs.x), r[2]);
            r[3] = fmaf(gz1, z1 - (nz + bs.y), r[3]);
            const float y0 = gz0 * dm.x, y1 = gz1 * dm.y;
            const bool st_ok = o != kRowMasked && !last;
            st_global_if(gy_step + o, pack_bf16(y0, y1), st_ok);
            if (kSplit) st_global_if(gyl_step + o, pack_bf16(y0 - bf16_round(y0), y1 - bf16_round(y1)), st_ok);
        }
    };

    unsigned xb[16];
#pragma unroll 1
    for (int c = 0; c < nsteps; ++c) {       // (a runtime loop: unrolled, the epilogue outgrows the instruction cache)
        {
            float acc[32];
            load_chunk(step0 + c, acc);
            if (c == nsteps - 1) release_acc();
            if (P.dbg_skip_epi) continue;
            if (any_invalid && !row_valid) {
#pragma unroll
                for (int j = 0; j < 32; ++j) acc[j] = 0.f;
            }
            float4* dst = reinterpret_cast<float4*>(ws->trans + lane * kTransStride);
#pragma unroll
            for (int j = 0; j < 8; ++j) dst[j] = make_float4(acc[4 * j], acc[4 * j + 1], acc[4 * j + 2], acc[4 * j + 3]);
        }
        if (c == nsteps - 1 && next) bwd_row_store(ws, buf ^ 1, lane, nrow);
        __syncwarp();
        if (c + 1 < nsteps) bwd_prefetch_x<BN>(P, ws, buf, cur, c + 1, lane, xb);
        else if (next) bwd_prefetch_x<BN>(P, ws, buf ^ 1, *next, 0, lane, xb);
        float r[10];
#pragma unroll
        for (int k = 0; k < 10; ++k) r[k] = 0.f;
        if (P.g_rgb && !last) step_body(std::true_type{}, c, r);
        else step_body(std::false_type{}, c, r);
#pragma unroll
        for (int cc = 0; cc < NSTEP; ++cc)
            if (cc == c) {
#pragma unroll
                for (int k = 0; k < 10; ++k) st.racc[cc][k] += r[k];
            }
        __syncwarp();           // the transpose tile may be overwritten from here on
#pragma unroll
        for (int i = 0; i < 16; ++i) xa[i] = xb[i];
    }
}

// Driver of the backward epilogue for one warp: walks the CTA's units with one-tile lookahead.
// get_tile(t, out_tile, out_advance) -> false at the end of the range.
template <int BN, int NSTEP, bool kSplit, class TileAt, class LoadChunkFor, class ReleaseFor>
__device__ __forceinline__ void bwd_warp_loop(const TapGemmParams& P, int q, int lane, WarpSmem* ws, int t_begin, int t_end, TileAt&& tile_at,
                                              LoadChunkFor&& chunk_loader, ReleaseFor&& releaser) {
    BwdState<NSTEP> st;
    bwd_state_init(st);
    BwdTile cur, nxt;
    int adv = 0;
    int t = t_begin;
    if (t >= t_end) return;
    tile_at(t, cur, adv);
    int buf = 0;
    bwd_row_store(ws, buf, lane, bwd_row_load(P, cur, q, lane));
    __syncwarp();
    unsigned xa[16];
    bwd_prefetch_x<BN>(P, ws, buf, cur, 0, lane, xa);
    int it = 0;
    while (t < t_end) {
        const int tn = t + adv;
        int adv_n = 0;
        const bool has_next = tn < t_end;
        if (has_next) tile_at(tn, nxt, adv_n);
        bwd_warp_tile<BN, NSTEP, kSplit>(P, cur, has_next ? &nxt : nullptr, q, lane, ws, buf, st, xa, chunk_loader(it, cur), releaser(it));
        cur = nxt; adv = adv_n; t = tn; buf ^= 1; ++it;
    }
    bwd_flush<BN, NSTEP>(P, st, lane);
}

// Work split of the 8 epilogue warps over a unit: with two M tiles, warps 0-3 take tile 0 and warps 4-7
// tile 1 (all columns); with one, the two warp groups split its columns.
template <int BN>
struct EpiSplit {
    int st;            // which M tile of the unit
    int ch_begin, ch_end;   // 32-column chunks
    bool whole;        // the warp covers the whole column block
};
template <int BN>
__device__ __forceinline__ EpiSplit<BN> epi_split(int mt, int sub) {
    constexpr int NCH = BN / 32;
    EpiSplit<BN> s;
    if (mt == 2) { s.st = sub; s.ch_begin = 0; s.ch_end = NCH; s.whole = true; }
    else { s.st = 0; s.ch_begin = sub * (NCH / 2); s.ch_end = (sub + 1) * (NCH / 2); s.whole = false; }
    return s;
}

// ------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long global_timer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

template <int BN, int EPI, bool kPair>
__global__ void __launch_bounds__(kThreads, 1) tapgemm_kernel(const __grid_constant__ TapGemmParams P) {
    using C = Cfg<BN, EPI, kPair>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // pointer arithmetic keeps the shared address space
    uint8_t* a_smem = smem;
    uint8_t* b_smem = smem + C::kAStages * C::kASlotBytes;
    uint8_t* epi_smem = b_smem + C::kBRing * C::kBSlotBytes;
    constexpr int kMaxAStages = 8;
    uint64_t* a_full = reinterpret_cast<uint64_t*>(epi_smem + C::kEpiSmemBytes);
    uint64_t* a_empty = a_full + kMaxAStages;
    uint64_t* b_full = a_empty + kMaxAStages;
    uint64_t* b_empty = b_full + C::kBRing;
    uint64_t* tfull_bar = b_empty + C::kBRing;
    uint64_t* tempty_bar = tfull_bar + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);
    static_assert((2 * kMaxAStages + 2 * C::kBRing + 4) * 8 + 4 <= 512, "barrier area");
    // A ring: slots of one M tile when the launch never pairs tiles (twice as many stages in flight)
    constexpr bool pair = kPair;                                    // CTA pair: M = 256 MMAs issued by cluster rank 0
    uint32_t rank = 0u;
    if constexpr (kPair) rank = cluster_ctarank();
    const int a_slot_bytes = (C::kMtMax == 2 && !(pair ? P.no_quad : P.no_pair)) ? 2 * kASubBytes : kASubBytes;
    const int a_stages = min(kMaxAStages, C::kABytes / a_slot_bytes);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    int t_begin, t_end;
    if (pair) tile_range(P, t_begin, t_end, static_cast<int>(blockIdx.x >> 1), static_cast<int>(gridDim.x >> 1));
    else tile_range(P, t_begin, t_end);
    auto unit_at = [&](int t) { return get_unit<C::kMtMax>(P, t, t_end); };                    // single-CTA launches
    auto pair_at = [&](int t) { return get_pair_work<C::kMtMax>(P, t, t_end); };                // CTA-pair launches
    unsigned long long dbg_c0 = 0, dbg_t0 = 0;
    if (P.dbg_clock && blockIdx.x == 0 && threadIdx.x == 64) {
        dbg_c0 = clock64();
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(dbg_t0));
    }

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&P.a_map[0]);
        prefetch_tmap(&P.b_map);
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < kMaxAStages; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], 1); }
        for (int s = 0; s < C::kBRing; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1); }
        for (int a = 0; a < 2; ++a) {
            mbar_init(&tfull_bar[a], 1);
            mbar_init(&tempty_bar[a], (pair ? 2 : 1) * (kEpiThreads / 32));      // (pair: the peer's warps arrive on the leader's)
        }
        fence_barrier_init();
    }
    if (warp == 2) {
        if constexpr (kPair) tmem_alloc_pair<C::kTmemCols>(tmem_slot);
        else tmem_alloc<C::kTmemCols>(tmem_slot);
    }
    tc_fence_before();
    if constexpr (kPair) cluster_sync_all();       // the peer's barriers must be initialised before anything arrives on them
    else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const uint32_t a_tx_bytes = static_cast<uint32_t>(P.nb * (P.th + P.halo) * P.tw) * 128u;
    const uint32_t dy_bytes = static_cast<uint32_t>(P.tw) * 128u;      // one tile row of pixels (1024 B when halo > 0)

    if (warp < 4) {
        setmaxnreg_dec<kRegsProducer>();
        if (warp == 0) {
            // ---------------------------------------------------------------- TMA producer of the A ring (whole warp, one elected lane issues)
            // (the two rings have separate producer threads: at 128^2 and 256^2 the activations come from DRAM with
            // 2-3 us of latency while the weights sit in L2 -- one thread issuing both in order stalls the A stream on
            // the shallow B ring and leaves most of the A ring empty)
            int as = 0;
            uint32_t aph = 0;
            const bool dbg = P.dbg_clock && blockIdx.x == 0 && lane == 0;
            int dbg_step = 0;
            for (int t = t_begin; t < t_end;) {
                Unit u;
                TileCoord tc0, tc1;          // pair: this CTA's own M tile(s)
                int nsub = 1;
                if constexpr (kPair) {
                    const PairWork w = pair_at(t);
                    t += w.adv;
                    u = w.a;
                    nsub = w.nsub;
                    tc0 = pair_tile(w.a, rank);
                    tc1 = pair_tile(w.b, rank);
                } else {
                    u = unit_at(t);
                    t += u.adv;
                    if (u.mt == 0) continue;
                    tc0 = u.tc0; tc1 = u.tc1;
                }
                const TapProblem& pr = P.prob[tc0.prob];
                for (int g = 0; g < pr.ngroups; ++g) {
                    const TapGroup grp = P.groups[pr.grp_begin + g];
                    const CUtensorMap* amap = &P.a_map[grp.src];
                    for (int kc = 0; kc < P.kchunks; ++kc) {
                        mbar_wait(&a_empty[as], aph ^ 1, P.err_flag, 1);
                        if (dbg && dbg_step < 28) P.dbg_clock[8 + 2 * dbg_step++] = global_timer_ns();
                        uint8_t* sa = a_smem + as * a_slot_bytes;
                        if (elect_one()) {
                            if constexpr (kPair) {
                                // all bytes of the pair are counted on the LEADER's barrier; it alone posts the expected total
                                const uint32_t lead = mapa_shared(smem_u32(&a_full[as]), 0);
                                if (rank == 0) mbar_expect_tx(&a_full[as], 2 * nsub * a_tx_bytes);
                                tma_load_4d_pair(sa, amap, lead, kc * kBlockK, tc0.w0 + grp.dx, tc0.h0 + grp.dy0, tc0.n0);
                                if (nsub == 2) tma_load_4d_pair(sa + kASubBytes, amap, lead, kc * kBlockK, tc1.w0 + grp.dx, tc1.h0 + grp.dy0, tc1.n0);
                            } else {
                                mbar_expect_tx(&a_full[as], a_tx_bytes * u.mt);
                                tma_load_4d(sa, amap, &a_full[as], kc * kBlockK, tc0.w0 + grp.dx, tc0.h0 + grp.dy0, tc0.n0);
                                if (u.mt == 2) tma_load_4d(sa + kASubBytes, amap, &a_full[as], kc * kBlockK, tc1.w0 + grp.dx, tc1.h0 + grp.dy0, tc1.n0);
                            }
                        }
                        __syncwarp();
                        if (++as == a_stages) { as = 0; aph ^= 1; }
                    }
                }
            }
        } else if (warp == 3) {
            // ---------------------------------------------------------------- TMA producer of the B ring (whole warp, one elected lane issues)
            int bs = 0;
            uint32_t bph = 0;
            const int b_row0 = kPair ? static_cast<int>(rank) * (BN / 2) : 0;      // (pair: this CTA's half of the column block)
            for (int t = t_begin; t < t_end;) {
                Unit u;
                if constexpr (kPair) {
                    const PairWork w = pair_at(t);
                    t += w.adv;
                    u = w.a;
                } else {
                    u = unit_at(t);
                    t += u.adv;
                    if (u.mt == 0) continue;
                }
                const TapProblem& pr = P.prob[u.tc0.prob];
                for (int g = 0; g < pr.ngroups; ++g) {
                    const TapGroup grp = P.groups[pr.grp_begin + g];
                    for (int kc = 0; kc < P.kchunks; ++kc) {
                        for (int j = 0; j < grp.ntaps; ++j) {
                            mbar_wait(&b_empty[bs], bph ^ 1, P.err_flag, 5);
                            uint8_t* sb = b_smem + bs * C::kBSlotBytes;
                            if (elect_one()) {
                                if constexpr (kPair) {
                                    if (rank == 0) mbar_expect_tx(&b_full[bs], C::kBBytes);
                                    tma_load_3d_pair(sb, &P.b_map, mapa_shared(smem_u32(&b_full[bs]), 0), kc * kBlockK, u.tc0.nblk * BN + b_row0,
                                                     P.gwidx[grp.tap_begin + j]);
                                } else {
                                    mbar_expect_tx(&b_full[bs], C::kBBytes);
                                    tma_load_3d(sb, &P.b_map, &b_full[bs], kc * kBlockK, u.tc0.nblk * BN, P.gwidx[grp.tap_begin + j]);
                                }
                            }
                            __syncwarp();
                            if (++bs == C::kBRing) { bs = 0; bph ^= 1; }
                        }
                    }
                }
            }
        } else if (kPair && warp == 1) {
            // ---------------------------------------------------------------- MMA issuer of a CTA pair (leader only)
            // (the whole warp walks the loop so that control flow and descriptors stay warp-uniform; one elected
            // lane issues -- a single diverged lane makes the compiler wrap every MMA in a broadcast loop)
            if (rank == 0) {
                constexpr uint32_t idesc2 = make_idesc_bf16(2 * kBlockM, BN);
                int as = 0, bs = 0;
                uint32_t aph = 0, bph = 0;
                int acc = 0;
                uint32_t acc_phase = 0;
                const bool dbg = P.dbg_clock && blockIdx.x == 0 && lane == 0;
                int dbg_units = 0, dbg_step = 0;
                unsigned long long dbg_wait_acc = 0, dbg_wait_a = 0, dbg_wait_b = 0, w0 = 0;
                if (dbg) P.dbg_clock[2] = global_timer_ns();
                for (int t = t_begin; t < t_end;) {
                    const PairWork w = pair_at(t);
                    t += w.adv;
                    const int nsub = w.nsub;
                    const TapProblem& pr = P.prob[w.a.tc0.prob];
                    if (dbg) w0 = global_timer_ns();
                    mbar_wait(&tempty_bar[acc], acc_phase ^ 1, P.err_flag, 2);
                    if (dbg) dbg_wait_acc += global_timer_ns() - w0;
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * C::kMtMax * BN);
                    bool first = true;
                    for (int g = 0; g < pr.ngroups; ++g) {
                        const TapGroup grp = P.groups[pr.grp_begin + g];
                        for (int kc = 0; kc < P.kchunks; ++kc) {
                            if (dbg) w0 = global_timer_ns();
                            mbar_wait(&a_full[as], aph, P.err_flag, 3);
                            if (dbg) dbg_wait_a += global_timer_ns() - w0;
                            if (dbg && dbg_step < 28) P.dbg_clock[9 + 2 * dbg_step++] = global_timer_ns();
                            const uint32_t sa = smem_u32(a_smem + as * a_slot_bytes);
                            for (int j = 0; j < grp.ntaps; ++j) {
                                if (dbg) w0 = global_timer_ns();
                                mbar_wait(&b_full[bs], bph, P.err_flag, 6);
                                if (dbg) dbg_wait_b += global_timer_ns() - w0;
                                tc_fence_after();
                                if (dbg && first && dbg_units == 0) P.dbg_clock[3] = global_timer_ns();
                                const uint64_t bdesc = make_sw128_kmajor_desc(smem_u32(b_smem + bs * C::kBSlotBytes));
                                const uint32_t a_tap = sa + P.gdyrel[grp.tap_begin + j] * dy_bytes;
                                if (elect_one()) {
                                    for (int sb = 0; sb < nsub; ++sb) {
                                        const uint64_t adesc = make_sw128_kmajor_desc(a_tap + sb * kASubBytes);
#pragma unroll
                                        for (int k = 0; k < kBlockK / 16; ++k)
                                            umma_bf16_pair(d_tmem + static_cast<uint32_t>(sb * BN), adesc + static_cast<uint64_t>(k * 2),
                                                           bdesc + static_cast<uint64_t>(k * 2), idesc2, (first && k == 0) ? 0u : 1u);
                                    }
                                    umma_commit_pair(&b_empty[bs]);
                                }
                                __syncwarp();
                                first = false;
                                if (++bs == C::kBRing) { bs = 0; bph ^= 1; }
                            }
                            if (elect_one()) umma_commit_pair(&a_empty[as]);
                            __syncwarp();
                            if (++as == a_stages) { as = 0; aph ^= 1; }
                        }
                    }
                    if (elect_one()) umma_commit_pair(&tfull_bar[acc]);
                    __syncwarp();
                    if (dbg && dbg_units++ == 0) P.dbg_clock[4] = global_timer_ns();
                    if (++acc == 2) { acc = 0; acc_phase ^= 1; }
                }
                if (dbg) {
                    P.dbg_clock[5] = global_timer_ns(); P.dbg_clock[6] = static_cast<unsigned long long>(dbg_units);
                    P.dbg_clock[60] = dbg_wait_acc; P.dbg_clock[61] = dbg_wait_a; P.dbg_clock[62] = dbg_wait_b;
                }
            }
        } else if (warp == 1) {
            // ---------------------------------------------------------------- MMA issuer (whole warp, one elected lane issues)
            constexpr uint32_t idesc = make_idesc_bf16(kBlockM, BN);
            int as = 0, bs = 0;
            uint32_t aph = 0, bph = 0;
            int acc = 0;
            uint32_t acc_phase = 0;
            const bool dbg = P.dbg_clock && blockIdx.x == 0 && lane == 0;
            int dbg_units = 0, dbg_step = 0;
            unsigned long long dbg_wait_acc = 0, dbg_wait_a = 0, dbg_wait_b = 0;
            if (dbg) P.dbg_clock[2] = global_timer_ns();
            for (int t = t_begin; t < t_end;) {
                const Unit u = get_unit<C::kMtMax>(P, t, t_end);
                t += u.adv;
                if (u.mt == 0) continue;
                const TapProblem& pr = P.prob[u.tc0.prob];
                unsigned long long w0 = dbg ? global_timer_ns() : 0ull;
                mbar_wait(&tempty_bar[acc], acc_phase ^ 1, P.err_flag, 2);
                if (dbg) dbg_wait_acc += global_timer_ns() - w0;
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * C::kMtMax * BN);
                bool first = true;
                for (int g = 0; g < pr.ngroups; ++g) {
                    const TapGroup grp = P.groups[pr.grp_begin + g];
                    for (int kc = 0; kc < P.kchunks; ++kc) {
                        w0 = dbg ? global_timer_ns() : 0ull;
                        mbar_wait(&a_full[as], aph, P.err_flag, 3);
                        if (dbg) dbg_wait_a += global_timer_ns() - w0;
                        if (dbg && dbg_step < 28) P.dbg_clock[9 + 2 * dbg_step++] = global_timer_ns();
                        const uint32_t sa = smem_u32(a_smem + as * a_slot_bytes);
                        for (int j = 0; j < grp.ntaps; ++j) {
                            w0 = dbg ? global_timer_ns() : 0ull;
                            mbar_wait(&b_full[bs], bph, P.err_flag, 6);
                            if (dbg) dbg_wait_b += global_timer_ns() - w0;
                            tc_fence_after();
                            if (dbg && first && dbg_units == 0) P.dbg_clock[3] = global_timer_ns();
                            const uint64_t bdesc = make_sw128_kmajor_desc(smem_u32(b_smem + bs * C::kBSlotBytes));
                            const uint32_t a_tap = sa + P.gdyrel[grp.tap_begin + j] * dy_bytes;
                            if (elect_one()) {
                                for (int s = 0; s < u.mt; ++s) {
                                    const uint64_t adesc = make_sw128_kmajor_desc(a_tap + s * kASubBytes);
#pragma unroll
                                    for (int k = 0; k < kBlockK / 16; ++k)
                                        umma_bf16(d_tmem + static_cast<uint32_t>(s * BN), adesc + static_cast<uint64_t>(k * 2),
                                                  bdesc + static_cast<uint64_t>(k * 2), idesc, (first && k == 0) ? 0u : 1u);
                                }
                                umma_commit(&b_empty[bs]);
                            }
                            __syncwarp();
                            first = false;
                            if (++bs == C::kBRing) { bs = 0; bph ^= 1; }
                        }
                        if (elect_one()) umma_commit(&a_empty[as]);
                        __syncwarp();
                        if (++as == a_stages) { as = 0; aph ^= 1; }
                    }
                }
                if (elect_one()) umma_commit(&tfull_bar[acc]);
                __syncwarp();
                if (dbg && dbg_units++ == 0) P.dbg_clock[4] = global_timer_ns();
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
            if (dbg) {
                P.dbg_clock[5] = global_timer_ns(); P.dbg_clock[6] = static_cast<unsigned long long>(dbg_units);
                P.dbg_clock[60] = dbg_wait_acc; P.dbg_clock[61] = dbg_wait_a; P.dbg_clock[62] = dbg_wait_b;
            }
        }
    } else {
        // -------------------------------------------------------------------- epilogue (8 independent warps)
        setmaxnreg_inc<kRegsEpilogue>();
        const int e = warp - 4;
        const int q = e & 3, sub = e >> 2;          // TMEM lane quarter (= warp % 4), warp group
        if constexpr (EPI == kEpiBwd) {
            WarpSmem* ws = reinterpret_cast<WarpSmem*>(epi_smem) + e;
            const uint32_t tempty_lead[2] = {pair ? mapa_shared(smem_u32(&tempty_bar[0]), 0) : 0u, pair ? mapa_shared(smem_u32(&tempty_bar[1]), 0) : 0u};
            auto tile_at = [&](int t, BwdTile& bt, int& adv) {
                EpiSplit<BN> sp;
                if constexpr (kPair) {
                    const PairWork w = pair_at(t);
                    sp = epi_split<BN>(w.nsub, sub);
                    bt.tc = pair_tile(sp.st ? w.b : w.a, rank);
                    adv = w.adv;
                } else {
                    const Unit u = unit_at(t);     // (the backward GEMMs are single-problem: never empty)
                    sp = epi_split<BN>(u.mt, sub);
                    bt.tc = u.tile(sp.st);
                    adv = u.adv;
                }
                bt.step0 = sp.ch_begin; bt.nsteps = sp.ch_end - sp.ch_begin; bt.sub_tile = sp.st;
            };
            auto chunk_loader = [&](int it, const BwdTile& bt) {
                const int acc = it & 1;
                const uint32_t ph = static_cast<uint32_t>(it >> 1) & 1u;
                const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) +
                                        static_cast<uint32_t>((acc * C::kMtMax + bt.sub_tile) * BN);
                uint64_t* bar = &tfull_bar[acc];
                int* err = P.err_flag;
                bool waited = false;
                return [=](int ch, float (&v)[32]) mutable {
                    if (!waited) {       // the row-data phase runs before this wait
                        mbar_wait(bar, ph, err, 4);
                        tc_fence_after();
                        waited = true;
                    }
                    uint32_t r[32];
                    tmem_ld32(t_addr + ch * 32, r);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
                };
            };
            auto releaser = [&](int it) {
                uint64_t* bar = &tempty_bar[it & 1];
                const uint32_t lead = tempty_lead[it & 1];
                const bool remote = pair && rank != 0;
                return [=]() {
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) {
                        if (remote) mbar_arrive_cluster(lead);
                        else mbar_arrive(bar);
                    }
                };
            };
            if (P.split) bwd_warp_loop<BN, C::kBwdSteps, true>(P, q, lane, ws, t_begin, t_end, tile_at, chunk_loader, releaser);
            else bwd_warp_loop<BN, C::kBwdSteps, false>(P, q, lane, ws, t_begin, t_end, tile_at, chunk_loader, releaser);
        } else {
            int acc = 0;
            uint32_t acc_phase = 0;
            int coef_key = -1;
            for (int t = t_begin; t < t_end;) {
                EpiSplit<BN> sp;
                TileCoord tc;
                if constexpr (kPair) {
                    const PairWork w = pair_at(t);
                    t += w.adv;
                    sp = epi_split<BN>(w.nsub, sub);
                    tc = pair_tile(sp.st ? w.b : w.a, rank);
                } else {
                    const Unit u = unit_at(t);
                    t += u.adv;
                    if (u.mt == 0) continue;
                    sp = epi_split<BN>(u.mt, sub);
                    tc = u.tile(sp.st);
                }
                const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) +
                                        static_cast<uint32_t>((acc * C::kMtMax + sp.st) * BN);
                bool waited = false;
                auto load_chunk = [&](int ch, float (&v)[32]) {
                    if (!waited) {
                        mbar_wait(&tfull_bar[acc], acc_phase, P.err_flag, 4);
                        tc_fence_after();
                        waited = true;
                    }
                    uint32_t r[32];
                    tmem_ld32(t_addr + ch * 32, r);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
                };
                uint8_t* stg = epi_smem + e * (2048 * C::kStageTensors);
                if (C::kStageTensors > 0 && P.staged) {
                    const float* ctab = nullptr;
                    if constexpr (EPI == kEpiFwd) {
                        // (re)fill the warp group's coefficient table when the (sample, column block) changes
                        float* tab = reinterpret_cast<float*>(epi_smem + 8 * 2048 * C::kStageTensors) + sub * (6 * BN);
                        const int key = tc.n0 * P.n_blocks + tc.nblk;
                        if (key != coef_key) {
                            asm volatile("bar.sync %0, 128;" ::"r"(1 + sub) : "memory");       // the group is done with the old table
                            const long long cb = static_cast<long long>(tc.n0) * P.n_total + tc.nblk * BN;
                            for (int i = q * 32 + lane; i < BN; i += 128) {
                                tab[i] = __ldg(P.demod + cb + i);
                                tab[BN + i] = P.s_next ? __ldg(P.s_next + cb + i) : 0.f;
                                const float4 w4 = P.rgbw ? __ldg(P.rgbw + cb + i) : make_float4(0.f, 0.f, 0.f, 0.f);
                                tab[2 * BN + i] = w4.x; tab[3 * BN + i] = w4.y; tab[4 * BN + i] = w4.z;
                                tab[5 * BN + i] = __ldg(P.bias + tc.nblk * BN + i);
                            }
                            asm volatile("bar.sync %0, 128;" ::"r"(1 + sub) : "memory");
                            coef_key = key;
                        }
                        ctab = tab;
                    }
                    rowowner_warp_tile<BN, EPI, (C::kStageTensors > 0)>(P, tc, q, lane, sp.ch_begin, sp.ch_end, sp.whole ? 0 : sub, sp.whole, stg, ctab, load_chunk);
                } else {
                    rowowner_warp_tile<BN, EPI, false>(P, tc, q, lane, sp.ch_begin, sp.ch_end, sp.whole ? 0 : sub, sp.whole, nullptr, nullptr, load_chunk);
                }
                if (!waited) {            // (a tile with every row masked may never have touched its accumulator)
                    mbar_wait(&tfull_bar[acc], acc_phase, P.err_flag, 4);
                    tc_fence_after();
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if (pair && rank != 0) mbar_arrive_cluster(mapa_shared(smem_u32(&tempty_bar[acc]), 0));
                    else mbar_arrive(&tempty_bar[acc]);
                }
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    }

    tc_fence_before();
    if constexpr (kPair) cluster_sync_all();       // no CTA may leave while its partner still arrives on its barriers or reads its operands
    else __syncthreads();
    if (P.dbg_clock && blockIdx.x == 0 && threadIdx.x == 64) {
        unsigned long long t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        P.dbg_clock[0] = clock64() - dbg_c0;
        P.dbg_clock[1] = t1 - dbg_t0;
        P.dbg_clock[7] = dbg_t0;
    }
    if (warp == 2) {
        if constexpr (kPair) tmem_dealloc_pair<C::kTmemCols>(tmem_base);
        else tmem_dealloc<C::kTmemCols>(tmem_base);
    }
}

// ------------------------------------------------------------------------------------
// SIMT twin: 8 warps with the SAME roles and the same epilogue code as the epilogue warps of the
// tensor-core kernel; the accumulator chunk is computed by brute force from the flat tap list.
// Debug cross-check of the tensor-core path (tests), never a fallback.
template <int BN, int EPI>
__global__ void __launch_bounds__(kEpiThreads) tapgemm_simt_kernel(const __grid_constant__ TapGemmParams P,
                                                                   const TapSimtOperands ops) {
    using C = Cfg<BN, EPI>;
    __shared__ WarpSmem wsm[EPI == kEpiBwd ? 8 : 1];
    const int e = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = e & 3, sub = e >> 2;
    int t_begin, t_end;
    tile_range(P, t_begin, t_end);
    const int K = P.kchunks * kBlockK;
    const int box_px = P.th * P.tw;
    // brute-force accumulator chunk of row (32q + lane) of tile tc
    auto brute = [&](const TileCoord& tc, int ch, float (&v)[32]) {
        const TapProblem& pr = P.prob[tc.prob];
        const int row = q * 32 + lane;
        const int ni = row / box_px, rem = row - ni * box_px;
        const int n = tc.n0 + ni, h = tc.h0 + rem / P.tw, w = tc.w0 + rem % P.tw;
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = 0.f;
        if (!(ni < P.nb && n < P.batch)) return;
        const int rows_total = (EPI == kEpiTopK || EPI == kEpiMember) ? P.n_codes : P.n_total;
        const int jmax = rows_total - (tc.nblk * BN + ch * 32);
        for (int ti = 0; ti < pr.ntaps; ++ti) {
            const Tap tap = P.taps[pr.tap_begin + ti];
            const int hh = h + tap.dy, ww = w + tap.dx;
            if (hh < 0 || hh >= ops.a_hs[tap.src] || ww < 0 || ww >= ops.a_ws[tap.src]) continue;
            const __nv_bfloat16* arow = reinterpret_cast<const __nv_bfloat16*>(ops.a_ptrs[tap.src]) +
                                        n * ops.a_sn + hh * ops.a_sh + ww * ops.a_sw;
            const __nv_bfloat16* wmat = reinterpret_cast<const __nv_bfloat16*>(ops.w) +
                                        (static_cast<long long>(tap.widx) * rows_total + tc.nblk * BN + ch * 32) * K;
            for (int k = 0; k < K; ++k) {
                const float a = __bfloat162float(arow[k]);
#pragma unroll
                for (int j = 0; j < 32; ++j)
                    if (j < jmax) v[j] = fmaf(a, __bfloat162float(wmat[static_cast<long long>(j) * K + k]), v[j]);
            }
        }
    };
    if constexpr (EPI == kEpiBwd) {
        auto tile_at = [&](int t, BwdTile& bt, int& adv) {
            const Unit u = get_unit<C::kMtMax>(P, t, t_end);
            const EpiSplit<BN> sp = epi_split<BN>(u.mt, sub);
            bt.tc = u.tile(sp.st); bt.step0 = sp.ch_begin; bt.nsteps = sp.ch_end - sp.ch_begin; bt.sub_tile = sp.st;
            adv = u.adv;
        };
        auto chunk_loader = [&](int, const BwdTile& bt) {
            const TileCoord tc = bt.tc;
            return [&brute, tc](int ch, float (&v)[32]) { brute(tc, ch, v); };
        };
        auto releaser = [&](int) { return [] {}; };
        if (P.split) bwd_warp_loop<BN, C::kBwdSteps, true>(P, q, lane, &wsm[e], t_begin, t_end, tile_at, chunk_loader, releaser);
        else bwd_warp_loop<BN, C::kBwdSteps, false>(P, q, lane, &wsm[e], t_begin, t_end, tile_at, chunk_loader, releaser);
    } else {
        for (int t = t_begin; t < t_end;) {
            const Unit u = get_unit<C::kMtMax>(P, t, t_end);
            t += u.adv;
            if (u.mt == 0) continue;
            const EpiSplit<BN> sp = epi_split<BN>(u.mt, sub);
            const TileCoord tc = u.tile(sp.st);
            auto load_chunk = [&](int ch, float (&v)[32]) { brute(tc, ch, v); };
            rowowner_warp_tile<BN, EPI, false>(P, tc, q, lane, sp.ch_begin, sp.ch_end, sp.whole ? 0 : sub, sp.whole, nullptr, nullptr, load_chunk);
        }
    }
}

// Seed of the backward chain: activation backward of the top layer from the toRGB gradient alone (the
// backward epilogue with a zero accumulator).  Streaming kernel: a block owns one sample, up to 128
// columns and a run of pixels; thread (cp, rl) owns a column pair and every (256 / pairs)-th pixel, so
// coefficients and the five column sums live in registers, each pixel row is one coalesced segment and
// many blocks fit an SM (HBM-bound: reads x, writes g_y).
constexpr int kSeedPixels = 2048;
__global__ void __launch_bounds__(256) seed_stream_kernel(const __grid_constant__ TapGemmParams P, int cpairs) {
    __shared__ float red[256 * 8];
    const int rlanes = 256 / cpairs;
    const int cp = threadIdx.x % cpairs, rl = threadIdx.x / cpairs;
    const int n = blockIdx.z;
    const int col = blockIdx.y * (2 * cpairs) + 2 * cp;
    const int img_px = P.OH * P.OW;
    const int p_begin = blockIdx.x * kSeedPixels;
    const int p_end = min(p_begin + kSeedPixels, img_px);
    const int half_n = P.n_total >> 1;
    const long long coff = static_cast<long long>(n) * P.n_total + col;
    const float2 dm = __ldg(reinterpret_cast<const float2*>(P.demod_prev + coff));
    const float2 bs = __ldg(reinterpret_cast<const float2*>(P.bias_prev + col));
    float4 rw0 = __ldg(P.rgbw_prev + coff), rw1 = __ldg(P.rgbw_prev + coff + 1);
    rw0.x *= P.act_gain; rw0.y *= P.act_gain; rw0.z *= P.act_gain;
    rw1.x *= P.act_gain; rw1.y *= P.act_gain; rw1.z *= P.act_gain;
    const float inv_gain = 1.f / P.act_gain, inv_gain_slope = 1.f / (P.act_gain * P.act_slope);
    const float saved_thr = act_saved_clamp(P.act_clamp, P.split);       // split: hi + lo read below
    const long long base = static_cast<long long>(n) * img_px;
    const unsigned* xh = reinterpret_cast<const unsigned*>(P.xp_hi) + base * half_n + (col >> 1);
    const unsigned* xl = P.split ? reinterpret_cast<const unsigned*>(P.xp_lo) + base * half_n + (col >> 1) : nullptr;
    unsigned* gh = reinterpret_cast<unsigned*>(P.gy_hi) + base * half_n + (col >> 1);
    unsigned* gl = P.split ? reinterpret_cast<unsigned*>(P.gy_lo) + base * half_n + (col >> 1) : nullptr;
    const float4* grgb = P.g_rgb + base;
    const float* nzp = P.noise_prev ? P.noise_prev + n * P.noise_prev_stride_n : nullptr;
    float r[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] = 0.f;
    constexpr int U = 4;                       // pixels in flight per thread
    for (int p0 = p_begin + rl; p0 < p_end; p0 += U * rlanes) {
        unsigned xu[U], xv[U];
        float4 g[U];
        float nz[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int p = p0 + u * rlanes;
            const bool ok = p < p_end;
            const long long o = static_cast<long long>(ok ? p : p_begin) * half_n;
            xu[u] = __ldg(xh + o);
            xv[u] = xl ? __ldg(xl + o) : 0u;
            g[u] = ok ? __ldg(grgb + p) : make_float4(0.f, 0.f, 0.f, 0.f);
            nz[u] = (nzp && ok) ? __ldg(nzp + p) * P.noise_prev_scale : 0.f;
            if (!ok) { xu[u] = 0u; xv[u] = 0u; }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int p = p0 + u * rlanes;
            const float x0 = bf16lo_f(xu[u]) + bf16lo_f(xv[u]), x1 = bf16hi_f(xu[u]) + bf16hi_f(xv[u]);
            const float g0 = fmaf(g[u].x, rw0.x, fmaf(g[u].y, rw0.y, g[u].z * rw0.z));
            const float g1 = fmaf(g[u].x, rw1.x, fmaf(g[u].y, rw1.y, g[u].z * rw1.z));
            r[2] = fmaf(x0, g[u].x, r[2]); r[3] = fmaf(x1, g[u].x, r[3]);
            r[4] = fmaf(x0, g[u].y, r[4]); r[5] = fmaf(x1, g[u].y, r[5]);
            r[6] = fmaf(x0, g[u].z, r[6]); r[7] = fmaf(x1, g[u].z, r[7]);
            const bool q0 = x0 > 0.f, q1 = x1 > 0.f;
            const float gz0 = act_grad(g0, x0, P.act_slope, saved_thr), gz1 = act_grad(g1, x1, P.act_slope, saved_thr);
            const float z0 = x0 * (q0 ? inv_gain : inv_gain_slope), z1 = x1 * (q1 ? inv_gain : inv_gain_slope);
            r[0] = fmaf(gz0, z0 - nz[u] - bs.x, r[0]);
            r[1] = fmaf(gz1, z1 - nz[u] - bs.y, r[1]);
            if (p < p_end) {
                const float y0 = gz0 * dm.x, y1 = gz1 * dm.y;
                const long long o = static_cast<long long>(p) * half_n;
                gh[o] = pack_bf16(y0, y1);
                if (gl) gl[o] = pack_bf16(y0 - bf16_round(y0), y1 - bf16_round(y1));
            }
        }
    }
    // reduce the row lanes of each column pair, then one atomic per (sum, column)
#pragma unroll
    for (int k = 0; k < 8; ++k) red[k * 256 + threadIdx.x] = r[k];
    __syncthreads();
    for (int e = threadIdx.x; e < 8 * cpairs; e += 256) {
        const int k = e / cpairs, c = e - k * cpairs;
        float v = 0.f;
        for (int j = 0; j < rlanes; ++j) v += red[k * 256 + j * cpairs + c];
        const int kind = k >> 1;                   // 0: red_d, 1..3: red_rgb
        float* dst = kind == 0 ? P.red_d : P.red_rgb + static_cast<long long>(kind - 1) * P.batch * P.n_total;
        atomicAdd(dst + static_cast<long long>(n) * P.n_total + blockIdx.y * (2 * cpairs) + 2 * c + (k & 1), v);
    }
}

// The same seed pass as an asynchronous pipeline (bf16 mode, N <= 256): a block streams runs of 32 pixels
// of one sample through shared memory with 1-D bulk copies -- x in, g_y out in place -- so the bytes in
// flight live in shared memory instead of registers and HBM stays busy.
constexpr int kSeedRows = 32, kSeedStages = 4;
__global__ void __launch_bounds__(128) seed_bulk_kernel(const __grid_constant__ TapGemmParams P, int px_per_block) {
    extern __shared__ __align__(128) uint8_t sraw[];
    const int N = P.n_total, pairs = N >> 1, rlanes = 128 / pairs, rows_per_thread = kSeedRows / rlanes;
    const uint32_t xbytes = kSeedRows * N * 2;
    const uint32_t stage_bytes = xbytes + kSeedRows * 16 + kSeedRows * 4;
    uint64_t* full = reinterpret_cast<uint64_t*>(sraw + kSeedStages * stage_bytes);
    float* red = reinterpret_cast<float*>(sraw);             // reused after the pipeline drained
    const int n = blockIdx.y;
    const int img_px = P.OH * P.OW;
    const int p_begin = blockIdx.x * px_per_block;
    const int p_end = min(p_begin + px_per_block, img_px);
    const int nchunks = (p_end - p_begin) / kSeedRows;       // img_px and px_per_block are multiples of 32
    const long long base = static_cast<long long>(n) * img_px;
    const __nv_bfloat16* xg = reinterpret_cast<const __nv_bfloat16*>(P.xp_hi) + base * N;
    __nv_bfloat16* gg = reinterpret_cast<__nv_bfloat16*>(P.gy_hi) + base * N;
    const float4* grgb = P.g_rgb + base;
    const float* nzp = P.noise_prev ? P.noise_prev + n * P.noise_prev_stride_n : nullptr;
    const int tid = threadIdx.x;
    if (tid == 0) {
        for (int s = 0; s < kSeedStages; ++s) mbar_init(&full[s], 1);
        fence_barrier_init();
    }
    __syncthreads();
    auto issue = [&](int chunk) {
        const int s = chunk % kSeedStages;
        uint8_t* st = sraw + s * stage_bytes;
        const int p = p_begin + chunk * kSeedRows;
        mbar_expect_tx(&full[s], xbytes + kSeedRows * 16 + (nzp ? kSeedRows * 4 : 0));
        bulk_load(st, xg + static_cast<long long>(p) * N, xbytes, &full[s]);
        bulk_load(st + xbytes, grgb + p, kSeedRows * 16, &full[s]);
        if (nzp) bulk_load(st + xbytes + kSeedRows * 16, nzp + p, kSeedRows * 4, &full[s]);
    };
    if (tid == 0)
        for (int c = 0; c < kSeedStages && c < nchunks; ++c) issue(c);

    const int cp = tid % pairs, rl = tid / pairs;
    const int col = 2 * cp;
    const long long coff = static_cast<long long>(n) * N + col;
    const float2 dm = __ldg(reinterpret_cast<const float2*>(P.demod_prev + coff));
    const float2 bs = __ldg(reinterpret_cast<const float2*>(P.bias_prev + col));
    float4 rw0 = __ldg(P.rgbw_prev + coff), rw1 = __ldg(P.rgbw_prev + coff + 1);
    rw0.x *= P.act_gain; rw0.y *= P.act_gain; rw0.z *= P.act_gain;
    rw1.x *= P.act_gain; rw1.y *= P.act_gain; rw1.z *= P.act_gain;
    const float inv_gain = 1.f / P.act_gain, inv_gain_slope = 1.f / (P.act_gain * P.act_slope);
    const float saved_thr = act_saved_clamp(P.act_clamp, false);         // hi plane only
    const float nscale = nzp ? P.noise_prev_scale : 0.f;
    float r[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) r[k] = 0.f;

    for (int it = 0; it < nchunks; ++it) {
        const int s = it % kSeedStages;
        uint8_t* st = sraw + s * stage_bytes;
        mbar_wait(&full[s], (it / kSeedStages) & 1, P.err_flag, 7);
        unsigned* xs = reinterpret_cast<unsigned*>(st);
        const float4* gs = reinterpret_cast<const float4*>(st + xbytes);
        const float* ns = reinterpret_cast<const float*>(st + xbytes + kSeedRows * 16);
#pragma unroll 8
        for (int j = 0; j < rows_per_thread; ++j) {
            const int row = rl + j * rlanes;
            const unsigned xu = xs[row * pairs + cp];
            const float4 g = gs[row];
            const float nz = nzp ? ns[row] * nscale : 0.f;
            const float x0 = bf16lo_f(xu), x1 = bf16hi_f(xu);
            const float g0 = fmaf(g.x, rw0.x, fmaf(g.y, rw0.y, g.z * rw0.z));
            const float g1 = fmaf(g.x, rw1.x, fmaf(g.y, rw1.y, g.z * rw1.z));
            r[2] = fmaf(x0, g.x, r[2]); r[3] = fmaf(x1, g.x, r[3]);
            r[4] = fmaf(x0, g.y, r[4]); r[5] = fmaf(x1, g.y, r[5]);
            r[6] = fmaf(x0, g.z, r[6]); r[7] = fmaf(x1, g.z, r[7]);
            const bool q0 = x0 > 0.f, q1 = x1 > 0.f;
            const float gz0 = act_grad(g0, x0, P.act_slope, saved_thr), gz1 = act_grad(g1, x1, P.act_slope, saved_thr);
            const float z0 = x0 * (q0 ? inv_gain : inv_gain_slope), z1 = x1 * (q1 ? inv_gain : inv_gain_slope);
            r[0] = fmaf(gz0, z0 - nz - bs.x, r[0]);
            r[1] = fmaf(gz1, z1 - nz - bs.y, r[1]);
            xs[row * pairs + cp] = pack_bf16(gz0 * dm.x, gz1 * dm.y);      // g_y in place
        }
        fence_proxy_async();          // generic-proxy writes -> visible to the bulk store
        __syncthreads();
        if (tid == 0) {
            bulk_store(gg + static_cast<long long>(p_begin + it * kSeedRows) * N, st, xbytes);
            bulk_commit();
            if (it >= 1 && it - 1 + kSeedStages < nchunks) {
                bulk_wait_read<1>();  // the store of the previous stage has read its buffer
                issue(it - 1 + kSeedStages);
            }
        }
    }
    if (tid == 0) bulk_wait_read<0>();
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 8; ++k) red[k * 128 + tid] = r[k];
    __syncthreads();
    for (int e = tid; e < 8 * pairs; e += 128) {
        const int k = e / pairs, c = e - k * pairs;
        float v = 0.f;
        for (int j = 0; j < rlanes; ++j) v += red[k * 128 + j * pairs + c];
        const int kind = k >> 1;                   // 0: red_d, 1..3: red_rgb
        float* dst = kind == 0 ? P.red_d : P.red_rgb + static_cast<long long>(kind - 1) * P.batch * N;
        atomicAdd(dst + static_cast<long long>(n) * N + 2 * c + (k & 1), v);
    }
}

template <int BN, int EPI, bool kPair>
int set_smem_attr() {
    static bool attr_set[kMaxDevices] = {};      // the attribute is per device (in-process multi-GPU: one engine per GPU id)
    const int dev = current_device_slot();
    if (!attr_set[dev]) {
        cudaError_t e = cudaFuncSetAttribute(tapgemm_kernel<BN, EPI, kPair>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             Cfg<BN, EPI, kPair>::kSmemBytes);
        if (e != cudaSuccess) return static_cast<int>(e);
        attr_set[dev] = true;
    }
    return 0;
}

template <int BN, int EPI>
int launch_bn_epi(const TapGemmParams& p, int num_sms, cudaStream_t stream) {
    static_assert(Cfg<BN, EPI>::kSmemBytes <= 232448, "shared memory budget");
    const int total = p.m_tiles * p.n_blocks;
    int grid = total < num_sms ? total : num_sms;
    if (grid <= 0) return 0;
    for (int i = 0; i < p.nprob; ++i)
        if (p.prob[i].ntaps <= 0 || p.prob[i].ngroups <= 0) return static_cast<int>(cudaErrorInvalidValue);   // accumulator would be undefined
    if (p.halo != 0 && (p.halo != 2 || p.tw != 8 || p.nb != 1 || p.th != 16)) return static_cast<int>(cudaErrorInvalidValue);
    if (p.interleave && (p.epilogue == kEpiBwd || p.m_tiles % (2 * p.nprob))) return static_cast<int>(cudaErrorInvalidValue);
    if (p.nb * (p.th + p.halo) * p.tw * 128 > kASubBytes) return static_cast<int>(cudaErrorInvalidValue);
    static const int cost_env = getenv("LA_TILE_COST") ? atoi(getenv("LA_TILE_COST")) : 0;      // tuning switch
    if (p.cta2) {
        // CTA pairs: clusters of two CTAs (one TPC), each cluster walks a cost-balanced range of tile pairs
        {
            if (p.interleave) return static_cast<int>(cudaErrorInvalidValue);
            if (int r = set_smem_attr<BN, EPI, true>()) return r;
            const int clusters = (total + 1) / 2 < num_sms / 2 ? (total + 1) / 2 : num_sms / 2;
            TapGemmParams q = p;
            // launches with at most one M tile per CTA never form four-tile work items: one-tile A slots, a ring twice
            // as deep (the K loop of the <= 16^2 layers is bound by the latency of the A loads in flight)
            q.no_pair = 0;
            q.no_quad = total <= num_sms ? 1 : 0;
            // (range balance: with the MMAs this much faster the fixed per-tile share weighs more; measured optimum)
            q.cost_fixed = cost_env ? cost_env : (BN == 128 ? 20 : 12);
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(static_cast<unsigned>(2 * clusters));
            cfg.blockDim = dim3(kThreads);
            cfg.dynamicSmemBytes = Cfg<BN, EPI, true>::kSmemBytes;
            cfg.stream = stream;
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeClusterDimension;
            attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
            cfg.attrs = attr;
            cfg.numAttrs = 1;
            return static_cast<int>(cudaLaunchKernelEx(&cfg, tapgemm_kernel<BN, EPI, true>, q));
        }
    }
    if (int r = set_smem_attr<BN, EPI, false>()) return r;
    TapGemmParams q = p;
    q.cost_fixed = 4;
    if (total <= num_sms && !p.no_pair) q.no_pair = 1;       // one tile per CTA: nothing to pair, so run the deeper unpaired A ring
    tapgemm_kernel<BN, EPI, false><<<grid, kThreads, Cfg<BN, EPI>::kSmemBytes, stream>>>(q);
    return static_cast<int>(cudaGetLastError());
}

template <int BN>
int launch_bn(const TapGemmParams& p, int num_sms, cudaStream_t stream) {
    switch (p.epilogue) {
        case kEpiRawF32: return launch_bn_epi<BN, kEpiRawF32>(p, num_sms, stream);
        case kEpiFwd: return launch_bn_epi<BN, kEpiFwd>(p, num_sms, stream);
        case kEpiBwd: return launch_bn_epi<BN, kEpiBwd>(p, num_sms, stream);
        case kEpiTopK: return launch_bn_epi<BN, kEpiTopK>(p, num_sms, stream);
        case kEpiMember: return launch_bn_epi<BN, kEpiMember>(p, num_sms, stream);
        case kEpiStoreBf16: return launch_bn_epi<BN, kEpiStoreBf16>(p, num_sms, stream);
        case kEpiLinear: return launch_bn_epi<BN, kEpiLinear>(p, num_sms, stream);
        default: return static_cast<int>(cudaErrorInvalidValue);
    }
}

template <int BN, int EPI>
int launch_simt_bn_epi(const TapGemmParams& p, const TapSimtOperands& ops, cudaStream_t stream) {
    const int total = p.m_tiles * p.n_blocks;
    int grid = total < 148 * 4 ? total : 148 * 4;
    if (grid <= 0) return 0;
    tapgemm_simt_kernel<BN, EPI><<<grid, kEpiThreads, 0, stream>>>(p, ops);
    return static_cast<int>(cudaGetLastError());
}

template <int BN>
int launch_simt_bn(const TapGemmParams& p, const TapSimtOperands& ops, cudaStream_t stream) {
    switch (p.epilogue) {
        case kEpiRawF32: return launch_simt_bn_epi<BN, kEpiRawF32>(p, ops, stream);
        case kEpiFwd: return launch_simt_bn_epi<BN, kEpiFwd>(p, ops, stream);
        case kEpiBwd: return launch_simt_bn_epi<BN, kEpiBwd>(p, ops, stream);
        case kEpiTopK: return launch_simt_bn_epi<BN, kEpiTopK>(p, ops, stream);
        case kEpiMember: return launch_simt_bn_epi<BN, kEpiMember>(p, ops, stream);
        case kEpiStoreBf16: return launch_simt_bn_epi<BN, kEpiStoreBf16>(p, ops, stream);
        case kEpiLinear: return launch_simt_bn_epi<BN, kEpiLinear>(p, ops, stream);
        default: return static_cast<int>(cudaErrorInvalidValue);
    }
}

}  // namespace

int tapgemm_finalize(TapGemmParams& p) {
    int ng = 0, nt = 0;
    for (int i = 0; i < p.nprob; ++i) {
        TapProblem& pr = p.prob[i];
        pr.grp_begin = ng;
        bool used[kMaxTaps] = {};
        for (int a = 0; a < pr.ntaps; ++a) {
            while (!used[a]) {       // groups keyed on (dx, src) of tap a; its lowest unused dy anchors the box
                const Tap ta = p.taps[pr.tap_begin + a];
                if (ng >= kMaxTaps) return -1;
                TapGroup g{};
                g.dx = ta.dx; g.src = ta.src; g.tap_begin = static_cast<uint16_t>(nt);
                int dy0 = ta.dy;
                if (p.halo > 0)
                    for (int b = a; b < pr.ntaps; ++b) {
                        const Tap tb = p.taps[pr.tap_begin + b];
                        if (!used[b] && tb.dx == ta.dx && tb.src == ta.src && tb.dy < dy0) dy0 = tb.dy;
                    }
                g.dy0 = static_cast<int8_t>(dy0);
                int cnt = 0;
                for (int b = a; b < pr.ntaps; ++b) {
                    const Tap tb = p.taps[pr.tap_begin + b];
                    const bool same = p.halo > 0 ? (tb.dx == ta.dx && tb.src == ta.src) : (b == a);
                    if (used[b] || !same) continue;
                    const int rel = tb.dy - dy0;
                    if (rel < 0 || rel > p.halo) continue;      // does not fit this box: a later group takes it
                    used[b] = true;
                    p.gdyrel[nt] = static_cast<uint8_t>(rel);
                    p.gwidx[nt] = tb.widx;
                    ++nt; ++cnt;
                }
                g.ntaps = static_cast<uint8_t>(cnt);
                p.groups[ng++] = g;
            }
        }
        pr.ngroups = ng - pr.grp_begin;
    }
    return 0;
}

int launch_tapgemm_seed(const TapGemmParams& p, int /*num_sms*/, cudaStream_t stream) {
    if (p.epilogue != kEpiBwd || !p.g_rgb || !p.rgbw_prev || p.n_total % 64) return static_cast<int>(cudaErrorInvalidValue);
    const int pairs = p.n_total / 2;
    const int img_px = p.OH * p.OW;
    if (!p.split && (pairs == 32 || pairs == 64 || pairs == 128) && img_px % kSeedRows == 0 && !getenv("LA_SEED_STREAM")) {
        const int smem = kSeedStages * (kSeedRows * p.n_total * 2 + kSeedRows * 20) + 64;
        static bool attr_set[kMaxDevices] = {};
        const int dev = current_device_slot();
        if (!attr_set[dev]) {
            cudaError_t e = cudaFuncSetAttribute(seed_bulk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 80 * 1024);
            if (e != cudaSuccess) return static_cast<int>(e);
            attr_set[dev] = true;
        }
        const int ppb = img_px < 2048 ? img_px : 2048;
        dim3 grid((img_px + ppb - 1) / ppb, p.batch);
        seed_bulk_kernel<<<grid, 128, smem, stream>>>(p, ppb);
        return static_cast<int>(cudaGetLastError());
    }
    const int cpairs = pairs >= 64 ? 64 : 32;
    dim3 grid((p.OH * p.OW + kSeedPixels - 1) / kSeedPixels, pairs / cpairs, p.batch);
    seed_stream_kernel<<<grid, 256, 0, stream>>>(p, cpairs);
    return static_cast<int>(cudaGetLastError());
}

int launch_tapgemm(const TapGemmParams& p, int num_sms, cudaStream_t stream) {
    const int bn = p.n_total / p.n_blocks;
    switch (bn) {
        case 256: return launch_bn<256>(p, num_sms, stream);
        case 128: return launch_bn<128>(p, num_sms, stream);
        case 64: return launch_bn<64>(p, num_sms, stream);
        default: return static_cast<int>(cudaErrorInvalidValue);
    }
}

int launch_tapgemm_simt(const TapGemmParams& p, const TapSimtOperands& ops, cudaStream_t stream) {
    const int bn = p.n_total / p.n_blocks;
    switch (bn) {
        case 256: return launch_simt_bn<256>(p, ops, stream);
        case 128: return launch_simt_bn<128>(p, ops, stream);
        case 64: return launch_simt_bn<64>(p, ops, stream);
        default: return static_cast<int>(cudaErrorInvalidValue);
    }
}

int encode_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides,
                     const uint32_t* box, int swizzle_bytes) {
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                 const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                 CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeFn fn = nullptr;
    if (!fn) {
        void* ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres);
        if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !ptr) return -1;
        fn = reinterpret_cast<EncodeFn>(ptr);
    }
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    cuuint64_t gdim[5], gstr[4];
    cuuint32_t bx[5];
    for (int i = 0; i < rank; ++i) { gdim[i] = dims[i]; bx[i] = box[i]; }
    for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides[i];
    CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, static_cast<cuuint32_t>(rank), const_cast<void*>(base), gdim, gstr,
                    bx, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    swizzle_bytes == 0 ? CU_TENSOR_MAP_SWIZZLE_NONE : (swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B), CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return static_cast<int>(r);
}

}  // namespace la
