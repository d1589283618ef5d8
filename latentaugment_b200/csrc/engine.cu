// Engine: owns the layer plan of one StyleGAN2 generator at one batch size -- prepared
// weights, activation buffers, the TapGemmParams of every forward / data-gradient GEMM --
// and runs the LatentAugment loop (reference augments/utils/util_latent_aug.py:207-310)
// as a CUDA graph.  Exposes the C ABI of include/latentaugment_b200.h.
#include <cuda_bf16.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/latentaugment_b200.h"
#include "kernels.cuh"
#include "tapgemm.cuh"
#include "plan.cuh"
#include "disc.cuh"
#include "lpips.cuh"

using namespace la;

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code ? code : -1;
}

#define CU(x)                                                                                              \
    do {                                                                                                   \
        cudaError_t e_ = (x);                                                                              \
        if (e_ != cudaSuccess) return fail(static_cast<int>(e_), "%s: %s (%s:%d)", #x, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)
#define LA(x)                                                                                              \
    do {                                                                                                   \
        int r_ = (x);                                                                                      \
        if (r_) return fail(r_, "%s: %s (%s:%d)", #x, r_ > 0 ? cudaGetErrorString(static_cast<cudaError_t>(r_)) : "error", __FILE__, __LINE__); \
    } while (0)

typedef __nv_bfloat16 bf16;

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

struct Conv {
    int res_in, res, cin, cout, up, block, last_in_block, ws_idx, soff, doff;
    la_conv_params p;
    bf16 *wf, *wb;
    float *w2, *w2t;
    bf16 *x_hi, *x_lo;
    long long noise_off;     // offset of this layer's slice in a random-noise buffer
    int split_up;            // x2 layer run as transposed-conv GEMM + FIR pass (vs FIR folded into 36 taps)
    UpFirParams fir;
    TapGemmParams fwd, bwd;
    TapSimtOperands fwd_ops, bwd_ops;
};
struct Rgb {
    int res, cin, ws_idx, soff, roff, nparts;
    la_torgb_params p;
    float4 *parts, *img, *g_img, *g_rgb;
};

}  // namespace

struct la_engine {
    la_generator_desc g;
    int batch, split, num_sms, num_ws;
    int S, D, R, nchunks;
    std::vector<Conv> conv;
    std::vector<Rgb> rgb;
    LayerTable table;
    // parameters / coefficients
    float *c_f32; bf16 *c_hi, *c_lo, *c_rep_hi, *c_rep_lo;
    float *a_cat, *b_cat, *s_cat, *d_cat, *g_s, *partial, *red_all, *red_s, *red_d, *red_rgb, *dummy_red;
    size_t red_bytes;
    float4* rgbw;
    int *chunk_soff, *chunk_cin;
    bf16 *xs_hi[2], *xs_lo[2], *gy_hi[2], *gy_lo[2];
    bf16 *t_hi, *t_lo;       // transposed-conv intermediate T / g_T of the split up-sampling layers
    int split_min_res;
    float fir_host[16];      // resample filter (host copy)
    // criteria
    float4* bank_mean; float* bank_m2; float* loss_parts; int n_loss_parts; int has_img_bank, has_lat_bank;
    float *w_sum, *lat_m2;
    int crop_off, crop_size;
    // loop state
    AdamConsts* consts; int* step; int* err_flag; unsigned long long* dbg_clock;
    float *w_opt, *m, *v, *w0, *w_aug, *loss_log, *map_a, *map_b;
    TapGemmParams seed; TapSimtOperands seed_ops;
    // execution
    cudaStream_t work = nullptr; cudaEvent_t ev_in = nullptr, ev_out = nullptr;
    cudaGraphExec_t step_graph = nullptr; bool warmed = false; bool graph_disabled = false;
    int use_simt = 0;
    long long launches = 0, launches_captured = 0, graph_kernels = 0;   // kernel launches (graph replays count their kernels)
    float cur_w_pix = -1.f, cur_w_disc = -1.f;
    la_disc* disc = nullptr;          // realism-term discriminator (optional)
    float* disc_loss = nullptr;
    la_lpips* lp = nullptr;           // perceptual term (optional)
    float* lpips_loss = nullptr;      // [batch]: the total in bank mode, the per-sample distances in projection
    float cur_w_lpips = -1.f;
    // projection (la_project): perturbed code the style GEMMs read, the device-resident schedule
    float* w_pert = nullptr;
    ProjConsts* proj = nullptr;
    int cur_project = 0;              // the captured step_graph is a projection step (it bakes the criterion launches)
    bool proj_warmed = false;         // a projection step has run eagerly (its launches differ from the augmentation's)
};

namespace {

// x2 layers with output resolution >= this run as transposed-conv GEMM + FIR pass (9 taps, the
// algorithmic MAC count); smaller ones keep the FIR folded into 36 taps (one launch, latency-bound anyway).
int upconv_split_min_res() {
    const char* v = getenv("LA_UPCONV_SPLIT_MIN_RES");
    return v ? atoi(v) : 8;
}

// Plans layers and carves the workspace.  With ws == nullptr only sizes are computed.
int plan(la_engine* e, char* ws, size_t* bytes_out) {
    const la_generator_desc& g = e->g;
    if (g.num_blocks < 2 || g.num_blocks > LA_MAX_BLOCKS || (4 << (g.num_blocks - 1)) != g.img_resolution)
        return fail(-2, "img_resolution %d does not match num_blocks %d", g.img_resolution, g.num_blocks);
    if (g.img_channels < 1 || g.img_channels > 3) return fail(-2, "img_channels must be 1..3");
    if (g.w_dim > 1024 || g.w_dim % 4) return fail(-2, "w_dim must be <= 1024");
    for (int b = 0; b < g.num_blocks; ++b)
        if (!pick_bn(g.channels[b]) || g.channels[b] > 1024) return fail(-2, "channels[%d]=%d unsupported (64 or a multiple of 128 up to 1024)", b, g.channels[b]);
    const int B = e->batch, split = e->split;
    e->num_ws = 2 * g.num_blocks;
    e->conv.clear();
    e->rgb.clear();
    int S = 0, D = 0, R = 0, widx = 0;
    long long noise_off = 0;
    for (int b = 0; b < g.num_blocks; ++b) {
        const int res = 4 << b, C = g.channels[b];
        if (b > 0) {
            Conv c{};
            c.res_in = res / 2; c.res = res; c.cin = g.channels[b - 1]; c.cout = C; c.up = 2; c.block = b; c.ws_idx = widx++;
            c.split_up = res >= e->split_min_res;
            e->conv.push_back(c);
        }
        Conv c{};
        c.res_in = res; c.res = res; c.cin = C; c.cout = C; c.up = 1; c.block = b; c.last_in_block = 1; c.ws_idx = widx++;
        e->conv.push_back(c);
        Rgb r{};
        r.res = res; r.cin = C; r.ws_idx = widx; r.p = g.torgb[b];
        r.nparts = 2 * (C / pick_bn(C, grid_m_tiles(res, e->batch)));      // two toRGB partial slots per column block
        e->rgb.push_back(r);
    }
    for (size_t l = 0; l < e->conv.size(); ++l) {
        Conv& c = e->conv[l];
        c.p = g.conv[l];
        c.soff = S; S += c.cin;
        c.doff = D; D += c.cout;
        c.noise_off = noise_off; noise_off += static_cast<long long>(B) * c.res * c.res;
    }
    for (Rgb& r : e->rgb) { r.soff = S; S += r.cin; r.roff = R; R += r.cin; }
    e->S = S; e->D = D; e->R = R; e->nchunks = S / 64;
    if (static_cast<int>(e->conv.size()) > kMaxLayers) return fail(-2, "too many layers");

    Bump bp;
    bp.base = ws;
    size_t max_xs = 0, max_gy = 0, max_t = 0;
    int max_n = 0;
    for (Conv& c : e->conv) {
        const int nmat = ((c.up == 2 && !c.split_up) ? 36 : 9) * (split ? 2 : 1);
        if (c.split_up) {
            const size_t tsz = static_cast<size_t>(B) * (c.res + 1) * (c.res + 2) * c.cout;
            max_t = tsz > max_t ? tsz : max_t;
        }
        const size_t wsz = static_cast<size_t>(nmat) * c.cout * c.cin;
        c.wf = bp.take<bf16>(wsz);
        c.wb = bp.take<bf16>(wsz);
        c.w2 = bp.take<float>(static_cast<size_t>(c.cout) * c.cin);
        c.w2t = bp.take<float>(static_cast<size_t>(c.cout) * c.cin);
        const size_t xsz = static_cast<size_t>(B) * c.res * c.res * c.cout;
        c.x_hi = bp.take<bf16>(xsz);
        c.x_lo = split ? bp.take<bf16>(xsz) : nullptr;
        max_gy = xsz > max_gy ? xsz : max_gy;
        const size_t isz = static_cast<size_t>(B) * c.res_in * c.res_in * c.cin;
        max_xs = isz > max_xs ? isz : max_xs;
        max_n = c.cout > max_n ? c.cout : max_n;
    }
    for (int i = 0; i < 2; ++i) {
        e->xs_hi[i] = bp.take<bf16>(max_xs);
        e->xs_lo[i] = split ? bp.take<bf16>(max_xs) : nullptr;
        e->gy_hi[i] = bp.take<bf16>(max_gy);
        e->gy_lo[i] = split ? bp.take<bf16>(max_gy) : nullptr;
    }
    e->t_hi = max_t ? bp.take<bf16>(max_t) : nullptr;
    e->t_lo = (max_t && split) ? bp.take<bf16>(max_t) : nullptr;
    const int C0 = g.channels[0];
    e->c_f32 = bp.take<float>(16 * C0);
    e->c_hi = bp.take<bf16>(16 * C0);
    e->c_lo = bp.take<bf16>(16 * C0);
    e->c_rep_hi = bp.take<bf16>(static_cast<size_t>(B) * 16 * C0);
    e->c_rep_lo = bp.take<bf16>(static_cast<size_t>(B) * 16 * C0);
    e->a_cat = bp.take<float>(static_cast<size_t>(S) * g.w_dim);
    e->b_cat = bp.take<float>(S);
    e->s_cat = bp.take<float>(static_cast<size_t>(B) * S);
    e->d_cat = bp.take<float>(static_cast<size_t>(B) * D);
    e->g_s = bp.take<float>(static_cast<size_t>(B) * S);
    e->partial = bp.take<float>(static_cast<size_t>(e->nchunks) * B * g.w_dim);
    const size_t red_floats = static_cast<size_t>(B) * (S + D + 3 * R);
    e->red_all = bp.take<float>(red_floats);
    e->red_bytes = red_floats * sizeof(float);
    e->red_s = e->red_all;
    e->red_d = e->red_all ? e->red_all + static_cast<size_t>(B) * S : nullptr;
    e->red_rgb = e->red_all ? e->red_d + static_cast<size_t>(B) * D : nullptr;
    e->dummy_red = bp.take<float>(static_cast<size_t>(B) * max_n);
    e->rgbw = bp.take<float4>(static_cast<size_t>(B) * R);
    e->chunk_soff = bp.take<int>(e->nchunks);
    e->chunk_cin = bp.take<int>(e->nchunks);
    for (Rgb& r : e->rgb) {
        const size_t px = static_cast<size_t>(B) * r.res * r.res;
        r.parts = bp.take<float4>(px * r.nparts);
        r.img = bp.take<float4>(px);
        r.g_img = bp.take<float4>(px);
        r.g_rgb = bp.take<float4>(px);
    }
    e->bank_mean = bp.take<float4>(static_cast<size_t>(g.img_resolution) * g.img_resolution);
    e->bank_m2 = bp.take<float>(4);
    e->loss_parts = bp.take<float>(1024);
    e->w_sum = bp.take<float>(g.w_dim);
    e->lat_m2 = bp.take<float>(1);
    e->consts = bp.take<AdamConsts>(1);
    e->step = bp.take<int>(1);
    e->err_flag = bp.take<int>(1);
    e->disc_loss = bp.take<float>(1);
    e->lpips_loss = bp.take<float>(B);
    e->proj = bp.take<ProjConsts>(1);
    e->dbg_clock = bp.take<unsigned long long>(64);
    const size_t wn = static_cast<size_t>(B) * g.w_dim;
    e->w_opt = bp.take<float>(wn); e->m = bp.take<float>(wn); e->v = bp.take<float>(wn);
    e->w0 = bp.take<float>(wn); e->w_aug = bp.take<float>(wn);
    e->w_pert = bp.take<float>(wn);
    e->loss_log = bp.take<float>(LA_MAX_STEPS * LA_LOSS_COLS);
    const size_t mapn = static_cast<size_t>(B) * (g.w_dim > g.z_dim ? g.w_dim : g.z_dim);
    e->map_a = bp.take<float>(mapn); e->map_b = bp.take<float>(mapn);
    bp.take<char>(1024);
    *bytes_out = bp.off;
    return 0;
}

int build_params(la_engine* e) {
    const int B = e->batch, split = e->split;
    const la_generator_desc& g = e->g;
    const int L = static_cast<int>(e->conv.size());
    for (int l = 0; l < L; ++l) {
        Conv& c = e->conv[l];
        const Conv* next = l + 1 < L ? &e->conv[l + 1] : nullptr;
        const Conv* prev = l > 0 ? &e->conv[l - 1] : nullptr;
        const Rgb* rgb = c.last_in_block ? &e->rgb[c.block] : nullptr;
        const int nmat = (c.up == 2 && !c.split_up) ? 36 : 9;
        // ---------------------------------------------------------------- forward
        TapGemmParams& F = c.fwd;
        memset(&F, 0, sizeof F);
        if (c.split_up) {       // T[2m+py, 2n+px]: even phases have one more row / column (T is (2H+1) x (2W+1))
            const int gh[4] = {c.res_in + 1, c.res_in + 1, c.res_in, c.res_in};
            const int gw[4] = {c.res_in + 1, c.res_in, c.res_in + 1, c.res_in};
            set_grid(F, c.res_in, B, 4, gh, gw);
            if (getenv("LA_INTERLEAVE")) set_interleaved(F);      // tuning switch: the cost-balanced contiguous split measured better
        } else {
            set_grid(F, c.res_in, B, c.up == 2 ? 4 : 1);
        }
        const bf16* a_hi = e->xs_hi[l & 1];
        const bf16* a_lo = e->xs_lo[l & 1];
        const long long sW = c.cin, sH = static_cast<long long>(c.res_in) * c.cin, sN = sH * c.res_in;
        LA(make_a_map(&F.a_map[0], a_hi, c.cin, c.res_in, c.res_in, B, sW, sH, sN, F.tw, F.th + F.halo, F.nb));
        if (split) LA(make_a_map(&F.a_map[1], a_lo, c.cin, c.res_in, c.res_in, B, sW, sH, sN, F.tw, F.th + F.halo, F.nb));
        c.fwd_ops = TapSimtOperands{};
        c.fwd_ops.a_ptrs[0] = a_hi; c.fwd_ops.a_ptrs[1] = a_lo;
        c.fwd_ops.a_sw = sW; c.fwd_ops.a_sh = sH; c.fwd_ops.a_sn = sN;
        set_ops_dims(c.fwd_ops, c.res_in, c.res_in);
        c.fwd_ops.w = c.wf;
        const int bn = pick_bn(c.cout, F.m_tiles);
        LA(make_b_map(F, c.wf, c.cin, c.cout, nmat * (split ? 2 : 1), bn, c.split_up ? 0 : 1));
        int nt = 0;
        for (int ph = 0; ph < F.nprob; ++ph) {
            F.prob[ph].tap_begin = nt;
            if (c.split_up) {   // transposed conv, stride 2: T[2i+a] += x[i] W[a]  ->  taps with a = phase (mod 2), x offset -(a >> 1)
                for (int ay = ph / 2; ay < 3; ay += 2)
                    for (int ax = ph % 2; ax < 3; ax += 2) add_tap(F, nt, -(ay >> 1), -(ax >> 1), ay * 3 + ax, 0, 1, nmat, split);
            } else {
                for (int t = 0; t < 9; ++t) add_tap(F, nt, t / 3 - 1, t % 3 - 1, ph * 9 + t, 0, 1, nmat, split);
            }
            F.prob[ph].ntaps = nt - F.prob[ph].tap_begin;
            F.prob[ph].oy0 = c.up == 2 ? ph / 2 : 0;
            F.prob[ph].ox0 = c.up == 2 ? ph % 2 : 0;
        }
        F.kchunks = c.cin / 64; F.n_total = c.cout; F.n_blocks = c.cout / bn;
        F.epilogue = kEpiFwd;
        F.OH = F.OW = c.res; F.osy = F.osx = c.up; F.split = split;
        F.act_gain = 1.41421356237309515f; F.act_clamp = g.conv_clamp; F.act_slope = 0.2f;
        F.demod = e->d_cat + static_cast<size_t>(B) * c.doff;
        F.bias = c.p.d_bias;
        F.noise = c.p.d_noise_const; F.noise_stride_n = 0; F.noise_scale = c.p.noise_strength;
        F.s_next = next ? e->s_cat + static_cast<size_t>(B) * next->soff : nullptr;
        F.x_hi = c.x_hi; F.x_lo = c.x_lo;
        F.xs_hi = e->xs_hi[(l + 1) & 1]; F.xs_lo = e->xs_lo[(l + 1) & 1];
        F.rgbw = rgb ? e->rgbw + static_cast<size_t>(B) * rgb->roff : nullptr;
        F.rgb_part = rgb ? rgb->parts : nullptr;
        F.err_flag = e->err_flag;
        const int TH = c.res + 1, TWp = c.res + 2;      // T rows / row pitch of the split up-sampling layers
        if (c.split_up) {
            UpFirParams& U = c.fir;
            memset(&U, 0, sizeof U);
            U.t_hi = e->t_hi; U.t_lo = e->t_lo;
            U.B = B; U.OH = U.OW = c.res; U.C = c.cout; U.TH = TH; U.TWp = TWp; U.split = split;
            U.demod = F.demod; U.bias = F.bias; U.noise = F.noise; U.noise_stride_n = 0; U.noise_scale = F.noise_scale;
            U.s_next = F.s_next; U.x_hi = F.x_hi; U.x_lo = F.x_lo; U.xs_hi = F.xs_hi; U.xs_lo = F.xs_lo;
            U.act_gain = F.act_gain; U.act_clamp = F.act_clamp; U.act_slope = F.act_slope;
            for (int jy = 0; jy < 4; ++jy)       // true convolution (flipped filter), gain up^2 = 4 (upfirdn2d.py:196-199)
                for (int jx = 0; jx < 4; ++jx) U.fk[jy * 4 + jx] = e->fir_host[(3 - jy) * 4 + (3 - jx)] * 4.f;
            {   // rank-1 test: fk = fy (x) fx with fy = column of the largest entry / that entry, fx = its row
                int bi = 0;
                for (int k = 1; k < 16; ++k) if (fabsf(U.fk[k]) > fabsf(U.fk[bi])) bi = k;
                const int by = bi / 4, bx = bi % 4;
                U.separable = U.fk[bi] != 0.f;
                for (int k = 0; k < 4 && U.separable; ++k) { U.fy[k] = U.fk[k * 4 + bx] / U.fk[bi]; U.fx[k] = U.fk[by * 4 + k]; }
                for (int k = 0; k < 16 && U.separable; ++k)
                    if (fabsf(U.fy[k / 4] * U.fx[k % 4] - U.fk[k]) > 1e-6f * fabsf(U.fk[bi])) U.separable = 0;
            }
            U.gy_hi = e->gy_hi[l & 1]; U.gy_lo = e->gy_lo[l & 1]; U.gt_hi = e->t_hi; U.gt_lo = e->t_lo;
            static const bool no_fir_tma = getenv("LA_NO_FIR_TMA") != nullptr;
            if (!split && U.separable && c.res >= 32 && c.cout % 64 == 0 && !no_fir_tma) {
                const uint64_t C = c.cout, R = c.res;
                const uint64_t tdims[4] = {C, R + 1, R + 1, static_cast<uint64_t>(B)};          // T: (2H+1) x (2W+1), row pitch TWp
                const uint64_t tstr[3] = {C * 2, static_cast<uint64_t>(TWp) * C * 2, static_cast<uint64_t>(TH) * TWp * C * 2};
                const uint64_t ydims[4] = {C, R, R, static_cast<uint64_t>(B)};
                const uint64_t ystr[3] = {C * 2, R * C * 2, R * R * C * 2};
                const uint32_t lbox[4] = {64, 35, 1, 1}, sbox[4] = {64, 8, 1, 1};
                int r = encode_tmap_bf16(&U.fwd_in, e->t_hi, 4, tdims, tstr, lbox, 0);
                r |= encode_tmap_bf16(&U.fwd_out_x, c.x_hi, 4, ydims, ystr, sbox, 0);
                if (next) r |= encode_tmap_bf16(&U.fwd_out_xs, e->xs_hi[(l + 1) & 1], 4, ydims, ystr, sbox, 0);
                r |= encode_tmap_bf16(&U.bwd_in, e->gy_hi[l & 1], 4, ydims, ystr, lbox, 0);
                r |= encode_tmap_bf16(&U.bwd_out, e->t_hi, 4, tdims, tstr, sbox, 0);
                if (r) return fail(-5, "tensor map encoding failed (FIR pass)");
                U.use_tma = 1;
            }
            // the GEMM only stores T
            F.epilogue = kEpiStoreBf16;
            F.OH = TH; F.OW = TWp;
            F.x_hi = e->t_hi; F.x_lo = e->t_lo;
            F.xs_hi = F.xs_lo = nullptr; F.s_next = nullptr; F.rgbw = nullptr;
        }

        // staged stores + coefficient tables in the row-owner epilogues (bf16 mode, one sample per tile)
        static const bool no_staged = getenv("LA_NO_STAGED") != nullptr;
        if (!split && !no_staged && F.nb == 1 && (c.split_up || c.up == 1)) F.staged = 1;

        // ---------------------------------------------------------------- data gradient
        TapGemmParams& G = c.bwd;
        memset(&G, 0, sizeof G);
        set_grid(G, c.res_in, B, 1);
        const bf16* gy_hi = e->gy_hi[l & 1];
        const bf16* gy_lo = e->gy_lo[l & 1];
        c.bwd_ops = TapSimtOperands{};
        c.bwd_ops.w = c.wb;
        nt = 0;
        G.prob[0].tap_begin = 0;
        if (c.up == 1) {
            const long long gW = c.cout, gH = static_cast<long long>(c.res) * c.cout, gN = gH * c.res;
            LA(make_a_map(&G.a_map[0], gy_hi, c.cout, c.res, c.res, B, gW, gH, gN, G.tw, G.th + G.halo, G.nb));
            if (split) LA(make_a_map(&G.a_map[1], gy_lo, c.cout, c.res, c.res, B, gW, gH, gN, G.tw, G.th + G.halo, G.nb));
            c.bwd_ops.a_ptrs[0] = gy_hi; c.bwd_ops.a_ptrs[1] = gy_lo;
            c.bwd_ops.a_sw = gW; c.bwd_ops.a_sh = gH; c.bwd_ops.a_sn = gN;
            set_ops_dims(c.bwd_ops, c.res, c.res);
            for (int t = 0; t < 9; ++t) add_tap(G, nt, 1 - t / 3, 1 - t % 3, t, 0, 1, nmat, split);
        } else if (c.split_up) {
            // g_xs[i] = sum_a g_T[2i + a] W[a]^T : four phase-strided views of g_T, 9 taps
            const long long gW = 2LL * c.cout, gH = 2LL * TWp * c.cout, gN = static_cast<long long>(TH) * TWp * c.cout;
            c.bwd_ops.a_sw = gW; c.bwd_ops.a_sh = gH; c.bwd_ops.a_sn = gN;
            for (int ph = 0; ph < 4; ++ph) {
                const int py = ph / 2, px = ph % 2;
                const int ph_h = c.res_in + (py == 0), ph_w = c.res_in + (px == 0);
                const long long off = (static_cast<long long>(py) * TWp + px) * c.cout;
                LA(make_a_map(&G.a_map[ph], e->t_hi + off, c.cout, ph_w, ph_h, B, gW, gH, gN, G.tw, G.th + G.halo, G.nb));
                c.bwd_ops.a_ptrs[ph] = e->t_hi + off;
                c.bwd_ops.a_ws[ph] = ph_w; c.bwd_ops.a_hs[ph] = ph_h;
                if (split) {
                    LA(make_a_map(&G.a_map[4 + ph], e->t_lo + off, c.cout, ph_w, ph_h, B, gW, gH, gN, G.tw, G.th + G.halo, G.nb));
                    c.bwd_ops.a_ptrs[4 + ph] = e->t_lo + off;
                    c.bwd_ops.a_ws[4 + ph] = ph_w; c.bwd_ops.a_hs[4 + ph] = ph_h;
                }
            }
            for (int ay = 0; ay < 3; ++ay)
                for (int ax = 0; ax < 3; ++ax) {
                    const int ph = (ay & 1) * 2 + (ax & 1);
                    add_tap(G, nt, ay >> 1, ax >> 1, ay * 3 + ax, ph, 4 + ph, nmat, split);
                }
        } else {
            const long long gW = 2LL * c.cout, gH = 2LL * c.res * c.cout, gN = static_cast<long long>(c.res) * c.res * c.cout;
            for (int ph = 0; ph < 4; ++ph) {
                const long long off = (static_cast<long long>(ph / 2) * c.res + (ph % 2)) * c.cout;
                LA(make_a_map(&G.a_map[ph], gy_hi + off, c.cout, c.res_in, c.res_in, B, gW, gH, gN, G.tw, G.th + G.halo, G.nb));
                c.bwd_ops.a_ptrs[ph] = gy_hi + off;
                if (split) {
                    LA(make_a_map(&G.a_map[4 + ph], gy_lo + off, c.cout, c.res_in, c.res_in, B, gW, gH, gN, G.tw, G.th + G.halo, G.nb));
                    c.bwd_ops.a_ptrs[4 + ph] = gy_lo + off;
                }
            }
            c.bwd_ops.a_sw = gW; c.bwd_ops.a_sh = gH; c.bwd_ops.a_sn = gN;
            set_ops_dims(c.bwd_ops, c.res_in, c.res_in);
            for (int ph = 0; ph < 4; ++ph)
                for (int t = 0; t < 9; ++t) add_tap(G, nt, -(t / 3 - 1), -(t % 3 - 1), ph * 9 + t, ph, 4 + ph, nmat, split);
        }
        G.prob[0].ntaps = nt;
        if (tapgemm_finalize(F) || tapgemm_finalize(G)) return fail(-2, "tap grouping failed");
        F.no_pair = G.no_pair = getenv("LA_NO_PAIR") != nullptr;
        F.dbg_skip_epi = G.dbg_skip_epi = getenv("LA_DBG_SKIP_EPI") != nullptr;     // timing experiment (DESIGN.md §7): wrong results
        const int bnb = pick_bn(c.cin, G.m_tiles);
        LA(make_b_map(G, c.wb, c.cout, c.cin, nmat * (split ? 2 : 1), bnb));
        G.kchunks = c.cout / 64; G.n_total = c.cin; G.n_blocks = c.cin / bnb;
        G.epilogue = kEpiBwd;
        G.OH = G.OW = c.res_in; G.osy = G.osx = 1; G.split = split;
        G.act_gain = F.act_gain; G.act_clamp = F.act_clamp; G.act_slope = F.act_slope;
        G.s_cur = e->s_cat + static_cast<size_t>(B) * c.soff;
        G.red_s = e->red_s + static_cast<size_t>(B) * c.soff;
        G.err_flag = e->err_flag;
        if (prev) {
            const Rgb* prgb = prev->last_in_block ? &e->rgb[prev->block] : nullptr;
            G.xp_hi = prev->x_hi; G.xp_lo = prev->x_lo;
            G.xp_stride_n = static_cast<long long>(prev->res) * prev->res * prev->cout;
            G.g_rgb = prgb ? prgb->g_rgb : nullptr;
            G.rgbw_prev = prgb ? e->rgbw + static_cast<size_t>(B) * prgb->roff : nullptr;
            G.red_rgb = prgb ? e->red_rgb + 3 * static_cast<size_t>(B) * prgb->roff : nullptr;
            G.demod_prev = e->d_cat + static_cast<size_t>(B) * prev->doff;
            G.bias_prev = prev->p.d_bias;
            G.noise_prev = prev->p.d_noise_const; G.noise_prev_stride_n = 0; G.noise_prev_scale = prev->p.noise_strength;
            G.gy_hi = e->gy_hi[(l - 1) & 1]; G.gy_lo = e->gy_lo[(l - 1) & 1];
            G.red_d = e->red_d + static_cast<size_t>(B) * prev->doff;
        } else {
            G.bwd_last = 1;
            G.xp_hi = e->c_rep_hi; G.xp_lo = e->c_rep_lo; G.xp_stride_n = 16LL * c.cin;      // the constant, replicated per sample
        }
    }
    // ---- seed of the backward chain: activation backward of the top layer from the toRGB gradient only
    {
        const Conv& top = e->conv[L - 1];
        const Rgb& rgb = e->rgb[top.block];
        TapGemmParams& Sd = e->seed;
        memset(&Sd, 0, sizeof Sd);
        set_grid(Sd, top.res, B, 1);
        Sd.prob[0].ntaps = 0;
        const int bn = pick_bn(top.cout, Sd.m_tiles);
        Sd.kchunks = 1; Sd.n_total = top.cout; Sd.n_blocks = top.cout / bn;
        Sd.epilogue = kEpiBwd;
        Sd.OH = Sd.OW = top.res; Sd.osy = Sd.osx = 1; Sd.split = split;
        Sd.act_gain = 1.41421356237309515f; Sd.act_clamp = g.conv_clamp; Sd.act_slope = 0.2f;
        Sd.s_cur = e->d_cat + static_cast<size_t>(B) * top.doff;   // multiplied by acc == 0
        Sd.red_s = e->dummy_red;
        Sd.xp_hi = top.x_hi; Sd.xp_lo = top.x_lo;
        Sd.xp_stride_n = static_cast<long long>(top.res) * top.res * top.cout;
        Sd.g_rgb = rgb.g_rgb;
        Sd.rgbw_prev = e->rgbw + static_cast<size_t>(B) * rgb.roff;
        Sd.red_rgb = e->red_rgb + 3 * static_cast<size_t>(B) * rgb.roff;
        Sd.demod_prev = e->d_cat + static_cast<size_t>(B) * top.doff;
        Sd.bias_prev = top.p.d_bias;
        Sd.noise_prev = top.p.d_noise_const; Sd.noise_prev_stride_n = 0; Sd.noise_prev_scale = top.p.noise_strength;
        Sd.gy_hi = e->gy_hi[(L - 1) & 1]; Sd.gy_lo = e->gy_lo[(L - 1) & 1];
        Sd.red_d = e->red_d + static_cast<size_t>(B) * top.doff;
        Sd.err_flag = e->err_flag;
        e->seed_ops = TapSimtOperands{};
    }
    // ---- layer table for the style kernels
    LayerTable& T = e->table;
    memset(&T, 0, sizeof T);
    T.nconv = L; T.nrgb = static_cast<int>(e->rgb.size());
    for (int l = 0; l < L; ++l) {
        const Conv& c = e->conv[l];
        T.conv[l] = ConvDesc{c.w2, c.w2t, c.cin, c.cout, c.soff, c.doff, c.ws_idx};
    }
    for (int r = 0; r < T.nrgb; ++r) {
        const Rgb& q = e->rgb[r];
        T.rgb[r] = RgbDesc{q.p.d_weight, q.cin, g.img_channels, q.soff, q.roff, q.ws_idx};
    }
    return 0;
}

int prepare_weights(la_engine* e, cudaStream_t s) {
    const la_generator_desc& g = e->g;
    const int split = e->split;
    std::vector<int> csoff(e->nchunks), ccin(e->nchunks);
    const float aff_gain = 1.f / sqrtf(static_cast<float>(g.w_dim));
    for (Conv& c : e->conv) {
        LA(prep_conv_weights(c.p.d_weight, c.cout, c.cin, c.split_up ? 1 : c.up, g.d_resample_filter, split, c.wf, c.wb, c.w2, c.w2t, s));
        LA(prep_affine(c.p.d_affine_weight, c.p.d_affine_bias, c.cin, g.w_dim, aff_gain, 1.f,
                       e->a_cat + static_cast<size_t>(c.soff) * g.w_dim, e->b_cat + c.soff, s));
        for (int r = 0; r < c.cin / 64; ++r) { csoff[c.soff / 64 + r] = c.soff; ccin[c.soff / 64 + r] = c.cin; }
    }
    for (Rgb& r : e->rgb) {
        const float wg = 1.f / sqrtf(static_cast<float>(r.cin));      // ToRGB weight_gain folded into the affine
        LA(prep_affine(r.p.d_affine_weight, r.p.d_affine_bias, r.cin, g.w_dim, aff_gain * wg, wg,
                       e->a_cat + static_cast<size_t>(r.soff) * g.w_dim, e->b_cat + r.soff, s));
        for (int q = 0; q < r.cin / 64; ++q) { csoff[r.soff / 64 + q] = r.soff; ccin[r.soff / 64 + q] = r.cin; }
    }
    LA(prep_const(g.d_const, g.channels[0], 16, e->c_f32, e->c_hi, e->c_lo, s));
    for (int n = 0; n < e->batch; ++n) {
        const size_t cn = static_cast<size_t>(16) * g.channels[0];
        CU(cudaMemcpyAsync(e->c_rep_hi + n * cn, e->c_hi, cn * sizeof(bf16), cudaMemcpyDeviceToDevice, s));
        CU(cudaMemcpyAsync(e->c_rep_lo + n * cn, e->c_lo, cn * sizeof(bf16), cudaMemcpyDeviceToDevice, s));
    }
    CU(cudaMemcpyAsync(e->chunk_soff, csoff.data(), sizeof(int) * e->nchunks, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(e->chunk_cin, ccin.data(), sizeof(int) * e->nchunks, cudaMemcpyHostToDevice, s));
    CU(cudaMemsetAsync(e->err_flag, 0, sizeof(int), s));
    CU(cudaMemsetAsync(e->bank_m2, 0, 4 * sizeof(float), s));
    CU(cudaMemsetAsync(e->lat_m2, 0, sizeof(float), s));
    CU(cudaMemsetAsync(e->w_sum, 0, sizeof(float) * g.w_dim, s));
    CU(cudaStreamSynchronize(s));     // host staging vectors go out of scope
    return 0;
}

int gemm(la_engine* e, const TapGemmParams& P, const TapSimtOperands& ops, cudaStream_t s) {
    e->launches++;
    if (e->use_simt) return launch_tapgemm_simt(P, ops, s);
    return launch_tapgemm(P, e->num_sms, s);
}

// styles + demod + the whole synthesis forward.  noise_mode / d_noise patch the epilogue noise source.
int run_forward(la_engine* e, const float* ws, long long sn, long long si, int noise_mode, const float* d_noise, float* d_img_nchw,
                cudaStream_t s) {
    const la_generator_desc& g = e->g;
    const int B = e->batch;
    LA(styles_forward(e->table, ws, sn, si, e->a_cat, e->b_cat, g.w_dim, B, e->s_cat, s));
    LA(demod_rgbw_forward(e->table, B, e->s_cat, e->d_cat, e->rgbw, s));
    LA(const_modulate(e->c_f32, e->s_cat + static_cast<size_t>(B) * e->conv[0].soff, B, 16, g.channels[0], e->split, e->xs_hi[0],
                      e->xs_lo[0], s));
    e->launches += 4;
    const int L = static_cast<int>(e->conv.size());
    for (int l = 0; l < L; ++l) {
        Conv& c = e->conv[l];
        if (c.split_up) {
            LA(gemm(e, c.fwd, c.fwd_ops, s));
            UpFirParams U = c.fir;
            if (noise_mode == LA_NOISE_NONE || c.p.noise_strength == 0.f) U.noise = nullptr;
            else if (noise_mode == LA_NOISE_RANDOM) { U.noise = d_noise + c.noise_off; U.noise_stride_n = static_cast<long long>(c.res) * c.res; }
            LA(upfir_forward(U, s));
            e->launches++;
        } else if (noise_mode == LA_NOISE_CONST) {
            LA(gemm(e, c.fwd, c.fwd_ops, s));
        } else {
            TapGemmParams P = c.fwd;
            if (noise_mode == LA_NOISE_NONE || c.p.noise_strength == 0.f) P.noise = nullptr;
            else { P.noise = d_noise + c.noise_off; P.noise_stride_n = static_cast<long long>(c.res) * c.res; }
            LA(gemm(e, P, c.fwd_ops, s));
        }
        if (c.last_in_block) {
            Rgb& r = e->rgb[c.block];
            const bool top = c.block == g.num_blocks - 1;
            LA(rgb_combine(r.parts, r.nparts, r.p.d_bias, g.img_channels, g.conv_clamp, c.block > 0 ? e->rgb[c.block - 1].img : nullptr,
                           B, r.res, r.img, top ? d_img_nchw : nullptr, s));
            e->launches++;
        }
    }
    return 0;
}

// project: the perceptual term alone, against the per-sample targets (la_project); opt is not read then
int run_backward(la_engine* e, const la_augment_options& opt, bool project, cudaStream_t s) {
    const la_generator_desc& g = e->g;
    const int B = e->batch;
    const int L = static_cast<int>(e->conv.size());
    Rgb& top = e->rgb.back();
    int nparts = 0;
    if (project) {
        CU(cudaMemsetAsync(top.g_img, 0, sizeof(float4) * static_cast<size_t>(B) * g.img_resolution * g.img_resolution, s));
        if (lpips_forward(e->lp, top.img, 1, s, &e->launches) || lpips_backward(e->lp, top.g_img, 1, e->lpips_loss, 1, s, &e->launches))
            return fail(-7, "lpips: %s", lpips_last_error());
    } else if (opt.w_pix > 0.f) {
        LA(pix_loss(top.img, e->bank_mean, e->bank_m2, B, g.img_resolution, g.img_channels, e->crop_off, e->crop_size, e->cur_w_pix,
                    top.g_img, e->loss_parts, &nparts, s));
    } else {
        CU(cudaMemsetAsync(top.g_img, 0, sizeof(float4) * static_cast<size_t>(B) * g.img_resolution * g.img_resolution, s));
    }
    e->n_loss_parts = nparts;
    if (!project && opt.w_disc > 0.f) {          // realism term (util_latent_aug.py:363-371): + w_disc * mean softplus(-D(x))
        if (disc_forward(e->disc, top.img, s, &e->launches) || disc_backward(e->disc, opt.w_disc, top.g_img, 1, e->disc_loss, s, &e->launches))
            return fail(-6, "discriminator: %s", disc_last_error());
    }
    if (!project && opt.w_lpips > 0.f) {   // perceptual term (util_latent_aug.py:387-424): - w_lpips * pair-normalised LPIPS distance to the bank
        if (lpips_forward(e->lp, top.img, 0, s, &e->launches) || lpips_backward(e->lp, top.g_img, 1, e->lpips_loss, 0, s, &e->launches))
            return fail(-7, "lpips: %s", lpips_last_error());
    }
    for (int b = g.num_blocks - 1; b >= 0; --b) {
        Rgb& r = e->rgb[b];
        LA(rgb_backward(r.g_img, r.parts, r.nparts, r.p.d_bias, g.img_channels, g.conv_clamp, B, r.res, r.g_rgb,
                        b > 0 ? e->rgb[b - 1].g_img : nullptr, s));
    }
    LA(launch_tapgemm_seed(e->seed, e->num_sms, s));
    e->launches += 2 + g.num_blocks;
    for (int l = L - 1; l >= 0; --l) {
        if (e->conv[l].split_up) { LA(upfir_backward(e->conv[l].fir, s)); e->launches++; }
        LA(gemm(e, e->conv[l].bwd, e->conv[l].bwd_ops, s));
    }
    LA(style_grad(e->table, B, e->s_cat, e->d_cat, e->red_s, e->red_d, e->red_rgb, e->g_s, s));
    LA(gw_partial(e->g_s, e->a_cat, e->chunk_soff, e->chunk_cin, e->nchunks, B, g.w_dim, e->partial, s));
    e->launches += 3;
    return 0;
}

int run_step(la_engine* e, const la_augment_options& opt, cudaStream_t s) {
    const la_generator_desc& g = e->g;
    const int B = e->batch;
    const bool synth = opt.w_pix > 0.f || opt.w_disc > 0.f || opt.w_lpips > 0.f;
    if (synth) {
        CU(cudaMemsetAsync(e->red_all, 0, e->red_bytes, s));
        LA(run_forward(e, e->w_opt, g.w_dim, 0, LA_NOISE_CONST, nullptr, nullptr, s));
        LA(run_backward(e, opt, false, s));
    }
    LA(adam_step(e->partial, e->nchunks, synth ? 1 : 0, e->w_sum, e->lat_m2, e->consts, e->step, e->w_opt, e->m, e->v, B, g.w_dim,
                 e->loss_parts, synth ? e->n_loss_parts : 0, e->bank_m2, opt.n_modalities, e->crop_size, e->loss_log, LA_MAX_STEPS,
                 opt.w_disc > 0.f ? e->disc_loss : nullptr, opt.w_lpips > 0.f ? e->lpips_loss : nullptr, s));
    e->launches += 3;
    return 0;
}

// one projection step: synthesis from the perturbed code, distance to the targets, scheduled Adam (which also writes the
// next step's perturbed code)
int run_project_step(la_engine* e, cudaStream_t s) {
    const la_generator_desc& g = e->g;
    la_augment_options unused{};
    CU(cudaMemsetAsync(e->red_all, 0, e->red_bytes, s));
    LA(run_forward(e, e->w_pert, g.w_dim, 0, LA_NOISE_CONST, nullptr, nullptr, s));
    LA(run_backward(e, unused, true, s));
    LA(adam_scheduled(e->partial, e->nchunks, e->proj, e->step, e->w_opt, e->m, e->v, e->w_pert, e->batch, g.w_dim, s));
    e->launches += 2;
    return 0;
}

// Runs num_steps of `step` on e->work: the first one ever eagerly (warm-up, flag `warmed`), the rest as replays of one
// captured graph.  after(it) enqueues per-step work outside the graph.
template <class Step, class After>
int run_loop(la_engine* e, int num_steps, bool graphable, bool& warmed, Step step, After after) {
    cudaStream_t w = e->work;
    for (int it = 0; it < num_steps; ++it) {
        if (!graphable || e->graph_disabled || !warmed) {
            LA(step());
            warmed = true;
        } else {
            if (!e->step_graph) {
                cudaGraph_t graph = nullptr;
                const long long before = e->launches;
                CU(cudaStreamBeginCapture(w, cudaStreamCaptureModeThreadLocal));
                int r = step();
                cudaError_t ce = cudaStreamEndCapture(w, &graph);
                e->launches_captured = e->launches - before;
                e->launches = before;
                if (r) { if (graph) cudaGraphDestroy(graph); return r; }
                CU(ce);
                e->graph_kernels = e->launches_captured;
                ce = cudaGraphInstantiate(&e->step_graph, graph, 0);
                cudaGraphDestroy(graph);
                CU(ce);
            }
            CU(cudaGraphLaunch(e->step_graph, w));
            e->launches += e->graph_kernels;
        }
        LA(after(it));
    }
    return 0;
}

int check_err_flag(la_engine* e, cudaStream_t s) {
    int flag = 0;
    CU(cudaMemcpyAsync(&flag, e->err_flag, sizeof(int), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    if (flag) return fail(-3, "tap-GEMM pipeline timeout at site %d", flag);
    return 0;
}

}  // namespace

int la_fail_msg(int code, const char* msg) { return fail(code, "%s", msg); }

// ======================================================================================= C ABI
#define LA_API __attribute__((visibility("default")))
extern "C" {

LA_API const char* la_last_error(void) { return g_err.c_str(); }
LA_API int la_version(void) { return LA_ABI_VERSION; }
LA_API int la_struct_sizes(size_t* out, int max) {
    static_assert(kLossCols == LA_LOSS_COLS, "loss-log row width");
    const size_t v[] = {sizeof(la_generator_desc), sizeof(la_augment_options), sizeof(la_disc_desc), sizeof(la_conv_params),
                        sizeof(la_torgb_params), sizeof(la_disc_block_params), sizeof(la_vgg_desc)};
    int n = 0;
    for (; out && n < max && n < static_cast<int>(sizeof v / sizeof v[0]); ++n) out[n] = v[n];
    return n;
}

LA_API int la_engine_workspace_bytes(const la_generator_desc* g, int batch, int precision, size_t* bytes) {
    if (!g || !bytes || batch < 1) return fail(-2, "bad arguments");
    la_engine tmp{};
    tmp.g = *g; tmp.batch = batch; tmp.split = precision == LA_PRECISION_FP32_PARITY;
    tmp.split_min_res = upconv_split_min_res();
    return plan(&tmp, nullptr, bytes);
}

LA_API int la_engine_create(const la_generator_desc* g, int batch, int precision, void* d_workspace, size_t workspace_bytes, la_stream stream,
                     la_engine** out) {
    if (!g || !out || !d_workspace || batch < 1) return fail(-2, "bad arguments");
    int dev = 0, major = 0, sms = 0;
    CU(cudaGetDevice(&dev));
    CU(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    if (major != 10) return fail(-4, "latentaugment_b200 needs an sm_100 device (found compute capability %d.x); there is no fallback", major);
    la_engine* e = new la_engine{};
    e->g = *g; e->batch = batch; e->split = precision == LA_PRECISION_FP32_PARITY; e->num_sms = sms;
    e->split_min_res = upconv_split_min_res();
    size_t need = 0;
    int r = plan(e, static_cast<char*>(d_workspace), &need);
    if (!r && need > workspace_bytes) r = fail(-2, "workspace too small: %zu < %zu", workspace_bytes, need);
    if (!r && (reinterpret_cast<uintptr_t>(d_workspace) & 1023)) r = fail(-2, "workspace must be 1024-byte aligned");
    const int res = g->img_resolution;
    e->crop_size = static_cast<int>(sqrt(static_cast<double>(res) * res / 2.0));          // util_dataset.py:317-323
    e->crop_off = static_cast<int>(nearbyint((res - e->crop_size) / 2.0));               // torchvision CenterCrop
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (!r) {
        cudaError_t ce = cudaMemcpyAsync(e->fir_host, g->d_resample_filter, sizeof e->fir_host, cudaMemcpyDeviceToHost, s);
        if (ce == cudaSuccess) ce = cudaStreamSynchronize(s);
        if (ce != cudaSuccess) r = fail(static_cast<int>(ce), "reading the resample filter: %s", cudaGetErrorString(ce));
    }
    if (!r) r = build_params(e);
    if (!r) r = prepare_weights(e, s);
    if (!r) {
        cudaError_t ce = cudaStreamCreateWithFlags(&e->work, cudaStreamNonBlocking);
        if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&e->ev_in, cudaEventDisableTiming);
        if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&e->ev_out, cudaEventDisableTiming);
        if (ce != cudaSuccess) r = fail(static_cast<int>(ce), "stream/event creation: %s", cudaGetErrorString(ce));
    }
    e->graph_disabled = getenv("LA_NO_GRAPH") != nullptr;
    if (r) { la_engine_destroy(e); return r; }
    *out = e;
    return 0;
}

LA_API void la_engine_destroy(la_engine* e) {
    if (!e) return;
    if (e->disc) disc_destroy(e->disc);
    if (e->lp) lpips_destroy(e->lp);
    if (e->step_graph) cudaGraphExecDestroy(e->step_graph);
    if (e->ev_in) cudaEventDestroy(e->ev_in);
    if (e->ev_out) cudaEventDestroy(e->ev_out);
    if (e->work) cudaStreamDestroy(e->work);
    delete e;
}

LA_API int la_set_latent_bank(la_engine* e, const float* d_W, int M, la_stream stream) {
    if (!e || !d_W || M < 1) return fail(-2, "bad arguments");
    LA(latent_bank_stats(d_W, M, e->num_ws, e->g.w_dim, e->w_sum, e->lat_m2, static_cast<cudaStream_t>(stream)));
    e->has_lat_bank = 1;
    return 0;
}

LA_API int la_set_image_bank(la_engine* e, const float* d_X, int M, la_stream stream) {
    if (!e || !d_X || M < 1) return fail(-2, "bad arguments");
    LA(image_bank_stats(d_X, M, e->g.img_channels, e->g.img_resolution, e->crop_off, e->crop_size, e->bank_mean, e->bank_m2,
                        static_cast<cudaStream_t>(stream)));
    e->has_img_bank = 1;
    return 0;
}

LA_API int la_mapping(la_engine* e, const float* d_z, int n, float psi, float* d_w, la_stream stream) {
    if (!e || !d_z || !d_w || n < 1 || n > e->batch) return fail(-2, "bad arguments");
    const la_generator_desc& g = e->g;
    if (g.mapping_layers < 1) return fail(-2, "engine was created without a mapping network");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    LA(mapping_normalize(d_z, n, g.z_dim, e->map_a, s));
    float* cur = e->map_a;
    float* nxt = e->map_b;
    int n_in = g.z_dim;
    for (int i = 0; i < g.mapping_layers; ++i) {
        const float wg = g.mapping_lr_multiplier / sqrtf(static_cast<float>(n_in));
        LA(mapping_fc(cur, g.d_mapping_weight[i], g.d_mapping_bias[i], n, n_in, g.w_dim, wg, g.mapping_lr_multiplier, 1, nxt, s));
        float* t = cur; cur = nxt; nxt = t;
        n_in = g.w_dim;
    }
    if (psi != 1.f) LA(mapping_truncate(cur, g.d_w_avg, psi, n, g.w_dim, d_w, s));
    else CU(cudaMemcpyAsync(d_w, cur, sizeof(float) * n * g.w_dim, cudaMemcpyDeviceToDevice, s));
    return 0;
}

LA_API size_t la_noise_floats(const la_engine* e) {
    size_t n = 0;
    for (const Conv& c : e->conv) n += static_cast<size_t>(e->batch) * c.res * c.res;
    return n;
}

static int bridge_in(la_engine* e, cudaStream_t s) {
    CU(cudaEventRecord(e->ev_in, s));
    CU(cudaStreamWaitEvent(e->work, e->ev_in, 0));
    return 0;
}
static int bridge_out(la_engine* e, cudaStream_t s) {
    CU(cudaEventRecord(e->ev_out, e->work));
    CU(cudaStreamWaitEvent(s, e->ev_out, 0));
    return 0;
}

LA_API int la_synthesis(la_engine* e, const float* d_ws, long long stride_n, long long stride_i, int noise_mode, const float* d_noise,
                 float* d_img, la_stream stream) {
    if (!e || !d_ws || !d_img) return fail(-2, "bad arguments");
    if (noise_mode == LA_NOISE_RANDOM && !d_noise) return fail(-2, "noise_mode random needs d_noise");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    LA(bridge_in(e, s));
    LA(run_forward(e, d_ws, stride_n, stride_i, noise_mode, d_noise, d_img, e->work));
    LA(bridge_out(e, s));
    return 0;
}

LA_API int la_augment(la_engine* e, const float* d_w0, const la_augment_options* opt, const float* d_final_noise, float* d_img, float* d_w_aug,
               float* d_loss_log, la_stream stream) {
    if (!e || !d_w0 || !opt || !d_img || !d_w_aug) return fail(-2, "bad arguments");
    if (opt->num_steps < 0) return fail(-2, "num_steps must be >= 0");      // (only the first LA_MAX_STEPS loss rows are logged)
    if (opt->w_pix > 0.f && !e->has_img_bank) return fail(-2, "w_pix > 0 needs la_set_image_bank");
    if (opt->w_latent > 0.f && !e->has_lat_bank) return fail(-2, "w_latent > 0 needs la_set_latent_bank");
    if (opt->final_noise_mode == LA_NOISE_RANDOM && !d_final_noise) return fail(-2, "final_noise_mode random needs d_final_noise");
    if (opt->n_modalities != e->g.img_channels) return fail(-2, "n_modalities must equal img_channels");
    if (opt->w_disc > 0.f && !e->disc) return fail(-2, "w_disc > 0 needs la_set_discriminator");
    if (opt->w_lpips > 0.f && (!e->lp || !lpips_has_bank(e->lp))) return fail(-2, "w_lpips > 0 needs la_set_lpips and la_set_feature_bank");
    const la_generator_desc& g = e->g;
    const int B = e->batch;
    const size_t wbytes = sizeof(float) * B * g.w_dim;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    cudaStream_t w = e->work;
    LA(bridge_in(e, s));
    AdamConsts hc{opt->lr, 0.9f, 0.999f, 1e-8f, opt->w_latent, opt->w_pix, e->num_ws, e->has_lat_bank};
    CU(cudaMemcpyAsync(e->consts, &hc, sizeof hc, cudaMemcpyHostToDevice, w));
    CU(cudaMemcpyAsync(e->w_opt, d_w0, wbytes, cudaMemcpyDeviceToDevice, w));
    CU(cudaMemcpyAsync(e->w0, d_w0, wbytes, cudaMemcpyDeviceToDevice, w));
    CU(cudaMemsetAsync(e->m, 0, wbytes, w));
    CU(cudaMemsetAsync(e->v, 0, wbytes, w));
    CU(cudaMemsetAsync(e->step, 0, sizeof(int), w));
    CU(cudaMemsetAsync(e->loss_log, 0, sizeof(float) * LA_LOSS_COLS * LA_MAX_STEPS, w));
    if (opt->w_lpips > 0.f) {        // crop window of this call (util_dataset.py:284-309,325-332), absolute image coordinates
        if (lpips_set_call(e->lp, opt->lpips_crop_x, opt->lpips_crop_y, opt->w_lpips, opt->lpips_norm_mode, w))
            return fail(-7, "lpips: %s", lpips_last_error());
    }
    if ((e->cur_project || e->cur_w_pix != opt->w_pix || e->cur_w_disc != opt->w_disc || (e->cur_w_lpips > 0.f) != (opt->w_lpips > 0.f)) &&
        e->step_graph) {   // baked into the criterion launches
        cudaGraphExecDestroy(e->step_graph);
        e->step_graph = nullptr;
    }
    e->cur_project = 0;
    e->cur_w_pix = opt->w_pix;
    e->cur_w_disc = opt->w_disc;
    e->cur_w_lpips = opt->w_lpips;
    const bool synth = opt->w_pix > 0.f || opt->w_disc > 0.f || opt->w_lpips > 0.f;
    LA(run_loop(e, opt->num_steps, synth, e->warmed, [&] { return run_step(e, *opt, w); }, [](int) { return 0; }));
    LA(finalize_w(e->w_opt, e->w0, opt->alpha, opt->soft_aug, B, g.w_dim, e->w_aug, w));
    LA(run_forward(e, e->w_aug, g.w_dim, 0, opt->final_noise_mode, d_final_noise, d_img, w));
    CU(cudaMemcpyAsync(d_w_aug, e->w_aug, wbytes, cudaMemcpyDeviceToDevice, w));
    if (d_loss_log && opt->num_steps > 0)
        CU(cudaMemcpyAsync(d_loss_log, e->loss_log, sizeof(float) * LA_LOSS_COLS * (opt->num_steps < LA_MAX_STEPS ? opt->num_steps : LA_MAX_STEPS),
                           cudaMemcpyDeviceToDevice, w));
    LA(bridge_out(e, s));
    return 0;
}

LA_API int la_set_projection_targets(la_engine* e, const float* d_img, la_stream stream) {
    if (!e || !d_img) return fail(-2, "bad arguments");
    if (!e->lp) return fail(-2, "la_set_projection_targets needs la_set_lpips (with per_sample_targets = 1)");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    Rgb& top = e->rgb.back();
    LA(bridge_in(e, s));
    LA(nchw_to_f4(d_img, e->batch, e->g.img_channels, e->g.img_resolution, top.img, e->work));
    if (lpips_set_targets(e->lp, top.img, e->work, &e->launches)) return fail(-7, "lpips: %s", lpips_last_error());
    LA(bridge_out(e, s));
    return 0;
}

LA_API int la_project(la_engine* e, const float* d_w0, int num_steps, const float* d_lr, const float* d_sigma, const float* d_wnoise,
                      float* d_w_out, float* d_loss_log, la_stream stream) {
    if (!e || !d_w0 || !d_w_out || num_steps < 0 || (num_steps > 0 && (!d_lr || !d_sigma))) return fail(-2, "bad arguments");
    if (!e->lp || !lpips_has_targets(e->lp)) return fail(-2, "la_project needs la_set_lpips and la_set_projection_targets");
    const int B = e->batch, wd = e->g.w_dim;
    const size_t wbytes = sizeof(float) * B * wd;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    cudaStream_t w = e->work;
    LA(bridge_in(e, s));
    const ProjConsts hc{d_lr, d_sigma, d_wnoise, num_steps};
    CU(cudaMemcpyAsync(e->proj, &hc, sizeof hc, cudaMemcpyHostToDevice, w));
    if (lpips_set_call(e->lp, 0, 0, 1.f, 1, w)) return fail(-7, "lpips: %s", lpips_last_error());      // whole-image window
    CU(cudaMemcpyAsync(e->w_opt, d_w0, wbytes, cudaMemcpyDeviceToDevice, w));
    CU(cudaMemsetAsync(e->m, 0, wbytes, w));
    CU(cudaMemsetAsync(e->v, 0, wbytes, w));
    CU(cudaMemsetAsync(e->step, 0, sizeof(int), w));
    LA(perturb_first(e->w_opt, e->proj, e->w_pert, B, wd, w));
    if (!e->cur_project && e->step_graph) {       // never replay an augmentation step here (nor the reverse, la_augment)
        cudaGraphExecDestroy(e->step_graph);
        e->step_graph = nullptr;
    }
    e->cur_project = 1;
    e->cur_w_pix = e->cur_w_disc = e->cur_w_lpips = -1.f;
    LA(run_loop(e, num_steps, true, e->proj_warmed, [&] { return run_project_step(e, w); },
                [&](int it) { return d_loss_log ? sum_floats(e->lpips_loss, B, d_loss_log + it, w) : 0; }));
    CU(cudaMemcpyAsync(d_w_out, e->w_opt, wbytes, cudaMemcpyDeviceToDevice, w));
    LA(bridge_out(e, s));
    return 0;
}

LA_API int la_disc_workspace_bytes(const la_disc_desc* d, int batch, int precision, size_t* bytes) {
    if (!d || !bytes || batch < 1) return fail(-2, "bad arguments");
    if (disc_workspace_bytes(*d, batch, precision == LA_PRECISION_FP32_PARITY, bytes)) return fail(-2, "%s", disc_last_error());
    return 0;
}

LA_API int la_set_discriminator(la_engine* e, const la_disc_desc* d, void* d_workspace, size_t workspace_bytes, la_stream stream) {
    if (!e || !d || !d_workspace) return fail(-2, "bad arguments");
    if (d->img_resolution != e->g.img_resolution || d->img_channels != e->g.img_channels)
        return fail(-2, "discriminator shape %dx%d (%d ch) does not match the generator", d->img_resolution, d->img_resolution, d->img_channels);
    if (e->disc) { disc_destroy(e->disc); e->disc = nullptr; }
    if (e->step_graph) { cudaGraphExecDestroy(e->step_graph); e->step_graph = nullptr; }
    if (disc_create(*d, e->batch, e->split, e->num_sms, d_workspace, workspace_bytes, static_cast<cudaStream_t>(stream), &e->disc))
        return fail(-6, "discriminator: %s", disc_last_error());
    return 0;
}

LA_API int la_disc_logits(la_engine* e, const float* d_img, float* d_logits, la_stream stream) {
    if (!e || !e->disc || !d_img || !d_logits) return fail(-2, "bad arguments (la_set_discriminator first)");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    Rgb& top = e->rgb.back();
    LA(bridge_in(e, s));
    LA(nchw_to_f4(d_img, e->batch, e->g.img_channels, e->g.img_resolution, top.img, e->work));
    if (disc_forward(e->disc, top.img, e->work, &e->launches)) return fail(-6, "discriminator: %s", disc_last_error());
    CU(cudaMemcpyAsync(d_logits, disc_logits(e->disc), sizeof(float) * e->batch, cudaMemcpyDeviceToDevice, e->work));
    LA(bridge_out(e, s));
    return 0;
}

LA_API int la_disc_loss_grad(la_engine* e, const float* d_img, float w_disc, float* d_loss, float* d_grad, la_stream stream) {
    if (!e || !e->disc || !d_img || !d_loss || !d_grad) return fail(-2, "bad arguments (la_set_discriminator first)");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    Rgb& top = e->rgb.back();
    LA(bridge_in(e, s));
    LA(nchw_to_f4(d_img, e->batch, e->g.img_channels, e->g.img_resolution, top.img, e->work));
    if (disc_forward(e->disc, top.img, e->work, &e->launches) ||
        disc_backward(e->disc, w_disc, top.g_img, 0, e->disc_loss, e->work, &e->launches))
        return fail(-6, "discriminator: %s", disc_last_error());
    LA(f4_to_nchw(top.g_img, e->batch, e->g.img_channels, e->g.img_resolution, d_grad, e->work));
    CU(cudaMemcpyAsync(d_loss, e->disc_loss, sizeof(float), cudaMemcpyDeviceToDevice, e->work));
    LA(bridge_out(e, s));
    return 0;
}

LA_API int la_lpips_workspace_bytes(const la_vgg_desc* v, int batch, int img_channels, int precision, size_t* bytes) {
    if (!v || !bytes || batch < 1) return fail(-2, "bad arguments");
    if (lpips_workspace_bytes(*v, batch, img_channels, precision == LA_PRECISION_FP32_PARITY, bytes)) return fail(-2, "%s", lpips_last_error());
    return 0;
}

LA_API int la_set_lpips(la_engine* e, const la_vgg_desc* v, void* d_workspace, size_t workspace_bytes, la_stream stream) {
    if (!e || !v || !d_workspace) return fail(-2, "bad arguments");
    if (e->lp) { lpips_destroy(e->lp); e->lp = nullptr; }
    if (e->step_graph) { cudaGraphExecDestroy(e->step_graph); e->step_graph = nullptr; }
    if (lpips_create(*v, e->batch, e->g.img_channels, e->g.img_resolution, e->split, e->num_sms, d_workspace, workspace_bytes,
                     static_cast<cudaStream_t>(stream), &e->lp))
        return fail(-7, "lpips: %s", lpips_last_error());
    return 0;
}

LA_API int la_set_feature_bank(la_engine* e, const float* d_crops, int M, la_stream stream) {
    if (!e || !e->lp || !d_crops || M < 1) return fail(-2, "bad arguments (la_set_lpips first)");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    LA(bridge_in(e, s));
    if (lpips_set_bank(e->lp, d_crops, M, e->work, &e->launches)) return fail(-7, "lpips: %s", lpips_last_error());
    LA(bridge_out(e, s));
    return 0;
}

LA_API int la_lpips_loss_grad(la_engine* e, const float* d_img, int crop_x, int crop_y, float w_lpips, int norm_mode, float* d_loss,
                              float* d_grad, la_stream stream) {
    if (!e || !e->lp || !d_img || !d_loss || !d_grad) return fail(-2, "bad arguments (la_set_lpips first)");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    Rgb& top = e->rgb.back();
    LA(bridge_in(e, s));
    LA(nchw_to_f4(d_img, e->batch, e->g.img_channels, e->g.img_resolution, top.img, e->work));
    if (norm_mode == 2) {             // the projection's per-sample distance to the targets: the window is the whole image
        if (crop_x != 0 || crop_y != 0) return fail(-2, "norm_mode 2 (per-sample targets) uses the whole image: crop_x = crop_y = 0");
        if (lpips_set_call(e->lp, 0, 0, 1.f, 1, e->work) || lpips_forward(e->lp, top.img, 1, e->work, &e->launches) ||
            lpips_backward(e->lp, top.g_img, 0, e->lpips_loss, 1, e->work, &e->launches))
            return fail(-7, "lpips: %s", lpips_last_error());
        LA(f4_to_nchw(top.g_img, e->batch, e->g.img_channels, e->g.img_resolution, d_grad, e->work));
        CU(cudaMemcpyAsync(d_loss, e->lpips_loss, sizeof(float) * e->batch, cudaMemcpyDeviceToDevice, e->work));
        LA(bridge_out(e, s));
        return 0;
    }
    // (the term enters the objective with a minus sign; the stand-alone call returns d loss / d img, hence -w)
    if (lpips_set_call(e->lp, crop_x, crop_y, -w_lpips, norm_mode, e->work) ||
        lpips_forward(e->lp, top.img, 0, e->work, &e->launches) || lpips_backward(e->lp, top.g_img, 0, e->lpips_loss, 0, e->work, &e->launches))
        return fail(-7, "lpips: %s", lpips_last_error());
    LA(f4_to_nchw(top.g_img, e->batch, e->g.img_channels, e->g.img_resolution, d_grad, e->work));
    LA(prep_scale(e->lpips_loss, -1.f, e->lpips_loss, 1, e->work));
    CU(cudaMemcpyAsync(d_loss, e->lpips_loss, sizeof(float), cudaMemcpyDeviceToDevice, e->work));
    LA(bridge_out(e, s));
    return 0;
}

LA_API int la_lpips_tap(la_engine* e, int k, float* d_out, size_t* count, la_stream stream) {
    if (!e || !e->lp) return fail(-2, "bad arguments (la_set_lpips first)");
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (d_out) LA(bridge_in(e, s));
    if (lpips_copy_tap(e->lp, k, d_out, count, e->work)) return fail(-7, "lpips: %s", lpips_last_error());
    if (d_out) LA(bridge_out(e, s));
    return 0;
}

LA_API int la_debug_set_simt(la_engine* e, int use_simt) {
    if (!e) return fail(-2, "bad arguments");
    e->use_simt = use_simt;
    if (e->step_graph) { cudaGraphExecDestroy(e->step_graph); e->step_graph = nullptr; }
    return 0;
}
LA_API long long la_debug_launch_count(const la_engine* e) { return e ? e->launches : 0; }

// Times every tap-GEMM launch of one optimisation step in isolation (CUDA events on the launch
// stream, `reps` back-to-back launches each; buffers hold whatever the last call left).
// h_ms: host array [4*L + 1] = forward GEMM[0..L), data-gradient GEMM[0..L), FIR pass fwd[0..L), FIR pass bwd[0..L), seed.
LA_API int la_debug_time_gemms(la_engine* e, int reps, float* h_ms, int* n_layers) {
    if (!e || !h_ms || reps < 1) return fail(-2, "bad arguments");
    const int L = static_cast<int>(e->conv.size());
    if (n_layers) *n_layers = L;
    cudaEvent_t a, b;
    CU(cudaEventCreate(&a));
    CU(cudaEventCreate(&b));
    cudaStream_t w = e->work;
    const bool dbg_clk = getenv("LA_DBG_CLK") != nullptr;
    auto timed = [&](int idx, const TapGemmParams& P0, const TapSimtOperands& ops, bool simt) -> int {
        TapGemmParams P = P0;
        if (dbg_clk && !simt) P.dbg_clock = e->dbg_clock;
        for (int warm = 0; warm < 2; ++warm) { int r = simt ? launch_tapgemm_seed(P, e->num_sms, w) : launch_tapgemm(P, e->num_sms, w); if (r) return r; }
        cudaEventRecord(a, w);
        for (int i = 0; i < reps; ++i) { int r = simt ? launch_tapgemm_seed(P, e->num_sms, w) : launch_tapgemm(P, e->num_sms, w); if (r) return r; }
        cudaEventRecord(b, w);
        cudaError_t ce = cudaEventSynchronize(b);
        if (ce != cudaSuccess) return static_cast<int>(ce);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, a, b);
        h_ms[idx] = ms / reps;
        if (dbg_clk && !simt) {
            unsigned long long hc[64] = {0, 1, 0, 0, 0, 0, 0, 0};
            cudaMemcpy(hc, e->dbg_clock, sizeof hc, cudaMemcpyDeviceToHost);
            fprintf(stderr, "[clk] gemm %2d: %.3f ms, CTA0 %.0f MHz over %.3f ms | us since CTA start: roles %.1f, first operands %.1f, unit 0 issued %.1f, all %llu units issued %.1f, exit %.1f\n",
                    idx, h_ms[idx], 1e3 * hc[0] / hc[1], hc[1] * 1e-6, (hc[2] - hc[7]) * 1e-3, (hc[3] - hc[7]) * 1e-3,
                    (hc[4] - hc[7]) * 1e-3, hc[6], (hc[5] - hc[7]) * 1e-3, hc[1] * 1e-3);
            fprintf(stderr, "[clk]    MMA thread waited (us): accumulator free %.1f, A landed %.1f, B landed %.1f\n", hc[60] * 1e-3, hc[61] * 1e-3, hc[62] * 1e-3);
            if (getenv("LA_DBG_STEPS")) {
                fprintf(stderr, "[clk]    A-group issue -> landed (us since CTA start):");
                for (int k = 0; k < 28; ++k) fprintf(stderr, " %.2f>%.2f", (hc[8 + 2 * k] - hc[7]) * 1e-3, (hc[9 + 2 * k] - hc[7]) * 1e-3);
                fprintf(stderr, "\n");
            }
        }
        return 0;
    };
    auto timed_fir = [&](int idx, const UpFirParams& U, bool fwd) -> int {
        for (int warm = 0; warm < 2; ++warm) { int r = fwd ? upfir_forward(U, w) : upfir_backward(U, w); if (r) return r; }
        cudaEventRecord(a, w);
        for (int i = 0; i < reps; ++i) { int r = fwd ? upfir_forward(U, w) : upfir_backward(U, w); if (r) return r; }
        cudaEventRecord(b, w);
        cudaError_t ce = cudaEventSynchronize(b);
        if (ce != cudaSuccess) return static_cast<int>(ce);
        float ms = 0.f;
        cudaEventElapsedTime(&ms, a, b);
        h_ms[idx] = ms / reps;
        return 0;
    };
    for (int l = 0; l < L; ++l) {
        LA(timed(l, e->conv[l].fwd, e->conv[l].fwd_ops, false));
        LA(timed(L + l, e->conv[l].bwd, e->conv[l].bwd_ops, false));
        h_ms[2 * L + l] = h_ms[3 * L + l] = 0.f;
        if (e->conv[l].split_up) {
            LA(timed_fir(2 * L + l, e->conv[l].fir, true));
            LA(timed_fir(3 * L + l, e->conv[l].fir, false));
        }
    }
    LA(timed(4 * L, e->seed, e->seed_ops, true));   // 'simt' flag selects the seed launcher here
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    return 0;
}

// Test hook: copies an internal per-step quantity of the LAST optimisation step to d_out (fp32) and reports its element count
// (d_out may be null).  what = 0: style gradients g_s [layer-blocked: batch * soff_l + n * cin_l + i, conv layers then toRGB
// layers]; 1: styles s (same layout); 2: demodulation coefficients d [batch * doff_l + n * cout_l + o]; 3: d loss / d w of the
// synthesis path [batch, w_dim] (sum of the per-chunk partials); 4: per-layer block offsets as floats [nconv + nrgb] (soff).
LA_API int la_debug_get(la_engine* e, int what, float* d_out, size_t* count, la_stream stream) {
    if (!e || !count) return fail(-2, "bad arguments");
    const size_t B = e->batch;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (what == 4) {
        std::vector<float> off;
        for (const Conv& c : e->conv) off.push_back(static_cast<float>(c.soff));
        for (const Rgb& r : e->rgb) off.push_back(static_cast<float>(r.soff));
        *count = off.size();
        if (d_out) { CU(cudaMemcpyAsync(d_out, off.data(), sizeof(float) * off.size(), cudaMemcpyHostToDevice, s)); CU(cudaStreamSynchronize(s)); }
        return 0;
    }
    const float* src = what == 0 ? e->g_s : (what == 1 ? e->s_cat : (what == 2 ? e->d_cat : nullptr));
    const size_t n = what == 2 ? B * e->D : (what == 3 ? B * e->g.w_dim : B * e->S);
    if (what < 0 || what > 3) return fail(-2, "unknown quantity %d", what);
    *count = n;
    if (!d_out) return 0;
    LA(bridge_in(e, s));
    if (what == 3) {
        CU(cudaMemsetAsync(d_out, 0, sizeof(float) * n, e->work));
        for (int c = 0; c < e->nchunks; ++c) LA(prep_axpy(e->partial + static_cast<size_t>(c) * n, 1.f, d_out, static_cast<long long>(n), e->work));
    } else {
        CU(cudaMemcpyAsync(d_out, src, sizeof(float) * n, cudaMemcpyDeviceToDevice, e->work));
    }
    LA(bridge_out(e, s));
    return 0;
}

LA_API int la_debug_check(la_engine* e, la_stream stream) { return e ? check_err_flag(e, static_cast<cudaStream_t>(stream)) : -2; }

}  // extern "C"
