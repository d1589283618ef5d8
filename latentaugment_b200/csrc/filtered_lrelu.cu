// filtered_lrelu: bias -> zero-insert up-sampling -> pad -> FIR (fu, gain up^2) -> leaky ReLU * gain -> clamp ->
// FIR (fd) -> decimation, fused per tile (reference models/stylegan3/torch_utils/ops/filtered_lrelu.py:56-153,
// composition of the ref path :121-153; the building block of the StyleGAN3 synthesis layers, SURVEY.md row a23).
//
// One block computes a 16 x 16 output tile of one (sample, channel) plane entirely in shared memory with
// separable passes:  x tile -> horizontal up-FIR (polyphase: only the non-zero taps) -> vertical up-FIR +
// activation -> horizontal down-FIR + decimation -> vertical down-FIR + decimation.  Every input element is read
// from global memory once per tile (+ halo), the up-sampled intermediate never leaves the SM.
// With `mask_out` the activation writes its derivative class per intermediate pixel (0 clamped, 1 positive,
// 2 negative); with `mask_in` the activation is replaced by that derivative -- the backward pass is the same
// kernel with the roles of the two filters swapped (python: latentaugment_b200/ops_sg3.py).
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/latentaugment_b200.h"
#include "common.cuh"

namespace {

constexpr int kTile = 16;          // output tile edge
constexpr int kMaxTaps = 32;

struct FlParams {
    const float* x; const float* b; float* y;
    const int8_t* mask_in; int8_t* mask_out;
    int N, C, H, W;                // input plane
    int up, down;
    int px0, py0;                  // leading pads (in up-sampled pixels; may be negative = crop)
    int mid_h, mid_w;              // intermediate (after the up FIR) extent
    int out_h, out_w;
    int fu_taps, fd_taps;
    float fu[kMaxTaps], fd[kMaxTaps];   // correlation-form taps (already flipped as needed), fu includes the gain `up` per axis
    float gain, slope, clamp;
    int in_t, mid_t;               // tile extents in shared memory: input rows/cols, intermediate rows/cols
    int mask_oy, mask_ox, mask_h, mask_w;   // the mask tensor [N*C, mask_h, mask_w] covers intermediate rows mask_oy.., cols mask_ox..
};

// UP / DOWN / FU / FD > 0 fix the factors and tap counts at compile time (unrolled tap loops); 0 = read them from P.
template <int UP, int DOWN, int FU, int FD>
__global__ void __launch_bounds__(256) filtered_lrelu_kernel(const __grid_constant__ FlParams P) {
    extern __shared__ float sm[];
    const int in_t = P.in_t, mid_t = P.mid_t;
    float* s_in = sm;                              // [in_t][in_t]
    float* s_h = s_in + in_t * in_t;               // [in_t][mid_t]   horizontally up-filtered
    float* s_mid = s_h + in_t * mid_t;             // [mid_t][mid_t]  activated intermediate
    float* s_d = s_mid + mid_t * mid_t;            // [mid_t][kTile]  horizontally down-filtered + decimated
    float* s_fu = s_d + mid_t * kTile;             // taps (dynamic per-thread indices: shared memory, not the constant bank)
    float* s_fd = s_fu + kMaxTaps;
    const int plane = blockIdx.z, c = plane % P.C;
    const int ox0 = blockIdx.x * kTile, oy0 = blockIdx.y * kTile;
    const int up = UP ? UP : P.up, down = DOWN ? DOWN : P.down, fu_taps = FU ? FU : P.fu_taps, fd_taps = FD ? FD : P.fd_taps;
    // intermediate window of this tile: rows/cols [my0, my0 + mid_t), m = o * down + k
    const int mx0 = ox0 * down, my0 = oy0 * down;
    // U[m] = sum_k fu[k] * P[m + k],  P[r] = xup[r - p0],  xup[r] = x[r / up] if r % up == 0
    // first input index that can contribute to the window: ceil((m0 - p0) / up)
    auto first_in = [&](int m0, int p0) { const int r = m0 - p0; return r >= 0 ? (r + up - 1) / up : -((-r) / up); };
    const int ix0 = first_in(mx0, P.px0), iy0 = first_in(my0, P.py0);
    if (threadIdx.x < kMaxTaps) {
        s_fu[threadIdx.x] = threadIdx.x < fu_taps ? P.fu[threadIdx.x] : 0.f;
        s_fd[threadIdx.x] = threadIdx.x < fd_taps ? P.fd[threadIdx.x] : 0.f;
    }
    const float bias = P.b ? P.b[c] : 0.f;
    const float* xp = P.x + static_cast<long long>(plane) * P.H * P.W;
    {   // input tile: thread = column, rows strided
        const int q = threadIdx.x % in_t, r0 = threadIdx.x / in_t, rs = blockDim.x / in_t;
        const int ix = ix0 + q;
        const bool cok = ix >= 0 && ix < P.W;
        if (r0 < rs)
            for (int r = r0; r < in_t; r += rs) {
                const int iy = iy0 + r;
                s_in[r * in_t + q] = (cok && iy >= 0 && iy < P.H) ? xp[static_cast<long long>(iy) * P.W + ix] + bias : 0.f;
            }
    }
    __syncthreads();
    {   // horizontal up-FIR: thread = intermediate column (its polyphase taps and first input are fixed), rows strided
        const int m = threadIdx.x % mid_t, r0 = threadIdx.x / mid_t, rs = blockDim.x / mid_t;
        const int mm = mx0 + m;
        const int k0 = ((P.px0 - mm) % up + up) % up;                 // taps k0, k0 + up, ... hit non-zero samples
        const int ib = (mm + k0 - P.px0) / up - ix0;                  // input column of tap k0 (>= 0 by construction of ix0)
        const bool cok = mm < P.mid_w;
        if (r0 < rs)
            for (int r = r0; r < in_t; r += rs) {
                float a = 0.f;
                if (cok) {
                    const float* src = s_in + r * in_t + ib;
#pragma unroll
                    for (int k = k0, i = 0; k < fu_taps; k += up, ++i) a = fmaf(s_fu[k], src[i], a);
                }
                s_h[r * mid_t + m] = a;
            }
    }
    __syncthreads();
    {   // vertical up-FIR + activation: thread = intermediate column, rows strided (the row fixes the polyphase)
        const int n = threadIdx.x % mid_t, r0 = threadIdx.x / mid_t, rs = blockDim.x / mid_t;
        const int nn = mx0 + n;
        const int mx = nn - P.mask_ox;
        const bool cok = nn < P.mid_w, mxok = mx >= 0 && mx < P.mask_w;
        if (r0 < rs)
            for (int m = r0; m < mid_t; m += rs) {
                const int mm = my0 + m;
                float a = 0.f;
                if (cok && mm < P.mid_h) {
                    const int k0 = ((P.py0 - mm) % up + up) % up;
                    const int ib = (mm + k0 - P.py0) / up - iy0;
                    const float* src = s_h + ib * mid_t + n;
#pragma unroll
                    for (int k = k0, i = 0; k < fu_taps; k += up, ++i) a = fmaf(s_fu[k], src[i * mid_t], a);
                    const int my = mm - P.mask_oy;
                    const bool m_ok = mxok && my >= 0 && my < P.mask_h;
                    const long long mi = (static_cast<long long>(plane) * P.mask_h + my) * P.mask_w + mx;
                    if (P.mask_in) {
                        const int8_t cls = m_ok ? P.mask_in[mi] : 0;
                        a = a * P.gain * (cls == 1 ? 1.f : (cls == 2 ? P.slope : 0.f));
                    } else {
                        int8_t cls = a > 0.f ? 1 : 2;     // (bias_act: the negative side includes 0)
                        a = (a > 0.f ? a : a * P.slope) * P.gain;
                        if (P.clamp >= 0.f && !(fabsf(a) < P.clamp)) { a = fminf(fmaxf(a, -P.clamp), P.clamp); cls = 0; }
                        // every tile that covers the pixel computes the same class: benign duplicate writes in the halo
                        if (P.mask_out && m_ok) P.mask_out[mi] = cls;
                    }
                }
                s_mid[m * mid_t + n] = a;
            }
    }
    __syncthreads();
    {   // horizontal down-FIR + decimation: s_d[m][o] = sum_k fd[k] * s_mid[m][o * down + k]; thread = output column
        const int o = threadIdx.x % kTile, r0 = threadIdx.x / kTile, rs = blockDim.x / kTile;
        for (int m = r0; m < mid_t; m += rs) {
            const float* row = s_mid + m * mid_t + o * down;
            float a = 0.f;
#pragma unroll
            for (int k = 0; k < fd_taps; ++k) a = fmaf(s_fd[k], row[k], a);
            s_d[m * kTile + o] = a;
        }
    }
    __syncthreads();
    {
        const int o = threadIdx.x / kTile, q = threadIdx.x % kTile;           // output (row, col) of the tile
        const int oy = oy0 + o, ox = ox0 + q;
        if (oy < P.out_h && ox < P.out_w) {
            float a = 0.f;
            const float* col = s_d + (o * down) * kTile + q;
#pragma unroll
            for (int k = 0; k < fd_taps; ++k) a = fmaf(s_fd[k], col[k * kTile], a);
            P.y[(static_cast<long long>(plane) * P.out_h + oy) * P.out_w + ox] = a;
        }
    }
}

}  // namespace

extern "C" __attribute__((visibility("default")))
int la_filtered_lrelu(const float* d_x, int N, int C, int H, int W, const float* h_fu, int fu_taps, const float* h_fd, int fd_taps,
                      const float* d_b, int up, int down, int px0, int px1, int py0, int py1, float gain, float slope, float clamp,
                      int flip_filter, const signed char* d_mask_in, signed char* d_mask_out, int mask_oy, int mask_ox, int mask_h, int mask_w,
                      float* d_y, la_stream stream) {
    if (!d_x || !d_y || N < 1 || C < 1 || H < 1 || W < 1) return la::fail(-2, "filtered_lrelu: bad arguments");
    if (up < 1 || up > 4 || down < 1 || down > 4) return la::fail(-2, "filtered_lrelu: up and down must be 1..4");
    if (fu_taps < 0 || fu_taps > kMaxTaps || fd_taps < 0 || fd_taps > kMaxTaps) return la::fail(-2, "filtered_lrelu: at most 32 separable taps per filter");
    FlParams P{};
    P.x = d_x; P.b = d_b; P.y = d_y; P.mask_in = reinterpret_cast<const int8_t*>(d_mask_in); P.mask_out = reinterpret_cast<int8_t*>(d_mask_out);
    P.N = N; P.C = C; P.H = H; P.W = W; P.up = up; P.down = down; P.px0 = px0; P.py0 = py0;
    P.fu_taps = h_fu && fu_taps > 0 ? fu_taps : 1;
    P.fd_taps = h_fd && fd_taps > 0 ? fd_taps : 1;
    // correlation-form taps: upfirdn2d convolves (flips the filter) unless flip_filter (upfirdn2d.py:196-199); gain up^2 over two axes
    for (int k = 0; k < P.fu_taps; ++k) P.fu[k] = (h_fu && fu_taps > 0 ? h_fu[flip_filter ? k : P.fu_taps - 1 - k] : 1.f) * up;
    for (int k = 0; k < P.fd_taps; ++k) P.fd[k] = h_fd && fd_taps > 0 ? h_fd[flip_filter ? k : P.fd_taps - 1 - k] : 1.f;
    P.gain = gain; P.slope = slope; P.clamp = clamp;
    P.mid_w = W * up + px0 + px1 - (P.fu_taps - 1);
    P.mid_h = H * up + py0 + py1 - (P.fu_taps - 1);
    P.out_w = (P.mid_w - (P.fd_taps - 1) + down - 1) / down;
    P.out_h = (P.mid_h - (P.fd_taps - 1) + down - 1) / down;
    if (P.mid_w < 1 || P.mid_h < 1 || P.out_w < 1 || P.out_h < 1) return la::fail(-2, "filtered_lrelu: empty output");
    if (d_mask_in || d_mask_out) {
        if (mask_h < 1 || mask_w < 1) { mask_oy = mask_ox = 0; mask_h = P.mid_h; mask_w = P.mid_w; }
        P.mask_oy = mask_oy; P.mask_ox = mask_ox; P.mask_h = mask_h; P.mask_w = mask_w;
    }
    P.mid_t = (kTile - 1) * down + P.fd_taps;
    P.in_t = (P.mid_t + P.fu_taps - 1 + up - 1) / up + 1;
    const size_t smem = sizeof(float) * (static_cast<size_t>(P.in_t) * P.in_t + static_cast<size_t>(P.in_t) * P.mid_t +
                                         static_cast<size_t>(P.mid_t) * P.mid_t + static_cast<size_t>(P.mid_t) * kTile + 2 * kMaxTaps);
    if (P.mid_t > 256 || P.in_t > 256) return la::fail(-2, "filtered_lrelu: filter footprint too large for one tile");
    if (smem > 200 * 1024) return la::fail(-2, "filtered_lrelu: filter footprint too large for one tile");
    dim3 grid((P.out_w + kTile - 1) / kTile, (P.out_h + kTile - 1) / kTile, N * C);
    cudaStream_t cs = static_cast<cudaStream_t>(stream);
    cudaError_t e = cudaSuccess;
#define LA_FL(U, D, A, B)                                                                                                          \
    do {                                                                                                                           \
        e = cudaFuncSetAttribute(filtered_lrelu_kernel<U, D, A, B>, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)); \
        if (e == cudaSuccess) filtered_lrelu_kernel<U, D, A, B><<<grid, 256, smem, cs>>>(P);                                       \
    } while (0)
    const int key = ((up * 8 + down) * 64 + P.fu_taps) * 64 + P.fd_taps;          // the StyleGAN3 layer shapes and their adjoints
    switch (key) {
        case ((2 * 8 + 2) * 64 + 12) * 64 + 12: LA_FL(2, 2, 12, 12); break;
        case ((4 * 8 + 2) * 64 + 24) * 64 + 12: LA_FL(4, 2, 24, 12); break;
        case ((2 * 8 + 4) * 64 + 12) * 64 + 24: LA_FL(2, 4, 12, 24); break;
        case ((2 * 8 + 1) * 64 + 12) * 64 + 1: LA_FL(2, 1, 12, 1); break;
        case ((1 * 8 + 2) * 64 + 1) * 64 + 12: LA_FL(1, 2, 1, 12); break;
        default: LA_FL(0, 0, 0, 0); break;
    }
#undef LA_FL
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) return la::fail(static_cast<int>(e), "filtered_lrelu: %s", cudaGetErrorString(e));
    return 0;
}
