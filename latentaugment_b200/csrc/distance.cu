// Distance-to-bank: exact pairwise squared L2 (reference l2_loss_vectorized, compute_mean=False,
// augments/utils/util_latent_aug.py:315-361) and the nearest-code / top-k extension
// (SURVEY.md F3): tensor-core candidate selection (tap-GEMM with the fused top-k epilogue, one
// bf16 pass) followed by an exact re-rank in the reference's association order whose margins
// make the result equal to the exhaustive search for any data (rerank_kernel).  The precision / recall entries
// (DESIGN.md §12) reuse the query split, the tap-GEMM and the re-rank over split (hi + lo) candidate passes, and add the
// membership pass (kEpiMember epilogue + member_recheck_kernel).
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "../../include/latentaugment_b200.h"
#include "common.cuh"
#include "tapgemm.cuh"

using namespace la;

namespace {

constexpr char kModule[] = "distance";
typedef __nv_bfloat16 bf16;
constexpr int kCand = 2;          // candidates kept per (query, 32-code chunk)
constexpr int kChunk = 32;
constexpr int kMemberCap = 256;   // ambiguous (probe, point) pairs listed per probe before the probe is rescanned exhaustively

// Error bound of the split candidate score s^ = |y|^2 - 2 (<xh,yh> + <xl,yh> + <xh,yl>) (three bf16 passes over the hi / lo
// planes of split_rows_kernel), as a multiple of |x| max_j |y_j|.  x = xh + xl + r with |xl| <= 2^-9 |x| and |r| <= 2^-18 |x|
// (r = 0 for fp16-valued rows), so the dropped terms xl.yl + r.y + x.r' - r.r' are <= 3.01 * 2^-18 sum|x_k y_k| < 2^-16 sum|x_k y_k|;
// every product of two bf16 values is exact in fp32 and the 3K fp32 additions add <= 3K * 2^-24 * 1.01 sum|x_k y_k|
// (worst case, partial sums bounded by the sum of the magnitudes).  Cauchy-Schwarz: sum|x_k y_k| <= |x| |y|; the factor 2 of
// the score doubles both.
__host__ __device__ __forceinline__ float split_eps_coef(int K) { return 3.0518e-5f + static_cast<float>(K) * 3.612e-7f; }

// rows -> bf16 (hi [, lo] planes) + |row|^2 (fp64 accumulate, rounded once to fp32).  Warp per row.
__global__ void split_rows_kernel(const float* __restrict__ src, int rows, int rows_padded, int K, bf16* hi, bf16* lo, float* sqnorm) {
    const int r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= rows_padded) return;
    double acc = 0.0;
    for (int k = lane; k < K; k += 32) {
        const float v = r < rows ? src[static_cast<long long>(r) * K + k] : 0.f;
        const bf16 h = __float2bfloat16_rn(v);
        hi[static_cast<long long>(r) * K + k] = h;
        if (lo) lo[static_cast<long long>(r) * K + k] = __float2bfloat16_rn(v - __bfloat162float(h));
        acc += static_cast<double>(v) * v;
    }
    acc = warp_sum_d(acc);
    if (lane == 0 && r < rows && sqnorm) sqnorm[r] = static_cast<float>(acc);
}

// D[j, i] = (|Y_j|^2 + |X_i|^2) - 2 <Y_j, X_i>; warp per (j, i); dot in fp64, one rounding.
__global__ void pairwise_kernel(const float* __restrict__ X, int n, const float* __restrict__ Y, int m, int K, float* D) {
    const long long pair = blockIdx.x * static_cast<long long>(blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (pair >= static_cast<long long>(m) * n) return;
    const int j = static_cast<int>(pair / n), i = static_cast<int>(pair % n);
    const float* x = X + static_cast<long long>(i) * K;
    const float* y = Y + static_cast<long long>(j) * K;
    double xx = 0.0, yy = 0.0, yx = 0.0;
    for (int k = lane; k < K; k += 32) {
        const double a = x[k], b = y[k];
        xx += a * a; yy += b * b; yx += a * b;
    }
    xx = warp_sum_d(xx); yy = warp_sum_d(yy); yx = warp_sum_d(yx);
    if (lane == 0) D[pair] = (static_cast<float>(yy) + static_cast<float>(xx)) - 2.f * static_cast<float>(yx);
}

// Exact re-rank, one block of kRerankWarps warps per query.  The tap-GEMM (ONE bf16 pass) left, per (query, 32-code chunk = "group"), the 2
// smallest approximate scores s^ = |y|^2 - 2 <bf16(x), bf16(y)> in ascending order.  With eps ~ 2^-7 * 1.02 |x| max_j|y_j|
// (>= the error of s^: two bf16 roundings of relative size 2^-9 each on every product, doubled by the factor -2, plus
// the fp32 accumulation error, Cauchy-Schwarz on sum |x_k y_k|) the exact k best are found as follows:
//   1. thr = the 8th smallest of the lanes' two best s^ (8 distinct candidates have s^ <= thr, so the k-th smallest EXACT
//      score T satisfies T <= thr + eps) and every exact top-k member has s^ <= T + eps, hence s^ <= cut = thr + 2 eps.
//   2. A member can be missing from the candidate lists only if 2 others of its group have smaller s^, i.e. only if
//      that group's 2nd kept score is <= cut: such groups ("overflowed") are rescanned exhaustively (their listed
//      candidates are dropped, the scan covers them); with more than kMaxOvf of them the whole shard is scanned.
//   3. every surviving candidate (s^ <= cut) and every code of an overflowed group is recomputed exactly -- fp64 dot,
//      one rounding, the reference's association (YY + XX) - 2 YX -- and the k smallest (distance, index) pairs are
//      kept, ties to the lowest index.
// So the result equals the exact search for ANY data, not only in probability; the margins only set the cost.
constexpr int kMaxOvf = 128, kMaxList = 512, kRerankWarps = 4;
// One BLOCK of kRerankWarps warps per query (the kernel is a chain of memory latencies: with a warp per query only 7 warps
// per SM were in flight at 1024 queries and it took 550 of the 770 us of a search): the warps split the groups of both
// passes and the exact evaluations, and every loop keeps several independent loads in flight.
template <int KQ>      // K / 128 (code rows as KQ independent 16-byte loads per lane), 0 = generic K
__global__ void __launch_bounds__(32 * kRerankWarps) rerank_kernel(const float* __restrict__ X, const float* __restrict__ xx, const float* __restrict__ Y,
                                                     const float* __restrict__ yy, int n, int m, int K, const float* __restrict__ cand_score,
                                                     const int* __restrict__ cand_idx, int ncand, int k, long long index_offset,
                                                     float* out_dist, long long* out_idx, int split, int* fallback) {
    __shared__ int s_list[kMaxList];
    __shared__ int s_ovf[kMaxOvf];
    __shared__ float s_thr[kRerankWarps * 8];
    static_assert(kRerankWarps * 8 <= 32, "one value per lane in the second level");
    __shared__ int s_cnt[2];                       // survivors, overflowed groups
    __shared__ float s_bd[kRerankWarps][8];
    __shared__ int s_bi[kRerankWarps][8];
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31, tid = threadIdx.x;
    const int i = blockIdx.x;
    if (i >= n) return;
    const float INF = __int_as_float(0x7f800000);
    const float2* cs2 = reinterpret_cast<const float2*>(cand_score + static_cast<long long>(i) * ncand);
    const int2* ci2 = reinterpret_cast<const int2*>(cand_idx + static_cast<long long>(i) * ncand);
    const int ngroups = ncand / kCand;
    constexpr int NT = 32 * kRerankWarps;
    if (tid < 2) s_cnt[tid] = 0;
    // pass 1 (branch-free): the two smallest approximate scores of this thread's strided share of the groups.  The 8th
    // smallest of the threads' pairs bounds the 8th smallest over ALL candidates from above (8 distinct candidates lie at
    // or below it), which is all that step 1 needs.
    float m1 = INF, m2 = INF;
#pragma unroll 4
    for (int g = tid; g < ngroups; g += NT) {
        const float2 sc = __ldg(cs2 + g);
        const int2 id = __ldg(ci2 + g);
        const float a = id.x >= 0 ? sc.x : INF, bq = id.y >= 0 ? sc.y : INF;        // a <= bq (ascending per group)
        const bool a1 = a < m1, a2 = a < m2;
        m2 = a1 ? m1 : (a2 ? a : m2);
        m1 = a1 ? a : m1;
        m2 = bq < m2 ? bq : m2;                                                     // bq >= a: it can only displace m2
    }
    // the warp's 8 smallest values (pop the minimum of the lane heads 8 times) -> shared; the 8th smallest of the
    // kRerankWarps * 8 values is the 8th smallest over all threads' pairs
    int head = 0;
    for (int r = 0; r < 8; ++r) {
        const float h = head == 0 ? m1 : (head == 1 ? m2 : INF);
        float mn = h;
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        if (lane == 0) s_thr[wib * 8 + r] = mn;
        const unsigned who = __ballot_sync(0xffffffffu, h == mn && mn != INF);
        if (who && lane == __ffs(who) - 1) ++head;
    }
    __syncthreads();
    float thr = INF;
    {
        float v = lane < kRerankWarps * 8 ? s_thr[lane] : INF;
        for (int r = 0; r < 8; ++r) {
            float mn = v;
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
            thr = mn;
            if (mn == INF) break;
            const unsigned who = __ballot_sync(0xffffffffu, v == mn);
            if (lane == __ffs(who) - 1) v = INF;
        }
    }
    const float xi = xx[i];
    // |s^ - s| <= 2 |<x,y> - <bf16 x, bf16 y>| <= 2 (2 * 2^-9 + 2^-18) sum|x_k y_k| + 2 K 2^-24 sum|x_k y_k| (fp32 accumulation,
    // worst case) <= 2^-7 (1.001 + K 2^-16) |x| |y| -- 1.02 covers K <= 1024, the K term takes over beyond; the last term
    // covers the roundings of the fp32 distance the final order is defined on (|y|^2, |x|^2, their sum, the result: 4 ulps)
    const float slack = fmaxf(1.02f, 1.004f + static_cast<float>(K) * 1.5259e-5f);
    // split candidates (three passes, split_eps_coef) leave only the lo.lo term and the longer fp32 accumulation
    const float eps = split ? split_eps_coef(K) * sqrtf(xi) * sqrtf(yy[m]) + 6e-7f * (xi + yy[m])
                            : 0.0078125f * slack * sqrtf(xi) * sqrtf(yy[m]) + 4.8e-7f * (xi + yy[m]);   // yy[m] = max_j |y_j|^2 (la_bank_prepare)
    const float cut = thr == INF ? INF : thr + 2.f * eps;
    // pass 2: overflowed groups (the last kept score is still within the cut: the group may hide more) go to the rescan
    // list, the candidates within the cut of the other groups to the survivor list (order is irrelevant: the final
    // selection orders by (distance, index))
#pragma unroll 4
    for (int g = tid; g < ngroups; g += NT) {
        const float2 sc = __ldg(cs2 + g);
        const int2 id = __ldg(ci2 + g);
        const bool ov = id.y >= 0 && sc.y <= cut;
        const bool k0 = !ov && id.x >= 0 && sc.x <= cut;           // (sc.y > cut here, so only the first entry can survive)
        if (ov) { const int slot = atomicAdd(&s_cnt[1], 1); if (slot < kMaxOvf) s_ovf[slot] = g; }
        if (k0) { const int slot = atomicAdd(&s_cnt[0], 1); if (slot < kMaxList) s_list[slot] = id.x; }
    }
    __syncthreads();
    const int cnt = s_cnt[0], novf = s_cnt[1];
    const bool scan_all = thr == INF || novf > kMaxOvf || cnt > kMaxList;
    if (scan_all && fallback && tid == 0) atomicAdd(fallback, 1);
    float bd[8];
    int bi[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) { bd[t] = INF; bi[t] = 0x7fffffff; }
    auto insert = [&](float d, int id) {
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            if (d < bd[t] || (d == bd[t] && id < bi[t])) {
                const float td = bd[t]; const int ti = bi[t];
                bd[t] = d; bi[t] = id; d = td; id = ti;
            }
        }
    };
    const float* x = X + static_cast<long long>(i) * K;
    // work list of this warp: entry e of [survivors | codes of the overflowed groups] (or every code), e = wib mod warps
    const int total = scan_all ? m : cnt + novf * kChunk;
    auto code_of = [&](int e) {
        if (scan_all) return e;
        if (e < cnt) return s_list[e];
        const int o = (e - cnt) / kChunk, j = s_ovf[o] * kChunk + (e - cnt) % kChunk;
        return j < m ? j : -1;
    };
    if constexpr (KQ > 0) {
        // query row in registers; a code row = KQ independent 16-byte loads per lane (occupancy hides their latency:
        // the first version also prefetched the next row and, at 196 registers, ran two blocks per SM)
        float4 xr[KQ];
#pragma unroll
        for (int q = 0; q < KQ; ++q) xr[q] = __ldg(reinterpret_cast<const float4*>(x) + q * 32 + lane);
        for (int e = wib; e < total; e += kRerankWarps) {
            const int j = code_of(e);
            if (j < 0) continue;
            const float4* y = reinterpret_cast<const float4*>(Y + static_cast<long long>(j) * K);
            float4 yr[KQ];
#pragma unroll
            for (int q = 0; q < KQ; ++q) yr[q] = __ldg(y + q * 32 + lane);
            double dot = 0.0;
#pragma unroll
            for (int q = 0; q < KQ; ++q) {
                dot += static_cast<double>(xr[q].x) * yr[q].x; dot += static_cast<double>(xr[q].y) * yr[q].y;
                dot += static_cast<double>(xr[q].z) * yr[q].z; dot += static_cast<double>(xr[q].w) * yr[q].w;
            }
            dot = warp_sum_d(dot);
            insert((yy[j] + xi) - 2.f * static_cast<float>(dot), j);
        }
    } else {
        for (int e = wib; e < total; e += kRerankWarps) {
            const int j = code_of(e);
            if (j < 0) continue;
            const float* y = Y + static_cast<long long>(j) * K;
            double dot = 0.0;
            for (int kk = lane; kk < K; kk += 32) dot += static_cast<double>(x[kk]) * y[kk];
            dot = warp_sum_d(dot);
            insert((yy[j] + xi) - 2.f * static_cast<float>(dot), j);
        }
    }
    // merge the warps' lists (every lane of a warp holds the same list)
#pragma unroll
    for (int t = 0; t < 8; ++t)
        if (lane == t) { s_bd[wib][t] = bd[t]; s_bi[wib][t] = bi[t]; }
    __syncthreads();
    if (wib == 0) {
        for (int w = 1; w < kRerankWarps; ++w)
            for (int t = 0; t < 8; ++t)
                if (s_bi[w][t] != 0x7fffffff) insert(s_bd[w][t], s_bi[w][t]);
        if (lane == 0)
            for (int t = 0; t < k; ++t) {
                out_dist[static_cast<long long>(i) * k + t] = bd[t];
                out_idx[static_cast<long long>(i) * k + t] = bi[t] == 0x7fffffff ? -1 : bi[t] + index_offset;
            }
    }
}

// max_j |y_j|^2 -> sqnorm[m]   (one block)
__global__ void max_sqnorm_kernel(float* sqnorm, int m) {
    float v = 0.f;
    for (int j = threadIdx.x; j < m; j += blockDim.x) v = fmaxf(v, sqnorm[j]);
    __shared__ float sm[32];
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (blockDim.x >> 5); ++w) v = fmaxf(v, sm[w]);
        sqnorm[m] = v;
    }
}

// Membership threshold (DESIGN.md §12): h(v) = fp16_rn(sqrt(max(v, 0))) is monotone, so h(d2) <= h(r2) <=> d2 <= T with
// b = the upper edge of the fp16 rounding interval of H = h(r2) (the midpoint to the next fp16 value; 65520 above 65504) and
// T = b^2 when H has an even significand (a tie at b rounds to H), else the fp32 value just below b^2.  b has at most 12
// significant bits, so b^2 is an exact fp32 value; H = +inf admits every distance.  (sqrt in fp64 then one rounding to fp16
// is h exactly: an fp32 v whose root lies off a 12-bit midpoint cannot have its fp64 root land on one.)
__device__ __forceinline__ float member_threshold(float r2) {
    const __half H = __double2half(sqrt(fmax(static_cast<double>(r2), 0.0)));
    const unsigned short hb = __half_as_ushort(H);
    if (hb >= 0x7c00) return __int_as_float(0x7f800000);
    const double hv = __half2float(H);
    const double nv = hb == 0x7bff ? 65536.0 : static_cast<double>(__half2float(__ushort_as_half(static_cast<unsigned short>(hb + 1))));
    const double b = 0.5 * (hv + nv);
    const float T = static_cast<float>(b * b);
    return (hb & 1) ? nextafterf(T, 0.f) : T;
}

// tab[j] = {|y_j|^2, T_j, 2.4e-7 T_j (the share of the membership margin that grows with T_j: the roundings of T_j - |x|^2
// and of the score difference), 0}
__global__ void member_table_kernel(const float* __restrict__ r2, const float* __restrict__ yy, int m, float4* tab) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    const float T = member_threshold(r2[j]);
    tab[j] = make_float4(yy[j], T, T == __int_as_float(0x7f800000) ? 0.f : 2.4e-7f * T, 0.f);
}

// One block per probe after the kEpiMember pass: a probe with a definite hit is a member; otherwise its listed ambiguous
// points (all points when the list overflowed: counted in *fallback) are evaluated with the exact distance
// (|y|^2 + |x|^2) - 2 <x,y> (fp64 dot, one rounding) against T_j, stopping at the first hit.
constexpr int kRecheckWarps = 4;
__global__ void __launch_bounds__(32 * kRecheckWarps) member_recheck_kernel(const float* __restrict__ X, const float* __restrict__ xx,
                                                                            const float* __restrict__ Y, const float4* __restrict__ tab,
                                                                            int n, int m, int K, const int* __restrict__ hit,
                                                                            const int* __restrict__ cnt, const int* __restrict__ list,
                                                                            unsigned char* member, int* fallback) {
    __shared__ int found;
    const int i = blockIdx.x, wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (i >= n) return;
    if (hit[i]) {
        if (threadIdx.x == 0) member[i] = 1;
        return;
    }
    const int c = cnt[i];
    const bool all = c > kMemberCap;
    if (threadIdx.x == 0) {
        found = 0;
        if (all && fallback) atomicAdd(fallback, 1);
    }
    __syncthreads();
    const int total = all ? m : c;
    const float xi = xx[i];
    const float* x = X + static_cast<long long>(i) * K;
    for (int e = wib; e < total; e += kRecheckWarps) {
        const int f = __shfl_sync(0xffffffffu, lane == 0 ? *reinterpret_cast<volatile int*>(&found) : 0, 0);
        if (f) break;
        const int j = all ? e : __ldg(list + static_cast<long long>(i) * kMemberCap + e);
        const float* y = Y + static_cast<long long>(j) * K;
        double dot = 0.0;
        for (int k = lane; k < K; k += 32) dot += static_cast<double>(x[k]) * y[k];
        dot = warp_sum_d(dot);
        const float4 t = __ldg(tab + j);
        if (lane == 0 && (t.x + xi) - 2.f * static_cast<float>(dot) <= t.y) found = 1;
    }
    __syncthreads();
    if (threadIdx.x == 0) member[i] = found ? 1 : 0;
}

// merge [shards, n, k] sorted lists -> k best per query (thread per query)
__global__ void merge_topk_kernel(const float* __restrict__ dist, const long long* __restrict__ idx, int shards, int n, int k,
                                  long long dist_stride, long long idx_stride, float* out_dist, long long* out_idx) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float bd[8];
    long long bi[8];
    for (int t = 0; t < 8; ++t) { bd[t] = __int_as_float(0x7f800000); bi[t] = 0x7fffffffffffffffLL; }
    for (int s = 0; s < shards; ++s)
        for (int t = 0; t < k; ++t) {
            float d = dist[s * dist_stride + static_cast<long long>(i) * k + t];
            long long id = idx[s * idx_stride + static_cast<long long>(i) * k + t];
            if (id < 0) continue;
            for (int u = 0; u < 8; ++u)
                if (d < bd[u] || (d == bd[u] && id < bi[u])) {
                    const float td = bd[u]; const long long ti = bi[u];
                    bd[u] = d; bi[u] = id; d = td; id = ti;
                }
        }
    for (int t = 0; t < k; ++t) {
        out_dist[static_cast<long long>(i) * k + t] = bd[t];
        out_idx[static_cast<long long>(i) * k + t] = bi[t] == 0x7fffffffffffffffLL ? -1 : bi[t];
    }
}

// kSearch: the nearest-code search (one bf16 pass);  kRadii: the same search over the hi + lo planes, plus its [n, k] results;
// kMember: the membership pass (hi + lo planes, the per-point table, per-probe flags and ambiguous lists)
enum DistanceMode { kSearch, kRadii, kMember };
struct NearestLayout {
    int Hq, rows_padded, n_blocks, ncand;
    size_t off_xhi, off_xx, off_cs, off_ci, off_err, off_xlo, off_dist, off_idx, off_tab, off_flags, off_list, total;
};
NearestLayout nearest_layout(int n, int m, int K, DistanceMode mode = kSearch, int k = 0) {
    NearestLayout L;
    L.Hq = (n + 15) / 16;
    L.Hq = (L.Hq + 7) / 8 * 8;                 // whole 8x16 query tiles
    L.rows_padded = L.Hq * 16;
    L.n_blocks = (m + 255) / 256;
    L.ncand = mode == kMember ? 0 : L.n_blocks * (256 / kChunk) * kCand;
    Bump bp;                                     // null base: offsets only
    auto take = [&](size_t b) { bp.take<char>(b); return bp.off - b; };
    L.off_xhi = take(static_cast<size_t>(L.rows_padded) * K * 2);
    L.off_xx = take(static_cast<size_t>(L.rows_padded) * 4);
    L.off_cs = take(static_cast<size_t>(n) * L.ncand * 4);
    L.off_ci = take(static_cast<size_t>(n) * L.ncand * 4);
    L.off_err = take(1024);                      // pipeline-timeout flag of the tap-GEMM (caller-owned like everything else)
    L.off_xlo = L.off_dist = L.off_idx = L.off_tab = L.off_flags = L.off_list = 0;
    if (mode != kSearch) L.off_xlo = take(static_cast<size_t>(L.rows_padded) * K * 2);
    if (mode == kRadii) {
        L.off_dist = take(static_cast<size_t>(n) * k * 4);
        L.off_idx = take(static_cast<size_t>(n) * k * 8);
    }
    if (mode == kMember) {
        L.off_tab = take(static_cast<size_t>(m) * 16);
        L.off_flags = take(static_cast<size_t>(n) * 8);          // [n] hit | [n] list count (one memset)
        L.off_list = take(static_cast<size_t>(n) * kMemberCap * 4);
    }
    L.total = bp.off + 1024;
    return L;
}

// The query side of every distance pass and the tap-GEMM over it: X -> bf16 planes + |x|^2, then candidate scores against
// the bank (kSearch: one bf16 pass; otherwise the three split passes (hi,hi) + (lo,hi) + (hi,lo) over the bank's
// [2, m, K] hi | lo planes) into the epilogue P.epilogue selects.  P arrives with the epilogue fields set.
int distance_gemm(TapGemmParams& P, const float* d_X, int n, const void* d_bank, int m, int K, const NearestLayout& L, char* ws,
                  bool split, cudaStream_t s) {
    bf16* xhi = reinterpret_cast<bf16*>(ws + L.off_xhi);
    bf16* xlo = split ? reinterpret_cast<bf16*>(ws + L.off_xlo) : nullptr;
    float* xx = reinterpret_cast<float*>(ws + L.off_xx);
    split_rows_kernel<<<(L.rows_padded + 7) / 8, 256, 0, s>>>(d_X, n, L.rows_padded, K, xhi, xlo, xx);
    CU(cudaGetLastError());

    int dev = 0, sms = 0;
    CU(cudaGetDevice(&dev));
    CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    P.th = 8; P.tw = 16; P.nb = 1;
    P.tiles_n = 1; P.batch = 1; P.nprob = 1;
    P.prob[0].tiles_h = L.Hq / 8; P.prob[0].tiles_w = 1; P.prob[0].vh = L.Hq; P.prob[0].vw = 16;
    P.m_tiles = P.prob[0].tiles_h;
    P.kchunks = K / 64;
    P.n_blocks = L.n_blocks; P.n_total = L.n_blocks * 256;
    P.OH = L.Hq; P.OW = 16; P.osy = P.osx = 1;
    P.n_codes = m; P.n_queries = n;
    if (split) {       // fp16-valued rows are held exactly by hi + lo: only lo.lo is dropped (split_eps_coef)
        P.taps[0] = Tap{0, 0, 0, 0}; P.taps[1] = Tap{0, 0, 0, 1}; P.taps[2] = Tap{0, 0, 1, 0};
        P.prob[0].tap_begin = 0; P.prob[0].ntaps = 3;
    } else {
        P.taps[0] = Tap{0, 0, 0, 0};      // one bf16 pass: bf16(x) . bf16(y); the exact re-rank absorbs its error (rerank_kernel)
        P.prob[0].tap_begin = 0; P.prob[0].ntaps = 1;
    }
    if (tapgemm_finalize(P)) return fail(-5, "tap grouping failed");
    uint64_t adims[4] = {static_cast<uint64_t>(K), 16, static_cast<uint64_t>(L.Hq), 1};
    uint64_t astr[3] = {static_cast<uint64_t>(K) * 2, static_cast<uint64_t>(K) * 32, static_cast<uint64_t>(K) * 32 * L.Hq};
    uint32_t abox[4] = {64, 16, 8, 1};
    if (encode_tmap_bf16(&P.a_map[0], xhi, 4, adims, astr, abox)) return fail(-5, "tensor map encoding failed (queries)");
    if (split && encode_tmap_bf16(&P.a_map[1], xlo, 4, adims, astr, abox)) return fail(-5, "tensor map encoding failed (queries, lo)");
    uint64_t bdims[3] = {static_cast<uint64_t>(K), static_cast<uint64_t>(m), split ? 2u : 1u};
    uint64_t bstr[2] = {static_cast<uint64_t>(K) * 2, static_cast<uint64_t>(K) * 2 * m};
    // CTA pairs (cta_group::2: two query tiles per MMA, each CTA loads half of every bank tile) halve the bank operand
    // traffic from L2 but MEASURED SLOWER here (0.346 vs 0.295 ms per search: the top-k epilogue, not operand delivery,
    // paces this launch): opt-in with LA_NEAREST_PAIR=1
    static const bool pair = getenv("LA_NEAREST_PAIR") && atoi(getenv("LA_NEAREST_PAIR")) == 1;
    P.cta2 = pair && L.Hq / 8 >= 2 ? 1 : 0;
    uint32_t bbox[3] = {64, static_cast<uint32_t>(P.cta2 ? 128 : 256), 1};
    if (encode_tmap_bf16(&P.b_map, d_bank, 3, bdims, bstr, bbox)) return fail(-5, "tensor map encoding failed (bank)");
    P.err_flag = reinterpret_cast<int*>(ws + L.off_err);
    CU(cudaMemsetAsync(P.err_flag, 0, sizeof(int), s));
    if (getenv("LA_DEBUG_SIMT_DIST")) {
        TapSimtOperands ops{};
        ops.a_ptrs[0] = xhi; ops.a_ptrs[1] = xlo;
        ops.a_sw = K; ops.a_sh = 16LL * K; ops.a_sn = 16LL * K * L.Hq;
        ops.a_ws[0] = ops.a_ws[1] = 16; ops.a_hs[0] = ops.a_hs[1] = L.Hq;
        ops.w = d_bank;
        int r = launch_tapgemm_simt(P, ops, s);
        if (r) return fail(r, "launch_tapgemm_simt failed");
    } else {
        int r = launch_tapgemm(P, sms, s);
        if (r) return fail(r, "launch_tapgemm failed");
    }
    return 0;
}

// The exact re-rank of distance_gemm's top-k candidates (kSearch / kRadii).
int launch_rerank(const float* d_X, const float* xx, const float* d_Y, const float* d_bank_sqnorm, int n, int m, int K, const float* cs,
                  const int* ci, int ncand, int k, long long index_offset, float* d_dist, long long* d_idx, int split, int* fallback,
                  cudaStream_t s) {
    const dim3 rb(32 * kRerankWarps);
    switch (K) {
        case 128: rerank_kernel<1><<<n, rb, 0, s>>>(d_X, xx, d_Y, d_bank_sqnorm, n, m, K, cs, ci, ncand, k, index_offset, d_dist, d_idx, split, fallback); break;
        case 256: rerank_kernel<2><<<n, rb, 0, s>>>(d_X, xx, d_Y, d_bank_sqnorm, n, m, K, cs, ci, ncand, k, index_offset, d_dist, d_idx, split, fallback); break;
        case 512: rerank_kernel<4><<<n, rb, 0, s>>>(d_X, xx, d_Y, d_bank_sqnorm, n, m, K, cs, ci, ncand, k, index_offset, d_dist, d_idx, split, fallback); break;
        case 1024: rerank_kernel<8><<<n, rb, 0, s>>>(d_X, xx, d_Y, d_bank_sqnorm, n, m, K, cs, ci, ncand, k, index_offset, d_dist, d_idx, split, fallback); break;
        default: rerank_kernel<0><<<n, rb, 0, s>>>(d_X, xx, d_Y, d_bank_sqnorm, n, m, K, cs, ci, ncand, k, index_offset, d_dist, d_idx, split, fallback); break;
    }
    CU(cudaGetLastError());
    return 0;
}

}  // namespace

extern "C" {

__attribute__((visibility("default")))
int la_pairwise_sqdist(const float* d_X, int n, const float* d_Y, int m, int K, float* d_D, la_stream stream) {
    if (!d_X || !d_Y || !d_D || n < 1 || m < 1 || K < 1) return fail(-2, "bad arguments");
    const long long pairs = static_cast<long long>(m) * n;
    pairwise_kernel<<<static_cast<unsigned>((pairs + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(d_X, n, d_Y, m, K, d_D);
    CU(cudaGetLastError());
    return 0;
}

__attribute__((visibility("default")))
int la_bank_prepare(const float* d_Y, int m, int K, void* d_bank_bf16, float* d_bank_sqnorm, la_stream stream) {
    if (!d_Y || !d_bank_bf16 || !d_bank_sqnorm || m < 1 || K < 64 || K % 64) return fail(-2, "bad arguments (K must be a multiple of 64)");
    bf16* hi = static_cast<bf16*>(d_bank_bf16);
    split_rows_kernel<<<(m + 7) / 8, 256, 0, static_cast<cudaStream_t>(stream)>>>(d_Y, m, m, K, hi, nullptr, d_bank_sqnorm);
    CU(cudaGetLastError());
    max_sqnorm_kernel<<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(d_bank_sqnorm, m);
    CU(cudaGetLastError());
    return 0;
}

__attribute__((visibility("default")))
int la_nearest_codes_workspace_bytes(int n, int m, int K, int k, size_t* bytes) {
    if (!bytes || n < 1 || m < 1 || K % 64 || k < 1 || k > 8) return fail(-2, "bad arguments (k <= 8, K %% 64 == 0)");
    *bytes = nearest_layout(n, m, K).total;
    return 0;
}

__attribute__((visibility("default")))
int la_nearest_codes(const float* d_X, int n, const float* d_Y, const void* d_bank_bf16, const float* d_bank_sqnorm, int m, int K, int k,
                     long long index_offset, void* d_workspace, size_t workspace_bytes, float* d_dist, long long* d_idx,
                     la_stream stream) {
    if (!d_X || !d_Y || !d_bank_bf16 || !d_bank_sqnorm || !d_workspace || !d_dist || !d_idx) return fail(-2, "bad arguments");
    if (k < 1 || k > 8 || K % 64 || K < 64) return fail(-2, "k must be 1..8 and K a multiple of 64");
    const NearestLayout L = nearest_layout(n, m, K);
    if (int r = check_workspace("nearest-codes", L.total, workspace_bytes, d_workspace)) return r;
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    char* ws = static_cast<char*>(d_workspace);
    float* cs = reinterpret_cast<float*>(ws + L.off_cs);
    int* ci = reinterpret_cast<int*>(ws + L.off_ci);
    TapGemmParams P;
    memset(&P, 0, sizeof P);
    P.epilogue = kEpiTopK;
    P.code_sqnorm = d_bank_sqnorm; P.topk = kCand;
    P.cand_score = cs; P.cand_idx = ci;
    if (int r = distance_gemm(P, d_X, n, d_bank_bf16, m, K, L, ws, false, s)) return r;
    return launch_rerank(d_X, reinterpret_cast<float*>(ws + L.off_xx), d_Y, d_bank_sqnorm, n, m, K, cs, ci, L.ncand, k, index_offset,
                         d_dist, d_idx, 0, nullptr, s);
}

__attribute__((visibility("default")))
int la_merge_topk(const float* d_dist, const long long* d_idx, int shards, int n, int k, float* d_out_dist, long long* d_out_idx,
                  la_stream stream) {
    if (!d_dist || !d_idx || !d_out_dist || !d_out_idx || shards < 1 || n < 1 || k < 1 || k > 8) return fail(-2, "bad arguments");
    const long long st = static_cast<long long>(n) * k;
    merge_topk_kernel<<<(n + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(d_dist, d_idx, shards, n, k, st, st, d_out_dist, d_out_idx);
    CU(cudaGetLastError());
    return 0;
}

__attribute__((visibility("default")))
int la_merge_topk_strided(const float* d_dist, const long long* d_idx, int shards, int n, int k, long long dist_shard_stride,
                          long long idx_shard_stride, float* d_out_dist, long long* d_out_idx, la_stream stream) {
    if (!d_dist || !d_idx || !d_out_dist || !d_out_idx || shards < 1 || n < 1 || k < 1 || k > 8) return fail(-2, "bad arguments");
    merge_topk_kernel<<<(n + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(d_dist, d_idx, shards, n, k, dist_shard_stride,
                                                                                      idx_shard_stride, d_out_dist, d_out_idx);
    CU(cudaGetLastError());
    return 0;
}

__attribute__((visibility("default")))
int la_pr_manifold_prepare(const float* d_Y, int m, int K, void* d_planes, float* d_sqnorm, la_stream stream) {
    if (!d_Y || !d_planes || !d_sqnorm || m < 1 || K < 64 || K % 64) return fail(-2, "bad arguments (K must be a multiple of 64)");
    bf16* hi = static_cast<bf16*>(d_planes);
    split_rows_kernel<<<(m + 7) / 8, 256, 0, static_cast<cudaStream_t>(stream)>>>(d_Y, m, m, K, hi, hi + static_cast<long long>(m) * K, d_sqnorm);
    CU(cudaGetLastError());
    max_sqnorm_kernel<<<1, 1024, 0, static_cast<cudaStream_t>(stream)>>>(d_sqnorm, m);
    CU(cudaGetLastError());
    return 0;
}

__attribute__((visibility("default")))
int la_pr_radii_workspace_bytes(int n, int m, int K, int nhood, size_t* bytes) {
    if (!bytes || n < 1 || K < 64 || K % 64) return fail(-2, "bad arguments (K must be a multiple of 64)");
    if (nhood < 1 || nhood > 7) return fail(-2, "nhood must be 1..7");
    if (m < nhood + 1) return fail(-2, "the manifold needs at least nhood + 1 points");
    *bytes = nearest_layout(n, m, K, kRadii, nhood + 1).total;
    return 0;
}

__attribute__((visibility("default")))
int la_pr_radii(const float* d_X, int n, const float* d_Y, const void* d_planes, const float* d_sqnorm, int m, int K, int nhood,
                void* d_workspace, size_t workspace_bytes, float* d_r2, int* d_fallback, la_stream stream) {
    size_t need = 0;
    if (!d_X || !d_Y || !d_planes || !d_sqnorm || !d_workspace || !d_r2) return fail(-2, "bad arguments");
    if (int r = la_pr_radii_workspace_bytes(n, m, K, nhood, &need)) return r;
    if (int r = check_workspace("radii", need, workspace_bytes, d_workspace)) return r;
    const int k = nhood + 1;
    const NearestLayout L = nearest_layout(n, m, K, kRadii, k);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    char* ws = static_cast<char*>(d_workspace);
    float* cs = reinterpret_cast<float*>(ws + L.off_cs);
    int* ci = reinterpret_cast<int*>(ws + L.off_ci);
    float* dist = reinterpret_cast<float*>(ws + L.off_dist);
    TapGemmParams P;
    memset(&P, 0, sizeof P);
    P.epilogue = kEpiTopK;
    P.code_sqnorm = d_sqnorm; P.topk = kCand;
    P.cand_score = cs; P.cand_idx = ci;
    if (int r = distance_gemm(P, d_X, n, d_planes, m, K, L, ws, true, s)) return r;
    if (int r = launch_rerank(d_X, reinterpret_cast<float*>(ws + L.off_xx), d_Y, d_sqnorm, n, m, K, cs, ci, L.ncand, k, 0, dist,
                              reinterpret_cast<long long*>(ws + L.off_idx), 1, d_fallback, s))
        return r;
    // r2[i] = dist[i][nhood]: the (nhood + 1)-th smallest distance, the point itself included
    CU(cudaMemcpy2DAsync(d_r2, sizeof(float), dist + nhood, static_cast<size_t>(k) * sizeof(float), sizeof(float), n,
                          cudaMemcpyDeviceToDevice, s));
    return 0;
}

__attribute__((visibility("default")))
int la_pr_member_workspace_bytes(int n, int m, int K, size_t* bytes) {
    if (!bytes || n < 1 || m < 1 || K < 64 || K % 64) return fail(-2, "bad arguments (K must be a multiple of 64)");
    *bytes = nearest_layout(n, m, K, kMember).total;
    return 0;
}

__attribute__((visibility("default")))
int la_pr_member(const float* d_X, int n, const float* d_Y, const void* d_planes, const float* d_sqnorm, const float* d_r2, int m, int K,
                 void* d_workspace, size_t workspace_bytes, unsigned char* d_member, int* d_fallback, la_stream stream) {
    size_t need = 0;
    if (!d_X || !d_Y || !d_planes || !d_sqnorm || !d_r2 || !d_workspace || !d_member) return fail(-2, "bad arguments");
    if (int r = la_pr_member_workspace_bytes(n, m, K, &need)) return r;
    if (int r = check_workspace("membership", need, workspace_bytes, d_workspace)) return r;
    const NearestLayout L = nearest_layout(n, m, K, kMember);
    cudaStream_t s = static_cast<cudaStream_t>(stream);
    char* ws = static_cast<char*>(d_workspace);
    float4* tab = reinterpret_cast<float4*>(ws + L.off_tab);
    int* hit = reinterpret_cast<int*>(ws + L.off_flags);
    int* cnt = hit + n;
    int* list = reinterpret_cast<int*>(ws + L.off_list);
    member_table_kernel<<<(m + 255) / 256, 256, 0, s>>>(d_r2, d_sqnorm, m, tab);
    CU(cudaGetLastError());
    CU(cudaMemsetAsync(hit, 0, static_cast<size_t>(n) * 8, s));
    TapGemmParams P;
    memset(&P, 0, sizeof P);
    P.epilogue = kEpiMember;
    P.code_sqnorm = d_sqnorm;
    P.member_tab = tab;
    P.query_sqnorm = reinterpret_cast<float*>(ws + L.off_xx);
    P.member_eps = split_eps_coef(K);
    P.member_hit = hit; P.member_cnt = cnt; P.member_list = list; P.member_cap = kMemberCap;
    if (int r = distance_gemm(P, d_X, n, d_planes, m, K, L, ws, true, s)) return r;
    member_recheck_kernel<<<n, 32 * kRecheckWarps, 0, s>>>(d_X, reinterpret_cast<float*>(ws + L.off_xx), d_Y, tab, n, m, K, hit, cnt,
                                                           list, d_member, d_fallback);
    CU(cudaGetLastError());
    return 0;
}

}  // extern "C"
