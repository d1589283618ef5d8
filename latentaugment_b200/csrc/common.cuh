// Plumbing shared by every host-side client of the tap-GEMM (engine, discriminator, perceptual term, VGG16 detector,
// distance entries): the one error channel behind la_last_error(), the workspace planner, and the helpers that store an
// fp32 value as split-bf16 (hi, lo) planes.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace la {

// ------------------------------------------------------------------------- errors
// Sets the thread-local text that la_last_error() returns; returns code (-1 for 0).  Defined in engine.cu.
int fail(int code, const char* fmt, ...) __attribute__((format(printf, 2, 3)));

// Return on a failed cudaError_t expression (CU) or a non-zero int-returning call (LA; > 0 is a cudaError_t).  The message
// starts with the calling file's `kModule`, the one place a client names itself.
#define CU(x)                                                                                                                \
    do {                                                                                                                     \
        cudaError_t e_ = (x);                                                                                                \
        if (e_ != cudaSuccess)                                                                                               \
            return ::la::fail(static_cast<int>(e_), "%s: %s: %s (%s:%d)", kModule, #x, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)
#define LA(x)                                                                                                                \
    do {                                                                                                                     \
        int r_ = (x);                                                                                                        \
        if (r_)                                                                                                              \
            return ::la::fail(r_, "%s: %s: %s (%s:%d)", kModule, #x, r_ > 0 ? cudaGetErrorString(static_cast<cudaError_t>(r_)) : "error", \
                              __FILE__, __LINE__);                                                                           \
    } while (0)

// ------------------------------------------------------------------------- workspace
struct Pl {                 // a bf16 tensor as (hi [, lo]) planes; lo only in split (fp32_parity) precision
    __nv_bfloat16* hi = nullptr;
    __nv_bfloat16* lo = nullptr;
};

// Places buffers in a caller-owned workspace, each 1024-byte aligned.  With a null base it only counts: `off` is then the
// size the same plan needs.
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
    Pl take_pl(size_t count, int split) {          // count elements as (hi [, lo]) planes
        Pl t;
        t.hi = take<__nv_bfloat16>(count);
        t.lo = split ? take<__nv_bfloat16>(count) : nullptr;
        return t;
    }
};

// A plan that needs `need` bytes, placed in the caller's workspace ws of `bytes` bytes: reject a short or misaligned one.
inline int check_workspace(const char* owner, size_t need, size_t bytes, const void* ws) {
    if (need > bytes) return fail(-2, "%s workspace too small: %zu < %zu", owner, bytes, need);
    if (reinterpret_cast<uintptr_t>(ws) & 1023) return fail(-2, "%s workspace must be 1024-byte aligned", owner);
    return 0;
}

inline int cdiv(long long a, long long b) { return static_cast<int>((a + b - 1) / b); }
// a bf16 plane as bf16x2 pairs
inline unsigned* U32(__nv_bfloat16* p) { return reinterpret_cast<unsigned*>(p); }
inline const unsigned* CU32(const __nv_bfloat16* p) { return reinterpret_cast<const unsigned*>(p); }

// ------------------------------------------------------------------------- split-bf16 planes
__device__ __forceinline__ unsigned pack2(float a, float b) {      // a in the low half, b in the high half
    __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<unsigned*>(&v);
}
__device__ __forceinline__ float lo_f(unsigned u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float hi_f(unsigned u) { return __uint_as_float(u & 0xffff0000u); }
__device__ __forceinline__ float rnd(float v) { return __bfloat162float(__float2bfloat16_rn(v)); }
// element i of a (hi [, lo]) pair: store / value
__device__ __forceinline__ void st_sp(__nv_bfloat16* hi, __nv_bfloat16* lo, long long i, float v) {
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    hi[i] = h;
    if (lo) lo[i] = __float2bfloat16_rn(v - __bfloat162float(h));
}
__device__ __forceinline__ float ld_sp(const __nv_bfloat16* hi, const __nv_bfloat16* lo, long long i) {
    float v = __bfloat162float(hi[i]);
    if (lo) v += __bfloat162float(lo[i]);
    return v;
}
// the same for element i of bf16x2 pairs
__device__ __forceinline__ void st_sp2(unsigned* hi, unsigned* lo, long long i, float a, float b) {
    hi[i] = pack2(a, b);
    if (lo) lo[i] = pack2(a - rnd(a), b - rnd(b));
}
__device__ __forceinline__ float2 ld_sp2(const unsigned* hi, const unsigned* lo, long long i) {
    const unsigned u = __ldg(hi + i);
    float2 v = make_float2(lo_f(u), hi_f(u));
    if (lo) { const unsigned l = __ldg(lo + i); v.x += lo_f(l); v.y += hi_f(l); }
    return v;
}

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

}  // namespace la
