// Shared device helpers for the sm_100a Mamba-block kernels (selective scan, causal conv1d, scan orders).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/mmunet_b200.h"

namespace mmu {

constexpr float kLog2e = 1.4426950408889634f;

// ---- host-side error plumbing (capi.cu) -------------------------------------------------------
int set_error(int code, const char *fmt, ...);
void count_launch(int n = 1);
int check_launch(const char *what);
int knob(const char *name, int dflt);   // MMU_* tuning knob (environment, read once: capi.cu)

// ---- deterministic mode (det_reduce.cu) -----------------------------------------------------------------------------------
// Ordered sum over `items` partial slots, added into a strided destination: column (a, r, c), extents (n0, n1, n2);
// src[i * item_stride + a * ss0 + r * ss1 + c], dst[a * ds0 + r * ds1 + c * ds2] += sum over i in a fixed order.
struct DetSum {
    const float *src;
    int64_t items, item_stride;
    int n0, n1, n2;
    int64_t ss0, ss1;
    float *dst;
    int64_t ds0, ds1, ds2;
};
int det_reduce(const DetSum &r, cudaStream_t st);
// Bump allocator over a caller's workspace: 256-byte aligned float slices.  size() of a dry run (base == nullptr) is the query.
struct DetWs {
    char *base;
    size_t used = 0;
    float *take(size_t floats) {
        float *p = base ? reinterpret_cast<float *>(base + used) : nullptr;
        used += (floats * sizeof(float) + 255) & ~(size_t)255;
        return p;
    }
};
// argument checks shared by every _det entry point: MMU_ERR_WORKSPACE when the caller's workspace is missing or too small
inline int det_ws_check(const void *ws, size_t ws_bytes, size_t need, const char *what) {
    if (need > 0 && (ws == nullptr || ws_bytes < need))
        return set_error(MMU_ERR_WORKSPACE, "%s: deterministic workspace %zu < %zu bytes", what, ws ? ws_bytes : (size_t)0, need);
    if (ws != nullptr && reinterpret_cast<uintptr_t>(ws) % 256 != 0) return set_error(MMU_ERR_INVALID, "%s: workspace must be 256-byte aligned", what);
    return MMU_OK;
}

// ---- element conversion -----------------------------------------------------------------------
template <typename T> struct Elem;
template <> struct Elem<float> {
    static constexpr int kVec = 4;   // elements per 16 bytes
    static __device__ __forceinline__ float to_f(float v) { return v; }
    static __device__ __forceinline__ float from_f(float v) { return v; }
};
template <> struct Elem<__nv_bfloat16> {
    static constexpr int kVec = 8;
    static __device__ __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
    static __device__ __forceinline__ __nv_bfloat16 from_f(float v) { return __float2bfloat16_rn(v); }
};
template <> struct Elem<__half> {
    static constexpr int kVec = 8;
    static __device__ __forceinline__ float to_f(__half v) { return __half2float(v); }
    static __device__ __forceinline__ __half from_f(float v) { return __float2half_rn(v); }
};

// 16-byte vector of elements
template <typename T> struct alignas(16) Vec16 { T v[Elem<T>::kVec]; };

// ---- packed fp32 (Blackwell FFMA2 / FMUL2 / FADD2: two fp32 lanes per issue slot) ----------------
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 splat(float a) { return make_float2(a, a); }

// MUFU.EX2
__device__ __forceinline__ float ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float2 ex2(float2 x) { return make_float2(ex2(x.x), ex2(x.y)); }

// softplus with the reference's threshold (selective_scan_fwd_kernel.cuh:153-156; F.softplus default)
// log1p(e^x) without the libm log1pf call: for small e = e^x the alternating series (error < e^5/5), otherwise
// log(1+e) through MUFU.LG2.  Relative error stays < 1e-5 over the whole range (delta feeds exp(delta*A), so it is the
// relative error that matters).
__device__ __forceinline__ float softplus_f(float x) {
    const float e = __expf(fminf(x, 20.f));
    const float series = e * fmaf(e, fmaf(e, fmaf(e, -0.25f, 0.33333334f), -0.5f), 1.f);
    const float lg = __logf(1.f + e);
    const float r = e < 1.5e-2f ? series : lg;
    return x <= 20.f ? r : x;
}
__device__ __forceinline__ float sigmoid_f(float x) { return __fdividef(1.f, 1.f + __expf(-x)); }

__device__ __forceinline__ float2 shfl_up2(float2 v, int delta, int width) {
    return make_float2(__shfl_up_sync(0xffffffffu, v.x, delta, width), __shfl_up_sync(0xffffffffu, v.y, delta, width));
}
__device__ __forceinline__ float2 shfl_down2(float2 v, int delta, int width) {
    return make_float2(__shfl_down_sync(0xffffffffu, v.x, delta, width),
                       __shfl_down_sync(0xffffffffu, v.y, delta, width));
}

// ---- scan-order index map -------------------------------------------------------------------------------------------------
// idx(l) = memory index of logical (scan-order) token l; the closed forms of the reference's permutations
// (NSLICES: requirements/mamba_simple.py:245-247, 263;  TWOROW: src/UM_Net/MMUNet.py:68-121).  Shared by the standalone gather /
// scatter kernels, the conv kernels (x / dx addressed through it) and the scan kernels (gate z, out, dout, dz addressed through it).
struct OrdMap {
    int kind;                 // MMU_ORDER_ROWMAJOR / FLIP / NSLICES / TWOROW
    int W, ns, L, Ls, even_tokens;   // Ls = L / ns, even_tokens = 2*(H/2)*W
    int ns_shift;                    // log2(ns) when ns is a power of two, else -1 (a runtime integer division costs ~25 instructions)
    __device__ __forceinline__ int operator()(int l) const {
        switch (kind) {
            case MMU_ORDER_FLIP: return L - 1 - l;
            case MMU_ORDER_NSLICES: {
                const int jj = ns_shift >= 0 ? l >> ns_shift : l / ns, s = l - jj * ns;
                return s * Ls + jj;
            }
            case MMU_ORDER_TWOROW: {
                if (l >= even_tokens) return l;   // odd tail row, appended row-major
                const int pair = l / (2 * W), rem = l - pair * 2 * W;
                return (2 * pair + (rem & 1)) * W + (rem >> 1);
            }
            default: return l;
        }
    }
    // 8 consecutive logical tokens t0 .. t0+7 with t0 % 8 == 0, for the fusable cases (NSLICES: ns % 8 == 0; TWOROW: W % 4 == 0, so
    // that a group never straddles a slice round / a row pair): one division per group
    __device__ __forceinline__ void idx8(int t0, int (&m)[8]) const {
        if (kind == MMU_ORDER_NSLICES) {
            const int jj = ns_shift >= 0 ? t0 >> ns_shift : t0 / ns, s0 = t0 - jj * ns;
#pragma unroll
            for (int i = 0; i < 8; ++i) m[i] = (s0 + i) * Ls + jj;
        } else if (kind == MMU_ORDER_TWOROW && t0 < even_tokens) {
            const int pair = t0 / (2 * W), rem = t0 - pair * 2 * W, base = 2 * pair * W + (rem >> 1);
#pragma unroll
            for (int i = 0; i < 8; ++i) m[i] = base + (i & 1) * W + (i >> 1);
        } else {
#pragma unroll
            for (int i = 0; i < 8; ++i) m[i] = t0 + i;
        }
    }
};
// host: fill the map; returns false when the arguments are inconsistent
inline bool make_ordmap(OrdMap &m, int order, int H, int W, int ns, int L) {
    m = OrdMap{order, W > 0 ? W : 1, ns > 0 ? ns : 1, L, 0, 0, -1};
    if (order == MMU_ORDER_NSLICES) {
        if (ns <= 0 || L % ns != 0) return false;
        m.Ls = L / ns;
        if ((ns & (ns - 1)) == 0)
            for (m.ns_shift = 0; (1 << m.ns_shift) < ns; ++m.ns_shift) {}
    } else if (order == MMU_ORDER_TWOROW) {
        if (H <= 0 || W <= 0 || (int64_t)H * W != L) return false;
        m.even_tokens = 2 * (H / 2) * W;
    }
    return true;
}
// the scan / conv kernels fuse an order only where 8-token groups map to simple strides (otherwise the caller permutes explicitly)
inline bool ordmap_fusable(int order, int H, int W, int ns, int L) {
    if (order == MMU_ORDER_ROWMAJOR) return true;
    if (L % 8 != 0) return false;
    if (order == MMU_ORDER_NSLICES) return ns > 0 && ns % 8 == 0 && L % ns == 0 && (L / ns) % 2 == 0;
    if (order == MMU_ORDER_TWOROW) return H > 0 && W > 0 && (int64_t)H * W == L && W % 4 == 0;
    return false;
}

// ---- shared-memory tile addressing ---------------------------------------------------------------
// A tile row holds TL fp32 tokens.  Thread j of a row-group reads T consecutive tokens with LDS.128; the
// 16-byte chunk index is XOR-swizzled so that the 8 lanes of a quarter-warp hit 8 distinct bank groups.
template <int T> __device__ __forceinline__ int swz_chunk(int c) {
    static_assert(T == 4 || T == 8 || T == 16, "T");
    return c ^ ((c >> 3) & (T / 4 - 1));
}
template <int T> __device__ __forceinline__ int swz_tok(int tok) { return (swz_chunk<T>(tok >> 2) << 2) | (tok & 3); }

}  // namespace mmu
