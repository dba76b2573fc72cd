// GroupNorm over channels-last (NHWC) feature maps with 4 channels per group, sm_100a - the normalisation that closes every
// MMConv (`self.gn = nn.GroupNorm(out_channels // 4, out_channels)`, src/UM_Net/MMUNet.py:46, 271; SURVEY.md section 8 row f2).
//
// ATen's CUDA GroupNorm is NCHW-only (a channels-last input is first copied to NCHW, the output comes back NCHW) and is
// up-cast to fp32 by autocast, so in a channels-last bf16 model each of the 47 MMConvs pays two layout copies and two dtype
// copies per direction around it.  Here x[b][p][c] is read in place: one thread owns the 4 channels of one group at one pixel
// (one 8/16-byte vector), statistics are fp32, the output is written in the requested dtype and stays channels-last.
//   forward : (1) per (b, group) sum / sum of squares -> (2) y = (x - mean) * rstd * gamma + beta
//   backward: (1) per (b, group) S1 = sum gamma*dy, S2 = sum gamma*dy*xhat, per channel dgamma = sum dy*xhat, dbeta = sum dy
//             (2) dx = rstd * (gamma*dy - (S1 + xhat*S2) / n)
// All four kernels are single-pass HBM-bound streams; the partial sums are reduced in the block, then by fp32 atomics into
// caller-zeroed accumulators.  Deterministic mode (the _det entry points): the reduction kernels store the block sums to
// [b][pixel block][G][2 | 10] slots instead, and the ordered reduce (det_reduce.cu) adds them into the same accumulators.
#include "common.cuh"

namespace mmu {

template <typename T> struct V4;
template <> struct V4<float> {
    static __device__ __forceinline__ void ld(const float *p, float (&v)[4]) {
        const float4 q = *reinterpret_cast<const float4 *>(p);
        v[0] = q.x, v[1] = q.y, v[2] = q.z, v[3] = q.w;
    }
    static __device__ __forceinline__ void st(float *p, const float (&v)[4]) { *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]); }
};
template <> struct V4<__nv_bfloat16> {
    static __device__ __forceinline__ void ld(const __nv_bfloat16 *p, float (&v)[4]) {
        const uint2 q = *reinterpret_cast<const uint2 *>(p);
        v[0] = __uint_as_float(q.x << 16), v[1] = __uint_as_float(q.x & 0xffff0000u);
        v[2] = __uint_as_float(q.y << 16), v[3] = __uint_as_float(q.y & 0xffff0000u);
    }
    static __device__ __forceinline__ void st(__nv_bfloat16 *p, const float (&v)[4]) {
        const __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]), b = __floats2bfloat162_rn(v[2], v[3]);
        *reinterpret_cast<uint2 *>(p) = make_uint2(*reinterpret_cast<const unsigned *>(&a), *reinterpret_cast<const unsigned *>(&b));
    }
};

struct GnGeom {
    int B, C, HW, G;       // G = C / 4
    int ppb;               // pixels per block (reduction kernels)
    float eps;
};

constexpr int kGnThreads = 256;

// Shift of the one-pass variance: the group's own first sample (pixel 0, first channel), the same value in every block.
// sums hold sum(x - K) and sum((x - K)^2); var = E[(x-K)^2] - E[x-K]^2 then cancels at the scale of (mean - K) ~ std
// instead of |mean| (ADVICE r1: E[x^2] - mean^2 lost all digits for inputs like x + 100).
template <typename TI> __device__ __forceinline__ float gn_shift(const TI *group_base) {
    float v[4];
    V4<TI>::ld(group_base, v);
    return v[0];
}

// thread layout of the reduction kernels: tid = lane_p * G + g  (G | 256 or G >= 256 handled by the g loop)
template <typename TI, bool DET = false>
__global__ void __launch_bounds__(kGnThreads) gn_stats_kernel(const TI *__restrict__ x, float *__restrict__ sums, GnGeom g) {
    extern __shared__ float sm[];                       // [2][kGnThreads]
    const int b = blockIdx.y, p0 = blockIdx.x * g.ppb, p1 = min(g.HW, p0 + g.ppb);
    const int G = g.G, lanes = max(1, kGnThreads / G), tid = threadIdx.x;
    for (int g0 = 0; g0 < G; g0 += kGnThreads) {
        const int gi = g0 + (G >= kGnThreads ? tid : tid % G), lp = G >= kGnThreads ? 0 : tid / G;
        float s = 0.f, ss = 0.f;
        if (gi < G && lp < lanes) {
            const TI *xp = x + ((int64_t)b * g.HW) * g.C + 4 * gi;
            const float K = gn_shift(xp);               // shifted sums: no cancellation when |mean| >> std
#pragma unroll 4
            for (int p = p0 + lp; p < p1; p += lanes) {
                float v[4];
                V4<TI>::ld(xp + (int64_t)p * g.C, v);
#pragma unroll
                for (int k = 0; k < 4; ++k) v[k] -= K;
                s += (v[0] + v[1]) + (v[2] + v[3]);
                ss += (v[0] * v[0] + v[1] * v[1]) + (v[2] * v[2] + v[3] * v[3]);
            }
        }
        sm[tid] = s, sm[kGnThreads + tid] = ss;
        __syncthreads();
        if (lp == 0 && gi < G) {
            for (int l = 1; l < lanes; ++l) s += sm[l * G + (tid % G)], ss += sm[kGnThreads + l * G + (tid % G)];
            if constexpr (DET) {      // sums = the slots [b][pixel block][G][2]
                float *slot = sums + (((int64_t)b * gridDim.x + blockIdx.x) * G + gi) * 2;
                slot[0] = s, slot[1] = ss;
            } else {
                atomicAdd(sums + ((int64_t)b * G + gi) * 2, s);
                atomicAdd(sums + ((int64_t)b * G + gi) * 2 + 1, ss);
            }
        }
        __syncthreads();
    }
}

__device__ __forceinline__ void gn_moments(const float *__restrict__ sums, int64_t bg, float n, float eps, float K, float &mean, float &rstd) {
    const float s = sums[bg * 2], ss = sums[bg * 2 + 1];
    const float m = s / n;                              // mean of (x - K)
    mean = K + m;
    rstd = rsqrtf(fmaxf(ss / n - m * m, 0.f) + eps);
}

template <typename TI, typename TO>
__global__ void __launch_bounds__(256) gn_apply_kernel(const TI *__restrict__ x, const float *__restrict__ sums, const float *__restrict__ gamma,
                                                       const float *__restrict__ beta, TO *__restrict__ y, float *__restrict__ mean_out,
                                                       float *__restrict__ rstd_out, GnGeom g) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;                  // (pixel, group) of batch element blockIdx.y
    if (i >= (unsigned)g.HW * (unsigned)g.G) return;
    const unsigned pix = i / (unsigned)g.G;                                    // 32-bit only: 64-bit div/mod would dominate
    const int gi = (int)(i - pix * (unsigned)g.G), b = blockIdx.y;
    const int64_t bp = (int64_t)b * g.HW + pix;
    float mean, rstd;
    gn_moments(sums, (int64_t)b * g.G + gi, 4.f * g.HW, g.eps, gn_shift(x + ((int64_t)b * g.HW) * g.C + 4 * gi), mean, rstd);
    if (pix == 0) mean_out[(int64_t)b * g.G + gi] = mean, rstd_out[(int64_t)b * g.G + gi] = rstd;
    float v[4], o[4];
    V4<TI>::ld(x + bp * g.C + 4 * gi, v);
    const float4 ga = *reinterpret_cast<const float4 *>(gamma + 4 * gi), be = *reinterpret_cast<const float4 *>(beta + 4 * gi);
    o[0] = fmaf((v[0] - mean) * rstd, ga.x, be.x), o[1] = fmaf((v[1] - mean) * rstd, ga.y, be.y);
    o[2] = fmaf((v[2] - mean) * rstd, ga.z, be.z), o[3] = fmaf((v[3] - mean) * rstd, ga.w, be.w);
    V4<TO>::st(y + bp * g.C + 4 * gi, o);
}

// backward reduction: sums2[b][g] = (S1, S2); dgb[c] = dgamma, dgb[C + c] = dbeta.  DET: sums2 = the slots [b][pixel block][G][10]
template <typename TI, typename TO, bool DET = false>
__global__ void __launch_bounds__(kGnThreads) gn_bwd_reduce_kernel(const TI *__restrict__ x, const TO *__restrict__ dy, const float *__restrict__ mean,
                                                                   const float *__restrict__ rstd, const float *__restrict__ gamma,
                                                                   float *__restrict__ sums2, float *__restrict__ dgb, GnGeom g) {
    extern __shared__ float sm[];                       // [10][kGnThreads]
    const int b = blockIdx.y, p0 = blockIdx.x * g.ppb, p1 = min(g.HW, p0 + g.ppb);
    const int G = g.G, lanes = max(1, kGnThreads / G), tid = threadIdx.x;
    for (int g0 = 0; g0 < G; g0 += kGnThreads) {
        const int gi = g0 + (G >= kGnThreads ? tid : tid % G), lp = G >= kGnThreads ? 0 : tid / G;
        float acc[10] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // S1, S2, dgamma[4], dbeta[4]
        if (gi < G && lp < lanes) {
            const float mu = mean[(int64_t)b * G + gi], rs = rstd[(int64_t)b * G + gi];
            const float4 ga = *reinterpret_cast<const float4 *>(gamma + 4 * gi);
            const float gam[4] = {ga.x, ga.y, ga.z, ga.w};
            const int64_t base = ((int64_t)b * g.HW) * g.C + 4 * gi;
#pragma unroll 4
            for (int p = p0 + lp; p < p1; p += lanes) {
                float v[4], d[4];
                V4<TI>::ld(x + base + (int64_t)p * g.C, v);
                V4<TO>::ld(dy + base + (int64_t)p * g.C, d);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float xh = (v[k] - mu) * rs, gd = gam[k] * d[k];
                    acc[0] += gd, acc[1] = fmaf(gd, xh, acc[1]);
                    acc[2 + k] = fmaf(d[k], xh, acc[2 + k]), acc[6 + k] += d[k];
                }
            }
        }
#pragma unroll
        for (int k = 0; k < 10; ++k) sm[k * kGnThreads + tid] = acc[k];
        __syncthreads();
        if (lp == 0 && gi < G) {
            for (int l = 1; l < lanes; ++l)
#pragma unroll
                for (int k = 0; k < 10; ++k) acc[k] += sm[k * kGnThreads + l * G + (tid % G)];
            if constexpr (DET) {
                float *slot = sums2 + (((int64_t)b * gridDim.x + blockIdx.x) * G + gi) * 10;
#pragma unroll
                for (int k = 0; k < 10; ++k) slot[k] = acc[k];
            } else {
                atomicAdd(sums2 + ((int64_t)b * G + gi) * 2, acc[0]);
                atomicAdd(sums2 + ((int64_t)b * G + gi) * 2 + 1, acc[1]);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    atomicAdd(dgb + 4 * gi + k, acc[2 + k]);
                    atomicAdd(dgb + g.C + 4 * gi + k, acc[6 + k]);
                }
            }
        }
        __syncthreads();
    }
}

template <typename TI, typename TO>
__global__ void __launch_bounds__(256) gn_bwd_apply_kernel(const TI *__restrict__ x, const TO *__restrict__ dy, const float *__restrict__ mean,
                                                           const float *__restrict__ rstd, const float *__restrict__ gamma,
                                                           const float *__restrict__ sums2, TI *__restrict__ dx, GnGeom g) {
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (unsigned)g.HW * (unsigned)g.G) return;
    const unsigned pix = i / (unsigned)g.G;
    const int gi = (int)(i - pix * (unsigned)g.G), b = blockIdx.y;
    const int64_t bp = (int64_t)b * g.HW + pix, bg = (int64_t)b * g.G + gi;
    const float mu = mean[bg], rs = rstd[bg], inv_n = 1.f / (4.f * g.HW);
    const float s1 = sums2[bg * 2] * inv_n, s2 = sums2[bg * 2 + 1] * inv_n;
    float v[4], d[4], o[4];
    V4<TI>::ld(x + bp * g.C + 4 * gi, v);
    V4<TO>::ld(dy + bp * g.C + 4 * gi, d);
    const float4 ga = *reinterpret_cast<const float4 *>(gamma + 4 * gi);
    const float gam[4] = {ga.x, ga.y, ga.z, ga.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float xh = (v[k] - mu) * rs;
        o[k] = rs * (gam[k] * d[k] - s1 - xh * s2);
    }
    V4<TI>::st(dx + bp * g.C + 4 * gi, o);
}

namespace {
// pixel blocks of the reduction grid: enough blocks to fill the GPU (~8 per SM), at least one pixel per lane
int gn_pblocks(int B, int HW, int G) {
    const int lanes = G >= kGnThreads ? 1 : kGnThreads / G;
    return (int)std::min<int64_t>((HW + lanes - 1) / lanes, std::max<int64_t>(1, (148 * 8 + B - 1) / B));
}
int gn_geom(GnGeom &g, int B, int C, int HW, int G, float eps, dim3 &rgrid, dim3 &agrid) {
    if (B <= 0 || C <= 0 || HW <= 0 || G <= 0) return set_error(MMU_ERR_INVALID, "group_norm: bad shape B%d C%d HW%d G%d", B, C, HW, G);
    if (C != 4 * G) return set_error(MMU_ERR_UNSUPPORTED, "group_norm (channels-last): only 4 channels per group (C=%d, G=%d)", C, G);
    if (G < kGnThreads && kGnThreads % G != 0) return set_error(MMU_ERR_UNSUPPORTED, "group_norm: G=%d must divide %d or be >= it", G, kGnThreads);
    const int64_t items = (int64_t)HW * G;                      // per batch element
    if (items > 0x7fffffffLL || B > 65535) return set_error(MMU_ERR_UNSUPPORTED, "group_norm: problem too large");
    const int pblocks = gn_pblocks(B, HW, G);
    g = {B, C, HW, G, (HW + pblocks - 1) / pblocks, eps};
    rgrid = dim3((unsigned)((HW + g.ppb - 1) / g.ppb), (unsigned)B);
    agrid = dim3((unsigned)((items + 255) / 256), (unsigned)B);
    return MMU_OK;
}
}  // namespace
}  // namespace mmu

#define MMU_GN_DISPATCH(KERNEL_CALL)                                                                       \
    if (in_dtype == MMU_F32 && out_dtype == MMU_F32) { using TI = float; using TO = float; KERNEL_CALL; }   \
    else if (in_dtype == MMU_F32 && out_dtype == MMU_BF16) { using TI = float; using TO = __nv_bfloat16; KERNEL_CALL; } \
    else if (in_dtype == MMU_BF16 && out_dtype == MMU_BF16) { using TI = __nv_bfloat16; using TO = __nv_bfloat16; KERNEL_CALL; } \
    else if (in_dtype == MMU_BF16 && out_dtype == MMU_F32) { using TI = __nv_bfloat16; using TO = float; KERNEL_CALL; } \
    else return set_error(MMU_ERR_UNSUPPORTED, "group_norm: dtypes %d -> %d", in_dtype, out_dtype);

namespace mmu {
namespace {
// slots of the deterministic reductions: [b][pixel block][G][per]
size_t gn_det_bytes(int B, int C, int HW, int G, int per) {
    if (B <= 0 || C <= 0 || HW <= 0 || G <= 0) return 0;
    DetWs w{nullptr};
    w.take((size_t)B * gn_pblocks(B, HW, G) * G * per);
    return w.used;
}

// part == nullptr: the atomic path; otherwise the block sums go to the slots `part` and are reduced into `sums` in order
int gn_fwd(const void *x, const float *gamma, const float *beta, void *y, float *sums, float *mean, float *rstd, int32_t in_dtype,
           int32_t out_dtype, int32_t B, int32_t C, int32_t HW, int32_t G, float eps, float *part, cudaStream_t st) {
    GnGeom g;
    dim3 rgrid, agrid;
    if (int rc = gn_geom(g, B, C, HW, G, eps, rgrid, agrid)) return rc;
    if (!x || !gamma || !beta || !y || !sums || !mean || !rstd) return set_error(MMU_ERR_INVALID, "group_norm_fwd: null pointer");
    const size_t smem = 2 * kGnThreads * sizeof(float);
    if (in_dtype == MMU_F32) {
        if (part) gn_stats_kernel<float, true><<<rgrid, kGnThreads, smem, st>>>((const float *)x, part, g);
        else gn_stats_kernel<float><<<rgrid, kGnThreads, smem, st>>>((const float *)x, sums, g);
    } else if (in_dtype == MMU_BF16) {
        if (part) gn_stats_kernel<__nv_bfloat16, true><<<rgrid, kGnThreads, smem, st>>>((const __nv_bfloat16 *)x, part, g);
        else gn_stats_kernel<__nv_bfloat16><<<rgrid, kGnThreads, smem, st>>>((const __nv_bfloat16 *)x, sums, g);
    } else {
        return set_error(MMU_ERR_UNSUPPORTED, "group_norm: input dtype %d", in_dtype);
    }
    if (part) {
        count_launch();
        if (int rc = check_launch("group_norm_nhwc_fwd(deterministic)")) return rc;
        if (int rc = det_reduce(DetSum{part, (int64_t)rgrid.x, (int64_t)G * 2, B, 1, 2 * G, (int64_t)rgrid.x * G * 2, 0, sums, 2 * G, 0, 1}, st))
            return rc;
    }
    MMU_GN_DISPATCH((gn_apply_kernel<TI, TO><<<agrid, 256, 0, st>>>((const TI *)x, sums, gamma, beta, (TO *)y, mean, rstd, g)))
    count_launch(part ? 1 : 2);
    return check_launch("group_norm_nhwc_fwd");
}

int gn_bwd(const void *x, const float *gamma, const void *dy, const float *mean, const float *rstd, void *dx, float *sums2,
           float *dgamma_dbeta, int32_t in_dtype, int32_t out_dtype, int32_t B, int32_t C, int32_t HW, int32_t G, float *part, cudaStream_t st) {
    GnGeom g;
    dim3 rgrid, agrid;
    if (int rc = gn_geom(g, B, C, HW, G, 0.f, rgrid, agrid)) return rc;
    if (!x || !gamma || !dy || !mean || !rstd || !dx || !sums2 || !dgamma_dbeta) return set_error(MMU_ERR_INVALID, "group_norm_bwd: null pointer");
    const size_t smem = 10 * kGnThreads * sizeof(float);
    if (part) {
        MMU_GN_DISPATCH((gn_bwd_reduce_kernel<TI, TO, true><<<rgrid, kGnThreads, smem, st>>>(
            (const TI *)x, (const TO *)dy, mean, rstd, gamma, part, dgamma_dbeta, g)))
        count_launch();
        if (int rc = check_launch("group_norm_nhwc_bwd(deterministic)")) return rc;
        const int64_t nb = rgrid.x;
        // sums2[b][g][0..1] = sum over pixel blocks of slot k = 0..1
        if (int rc = det_reduce(DetSum{part, nb, (int64_t)G * 10, B, G, 2, nb * G * 10, 10, sums2, 2 * G, 2, 1}, st)) return rc;
        // dgamma[4g + k] (slot 2 + k), dbeta[4g + k] (slot 6 + k): summed over batch and pixel blocks
        if (int rc = det_reduce(DetSum{part + 2, (int64_t)B * nb, (int64_t)G * 10, 2, G, 4, 4, 10, dgamma_dbeta, C, 4, 1}, st)) return rc;
    } else {
        MMU_GN_DISPATCH((gn_bwd_reduce_kernel<TI, TO><<<rgrid, kGnThreads, smem, st>>>(
            (const TI *)x, (const TO *)dy, mean, rstd, gamma, sums2, dgamma_dbeta, g)))
        count_launch();
    }
    MMU_GN_DISPATCH((gn_bwd_apply_kernel<TI, TO><<<agrid, 256, 0, st>>>((const TI *)x, (const TO *)dy, mean, rstd, gamma, sums2, (TI *)dx, g)))
    count_launch();
    return check_launch("group_norm_nhwc_bwd");
}
}  // namespace
}  // namespace mmu

extern "C" int mmu_group_norm_nhwc_fwd(const void *x, const float *gamma, const float *beta, void *y, float *sums, float *mean, float *rstd,
                                       int32_t in_dtype, int32_t out_dtype, int32_t B, int32_t C, int32_t HW, int32_t G, float eps, void *stream) {
    return mmu::gn_fwd(x, gamma, beta, y, sums, mean, rstd, in_dtype, out_dtype, B, C, HW, G, eps, nullptr, static_cast<cudaStream_t>(stream));
}

// dy has dtype out_dtype (the forward's output dtype), dx has in_dtype.  sums2 (B*G*2) and dgamma_dbeta (2*C) are accumulated
// into: the caller zero-fills them.
extern "C" int mmu_group_norm_nhwc_bwd(const void *x, const float *gamma, const void *dy, const float *mean, const float *rstd, void *dx,
                                       float *sums2, float *dgamma_dbeta, int32_t in_dtype, int32_t out_dtype, int32_t B, int32_t C, int32_t HW,
                                       int32_t G, void *stream) {
    return mmu::gn_bwd(x, gamma, dy, mean, rstd, dx, sums2, dgamma_dbeta, in_dtype, out_dtype, B, C, HW, G, nullptr,
                       static_cast<cudaStream_t>(stream));
}

extern "C" size_t mmu_group_norm_nhwc_fwd_det_workspace(int32_t B, int32_t C, int32_t HW, int32_t G) { return mmu::gn_det_bytes(B, C, HW, G, 2); }
extern "C" size_t mmu_group_norm_nhwc_bwd_det_workspace(int32_t B, int32_t C, int32_t HW, int32_t G) { return mmu::gn_det_bytes(B, C, HW, G, 10); }

extern "C" int mmu_group_norm_nhwc_fwd_det(const void *x, const float *gamma, const float *beta, void *y, float *sums, float *mean, float *rstd,
                                           int32_t in_dtype, int32_t out_dtype, int32_t B, int32_t C, int32_t HW, int32_t G, float eps, void *ws,
                                           size_t ws_bytes, void *stream) {
    using namespace mmu;
    const size_t need = mmu_group_norm_nhwc_fwd_det_workspace(B, C, HW, G);
    if (need == 0) return set_error(MMU_ERR_INVALID, "group_norm_fwd_det: bad shape B%d C%d HW%d G%d", B, C, HW, G);
    if (int rc = det_ws_check(ws, ws_bytes, need, "group_norm_nhwc_fwd_det")) return rc;
    return gn_fwd(x, gamma, beta, y, sums, mean, rstd, in_dtype, out_dtype, B, C, HW, G, eps, static_cast<float *>(ws), static_cast<cudaStream_t>(stream));
}

extern "C" int mmu_group_norm_nhwc_bwd_det(const void *x, const float *gamma, const void *dy, const float *mean, const float *rstd, void *dx,
                                           float *sums2, float *dgamma_dbeta, int32_t in_dtype, int32_t out_dtype, int32_t B, int32_t C,
                                           int32_t HW, int32_t G, void *ws, size_t ws_bytes, void *stream) {
    using namespace mmu;
    const size_t need = mmu_group_norm_nhwc_bwd_det_workspace(B, C, HW, G);
    if (need == 0) return set_error(MMU_ERR_INVALID, "group_norm_bwd_det: bad shape B%d C%d HW%d G%d", B, C, HW, G);
    if (int rc = det_ws_check(ws, ws_bytes, need, "group_norm_nhwc_bwd_det")) return rc;
    return gn_bwd(x, gamma, dy, mean, rstd, dx, sums2, dgamma_dbeta, in_dtype, out_dtype, B, C, HW, G, static_cast<float *>(ws),
                  static_cast<cudaStream_t>(stream));
}
