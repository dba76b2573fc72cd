// Deterministic backward of F.interpolate(x, size=(Ho, Wo), mode="bilinear", align_corners=True) on 4-D maps, gather-side.
//
// The forward (ATen's) sends output o of an axis to inputs i0 and i0 + p with weights l0 and l1:
//   scale = (in - 1) / (out - 1) in fp32 (0 when out == 1), r = scale * o, i0 = (int)r, p = (i0 < in - 1), l1 = r - i0, l0 = 1 - l1.
// ATen's backward scatters with atomics.  Here every thread owns one dx element (NCHW) or one 16-byte channel vector (NHWC), walks a
// conservative window of candidate outputs along each axis, recomputes each candidate's (i0, p, l0, l1) exactly as above and keeps the
// taps that land on its input.  The sum runs over output rows ascending, then output columns ascending, in fp32, and is rounded once
// to dx's dtype: no atomics, no workspace, no zero-fill, the same bits on every run.
#include "common.cuh"

namespace mmu {

struct ResizeGeom {
    int C, hi, wi, ho, wo;
    float sh, sw;              // per-axis scale, as ATen computes it
    float inv_h, inv_w;        // 1 / scale (0 when the scale is 0)
    float margin_h, margin_w;  // window widening, see resize_window
    int64_t planes;            // NCHW: B * C;  NHWC: B
    int nv;                    // NHWC: channel vectors per pixel
};

// weight of output o on input i along one axis; false when o sends nothing to i
__device__ __forceinline__ bool resize_tap(float s, int o, int i, int in, float &w) {
    const float r = __fmul_rn(s, (float)o);
    const int i0 = (int)r;
    const int i1 = i0 + (i0 < in - 1 ? 1 : 0);
    const float l1 = __fsub_rn(r, (float)i0), l0 = 1.f - l1;
    w = (i0 == i ? l0 : 0.f) + (i1 == i ? l1 : 0.f);          // i1 == i0 (p == 0): both weights go to i0
    return i0 == i || i1 == i;
}

// candidate outputs [lo, hi] for input i: the outputs with i0 in {i - 1, i}, i.e. r in [i - 1, i + 1), so o in [(i - 1) / scale,
// (i + 1) / scale).  inv = 1 / scale in fp32; margin (host: 2 + out * 2^-22 outputs) covers the rounding of r = fl(scale * o) and of
// (i +- 1) * inv, each below out * 2^-23 outputs.
__device__ __forceinline__ void resize_window(float inv, float margin, int i, int out, int &lo, int &hi) {
    if (inv == 0.f) {          // scale 0 (in == 1 or out == 1): every output reads input 0 (and sends l1 = 0 to input 1)
        lo = 0;
        hi = i <= 1 ? out - 1 : -1;
        return;
    }
    const float a = (float)(i - 1) * inv - margin, b = (float)(i + 1) * inv + margin;
    lo = a <= 0.f ? 0 : (int)fminf(floorf(a), (float)out);
    hi = b >= (float)(out - 1) ? out - 1 : (int)ceilf(b);
}

// grid: (ceil(hi * wi / 256), min(ceil(B * C / 4), 65535)); one thread per input pixel of 4 or more (b, c) planes (the window is
// computed once for all of them)
template <typename T>
__global__ void __launch_bounds__(256) resize_bilinear_bwd_nchw_kernel(const T *__restrict__ dout, T *__restrict__ dx, ResizeGeom g) {
    const int pix = blockIdx.x * blockDim.x + threadIdx.x;
    if (pix >= g.hi * g.wi) return;
    const int ih = pix / g.wi, iw = pix - ih * g.wi;
    int oh0, oh1, ow0, ow1;
    resize_window(g.inv_h, g.margin_h, ih, g.ho, oh0, oh1);
    resize_window(g.inv_w, g.margin_w, iw, g.wo, ow0, ow1);
    const int64_t oplane = (int64_t)g.ho * g.wo, iplane = (int64_t)g.hi * g.wi;
    for (int64_t pl = blockIdx.y; pl < g.planes; pl += gridDim.y) {
        const T *src = dout + pl * oplane;
        float acc = 0.f;
        for (int oh = oh0; oh <= oh1; ++oh) {
            float wh;
            if (!resize_tap(g.sh, oh, ih, g.hi, wh)) continue;
            const T *row = src + (int64_t)oh * g.wo;
            for (int ow = ow0; ow <= ow1; ++ow) {
                float ww;
                if (!resize_tap(g.sw, ow, iw, g.wi, ww)) continue;
                acc = fmaf(Elem<T>::to_f(row[ow]), wh * ww, acc);
            }
        }
        dx[pl * iplane + pix] = Elem<T>::from_f(acc);
    }
}

// 16-byte load / store of 4 fp32 / 8 bf16 values, converted in registers
__device__ __forceinline__ void load16(const float *src, float (&v)[4]) {
    const float4 q = *reinterpret_cast<const float4 *>(src);
    v[0] = q.x, v[1] = q.y, v[2] = q.z, v[3] = q.w;
}
__device__ __forceinline__ void load16(const __nv_bfloat16 *src, float (&v)[8]) {
    const uint4 q = *reinterpret_cast<const uint4 *>(src);
    const uint32_t u[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) v[2 * j] = __uint_as_float(u[j] << 16), v[2 * j + 1] = __uint_as_float(u[j] & 0xffff0000u);
}
__device__ __forceinline__ void store16(float *dst, const float (&a)[4]) { *reinterpret_cast<float4 *>(dst) = make_float4(a[0], a[1], a[2], a[3]); }
__device__ __forceinline__ void store16(__nv_bfloat16 *dst, const float (&a)[8]) {
    uint32_t u[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const __nv_bfloat162 h = __floats2bfloat162_rn(a[2 * j], a[2 * j + 1]);
        u[j] = (uint32_t)__bfloat16_as_ushort(h.x) | ((uint32_t)__bfloat16_as_ushort(h.y) << 16);
    }
    *reinterpret_cast<uint4 *>(dst) = make_uint4(u[0], u[1], u[2], u[3]);
}

// grid: (ceil(hi * wi * nv / 256), min(B, 65535)); one thread per (input pixel, vector of Elem<T>::kVec channels).  VEC: C is a
// multiple of the vector width (16-byte loads and stores); otherwise the channels of the vector are walked one by one (C = 1 logits).
template <typename T, bool VEC>
__global__ void __launch_bounds__(256) resize_bilinear_bwd_nhwc_kernel(const T *__restrict__ dout, T *__restrict__ dx, ResizeGeom g) {
    constexpr int V = Elem<T>::kVec;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= g.hi * g.wi * g.nv) return;
    const int pix = t / g.nv, cv = t - pix * g.nv;
    const int ih = pix / g.wi, iw = pix - ih * g.wi;
    const int c0 = cv * V, nc = VEC ? V : min(V, g.C - c0);
    int oh0, oh1, ow0, ow1;
    resize_window(g.inv_h, g.margin_h, ih, g.ho, oh0, oh1);
    resize_window(g.inv_w, g.margin_w, iw, g.wo, ow0, ow1);
    for (int b = blockIdx.y; b < g.planes; b += gridDim.y) {
        float acc[V];
#pragma unroll
        for (int j = 0; j < V; ++j) acc[j] = 0.f;
        for (int oh = oh0; oh <= oh1; ++oh) {
            float wh;
            if (!resize_tap(g.sh, oh, ih, g.hi, wh)) continue;
            const T *row = dout + (((int64_t)b * g.ho + oh) * g.wo) * g.C + c0;
            for (int ow = ow0; ow <= ow1; ++ow) {
                float ww;
                if (!resize_tap(g.sw, ow, iw, g.wi, ww)) continue;
                const float w = wh * ww;
                const T *src = row + (int64_t)ow * g.C;
                if constexpr (VEC) {
                    float v[V];
                    load16(src, v);
#pragma unroll
                    for (int j = 0; j < V; ++j) acc[j] = fmaf(v[j], w, acc[j]);
                } else {
#pragma unroll
                    for (int j = 0; j < V; ++j)
                        if (j < nc) acc[j] = fmaf(Elem<T>::to_f(src[j]), w, acc[j]);
                }
            }
        }
        T *dst = dx + (((int64_t)b * g.hi + ih) * g.wi + iw) * g.C + c0;
        if constexpr (VEC) {
            store16(dst, acc);
        } else {
#pragma unroll
            for (int j = 0; j < V; ++j)
                if (j < nc) dst[j] = Elem<T>::from_f(acc[j]);
        }
    }
}

namespace {
// a * b * c * d without overflowing int64 (all positive); false on overflow
bool count4(int64_t a, int64_t b, int64_t c, int64_t d, int64_t &n) {
    const int64_t f[3] = {b, c, d};
    n = a;
    for (int k = 0; k < 3; ++k) {
        if (n > INT64_MAX / f[k]) return false;
        n *= f[k];
    }
    return true;
}

template <typename T>
void launch_resize_bwd(const void *dout, void *dx, const ResizeGeom &g, bool channels_last, bool vec, cudaStream_t st) {
    const int64_t rows = channels_last ? g.planes : (g.planes + 3) / 4;
    const unsigned ys = (unsigned)(rows < 65535 ? rows : 65535);
    if (channels_last) {
        const dim3 grid((unsigned)(((int64_t)g.hi * g.wi * g.nv + 255) / 256), ys);
        if (vec) resize_bilinear_bwd_nhwc_kernel<T, true><<<grid, 256, 0, st>>>((const T *)dout, (T *)dx, g);
        else resize_bilinear_bwd_nhwc_kernel<T, false><<<grid, 256, 0, st>>>((const T *)dout, (T *)dx, g);
    } else {
        const dim3 grid((unsigned)(((int64_t)g.hi * g.wi + 255) / 256), ys);
        resize_bilinear_bwd_nchw_kernel<T><<<grid, 256, 0, st>>>((const T *)dout, (T *)dx, g);
    }
}
}  // namespace
}  // namespace mmu

extern "C" int mmu_resize_bilinear_bwd_det(const void *dout, void *dx, int32_t dtype, int32_t B, int32_t C, int32_t H_in, int32_t W_in,
                                           int32_t H_out, int32_t W_out, int32_t channels_last, void *stream) {
    using namespace mmu;
    if (!dout || !dx) return set_error(MMU_ERR_INVALID, "resize_bilinear_bwd_det: null pointer");
    if (dtype != MMU_F32 && dtype != MMU_BF16) return set_error(MMU_ERR_INVALID, "resize_bilinear_bwd_det: dtype %d (fp32 or bf16 only)", dtype);
    if (B <= 0 || C <= 0 || H_in <= 0 || W_in <= 0 || H_out <= 0 || W_out <= 0)
        return set_error(MMU_ERR_INVALID, "resize_bilinear_bwd_det: bad shape B%d C%d %dx%d -> %dx%d", B, C, H_in, W_in, H_out, W_out);
    const int V = dtype == MMU_F32 ? 4 : 8;
    const int nv = (C + V - 1) / V;
    int64_t n_in, n_out;
    // per-plane indices are int32 (threads of one plane: H_in * W_in, or H_in * W_in * channel vectors); element offsets are int64
    if (!count4(B, C, H_in, W_in, n_in) || !count4(B, C, H_out, W_out, n_out) || (int64_t)H_in * W_in * (channels_last ? nv : 1) > INT32_MAX ||
        (int64_t)H_out * W_out > INT32_MAX)
        return set_error(MMU_ERR_INVALID, "resize_bilinear_bwd_det: B%d C%d %dx%d -> %dx%d overflows the kernel's index range", B, C, H_in, W_in,
                         H_out, W_out);
    ResizeGeom g;
    g.C = C, g.hi = H_in, g.wi = W_in, g.ho = H_out, g.wo = W_out, g.nv = nv;
    g.sh = H_out > 1 ? (float)(H_in - 1) / (float)(H_out - 1) : 0.f;
    g.sw = W_out > 1 ? (float)(W_in - 1) / (float)(W_out - 1) : 0.f;
    g.inv_h = g.sh > 0.f ? (float)(1.0 / g.sh) : 0.f;
    g.inv_w = g.sw > 0.f ? (float)(1.0 / g.sw) : 0.f;
    g.margin_h = 2.f + (float)H_out * 0x1p-22f;
    g.margin_w = 2.f + (float)W_out * 0x1p-22f;
    g.planes = channels_last ? (int64_t)B : (int64_t)B * C;
    const bool vec = C % V == 0 && reinterpret_cast<uintptr_t>(dout) % 16 == 0 && reinterpret_cast<uintptr_t>(dx) % 16 == 0;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (dtype == MMU_F32) launch_resize_bwd<float>(dout, dx, g, channels_last != 0, vec, st);
    else launch_resize_bwd<__nv_bfloat16>(dout, dx, g, channels_last != 0, vec, st);
    count_launch();
    return check_launch("resize_bilinear_bwd_det");
}
