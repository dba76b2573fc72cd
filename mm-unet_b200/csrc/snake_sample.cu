// Snake (dynamic-snake-conv) row sampler for MMConv, sm_100a: the bilinear gather that follows the Mamba-refined row
// coordinates (the caller of the hot path, SURVEY.md section 8 row f2).
//
// Reference: src/UM_Net/MMUNet.py:190-224 builds, per tap k of a K-tap vertical snake kernel, a coordinate map
//   y[b,k,h,w] (learned, fractional) and x = w + (k - K/2) (integer), clamps both to the image, rescales them to [-1,1]
//   (:229-242) and calls F.grid_sample(bilinear, zeros, align_corners=True) on a (B, H*K, W, 2) grid -> (B, C, H*K, W).
// With integer x the bilinear stencil degenerates to a 2-tap interpolation along rows:
//   yc = clamp(y, 0, H-1), r0 = floor(yc), f = yc - r0, xk = clamp(w + k - K/2, 0, W-1)
//   out[b,c,h*K+k,w] = (1-f) * feat[b,c,r0,xk] + f * feat[b,c,r0+1,xk]          (row r0+1 == H contributes 0: then f == 0)
// One thread owns one (b, h, k, w) sample - r0, f, xk are computed once - and walks a block of channels; consecutive
// threads are consecutive w, so loads and stores are coalesced rows.  No (B,H*K,W,2) grid, no fp32 up-cast of the feature
// map, output written directly in the consumer's dtype.
// Backward: d_feat (fp32, caller zero-fills) receives the two taps by red.global.add.f32; d_y[b,k,h,w] = sum_c dout * (v1 - v0)
// inside the clamp range (torch.clamp passes the gradient on the closed interval), accumulated across channel blocks.
// Deterministic backward (mmu_snake_sample_bwd_det): gather-side, no float atomics - see snake_bwd_det_dfeat_kernel.
#include "common.cuh"

namespace mmu {

template <typename T> __device__ __forceinline__ float ldf(const T *p) { return Elem<T>::to_f(*p); }

struct SnakeGeom {
    int B, C, H, W, K, cpb;   // cpb = channels per thread
};

// Sample coordinates.  `row` = (b*H + h)*K + k (one output row of W samples), decomposed with 32-bit arithmetic only (64-bit
// div/mod by runtime values costs hundreds of instructions per thread and dominated the first version of these kernels).
__device__ __forceinline__ void snake_coord(const SnakeGeom &g, const float *__restrict__ y, unsigned row, int w, int &b, int &h, int &k,
                                            int &r0, int &r1ok, float &f, int &xk, bool &inside) {
    const unsigned bh = row / (unsigned)g.K;
    k = (int)(row - bh * (unsigned)g.K);
    b = (int)(bh / (unsigned)g.H);
    h = (int)(bh - (unsigned)b * (unsigned)g.H);
    const float yv = y[(((int64_t)b * g.K + k) * g.H + h) * g.W + w];
    const float hi = (float)(g.H - 1);
    const bool is_nan = yv != yv;                // a NaN coordinate must poison the sample and its gradients, as torch.clamp +
    inside = (yv >= 0.f && yv <= hi) || is_nan;  // grid_sample do (fminf/fmaxf alone would silently map it to row 0)
    const float yc = fminf(fmaxf(yv, 0.f), hi);
    const float fl = floorf(yc);
    r0 = (int)fl;
    f = is_nan ? yv : yc - fl;
    r1ok = r0 + 1 < g.H;
    xk = min(max(w + k - g.K / 2, 0), g.W - 1);
}

template <typename TI, typename TO>
__global__ void __launch_bounds__(256) snake_fwd_kernel(const TI *__restrict__ feat, const float *__restrict__ y, TO *__restrict__ out,
                                                        SnakeGeom g) {
    int b, h, k, r0, r1ok, xk;
    float f;
    bool inside;
    const int w = blockIdx.y * blockDim.x + threadIdx.x;          // grid: (output row, w block, channel block)
    if (w >= g.W) return;
    snake_coord(g, y, blockIdx.x, w, b, h, k, r0, r1ok, f, xk, inside);
    const int c0 = blockIdx.z * g.cpb, c1 = min(g.C, c0 + g.cpb);
    const int64_t plane = (int64_t)g.H * g.W;
    const TI *p0 = feat + ((int64_t)b * g.C + c0) * plane + (int64_t)r0 * g.W + xk;
    TO *o = out + (((int64_t)b * g.C + c0) * g.H + h) * g.K * g.W + (int64_t)k * g.W + w;
    const int64_t oplane = plane * g.K;
    const float f0 = 1.f - f;
    const int d1 = r1ok ? g.W : 0;           // row r0+1 outside the map: weight f is 0, re-read row r0
#pragma unroll 4
    for (int c = c0; c < c1; ++c, p0 += plane, o += oplane) {
        const float v0 = ldf(p0), v1 = ldf(p0 + d1);
        *o = Elem<TO>::from_f(fmaf(f, v1, f0 * v0));
    }
}

template <typename TI, typename TO>
__global__ void __launch_bounds__(256) snake_bwd_kernel(const TI *__restrict__ feat, const float *__restrict__ y, const TO *__restrict__ dout,
                                                        float *__restrict__ dfeat, float *__restrict__ dy, SnakeGeom g) {
    int b, h, k, r0, r1ok, xk;
    float f;
    bool inside;
    const int w = blockIdx.y * blockDim.x + threadIdx.x;          // grid: (output row, w block, channel block)
    if (w >= g.W) return;
    snake_coord(g, y, blockIdx.x, w, b, h, k, r0, r1ok, f, xk, inside);
    const int c0 = blockIdx.z * g.cpb, c1 = min(g.C, c0 + g.cpb);
    const int64_t plane = (int64_t)g.H * g.W, oplane = plane * g.K;
    const int64_t fo = ((int64_t)b * g.C + c0) * plane + (int64_t)r0 * g.W + xk;
    const TI *p0 = feat + fo;
    float *d0 = dfeat + fo;
    const TO *go = dout + (((int64_t)b * g.C + c0) * g.H + h) * g.K * g.W + (int64_t)k * g.W + w;
    const float f0 = 1.f - f;
    float acc = 0.f;
#pragma unroll 4
    for (int c = c0; c < c1; ++c, p0 += plane, d0 += plane, go += oplane) {
        const float gv = ldf(go);
        const float v0 = ldf(p0);
        atomicAdd(d0, f0 * gv);
        if (r1ok) {
            const float v1 = ldf(p0 + g.W);
            atomicAdd(d0 + g.W, f * gv);
            acc = fmaf(gv, v1 - v0, acc);
        } else {
            acc = fmaf(gv, -v0, acc);       // zero padding below the last row
        }
    }
    if (dy != nullptr && inside) atomicAdd(dy + (((int64_t)b * g.K + k) * g.H + h) * g.W + w, fmaf(f, 0.f, acc));   // NaN f -> NaN dy
}

// ---- channels-last (NHWC) variants: feat[b][r][x][c], out[b][h*K+k][w][c].  A thread owns 4 consecutive channels of one sample,
// consecutive threads walk the channel axis: every access is a coalesced 8/16-byte vector; the backward uses
// red.global.add.v4.f32 for the two taps and a shuffle reduction over the sample's channel threads for d_y.
template <typename T> struct Vec4;
template <> struct Vec4<float> {
    static __device__ __forceinline__ void ld(const float *p, float (&v)[4]) {
        const float4 q = *reinterpret_cast<const float4 *>(p);
        v[0] = q.x, v[1] = q.y, v[2] = q.z, v[3] = q.w;
    }
    static __device__ __forceinline__ void st(float *p, const float (&v)[4]) { *reinterpret_cast<float4 *>(p) = make_float4(v[0], v[1], v[2], v[3]); }
};
template <> struct Vec4<__nv_bfloat16> {
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

template <typename TI, typename TO>
__global__ void __launch_bounds__(256) snake_fwd_nhwc_kernel(const TI *__restrict__ feat, const float *__restrict__ y, TO *__restrict__ out,
                                                             SnakeGeom g) {
    const unsigned cv = (unsigned)g.C >> 2;                     // channel vectors per sample (a power of two)
    const unsigned tix = blockIdx.y * blockDim.x + threadIdx.x;  // (w, channel vector) inside output row blockIdx.x
    const int w = (int)(tix >> g.cpb);                          // cpb holds log2(cv) for the channels-last kernels
    if (w >= g.W) return;
    int b, h, k, r0, r1ok, xk;
    float f;
    bool inside;
    snake_coord(g, y, blockIdx.x, w, b, h, k, r0, r1ok, f, xk, inside);
    const int c = (int)(tix & (cv - 1)) << 2;
    const TI *p0 = feat + (((int64_t)b * g.H + r0) * g.W + xk) * g.C + c;
    float v0[4], v1[4], o[4];
    Vec4<TI>::ld(p0, v0);
    Vec4<TI>::ld(p0 + (r1ok ? (int64_t)g.W * g.C : 0), v1);
    const float f0 = 1.f - f;
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = fmaf(f, v1[i], f0 * v0[i]);
    Vec4<TO>::st(out + ((((int64_t)b * g.H + h) * g.K + k) * g.W + w) * g.C + c, o);
}

template <typename TI, typename TO>
__global__ void __launch_bounds__(256) snake_bwd_nhwc_kernel(const TI *__restrict__ feat, const float *__restrict__ y, const TO *__restrict__ dout,
                                                             float *__restrict__ dfeat, float *__restrict__ dy, SnakeGeom g) {
    const unsigned cv = (unsigned)g.C >> 2;
    const unsigned tix = blockIdx.y * blockDim.x + threadIdx.x;
    const int w = (int)(tix >> g.cpb);
    int b = 0, h = 0, k = 0, r0 = 0, r1ok = 0, xk = 0;
    float f = 0.f;
    bool inside = false;
    const bool live = w < g.W;
    float acc = 0.f;
    if (live) {
        snake_coord(g, y, blockIdx.x, w, b, h, k, r0, r1ok, f, xk, inside);
        const int c = (int)(tix & (cv - 1)) << 2;
        const int64_t fo = (((int64_t)b * g.H + r0) * g.W + xk) * g.C + c;
        float gv[4], v0[4], v1[4] = {0.f, 0.f, 0.f, 0.f};
        Vec4<TO>::ld(dout + ((((int64_t)b * g.H + h) * g.K + k) * g.W + w) * g.C + c, gv);
        Vec4<TI>::ld(feat + fo, v0);
        const float f0 = 1.f - f;
        asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dfeat + fo), "f"(f0 * gv[0]), "f"(f0 * gv[1]), "f"(f0 * gv[2]),
                     "f"(f0 * gv[3]) : "memory");
        if (r1ok) {
            const int64_t f1 = fo + (int64_t)g.W * g.C;
            Vec4<TI>::ld(feat + f1, v1);
            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dfeat + f1), "f"(f * gv[0]), "f"(f * gv[1]), "f"(f * gv[2]),
                         "f"(f * gv[3]) : "memory");
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) acc = fmaf(gv[i], v1[i] - v0[i], acc);
        acc = fmaf(f, 0.f, acc);                 // NaN f -> NaN dy
        if (!inside) acc = 0.f;
    }
    // d_y: sum over the sample's channel threads.  cv is a power of two (checked by the host): groups of min(cv, 32) lanes
    const int grp = cv < 32 ? (int)cv : 32;
    for (int o = grp >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (live && dy != nullptr && (threadIdx.x & (grp - 1)) == 0 && acc != 0.f)
        atomicAdd(dy + (((int64_t)b * g.K + k) * g.H + h) * g.W + w, acc);
}

// ---- deterministic backward -------------------------------------------------------------------------------------------------
// d_feat: the scatter targets are data-dependent rows, so the work is organised by TARGET column instead.  One thread owns the column
// dfeat[b, c (or 4 channels), :, x] - nobody else writes it - and walks every sample that reads column x, i.e. every (k, h, w) with
// clamp(w + k - K/2, 0, W-1) == x, in the fixed order k, h, w.  The two taps of consecutive samples mostly hit the same or the next
// row, so they are summed in registers over a window of rows (rc, rc + 1) and added to global memory (plain read-modify-write) when
// the window moves.  Consecutive threads own consecutive x (NCHW) or channel vectors (NHWC): the dout / y / dfeat accesses coalesce.
// d_y: one thread per sample sums over ALL channels in channel order (snake_bwd_det_dy_kernel).
__device__ __forceinline__ void snake_rowf(float yv, int H, int &r0, bool &r1ok, float &f, bool &inside) {
    const float hi = (float)(H - 1);
    const bool is_nan = yv != yv;                // as snake_coord: NaN poisons the sample and its gradients
    inside = (yv >= 0.f && yv <= hi) || is_nan;
    const float yc = fminf(fmaxf(yv, 0.f), hi);
    const float fl = floorf(yc);
    r0 = (int)fl;
    f = is_nan ? yv : yc - fl;
    r1ok = r0 + 1 < H;
}

template <int NV> struct RowWin {      // pending contributions to rows rc and rc + 1 of one owned column (NV channels)
    int rc = -2;
    float a0[NV] = {}, a1[NV] = {};
    __device__ __forceinline__ void flush(float *col, int64_t rstride, int H) {
        if (rc < 0) return;
        float *p = col + (int64_t)rc * rstride;
#pragma unroll
        for (int i = 0; i < NV; ++i) p[i] += a0[i];
        if (rc + 1 < H) {
#pragma unroll
            for (int i = 0; i < NV; ++i) p[rstride + i] += a1[i];
        }
    }
    __device__ __forceinline__ void add(int r0, bool r1ok, float f, const float (&gv)[NV], float *col, int64_t rstride, int H) {
        const float f0 = 1.f - f;
        if (r0 == rc + 1) {              // the window slides by one row: row rc is complete
            flush_row0(col, rstride);
#pragma unroll
            for (int i = 0; i < NV; ++i) a0[i] = a1[i], a1[i] = 0.f;
            rc = r0;
        } else if (r0 != rc) {
            flush(col, rstride, H);
#pragma unroll
            for (int i = 0; i < NV; ++i) a0[i] = 0.f, a1[i] = 0.f;
            rc = r0;
        }
#pragma unroll
        for (int i = 0; i < NV; ++i) {
            a0[i] = fmaf(f0, gv[i], a0[i]);
            if (r1ok) a1[i] = fmaf(f, gv[i], a1[i]);
        }
    }
    __device__ __forceinline__ void flush_row0(float *col, int64_t rstride) {
        if (rc < 0) return;
        float *p = col + (int64_t)rc * rstride;
#pragma unroll
        for (int i = 0; i < NV; ++i) p[i] += a0[i];
    }
};

// NCHW: grid (x blocks, b*C + c); NHWC (NV = 4): grid (blocks over (x, channel vector), b)
template <typename TO, bool NHWC>
__global__ void __launch_bounds__(256) snake_bwd_det_dfeat_kernel(const float *__restrict__ y, const TO *__restrict__ dout,
                                                                  float *__restrict__ dfeat, SnakeGeom g) {
    constexpr int NV = NHWC ? 4 : 1;
    const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
    const int x = NHWC ? (int)(t >> g.cpb) : (int)t;
    const int b = NHWC ? (int)blockIdx.y : (int)(blockIdx.y / (unsigned)g.C);
    const int c = NHWC ? (int)(t & (((unsigned)g.C >> 2) - 1)) << 2 : (int)blockIdx.y - b * g.C;
    if (x >= g.W) return;
    const int H = g.H, W = g.W, K = g.K;
    float *col = NHWC ? dfeat + ((int64_t)b * H * W + x) * g.C + c : dfeat + ((int64_t)b * g.C + c) * H * W + x;
    const int64_t rstride = NHWC ? (int64_t)W * g.C : W;
    RowWin<NV> win;
    for (int k = 0; k < K; ++k) {
        const int s = k - K / 2;
        const int wa = x == 0 ? 0 : max(0, x - s), wb = x == W - 1 ? W - 1 : min(W - 1, x - s);
        if (wa > wb) continue;
        const float *yk = y + ((int64_t)b * K + k) * H * W;
#pragma unroll 1
        for (int h = 0; h < H; ++h) {
#pragma unroll 1
            for (int w = wa; w <= wb; ++w) {
                int r0;
                bool r1ok, inside;
                float f, gv[NV];
                snake_rowf(yk[(int64_t)h * W + w], H, r0, r1ok, f, inside);
                if constexpr (NHWC) {
                    Vec4<TO>::ld(dout + ((((int64_t)b * H + h) * K + k) * W + w) * g.C + c, gv);
                } else {
                    gv[0] = ldf(dout + (((int64_t)b * g.C + c) * H + h) * K * W + (int64_t)k * W + w);
                }
                win.add(r0, r1ok, f, gv, col, rstride, H);
            }
        }
    }
    win.flush(col, rstride, H);
}

// d_y[b,k,h,w] += sum over every channel, in channel order, of dout * (v1 - v0) (inside the clamp range).  Grid as snake_fwd_kernel
// with one channel block (NCHW), or (output row, w blocks of 256) (NHWC).
template <typename TI, typename TO, bool NHWC>
__global__ void __launch_bounds__(256) snake_bwd_det_dy_kernel(const TI *__restrict__ feat, const float *__restrict__ y, const TO *__restrict__ dout,
                                                               float *__restrict__ dy, SnakeGeom g) {
    int b, h, k, r0, r1ok, xk;
    float f;
    bool inside;
    const int w = blockIdx.y * blockDim.x + threadIdx.x;
    if (w >= g.W) return;
    snake_coord(g, y, blockIdx.x, w, b, h, k, r0, r1ok, f, xk, inside);
    const int64_t plane = (int64_t)g.H * g.W;
    float acc = 0.f;
    if constexpr (NHWC) {
        const TI *p0 = feat + (((int64_t)b * g.H + r0) * g.W + xk) * g.C;
        const TO *go = dout + ((((int64_t)b * g.H + h) * g.K + k) * g.W + w) * g.C;
        for (int c = 0; c < g.C; c += 4) {
            float gv[4], v0[4], v1[4] = {0.f, 0.f, 0.f, 0.f};
            Vec4<TO>::ld(go + c, gv);
            Vec4<TI>::ld(p0 + c, v0);
            if (r1ok) Vec4<TI>::ld(p0 + (int64_t)g.W * g.C + c, v1);
#pragma unroll
            for (int i = 0; i < 4; ++i) acc = fmaf(gv[i], v1[i] - v0[i], acc);
        }
    } else {
        const TI *p0 = feat + (int64_t)b * g.C * plane + (int64_t)r0 * g.W + xk;
        const TO *go = dout + (((int64_t)b * g.C) * g.H + h) * g.K * g.W + (int64_t)k * g.W + w;
#pragma unroll 4
        for (int c = 0; c < g.C; ++c, p0 += plane, go += plane * g.K) {
            const float gv = ldf(go), v0 = ldf(p0);
            acc = r1ok ? fmaf(gv, ldf(p0 + g.W) - v0, acc) : fmaf(gv, -v0, acc);
        }
    }
    if (inside) dy[(((int64_t)b * g.K + k) * g.H + h) * g.W + w] += fmaf(f, 0.f, acc);   // NaN f -> NaN dy; one owner per sample
}

namespace {
int geom_nhwc(SnakeGeom &g, int B, int C, int H, int W, int K, dim3 &grid, int &threads) {
    threads = 256;
    if (B <= 0 || C <= 0 || H <= 0 || W <= 0 || K <= 0) return set_error(MMU_ERR_INVALID, "snake_sample: bad shape B%d C%d H%d W%d K%d", B, C, H, W, K);
    if (C % 4 != 0 || ((C / 4) & (C / 4 - 1)) != 0)
        return set_error(MMU_ERR_UNSUPPORTED, "snake_sample (channels-last): C=%d must be 4 * a power of two", C);
    const int64_t rows = (int64_t)B * H * K, per_row = (int64_t)W * (C / 4);
    if (rows > 0x7fffffffLL || (per_row + 255) / 256 > 65535) return set_error(MMU_ERR_UNSUPPORTED, "snake_sample: problem too large");
    int lg = 0;
    while ((1 << lg) < C / 4) ++lg;
    g = {B, C, H, W, K, lg};                       // cpb = log2(channel vectors per sample)
    grid = dim3((unsigned)rows, (unsigned)((per_row + 255) / 256));
    return MMU_OK;
}

int geom(SnakeGeom &g, int B, int C, int H, int W, int K, dim3 &grid, int &threads) {
    if (B <= 0 || C <= 0 || H <= 0 || W <= 0 || K <= 0) return set_error(MMU_ERR_INVALID, "snake_sample: bad shape B%d C%d H%d W%d K%d", B, C, H, W, K);
    const int64_t rows = (int64_t)B * H * K;
    if (rows > 0x7fffffffLL) return set_error(MMU_ERR_UNSUPPORTED, "snake_sample: too many rows");
    // channel blocks: enough CTAs to fill the GPU a few times over, at least 8 channels per thread to amortise the coordinates
    threads = W >= 128 ? 128 : ((W + 31) / 32) * 32;           // one output row per block row; narrow maps use narrow blocks
    const int wblocks = (W + threads - 1) / threads;
    const int64_t blocks = rows * wblocks;
    int cblocks = 1;
    while (blocks * cblocks < 148 * 16 && C / (cblocks * 2) >= 8 && cblocks < 32768) cblocks *= 2;
    g = {B, C, H, W, K, (C + cblocks - 1) / cblocks};
    if (wblocks > 65535) return set_error(MMU_ERR_UNSUPPORTED, "snake_sample: W too large");
    grid = dim3((unsigned)rows, (unsigned)wblocks, (unsigned)((C + g.cpb - 1) / g.cpb));
    return MMU_OK;
}
}  // namespace
}  // namespace mmu

extern "C" int mmu_snake_sample_fwd(const void *feat, const float *y, void *out, int32_t in_dtype, int32_t out_dtype, int32_t B,
                                    int32_t C, int32_t H, int32_t W, int32_t K, int32_t channels_last, void *stream) {
    using namespace mmu;
    SnakeGeom g;
    dim3 grid;
    int nthr = 0;
    if (int rc = channels_last ? geom_nhwc(g, B, C, H, W, K, grid, nthr) : geom(g, B, C, H, W, K, grid, nthr)) return rc;
    if (!feat || !y || !out) return set_error(MMU_ERR_INVALID, "snake_sample_fwd: null pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (channels_last) {
        if (in_dtype == MMU_F32 && out_dtype == MMU_F32)
            snake_fwd_nhwc_kernel<float, float><<<grid, 256, 0, st>>>((const float *)feat, y, (float *)out, g);
        else if (in_dtype == MMU_F32 && out_dtype == MMU_BF16)
            snake_fwd_nhwc_kernel<float, __nv_bfloat16><<<grid, 256, 0, st>>>((const float *)feat, y, (__nv_bfloat16 *)out, g);
        else if (in_dtype == MMU_BF16 && out_dtype == MMU_BF16)
            snake_fwd_nhwc_kernel<__nv_bfloat16, __nv_bfloat16><<<grid, 256, 0, st>>>((const __nv_bfloat16 *)feat, y, (__nv_bfloat16 *)out, g);
        else if (in_dtype == MMU_BF16 && out_dtype == MMU_F32)
            snake_fwd_nhwc_kernel<__nv_bfloat16, float><<<grid, 256, 0, st>>>((const __nv_bfloat16 *)feat, y, (float *)out, g);
        else
            return set_error(MMU_ERR_UNSUPPORTED, "snake_sample_fwd: dtypes %d -> %d", in_dtype, out_dtype);
        count_launch();
        return check_launch("snake_sample_fwd (channels-last)");
    }
    if (in_dtype == MMU_F32 && out_dtype == MMU_F32)
        snake_fwd_kernel<float, float><<<grid, nthr, 0, st>>>((const float *)feat, y, (float *)out, g);
    else if (in_dtype == MMU_F32 && out_dtype == MMU_BF16)
        snake_fwd_kernel<float, __nv_bfloat16><<<grid, nthr, 0, st>>>((const float *)feat, y, (__nv_bfloat16 *)out, g);
    else if (in_dtype == MMU_BF16 && out_dtype == MMU_BF16)
        snake_fwd_kernel<__nv_bfloat16, __nv_bfloat16><<<grid, nthr, 0, st>>>((const __nv_bfloat16 *)feat, y, (__nv_bfloat16 *)out, g);
    else if (in_dtype == MMU_BF16 && out_dtype == MMU_F32)
        snake_fwd_kernel<__nv_bfloat16, float><<<grid, nthr, 0, st>>>((const __nv_bfloat16 *)feat, y, (float *)out, g);
    else
        return set_error(MMU_ERR_UNSUPPORTED, "snake_sample_fwd: dtypes %d -> %d", in_dtype, out_dtype);
    count_launch();
    return check_launch("snake_sample_fwd");
}

extern "C" int mmu_snake_sample_bwd(const void *feat, const float *y, const void *dout, float *dfeat, float *dy, int32_t in_dtype,
                                    int32_t out_dtype, int32_t B, int32_t C, int32_t H, int32_t W, int32_t K, int32_t channels_last,
                                    void *stream) {
    using namespace mmu;
    SnakeGeom g;
    dim3 grid;
    int nthr = 0;
    if (int rc = channels_last ? geom_nhwc(g, B, C, H, W, K, grid, nthr) : geom(g, B, C, H, W, K, grid, nthr)) return rc;
    if (!feat || !y || !dout || !dfeat) return set_error(MMU_ERR_INVALID, "snake_sample_bwd: null pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (channels_last) {
        if (in_dtype == MMU_F32 && out_dtype == MMU_F32)
            snake_bwd_nhwc_kernel<float, float><<<grid, 256, 0, st>>>((const float *)feat, y, (const float *)dout, dfeat, dy, g);
        else if (in_dtype == MMU_F32 && out_dtype == MMU_BF16)
            snake_bwd_nhwc_kernel<float, __nv_bfloat16><<<grid, 256, 0, st>>>((const float *)feat, y, (const __nv_bfloat16 *)dout, dfeat, dy, g);
        else if (in_dtype == MMU_BF16 && out_dtype == MMU_BF16)
            snake_bwd_nhwc_kernel<__nv_bfloat16, __nv_bfloat16><<<grid, 256, 0, st>>>((const __nv_bfloat16 *)feat, y, (const __nv_bfloat16 *)dout, dfeat, dy, g);
        else if (in_dtype == MMU_BF16 && out_dtype == MMU_F32)
            snake_bwd_nhwc_kernel<__nv_bfloat16, float><<<grid, 256, 0, st>>>((const __nv_bfloat16 *)feat, y, (const float *)dout, dfeat, dy, g);
        else
            return set_error(MMU_ERR_UNSUPPORTED, "snake_sample_bwd: dtypes %d -> %d", in_dtype, out_dtype);
        count_launch();
        return check_launch("snake_sample_bwd (channels-last)");
    }
    if (in_dtype == MMU_F32 && out_dtype == MMU_F32)
        snake_bwd_kernel<float, float><<<grid, nthr, 0, st>>>((const float *)feat, y, (const float *)dout, dfeat, dy, g);
    else if (in_dtype == MMU_F32 && out_dtype == MMU_BF16)
        snake_bwd_kernel<float, __nv_bfloat16><<<grid, nthr, 0, st>>>((const float *)feat, y, (const __nv_bfloat16 *)dout, dfeat, dy, g);
    else if (in_dtype == MMU_BF16 && out_dtype == MMU_BF16)
        snake_bwd_kernel<__nv_bfloat16, __nv_bfloat16><<<grid, nthr, 0, st>>>((const __nv_bfloat16 *)feat, y, (const __nv_bfloat16 *)dout, dfeat, dy, g);
    else if (in_dtype == MMU_BF16 && out_dtype == MMU_F32)
        snake_bwd_kernel<__nv_bfloat16, float><<<grid, nthr, 0, st>>>((const __nv_bfloat16 *)feat, y, (const float *)dout, dfeat, dy, g);
    else
        return set_error(MMU_ERR_UNSUPPORTED, "snake_sample_bwd: dtypes %d -> %d", in_dtype, out_dtype);
    count_launch();
    return check_launch("snake_sample_bwd");
}

// Deterministic backward: no workspace (every output element has exactly one writer); the query exists for a uniform interface.
extern "C" size_t mmu_snake_sample_bwd_det_workspace(int32_t B, int32_t C, int32_t H, int32_t W, int32_t K, int32_t channels_last) {
    (void)B, (void)C, (void)H, (void)W, (void)K, (void)channels_last;
    return 0;
}

extern "C" int mmu_snake_sample_bwd_det(const void *feat, const float *y, const void *dout, float *dfeat, float *dy, int32_t in_dtype,
                                        int32_t out_dtype, int32_t B, int32_t C, int32_t H, int32_t W, int32_t K, int32_t channels_last,
                                        void *ws, size_t ws_bytes, void *stream) {
    using namespace mmu;
    (void)ws, (void)ws_bytes;
    SnakeGeom g;
    dim3 grid;
    int nthr = 0;
    if (int rc = channels_last ? geom_nhwc(g, B, C, H, W, K, grid, nthr) : geom(g, B, C, H, W, K, grid, nthr)) return rc;
    if (!feat || !y || !dout || !dfeat) return set_error(MMU_ERR_INVALID, "snake_sample_bwd_det: null pointer");
    const bool f32in = in_dtype == MMU_F32, f32out = out_dtype == MMU_F32;
    if ((in_dtype != MMU_F32 && in_dtype != MMU_BF16) || (out_dtype != MMU_F32 && out_dtype != MMU_BF16))
        return set_error(MMU_ERR_UNSUPPORTED, "snake_sample_bwd: dtypes %d -> %d", in_dtype, out_dtype);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const unsigned rows = (unsigned)((int64_t)B * H * K);
    // d_feat by target column
    if (channels_last) {
        const int64_t per_b = (int64_t)W * (C / 4);
        if ((per_b + 255) / 256 > 0x7fffffffLL || B > 65535) return set_error(MMU_ERR_UNSUPPORTED, "snake_sample_bwd_det: problem too large");
        const dim3 dg((unsigned)((per_b + 255) / 256), (unsigned)B);
        if (f32out) snake_bwd_det_dfeat_kernel<float, true><<<dg, 256, 0, st>>>(y, (const float *)dout, dfeat, g);
        else snake_bwd_det_dfeat_kernel<__nv_bfloat16, true><<<dg, 256, 0, st>>>(y, (const __nv_bfloat16 *)dout, dfeat, g);
    } else {
        if ((int64_t)B * C > 65535) return set_error(MMU_ERR_UNSUPPORTED, "snake_sample_bwd_det: B * C > 65535");
        const int nt = W >= 128 ? 128 : ((W + 31) / 32) * 32;
        const dim3 dg((unsigned)((W + nt - 1) / nt), (unsigned)(B * C));
        if (f32out) snake_bwd_det_dfeat_kernel<float, false><<<dg, nt, 0, st>>>(y, (const float *)dout, dfeat, g);
        else snake_bwd_det_dfeat_kernel<__nv_bfloat16, false><<<dg, nt, 0, st>>>(y, (const __nv_bfloat16 *)dout, dfeat, g);
    }
    count_launch();
    if (int rc = check_launch("snake_sample_bwd_det (d_feat)")) return rc;
    if (dy == nullptr) return MMU_OK;
    // d_y by sample, all channels in one thread
    const int nt = channels_last ? 256 : nthr;
    const dim3 yg(rows, (unsigned)((W + nt - 1) / nt));
#define MMU_SNAKE_DY(TI_, TO_)                                                                                                         \
    (channels_last ? snake_bwd_det_dy_kernel<TI_, TO_, true><<<yg, nt, 0, st>>>((const TI_ *)feat, y, (const TO_ *)dout, dy, g)         \
                   : snake_bwd_det_dy_kernel<TI_, TO_, false><<<yg, nt, 0, st>>>((const TI_ *)feat, y, (const TO_ *)dout, dy, g))
    if (f32in && f32out) MMU_SNAKE_DY(float, float);
    else if (f32in) MMU_SNAKE_DY(float, __nv_bfloat16);
    else if (f32out) MMU_SNAKE_DY(__nv_bfloat16, float);
    else MMU_SNAKE_DY(__nv_bfloat16, __nv_bfloat16);
#undef MMU_SNAKE_DY
    count_launch();
    return check_launch("snake_sample_bwd_det (d_y)");
}
