// Prologue / epilogue kernels of a NARROW Mamba block (d_model = 3: MMConv's offset-refining Mamba, SURVEY.md section 8 row f3).
//
// The reference runs in_proj -> conv1d -> x_proj -> dt_proj -> scan -> out_proj as separate ops
// (requirements/mamba_simple.py:201-270, mamba_ssm/ops/selective_scan_interface.py:181-207, backward :256-277).  With d_model = 3,
// d_inner = 6, dt_rank = 1 those projections are 3..33-row matrix products: ~25 launches per block per direction whose cost is launch
// latency and skinny-GEMM inefficiency, 47 times per MM-UNet step.  Here everything between the token tensor and the scan - and
// between the scan and the block's output - is ONE kernel each way, one thread per token, weights in shared memory:
//   pre_fwd  : hidden (natural token order, addressed through the scan-order map) -> in_proj -> causal conv (w = 4) + SiLU -> x_proj
//              -> dt_proj;  writes u | delta | z | B | C in scan order, ready for mmu_selective_scan_fwd (which adds dt bias + softplus)
//   post_fwd : out_proj of the gated scan output, written back to natural token order through the map
//   post_bwd : dout (natural) -> d(out_z) (scan order);  d(out_proj.weight)
//   pre_bwd  : the scan's du | ddelta | dz, dB | dC -> d(hidden) (natural order) and every weight gradient of the prologue.
//              Per 256-token tile: (1) per token d(x_dbl), d(u) and d(conv pre-activation) (+3 halo tokens), (2) conv transposed,
//              in_proj transposed, (3) the x_proj / dt_proj / in_proj weight gradients as sums over the tile of products of two
//              entries of a per-token record kept in shared memory (one accumulator per thread, one atomic per accumulator and tile).
// MMConv epilogue (coord_mode): the block's output is consumed only as  y = gain * refined + rows + snake_offsets(dy) * extend_scope
// (src/UM_Net/MMUNet.py:156-188: gain = clamp(softplus(altho), 0.01), rows = the row index h, offsets = cumulative sums of dy away
// from the centre tap, dy = the block's own input).  post_fwd writes y (fp32) instead of the block output, post_bwd takes d(y) and
// accumulates d(altho), pre_bwd adds the offsets' gradient to d(hidden): ~35 element-wise launches per MMConv disappear.
// All arithmetic in fp32 from fp32 weights; scan-side activations in the I/O dtype IN_T, hidden / d(hidden) in HID_T.
#include "scan_tiles.cuh"

namespace mmu {
namespace {

constexpr int kNarT = 256;      // tokens per block, one thread each

template <int DM> struct Nar {
    static constexpr int DI = 2 * DM, N = 16, R = 1, XD = R + 2 * N, KW = 4;
    // weight block (floats), the same offsets in shared memory and in the gradient accumulator
    static constexpr int oWin = 0, oWc = oWin + 2 * DI * DM, oBc = oWc + DI * KW, oWx = oBc + DI, oWdt = oWx + XD * DI,
                         oWout = oWdt + DI * R, kNW = oWout + DM * DI;
    // rows of the scan-order workspace `pre` (batch, kPreRows, L) and of `gpre` (batch, 3*DI, L)
    static constexpr int rU = 0, rDl = DI, rZ = 2 * DI, rB = 3 * DI, kPreRows = 3 * DI + 2 * N;      // C follows B
    // per-token record of pre_bwd (floats): d(x_dbl) | u | ddelta | dt_in | d(xz) | hidden
    static constexpr int qX = 0, qU = XD, qDd = qU + DI, qDt = qDd + DI, qDxz = qDt + 1, qH = qDxz + 2 * DI, kRec = (qH + DM) | 1;
    static constexpr int kAcc = XD * DI + DI + 2 * DI * DM;      // x_proj, dt_proj, in_proj gradients
};

struct NarArgs {
    const float *in_w, *conv_w, *conv_b, *x_w, *dt_w, *out_w;
    const void *hidden, *out_z, *dout, *gpre;
    const float *dBC;
    void *pre, *out, *dout_y, *dhidden;
    float *dW;
    int64_t h_bs, h_cs, o_bs, o_cs, g_bs, g_cs, dh_bs, dh_cs;
    int B, L;
    OrdMap ord;
    // MMConv coordinate epilogue
    int coord_mode, map_w;
    float scope;
    const float *altho, *dcoords;
    float *coords;
    float *part;             // deterministic backward: per (batch, tile) slots of the weight-gradient sums (NarDet)
};

__device__ __forceinline__ float coord_gain(float altho, float *dgain_daltho = nullptr) {
    const float sp = altho > 20.f ? altho : log1pf(__expf(altho));        // F.softplus (threshold 20)
    if (dgain_daltho != nullptr) *dgain_daltho = sp > 0.01f ? sigmoid_f(altho) : 0.f;
    return fmaxf(sp, 0.01f);
}
// cumulative offsets away from the centre tap (MMUNet.py:156-174) and the transposed map for gradients
template <int DM> __device__ __forceinline__ void snake_offsets(const float (&dy)[DM], float (&off)[DM]) {
    constexpr int c = DM / 2;
    off[c] = 0.f;
#pragma unroll
    for (int k = c + 1; k < DM; ++k) off[k] = off[k - 1] + dy[k];
#pragma unroll
    for (int k = c - 1; k >= 0; --k) off[k] = off[k + 1] + dy[k];
}
template <int DM> __device__ __forceinline__ void snake_offsets_t(const float (&g)[DM], float (&d)[DM]) {
    constexpr int c = DM / 2;
    d[c] = 0.f;
    float acc = 0.f;
#pragma unroll
    for (int k = DM - 1; k > c; --k) acc += g[k], d[k] = acc;
    acc = 0.f;
#pragma unroll
    for (int k = 0; k < c; ++k) acc += g[k], d[k] = acc;
}

template <int DM> __device__ __forceinline__ void load_weights(const NarArgs &p, float *s_w) {
    using C = Nar<DM>;
    for (int i = threadIdx.x; i < C::kNW; i += kNarT) {
        float v;
        if (i < C::oWc) v = p.in_w[i];
        else if (i < C::oBc) v = p.conv_w[i - C::oWc];
        else if (i < C::oWx) v = p.conv_b != nullptr ? p.conv_b[i - C::oBc] : 0.f;
        else if (i < C::oWdt) v = p.x_w[i - C::oWx];
        else if (i < C::oWout) v = p.dt_w[i - C::oWdt];
        else v = p.out_w[i - C::oWout];
        s_w[i] = v;
    }
}

// hidden of the 4 conv taps of scan token l (tap k = scan token l-3+k; zeros before the sequence start)
template <typename HID_T, int DM>
__device__ __forceinline__ void load_taps_hidden(const NarArgs &p, int b, int l, float (&h)[4][DM]) {
    const HID_T *hp = reinterpret_cast<const HID_T *>(p.hidden) + (int64_t)b * p.h_bs;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int lt = l - 3 + k;
        const int m = lt >= 0 ? p.ord(lt) : 0;
#pragma unroll
        for (int c = 0; c < DM; ++c) h[k][c] = lt >= 0 ? Elem<HID_T>::to_f(hp[(int64_t)c * p.h_cs + m]) : 0.f;
    }
}

// conv pre-activation of the DI channels at scan token l and the in_proj x rows of its last tap (xl = in_proj x of token l itself)
template <int DM>
__device__ __forceinline__ void conv_pre(const float *s_w, const float (&h)[4][DM], float (&pre)[2 * DM], float (&xtap)[4][2 * DM]) {
    using C = Nar<DM>;
#pragma unroll
    for (int d = 0; d < C::DI; ++d) {
        float acc = s_w[C::oBc + d];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float x = 0.f;
#pragma unroll
            for (int c = 0; c < DM; ++c) x = fmaf(s_w[C::oWin + d * DM + c], h[k][c], x);
            xtap[k][d] = x;
            acc = fmaf(s_w[C::oWc + d * 4 + k], x, acc);
        }
        pre[d] = acc;
    }
}

template <typename IN_T, typename HID_T, int DM> __global__ void __launch_bounds__(kNarT) narrow_pre_fwd_kernel(const __grid_constant__ NarArgs p) {
    using C = Nar<DM>;
    __shared__ float s_w[C::kNW];
    load_weights<DM>(p, s_w);
    __syncthreads();
    const int b = blockIdx.y, l = blockIdx.x * kNarT + threadIdx.x;
    if (l >= p.L) return;
    float h[4][DM], pre[C::DI], xtap[4][C::DI];
    load_taps_hidden<HID_T, DM>(p, b, l, h);
    conv_pre<DM>(s_w, h, pre, xtap);
    IN_T *P = reinterpret_cast<IN_T *>(p.pre) + (int64_t)b * C::kPreRows * p.L + l;
    float u[C::DI];
#pragma unroll
    for (int d = 0; d < C::DI; ++d) {
        const IN_T ur = Elem<IN_T>::from_f(pre[d] * sigmoid_f(pre[d]));
        u[d] = Elem<IN_T>::to_f(ur);        // the projections see the value the scan reads
        P[(int64_t)(C::rU + d) * p.L] = ur;
        float z = 0.f;
#pragma unroll
        for (int c = 0; c < DM; ++c) z = fmaf(s_w[C::oWin + (C::DI + d) * DM + c], h[3][c], z);
        P[(int64_t)(C::rZ + d) * p.L] = Elem<IN_T>::from_f(z);
    }
    float dt = 0.f;
#pragma unroll
    for (int d = 0; d < C::DI; ++d) dt = fmaf(s_w[C::oWx + d], u[d], dt);
#pragma unroll
    for (int d = 0; d < C::DI; ++d) P[(int64_t)(C::rDl + d) * p.L] = Elem<IN_T>::from_f(s_w[C::oWdt + d] * dt);
#pragma unroll
    for (int r = 0; r < 2 * C::N; ++r) {
        float v = 0.f;
#pragma unroll
        for (int d = 0; d < C::DI; ++d) v = fmaf(s_w[C::oWx + (C::R + r) * C::DI + d], u[d], v);
        P[(int64_t)(C::rB + r) * p.L] = Elem<IN_T>::from_f(v);
    }
}

template <typename IN_T, typename HID_T, int DM> __global__ void __launch_bounds__(kNarT) narrow_post_fwd_kernel(const __grid_constant__ NarArgs p) {
    using C = Nar<DM>;
    __shared__ float s_wo[DM * C::DI];
    for (int i = threadIdx.x; i < DM * C::DI; i += kNarT) s_wo[i] = p.out_w[i];
    __syncthreads();
    const int b = blockIdx.y, l = blockIdx.x * kNarT + threadIdx.x;
    if (l >= p.L) return;
    const IN_T *oz = reinterpret_cast<const IN_T *>(p.out_z) + (int64_t)b * C::DI * p.L + l;
    float y[C::DI];
#pragma unroll
    for (int d = 0; d < C::DI; ++d) y[d] = Elem<IN_T>::to_f(oz[(int64_t)d * p.L]);
    const int m = p.ord(l);
    float v[DM];
#pragma unroll
    for (int e = 0; e < DM; ++e) {
        v[e] = 0.f;
#pragma unroll
        for (int d = 0; d < C::DI; ++d) v[e] = fmaf(s_wo[e * C::DI + d], y[d], v[e]);
    }
    if (p.coord_mode) {       // y coordinates of the K snake taps at pixel m = (h, w)
        const HID_T *hp = reinterpret_cast<const HID_T *>(p.hidden) + (int64_t)b * p.h_bs + m;
        float dyv[DM], off[DM];
#pragma unroll
        for (int c = 0; c < DM; ++c) dyv[c] = Elem<HID_T>::to_f(hp[(int64_t)c * p.h_cs]);
        snake_offsets<DM>(dyv, off);
        const float gain = coord_gain(*p.altho), row = (float)(m / p.map_w);
        float *cp = p.coords + (int64_t)b * DM * p.L + m;
#pragma unroll
        for (int e = 0; e < DM; ++e) cp[(int64_t)e * p.L] = fmaf(gain, v[e], fmaf(off[e], p.scope, row));
        return;
    }
    IN_T *op = reinterpret_cast<IN_T *>(p.out) + (int64_t)b * p.o_bs + m;
#pragma unroll
    for (int e = 0; e < DM; ++e) op[(int64_t)e * p.o_cs] = Elem<IN_T>::from_f(v[e]);
}

// sum of v[i] over the block -> one atomicAdd per i (DET: one plain store per i into the block's own slot)
template <int NV, bool DET> __device__ __forceinline__ void block_sum(float (&v)[NV], float *dst, float *s_red /* [kNarT/32][NV] */) {
#pragma unroll
    for (int i = 0; i < NV; ++i) {
        float x = v[i];
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) x += __shfl_xor_sync(0xffffffffu, x, s);
        if ((threadIdx.x & 31) == 0) s_red[(threadIdx.x >> 5) * NV + i] = x;
    }
    __syncthreads();
    if (threadIdx.x < NV) {
        float x = 0.f;
#pragma unroll
        for (int w = 0; w < kNarT / 32; ++w) x += s_red[w * NV + threadIdx.x];
        if constexpr (DET) dst[threadIdx.x] = x;
        else atomicAdd(dst + threadIdx.x, x);
    }
}

// Deterministic backward: the (batch, tile) work item's sums go to slot b * gridDim.x + tile of p.part - post_bwd: the out_proj | altho
// floats [oWout, kNW], pre_bwd: every float below oWout - and the ordered reduce adds the slots into dweights.
template <int DM> struct NarDet {
    static constexpr int kPost = DM * Nar<DM>::DI + 1, kPre = Nar<DM>::oWout;
};

template <typename IN_T, int DM, bool DET = false> __global__ void __launch_bounds__(kNarT) narrow_post_bwd_kernel(const __grid_constant__ NarArgs p) {
    using C = Nar<DM>;
    __shared__ float s_wo[DM * C::DI];
    __shared__ float s_red[(kNarT / 32) * (DM * C::DI + 1)];
    for (int i = threadIdx.x; i < DM * C::DI; i += kNarT) s_wo[i] = p.out_w[i];
    __syncthreads();
    const int b = blockIdx.y, l = blockIdx.x * kNarT + threadIdx.x;
    float dw[DM * C::DI + 1];       // out_proj weight gradient | d(altho) (coord_mode; the two are adjacent in the accumulator)
#pragma unroll
    for (int i = 0; i < DM * C::DI + 1; ++i) dw[i] = 0.f;
    float gain = 1.f, dgain_daltho = 0.f;
    if (p.coord_mode) gain = coord_gain(*p.altho, &dgain_daltho);
    if (l < p.L) {
        const int m = p.ord(l);
        const IN_T *oz = reinterpret_cast<const IN_T *>(p.out_z) + (int64_t)b * C::DI * p.L + l;
        IN_T *dy = reinterpret_cast<IN_T *>(p.dout_y) + (int64_t)b * C::DI * p.L + l;
        float g[DM], y[C::DI];
#pragma unroll
        for (int d = 0; d < C::DI; ++d) y[d] = Elem<IN_T>::to_f(oz[(int64_t)d * p.L]);
        if (p.coord_mode) {       // d(refined) = gain * d(coords);  d(gain) = sum d(coords) * refined
            const float *gc = p.dcoords + (int64_t)b * DM * p.L + m;
            float dgain = 0.f;
#pragma unroll
            for (int e = 0; e < DM; ++e) {
                const float gce = gc[(int64_t)e * p.L];
                float refined = 0.f;
#pragma unroll
                for (int d = 0; d < C::DI; ++d) refined = fmaf(s_wo[e * C::DI + d], y[d], refined);
                dgain = fmaf(gce, refined, dgain);
                g[e] = gain * gce;
            }
            dw[DM * C::DI] = dgain * dgain_daltho;
        } else {
            const IN_T *gp = reinterpret_cast<const IN_T *>(p.dout) + (int64_t)b * p.g_bs + m;
#pragma unroll
            for (int e = 0; e < DM; ++e) g[e] = Elem<IN_T>::to_f(gp[(int64_t)e * p.g_cs]);
        }
#pragma unroll
        for (int d = 0; d < C::DI; ++d) {
            float v = 0.f;
#pragma unroll
            for (int e = 0; e < DM; ++e) v = fmaf(s_wo[e * C::DI + d], g[e], v);
            dy[(int64_t)d * p.L] = Elem<IN_T>::from_f(v);
#pragma unroll
            for (int e = 0; e < DM; ++e) dw[e * C::DI + d] = g[e] * y[d];
        }
    }
    block_sum<DM * C::DI + 1, DET>(dw, DET ? p.part + ((int64_t)b * gridDim.x + blockIdx.x) * NarDet<DM>::kPost : p.dW + C::oWout,
                                   s_red);       // slot kNW = d(altho)
}

template <typename IN_T, typename HID_T, int DM, bool DET = false> __global__ void __launch_bounds__(kNarT) narrow_pre_bwd_kernel(const __grid_constant__ NarArgs p) {
    using C = Nar<DM>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float *s_w = reinterpret_cast<float *>(smem_raw);                 // [kNW]
    float *s_dpre = s_w + ((C::kNW + 3) & ~3);                        // [DI][kNarT + 3]
    float *s_red = s_dpre + C::DI * (kNarT + 3) + 1;                  // [kNarT/32][DI*5]
    float *s_rec = s_red + (kNarT / 32) * C::DI * 5;                  // [kNarT][kRec]
    load_weights<DM>(p, s_w);
    __syncthreads();
    const int b = blockIdx.y, t0 = blockIdx.x * kNarT, tid = threadIdx.x;
    const IN_T *P = reinterpret_cast<const IN_T *>(p.pre) + (int64_t)b * C::kPreRows * p.L;
    const IN_T *G = reinterpret_cast<const IN_T *>(p.gpre) + (int64_t)b * 3 * C::DI * p.L;
    const float *BC = p.dBC + (int64_t)b * 2 * C::N * p.L;
    float *rec = s_rec + tid * C::kRec;
    float cw[C::DI * 5];             // conv weight / bias gradient partials of this thread's own token
#pragma unroll
    for (int i = 0; i < C::DI * 5; ++i) cw[i] = 0.f;

    // (1) d(conv pre-activation) of token l; own = this thread's token (fills the record), otherwise a halo token of the next tile
    auto token = [&](int l, int slot, bool own) {
        float dpre[C::DI];
#pragma unroll
        for (int d = 0; d < C::DI; ++d) dpre[d] = 0.f;
        if (l < p.L) {
            float u[C::DI], dxd[C::XD], dd[C::DI];
#pragma unroll
            for (int d = 0; d < C::DI; ++d) {
                u[d] = Elem<IN_T>::to_f(P[(int64_t)(C::rU + d) * p.L + l]);
                dd[d] = Elem<IN_T>::to_f(G[(int64_t)(C::DI + d) * p.L + l]);
            }
            float dt_in = 0.f, ddt = 0.f;
#pragma unroll
            for (int d = 0; d < C::DI; ++d) {
                dt_in = fmaf(s_w[C::oWx + d], u[d], dt_in);
                ddt = fmaf(s_w[C::oWdt + d], dd[d], ddt);
            }
            dxd[0] = ddt;
#pragma unroll
            for (int r = 0; r < 2 * C::N; ++r) dxd[C::R + r] = BC[(int64_t)r * p.L + l];
            float h[4][DM], pre[C::DI], xtap[4][C::DI];
            load_taps_hidden<HID_T, DM>(p, b, l, h);
            conv_pre<DM>(s_w, h, pre, xtap);
#pragma unroll
            for (int d = 0; d < C::DI; ++d) {
                float du = Elem<IN_T>::to_f(G[(int64_t)d * p.L + l]);
#pragma unroll
                for (int r = 0; r < C::XD; ++r) du = fmaf(s_w[C::oWx + r * C::DI + d], dxd[r], du);
                const float s = sigmoid_f(pre[d]);
                dpre[d] = du * s * fmaf(pre[d], 1.f - s, 1.f);
            }
            if (own) {
#pragma unroll
                for (int r = 0; r < C::XD; ++r) rec[C::qX + r] = dxd[r];
#pragma unroll
                for (int d = 0; d < C::DI; ++d) {
                    rec[C::qU + d] = u[d];
                    rec[C::qDd + d] = dd[d];
                    rec[C::qDxz + C::DI + d] = Elem<IN_T>::to_f(G[(int64_t)(2 * C::DI + d) * p.L + l]);     // dz
#pragma unroll
                    for (int k = 0; k < 4; ++k) cw[d * 4 + k] = dpre[d] * xtap[k][d];
                    cw[C::DI * 4 + d] = dpre[d];
                }
                rec[C::qDt] = dt_in;
#pragma unroll
                for (int c = 0; c < DM; ++c) rec[C::qH + c] = h[3][c];
            }
        } else if (own) {
#pragma unroll
            for (int i = 0; i < C::kRec; ++i) rec[i] = 0.f;
        }
#pragma unroll
        for (int d = 0; d < C::DI; ++d) s_dpre[d * (kNarT + 3) + slot] = dpre[d];
    };
    token(t0 + tid, tid, true);
    if (tid < 3) token(t0 + kNarT + tid, kNarT + tid, false);
    __syncthreads();

    // (2) conv transposed: dx[d][l] = sum_k w[d][k] dpre[d][l + 3 - k];  in_proj transposed -> d(hidden)
    const int l = t0 + tid;
    if (l < p.L) {
        float dxz[2 * C::DI];
#pragma unroll
        for (int d = 0; d < C::DI; ++d) {
            float acc = 0.f;
#pragma unroll
            for (int k = 0; k < 4; ++k) acc = fmaf(s_w[C::oWc + d * 4 + k], s_dpre[d * (kNarT + 3) + tid + 3 - k], acc);
            dxz[d] = acc;
            rec[C::qDxz + d] = acc;
            dxz[C::DI + d] = rec[C::qDxz + C::DI + d];
        }
        const int m = p.ord(l);
        float doff[DM];
#pragma unroll
        for (int c = 0; c < DM; ++c) doff[c] = 0.f;
        if (p.coord_mode) {       // the snake offsets' path from d(coords) straight back to dy = hidden
            const float *gc = p.dcoords + (int64_t)b * DM * p.L + m;
            float g[DM];
#pragma unroll
            for (int c = 0; c < DM; ++c) g[c] = gc[(int64_t)c * p.L] * p.scope;
            snake_offsets_t<DM>(g, doff);
        }
        HID_T *dh = reinterpret_cast<HID_T *>(p.dhidden) + (int64_t)b * p.dh_bs + m;
#pragma unroll
        for (int c = 0; c < DM; ++c) {
            float v = doff[c];
#pragma unroll
            for (int j = 0; j < 2 * C::DI; ++j) v = fmaf(s_w[C::oWin + j * DM + c], dxz[j], v);
            dh[(int64_t)c * p.dh_cs] = Elem<HID_T>::from_f(v);
        }
    }
    // conv weight / bias gradients: block sum of the per-token partials
    float *dW = DET ? p.part + ((int64_t)b * gridDim.x + blockIdx.x) * NarDet<DM>::kPre : p.dW;
    block_sum<C::DI * 5, DET>(cw, dW + C::oWc, s_red);       // conv_w (DI*4) and conv_b (DI) are adjacent in the weight block
    __syncthreads();

    // (3) x_proj / dt_proj / in_proj weight gradients: accumulator j = sum over the tile of rec[a_j] * rec[b_j]
    const int ntok = min(kNarT, p.L - t0);
    for (int j = tid; j < C::kAcc; j += kNarT) {
        int a, bb, dst;
        if (j < C::XD * C::DI) {
            a = C::qX + j / C::DI, bb = C::qU + j % C::DI, dst = C::oWx + j;
        } else if (j < C::XD * C::DI + C::DI) {
            a = C::qDd + (j - C::XD * C::DI), bb = C::qDt, dst = C::oWdt + (j - C::XD * C::DI);
        } else {
            const int q = j - C::XD * C::DI - C::DI;
            a = C::qDxz + q / DM, bb = C::qH + q % DM, dst = C::oWin + q;
        }
        float acc0 = 0.f, acc1 = 0.f;
        int t = 0;
        for (; t + 1 < ntok; t += 2) {
            acc0 = fmaf(s_rec[t * C::kRec + a], s_rec[t * C::kRec + bb], acc0);
            acc1 = fmaf(s_rec[(t + 1) * C::kRec + a], s_rec[(t + 1) * C::kRec + bb], acc1);
        }
        if (t < ntok) acc0 = fmaf(s_rec[t * C::kRec + a], s_rec[t * C::kRec + bb], acc0);
        if constexpr (DET) dW[dst] = acc0 + acc1;
        else atomicAdd(p.dW + dst, acc0 + acc1);
    }
}

template <int DM> constexpr size_t pre_bwd_smem() {
    using C = Nar<DM>;
    return sizeof(float) * (((C::kNW + 3) & ~3) + C::DI * (kNarT + 3) + 1 + (kNarT / 32) * C::DI * 5 + kNarT * C::kRec);
}

enum NarKernel { kPreFwd, kPostFwd, kPostBwd, kPreBwd };

template <typename IN_T, typename HID_T> int launch_narrow(const NarArgs &a, NarKernel which, cudaStream_t st) {
    constexpr int DM = 3;
    dim3 grid((a.L + kNarT - 1) / kNarT, a.B);
    if (a.part != nullptr) {
        const int64_t items = (int64_t)a.B * grid.x;
        if (which == kPostBwd) {
            narrow_post_bwd_kernel<IN_T, DM, true><<<grid, kNarT, 0, st>>>(a);
        } else {
            auto k = narrow_pre_bwd_kernel<IN_T, HID_T, DM, true>;
            constexpr size_t smem = pre_bwd_smem<DM>();
            cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            k<<<grid, kNarT, smem, st>>>(a);
        }
        count_launch();
        if (int rc = check_launch("mamba_narrow(deterministic)")) return rc;
        const int nv = which == kPostBwd ? NarDet<DM>::kPost : NarDet<DM>::kPre;
        return det_reduce(DetSum{a.part, items, nv, 1, 1, nv, 0, 0, a.dW + (which == kPostBwd ? Nar<DM>::oWout : 0), 0, 0, 1}, st);
    }
    switch (which) {
        case kPreFwd: narrow_pre_fwd_kernel<IN_T, HID_T, DM><<<grid, kNarT, 0, st>>>(a); break;
        case kPostFwd: narrow_post_fwd_kernel<IN_T, HID_T, DM><<<grid, kNarT, 0, st>>>(a); break;
        case kPostBwd: narrow_post_bwd_kernel<IN_T, DM><<<grid, kNarT, 0, st>>>(a); break;
        case kPreBwd: {
            auto k = narrow_pre_bwd_kernel<IN_T, HID_T, DM>;
            constexpr size_t smem = pre_bwd_smem<DM>();
            cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            k<<<grid, kNarT, smem, st>>>(a);
            break;
        }
    }
    count_launch();
    return check_launch("mamba_narrow");
}

int narrow_entry(const mmu_narrow_params *p, NarKernel which, float *part, void *stream) {
    if (p == nullptr) return set_error(MMU_ERR_INVALID, "mamba_narrow: null params");
    if (!mmu_mamba_narrow_supported(p->d_model, p->d_inner, p->d_state, p->dt_rank, p->d_conv, p->dtype))
        return set_error(MMU_ERR_UNSUPPORTED, "mamba_narrow: d_model %d d_inner %d d_state %d dt_rank %d d_conv %d dtype %d is not a narrow block",
                         p->d_model, p->d_inner, p->d_state, p->dt_rank, p->d_conv, p->dtype);
    if (p->batch <= 0 || p->seqlen <= 0 || p->batch > 65535) return set_error(MMU_ERR_INVALID, "mamba_narrow: bad shape");
    NarArgs a{};
    a.in_w = p->in_proj_w, a.conv_w = p->conv_w, a.conv_b = p->conv_b, a.x_w = p->x_proj_w, a.dt_w = p->dt_proj_w, a.out_w = p->out_proj_w;
    a.hidden = p->hidden, a.out_z = p->out_z, a.dout = p->dout, a.gpre = p->gpre, a.dBC = p->dBC;
    a.pre = p->pre, a.out = p->out, a.dout_y = p->dout_y, a.dhidden = p->dhidden, a.dW = p->dweights;
    a.h_bs = p->hidden_bs, a.h_cs = p->hidden_cs, a.o_bs = p->out_bs, a.o_cs = p->out_cs;
    a.g_bs = p->dout_bs, a.g_cs = p->dout_cs, a.dh_bs = p->dhidden_bs, a.dh_cs = p->dhidden_cs;
    a.B = p->batch, a.L = p->seqlen;
    a.part = part;
    if (!make_ordmap(a.ord, p->order, p->order_h, p->order_w, p->order_ns, p->seqlen) || p->order == MMU_ORDER_FLIP)
        return set_error(MMU_ERR_INVALID, "mamba_narrow: bad scan order %d (H=%d W=%d nslices=%d, L=%d)", p->order, p->order_h, p->order_w,
                         p->order_ns, p->seqlen);
    a.coord_mode = p->coord_mode, a.map_w = p->map_w, a.scope = p->extend_scope, a.altho = p->altho, a.dcoords = p->dcoords, a.coords = p->coords;
    const bool cm = p->coord_mode != 0;
    if (cm && (p->map_h <= 0 || p->map_w <= 0 || (int64_t)p->map_h * p->map_w != p->seqlen || p->altho == nullptr))
        return set_error(MMU_ERR_INVALID, "mamba_narrow: coord_mode needs map_h * map_w == seqlen and altho");
    bool ok = true;
    switch (which) {
        case kPreFwd: ok = a.in_w && a.conv_w && a.x_w && a.dt_w && a.hidden && a.pre; break;
        case kPostFwd: ok = a.out_w && a.out_z && (cm ? (a.coords && a.hidden) : a.out != nullptr); break;
        case kPostBwd: ok = a.out_w && a.out_z && (cm ? a.dcoords != nullptr : a.dout != nullptr) && a.dout_y && a.dW; break;
        case kPreBwd:
            ok = a.in_w && a.conv_w && a.x_w && a.dt_w && a.hidden && a.pre && a.gpre && a.dBC && a.dhidden && a.dW && (!cm || a.dcoords);
            break;
    }
    if (!ok) return set_error(MMU_ERR_INVALID, "mamba_narrow: null tensor pointer");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (p->dtype == MMU_F32 && p->hidden_dtype == MMU_F32) return launch_narrow<float, float>(a, which, st);
    if (p->dtype == MMU_BF16 && p->hidden_dtype == MMU_BF16) return launch_narrow<__nv_bfloat16, __nv_bfloat16>(a, which, st);
    if (p->dtype == MMU_BF16 && p->hidden_dtype == MMU_F32) return launch_narrow<__nv_bfloat16, float>(a, which, st);
    return set_error(MMU_ERR_UNSUPPORTED, "mamba_narrow: dtype %d with hidden dtype %d", p->dtype, p->hidden_dtype);
}
}  // namespace
}  // namespace mmu

extern "C" int32_t mmu_mamba_narrow_supported(int32_t d_model, int32_t d_inner, int32_t d_state, int32_t dt_rank, int32_t d_conv, int32_t dtype) {
    return d_model == 3 && d_inner == 6 && d_state == 16 && dt_rank == 1 && d_conv == 4 && (dtype == MMU_F32 || dtype == MMU_BF16);
}
extern "C" int32_t mmu_mamba_narrow_rows(int32_t d_inner, int32_t d_state) { return 3 * d_inner + 2 * d_state; }
extern "C" int32_t mmu_mamba_narrow_weight_floats(int32_t d_model, int32_t d_inner, int32_t d_state, int32_t dt_rank, int32_t d_conv) {
    return 2 * d_inner * d_model + d_inner * d_conv + d_inner + (dt_rank + 2 * d_state) * d_inner + d_inner * dt_rank + d_model * d_inner + 1;
}
extern "C" int mmu_mamba_narrow_pre_fwd(const mmu_narrow_params *p, void *stream) { return mmu::narrow_entry(p, mmu::kPreFwd, nullptr, stream); }
extern "C" int mmu_mamba_narrow_post_fwd(const mmu_narrow_params *p, void *stream) { return mmu::narrow_entry(p, mmu::kPostFwd, nullptr, stream); }
extern "C" int mmu_mamba_narrow_post_bwd(const mmu_narrow_params *p, void *stream) { return mmu::narrow_entry(p, mmu::kPostBwd, nullptr, stream); }
extern "C" int mmu_mamba_narrow_pre_bwd(const mmu_narrow_params *p, void *stream) { return mmu::narrow_entry(p, mmu::kPreBwd, nullptr, stream); }

namespace mmu {
namespace {
size_t narrow_det_bytes(int32_t batch, int32_t seqlen, int per_tile) {
    if (batch <= 0 || seqlen <= 0) return 0;
    DetWs w{nullptr};
    w.take((size_t)batch * ((seqlen + kNarT - 1) / kNarT) * per_tile);
    return w.used;
}
int narrow_det(const mmu_narrow_params *p, NarKernel which, void *ws, size_t ws_bytes, void *stream) {
    const char *what = which == kPostBwd ? "mamba_narrow_post_bwd_det" : "mamba_narrow_pre_bwd_det";
    if (p == nullptr) return set_error(MMU_ERR_INVALID, "%s: null params", what);
    const size_t need = which == kPostBwd ? mmu_mamba_narrow_post_bwd_det_workspace(p->batch, p->seqlen)
                                          : mmu_mamba_narrow_pre_bwd_det_workspace(p->batch, p->seqlen);
    if (need == 0) return set_error(MMU_ERR_INVALID, "%s: bad shape", what);
    if (int rc = det_ws_check(ws, ws_bytes, need, what)) return rc;
    return narrow_entry(p, which, static_cast<float *>(ws), stream);
}
}  // namespace
}  // namespace mmu

extern "C" size_t mmu_mamba_narrow_post_bwd_det_workspace(int32_t batch, int32_t seqlen) {
    return mmu::narrow_det_bytes(batch, seqlen, mmu::NarDet<3>::kPost);
}
extern "C" size_t mmu_mamba_narrow_pre_bwd_det_workspace(int32_t batch, int32_t seqlen) {
    return mmu::narrow_det_bytes(batch, seqlen, mmu::NarDet<3>::kPre);
}
extern "C" int mmu_mamba_narrow_post_bwd_det(const mmu_narrow_params *p, void *ws, size_t ws_bytes, void *stream) {
    return mmu::narrow_det(p, mmu::kPostBwd, ws, ws_bytes, stream);
}
extern "C" int mmu_mamba_narrow_pre_bwd_det(const mmu_narrow_params *p, void *ws, size_t ws_bytes, void *stream) {
    return mmu::narrow_det(p, mmu::kPreBwd, ws, ws_bytes, stream);
}
