// Depthwise causal conv1d (width 2..4) forward / backward for sm_100a.
//
// Replaces causal_conv1d_fwd_kernel / causal_conv1d_bwd_kernel
// (requirements/Mamba/causal-conv1d/csrc/causal_conv1d_fwd.cu:39-130, causal_conv1d_bwd.cu:46-240).
// The reference walks one (batch, channel) row per CTA, chunk after chunk; a conv has no long-range dependency, so
// here the grid is (token-blocks, channel, batch): MM-UNet's D=6 / L=65536 rows spread over all SMs.
// Each thread owns VT consecutive tokens - 8 for fp32, 16 for the 2-byte types, i.e. 32 bytes per tensor in flight either way -
// plus a 3-token halo that hits L1.
//   fwd : out[l]  = act(bias + sum_k w[k] x[l-(W-1-k)])
//   bwd : dpre[l] = dout[l] * silu'(pre[l]) (pre recomputed, causal_conv1d_bwd.cu:153-164)
//         dx[l]   = sum_k w[k] dpre[l+(W-1-k)]        dw[k] = sum_{b,l} x[l-(W-1-k)] dpre[l]       db = sum dpre
// Widths < 4 are handled as width 4 with zero leading taps.
#include "scan_tiles.cuh"

namespace mmu {

struct ConvArgs {
    const void *x, *dout;
    const float *w, *bias;
    void *out, *dx;
    float *dw, *db;
    int64_t x_bs, x_ds, o_bs, o_ds, w_ds, w_ws, g_bs, g_ds, dx_bs, dx_ds;
    int B, D, L, W;
    int silu, reverse;
    unsigned vec_mask;   // bit0 x, bit1 out/dx, bit2 dout
    OrdMap ord;          // fused scan order: x / dx live at ord(l), out / dout at l
    float *part;         // deterministic backward: [b][token block][d][5] partials (4 taps, width-padded | bias)
};

constexpr int kConvNT = 128;
template <typename IN_T> struct ConvVT { static constexpr int value = sizeof(IN_T) == 4 ? 8 : 16; };

// logical token t lives at memory position t (forward) or L-1-t (reverse)
__device__ __forceinline__ int mpos(int t, int L, bool rev) { return rev ? L - 1 - t : t; }

template <typename IN_T, int VT>
__device__ __forceinline__ void loadv(const IN_T *rp, int t, int L, bool vec, bool rev, float *v) {
    if (vec && t + VT <= L) {
#pragma unroll
        for (int h = 0; h < VT / 4; ++h) {
            const Quad<IN_T> q = *reinterpret_cast<const Quad<IN_T> *>(rp + (rev ? L - 4 - (t + 4 * h) : t + 4 * h));
#pragma unroll
            for (int k = 0; k < 4; ++k) v[4 * h + k] = Elem<IN_T>::to_f(q.v[rev ? 3 - k : k]);
        }
    } else {
#pragma unroll
        for (int k = 0; k < VT; ++k) v[k] = (t + k < L) ? Elem<IN_T>::to_f(rp[mpos(t + k, L, rev)]) : 0.f;
    }
}

// x addressed through the scan-order map (element-wise: the map scatters consecutive tokens)
template <typename IN_T, int N> __device__ __forceinline__ void load_ord(const IN_T *rp, int t, int L, const OrdMap &ord, float *v) {
#pragma unroll
    for (int k = 0; k < N; ++k) v[k] = (t + k >= 0 && t + k < L) ? Elem<IN_T>::to_f(rp[ord(t + k)]) : 0.f;
}

// NSLICES through shared memory (the nslices_tiled_kernel idea, scan_order.cu): a CTA's TB = 128*VT consecutive LOGICAL tokens
// are, in memory, ns runs of RL = TB/ns consecutive elements (run s starts at s*Ls + T0/ns).  The runs are moved with coalesced
// accesses and the threads pick their tokens out of the tile: element-wise global gathers would touch one sector per token
// (measured: 551 vs 132 us for the RCG stage at L = 65 536, ns = 64).  Tile layout [s][RL + pad], pad keeps a thread's walk over
// consecutive s (stride RL + pad) off a single bank.
template <typename IN_T> struct OrdTile {
    static constexpr int VT = sizeof(IN_T) == 4 ? 8 : 16, TB = 128 * VT;
    static constexpr int kPad = sizeof(IN_T) == 4 ? 1 : 2;
    static constexpr int kElems = TB + 128 * kPad;        // ns <= 128 runs
    static __device__ __forceinline__ int at(int lt, int sh, int RL) {      // logical offset inside the block -> tile index (ns = 1 << sh)
        const int jj = lt >> sh, sl = lt - (jj << sh);
        return sl * (RL + kPad) + jj;
    }
};
// usable when the block's tokens split into whole runs (ns a power of two: shifts instead of divisions)
__device__ __forceinline__ bool ord_tiled(const OrdMap &o, int TB) {
    return o.kind == MMU_ORDER_NSLICES && o.ns_shift >= 0 && o.ns <= 128 && TB % o.ns == 0 && o.L % TB == 0;
}

template <typename OUT_T, int VT>
__device__ __forceinline__ void storev(OUT_T *rp, int t, int L, bool vec, bool rev, const float *v) {
    if (vec && t + VT <= L) {
#pragma unroll
        for (int h = 0; h < VT / 4; ++h) {
            Quad<OUT_T> q;
#pragma unroll
            for (int k = 0; k < 4; ++k) q.v[rev ? 3 - k : k] = Elem<OUT_T>::from_f(v[4 * h + k]);
            *reinterpret_cast<Quad<OUT_T> *>(rp + (rev ? L - 4 - (t + 4 * h) : t + 4 * h)) = q;
        }
    } else {
#pragma unroll
        for (int k = 0; k < VT; ++k)
            if (t + k < L) rp[mpos(t + k, L, rev)] = Elem<OUT_T>::from_f(v[k]);
    }
}

__device__ __forceinline__ void load_taps(const ConvArgs &p, int d, float w4[4], float &bias) {
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int kk = k - (4 - p.W);
        w4[k] = kk >= 0 ? p.w[(int64_t)d * p.w_ds + (int64_t)kk * p.w_ws] : 0.f;
    }
    bias = p.bias != nullptr ? p.bias[d] : 0.f;
}

// ORD = false: the plain / reversed path only (no tile, no index map in the instruction stream)
template <typename IN_T, bool ORD> __global__ void __launch_bounds__(kConvNT) conv1d_fwd_kernel(const __grid_constant__ ConvArgs p) {
    constexpr int kConvVT = ConvVT<IN_T>::value;
    const int d = blockIdx.y, b = blockIdx.z;
    const int t = (blockIdx.x * kConvNT + threadIdx.x) * kConvVT;
    const IN_T *xr = reinterpret_cast<const IN_T *>(p.x) + (int64_t)b * p.x_bs + (int64_t)d * p.x_ds;
    float xv[kConvVT + 3];
    __shared__ IN_T s_x[ORD ? OrdTile<IN_T>::kElems : 1];
    __shared__ float s_halo[3];
    const bool tiled = ORD && ord_tiled(p.ord, OrdTile<IN_T>::TB);
    if (tiled) {       // block-uniform
        constexpr int TB = OrdTile<IN_T>::TB;
        const int sh = p.ord.ns_shift, RL = TB >> sh, rsh = 31 - __clz(RL), T0 = blockIdx.x * TB, j0 = T0 >> sh;
        for (int e = threadIdx.x; e < TB; e += kConvNT) {
            const int sl = e >> rsh, jj = e - (sl << rsh);
            s_x[sl * (RL + OrdTile<IN_T>::kPad) + jj] = xr[(int64_t)sl * p.ord.Ls + j0 + jj];
        }
        if (threadIdx.x < 3) s_halo[threadIdx.x] = T0 - 3 + (int)threadIdx.x >= 0 ? Elem<IN_T>::to_f(xr[p.ord(T0 - 3 + (int)threadIdx.x)]) : 0.f;
        __syncthreads();
#pragma unroll
        for (int k = 0; k < kConvVT + 3; ++k) {
            const int lt = (int)threadIdx.x * kConvVT + k - 3;
            xv[k] = lt >= 0 ? Elem<IN_T>::to_f(s_x[OrdTile<IN_T>::at(lt, sh, RL)]) : s_halo[lt + 3];
        }
    }
    if (t >= p.L) return;
    float w4[4], bias;
    load_taps(p, d, w4, bias);
    const bool rev = p.reverse != 0;
    if (tiled) {
    } else if (ORD && p.ord.kind != MMU_ORDER_ROWMAJOR) {
        load_ord<IN_T, kConvVT + 3>(xr, t - 3, p.L, p.ord, xv);
    } else {
#pragma unroll
        for (int k = 0; k < 3; ++k) xv[k] = (t - 3 + k >= 0) ? Elem<IN_T>::to_f(xr[mpos(t - 3 + k, p.L, rev)]) : 0.f;
        loadv<IN_T, kConvVT>(xr, t, p.L, p.vec_mask & 1u, rev, xv + 3);
    }
    float o[kConvVT];
#pragma unroll
    for (int i = 0; i < kConvVT; ++i) {
        float acc = bias;
#pragma unroll
        for (int k = 0; k < 4; ++k) acc = fmaf(w4[k], xv[i + k], acc);
        o[i] = p.silu ? acc * sigmoid_f(acc) : acc;
    }
    storev<IN_T, kConvVT>(reinterpret_cast<IN_T *>(p.out) + (int64_t)b * p.o_bs + (int64_t)d * p.o_ds, t, p.L, p.vec_mask & 2u,
                 rev, o);
}

// DET: the block's dw / db sums go to its own slot of p.part instead of atomics (the ordered reduce in det_reduce.cu adds them)
template <typename IN_T, bool ORD, bool DET = false> __global__ void __launch_bounds__(kConvNT) conv1d_bwd_kernel(const __grid_constant__ ConvArgs p) {
    constexpr int kConvVT = ConvVT<IN_T>::value;
    const int d = blockIdx.y, b = blockIdx.z;
    const int t = (blockIdx.x * kConvNT + threadIdx.x) * kConvVT;
    float w4[4], bias;
    load_taps(p, d, w4, bias);
    float part[5] = {0.f, 0.f, 0.f, 0.f, 0.f};   // dw4[0..3], dbias
    const bool rev = p.reverse != 0;
    __shared__ IN_T s_x[ORD ? OrdTile<IN_T>::kElems : 1];
    __shared__ IN_T s_dx[ORD ? OrdTile<IN_T>::kElems : 1];
    __shared__ float s_halo[6];
    const bool tiled = ORD && ord_tiled(p.ord, OrdTile<IN_T>::TB);
    if (tiled) {       // block-uniform: x of logical tokens [T0 - 3, T0 + TB + 3)
        constexpr int TB = OrdTile<IN_T>::TB;
        const IN_T *xr = reinterpret_cast<const IN_T *>(p.x) + (int64_t)b * p.x_bs + (int64_t)d * p.x_ds;
        const int sh = p.ord.ns_shift, RL = TB >> sh, rsh = 31 - __clz(RL), T0 = blockIdx.x * TB, j0 = T0 >> sh;
        for (int e = threadIdx.x; e < TB; e += kConvNT) {
            const int sl = e >> rsh, jj = e - (sl << rsh);
            s_x[sl * (RL + OrdTile<IN_T>::kPad) + jj] = xr[(int64_t)sl * p.ord.Ls + j0 + jj];
        }
        if (threadIdx.x < 6) {
            const int lt = threadIdx.x < 3 ? T0 - 3 + (int)threadIdx.x : T0 + TB + (int)threadIdx.x - 3;
            s_halo[threadIdx.x] = (lt >= 0 && lt < p.L) ? Elem<IN_T>::to_f(xr[p.ord(lt)]) : 0.f;
        }
        __syncthreads();
    }
    if (t < p.L) {
        const IN_T *xr = reinterpret_cast<const IN_T *>(p.x) + (int64_t)b * p.x_bs + (int64_t)d * p.x_ds;
        const IN_T *gr = reinterpret_cast<const IN_T *>(p.dout) + (int64_t)b * p.g_bs + (int64_t)d * p.g_ds;
        float xv[kConvVT + 6], gv[kConvVT + 3];   // x[t-3 .. t+10], dout[t .. t+10]
        const bool ordered = ORD && p.ord.kind != MMU_ORDER_ROWMAJOR;
        if (tiled) {
#pragma unroll
            for (int k = 0; k < kConvVT + 6; ++k) {
                const int lt = (int)threadIdx.x * kConvVT + k - 3;
                xv[k] = lt < 0 ? s_halo[lt + 3] : (lt < OrdTile<IN_T>::TB ? Elem<IN_T>::to_f(s_x[OrdTile<IN_T>::at(lt, p.ord.ns_shift, OrdTile<IN_T>::TB >> p.ord.ns_shift)])
                                                                           : s_halo[3 + lt - OrdTile<IN_T>::TB]);
            }
        } else if (ordered) {
            load_ord<IN_T, kConvVT + 6>(xr, t - 3, p.L, p.ord, xv);
        } else {
#pragma unroll
            for (int k = 0; k < 3; ++k) xv[k] = (t - 3 + k >= 0) ? Elem<IN_T>::to_f(xr[mpos(t - 3 + k, p.L, rev)]) : 0.f;
            loadv<IN_T, kConvVT>(xr, t, p.L, p.vec_mask & 1u, rev, xv + 3);
        }
        loadv<IN_T, kConvVT>(gr, t, p.L, p.vec_mask & 4u, rev, gv);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const int tt = t + kConvVT + k;
            if (!ordered) xv[3 + kConvVT + k] = tt < p.L ? Elem<IN_T>::to_f(xr[mpos(tt, p.L, rev)]) : 0.f;
            gv[kConvVT + k] = tt < p.L ? Elem<IN_T>::to_f(gr[mpos(tt, p.L, rev)]) : 0.f;
        }
        float dpre[kConvVT + 3];
#pragma unroll
        for (int i = 0; i < kConvVT + 3; ++i) {
            float g = gv[i];
            if (p.silu) {
                float pre = bias;
#pragma unroll
                for (int k = 0; k < 4; ++k) pre = fmaf(w4[k], xv[i + k], pre);
                const float s = sigmoid_f(pre);
                g *= s * fmaf(pre, 1.f - s, 1.f);
            }
            dpre[i] = g;   // zero beyond L because dout is zero there
        }
        float dxv[kConvVT];
#pragma unroll
        for (int i = 0; i < kConvVT; ++i) {
            float acc = 0.f;
#pragma unroll
            for (int k = 0; k < 4; ++k) acc = fmaf(w4[k], dpre[i + 3 - k], acc);
            dxv[i] = acc;
            part[4] += dpre[i];
#pragma unroll
            for (int k = 0; k < 4; ++k) part[k] = fmaf(xv[i + k], dpre[i], part[k]);
        }
        IN_T *dxr = reinterpret_cast<IN_T *>(p.dx) + (int64_t)b * p.dx_bs + (int64_t)d * p.dx_ds;
        if (tiled) {
#pragma unroll
            for (int k = 0; k < kConvVT; ++k)
                s_dx[OrdTile<IN_T>::at((int)threadIdx.x * kConvVT + k, p.ord.ns_shift, OrdTile<IN_T>::TB >> p.ord.ns_shift)] = Elem<IN_T>::from_f(dxv[k]);
        } else if (ordered) {
#pragma unroll
            for (int k = 0; k < kConvVT; ++k)
                if (t + k < p.L) dxr[p.ord(t + k)] = Elem<IN_T>::from_f(dxv[k]);
        } else {
            storev<IN_T, kConvVT>(dxr, t, p.L, p.vec_mask & 2u, rev, dxv);
        }
    }
    if (tiled) {       // the block's dx runs, coalesced
        constexpr int TB = OrdTile<IN_T>::TB;
        __syncthreads();
        IN_T *dxr = reinterpret_cast<IN_T *>(p.dx) + (int64_t)b * p.dx_bs + (int64_t)d * p.dx_ds;
        const int sh = p.ord.ns_shift, RL = TB >> sh, rsh = 31 - __clz(RL), j0 = (blockIdx.x * TB) >> sh;
        for (int e = threadIdx.x; e < TB; e += kConvNT) {
            const int sl = e >> rsh, jj = e - (sl << rsh);
            dxr[(int64_t)sl * p.ord.Ls + j0 + jj] = s_dx[sl * (RL + OrdTile<IN_T>::kPad) + jj];
        }
    }
    // block reduce -> one atomic per (channel, tap) per CTA
    __shared__ float red[kConvNT / 32][5];
#pragma unroll
    for (int k = 0; k < 5; ++k) {
        float v = part[k];
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][k] = v;
    }
    __syncthreads();
    if (threadIdx.x < 5) {
        float v = 0.f;
#pragma unroll
        for (int wdx = 0; wdx < kConvNT / 32; ++wdx) v += red[wdx][threadIdx.x];
        if constexpr (DET) {
            p.part[(((int64_t)b * gridDim.x + blockIdx.x) * p.D + d) * 5 + threadIdx.x] = v;
        } else if (threadIdx.x == 4) {
            if (p.db != nullptr) atomicAdd(p.db + d, v);
        } else {
            const int kk = (int)threadIdx.x - (4 - p.W);
            if (kk >= 0) atomicAdd(p.dw + (int64_t)d * p.W + kk, v);
        }
    }
}

namespace {
template <typename IN_T> constexpr int conv_block_tokens() { return kConvNT * ConvVT<IN_T>::value; }

// deterministic backward: the partial slots, [b][token block][d][5]
size_t conv_det_floats(int B, int D, int L, int dtype) {
    const int per_block = dtype == MMU_F32 ? conv_block_tokens<float>() : conv_block_tokens<__nv_bfloat16>();
    return (size_t)B * ((L + per_block - 1) / per_block) * D * 5;
}

template <typename IN_T> int run_conv(const mmu_conv_params *p, bool bwd, float *part, cudaStream_t st) {
    ConvArgs a{};
    a.part = part;
    a.x = p->x, a.dout = p->dout, a.w = p->weight, a.bias = p->bias, a.out = p->out, a.dx = p->dx;
    a.dw = p->dweight, a.db = p->dbias;
    a.x_bs = p->x_bs, a.x_ds = p->x_ds, a.o_bs = p->out_bs, a.o_ds = p->out_ds, a.w_ds = p->w_ds, a.w_ws = p->w_ws;
    a.g_bs = p->dout_bs, a.g_ds = p->dout_ds, a.dx_bs = p->dx_bs, a.dx_ds = p->dx_ds;
    a.B = p->batch, a.D = p->dim, a.L = p->seqlen, a.W = p->width, a.silu = p->silu, a.reverse = p->reverse;
    if (!make_ordmap(a.ord, p->order, p->order_h, p->order_w, p->order_ns, p->seqlen) || (p->order == MMU_ORDER_FLIP) ||
        (p->order != MMU_ORDER_ROWMAJOR && p->reverse))
        return set_error(MMU_ERR_INVALID, "causal_conv1d: bad scan order %d (H=%d W=%d nslices=%d, L=%d, reverse=%d)", p->order, p->order_h,
                         p->order_w, p->order_ns, p->seqlen, p->reverse);
    const int L = p->seqlen;
    const bool rv = p->reverse != 0;
    a.vec_mask = quad_ok<IN_T>(p->x, p->x_bs, p->x_ds, L, rv) ? 1u : 0u;
    if (!bwd) {
        a.vec_mask |= quad_ok<IN_T>(p->out, p->out_bs, p->out_ds, L, rv) ? 2u : 0u;
    } else {
        a.vec_mask |= quad_ok<IN_T>(p->dx, p->dx_bs, p->dx_ds, L, rv) ? 2u : 0u;
        a.vec_mask |= quad_ok<IN_T>(p->dout, p->dout_bs, p->dout_ds, L, rv) ? 4u : 0u;
    }
    const int per_block = kConvNT * ConvVT<IN_T>::value;
    dim3 grid((L + per_block - 1) / per_block, p->dim, p->batch);
    if (grid.y > 65535 || grid.z > 65535) return set_error(MMU_ERR_UNSUPPORTED, "causal_conv1d: dim/batch > 65535");
    const bool ord = p->order != MMU_ORDER_ROWMAJOR;
    if (bwd && part != nullptr) {
        if (ord) conv1d_bwd_kernel<IN_T, true, true><<<grid, kConvNT, 0, st>>>(a);
        else conv1d_bwd_kernel<IN_T, false, true><<<grid, kConvNT, 0, st>>>(a);
        count_launch();
        if (int rc = check_launch("causal_conv1d_bwd(deterministic)")) return rc;
        const int64_t items = (int64_t)p->batch * grid.x;
        // dweight[d][k] = sum of slot (d, 4 - W + k);  dbias[d] = sum of slot (d, 4)
        if (int rc = det_reduce(DetSum{part + (4 - p->width), items, (int64_t)p->dim * 5, 1, p->dim, p->width, 0, 5, p->dweight, 0,
                                       p->width, 1}, st))
            return rc;
        if (p->dbias == nullptr) return MMU_OK;
        return det_reduce(DetSum{part + 4, items, (int64_t)p->dim * 5, 1, p->dim, 1, 0, 5, p->dbias, 0, 1, 0}, st);
    }
    if (bwd) {
        if (ord) conv1d_bwd_kernel<IN_T, true><<<grid, kConvNT, 0, st>>>(a);
        else conv1d_bwd_kernel<IN_T, false><<<grid, kConvNT, 0, st>>>(a);
    } else {
        if (ord) conv1d_fwd_kernel<IN_T, true><<<grid, kConvNT, 0, st>>>(a);
        else conv1d_fwd_kernel<IN_T, false><<<grid, kConvNT, 0, st>>>(a);
    }
    count_launch();
    return check_launch(bwd ? "causal_conv1d_bwd" : "causal_conv1d_fwd");
}

int conv_entry(const mmu_conv_params *p, bool bwd, float *part, void *stream) {
    if (p == nullptr) return set_error(MMU_ERR_INVALID, "causal_conv1d: null params");
    if (p->batch <= 0 || p->dim <= 0 || p->seqlen <= 0) return set_error(MMU_ERR_INVALID, "causal_conv1d: empty shape");
    if (p->width < 2 || p->width > 4) return set_error(MMU_ERR_INVALID, "causal_conv1d only supports width between 2 and 4");
    if (!p->x || !p->weight) return set_error(MMU_ERR_INVALID, "causal_conv1d: null tensor pointer");
    if (!bwd && !p->out) return set_error(MMU_ERR_INVALID, "causal_conv1d_fwd: null out");
    if (bwd && (!p->dout || !p->dx || !p->dweight)) return set_error(MMU_ERR_INVALID, "causal_conv1d_bwd: null tensor pointer");
    if (bwd && p->bias != nullptr && !p->dbias) return set_error(MMU_ERR_INVALID, "causal_conv1d_bwd: dbias missing");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (p->dtype) {
        case MMU_F32: return run_conv<float>(p, bwd, part, st);
        case MMU_BF16: return run_conv<__nv_bfloat16>(p, bwd, part, st);
        case MMU_F16: return run_conv<__half>(p, bwd, part, st);
        default: return set_error(MMU_ERR_UNSUPPORTED, "causal_conv1d: dtype %d", p->dtype);
    }
}
}  // namespace
}  // namespace mmu

extern "C" int mmu_causal_conv1d_fwd(const mmu_conv_params *p, void *stream) { return mmu::conv_entry(p, false, nullptr, stream); }
extern "C" int mmu_causal_conv1d_bwd(const mmu_conv_params *p, void *stream) { return mmu::conv_entry(p, true, nullptr, stream); }

extern "C" size_t mmu_causal_conv1d_bwd_det_workspace(int32_t batch, int32_t dim, int32_t seqlen, int32_t dtype) {
    if (batch <= 0 || dim <= 0 || seqlen <= 0) return 0;
    mmu::DetWs w{nullptr};
    w.take(mmu::conv_det_floats(batch, dim, seqlen, dtype));
    return w.used;
}
extern "C" int mmu_causal_conv1d_bwd_det(const mmu_conv_params *p, void *ws, size_t ws_bytes, void *stream) {
    using namespace mmu;
    if (p == nullptr) return set_error(MMU_ERR_INVALID, "causal_conv1d_bwd_det: null params");
    const size_t need = mmu_causal_conv1d_bwd_det_workspace(p->batch, p->dim, p->seqlen, p->dtype);
    if (need == 0) return set_error(MMU_ERR_INVALID, "causal_conv1d_bwd_det: empty shape");
    if (int rc = det_ws_check(ws, ws_bytes, need, "causal_conv1d_bwd_det")) return rc;
    return conv_entry(p, true, static_cast<float *>(ws), stream);
}
