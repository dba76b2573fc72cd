// Selective scan backward for sm_100a (recompute-based; never materialises the L x N state in HBM).
//
// Replaces selective_scan_bwd_kernel (requirements/Mamba/mamba/csrc/selective_scan/selective_scan_bwd_kernel.cuh:75-489).
// Math: SURVEY.md Appendix A.  Decomposition (DESIGN.md "scan backward"):
//
//   * chunks of 64 tokens are walked last -> first; the forward state entering a chunk comes from the x buffer
//     the forward kernel saved every MMU_STATE_STRIDE tokens, the reverse state dh is carried in shared memory;
//   * a warp owns 4 channel rows x 8 token-lanes x 8 tokens; both in-chunk scans (forward recompute, reverse dh)
//     are 3-step 8-lane shuffle scans; the dstate axis is split over NGW warps and walked two states at a time
//     with packed FFMA2;
//   * dB/dC (sums over channels) are reduced across the 4 rows of a warp with a select/shuffle butterfly, across
//     the row-warps of the CTA in shared memory, and only then added to global memory - (D / rows-per-CTA)
//     atomics per element instead of the reference's D (selective_scan_bwd_kernel.cuh:306-315);
//   * the pre-gate output y is recomputed (one extra FFMA2 per state pair), so `out` is never read;
//   * like the forward, the sequence can be split over CTAs: an aggregate pass yields per-segment
//     (dh at segment start | zero inflow, sum(delta), delta_first), a tiny kernel chains them right-to-left.
#include <algorithm>
#include <cstdlib>

#include "scan3_bwd.cuh"
#include "tma_map.cuh"
#include "scan4_bwd.cuh"
#include "scan_tiles.cuh"

namespace mmu {

struct BwdArgs {
    const void *u, *delta, *z, *dout, *Bm, *Cm;
    const float *A, *Dv, *dbias, *x;
    void *du, *ddelta, *dz;
    float *dA, *dB, *dC, *dD, *ddbias;
    float *seg_dh, *seg_dsum, *seg_dfirst;
    const float *dhin;
    int64_t u_bs, u_ds, dl_bs, dl_ds, z_bs, z_ds, g_bs, g_ds, B_bs, B_ns, C_bs, C_ns;
    int64_t du_bs, du_ds, ddl_bs, ddl_ds, dz_bs, dz_ds;
    int64_t dB_bs, dC_bs, dB_ns, dC_ns;
    int B, D, L, N, Ne;
    int nseg, cps, nchunks, nx;
    int softplus, reverse;
    unsigned vec_mask;   // bit0 u, 1 delta, 2 z, 3 dout, 4 B, 5 C, 6 du, 7 ddelta, 8 dz
    int64_t det_rgs;     // DET kernels: row-group stride of the dB / dC slots
};

template <int RQ, int NGW> struct BwdCfg {
    static constexpr int T = 8, LS = 8, RG = 4;
    static constexpr int R = RQ * RG, TL = LS * T, NT = 32 * RQ * NGW, NW = RQ * NGW;
    static_assert(TL == MMU_STATE_STRIDE, "backward chunk == saved-state stride");
    static size_t smem_floats(int Ne) {
        return (size_t)4 * R * TL + 2 * (size_t)Ne * TL + (size_t)NGW * 3 * R * TL + (size_t)RQ * (Ne / 2) * 4 * TL +
               (size_t)NW * 1024 + (size_t)5 * R * Ne + (size_t)R * Ne * 8 + 4 * R;
    }
};

// DET (deterministic mode, main pass only): as scan3_bwd_kernel's DET - dB / dC / dA / dD / ddbias point at the caller's slots, the
// CTA stores its sums there, and dD / ddbias are summed over the CTA in a fixed order instead of with shared-memory atomics.
template <typename IN_T, int RQ, int NGW, bool AGG, int MINB, bool DET = false>
__global__ void __launch_bounds__(32 * RQ * NGW, AGG ? 512 / (32 * RQ * NGW) : MINB) scan_bwd_kernel(const __grid_constant__ BwdArgs p) {
    using Cfg = BwdCfg<RQ, NGW>;
    constexpr int T = Cfg::T, R = Cfg::R, TL = Cfg::TL, NT = Cfg::NT, NW = Cfg::NW;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int wq = warp / NGW, g = warp % NGW, rg = lane >> 3, j = lane & 7;
    const int b = blockIdx.y, row0 = blockIdx.x * R, seg = blockIdx.z;
    const int N = p.N, Ne = p.Ne, NP = Ne >> 1, D = p.D, L = p.L;
    const bool has_z = p.z != nullptr, rev = p.reverse != 0, sp = p.softplus != 0;

    extern __shared__ __align__(128) unsigned char smem_raw[];
    float *s_u = reinterpret_cast<float *>(smem_raw);   // [R][TL]  u, later du
    float *s_dl = s_u + R * TL;                          // [R][TL]  softplus(delta+bias), later ddelta
    float *s_z = s_dl + R * TL;                          // [R][TL]  z -> dz factor -> dz
    float *s_g = s_z + R * TL;                           // [R][TL]  dout -> dy
    float *s_B = s_g + R * TL;                           // [NP][TL][2]  pair-interleaved
    float *s_C = s_B + Ne * TL;                          // [NP][TL][2]
    float *s_part = s_C + Ne * TL;                       // [NGW][3][R][TL]  partial S1, S2, y
    float *s_dbc = s_part + NGW * 3 * R * TL;            // [RQ][NP][8 i][8 j][4]  row-reduced (dB.x dB.y dC.x dC.y), token = 8j+i
    float *s_stg = s_dbc + RQ * NP * 4 * TL;             // [NW][4 rows][8 i][8 j][4]  per-warp products awaiting the row sum
    float *s_A2 = s_stg + NW * 1024;                     // [R][Ne]  A*log2e
    float *s_A = s_A2 + R * Ne;                          // [R][Ne]
    float *s_hin = s_A + R * Ne;                         // [R][Ne]  forward state entering the chunk
    float *s_dhc = s_hin + R * Ne;                       // [R][Ne]  dh at the first token of the next chunk
    float *s_an = s_dhc + R * Ne;                        // [R][Ne]  a at the first token of the next chunk
    float *s_dA = s_an + R * Ne;                         // [R][NP][8 lanes][2]
    float *s_bias = s_dA + R * Ne * 8;                   // [R]
    float *s_D = s_bias + R;                             // [R]
    float *s_dD = s_D + R;                               // [R]
    float *s_db = s_dD + R;                              // [R]

    const int c_begin = seg * p.cps, c_end = min(p.nchunks, c_begin + p.cps);
    const IN_T *dl_b = reinterpret_cast<const IN_T *>(p.delta) + (int64_t)b * p.dl_bs;

    for (int r = tid; r < R; r += NT) {
        const int row = row0 + r;
        s_bias[r] = (row < D && p.dbias != nullptr) ? p.dbias[row] : 0.f;
        s_D[r] = (row < D && p.Dv != nullptr) ? p.Dv[row] : 0.f;
        s_dD[r] = 0.f;
        s_db[r] = 0.f;
    }
    __syncthreads();
    for (int i = tid; i < R * Ne; i += NT) {
        const int r = i / Ne, n = i - r * Ne, row = row0 + r;
        const bool ok = row < D && n < N;
        const float A = ok ? p.A[(int64_t)row * N + n] : 0.f;
        s_A[i] = A;
        s_A2[i] = A * kLog2e;
        float dh0 = 0.f, an = 1.f;
        const int tn = c_end * TL;   // first logical token of the next segment
        if (ok && tn < L) {
            const float raw = Elem<IN_T>::to_f(dl_b[(int64_t)row * p.dl_ds + (rev ? L - 1 - tn : tn)]) + s_bias[r];
            an = ex2(A * kLog2e * (sp ? softplus_f(raw) : raw));
            if (!AGG && p.dhin != nullptr) dh0 = p.dhin[(((int64_t)b * D + row) * p.nseg + seg) * Ne + n];
        }
        s_dhc[i] = dh0;
        s_an[i] = an;
    }
    for (int i = tid; i < R * Ne * 8; i += NT) s_dA[i] = 0.f;

    const IN_T *u_b = reinterpret_cast<const IN_T *>(p.u) + (int64_t)b * p.u_bs;
    const IN_T *z_b = has_z ? reinterpret_cast<const IN_T *>(p.z) + (int64_t)b * p.z_bs : nullptr;
    const IN_T *g_b = reinterpret_cast<const IN_T *>(p.dout) + (int64_t)b * p.g_bs;
    const IN_T *B_b = reinterpret_cast<const IN_T *>(p.Bm) + (int64_t)b * p.B_bs;
    const IN_T *C_b = reinterpret_cast<const IN_T *>(p.Cm) + (int64_t)b * p.C_bs;

    const int npw = (NP + NGW - 1) / NGW;
    const int pair0 = g * npw, pair1 = min(NP, pair0 + npw);
    const int lr = wq * 4 + rg;
    float dsum = 0.f, dfirst = 0.f;

    // per-thread constant shared-memory offsets (hoisted out of every loop)
    const int off_t0 = lr * TL + 4 * swz_chunk<T>(j * 2), off_t1 = lr * TL + 4 * swz_chunk<T>(j * 2 + 1);
    int off_bc[4];
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) off_bc[cc] = bc_off(j * 4 + cc);

    // ---- chunk loop (last -> first) with register prefetch of the next chunk's tiles -----------------------------------
    constexpr int QT = R * (TL / 4);                      // quads of a row tile
    constexpr int KR = (QT + NT - 1) / NT;
    constexpr int K2 = (8 * (TL / 4) + NT - 1) / NT;      // pair-quads per thread of a B / C tile (fast path: dstate <= 16)
    constexpr int KH = (R * 16 + NT - 1) / NT;
    const bool fast_all = (p.vec_mask & 0x8000u) != 0;
    Quad<IN_T> q_u[KR], q_dl[KR], q_z[KR], q_g[KR], q_B[2 * K2], q_C[2 * K2];
    float q_h[KH];
    auto ident = [](int, float v) { return v; };
    auto dl_xf = [&](int r, float v) {
        const float xx = v + s_bias[r];
        return sp ? softplus_f(xx) : xx;
    };
    auto load_hin = [&](int c, int i) -> float {
        const int r = i / Ne, n = i - r * Ne, row = row0 + r;
        return (c > 0 && row < D && n < N) ? p.x[(((int64_t)b * D + row) * p.nx + (c - 1)) * N + n] : 0.f;
    };
    auto prefetch = [&](int c) {
        const int t0 = c * TL;
        tile_prefetch<IN_T, TL, NT, KR>(q_dl, dl_b, p.dl_ds, row0, D, QT, t0, L, rev, tid);
        tile_prefetch<IN_T, TL, NT, KR>(q_g, g_b, p.g_ds, row0, D, QT, t0, L, rev, tid);
        bc_prefetch<IN_T, TL, NT, K2>(q_C, C_b, p.C_ns, N, NP, t0, L, rev, tid);
        if (has_z) tile_prefetch<IN_T, TL, NT, KR>(q_z, z_b, p.z_ds, row0, D, QT, t0, L, rev, tid);
        if (!AGG) {
            tile_prefetch<IN_T, TL, NT, KR>(q_u, u_b, p.u_ds, row0, D, QT, t0, L, rev, tid);
            bc_prefetch<IN_T, TL, NT, K2>(q_B, B_b, p.B_ns, N, NP, t0, L, rev, tid);
#pragma unroll
            for (int k = 0; k < KH; ++k) q_h[k] = (tid + k * NT < R * Ne) ? load_hin(c, tid + k * NT) : 0.f;
        }
    };
    float acc_dD[KR], acc_db[KR];    // per-thread partial dD / ddelta_bias of the row its epilogue quad belongs to
#pragma unroll
    for (int k = 0; k < KR; ++k) acc_dD[k] = acc_db[k] = 0.f;

    bool cur_fast = fast_all && c_end * TL <= L;
    if (cur_fast) prefetch(c_end - 1);
    for (int c = c_end - 1; c >= c_begin; --c) {
        const int t0 = c * TL;
        __syncthreads();
        if (cur_fast) {
            tile_commit<IN_T, T, TL, NT, KR>(s_dl, q_dl, QT, rev, tid, dl_xf);
            tile_commit<IN_T, T, TL, NT, KR>(s_g, q_g, QT, rev, tid, ident);
            bc_commit<IN_T, TL, NT, K2>(s_C, q_C, NP, rev, tid);
            if (has_z) tile_commit<IN_T, T, TL, NT, KR>(s_z, q_z, QT, rev, tid, ident);
            if (!AGG) {
                tile_commit<IN_T, T, TL, NT, KR>(s_u, q_u, QT, rev, tid, ident);
                bc_commit<IN_T, TL, NT, K2>(s_B, q_B, NP, rev, tid);
#pragma unroll
                for (int k = 0; k < KH; ++k)
                    if (tid + k * NT < R * Ne) s_hin[tid + k * NT] = q_h[k];
            }
        } else {
            load_tile<IN_T, T, TL, NT>(s_dl, dl_b, p.dl_ds, row0, R, D, t0, L, rev, p.vec_mask & 2u, tid, 0.f, dl_xf);
            load_tile<IN_T, T, TL, NT>(s_g, g_b, p.g_ds, row0, R, D, t0, L, rev, p.vec_mask & 8u, tid, 0.f, ident);
            bc_load_generic<IN_T, TL, NT>(s_C, C_b, p.C_ns, N, Ne, t0, L, rev, tid);
            if (has_z) load_tile<IN_T, T, TL, NT>(s_z, z_b, p.z_ds, row0, R, D, t0, L, rev, p.vec_mask & 4u, tid, 0.f, ident);
            if (!AGG) {
                load_tile<IN_T, T, TL, NT>(s_u, u_b, p.u_ds, row0, R, D, t0, L, rev, p.vec_mask & 1u, tid, 0.f, ident);
                bc_load_generic<IN_T, TL, NT>(s_B, B_b, p.B_ns, N, Ne, t0, L, rev, tid);
                for (int i = tid; i < R * Ne; i += NT) s_hin[i] = load_hin(c, i);
            }
        }
        if (has_z) {
            // same thread, same elements as it just wrote: dy = dout*silu(z); s_z <- factor such that dz = y * s_z
            for (int idx = tid; idx < QT; idx += NT) {
                const int rr = idx / (TL / 4), ch = idx - rr * (TL / 4);
                const int zoff = rr * TL + 4 * swz_chunk<T>(ch);
                float4 z4 = *reinterpret_cast<const float4 *>(s_z + zoff);
                float4 g4 = *reinterpret_cast<const float4 *>(s_g + zoff);
                float *zz = reinterpret_cast<float *>(&z4), *gg = reinterpret_cast<float *>(&g4);
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float s = sigmoid_f(zz[k]);
                    const float gz = gg[k] * s;
                    gg[k] = gz * zz[k];                               // dy   (bwd_kernel.cuh:186-191)
                    zz[k] = gz * fmaf(zz[k], 1.f - s, 1.f);           // dz = y * this
                }
                *reinterpret_cast<float4 *>(s_z + zoff) = z4;
                *reinterpret_cast<float4 *>(s_g + zoff) = g4;
            }
        }
        __syncthreads();
        cur_fast = fast_all && c > c_begin;    // every chunk before the last one of the sequence is full
        if (cur_fast) prefetch(c - 1);

        float dl[T], dlu[T], dy[T];
#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
            const int off = cc ? off_t1 : off_t0;
            const float4 d4 = *reinterpret_cast<const float4 *>(s_dl + off);
            const float4 g4 = *reinterpret_cast<const float4 *>(s_g + off);
            float4 u4 = make_float4(0.f, 0.f, 0.f, 0.f);
            if (!AGG) u4 = *reinterpret_cast<const float4 *>(s_u + off);
            dl[4 * cc] = d4.x, dl[4 * cc + 1] = d4.y, dl[4 * cc + 2] = d4.z, dl[4 * cc + 3] = d4.w;
            dy[4 * cc] = g4.x, dy[4 * cc + 1] = g4.y, dy[4 * cc + 2] = g4.z, dy[4 * cc + 3] = g4.w;
            dlu[4 * cc] = d4.x * u4.x, dlu[4 * cc + 1] = d4.y * u4.y, dlu[4 * cc + 2] = d4.z * u4.z,
                     dlu[4 * cc + 3] = d4.w * u4.w;
        }
        if (AGG) {
#pragma unroll
            for (int i = 0; i < T; ++i) dsum += dl[i];
            if (c == c_begin) dfirst = dl[0];   // meaningful in lane j == 0
        }
        float2 S1[T], S2[T], yv[T];
#pragma unroll
        for (int i = 0; i < T; ++i) S1[i] = S2[i] = yv[i] = make_float2(0.f, 0.f);

        const float *pB = s_B + pair0 * 2 * TL, *pC = s_C + pair0 * 2 * TL;
        int tab = lr * Ne + 2 * pair0;          // offset of my (row, pair) in the [R][Ne] tables
        float *pdbc = s_dbc + (wq * NP + pair0) * 4 * TL + lane * 4;   // my two row-summed entries: e = lane, lane + 32
        float *stg_w = s_stg + warp * 1024 + rg * 256 + j * 4;          // my slot for token i: + i * 32
        float2 *pdA = reinterpret_cast<float2 *>(s_dA) + (lr * NP + pair0) * 8 + j;
        for (int pr = pair0; pr < pair1; ++pr, pB += 2 * TL, pC += 2 * TL, tab += 2, pdbc += 4 * TL, pdA += 8) {
            const float2 A2 = *reinterpret_cast<const float2 *>(s_A2 + tab);
            float2 a[T], Cv[T], Bv[T];
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
                const float4 c4 = *reinterpret_cast<const float4 *>(pC + off_bc[cc]);
                Cv[2 * cc] = make_float2(c4.x, c4.y), Cv[2 * cc + 1] = make_float2(c4.z, c4.w);
                if (!AGG) {
                    const float4 b4 = *reinterpret_cast<const float4 *>(pB + off_bc[cc]);
                    Bv[2 * cc] = make_float2(b4.x, b4.y), Bv[2 * cc + 1] = make_float2(b4.z, b4.w);
                }
            }
#pragma unroll
            for (int i = 0; i < T; ++i) a[i] = ex2(fmul2(splat(dl[i]), A2));

            // ---- forward recompute: state before my first token ------------------------------------------
            float2 hs = make_float2(0.f, 0.f);
            if (!AGG) {
                float2 P = make_float2(1.f, 1.f), hl = make_float2(0.f, 0.f);
#pragma unroll
                for (int i = 0; i < T; ++i) {
                    hl = ffma2(a[i], hl, fmul2(splat(dlu[i]), Bv[i]));
                    P = fmul2(P, a[i]);
                }
#pragma unroll
                for (int k = 1; k < 8; k <<= 1) {
                    const float2 Pn = shfl_up2(P, k, 8), Hn = shfl_up2(hl, k, 8);
                    if (j >= k) {
                        hl = ffma2(P, Hn, hl);
                        P = fmul2(P, Pn);
                    }
                }
                const float2 hc = *reinterpret_cast<const float2 *>(s_hin + tab);
                const float2 send = ffma2(P, hc, hl);
                hs = shfl_up2(send, 1, 8);
                if (j == 0) hs = hc;
            }
            // ---- reverse: dh at the first token of the lane to my right ---------------------------------------
            float *dhc_p = s_dhc + tab, *an_p = s_an + tab;
            float2 a_nl = shfl_down2(a[0], 1, 8);   // a of the first token of the next lane
            if (j == 7) a_nl = *reinterpret_cast<const float2 *>(an_p);
            float2 dhn;
            {
                float2 Pr = a_nl, dhl = fmul2(Cv[T - 1], splat(dy[T - 1]));
#pragma unroll
                for (int i = T - 2; i >= 0; --i) {
                    dhl = ffma2(a[i + 1], dhl, fmul2(Cv[i], splat(dy[i])));
                    Pr = fmul2(Pr, a[i + 1]);
                }
#pragma unroll
                for (int k = 1; k < 8; k <<= 1) {
                    const float2 Pn = shfl_down2(Pr, k, 8), Hn = shfl_down2(dhl, k, 8);
                    if (j + k < 8) {
                        dhl = ffma2(Pr, Hn, dhl);
                        Pr = fmul2(Pr, Pn);
                    }
                }
                const float2 dhc = *reinterpret_cast<const float2 *>(dhc_p);
                const float2 dfirst_tok = ffma2(Pr, dhc, dhl);   // dh at my first token
                dhn = shfl_down2(dfirst_tok, 1, 8);
                if (j == 7) dhn = dhc;
                __syncwarp();
                if (j == 0) {
                    *reinterpret_cast<float2 *>(dhc_p) = dfirst_tok;
                    *reinterpret_cast<float2 *>(an_p) = a[0];
                }
            }
            if (AGG) continue;

            // ---- forward states of my tokens -------------------------------------------------------------------
            float2 h[T];
            {
                float2 hp = hs;
#pragma unroll
                for (int i = 0; i < T; ++i) {
                    hp = ffma2(a[i], hp, fmul2(splat(dlu[i]), Bv[i]));
                    h[i] = hp;
                }
            }
            // ---- reverse sweep: consume -----------------------------------------------------------------------------
            const float2 Av = *reinterpret_cast<const float2 *>(s_A + tab);
            float2 e = fmul2(a_nl, dhn);   // a_{t+1} * dh_{t+1} for my last token
            float2 dAacc = make_float2(0.f, 0.f);
#pragma unroll
            for (int i = T - 1; i >= 0; --i) {
                const float2 dh = ffma2(Cv[i], splat(dy[i]), e);
                const float2 hprev = i > 0 ? h[i - 1] : hs;
                e = fmul2(a[i], dh);
                const float2 q = fmul2(e, hprev);                    // dh * a_t * h_{t-1}
                S1[i] = ffma2(dh, Bv[i], S1[i]);
                S2[i] = ffma2(Av, q, S2[i]);
                dAacc = ffma2(splat(dl[i]), q, dAacc);
                yv[i] = ffma2(Cv[i], h[i], yv[i]);
                const float2 dBv = fmul2(dh, splat(dlu[i]));
                const float2 dCv = fmul2(h[i], splat(dy[i]));
                // products of my row; the 4 rows of the warp are summed below through the warp's staging area
                *reinterpret_cast<float4 *>(stg_w + i * 32) = make_float4(dBv.x, dBv.y, dCv.x, dCv.y);
            }
            __syncwarp();
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                const float *src = s_stg + warp * 1024 + (lane + 32 * q) * 4;      // entry e = 8*i + j
                float4 v0 = *reinterpret_cast<const float4 *>(src);
                const float4 v1 = *reinterpret_cast<const float4 *>(src + 256);
                const float4 v2 = *reinterpret_cast<const float4 *>(src + 512);
                const float4 v3 = *reinterpret_cast<const float4 *>(src + 768);
                v0.x += v1.x + (v2.x + v3.x), v0.y += v1.y + (v2.y + v3.y);
                v0.z += v1.z + (v2.z + v3.z), v0.w += v1.w + (v2.w + v3.w);
                *reinterpret_cast<float4 *>(pdbc + 128 * q) = v0;
            }
            __syncwarp();
            *pdA = fadd2(*pdA, dAacc);
        }
        if (AGG) continue;

#pragma unroll
        for (int cc = 0; cc < 2; ++cc) {
            float *pp = s_part + (g * 3) * R * TL + (cc ? off_t1 : off_t0);
            *reinterpret_cast<float4 *>(pp) = make_float4(S1[4 * cc].x + S1[4 * cc].y, S1[4 * cc + 1].x + S1[4 * cc + 1].y,
                                                          S1[4 * cc + 2].x + S1[4 * cc + 2].y, S1[4 * cc + 3].x + S1[4 * cc + 3].y);
            *reinterpret_cast<float4 *>(pp + R * TL) =
                make_float4(S2[4 * cc].x + S2[4 * cc].y, S2[4 * cc + 1].x + S2[4 * cc + 1].y,
                            S2[4 * cc + 2].x + S2[4 * cc + 2].y, S2[4 * cc + 3].x + S2[4 * cc + 3].y);
            *reinterpret_cast<float4 *>(pp + 2 * R * TL) =
                make_float4(yv[4 * cc].x + yv[4 * cc].y, yv[4 * cc + 1].x + yv[4 * cc + 1].y,
                            yv[4 * cc + 2].x + yv[4 * cc + 2].y, yv[4 * cc + 3].x + yv[4 * cc + 3].y);
        }
        __syncthreads();

        // ---- epilogue A: per-(row,token) gradients, one quad per thread, stored straight to global ------------------------
        {
            IN_T *du_b = reinterpret_cast<IN_T *>(p.du) + (int64_t)b * p.du_bs;
            IN_T *dd_b = reinterpret_cast<IN_T *>(p.ddelta) + (int64_t)b * p.ddl_bs;
            IN_T *dz_b = has_z ? reinterpret_cast<IN_T *>(p.dz) + (int64_t)b * p.dz_bs : nullptr;
#pragma unroll
            for (int k = 0; k < KR; ++k) {
                const int idx = tid + k * NT;
                if (idx >= QT) continue;
                const int r = idx / (TL / 4), cs = idx - r * (TL / 4);
                const int off = idx * 4;   // raw (swizzled) position
                float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s1, yy = s1;
#pragma unroll
                for (int gg = 0; gg < NGW; ++gg) {
                    const float *pp = s_part + (gg * 3) * R * TL + off;
                    const float4 a1 = *reinterpret_cast<const float4 *>(pp);
                    const float4 a2 = *reinterpret_cast<const float4 *>(pp + R * TL);
                    const float4 a3 = *reinterpret_cast<const float4 *>(pp + 2 * R * TL);
                    s1.x += a1.x, s1.y += a1.y, s1.z += a1.z, s1.w += a1.w;
                    s2.x += a2.x, s2.y += a2.y, s2.z += a2.z, s2.w += a2.w;
                    yy.x += a3.x, yy.y += a3.y, yy.z += a3.z, yy.w += a3.w;
                }
                const float4 u4 = *reinterpret_cast<const float4 *>(s_u + off);
                const float4 d4 = *reinterpret_cast<const float4 *>(s_dl + off);
                const float4 g4 = *reinterpret_cast<const float4 *>(s_g + off);
                const float Dk = s_D[r];
                const float uu[4] = {u4.x, u4.y, u4.z, u4.w}, dd_[4] = {d4.x, d4.y, d4.z, d4.w};
                const float gg_[4] = {g4.x, g4.y, g4.z, g4.w}, S1[4] = {s1.x, s1.y, s1.z, s1.w};
                const float S2[4] = {s2.x, s2.y, s2.z, s2.w}, Y[4] = {yy.x, yy.y, yy.z, yy.w};
                float du[4], dd[4], dzv[4];
                float4 zf = make_float4(0.f, 0.f, 0.f, 0.f);
                if (has_z) zf = *reinterpret_cast<const float4 *>(s_z + off);
                const float ZF[4] = {zf.x, zf.y, zf.z, zf.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    du[e] = fmaf(dd_[e], S1[e], Dk * gg_[e]);          // D*dy + delta*S1   (bwd_kernel.cuh:211,280-281)
                    float t_ = fmaf(uu[e], S1[e], S2[e]);               // u*S1 + S2         (:282-283)
                    if (sp) t_ *= 1.f - __expf(-dd_[e]);                // softplus' = sigmoid(x) = 1 - exp(-softplus(x))
                    dd[e] = t_;
                    dzv[e] = fmaf(Dk, uu[e], Y[e]) * ZF[e];
                    acc_dD[k] = fmaf(gg_[e], uu[e], acc_dD[k]);
                    acc_db[k] += t_;
                }
                const int row = row0 + r, t = t0 + 4 * swz_chunk<T>(cs);
                if (row < D && t < L) {
                    store_quad<IN_T>(du_b + (int64_t)row * p.du_ds, t, L, rev, p.vec_mask & 64u, du);
                    store_quad<IN_T>(dd_b + (int64_t)row * p.ddl_ds, t, L, rev, p.vec_mask & 128u, dd);
                    if (has_z) store_quad<IN_T>(dz_b + (int64_t)row * p.dz_ds, t, L, rev, p.vec_mask & 256u, dzv);
                }
            }
        }
        // ---- epilogue B: dB / dC -> global (sum over the CTA's row-warps, then one atomic per element) ---------------
        {
            float *dB_b = p.dB + (int64_t)b * p.dB_bs + (DET ? (int64_t)blockIdx.x * p.det_rgs : 0);
            float *dC_b = p.dC + (int64_t)b * p.dC_bs + (DET ? (int64_t)blockIdx.x * p.det_rgs : 0);
            for (int idx = tid; idx < NP * TL; idx += NT) {
                const int tok = idx % TL, pr = idx / TL;
                const int e = ((tok & 7) << 3) | (tok >> 3);            // staging order: e = 8*i + j for token 8*j + i
                const float *src = s_dbc + (pr * TL + e) * 4;
                float4 v = *reinterpret_cast<const float4 *>(src);
#pragma unroll
                for (int q = 1; q < RQ; ++q) {
                    const float4 w = *reinterpret_cast<const float4 *>(src + q * NP * 4 * TL);
                    v.x += w.x, v.y += w.y, v.z += w.z, v.w += w.w;
                }
                const int t = t0 + tok, n0 = 2 * pr;
                if (t < L) {
                    const int64_t m = rev ? L - 1 - t : t;
                    if constexpr (DET) {
                        dB_b[(int64_t)n0 * p.dB_ns + m] = v.x;
                        dC_b[(int64_t)n0 * p.dC_ns + m] = v.z;
                        if (n0 + 1 < N) {
                            dB_b[(int64_t)(n0 + 1) * p.dB_ns + m] = v.y;
                            dC_b[(int64_t)(n0 + 1) * p.dC_ns + m] = v.w;
                        }
                    } else {
                        atomicAdd(dB_b + (int64_t)n0 * p.dB_ns + m, v.x);
                        atomicAdd(dC_b + (int64_t)n0 * p.dC_ns + m, v.z);
                        if (n0 + 1 < N) {
                            atomicAdd(dB_b + (int64_t)(n0 + 1) * p.dB_ns + m, v.y);
                            atomicAdd(dC_b + (int64_t)(n0 + 1) * p.dC_ns + m, v.w);
                        }
                    }
                }
            }
        }
    }

    __syncthreads();
    if (AGG) {
        for (int i = tid; i < R * Ne; i += NT) {
            const int r = i / Ne, n = i - r * Ne, row = row0 + r;
            if (row < D) p.seg_dh[(((int64_t)b * D + row) * p.nseg + seg) * Ne + n] = s_dhc[i];
        }
        if (g == 0) {
            float s = dsum;
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
            s += __shfl_xor_sync(0xffffffffu, s, 4);
            const int row = row0 + lr;
            if (j == 0 && row < D) {
                p.seg_dsum[((int64_t)b * D + row) * p.nseg + seg] = s;
                p.seg_dfirst[((int64_t)b * D + row) * p.nseg + seg] = dfirst;
            }
        }
    } else {
        for (int i = tid; i < R * Ne; i += NT) {
            const int r = i / Ne, n = i - r * Ne, row = row0 + r;
            if (row < D && n < N) {
                const float *src = s_dA + ((r * NP + (n >> 1)) * 8) * 2 + (n & 1);
                float v = 0.f;
#pragma unroll
                for (int k = 0; k < 8; ++k) v += src[2 * k];
                if constexpr (DET) p.dA[((int64_t)b * p.nseg + seg) * D * N + (int64_t)row * N + n] = v;
                else atomicAdd(p.dA + (int64_t)row * N + n, v);           // sum over batch and segments
            }
        }
        if constexpr (DET) {      // dD / ddelta_bias: the row's TL/4 quad partials (s_part is free now), summed in quad order
#pragma unroll
            for (int k = 0; k < KR; ++k) {
                const int idx = tid + k * NT;
                if (idx < QT) s_part[idx] = acc_dD[k], s_part[QT + idx] = acc_db[k];
            }
            __syncthreads();
            for (int r = tid; r < R; r += NT) {
                const int row = row0 + r;
                if (row < D) {
                    float sd = 0.f, sb = 0.f;
                    for (int q = 0; q < TL / 4; ++q) sd += s_part[r * (TL / 4) + q], sb += s_part[QT + r * (TL / 4) + q];
                    const int64_t slot = ((int64_t)b * p.nseg + seg) * D + row;
                    if (p.dD != nullptr) p.dD[slot] = sd;
                    if (p.ddbias != nullptr) p.ddbias[slot] = sb;
                }
            }
            return;
        }
#pragma unroll
        for (int k = 0; k < KR; ++k) {
            const int idx = tid + k * NT;
            if (idx < QT) {
                atomicAdd(s_dD + idx / (TL / 4), acc_dD[k]);
                atomicAdd(s_db + idx / (TL / 4), acc_db[k]);
            }
        }
        __syncthreads();
        for (int r = tid; r < R; r += NT) {
            const int row = row0 + r;
            if (row < D) {
                if (p.dD != nullptr) atomicAdd(p.dD + row, s_dD[r]);
                if (p.ddbias != nullptr) atomicAdd(p.ddbias + row, s_db[r]);
            }
        }
    }
}

// chain reverse aggregates right-to-left: dhin[s] = dh at the first token of segment s+1
__global__ void scan_bwd_chain_kernel(const float *__restrict__ A, const float *__restrict__ seg_dh,
                                      const float *__restrict__ seg_dsum, const float *__restrict__ seg_dfirst,
                                      float *__restrict__ dhin, int B, int D, int N, int Ne, int nseg) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)B * D * Ne) return;
    const int n = (int)(i % Ne);
    const int64_t bd = i / Ne;
    const int row = (int)(bd % D);
    const float a2 = n < N ? A[(int64_t)row * N + n] * kLog2e : 0.f;
    float carry = 0.f;
    for (int s = nseg - 1; s >= 0; --s) {
        dhin[(bd * nseg + s) * Ne + n] = carry;
        // product of a_{t+1} over the tokens t of segment s
        const float dnext = s + 1 < nseg ? seg_dfirst[bd * nseg + s + 1] : 0.f;
        const float P = ex2(a2 * (seg_dsum[bd * nseg + s] - seg_dfirst[bd * nseg + s] + dnext));
        carry = fmaf(P, carry, seg_dh[(bd * nseg + s) * Ne + n]);
    }
}

namespace {

int env_int(const char *name, int dflt) { return knob(name, dflt); }
size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

constexpr int kNumBwdCfg = 5;
constexpr int kBwdCfg[kNumBwdCfg][2] = {{2, 2}, {1, 4}, {2, 4}, {2, 2}, {2, 2}};   // {RQ, NGW}; 3/4 differ in regs cap

struct BwdPlan {
    int cfg, R, nseg, cps, nchunks;
};

BwdPlan plan_bwd(int B, int D, int L) {
    BwdPlan pl;
    pl.cfg = D <= 4 ? 1 : 3;   // 3 = 8 rows x 2 dstate groups, no register cap (no spills): fastest measured on B200
    pl.cfg = env_int("MMU_BWD_CFG", pl.cfg);
    if (pl.cfg < 0 || pl.cfg >= kNumBwdCfg) pl.cfg = 0;
    const int RQ = kBwdCfg[pl.cfg][0], NGW = kBwdCfg[pl.cfg][1];
    pl.R = 4 * RQ;
    pl.nchunks = (L + 63) / 64;
    const int warps = B * ((D + pl.R - 1) / pl.R) * RQ * NGW;
    const int target = 148 * 12;
    int nseg = warps >= 148 * 6 ? 1 : (target + warps - 1) / warps;   // splitting costs a second pass: only when starved
    nseg = std::min(nseg, std::max(1, pl.nchunks / 8));
    nseg = std::max(1, std::min(nseg, 64));
    nseg = env_int("MMU_BWD_NSEG", nseg);
    nseg = std::max(1, std::min(nseg, pl.nchunks));
    pl.cps = (pl.nchunks + nseg - 1) / nseg;
    pl.nseg = (pl.nchunks + pl.cps - 1) / pl.cps;
    return pl;
}

template <typename IN_T, int RQ, int NGW, int MINB> int launch_bwd(const BwdArgs &a, bool agg, bool det, cudaStream_t st) {
    using Cfg = BwdCfg<RQ, NGW>;
    const size_t smem = Cfg::smem_floats(a.Ne) * sizeof(float);
    if (smem > 227 * 1024) return set_error(MMU_ERR_UNSUPPORTED, "selective_scan_bwd: dstate %d needs %zu B smem", a.N, smem);
    dim3 grid((a.D + Cfg::R - 1) / Cfg::R, a.B, a.nseg), block(Cfg::NT);
    if (det && !agg) {
        auto k = scan_bwd_kernel<IN_T, RQ, NGW, false, MINB, true>;
        cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        k<<<grid, block, smem, st>>>(a);
    } else if (agg) {
        auto k = scan_bwd_kernel<IN_T, RQ, NGW, true, MINB>;
        cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        k<<<grid, block, smem, st>>>(a);
    } else {
        auto k = scan_bwd_kernel<IN_T, RQ, NGW, false, MINB>;
        cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        k<<<grid, block, smem, st>>>(a);
    }
    count_launch();
    return check_launch("selective_scan_bwd");
}

template <typename IN_T> int dispatch_bwd(int cfg, const BwdArgs &a, bool agg, cudaStream_t st, bool det = false) {
    switch (cfg) {
        case 0: return launch_bwd<IN_T, 2, 2, 3>(a, agg, det, st);
        case 1: return launch_bwd<IN_T, 1, 4, 3>(a, agg, det, st);
        case 2: return launch_bwd<IN_T, 2, 4, 1>(a, agg, det, st);
        case 3: return launch_bwd<IN_T, 2, 2, 2>(a, agg, det, st);
        default: return launch_bwd<IN_T, 2, 2, 4>(a, agg, det, st);
    }
}

// ---- deterministic mode: partial slots in the caller's workspace, then ordered reduces -----------------------------------------
// Slot layout (fixed for a shape, whichever kernel runs): dB and dC [row group][batch][dstate][seqlen], dA [batch][segment][dim][dstate],
// dD and ddelta_bias [batch][segment][dim], each sized for the most row groups / segments any plan of this shape can use.
struct ScanDet {
    float *pB, *pC, *pA, *pD, *pdb;
};
struct ScanDetBound {
    int64_t nrg, nseg;
};
ScanDetBound scan_det_bound(int B, int D, int L);   // below the plans
size_t scan_det_carve(int B, int D, int L, int N, char *base, ScanDet *d) {
    const ScanDetBound bd = scan_det_bound(B, D, L);
    DetWs w{base};
    const size_t bc = (size_t)bd.nrg * B * N * L, a = (size_t)B * bd.nseg * D * N, r = (size_t)B * bd.nseg * D;
    ScanDet t{w.take(bc), w.take(bc), w.take(a), w.take(r), w.take(r)};
    if (d != nullptr) *d = t;
    return w.used;
}
// point the kernel's gradient outputs at the slots
template <typename Args> void scan_det_args(Args &a, const ScanDet &d) {
    a.dB = d.pB, a.dC = d.pC, a.dA = d.pA;
    a.dD = a.dD ? d.pD : nullptr, a.ddbias = a.ddbias ? d.pdb : nullptr;
    a.dB_bs = a.dC_bs = (int64_t)a.N * a.L, a.dB_ns = a.dC_ns = a.L;
    a.det_rgs = (int64_t)a.B * a.N * a.L;
}
// sum the slots of the nrg row groups / nseg segments the kernel used into the caller's outputs
int scan_det_reduce(const mmu_scan_bwd_params *p, const ScanDet &d, int nrg, int nseg, cudaStream_t st) {
    const mmu_scan_fwd_params &f = p->f;
    const int B = f.batch, D = f.dim, L = f.seqlen, N = f.dstate;
    const int64_t dB_bs = p->dB_bs ? p->dB_bs : (int64_t)N * L, dC_bs = p->dC_bs ? p->dC_bs : (int64_t)N * L;
    const int64_t dB_ns = p->dB_ns ? p->dB_ns : L, dC_ns = p->dC_ns ? p->dC_ns : L;
    const int64_t rgs = (int64_t)B * N * L, items = (int64_t)B * nseg;
    if (int rc = det_reduce(DetSum{d.pB, nrg, rgs, B, N, L, (int64_t)N * L, L, p->dB, dB_bs, dB_ns, 1}, st)) return rc;
    if (int rc = det_reduce(DetSum{d.pC, nrg, rgs, B, N, L, (int64_t)N * L, L, p->dC, dC_bs, dC_ns, 1}, st)) return rc;
    if (int rc = det_reduce(DetSum{d.pA, items, (int64_t)D * N, 1, 1, D * N, 0, 0, p->dA, 0, 0, 1}, st)) return rc;
    if (p->dD != nullptr)
        if (int rc = det_reduce(DetSum{d.pD, items, D, 1, 1, D, 0, 0, p->dD, 0, 0, 1}, st)) return rc;
    if (p->ddelta_bias != nullptr)
        if (int rc = det_reduce(DetSum{d.pdb, items, D, 1, 1, D, 0, 0, p->ddelta_bias, 0, 0, 1}, st)) return rc;
    return MMU_OK;
}

// ---- v3 host side (scan3_bwd.cuh) ------------------------------------------------------------------------------------------
template <typename IN_T> bool row_aligned16(const void *p, int64_t s0, int64_t s1) {
    return reinterpret_cast<uintptr_t>(p) % 16 == 0 && (s0 * (int64_t)sizeof(IN_T)) % 16 == 0 && (s1 * (int64_t)sizeof(IN_T)) % 16 == 0;
}

template <typename IN_T> bool bwd3_eligible(const mmu_scan_bwd_params *p) {
    const mmu_scan_fwd_params &f = p->f;
    if (env_int("MMU_SCAN_V", 3) < 3 || env_int("MMU_BWD_V", 3) < 3) return false;
    if (f.dstate > 16 || f.seqlen % 8 != 0) return false;
    if (f.z && !f.y) return false;                       // dz needs the pre-gate y the forward saved
    if (f.seqlen > MMU_STATE_STRIDE && !f.x) return false;
    if (!row_aligned16<IN_T>(f.u, f.u_bs, f.u_ds) || !row_aligned16<IN_T>(f.delta, f.delta_bs, f.delta_ds) ||
        !row_aligned16<IN_T>(p->dout, p->dout_bs, p->dout_ds) || !row_aligned16<IN_T>(f.B, f.B_bs, f.B_ns) ||
        !row_aligned16<IN_T>(f.C, f.C_bs, f.C_ns) || !row_aligned16<IN_T>(p->du, p->du_bs, p->du_ds) ||
        !row_aligned16<IN_T>(p->ddelta, p->ddelta_bs, p->ddelta_ds))
        return false;
    if (f.z && (!row_aligned16<IN_T>(f.z, f.z_bs, f.z_ds) || !row_aligned16<IN_T>(f.y, f.y_bs, f.y_ds) ||
                !row_aligned16<IN_T>(p->dz, p->dz_bs, p->dz_ds)))
        return false;
    if (reinterpret_cast<uintptr_t>(p->dB) % 16 != 0 || reinterpret_cast<uintptr_t>(p->dC) % 16 != 0) return false;
    if ((p->dB_bs * 4) % 16 != 0 || (p->dC_bs * 4) % 16 != 0 || (p->dB_ns * 4) % 16 != 0 || (p->dC_ns * 4) % 16 != 0) return false;
    return true;
}

struct Bwd3Plan {
    int W, nseg, cps, nchunks;
    bool chain;     // segments are chained CTAs (no aggregate pass)
};

Bwd3Plan plan_bwd3(int B, int D, int L, bool ordered = false) {
    Bwd3Plan pl;
    pl.W = env_int("MMU_BWD3_W", D <= 2 ? 1 : (D <= 4 ? 2 : 4));   // W = 3 (6 rows) measured slower than 4 with idle lanes
    if (pl.W != 8 && (pl.W < 1 || pl.W > 4)) pl.W = 4;
    if (ordered && pl.W == 8) pl.W = 4;
    const int R = 2 * pl.W;
    pl.nchunks = (L + 255) / 256;
    const int warps = B * ((D + R - 1) / R) * pl.W;
    int nseg = warps >= 148 * 4 ? 1 : (148 * 8 + warps - 1) / warps;   // splitting costs a second (aggregate) pass
    nseg = std::min(nseg, std::max(1, pl.nchunks / 2));
    nseg = std::max(1, std::min(nseg, 64));
    nseg = env_int("MMU_BWD_NSEG", nseg);
    pl.chain = false;
    {
        // Wide problem: one CTA per row group walks the whole sequence.  When those CTAs do not fill whole waves (2 CTAs of
        // 4 warps per SM), cut the sequence into chained segments so the tail wave shrinks (measured at config 2: 578 ->
        // 482 us with 3 segments).  MMU_BWD_CHAIN=k forces k chained segments (tests), 1 disables.
        const int slots = 148 * (pl.W == 8 ? 1 : 2), ctas = warps / pl.W, rem = ctas % slots;
        int want = (nseg == 1 && warps >= 148 * 4 && ctas > slots && rem != 0 && rem < slots * 3 / 4 && pl.nchunks >= 6) ? 3 : 1;
        want = env_int("MMU_BWD_CHAIN", want);
        if (want > 1 && pl.nchunks >= want) nseg = want, pl.chain = true;
    }
    nseg = std::max(1, std::min(nseg, pl.nchunks));
    pl.cps = (pl.nchunks + nseg - 1) / nseg;
    pl.nseg = (pl.nchunks + pl.cps - 1) / pl.cps;
    if (pl.nseg == 1) pl.chain = false;
    return pl;
}

template <typename IN_T, int W, bool REV, bool AGG, bool ORD = false, bool DET = false> int launch_bwd3(const Bwd3Args &a, cudaStream_t st) {
    using Cfg = Bwd3Cfg<IN_T, W>;
    dim3 grid((a.D + Cfg::R - 1) / Cfg::R, a.B, a.nseg), block(Cfg::NT);
    auto k = scan3_bwd_kernel<IN_T, W, REV, AGG, ORD, DET>;
    const size_t smem = Cfg::smem_bytes;
    cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    k<<<grid, block, smem, st>>>(a);
    count_launch();
    return check_launch("selective_scan_bwd(v3)");
}

template <typename IN_T, bool AGG, bool DET = false> int dispatch_bwd3(const Bwd3Args &a, int W, bool rev, cudaStream_t st) {
    if (a.ord.kind != MMU_ORDER_ROWMAJOR) {         // fused scan order: z / dout / dz permuted by the kernel (never with rev)
        if (W == 1) return launch_bwd3<IN_T, 1, false, AGG, true, DET>(a, st);
        if (W == 2) return launch_bwd3<IN_T, 2, false, AGG, true, DET>(a, st);
        if (W == 3) return launch_bwd3<IN_T, 3, false, AGG, true, DET>(a, st);
        return launch_bwd3<IN_T, 4, false, AGG, true, DET>(a, st);
    }
#define MMU_B3(W_) (rev ? launch_bwd3<IN_T, W_, true, AGG, false, DET>(a, st) : launch_bwd3<IN_T, W_, false, AGG, false, DET>(a, st))
    if (W == 1) return MMU_B3(1);
    if (W == 2) return MMU_B3(2);
    if (W == 3) return MMU_B3(3);
    if (W == 8) return MMU_B3(8);
    return MMU_B3(4);
#undef MMU_B3
}

// the main pass; det != nullptr: the DET kernels into the slots, then the ordered reduces
template <typename IN_T> int run_bwd3_main(const Bwd3Args &a0, const mmu_scan_bwd_params *p, const Bwd3Plan &pl, const ScanDet *det,
                                           cudaStream_t st) {
    const bool rev = p->f.reverse != 0;
    if (det == nullptr) return dispatch_bwd3<IN_T, false>(a0, pl.W, rev, st);
    Bwd3Args a = a0;
    scan_det_args(a, *det);
    if (int rc = dispatch_bwd3<IN_T, false, true>(a, pl.W, rev, st)) return rc;
    return scan_det_reduce(p, *det, (a.D + 2 * pl.W - 1) / (2 * pl.W), pl.nseg, st);
}

template <typename IN_T> int run_bwd3(const mmu_scan_bwd_params *p, cudaStream_t st, const ScanDet *det) {
    const mmu_scan_fwd_params &f = p->f;
    const Bwd3Plan pl = plan_bwd3(f.batch, f.dim, f.seqlen, f.order != MMU_ORDER_ROWMAJOR);
    Bwd3Args a{};
    make_ordmap(a.ord, f.order, f.order_h, f.order_w, f.order_ns, f.seqlen);
    a.u = f.u, a.delta = f.delta, a.z = f.z, a.dout = p->dout, a.ysave = f.y, a.Bm = f.B, a.Cm = f.C;
    a.A = f.A, a.Dv = f.D, a.dbias = f.delta_bias, a.x = f.x;
    a.du = p->du, a.ddelta = p->ddelta, a.dz = p->dz;
    a.dA = p->dA, a.dB = p->dB, a.dC = p->dC, a.dD = p->dD, a.ddbias = p->ddelta_bias;
    a.u_bs = f.u_bs, a.u_ds = f.u_ds, a.dl_bs = f.delta_bs, a.dl_ds = f.delta_ds, a.z_bs = f.z_bs, a.z_ds = f.z_ds;
    a.g_bs = p->dout_bs, a.g_ds = p->dout_ds, a.y_bs = f.y_bs, a.y_ds = f.y_ds;
    a.B_bs = f.B_bs, a.B_ns = f.B_ns, a.C_bs = f.C_bs, a.C_ns = f.C_ns;
    a.du_bs = p->du_bs, a.du_ds = p->du_ds, a.ddl_bs = p->ddelta_bs, a.ddl_ds = p->ddelta_ds;
    a.dz_bs = p->dz_bs, a.dz_ds = p->dz_ds;
    a.dB_bs = p->dB_bs ? p->dB_bs : (int64_t)f.dstate * f.seqlen, a.dC_bs = p->dC_bs ? p->dC_bs : (int64_t)f.dstate * f.seqlen;
    a.dB_ns = p->dB_ns ? p->dB_ns : f.seqlen, a.dC_ns = p->dC_ns ? p->dC_ns : f.seqlen;
    a.B = f.batch, a.D = f.dim, a.L = f.seqlen, a.N = f.dstate;
    a.nseg = pl.nseg, a.cps = pl.cps, a.nchunks = pl.nchunks;
    a.nx = (f.seqlen + MMU_STATE_STRIDE - 1) / MMU_STATE_STRIDE;
    a.softplus = f.delta_softplus;
    const bool rev = f.reverse != 0;
#if MMU_TMA_TILE
    if constexpr (sizeof(IN_T) == 4) {
        if (int rc = encode_bc_map(a.tmB, f.B, f.seqlen, f.dstate, f.batch, f.B_ns, f.B_bs)) return rc;
        if (int rc = encode_bc_map(a.tmC, f.C, f.seqlen, f.dstate, f.batch, f.C_ns, f.C_bs)) return rc;
    }
#endif
    if (pl.nseg > 1 && pl.chain) {
        const size_t n_state = (size_t)a.B * a.D * pl.nseg * 16;
        const size_t n_flags = (size_t)a.B * ((a.D + 2 * pl.W - 1) / (2 * pl.W)) * pl.nseg + 1;
        const size_t need = align256(n_state * 4) + align256(n_flags * 4);
        if (f.workspace == nullptr || f.workspace_bytes < need)
            return set_error(MMU_ERR_WORKSPACE, "selective_scan_bwd: workspace %zu < %zu", f.workspace_bytes, need);
        char *w = static_cast<char *>(f.workspace);
        a.ein = reinterpret_cast<float *>(w);
        a.chain_flags = reinterpret_cast<int *>(w + align256(n_state * 4));
        a.chain_ticket = a.chain_flags + (n_flags - 1);
        cudaMemsetAsync(a.chain_flags, 0, n_flags * 4, st);
        return run_bwd3_main<IN_T>(a, p, pl, det, st);
    }
    if (pl.nseg > 1) {
        const size_t n_state = (size_t)a.B * a.D * pl.nseg * 16, n_row = (size_t)a.B * a.D * pl.nseg;
        const size_t need = 2 * align256(n_state * 4) + 2 * align256(n_row * 4);
        if (f.workspace == nullptr || f.workspace_bytes < need)
            return set_error(MMU_ERR_WORKSPACE, "selective_scan_bwd: workspace %zu < %zu", f.workspace_bytes, need);
        char *w = static_cast<char *>(f.workspace);
        a.seg_E = reinterpret_cast<float *>(w);
        float *ein = reinterpret_cast<float *>(w + align256(n_state * 4));
        a.seg_dsum = reinterpret_cast<float *>(w + 2 * align256(n_state * 4));
        a.ein = nullptr;
        int rc = dispatch_bwd3<IN_T, true>(a, pl.W, rev, st);
        if (rc) return rc;
        const int64_t tot = (int64_t)a.B * a.D * 16;
        scan3_bwd_chain_kernel<<<(unsigned)((tot + 127) / 128), 128, 0, st>>>(a.A, a.seg_E, a.seg_dsum, ein, a.B, a.D, a.N, pl.nseg);
        count_launch();
        rc = check_launch("scan3_bwd_chain");
        if (rc) return rc;
        a.ein = ein;
    }
    return run_bwd3_main<IN_T>(a, p, pl, det, st);
}


// ---- v4 host side (scan4_bwd.cuh): wide problems, rows in lanes; needs x saved every 8 tokens ---------------------------------
struct Bwd4Plan {
    int nseg, sps, nstage, nrg;
};

Bwd4Plan plan_bwd4(int B, int D, int L) {
    Bwd4Plan pl;
    pl.nstage = L / 8;
    pl.nrg = (D + kS4Rows - 1) / kS4Rows;
    const int wps = B * pl.nrg;                                          // warps per segment
    int nseg = (148 * env_int("MMU_V4_BWD_WPSM", 16) + wps - 1) / wps;   // about two waves of the 8 resident warps
    nseg = std::min(nseg, std::max(1, pl.nstage / 4));                   // at least 32 tokens per segment
    nseg = env_int("MMU_BWD_NSEG", nseg);
    nseg = std::max(1, std::min(nseg, std::min(pl.nstage, kS4MaxSeg)));
    pl.sps = (pl.nstage + nseg - 1) / nseg;
    pl.nseg = (pl.nstage + pl.sps - 1) / pl.sps;
    return pl;
}

template <typename IN_T> bool bwd4_eligible(const mmu_scan_bwd_params *p) {
    const mmu_scan_fwd_params &f = p->f;
    if (env_int("MMU_SCAN_V", 3) < 4 || env_int("MMU_BWD_V", 4) < 4) return false;
    if (f.x_stride != 8 || f.dstate != 16 || f.dim < env_int("MMU_V4_MIN_DIM", 64)) return false;
    if (reinterpret_cast<uintptr_t>(f.x) % 16 != 0) return false;
    if (f.seqlen > 8 && !f.x) return false;
    return bwd3_eligible<IN_T>(p);
}

template <typename IN_T> int run_bwd4(const mmu_scan_bwd_params *p, cudaStream_t st) {
    const mmu_scan_fwd_params &f = p->f;
    const Bwd4Plan pl = plan_bwd4(f.batch, f.dim, f.seqlen);
    Bwd4Args a{};
    a.u = f.u, a.delta = f.delta, a.z = f.z, a.dout = p->dout, a.ysave = f.y, a.Bm = f.B, a.Cm = f.C;
    a.A = f.A, a.Dv = f.D, a.dbias = f.delta_bias, a.x = f.x;
    a.du = p->du, a.ddelta = p->ddelta, a.dz = p->dz;
    a.dA = p->dA, a.dB = p->dB, a.dC = p->dC, a.dD = p->dD, a.ddbias = p->ddelta_bias;
    a.u_bs = f.u_bs, a.u_ds = f.u_ds, a.dl_bs = f.delta_bs, a.dl_ds = f.delta_ds, a.z_bs = f.z_bs, a.z_ds = f.z_ds;
    a.g_bs = p->dout_bs, a.g_ds = p->dout_ds, a.y_bs = f.y_bs, a.y_ds = f.y_ds;
    a.B_bs = f.B_bs, a.B_ns = f.B_ns, a.C_bs = f.C_bs, a.C_ns = f.C_ns;
    a.du_bs = p->du_bs, a.du_ds = p->du_ds, a.ddl_bs = p->ddelta_bs, a.ddl_ds = p->ddelta_ds;
    a.dz_bs = p->dz_bs, a.dz_ds = p->dz_ds;
    a.dB_bs = p->dB_bs ? p->dB_bs : (int64_t)f.dstate * f.seqlen, a.dC_bs = p->dC_bs ? p->dC_bs : (int64_t)f.dstate * f.seqlen;
    a.dB_ns = p->dB_ns ? p->dB_ns : f.seqlen, a.dC_ns = p->dC_ns ? p->dC_ns : f.seqlen;
    a.B = f.batch, a.D = f.dim, a.L = f.seqlen, a.N = f.dstate;
    a.nseg = pl.nseg, a.sps = pl.sps, a.nstage = pl.nstage, a.nrg = pl.nrg;
    a.nx = (f.seqlen + 7) / 8;
    a.softplus = f.delta_softplus;
    const bool rev = f.reverse != 0;
    if (pl.nseg > 1) {
        const size_t n_state = (size_t)a.B * a.D * pl.nseg * 16, n_row = (size_t)a.B * a.D * pl.nseg;
        const size_t need = 2 * align256(n_state * 4) + 2 * align256(n_row * 4);
        if (f.workspace == nullptr || f.workspace_bytes < need)
            return set_error(MMU_ERR_WORKSPACE, "selective_scan_bwd: workspace %zu < %zu", f.workspace_bytes, need);
        char *w = static_cast<char *>(f.workspace);
        a.seg_E = reinterpret_cast<float *>(w);
        float *ein = reinterpret_cast<float *>(w + align256(n_state * 4));
        a.seg_dsum = reinterpret_cast<float *>(w + 2 * align256(n_state * 4));
        a.ein = nullptr;
        a.nitems = a.B * a.nrg * (pl.nseg - 1);
        {
            using Sm = S4Fwd<IN_T, 3>;
            const size_t smem = (size_t)kS4W * Sm::kWarpBytes;
            auto k = rev ? scan4_bwd_agg_kernel<IN_T, true> : scan4_bwd_agg_kernel<IN_T, false>;
            cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            k<<<(a.nitems + kS4W - 1) / kS4W, 32 * kS4W, smem, st>>>(a);
            count_launch();
            int rc = check_launch("selective_scan_bwd(v4 aggregates)");
            if (rc) return rc;
        }
        const int64_t tot = (int64_t)a.B * a.D * 16;
        scan3_bwd_chain_kernel<<<(unsigned)((tot + 127) / 128), 128, 0, st>>>(a.A, a.seg_E, a.seg_dsum, ein, a.B, a.D, a.N, pl.nseg);
        count_launch();
        int rc = check_launch("scan3_bwd_chain");
        if (rc) return rc;
        a.ein = ein;
    }
    a.nitems = a.B * a.nrg * pl.nseg;
    using Sm = S4Bwd<IN_T>;
    const size_t smem = (size_t)kS4W * Sm::kWarpBytes;
    auto k = rev ? scan4_bwd_kernel<IN_T, true> : scan4_bwd_kernel<IN_T, false>;
    cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    k<<<(a.nitems + kS4W - 1) / kS4W, 32 * kS4W, smem, st>>>(a);
    count_launch();
    return check_launch("selective_scan_bwd(v4)");
}

template <typename IN_T> struct HasV3 { static constexpr bool value = false; };
template <> struct HasV3<float> { static constexpr bool value = true; };
template <> struct HasV3<__nv_bfloat16> { static constexpr bool value = true; };

template <typename IN_T> int run_bwd(const mmu_scan_bwd_params *p, cudaStream_t st, const ScanDet *det) {
    if (p->f.order != MMU_ORDER_ROWMAJOR) {      // fused scan order: only on the dstate <= 16 kernels, only for the fusable maps
        const mmu_scan_fwd_params &f = p->f;
        bool ok = f.order != MMU_ORDER_FLIP && !f.reverse && ordmap_fusable(f.order, f.order_h, f.order_w, f.order_ns, f.seqlen) &&
                  (f.x_stride == 0 || f.x_stride == MMU_STATE_STRIDE);
        if constexpr (HasV3<IN_T>::value) ok = ok && bwd3_eligible<IN_T>(p);
        else ok = false;
        if (!ok)
            return set_error(MMU_ERR_UNSUPPORTED, "selective_scan_bwd: scan order %d (H=%d W=%d nslices=%d) cannot be fused for this problem "
                             "(see mmu_scan_order_fusable)", f.order, f.order_h, f.order_w, f.order_ns);
        if constexpr (HasV3<IN_T>::value) return run_bwd3<IN_T>(p, st, det);
    }
    if constexpr (HasV3<IN_T>::value) {
        if (det == nullptr && bwd4_eligible<IN_T>(p)) return run_bwd4<IN_T>(p, st);      // opt-in experiment: never deterministic
    }
    if (p->f.x_stride != 0 && p->f.x_stride != MMU_STATE_STRIDE)
        return set_error(MMU_ERR_UNSUPPORTED, "selective_scan_bwd: x_stride %d needs the wide (v4) kernels (dim >= 64, dstate <= 16, "
                         "seqlen %% 8 == 0, 16-byte aligned rows)", p->f.x_stride);
    if constexpr (HasV3<IN_T>::value) {
        if (bwd3_eligible<IN_T>(p)) return run_bwd3<IN_T>(p, st, det);
    }
    const mmu_scan_fwd_params &f = p->f;
    const BwdPlan pl = plan_bwd(f.batch, f.dim, f.seqlen);
    BwdArgs a{};
    a.u = f.u, a.delta = f.delta, a.z = f.z, a.dout = p->dout, a.Bm = f.B, a.Cm = f.C;
    a.A = f.A, a.Dv = f.D, a.dbias = f.delta_bias, a.x = f.x;
    a.du = p->du, a.ddelta = p->ddelta, a.dz = p->dz;
    a.dA = p->dA, a.dB = p->dB, a.dC = p->dC, a.dD = p->dD, a.ddbias = p->ddelta_bias;
    a.u_bs = f.u_bs, a.u_ds = f.u_ds, a.dl_bs = f.delta_bs, a.dl_ds = f.delta_ds, a.z_bs = f.z_bs, a.z_ds = f.z_ds;
    a.g_bs = p->dout_bs, a.g_ds = p->dout_ds, a.B_bs = f.B_bs, a.B_ns = f.B_ns, a.C_bs = f.C_bs, a.C_ns = f.C_ns;
    a.du_bs = p->du_bs, a.du_ds = p->du_ds, a.ddl_bs = p->ddelta_bs, a.ddl_ds = p->ddelta_ds;
    a.dz_bs = p->dz_bs, a.dz_ds = p->dz_ds;
    a.dB_bs = p->dB_bs ? p->dB_bs : (int64_t)f.dstate * f.seqlen, a.dC_bs = p->dC_bs ? p->dC_bs : (int64_t)f.dstate * f.seqlen;
    a.dB_ns = p->dB_ns ? p->dB_ns : f.seqlen, a.dC_ns = p->dC_ns ? p->dC_ns : f.seqlen;
    a.B = f.batch, a.D = f.dim, a.L = f.seqlen, a.N = f.dstate, a.Ne = (f.dstate + 1) & ~1;
    a.nseg = pl.nseg, a.cps = pl.cps, a.nchunks = pl.nchunks;
    a.nx = (f.seqlen + MMU_STATE_STRIDE - 1) / MMU_STATE_STRIDE;
    a.softplus = f.delta_softplus, a.reverse = f.reverse;
    const bool rev = f.reverse != 0;
    const int L = f.seqlen;
    a.vec_mask = (quad_ok<IN_T>(f.u, f.u_bs, f.u_ds, L, rev) ? 1u : 0u) |
                 (quad_ok<IN_T>(f.delta, f.delta_bs, f.delta_ds, L, rev) ? 2u : 0u) |
                 ((f.z && quad_ok<IN_T>(f.z, f.z_bs, f.z_ds, L, rev)) ? 4u : 0u) |
                 (quad_ok<IN_T>(p->dout, p->dout_bs, p->dout_ds, L, rev) ? 8u : 0u) |
                 (quad_ok<IN_T>(f.B, f.B_bs, f.B_ns, L, rev) ? 16u : 0u) |
                 (quad_ok<IN_T>(f.C, f.C_bs, f.C_ns, L, rev) ? 32u : 0u) |
                 (quad_ok<IN_T>(p->du, p->du_bs, p->du_ds, L, rev) ? 64u : 0u) |
                 (quad_ok<IN_T>(p->ddelta, p->ddelta_bs, p->ddelta_ds, L, rev) ? 128u : 0u) |
                 ((p->dz && quad_ok<IN_T>(p->dz, p->dz_bs, p->dz_ds, L, rev)) ? 256u : 0u);
    const unsigned need = 1u | 2u | 8u | 16u | 32u | (f.z ? 4u : 0u);
    if ((a.vec_mask & need) == need && a.Ne <= 16 && env_int("MMU_NO_PREFETCH", 0) == 0) a.vec_mask |= 0x8000u;
    if (pl.nseg > 1) {
        const size_t n_state = (size_t)a.B * a.D * pl.nseg * a.Ne, n_row = (size_t)a.B * a.D * pl.nseg;
        const size_t need = 2 * align256(n_state * 4) + 2 * align256(n_row * 4);
        if (f.workspace == nullptr || f.workspace_bytes < need)
            return set_error(MMU_ERR_WORKSPACE, "selective_scan_bwd: workspace %zu < %zu", f.workspace_bytes, need);
        char *w = static_cast<char *>(f.workspace);
        a.seg_dh = reinterpret_cast<float *>(w);
        float *dhin = reinterpret_cast<float *>(w + align256(n_state * 4));
        a.seg_dsum = reinterpret_cast<float *>(w + 2 * align256(n_state * 4));
        a.seg_dfirst = reinterpret_cast<float *>(w + 2 * align256(n_state * 4) + align256(n_row * 4));
        a.dhin = nullptr;
        int rc = dispatch_bwd<IN_T>(pl.cfg, a, true, st);
        if (rc) return rc;
        const int64_t tot = (int64_t)a.B * a.D * a.Ne;
        scan_bwd_chain_kernel<<<(unsigned)((tot + 127) / 128), 128, 0, st>>>(a.A, a.seg_dh, a.seg_dsum, a.seg_dfirst, dhin,
                                                                             a.B, a.D, a.N, a.Ne, pl.nseg);
        count_launch();
        rc = check_launch("scan_bwd_chain");
        if (rc) return rc;
        a.dhin = dhin;
    }
    if (det == nullptr) return dispatch_bwd<IN_T>(pl.cfg, a, false, st);
    scan_det_args(a, *det);
    if (int rc = dispatch_bwd<IN_T>(pl.cfg, a, false, st, true)) return rc;
    return scan_det_reduce(p, *det, (a.D + pl.R - 1) / pl.R, pl.nseg, st);
}

ScanDetBound scan_det_bound(int B, int D, int L) {
    const Bwd3Plan a = plan_bwd3(B, D, L, false), o = plan_bwd3(B, D, L, true);
    const BwdPlan v1 = plan_bwd(B, D, L);
    ScanDetBound bd;
    bd.nrg = std::max({(D + 2 * a.W - 1) / (2 * a.W), (D + 2 * o.W - 1) / (2 * o.W), (D + v1.R - 1) / v1.R});
    bd.nseg = std::max({a.nseg, o.nseg, v1.nseg});
    return bd;
}

}  // namespace
}  // namespace mmu

extern "C" size_t mmu_selective_scan_bwd_workspace(int32_t batch, int32_t dim, int32_t seqlen, int32_t dstate) {
    const int Ne = dstate <= 16 ? 16 : ((dstate + 1) & ~1);
    const int nchunks = (seqlen + 63) / 64;
    const size_t nseg = (size_t)std::max(1, std::min(nchunks, std::max(64, mmu::env_int("MMU_BWD_NSEG", 1))));
    const size_t n_state = (size_t)batch * dim * nseg * Ne, n_row = (size_t)batch * dim * nseg;
    size_t need = 2 * mmu::align256(n_state * 4) + 2 * mmu::align256(n_row * 4);
    if (dstate <= 16 && seqlen % 8 == 0 && seqlen >= 8) {   // the wide (v4) plan
        const mmu::Bwd4Plan pl = mmu::plan_bwd4(batch, dim, seqlen);
        const size_t n4 = (size_t)batch * dim * pl.nseg * 16, r4 = (size_t)batch * dim * pl.nseg;
        need = std::max(need, 2 * mmu::align256(n4 * 4) + 2 * mmu::align256(r4 * 4));
    }
    return need;
}

extern "C" int32_t mmu_scan_state_stride(int32_t batch, int32_t dim, int32_t seqlen, int32_t dstate, int32_t dtype) {
    using namespace mmu;
    (void)batch;
    const bool v4 = env_int("MMU_SCAN_V", 3) >= 4 && env_int("MMU_BWD_V", 4) >= 4 && dim >= env_int("MMU_V4_MIN_DIM", 64) &&
                    dstate == 16 && seqlen % 8 == 0 && (dtype == MMU_F32 || dtype == MMU_BF16);
    return v4 ? 8 : MMU_STATE_STRIDE;
}

namespace mmu {
namespace {
int scan_bwd_entry(const mmu_scan_bwd_params *p, const ScanDet *det, void *stream);
}
}  // namespace mmu

extern "C" size_t mmu_selective_scan_bwd_det_workspace(int32_t batch, int32_t dim, int32_t seqlen, int32_t dstate) {
    if (batch <= 0 || dim <= 0 || seqlen <= 0 || dstate <= 0) return 0;
    return mmu::scan_det_carve(batch, dim, seqlen, dstate, nullptr, nullptr);
}

extern "C" int mmu_selective_scan_bwd_det(const mmu_scan_bwd_params *p, void *ws, size_t ws_bytes, void *stream) {
    using namespace mmu;
    if (p == nullptr) return set_error(MMU_ERR_INVALID, "selective_scan_bwd_det: null params");
    const mmu_scan_fwd_params &f = p->f;
    const size_t need = mmu_selective_scan_bwd_det_workspace(f.batch, f.dim, f.seqlen, f.dstate);
    if (need == 0) return set_error(MMU_ERR_INVALID, "selective_scan_bwd_det: empty shape");
    if (int rc = det_ws_check(ws, ws_bytes, need, "selective_scan_bwd_det")) return rc;
    ScanDet d;
    scan_det_carve(f.batch, f.dim, f.seqlen, f.dstate, static_cast<char *>(ws), &d);
    return scan_bwd_entry(p, &d, stream);
}

extern "C" int mmu_selective_scan_bwd(const mmu_scan_bwd_params *p, void *stream) { return mmu::scan_bwd_entry(p, nullptr, stream); }

namespace mmu {
namespace {
int scan_bwd_entry(const mmu_scan_bwd_params *p, const ScanDet *det, void *stream) {
    if (p == nullptr) return set_error(MMU_ERR_INVALID, "selective_scan_bwd: null params");
    const mmu_scan_fwd_params &f = p->f;
    if (f.batch <= 0 || f.dim <= 0 || f.seqlen <= 0 || f.dstate <= 0)
        return set_error(MMU_ERR_INVALID, "selective_scan_bwd: empty shape");
    if (f.dstate > 256) return set_error(MMU_ERR_INVALID, "selective_scan only supports state dimension <= 256");
    if (!f.u || !f.delta || !f.A || !f.B || !f.C || !p->dout || !p->du || !p->ddelta || !p->dA || !p->dB || !p->dC)
        return set_error(MMU_ERR_INVALID, "selective_scan_bwd: null tensor pointer");
    if (f.seqlen > (f.x_stride ? f.x_stride : MMU_STATE_STRIDE) && !f.x)
        return set_error(MMU_ERR_INVALID, "selective_scan_bwd: x (saved states from the forward) is required");
    if ((f.z != nullptr) != (p->dz != nullptr)) return set_error(MMU_ERR_INVALID, "selective_scan_bwd: dz must be given iff z is");
    if ((f.D != nullptr && !p->dD) || (f.delta_bias != nullptr && !p->ddelta_bias))
        return set_error(MMU_ERR_INVALID, "selective_scan_bwd: dD / ddelta_bias missing");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (f.dtype) {
        case MMU_F32: return run_bwd<float>(p, st, det);
        case MMU_BF16: return run_bwd<__nv_bfloat16>(p, st, det);
        case MMU_F16: return run_bwd<__half>(p, st, det);
        default: return set_error(MMU_ERR_UNSUPPORTED, "selective_scan_bwd: dtype %d", f.dtype);
    }
}
}  // namespace
}  // namespace mmu
