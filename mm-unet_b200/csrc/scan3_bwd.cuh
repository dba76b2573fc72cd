// Selective scan backward, v3 kernel (dstate <= 16, seqlen % 8 == 0, 16-byte aligned rows).  Recompute based: the L x N state is
// never materialised.  Math: SURVEY.md Appendix A; replaces selective_scan_bwd_kernel (selective_scan_bwd_kernel.cuh:75-489).
//
// Geometry as the forward (scan3.cuh): a lane owns 8 tokens of two rows (packed in the halves of FFMA2), 32 lanes = one
// 256-token chunk of a row pair; chunks are walked last -> first.  Per chunk and state n:
//   forward recompute   a_i = exp(delta_i A), H = a H + delta_i u_i B_i from zero; the forward kernel saved the true state every
//                       64 tokens (x), so an 8-lane shuffle scan seeded from x gives each lane its entering state hs, then h_i;
//   reverse             "e form": e_i = a_i (C_i dy_i + e_{i+1}) with dh_i = C_i dy_i + e_{i+1}; it shares its multipliers with
//                       the forward, so the lanes' (prod a, e) close with one 32-lane shuffle scan plus a chunk carry;
//   contributions       dB, dC (summed over the two rows in registers, then red.global.add.v4), S1 = sum_n dh B,
//                       S2 = sum_n dh a h_prev A (registers, per token), dA (lane-private shared accumulators).
// The per (row, token) epilogue turns S1, S2 into du, ddelta, and uses the pre-gate y saved by the forward for dz.
#pragma once
#include <type_traits>

#include "scan3.cuh"

namespace mmu {

struct Bwd3Args {
    const void *u, *delta, *z, *dout, *ysave, *Bm, *Cm;
    const float *A, *Dv, *dbias, *x;
    void *du, *ddelta, *dz;
    float *dA, *dB, *dC, *dD, *ddbias;
    float *seg_E, *seg_dsum;       // AGG pass outputs
    float *ein;                    // reverse carry entering each segment (main pass, nseg > 1); written by the chained kernel
    int *chain_flags, *chain_ticket;   // chained segments (no aggregate pass): carry-ready flags [group][seg], work ticket
    int64_t u_bs, u_ds, dl_bs, dl_ds, z_bs, z_ds, g_bs, g_ds, y_bs, y_ds, B_bs, B_ns, C_bs, C_ns;
    int64_t du_bs, du_ds, ddl_bs, ddl_ds, dz_bs, dz_ds;
    int64_t dB_bs, dC_bs, dB_ns, dC_ns;   // batch / state strides of dB / dC (elements)
    int B, D, L, N;
    int nseg, cps, nchunks, nx;
    int softplus;
    OrdMap ord;                    // ORD kernels: z, dout and dz live at ord(l) (natural token order), everything else at l
    int64_t det_rgs;               // DET kernels: row-group stride of the dB / dC slots (dB, dC point at the slots)
#if MMU_TMA_TILE
    alignas(64) unsigned char tmB[128], tmC[128];   // CUtensorMap of B and C (see Fwd3Args)
#endif
};

template <typename IN_T, int W> struct Bwd3Cfg {
    static constexpr int LPR = 32;
    static constexpr bool kF32 = sizeof(IN_T) == 4;
    static constexpr int CH = LPR * kS3T, R = 2 * W, NT = 32 * W, NRP = W;
    static constexpr int NCK = CH / MMU_STATE_STRIDE;                     // 4 saved states per chunk
    static constexpr int kRawBytes = kF32 ? 0 : 2 * 16 * CH * 2;
    static constexpr int NQ = Raw8<IN_T>::kQuads;
    static constexpr int kLandBytes = 5 * 2 * NQ * NT * 16;               // u | delta | z | dout | y : [tensor][row][quad][thread] x 16 B
    static constexpr int kZfBytes = 2 * 2 * NT * 16;                      // dz factor, fp32: [row][quad][thread] x 16 B
    static constexpr int kDABytes = 16 * W * 8 * 8;                       // dA partials [state][warp][8 lanes] float2
    static constexpr int kSlabBytes = 2 * W * 2 * 2 * 32 * 16;            // dB | dC partials of one state: [buf][warp][tensor][quad][lane] float4
    static constexpr int kSeedBytes = 2 * W * NCK * 16 * 8;               // x seeds [buf][warp][ck][state] float2
    static constexpr int kTabBytes = 2 * NRP * 16 * 8;                    // A*log2e | e carry
    static constexpr size_t smem_bytes = (size_t)BcTile<LPR>::kBytes + kRawBytes + kLandBytes + kZfBytes + kDABytes + kSlabBytes + kSeedBytes + kTabBytes;
};

__device__ __forceinline__ void red_add_v4(float *p, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// ORD: fused scan order (NSLICES / TWOROW): z and dout are gathered, dz is scattered through p.ord (ord_issue8 / ord_store8 in
// scan3.cuh); never together with REV.
// DET (deterministic mode, main pass only): no float atomics.  dB / dC / dA / dD / ddbias point at slots of the caller's workspace:
// the CTA STORES its slab sums to dB / dC + row group * det_rgs (each (row group, batch, state, token) has exactly one writer), and
// dA / dD / ddbias to [batch][segment][row](x dstate).  The ordered reduce (det_reduce.cu) adds the slots to the real outputs.
template <typename IN_T, int W, bool REV, bool AGG, bool ORD = false, bool DET = false>
__global__ void __launch_bounds__(32 * W, AGG ? 1 : 8 / W) scan3_bwd_kernel(const __grid_constant__ Bwd3Args p) {
    static_assert(!ORD || !REV, "ordered gate / output gradient: forward direction only");
    using Cfg = Bwd3Cfg<IN_T, W>;
    constexpr int LPR = 32;
    constexpr bool kTmaTile = MMU_TMA_TILE != 0 && sizeof(IN_T) == 4 && LPR == 32;   // B/C tile by two tensor-map copies (scan3_fwd.cuh)
    using Tl = typename std::conditional<kTmaTile, BcTileDense<LPR>, BcTile<LPR>>::type;
    constexpr int CH = Cfg::CH, R = Cfg::R, NT = Cfg::NT, NRP = Cfg::NRP, T = kS3T, NQ = Cfg::NQ, NCK = Cfg::NCK;
    constexpr int EPQ = 16 / (int)sizeof(IN_T);
    constexpr bool kF32 = Cfg::kF32;
    const int tid = threadIdx.x, warp = tid >> 5, j = tid & 31;
    const int D = p.D, L = p.L, N = p.N;
    const bool has_z = p.z != nullptr, sp = p.softplus != 0;
    // Work item.  Plain launch: (row group, batch, segment) = blockIdx.  Chained launch (wide problems whose CTAs do not fill
    // whole waves): segments of one row group are separate CTAs, LAST segment first; a CTA takes its item from a ticket
    // counter, so the CTA that owns the segment to its right always started earlier and a spin-wait on its carry cannot
    // deadlock.  No aggregate pass is needed: the forward states come from x, only e flows between segments.
    __shared__ int s_item;
    const bool chained = !AGG && p.chain_ticket != nullptr;
    int bx = blockIdx.x, b = blockIdx.y, seg = blockIdx.z;
    int gidx = 0;
    if (chained) {
        if (tid == 0) s_item = atomicAdd(p.chain_ticket, 1);
        __syncthreads();
        const int G = gridDim.x * gridDim.y;
        gidx = s_item % G;
        seg = p.nseg - 1 - s_item / G;
        bx = gidx % gridDim.x, b = gidx / gridDim.x;
    }
    const int row0 = bx * R;
    const int NS = (N + 1) & ~1;           // states are walked two at a time (a padding state has A = B = C = 0)

    extern __shared__ __align__(128) unsigned char smem_raw[];
    unsigned char *s_tile = smem_raw;
    unsigned char *s_rawbc = s_tile + BcTile<LPR>::kBytes;
    unsigned char *s_land = s_rawbc + Cfg::kRawBytes;
    unsigned char *s_zf = s_land + Cfg::kLandBytes;
    float2 *s_dA = reinterpret_cast<float2 *>(s_zf + Cfg::kZfBytes);       // [16][W][8]
    float4 *s_slab = reinterpret_cast<float4 *>(s_zf + Cfg::kZfBytes + Cfg::kDABytes);   // [2][W][2][2][32]
    float2 *s_seed = reinterpret_cast<float2 *>(s_zf + Cfg::kZfBytes + Cfg::kDABytes + Cfg::kSlabBytes);   // [2][W][NCK][16]
    float2 *s_A = s_seed + 2 * W * NCK * 16;                               // [NRP][16]  A*log2e of (row A, row B)
    float2 *s_ec = s_A + NRP * 16;                                         // [NRP][16]  e entering the chunk from the right

    for (int i = tid; i < (int)((BcTile<LPR>::kBytes + Cfg::kRawBytes + Cfg::kLandBytes + Cfg::kZfBytes + Cfg::kDABytes + Cfg::kSlabBytes + Cfg::kSeedBytes) / 16); i += NT)
        reinterpret_cast<uint4 *>(smem_raw)[i] = make_uint4(0u, 0u, 0u, 0u);
    if (chained && seg + 1 < p.nseg) {
        if (tid == 0) {
            volatile int *f = p.chain_flags + gidx * p.nseg + seg;
            while (*f == 0) __nanosleep(200);
            __threadfence();
        }
        __syncthreads();
    }
    for (int i = tid; i < NRP * 16; i += NT) {
        const int g = i >> 4, n = i & 15;
        float a[2], e[2];
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int row = row0 + 2 * g + r;
            const bool ok = row < D && n < N;
            a[r] = ok ? p.A[(int64_t)row * N + n] * kLog2e : 0.f;
            e[r] = 0.f;
            if (!AGG && ok && p.ein != nullptr && seg + 1 < p.nseg) e[r] = __ldcg(p.ein + (((int64_t)b * D + row) * p.nseg + seg) * 16 + n);
        }
        s_A[i] = make_float2(a[0], a[1]);
        s_ec[i] = make_float2(e[0], e[1]);
    }

    // ---- my two rows; chunks are walked from c_end-1 down to c_begin ------------------------------------------------------
    const int rowA = row0 + 2 * warp;
    const int c_begin = seg * p.cps, c_end = min(p.nchunks, c_begin + p.cps);
    int tl = (c_end - 1) * CH + T * j;                  // first logical token of my 8 in the current chunk
    constexpr int STEP = REV ? CH : -CH;                // memory step to the next (= previous in time) chunk
    // Every pointer starts ONE STEP BEHIND and is advanced just before it is used: a cp.async / store keeps its address
    // registers busy until it has been accepted by the memory pipe, and advancing them right AFTER the access (the natural
    // form) stalled on that release at the top of every chunk (long-scoreboard samples on the pointer updates in ncu).
    const int mo0 = (REV ? L - T - tl : tl) - STEP;
    bool row_ok[2];
    const IN_T *u_p[2], *d_p[2], *z_p[2], *g_p[2], *y_p[2];     // prefetch pointers
    IN_T *du_p[2], *dd_p[2], *dz_p[2];                            // output pointers (current chunk)
    float bias[2], Dsk[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        row_ok[r] = rowA + r < D;
        const int row = min(rowA + r, D - 1);
        u_p[r] = reinterpret_cast<const IN_T *>(p.u) + (int64_t)b * p.u_bs + (int64_t)row * p.u_ds + mo0;
        d_p[r] = reinterpret_cast<const IN_T *>(p.delta) + (int64_t)b * p.dl_bs + (int64_t)row * p.dl_ds + mo0;
        g_p[r] = reinterpret_cast<const IN_T *>(p.dout) + (int64_t)b * p.g_bs + (int64_t)row * p.g_ds + mo0;
        z_p[r] = has_z ? reinterpret_cast<const IN_T *>(p.z) + (int64_t)b * p.z_bs + (int64_t)row * p.z_ds + mo0 : nullptr;
        y_p[r] = has_z ? reinterpret_cast<const IN_T *>(p.ysave) + (int64_t)b * p.y_bs + (int64_t)row * p.y_ds + mo0 : nullptr;
        du_p[r] = AGG ? nullptr : reinterpret_cast<IN_T *>(p.du) + (int64_t)b * p.du_bs + (int64_t)row * p.du_ds + mo0;
        dd_p[r] = AGG ? nullptr : reinterpret_cast<IN_T *>(p.ddelta) + (int64_t)b * p.ddl_bs + (int64_t)row * p.ddl_ds + mo0;
        dz_p[r] = (AGG || !has_z) ? nullptr : reinterpret_cast<IN_T *>(p.dz) + (int64_t)b * p.dz_bs + (int64_t)row * p.dz_ds + mo0;
        bias[r] = p.dbias != nullptr ? p.dbias[row] : 0.f;
        Dsk[r] = p.Dv != nullptr ? p.Dv[row] : 0.f;
    }
    [[maybe_unused]] const IN_T *z_row[2], *g_row[2];
    [[maybe_unused]] IN_T *dz_row[2];
    if constexpr (ORD) {
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            const int row = min(rowA + r, D - 1);
            z_row[r] = has_z ? reinterpret_cast<const IN_T *>(p.z) + (int64_t)b * p.z_bs + (int64_t)row * p.z_ds : nullptr;
            g_row[r] = reinterpret_cast<const IN_T *>(p.dout) + (int64_t)b * p.g_bs + (int64_t)row * p.g_ds;
            dz_row[r] = (AGG || !has_z) ? nullptr : reinterpret_cast<IN_T *>(p.dz) + (int64_t)b * p.dz_bs + (int64_t)row * p.dz_ds;
        }
    }
    [[maybe_unused]] int tin = tl + CH;      // ORD: first logical token of my 8 in the chunk being prefetched (one step behind, like the pointers)
    const IN_T *B_b = reinterpret_cast<const IN_T *>(p.Bm) + (int64_t)b * p.B_bs;
    const IN_T *C_b = reinterpret_cast<const IN_T *>(p.Cm) + (int64_t)b * p.C_bs;
    float *dB_b = AGG ? nullptr : p.dB + (int64_t)b * p.dB_bs + (DET ? (int64_t)bx * p.det_rgs : 0);
    float *dC_b = AGG ? nullptr : p.dC + (int64_t)b * p.dC_bs + (DET ? (int64_t)bx * p.det_rgs : 0);

    bool ge_up[3], ge_dn[5];
#pragma unroll
    for (int s = 0; s < 3; ++s) ge_up[s] = (j & 7) >= (1 << s);
#pragma unroll
    for (int s = 0; s < 5; ++s) ge_dn[s] = j + (1 << s) < 32;
    const int qa = REV ? 2 * (LPR - 1 - j) : 2 * j;
    const unsigned char *tile = s_tile + Tl::quad_off(qa);
    const unsigned s_tile_u32 = smem_u32(s_tile), s_raw_u32 = smem_u32(s_rawbc);
    const unsigned s_land_u32 = smem_u32(s_land) + tid * 16;
    const unsigned char *s_land_t = s_land + tid * 16;
    unsigned char *s_zf_t = s_zf + tid * 16;
    float2 dDacc = make_float2(0.f, 0.f), dbacc = make_float2(0.f, 0.f);
    float dsum[2] = {0.f, 0.f};

    __shared__ __align__(8) unsigned long long s_mbar;       // tensor-map variant only
    const unsigned mbar = smem_u32(&s_mbar);
    [[maybe_unused]] unsigned tile_phase = 0;
    if constexpr (kTmaTile) {
        if (tid == 0) {
            mbar_init(mbar, 1);
            fence_mbar_init();
        }
    }
    auto issue_tile = [&](int c) {
#if MMU_TMA_TILE
        if constexpr (kTmaTile) {
            if (tid == 0) {
                const int m0 = REV ? L - (c + 1) * CH : c * CH;
                fence_proxy_async();
                mbar_arrive_expect_tx(mbar, 2u * 16u * CH * 4u);
                tma_tile_3d(s_tile_u32, p.tmB, m0, 0, b, mbar);
                tma_tile_3d(s_tile_u32 + 16 * Tl::kRowBytes, p.tmC, m0, 0, b, mbar);
            }
            return;
        }
#endif
        if constexpr (kF32) {
            tile_async_f32<LPR, NT, REV, true>(s_tile_u32, reinterpret_cast<const float *>(B_b), reinterpret_cast<const float *>(C_b), p.B_ns,
                                               p.C_ns, N, c * CH, L, tid);
        } else {
            raw_async_bf16<LPR, NT, REV, true>(s_raw_u32, reinterpret_cast<const __nv_bfloat16 *>(B_b),
                                               reinterpret_cast<const __nv_bfloat16 *>(C_b), p.B_ns, p.C_ns, N, c * CH, L, tid);
        }
    };
    // landing slots: tensor 0 u, 1 delta, 2 z, 3 dout, 4 y
    auto issue_in = [&](bool in_seq) {      // move the prefetch pointers on to the next chunk, then fetch its u, delta, z, dout, y
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            u_p[r] += STEP, d_p[r] += STEP, g_p[r] += STEP;
            if (has_z) z_p[r] += STEP;
            if (!AGG && has_z) y_p[r] += STEP;
        }
        if constexpr (ORD) tin -= CH;
        if (in_seq) {
#pragma unroll
            for (int r = 0; r < 2; ++r)
#pragma unroll
                for (int q = 0; q < NQ; ++q) {
                    cp_async16(s_land_u32 + ((1 * 2 + r) * NQ + q) * NT * 16, d_p[r] + q * EPQ);
                    if (!ORD) cp_async16(s_land_u32 + ((3 * 2 + r) * NQ + q) * NT * 16, g_p[r] + q * EPQ);
                    if (!AGG) cp_async16(s_land_u32 + ((0 * 2 + r) * NQ + q) * NT * 16, u_p[r] + q * EPQ);
                    if (!ORD && has_z) cp_async16(s_land_u32 + ((2 * 2 + r) * NQ + q) * NT * 16, z_p[r] + q * EPQ);
                    if (!AGG && has_z) cp_async16(s_land_u32 + ((4 * 2 + r) * NQ + q) * NT * 16, y_p[r] + q * EPQ);
                }
            if constexpr (ORD) {
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    ord_issue8<IN_T>(p.ord, tin, g_row[r], s_land_u32 + ((3 * 2 + r) * NQ) * NT * 16, s_land_u32 + ((3 * 2 + r) * NQ + NQ - 1) * NT * 16);
                    if (has_z)
                        ord_issue8<IN_T>(p.ord, tin, z_row[r], s_land_u32 + ((2 * 2 + r) * NQ) * NT * 16, s_land_u32 + ((2 * 2 + r) * NQ + NQ - 1) * NT * 16);
                }
            }
        }
    };
    // ordered tensor `which` (2 = z, 3 = dout), row r -> logical token order
    auto load_ord8 = [&](int which, int r, int t0, float (&v)[T]) {
        uint4 q[NQ];
#pragma unroll
        for (int k = 0; k < NQ; ++k) q[k] = *reinterpret_cast<const uint4 *>(s_land_t + ((which * 2 + r) * NQ + k) * NT * 16);
        float e[8];
        Raw8<IN_T>::unpack(q, e);
        ord_to_tokens(p.ord, t0, e, v);
    };
    auto load_land = [&](int which, int r, float (&v)[T]) {
        uint4 q[NQ];
#pragma unroll
        for (int k = 0; k < NQ; ++k) q[k] = *reinterpret_cast<const uint4 *>(s_land_t + ((which * 2 + r) * NQ + k) * NT * 16);
        float e[8];
        Raw8<IN_T>::unpack(q, e);
        order8<REV>(e, v);
    };
    // x seeds of chunk c: state entering the chunk's k-th 64-token block, k = 0..3  ->  s_seed[buf][warp][k][n] (row A, row B)
    const unsigned s_seed_u32 = smem_u32(s_seed);
    auto load_seeds = [&](int c, int buf) {       // asynchronous: part of the chunk's cp.async group
        if (AGG) return;
#pragma unroll
        for (int it = 0; it < NCK * 16 / 32; ++it) {
            const int e = j + 32 * it, ck = e >> 4, n = e & 15;
            const int kx = c * NCK + ck - 1;
            const unsigned dst = s_seed_u32 + (((buf * W + warp) * NCK + ck) * 16 + n) * 8;
            if (kx >= 0 && n < N) {
#pragma unroll
                for (int r = 0; r < 2; ++r) cp_async4(dst + 4 * r, p.x + (((int64_t)b * D + min(rowA + r, D - 1)) * p.nx + kx) * N + n);
            } else {
                s_seed[((buf * W + warp) * NCK + ck) * 16 + n] = make_float2(0.f, 0.f);
            }
        }
    };

    // Two cp.async groups per chunk: (A) this thread's u / delta / z / dout / y slots and the x seeds, issued a whole chunk ahead;
    // (B) the B/C tile, which can only be refilled after the state loop.  The prologue needs A only, so the tile's latency
    // hides under the per-(row, token) prologue instead of stalling the top of the chunk.
    __syncthreads();
    issue_in(tl < L);
    load_seeds(c_end - 1, (c_end - 1) & 1);
    cp_async_commit();
    issue_tile(c_end - 1);
    cp_async_commit();

    for (int c = c_end - 1; c >= c_begin; --c, tl -= CH) {
        const bool ok = tl < L;
        cp_async_wait_but_last();       // group A of this chunk (my own landing slots: no barrier needed to read them)
        // ---- per (row, token) registers (.x = row A, .y = row B) ---------------------------------------------------------------
        float2 dl[T], dlu[T], dy[T];
        {
            float uu[2][T], dd[2][T], gg[2][T], zf[2][T];
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                load_land(1, r, dd[r]);
                if constexpr (ORD) load_ord8(3, r, tl, gg[r]);
                else load_land(3, r, gg[r]);
                if (!AGG) load_land(0, r, uu[r]);
                if (has_z) {
                    float zz[T], yv[T];
                    if constexpr (ORD) load_ord8(2, r, tl, zz);
                    else load_land(2, r, zz);
                    if (!AGG) load_land(4, r, yv);
#pragma unroll
                    for (int i = 0; i < T; ++i) {
                        const float s = sigmoid3(zz[i]);
                        const float gz = gg[r][i] * s;
                        zf[r][i] = AGG ? 0.f : yv[i] * (gz * fmaf(zz[i], 1.f - s, 1.f));   // dz = y * g * d silu(z)/dz  (bwd_kernel.cuh:186-191)
                        gg[r][i] = gz * zz[i];                              // dy
                    }
                    // dz needs nothing from the state loop: store it now, so that neither y nor the gate factor has to be kept
                    if (!AGG) {
                        dz_p[r] += STEP;
                        if (ok && row_ok[r]) {
                            if constexpr (ORD) {
                                ord_store8<IN_T>(p.ord, tl, dz_row[r], zf[r]);
                            } else {
                                store8<IN_T, REV>(dz_p[r], zf[r]);
                            }
                        }
                    }
                }
#pragma unroll
                for (int i = 0; i < T; ++i) {
                    const float xx = dd[r][i] + bias[r];
                    const float v = sp ? softplus3(xx) : xx;
                    dd[r][i] = (ok && row_ok[r]) ? v : 0.f;        // padding tokens / rows: delta = 0, dy = 0 -> no contribution
                    gg[r][i] = (ok && row_ok[r]) ? gg[r][i] : 0.f;
                    if (AGG) dsum[r] += dd[r][i];
                }
                if (!AGG) {      // u is needed again by the epilogue (ddelta = u*S1 + S2): keep it in shared memory, not in registers
                    *reinterpret_cast<float4 *>(s_zf_t + (r * 2 + 0) * NT * 16) = make_float4(uu[r][0], uu[r][1], uu[r][2], uu[r][3]);
                    *reinterpret_cast<float4 *>(s_zf_t + (r * 2 + 1) * NT * 16) = make_float4(uu[r][4], uu[r][5], uu[r][6], uu[r][7]);
                }
            }
#pragma unroll
            for (int i = 0; i < T; ++i) {
                dl[i] = make_float2(dd[0][i], dd[1][i]);
                dy[i] = make_float2(gg[0][i], gg[1][i]);
                if (!AGG) {
                    const float2 u2 = make_float2(uu[0][i], uu[1][i]);
                    dlu[i] = fmul2(dl[i], u2);
                    dDacc = ffma2(dy[i], u2, dDacc);
                }
            }
        }
        // inputs of the next chunk (c-1): the landing slots are private to this thread and were just consumed
        cp_async_wait_all();            // group B: the B/C tile (and everybody's seeds) of this chunk
        __syncthreads();
        if constexpr (kTmaTile) mbar_wait(mbar, tile_phase++ & 1u);
        if constexpr (!kF32) {
            widen_bf16_tile<LPR, NT, true>(s_tile, s_rawbc, tid);
            __syncthreads();
        }
        if (c > c_begin) {
            issue_in(true);
            load_seeds(c - 1, (c - 1) & 1);
        }
        cp_async_commit();              // group A of chunk c-1

        float2 s1[T], s2[T];
#pragma unroll
        for (int i = 0; i < T; ++i) s1[i] = s2[i] = make_float2(0.f, 0.f);
        const float2 *seedp = s_seed + (((c & 1) * W + warp) * NCK + (j >> 3)) * 16;

        // ---- state loop, software pipelined: phase 1 of state n+1 (a, lane aggregates, both shuffle scans) is independent of
        //      phase 2 of state n (h, reverse sweep, contributions) and hides the scans' shuffle latency -----------------------
        auto load_bc = [&](int n, float (&Bn)[T], float (&Cn)[T]) {
            const unsigned char *rowB = tile + n * Tl::kRowBytes, *rowC = rowB + 16 * Tl::kRowBytes;
            const float4 c0 = *reinterpret_cast<const float4 *>(rowC), c1 = *reinterpret_cast<const float4 *>(rowC + 16);
            const float ec_[8] = {c0.x, c0.y, c0.z, c0.w, c1.x, c1.y, c1.z, c1.w};
            order8<REV>(ec_, Cn);
            if (!AGG) {
                const float4 b0 = *reinterpret_cast<const float4 *>(rowB), b1 = *reinterpret_cast<const float4 *>(rowB + 16);
                const float eb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
                order8<REV>(eb, Bn);
            }
        };
        // phase 1: a_i, the state hs entering my first token, the e entering my last token from the right
        auto phase1 = [&](int n, float2 (&a)[T], float2 &hs, float2 &ein) {
            const float2 A2l = s_A[warp * 16 + n];
            const float2 ec = s_ec[warp * 16 + n];
            float Bn[T], Cn[T];
            load_bc(n, Bn, Cn);
            float2 H = make_float2(0.f, 0.f), P, E = make_float2(0.f, 0.f);
#pragma unroll
            for (int i = 0; i < T; ++i) {
                a[i] = ex2(fmul2(dl[i], A2l));
                P = i == 0 ? a[0] : fmul2(P, a[i]);
                if (!AGG) H = ffma2(a[i], H, fmul2(dlu[i], splat(Bn[i])));
            }
#pragma unroll
            for (int i = T - 1; i >= 0; --i) E = fmul2(a[i], ffma2(dy[i], splat(Cn[i]), E));
            {   // lane 31 absorbs the e entering the chunk from the right
                const float2 E31 = ffma2(P, ec, E);
                if (j == 31) E = E31;
            }
            float2 seed = make_float2(0.f, 0.f);
            if (!AGG) {
                seed = seedp[n];
                const float2 H0 = ffma2(P, seed, H);
                if ((j & 7) == 0) H = H0;
            }
            float2 Pr = P, Pf = P;
#pragma unroll
            for (int st = 0; st < 5; ++st) {
                const float2 En = shfl_down2(E, 1 << st, 32);
                float2 Pn, Hn, Pfn;
                if (st < 4) Pn = shfl_down2(Pr, 1 << st, 32);
                if (!AGG && st < 3) {
                    Hn = shfl_up2(H, 1 << st, 8);
                    if (st < 2) Pfn = shfl_up2(Pf, 1 << st, 8);
                }
                if (ge_dn[st]) {
                    E = ffma2(Pr, En, E);
                    if (st < 4) Pr = fmul2(Pr, Pn);
                }
                if (!AGG && st < 3 && ge_up[st]) {
                    H = ffma2(Pf, Hn, H);
                    if (st < 2) Pf = fmul2(Pf, Pfn);
                }
            }
            if (j == 0) s_ec[warp * 16 + n] = E;                            // e at the chunk's first token: carry for chunk c-1
            ein = shfl_down2(E, 1, 32);
            if (j == 31) ein = ec;
            if (!AGG) {
                hs = shfl_up2(H, 1, 8);
                if ((j & 7) == 0) hs = seed;
            }
        };
        // phase 2: forward states, reverse sweep, contributions
        auto phase2 = [&](int n, const float2 (&a)[T], float2 hs, float2 e) {
            float Bn[T], Cn[T];
            load_bc(n, Bn, Cn);
            float2 h[T];
#pragma unroll
            for (int i = 0; i < T; ++i) h[i] = ffma2(a[i], i == 0 ? hs : h[i - 1], fmul2(dlu[i], splat(Bn[i])));
            const float2 A2 = fmul2(s_A[warp * 16 + n], splat(0.69314718056f));
            float dBn[T], dCn[T];
            float2 dAacc = make_float2(0.f, 0.f);
#pragma unroll
            for (int i = T - 1; i >= 0; --i) {
                const float2 dh = ffma2(dy[i], splat(Cn[i]), e);
                e = fmul2(a[i], dh);
                const float2 q = fmul2(e, i == 0 ? hs : h[i - 1]);          // dh * a_i * h_{i-1}
                const float2 pc = fmul2(dy[i], h[i]);
                const float2 pb = fmul2(dlu[i], dh);
                dCn[i] = pc.x + pc.y;
                dBn[i] = pb.x + pb.y;
                s1[i] = ffma2(dh, splat(Bn[i]), s1[i]);
                s2[i] = ffma2(q, A2, s2[i]);
                dAacc = ffma2(q, dl[i], dAacc);
            }
            // dB / dC: my 8 tokens of state n, summed over my two rows -> CTA slab -> summed over the CTA's warps -> one
            // red.global.add.v4 per 4 tokens (8x fewer L2 atomics than one per row pair)
            {
                float4 *sl = s_slab + (((n & 1) * W + warp) * 4) * 32 + j;
                sl[0 * 32] = make_float4(dBn[0], dBn[1], dBn[2], dBn[3]);
                sl[1 * 32] = make_float4(dBn[4], dBn[5], dBn[6], dBn[7]);
                sl[2 * 32] = make_float4(dCn[0], dCn[1], dCn[2], dCn[3]);
                sl[3 * 32] = make_float4(dCn[4], dCn[5], dCn[6], dCn[7]);
            }
            // publish the slab: named barrier 1 + (n & 1); the matching sync sits in reduce_state(n), one phase of work later
            asm volatile("bar.arrive %0, %1;" ::"r"(1 + (n & 1)), "r"(2 * NT) : "memory");
            // dA: fold the 32 lane partials to 8, accumulate those in (warp-private) shared memory.  After the arrive, so that the
            // shuffle latency overlaps the next phase instead of delaying the barrier.
            dAacc.x += __shfl_xor_sync(0xffffffffu, dAacc.x, 16), dAacc.y += __shfl_xor_sync(0xffffffffu, dAacc.y, 16);
            dAacc.x += __shfl_xor_sync(0xffffffffu, dAacc.x, 8), dAacc.y += __shfl_xor_sync(0xffffffffu, dAacc.y, 8);
            if (j < 8) s_dA[(n * W + warp) * 8 + j] = fadd2(s_dA[(n * W + warp) * 8 + j], dAacc);
        };
        // sum the CTA's slabs of state n and add them to global memory
        auto reduce_state = [&](int n) {
            asm volatile("bar.sync %0, %1;" ::"r"(1 + (n & 1)), "r"(2 * NT) : "memory");
            if (n < N) {
                const int t0c = tl - T * j;                                 // first token of the chunk
                for (int idx = tid; idx < 128; idx += NT) {
                    const int which = idx >> 6, q = (idx >> 5) & 1, l = idx & 31;
                    const float4 *src = s_slab + (((n & 1) * W) * 4 + which * 2 + q) * 32 + l;
                    float4 v = src[0];
#pragma unroll
                    for (int w = 1; w < W; ++w) {
                        const float4 t = src[w * 4 * 32];
                        v.x += t.x, v.y += t.y, v.z += t.z, v.w += t.w;
                    }
                    const int tq = t0c + 8 * l + 4 * q;
                    if (tq < L) {
                        float *dst = (which ? dC_b + (int64_t)n * p.dC_ns : dB_b + (int64_t)n * p.dB_ns) + (REV ? L - 4 - tq : tq);
                        if constexpr (DET) *reinterpret_cast<float4 *>(dst) = REV ? make_float4(v.w, v.z, v.y, v.x) : v;
                        else if (REV) red_add_v4(dst, v.w, v.z, v.y, v.x);
                        else red_add_v4(dst, v.x, v.y, v.z, v.w);
                    }
                }
            }
        };

        if (AGG) {
#pragma unroll 1
            for (int n = 0; n < NS; ++n) {
                float2 a0[T], hs0, e0;
                phase1(n, a0, hs0, e0);
            }
        } else {
            float2 a0[T], a1[T], hs0, hs1, e0, e1;
            phase1(0, a0, hs0, e0);
#pragma unroll 1
            for (int n = 0; n < NS; n += 2) {
                phase1(n + 1, a1, hs1, e1);
                if (n > 0) reduce_state(n - 1);
                phase2(n, a0, hs0, e0);
                if (n + 2 < NS) phase1(n + 2, a0, hs0, e0);
                reduce_state(n);
                phase2(n + 1, a1, hs1, e1);
            }
            reduce_state(NS - 1);
        }

        __syncthreads();                // everybody is done with the B/C tile: fetch the next one under the epilogue
        if (c > c_begin) issue_tile(c - 1);
        if (!AGG) {
            // ---- epilogue: du, ddelta, dz ---------------------------------------------------------------------------------------------
            float uu[2][T];
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                du_p[r] += STEP, dd_p[r] += STEP;
                const float4 f0 = *reinterpret_cast<const float4 *>(s_zf_t + (r * 2 + 0) * NT * 16);
                const float4 f1 = *reinterpret_cast<const float4 *>(s_zf_t + (r * 2 + 1) * NT * 16);
                uu[r][0] = f0.x, uu[r][1] = f0.y, uu[r][2] = f0.z, uu[r][3] = f0.w;
                uu[r][4] = f1.x, uu[r][5] = f1.y, uu[r][6] = f1.z, uu[r][7] = f1.w;
            }
            cp_async_commit();
            float2 duv[T], ddv[T];
#pragma unroll
            for (int i = 0; i < T; ++i) {
                duv[i] = ffma2(dl[i], s1[i], fmul2(make_float2(Dsk[0], Dsk[1]), dy[i]));      // delta*S1 + D*dy   (bwd_kernel.cuh:211,280-281)
                float2 t = ffma2(make_float2(uu[0][i], uu[1][i]), s1[i], s2[i]);                  // u*S1 + S2         (:282-283)
                if (sp) {
                    // softplus'(x) = sigmoid(x) = 1 - exp(-softplus(x)); series where delta is tiny (no cancellation)
                    const float2 d = dl[i];
                    const float sx = d.x < 1e-2f ? d.x * fmaf(d.x, fmaf(d.x, 0.16666667f, -0.5f), 1.f) : 1.f - ex2(-d.x * kLog2e);
                    const float sy = d.y < 1e-2f ? d.y * fmaf(d.y, fmaf(d.y, 0.16666667f, -0.5f), 1.f) : 1.f - ex2(-d.y * kLog2e);
                    t = fmul2(t, make_float2(sx, sy));
                }
                if (!ok) t = make_float2(0.f, 0.f);
                ddv[i] = t;
                dbacc = fadd2(dbacc, t);
            }
            if (ok) {
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    if (row_ok[r]) {
                        float v[T];
#pragma unroll
                        for (int i = 0; i < T; ++i) v[i] = r ? duv[i].y : duv[i].x;
                        store8<IN_T, REV>(du_p[r], v);
#pragma unroll
                        for (int i = 0; i < T; ++i) v[i] = r ? ddv[i].y : ddv[i].x;
                        store8<IN_T, REV>(dd_p[r], v);
                    }
                }
            }
        } else {
            cp_async_commit();
        }
    }

    // ---- end of the segment ---------------------------------------------------------------------------------------------------------
    __syncthreads();
    if (AGG) {
        for (int i = tid; i < NRP * 16; i += NT) {
            const int g = i >> 4, n = i & 15;
            const float2 e = s_ec[i];
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const int row = row0 + 2 * g + r;
                if (row < D) p.seg_E[(((int64_t)b * D + row) * p.nseg + seg) * 16 + n] = r ? e.y : e.x;
            }
        }
#pragma unroll
        for (int r = 0; r < 2; ++r) {
            float s = dsum[r];
#pragma unroll
            for (int k = 1; k < 32; k <<= 1) s += __shfl_xor_sync(0xffffffffu, s, k);
            if (j == 0 && row_ok[r]) p.seg_dsum[((int64_t)b * D + rowA + r) * p.nseg + seg] = s;
        }
    } else {
        if (chained && seg > 0) {   // publish e at my first token: the carry entering the segment to my left
            for (int i = tid; i < NRP * 16; i += NT) {
                const int g = i >> 4, n = i & 15;
                const float2 e = s_ec[i];
#pragma unroll
                for (int r = 0; r < 2; ++r) {
                    const int row = row0 + 2 * g + r;
                    if (row < D) __stcg(p.ein + (((int64_t)b * D + row) * p.nseg + seg - 1) * 16 + n, r ? e.y : e.x);
                }
            }
            __threadfence();
            __syncthreads();
            if (tid == 0) atomicExch(p.chain_flags + gidx * p.nseg + seg - 1, 1);
        }
        // dA: sum the 8 lane partials of my warp (its row pair), one atomic per (row, state)
        for (int n = 0; n < N; ++n) {
            float2 v = j < 8 ? s_dA[(n * W + warp) * 8 + j] : make_float2(0.f, 0.f);
#pragma unroll
            for (int k = 1; k < 8; k <<= 1) {
                v.x += __shfl_xor_sync(0xffffffffu, v.x, k);
                v.y += __shfl_xor_sync(0xffffffffu, v.y, k);
            }
            if (j == 0) {
                if constexpr (DET) {
                    float *slot = p.dA + ((int64_t)b * p.nseg + seg) * D * N;
                    if (row_ok[0]) slot[(int64_t)rowA * N + n] = v.x;
                    if (row_ok[1]) slot[(int64_t)(rowA + 1) * N + n] = v.y;
                } else {
                    if (row_ok[0]) atomicAdd(p.dA + (int64_t)rowA * N + n, v.x);
                    if (row_ok[1]) atomicAdd(p.dA + (int64_t)(rowA + 1) * N + n, v.y);
                }
            }
        }
        float2 dd = dDacc, db = dbacc;
#pragma unroll
        for (int k = 1; k < 32; k <<= 1) {
            dd.x += __shfl_xor_sync(0xffffffffu, dd.x, k), dd.y += __shfl_xor_sync(0xffffffffu, dd.y, k);
            db.x += __shfl_xor_sync(0xffffffffu, db.x, k), db.y += __shfl_xor_sync(0xffffffffu, db.y, k);
        }
        if (j == 0) {
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                if (row_ok[r]) {
                    if constexpr (DET) {
                        const int64_t slot = ((int64_t)b * p.nseg + seg) * D + rowA + r;
                        if (p.dD != nullptr) p.dD[slot] = r ? dd.y : dd.x;
                        if (p.ddbias != nullptr) p.ddbias[slot] = r ? db.y : db.x;
                    } else {
                        if (p.dD != nullptr) atomicAdd(p.dD + rowA + r, r ? dd.y : dd.x);
                        if (p.ddbias != nullptr) atomicAdd(p.ddbias + rowA + r, r ? db.y : db.x);
                    }
                }
            }
        }
    }
}

// chain the per-segment reverse aggregates right-to-left: ein[s] = e entering segment s from segment s+1
__global__ void scan3_bwd_chain_kernel(const float *__restrict__ A, const float *__restrict__ seg_E, const float *__restrict__ seg_dsum,
                                       float *__restrict__ ein, int B, int D, int N, int nseg) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)B * D * 16) return;
    const int n = (int)(i & 15);
    const int64_t bd = i >> 4;
    const int row = (int)(bd % D);
    const float a2 = n < N ? A[(int64_t)row * N + n] * kLog2e : 0.f;
    float carry = 0.f;
    for (int s0 = nseg - 1; s0 >= 0; s0 -= 8) {      // loads batched 8 segments at a time (they do not depend on the carry)
        float pa[8], ev[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int s = max(s0 - k, 0);
            pa[k] = seg_dsum[bd * nseg + s], ev[k] = seg_E[(bd * nseg + s) * 16 + n];
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const int s = s0 - k;
            if (s >= 0) {
                ein[(bd * nseg + s) * 16 + n] = carry;
                if (s > 0) carry = fmaf(ex2(a2 * pa[k]), carry, ev[k]);
            }
        }
    }
}


}  // namespace mmu
