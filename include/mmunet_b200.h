/*
 * mmunet_b200 — C-ABI of the B200-native (sm_100a) Mamba-block hot path of MM-UNet.
 *
 * Drop-in boundary: these entry points replace the reference's two pybind11/torch-C++ extension
 * modules (which are torch-ABI, not C-ABI):
 *
 *   selective_scan_cuda.fwd / .bwd        requirements/Mamba/mamba/csrc/selective_scan/selective_scan.cpp:226-232, 338-349, 494-497
 *   causal_conv1d_cuda.causal_conv1d_fwd / _bwd
 *                                         requirements/Mamba/causal-conv1d/csrc/causal_conv1d.cpp:130-133, 191-196, 329-333
 *   (parameter blocks mirror SSMParamsBase/SSMParamsBwd  selective_scan.h:26-101  and
 *    ConvParamsBase/ConvParamsBwd  causal_conv1d.h:9-52)
 *
 * plus the scan-order gather/scatter that the reference expresses as torch view/permute/flip/stack
 * copies (src/UM_Net/MMUNet.py:68-121, requirements/mamba_simple.py:230,245-247,263).
 *
 * Conventions
 *   - plain pointers + sizes + element strides; no torch types.  All pointers are DEVICE pointers.
 *   - the caller allocates every output and workspace (the library never owns memory).
 *   - every call enqueues work on `stream` (a cudaStream_t passed as void*) and returns without
 *     synchronising.  Re-entrant: no global scratch.
 *   - return value: 0 on success; MMU_ERR_* (<0) for argument errors, or a positive cudaError_t
 *     for launch failures.  mmu_last_error() gives a thread-local human readable message.
 *   - the innermost (sequence) stride of every activation tensor must be 1 (same rule as the
 *     reference: selective_scan.cpp:252-253, causal_conv1d.cpp:151).  Batch / channel strides are
 *     free, which is what the (L, B*L, 1)-strided `xz` produced by in_proj needs (SURVEY.md App. B).
 *
 * Supported subset (everything MM-UNet uses; the rest is rejected with MMU_ERR_UNSUPPORTED):
 *   real A (fp32), input-dependent B and C of shape (batch, 1, dstate, L) [n_groups == 1],
 *   dstate <= 256, activations fp32 / bf16 / fp16, conv width 2..4.
 */
#ifndef MMUNET_B200_H
#define MMUNET_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMU_VERSION 100

enum mmu_dtype { MMU_F32 = 0, MMU_BF16 = 1, MMU_F16 = 2 };

enum mmu_error {
    MMU_OK = 0,
    MMU_ERR_INVALID = -1,      /* bad shape / null pointer / bad stride */
    MMU_ERR_UNSUPPORTED = -2,  /* valid for the reference, not implemented here */
    MMU_ERR_WORKSPACE = -3     /* workspace too small */
};

/* x[b][d][k][n] holds the scan state h after token (k+1)*stride-1 (fp32), stride = x_stride (default MMU_STATE_STRIDE).
 * It plays the role of the reference's `x` / scan_intermediates tensor (selective_scan.cpp:313) at a finer grain. */
#define MMU_STATE_STRIDE 64

/* ---------------------------------------------------------------------------------------------
 * selective scan.  replaces selective_scan_cuda.fwd  (selective_scan.cpp:226-336)
 *   u, delta, z, out : (batch, dim, seqlen)   dtype `dtype`, seqlen-stride 1
 *   A               : (dim, dstate) fp32 contiguous
 *   B, C            : (batch, 1, dstate, seqlen) dtype `dtype`; strides (B_bs, B_ns, 1)
 *   D, delta_bias   : (dim) fp32 or NULL;  z / out_z NULL when there is no gate
 *   out             : y*silu(z) when z != NULL, else y.  (The reference's separate pre-gate `out`
 *                     tensor is not produced: the backward recomputes it.)
 *   x               : (batch, dim, ceil(seqlen/x_stride), dstate) fp32, contiguous; NULL allowed
 *                     for inference (no backward).
 *   last_state      : (batch, dim, dstate) fp32 or NULL
 *   workspace       : mmu_selective_scan_fwd_workspace() bytes (may be NULL when that is 0)
 * --------------------------------------------------------------------------------------------- */
typedef struct mmu_scan_fwd_params {
    int32_t batch, dim, seqlen, dstate;
    int32_t dtype;           /* enum mmu_dtype */
    int32_t delta_softplus;  /* 0/1 */
    int32_t reverse;         /* 0: scan l = 0..L-1.  1: scan l = L-1..0 (fused flip, mamba_simple.py:230) */
    int32_t x_stride;        /* tokens between saved states in x; 0 = MMU_STATE_STRIDE.  Use mmu_scan_state_stride() */
    const void *u, *delta, *z, *B, *C;
    const float *A, *D, *delta_bias;
    void *out;
    float *x;
    float *last_state;
    int64_t u_bs, u_ds, delta_bs, delta_ds, z_bs, z_ds, out_bs, out_ds;   /* element strides */
    int64_t B_bs, B_ns, C_bs, C_ns;
    void *workspace;
    size_t workspace_bytes;
    /* pre-gate y = C.h + D*u (dtype `dtype`): written by the forward when non-NULL, read by the backward when non-NULL
     * (the role of the reference's saved `out`, selective_scan.cpp:311, selective_scan_interface.py:218).  NULL: the
     * backward recomputes it.  Ignored when z == NULL (then out == y). */
    void *y;
    int64_t y_bs, y_ds;
    /* Fused scan order (enum mmu_order; 0 = none).  NSLICES / TWOROW: logical token l of the scan lives at memory index idx(l)
     * (the index map of mmu_scan_order_*) in the GATE and OUTPUT tensors - z and out in the forward, z, dout and dz in the
     * backward - i.e. those tensors stay in the image's natural token order and are permuted by the kernels' own loads and
     * stores (requirements/mamba_simple.py:245-247, 263; src/UM_Net/MMUNet.py:68-121), while u, delta, B, C, y, x, du, ddelta,
     * dB, dC are in scan order (they are produced / consumed in that order by the conv and the projections).  Only where
     * mmu_scan_order_fusable() says so; FLIP is the `reverse` flag. */
    int32_t order, order_h, order_w, order_ns;
} mmu_scan_fwd_params;

size_t mmu_selective_scan_fwd_workspace(int32_t batch, int32_t dim, int32_t seqlen, int32_t dstate);
int mmu_selective_scan_fwd(const mmu_scan_fwd_params *p, void *stream);
/* Tokens between the states the backward wants in x for this problem: 8 for the wide (rows-in-lanes) kernels
 * (dim >= 64, dstate <= 16, seqlen % 8 == 0, fp32 / bf16), MMU_STATE_STRIDE otherwise.  Pass it as x_stride to BOTH passes
 * and size x as (batch, dim, ceil(seqlen / stride), dstate). */
int32_t mmu_scan_state_stride(int32_t batch, int32_t dim, int32_t seqlen, int32_t dstate, int32_t dtype);

/* ---------------------------------------------------------------------------------------------
 * selective scan backward.  replaces selective_scan_cuda.bwd  (selective_scan.cpp:338-492)
 *   inputs as forward + dout (batch, dim, seqlen) and x from the forward.
 *   du, ddelta, dz : (batch, dim, seqlen) dtype `dtype` (dz NULL iff z NULL)
 *   dA (dim,dstate), dD (dim), ddelta_bias (dim), dB, dC (batch,1,dstate,seqlen; rows contiguous, batch strides
 *   dB_bs / dC_bs and state strides dB_ns / dC_ns, 0 = contiguous): fp32,
 *   ACCUMULATED INTO (atomics) — the caller zero-fills them, as the reference does
 *   (selective_scan.cpp:458-466).  dD / ddelta_bias may be NULL when D / delta_bias are NULL.
 * --------------------------------------------------------------------------------------------- */
typedef struct mmu_scan_bwd_params {
    mmu_scan_fwd_params f;   /* f.out, f.last_state unused */
    const void *dout;
    int64_t dout_bs, dout_ds;
    void *du, *ddelta, *dz;
    int64_t du_bs, du_ds, ddelta_bs, ddelta_ds, dz_bs, dz_ds;
    float *dA, *dB, *dC, *dD, *ddelta_bias;
    /* batch and state strides (elements) of dB / dC; 0 = contiguous (dstate*seqlen, seqlen).  Lets both accumulate into row
     * slices of the gradient buffer of the x_proj output in whatever layout the caller keeps it - (batch, R + 2*dstate, seqlen)
     * or the GEMM-friendly (R + 2*dstate, batch, seqlen) (selective_scan_interface.py:256-262). */
    int64_t dB_bs, dC_bs, dB_ns, dC_ns;
} mmu_scan_bwd_params;

size_t mmu_selective_scan_bwd_workspace(int32_t batch, int32_t dim, int32_t seqlen, int32_t dstate);
int mmu_selective_scan_bwd(const mmu_scan_bwd_params *p, void *stream);

/* ---------------------------------------------------------------------------------------------
 * causal depthwise conv1d.  replaces causal_conv1d_cuda.causal_conv1d_fwd/_bwd
 *   (causal_conv1d.cpp:130-268)
 *   x, out, dout, dx : (batch, dim, seqlen) dtype `dtype`, seqlen-stride 1
 *   weight (dim, width) fp32 with strides (w_ds, w_ws); bias (dim) fp32 or NULL
 *   dweight (dim, width) fp32 contiguous, dbias (dim) fp32: accumulated into (caller zero-fills)
 * --------------------------------------------------------------------------------------------- */
typedef struct mmu_conv_params {
    int32_t batch, dim, seqlen, width;
    int32_t dtype;
    int32_t silu;            /* 0/1 */
    int32_t reverse;         /* 1: anti-causal == conv of the flipped sequence, stored un-flipped (mamba_simple.py:230) */
    int32_t reserved;
    const void *x;
    const float *weight, *bias;
    void *out;               /* fwd */
    int64_t x_bs, x_ds, out_bs, out_ds, w_ds, w_ws;
    /* backward only */
    const void *dout;
    void *dx;
    float *dweight, *dbias;
    int64_t dout_bs, dout_ds, dx_bs, dx_ds;
    /* Fused scan order (0 = none): x (and dx) are addressed through idx(l), i.e. they stay in natural token order, while out /
     * dout are in scan order: out[l] = act(bias + sum_k w[k] x[idx(l - (W-1-k))]).  Not combined with `reverse`. */
    int32_t order, order_h, order_w, order_ns;
} mmu_conv_params;

int mmu_causal_conv1d_fwd(const mmu_conv_params *p, void *stream);
int mmu_causal_conv1d_bwd(const mmu_conv_params *p, void *stream);

/* ---------------------------------------------------------------------------------------------
 * scan-order gather / scatter over the last (token) axis of a (rows, L) matrix with row stride.
 *   order: MMU_ORDER_*;  gather:  dst[r][l] = src[r][idx(l)];  scatter: dst[r][idx(l)] = src[r][l]
 *   idx(l) is the closed form of the reference permutations (bit-exact):
 *     FLIP      idx = L-1-l                                   mamba_simple.py:230
 *     NSLICES   idx(j*ns+s) = s*(L/ns)+j     (L % ns == 0)    mamba_simple.py:245-247 (scatter = :263)
 *     TWOROW    rows of an (H, W) map taken in pairs, column-interleaved, odd last row appended
 *                                                             MMUNet.py:68-93 (scatter = :95-121)
 *   rows = product of leading dims; src/dst row strides in elements; L = H*W.
 *   mmu_scan_order_index writes idx as int64 (for tests and host-side index building).
 * --------------------------------------------------------------------------------------------- */
enum mmu_order { MMU_ORDER_ROWMAJOR = 0, MMU_ORDER_FLIP = 1, MMU_ORDER_NSLICES = 2, MMU_ORDER_TWOROW = 3 };

int mmu_scan_order_gather(const void *src, void *dst, int32_t dtype, int64_t rows, int64_t src_rs, int64_t dst_rs,
                          int32_t order, int32_t H, int32_t W, int32_t nslices, void *stream);
int mmu_scan_order_scatter(const void *src, void *dst, int32_t dtype, int64_t rows, int64_t src_rs, int64_t dst_rs,
                           int32_t order, int32_t H, int32_t W, int32_t nslices, void *stream);
int mmu_scan_order_index(int64_t *idx_dev, int32_t order, int32_t H, int32_t W, int32_t nslices, void *stream);
/* 1 when the conv / scan kernels can apply `order` themselves for a sequence of H*W tokens (their `order` fields): 8-token groups
 * must map to simple strides - NSLICES: nslices % 8 == 0, (L / nslices) even; TWOROW: W % 4 == 0 - and the scan must run on the
 * dstate <= 16 kernels (seqlen % 8 == 0, fp32 / bf16).  Otherwise permute with mmu_scan_order_gather / _scatter. */
int32_t mmu_scan_order_fusable(int32_t order, int32_t H, int32_t W, int32_t nslices, int32_t dstate, int32_t dtype);

/* ---------------------------------------------------------------------------------------------
 * snake row sampler of MMConv (the caller of the Mamba block; SURVEY.md section 8 row f2).  replaces the
 * coordinate rescale + F.grid_sample(bilinear, zeros, align_corners=True) of src/UM_Net/MMUNet.py:190-224
 * (get_coordinate_map_2D's rearrange, _coordinate_map_scaling, get_interpolated_feature), morph 0:
 *   feat (B, C, H, W) contiguous, dtype in_dtype;  y (B, K, H, W) fp32 row coordinates in pixels (unclamped)
 *   out  (B, C, H*K, W) contiguous, dtype out_dtype:
 *        out[b,c,h*K+k,w] = lerp over rows of feat[b,c,:,clamp(w+k-K/2, 0, W-1)] at clamp(y[b,k,h,w], 0, H-1)
 *   bwd: dout (B, C, H*K, W) dtype out_dtype;  dfeat (B, C, H, W) fp32 and dy (B, K, H, W) fp32 are ACCUMULATED INTO
 *        (caller zero-fills); dy may be NULL.
 *   dtypes: MMU_F32 / MMU_BF16 in any combination.
 *   channels_last != 0: feat, out, dout, dfeat are NHWC in memory (feat[b][h][w][c], out[b][h*K+k][w][c]); C must be
 *        4 * a power of two.  y / dy stay (B, K, H, W).
 * --------------------------------------------------------------------------------------------- */
int mmu_snake_sample_fwd(const void *feat, const float *y, void *out, int32_t in_dtype, int32_t out_dtype, int32_t B,
                         int32_t C, int32_t H, int32_t W, int32_t K, int32_t channels_last, void *stream);
int mmu_snake_sample_bwd(const void *feat, const float *y, const void *dout, float *dfeat, float *dy, int32_t in_dtype,
                         int32_t out_dtype, int32_t B, int32_t C, int32_t H, int32_t W, int32_t K, int32_t channels_last,
                         void *stream);

/* ---------------------------------------------------------------------------------------------
 * GroupNorm that closes every MMConv (`nn.GroupNorm(out_channels // 4, out_channels)`, src/UM_Net/MMUNet.py:46, 271) for
 * channels-last maps: x, y, dy, dx are (B, HW, C) in memory with C = 4 * G (4 channels per group); gamma, beta (C) fp32.
 *   fwd: sums (B*G*2 fp32, caller zero-fills) is scratch; mean, rstd (B*G fp32) are written for the backward.
 *   bwd: dy has dtype out_dtype, dx has in_dtype; sums2 (B*G*2) and dgamma_dbeta (2*C: dgamma | dbeta) are fp32 accumulators
 *        the caller zero-fills.
 * Replaces at::native_group_norm(+backward), which is NCHW-only.
 * --------------------------------------------------------------------------------------------- */
int mmu_group_norm_nhwc_fwd(const void *x, const float *gamma, const float *beta, void *y, float *sums, float *mean, float *rstd,
                            int32_t in_dtype, int32_t out_dtype, int32_t B, int32_t C, int32_t HW, int32_t G, float eps, void *stream);
int mmu_group_norm_nhwc_bwd(const void *x, const float *gamma, const void *dy, const float *mean, const float *rstd, void *dx,
                            float *sums2, float *dgamma_dbeta, int32_t in_dtype, int32_t out_dtype, int32_t B, int32_t C, int32_t HW,
                            int32_t G, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Narrow Mamba block (d_model = 3, d_inner = 6, dt_rank = 1, d_state = 16, d_conv = 4: the Mamba inside every MMConv,
 * src/UM_Net/MMUNet.py:56, 178-183) - SURVEY.md section 8 row f3.  Replaces, around the selective scan, the separate
 * in_proj / causal_conv1d / x_proj / dt_proj / out_proj ops of requirements/mamba_simple.py:201-270 and
 * mamba_ssm/ops/selective_scan_interface.py:181-207 (backward :256-277) by one kernel each way:
 *   pre_fwd  : hidden -> pre   = rows [u (d_inner) | delta (d_inner) | z (d_inner) | B (d_state) | C (d_state)] in SCAN order;
 *              the caller then runs mmu_selective_scan_fwd on row views of `pre` (delta bias + softplus inside the scan)
 *   post_fwd : out_z (scan order, the gated scan output) -> out = out_proj(out_z) in natural token order
 *   post_bwd : dout (natural order) -> dout_y (scan order);  d(out_proj.weight) accumulated
 *   pre_bwd  : gpre = rows [du | ddelta | dz] and dBC = rows [dB | dC] (fp32) from mmu_selective_scan_bwd -> dhidden (natural
 *              order) and the in_proj / conv / x_proj / dt_proj weight gradients accumulated
 * hidden, out, dout, dhidden: (batch, d_model, L), token stride 1, tokens in NATURAL order; the scan visits them in the order
 * idx(l) (order fields as in mmu_conv_params; 0 = natural order).  pre (batch, mmu_mamba_narrow_rows(), L), out_z / dout_y
 * (batch, d_inner, L), gpre (batch, 3*d_inner, L), dBC (batch, 2*d_state, L) fp32: contiguous.  Weights fp32 contiguous, no in_proj /
 * out_proj bias.  dweights: fp32, caller zero-fills, mmu_mamba_narrow_weight_floats() long, laid out
 * [in_proj (2*d_inner, d_model) | conv_w (d_inner, d_conv) | conv_b (d_inner) | x_proj (dt_rank + 2*d_state, d_inner) |
 *  dt_proj (d_inner, dt_rank) | out_proj (d_model, d_inner) | d(altho) (1, coord_mode only)].
 * --------------------------------------------------------------------------------------------- */
typedef struct mmu_narrow_params {
    int32_t dtype;
    int32_t batch, seqlen;
    int32_t d_model, d_inner, d_state, dt_rank, d_conv;
    int32_t order, order_h, order_w, order_ns;
    const float *in_proj_w, *conv_w, *conv_b /* or NULL */, *x_proj_w, *dt_proj_w, *out_proj_w;
    const void *hidden;
    int64_t hidden_bs, hidden_cs;
    void *pre;               /* written by pre_fwd, read by pre_bwd */
    const void *out_z;       /* post_fwd, post_bwd */
    void *out;
    int64_t out_bs, out_cs;
    const void *dout;
    int64_t dout_bs, dout_cs;
    void *dout_y;
    const void *gpre;
    const float *dBC;
    void *dhidden;
    int64_t dhidden_bs, dhidden_cs;
    float *dweights;
    int32_t hidden_dtype;    /* dtype of hidden / dhidden: equal to `dtype`, or MMU_F32 with dtype MMU_BF16 (autocast) */
    /* MMConv coordinate epilogue (src/UM_Net/MMUNet.py:156-188), coord_mode = 1:  post_fwd writes, instead of `out`,
     *   coords[b][k][h*map_w + w] = gain * refined + h + snake_offsets(hidden)[k] * extend_scope      (fp32, (batch, d_model, L))
     * with gain = max(softplus(*altho), 0.01) and refined the block's output; post_bwd reads dcoords (fp32, same shape) instead of
     * dout and accumulates d(altho) into the LAST float of dweights; pre_bwd adds the offsets' gradient to dhidden. */
    int32_t coord_mode, map_h, map_w;
    float extend_scope;
    const float *altho;
    float *coords;
    const float *dcoords;
} mmu_narrow_params;

int32_t mmu_mamba_narrow_supported(int32_t d_model, int32_t d_inner, int32_t d_state, int32_t dt_rank, int32_t d_conv, int32_t dtype);
int32_t mmu_mamba_narrow_rows(int32_t d_inner, int32_t d_state);
int32_t mmu_mamba_narrow_weight_floats(int32_t d_model, int32_t d_inner, int32_t d_state, int32_t dt_rank, int32_t d_conv);
int mmu_mamba_narrow_pre_fwd(const mmu_narrow_params *p, void *stream);
int mmu_mamba_narrow_post_fwd(const mmu_narrow_params *p, void *stream);
int mmu_mamba_narrow_post_bwd(const mmu_narrow_params *p, void *stream);
int mmu_mamba_narrow_pre_bwd(const mmu_narrow_params *p, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Deterministic mode.  Every entry point above that sums floats across CTAs does it with fp32 atomics, so those sums differ in
 * the last bits from run to run.  The _det variants below compute the same results without floating-point atomics: each CTA
 * stores its partial sums to a slot of the caller's workspace indexed by its work item (row group, batch, segment, token block,
 * pixel block), and one ordered-reduce kernel adds the slots, in a fixed order, into the same outputs.  For the same inputs,
 * shapes, strides, dtypes, library build, MMU_* knobs and device, every output is then bitwise identical from call to call,
 * on any stream and in CUDA-graph replays.
 *   - Arguments are those of the plain entry point plus `ws` / `ws_bytes`: a caller-allocated device workspace (256-byte
 *     aligned; its contents on entry do not matter) of at least the size the matching ..._det_workspace() query returns.  The
 *     query is a pure host function: an upper bound for whichever kernel the dispatcher picks for that shape.
 *   - MMU_ERR_WORKSPACE when ws is NULL or smaller than that, before any work is enqueued.
 *   - The accumulate-into contract is unchanged: the caller zero-fills the accumulated outputs, the kernels add into them.
 *   - mmu_deterministic_default(): 1 when the environment knob MMU_DETERMINISTIC is a non-zero integer (read once, like the other
 *     MMU_* knobs), for callers that select the mode without an API of their own.
 * --------------------------------------------------------------------------------------------- */
int32_t mmu_deterministic_default(void);

/* selective scan backward.  Partials: dB and dC as [row group][batch][dstate][seqlen] (the sums over the rows of one CTA), dA as
 * [batch][segment][dim][dstate], dD and ddelta_bias as [batch][segment][dim].  The opt-in v4 kernels are never used here.
 * The workspace grows with batch * ceil(dim / rows per CTA) * dstate * seqlen * 8 bytes; callers slice the batch to bound it. */
size_t mmu_selective_scan_bwd_det_workspace(int32_t batch, int32_t dim, int32_t seqlen, int32_t dstate);
int mmu_selective_scan_bwd_det(const mmu_scan_bwd_params *p, void *ws, size_t ws_bytes, void *stream);
/* causal conv1d backward.  Partials [batch][token block][dim][5] (4 width-padded taps | bias). */
size_t mmu_causal_conv1d_bwd_det_workspace(int32_t batch, int32_t dim, int32_t seqlen, int32_t dtype);
int mmu_causal_conv1d_bwd_det(const mmu_conv_params *p, void *ws, size_t ws_bytes, void *stream);
/* narrow Mamba block backward.  Partials [batch][256-token tile][floats]: post_bwd the out_proj | d(altho) block of dweights,
 * pre_bwd every float of dweights before out_proj. */
size_t mmu_mamba_narrow_post_bwd_det_workspace(int32_t batch, int32_t seqlen);
size_t mmu_mamba_narrow_pre_bwd_det_workspace(int32_t batch, int32_t seqlen);
int mmu_mamba_narrow_post_bwd_det(const mmu_narrow_params *p, void *ws, size_t ws_bytes, void *stream);
int mmu_mamba_narrow_pre_bwd_det(const mmu_narrow_params *p, void *ws, size_t ws_bytes, void *stream);
/* channels-last GroupNorm.  Partials [B][pixel block][G][2] (forward statistics, reduced into `sums`) and [B][pixel block][G][10]
 * (backward: S1, S2, dgamma[4], dbeta[4]). */
size_t mmu_group_norm_nhwc_fwd_det_workspace(int32_t B, int32_t C, int32_t HW, int32_t G);
size_t mmu_group_norm_nhwc_bwd_det_workspace(int32_t B, int32_t C, int32_t HW, int32_t G);
int mmu_group_norm_nhwc_fwd_det(const void *x, const float *gamma, const float *beta, void *y, float *sums, float *mean, float *rstd,
                                int32_t in_dtype, int32_t out_dtype, int32_t B, int32_t C, int32_t HW, int32_t G, float eps, void *ws,
                                size_t ws_bytes, void *stream);
int mmu_group_norm_nhwc_bwd_det(const void *x, const float *gamma, const void *dy, const float *mean, const float *rstd, void *dx,
                                float *sums2, float *dgamma_dbeta, int32_t in_dtype, int32_t out_dtype, int32_t B, int32_t C, int32_t HW,
                                int32_t G, void *ws, size_t ws_bytes, void *stream);
/* snake sampler backward.  Gather-side: one thread owns a column of dfeat (b, channel(s), all rows, x) and walks the samples that read
 * column x in a fixed order; dy is summed over all channels by one thread per sample.  Needs no workspace (the query returns 0,
 * ws may be NULL). */
size_t mmu_snake_sample_bwd_det_workspace(int32_t B, int32_t C, int32_t H, int32_t W, int32_t K, int32_t channels_last);
int mmu_snake_sample_bwd_det(const void *feat, const float *y, const void *dout, float *dfeat, float *dy, int32_t in_dtype,
                             int32_t out_dtype, int32_t B, int32_t C, int32_t H, int32_t W, int32_t K, int32_t channels_last, void *ws,
                             size_t ws_bytes, void *stream);
/* bilinear-resize backward: the adjoint of F.interpolate(x, size=(H_out, W_out), mode="bilinear", align_corners=True) for a
 * (B, C, H_in, W_in) map, dx from dout (B, C, H_out, W_out).  dout and dx share the dtype (MMU_F32 or MMU_BF16) and the layout: dense
 * NCHW, or NHWC when channels_last != 0.  Gather-side: every dx element is written exactly once (no zero-fill, no workspace) with the
 * sum, in fp32 and in a fixed order (output row, then output column, ascending), of dout times the forward's weights, recomputed as
 * ATen computes them (scale (in - 1) / (out - 1) in fp32, 0 when out == 1), and rounded once to the dtype.  MMU_ERR_INVALID, before
 * anything is enqueued, for NULL pointers, another dtype, a size <= 0, or more elements than the kernels index (H_in * W_in and
 * H_out * W_out, times ceil(C / 16-byte vector) for NHWC input pixels, must fit int32; B * C * H * W must fit int64). */
int mmu_resize_bilinear_bwd_det(const void *dout, void *dx, int32_t dtype, int32_t B, int32_t C, int32_t H_in, int32_t W_in,
                                int32_t H_out, int32_t W_out, int32_t channels_last, void *stream);

/* ---------------------------------------------------------------------------------------------
 * Sliding-window stitch of MM_Net's five head maps (out2, out3, out4, out5, p_c): the window blending of monai's
 * SlidingWindowInferer(roi_size = roi, overlap, mode="constant") as used by the reference's validation (train.py:180), with the
 * model's own final resize-and-sum (MMUNet.py:577) fused in.  Per axis of the zero-padded image (size n >= roi):
 *   interval = roi if n == roi, else max((int)(roi * (1 - overlap)), 1)   (the caller passes it; 1 <= interval <= roi)
 *   count    = 1 + the first d >= 0 with d * interval + roi >= n;   window d starts at min(d * interval, n - roi)
 *   windows are numbered row-major (row window index first); the image sits at (pad_top, pad_left) of the padded one.
 * For every pixel (y, x) of the un-padded H x W image, in padded coordinates (y + pad_top, x + pad_left), and for every window
 * covering it, in window order, with (a, b) the window-local coordinate:
 *   v = up(out2) + up(out3) + up(out4) + up(out5) + up(p_c)   (fp32, in that order)
 *   up(m) = F.interpolate(m, (roi, roi), mode="bilinear", align_corners=True)[a, b] computed as ATen does (scale (h_m - 1) / (roi - 1)
 *           in fp32, 0 when roi == 1);   acc += v
 * and logits[b][y][x] = acc / (number of covering windows), fp32.  Every logit is written once, without float atomics: the same bits
 * on every run, on any stream and in CUDA-graph replays.
 *   heads[k]  : C = 1 maps of head_h[k] x head_w[k], dtype `dtype` (MMU_F32 or MMU_BF16), column stride 1; the map of window w of
 *               image i at heads[k] + i * head_bs[k] + w * head_ws[k] (+ row * head_rs[k] + column), element strides >= 0.
 *   logits    : (batch, H, W) fp32, strides (logits_bs, logits_rs, 1).
 *   target, fov: uint8 (batch, H, W) maps with their own strides, or NULL; target is required with counts.
 *   counts    : int64 [batch][4] or NULL, ACCUMULATED INTO (caller zero-fills): TP, FP, FN, TN over the pixels with fov != 0 (all
 *               pixels without fov), positive meaning logit > 0 and target != 0.  Per-block sums added with 64-bit integer atomics.
 * MMU_ERR_INVALID, before anything is enqueued, for a NULL required pointer, another dtype, a size <= 0, n < roi, a pad outside
 * [0, n - size], an interval outside [1, roi], a negative stride, or offsets / grid sizes the kernel cannot index (batch and
 * ceil(H / 8) <= 65535, element offsets within int64).
 * --------------------------------------------------------------------------------------------- */
#define MMU_SW_HEADS 5
typedef struct mmu_sw_stitch_params {
    int32_t dtype;                       /* of the head maps */
    int32_t batch;                       /* images of the same size */
    int32_t H, W;                        /* image size: logits, target, fov */
    int32_t roi;                         /* window side */
    int32_t n_h, n_w;                    /* padded image size (>= roi) */
    int32_t pad_top, pad_left;           /* zeros before the image in the padded one */
    int32_t interval_h, interval_w;      /* window stride per axis */
    int32_t head_h[MMU_SW_HEADS], head_w[MMU_SW_HEADS];
    const void *heads[MMU_SW_HEADS];
    int64_t head_bs[MMU_SW_HEADS], head_ws[MMU_SW_HEADS], head_rs[MMU_SW_HEADS];
    float *logits;
    int64_t logits_bs, logits_rs;
    const uint8_t *target;
    int64_t target_bs, target_rs;
    const uint8_t *fov;
    int64_t fov_bs, fov_rs;
    int64_t *counts;
} mmu_sw_stitch_params;

int mmu_sw_stitch(const mmu_sw_stitch_params *p, void *stream);

/* ---------------------------------------------------------------------------------------------
 * misc
 * --------------------------------------------------------------------------------------------- */
int mmu_version(void);
/* MMU_* environment knobs (kernel generation / tiling overrides for tests and experiments) are read once, at the first dispatch;
 * call this after changing the environment of a live process. */
void mmu_reload_knobs(void);
const char *mmu_last_error(void);
/* number of kernel launches issued through this library by the calling process (bench.py's gpu_launches) */
uint64_t mmu_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* MMUNET_B200_H */
