// Sliding-window stitch of MM_Net's head maps: the epilogue of monai's SlidingWindowInferer (constant blending) fused into one
// gather-side kernel.
//
// Per axis of the zero-padded image (size n >= S = roi, stride `interval`): window d starts at min(d * interval, n - S), count = 1 +
// (the first d >= 0 with d * interval + S >= n); windows are numbered row-major.  The windows covering padded coordinate p are the
// regular ones d in [ceil((p - S + 1) / interval), min(p / interval, count - 2)] (start d * interval) and, when p >= n - S, the last
// one (start n - S): found in closed form, no list of starts.
//
// One thread per output pixel of the un-padded image walks its covering windows in window order; for each it sums the five heads'
// align_corners=True bilinear taps at the window-local coordinate (ATen's arithmetic, as resize_bilinear.cu's resize_tap) in head
// order, in fp32, adds the sum to its accumulator, and writes acc / (number of covering windows) once.  No atomics on floats: the
// logits have the same bits on every run.  The optional confusion counts (TP, FP, FN, TN of logit > 0 against target != 0 inside
// the FOV) are reduced per block and added with 64-bit integer atomics, which are exact.
#include "common.cuh"

namespace mmu {

constexpr int kSwHeads = 5;
constexpr int kSwTileW = 32, kSwTileH = 8;       // 256 threads: a 32 x 8 pixel tile

struct SwGeom {
    const void *head[kSwHeads];
    int64_t hbs[kSwHeads], hws[kSwHeads], hrs[kSwHeads];
    int hh[kSwHeads], hw[kSwHeads];
    float sh[kSwHeads], sw[kSwHeads];
    int S, H, W, pad_t, pad_l, n_h, n_w, iv_h, iv_w, cnt_h, cnt_w;
    float *logits;
    int64_t lbs, lrs;
    const uint8_t *tgt;
    int64_t tbs, trs;
    const uint8_t *fov;
    int64_t fbs, frs;
    unsigned long long *counts;
};

// covering windows of padded coordinate p along one axis: regular windows lo .. lo + nreg - 1, then window cnt - 1 when `last`
__device__ __forceinline__ void sw_cover(int p, int n, int S, int iv, int cnt, int &lo, int &nreg, bool &last) {
    lo = p < S ? 0 : (p - S) / iv + 1;
    nreg = max(min(p / iv, cnt - 2) - lo + 1, 0);
    last = p >= n - S;
}

// ATen's upsample_bilinear2d (align_corners=True) value of a (hh, hw) map at output (a, b) of an S x S window
template <typename T>
__device__ __forceinline__ float sw_up(const T *__restrict__ m, int64_t rs, float sh, float sw, int hh, int hw, int a, int b) {
    const float rh = __fmul_rn(sh, (float)a), rw = __fmul_rn(sw, (float)b);
    const int h0 = (int)rh, w0 = (int)rw;
    const int hp = h0 < hh - 1 ? 1 : 0, wp = w0 < hw - 1 ? 1 : 0;
    const float h1l = __fsub_rn(rh, (float)h0), h0l = 1.f - h1l;
    const float w1l = __fsub_rn(rw, (float)w0), w0l = 1.f - w1l;
    const T *r0 = m + (int64_t)h0 * rs, *r1 = r0 + hp * rs;
    return h0l * (w0l * Elem<T>::to_f(r0[w0]) + w1l * Elem<T>::to_f(r0[w0 + wp])) +
           h1l * (w0l * Elem<T>::to_f(r1[w0]) + w1l * Elem<T>::to_f(r1[w0 + wp]));
}

// grid: (ceil(W / 32), ceil(H / 8), batch)
template <typename T>
__global__ void __launch_bounds__(kSwTileW * kSwTileH) sw_stitch_kernel(const SwGeom g) {
    const int x = blockIdx.x * kSwTileW + (threadIdx.x % kSwTileW), y = blockIdx.y * kSwTileH + (threadIdx.x / kSwTileW);
    const int64_t b = blockIdx.z;
    bool counted = false, pos = false, t = false;         // this thread's pixel: inside the FOV, logit > 0, target != 0
    if (x < g.W && y < g.H) {
        const int py = y + g.pad_t, px = x + g.pad_l;
        int lo_h, nr_h, lo_w, nr_w;
        bool last_h, last_w;
        sw_cover(py, g.n_h, g.S, g.iv_h, g.cnt_h, lo_h, nr_h, last_h);
        sw_cover(px, g.n_w, g.S, g.iv_w, g.cnt_w, lo_w, nr_w, last_w);
        const int nh = nr_h + (last_h ? 1 : 0), nw = nr_w + (last_w ? 1 : 0);
        float acc = 0.f;
        for (int i = 0; i < nh; ++i) {
            const int dh = i < nr_h ? lo_h + i : g.cnt_h - 1;
            const int a = py - (i < nr_h ? dh * g.iv_h : g.n_h - g.S);
            for (int j = 0; j < nw; ++j) {
                const int dw = j < nr_w ? lo_w + j : g.cnt_w - 1;
                const int bc = px - (j < nr_w ? dw * g.iv_w : g.n_w - g.S);
                const int64_t win = (int64_t)dh * g.cnt_w + dw;
                float v = 0.f;
#pragma unroll
                for (int k = 0; k < kSwHeads; ++k) {
                    const T *m = static_cast<const T *>(g.head[k]) + b * g.hbs[k] + win * g.hws[k];
                    v += sw_up(m, g.hrs[k], g.sh[k], g.sw[k], g.hh[k], g.hw[k], a, bc);
                }
                acc += v;
            }
        }
        const float logit = acc / (float)(nh * nw);
        g.logits[b * g.lbs + (int64_t)y * g.lrs + x] = logit;
        if (g.counts != nullptr && (g.fov == nullptr || g.fov[b * g.fbs + (int64_t)y * g.frs + x] != 0)) {
            counted = true;
            pos = logit > 0.f;
            t = g.tgt[b * g.tbs + (int64_t)y * g.trs + x] != 0;
        }
    }
    if (g.counts == nullptr) return;                      // uniform over the grid
    __shared__ unsigned s_c[kSwTileH][4];
    const int lane = threadIdx.x % 32, warp = threadIdx.x / 32;
    const unsigned tp = __reduce_add_sync(0xffffffffu, counted && pos && t), fp = __reduce_add_sync(0xffffffffu, counted && pos && !t);
    const unsigned fn = __reduce_add_sync(0xffffffffu, counted && !pos && t), tn = __reduce_add_sync(0xffffffffu, counted && !pos && !t);
    if (lane == 0) s_c[warp][0] = tp, s_c[warp][1] = fp, s_c[warp][2] = fn, s_c[warp][3] = tn;
    __syncthreads();
    if (threadIdx.x < 4) {
        unsigned long long s = 0;
        for (int w = 0; w < kSwTileH; ++w) s += s_c[w][threadIdx.x];
        if (s) atomicAdd(g.counts + b * 4 + threadIdx.x, s);
    }
}

namespace {
// acc += (n - 1) * stride without overflowing int64; false on overflow
bool span(int64_t &acc, int64_t n, int64_t stride) {
    int64_t t;
    return !__builtin_mul_overflow(n - 1, stride, &t) && !__builtin_add_overflow(acc, t, &acc);
}

bool axis_ok(int32_t size, int32_t pad, int32_t n, int32_t S, int32_t iv) {
    return size > 0 && pad >= 0 && n >= S && (int64_t)pad + size <= n && iv >= 1 && iv <= S;
}
}  // namespace
}  // namespace mmu

extern "C" int mmu_sw_stitch(const mmu_sw_stitch_params *p, void *stream) {
    using namespace mmu;
    if (p == nullptr) return set_error(MMU_ERR_INVALID, "sw_stitch: null params");
    if (p->dtype != MMU_F32 && p->dtype != MMU_BF16) return set_error(MMU_ERR_INVALID, "sw_stitch: dtype %d (fp32 or bf16 only)", p->dtype);
    if (p->batch <= 0 || p->H <= 0 || p->W <= 0 || p->roi <= 0)
        return set_error(MMU_ERR_INVALID, "sw_stitch: bad shape batch %d image %dx%d roi %d", p->batch, p->H, p->W, p->roi);
    if (!axis_ok(p->H, p->pad_top, p->n_h, p->roi, p->interval_h) || !axis_ok(p->W, p->pad_left, p->n_w, p->roi, p->interval_w))
        return set_error(MMU_ERR_INVALID, "sw_stitch: bad window geometry: image %dx%d, pads (%d, %d), padded %dx%d, roi %d, intervals (%d, %d) "
                         "(need n >= roi, 0 <= pad, pad + size <= n, 1 <= interval <= roi)", p->H, p->W, p->pad_top, p->pad_left, p->n_h,
                         p->n_w, p->roi, p->interval_h, p->interval_w);
    if (p->logits == nullptr) return set_error(MMU_ERR_INVALID, "sw_stitch: null logits");
    if (p->counts != nullptr && p->target == nullptr) return set_error(MMU_ERR_INVALID, "sw_stitch: counts need a target (null pointer)");
    if (p->counts != nullptr && reinterpret_cast<uintptr_t>(p->counts) % 8 != 0)
        return set_error(MMU_ERR_INVALID, "sw_stitch: counts must be 8-byte aligned");
    SwGeom g{};
    g.S = p->roi, g.H = p->H, g.W = p->W, g.pad_t = p->pad_top, g.pad_l = p->pad_left, g.n_h = p->n_h, g.n_w = p->n_w;
    g.iv_h = p->interval_h, g.iv_w = p->interval_w;
    g.cnt_h = (p->n_h - p->roi + p->interval_h - 1) / p->interval_h + 1;
    g.cnt_w = (p->n_w - p->roi + p->interval_w - 1) / p->interval_w + 1;
    const int64_t nwin = (int64_t)g.cnt_h * g.cnt_w;
    for (int k = 0; k < kSwHeads; ++k) {
        if (p->heads[k] == nullptr) return set_error(MMU_ERR_INVALID, "sw_stitch: null head %d", k);
        if (p->head_h[k] <= 0 || p->head_w[k] <= 0)
            return set_error(MMU_ERR_INVALID, "sw_stitch: bad shape of head %d: %dx%d", k, p->head_h[k], p->head_w[k]);
        if (p->head_bs[k] < 0 || p->head_ws[k] < 0 || p->head_rs[k] < 0)
            return set_error(MMU_ERR_INVALID, "sw_stitch: negative stride of head %d", k);
        int64_t last = p->head_w[k] - 1;
        if (!span(last, p->batch, p->head_bs[k]) || !span(last, nwin, p->head_ws[k]) || !span(last, p->head_h[k], p->head_rs[k]))
            return set_error(MMU_ERR_INVALID, "sw_stitch: head %d overflows the kernel's index range", k);
        g.head[k] = p->heads[k], g.hbs[k] = p->head_bs[k], g.hws[k] = p->head_ws[k], g.hrs[k] = p->head_rs[k];
        g.hh[k] = p->head_h[k], g.hw[k] = p->head_w[k];
        g.sh[k] = p->roi > 1 ? (float)(p->head_h[k] - 1) / (float)(p->roi - 1) : 0.f;   // ATen's area_pixel_compute_scale
        g.sw[k] = p->roi > 1 ? (float)(p->head_w[k] - 1) / (float)(p->roi - 1) : 0.f;
    }
    const struct { const void *ptr; int64_t bs, rs; const char *name; } maps[3] = {
        {p->logits, p->logits_bs, p->logits_rs, "logits"}, {p->target, p->target_bs, p->target_rs, "target"}, {p->fov, p->fov_bs, p->fov_rs, "fov"}};
    for (const auto &m : maps) {
        if (m.ptr == nullptr) continue;
        int64_t last = p->W - 1;
        if (m.bs < 0 || m.rs < 0) return set_error(MMU_ERR_INVALID, "sw_stitch: negative stride of %s", m.name);
        if (!span(last, p->batch, m.bs) || !span(last, p->H, m.rs))
            return set_error(MMU_ERR_INVALID, "sw_stitch: %s overflows the kernel's index range", m.name);
    }
    if (p->batch > 65535 || (p->H + kSwTileH - 1) / kSwTileH > 65535 || nwin > INT32_MAX)
        return set_error(MMU_ERR_INVALID, "sw_stitch: batch %d, image %dx%d, %lld windows overflow the kernel's index range", p->batch, p->H,
                         p->W, (long long)nwin);
    g.logits = p->logits, g.lbs = p->logits_bs, g.lrs = p->logits_rs;
    g.tgt = p->target, g.tbs = p->target_bs, g.trs = p->target_rs;
    g.fov = p->fov, g.fbs = p->fov_bs, g.frs = p->fov_rs;
    g.counts = reinterpret_cast<unsigned long long *>(p->counts);
    const dim3 grid((unsigned)((p->W + kSwTileW - 1) / kSwTileW), (unsigned)((p->H + kSwTileH - 1) / kSwTileH), (unsigned)p->batch);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (p->dtype == MMU_F32) sw_stitch_kernel<float><<<grid, kSwTileW * kSwTileH, 0, st>>>(g);
    else sw_stitch_kernel<__nv_bfloat16><<<grid, kSwTileW * kSwTileH, 0, st>>>(g);
    count_launch();
    return check_launch("sw_stitch");
}
