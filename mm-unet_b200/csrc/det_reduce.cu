// Ordered reduction of per-work-item partial sums: the second half of every deterministic (`_det`) entry point.
//
// The deterministic kernels never add floats with atomics.  Each CTA writes its partial sum to a slot indexed by its WORK ITEM
// (row group, batch, segment, token block, pixel block), never by blockIdx or arrival order, and this kernel sums the slots of every
// destination element in a fixed order and adds the total into the caller's (zero-filled, possibly strided) destination.  The order
// depends only on the number of items, so the result is bitwise reproducible for a given shape.
//
// Column j of the reduction is split as (a, r, c) with c fastest, extents (n0, n1, n2):
//   src  item i, column j : r.src[i * item_stride + a * ss0 + r * ss1 + c]
//   dst             column j : r.dst[a * ds0 + r * ds1 + c * ds2]  (+= the sum)
// Lanes: with >= 8 items, 8 threads of a column each sum every 8th item in order, then lane 0 adds the 8 lane sums in order.
#include "common.cuh"

namespace mmu {
namespace {

constexpr int kDetThreads = 256;

__global__ void __launch_bounds__(kDetThreads) det_reduce_kernel(const DetSum r, int ly) {
    __shared__ float s_part[kDetThreads];
    const int cx = kDetThreads / ly;                     // columns per block
    const int tx = threadIdx.x % cx, ty = threadIdx.x / cx;
    const int64_t ncol = (int64_t)r.n0 * r.n1 * r.n2;
    const int64_t jc = (int64_t)blockIdx.x * cx + tx;
    float s = 0.f;
    int64_t so = 0;
    if (jc < ncol) {
        const int64_t c = jc % r.n2, rr = (jc / r.n2) % r.n1, a = jc / ((int64_t)r.n1 * r.n2);
        so = a * r.ss0 + rr * r.ss1 + c;
        const float *p = r.src + so;
        int64_t i = ty;
#pragma unroll 1
        for (; i + 3 * ly < r.items; i += 4 * ly) {      // four loads in flight, summed in item order
            const float v0 = __ldcg(p + i * r.item_stride), v1 = __ldcg(p + (i + ly) * r.item_stride);
            const float v2 = __ldcg(p + (i + 2 * ly) * r.item_stride), v3 = __ldcg(p + (i + 3 * ly) * r.item_stride);
            s = (((s + v0) + v1) + v2) + v3;
        }
        for (; i < r.items; i += ly) s += __ldcg(p + i * r.item_stride);
    }
    if (ly > 1) {
        s_part[threadIdx.x] = s;
        __syncthreads();
        if (ty != 0) return;
        for (int k = 1; k < ly; ++k) s += s_part[k * cx + tx];
    }
    if (jc < ncol) {
        const int64_t c = jc % r.n2, rr = (jc / r.n2) % r.n1, a = jc / ((int64_t)r.n1 * r.n2);
        float *d = r.dst + a * r.ds0 + rr * r.ds1 + c * r.ds2;
        *d += s;
    }
}

}  // namespace

int det_reduce(const DetSum &r, cudaStream_t st) {
    const int64_t ncol = (int64_t)r.n0 * r.n1 * r.n2;
    if (ncol <= 0 || r.items <= 0) return MMU_OK;
    const int ly = r.items >= 8 ? 8 : 1;
    const int64_t blocks = (ncol + kDetThreads / ly - 1) / (kDetThreads / ly);
    if (blocks > 0x7fffffffLL) return set_error(MMU_ERR_UNSUPPORTED, "deterministic reduce: %lld columns", (long long)ncol);
    det_reduce_kernel<<<(unsigned)blocks, kDetThreads, 0, st>>>(r, ly);
    count_launch();
    return check_launch("deterministic reduce");
}

}  // namespace mmu
