// C-ABI plumbing shared by all entry points: thread-local error text, launch accounting.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "common.cuh"

namespace mmu {
namespace {
thread_local char g_err[512] = "";
std::atomic<uint64_t> g_launches{0};
}  // namespace

int set_error(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

// ---- tuning knobs -------------------------------------------------------------------------------------------------------
// MMU_* environment variables select kernel generations / tilings for tests and experiments.  They are read ONCE (first
// dispatch, or mmu_reload_knobs()), not per launch.
namespace {
constexpr const char *kKnobNames[] = {
    "MMU_SCAN_V", "MMU_BWD_V", "MMU_FWD_CFG", "MMU_BWD_CFG", "MMU_FWD_NSEG", "MMU_BWD_NSEG", "MMU_NO_PREFETCH", "MMU_FWD3_LPR",
    "MMU_FWD3_W", "MMU_BWD3_W", "MMU_BWD_CHAIN", "MMU_V4_WPSM", "MMU_V4_BWD_WPSM", "MMU_V4_MIN_DIM", "MMU_V5_MIN_DIM", "MMU_FUSE", "MMU_RING", "MMU_V5_W", "MMU_V5_MIN_WARPS", "MMU_RING_BF16",
    "MMU_DETERMINISTIC"};
constexpr int kNumKnobs = sizeof(kKnobNames) / sizeof(kKnobNames[0]);
struct KnobTable {
    bool set[kNumKnobs];
    int value[kNumKnobs];
};
KnobTable g_knobs;
std::once_flag g_knobs_once;
std::mutex g_knobs_mu;
void load_knobs() {
    std::lock_guard<std::mutex> lk(g_knobs_mu);
    for (int i = 0; i < kNumKnobs; ++i) {
        const char *v = getenv(kKnobNames[i]);
        g_knobs.set[i] = v != nullptr && *v != 0;
        g_knobs.value[i] = g_knobs.set[i] ? atoi(v) : 0;
    }
}
}  // namespace

int knob(const char *name, int dflt) {
    std::call_once(g_knobs_once, load_knobs);
    for (int i = 0; i < kNumKnobs; ++i)
        if (strcmp(name, kKnobNames[i]) == 0) return g_knobs.set[i] ? g_knobs.value[i] : dflt;
    return dflt;    // unknown name: not a knob
}

void count_launch(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

int check_launch(const char *what) {
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error((int)e, "%s: launch failed: %s", what, cudaGetErrorString(e));
    return MMU_OK;
}
}  // namespace mmu

extern "C" int mmu_version(void) { return MMU_VERSION; }
extern "C" void mmu_reload_knobs(void) {
    std::call_once(mmu::g_knobs_once, mmu::load_knobs);
    mmu::load_knobs();
}
extern "C" const char *mmu_last_error(void) { return mmu::g_err; }
extern "C" int32_t mmu_deterministic_default(void) { return mmu::knob("MMU_DETERMINISTIC", 0) != 0 ? 1 : 0; }
extern "C" uint64_t mmu_launch_count(void) { return mmu::g_launches.load(std::memory_order_relaxed); }
