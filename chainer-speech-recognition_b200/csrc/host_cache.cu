// host_cache.cu -- per-process caches of the host launch path.
//
// A forward+backward pair is five launches of a few hundred microseconds in total; what the host does per call
// has to stay well below that.  Everything that does not change between calls is looked up once:
//   * the SM count of each device (cudaDeviceGetAttribute is a driver round trip),
//   * the opt-in dynamic shared memory size and carve-out preference of each kernel (cudaFuncSetAttribute is only
//     called again when a launch needs MORE than what was granted before).
#include <mutex>

#include "kernels.h"

namespace b200ctc {

namespace {
constexpr int kMaxDevices = 64;
int g_sm_count[kMaxDevices];              // 0 = not looked up yet
struct FuncAttr { const void *func; int device; size_t granted; };
constexpr int kMaxFuncs = 256;
FuncAttr g_funcs[kMaxFuncs];
int g_nfuncs = 0;
std::mutex g_mu;
}  // namespace

namespace { thread_local const char *g_where = ""; }
void note_failure_site(const char *where) { g_where = where; }
const char *failure_site() { const char *w = g_where; g_where = ""; return w; }

int current_device() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    return dev;
}

int sm_count() {
    const int dev = current_device();
    if (dev >= 0 && dev < kMaxDevices && g_sm_count[dev] > 0) return g_sm_count[dev];
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (dev >= 0 && dev < kMaxDevices) g_sm_count[dev] = sms;
    return sms;
}

cudaError_t ensure_dynamic_smem(const void *func, size_t bytes) {
    const int dev = current_device();
    std::lock_guard<std::mutex> lock(g_mu);
    FuncAttr *slot = nullptr;
    for (int i = 0; i < g_nfuncs; ++i)
        if (g_funcs[i].func == func && g_funcs[i].device == dev) { slot = &g_funcs[i]; break; }
    if (slot && slot->granted >= bytes) return cudaSuccess;
    if (bytes > 48 * 1024 || !slot) {
        // default limit without opt-in: 48 KB; always state the carve-out preference once, so that a lattice CTA and a
        // ring CTA (both ask for the maximum) can share an SM
        if (bytes > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
            if (e != cudaSuccess) return e;
        }
        cudaFuncSetAttribute(func, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    }
    if (!slot && g_nfuncs < kMaxFuncs) {
        slot = &g_funcs[g_nfuncs++];
        slot->func = func; slot->device = dev; slot->granted = 0;
    }
    if (slot && bytes > slot->granted) slot->granted = bytes > 48 * 1024 ? bytes : 48 * 1024;
    return cudaSuccess;
}

}  // namespace b200ctc
