// pcd_host.cu -- host-side state shared by every entry point of the library: the error string, the version
// query and the memo of kernel attributes and occupancies (see pcd_common.cuh).
#include <cstdarg>
#include <cstdio>

#include <mutex>

#include "pcd_common.cuh"

namespace pcd {

// ------------------------------------------------------------------------------ error state
static thread_local char g_err[512] = "";
void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
int cuda_fail(cudaError_t e, const char *what) {
    set_error("CUDA error %d (%s) at %s", (int)e, cudaGetErrorString(e), what);
    return PCD_ERR_CUDA;
}

// ------------------------------------------------------------- kernel attribute / occupancy memo
// Entries are filled in order and never removed, so a lookup stops at the first free slot.  A full table only means that
// the attribute is set, or the occupancy queried, again on the next call.
static std::mutex g_memo_mu;

cudaError_t opt_in_smem_fn(const void *kernel, size_t bytes, bool max_carveout) {
    struct Entry { const void *fn; int bytes[64]; };
    static Entry table[128] = {};
    const int dev = current_device();
    if (dev < 0) return cudaErrorInvalidDevice;
    std::lock_guard<std::mutex> lock(g_memo_mu);
    Entry *slot = nullptr;
    for (Entry &e : table) {
        if (e.fn == kernel || e.fn == nullptr) { slot = &e; break; }
    }
    if (slot && slot->fn == kernel && slot->bytes[dev] >= (int)bytes) return cudaSuccess;
    cudaError_t err = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (err == cudaSuccess && max_carveout)
        err = cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    if (err == cudaSuccess && slot) {
        slot->fn = kernel;
        slot->bytes[dev] = (int)bytes;
    }
    return err;
}

cudaError_t ctas_per_sm_fn(const void *kernel, int threads, size_t smem, int *ctas) {
    struct Entry { const void *fn; int dev, threads; size_t smem; int ctas; };
    static Entry table[512] = {};
    const int dev = current_device();
    if (dev < 0) return cudaErrorInvalidDevice;
    std::lock_guard<std::mutex> lock(g_memo_mu);
    Entry *slot = nullptr;
    for (Entry &e : table) {
        if (e.fn == nullptr || (e.fn == kernel && e.dev == dev && e.threads == threads && e.smem == smem)) { slot = &e; break; }
    }
    if (slot && slot->fn) {
        *ctas = slot->ctas;
        return cudaSuccess;
    }
    int occ = 0;
    const cudaError_t err = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, smem);
    if (err != cudaSuccess) return err;
    *ctas = occ < 1 ? 1 : occ;
    if (slot) *slot = Entry{kernel, dev, threads, smem, *ctas};
    return cudaSuccess;
}

}  // namespace pcd

extern "C" int pcd_version(void) { return PCD_VERSION; }
extern "C" const char *pcd_last_error(void) { return pcd::g_err; }
