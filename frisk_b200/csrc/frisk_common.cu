// frisk_b200: the library-wide part of the C ABI -- error text, ABI version, devices, device and pinned host
// allocation -- and the per-device state the other translation units share (the memory pool's setting, the SM count).
// Nothing here replaces code of the reference.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "../../include/frisk_b200.h"
#include "frisk_internal.h"

namespace {
thread_local char g_cuda_err[512] = "";
#define CK(call) FRISK_CK(call)
}  // namespace

int frisk_internal::cuda_fail(cudaError_t e, const char* what) {
    snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
    return FRISK_E_CUDA;
}

int frisk_internal::sm_count_cached() {
    static std::atomic<int> cached[64];
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    if ((n = cached[dev & 63].load(std::memory_order_acquire)) > 0) return n;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
    cached[dev & 63].store(n, std::memory_order_release);
    return n;
}

int frisk_internal::pool_ready() {
    static bool done[64] = {};
    int dev = 0;
    CK(cudaGetDevice(&dev));
    if (!done[dev & 63]) {
        cudaMemPool_t pool;
        CK(cudaDeviceGetDefaultMemPool(&pool, dev));
        // Freed stream-ordered scratch stays cached in the pool up to this size.  Above it every cudaFreeAsync hands the
        // memory back to the driver and the next call pays a real allocation: measured ~50 ms per call for the 1.8 GB text
        // buffer of a C5 shard and 39 ms for a 1.25 GB slab, against microseconds from the cache (180 GB of HBM: 32 GiB is cheap).
        uint64_t keep = 32ull << 30;
        CK(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
        done[dev & 63] = true;
    }
    return FRISK_OK;
}

extern "C" {

const char* frisk_b200_strerror(int code) {
    switch (code) {
        case FRISK_OK: return "ok";
        case FRISK_E_INVALID: return "invalid argument";
        case FRISK_E_UNSUPPORTED: return "unsupported: kmax > 12, more than 2^32-1 windows, or a table dump of windows > 65535 bases";
        case FRISK_E_CUDA: return "CUDA error (see frisk_b200_last_cuda_error)";
        case FRISK_E_NO_DEVICE: return "no CUDA device (frisk_b200 has no CPU fallback)";
        case FRISK_E_CAPACITY: return "output capacity too small";
        case FRISK_E_FORMAT: return "malformed input";
        default: return "unknown error";
    }
}

const char* frisk_b200_last_cuda_error(void) { return g_cuda_err; }
int frisk_b200_abi_version(void) { return FRISK_B200_ABI_VERSION; }

int frisk_b200_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int frisk_b200_device_alloc(void** ptr, uint64_t bytes) {
    if (!ptr) return FRISK_E_INVALID;
    if (frisk_b200_device_count() <= 0) return FRISK_E_NO_DEVICE;
    CK(cudaMalloc(ptr, bytes ? bytes : 1));
    return FRISK_OK;
}

int frisk_b200_device_free(void* ptr) {
    if (ptr) CK(cudaFree(ptr));
    return FRISK_OK;
}

int frisk_b200_set_device(int index) {
    if (frisk_b200_device_count() <= 0) return FRISK_E_NO_DEVICE;
    CK(cudaSetDevice(index));
    return FRISK_OK;
}

int frisk_b200_host_alloc(void** ptr, uint64_t bytes) {
    if (!ptr) return FRISK_E_INVALID;
    if (frisk_b200_device_count() <= 0) return FRISK_E_NO_DEVICE;
    CK(cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocDefault));
    return FRISK_OK;
}

int frisk_b200_host_free(void* ptr) {
    if (ptr) CK(cudaFreeHost(ptr));
    return FRISK_OK;
}

}  // extern "C"
