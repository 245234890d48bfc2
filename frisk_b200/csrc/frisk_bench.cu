// frisk_b200: micro-benchmarks that measure the roofline denominators of the window kernels on the GPU at hand
// (bench.py calls them live; SURVEY.md section 8d asks for measured, not assumed, rates):
//   frisk_b200_bench_l2_gather   random 16-byte gathers from an L2-resident table (the genome-IVOM lookup: one
//                                {I_g, log2 I_g} pair per distinct K-mer out of a 1 MiB table); mode 7: 32-byte entries
//                                with one 256-bit load each (the nibble kernel's (K+1)-mer pair table)
//   frisk_b200_bench_smem_loads  random 4/8/16-byte loads from a 32 KiB shared-memory table (bank-conflicted reads:
//                                what a position-ordered epilogue does to its count tables)
//   frisk_b200_bench_smem_atomics  u32 shared-memory atomics on a 64 KiB table: one lane per bank, random bins or one
//                                address (the counting step of the window and table kernels)
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/frisk_b200.h"
#include "frisk_internal.h"
#include "frisk_device.cuh"

namespace {
#define CK(call) FRISK_CK(call)

__device__ __forceinline__ uint32_t lcg(uint32_t& x) { x = x * 1664525u + 1013904223u; return x >> 8; }

// mode 0: every lane an independent uniformly random entry (position-ordered epilogue)
// mode 1: a warp's lanes read increasing entries with random gaps of mean `gap` (sorted epilogue: 4,794 of 65,536)
__global__ void __launch_bounds__(256, 4)
l2_gather_kernel(const double2* __restrict__ tab, uint32_t n_mask, int iters, int mode, uint32_t gap, double* sink) {
    uint32_t x = (blockIdx.x * 256u + threadIdx.x) * 2654435761u + 12345u;
    const uint32_t lane = threadIdx.x & 31u;
    double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
    for (int it = 0; it < iters; it += 4) {
        uint32_t i0, i1, i2, i3;
        if (mode == 0) { i0 = lcg(x); i1 = lcg(x); i2 = lcg(x); i3 = lcg(x); }
        else {
            // inclusive scan of random gaps over the lanes -> increasing indices inside the warp
            uint32_t g = 1u + lcg(x) % (2u * gap - 1u);
            for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync(0xffffffffu, g, o); if ((int)lane >= o) g += y; }
            const uint32_t base = __shfl_sync(0xffffffffu, lcg(x), 0);
            i0 = base + g; i1 = i0 + 32u * gap; i2 = i1 + 32u * gap; i3 = i2 + 32u * gap;
        }
        const double2 v0 = __ldg(tab + (i0 & n_mask)), v1 = __ldg(tab + (i1 & n_mask));
        const double2 v2 = __ldg(tab + (i2 & n_mask)), v3 = __ldg(tab + (i3 & n_mask));
        a0 += v0.x + v0.y; a1 += v1.x + v1.y; a2 += v2.x + v2.y; a3 += v3.x + v3.y;
    }
    const double s = a0 + a1 + a2 + a3;
    if (s == 1.2345e-300) sink[0] = s;
}

// mode 6: the random gather of mode 0 through the TEXTURE path (tex1Dfetch of 16-byte texels from linear memory): does the
// texture unit look up more than one cache line per clock?
__global__ void __launch_bounds__(256, 4)
l2_gather_tex_kernel(cudaTextureObject_t tex, uint32_t n_mask, int iters, double* sink) {
    uint32_t x = (blockIdx.x * 256u + threadIdx.x) * 2654435761u + 12345u;
    double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
    for (int it = 0; it < iters; it += 4) {
        const uint32_t i0 = lcg(x), i1 = lcg(x), i2 = lcg(x), i3 = lcg(x);
        const uint4 v0 = tex1Dfetch<uint4>(tex, (int)(i0 & n_mask)), v1 = tex1Dfetch<uint4>(tex, (int)(i1 & n_mask));
        const uint4 v2 = tex1Dfetch<uint4>(tex, (int)(i2 & n_mask)), v3 = tex1Dfetch<uint4>(tex, (int)(i3 & n_mask));
        a0 += __hiloint2double(v0.y, v0.x) + __hiloint2double(v0.w, v0.z);
        a1 += __hiloint2double(v1.y, v1.x) + __hiloint2double(v1.w, v1.z);
        a2 += __hiloint2double(v2.y, v2.x) + __hiloint2double(v2.w, v2.z);
        a3 += __hiloint2double(v3.y, v3.x) + __hiloint2double(v3.w, v3.z);
    }
    const double s = a0 + a1 + a2 + a3;
    if (s == 1.2345e-300) sink[0] = s;
}

// mode 2: the same random gather as mode 0, but as cp.async (LDGSTS) of 16 bytes per lane into shared memory, read back
// coalesced -- does a divergent gather cost fewer data-pipe cycles when it does not return through the register file?
__global__ void __launch_bounds__(256, 4)
l2_gather_async_kernel(const double2* __restrict__ tab, uint32_t n_mask, int iters, double* sink) {
    __shared__ __align__(16) double2 stage[2][4][256];
    uint32_t x = (blockIdx.x * 256u + threadIdx.x) * 2654435761u + 12345u;
    double a0 = 0;
    auto issue = [&](int buf) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t i = lcg(x) & n_mask;
            const uint32_t dst = (uint32_t)__cvta_generic_to_shared(&stage[buf][j][threadIdx.x]);
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(tab + i) : "memory");
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    issue(0);
    int buf = 0;
    for (int it = 0; it < iters; it += 4) {
        if (it + 4 < iters) { issue(buf ^ 1); asm volatile("cp.async.wait_group 1;" ::: "memory"); }
        else asm volatile("cp.async.wait_group 0;" ::: "memory");
#pragma unroll
        for (int j = 0; j < 4; ++j) { const double2 v = stage[buf][j][threadIdx.x]; a0 += v.x + v.y; }
        buf ^= 1;
    }
    if (a0 == 1.2345e-300) sink[0] = a0;
}

// mode 4: the gather as 16-byte BULK async copies (cp.async.bulk, the TMA engine) into shared memory, completion on an
// mbarrier, read back coalesced -- does the copy engine take small random pieces off the LSU data pipe, and how fast?
__global__ void __launch_bounds__(256, 4)
l2_gather_bulk_kernel(const double2* __restrict__ tab, uint32_t n_mask, int iters, double* sink) {
    __shared__ __align__(16) double2 stage[4][256];
    __shared__ __align__(8) unsigned long long bar;
    uint32_t x = (blockIdx.x * 256u + threadIdx.x) * 2654435761u + 12345u;
    const uint32_t bar_a = (uint32_t)__cvta_generic_to_shared(&bar);
    if (threadIdx.x == 0) asm volatile("mbarrier.init.shared::cta.b64 [%0], 256;" ::"r"(bar_a));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();
    double a0 = 0;
    uint32_t phase = 0;
    for (int it = 0; it < iters; it += 4) {
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], 64;" ::"r"(bar_a) : "memory");
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const uint32_t i = lcg(x) & n_mask;
            const uint32_t dst = (uint32_t)__cvta_generic_to_shared(&stage[j][threadIdx.x]);
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], 16, [%2];"
                         ::"r"(dst), "l"(tab + i), "r"(bar_a) : "memory");
        }
        uint32_t done = 0;
        while (!done)
            asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                         : "=r"(done) : "r"(bar_a), "r"(phase) : "memory");
        phase ^= 1u;
#pragma unroll
        for (int j = 0; j < 4; ++j) { const double2 v = stage[j][threadIdx.x]; a0 += v.x + v.y; }
        __syncthreads();                                   // the stage is rewritten by the next round's copies
    }
    if (a0 == 1.2345e-300) sink[0] = a0;
}

// mode 5: the gather as TMA tile::gather4 loads (four rows of a 2-D tensor per instruction; tensor map with a box of one
// row), completion on an mbarrier, read back.  The table holds {i, -i} in entry i so that the kernel can
// check what arrived; a poll budget turns a descriptor the hardware does not like into an error instead of a hang.
__global__ void __launch_bounds__(256, 4)
l2_gather4_kernel(const __grid_constant__ CUtensorMap map, uint32_t n_mask, int iters, double* sink, unsigned int* bad) {
    __shared__ __align__(128) double2 stage[256][8];      // 128 bytes per thread: every destination 128-byte aligned
    __shared__ __align__(8) unsigned long long bar;
    uint32_t x = (blockIdx.x * 256u + threadIdx.x) * 2654435761u + 12345u;
    const uint32_t bar_a = (uint32_t)__cvta_generic_to_shared(&bar);
    if (threadIdx.x == 0) asm volatile("mbarrier.init.shared::cta.b64 [%0], 256;" ::"r"(bar_a));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    double a0 = 0;
    uint32_t phase = 0;
    bool dead = false;
    for (int it = 0; it < iters && !dead; it += 4) {
        const int32_t r0 = (int32_t)(lcg(x) & n_mask), r1 = (int32_t)(lcg(x) & n_mask), r2 = (int32_t)(lcg(x) & n_mask), r3 = (int32_t)(lcg(x) & n_mask);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], 64;" ::"r"(bar_a) : "memory");
        const uint32_t dst = (uint32_t)__cvta_generic_to_shared(&stage[threadIdx.x][0]);
        asm volatile("cp.async.bulk.tensor.2d.shared::cta.global.tile::gather4.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];"
                     ::"r"(dst), "l"(&map), "r"(0), "r"(r0), "r"(r1), "r"(r2), "r"(r3), "r"(bar_a) : "memory");
        uint32_t done = 0;
        for (int poll = 0; !done && poll < 4000000; ++poll)
            asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                         : "=r"(done) : "r"(bar_a), "r"(phase) : "memory");
        if (!done) { atomicAdd(bad, 1000000u); dead = true; break; }
        phase ^= 1u;
        const int32_t rr[4] = {r0, r1, r2, r3};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double2 v = stage[threadIdx.x][j];
            if (v.x != (double)rr[j] || v.y != -(double)rr[j]) atomicAdd(bad, 1u);
            a0 += v.x + v.y;
        }
        __syncthreads();
    }
    if (a0 == 1.2345e-300) sink[0] = a0;
}

// mode 7: the random gather of mode 0 with 32-byte entries, each read by one 256-bit load (ldcg_pair): the nibble kernel's
// (K+1)-mer pair table, 8 MiB at K = 8 and 2 MiB at K = 7
__global__ void __launch_bounds__(256, 4)
l2_gather32_kernel(const double2* __restrict__ tab, uint32_t n_mask, int iters, double* sink) {
    uint32_t x = (blockIdx.x * 256u + threadIdx.x) * 2654435761u + 12345u;
    double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
    for (int it = 0; it < iters; it += 4) {
        const uint32_t i0 = lcg(x), i1 = lcg(x), i2 = lcg(x), i3 = lcg(x);
        double2 u0, v0, u1, v1, u2, v2, u3, v3;
        ldcg_pair(tab + 2u * (i0 & n_mask), u0, v0); ldcg_pair(tab + 2u * (i1 & n_mask), u1, v1);
        ldcg_pair(tab + 2u * (i2 & n_mask), u2, v2); ldcg_pair(tab + 2u * (i3 & n_mask), u3, v3);
        a0 += u0.x + v0.y; a1 += u1.x + v1.y; a2 += u2.x + v2.y; a3 += u3.x + v3.y;
    }
    const double s = a0 + a1 + a2 + a3;
    if (s == 1.2345e-300) sink[0] = s;
}

__global__ void fill_pattern_kernel(double2* tab, uint32_t n) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) tab[i] = make_double2((double)i, -(double)i);
}

// mode 3: 8-byte entries (half the table bytes for the same number of entries)
__global__ void __launch_bounds__(256, 4)
l2_gather8_kernel(const double* __restrict__ tab, uint32_t n_mask, int iters, double* sink) {
    uint32_t x = (blockIdx.x * 256u + threadIdx.x) * 2654435761u + 12345u;
    double a0 = 0, a1 = 0, a2 = 0, a3 = 0;
    for (int it = 0; it < iters; it += 4) {
        const uint32_t i0 = lcg(x), i1 = lcg(x), i2 = lcg(x), i3 = lcg(x);
        a0 += __ldg(tab + (i0 & n_mask)); a1 += __ldg(tab + (i1 & n_mask));
        a2 += __ldg(tab + (i2 & n_mask)); a3 += __ldg(tab + (i3 & n_mask));
    }
    const double s = a0 + a1 + a2 + a3;
    if (s == 1.2345e-300) sink[0] = s;
}

template <typename T>
__global__ void __launch_bounds__(256, 4)
smem_load_kernel(int iters, T* sink) {
    __shared__ __align__(16) unsigned char raw[32768];
    T* tab = reinterpret_cast<T*>(raw);
    constexpr uint32_t N = 32768u / sizeof(T);
    for (uint32_t i = threadIdx.x; i < 32768u / 4u; i += 256) reinterpret_cast<uint32_t*>(raw)[i] = i;
    __syncthreads();
    uint32_t x = (blockIdx.x * 256u + threadIdx.x) * 2654435761u + 777u;
    uint32_t acc = 0;
    for (int it = 0; it < iters; it += 4) {
        const uint32_t i0 = lcg(x) & (N - 1), i1 = lcg(x) & (N - 1), i2 = lcg(x) & (N - 1), i3 = lcg(x) & (N - 1);
        const T v0 = tab[i0], v1 = tab[i1], v2 = tab[i2], v3 = tab[i3];
        acc += *reinterpret_cast<const uint32_t*>(&v0) + *reinterpret_cast<const uint32_t*>(&v1) +
               *reinterpret_cast<const uint32_t*>(&v2) + *reinterpret_cast<const uint32_t*>(&v3);
    }
    if (acc == 0xdeadbeefu) *reinterpret_cast<uint32_t*>(sink) = acc;
}

// Shared-memory atomic micro-benchmark (roofline denominator for the counting step): one CTA of 1,024 threads per SM
constexpr int kThreads = 1024;

__global__ void __launch_bounds__(kThreads, 1) smem_atomic_bench_kernel(int iters, int mode, uint32_t* sink) {
    extern __shared__ __align__(16) uint32_t tab[];
    constexpr uint32_t N = 16384;   // 64 KiB of u32 bins
    for (uint32_t i = threadIdx.x; i < N; i += kThreads) tab[i] = 0;
    __syncthreads();
    uint32_t x = threadIdx.x * 2654435761u + blockIdx.x * 40503u + 12345u;
    for (int it = 0; it < iters; ++it) {
        uint32_t idx;
        if (mode == 0) idx = (threadIdx.x + 32u * (uint32_t)it) & (N - 1);        // one lane per bank
        else if (mode == 1) { x = x * 1664525u + 1013904223u; idx = (x >> 10) & (N - 1); }   // random bins
        else idx = 0;                                                              // one address
        atomicAdd(&tab[idx], 1u);
    }
    __syncthreads();
    uint32_t s = 0;
    for (uint32_t i = threadIdx.x; i < N; i += kThreads) s += tab[i];
    if (s == 0xdeadbeefu) sink[0] = s;
}

template <typename F>
int time_twice(F launch, cudaStream_t st, float* ms) {
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a));
    CK(cudaEventCreate(&b));
    launch();                                            // warm-up
    CK(cudaEventRecord(a, st));
    launch();
    CK(cudaEventRecord(b, st));
    CK(cudaEventSynchronize(b));
    CK(cudaEventElapsedTime(ms, a, b));
    CK(cudaEventDestroy(a));
    CK(cudaEventDestroy(b));
    CK(cudaGetLastError());
    return FRISK_OK;
}
}  // namespace

extern "C" {

int frisk_b200_bench_l2_gather(int blocks, int iters, uint64_t table_bytes, int mode, float* ms, void* stream) {
    if (blocks <= 0 || iters <= 0 || (iters & 3) || !ms || table_bytes < 4096 || (table_bytes & (table_bytes - 1)) || mode < 0 || mode > 7)
        return FRISK_E_INVALID;
    if (frisk_b200_device_count() <= 0) return FRISK_E_NO_DEVICE;
    cudaStream_t st = (cudaStream_t)stream;
    double2* tab = nullptr;
    double* sink = nullptr;
    CK(cudaMalloc(&tab, table_bytes));
    CK(cudaMalloc(&sink, 8));
    CK(cudaMemsetAsync(tab, 0, table_bytes, st));
    const uint32_t n_mask = (uint32_t)(table_bytes / 16u) - 1u;
    const uint32_t gap = 14u;                            // 65,536 entries / ~4,794 distinct K-mers of a 5 kb window
    int rc;
    if (mode == 6) {
        cudaResourceDesc rd{};
        rd.resType = cudaResourceTypeLinear;
        rd.res.linear.devPtr = tab;
        rd.res.linear.desc = cudaCreateChannelDesc<uint4>();
        rd.res.linear.sizeInBytes = table_bytes;
        cudaTextureDesc td{};
        td.readMode = cudaReadModeElementType;
        cudaTextureObject_t tex = 0;
        CK(cudaCreateTextureObject(&tex, &rd, &td, nullptr));
        rc = time_twice([&] { l2_gather_tex_kernel<<<blocks, 256, 0, st>>>(tex, n_mask, iters, sink); }, st, ms);
        cudaDestroyTextureObject(tex);
    } else if (mode == 5) {
        // tensor map of the table as a [rows][2 doubles] tensor; the driver entry point comes through the runtime
        typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                     const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                     CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        CK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (!fn || qres != cudaDriverEntryPointSuccess) { cudaFree(tab); cudaFree(sink); return FRISK_E_UNSUPPORTED; }
        CUtensorMap map;
        const cuuint64_t gdim[2] = {2, (cuuint64_t)n_mask + 1};
        const cuuint64_t gstride[1] = {16};
        const cuuint32_t box[2] = {2, 1};                  // (a box of 4 rows is rejected; destinations must be 128-byte aligned:
                                                           //  64- and 80-byte slot strides fault with cudaErrorMisalignedAddress)
        const cuuint32_t estride[2] = {1, 1};
        const CUresult cr = ((EncodeFn)fn)(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, tab, gdim, gstride, box, estride,
                                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (cr != CUDA_SUCCESS) { cudaFree(tab); cudaFree(sink); return FRISK_E_UNSUPPORTED; }
        unsigned int* bad = nullptr;
        CK(cudaMalloc(&bad, 4));
        CK(cudaMemsetAsync(bad, 0, 4, st));
        fill_pattern_kernel<<<(n_mask + 256) / 256, 256, 0, st>>>(tab, n_mask + 1);
        rc = time_twice([&] { l2_gather4_kernel<<<blocks, 256, 0, st>>>(map, n_mask, iters, sink, bad); }, st, ms);
        unsigned int h_bad = 0;
        if (cudaMemcpy(&h_bad, bad, 4, cudaMemcpyDeviceToHost) != cudaSuccess) rc = FRISK_E_CUDA;
        cudaFree(bad);
        if (!rc && h_bad) rc = h_bad >= 1000000u ? FRISK_E_UNSUPPORTED : FRISK_E_FORMAT;   // never completed / wrong data
    } else if (mode == 2) rc = time_twice([&] { l2_gather_async_kernel<<<blocks, 256, 0, st>>>(tab, n_mask, iters, sink); }, st, ms);
    else if (mode == 4) rc = time_twice([&] { l2_gather_bulk_kernel<<<blocks, 256, 0, st>>>(tab, n_mask, iters, sink); }, st, ms);
    else if (mode == 7) rc = time_twice([&] { l2_gather32_kernel<<<blocks, 256, 0, st>>>(tab, (n_mask - 1u) / 2u, iters, sink); }, st, ms);
    else if (mode == 3) rc = time_twice([&] { l2_gather8_kernel<<<blocks, 256, 0, st>>>((const double*)tab, 2u * n_mask + 1u, iters, sink); }, st, ms);
    else rc = time_twice([&] { l2_gather_kernel<<<blocks, 256, 0, st>>>(tab, n_mask, iters, mode, gap, sink); }, st, ms);
    cudaFree(tab);
    cudaFree(sink);
    return rc;
}

int frisk_b200_bench_smem_loads(int blocks, int iters, int elem_bytes, float* ms, void* stream) {
    if (blocks <= 0 || iters <= 0 || (iters & 3) || !ms) return FRISK_E_INVALID;
    if (frisk_b200_device_count() <= 0) return FRISK_E_NO_DEVICE;
    cudaStream_t st = (cudaStream_t)stream;
    void* sink = nullptr;
    CK(cudaMalloc(&sink, 16));
    int rc;
    if (elem_bytes == 4) rc = time_twice([&] { smem_load_kernel<uint32_t><<<blocks, 256, 0, st>>>(iters, (uint32_t*)sink); }, st, ms);
    else if (elem_bytes == 8) rc = time_twice([&] { smem_load_kernel<uint2><<<blocks, 256, 0, st>>>(iters, (uint2*)sink); }, st, ms);
    else if (elem_bytes == 16) rc = time_twice([&] { smem_load_kernel<uint4><<<blocks, 256, 0, st>>>(iters, (uint4*)sink); }, st, ms);
    else rc = FRISK_E_INVALID;
    cudaFree(sink);
    return rc;
}

int frisk_b200_bench_smem_atomics(int blocks, int iters, int mode, float* ms, void* stream) {
    if (blocks <= 0 || iters <= 0 || !ms) return FRISK_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    CK(cudaFuncSetAttribute(smem_atomic_bench_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 65536));
    uint32_t* sink = nullptr;
    CK(cudaMalloc(&sink, 4));
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a));
    CK(cudaEventCreate(&b));
    smem_atomic_bench_kernel<<<blocks, kThreads, 65536, st>>>(iters, mode, sink);   // warm-up
    CK(cudaEventRecord(a, st));
    smem_atomic_bench_kernel<<<blocks, kThreads, 65536, st>>>(iters, mode, sink);
    CK(cudaEventRecord(b, st));
    CK(cudaEventSynchronize(b));
    CK(cudaEventElapsedTime(ms, a, b));
    CK(cudaEventDestroy(a));
    CK(cudaEventDestroy(b));
    CK(cudaFree(sink));
    CK(cudaGetLastError());
    return FRISK_OK;
}

}  // extern "C"
