// frisk_b200: the window-kernel layer -- which window kernel frisk_b200_score runs (plan_score), how a persistent window
// kernel is launched, the hand-over to the small-K and bucketed kernels, the score entry points of the C ABI and the
// options that force a kernel -- and the KLD of two IVOM vectors.
//
// Replaces the reference's per-window loop (/root/reference/frisk/__init__.py F:1478-1494) by a choice of one kernel
// for all windows; the kernels are in frisk_small.cu, frisk_bucket.cu, frisk_dense.cu, frisk_direct.cu, frisk_nibble.cu,
// frisk_nibble_ext.cu and frisk_general.cu.  kld_kernel replaces F:459-472 for the dict-level compatibility API.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <tuple>

#include "../../include/frisk_b200.h"
#include "frisk_internal.h"
#include "frisk_device.cuh"

namespace {
using frisk_internal::sm_count_cached;
using frisk_internal::LaunchShape;
using frisk_internal::WinKernel;
using frisk_internal::WinPlan;
using frisk_internal::kSmemMaxWindow;
using frisk_internal::check_k;
#define CK(call) FRISK_CK(call)

constexpr int kThreads = 1024;          // kld_kernel: one CTA
constexpr int kWarps = kThreads / 32;

// KLD of two already-normalised IVOM vectors (F:459-472): sum w*log2(w/G), G == 0 skipped.
// One CTA, fixed reduction tree.  Only used by the dict-level compatibility API; the batch path
// computes the same quantity inside score_windows_kernel.
__global__ void __launch_bounds__(kThreads, 1)
kld_kernel(const double* __restrict__ g, const double* __restrict__ w, uint32_t n, double* __restrict__ out) {
    __shared__ double red[kWarps];
    double acc = 0.0;
    for (uint32_t i = threadIdx.x; i < n; i += kThreads) {
        const double gv = g[i], wv = w[i];
        if (gv != 0.0) acc = fma(wv, log2(wv / gv), acc);
    }
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(kFull, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int wp = 0; wp < kWarps; ++wp) s += red[wp];
        *out = s;
    }
}

int g_forced = -1;          // the WinKernel forced through frisk_b200_set_option (tests, A/B measurements), -1: none

bool forced(WinKernel k) { return g_forced == (int)k; }

constexpr bool nibble_default(int kmax, uint32_t len) { return kmax == 8 || (kmax == 7 && len > 1500u); }   // measured: tools/k8_ab.py
constexpr bool direct_default(int kmax) { return kmax == 7; }   // (reached for short windows only: w = 1000 / 500: 1.00 / 1.59 ms vs 1.05 / 1.76 nibble, 1.14 / 1.85 bucketed)

}  // namespace

// Which window kernel frisk_b200_score runs.  kmax 9..12: the extension kernel on windows the shared-memory kernels hold,
// the general one otherwise (and for the test-only table dump).  kmax <= 8: the small-K kernel up to kmax 6 (no sorting,
// 6 CTAs/SM, any window up to 65,535 bases); for kmax 7 and 8 the nibble kernel (4-bit counters, one atomic per position)
// or the direct kernel (byte table) as measured on C2 (nibble_default / direct_default), then the bucketed
// one over whatever they hand back; the dense-table kernel for windows longer than the shared-memory buffer.  A forced
// kernel wins wherever it can run.
int frisk_internal::plan_score(int kmin, int kmax, uint32_t len, bool dump, WinPlan* out) {
    int rc = check_k(kmin, kmax);
    if (rc) return rc;
    const bool smem = len <= kSmemMaxWindow;
    WinKernel k;
    if (forced(WinKernel::General) || len > 65535u) k = WinKernel::General;
    else if (kmax > FRISK_B200_FAST_K) k = kmax <= 12 && smem && !dump ? WinKernel::NibbleExt : WinKernel::General;
    else if (forced(WinKernel::Dense)) k = WinKernel::Dense;
    else if (kmax <= 6 && !forced(WinKernel::Bucket)) k = WinKernel::Small;
    else if (kmax < 4 || !smem) k = WinKernel::Dense;
    else if (kmax >= 7 && (forced(WinKernel::Nibble) ||
                           (!forced(WinKernel::Bucket) && !forced(WinKernel::Direct) && nibble_default(kmax, len))))
        k = WinKernel::Nibble;
    else if (kmax >= 7 && (forced(WinKernel::Direct) || (!forced(WinKernel::Bucket) && direct_default(kmax))))
        k = WinKernel::Direct;
    else k = WinKernel::Bucket;
    *out = {k, window_variant(k, len), dump, kmin == 1 && !dump};
    return FRISK_OK;
}

int frisk_internal::check_k(int kmin, int kmax) {
    if (kmin < 1 || kmin > kmax) return FRISK_E_INVALID;
    if (kmax > FRISK_B200_MAX_K) return FRISK_E_UNSUPPORTED;
    return FRISK_OK;
}

// Positions per thread, from the longest window (the K-mer codes stay in registers between the counting and the scoring
// pass; shorter windows of the same launch use fewer).  All four kernels run 256 threads; a bucketed or direct round is
// 4 positions and keeps 6 bases of look-ahead.
int frisk_internal::window_variant(WinKernel kind, uint32_t len) {
    constexpr uint32_t kT = 256;        // threads per CTA of the four kernels
    if (kind == WinKernel::Bucket || kind == WinKernel::Direct)
        return len <= kT * 4u * 2u - 6u ? 2 : (len <= kT * 4u * 5u - 6u ? 5 : 8);
    if (kind == WinKernel::Nibble || kind == WinKernel::NibbleExt) return len <= kT * 8u ? 8 : (len <= kT * 20u ? 20 : 32);
    return 0;
}

namespace {
// CTAs per SM by (device, kernel, dynamic shared memory), and the largest dynamic shared memory a kernel has been allowed
// on a device: the attribute is only ever raised, so that a launch with a smaller cached size stays valid
std::mutex g_occ_mu;
std::map<std::tuple<int, const void*, size_t>, int> g_occ;
std::map<std::pair<int, const void*>, size_t> g_smem_attr;
}  // namespace

int frisk_internal::ctas_per_sm(const LaunchShape& s, int* out) {
    int dev = 0;
    CK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_occ_mu);
    auto it = g_occ.find({dev, s.fn, s.smem});
    if (it == g_occ.end()) {
        size_t& attr = g_smem_attr[{dev, s.fn}];
        if (s.smem > attr) {
            CK(cudaFuncSetAttribute(s.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s.smem));
            attr = s.smem;
        }
        if (s.max_carveout)
            CK(cudaFuncSetAttribute(s.fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        int n = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, s.fn, s.threads, s.smem));
        it = g_occ.emplace(std::make_tuple(dev, s.fn, s.smem), n).first;
    }
    *out = it->second;
    return FRISK_OK;
}

int frisk_internal::launch_persistent(const LaunchShape& s, uint64_t n_win, void** args, cudaStream_t st) {
    int per_sm = 0;
    int rc = ctas_per_sm(s, &per_sm);
    if (rc) return rc;
    const int sms = sm_count_cached();
    if (sms <= 0) return FRISK_E_NO_DEVICE;
    const uint64_t grid = std::min<uint64_t>((uint64_t)sms * (uint64_t)std::max(per_sm, 1), n_win);
    CK(cudaLaunchKernel(s.fn, dim3((unsigned)grid), dim3((unsigned)s.threads), args, s.smem, st));
    return FRISK_OK;
}

int frisk_internal::score_bucket_redo(const uint32_t* codes, const uint32_t* inv, const uint32_t* low, const uint64_t* win_off,
                                      const uint32_t* win_len, uint64_t n_win, uint32_t max_len, const double* ig, int kmin, int K,
                                      int want_rip, double* rows, uint32_t* status, uint16_t* dump, const uint32_t* redo_src,
                                      cudaStream_t st) {
    if (max_len > kSmemMaxWindow || !redo_src) return FRISK_E_UNSUPPORTED;
    // the generic instantiation (any kmin, optional dump); the k sweep hands a window over for EVERY kmax': 4..6 on the
    // bucketed kernel too, 1..3 on the small-K kernel
    const WinPlan p{K <= 3 ? WinKernel::Small : WinKernel::Bucket, window_variant(WinKernel::Bucket, max_len), dump != nullptr, false};
    if (K <= 3)
        return score_small(p, codes, inv, low, win_off, win_len, n_win, ig, kmin, K, want_rip, rows, status, dump, st, redo_src);
    return score_bucket(p, codes, inv, low, win_off, win_len, n_win, max_len, ig, kmin, K, want_rip, rows, status, dump, st, redo_src);
}

extern "C" {

int frisk_b200_score(const uint32_t* d_codes, const uint32_t* d_inv, const uint32_t* d_low, const uint64_t* d_win_off,
                     const uint32_t* d_win_len, uint64_t n_win, uint32_t max_win_len, const double* d_ig, int kmin,
                     int kmax, int want_rip, double* d_rows, uint32_t* d_status, uint16_t* d_dump, void* stream) {
    if (n_win == 0) return FRISK_OK;
    if (!d_codes || !d_inv || !d_win_off || !d_win_len || !d_ig || !d_rows || !d_status) return FRISK_E_INVALID;
    WinPlan p;
    int rc = frisk_internal::plan_score(kmin, kmax, max_win_len, d_dump != nullptr, &p);
    if (rc) return rc;
    if (max_win_len > FRISK_B200_MAX_WINDOW || n_win > 0xffffffffull) return FRISK_E_UNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    const int rip = want_rip && kmin <= 2 && kmax >= 2;
    switch (p.kind) {
        case WinKernel::NibbleExt:
            return frisk_internal::score_nibble_ext(p, d_codes, d_inv, d_low, d_win_off, d_win_len, n_win, max_win_len, d_ig, kmin, kmax,
                                                    rip, d_rows, d_status, st);
        case WinKernel::General:
            return frisk_internal::general_score(d_codes, d_inv, d_low, d_win_off, d_win_len, n_win, max_win_len, d_ig, kmin, kmax, rip,
                                                 d_rows, d_status, d_dump, st);
        case WinKernel::Nibble:
            return frisk_internal::score_nibble(p, d_codes, d_inv, d_low, d_win_off, d_win_len, n_win, max_win_len, d_ig, kmin, kmax, rip,
                                                d_rows, d_status, d_dump, st);
        case WinKernel::Direct:
            return frisk_internal::score_direct(p, d_codes, d_inv, d_low, d_win_off, d_win_len, n_win, max_win_len, d_ig, kmin, kmax, rip,
                                                d_rows, d_status, d_dump, st);
        case WinKernel::Small:
            return frisk_internal::score_small(p, d_codes, d_inv, d_low, d_win_off, d_win_len, n_win, d_ig, kmin, kmax, rip, d_rows,
                                               d_status, d_dump, st);
        case WinKernel::Bucket:
            return frisk_internal::score_bucket(p, d_codes, d_inv, d_low, d_win_off, d_win_len, n_win, max_win_len, d_ig, kmin, kmax, rip,
                                                d_rows, d_status, d_dump, st);
        case WinKernel::Dense:
            return frisk_internal::score_dense(d_codes, d_inv, d_low, d_win_off, d_win_len, n_win, max_win_len, d_ig, kmin, kmax, rip,
                                               d_rows, d_status, d_dump, st);
    }
    return FRISK_E_UNSUPPORTED;
}

int frisk_b200_score_sweep(const uint32_t* d_codes, const uint32_t* d_inv, const uint32_t* d_low, const uint64_t* d_win_off,
                           const uint32_t* d_win_len, uint64_t n_win, uint32_t max_win_len, const double* const* d_ig, int kmax,
                           int want_rip, double* const* d_rows, uint32_t* const* d_status, void* stream) {
    if (n_win == 0) return FRISK_OK;
    if (!d_codes || !d_inv || !d_win_off || !d_win_len || !d_ig || !d_rows || !d_status) return FRISK_E_INVALID;
    if (kmax != 8 || max_win_len > kSmemMaxWindow || n_win > 0xffffffffull) return FRISK_E_UNSUPPORTED;
    return frisk_internal::score_sweep(d_codes, d_inv, d_low, d_win_off, d_win_len, n_win, max_win_len, d_ig, want_rip, d_rows, d_status,
                                       (cudaStream_t)stream);
}

int frisk_b200_score_occupancy(int kmax, uint32_t max_win_len, int* ctas_per_sm, int* threads_per_cta) {
    if (!ctas_per_sm || !threads_per_cta) return FRISK_E_INVALID;
    WinPlan p;
    int rc = frisk_internal::plan_score(1, kmax, max_win_len, false, &p);
    if (rc) return rc;
    LaunchShape s;
    switch (p.kind) {
        case WinKernel::Dense:                              // one CTA per SM (see score_dense)
            *ctas_per_sm = 1; *threads_per_cta = frisk_internal::dense_shape(kmax).threads; return FRISK_OK;
        case WinKernel::General: *ctas_per_sm = 1; *threads_per_cta = 1024; return FRISK_OK;   // gen_score_kernel: one per SM
        case WinKernel::Small: s = frisk_internal::small_shape(p, kmax); break;
        case WinKernel::Bucket: s = frisk_internal::bucket_shape(p, kmax, max_win_len); break;
        case WinKernel::Nibble: s = frisk_internal::nibble_shape(p, kmax); break;
        case WinKernel::Direct: s = frisk_internal::direct_shape(p, kmax); break;
        case WinKernel::NibbleExt: s = frisk_internal::ext_shape(p); break;
    }
    *threads_per_cta = s.threads;
    return frisk_internal::ctas_per_sm(s, ctas_per_sm);
}

// Which window kernel frisk_b200_score launches for these parameters (the plan), spelled the way ncu prints it (without
// the "<unnamed>::" prefix and the argument list), so that a profile or a bench line is labelled from the launcher's own
// selection instead of a string constant.
int frisk_b200_score_kernel_name(int kmin, int kmax, uint32_t max_win_len, char* buf, uint64_t cap) {
    if (!buf || cap < 8) return FRISK_E_INVALID;
    WinPlan p;
    int rc = frisk_internal::plan_score(kmin, kmax, max_win_len, false, &p);
    if (rc) return rc;
    const int v = p.variant, allk = p.allk;
    switch (p.kind) {
        case WinKernel::Small: snprintf(buf, cap, "score_windows_small_kernel<%d, 0>", kmax); break;
        case WinKernel::Nibble: snprintf(buf, cap, "score_windows_nibble_kernel<%d, %d, 0, %d, 0>", kmax, v, allk); break;
        case WinKernel::Direct: snprintf(buf, cap, "score_windows_direct_kernel<%d, 256, %d, 0, %d>", kmax, v, allk); break;
        case WinKernel::Bucket: snprintf(buf, cap, "score_windows_bucket_kernel<%d, %d, 0, %d>", kmax, v, allk); break;
        case WinKernel::Dense: snprintf(buf, cap, "score_windows_kernel<%d>", kmax); break;
        case WinKernel::NibbleExt: snprintf(buf, cap, "score_windows_nibble_ext_kernel<%d, %d>", v, allk); break;
        case WinKernel::General: snprintf(buf, cap, "gen_score_kernel"); break;
    }
    return FRISK_OK;
}

int frisk_b200_set_option(const char* name, int value) {
    if (!name) return FRISK_E_INVALID;
    static const struct { const char* name; WinKernel kind; } kForce[] = {
        {"force_dense_kernel", WinKernel::Dense},   {"force_general_kernel", WinKernel::General}, {"force_bucket_kernel", WinKernel::Bucket},
        {"force_direct_kernel", WinKernel::Direct}, {"force_nibble_kernel", WinKernel::Nibble}};
    for (const auto& f : kForce)
        if (strcmp(name, f.name) == 0) {                    // the last switch set wins; clearing another one changes nothing
            if (value) g_forced = (int)f.kind;
            else if (g_forced == (int)f.kind) g_forced = -1;
            return FRISK_OK;
        }
    if (strcmp(name, "ingest_exact_open") == 0) { frisk_internal::g_ingest_exact = value; return FRISK_OK; }
    if (strcmp(name, "ingest_chunk_tiles") == 0) { frisk_internal::g_ingest_chunk_tiles = value; return FRISK_OK; }
    if (strcmp(name, "gzip_chunk_bytes") == 0) { frisk_internal::g_gzip_chunk_bytes = value; return FRISK_OK; }
    return FRISK_E_INVALID;
}

int frisk_b200_kld(const double* d_genome_ivom, const double* d_window_ivom, uint64_t n, double* d_out, void* stream) {
    if (!d_out || (n && (!d_genome_ivom || !d_window_ivom)) || n > 0xffffffffull) return FRISK_E_INVALID;
    kld_kernel<<<1, kThreads, 0, (cudaStream_t)stream>>>(d_genome_ivom, d_window_ivom, (uint32_t)n, d_out);
    CK(cudaGetLastError());
    return FRISK_OK;
}

}  // extern "C"
