// frisk_b200 general path: runtime K (1..12) and windows of any length.
//
// The reference accepts any --minWordSize/--maxWordSize/--windowlen (F:1197-1216); its defaults are
// 1..8 and 5,000.  The tuned window kernels keep a window's tables in shared memory,
// which caps them at K <= 8 and 65,535 bases.  Everything beyond that comes here: same arithmetic,
// same table/row conventions, but the tables of orders >= 7 live in a per-CTA slab of global memory
// (L2-resident for the sizes that matter) and K is a run-time value.
//
//   gen_bg_kernel            forward-strand counts, one global u64 atomic per position
//   gen_top/marginal/sym     finalise: F_x = short words + marginal of F_{x+1}; tables = F + F(revcomp)
//   gen_ivom_kernel          genome IVOM value + log2 per K-mer
//   gen_score_kernel         per window: count (orders <= 6 in shared memory, 7..K in the slab, first
//                            occurrence of every K-mer by atomicMin), score the first occurrences
//                            (summation order = position order: bit-reproducible), clean the slab by
//                            walking the positions again
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "../../include/frisk_b200.h"
#include "frisk_internal.h"

namespace {

constexpr int kGT = 1024;                 // threads per CTA of the score kernel
constexpr int kGW = kGT / 32;
constexpr int kSmemOrders = 6;            // orders 1..6 of a window are counted in shared memory
constexpr uint32_t kFullMask = 0xffffffffu;

__host__ __device__ inline uint64_t p4(int k) { return 1ull << (2 * k); }
__host__ __device__ inline uint64_t loff(int x) { return (p4(x) - 4ull) / 3ull; }   // entries of orders 1..x-1

__device__ __forceinline__ uint64_t revcomp64(uint64_t idx, int x) {
    uint64_t r = 0;
    for (int i = 0; i < x; ++i) { r = (r << 2) | ((idx & 3ull) ^ 1ull); idx >>= 2; }
    return r;
}

// ---- background ------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
gen_bg_kernel(const uint32_t* __restrict__ codes, const uint32_t* __restrict__ inv, const uint32_t* __restrict__ low,
              uint64_t word_lo, uint64_t word_hi, int K, int mask_host, unsigned long long* __restrict__ fwd) {
    const bool use_low = mask_host && low != nullptr;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t wd = word_lo + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; wd < word_hi; wd += stride) {
        uint32_t m0 = __ldg(inv + wd), m1 = __ldg(inv + wd + 1);
        if (use_low) { m0 |= __ldg(low + wd); m1 |= __ldg(low + wd + 1); }
        const uint32_t c0 = __ldg(codes + 2 * wd), c1 = __ldg(codes + 2 * wd + 1), c2 = __ldg(codes + 2 * wd + 2);
        for (int p = 0; p < 32; ++p) {
            const uint32_t c32 = p < 16 ? __funnelshift_l(c1, c0, 2 * p) : __funnelshift_l(c2, c1, 2 * (p - 16));
            const int v = min(__clz(__funnelshift_l(m1, m0, p)), K);
            if (v > 0) atomicAdd(&fwd[loff(v) + (c32 >> (32 - 2 * v))], 1ull);
        }
    }
}

// ---- finalise ----------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
gen_top_kernel(const unsigned long long* __restrict__ fwd, unsigned long long* __restrict__ tables, int K,
               unsigned long long* __restrict__ valid_kmax) {
    __shared__ unsigned long long red[8];
    const uint64_t i = (uint64_t)blockIdx.x * 256u + threadIdx.x;
    unsigned long long v = 0;
    if (i < p4(K)) { v = fwd[loff(K) + i]; tables[loff(K) + i] = v; }
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(kFullMask, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0 && valid_kmax) {
        unsigned long long s = 0;
        for (int w = 0; w < 8; ++w) s += red[w];
        if (s) atomicAdd(valid_kmax, s);
    }
}

__global__ void __launch_bounds__(256)
gen_marginal_kernel(const unsigned long long* __restrict__ fwd, unsigned long long* __restrict__ tables, int x) {
    const uint64_t t = (uint64_t)blockIdx.x * 256u + threadIdx.x;
    if (t >= p4(x)) return;
    const unsigned long long* ch = tables + loff(x + 1) + 4 * t;
    tables[loff(x) + t] = fwd[loff(x) + t] + ch[0] + ch[1] + ch[2] + ch[3];
}

__global__ void __launch_bounds__(256)
gen_sym_kernel(unsigned long long* __restrict__ tables, int K) {
    const uint64_t i = (uint64_t)blockIdx.x * 256u + threadIdx.x;
    if (i >= loff(K + 1)) return;
    int x = 1;
    for (int y = 2; y <= K; ++y) x += (i >= loff(y));
    const uint64_t b = i - loff(x), r = revcomp64(b, x);
    if (b < r) {
        const unsigned long long s = tables[i] + tables[loff(x) + r];
        tables[i] = s;
        tables[loff(x) + r] = s;
    } else if (b == r) {
        tables[i] *= 2ull;
    }
}

// ---- genome IVOM (closed form, see genome_ivom_kernel in frisk_tables.cu) ------------------------
__global__ void __launch_bounds__(256)
gen_ivom_kernel(const unsigned long long* __restrict__ tables, int kmin, int K, long long space, double2* __restrict__ ig) {
    const uint64_t kappa = (uint64_t)blockIdx.x * 256u + threadIdx.x;
    if (kappa >= p4(K)) return;
    double num = 0.0;
    unsigned long long den = 0;
    bool bad = false;
    for (int x = kmin; x <= K; ++x) {
        const unsigned long long c = tables[loff(x) + (kappa >> (2 * (K - x)))];
        const long long d = (space - (long long)(x - 1)) * 2;
        if (d == 0) bad = true;
        const double q = (double)p4(x) / (double)d;
        const double cd = (double)c;
        num = fma(q, cd * cd, num);
        den += c << (2 * x);
        if (x == kmin && c == 0) bad = true;         // W_kmin == 0: ZeroDivisionError at F:437
    }
    const double v = bad ? CUDART_NAN : num / (double)den;
    ig[kappa] = make_double2(v, log2(v));
}

// ---- window scoring ------------------------------------------------------------------------------
struct GenSmem {
    double q[12];
    double red[3][kGW];
    int n_non, n_gc, flags;
};

__global__ void __launch_bounds__(kGT, 1)
gen_score_kernel(const uint32_t* __restrict__ codes, const uint32_t* __restrict__ inv, const uint32_t* __restrict__ low,
                 const unsigned long long* __restrict__ win_off, const uint32_t* __restrict__ win_len, uint32_t n_win,
                 const double2* __restrict__ ig, int kmin, int K, int want_rip, uint32_t* __restrict__ slab, uint64_t slab_words,
                 double* __restrict__ rows, uint32_t* __restrict__ status, uint16_t* __restrict__ dump,
                 const uint32_t* __restrict__ redo_list, const uint32_t* __restrict__ redo_count) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    GenSmem& ss = *reinterpret_cast<GenSmem*>(smem_raw);
    uint32_t* stab = reinterpret_cast<uint32_t*>(smem_raw + ((sizeof(GenSmem) + 15) & ~(size_t)15));   // orders 1..min(K,6)
    const int KS = K < kSmemOrders ? K : kSmemOrders;
    const uint32_t n_stab = (uint32_t)loff(KS + 1);
    uint32_t* sfirst = stab + n_stab;                                  // first-occurrence table when K <= 6
    uint32_t* gtab = slab + (uint64_t)blockIdx.x * slab_words;         // orders 7..K, then first occurrence (K >= 7)
    uint32_t* first = K <= kSmemOrders ? sfirst : gtab + (loff(K + 1) - loff(kSmemOrders + 1));
    const uint32_t n_first_smem = K <= kSmemOrders ? (uint32_t)p4(K) : 0u;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    auto cnt = [&](int x) -> uint32_t* {      // table of order x
        return x <= kSmemOrders ? stab + loff(x) : gtab + (loff(x) - loff(kSmemOrders + 1));
    };

    for (uint32_t i = tid; i < n_stab; i += kGT) stab[i] = 0;
    for (uint32_t i = tid; i < n_first_smem; i += kGT) sfirst[i] = kFullMask;
    if (tid == 0) { ss.n_non = 0; ss.n_gc = 0; ss.flags = 0; }
    __syncthreads();

    // Second launch behind the kmax 9..12 kernel (frisk_nibble_ext.cu): only the windows it handed over, as a compacted
    // list.  A CTA without work leaves at once; one with work initialises its own slab (the host skipped that: the slab
    // of a launch that usually has nothing to do is not worth 100+ MB of memset per CTA).
    const uint32_t n_todo = redo_list ? *redo_count : n_win;
    if (redo_list) {
        if (blockIdx.x >= n_todo) return;
        if (K > kSmemOrders) {
            const uint64_t count_words = loff(K + 1) - loff(kSmemOrders + 1);
            for (uint64_t i = tid; i < count_words; i += kGT) gtab[i] = 0u;
            for (uint64_t i = tid; i < (uint64_t)p4(K); i += kGT) gtab[count_words + i] = kFullMask;
        }
        __syncthreads();
    }
    for (uint32_t todo = blockIdx.x; todo < n_todo; todo += gridDim.x) {
        const uint32_t win = redo_list ? redo_list[todo] : todo;
        const uint64_t o = win_off[win];
        const uint32_t len = win_len[win];
        // one position: 16 bases of codes from it, unresolved mask of the 32 bases from it, v = longest valid word (<= K)
        auto fetch = [&](uint32_t p, uint32_t& c32, int& v, uint32_t& unres) {
            const uint64_t a = o + p, wi = a >> 4, mi = a >> 5;
            c32 = __funnelshift_l(__ldg(codes + wi + 1), __ldg(codes + wi), (uint32_t)(a & 15) * 2u);
            const uint32_t m = __funnelshift_l(__ldg(inv + mi + 1), __ldg(inv + mi), (uint32_t)(a & 31));
            const uint32_t lb = low ? (__ldg(low + mi) << (uint32_t)(a & 31)) >> 31 : 0u;
            unres = (m >> 31) | lb;
            const uint32_t rest = len - p;
            v = min(min(__clz(m), K), (int)(rest < 12u ? rest : 12u));
        };

        // ---- P1: count every order, elect the first occurrence of every K-mer -------------------
        int non = 0, gc = 0;
        for (uint32_t p = tid; p < len; p += kGT) {
            uint32_t c32, unres; int v;
            fetch(p, c32, v, unres);
            non += (int)unres;
            gc += (int)((1u - unres) & (c32 >> 31));                    // G = 2, C = 3: high bit of the first base
            for (int x = 1; x <= v; ++x) atomicAdd(cnt(x) + (c32 >> (32 - 2 * x)), 1u);
            if (v == K) atomicMin(first + (c32 >> (32 - 2 * K)), p);
        }
        non = __reduce_add_sync(kFullMask, non);
        gc = __reduce_add_sync(kFullMask, gc);
        if (lane == 0 && (non | gc)) { atomicAdd(&ss.n_non, non); atomicAdd(&ss.n_gc, gc); }
        __syncthreads();
        const int n_non = ss.n_non, n_gc = ss.n_gc, n_up = (int)len - n_non;
        const bool excluded = (double)n_non >= 0.3 * (double)len;      // F:238 / F:213
        if (tid < K) {
            const int x = tid + 1;
            const long long d = ((long long)n_up - (long long)(x - 1)) * 2;
            ss.q[tid] = (double)p4(x) / (double)d;
        }
        uint32_t n_at = 0, n_ta = 0, n_sub = 0, n_prod = 0;
        if (tid == 0 && want_rip && K >= 2) {                           // calcRIP's dinucleotides (F:474-495)
            const uint32_t* di = cnt(2);
            n_at = di[1]; n_ta = di[4]; n_sub = di[3] + di[9]; n_prod = di[12] + di[6];
        }
        __syncthreads();

        // ---- P2: score the first occurrences ----------------------------------------------------
        double s_w = 0.0, s_g = 0.0, s_t = 0.0;
        uint32_t n_kmers = 0;
        if (!excluded) {
            for (uint32_t p = tid; p < len; p += kGT) {
                uint32_t c32, unres; int v;
                fetch(p, c32, v, unres);
                if (dump) {                                             // tests only (windows <= 65,535 bases)
                    uint16_t* d = dump + (size_t)win * loff(K + 1);
                    for (int x = 1; x <= v; ++x) {
                        const uint32_t idx = c32 >> (32 - 2 * x);
                        d[loff(x) + idx] = (uint16_t)cnt(x)[idx];
                    }
                }
                if (v != K) continue;
                const uint32_t kappa = c32 >> (32 - 2 * K);
                if (first[kappa] != p) continue;
                double num = 0.0, den = 0.0;
                for (int x = kmin; x <= K; ++x) {
                    const double c = (double)cnt(x)[c32 >> (32 - 2 * x)];
                    num = fma(ss.q[x - 1], c * c, num);
                    den = fma((double)p4(x), c, den);
                }
                const double iw = num / den;
                const double2 g = __ldg(ig + kappa);
                s_w += iw;
                s_g += g.x;
                s_t = fma(iw, log2(iw) - g.y, s_t);
                ++n_kmers;
            }
        }
#pragma unroll
        for (int ofs = 16; ofs; ofs >>= 1) {
            s_w += __shfl_xor_sync(kFullMask, s_w, ofs);
            s_g += __shfl_xor_sync(kFullMask, s_g, ofs);
            s_t += __shfl_xor_sync(kFullMask, s_t, ofs);
        }
        n_kmers = __reduce_add_sync(kFullMask, n_kmers);
        if (lane == 0) {
            ss.red[0][warp] = s_w; ss.red[1][warp] = s_g; ss.red[2][warp] = s_t;
            if (n_kmers) atomicOr(&ss.flags, 1);
        }
        __syncthreads();

        // ---- P3: the row; clean the tables by walking the positions once more ---------------------
        if (tid == 0) {
            double* row = rows + (size_t)win * 5;
            if (excluded) {
                status[win] = FRISK_ROW_EXCLUDED;
                for (int c = 0; c < 5; ++c) row[c] = CUDART_NAN;
            } else {
                double a = 0, b = 0, c = 0;
                for (int w = 0; w < kGW; ++w) { a += ss.red[0][w]; b += ss.red[1][w]; c += ss.red[2][w]; }
                uint32_t st = 0;
                double kld = 0.0;                                        // no kmax-mer in the window: the reference returns 0
                if (ss.flags & 1) {
                    bool zd = b != b;                                    // NaN genome entry: ZeroDivisionError at F:437
                    for (int x = kmin; x <= K; ++x) zd |= ((long long)n_up - (long long)(x - 1)) == 0;
                    if (zd) { st |= FRISK_ROW_KLD_ZERODIV; kld = CUDART_NAN; }
                    else {
                        kld = c / a + (log2(b) - log2(a));
                        if (!(kld == kld) || isinf(kld)) st |= FRISK_ROW_LOG_DOMAIN;
                    }
                }
                row[0] = kld;
                if (n_up == 0) { st |= FRISK_ROW_GC_ZERODIV; row[1] = CUDART_NAN; }
                else row[1] = (double)n_gc / (double)n_up;               // F:136
                double pi = CUDART_NAN, si = CUDART_NAN, cri = CUDART_NAN;
                if (want_rip && K >= 2) {
                    if (n_at > 0) pi = (double)n_ta / (double)n_at;
                    if (n_sub > 0) si = (double)n_prod / (double)n_sub;
                    if (pi != 0.0 && si != 0.0) cri = pi - si;           // F:491: 0.0 falsy, NaN truthy
                }
                row[2] = pi; row[3] = si; row[4] = cri;
                status[win] = st;
            }
            ss.n_non = 0; ss.n_gc = 0; ss.flags = 0;
        }
        if (K > kSmemOrders) {
            for (uint32_t p = tid; p < len; p += kGT) {
                uint32_t c32, unres; int v;
                fetch(p, c32, v, unres);
                for (int x = kSmemOrders + 1; x <= v; ++x) cnt(x)[c32 >> (32 - 2 * x)] = 0;
                if (v == K) first[c32 >> (32 - 2 * K)] = kFullMask;
            }
        }
        for (uint32_t i = tid; i < n_stab; i += kGT) stab[i] = 0;
        for (uint32_t i = tid; i < n_first_smem; i += kGT) sfirst[i] = kFullMask;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256) gen_zero_dump_kernel(uint16_t* dump, uint64_t n) {
    const uint64_t stride = (uint64_t)gridDim.x * 256u;
    for (uint64_t i = (uint64_t)blockIdx.x * 256u + threadIdx.x; i < n; i += stride) dump[i] = 0;
}

int sms() {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
    return n;
}

// indices of the windows marked kRowRedo, in any order
__global__ void __launch_bounds__(256)
gen_compact_kernel(const uint32_t* __restrict__ marks, uint32_t n, uint32_t* __restrict__ list, uint32_t* __restrict__ count) {
    const uint32_t i = blockIdx.x * 256u + threadIdx.x;
    if (i < n && (marks[i] & frisk_internal::kRowRedo)) list[atomicAdd(count, 1u)] = i;
}

}  // namespace

namespace frisk_internal {

int general_background(const uint32_t* codes, const uint32_t* inv, const uint32_t* low, uint64_t w_lo, uint64_t w_hi, int K,
                       int mask_host, uint64_t* fwd, cudaStream_t st) {
    const int n = sms();
    if (n <= 0) return FRISK_E_NO_DEVICE;
    uint64_t grid = (w_hi - w_lo + 255) / 256;
    if (grid > (uint64_t)n * 8) grid = (uint64_t)n * 8;
    if (grid == 0) return FRISK_OK;
    gen_bg_kernel<<<(unsigned)grid, 256, 0, st>>>(codes, inv, low, w_lo, w_hi, K, mask_host,
                                                  reinterpret_cast<unsigned long long*>(fwd));
    FRISK_CK(cudaGetLastError());
    return FRISK_OK;
}

int general_finalize(const uint64_t* fwd, int K, int symmetric, uint64_t* tables, uint64_t* valid, cudaStream_t st) {
    auto f = reinterpret_cast<const unsigned long long*>(fwd);
    auto t = reinterpret_cast<unsigned long long*>(tables);
    if (valid) FRISK_CK(cudaMemsetAsync(valid, 0, sizeof(uint64_t), st));
    gen_top_kernel<<<(unsigned)((p4(K) + 255) / 256), 256, 0, st>>>(f, t, K, reinterpret_cast<unsigned long long*>(valid));
    for (int x = K - 1; x >= 1; --x)
        gen_marginal_kernel<<<(unsigned)((p4(x) + 255) / 256), 256, 0, st>>>(f, t, x);
    if (symmetric) gen_sym_kernel<<<(unsigned)((loff(K + 1) + 255) / 256), 256, 0, st>>>(t, K);
    FRISK_CK(cudaGetLastError());
    return FRISK_OK;
}

int general_genome_ivom(const uint64_t* tables, int kmin, int K, int64_t space, double* ig, cudaStream_t st) {
    gen_ivom_kernel<<<(unsigned)((p4(K) + 255) / 256), 256, 0, st>>>(reinterpret_cast<const unsigned long long*>(tables), kmin, K,
                                                                    (long long)space, reinterpret_cast<double2*>(ig));
    FRISK_CK(cudaGetLastError());
    return FRISK_OK;
}

int general_score(const WinPlan&, const WinJob& j, const uint32_t* redo_src, int grid_cap) {
    const uint64_t n_win = j.n_win;
    const int K = j.K;
    const cudaStream_t st = j.st;
    if (j.dump && j.max_len > 65535u) return FRISK_E_UNSUPPORTED;      // the test dump is 16-bit
    const int n = sms();
    if (n <= 0) return FRISK_E_NO_DEVICE;
    uint64_t grid = (uint64_t)n;
    if (grid_cap > 0 && grid > (uint64_t)grid_cap) grid = (uint64_t)grid_cap;   // a hand-over launch: few windows, small slab
    if (grid > n_win) grid = n_win;
    // per-CTA slab: orders 7..K (u32 counts) + first-occurrence position per K-mer
    const uint64_t slab_words = K > kSmemOrders ? (loff(K + 1) - loff(kSmemOrders + 1)) + p4(K) : 0;
    uint32_t* slab = nullptr;
    if (slab_words) {
        const uint64_t count_words = loff(K + 1) - loff(kSmemOrders + 1);
        { const int rc = pool_ready(); if (rc) return rc; }
        // stream-ordered: up to 156 MB per CTA at K = 12, handed back as soon as the kernel is done
        FRISK_CK(cudaMallocAsync((void**)&slab, (size_t)(grid * slab_words * 4), st));
        for (uint64_t c = 0; c < grid && !redo_src; ++c) {             // counts = 0, first = "none" (hand-over launch: in the kernel)
            FRISK_CK(cudaMemsetAsync(slab + c * slab_words, 0, count_words * 4, st));
            FRISK_CK(cudaMemsetAsync(slab + c * slab_words + count_words, 0xff, p4(K) * 4, st));
        }
    }
    // hand-over launch: compact the marked windows into a list first (a CTA scanning the marks one by one would spend a
    // global-memory round trip per window)
    uint32_t* redo_list = nullptr;
    uint32_t* redo_count = nullptr;
    if (redo_src) {
        { const int rc = pool_ready(); if (rc) return rc; }
        FRISK_CK(cudaMallocAsync((void**)&redo_list, (size_t)(n_win + 1) * 4, st));
        redo_count = redo_list + n_win;
        FRISK_CK(cudaMemsetAsync(redo_count, 0, 4, st));
        gen_compact_kernel<<<(unsigned)((n_win + 255) / 256), 256, 0, st>>>(redo_src, (uint32_t)n_win, redo_list, redo_count);
    }
    const int KS = K < kSmemOrders ? K : kSmemOrders;
    const size_t smem = ((sizeof(GenSmem) + 15) & ~(size_t)15) + (size_t)loff(KS + 1) * 4 + (K <= kSmemOrders ? (size_t)p4(K) * 4 : 0);
    FRISK_CK(cudaFuncSetAttribute(gen_score_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (j.dump) gen_zero_dump_kernel<<<1024, 256, 0, st>>>(j.dump, n_win * loff(K + 1));
    gen_score_kernel<<<(unsigned)grid, kGT, smem, st>>>(j.codes, j.inv, j.low, reinterpret_cast<const unsigned long long*>(j.win_off),
                                                       j.win_len, (uint32_t)n_win, reinterpret_cast<const double2*>(j.ig), j.kmin, K,
                                                       j.rip, slab, slab_words, j.rows, j.status, j.dump, redo_list, redo_count);
    FRISK_CK(cudaGetLastError());
    if (redo_list) FRISK_CK(cudaFreeAsync(redo_list, st));
    if (slab) FRISK_CK(cudaFreeAsync(slab, st));
    return FRISK_OK;
}

}  // namespace frisk_internal
