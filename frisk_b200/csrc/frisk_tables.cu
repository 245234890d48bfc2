// frisk_b200: the genome tables -- forward-strand k-mer counts of the genome, the tables of orders 1..K (both strands)
// and the genome IVOM of every kmax-mer -- and their C-ABI launchers.
//
// Replaces the reference's genome pass (/root/reference/frisk/__init__.py F:321-351: computeKmers over the host, the
// lower orders and the reverse strand) and its genome-side IvomBuild (F:411-450).  Nothing here is a translation of it
// (the reference is a Python dict loop); see DESIGN.md for the derivation.
//
//   bg_count_kernel, bg_reduce_kernel      forward-strand k-mer counts of the genome (F:321-351, counting)
//   forward_totals_kernel,                 marginalise orders K-1..1 + add the reverse strand (F:348-351), as the
//   forward_low_kernel, symmetrise_kernel  staged entry points frisk_b200_finalize_tables(_peers) launch them
//   genome_ivom_kernel                     per-kmax-mer genome IVOM value and its log2 (F:411-450)
//   finalize_ivom_kernel                   the finalising steps and the genome IVOM as one cooperative launch
//
// Table index convention everywhere: base-4 number, digits A=0 T=1 G=2 C=3, first base most
// significant (the reference's dict key order, F:70/F:253-274); complement = digit ^ 1.
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include <atomic>

#include "../../include/frisk_b200.h"
#include "frisk_internal.h"
#include "frisk_device.cuh"

namespace {

constexpr int kThreads = 1024;          // bg_count_kernel: one CTA per SM, the 4^8 u16 counters take 128 KiB of smem

// reverse complement of the x-mer with index idx (F:276-278): reverse the digits, xor each with 1
__device__ __forceinline__ uint32_t revcomp_idx(uint32_t idx, int x) {
    uint32_t r = __brev(idx) >> (32 - 2 * x);                       // digits reversed, bits inside a digit swapped
    r = ((r >> 1) & 0x55555555u) | ((r & 0x55555555u) << 1);         // swap them back
    return r ^ (0x55555555u & (pow4(x) - 1u));
}

// ============================================================================================
// Background: forward-strand counts.  Each CTA owns a contiguous run of 32-base mask words and
// histograms the order-K codes into a shared-memory table of u16 counters, two per 32-bit word
// (4^8 bins = 128 KiB: the whole code space in one pass), then stores the table as its partial
// result; bg_reduce_kernel sums the partials into the global u64 table.  A 16-bit counter that
// wraps is made exact by the thread whose atomic caused the wrap (it sees the old word): it adds
// 65,536 to the global bin and, when the low half's carry leaked into the high half, takes that 1
// back out of the neighbour's global bin -- no second shared-memory operation, so no transient
// state another thread could misread.  Positions whose K-word is invalid but which start a shorter
// valid word (scaffold ends, N boundaries) add 1 to the order-v table directly in global memory.
// ============================================================================================
__device__ __noinline__ void bg_wrapped(unsigned long long* __restrict__ fwd_k, uint32_t code, uint32_t old) {
    atomicAdd(&fwd_k[code], 65536ull);
    if (!(code & 1u))       // low half: its carry bumped the high half (or wrapped it: old word all ones)
        atomicAdd(&fwd_k[code | 1u], old == 0xffffffffu ? 65535ull : ~0ull);
}

__device__ __forceinline__ void bg_add(uint32_t* tab, unsigned long long* __restrict__ fwd_k, uint32_t code) {
    const uint32_t sh = (code & 1u) * 16u;
    const uint32_t old = atomicAdd(&tab[code >> 1], 1u << sh);
    if (((old >> sh) & 0xffffu) == 0xffffu) bg_wrapped(fwd_k, code, old);
}

// ~(old | other half) == 0  <=>  the half that was incremented held 0xffff
__device__ __forceinline__ uint32_t bg_room(uint32_t old, uint32_t sh) { return ~(old | (0xffff0000u >> sh)); }

template <int K>
__global__ void __launch_bounds__(kThreads, 1)
bg_count_kernel(const uint32_t* __restrict__ codes, const uint32_t* __restrict__ inv, const uint32_t* __restrict__ low,
                uint64_t word_lo, uint64_t word_hi, int mask_host, unsigned long long* __restrict__ fwd,
                uint32_t* __restrict__ partial, const unsigned long long* __restrict__ d_range) {
    constexpr uint32_t NB = pow4(K);
    constexpr uint32_t NW = NB / 2u;                       // shared words: two u16 bins each
    extern __shared__ __align__(16) uint32_t tab[];
    if (d_range) { word_lo = d_range[0]; word_hi = d_range[1]; }     // range produced on the device (streamed FASTA ingest)
    const uint64_t n_words = word_hi - word_lo;
    const uint64_t per = (n_words + gridDim.x - 1) / gridDim.x;
    const uint64_t w0 = word_lo + per * blockIdx.x;
    uint64_t w1 = w0 + per;
    if (w1 > word_hi) w1 = word_hi;
    const bool use_low = mask_host && low != nullptr;
    unsigned long long* fwd_k = fwd + lvl_off(K);

    for (uint32_t b = threadIdx.x; b < NW; b += kThreads) tab[b] = 0;
    __syncthreads();
    for (uint64_t wd = w0 + threadIdx.x; wd < w1; wd += kThreads) {
        uint32_t m0 = __ldg(inv + wd), m1 = __ldg(inv + wd + 1);
        if (use_low) { m0 |= __ldg(low + wd); m1 |= __ldg(low + wd + 1); }
        const uint32_t c0 = __ldg(codes + 2 * wd), c1 = __ldg(codes + 2 * wd + 1), c2 = __ldg(codes + 2 * wd + 2);
        const bool all_valid = (m0 == 0u) && (K == 1 || (m1 >> ((33 - K) & 31)) == 0u);
        if (all_valid) {                                   // the common word: 32 full K-words, no per-position checks
            // all 32 atomics are issued before any of their results is looked at; a wrap (rare) is
            // detected through one running minimum and handled after the fact
            uint32_t olds[32], room = 0xffffffffu;
#pragma unroll
            for (int p = 0; p < 32; ++p) {
                const uint32_t code = (p < 16 ? __funnelshift_l(c1, c0, 2 * p) : __funnelshift_l(c2, c1, 2 * (p - 16)))
                                      >> (32 - 2 * K);
                const uint32_t sh = (code & 1u) * 16u;
                olds[p] = atomicAdd(&tab[code >> 1], 1u << sh);
                room = min(room, bg_room(olds[p], sh));
            }
            if (room == 0u) {
#pragma unroll 1
                for (int p = 0; p < 32; ++p) {
                    const uint32_t code = (p < 16 ? __funnelshift_l(c1, c0, 2 * p) : __funnelshift_l(c2, c1, 2 * (p - 16)))
                                          >> (32 - 2 * K);
                    uint32_t old = 0;
#pragma unroll
                    for (int q = 0; q < 32; ++q) if (q == p) old = olds[q];
                    if (bg_room(old, (code & 1u) * 16u) == 0u) bg_wrapped(fwd_k, code, old);
                }
            }
        } else {
#pragma unroll 4
            for (int p = 0; p < 32; ++p) {
                const uint32_t code = (p < 16 ? __funnelshift_l(c1, c0, 2 * p) : __funnelshift_l(c2, c1, 2 * (p - 16)))
                                      >> (32 - 2 * K);
                const int v = min(__clz(__funnelshift_l(m1, m0, p)), K);
                if (v == K) bg_add(tab, fwd_k, code);
                else if (v > 0) atomicAdd(&fwd[lvl_off(v) + (code >> (2 * (K - v)))], 1ull);
            }
        }
    }
    __syncthreads();
    if (partial) {   // per-CTA partial table (raw words), coalesced stores
        uint32_t* dst = partial + (size_t)blockIdx.x * NW;
        if constexpr (NW >= 4u * kThreads) {
            for (uint32_t b = threadIdx.x * 4u; b < NW; b += kThreads * 4u)
                *reinterpret_cast<uint4*>(dst + b) = *reinterpret_cast<const uint4*>(tab + b);
        } else {
            for (uint32_t b = threadIdx.x; b < NW; b += kThreads) dst[b] = tab[b];
        }
    } else {
        for (uint32_t b = threadIdx.x; b < NW; b += kThreads) {
            const uint32_t c = tab[b];
            if (c & 0xffffu) atomicAdd(&fwd_k[2u * b], (unsigned long long)(c & 0xffffu));
            if (c >> 16) atomicAdd(&fwd_k[2u * b + 1u], (unsigned long long)(c >> 16));
        }
    }
}

// fwd[order K][2w], [2w+1] += sum over CTAs of the two halves of partial[cta][w].  A CTA handles 32
// consecutive words (coalesced across lanes); its 8 warps split the partial tables between them.
template <int K>
__global__ void __launch_bounds__(256)
bg_reduce_kernel(const uint32_t* __restrict__ partial, int n_parts, unsigned long long* __restrict__ fwd) {
    constexpr uint32_t NW = pow4(K) / 2u;
    __shared__ unsigned long long acc[8][32][2];
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    const uint32_t w = blockIdx.x * 32u + lane;
    unsigned long long lo = 0, hi = 0;
    if (w < NW) {
#pragma unroll 4
        for (int c = (int)warp; c < n_parts; c += 8) {
            const uint32_t v = partial[(size_t)c * NW + w];
            lo += v & 0xffffu;
            hi += v >> 16;
        }
    }
    acc[warp][lane][0] = lo; acc[warp][lane][1] = hi;
    __syncthreads();
    if (warp == 0 && w < NW) {
#pragma unroll
        for (int j = 1; j < 8; ++j) { lo += acc[j][lane][0]; hi += acc[j][lane][1]; }
        if (lo) fwd[lvl_off(K) + 2u * w] += lo;
        if (hi) fwd[lvl_off(K) + 2u * w + 1u] += hi;
    }
}

// Finalising the tables: F_x = short-word counts of order x + marginal of F_{x+1}; then
// tables = F + F(revcomp).  Three small launches instead of one serial CTA:
//   forward_totals_kernel   one CTA per order-R subtree (R = K-4): F_x for x = R..K
//   forward_low_kernel      one CTA: F_x for x = R-1..1 (<= 84 bins)
//   symmetrise_kernel       one thread per table entry, each {kmer, revcomp} pair handled once
// Where the forward counters come from: this GPU's buffer, or -- multi-GPU, fused all-reduce -- the sum
// over every rank's buffer read directly through NVLink peer mappings (no separate collective, no
// staging copy: the reduction happens in the registers of the kernel that needs the sums).
struct LocalFwd {
    const unsigned long long* p;
    const long long* space_dev = nullptr;     // genome space in device memory (frisk_b200_run_fasta: the host does not know it yet)
    __device__ __forceinline__ unsigned long long operator()(uint32_t i) const { return p[i]; }
    __device__ __forceinline__ void arrive_and_wait() const {}
    __device__ __forceinline__ long long space(long long by_value) const { return space_dev ? *space_dev : by_value; }
};
using frisk_internal::kMaxPeers;
struct PeerFwd {
    const unsigned long long* p[kMaxPeers];
    unsigned long long* flags[kMaxPeers];     // flags[q][r]: "rank r's counters of epoch >= value are complete", in rank q's memory
    int n, rank;
    unsigned long long epoch;                 // 0: the caller already synchronised the GPUs
    __device__ __forceinline__ long long space(long long by_value) const { return by_value; }
    __device__ __forceinline__ unsigned long long operator()(uint32_t i) const {
        // every peer's load is issued before any of them is consumed: a loop over the run-time `n` with the running sum in
        // it makes each NVLink round trip wait for the one before (8 ranks: 8 exposed latencies per counter instead of 1)
        unsigned long long v[kMaxPeers];
#pragma unroll
        for (int q = 0; q < kMaxPeers; ++q) v[q] = q < n ? __ldcv(p[q] + i) : 0ull;   // written before the peers' arrival below
        unsigned long long s = 0;
#pragma unroll
        for (int q = 0; q < kMaxPeers; ++q) s += v[q];
        return s;
    }
    // Cross-GPU barrier folded into the first kernel that needs the peers' counters: this rank's count
    // kernels are complete (stream order), so CTA 0 posts the epoch into every peer's flag array; every
    // CTA then waits until all ranks have posted into ours.  A peer that never arrives (a rank died) traps
    // after ~10 s instead of hanging the GPU.
    __device__ __forceinline__ void arrive_and_wait() const {
        if (epoch == 0) return;
        if (blockIdx.x == 0 && (int)threadIdx.x < n) {
            __threadfence_system();
            asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(flags[threadIdx.x] + rank), "l"(epoch) : "memory");
        }
        if (threadIdx.x == 0) {
            const long long t0 = clock64();
            for (int q = 0; q < n; ++q) {
                unsigned long long seen;
                do {
                    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(seen) : "l"(flags[rank] + q) : "memory");
                    if (seen < epoch && clock64() - t0 > 20000000000ll) __trap();
                } while (seen < epoch);
            }
        }
        __syncthreads();
    }
};

template <int K, typename Fwd>
__device__ __forceinline__ void forward_totals_body(const Fwd& fwd, unsigned long long* __restrict__ tables,
                                                    unsigned long long* __restrict__ valid_kmax, uint32_t root,
                                                    unsigned long long (*lvl)[256], unsigned long long* red) {
    constexpr int R = K > 4 ? K - 4 : 0;
    const uint32_t t = threadIdx.x;
    uint32_t n = pow4(K - R);                         // subtree nodes at the current order
    // every counter this thread will need is requested up front (with peer buffers each is a round
    // trip over NVLink: one exposed latency instead of one per level)
    constexpr int LV = K - (R > 1 ? R : 1);           // levels below the top handled here
    unsigned long long own[LV > 0 ? LV : 1];
    unsigned long long v = 0;
    if (t < n) v = fwd(lvl_off(K) + root * n + t);
    {
        uint32_t m = n;
#pragma unroll
        for (int i = 0; i < LV; ++i) {
            m >>= 2;
            own[i] = (t < m) ? fwd(lvl_off(K - 1 - i) + root * m + t) : 0ull;
        }
    }
    if (t < n) {
        tables[lvl_off(K) + root * n + t] = v;
        lvl[0][t] = v;
    }
    unsigned long long local = v;                     // valid K-words of this subtree
    for (int o = 16; o; o >>= 1) local += __shfl_xor_sync(kFull, local, o);
    if ((t & 31) == 0) red[t >> 5] = local;
    __syncthreads();
    if (t == 0 && valid_kmax) {
        unsigned long long sum = 0;
        for (int w = 0; w < 8; ++w) sum += red[w];
        if (sum) atomicAdd(valid_kmax, sum);
    }
    int cur = 0;
#pragma unroll
    for (int i = 0; i < LV; ++i) {
        const int x = K - 1 - i;
        n >>= 2;
        if (t < n) {
            const unsigned long long* ch = &lvl[cur][4 * t];
            const unsigned long long f = own[i] + ch[0] + ch[1] + ch[2] + ch[3];
            tables[lvl_off(x) + root * n + t] = f;
            lvl[cur ^ 1][t] = f;
        }
        cur ^= 1;
        __syncthreads();
    }
}

template <int K, typename Fwd>
__global__ void __launch_bounds__(256)
forward_totals_kernel(const Fwd fwd, unsigned long long* __restrict__ tables,
                      unsigned long long* __restrict__ valid_kmax) {
    __shared__ unsigned long long lvl[2][256];
    __shared__ unsigned long long red[8];
    fwd.arrive_and_wait();
    forward_totals_body<K, Fwd>(fwd, tables, valid_kmax, blockIdx.x, lvl, red);
}

template <int K, typename Fwd>
__device__ __forceinline__ void forward_low_body(const Fwd& fwd, unsigned long long* __restrict__ tables) {
    constexpr int R = K > 4 ? K - 4 : 0;
    const uint32_t t = threadIdx.x;
    unsigned long long own[R > 1 ? R - 1 : 1];         // this thread's counter of every level, requested up front
#pragma unroll
    for (int x = R - 1; x >= 1; --x) own[x - 1] = (t < pow4(x)) ? fwd(lvl_off(x) + t) : 0ull;
#pragma unroll
    for (int x = R - 1; x >= 1; --x) {
        if (t < pow4(x)) {
            // (L2 loads: in the fused kernel these entries were written by other CTAs earlier in the same launch)
            const unsigned long long* ch = tables + lvl_off(x + 1) + 4 * t;
            tables[lvl_off(x) + t] = own[x - 1] + __ldcg(ch) + __ldcg(ch + 1) + __ldcg(ch + 2) + __ldcg(ch + 3);
        }
        __syncthreads();
    }
}

template <int K, typename Fwd>
__global__ void __launch_bounds__(64)
forward_low_kernel(const Fwd fwd, unsigned long long* __restrict__ tables) {
    forward_low_body<K, Fwd>(fwd, tables);
}

template <int K>
__device__ __forceinline__ void symmetrise_entry(unsigned long long* __restrict__ tables, uint32_t i) {
    int x = 1;
#pragma unroll
    for (int y = 2; y <= K; ++y) x += (i >= lvl_off(y));
    const uint32_t b = i - lvl_off(x);
    const uint32_t r = revcomp_idx(b, x);
    if (b < r) {
        const unsigned long long sum = __ldcg(tables + i) + __ldcg(tables + lvl_off(x) + r);
        tables[i] = sum;
        tables[lvl_off(x) + r] = sum;
    } else if (b == r) {
        tables[i] = 2ull * __ldcg(tables + i);      // palindrome: +1 word, +1 its own reverse complement
    }
}

template <int K>
__global__ void __launch_bounds__(256)
symmetrise_kernel(unsigned long long* __restrict__ tables) {
    const uint32_t i = blockIdx.x * 256 + threadIdx.x;
    if (i < lvl_off(K + 1)) symmetrise_entry<K>(tables, i);
}

// Genome-side IVOM of every K-mer.  The reference's recurrence (F:426-446)
//     a_x = w_x / W_x,  I_x = a_x p_x + (1 - a_x) I_{x-1},  W_x = sum_{y<=x} w_y
// telescopes (multiply by W_x):  W_x I_x = w_x p_x + W_{x-1} I_{x-1}, hence
//     I_K = sum_x w_x p_x / sum_x w_x,   w_x = C_x 4^x,  p_x = C_x / ((S-(x-1)) 2).
// One division per k-mer instead of sixteen; agreement with the sequential form ~1e-15 relative.
template <int K>
__device__ __forceinline__ void genome_ivom_entry(const unsigned long long* __restrict__ tables, int kmin, long long space,
                                                  double2* __restrict__ ig, uint32_t kappa) {
    double num = 0.0;
    unsigned long long den = 0;
    bool bad = false;
#pragma unroll
    for (int x = 1; x <= K; ++x) {
        if (x < kmin) continue;
        const unsigned long long c = __ldcg(tables + lvl_off(x) + (kappa >> (2 * (K - x))));
        const long long d = (space - (long long)(x - 1)) * 2;
        if (d == 0) bad = true;
        const double q = (double)pow4(x) / (double)d;
        const double cd = (double)c;
        num = fma(q, cd * cd, num);
        den += c << (2 * x);
        if (x == kmin && c == 0) bad = true;      // W_kmin == 0: ZeroDivisionError at F:437
    }
    double v = bad ? CUDART_NAN : num / (double)den;
    ig[kappa] = make_double2(v, log2(v));
}

template <int K>
__global__ void genome_ivom_kernel(const unsigned long long* __restrict__ tables, int kmin, long long space,
                                   double2* __restrict__ ig) {
    const uint32_t kappa = blockIdx.x * blockDim.x + threadIdx.x;
    if (kappa < pow4(K)) genome_ivom_entry<K>(tables, kmin, space, ig, kappa);
}

// The four finalising steps + the genome IVOM table as ONE cooperative launch (grid-wide barriers instead
// of five launch boundaries: 23 us -> ~10 us).  With peer counters the cross-GPU arrival happens first.
template <int K, typename Fwd>
__global__ void __launch_bounds__(256)
finalize_ivom_kernel(const Fwd fwd, unsigned long long* __restrict__ tables, unsigned long long* __restrict__ valid_kmax,
                     int kmin, long long space, double2* __restrict__ ig) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    constexpr int R = K > 4 ? K - 4 : 0;
    __shared__ unsigned long long lvl[2][256];
    __shared__ unsigned long long red[8];
    fwd.arrive_and_wait();
    for (uint32_t root = blockIdx.x; root < pow4(R); root += gridDim.x) {
        forward_totals_body<K, Fwd>(fwd, tables, valid_kmax, root, lvl, red);
        __syncthreads();
    }
    grid.sync();
    if (R > 1) {
        if (blockIdx.x == 0) forward_low_body<K, Fwd>(fwd, tables);
        grid.sync();
    }
    const uint32_t gtid = blockIdx.x * 256 + threadIdx.x, gstride = gridDim.x * 256;
    for (uint32_t i = gtid; i < lvl_off(K + 1); i += gstride) symmetrise_entry<K>(tables, i);
    grid.sync();
    const long long sp = fwd.space(space);
    for (uint32_t kappa = gtid; kappa < pow4(K); kappa += gstride) genome_ivom_entry<K>(tables, kmin, sp, ig, kappa);
}

using frisk_internal::check_k;
using frisk_internal::sm_count_cached;
#define CK(call) FRISK_CK(call)

template <int K>
int launch_background(const uint32_t* codes, const uint32_t* inv, const uint32_t* low, uint64_t w_lo, uint64_t w_hi,
                      int mask_host, uint64_t* fwd, cudaStream_t st, const unsigned long long* d_range = nullptr) {
    // d_range: the kernel reads its range from device memory; [w_lo, w_hi) then only sizes the grid
    constexpr uint32_t NB = pow4(K);
    constexpr uint32_t NW = NB / 2u;
    const size_t smem = (size_t)NW * 4;
    CK(cudaFuncSetAttribute(bg_count_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const uint64_t n_words = w_hi - w_lo;
    int grid = sm_count_cached();
    if (grid <= 0) return FRISK_E_NO_DEVICE;
    // at least ~2 rounds of 1024 words per CTA, otherwise fewer CTAs
    const uint64_t want = (n_words + 2047) / 2048;
    if ((uint64_t)grid > want) grid = want ? (int)want : 1;
    // large tables: per-CTA partial tables + one reduction instead of ~65 k global atomics per CTA.
    // Stream-ordered scratch (cached by the device's memory pool): concurrent calls on different
    // streams never share it.
    uint32_t* partial = nullptr;
    if (NB >= 4096u && grid > 1) {
        int rc = frisk_internal::pool_ready();
        if (rc) return rc;
        CK(cudaMallocAsync((void**)&partial, (size_t)grid * NW * sizeof(uint32_t), st));
    }
    bg_count_kernel<K><<<grid, kThreads, smem, st>>>(codes, inv, low, w_lo, w_hi, mask_host,
                                                      reinterpret_cast<unsigned long long*>(fwd), partial, d_range);
    if (partial) {
        bg_reduce_kernel<K><<<(NW + 31) / 32, 256, 0, st>>>(partial, grid, reinterpret_cast<unsigned long long*>(fwd));
        CK(cudaFreeAsync(partial, st));
    }
    CK(cudaGetLastError());
    return FRISK_OK;
}

template <int K, typename Fwd>
int launch_finalize(const Fwd f, int symmetric, uint64_t* tables, uint64_t* valid, cudaStream_t st) {
    constexpr int R = K > 4 ? K - 4 : 0;
    auto t = reinterpret_cast<unsigned long long*>(tables);
    if (valid) CK(cudaMemsetAsync(valid, 0, sizeof(uint64_t), st));
    forward_totals_kernel<K, Fwd><<<pow4(R), 256, 0, st>>>(f, t, reinterpret_cast<unsigned long long*>(valid));
    if (R > 1) forward_low_kernel<K, Fwd><<<1, 64, 0, st>>>(f, t);
    if (symmetric) symmetrise_kernel<K><<<(lvl_off(K + 1) + 255) / 256, 256, 0, st>>>(t);
    CK(cudaGetLastError());
    return FRISK_OK;
}

template <int K, typename Fwd>
int launch_finalize_ivom(Fwd f, int kmin, int64_t space, uint64_t* tables, uint64_t* valid, double* ig, cudaStream_t st) {
    auto kern = finalize_ivom_kernel<K, Fwd>;
    static std::atomic<int> cached[64];                                  // occupancy once per device and instantiation
    int dev = 0;
    CK(cudaGetDevice(&dev));
    int per_sm = cached[dev & 63].load(std::memory_order_acquire);
    if (per_sm == 0) {
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, 256, 0));
        if (per_sm > 0) cached[dev & 63].store(per_sm, std::memory_order_release);
    }
    const int sms = sm_count_cached();
    if (sms <= 0) return FRISK_E_NO_DEVICE;
    if (per_sm < 1) return FRISK_E_UNSUPPORTED;
    int grid = sms * (per_sm > 2 ? 2 : per_sm);                          // every CTA resident (grid-wide barriers); 2 per SM measured best
    if (valid) CK(cudaMemsetAsync(valid, 0, sizeof(uint64_t), st));
    unsigned long long* t = reinterpret_cast<unsigned long long*>(tables);
    unsigned long long* v = reinterpret_cast<unsigned long long*>(valid);
    long long sp = (long long)space;
    double2* g = reinterpret_cast<double2*>(ig);
    void* args[] = {(void*)&f, (void*)&t, (void*)&v, (void*)&kmin, (void*)&sp, (void*)&g};
    CK(cudaLaunchCooperativeKernel((const void*)kern, dim3((unsigned)grid), dim3(256), args, 0, st));
    return FRISK_OK;
}

template <int K>
int launch_genome_ivom(const uint64_t* tables, int kmin, int64_t space, double* ig, cudaStream_t st) {
    const uint32_t n = pow4(K);
    const int bs = 256;
    genome_ivom_kernel<K><<<(n + bs - 1) / bs, bs, 0, st>>>(reinterpret_cast<const unsigned long long*>(tables), kmin,
                                                           (long long)space, reinterpret_cast<double2*>(ig));
    CK(cudaGetLastError());
    return FRISK_OK;
}

// the peers' forward tables and ready flags of a sharded finalize
int peer_fwd(const uint64_t* const* d_fwd_peers, uint64_t* const* d_flag_peers, int rank, int world, uint64_t epoch, PeerFwd* f) {
    if (world > kMaxPeers) return FRISK_E_UNSUPPORTED;
    f->n = world;
    f->rank = rank;
    f->epoch = d_flag_peers ? epoch : 0;
    for (int q = 0; q < kMaxPeers; ++q) { f->p[q] = nullptr; f->flags[q] = nullptr; }
    for (int q = 0; q < world; ++q) {
        if (!d_fwd_peers[q] || (d_flag_peers && !d_flag_peers[q])) return FRISK_E_INVALID;
        f->p[q] = reinterpret_cast<const unsigned long long*>(d_fwd_peers[q]);
        if (d_flag_peers) f->flags[q] = reinterpret_cast<unsigned long long*>(d_flag_peers[q]);
    }
    return FRISK_OK;
}

}  // namespace

int frisk_internal::finalize_ivom(const uint64_t* d_fwd, const uint64_t* const* d_fwd_peers, uint64_t* const* d_flag_peers, int rank,
                                  int world, uint64_t epoch, int kmin, int kmax, int64_t space, const long long* space_dev,
                                  uint64_t* tables, uint64_t* valid, double* ig, cudaStream_t st) {
    int rc;
    if (kmax > FRISK_B200_FAST_K) {                                   // general path: separate launches
        if (world > 0 || space_dev) return FRISK_E_UNSUPPORTED;
        if ((rc = frisk_internal::general_finalize(d_fwd, kmax, 1, tables, valid, st))) return rc;
        return frisk_internal::general_genome_ivom(tables, kmin, kmax, space, ig, st);
    }
    if (world == 0) {
        const LocalFwd f{reinterpret_cast<const unsigned long long*>(d_fwd), space_dev};
        DISPATCH_K(kmax, (launch_finalize_ivom<K, LocalFwd>(f, kmin, space, tables, valid, ig, st)));
    }
    if (space_dev) return FRISK_E_UNSUPPORTED;
    PeerFwd f;
    if ((rc = peer_fwd(d_fwd_peers, d_flag_peers, rank, world, epoch, &f))) return rc;
    DISPATCH_K(kmax, (launch_finalize_ivom<K, PeerFwd>(f, kmin, space, tables, valid, ig, st)));
}

extern "C" {

int frisk_b200_background(const uint32_t* d_codes, const uint32_t* d_inv, const uint32_t* d_low, uint64_t first_base,
                          uint64_t last_base, int kmax, int mask_host, uint64_t* d_fwd, void* stream) {
    if (!d_codes || !d_inv || !d_fwd || (first_base & 31) || (last_base & 31) || last_base < first_base)
        return FRISK_E_INVALID;
    int rc = check_k(1, kmax);
    if (rc) return rc;
    if (last_base == first_base) return FRISK_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (kmax > FRISK_B200_FAST_K)
        return frisk_internal::general_background(d_codes, d_inv, d_low, first_base >> 5, last_base >> 5, kmax, mask_host, d_fwd, st);
    DISPATCH_K(kmax, launch_background<K>(d_codes, d_inv, d_low, first_base >> 5, last_base >> 5, mask_host, d_fwd, st));
}

}  // extern "C"

int frisk_internal::background_device_range(const uint32_t* codes, const uint32_t* inv, const uint32_t* low,
                                            const unsigned long long* d_word_range, uint64_t words_hint, int kmax, int mask_host,
                                            uint64_t* fwd, cudaStream_t st) {
    if (!codes || !inv || !fwd || !d_word_range) return FRISK_E_INVALID;
    int rc = check_k(1, kmax);
    if (rc) return rc;
    if (kmax > FRISK_B200_FAST_K) return FRISK_E_UNSUPPORTED;
    DISPATCH_K(kmax, launch_background<K>(codes, inv, low, 0, words_hint ? words_hint : 1, mask_host, fwd, st, d_word_range));
}

extern "C" {

int frisk_b200_finalize_tables(const uint64_t* d_fwd, int kmax, int symmetric, uint64_t* d_tables, uint64_t* d_valid_kmax,
                               void* stream) {
    if (!d_fwd || !d_tables) return FRISK_E_INVALID;
    int rc = check_k(1, kmax);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (kmax > FRISK_B200_FAST_K) return frisk_internal::general_finalize(d_fwd, kmax, symmetric, d_tables, d_valid_kmax, st);
    const LocalFwd f{reinterpret_cast<const unsigned long long*>(d_fwd)};
    DISPATCH_K(kmax, (launch_finalize<K, LocalFwd>(f, symmetric, d_tables, d_valid_kmax, st)));
}

int frisk_b200_finalize_tables_peers(const uint64_t* const* d_fwd_peers, uint64_t* const* d_flag_peers, int rank, int world,
                                     uint64_t epoch, int kmax, int symmetric, uint64_t* d_tables, uint64_t* d_valid_kmax,
                                     void* stream) {
    if (!d_fwd_peers || !d_tables || world < 1 || rank < 0 || rank >= world) return FRISK_E_INVALID;
    if (d_flag_peers && epoch == 0) return FRISK_E_INVALID;
    int rc = check_k(1, kmax);
    if (rc) return rc;
    if (kmax > FRISK_B200_FAST_K) return FRISK_E_UNSUPPORTED;
    PeerFwd f;
    if ((rc = peer_fwd(d_fwd_peers, d_flag_peers, rank, world, epoch, &f))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    DISPATCH_K(kmax, (launch_finalize<K, PeerFwd>(f, symmetric, d_tables, d_valid_kmax, st)));
}

int frisk_b200_finalize_ivom(const uint64_t* d_fwd, const uint64_t* const* d_fwd_peers, uint64_t* const* d_flag_peers, int rank,
                             int world, uint64_t epoch, int kmin, int kmax, int64_t genome_space, uint64_t* d_tables,
                             uint64_t* d_valid_kmax, double* d_ig, void* stream) {
    if (!d_tables || !d_ig || (world == 0 && !d_fwd) || (world > 0 && (!d_fwd_peers || rank < 0 || rank >= world)))
        return FRISK_E_INVALID;
    if (world > 0 && d_flag_peers && epoch == 0) return FRISK_E_INVALID;
    int rc = check_k(kmin, kmax);
    if (rc) return rc;
    return frisk_internal::finalize_ivom(d_fwd, d_fwd_peers, d_flag_peers, rank, world, epoch, kmin, kmax, genome_space, nullptr,
                                         d_tables, d_valid_kmax, d_ig, (cudaStream_t)stream);
}

int frisk_b200_genome_ivom(const uint64_t* d_tables, int kmin, int kmax, int64_t genome_space, double* d_ig, void* stream) {
    if (!d_tables || !d_ig) return FRISK_E_INVALID;
    int rc = check_k(kmin, kmax);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (kmax > FRISK_B200_FAST_K) return frisk_internal::general_genome_ivom(d_tables, kmin, kmax, genome_space, d_ig, st);
    DISPATCH_K(kmax, launch_genome_ivom<K>(d_tables, kmin, genome_space, d_ig, st));
}

}  // extern "C"
