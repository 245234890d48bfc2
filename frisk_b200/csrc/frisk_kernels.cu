// frisk_b200 device code: sm_100a kernels for the frisk hot path and their C-ABI launchers.
//
// Reference being replaced: /root/reference/frisk/__init__.py ("F:").  Nothing here is a
// translation of it (the reference is a Python dict loop); see DESIGN.md for the derivation.
//
//   bg_count_kernel        forward-strand k-mer counts of the genome       (F:321-351, counting)
//   finalize_tables_kernel marginalise orders K-1..1 + add reverse strand   (F:348-351)
//   genome_ivom_kernel     per-kmax-mer genome IVOM value and its log2      (F:411-450)
//   score_windows_kernel   window tables + IVOM x2 + KLD + GC + RIP, fused  (F:1478-1488)
//
// Table index convention everywhere: base-4 number, digits A=0 T=1 G=2 C=3, first base most
// significant (the reference's dict key order, F:70/F:253-274); complement = digit ^ 1.
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <map>
#include <mutex>
#include <tuple>

#include "../../include/frisk_b200.h"
#include "frisk_internal.h"
#include "frisk_device.cuh"

namespace {

constexpr int kThreads = 1024;          // one CTA per SM: the 4^8 u16 window table takes 128 KiB of smem
constexpr int kWarps = kThreads / 32;
constexpr uint32_t kListCap = 8192;     // compacted (kmer, count) entries per segment
constexpr int kMaxSeg = 8;

// reverse complement of the x-mer with index idx (F:276-278): reverse the digits, xor each with 1
__device__ __forceinline__ uint32_t revcomp_idx(uint32_t idx, int x) {
    uint32_t r = __brev(idx) >> (32 - 2 * x);                       // digits reversed, bits inside a digit swapped
    r = ((r >> 1) & 0x55555555u) | ((r & 0x55555555u) << 1);         // swap them back
    return r ^ (0x55555555u & (pow4(x) - 1u));
}

// gather bit1 of each of the 16 2-bit codes of a word into 16 contiguous bits (order kept)
__device__ __forceinline__ uint32_t high_bits16(uint32_t w) {
    uint32_t x = (w >> 1) & 0x55555555u;
    x = (x | (x >> 1)) & 0x33333333u;
    x = (x | (x >> 2)) & 0x0f0f0f0fu;
    x = (x | (x >> 4)) & 0x00ff00ffu;
    x = (x | (x >> 8)) & 0x0000ffffu;
    return x;
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

// ============================================================================================
// Window scoring.  One persistent CTA per SM (the 4^8 u16 order-K table alone is 128 KiB).
// Per window:
//   0. word-wise popcounts: unresolved count (30 % rule, F:238), upper-case base and G+C counts
//   1. count: per position one u16 shared-memory atomic on each of the orders LD..K (LD = 5: the
//      orders with >= 1024 bins, where a warp's 32 updates rarely collide) plus one atomicOr on an
//      occupancy bitmap of the order-K table.  A position whose longest valid word is v < LD
//      (window end, N boundary) adds 1 to order v only.
//   2. orders LD-1..1 by marginalisation (4 children -> parent) in one warp: <= 340 bins.
//   3. per order-LP node (LP = 5) the partial sums  sum_{x<=LP} q_x c_x^2  and  sum_{x<=LP} 4^x c_x
//      shared by every k-mer below it; bitmap popcounts + block scan -> sorted list of the
//      distinct K-mers (no pass over the 65,536 bins, 93 % of which are empty).
//   4. per distinct K-mer: window IVOM = N/D (closed form, see genome_ivom_kernel) from the prefix
//      counts, genome IVOM and its log2 from the precomputed table, three fp64 sums;
//      KLD = T/Sw + log2(Sg/Sw)  ==  sum_k w_k log2(w_k/g_k) with w, g normalised (F:448-454, F:466-470)
// ============================================================================================
struct ScoreSmem {
    double q[8];              // q_x = 4^x / ((S-(x-1)) 2) for the current window
    double red[3][kWarps];
    int n_non, n_gc, n_up, flags;
    uint32_t warp_tot[kWarps];
    uint32_t seg_base[kMaxSeg + 1];
};

template <int K>
struct ScoreLayout {
    static constexpr uint32_t NB = pow4(K);
    static constexpr int LD = K < 5 ? K : 5;                            // lowest order counted by atomics
    static constexpr int LP = K > 5 ? 5 : K - 1;                        // order of the shared partial sums (0: none)
    static constexpr uint32_t NPRE = LP > 0 ? pow4(LP) : 1u;
    static constexpr uint32_t NLOW = lvl_off(K);                       // entries of orders 1..K-1
    static constexpr uint32_t BM_WORDS = NB >= 32u ? NB / 32u : 1u;
    static constexpr uint32_t TOP_BYTES = (NB * 2u + 15u) & ~15u;
    static constexpr uint32_t LOW_BYTES = (NLOW * 2u + 15u) & ~15u;
    static constexpr uint32_t BM_BYTES = (BM_WORDS * 4u + 15u) & ~15u;
    static constexpr uint32_t LIST_BYTES = kListCap * 2u;
    static constexpr uint32_t PRE_BYTES = NPRE * 16u;                  // double num + u64 den per node
    static constexpr uint32_t LOG_BYTES = 128u * 16u;
    static constexpr uint32_t OFF_LOW = TOP_BYTES;
    static constexpr uint32_t OFF_BM = OFF_LOW + LOW_BYTES;
    static constexpr uint32_t OFF_LIST = OFF_BM + BM_BYTES;
    static constexpr uint32_t OFF_PRE = OFF_LIST + LIST_BYTES;
    static constexpr uint32_t OFF_LOG = OFF_PRE + PRE_BYTES;
    static constexpr uint32_t OFF_SS = OFF_LOG + LOG_BYTES;
    static constexpr uint32_t TOTAL = OFF_SS + (uint32_t)sizeof(ScoreSmem);
};

template <int K>
__global__ void __launch_bounds__(kThreads, 1)
score_windows_kernel(const uint32_t* __restrict__ codes, const uint32_t* __restrict__ inv, const uint32_t* __restrict__ low,
                     const unsigned long long* __restrict__ win_off, const uint32_t* __restrict__ win_len, uint32_t n_win,
                     const double2* __restrict__ ig, int kmin, int want_rip, int nseg,
                     double* __restrict__ rows, uint32_t* __restrict__ status, uint16_t* __restrict__ dump) {
    using L = ScoreLayout<K>;
    constexpr uint32_t NB = L::NB;
    constexpr int LD = L::LD, LP = L::LP;
    extern __shared__ __align__(16) unsigned char smem[];
    uint16_t* top16 = reinterpret_cast<uint16_t*>(smem);
    uint32_t* top32 = reinterpret_cast<uint32_t*>(smem);
    uint16_t* low16 = reinterpret_cast<uint16_t*>(smem + L::OFF_LOW);
    uint32_t* low32 = reinterpret_cast<uint32_t*>(smem + L::OFF_LOW);
    uint32_t* bitmap = reinterpret_cast<uint32_t*>(smem + L::OFF_BM);
    uint16_t* list = reinterpret_cast<uint16_t*>(smem + L::OFF_LIST);
    double2* pre = reinterpret_cast<double2*>(smem + L::OFF_PRE);       // .x = num, .y = den (as a double bit pattern of u64)
    double2* logtab = reinterpret_cast<double2*>(smem + L::OFF_LOG);
    ScoreSmem& ss = *reinterpret_cast<ScoreSmem*>(smem + L::OFF_SS);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // zero tables + bitmap once; afterwards every window leaves them zeroed
    for (uint32_t i = tid; i < L::OFF_LIST / 16u; i += kThreads)
        reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
    if (tid == 0) { ss.n_non = 0; ss.n_gc = 0; ss.n_up = 0; ss.flags = 0; }
    if (tid < 128) {
        const double c = 1.0 + ((double)tid + 0.5) / 128.0;
        const double ic = 1.0 / c;
        logtab[tid] = make_double2(ic, -log2(ic));
    }
    __syncthreads();

    for (uint32_t win = blockIdx.x; win < n_win; win += gridDim.x) {
        const uint64_t o = win_off[win];
        const uint32_t len = win_len[win];

        // ---- 0. composition counts, word-wise (32 bases per thread) ---------------------------
        {
            const uint64_t mw_first = o >> 5, mw_last = (o + len - 1) >> 5;
            int non = 0, gc = 0, upc = 0;
            for (uint64_t mw = mw_first + tid; mw <= mw_last && len > 0; mw += kThreads) {
                uint32_t range = kFull;
                if (mw == mw_first) range &= kFull >> (uint32_t)(o & 31);
                if (mw == mw_last) range &= kFull << (31u - (uint32_t)((o + len - 1) & 31));
                uint32_t bad = __ldg(inv + mw);
                if (low) bad |= __ldg(low + mw);
                const uint32_t good = ~bad & range;
                const uint32_t g = (high_bits16(__ldg(codes + 2 * mw)) << 16) | high_bits16(__ldg(codes + 2 * mw + 1));
                non += __popc(bad & range);
                upc += __popc(good);
                gc += __popc(g & good);
            }
            if (__any_sync(kFull, (non | upc) != 0)) {
                non = __reduce_add_sync(kFull, non);
                gc = __reduce_add_sync(kFull, gc);
                upc = __reduce_add_sync(kFull, upc);
                if (lane == 0) { atomicAdd(&ss.n_non, non); atomicAdd(&ss.n_gc, gc); atomicAdd(&ss.n_up, upc); }
            }
        }
        __syncthreads();
        const int n_non = ss.n_non, n_gc = ss.n_gc, n_up = ss.n_up;
        // F:238 / F:213: excluded when winN >= 0.3 * len (same double comparison as the reference)
        const bool excluded = (double)n_non >= 0.3 * (double)len;
        __syncthreads();                                   // everyone has read the counters
        if (tid == 0) { ss.n_non = 0; ss.n_gc = 0; ss.n_up = 0; ss.flags = 0; }
        if (excluded) {
            if (tid == 0) {
                status[win] = FRISK_ROW_EXCLUDED;
                for (int c = 0; c < 5; ++c) rows[(size_t)win * 5 + c] = CUDART_NAN;
            }
            if (dump) for (uint32_t i = tid; i < lvl_off(K + 1); i += kThreads) dump[(size_t)win * lvl_off(K + 1) + i] = 0;
            __syncthreads();                               // counters are reset before the next window adds to them
            continue;
        }
        // window space S = totalLen - nnTotal (F:380) = number of upper-case ATGC characters
        if (tid < K) {
            const int x = tid + 1;
            const long long d = ((long long)n_up - (long long)(x - 1)) * 2;
            ss.q[tid] = (double)pow4(x) / (double)d;       // inf if d == 0: flagged below when used
        }

        // ---- 1. count ---------------------------------------------------------------------------
        for (uint32_t p = tid; p < len; p += kThreads) {
            const uint64_t a = o + p;
            const uint64_t wi = a >> 4, mi = a >> 5;
            const uint32_t code = __funnelshift_l(__ldg(codes + wi + 1), __ldg(codes + wi), (uint32_t)(a & 15) * 2u)
                                  >> (32 - 2 * K);
            const uint32_t m = __funnelshift_l(__ldg(inv + mi + 1), __ldg(inv + mi), (uint32_t)(a & 31));
            const int v = min(min(__clz(m), K), (int)min(len - p, (uint32_t)K));
            if (v == K) {
                atomicAdd(&top32[code >> 1], 1u << ((code & 1u) * 16u));
                atomicOr(&bitmap[code >> 5], 1u << (code & 31u));
            }
            if (v >= LD) {
#pragma unroll
                for (int x = LD; x < K; ++x) {
                    if (x <= v) {
                        const uint32_t g = lvl_off(x) + (code >> (2 * (K - x)));
                        atomicAdd(&low32[g >> 1], 1u << ((g & 1u) * 16u));
                    }
                }
            } else if (v > 0) {
                const uint32_t g = lvl_off(v) + (code >> (2 * (K - v)));
                atomicAdd(&low32[g >> 1], 1u << ((g & 1u) * 16u));
            }
        }
        __syncthreads();

        // ---- 2. orders LD-1..1 from order LD (warp 0); every thread: its two bitmap words ----------
        if (warp == 0) {
#pragma unroll
            for (int x = LD - 1; x >= 1; --x) {
                const uint16_t* child = (x + 1 == K) ? top16 : low16 + lvl_off(x + 1);
                for (uint32_t t = lane; t < pow4(x); t += 32) {
                    const uint2 ch = *reinterpret_cast<const uint2*>(child + 4 * t);
                    low16[lvl_off(x) + t] += (uint16_t)((ch.x & 0xffffu) + (ch.x >> 16) + (ch.y & 0xffffu) + (ch.y >> 16));
                }
                __syncwarp();
            }
        }
        uint32_t w0 = 0, w1 = 0;
        if (2u * tid < L::BM_WORDS) {
            if (L::BM_WORDS >= 2u) {
                const uint2 ww = *reinterpret_cast<const uint2*>(bitmap + 2 * tid);
                w0 = ww.x; w1 = ww.y;
                if (w0 | w1) *reinterpret_cast<uint2*>(bitmap + 2 * tid) = make_uint2(0, 0);
            } else {
                w0 = bitmap[0];
                bitmap[0] = 0;
            }
        }
        const uint32_t cnt = __popc(w0) + __popc(w1);
        uint32_t incl = cnt;
#pragma unroll
        for (int ofs = 1; ofs < 32; ofs <<= 1) {
            const uint32_t y = __shfl_up_sync(kFull, incl, ofs);
            if (lane >= ofs) incl += y;
        }
        if (lane == 31) ss.warp_tot[warp] = incl;
        __syncthreads();

        // ---- 3. shared partial sums per order-LP node; offsets of every thread's k-mers ------------
        const uint32_t wt = ss.warp_tot[lane];
        const uint32_t n_total = __reduce_add_sync(kFull, wt);
        uint32_t my_off = __reduce_add_sync(kFull, lane < warp ? wt : 0u) + incl - cnt;   // exclusive, window-wide
        constexpr int OWN = L::BM_WORDS >= 2u ? (int)(L::BM_WORDS / 2u) : 1;   // threads that own bitmap words
        const int tps = OWN / nseg > 0 ? OWN / nseg : 1;                       // of them, per segment
        if (tid < OWN && tid % tps == 0) ss.seg_base[tid / tps] = my_off;
        if (tid == 0) ss.seg_base[nseg] = n_total;
        if (LP > 0 && tid < (int)L::NPRE) {
            double num = 0.0;
            unsigned long long den = 0;
#pragma unroll
            for (int x = 1; x <= LP; ++x) {
                if (x >= kmin) {
                    const uint32_t c = low16[lvl_off(x) + ((uint32_t)tid >> (2 * (LP - x)))];
                    den += (unsigned long long)c << (2 * x);
                    num = fma(ss.q[x - 1], u32_to_double(c * c), num);
                }
            }
            pre[tid] = make_double2(num, __longlong_as_double((long long)den));
        }
        // dinucleotide counts for calcRIP (F:474-495), read before the epilogue wipes the top table
        uint32_t n_at = 0, n_ta = 0, n_sub = 0, n_prod = 0;
        if constexpr (K >= 2) {
            if (tid == 0 && want_rip) {
                const uint16_t* di = (K == 2) ? top16 : low16 + lvl_off(2);
                n_at = di[1]; n_ta = di[4];                 // AT = 0*4+1, TA = 1*4+0
                n_sub = (uint32_t)di[3] + di[9];            // AC + GT
                n_prod = (uint32_t)di[12] + di[6];          // CA + TG
            }
        }
        if (dump) {   // tests only: window tables, orders 1..K (orders < LD are final: warp 0 finished before the barrier)
            uint16_t* d = dump + (size_t)win * lvl_off(K + 1);
            for (uint32_t i = tid; i < lvl_off(K); i += kThreads) d[i] = low16[i];
            for (uint32_t i = tid; i < NB; i += kThreads) d[lvl_off(K) + i] = top16[i];
        }
        __syncthreads();

        // ---- 4. per segment: expand bitmap words into the sorted k-mer list, then score -----------
        double s_w = 0.0, s_g = 0.0, s_t = 0.0;
        int bad = 0;
        for (int seg = 0; seg < nseg; ++seg) {
            const uint32_t base = ss.seg_base[seg];
            const uint32_t n_list = ss.seg_base[seg + 1] - base;
            if (tid < OWN && tid / tps == seg) {
                uint32_t pos = my_off - base;
                uint32_t w = w0;
                while (w) { const int b = __ffs(w) - 1; w &= w - 1; list[pos++] = (uint16_t)(64u * tid + b); }
                w = w1;
                while (w) { const int b = __ffs(w) - 1; w &= w - 1; list[pos++] = (uint16_t)(64u * tid + 32u + b); }
            }
            __syncthreads();

            for (uint32_t e = tid; e < n_list; e += kThreads) {
                const uint32_t kappa = list[e];
                const uint32_t ck = top16[kappa];
                top16[kappa] = 0;                              // leave the table zeroed for the next window
                double num = 0.0;
                unsigned long long den = 0;
                if (LP > 0) {
                    const double2 pp = pre[kappa >> (2 * (K - LP))];
                    num = pp.x;
                    den = (unsigned long long)__double_as_longlong(pp.y);
                }
#pragma unroll
                for (int x = LP + 1; x <= K; ++x) {
                    if (x >= kmin) {
                        const uint32_t c = (x == K) ? ck : (uint32_t)low16[lvl_off(x) + (kappa >> (2 * (K - x)))];
                        den += (unsigned long long)c << (2 * x);
                        num = fma(ss.q[x - 1], u32_to_double(c * c), num);
                    }
                }
                const double iw = div_pos(num, __ull2double_rn(den));
                const double2 g = __ldg(ig + kappa);
                s_w += iw;
                s_g += g.x;
                s_t = fma(iw, log2_pos(iw, logtab) - g.y, s_t);
                bad |= (g.x != g.x);
            }
            __syncthreads();                               // list is reused by the next segment
        }

        // ---- block reduction (fixed tree -> bit-reproducible) and the row ----------------------
#pragma unroll
        for (int ofs = 16; ofs; ofs >>= 1) {
            s_w += __shfl_xor_sync(kFull, s_w, ofs);
            s_g += __shfl_xor_sync(kFull, s_g, ofs);
            s_t += __shfl_xor_sync(kFull, s_t, ofs);
        }
        bad = __any_sync(kFull, bad);
        if (lane == 0) {
            ss.red[0][warp] = s_w; ss.red[1][warp] = s_g; ss.red[2][warp] = s_t;
            if (bad) atomicOr(&ss.flags, 1);
        }
        // re-zero the lower-order tables for the next window (top table and bitmap are already clean)
        for (uint32_t i = tid; i < L::LOW_BYTES / 16u; i += kThreads)
            reinterpret_cast<uint4*>(low16)[i] = make_uint4(0, 0, 0, 0);
        __syncthreads();
        if (tid == 0) {
            double a = 0, b = 0, c = 0;
            for (int w = 0; w < kWarps; ++w) { a += ss.red[0][w]; b += ss.red[1][w]; c += ss.red[2][w]; }
            uint32_t st = 0;
            double kld = 0.0;                              // the reference returns 0 for a window without kmax-mers
            if (n_total) {
                bool zd = ss.flags & 1;
                for (int x = kmin; x <= K; ++x) zd |= ((long long)n_up - (long long)(x - 1)) == 0;
                if (zd) { st |= FRISK_ROW_KLD_ZERODIV; kld = CUDART_NAN; }
                else {
                    kld = c / a + (log2(b) - log2(a));
                    if (!(kld == kld) || isinf(kld)) st |= FRISK_ROW_LOG_DOMAIN;
                }
            }
            double* row = rows + (size_t)win * 5;
            row[0] = kld;
            if (n_up == 0) { st |= FRISK_ROW_GC_ZERODIV; row[1] = CUDART_NAN; }
            else row[1] = (double)n_gc / (double)n_up;       // F:136
            double pi = CUDART_NAN, si = CUDART_NAN, cri = CUDART_NAN;
            if (K >= 2 && want_rip) {
                if (n_at > 0) pi = (double)n_ta / (double)n_at;        // F:480-483
                if (n_sub > 0) si = (double)n_prod / (double)n_sub;    // F:485-489
                if (pi != 0.0 && si != 0.0) cri = pi - si;             // F:491: 0.0 falsy, NaN truthy
            }
            row[2] = pi; row[3] = si; row[4] = cri;
            status[win] = st;
        }
    }
}

// ============================================================================================
// Window scoring, bucketed formulation: the default path (4 <= K <= 8, windows <= 8192 bases).
//
// The dense 4^K table of score_windows_kernel costs 128 KiB and forces one CTA per SM, whose phases
// (count / scan / score) then run back to back with barriers between them.  A window of L bases has
// at most L distinct K-mers, so instead the K-mers are counting-sorted by their (K-2)-prefix:
//   P1  per position: ONE u16 shared-memory atomic, on order B = K-2 (4^B buckets), or on order v
//       for a word valid for v < B bases only; composition counts on the way (30 % rule, GC)
//   P2  exclusive scan of the order-B counts -> bucket cursors; orders B-1..1 by marginalisation
//       (4 children -> parent) inside the same pass
//   P3  per position: claim a slot in its bucket (atomic on the cursor) and store a 5-bit code: the
//       2-base suffix (0..15), or 16+b for a word valid for K-1 bases only, or 20 for K-2 only;
//       OR the suffix into the bucket's 16-bit presence mask.  Per order-LP node (LP = min(4,B)) the
//       partial sums  sum q_x c_x^2 ,  sum 4^x c_x  shared by every K-mer below it.
//   P4a popcounts of the presence masks + block scan -> sorted list of the distinct K-mers
//   P4b one list entry per thread per round (converged): order-K / order-(K-1) counts are 1 and
//       popc(mask group) when every entry of the bucket is a distinct K-mer (the common case),
//       otherwise recounted from the bucket; then the same closed-form IVOM / KLD terms as above.
// Footprint for K = 8, w = 5000: 48 KiB -> 4 CTAs of 256 threads per SM: four windows in
// different phases overlap on every SM and barriers span 8 warps only.
// ============================================================================================
constexpr int kT3 = 256;
constexpr int kW3 = kT3 / 32;

struct Score3Smem {
    double q[8];
    double red[3][kW3];
    int cnt[2][4];                    // [window parity][n_non, n_gc, n_up, -]
    int flags[2];
    uint32_t warp_tot[kW3];
    uint32_t warp_tot2[kW3];
};

template <int K>
struct Score3Layout {
    static constexpr int B = K - 2;                                     // bucket order
    static constexpr uint32_t NBK = pow4(B);
    static constexpr int LP = B < 4 ? B : 4;                            // order of the shared partial sums
    static constexpr uint32_t NPRE = pow4(LP);
    static constexpr uint32_t PER = NBK >= (uint32_t)kT3 ? NBK / kT3 : 1u;   // buckets per thread (contiguous)
    static constexpr uint32_t TAB_BYTES = (lvl_off(B + 1) * 2u + 15u) & ~15u;  // orders 1..B, u16
    static constexpr uint32_t MASK_BYTES = (NBK * 2u + 15u) & ~15u;     // suffix-presence masks, u16 per bucket
    static constexpr uint32_t OFF_MASK = TAB_BYTES;                     // (tables and masks are zeroed together)
    static constexpr uint32_t ZERO_BYTES = TAB_BYTES + MASK_BYTES;
    static constexpr uint32_t OFF_CUR = ZERO_BYTES;                     // u32 per bucket (list start, dirty flag, buf start)
    static constexpr uint32_t OFF_PRE = OFF_CUR + 2u * MASK_BYTES;
    static constexpr uint32_t OFF_LOG = OFF_PRE + NPRE * 16u;
    static constexpr uint32_t OFF_SS = OFF_LOG + 128u * 16u;
    static constexpr uint32_t OFF_BUF = (OFF_SS + (uint32_t)sizeof(Score3Smem) + 15u) & ~15u;
    // then: buf[cap] (suffix codes, one byte per position) and list[cap] (u16 distinct K-mers),
    // cap = longest window of the launch rounded up to 16
    static constexpr uint32_t total(uint32_t cap) { return OFF_BUF + cap + 2u * cap; }
};

// PER consecutive u16 values starting at p (8-byte aligned when PER >= 4) with the widest loads:
// a thread's contiguous bins are 32 bytes apart from its neighbour's, so single u16 loads would be
// 8-way bank-conflicted.
template <uint32_t PER>
__device__ __forceinline__ void load_u16s(const uint16_t* p, uint32_t (&out)[PER]) {
    if constexpr (PER >= 4) {
#pragma unroll
        for (uint32_t g = 0; g < PER / 4; ++g) {
            const uint2 v = *reinterpret_cast<const uint2*>(p + 4 * g);
            out[4 * g] = v.x & 0xffffu; out[4 * g + 1] = v.x >> 16; out[4 * g + 2] = v.y & 0xffffu; out[4 * g + 3] = v.y >> 16;
        }
    } else {
#pragma unroll
        for (uint32_t g = 0; g < PER; ++g) out[g] = p[g];
    }
}

// ROUNDS rounds of 4 positions per thread cover a window of up to 4*NT*ROUNDS - 3 bases; what a
// position contributes (bucket, suffix code, arrival rank in its bucket) stays in registers
// between the counting pass and the placement pass, so the sequence is read and decoded once.
template <int K, int ROUNDS, bool DUMP, bool ALLK>
__global__ void __launch_bounds__(kT3, 4)
score_windows_bucket_kernel(const uint32_t* __restrict__ codes, const uint32_t* __restrict__ inv, const uint32_t* __restrict__ low,
                            const unsigned long long* __restrict__ win_off, const uint32_t* __restrict__ win_len, uint32_t n_win,
                            const double2* __restrict__ ig, int kmin_arg, int want_rip, uint32_t cap, uint32_t len_min,
                            uint32_t len_max, double* __restrict__ rows, uint32_t* __restrict__ status, uint16_t* __restrict__ dump,
                            const uint32_t* __restrict__ redo_src) {
    using L = Score3Layout<K>;
    constexpr int B = L::B, LP = L::LP;
    constexpr uint32_t NBK = L::NBK, PER = L::PER;
    constexpr uint32_t kNone = 31u;                                      // suffix code of "nothing to place"
    const int kmin = ALLK ? 1 : kmin_arg;                                // ALLK: the default --minWordSize 1, predicates fold away
    extern __shared__ __align__(16) unsigned char smem[];
    uint16_t* tab16 = reinterpret_cast<uint16_t*>(smem);                 // orders 1..B
    uint32_t* tab32 = reinterpret_cast<uint32_t*>(smem);
    uint16_t* mask16 = reinterpret_cast<uint16_t*>(smem + L::OFF_MASK);
    uint32_t* mask32 = reinterpret_cast<uint32_t*>(smem + L::OFF_MASK);
    // per bucket: clean: bits 0-12 start of its K-mers in the list, bit 15 = 0, bits 16-31 its presence mask;
    //             dirty: bits 0-14 start in the dirty list, bit 15 = 1, bits 16-31 start of its entries in buf
    uint32_t* dst32 = reinterpret_cast<uint32_t*>(smem + L::OFF_CUR);
    double2* pre = reinterpret_cast<double2*>(smem + L::OFF_PRE);       // .x = num, .y = den (u32 bit pattern)
    double2* logtab = reinterpret_cast<double2*>(smem + L::OFF_LOG);
    Score3Smem& ss = *reinterpret_cast<Score3Smem*>(smem + L::OFF_SS);
    uint8_t* buf = smem + L::OFF_BUF;
    uint16_t* list = reinterpret_cast<uint16_t*>(smem + L::OFF_BUF + cap);
    const uint16_t* tabB = tab16 + lvl_off(B);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (redo_src) {
        // hand-over launch: nearly always there is nothing to do.  All threads look at this CTA's marks at once and the CTA
        // leaves if none is set (walking them one window at a time cost 26 us per step: a global round trip per window)
        bool any = false;
        for (uint32_t w = blockIdx.x + (uint32_t)tid * gridDim.x; w < n_win; w += gridDim.x * (uint32_t)kT3)
            any |= (redo_src[w] & frisk_internal::kRowRedo) != 0u;
        if (!__syncthreads_or(any)) return;
    }
    for (uint32_t i = tid; i < L::ZERO_BYTES / 16u; i += kT3) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
    if (tid < 8) { ss.cnt[tid >> 2][tid & 3] = 0; ss.flags[tid & 1] = 0; }
    if (tid < 128) {
        const double c = 1.0 + ((double)tid + 0.5) / 128.0;
        const double ic = 1.0 / c;
        logtab[tid] = make_double2(ic, -log2(ic));
    }
    __syncthreads();

    int par = 1;                                         // flipped by every window this launch processes
    for (uint32_t win = blockIdx.x; win < n_win; win += gridDim.x) {
        const uint64_t o = win_off[win];                 // (both descriptor loads are in flight before the length test)
        const uint32_t len = win_len[win];
        if (len < len_min || len > len_max) continue;    // another launch (other buffer size) takes this one
        // second launch behind the direct kernel (frisk_direct.cu): only the windows it handed over
        if (redo_src && !(redo_src[win] & frisk_internal::kRowRedo)) continue;
        par ^= 1;
        // 32-bit addressing relative to the window's first mask word
        const uint32_t o_lo = (uint32_t)(o & 31);
        const uint32_t* __restrict__ cw = codes + (o >> 5) * 2;
        const uint32_t* __restrict__ mw = inv + (o >> 5);
        const uint32_t* __restrict__ lw = low ? low + (o >> 5) : nullptr;
        const uint32_t g0 = o_lo >> 2;
        const uint32_t ngroups = ((o_lo + len + 3u) >> 2) - g0;          // <= NT * ROUNDS (checked by the launcher)

        // ---- P1: one pass over the positions: composition, order-B counts (-> rank), presence masks ---
        uint32_t place[4 * ROUNDS];                    // per position: bucket << 18 | rank << 5 | suffix code
        {
            int non = 0, gc = 0;
            GroupWords gw = load_group(cw, mw, lw, (g0 + (tid < (int)ngroups ? tid : 0)) << 2);
#pragma unroll
            for (int r = 0; r < ROUNDS; ++r) {
                const uint32_t gi = tid + r * kT3;
                // next round's words are requested before this round is processed (hides the L2 latency)
                const uint32_t gn = gi + kT3;
                GroupWords nx = gw;
                if (r + 1 < ROUNDS) nx = load_group(cw, mw, lw, (g0 + (gn < ngroups ? gn : 0u)) << 2);
#pragma unroll
                for (int j = 0; j < 4; ++j) place[4 * r + j] = kNone;
                if (gi < ngroups) {
                    visit_group(gw, (g0 + gi) << 2, o_lo, len, [&](uint32_t j, uint32_t p, uint32_t c32, uint32_t m, uint32_t lowbit) {
                        const uint32_t unres = (m >> 31) | lowbit;               // not an upper-case ATGC (F:106-118)
                        non += unres;
                        gc += (1 - unres) & (c32 >> 31);                         // G = 2, C = 3: bit 1 of the first base
                        const uint32_t b = c32 >> (32 - 2 * B);
                        const uint32_t sfx = (c32 >> (32 - 2 * K)) & 15u;
                        const uint32_t sh = (b & 1u) * 16u;
                        if ((m >> (32 - K)) == 0u && p + K <= len) {             // the common case: a full K-word
                            const uint32_t old = atomicAdd(&tab32[(lvl_off(B) + b) >> 1], 1u << sh);
                            atomicOr(&mask32[b >> 1], (1u << sfx) << sh);
                            place[4 * r + j] = (b << 18) | (((old >> sh) & 0x1fffu) << 5) | sfx;
                        } else {                                                 // window end / N boundary
                            const int v = min(__clz(m), (int)(len - p));
                            if (v >= B) {                                        // valid for K-1 or K-2 bases only
                                const uint32_t old = atomicAdd(&tab32[(lvl_off(B) + b) >> 1], 1u << sh);
                                place[4 * r + j] = (b << 18) | (((old >> sh) & 0x1fffu) << 5) | (v == K - 1 ? 16u + (sfx >> 2) : 20u);
                            } else if (v > 0) {                                  // order v < B only
                                const uint32_t g = lvl_off(v) + (c32 >> (32 - 2 * v));
                                atomicAdd(&tab32[g >> 1], 1u << ((g & 1u) * 16u));
                            }
                        }
                    });
                }
                gw = nx;
            }
            non = __reduce_add_sync(kFull, non);
            gc = __reduce_add_sync(kFull, gc);
            if (lane == 0) { atomicAdd(&ss.cnt[par][0], non); atomicAdd(&ss.cnt[par][1], gc); }
        }
        __syncthreads();                                                   // (1)
        const int n_non = ss.cnt[par][0], n_gc = ss.cnt[par][1], n_up = (int)len - n_non;
        if (tid < 4) ss.cnt[par ^ 1][tid] = 0;                              // next window's counters (idle until its P1)
        if (tid == 4) ss.flags[par ^ 1] = 0;
        const bool excluded = (double)n_non >= 0.3 * (double)len;          // F:238 / F:213
        uint16_t* dmp = DUMP ? dump + (size_t)win * lvl_off(K + 1) : nullptr;
        if (excluded) {
            for (uint32_t i = tid; i < L::ZERO_BYTES / 16u; i += kT3) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
            if (tid == 0) {
                status[win] = FRISK_ROW_EXCLUDED;
                for (int c = 0; c < 5; ++c) rows[(size_t)win * 5 + c] = CUDART_NAN;
            }
            if (DUMP) for (uint32_t i = tid; i < lvl_off(K + 1); i += kT3) dmp[i] = 0;
            __syncthreads();
            continue;
        }
        if (tid < K) {
            const int x = tid + 1;
            const long long d = ((long long)n_up - (long long)(x - 1)) * 2;
            ss.q[tid] = (double)pow4(x) / (double)d;
        }

        // ---- P2: per bucket: clean (every entry a distinct K-mer) or dirty; three exclusive scans
        //          (clean K-mers, dirty K-mers, dirty entries); orders B-1..1 by marginalisation -----------
        // Bucket ownership: a thread owns G groups of GS contiguous buckets; group g of lane l in warp w
        // starts at bucket w*32*PER + g*32*GS + l*GS, so a warp's lanes read contiguous 8-byte units (no
        // bank conflicts) and (warp, group, lane, bucket-in-group) order is bucket order: the lists stay sorted.
        constexpr uint32_t GS = PER >= 4 ? 4u : PER, G = PER / GS;
        const bool owner = (uint32_t)tid * PER < NBK;
        const uint32_t wbase = (uint32_t)warp * 32u * PER + (uint32_t)lane * GS;
        uint32_t gA[G], gB[G];                         // per group: A = clean K-mers | dirty K-mers << 16;  B = entries of dirty buckets
#pragma unroll
        for (uint32_t g = 0; g < G; ++g) {
            gA[g] = 0; gB[g] = 0;
            uint32_t sum4 = 0;
            if (owner) {
                uint32_t nbs[GS], mks[GS];
                load_u16s<GS>(tabB + wbase + g * 32u * GS, nbs);
                load_u16s<GS>(mask16 + wbase + g * 32u * GS, mks);
#pragma unroll
                for (uint32_t j = 0; j < GS; ++j) {
                    const uint32_t pc = __popc(mks[j]);
                    const bool dirty = nbs[j] != pc;
                    gA[g] += dirty ? pc << 16 : pc;
                    gB[g] += dirty ? nbs[j] : 0u;
                    sum4 += nbs[j];
                }
                if constexpr (PER >= 4) {              // the four buckets are the children of one order-(B-1) bin
                    uint16_t* par1 = tab16 + lvl_off(B - 1) + (wbase + g * 32u * GS) / 4;
                    sum4 += *par1;                     // + the short words of order B-1
                    *par1 = (uint16_t)sum4;
                }
            }
            if constexpr (PER >= 16) {                 // four consecutive lanes hold the children of one order-(B-2) bin
                sum4 += __shfl_xor_sync(kFull, sum4, 1);
                sum4 += __shfl_xor_sync(kFull, sum4, 2);
                if (owner && (lane & 3) == 0) tab16[lvl_off(B - 2) + (wbase + g * 32u * GS) / 16] += (uint16_t)sum4;
            }
        }
        // inclusive scans over lanes per group, then groups chained inside the warp
        uint32_t iA[G], iB[G], warpA = 0, warpB = 0;
#pragma unroll
        for (uint32_t g = 0; g < G; ++g) {
            iA[g] = gA[g]; iB[g] = gB[g];
#pragma unroll
            for (int ofs = 1; ofs < 32; ofs <<= 1) {
                const uint32_t ya = __shfl_up_sync(kFull, iA[g], ofs), yb = __shfl_up_sync(kFull, iB[g], ofs);
                if (lane >= ofs) { iA[g] += ya; iB[g] += yb; }
            }
            const uint32_t ta = __shfl_sync(kFull, iA[g], 31), tb = __shfl_sync(kFull, iB[g], 31);
            iA[g] += warpA - gA[g];                    // -> exclusive prefix inside the warp
            iB[g] += warpB - gB[g];
            warpA += ta; warpB += tb;
        }
        if (lane == 31) { ss.warp_tot[warp] = warpA; ss.warp_tot2[warp] = warpB; }
        __syncthreads();                                                   // (2a)
        if (warp == 0) {
            constexpr int LW = B - (PER >= 16 ? 2 : (PER >= 4 ? 1 : 0));  // lowest order that is complete by now
#pragma unroll
            for (int x = LW - 1; x >= 1; --x) {
                for (uint32_t t = lane; t < pow4(x); t += 32) {
                    const uint2 ch = *reinterpret_cast<const uint2*>(tab16 + lvl_off(x + 1) + 4 * t);
                    tab16[lvl_off(x) + t] += (uint16_t)((ch.x & 0xffffu) + (ch.x >> 16) + (ch.y & 0xffffu) + (ch.y >> 16));
                }
                __syncwarp();
            }
        }
        uint32_t n_clean, n_dirty;
        {
            uint32_t totA = 0, preA = 0, preB = 0;
#pragma unroll
            for (int w = 0; w < kW3; ++w) {
                const uint32_t ta = ss.warp_tot[w], tb = ss.warp_tot2[w];
                totA += ta;
                if (w < warp) { preA += ta; preB += tb; }
            }
            n_clean = totA & 0xffffu; n_dirty = totA >> 16;
            if (owner) {
#pragma unroll
                for (uint32_t g = 0; g < G; ++g) {
                    uint32_t nbs[GS], mks[GS], outv[GS];
                    load_u16s<GS>(tabB + wbase + g * 32u * GS, nbs);
                    load_u16s<GS>(mask16 + wbase + g * 32u * GS, mks);
                    uint32_t runA = preA + iA[g], runB = preB + iB[g];
#pragma unroll
                    for (uint32_t j = 0; j < GS; ++j) {
                        const uint32_t pc = __popc(mks[j]);
                        if (nbs[j] != pc) {                                // dirty: list start | flag, and the start of its entries in buf
                            outv[j] = 0x8000u | (runA >> 16) | (runB << 16);
                            runA += pc << 16;
                            runB += nbs[j];
                        } else {                                           // clean: list start | presence mask << 16 (all P3/P4 need)
                            outv[j] = (runA & 0x1fffu) | (mks[j] << 16);
                            runA += pc;
                        }
                    }
                    if constexpr (GS == 4) {
                        *reinterpret_cast<uint4*>(dst32 + wbase + g * 32u * GS) = make_uint4(outv[0], outv[1], outv[2], outv[3]);
                    } else {
#pragma unroll
                        for (uint32_t j = 0; j < GS; ++j) dst32[wbase + g * 32u * GS + j] = outv[j];
                    }
                }
            }
        }
        __syncthreads();                                                   // (2b)

        // ---- P3: place every remembered position: its K-mer into the sorted list of distinct K-mers
        //          (slot = bucket start + rank of the suffix among the bucket's present suffixes: the same
        //          for every occurrence, so duplicates write the same value), dirty buckets' entries into buf --
#pragma unroll
        for (int i = 0; i < 4 * ROUNDS; ++i) {
            const uint32_t pl = place[i], c5 = pl & 31u;
            if (c5 != kNone) {
                const uint32_t b = pl >> 18, rank = (pl >> 5) & 0x1fffu;
                const uint32_t d = dst32[b];
                if (c5 < 16u) {
                    const uint16_t kappa = (uint16_t)((b << 4) | c5);
                    const uint32_t below = (1u << c5) - 1u;
                    // clean bucket: cursor and mask come in the one word; a dirty one (rare) reads its mask too
                    uint32_t slot = (d & 0x1fffu) + __popc((d >> 16) & below);
                    if (d & 0x8000u) {
                        slot = cap - 1u - ((d & 0x7fffu) + __popc((uint32_t)mask16[b] & below));
                        buf[(d >> 16) + rank] = (uint8_t)c5;
                    }
                    list[slot] = kappa;
                } else {
                    buf[(d >> 16) + rank] = (uint8_t)c5;                   // a short word makes its bucket dirty
                }
            }
        }
        for (uint32_t node = tid; node < L::NPRE; node += kT3) {
            double num = 0.0;
            uint32_t den = 0;
#pragma unroll
            for (int x = 1; x <= LP; ++x) {
                if (x >= kmin) {
                    const uint32_t c = tab16[lvl_off(x) + (node >> (2 * (LP - x)))];
                    den += c << (2 * x);
                    num = fma(ss.q[x - 1], u32_to_double(c * c), num);
                }
            }
            pre[node] = make_double2(num, __hiloint2double(0, (int)den));
        }
        uint32_t n_at = 0, n_ta = 0, n_sub = 0, n_prod = 0;
        if (tid == 0 && want_rip) {                        // all orders are final since barrier (2b); K >= 4 so B >= 2
            const uint16_t* di = tab16 + lvl_off(2);
            n_at = di[1]; n_ta = di[4];
            n_sub = (uint32_t)di[3] + di[9];
            n_prod = (uint32_t)di[12] + di[6];
        }
        if (DUMP) {
            for (uint32_t i = tid; i < lvl_off(B + 1); i += kT3) dmp[i] = tab16[i];
            for (uint32_t i = lvl_off(B + 1) + tid; i < lvl_off(K + 1); i += kT3) dmp[i] = 0;
        }
        __syncthreads();                                                   // (3)
        if (DUMP) {   // tests only: order K-1 counts of the window, per bucket
            for (uint32_t b = tid; b < NBK; b += kT3) {
                const uint32_t nb = tabB[b], msk = mask16[b];
                if (nb == 0) continue;
                uint32_t c7[4] = {0, 0, 0, 0};
                if (!(dst32[b] & 0x8000u)) {
                    for (int j = 0; j < 4; ++j) c7[j] = __popc((msk >> (4 * j)) & 15u);
                } else {
                    const uint32_t beg = dst32[b] >> 16;
                    for (uint32_t e = beg; e < beg + nb; ++e) {
                        const uint32_t c5 = buf[e];
                        if (c5 < 16u) c7[c5 >> 2]++; else if (c5 < 20u) c7[c5 - 16u]++;
                    }
                }
                for (int j = 0; j < 4; ++j) dmp[lvl_off(K - 1) + 4 * b + j] = (uint16_t)c7[j];
            }
        }

        // ---- P4: score the distinct K-mers, one list entry per thread per round -------------------
        double s_w = 0.0, s_g = 0.0, s_t = 0.0;
        double qr[K - LP];                                                 // q of the orders LP+1..K
#pragma unroll
        for (int x = LP + 1; x <= K; ++x) qr[x - LP - 1] = ss.q[x - 1];
        auto score_one = [&](uint32_t kappa, uint32_t b, uint32_t nb, uint32_t c7, uint32_t c8) {
            if (DUMP) dmp[lvl_off(K) + kappa] = (uint16_t)c8;
            // orders <= LP from `pre`, orders LP+1..B from the tables, then K-1 and K
            const double2 pp = pre[b >> (2 * (B - LP))];
            double num = pp.x;
            uint32_t den = (uint32_t)__double2loint(pp.y);
#pragma unroll
            for (int x = LP + 1; x <= B; ++x) {
                if (x >= kmin) {
                    const uint32_t c = (x == B) ? nb : (uint32_t)tab16[lvl_off(x) + (b >> (2 * (B - x)))];
                    den += c << (2 * x);
                    num = fma(qr[x - LP - 1], u32_to_double(c * c), num);
                }
            }
            if (K - 1 >= kmin) {
                den += c7 << (2 * (K - 1));
                num = fma(qr[K - LP - 2], u32_to_double(c7 * c7), num);
            }
            den += c8 << (2 * K);
            num = fma(qr[K - LP - 1], u32_to_double(c8 * c8), num);
            const double iw = div_pos(num, (double)den);
            const double2 g = __ldg(ig + kappa);
            s_w += iw;
            s_g += g.x;                                    // a NaN entry (reference: ZeroDivisionError) poisons the sum
            s_t = fma(iw, log2_pos(iw, logtab) - g.y, s_t);
        };
        for (uint32_t e = tid; e < n_clean; e += kT3) {
            const uint32_t kappa = list[e];
            const uint32_t b = kappa >> 4, j = (kappa >> 2) & 3u;
            const uint32_t msk = dst32[b] >> 16;                               // clean bucket: count = popc(mask)
            score_one(kappa, b, __popc(msk), __popc((msk >> (4 * j)) & 15u), 1u);
        }
        for (uint32_t e = tid; e < n_dirty; e += kT3) {
            const uint32_t kappa = list[cap - 1u - e];
            const uint32_t b = kappa >> 4, sfx = kappa & 15u, j = sfx >> 2;
            const uint32_t nb = tabB[b], beg = dst32[b] >> 16;
            uint32_t c8 = 0, c7 = 0;
            for (uint32_t i = beg; i < beg + nb; ++i) {
                const uint32_t c5 = buf[i];
                c8 += (c5 == sfx);
                c7 += (c5 < 16u) ? ((c5 >> 2) == j) : (c5 == 16u + j);
            }
            score_one(kappa, b, nb, c7, c8);
        }
        const uint32_t n_list = n_clean + n_dirty;
#pragma unroll
        for (int ofs = 16; ofs; ofs >>= 1) {
            s_w += __shfl_xor_sync(kFull, s_w, ofs);
            s_g += __shfl_xor_sync(kFull, s_g, ofs);
            s_t += __shfl_xor_sync(kFull, s_t, ofs);
        }
        if (lane == 0) { ss.red[0][warp] = s_w; ss.red[1][warp] = s_g; ss.red[2][warp] = s_t; }
        __syncthreads();                                                   // (4) everyone is done with the tables
        for (uint32_t i = tid; i < L::ZERO_BYTES / 16u; i += kT3) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
        if (tid == 0) {
            double a = 0, bsum = 0, c = 0;
            for (int w = 0; w < kW3; ++w) { a += ss.red[0][w]; bsum += ss.red[1][w]; c += ss.red[2][w]; }
            uint32_t st = 0;
            double kld = 0.0;                              // the reference returns 0 for a window without kmax-mers
            if (n_list) {
                bool zd = bsum != bsum;                    // NaN genome IVOM entry: ZeroDivisionError at F:437
                for (int x = kmin; x <= K; ++x) zd |= ((long long)n_up - (long long)(x - 1)) == 0;
                if (zd) { st |= FRISK_ROW_KLD_ZERODIV; kld = CUDART_NAN; }
                else {
                    kld = c / a + (log2(bsum) - log2(a));
                    if (!(kld == kld) || isinf(kld)) st |= FRISK_ROW_LOG_DOMAIN;
                }
            }
            double* row = rows + (size_t)win * 5;
            row[0] = kld;
            if (n_up == 0) { st |= FRISK_ROW_GC_ZERODIV; row[1] = CUDART_NAN; }
            else row[1] = (double)n_gc / (double)n_up;       // F:136
            double pi = CUDART_NAN, si = CUDART_NAN, cri = CUDART_NAN;
            if (want_rip) {
                if (n_at > 0) pi = (double)n_ta / (double)n_at;        // F:480-483
                if (n_sub > 0) si = (double)n_prod / (double)n_sub;    // F:485-489
                if (pi != 0.0 && si != 0.0) cri = pi - si;             // F:491: 0.0 falsy, NaN truthy
            }
            row[2] = pi; row[3] = si; row[4] = cri;
            status[win] = st;
        }
        __syncthreads();                                                   // (5) tables zeroed, ss.red consumed
    }
}

// ============================================================================================
// Window scoring for small word sizes (K <= 6): no sorting at all.  The whole order-K table has at most
// 4,096 bins, so every position does ONE u16 shared-memory atomic on order K (or on the order of its
// longest valid word), lower orders follow by marginalisation, and the epilogue simply walks the bins
// of order K in order (coalesced genome-IVOM reads, fixed summation order -> bit-reproducible).
// 11 KB of shared memory: 6 CTAs of 256 threads per SM.  Windows up to 65,535 bases (16-bit counters).
// ============================================================================================
struct SmallSmem {
    double q[8];
    double red[3][kW3];
    int n_non, n_gc, flags, pad;
};

template <int K>
struct SmallLayout {
    static constexpr uint32_t NTAB = lvl_off(K + 1);                       // u16 entries, orders 1..K
    static constexpr uint32_t TAB_BYTES = (NTAB * 2u + 15u) & ~15u;
    static constexpr int P = K >= 3 ? (K - 1 < 4 ? K - 1 : 4) : 0;          // orders <= P are folded into one pair per order-P prefix
    static constexpr uint32_t NPRE = P ? pow4(P) : 0u;
    static constexpr uint32_t OFF_LOG = TAB_BYTES;
    static constexpr uint32_t OFF_PRE = OFF_LOG + 128u * 16u;
    static constexpr uint32_t OFF_SS = OFF_PRE + NPRE * 16u;
    static constexpr uint32_t TOTAL = OFF_SS + (uint32_t)sizeof(SmallSmem);
};

template <int K, bool DUMP>
__global__ void __launch_bounds__(kT3, 6)
score_windows_small_kernel(const uint32_t* __restrict__ codes, const uint32_t* __restrict__ inv, const uint32_t* __restrict__ low,
                           const unsigned long long* __restrict__ win_off, const uint32_t* __restrict__ win_len, uint32_t n_win,
                           const double2* __restrict__ ig, int kmin, int want_rip,
                           double* __restrict__ rows, uint32_t* __restrict__ status, uint16_t* __restrict__ dump,
                           const uint32_t* __restrict__ redo_src) {
    using L = SmallLayout<K>;
    extern __shared__ __align__(16) unsigned char smem[];
    uint16_t* tab16 = reinterpret_cast<uint16_t*>(smem);
    uint32_t* tab32 = reinterpret_cast<uint32_t*>(smem);
    double2* logtab = reinterpret_cast<double2*>(smem + L::OFF_LOG);
    double2* pre = reinterpret_cast<double2*>(smem + L::OFF_PRE);          // .x = num, .y = den (low word) of the orders <= P
    SmallSmem& ss = *reinterpret_cast<SmallSmem*>(smem + L::OFF_SS);
    constexpr int P = L::P;
    (void)pre;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (redo_src) {                                                        // hand-over launch: leave at once when no window of this CTA is marked
        bool any = false;
        for (uint32_t w = blockIdx.x + (uint32_t)tid * gridDim.x; w < n_win; w += gridDim.x * (uint32_t)kT3)
            any |= (redo_src[w] & frisk_internal::kRowRedo) != 0u;
        if (!__syncthreads_or(any)) return;
    }

    for (uint32_t i = tid; i < L::TAB_BYTES / 16u; i += kT3) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
    if (tid == 0) { ss.n_non = 0; ss.n_gc = 0; ss.flags = 0; }
    if (tid < 128) {
        const double c = 1.0 + ((double)tid + 0.5) / 128.0;
        const double ic = 1.0 / c;
        logtab[tid] = make_double2(ic, -log2(ic));
    }
    __syncthreads();

    for (uint32_t win = blockIdx.x; win < n_win; win += gridDim.x) {
        // second launch behind the k sweep (frisk_nibble.cu): only the windows it handed over
        if (redo_src && !(redo_src[win] & frisk_internal::kRowRedo)) continue;
        const uint64_t o = win_off[win];
        const uint32_t len = win_len[win];
        const uint32_t o_lo = (uint32_t)(o & 31);
        const uint32_t* __restrict__ cw = codes + (o >> 5) * 2;
        const uint32_t* __restrict__ mw = inv + (o >> 5);
        const uint32_t* __restrict__ lw = low ? low + (o >> 5) : nullptr;
        const uint32_t g0 = o_lo >> 2;
        const uint32_t ngroups = ((o_lo + len + 3u) >> 2) - g0;

        // ---- count: one atomic per position, on the order of its longest valid word (<= K) -----------
        int non = 0, gc = 0;
        for (uint32_t gi = tid; gi < ngroups; gi += kT3) {
            const GroupWords gw = load_group(cw, mw, lw, (g0 + gi) << 2);
            visit_group(gw, (g0 + gi) << 2, o_lo, len, [&](uint32_t, uint32_t p, uint32_t c32, uint32_t m, uint32_t lowbit) {
                const uint32_t unres = (m >> 31) | lowbit;                       // not an upper-case ATGC (F:106-118)
                non += unres;
                gc += (1 - unres) & (c32 >> 31);
                const uint32_t rest = len - p;
                const int v = min(min(__clz(m), K), (int)(rest < (uint32_t)K ? rest : (uint32_t)K));
                if (v > 0) {
                    const uint32_t g = lvl_off(v) + (c32 >> (32 - 2 * v));
                    if constexpr (K == 1) {
                        // 4 bins for 32 lanes: same-address atomics serialise (5,000 positions on two words cost 0.15 ms
                        // per 120 Mbp), so the lanes that hit the same bin send one atomic between them (measured: 0.83 ->
                        // 0.68 ms; at K = 2, 20 bins, the match costs more than it saves: 0.65 -> 0.94 ms)
                        const uint32_t peers = __match_any_sync(__activemask(), g);
                        if ((uint32_t)lane == (uint32_t)__ffs((int)peers) - 1u)
                            atomicAdd(&tab32[g >> 1], (uint32_t)__popc(peers) << ((g & 1u) * 16u));
                    } else {
                        atomicAdd(&tab32[g >> 1], 1u << ((g & 1u) * 16u));
                    }
                }
            });
        }
        non = __reduce_add_sync(kFull, non);
        gc = __reduce_add_sync(kFull, gc);
        if (lane == 0 && (non | gc)) { atomicAdd(&ss.n_non, non); atomicAdd(&ss.n_gc, gc); }
        __syncthreads();
        // ---- lower orders: F_x = words that end at order x + marginal of F_{x+1} ----------------------
#pragma unroll
        for (int x = K - 1; x >= 1; --x) {
            for (uint32_t t = tid; t < pow4(x); t += kT3) {
                const uint2 ch = *reinterpret_cast<const uint2*>(tab16 + lvl_off(x + 1) + 4 * t);
                tab16[lvl_off(x) + t] += (uint16_t)((ch.x & 0xffffu) + (ch.x >> 16) + (ch.y & 0xffffu) + (ch.y >> 16));
            }
            __syncthreads();
        }
        const int n_non = ss.n_non, n_gc = ss.n_gc, n_up = (int)len - n_non;
        const bool excluded = (double)n_non >= 0.3 * (double)len;              // F:238 / F:213
        if (tid < K) {
            const int x = tid + 1;
            const long long d = ((long long)n_up - (long long)(x - 1)) * 2;
            ss.q[tid] = (double)pow4(x) / (double)d;
        }
        uint32_t n_at = 0, n_ta = 0, n_sub = 0, n_prod = 0;
        if (K >= 2 && tid == 0 && want_rip) {
            const uint16_t* di = tab16 + lvl_off(2);
            n_at = di[1]; n_ta = di[4]; n_sub = (uint32_t)di[3] + di[9]; n_prod = (uint32_t)di[12] + di[6];
        }
        if (DUMP) {
            uint16_t* d = dump + (size_t)win * lvl_off(K + 1);
            for (uint32_t i = tid; i < lvl_off(K + 1); i += kT3) d[i] = excluded ? (uint16_t)0 : tab16[i];
        }
        __syncthreads();
        if constexpr (P > 0) {           // the low orders' share of numerator and denominator, once per order-P prefix
            if (!excluded) {
                for (uint32_t node = tid; node < pow4(P); node += kT3) {
                    double num = 0.0;
                    uint32_t den = 0;
#pragma unroll
                    for (int x = 1; x <= P; ++x) {
                        if (x >= kmin) {
                            const uint32_t c = tab16[lvl_off(x) + (node >> (2 * (P - x)))];
                            den += c << (2 * x);
                            num = fma(ss.q[x - 1], u32_to_double(c * c), num);
                        }
                    }
                    pre[node] = make_double2(num, __hiloint2double(0, (int)den));
                }
            }
            __syncthreads();
        }

        // ---- epilogue: every occupied bin of order K, in table order ------------------------------------
        double s_w = 0.0, s_g = 0.0, s_t = 0.0;
        uint32_t any = 0;
        if (!excluded) {
            for (uint32_t kappa = tid; kappa < pow4(K); kappa += kT3) {
                const uint32_t ck = tab16[lvl_off(K) + kappa];
                if (ck == 0) continue;
                double num = 0.0;
                uint32_t den = 0;
                if constexpr (P > 0) {
                    const double2 pp = pre[kappa >> (2 * (K - P))];
                    num = pp.x;
                    den = (uint32_t)__double2loint(pp.y);
                }
#pragma unroll
                for (int x = P + 1; x <= K; ++x) {
                    if (x >= kmin) {
                        const uint32_t c = (x == K) ? ck : (uint32_t)tab16[lvl_off(x) + (kappa >> (2 * (K - x)))];
                        den += c << (2 * x);
                        num = fma(ss.q[x - 1], u32_to_double(c * c), num);
                    }
                }
                const double iw = div_pos(num, (double)den);
                const double2 g = __ldg(ig + kappa);
                s_w += iw;
                s_g += g.x;
                s_t = fma(iw, log2_pos(iw, logtab) - g.y, s_t);
                any = 1;
            }
        }
#pragma unroll
        for (int ofs = 16; ofs; ofs >>= 1) {
            s_w += __shfl_xor_sync(kFull, s_w, ofs);
            s_g += __shfl_xor_sync(kFull, s_g, ofs);
            s_t += __shfl_xor_sync(kFull, s_t, ofs);
        }
        any = __any_sync(kFull, any);
        if (lane == 0) {
            ss.red[0][warp] = s_w; ss.red[1][warp] = s_g; ss.red[2][warp] = s_t;
            if (any) atomicOr(&ss.flags, 1);
        }
        __syncthreads();                                                       // everyone is done with the tables
        for (uint32_t i = tid; i < L::TAB_BYTES / 16u; i += kT3) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
        if (tid == 0) {
            double* row = rows + (size_t)win * 5;
            if (excluded) {
                status[win] = FRISK_ROW_EXCLUDED;
                for (int c = 0; c < 5; ++c) row[c] = CUDART_NAN;
            } else {
                double a = 0, bsum = 0, c = 0;
                for (int w = 0; w < kW3; ++w) { a += ss.red[0][w]; bsum += ss.red[1][w]; c += ss.red[2][w]; }
                uint32_t st = 0;
                double kld = 0.0;                          // the reference returns 0 for a window without kmax-mers
                if (ss.flags & 1) {
                    bool zd = bsum != bsum;                // NaN genome IVOM entry: ZeroDivisionError at F:437
                    for (int x = kmin; x <= K; ++x) zd |= ((long long)n_up - (long long)(x - 1)) == 0;
                    if (zd) { st |= FRISK_ROW_KLD_ZERODIV; kld = CUDART_NAN; }
                    else {
                        kld = c / a + (log2(bsum) - log2(a));
                        if (!(kld == kld) || isinf(kld)) st |= FRISK_ROW_LOG_DOMAIN;
                    }
                }
                row[0] = kld;
                if (n_up == 0) { st |= FRISK_ROW_GC_ZERODIV; row[1] = CUDART_NAN; }
                else row[1] = (double)n_gc / (double)n_up;   // F:136
                double pi = CUDART_NAN, si = CUDART_NAN, cri = CUDART_NAN;
                if (K >= 2 && want_rip) {
                    if (n_at > 0) pi = (double)n_ta / (double)n_at;        // F:480-483
                    if (n_sub > 0) si = (double)n_prod / (double)n_sub;    // F:485-489
                    if (pi != 0.0 && si != 0.0) cri = pi - si;             // F:491: 0.0 falsy, NaN truthy
                }
                row[2] = pi; row[3] = si; row[4] = cri;
                status[win] = st;
            }
            ss.n_non = 0; ss.n_gc = 0; ss.flags = 0;
        }
        __syncthreads();
    }
}

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
}  // namespace

// ============================================================================================
// Shared-memory atomic micro-benchmark (roofline denominator for the counting step)
// ============================================================================================
namespace {
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

thread_local char g_cuda_err[512] = "";
int g_forced = -1;          // the WinKernel forced through frisk_b200_set_option (tests, A/B measurements), -1: none
}  // namespace

int frisk_internal::cuda_fail(cudaError_t e, const char* what) {
    snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
    return FRISK_E_CUDA;
}

namespace {
using frisk_internal::sm_count_cached;
using frisk_internal::LaunchShape;
using frisk_internal::WinKernel;
using frisk_internal::WinPlan;
using frisk_internal::kSmemMaxWindow;
using frisk_internal::check_k;
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

template <int K>
int launch_score(const uint32_t* codes, const uint32_t* inv, const uint32_t* low, const uint64_t* win_off,
                 const uint32_t* win_len, uint64_t n_win, uint32_t max_len, const double* ig, int kmin, int want_rip,
                 double* rows, uint32_t* status, uint16_t* dump, cudaStream_t st) {
    using L = ScoreLayout<K>;
    constexpr uint32_t NB = pow4(K);
    // a segment = a contiguous 1/nseg of the k-mer space (and of the threads owning its bitmap words);
    // its distinct k-mers (<= bins in it, <= window length) must fit the list
    int nseg = 1;
    while ((NB / (uint32_t)nseg < max_len ? NB / (uint32_t)nseg : max_len) > kListCap) nseg *= 2;
    if (nseg > kMaxSeg || (uint32_t)nseg > (L::BM_WORDS >= 2u ? L::BM_WORDS / 2u : 1u)) return FRISK_E_UNSUPPORTED;
    CK(cudaFuncSetAttribute(score_windows_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L::TOTAL));
    int grid = sm_count_cached();
    if (grid <= 0) return FRISK_E_NO_DEVICE;
    if ((uint64_t)grid > n_win) grid = (int)n_win;
    score_windows_kernel<K><<<grid, kThreads, L::TOTAL, st>>>(
        codes, inv, low, reinterpret_cast<const unsigned long long*>(win_off), win_len, (uint32_t)n_win,
        reinterpret_cast<const double2*>(ig), kmin, want_rip, nseg, rows, status, dump);
    CK(cudaGetLastError());
    return FRISK_OK;
}

// The small-K kernel (K <= 6: the whole order-K table in shared memory; its L1 / shared split is left to the driver) or the
// bucketed kernel (K >= 4: buffer sized by the longest window; four CTAs of 57 KB need the whole 228 KB carve-out, which
// the driver's per-launch heuristic does not always give: 0.73 vs 0.83 ms).
template <int K>
int table_shape(const WinPlan& p, uint32_t max_len, LaunchShape* s) {
    if constexpr (K <= 6) {
        if (p.kind == WinKernel::Small) {
            *s = {p.dump ? (const void*)score_windows_small_kernel<K, true> : (const void*)score_windows_small_kernel<K, false>, kT3,
                  SmallLayout<K>::TOTAL, false};
            return FRISK_OK;
        }
    }
    if constexpr (K >= 4) {
        if (p.kind == WinKernel::Bucket) {
            *s = {p.variant == 2   ? FRISK_WIN_INSTANCE(p, score_windows_bucket_kernel, K, 2)
                  : p.variant == 5 ? FRISK_WIN_INSTANCE(p, score_windows_bucket_kernel, K, 5)
                                   : FRISK_WIN_INSTANCE(p, score_windows_bucket_kernel, K, 8),
                  kT3, Score3Layout<K>::total((max_len + 15u) & ~15u), true};
            return FRISK_OK;
        }
    }
    return FRISK_E_UNSUPPORTED;
}

// one launch of the small-K or the bucketed kernel; the bucketed one takes the windows of [len_min, len_max] only, and with
// redo_src only those marked kRowRedo there
template <int K>
int launch_table(const WinPlan& p, const uint32_t* codes, const uint32_t* inv, const uint32_t* low, const uint64_t* win_off,
                 const uint32_t* win_len, uint64_t n_win, uint32_t max_len, const double* ig, int kmin, int want_rip, double* rows,
                 uint32_t* status, uint16_t* dump, cudaStream_t st, uint32_t len_min = 0, uint32_t len_max = 0xffffffffu,
                 const uint32_t* redo_src = nullptr) {
    LaunchShape s;
    int rc = table_shape<K>(p, max_len, &s);
    if (rc) return rc;
    const unsigned long long* off = reinterpret_cast<const unsigned long long*>(win_off);
    const double2* g = reinterpret_cast<const double2*>(ig);
    uint32_t n = (uint32_t)n_win, cap = (max_len + 15u) & ~15u;
    if (p.kind == WinKernel::Small) {
        void* args[] = {&codes, &inv, &low, &off, &win_len, &n, &g, &kmin, &want_rip, &rows, &status, &dump, &redo_src};
        return frisk_internal::launch_persistent(s, n_win, args, st);
    }
    void* args[] = {&codes, &inv, &low, &off, &win_len, &n, &g, &kmin, &want_rip, &cap, &len_min, &len_max, &rows, &status, &dump, &redo_src};
    return frisk_internal::launch_persistent(s, n_win, args, st);
}

// frisk_b200_score on the small-K or the bucketed kernel.  Bucketed windows longer than 5 rounds need a bigger buffer, which
// costs a CTA per SM.  With --scaffoldsAll nearly all windows are still the standard length and only whole short scaffolds
// (up to 1.25 w) are longer: two launches, each taking the windows of its length class, keep the standard ones at four
// CTAs per SM.
template <int K>
int score_table(const WinPlan& p, const uint32_t* codes, const uint32_t* inv, const uint32_t* low, const uint64_t* win_off,
                const uint32_t* win_len, uint64_t n_win, uint32_t max_len, const double* ig, int kmin, int want_rip, double* rows,
                uint32_t* status, uint16_t* dump, cudaStream_t st) {
    constexpr uint32_t kStd = 5104u;                   // largest buffer that still fits four CTAs
    if (p.kind == WinKernel::Bucket && p.variant == 8 && n_win >= 4096) {
        const WinPlan std5{p.kind, 5, p.dump, p.allk};
        int rc = launch_table<K>(std5, codes, inv, low, win_off, win_len, n_win, kStd, ig, kmin, want_rip, rows, status, dump, st, 0u, kStd);
        if (rc) return rc;
        return launch_table<K>(p, codes, inv, low, win_off, win_len, n_win, max_len, ig, kmin, want_rip, rows, status, dump, st, kStd + 1u);
    }
    return launch_table<K>(p, codes, inv, low, win_off, win_len, n_win, max_len, ig, kmin, want_rip, rows, status, dump, st);
}

#define DISPATCH_K(kmax, expr)                      \
    switch (kmax) {                                 \
        case 1: { constexpr int K = 1; return expr; } \
        case 2: { constexpr int K = 2; return expr; } \
        case 3: { constexpr int K = 3; return expr; } \
        case 4: { constexpr int K = 4; return expr; } \
        case 5: { constexpr int K = 5; return expr; } \
        case 6: { constexpr int K = 6; return expr; } \
        case 7: { constexpr int K = 7; return expr; } \
        case 8: { constexpr int K = 8; return expr; } \
        default: return FRISK_E_UNSUPPORTED;        \
    }

int table_shape_k(const WinPlan& p, int K, uint32_t max_len, LaunchShape* s) { DISPATCH_K(K, table_shape<K>(p, max_len, s)); }

bool forced(WinKernel k) { return g_forced == (int)k; }

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

// Positions per thread, from the longest window (the K-mer codes stay in registers between the counting and the scoring
// pass; shorter windows of the same launch use fewer).  All four kernels run 256 threads; a bucketed or direct round is
// 4 positions and keeps 6 bases of look-ahead.
int frisk_internal::check_k(int kmin, int kmax) {
    if (kmin < 1 || kmin > kmax) return FRISK_E_INVALID;
    if (kmax > FRISK_B200_MAX_K) return FRISK_E_UNSUPPORTED;
    return FRISK_OK;
}

int frisk_internal::window_variant(WinKernel kind, uint32_t len) {
    if (kind == WinKernel::Bucket || kind == WinKernel::Direct)
        return len <= kT3 * 4u * 2u - 6u ? 2 : (len <= kT3 * 4u * 5u - 6u ? 5 : 8);
    if (kind == WinKernel::Nibble || kind == WinKernel::NibbleExt) return len <= kT3 * 8u ? 8 : (len <= kT3 * 20u ? 20 : 32);
    return 0;
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
    DISPATCH_K(K, launch_table<K>(p, codes, inv, low, win_off, win_len, n_win, max_len, ig, kmin, want_rip, rows, status, dump, st, 0u,
                                  0xffffffffu, redo_src));
}

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
        case WinKernel::Bucket:
            DISPATCH_K(kmax, score_table<K>(p, d_codes, d_inv, d_low, d_win_off, d_win_len, n_win, max_win_len, d_ig, kmin, rip, d_rows,
                                            d_status, d_dump, st));
        case WinKernel::Dense:
            DISPATCH_K(kmax, launch_score<K>(d_codes, d_inv, d_low, d_win_off, d_win_len, n_win, max_win_len, d_ig, kmin, rip, d_rows,
                                             d_status, d_dump, st));
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
        case WinKernel::Dense:                              // one CTA of 1,024 threads per SM, like the general kernel
        case WinKernel::General: *ctas_per_sm = 1; *threads_per_cta = kThreads; return FRISK_OK;
        case WinKernel::Nibble: s = frisk_internal::nibble_shape(p, kmax); break;
        case WinKernel::Direct: s = frisk_internal::direct_shape(p, kmax); break;
        case WinKernel::NibbleExt: s = frisk_internal::ext_shape(p); break;
        default: if ((rc = table_shape_k(p, kmax, max_win_len, &s))) return rc;
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
