// frisk_b200: the "nibble" window-score kernel for kmax 7 and 8 (windows <= 8,186 bases).
//
// Replaces, per window, the reference's computeKmers(window) + IvomBuild x2 + KLD + calcGC + calcRIP
// (/root/reference/frisk/__init__.py F:1478-1494, F:280-367, F:369-472, F:120-137, F:474-495).
//
// ONE shared-memory atomic per position and no sorting.  The order-K code space is one 4-BIT counter per K-mer:
// the 16 K-mers below an order-(K-2) prefix ("bucket") share one 64-bit word (4^6 buckets x 8 B = 32 KiB at K = 8).
//   * a position adds 1 to its K-mer's nibble; afterwards every POSITION scores its own K-mer with weight 1/c_K
//     (c_K = its count in the window), so the sum over positions equals the sum over distinct K-mers (F:448-472
//     iterate the distinct keys) without enumerating or sorting them.  (Letting only the first arrival at a nibble
//     score it would save the weights, but which occurrence arrives first is a race: the rows would no longer be
//     bit-reproducible.)
//   * one 64-bit load gives the three highest orders of a K-mer: its nibble (order K), the sum of the 4 nibbles of
//     its 16-bit quarter (order K-1) and the sum of all 16 (order K-2);
//   * order A = K-3 is the sum of four buckets' nibble sums (one pass over the table, coalesced, warp shuffles), the
//     orders below follow by marginalisation, orders <= 4 are folded into one {numerator, denominator} pair per
//     order-4 prefix (`pre`);
//   * a thread's positions are fixed and so is the reduction tree -> bit-reproducible rows.
// 40-56 KB of shared memory per CTA (K = 8).
//
// What a nibble cannot hold is handed to the bucketed kernel (frisk_bucket.cu), exactly: a window in which some
// K-mer occurs 16+ times (the thread whose increment wraps the nibble sees 15 in the word it got back), or with
// more than kSideCap words cut short by an N / the window end at K-1 or K-2 bases, is marked kRowRedo and re-done
// by the launch that follows on the same stream.  Short words of K-1 / K-2 bases (every window has two at its
// end) are not in the nibble table: they go to a small side list, and bit 15 of their order-A bin sends the (few)
// K-mers below that bin through the list.
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "../../include/frisk_b200.h"
#include "frisk_internal.h"
#include "frisk_device.cuh"

namespace {
using frisk_internal::kRowRedo;

constexpr uint32_t kSideCap = 64;
constexpr int kNT = 256;

struct NibSmem {
    double q[8];
    double red[3][kNT / 32];
    int cnt[2][6];                    // [window parity][n_non, n_gc, full K-words counted, n_side, sum of all nibbles, -]
    uint32_t c2[16];                  // final dinucleotide counts (RIP, and the way up to order 1)
    uint32_t c1[4];                   // sweep: final base counts
    uint32_t side[kSideCap];          // v << 16 | code of a word valid for v = K-1 or K-2 bases only
};

template <int K>
struct NibLayout {
    static_assert(K == 7 || K == 8, "nibble kernel: K = 7 or 8");
    static constexpr int B = K - 2;                                      // bucket order: 16 K-mers per bucket
    static constexpr int A = K - 3;                                      // highest order kept as u16 counts
    static constexpr int LP = 4;                                         // orders <= LP live in `pre`
    static constexpr uint32_t NBK = pow4(B);
    static constexpr uint32_t NPRE = pow4(LP);
    static constexpr uint32_t NIB_BYTES = NBK * 8u;                      // 16 nibbles per bucket
    static constexpr uint32_t LOW_BYTES = (lvl_off(A + 1) * 2u + 15u) & ~15u;   // orders 1..A, u16
    static constexpr uint32_t ZERO_BYTES = NIB_BYTES + LOW_BYTES;
    static constexpr uint32_t OFF_LOW = NIB_BYTES;
    static constexpr uint32_t OFF_PRE = ZERO_BYTES;
    // K = 8: `pre` extended to order A (its own array, after the order-4 one): one 16-byte read instead of 16 + 2
    static constexpr bool FOLD_A = A > LP;
    static constexpr uint32_t NPREA = FOLD_A ? pow4(A) : 0u;
    static constexpr uint32_t OFF_PREA = OFF_PRE + NPRE * 16u;
    static constexpr uint32_t OFF_SS = OFF_PREA + NPREA * 16u;
    static constexpr uint32_t TOTAL = OFF_SS + (uint32_t)sizeof(NibSmem);
};

// Per-thread position masks: position i of the thread's chunk is bit (MB - 1 - i).  32 bits when the chunk and the
// K - 1 bases of look-ahead fit (PP + K - 1 <= 32), 64 bits otherwise.
template <bool WIDE> struct MaskT { using type = uint32_t; };
template <> struct MaskT<true> { using type = unsigned long long; };
__device__ __forceinline__ int popc_m(uint32_t x) { return __popc(x); }
__device__ __forceinline__ int popc_m(unsigned long long x) { return __popcll(x); }
__device__ __forceinline__ int clz_m(uint32_t x) { return __clz((int)x); }
__device__ __forceinline__ int clz_m(unsigned long long x) { return __clzll((long long)x); }
template <typename MT> __device__ __forceinline__ MT top_bits(int n) {       // the n leading bits set, 0 <= n
    constexpr int MB = (int)sizeof(MT) * 8;
    return n >= MB ? ~MT(0) : ~(~MT(0) >> n);
}

// The k sweep of BASELINE config C3 (scores for kmax' = 1..K with kmin = 1, i.e. K reference runs `-m 1 -k k'`, F:1197-1206)
// from ONE pass over the window: the counts of every order are there after the marginalisation, so the SWEEP
// instantiation evaluates all K scores -- kmax' <= K-2 by walking that order's bins (coalesced genome-IVOM reads),
// K-1 and K per position with weights 1/c -- and writes K rows per window.
struct NibSweep {
    const unsigned long long* n_win_dev;   // nullable: the number of windows lives in device memory (frisk_b200_run_fasta builds
                                           // its window list on the device); the n_win argument is then the capacity
    const double2* ig[8];             // genome IVOM table of kmax' = i + 1
    double* rows[8];
    uint32_t* status[8];
};

// PP = positions per thread: a thread owns ONE chunk of cs <= PP consecutive positions of the window
// (cs = the window length spread over the CTA, a multiple of 4), reads the three or four code words and two or three
// mask words that cover it once, and issues the atomics of its full K-words back to back from registers.
template <int K, int PP, bool DUMP, bool ALLK, bool SWEEP = false>
__global__ void __launch_bounds__(kNT, 4)
score_windows_nibble_kernel(const uint32_t* __restrict__ codes, const uint32_t* __restrict__ inv, const uint32_t* __restrict__ low,
                            const unsigned long long* __restrict__ win_off, const uint32_t* __restrict__ win_len, uint32_t n_win,
                            const double2* __restrict__ pair, int kmin_arg, int want_rip,
                            double* __restrict__ rows, uint32_t* __restrict__ status, uint16_t* __restrict__ dump,
                            uint32_t* redo_dst, const NibSweep sw) {
    static_assert(!SWEEP || (K == 8 && ALLK && !DUMP), "the sweep instantiation: K = 8, kmin = 1");
    using L = NibLayout<K>;
    static_assert(PP % 4 == 0 && PP >= 4 && PP + K - 1 <= 64, "chunk size");
    constexpr int A = L::A, LP = L::LP, NT = kNT, NW = NT / 32;
    constexpr bool WIDE = PP + K - 1 > 32;
    using MT = typename MaskT<WIDE>::type;
    constexpr int MB = (int)sizeof(MT) * 8;
    constexpr int NA = ((PP - 1) * 2 + 2 * K + 31) / 32;                 // aligned code words a chunk's K-mers touch
    constexpr int NM = WIDE ? 3 : 2;                                     // raw mask words
    const int kmin = ALLK ? 1 : kmin_arg;                                // ALLK: the default --minWordSize 1
    extern __shared__ __align__(16) unsigned char smem[];
    uint32_t* nib32 = reinterpret_cast<uint32_t*>(smem);                // word kappa >> 3, nibble kappa & 7
    const uint2* nib64 = reinterpret_cast<const uint2*>(smem);          // bucket kappa >> 4
    uint16_t* tab16 = reinterpret_cast<uint16_t*>(smem + L::OFF_LOW);    // orders 1..A at lvl_off(x)
    uint32_t* tab32 = reinterpret_cast<uint32_t*>(smem + L::OFF_LOW);
    double2* pre = reinterpret_cast<double2*>(smem + L::OFF_PRE);       // .x = num, .y = {flag, den} as two u32
    double2* preA = reinterpret_cast<double2*>(smem + L::OFF_PREA);     // FOLD_A: the same pair through order A, per order-A prefix
    NibSmem& ss = *reinterpret_cast<NibSmem*>(smem + L::OFF_SS);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (uint32_t i = tid; i < L::ZERO_BYTES / 16u; i += NT) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
    if (tid < 12) ss.cnt[tid / 6][tid % 6] = 0;
    __syncthreads();

    if (sw.n_win_dev) n_win = (uint32_t)min((unsigned long long)n_win, *sw.n_win_dev);
    int par = 1;
    for (uint32_t win = blockIdx.x; win < n_win; win += gridDim.x) {
        const uint64_t o = win_off[win];
        const uint32_t len = win_len[win];
        par ^= 1;
        // 32-bit addressing relative to the window's first mask word
        const uint32_t o_lo = (uint32_t)(o & 31);
        const uint32_t* __restrict__ cw = codes + (o >> 5) * 2;
        const uint32_t* __restrict__ mw = inv + (o >> 5);
        const uint32_t* __restrict__ lw = low ? low + (o >> 5) : nullptr;
        const uint32_t cs = max(4u, ((len + NT - 1) / NT + 3u) & ~3u);    // positions per thread (<= PP: checked by the launcher)
        const uint32_t p0 = (uint32_t)tid * cs;                          // this thread's first position

        // ---- P1: composition + ONE atomic per full K-word, all from registers ----------------------------
        uint32_t kk[PP / 2];                                             // two K-mer codes per register
        MT vm = 0;                                                       // position i (bit MB-1-i) holds a full K-word
        {
            int non = 0, gc = 0, nfull = 0;
#pragma unroll
            for (int i = 0; i < PP / 2; ++i) kk[i] = 0;
            if (p0 < len) {
                const uint32_t r0 = o_lo + p0;
                uint32_t raw[NA + 1], mraw[NM], lraw[NM];
#pragma unroll
                for (int j = 0; j <= NA; ++j) raw[j] = __ldg(cw + (r0 >> 4) + j);
#pragma unroll
                for (int j = 0; j < NM; ++j) mraw[j] = __ldg(mw + (r0 >> 5) + j);
#pragma unroll
                for (int j = 0; j < NM; ++j) lraw[j] = lw ? __ldg(lw + (r0 >> 5) + j) : 0u;
                uint32_t W[NA];                                          // W[j]: the 16 bases from position 16 j
                const uint32_t sc = (r0 & 15u) * 2u, ms = r0 & 31u;
#pragma unroll
                for (int j = 0; j < NA; ++j) W[j] = __funnelshift_l(raw[j + 1], raw[j], sc);
                MT M, Lm;
                if constexpr (WIDE) {
                    M = ((MT)__funnelshift_l(mraw[1], mraw[0], ms) << 32) | (MT)__funnelshift_l(mraw[2], mraw[1], ms);
                    Lm = ((MT)__funnelshift_l(lraw[1], lraw[0], ms) << 32) | (MT)__funnelshift_l(lraw[2], lraw[1], ms);
                } else {
                    M = __funnelshift_l(mraw[1], mraw[0], ms);
                    Lm = __funnelshift_l(lraw[1], lraw[0], ms);
                }
                const int left = (int)(len - p0);                        // positions from p0 to the window end
                const MT in_p = top_bits<MT>(left < (int)cs ? left : (int)cs);   // this thread's positions
                const MT bad = M | ~top_bits<MT>(left);                  // invalid character or beyond the window end
                MT sm = bad | (bad << 1);                                // position i: any bad base among i .. i+K-1
                sm |= sm << 2;
                sm |= sm << (K - 4);
                vm = ~sm & in_p;
                const MT unres = (M | Lm) & in_p;                        // not an upper-case ATGC (F:106-118)
                MT G = 0;                                                // bit 1 of the code: G = 2, C = 3 (invalid bases carry code 0)
#pragma unroll
                for (int j = 0; j < NA; ++j)
                    if (MB - 16 - 16 * j >= 0) G |= (MT)high_bits16(W[j]) << (MB - 16 - 16 * j);
                non = popc_m(unres);
                gc = popc_m(G & in_p & ~unres);
                nfull = popc_m(vm);
                // the full K-words: decode, address/value, one atomic each, no result awaited.  A chunk of PP positions
                // without an N (nearly all of them) runs the straight-line version: no per-position test
                auto kmer_at = [&](int i) -> uint32_t {
                    const int wi = i >> 4, oi = (i & 15) * 2;
                    if (oi + 2 * K <= 32) return (W[wi] << oi) >> (32 - 2 * K);
                    return __funnelshift_l(W[wi + 1 < NA ? wi + 1 : wi], W[wi], oi) >> (32 - 2 * K);
                };
                if (vm == top_bits<MT>(PP)) {
#pragma unroll
                    for (int i = 0; i < PP; i += 2) {
                        const uint32_t k0 = kmer_at(i), k1 = kmer_at(i + 1);
                        atomicAdd(&nib32[k0 >> 3], 1u << ((k0 & 7u) * 4u));
                        atomicAdd(&nib32[k1 >> 3], 1u << ((k1 & 7u) * 4u));
                        kk[i >> 1] = k0 | (k1 << 16);
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < PP; ++i) {
                        if (vm & (MT(1) << (MB - 1 - i))) {
                            const uint32_t kap = kmer_at(i);
                            atomicAdd(&nib32[kap >> 3], 1u << ((kap & 7u) * 4u));
                            kk[i >> 1] |= kap << (16 * (i & 1));
                        }
                    }
                }
                // words cut short by an N or the window end (rare): valid for v < K bases
                MT slow = in_p & ~vm & ~bad;
                while (slow) {
                    const int i = clz_m(slow);
                    slow &= ~(MT(1) << (MB - 1 - i));
                    const int v = clz_m((MT)(bad << i));                 // 1 <= v < K
                    const uint32_t r = r0 + (uint32_t)i;
                    const uint32_t c32 = __funnelshift_l(__ldg(cw + (r >> 4) + 1), __ldg(cw + (r >> 4)), (r & 15u) * 2u);
                    if (v >= A) {
                        const uint32_t ga = lvl_off(A) + (c32 >> (32 - 2 * A));
                        atomicAdd(&tab32[ga >> 1], 1u << ((ga & 1u) * 16u));
                        if (v > A) {                                     // K-1 or K-2 bases: side list + flag on its bin
                            atomicOr(&tab32[ga >> 1], 0x8000u << ((ga & 1u) * 16u));
                            const uint32_t slot = (uint32_t)atomicAdd(&ss.cnt[par][3], 1);
                            if (slot < kSideCap) ss.side[slot] = ((uint32_t)v << 16) | (c32 >> (32 - 2 * v));
                        }
                    } else {                                             // order v < A only
                        const uint32_t g = lvl_off(v) + (c32 >> (32 - 2 * v));
                        atomicAdd(&tab32[g >> 1], 1u << ((g & 1u) * 16u));
                    }
                }
            }
            non = __reduce_add_sync(kFull, non);
            gc = __reduce_add_sync(kFull, gc);
            nfull = __reduce_add_sync(kFull, nfull);
            if (lane == 0) { atomicAdd(&ss.cnt[par][0], non); atomicAdd(&ss.cnt[par][1], gc); atomicAdd(&ss.cnt[par][2], nfull); }
        }
        __syncthreads();                                                   // (1)
        const int n_non = ss.cnt[par][0], n_gc = ss.cnt[par][1], n_up = (int)len - n_non;
        const uint32_t n_side = (uint32_t)ss.cnt[par][3];
        if (tid < 6) ss.cnt[par ^ 1][tid] = 0;                              // next window's counters (idle until its P1)
        const bool excluded = (double)n_non >= 0.3 * (double)len;          // F:238 / F:213
        uint16_t* dmp = DUMP ? dump + (size_t)win * lvl_off(K + 1) : nullptr;
        if (excluded) {
            for (uint32_t i = tid; i < L::ZERO_BYTES / 16u; i += NT) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
            if (SWEEP) {
                if (tid < K) {
                    sw.status[tid][win] = FRISK_ROW_EXCLUDED;
                    for (int c = 0; c < 5; ++c) sw.rows[tid][(size_t)win * 5 + c] = CUDART_NAN;
                }
                if (tid == 0) redo_dst[win] = 0;
            } else if (tid == 0) {
                status[win] = FRISK_ROW_EXCLUDED;
                for (int c = 0; c < 5; ++c) rows[(size_t)win * 5 + c] = CUDART_NAN;
                if (redo_dst != status) redo_dst[win] = 0;
            }
            if (DUMP) for (uint32_t i = tid; i < lvl_off(K + 1); i += NT) dmp[i] = 0;
            __syncthreads();
            continue;
        }
        if (tid < K) {
            const int x = tid + 1;
            const long long d = ((long long)n_up - (long long)(x - 1)) * 2;
            ss.q[tid] = (double)pow4(x) / (double)d;
        }

        // ---- P2a: order A = the nibble sums of four consecutive buckets (+ the short words already there).  Per word:
        //      sum of bytes = lo-nibbles + 16 hi-nibbles, and the lo-nibbles alone -- two dp4a.  A wrapped nibble (a
        //      K-mer seen 16+ times) loses 15 or 16 from the grand total: that is how overflow is detected, for free.
        {
            uint32_t tot = 0;
            const uint32_t sw = (lane >> 2) & 1u;                          // lanes j and j+4 would share banks: swap their halves
            for (uint32_t b5 = tid; b5 < pow4(A); b5 += NT) {
                const uint4* src = reinterpret_cast<const uint4*>(smem) + 2u * b5;
                const uint4 v0 = src[sw], v1 = src[sw ^ 1u];
                uint32_t by = 0, lo = 0;
                const uint32_t w8[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
                for (int j = 0; j < 8; ++j) { by = __dp4a(w8[j], 0x01010101u, by); lo = __dp4a(w8[j] & 0x0f0f0f0fu, 0x01010101u, lo); }
                const uint32_t s = lo + ((by - lo) >> 4);
                tot += s;
                if (s) tab16[lvl_off(A) + b5] += (uint16_t)s;              // < 2^15 in total: the flag bit survives
            }
            tot = __reduce_add_sync(kFull, tot);
            if (lane == 0) atomicAdd(&ss.cnt[par][4], (int)tot);
        }
        __syncthreads();                                                   // (1b)
        if (ss.cnt[par][4] != ss.cnt[par][2] || n_side > kSideCap) {        // a nibble wrapped / too many cut words
            for (uint32_t i = tid; i < L::ZERO_BYTES / 16u; i += NT) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
            if (tid == 0) redo_dst[win] = kRowRedo;                        // the bucketed kernel takes this window (sweep: per kmax')
            __syncthreads();
            continue;
        }

        // ---- P2: orders 4..1 by marginalisation: thread t owns order-4 bin t; orders 3 and 2 by shuffles -----
        uint32_t c4 = 0, c3 = 0, c2 = 0, flag4 = 0;
        if (tid < 256) {
            if constexpr (A == 5) {
                const uint2 ch = *reinterpret_cast<const uint2*>(tab16 + lvl_off(5) + 4 * tid);
                c4 = (ch.x & 0x7fffu) + ((ch.x >> 16) & 0x7fffu) + (ch.y & 0x7fffu) + ((ch.y >> 16) & 0x7fffu)
                     + tab16[lvl_off(4) + tid];                              // + the short words of order 4
            } else {
                const uint32_t raw = tab16[lvl_off(4) + tid];
                c4 = raw & 0x7fffu; flag4 = raw >> 15;
            }
            uint32_t x = c4;
            x += __shfl_xor_sync(kFull, x, 1);
            x += __shfl_xor_sync(kFull, x, 2);
            c3 = x + tab16[lvl_off(3) + (tid >> 2)];
            uint32_t y = c3;
            y += __shfl_xor_sync(kFull, y, 4);
            y += __shfl_xor_sync(kFull, y, 8);
            c2 = y + tab16[lvl_off(2) + (tid >> 4)];
            if ((tid & 15) == 0) ss.c2[tid >> 4] = c2;
        }
        __syncthreads();                                                   // (2)
        if (tid < 256) {
            const uint32_t* q2 = ss.c2 + (tid >> 6) * 4;
            const uint32_t c1 = q2[0] + q2[1] + q2[2] + q2[3] + tab16[lvl_off(1) + (tid >> 6)];
            const uint32_t cs4[4] = {c1, c2, c3, c4};
            double num = 0.0;
            uint32_t den = 0;
#pragma unroll
            for (int x = 1; x <= LP; ++x) {
                if (x >= kmin) {
                    const uint32_t c = cs4[x - 1];
                    den += c << (2 * x);
                    num = fma(ss.q[x - 1], u32_to_double(c * c), num);
                }
            }
            pre[tid] = make_double2(num, __hiloint2double((int)flag4, (int)den));
            if (SWEEP) {                                                   // the bin walks of kmax' <= 4 read the TOTALS
                tab16[lvl_off(4) + tid] = (uint16_t)c4;
                if ((tid & 3) == 0) tab16[lvl_off(3) + (tid >> 2)] = (uint16_t)c3;
                if ((tid & 15) == 0) tab16[lvl_off(2) + (tid >> 4)] = (uint16_t)c2;
                if ((tid & 63) == 0) ss.c1[tid >> 6] = c1;                 // (its table entry is still being read by the others)
            }
            if (DUMP) {
                dmp[lvl_off(4) + tid] = (uint16_t)c4;
                if ((tid & 3) == 0) dmp[lvl_off(3) + (tid >> 2)] = (uint16_t)c3;
                if ((tid & 15) == 0) dmp[lvl_off(2) + (tid >> 4)] = (uint16_t)c2;
                if ((tid & 63) == 0) dmp[lvl_off(1) + (tid >> 6)] = (uint16_t)c1;
            }
        }
        __syncthreads();                                                   // (3)
        if constexpr (L::FOLD_A) {                                         // order A joins the folded pair: P3 reads one entry per K-mer
            const double qa = ss.q[A - 1];
            for (uint32_t b = tid; b < pow4(A); b += NT) {
                const uint32_t raw = tab16[lvl_off(A) + b], cA = raw & 0x7fffu;
                const double2 pp = pre[b >> 2];
                double num = pp.x;
                uint32_t den = (uint32_t)__double2loint(pp.y);
                if (A >= kmin) { den += cA << (2 * A); num = fma(qa, u32_to_double(cA * cA), num); }
                preA[b] = make_double2(num, __hiloint2double((int)(raw >> 15), (int)den));
            }
            __syncthreads();                                               // (3b)
        }
        if (DUMP) {                                                        // tests only: the window's tables, all orders
            if constexpr (A == 5)
                for (uint32_t i = tid; i < pow4(5); i += NT) dmp[lvl_off(5) + i] = tab16[lvl_off(5) + i] & 0x7fffu;
            for (uint32_t i = tid; i < pow4(K); i += NT) dmp[lvl_off(K) + i] = (uint16_t)((nib32[i >> 3] >> ((i & 7u) * 4u)) & 15u);
            for (uint32_t i = tid; i < pow4(K - 1); i += NT) {
                const uint32_t h = (nib32[i >> 1] >> ((i & 1u) * 16u)) & 0xffffu;
                dmp[lvl_off(K - 1) + i] = (uint16_t)((h & 15u) + ((h >> 4) & 15u) + ((h >> 8) & 15u) + (h >> 12));
            }
            for (uint32_t i = tid; i < pow4(K - 2); i += NT) {
                const uint2 v = nib64[i];
                dmp[lvl_off(K - 2) + i] = (uint16_t)__dp4a(nib_pairs(v.x) + nib_pairs(v.y), 0x01010101u, 0u);
            }
            __syncthreads();
            if (tid == 0) {
                for (uint32_t i = 0; i < n_side; ++i) {
                    const uint32_t e = ss.side[i], v = e >> 16, code = e & 0xffffu;
                    if (v == (uint32_t)(K - 1)) { dmp[lvl_off(K - 1) + code] += 1; dmp[lvl_off(K - 2) + (code >> 2)] += 1; }
                    else dmp[lvl_off(K - 2) + code] += 1;
                }
            }
        }

        if constexpr (SWEEP) {
            // ======== all K scores of this window (kmax' = 1..K, kmin = 1) ========
            double (*sred)[3][NW] = reinterpret_cast<double (*)[3][NW]>(pre);   // [kmax' - 1][sum][warp]; `pre` is dead after the kmax' = 4 walk
            auto warp_store = [&](int ks, double a, double b, double c) {
#pragma unroll
                for (int ofs = 16; ofs; ofs >>= 1) {
                    a += __shfl_xor_sync(kFull, a, ofs); b += __shfl_xor_sync(kFull, b, ofs); c += __shfl_xor_sync(kFull, c, ofs);
                }
                if (lane == 0) { sred[ks][0][warp] = a; sred[ks][1][warp] = b; sred[ks][2][warp] = c; }
            };
            auto accum = [&](double num, uint32_t den, const double2 g, double& a, double& b, double& c) {
                const double iw = div_pos(num, u32_to_double(den));
                a += iw; b += g.x; c = fma(iw, log2_series(iw) - g.y, c);
            };
            // kmax' = 4: one bin per thread, straight from `pre`; its sums wait in registers for the barrier that retires `pre`
            double w4 = 0.0, g4 = 0.0, t4 = 0.0;
            if (tab16[lvl_off(4) + tid]) {
                const double2 pp = pre[tid];
                accum(pp.x, (uint32_t)__double2loint(pp.y), __ldg(sw.ig[3] + tid), w4, g4, t4);
            }
            __syncthreads();                                               // (3c)
            warp_store(3, w4, g4, t4);
            // kmax' = 1..3: from the totals
#pragma unroll
            for (int kq = 1; kq <= 3; ++kq) {
                double a = 0.0, b = 0.0, c = 0.0;
                if ((uint32_t)tid < pow4(kq)) {
                    double num = 0.0;
                    uint32_t den = 0, ck = 0;
#pragma unroll
                    for (int x = 1; x <= kq; ++x) {
                        const uint32_t idx = (uint32_t)tid >> (2 * (kq - x));
                        ck = x == 1 ? ss.c1[idx] : (uint32_t)tab16[lvl_off(x) + idx];
                        den += ck << (2 * x);
                        num = fma(ss.q[x - 1], u32_to_double(ck * ck), num);
                    }
                    if (ck) accum(num, den, __ldg(sw.ig[kq - 1] + tid), a, b, c);
                }
                warp_store(kq - 1, a, b, c);
            }
            // kmax' = 5: the folded pair of every occupied order-5 bin
            {
                double a = 0.0, b = 0.0, c = 0.0;
                for (uint32_t bin = tid; bin < pow4(5); bin += NT) {
                    if (tab16[lvl_off(5) + bin] & 0x7fffu) {
                        const double2 pp = preA[bin];
                        accum(pp.x, (uint32_t)__double2loint(pp.y), __ldg(sw.ig[4] + bin), a, b, c);
                    }
                }
                warp_store(4, a, b, c);
            }
            const double q6 = ss.q[5], q7 = ss.q[6], q8 = ss.q[7];
            // the words cut at 7 / 6 bases (side list) that fall below a bucket / a quarter
            auto side_counts = [&](uint32_t bucket, uint32_t code7, uint32_t& c6, uint32_t& c7) {
                for (uint32_t i = 0; i < n_side; ++i) {
                    const uint32_t e = ss.side[i], sv = e >> 16, code = e & 0xffffu;
                    if (sv == 7u) { c7 += (code == code7); c6 += ((code >> 2) == bucket); }
                    else c6 += (code == bucket);
                }
            };
            // kmax' = 6: one bucket = one 6-mer
            {
                double a = 0.0, b = 0.0, c = 0.0;
                for (uint32_t bk = tid; bk < L::NBK; bk += NT) {
                    const uint2 v = nib64[bk];
                    uint32_t c6 = __dp4a(nib_pairs(v.x) + nib_pairs(v.y), 0x01010101u, 0u), c7 = 0;
                    const double2 pp = preA[bk >> 2];
                    if (__double2hiint(pp.y)) side_counts(bk, 0xffffffffu, c6, c7);
                    if (c6) accum(fma(q6, u32_to_double(c6 * c6), pp.x), (uint32_t)__double2loint(pp.y) + (c6 << 12), __ldg(sw.ig[5] + bk), a, b, c);
                }
                warp_store(5, a, b, c);
            }
            // kmax' = 7 and 8: every position, weights 1 / c7 and 1 / c8
            double w7 = 0.0, g7 = 0.0, t7 = 0.0, w8 = 0.0, g8 = 0.0, t8 = 0.0;
            auto weighted = [&](double num, uint32_t den, uint32_t cnt, const double2 g, double& a, double& b, double& c) {
                const double dden = u32_to_double(den), dc = u32_to_double(cnt);
                const double D = dden * dc;
                double r;
                asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(D));
                r = fma(r, fma(-D, r, 1.0), r);
                r = fma(r, fma(-D, r, 1.0), r);
                double x = num * r;
                x = fma(fma(-D, x, num), r, x);                            // I_w / cnt
                a += x;
                b = fma(g.x, dden * r, b);                                 // I_g / cnt
                c = fma(x, log2_series(x * dc) - g.y, c);
            };
            auto eval7 = [&](uint32_t code7, const uint2 v, const double2 pp, uint32_t c6, uint32_t c7) {
                weighted(fma(q7, u32_to_double(c7 * c7), fma(q6, u32_to_double(c6 * c6), pp.x)),
                         (uint32_t)__double2loint(pp.y) + (c6 << 12) + (c7 << 14), c7, __ldcg(sw.ig[6] + code7), w7, g7, t7);
                (void)v;
            };
            {
                const int rounds = (int)(cs >> 2);
#pragma unroll 1
                for (int r = 0; r < rounds; ++r) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        if (vm & (MT(1) << (MB - 1 - j))) {
                            const uint32_t kap = (kk[j >> 1] >> (16 * (j & 1))) & 0xffffu;
                            const double2 gg8 = __ldcg(sw.ig[7] + kap);           // L2 only, as in P3
                            const uint2 v = nib64[kap >> 4];
                            const uint32_t ws = (kap & 8u) ? v.y : v.x, wo = (kap & 8u) ? v.x : v.y;
                            const uint32_t c8 = (ws >> ((kap & 7u) * 4u)) & 15u;
                            const uint32_t ps = nib_pairs(ws);
                            const uint32_t hs = ps >> ((kap & 4u) * 4u);
                            uint32_t c7 = (hs & 0xffu) + ((hs >> 8) & 0xffu);
                            uint32_t c6 = __dp4a(ps + nib_pairs(wo), 0x01010101u, 0u);
                            const double2 pp = preA[kap >> 6];
                            if (__double2hiint(pp.y)) side_counts(kap >> 4, kap >> 2, c6, c7);
                            eval7(kap >> 2, v, pp, c6, c7);
                            const double n7 = fma(q7, u32_to_double(c7 * c7), fma(q6, u32_to_double(c6 * c6), pp.x));
                            weighted(fma(q8, u32_to_double(c8 * c8), n7), (uint32_t)__double2loint(pp.y) + (c6 << 12) + (c7 << 14) + (c8 << 16), c8, gg8,
                                     w8, g8, t8);
                        }
                    }
                    vm <<= 4;
#pragma unroll
                    for (int i = 0; i + 2 < PP / 2; ++i) kk[i] = kk[i + 2];
                }
            }
            if ((uint32_t)tid < n_side) {                                  // a word of exactly 7 bases is an occurrence of its 7-mer too
                const uint32_t e = ss.side[tid];
                if ((e >> 16) == 7u) {
                    const uint32_t code7 = e & 0xffffu, bk = code7 >> 2;
                    const uint2 v = nib64[bk];
                    const uint32_t h = ((code7 & 2u) ? v.y : v.x) >> ((code7 & 1u) * 16u);
                    uint32_t c7 = (h & 15u) + ((h >> 4) & 15u) + ((h >> 8) & 15u) + ((h >> 12) & 15u);
                    uint32_t c6 = __dp4a(nib_pairs(v.x) + nib_pairs(v.y), 0x01010101u, 0u);
                    side_counts(bk, code7, c6, c7);
                    eval7(code7, v, preA[bk >> 2], c6, c7);
                }
            }
            warp_store(6, w7, g7, t7);
            warp_store(7, w8, g8, t8);
            __syncthreads();                                               // (4) everyone is done with the tables
            for (uint32_t i = tid; i < L::ZERO_BYTES / 16u; i += NT) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
            if (warp == 0) {                                               // lane i finalises the row of kmax' = i + 1
                const int kq = lane < K ? lane + 1 : K;
                double a = 0, bsum = 0, c = 0;
                for (int w = 0; w < NW; ++w) { a += sred[kq - 1][0][w]; bsum += sred[kq - 1][1][w]; c += sred[kq - 1][2][w]; }
                uint32_t st = 0;
                double kld = 0.0;
                if (!(a == 0.0)) {
                    bool zd = bsum != bsum;
                    for (int x = 1; x <= kq; ++x) zd |= ((long long)n_up - (long long)(x - 1)) == 0;
                    if (zd) { st |= FRISK_ROW_KLD_ZERODIV; kld = CUDART_NAN; }
                    else {
                        kld = c / a + (log2(bsum) - log2(a));
                        if (!(kld == kld) || isinf(kld)) st |= FRISK_ROW_LOG_DOMAIN;
                    }
                }
                double gcv = CUDART_NAN;
                if (n_up == 0) st |= FRISK_ROW_GC_ZERODIV; else gcv = (double)n_gc / (double)n_up;
                double pi = CUDART_NAN, si = CUDART_NAN, cri = CUDART_NAN;
                if (want_rip && kq >= 2) {
                    const uint32_t n_at = ss.c2[1], n_ta = ss.c2[4], n_sub = ss.c2[3] + ss.c2[9], n_prod = ss.c2[12] + ss.c2[6];
                    if (n_at > 0) pi = (double)n_ta / (double)n_at;
                    if (n_sub > 0) si = (double)n_prod / (double)n_sub;
                    if (pi != 0.0 && si != 0.0) cri = pi - si;
                }
                if (lane < K) {
                    double* row = sw.rows[lane] + (size_t)win * 5;
                    row[0] = kld; row[1] = gcv; row[2] = pi; row[3] = si; row[4] = cri;
                    sw.status[lane][win] = st;
                }
                if (lane == 0) redo_dst[win] = 0;
            }
            __syncthreads();                                               // (5)
            continue;
        }

        // ---- P3: every position scores its own K-mer with weight 1 / (its count) --------------------
        double s_w = 0.0, s_g = 0.0, s_t = 0.0;
        const double qK2 = ss.q[K - 3], qK1 = ss.q[K - 2], qK = ss.q[K - 1];
        auto score_one = [&](uint32_t kap, const double2 g) {
            const uint2 v = nib64[kap >> 4];
            const uint32_t ws = (kap & 8u) ? v.y : v.x, wo = (kap & 8u) ? v.x : v.y;
            const uint32_t cK = (ws >> ((kap & 7u) * 4u)) & 15u;
            const uint32_t ps = nib_pairs(ws);
            const uint32_t hs = ps >> ((kap & 4u) * 4u);                   // the quarter of the (K-1)-prefix: two pair sums
            uint32_t cK1 = (hs & 0xffu) + ((hs >> 8) & 0xffu);
            uint32_t cK2 = __dp4a(ps + nib_pairs(wo), 0x01010101u, 0u);
            const double2 pp = L::FOLD_A ? preA[kap >> (2 * (K - A))] : pre[kap >> (2 * (K - LP))];
            double num = pp.x;
            uint32_t den = (uint32_t)__double2loint(pp.y);
            if (__double2hiint(pp.y)) {                    // rare: a short word of K-1 / K-2 bases lies below this bin
                for (uint32_t i = 0; i < n_side; ++i) {
                    const uint32_t e = ss.side[i], sv = e >> 16, code = e & 0xffffu;
                    if (sv == (uint32_t)(K - 1)) { cK1 += (code == (kap >> 2)); cK2 += ((code >> 2) == (kap >> 4)); }
                    else cK2 += (code == (kap >> 4));
                }
            }
            if (K - 2 >= kmin) { den += cK2 << (2 * (K - 2)); num = fma(qK2, u32_to_double(cK2 * cK2), num); }
            if (K - 1 >= kmin) { den += cK1 << (2 * (K - 1)); num = fma(qK1, u32_to_double(cK1 * cK1), num); }
            den += cK << (2 * K);
            num = fma(qK, u32_to_double(cK * cK), num);
            // a = I_w / c_K, om = 1 / c_K from ONE reciprocal, of den * c_K (exact product, < 2^37)
            const double dden = u32_to_double(den), dc = u32_to_double(cK);
            const double D = dden * dc;
            double r;
            asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(D));
            r = fma(r, fma(-D, r, 1.0), r);
            r = fma(r, fma(-D, r, 1.0), r);
            double a = num * r;
            a = fma(fma(-D, a, num), r, a);
            const double iw = a * dc;
            const double om = dden * r;
            s_w += a;
            s_g = fma(g.x, om, s_g);                       // a NaN entry (reference: ZeroDivisionError) poisons the sum
            s_t = fma(a, log2_series(iw) - g.y, s_t);
        };
        const int rounds = (int)(cs >> 2);
#pragma unroll 1
        for (int r = 0; r < rounds; ++r) {
            uint32_t kp[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) kp[j] = (kk[j >> 1] >> (16 * (j & 1))) & 0xffffu;
            // positions j and j + 1 fetch both genome-IVOM entries with ONE 32-byte load from the pair table, at the
            // (K+1)-mer of bases j .. j+K.  Only j + 1 valid: its K-mer with a leading A (the second half is still its
            // entry).  Only j valid: the first half is used, kp[j + 1] & 3 only keeps mu in range.  L2 only (.cg): the
            // table never survives in a ~30 KB L1 anyway, and not allocating there measured faster (0.703 -> 0.671 ms on C2)
#pragma unroll
            for (int j = 0; j < 4; j += 2) {
                const bool v0 = vm & (MT(1) << (MB - 1 - j)), v1 = vm & (MT(1) << (MB - 2 - j));
                if (v0 || v1) {
                    const uint32_t mu = v0 ? ((kp[j] << 2) | (kp[j + 1] & 3u)) : kp[j + 1];
                    double2 g0, g1;
                    ldcg_pair(pair + 2u * mu, g0, g1);
                    if (v0) score_one(kp[j], g0);
                    if (v1) score_one(kp[j + 1], g1);
                }
            }
            vm <<= 4;
#pragma unroll
            for (int i = 0; i + 2 < PP / 2; ++i) kk[i] = kk[i + 2];         // rotate: the loop body stays one round long
#pragma unroll
            for (int i = (PP / 2 > 2 ? PP / 2 - 2 : 0); i < PP / 2; ++i) kk[i] = 0;
        }
#pragma unroll
        for (int ofs = 16; ofs; ofs >>= 1) {
            s_w += __shfl_xor_sync(kFull, s_w, ofs);
            s_g += __shfl_xor_sync(kFull, s_g, ofs);
            s_t += __shfl_xor_sync(kFull, s_t, ofs);
        }
        if (lane == 0) { ss.red[0][warp] = s_w; ss.red[1][warp] = s_g; ss.red[2][warp] = s_t; }
        __syncthreads();                                                   // (4) everyone is done with the tables
        for (uint32_t i = tid; i < L::ZERO_BYTES / 16u; i += NT) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
        if (warp == 0) {
            // the row: four IEEE divisions and two logarithms, one per LANE instead of one after the other in a single
            // thread (the other seven warps of the CTA wait for this at the barrier below)
            double a = 0, bsum = 0, c = 0;
            for (int w = 0; w < NW; ++w) { a += ss.red[0][w]; bsum += ss.red[1][w]; c += ss.red[2][w]; }
            double nu = 0.0, de = 1.0;
            if (lane == 0) { nu = c; de = a; }
            else if (lane == 1) { nu = (double)n_gc; de = (double)n_up; }                                   // F:136
            else if (lane == 2) { nu = (double)ss.c2[4]; de = (double)ss.c2[1]; }                          // TA / AT, F:480-483
            else if (lane == 3) { nu = (double)(ss.c2[12] + ss.c2[6]); de = (double)(ss.c2[3] + ss.c2[9]); }  // (CA+TG) / (AC+GT), F:485-489
            const double qv = nu / de;
            const double lgv = log2(lane == 0 ? bsum : a);
            const double q_gc = __shfl_sync(kFull, qv, 1), q_pi = __shfl_sync(kFull, qv, 2), q_si = __shfl_sync(kFull, qv, 3);
            const double lg_a = __shfl_sync(kFull, lgv, 1);
            if (lane == 0) {
                uint32_t st = 0;
                double kld = 0.0;                          // the reference returns 0 for a window without kmax-mers
                if (!(a == 0.0)) {
                    bool zd = bsum != bsum;                // NaN genome IVOM entry: ZeroDivisionError at F:437
                    for (int x = kmin; x <= K; ++x) zd |= ((long long)n_up - (long long)(x - 1)) == 0;
                    if (zd) { st |= FRISK_ROW_KLD_ZERODIV; kld = CUDART_NAN; }
                    else {
                        kld = qv + (lgv - lg_a);
                        if (!(kld == kld) || isinf(kld)) st |= FRISK_ROW_LOG_DOMAIN;
                    }
                }
                double* row = rows + (size_t)win * 5;
                row[0] = kld;
                if (n_up == 0) { st |= FRISK_ROW_GC_ZERODIV; row[1] = CUDART_NAN; }
                else row[1] = q_gc;
                double pi = CUDART_NAN, si = CUDART_NAN, cri = CUDART_NAN;
                if (want_rip) {
                    if (ss.c2[1] > 0) pi = q_pi;
                    if (ss.c2[3] + ss.c2[9] > 0) si = q_si;
                    if (pi != 0.0 && si != 0.0) cri = pi - si;         // F:491: 0.0 falsy, NaN truthy
                }
                row[2] = pi; row[3] = si; row[4] = cri;
                status[win] = st;
                if (redo_dst != status) redo_dst[win] = 0;
            }
        }
        __syncthreads();                                                   // (5) tables zeroed, ss.red consumed
    }
}

// The pair table of P3: P[mu] = {ig[mu >> 2], ig[mu & (4^K - 1)]} for every (K+1)-mer mu, i.e. the genome-IVOM entries of
// the K-mers at two adjacent positions p, p + 1 (bases p .. p+K) in one 32-byte entry, 4^(K+1) x 32 B (8 MiB at K = 8, 2 MiB
// at K = 7).  Bits are copied: a NaN entry (query k-mer absent from the host, the reference's ZeroDivisionError) stays NaN.
template <int K>
__global__ void __launch_bounds__(256) ivom_pair_kernel(const uint4* __restrict__ ig, uint4* __restrict__ pair) {
    const uint32_t mu = blockIdx.x * 256u + threadIdx.x;                 // the grid covers 4^(K+1) exactly
    pair[2u * mu] = __ldg(ig + (mu >> 2));
    pair[2u * mu + 1u] = __ldg(ig + (mu & (pow4(K) - 1u)));
}

template <int K>
const void* nibble_fn(const frisk_internal::WinPlan& p) {
    if (p.variant == 8) return FRISK_WIN_INSTANCE(p, score_windows_nibble_kernel, K, 8);
    if (p.variant == 20) return FRISK_WIN_INSTANCE(p, score_windows_nibble_kernel, K, 20);
    return FRISK_WIN_INSTANCE(p, score_windows_nibble_kernel, K, 32);
}

// one launch of a nibble-kernel instantiation, the sweep's included (they share the signature)
int launch_nibble(const frisk_internal::LaunchShape& s, const uint32_t* codes, const uint32_t* inv, const uint32_t* low,
                  const uint64_t* win_off, const uint32_t* win_len, uint64_t n_win, const double2* pair, int kmin, int want_rip,
                  double* rows, uint32_t* status, uint16_t* dump, uint32_t* redo_dst, NibSweep sw, cudaStream_t st) {
    const unsigned long long* off = reinterpret_cast<const unsigned long long*>(win_off);
    uint32_t n = (uint32_t)n_win;
    void* args[] = {&codes, &inv, &low, &off, &win_len, &n, &pair, &kmin, &want_rip, &rows, &status, &dump, &redo_dst, &sw};
    return frisk_internal::launch_persistent(s, n_win, args, st);
}

}  // namespace

frisk_internal::LaunchShape frisk_internal::nibble_shape(const WinPlan& p, int K) {
    if (K == 8) return {nibble_fn<8>(p), kNT, NibLayout<8>::TOTAL, true};
    return {nibble_fn<7>(p), kNT, NibLayout<7>::TOTAL, true};
}

int frisk_internal::score_nibble(const WinPlan& p, const uint32_t* codes, const uint32_t* inv, const uint32_t* low,
                                 const uint64_t* win_off, const uint32_t* win_len, uint64_t n_win, uint32_t max_len, const double* ig,
                                 int kmin, int K, int want_rip, double* rows, uint32_t* status, uint16_t* dump, cudaStream_t st,
                                 const unsigned long long* n_win_dev) {
    if (K != 7 && K != 8) return FRISK_E_UNSUPPORTED;
    NibSweep sw{};
    sw.n_win_dev = n_win_dev;
    // the pair table: stream-ordered scratch, built from ig right before the window kernel, freed behind the hand-over
    int rc = pool_ready();
    if (rc) return rc;
    const uint32_t n_pair = pow4(K + 1);
    uint4* pair = nullptr;
    FRISK_CK(cudaMallocAsync((void**)&pair, (size_t)n_pair * 32u, st));
    (K == 8 ? ivom_pair_kernel<8> : ivom_pair_kernel<7>)<<<n_pair / 256u, 256, 0, st>>>(reinterpret_cast<const uint4*>(ig), pair);
    const cudaError_t le = cudaGetLastError();
    if (le != cudaSuccess) rc = cuda_fail(le, "ivom_pair_kernel");
    if (!rc)
        rc = with_redo_marks(status, n_win, n_win_dev != nullptr, st, [&](uint32_t* redo) {
            int rc2 = launch_nibble(nibble_shape(p, K), codes, inv, low, win_off, win_len, n_win, reinterpret_cast<const double2*>(pair),
                                    kmin, want_rip, rows, status, dump, redo, sw, st);
            // windows the nibble table could not hold (marked kRowRedo): exact re-run on the bucketed kernel, which reads ig
            return rc2 ? rc2 : score_bucket_redo(codes, inv, low, win_off, win_len, n_win, max_len, ig, kmin, K, want_rip, rows, status,
                                                 dump, redo, st);
        });
    const cudaError_t e = cudaFreeAsync(pair, st);                     // stream-ordered: behind the launches above
    if (!rc && e != cudaSuccess) return cuda_fail(e, "cudaFreeAsync(pair table)");
    return rc;
}

// The k sweep: rows of kmax' = 1..8 (kmin 1) for every window from one pass (see NibSweep).  A window the 4-bit counters
// cannot hold is handed, for every kmax', to the kernel that serves that kmax' on its own.
int frisk_internal::score_sweep(const uint32_t* codes, const uint32_t* inv, const uint32_t* low, const uint64_t* win_off,
                                const uint32_t* win_len, uint64_t n_win, uint32_t max_len, const double* const* ig, int want_rip,
                                double* const* rows, uint32_t* const* status, cudaStream_t st) {
    if (max_len > kSmemMaxWindow) return FRISK_E_UNSUPPORTED;
    NibSweep sw{};
    for (int k = 0; k < 8; ++k) {
        if (!ig[k] || !rows[k] || !status[k]) return FRISK_E_INVALID;
        sw.ig[k] = reinterpret_cast<const double2*>(ig[k]); sw.rows[k] = rows[k]; sw.status[k] = status[k];
    }
    const int pp = window_variant(WinKernel::Nibble, max_len);
    const void* fn = pp == 8    ? (const void*)score_windows_nibble_kernel<8, 8, false, true, true>
                     : pp == 20 ? (const void*)score_windows_nibble_kernel<8, 20, false, true, true>
                                : (const void*)score_windows_nibble_kernel<8, 32, false, true, true>;
    return with_redo_marks(nullptr, n_win, false, st, [&](uint32_t* redo) {
        int rc = launch_nibble({fn, kNT, NibLayout<8>::TOTAL, true}, codes, inv, low, win_off, win_len, n_win, nullptr, 1, want_rip,
                               nullptr, nullptr, nullptr, redo, sw, st);
        for (int k = 1; k <= 8 && !rc; ++k)
            rc = score_bucket_redo(codes, inv, low, win_off, win_len, n_win, max_len, ig[k - 1], 1, k, want_rip && k >= 2, rows[k - 1],
                                   status[k - 1], nullptr, redo, st);
        return rc;
    });
}
