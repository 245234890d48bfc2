// frisk_b200: window scores for kmax 9..12 (windows <= 8,186 bases) at nearly the cost of kmax 8.
//
// Replaces, per window, the reference's computeKmers(window) + IvomBuild x2 + KLD + calcGC + calcRIP for `-k 9..12`
// (/root/reference/frisk/__init__.py F:1197-1206 accepts any k; F:1478-1494, F:280-367, F:369-472).
//
// The orders 1..8 are counted exactly as in the kmax-8 nibble kernel (frisk_nibble.cu: one 4-bit counter per 8-mer,
// one shared-memory atomic per position, lower orders by marginalisation).  The orders 9..K need no table at all:
//   * a position whose 8-mer occurs ONCE in the window has c_9 = ... = c_K = 1 (any extension of a unique word is unique);
//     in a 5 kb window that is ~96 % of the positions;
//   * the positions whose 8-mer repeats (c_8 >= 2) put their order-9 prefix into a small open-addressing hash table in
//     shared memory (tag = order + prefix, 4-bit count in the same 32-bit slot); those whose 9-mer still repeats their
//     order-10 prefix, and so on: the set shrinks about four-fold per order, and only its members look the table up.
// Every position that starts a full K-word scores its K-mer with weight 1/c_K (sum over positions = sum over distinct
// K-mers, F:448-472), fixed thread -> positions mapping, fixed reduction tree: bit-reproducible rows.
// The K-mer codes are not kept in registers between the passes: each pass re-reads the thread's four code words (L1/L2
// hits) and walks them with a 2-bit shift register, so the loops are not unrolled and the code stays small.
//
// What this cannot hold -- an 8-mer seen 16+ times, more than 64 words cut at 7 / 6 bases, a hash table more than 5/8
// full (a window made of repeats) -- is marked kRowRedo and re-done by the general kernel (frisk_general.cu) behind it.
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
constexpr int NW = kNT / 32;
constexpr uint32_t kHashSlots = 4096;                 // u32 each: tag << 4 | count
constexpr uint32_t kHashMaxKeys = kHashSlots * 5 / 8;
constexpr int kMaxProbe = 64;

struct ExtSmem {
    double q[12];
    double red[3][NW];
    int cnt[2][8];                    // [parity][n_non, n_gc, full 8-words counted, n_side, sum of nibbles, hash keys, hash overflow, -]
    uint32_t c2[16];
    uint32_t side[kSideCap];
};

// shared-memory layout: [nibbles of order 8 | u16 counts of orders 1..5 | hash] zeroed per window, then the folded pairs
struct ExtLayout {
    static constexpr int A = 5, LP = 4;
    static constexpr uint32_t NBK = pow4(6);
    static constexpr uint32_t NIB_BYTES = NBK * 8u;
    static constexpr uint32_t LOW_BYTES = (lvl_off(A + 1) * 2u + 15u) & ~15u;
    static constexpr uint32_t OFF_LOW = NIB_BYTES;
    static constexpr uint32_t OFF_HASH = OFF_LOW + LOW_BYTES;
    static constexpr uint32_t ZERO_BYTES = OFF_HASH + kHashSlots * 4u;
    static constexpr uint32_t OFF_PRE = ZERO_BYTES;
    static constexpr uint32_t OFF_PREA = OFF_PRE + pow4(LP) * 16u;
    static constexpr uint32_t OFF_SS = OFF_PREA + pow4(A) * 16u;
    static constexpr uint32_t TOTAL = OFF_SS + (uint32_t)sizeof(ExtSmem);
};

__device__ __forceinline__ unsigned long long top_bits64(int n) { return n >= 64 ? ~0ull : ~(~0ull >> n); }

// tag of the order-x prefix `code` (2x bits, x = 9..12): never 0
__device__ __forceinline__ uint32_t ext_tag(int x, uint32_t code) { return 1u + (((uint32_t)(x - 9) << 24) | code); }
__device__ __forceinline__ uint32_t ext_slot(uint32_t tag) { return (tag * 2654435761u) >> 20; }          // 12 bits: kHashSlots = 4096

// PP = positions per thread (one chunk of consecutive positions, as in the kmax-8 kernel); the masks are 64 bits wide:
// PP + K - 1 <= 43
template <int PP, bool ALLK>
__global__ void __launch_bounds__(kNT, 3)
score_windows_nibble_ext_kernel(const uint32_t* __restrict__ codes, const uint32_t* __restrict__ inv, const uint32_t* __restrict__ low,
                                const unsigned long long* __restrict__ win_off, const uint32_t* __restrict__ win_len, uint32_t n_win,
                                const double2* __restrict__ ig, int kmin_arg, int K, int want_rip,
                                double* __restrict__ rows, uint32_t* __restrict__ status, uint32_t* redo_dst) {
    using L = ExtLayout;
    constexpr int A = L::A, LP = L::LP, NT = kNT;
    using MT = unsigned long long;
    constexpr int MB = 64;
    constexpr int NAW = (PP + 12 - 1 + 15 + 15) / 16;                    // aligned code words: the chunk, 11 bases of look-ahead, 16 for the walk
    const int kmin = ALLK ? 1 : kmin_arg;
    extern __shared__ __align__(16) unsigned char smem[];
    uint32_t* nib32 = reinterpret_cast<uint32_t*>(smem);
    const uint2* nib64 = reinterpret_cast<const uint2*>(smem);
    uint16_t* tab16 = reinterpret_cast<uint16_t*>(smem + L::OFF_LOW);
    uint32_t* tab32 = reinterpret_cast<uint32_t*>(smem + L::OFF_LOW);
    uint32_t* hash = reinterpret_cast<uint32_t*>(smem + L::OFF_HASH);
    double2* pre = reinterpret_cast<double2*>(smem + L::OFF_PRE);
    double2* preA = reinterpret_cast<double2*>(smem + L::OFF_PREA);
    ExtSmem& ss = *reinterpret_cast<ExtSmem*>(smem + L::OFF_SS);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (uint32_t i = tid; i < L::ZERO_BYTES / 16u; i += NT) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
    if (tid < 16) ss.cnt[tid >> 3][tid & 7] = 0;
    __syncthreads();

    int par = 1;
    for (uint32_t win = blockIdx.x; win < n_win; win += gridDim.x) {
        const uint64_t o = win_off[win];
        const uint32_t len = win_len[win];
        par ^= 1;
        const uint32_t o_lo = (uint32_t)(o & 31);
        const uint32_t* __restrict__ cw = codes + (o >> 5) * 2;
        const uint32_t* __restrict__ mw = inv + (o >> 5);
        const uint32_t* __restrict__ lw = low ? low + (o >> 5) : nullptr;
        const uint32_t cs = max(4u, ((len + NT - 1) / NT + 3u) & ~3u);    // positions per thread (<= PP: checked by the launcher)
        const uint32_t p0 = (uint32_t)tid * cs;
        const uint32_t r0 = o_lo + p0;
        const int left = (int)len - (int)p0;                             // positions from p0 to the window end (<= 0: idle thread)

        // the thread's chunk: aligned code words, invalid / beyond-the-window mask, own positions
        uint32_t W[NAW];
        MT bad = ~0ull, in_p = 0;
        auto load_chunk = [&](MT* lower) {
            uint32_t raw[NAW + 1];
#pragma unroll
            for (int j = 0; j <= NAW; ++j) raw[j] = __ldg(cw + (r0 >> 4) + j);
            const uint32_t m0 = __ldg(mw + (r0 >> 5)), m1 = __ldg(mw + (r0 >> 5) + 1), m2 = __ldg(mw + (r0 >> 5) + 2);
            const uint32_t sc = (r0 & 15u) * 2u, ms = r0 & 31u;
#pragma unroll
            for (int j = 0; j < NAW; ++j) W[j] = __funnelshift_l(raw[j + 1], raw[j], sc);
            const MT M = ((MT)__funnelshift_l(m1, m0, ms) << 32) | (MT)__funnelshift_l(m2, m1, ms);
            in_p = top_bits64(left < (int)cs ? left : (int)cs);
            bad = M | ~top_bits64(left);
            if (lower) {
                MT Lm = 0;
                if (lw) {
                    const uint32_t l0 = __ldg(lw + (r0 >> 5)), l1 = __ldg(lw + (r0 >> 5) + 1), l2 = __ldg(lw + (r0 >> 5) + 2);
                    Lm = ((MT)__funnelshift_l(l1, l0, ms) << 32) | (MT)__funnelshift_l(l2, l1, ms);
                }
                *lower = (M | Lm) & in_p;                               // not an upper-case ATGC (F:106-118)
            }
        };

        // ---- P1: composition + ONE atomic per position that starts a word of 8+ valid bases ---------------
        {
            int non = 0, gc = 0, nfull = 0;
            if (left > 0) {
                MT unres;
                load_chunk(&unres);
                MT sm = bad | (bad << 1);
                sm |= sm << 2;
                sm |= sm << 4;
                const MT vm8 = ~sm & in_p;                               // 8+ valid bases from here
                MT G = 0;
#pragma unroll
                for (int j = 0; j < NAW && j < 4; ++j) G |= (MT)high_bits16(W[j]) << (MB - 16 - 16 * j);
                non = __popcll(unres);
                gc = __popcll(G & in_p & ~unres);
                nfull = __popcll(vm8);
                auto kmer8_at = [&](int i) -> uint32_t {
                    const int wi = i >> 4, oi = (i & 15) * 2;
                    if (oi <= 16) return (W[wi] << oi) >> 16;
                    return __funnelshift_l(W[wi + 1 < NAW ? wi + 1 : wi], W[wi], oi) >> 16;
                };
                if (vm8 == top_bits64(PP)) {
#pragma unroll
                    for (int i = 0; i < PP; ++i) {
                        const uint32_t k8 = kmer8_at(i);
                        atomicAdd(&nib32[k8 >> 3], 1u << ((k8 & 7u) * 4u));
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < PP; ++i) {
                        if (vm8 & (MT(1) << (MB - 1 - i))) {
                            const uint32_t k8 = kmer8_at(i);
                            atomicAdd(&nib32[k8 >> 3], 1u << ((k8 & 7u) * 4u));
                        }
                    }
                }
                MT slow = in_p & ~vm8 & ~bad;                            // words cut short at v < 8 bases
                while (slow) {
                    const int i = __clzll((long long)slow);
                    slow &= ~(MT(1) << (MB - 1 - i));
                    const int v = __clzll((long long)(bad << i));        // 1 <= v < 8
                    const uint32_t r = r0 + (uint32_t)i;
                    const uint32_t c32 = __funnelshift_l(__ldg(cw + (r >> 4) + 1), __ldg(cw + (r >> 4)), (r & 15u) * 2u);
                    if (v >= A) {
                        const uint32_t ga = lvl_off(A) + (c32 >> (32 - 2 * A));
                        atomicAdd(&tab32[ga >> 1], 1u << ((ga & 1u) * 16u));
                        if (v > A) {                                     // 7 or 6 bases: side list + flag on its order-5 bin
                            atomicOr(&tab32[ga >> 1], 0x8000u << ((ga & 1u) * 16u));
                            const uint32_t slot = (uint32_t)atomicAdd(&ss.cnt[par][3], 1);
                            if (slot < kSideCap) ss.side[slot] = ((uint32_t)v << 16) | (c32 >> (32 - 2 * v));
                        }
                    } else {
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
        if (tid < 8) ss.cnt[par ^ 1][tid] = 0;
        const bool excluded = (double)n_non >= 0.3 * (double)len;          // F:238 / F:213
        auto give_up = [&](bool excl) {                                    // clear the tables; excluded row or hand-over mark
            for (uint32_t i = tid; i < L::ZERO_BYTES / 16u; i += NT) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
            if (tid == 0) {
                if (excl) {
                    status[win] = FRISK_ROW_EXCLUDED;
                    for (int c = 0; c < 5; ++c) rows[(size_t)win * 5 + c] = CUDART_NAN;
                    if (redo_dst != status) redo_dst[win] = 0;
                } else {
                    redo_dst[win] = kRowRedo;
                }
            }
            __syncthreads();
        };
        if (excluded) { give_up(true); continue; }
        if (tid < K) {
            const int x = tid + 1;
            const long long d = ((long long)n_up - (long long)(x - 1)) * 2;
            ss.q[tid] = (double)(1ull << (2 * x)) / (double)d;
        }

        // ---- P2a: order 5 = the nibble sums of four consecutive buckets (as in frisk_nibble.cu) ---------------
        {
            uint32_t tot = 0;
            const uint32_t sw = (lane >> 2) & 1u;
            for (uint32_t b5 = tid; b5 < pow4(A); b5 += NT) {
                const uint4* src = reinterpret_cast<const uint4*>(smem) + 2u * b5;
                const uint4 v0 = src[sw], v1 = src[sw ^ 1u];
                uint32_t by = 0, lo = 0;
                const uint32_t w8[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
                for (int j = 0; j < 8; ++j) { by = __dp4a(w8[j], 0x01010101u, by); lo = __dp4a(w8[j] & 0x0f0f0f0fu, 0x01010101u, lo); }
                const uint32_t s = lo + ((by - lo) >> 4);
                tot += s;
                if (s) tab16[lvl_off(A) + b5] += (uint16_t)s;
            }
            tot = __reduce_add_sync(kFull, tot);
            if (lane == 0) atomicAdd(&ss.cnt[par][4], (int)tot);
        }
        __syncthreads();                                                   // (1b)
        if (ss.cnt[par][4] != ss.cnt[par][2] || n_side > kSideCap) { give_up(false); continue; }   // a nibble wrapped / too many cut words

        // ---- P2: orders 4..1 by marginalisation, the folded {numerator, denominator} pairs per order-4 / order-5 prefix ----
        uint32_t c4 = 0, c3 = 0, c2 = 0;
        {
            const uint2 ch = *reinterpret_cast<const uint2*>(tab16 + lvl_off(5) + 4 * tid);
            c4 = (ch.x & 0x7fffu) + ((ch.x >> 16) & 0x7fffu) + (ch.y & 0x7fffu) + ((ch.y >> 16) & 0x7fffu) + tab16[lvl_off(4) + tid];
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
        {
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
            pre[tid] = make_double2(num, __hiloint2double(0, (int)den));
        }
        __syncthreads();                                                   // (3)
        {
            const double qa = ss.q[A - 1];
            for (uint32_t b = tid; b < pow4(A); b += NT) {
                const uint32_t raw = tab16[lvl_off(A) + b], cA = raw & 0x7fffu;
                const double2 pp = pre[b >> 2];
                double num = pp.x;
                uint32_t den = (uint32_t)__double2loint(pp.y);
                if (A >= kmin) { den += cA << (2 * A); num = fma(qa, u32_to_double(cA * cA), num); }
                preA[b] = make_double2(num, __hiloint2double((int)(raw >> 15), (int)den));
            }
        }
        // (no barrier: the next pass reads only the nibbles and writes only the hash)

        // ---- P3: order by order (9..K), the positions whose prefix of the order below REPEATS register their prefix of this
        //      order; everything else is unique from there on.  One walk over the chunk per order: Wa = the 16 bases from
        //      the current position (an x-mer is its top 2x <= 24 bits), bd = the invalid mask from it.
        if (left > 0) load_chunk(nullptr);
        {
            MT cm = 0;                                                     // positions whose prefix of the previous order repeats
            int mine = 0;
            bool over = false;
            const int n_pos = left > 0 ? (left < (int)cs ? left : (int)cs) : 0;
            auto lookup = [&](uint32_t tag) -> uint32_t {
                uint32_t s = ext_slot(tag);
                for (int probe = 0; probe < kMaxProbe; ++probe) {
                    const uint32_t cur = hash[s];
                    if ((cur >> 4) == tag) return cur & 15u;
                    if (cur == 0u) break;
                    s = (s + 1u) & (kHashSlots - 1u);
                }
                return 0u;
            };
            for (int x = 9; x <= K; ++x) {
                uint32_t Wa = W[0], Wb = W[1], Wc = NAW > 2 ? W[2] : 0u, Wd = NAW > 3 ? W[3] : 0u;
                MT bd = bad, ncm = 0;
                for (int i = 0; i < n_pos; ++i) {
                    if (min(__clzll((long long)bd), K) >= x) {             // x valid bases from this position
                        bool rep;
                        if (x == 9) {
                            const uint32_t k8 = Wa >> 16;
                            rep = ((nib32[k8 >> 3] >> ((k8 & 7u) * 4u)) & 15u) >= 2u;
                        } else {
                            rep = (cm >> (MB - 1 - i)) & 1ull ? lookup(ext_tag(x - 1, Wa >> (34 - 2 * x))) >= 2u : false;
                        }
                        if (rep) {
                            const uint32_t tag = ext_tag(x, Wa >> (32 - 2 * x));
                            uint32_t s = ext_slot(tag);
                            int probe = 0;
                            for (; probe < kMaxProbe; ++probe) {
                                uint32_t cur = reinterpret_cast<volatile uint32_t*>(hash)[s];
                                if (cur == 0u) {
                                    cur = atomicCAS(&hash[s], 0u, (tag << 4) | 1u);
                                    if (cur == 0u) break;                  // claimed the empty slot: count 1
                                }
                                if ((cur >> 4) == tag) { atomicAdd(&hash[s], 1u); break; }
                                s = (s + 1u) & (kHashSlots - 1u);
                            }
                            if (probe == kMaxProbe) over = true;
                            ncm |= MT(1) << (MB - 1 - i);
                            ++mine;
                        }
                    }
                    Wa = __funnelshift_l(Wb, Wa, 2); Wb = __funnelshift_l(Wc, Wb, 2); Wc = __funnelshift_l(Wd, Wc, 2); Wd <<= 2;
                    bd <<= 1;
                }
                cm = ncm;
                if (x < K) __syncthreads();                                // this order's counts are final before the next order reads them
            }
            if (mine) atomicAdd(&ss.cnt[par][5], mine);
            if (over) ss.cnt[par][6] = 1;
        }
        __syncthreads();                                                   // (3b)
        if ((uint32_t)ss.cnt[par][5] > kHashMaxKeys || ss.cnt[par][6]) { give_up(false); continue; }   // a window of repeats

        // ---- P4: every position that starts a full K-word scores its K-mer with weight 1 / c_K ------------------
        double s_w = 0.0, s_g = 0.0, s_t = 0.0;
        if (left > 0) {
            const double q6 = ss.q[5], q7 = ss.q[6], q8 = ss.q[7];
            double qsum = 0.0;                                             // orders 9..K of a K-mer whose 8-mer is unique: all counts 1
            uint32_t dsum = 0;
            for (int x = 9; x <= K; ++x)
                if (x >= kmin) { qsum += ss.q[x - 1]; dsum += 1u << (2 * x); }
            uint32_t Wa = W[0], Wb = W[1], Wc = NAW > 2 ? W[2] : 0u, Wd = NAW > 3 ? W[3] : 0u;
            MT bd = bad;
            const int n_pos = left < (int)cs ? left : (int)cs;
#pragma unroll 1
            for (int i = 0; i < n_pos; ++i) {
                if (__clzll((long long)bd) >= K) {
                    const uint32_t kap = Wa >> 16;                         // the 8-mer
                    const uint32_t kK = Wa >> (32 - 2 * K);                // the K-mer
                    const double2 g = __ldcg(ig + kK);
                    const uint2 v = nib64[kap >> 4];
                    const uint32_t ws = (kap & 8u) ? v.y : v.x, wo = (kap & 8u) ? v.x : v.y;
                    const uint32_t c8 = (ws >> ((kap & 7u) * 4u)) & 15u;
                    const uint32_t ps = nib_pairs(ws);
                    const uint32_t hs = ps >> ((kap & 4u) * 4u);
                    uint32_t c7 = (hs & 0xffu) + ((hs >> 8) & 0xffu);
                    uint32_t c6 = __dp4a(ps + nib_pairs(wo), 0x01010101u, 0u);
                    const double2 pp = preA[kap >> 6];
                    if (__double2hiint(pp.y)) {                            // rare: a word of 7 / 6 bases lies below this order-5 bin
                        for (uint32_t s = 0; s < n_side; ++s) {
                            const uint32_t e = ss.side[s], sv = e >> 16, code = e & 0xffffu;
                            if (sv == 7u) { c7 += (code == (kap >> 2)); c6 += ((code >> 2) == (kap >> 4)); }
                            else c6 += (code == (kap >> 4));
                        }
                    }
                    double num = pp.x;
                    uint32_t den = (uint32_t)__double2loint(pp.y);
                    if (6 >= kmin) { den += c6 << 12; num = fma(q6, u32_to_double(c6 * c6), num); }
                    if (7 >= kmin) { den += c7 << 14; num = fma(q7, u32_to_double(c7 * c7), num); }
                    if (8 >= kmin) { den += c8 << 16; num = fma(q8, u32_to_double(c8 * c8), num); }
                    uint32_t cK = 1u;
                    if (c8 == 1u) { num += qsum; den += dsum; }
                    else {
                        uint32_t cx = c8;                                  // counts stay 1 once a prefix is unique
                        for (int x = 9; x <= K; ++x) {
                            if (cx >= 2u) {
                                const uint32_t tag = ext_tag(x, Wa >> (32 - 2 * x));
                                uint32_t s = ext_slot(tag);
                                cx = 0;
                                for (int probe = 0; probe < kMaxProbe; ++probe) {
                                    const uint32_t cur = hash[s];
                                    if ((cur >> 4) == tag) { cx = cur & 15u; break; }
                                    if (cur == 0u) break;                  // (cannot happen: a repeated prefix registered its extensions)
                                    s = (s + 1u) & (kHashSlots - 1u);
                                }
                            }
                            if (x >= kmin) { den += cx << (2 * x); num = fma(ss.q[x - 1], u32_to_double(cx * cx), num); }
                        }
                        cK = cx;
                    }
                    // a = I_w / c_K, om = 1 / c_K from ONE reciprocal, of den * c_K (exact product)
                    const double dden = u32_to_double(den), dc = u32_to_double(cK);
                    const double D = dden * dc;
                    double r;
                    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(D));
                    r = fma(r, fma(-D, r, 1.0), r);
                    r = fma(r, fma(-D, r, 1.0), r);
                    double a = num * r;
                    a = fma(fma(-D, a, num), r, a);
                    s_w += a;
                    s_g = fma(g.x, dden * r, s_g);                         // a NaN entry (reference: ZeroDivisionError) poisons the sum
                    s_t = fma(a, log2_series(a * dc) - g.y, s_t);
                }
                Wa = __funnelshift_l(Wb, Wa, 2); Wb = __funnelshift_l(Wc, Wb, 2); Wc = __funnelshift_l(Wd, Wc, 2); Wd <<= 2;
                bd <<= 1;
            }
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
        if (warp == 0) {                                                   // the row: divisions and logarithms one per lane
            double a = 0, bsum = 0, c = 0;
            for (int w = 0; w < NW; ++w) { a += ss.red[0][w]; bsum += ss.red[1][w]; c += ss.red[2][w]; }
            double nu = 0.0, de = 1.0;
            if (lane == 0) { nu = c; de = a; }
            else if (lane == 1) { nu = (double)n_gc; de = (double)n_up; }
            else if (lane == 2) { nu = (double)ss.c2[4]; de = (double)ss.c2[1]; }
            else if (lane == 3) { nu = (double)(ss.c2[12] + ss.c2[6]); de = (double)(ss.c2[3] + ss.c2[9]); }
            const double qv = nu / de;
            const double lgv = log2(lane == 0 ? bsum : a);
            const double q_gc = __shfl_sync(kFull, qv, 1), q_pi = __shfl_sync(kFull, qv, 2), q_si = __shfl_sync(kFull, qv, 3);
            const double lg_a = __shfl_sync(kFull, lgv, 1);
            if (lane == 0) {
                uint32_t st = 0;
                double kld = 0.0;
                if (!(a == 0.0)) {
                    bool zd = bsum != bsum;                                // NaN genome IVOM entry: ZeroDivisionError at F:437
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
                    if (pi != 0.0 && si != 0.0) cri = pi - si;             // F:491: 0.0 falsy, NaN truthy
                }
                row[2] = pi; row[3] = si; row[4] = cri;
                status[win] = st;
                if (redo_dst != status) redo_dst[win] = 0;
            }
        }
        __syncthreads();                                                   // (5)
    }
}

}  // namespace

frisk_internal::LaunchShape frisk_internal::ext_shape(const WinPlan& p) {
#define FRISK_EXT(PP) (p.allk ? (const void*)score_windows_nibble_ext_kernel<PP, true> : (const void*)score_windows_nibble_ext_kernel<PP, false>)
    const void* fn = p.variant == 8 ? FRISK_EXT(8) : (p.variant == 20 ? FRISK_EXT(20) : FRISK_EXT(32));
#undef FRISK_EXT
    return {fn, kNT, ExtLayout::TOTAL, true};
}

int frisk_internal::score_nibble_ext(const WinPlan& p, const uint32_t* codes, const uint32_t* inv, const uint32_t* low,
                                     const uint64_t* win_off, const uint32_t* win_len, uint64_t n_win, uint32_t max_len, const double* ig,
                                     int kmin, int K, int want_rip, double* rows, uint32_t* status, cudaStream_t st) {
    if (K < 9 || K > 12) return FRISK_E_UNSUPPORTED;
    return with_redo_marks(status, n_win, false, st, [&](uint32_t* redo) {
        const unsigned long long* off = reinterpret_cast<const unsigned long long*>(win_off);
        const double2* g = reinterpret_cast<const double2*>(ig);
        uint32_t n = (uint32_t)n_win;
        void* args[] = {&codes, &inv, &low, &off, &win_len, &n, &g, &kmin, &K, &want_rip, &rows, &status, &redo};
        int rc = launch_persistent(ext_shape(p), n_win, args, st);
        // the windows this kernel could not hold: exact re-run on the general kernel (few CTAs: the slab is 156 MB per CTA
        // at kmax 12, and a hand-over launch usually has nothing to do)
        return rc ? rc : general_score(codes, inv, low, win_off, win_len, n_win, max_len, ig, kmin, K, want_rip, rows, status, nullptr, st,
                                       redo, K <= 10 ? 8 : 2);
    });
}
