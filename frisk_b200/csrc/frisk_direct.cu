// frisk_b200: the "direct" window-score kernel -- the default path for kmax 7 and 8 (windows <= 8,186 bases).
//
// Replaces, per window, the reference's computeKmers(window) + IvomBuild x2 + KLD + calcGC + calcRIP
// (/root/reference/frisk/__init__.py F:1478-1494, F:280-367, F:369-472, F:120-137, F:474-495).
//
// No sorting and no list of distinct K-mers.  The whole order-K code space is ONE BYTE per K-mer in shared
// memory (4^8 = 64 KiB), so that
//   * the count of a K-mer is a byte, the count of its (K-1)-prefix the sum of the 4 bytes of its aligned word,
//     the count of its (K-2)-prefix the sum of its aligned 16 bytes: one 128-bit shared-memory load gives the
//     three highest orders;
//   * order A = K-3 is counted by a second atomic (u16 bins), orders below it follow by marginalisation, and the
//     orders <= 4 are folded into one {numerator, denominator} pair per order-4 prefix (`pre`);
//   * every POSITION scores its own K-mer with weight 1/c_K (c_K = its count in the window), so the sum over
//     positions equals the sum over distinct K-mers (F:448-472 iterate the distinct keys) without ever
//     enumerating them; a thread's positions are fixed and so is the reduction tree -> bit-reproducible rows.
// Two atomics and one epilogue per position; 3 CTAs per SM (73 KB each).
//
// What a byte cannot hold is handed to the bucketed kernel (frisk_bucket.cu), exactly: a window in which some
// K-mer occurs 256+ times (the thread whose increment wraps the byte sees 255 in the word it got back), or
// with more than kSideCap words cut short by an N / the window end at K-1 or K-2 bases, is marked kRowRedo in
// `status` and re-done by the launch that follows on the same stream.  Short words of K-1 / K-2 bases (every
// window has two at its end) are not in the byte table: they go to a small side list, and bit 15 of their
// order-A bin sends the (few) K-mers below that bin through the list.
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "../../include/frisk_b200.h"
#include "frisk_internal.h"
#include "frisk_device.cuh"

namespace {
using frisk_internal::kRowRedo;

constexpr uint32_t kSideCap = 64;

template <int NT>
struct DirectSmem {
    double q[8];
    double red[3][NT / 32];
    int cnt[2][4];                    // [window parity][n_non, n_gc, redo, n_side]
    uint32_t c2[16];                  // final dinucleotide counts (RIP, and the way up to order 1)
    uint32_t side[kSideCap];          // v << 16 | code of a word valid for v = K-1 or K-2 bases only
};

template <int K, int NT>
struct DirectLayout {
    static_assert(K == 7 || K == 8, "direct kernel: K = 7 or 8");
    static constexpr int A = K - 3;                                      // order of the second atomic
    static constexpr int LP = 4;                                         // orders <= LP live in `pre`
    static constexpr uint32_t NPRE = pow4(LP);
    static constexpr uint32_t TOP_BYTES = pow4(K);                       // u8 per K-mer
    static constexpr uint32_t LOW_BYTES = (lvl_off(A + 1) * 2u + 15u) & ~15u;   // orders 1..A, u16
    static constexpr uint32_t ZERO_BYTES = TOP_BYTES + LOW_BYTES;
    static constexpr uint32_t OFF_LOW = TOP_BYTES;
    static constexpr uint32_t OFF_PRE = ZERO_BYTES;
    static constexpr uint32_t OFF_SS = OFF_PRE + NPRE * 16u;
    static constexpr uint32_t TOTAL = OFF_SS + (uint32_t)sizeof(DirectSmem<NT>);
};

__device__ __forceinline__ uint32_t bytes_sum(uint32_t w, uint32_t acc) { return __dp4a(w, 0x01010101u, acc); }

// CTAs per SM: K = 8: 73 KB of shared memory each; K = 7: registers decide
template <int K, int NT, int ROUNDS, bool DUMP, bool ALLK>
__global__ void __launch_bounds__(NT, K == 7 ? 4 : 3)
score_windows_direct_kernel(const uint32_t* __restrict__ codes, const uint32_t* __restrict__ inv, const uint32_t* __restrict__ low,
                            const unsigned long long* __restrict__ win_off, const uint32_t* __restrict__ win_len, uint32_t n_win,
                            const double2* __restrict__ ig, int kmin_arg, int want_rip,
                            double* __restrict__ rows, uint32_t* __restrict__ status, uint16_t* __restrict__ dump,
                            uint32_t* redo_dst) {
    using L = DirectLayout<K, NT>;
    constexpr int A = L::A, LP = L::LP, NW = NT / 32;
    const int kmin = ALLK ? 1 : kmin_arg;                                // ALLK: the default --minWordSize 1
    extern __shared__ __align__(16) unsigned char smem[];
    uint32_t* top32 = reinterpret_cast<uint32_t*>(smem);
    uint16_t* tab16 = reinterpret_cast<uint16_t*>(smem + L::OFF_LOW);    // orders 1..A at lvl_off(x)
    uint32_t* tab32 = reinterpret_cast<uint32_t*>(smem + L::OFF_LOW);
    double2* pre = reinterpret_cast<double2*>(smem + L::OFF_PRE);       // .x = num, .y = {flag, den} as two u32
    DirectSmem<NT>& ss = *reinterpret_cast<DirectSmem<NT>*>(smem + L::OFF_SS);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (uint32_t i = tid; i < L::ZERO_BYTES / 16u; i += NT) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
    if (tid < 8) ss.cnt[tid >> 2][tid & 3] = 0;
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
        const uint32_t g0 = o_lo >> 2;
        const uint32_t ngroups = ((o_lo + len + 3u) >> 2) - g0;          // <= NT * ROUNDS (checked by the launcher)

        // ---- P1: one pass over the positions: composition, the byte table, order A --------------------
        uint32_t kk[2 * ROUNDS];                                         // two K-mer codes per register
        uint32_t vm = 0;                                                 // bit 4r+j: position holds a full K-word
        {
            int non = 0, gc = 0, redo = 0;
            GroupWords gw = load_group(cw, mw, lw, (g0 + (tid < (int)ngroups ? tid : 0)) << 2);
#pragma unroll
            for (int r = 0; r < ROUNDS; ++r) {
                const uint32_t gi = tid + r * NT;
                const uint32_t gn = gi + NT;
                GroupWords nx = gw;
                if (r + 1 < ROUNDS) nx = load_group(cw, mw, lw, (g0 + (gn < ngroups ? gn : 0u)) << 2);
                kk[2 * r] = 0; kk[2 * r + 1] = 0;
                if (gi < ngroups) {
                    visit_group(gw, (g0 + gi) << 2, o_lo, len, [&](uint32_t j, uint32_t p, uint32_t c32, uint32_t m, uint32_t lowbit) {
                        const uint32_t unres = (m >> 31) | lowbit;               // not an upper-case ATGC (F:106-118)
                        non += unres;
                        gc += (1 - unres) & (c32 >> 31);                         // G = 2, C = 3: bit 1 of the first base
                        const uint32_t a = c32 >> (32 - 2 * A);
                        const uint32_t ga = lvl_off(A) + a;
                        if ((m >> (32 - K)) == 0u && p + K <= len) {             // the common case: a full K-word
                            const uint32_t kap = c32 >> (32 - 2 * K);
                            const uint32_t sh = (kap & 3u) * 8u;
                            const uint32_t old = atomicAdd(&top32[kap >> 2], 1u << sh);
                            atomicAdd(&tab32[ga >> 1], 1u << ((ga & 1u) * 16u));
                            redo |= (((old >> sh) & 255u) == 255u);
                            kk[2 * r + (j >> 1)] |= kap << (16u * (j & 1u));
                            vm |= 1u << (4 * r + j);
                        } else {                                                 // window end / N boundary
                            const int v = min(__clz(m), (int)(len - p));
                            if (v >= A) {
                                atomicAdd(&tab32[ga >> 1], 1u << ((ga & 1u) * 16u));
                                if (v > A) {                                     // K-1 or K-2 bases: side list + flag on its bin
                                    atomicOr(&tab32[ga >> 1], 0x8000u << ((ga & 1u) * 16u));
                                    const uint32_t slot = (uint32_t)atomicAdd(&ss.cnt[par][3], 1);
                                    if (slot < kSideCap) ss.side[slot] = ((uint32_t)v << 16) | (c32 >> (32 - 2 * v));
                                }
                            } else if (v > 0) {                                  // order v < A only
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
            redo = __any_sync(kFull, redo);
            if (lane == 0) {
                atomicAdd(&ss.cnt[par][0], non); atomicAdd(&ss.cnt[par][1], gc);
                if (redo) ss.cnt[par][2] = 1;
            }
        }
        __syncthreads();                                                   // (1)
        const int n_non = ss.cnt[par][0], n_gc = ss.cnt[par][1], n_up = (int)len - n_non;
        const uint32_t n_side = (uint32_t)ss.cnt[par][3];
        const bool redo_win = ss.cnt[par][2] != 0 || n_side > kSideCap;
        if (tid < 4) ss.cnt[par ^ 1][tid] = 0;                              // next window's counters (idle until its P1)
        const bool excluded = (double)n_non >= 0.3 * (double)len;          // F:238 / F:213
        uint16_t* dmp = DUMP ? dump + (size_t)win * lvl_off(K + 1) : nullptr;
        if (excluded || redo_win) {
            for (uint32_t i = tid; i < L::ZERO_BYTES / 16u; i += NT) reinterpret_cast<uint4*>(smem)[i] = make_uint4(0, 0, 0, 0);
            if (tid == 0) {
                if (excluded) {
                    status[win] = FRISK_ROW_EXCLUDED;
                    for (int c = 0; c < 5; ++c) rows[(size_t)win * 5 + c] = CUDART_NAN;
                    if (redo_dst != status) redo_dst[win] = 0;
                } else {
                    redo_dst[win] = kRowRedo;                              // the bucketed kernel takes this window
                }
            }
            if (DUMP && excluded) for (uint32_t i = tid; i < lvl_off(K + 1); i += NT) dmp[i] = 0;
            __syncthreads();
            continue;
        }
        if (tid < K) {
            const int x = tid + 1;
            const long long d = ((long long)n_up - (long long)(x - 1)) * 2;
            ss.q[tid] = (double)pow4(x) / (double)d;
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
        uint32_t n_at = 0, n_ta = 0, n_sub = 0, n_prod = 0;
        if (tid < 256) {
            const uint32_t* q2 = ss.c2 + (tid >> 6) * 4;
            const uint32_t c1 = q2[0] + q2[1] + q2[2] + q2[3] + tab16[lvl_off(1) + (tid >> 6)];
            const uint32_t cs[4] = {c1, c2, c3, c4};
            double num = 0.0;
            uint32_t den = 0;
#pragma unroll
            for (int x = 1; x <= LP; ++x) {
                if (x >= kmin) {
                    const uint32_t c = cs[x - 1];
                    den += c << (2 * x);
                    num = fma(ss.q[x - 1], u32_to_double(c * c), num);
                }
            }
            pre[tid] = make_double2(num, __hiloint2double((int)flag4, (int)den));
            if (DUMP) {
                dmp[lvl_off(4) + tid] = (uint16_t)c4;
                if ((tid & 3) == 0) dmp[lvl_off(3) + (tid >> 2)] = (uint16_t)c3;
                if ((tid & 15) == 0) dmp[lvl_off(2) + (tid >> 4)] = (uint16_t)c2;
                if ((tid & 63) == 0) dmp[lvl_off(1) + (tid >> 6)] = (uint16_t)c1;
            }
        }
        if (tid == 0 && want_rip) {                                        // K >= 7 so order 2 always exists
            n_at = ss.c2[1]; n_ta = ss.c2[4];
            n_sub = ss.c2[3] + ss.c2[9];
            n_prod = ss.c2[12] + ss.c2[6];
        }
        __syncthreads();                                                   // (3)
        if (DUMP) {                                                        // tests only: the window's tables, all orders
            if constexpr (A == 5)
                for (uint32_t i = tid; i < pow4(5); i += NT) dmp[lvl_off(5) + i] = tab16[lvl_off(5) + i] & 0x7fffu;
            for (uint32_t i = tid; i < pow4(K); i += NT) dmp[lvl_off(K) + i] = smem[i];
            for (uint32_t i = tid; i < pow4(K - 1); i += NT) dmp[lvl_off(K - 1) + i] = (uint16_t)bytes_sum(top32[i], 0u);
            for (uint32_t i = tid; i < pow4(K - 2); i += NT) {
                const uint4 v = reinterpret_cast<const uint4*>(smem)[i];
                dmp[lvl_off(K - 2) + i] = (uint16_t)bytes_sum(v.x, bytes_sum(v.y, bytes_sum(v.z, bytes_sum(v.w, 0u))));
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

        // ---- P3: every position scores its own K-mer with weight 1 / (its count) --------------------
        double s_w = 0.0, s_g = 0.0, s_t = 0.0;
        const double qA = ss.q[A - 1], qK2 = ss.q[K - 3], qK1 = ss.q[K - 2], qK = ss.q[K - 1];
        auto score_one = [&](uint32_t kap, const double2 g) {
            const uint4 v = *reinterpret_cast<const uint4*>(smem + (kap & ~15u));
            const uint32_t jw = (kap >> 2) & 3u;
            const uint32_t w = (jw & 2u) ? ((jw & 1u) ? v.w : v.z) : ((jw & 1u) ? v.y : v.x);
            const uint32_t cK = (w >> ((kap & 3u) * 8u)) & 255u;
            uint32_t cK1 = bytes_sum(w, 0u);
            uint32_t cK2 = bytes_sum(v.x, bytes_sum(v.y, bytes_sum(v.z, bytes_sum(v.w, 0u))));
            const double2 pp = pre[kap >> (2 * (K - LP))];
            double num = pp.x;
            uint32_t den = (uint32_t)__double2loint(pp.y);
            uint32_t cA = 0, flag;
            if constexpr (A > LP) {
                const uint32_t raw = tab16[lvl_off(A) + (kap >> (2 * (K - A)))];
                cA = raw & 0x7fffu; flag = raw >> 15;
            } else {
                flag = (uint32_t)__double2hiint(pp.y);
            }
            if (flag) {                                    // rare: a short word of K-1 / K-2 bases lies below this bin
                for (uint32_t i = 0; i < n_side; ++i) {
                    const uint32_t e = ss.side[i], sv = e >> 16, code = e & 0xffffu;
                    if (sv == (uint32_t)(K - 1)) { cK1 += (code == (kap >> 2)); cK2 += ((code >> 2) == (kap >> 4)); }
                    else cK2 += (code == (kap >> 4));
                }
            }
            if constexpr (A > LP) {
                if (A >= kmin) { den += cA << (2 * A); num = fma(qA, u32_to_double(cA * cA), num); }
            }
            if (K - 2 >= kmin) { den += cK2 << (2 * (K - 2)); num = fma(qK2, u32_to_double(cK2 * cK2), num); }
            if (K - 1 >= kmin) { den += cK1 << (2 * (K - 1)); num = fma(qK1, u32_to_double(cK1 * cK1), num); }
            den += cK << (2 * K);
            num = fma(qK, u32_to_double(cK * cK), num);
            // a = I_w / c_K, om = 1 / c_K from ONE reciprocal, of den * c_K (exact product, < 2^41)
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
#pragma unroll 1
        for (int r = 0; r < ROUNDS; ++r) {
            uint32_t kp[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) kp[j] = (kk[j >> 1] >> (16 * (j & 1))) & 0xffffu;
            // the gather is issued where it is used: four at the top of the round cost 12 % (0.771 -> 0.886 ms), one
            // K-mer ahead 4 % -- they queue in front of the other warps' shared-memory traffic (DESIGN.md section 5)
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (vm & (1u << j)) score_one(kp[j], __ldg(ig + kp[j]));
            vm >>= 4;
#pragma unroll
            for (int i = 0; i + 2 < 2 * ROUNDS; ++i) kk[i] = kk[i + 2];     // rotate: the loop body stays one round long
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
        if (tid == 0) {
            double a = 0, bsum = 0, c = 0;
            for (int w = 0; w < NW; ++w) { a += ss.red[0][w]; bsum += ss.red[1][w]; c += ss.red[2][w]; }
            uint32_t st = 0;
            double kld = 0.0;                              // the reference returns 0 for a window without kmax-mers
            if (!(a == 0.0)) {
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
            if (redo_dst != status) redo_dst[win] = 0;
        }
        __syncthreads();                                                   // (5) tables zeroed, ss.red consumed
    }
}

template <int K>
const void* direct_fn(const frisk_internal::WinPlan& p) {
    if (p.variant == 2) return FRISK_WIN_INSTANCE(p, score_windows_direct_kernel, K, 256, 2);
    if (p.variant == 5) return FRISK_WIN_INSTANCE(p, score_windows_direct_kernel, K, 256, 5);
    return FRISK_WIN_INSTANCE(p, score_windows_direct_kernel, K, 256, 8);
}

}  // namespace

// 256 threads; at K = 8 three CTAs of 73 KB need the whole 228 KB carve-out
frisk_internal::LaunchShape frisk_internal::direct_shape(const WinPlan& p, int K) {
    if (K == 8) return {direct_fn<8>(p), 256, DirectLayout<8, 256>::TOTAL, true};
    return {direct_fn<7>(p), 256, DirectLayout<7, 256>::TOTAL, true};
}

int frisk_internal::score_direct(const WinPlan& p, const WinJob& j) {
    if (j.K != 7 && j.K != 8) return FRISK_E_UNSUPPORTED;
    return with_redo_marks(j.status, j.n_win, false, j.st, [&](uint32_t* redo) {
        WinJob a = j;                                  // the kernel arguments are read from their addresses
        const unsigned long long* off = reinterpret_cast<const unsigned long long*>(a.win_off);
        const double2* g = reinterpret_cast<const double2*>(a.ig);
        uint32_t n = (uint32_t)a.n_win;
        void* args[] = {&a.codes, &a.inv, &a.low, &off, &a.win_len, &n, &g, &a.kmin, &a.rip, &a.rows, &a.status, &a.dump, &redo};
        int rc = launch_persistent(direct_shape(p, a.K), a.n_win, args, a.st);
        // windows the byte table could not hold (marked kRowRedo): exact re-run on the bucketed kernel
        return rc ? rc : score_bucket_redo(j, redo);
    });
}
