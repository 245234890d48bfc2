// frisk_b200: the small-K window-score kernel for kmax 1..6 (windows <= 65,535 bases).
//
// Replaces, per window, the reference's computeKmers(window) + IvomBuild x2 + KLD + calcGC + calcRIP
// (/root/reference/frisk/__init__.py F:1478-1494, F:280-367, F:369-472, F:120-137, F:474-495).
//
// No sorting: the whole order-K table of a window is at most 4,096 u16 bins in shared memory (see the comment at
// score_windows_small_kernel).  It also re-does, for kmax 1..3, the windows the k sweep hands over.
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "../../include/frisk_b200.h"
#include "frisk_internal.h"
#include "frisk_device.cuh"

namespace {
using frisk_internal::LaunchShape;
using frisk_internal::WinPlan;

constexpr int kT3 = 256;
constexpr int kW3 = kT3 / 32;

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

template <int K>
LaunchShape small_shape_k(const WinPlan& p) {
    return {p.dump ? (const void*)score_windows_small_kernel<K, true> : (const void*)score_windows_small_kernel<K, false>, kT3,
            SmallLayout<K>::TOTAL, false};
}

}  // namespace

// 256 threads; the L1 / shared split is left to the driver
frisk_internal::LaunchShape frisk_internal::small_shape(const WinPlan& p, int K) {
    switch (K) {
        case 1: return small_shape_k<1>(p);
        case 2: return small_shape_k<2>(p);
        case 3: return small_shape_k<3>(p);
        case 4: return small_shape_k<4>(p);
        case 5: return small_shape_k<5>(p);
        default: return small_shape_k<6>(p);
    }
}

int frisk_internal::score_small(const WinPlan& p, const uint32_t* codes, const uint32_t* inv, const uint32_t* low,
                                const uint64_t* win_off, const uint32_t* win_len, uint64_t n_win, const double* ig, int kmin, int K,
                                int want_rip, double* rows, uint32_t* status, uint16_t* dump, cudaStream_t st,
                                const uint32_t* redo_src) {
    if (K < 1 || K > 6) return FRISK_E_UNSUPPORTED;
    const unsigned long long* off = reinterpret_cast<const unsigned long long*>(win_off);
    const double2* g = reinterpret_cast<const double2*>(ig);
    uint32_t n = (uint32_t)n_win;
    void* args[] = {&codes, &inv, &low, &off, &win_len, &n, &g, &kmin, &want_rip, &rows, &status, &dump, &redo_src};
    return launch_persistent(small_shape(p, K), n_win, args, st);
}
