// frisk_b200: the dense-table window-score kernel: kmax 7 and 8 on windows longer than the shared-memory kernels hold
// (8,187..65,535 bases), and kmax <= 8 where it is forced (force_dense_kernel; kmax <= 3 under force_bucket_kernel).
//
// Replaces, per window, the reference's computeKmers(window) + IvomBuild x2 + KLD + calcGC + calcRIP
// (/root/reference/frisk/__init__.py F:1478-1494, F:280-367, F:369-472, F:120-137, F:474-495).
//
// The whole 4^K table of a window in shared memory as u16 counters (128 KiB at K = 8) with an occupancy bitmap, so one
// CTA of 1,024 threads per SM.  The distinct K-mers are listed from the bitmap in segments of the K-mer space; each
// segment's list must fit kListCap entries.
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "../../include/frisk_b200.h"
#include "frisk_internal.h"
#include "frisk_device.cuh"

namespace {
using frisk_internal::LaunchShape;
using frisk_internal::WinJob;
using frisk_internal::sm_count_cached;
#define CK(call) FRISK_CK(call)

constexpr int kThreads = 1024;          // one CTA per SM: the 4^8 u16 window table takes 128 KiB of smem
constexpr int kWarps = kThreads / 32;
constexpr uint32_t kListCap = 8192;     // compacted (kmer, count) entries per segment
constexpr int kMaxSeg = 8;

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

template <int K>
LaunchShape dense_shape_k() {
    return {(const void*)score_windows_kernel<K>, kThreads, ScoreLayout<K>::TOTAL, false};
}

// grid: one CTA per SM (or per window, when there are fewer windows than SMs)
template <int K>
int score_dense_k(const WinJob& j) {
    using L = ScoreLayout<K>;
    constexpr uint32_t NB = pow4(K);
    const LaunchShape s = dense_shape_k<K>();
    // a segment = a contiguous 1/nseg of the k-mer space (and of the threads owning its bitmap words);
    // its distinct k-mers (<= bins in it, <= window length) must fit the list
    int nseg = 1;
    while ((NB / (uint32_t)nseg < j.max_len ? NB / (uint32_t)nseg : j.max_len) > kListCap) nseg *= 2;
    if (nseg > kMaxSeg || (uint32_t)nseg > (L::BM_WORDS >= 2u ? L::BM_WORDS / 2u : 1u)) return FRISK_E_UNSUPPORTED;
    CK(cudaFuncSetAttribute(s.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s.smem));
    int grid = sm_count_cached();
    if (grid <= 0) return FRISK_E_NO_DEVICE;
    if ((uint64_t)grid > j.n_win) grid = (int)j.n_win;
    score_windows_kernel<K><<<grid, s.threads, s.smem, j.st>>>(
        j.codes, j.inv, j.low, reinterpret_cast<const unsigned long long*>(j.win_off), j.win_len, (uint32_t)j.n_win,
        reinterpret_cast<const double2*>(j.ig), j.kmin, j.rip, nseg, j.rows, j.status, j.dump);
    CK(cudaGetLastError());
    return FRISK_OK;
}

}  // namespace

frisk_internal::LaunchShape frisk_internal::dense_shape(int K) {
    switch (K) {
        case 1: return dense_shape_k<1>();
        case 2: return dense_shape_k<2>();
        case 3: return dense_shape_k<3>();
        case 4: return dense_shape_k<4>();
        case 5: return dense_shape_k<5>();
        case 6: return dense_shape_k<6>();
        case 7: return dense_shape_k<7>();
        default: return dense_shape_k<8>();
    }
}

int frisk_internal::score_dense(const WinPlan&, const WinJob& j) {
    DISPATCH_K(j.K, score_dense_k<K>(j));
}
