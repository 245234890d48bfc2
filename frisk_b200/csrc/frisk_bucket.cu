// frisk_b200: the bucketed window-score kernel for kmax 4..8 (windows <= 8,186 bases): the round-1 default, now the
// kernel that re-does the windows the nibble and direct kernels hand over, and kmax 4..8 when forced.
//
// Replaces, per window, the reference's computeKmers(window) + IvomBuild x2 + KLD + calcGC + calcRIP
// (/root/reference/frisk/__init__.py F:1478-1494, F:280-367, F:369-472, F:120-137, F:474-495).
//
// The K-mers of a window are counting-sorted by their (K-2)-prefix into a list of the distinct K-mers, which is then
// scored (see the comment at score_windows_bucket_kernel).
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "../../include/frisk_b200.h"
#include "frisk_internal.h"
#include "frisk_device.cuh"

namespace {
using frisk_internal::LaunchShape;
using frisk_internal::WinPlan;

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

template <int K>
LaunchShape bucket_shape_k(const WinPlan& p, uint32_t max_len) {
    return {p.variant == 2   ? FRISK_WIN_INSTANCE(p, score_windows_bucket_kernel, K, 2)
            : p.variant == 5 ? FRISK_WIN_INSTANCE(p, score_windows_bucket_kernel, K, 5)
                             : FRISK_WIN_INSTANCE(p, score_windows_bucket_kernel, K, 8),
            kT3, Score3Layout<K>::total((max_len + 15u) & ~15u), true};
}

// one launch; it takes the windows of [len_min, len_max] only, and with redo_src only those marked kRowRedo there
int launch_bucket(const WinPlan& p, const uint32_t* codes, const uint32_t* inv, const uint32_t* low, const uint64_t* win_off,
                  const uint32_t* win_len, uint64_t n_win, uint32_t max_len, const double* ig, int kmin, int K, int want_rip,
                  double* rows, uint32_t* status, uint16_t* dump, cudaStream_t st, uint32_t len_min, uint32_t len_max,
                  const uint32_t* redo_src) {
    const LaunchShape s = frisk_internal::bucket_shape(p, K, max_len);
    const unsigned long long* off = reinterpret_cast<const unsigned long long*>(win_off);
    const double2* g = reinterpret_cast<const double2*>(ig);
    uint32_t n = (uint32_t)n_win, cap = (max_len + 15u) & ~15u;
    void* args[] = {&codes, &inv, &low, &off, &win_len, &n, &g, &kmin, &want_rip, &cap, &len_min, &len_max, &rows, &status, &dump, &redo_src};
    return frisk_internal::launch_persistent(s, n_win, args, st);
}

}  // namespace

// 256 threads, buffer sized by the longest window; four CTAs of 57 KB need the whole 228 KB carve-out, which the driver's
// per-launch heuristic does not always give (0.73 vs 0.83 ms)
frisk_internal::LaunchShape frisk_internal::bucket_shape(const WinPlan& p, int K, uint32_t max_len) {
    switch (K) {
        case 4: return bucket_shape_k<4>(p, max_len);
        case 5: return bucket_shape_k<5>(p, max_len);
        case 6: return bucket_shape_k<6>(p, max_len);
        case 7: return bucket_shape_k<7>(p, max_len);
        default: return bucket_shape_k<8>(p, max_len);
    }
}

// Windows longer than 5 rounds need a bigger buffer, which costs a CTA per SM.  With --scaffoldsAll nearly all windows are
// still the standard length and only whole short scaffolds (up to 1.25 w) are longer: two launches, each taking the
// windows of its length class, keep the standard ones at four CTAs per SM.  A hand-over launch (redo_src) is one launch.
int frisk_internal::score_bucket(const WinPlan& p, const uint32_t* codes, const uint32_t* inv, const uint32_t* low,
                                 const uint64_t* win_off, const uint32_t* win_len, uint64_t n_win, uint32_t max_len, const double* ig,
                                 int kmin, int K, int want_rip, double* rows, uint32_t* status, uint16_t* dump, cudaStream_t st,
                                 const uint32_t* redo_src) {
    if (K < 4 || K > 8) return FRISK_E_UNSUPPORTED;
    constexpr uint32_t kStd = 5104u;                   // largest buffer that still fits four CTAs
    if (!redo_src && p.variant == 8 && n_win >= 4096) {
        const WinPlan std5{p.kind, 5, p.dump, p.allk};
        int rc = launch_bucket(std5, codes, inv, low, win_off, win_len, n_win, kStd, ig, kmin, K, want_rip, rows, status, dump, st, 0u,
                               kStd, nullptr);
        if (rc) return rc;
        return launch_bucket(p, codes, inv, low, win_off, win_len, n_win, max_len, ig, kmin, K, want_rip, rows, status, dump, st,
                             kStd + 1u, 0xffffffffu, nullptr);
    }
    return launch_bucket(p, codes, inv, low, win_off, win_len, n_win, max_len, ig, kmin, K, want_rip, rows, status, dump, st, 0u,
                         0xffffffffu, redo_src);
}
