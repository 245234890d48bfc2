// Device helpers shared by the translation units that hold the table and window kernels.
#ifndef FRISK_DEVICE_CUH
#define FRISK_DEVICE_CUH

#include <cuda_runtime.h>
#include <stdint.h>

namespace {

constexpr uint32_t kFull = 0xffffffffu;

__host__ __device__ constexpr uint32_t pow4(int k) { return 1u << (2 * k); }
// offset (in entries) of order x inside a concatenation of orders 1..: sum_{y<x} 4^y
__host__ __device__ constexpr uint32_t lvl_off(int x) { return (pow4(x) - 4u) / 3u; }

// gather bit1 of each of the 16 2-bit codes of a word into 16 contiguous bits (order kept)
__device__ __forceinline__ uint32_t high_bits16(uint32_t w) {
    uint32_t x = (w >> 1) & 0x55555555u;
    x = (x | (x >> 1)) & 0x33333333u;
    x = (x | (x >> 2)) & 0x0f0f0f0fu;
    x = (x | (x >> 4)) & 0x00ff00ffu;
    x = (x | (x >> 8)) & 0x0000ffffu;
    return x;
}

// bytes of the result = sums of the two nibbles of each byte of w (<= 30)
__device__ __forceinline__ uint32_t nib_pairs(uint32_t w) { return (w & 0x0f0f0f0fu) + ((w >> 4) & 0x0f0f0f0fu); }

__device__ __forceinline__ double u32_to_double(uint32_t v) {
    // exact: 2^52 + v has v in the low mantissa bits
    return __hiloint2double(0x43300000, (int)v) - 4503599627370496.0;
}

// log2 of a positive normal double: x = 2^e * m, m in [1,2); m = c (1 + r) with c the midpoint of
// one of 128 mantissa intervals, |r| <= 2^-8; log2(1+r) by a degree-6 Taylor polynomial
// (truncation < 3e-18).  tab[i] = {1/c_i rounded, -log2 of that rounded value}.  ~20 instructions
// against ~75 for the library log2 (which also handles zero, denormals, inf, NaN).
__device__ __forceinline__ double log2_pos(double x, const double2* __restrict__ tab) {
    const int hi = __double2hiint(x);
    const double2 t = tab[(hi >> 13) & 127];
    const double m = __hiloint2double((hi & 0x000fffff) | 0x3ff00000, __double2loint(x));
    const double r = fma(m, t.x, -1.0);
    double p = fma(r, -0.24044917348149390, 0.28853900817779268);
    p = fma(r, p, -0.36067376022224085);
    p = fma(r, p, 0.48089834696298783);
    p = fma(r, p, -0.72134752044448170);
    p = fma(r, p, 1.4426950408889634);
    return fma(r, p, (double)((hi >> 20) - 1023) + t.y);
}

// log2 of a positive normal double without a table (the table lookup of log2_pos is a random 16-byte shared-memory
// read: ~10 wavefronts per warp; the kernels that use it are bound by the LSU data pipe, not by issue slots).
// x = 2^e * m with m in [sqrt(1/2), sqrt(2)); t = (m - 1) / (m + 1), |t| <= 0.1716;
// log2(m) = (2 / ln 2) * atanh(t) = t * sum_k c_k t^(2k), k = 0..7 (first dropped term < 1.7e-14 absolute).
// coefficients (2 / ln 2) / (2k + 1), k = 7 .. 0, in constant memory: a DFMA takes them straight from the constant bank
// (as immediates each costs two moves into uniform registers per use)
__constant__ double kLog2Series[8] = {0.19235933878519512, 0.22195308321368667, 0.2623081892525388, 0.3205988979753252,
                                      0.4121985831111324,  0.5770780163555853,  0.9617966939259756, 2.8853900817779268};

__device__ __forceinline__ double log2_series(double x) {
    int hi = __double2hiint(x);
    const int big = ((hi & 0x000fffff) >= 0x6a09f) ? 1 : 0;           // mantissa above sqrt(2): halve it, e + 1
    const int e = (hi >> 20) - 1023 + big;
    hi = (hi & 0x000fffff) | ((0x3ff - big) << 20);
    const double m = __hiloint2double(hi, __double2loint(x));
    const double n = m - 1.0, d = m + 1.0;
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
    r = fma(r, fma(-d, r, 1.0), r);
    r = fma(r, fma(-d, r, 1.0), r);
    double t = n * r;
    t = fma(fma(-d, t, n), r, t);
    const double s = t * t;
    double p = fma(s, kLog2Series[0], kLog2Series[1]);                // (2/ln2)/15, (2/ln2)/13
    p = fma(s, p, kLog2Series[2]);                                   // /11
    p = fma(s, p, kLog2Series[3]);                                   // /9
    p = fma(s, p, kLog2Series[4]);                                   // /7
    p = fma(s, p, kLog2Series[5]);                                   // /5
    p = fma(s, p, kLog2Series[6]);                                   // /3
    p = fma(s, p, kLog2Series[7]);                                   // 2/ln2
    return fma(t, p, (double)e);
}

// n / d for a positive normal d: hardware reciprocal seed + two Newton steps + one residual step
__device__ __forceinline__ double div_pos(double n, double d) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(d));
    r = fma(r, fma(-d, r, 1.0), r);
    r = fma(r, fma(-d, r, 1.0), r);
    const double q = n * r;
    return fma(fma(-d, q, n), r, q);
}

// The 32-byte entry at p (32-byte aligned) as two double2, with ONE 256-bit load cached in L2 only (as __ldcg): on sm_100
// this is a single LDG.E.ENL2.256, so a fully divergent gather of 32-byte entries costs a warp no more wavefronts than one
// of 16-byte entries.
__device__ __forceinline__ void ldcg_pair(const double2* p, double2& a, double2& b) {
    asm volatile("ld.global.cg.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(a.x), "=d"(a.y), "=d"(b.x), "=d"(b.y) : "l"(p));
}

// One round of the position walk: the four absolute-aligned bases of group `gi` (see below), with
// the words they need loaded once.  f(j, p, c32, m, low_bit) for the positions inside the window:
// j = 0..3, p = position in the window, c32 = the 16 bases from p (2 bits each, first base on top),
// m = unresolved mask of the 32 bases from p (bit 31 = p), low_bit = 1 when base p is lower case.
struct GroupWords { uint32_t chi, clo, mhi, mlo, lhi; };

__device__ __forceinline__ GroupWords load_group(const uint32_t* __restrict__ cw, const uint32_t* __restrict__ mw,
                                                 const uint32_t* __restrict__ lw, uint32_t a0) {
    GroupWords g;
    g.chi = __ldg(cw + (a0 >> 4)); g.clo = __ldg(cw + (a0 >> 4) + 1);
    g.mhi = __ldg(mw + (a0 >> 5)); g.mlo = __ldg(mw + (a0 >> 5) + 1);
    g.lhi = lw ? __ldg(lw + (a0 >> 5)) : 0u;
    return g;
}

template <typename F>
__device__ __forceinline__ void visit_group(const GroupWords& g, uint32_t a0, uint32_t o_lo, uint32_t len, F f) {
    const uint32_t cs = (a0 & 15u) * 2u, ms = a0 & 31u;               // cs <= 24, ms <= 28
#pragma unroll
    for (uint32_t j = 0; j < 4; ++j) {
        const uint32_t p = a0 + j - o_lo;                              // wraps for bases before the window
        if (p < len)
            f(j, p, __funnelshift_l(g.clo, g.chi, cs + 2u * j), __funnelshift_l(g.mlo, g.mhi, ms + j), (g.lhi << (ms + j)) >> 31);
    }
}

}  // namespace

#endif
