// frisk_b200 device-side FASTA ingest: FASTA text in, packed 2-bit planes out, on the GPU.
//
// Replaces the reference's iterFasta (F:139-164: line.strip(), blank lines skipped, '>' lines start
// a record, everything else is sequence) and countN (F:106-118) -- which the reference runs three
// times per file (F:170, F:203, F:297) in pure Python -- and this library's own host packer
// (frisk_b200_fasta_scan + frisk_b200_pack), whose outputs it reproduces bit for bit.  The host
// only copies the raw text to the device and reads back one small record table.
//
// The text is cut into tiles of 4096 bytes (256 threads x 16 bytes).  What a byte means depends on the line it is in (header
// or sequence), on the record it belongs to and on where that record starts in the packed planes, i.e. on everything before
// it.  Two passes over the text with one scan over per-tile summaries between them:
//   fasta_summary_kernel   per tile: header lines, state of the last line start, bases before the first line start / before
//                          the first header / after the last header, packed space of the records inside the tile
//   fasta_tilescan_kernel  over tiles (one CTA, batches of 4096 tiles in registers): records before every tile, the line state
//                          it starts in, bases and packed offset of the record open there -- frisk_b200_pack_layout's layout
//                          computed on the device -- and which plane words are final (what the caller may count already)
//   fasta_pack_kernel      per tile: planes (a word-wide path for plain ACGT lines, byte by byte for anything else), record
//                          table (header position, length, offset: written once, by the thread that sees the next header),
//                          padding flags, countN statistics
// The text travels in chunks on a second stream; the three kernels of a chunk run while the next chunk is on the bus, with
// the state between chunks in device memory.  Record table and planes are sized by a guess so that the host synchronises
// once; a text that does not fit the guesses, or a line decision that needs a byte of a later chunk, is redone in one piece
// with exact sizes (open_any).  The planes belong to the handle.
// A BGZF source (frisk_b200_fasta_open_bgzf, frisk_b200_run_fasta_bgzf) shares all of it: the compressed bytes go up on the
// upload lane, frisk_bgzf.cu inflates them into the text buffer, and the passes wait on that instead of on the text's copy.
// A gzip source (frisk_b200_fasta_open_gzip, frisk_b200_run_fasta_gzip) is inflated first (frisk_gzip.cu synchronises: its
// text length is only known at the end) and the open takes over the text buffer it filled, as the BGZF exact re-open does.
// A .2bit file (frisk_b200_fasta_open_2bit, frisk_b200_run_2bit) is not text: frisk_twobit.cu decodes it into planes and a
// record table of its own, and fasta_adopt makes the handle and does what the passes above do behind the last chunk.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <mutex>
#include <new>
#include <vector>

#include "../../include/frisk_b200.h"
#include "frisk_internal.h"

namespace frisk_internal {
int g_ingest_exact = 0;          // tests: always take the one-copy, count-first open
int g_ingest_chunk_tiles = 0;    // tests: tiles per upload chunk at least this (0 = default), so small texts are chunked too
}  // namespace frisk_internal

namespace {

constexpr int kTT = 256;                    // threads per tile
constexpr uint32_t kTile = kTT * 16u;       // text bytes per tile
constexpr int kST = 1024;                   // threads of the (single-CTA) tile scans
constexpr uint32_t kFullMask = 0xffffffffu;
// device counters of one open(): records, countN statistics (2), interior whitespace seen, and the state of a chunked open
enum { kCtrRecords = 0, kCtrNonUpper = 1, kCtrLower = 2, kCtrWhitespace = 3, kCtrAmbig = 4, kCtrOverflow = 5,
       // state carried from one chunk's tile scan to the next: line state, bases and packed offset of the open record
       kCtrKeyCarry = 6, kCtrBaseCarry = 7, kCtrOffCarry = 8,
       kLayCounted = 9,        // plane words already handed to the count hook
       kLayPaddedLen = 10,     // padded length of the finished layout
       kCtrCount = 12,
       kRangeSlots = 2 };      // per chunk, behind the counters: {word_lo, word_hi}

static_assert((int)kCtrRecords == (int)frisk_internal::kIngestRecords && (int)kCtrNonUpper == (int)frisk_internal::kIngestNonUpper &&
              (int)kCtrLower == (int)frisk_internal::kIngestLower && (int)kCtrOverflow == (int)frisk_internal::kIngestOverflow &&
              (int)kCtrCount == (int)frisk_internal::kIngestRange, "frisk_internal.h names these counters");

// class of a byte: 0..3 = A,T,G,C (F:70 order); 4..7 = a,t,g,c; 8 = anything else; 9 = whitespace
// removed by the reference's line.strip() (F:149)
__device__ __forceinline__ uint32_t class_of(uint32_t c) {
    switch (c) {
        case 'A': return 0; case 'T': return 1; case 'G': return 2; case 'C': return 3;
        case 'a': return 4; case 't': return 5; case 'g': return 6; case 'c': return 7;
        case ' ': case '\t': case '\n': case '\r': case '\v': case '\f': return 9;
        default: return 8;
    }
}

__device__ __forceinline__ uint32_t byte_of(const uint4& v, int k) {
    const uint32_t w = k < 4 ? v.x : (k < 8 ? v.y : (k < 12 ? v.z : v.w));
    return (w >> (8 * (k & 3))) & 0xffu;
}

// Is the line starting at byte i a header?  Its first non-blank character decides (the reference
// strips the line before looking at it, F:149-153).
// `avail` (<= n): bytes already on the device (chunked upload).  A decision that would need a byte beyond it is reported
// through *ambig (the caller then falls back to the one-shot path); with avail == n it cannot happen.
__device__ bool line_is_header(const uint8_t* __restrict__ t, uint64_t i, uint64_t n, uint64_t avail, uint32_t* ambig) {
    while (i < n) {
        if (i >= avail) { *ambig = 1u; return false; }
        const uint32_t c = t[i];
        if (c == '\n') return false;                 // blank line
        if (class_of(c) != 9u) return c == '>';
        ++i;
    }
    return false;
}

// state of the last line start of a thread / tile: 0 = no line starts here, 1 = sequence line, 2 = header
__device__ __forceinline__ uint32_t last_key(uint32_t start_mask, uint32_t hdr_mask) {
    return start_mask ? 1u + ((hdr_mask >> (31 - __clz(start_mask))) & 1u) : 0u;
}

// ---- block-wide scans (blockDim.x a multiple of 32, <= 1024); sm: >= 64 words of shared memory ----------
// Two levels: a shuffle scan inside every warp, the warp totals through shared memory, and -- instead of every thread walking
// the totals one by one -- the same shuffle scan over the (<= 32) totals, done by every warp for itself.
template <typename T>
__device__ __forceinline__ T block_excl_sum(T v, T* sm, T* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    T incl = v;
#pragma unroll
    for (int ofs = 1; ofs < 32; ofs <<= 1) {
        const T y = __shfl_up_sync(kFullMask, incl, ofs);
        if (lane >= ofs) incl += y;
    }
    if (lane == 31) sm[warp] = incl;
    __syncthreads();
    T w = lane < nw ? sm[lane] : T(0);
#pragma unroll
    for (int ofs = 1; ofs < 32; ofs <<= 1) {
        const T y = __shfl_up_sync(kFullMask, w, ofs);
        if (lane >= ofs) w += y;
    }
    const T before = __shfl_sync(kFullMask, w, warp ? warp - 1 : 0);
    *total = __shfl_sync(kFullMask, w, nw - 1);
    __syncthreads();
    return (warp ? before : T(0)) + incl - v;
}

// "last writer wins": the last non-zero key among the threads before this one (0 if none);
// *last = the last non-zero key of the whole block
__device__ __forceinline__ uint32_t block_excl_last(uint32_t key, uint32_t* sm, uint32_t* last) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const uint32_t ball = __ballot_sync(kFullMask, key != 0u);
    const uint32_t prior = ball & ((1u << lane) - 1u);
    uint32_t v = __shfl_sync(kFullMask, key, prior ? 31 - __clz(prior) : 0);
    if (!prior) v = 0;
    const uint32_t wl = __shfl_sync(kFullMask, key, ball ? 31 - __clz(ball) : 0);
    if (lane == 0) sm[warp] = ball ? wl : 0u;
    __syncthreads();
    const uint32_t x = lane < nw ? sm[lane] : 0u;
    const uint32_t wb = __ballot_sync(kFullMask, x != 0u);
    const uint32_t wprior = wb & ((1u << warp) - 1u);
    uint32_t carry = __shfl_sync(kFullMask, x, wprior ? 31 - __clz(wprior) : 0);
    if (!wprior) carry = 0;
    const uint32_t tot = __shfl_sync(kFullMask, x, wb ? 31 - __clz(wb) : 0);
    __syncthreads();
    *last = wb ? tot : 0u;
    return v ? v : carry;
}

// Segmented sum.  Element = (f, v): f = "a reset happens inside this element", v = the amount after
// its last reset (the whole amount when !f).  Returns the amount accumulated since the last reset
// before this thread; *reset_before = some earlier thread has a reset.
template <typename T>
__device__ __forceinline__ T block_excl_seg(bool f, T v, T* smv, uint32_t* smf, bool* reset_before) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    T iv = v;
    uint32_t fl = f ? 1u : 0u;
#pragma unroll
    for (int ofs = 1; ofs < 32; ofs <<= 1) {
        const T uv = __shfl_up_sync(kFullMask, iv, ofs);
        const uint32_t uf = __shfl_up_sync(kFullMask, fl, ofs);
        if (lane >= ofs) { if (!fl) iv += uv; fl |= uf; }
    }
    T ev = __shfl_up_sync(kFullMask, iv, 1);
    uint32_t ef = __shfl_up_sync(kFullMask, fl, 1);
    if (lane == 0) { ev = 0; ef = 0; }
    if (lane == 31) { smv[warp] = iv; smf[warp] = fl; }
    __syncthreads();
    T wv = lane < nw ? smv[lane] : T(0);                     // the same segmented scan over the warp totals
    uint32_t wf = lane < nw ? smf[lane] : 0u;
#pragma unroll
    for (int ofs = 1; ofs < 32; ofs <<= 1) {
        const T uv = __shfl_up_sync(kFullMask, wv, ofs);
        const uint32_t uf = __shfl_up_sync(kFullMask, wf, ofs);
        if (lane >= ofs) { if (!wf) wv += uv; wf |= uf; }
    }
    T c = __shfl_sync(kFullMask, wv, warp ? warp - 1 : 0);
    uint32_t cf = __shfl_sync(kFullMask, wf, warp ? warp - 1 : 0);
    if (!warp) { c = 0; cf = 0; }
    __syncthreads();
    if (!ef) ev += c;
    *reset_before = (ef | cf) != 0u;
    return ev;
}

// ---- the lines of a thread's 16 bytes ------------------------------------------------------------------------------------
// 16-bit masks, bit k = byte k: '\n', other blanks (the characters line.strip() removes, F:149), line starts, header line
// starts, and the bytes that are not blank.  Ordinary sequence bytes never enter a per-byte branch: the bytes below 0x21 and
// the '>' are found with four word-wide tests, and only those (one newline per 61 bytes of a 60-column file) are looked at.
struct Lines { uint32_t nl, ws, start, hdr, nonblank; };

__device__ __forceinline__ uint32_t special_bytes(uint32_t x) {              // bit 7 of every byte that is < 0x21 or '>'
    const uint32_t lt = ~(((x | 0x80808080u) - 0x21212121u) | x);
    const uint32_t v = x ^ 0x3E3E3E3Eu;
    const uint32_t gt = ~(((v & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | v);
    return (lt | gt) & 0x80808080u;
}
__device__ __forceinline__ uint32_t flags_to_nibble(uint32_t w) {           // bit 7 of byte j -> bit j
    return (((w >> 7) & 0x01010101u) * 0x01020408u) >> 24;
}
__device__ __forceinline__ uint32_t below(int k) { return (1u << k) - 1u; }  // k <= 16

__device__ __forceinline__ Lines thread_lines(const uint8_t* __restrict__ t, uint64_t n, uint64_t i0, const uint4& raw, uint32_t prev,
                                              uint64_t avail, uint32_t* ambig) {
    const uint32_t sp = flags_to_nibble(special_bytes(raw.x)) | (flags_to_nibble(special_bytes(raw.y)) << 4) |
                        (flags_to_nibble(special_bytes(raw.z)) << 8) | (flags_to_nibble(special_bytes(raw.w)) << 12);
    Lines L;
    L.nl = 0; L.ws = 0;
    uint32_t gt = 0;
    for (uint32_t m = sp; m; m &= m - 1u) {
        const int k = __ffs(m) - 1;
        const uint32_t c = byte_of(raw, k);
        if (c == '\n') L.nl |= 1u << k;
        else if (c == '>') gt |= 1u << k;
        else if (c == ' ' || (c >= 9u && c <= 13u)) L.ws |= 1u << k;
    }
    L.start = ((L.nl << 1) | (prev == '\n' ? 1u : 0u)) & 0xffffu;
    L.hdr = L.start & gt;                                   // its first non-blank character decides (F:149-153)
    for (uint32_t lead = L.start & L.ws; lead; lead &= lead - 1u) {         // a line that begins with blanks (rare): look further
        const int k = __ffs(lead) - 1;
        if (line_is_header(t, i0 + k, n, avail, ambig)) L.hdr |= 1u << k;
    }
    L.nonblank = ~(L.nl | L.ws) & 0xffffu;
    return L;
}

__device__ __forceinline__ unsigned long long align128(unsigned long long v) { return (v + 127ull) & ~127ull; }

// What a thread's bytes add up to: bases before its first line start (`head`: whether they count depends on the line they
// continue), bases after it and before its first header line (`pre`; all of them when there is no header), after its last
// header (`post`), and the packed space of the records opened AND closed inside the thread (frisk_b200_pack_layout's rule:
// every record takes align128(len + 1) bases).
struct ThreadSum { uint32_t n_hdr, head, pre, post, inner, key; };

__device__ __forceinline__ ThreadSum thread_sum(const Lines& L) {
    ThreadSum s;
    s.n_hdr = 0; s.pre = 0; s.post = 0; s.inner = 0;
    const int first = L.start ? __ffs(L.start) - 1 : 16;
    s.head = __popc(L.nonblank & below(first));
    uint32_t cur = 0;
    for (uint32_t m = L.start; m;) {
        const int k = __ffs(m) - 1;
        m &= m - 1u;
        const int nx = m ? __ffs(m) - 1 : 16;
        if ((L.hdr >> k) & 1u) {
            if (s.n_hdr == 0) s.pre = cur; else s.inner += (uint32_t)align128(cur + 1u);
            ++s.n_hdr;
            cur = 0;                                        // the header line itself holds no bases
        } else {
            cur += __popc(L.nonblank & below(nx) & ~below(k));
        }
    }
    if (s.n_hdr) s.post = cur; else s.pre = cur;
    s.key = last_key(L.start, L.hdr);
    return s;
}

__device__ __forceinline__ uint32_t prev_byte(const uint8_t* __restrict__ t, uint64_t i0, const uint4& raw) {
    const uint32_t up = __shfl_up_sync(kFullMask, raw.w, 1);
    return (threadIdx.x & 31) ? up >> 24 : (i0 ? (uint32_t)t[i0 - 1] : (uint32_t)'\n');
}

// Does a line start in an earlier thread of the tile?  (header-free tiles: all that the line state needs)  One barrier.
__device__ __forceinline__ bool start_before(bool has_start, uint32_t* s_ball, bool* any_start) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t ball = __ballot_sync(kFullMask, has_start);
    if (lane == 0) s_ball[warp] = ball;
    __syncthreads();
    uint32_t earlier = ball & ((1u << lane) - 1u), any = 0;
#pragma unroll
    for (int w = 0; w < kTT / 32; ++w) {
        const uint32_t b = s_ball[w];
        any |= b;
        if (w < warp) earlier |= b;
    }
    *any_start = any != 0u;
    return earlier != 0u;
}

// ---- pass A: what every tile adds up to --------------------------------------------------------------------------------
__global__ void __launch_bounds__(kTT)
fasta_summary_kernel(const uint8_t* __restrict__ t, uint64_t n, uint64_t tile0, uint64_t avail, unsigned long long* __restrict__ counters,
                     uint32_t* __restrict__ tile_nhdr, uint8_t* __restrict__ tile_key, uint32_t* __restrict__ tile_head,
                     uint32_t* __restrict__ tile_pre, uint32_t* __restrict__ tile_post, uint32_t* __restrict__ tile_inner) {
    __shared__ unsigned long long sm[64];
    __shared__ uint32_t smf[32];
    const uint64_t tile = tile0 + blockIdx.x;
    const uint64_t i0 = tile * kTile + threadIdx.x * 16u;
    const uint4 raw = *reinterpret_cast<const uint4*>(t + i0);
    const Lines L = thread_lines(t, n, i0, raw, prev_byte(t, i0, raw), avail, reinterpret_cast<uint32_t*>(counters + kCtrAmbig));
    const ThreadSum s = thread_sum(L);
    if (!__syncthreads_or(s.n_hdr != 0u)) {
        // no header line in this tile (almost every tile): two sums -- the bases before the tile's first line start, and the rest
        __shared__ uint32_t s_ball[kTT / 32], s_part[kTT / 32];
        bool any_start;
        const bool sb = start_before(L.start != 0u, s_ball, &any_start);
        const uint32_t part = __reduce_add_sync(kFullMask, sb ? (s.head + s.pre) << 16 : s.head | (s.pre << 16));
        if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = part;
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t tot = 0;
#pragma unroll
            for (int w = 0; w < kTT / 32; ++w) tot += s_part[w];
            tile_nhdr[tile] = 0; tile_inner[tile] = 0;
            tile_key[tile] = any_start ? 1 : 0;
            tile_head[tile] = tot & 0xffffu;
            tile_pre[tile] = tile_post[tile] = tot >> 16;
        }
        return;
    }
    uint32_t last;
    const uint32_t key_before = block_excl_last(s.key, reinterpret_cast<uint32_t*>(sm), &last);
    // bytes before the thread's first line start continue a line that began earlier in the tile -- or before the tile, and
    // then they are the tile's `head`, resolved by the scan over tiles
    const uint32_t pre_def = (key_before == 1u ? s.head : 0u) + s.pre;
    const bool f = s.n_hdr != 0u;
    bool reset_before;
    const uint32_t carry = block_excl_seg<uint32_t>(f, f ? s.post : pre_def, reinterpret_cast<uint32_t*>(sm), smf, &reset_before);
    unsigned long long inner = s.inner;
    if (f && reset_before) inner += align128((unsigned long long)carry + pre_def + 1ull);   // closes a record opened in this tile
    unsigned long long total;
    block_excl_sum<unsigned long long>((unsigned long long)s.n_hdr | ((unsigned long long)(key_before ? 0u : s.head) << 16) | (inner << 32),
                                       sm, &total);
    if (f && !reset_before) tile_pre[tile] = carry + pre_def;           // the tile's first header: bases before it
    if (threadIdx.x == kTT - 1) {
        const uint32_t after = f ? s.post : carry + pre_def;            // bases after the tile's last header (all, if none)
        tile_post[tile] = after;
        if (!f && !reset_before) tile_pre[tile] = after;
        tile_nhdr[tile] = (uint32_t)(total & 0xffffu);
        tile_head[tile] = (uint32_t)((total >> 16) & 0xffffu);
        tile_inner[tile] = (uint32_t)(total >> 32);
        tile_key[tile] = (uint8_t)last;
    }
}

// ---- the scan over tiles (one CTA): records before every tile, the line state it starts in, the bases and the packed
// offset of the record that is open there -- frisk_b200_pack_layout's layout, computed on the device ---------------------
// Tiles [tile_lo, tile_hi): one chunk of a chunked upload, or everything.  The state at tile_lo comes from `counters`
// (records, line state, open record's bases and offset) and the state at tile_hi goes back there.  range_out[0..1]: the
// plane words that are final once the chunk is packed and have not been handed out yet (count_now; the count kernel looks
// one word ahead).  final: the text ends at tile_hi -- the open record closes, counters[kLayPaddedLen] is the layout's length.
constexpr int kSP = 4;                      // tiles per thread and batch of the tile scan (vector loads)

__global__ void __launch_bounds__(kST)
fasta_tilescan_kernel(const uint32_t* __restrict__ tile_nhdr, const uint8_t* __restrict__ tile_key, const uint32_t* __restrict__ tile_head,
                      const uint32_t* __restrict__ tile_pre, const uint32_t* __restrict__ tile_post, const uint32_t* __restrict__ tile_inner,
                      uint64_t tile_lo, uint64_t tile_hi, uint32_t* __restrict__ tile_rec_base, uint8_t* __restrict__ tile_carry_hdr,
                      unsigned long long* __restrict__ tile_base_in, unsigned long long* __restrict__ tile_open_off,
                      unsigned long long* __restrict__ counters, unsigned long long* __restrict__ range_out, uint64_t rec_cap,
                      uint64_t plane_cap, int count_now, int final) {
    // tile_lo is a multiple of kSP and the arrays are padded to one: a thread owns kSP consecutive tiles of a batch of
    // kST * kSP, loaded as vectors and kept in registers through the three scans; batches follow each other with the carries
    __shared__ unsigned long long sm[64];
    __shared__ uint32_t smf[32];
    __shared__ unsigned long long s_bases;
    unsigned long long rec_c = counters[kCtrRecords], base_c = counters[kCtrBaseCarry], off_c = counters[kCtrOffCarry];
    uint32_t key_c = (uint32_t)counters[kCtrKeyCarry];
    for (uint64_t b0 = tile_lo; b0 < tile_hi; b0 += (uint64_t)kST * kSP) {
        const uint64_t i = b0 + (uint64_t)threadIdx.x * kSP;
        uint32_t nh[kSP] = {0, 0, 0, 0}, hd[kSP] = {0, 0, 0, 0}, pr[kSP] = {0, 0, 0, 0}, po[kSP] = {0, 0, 0, 0}, in[kSP] = {0, 0, 0, 0},
                 ky[kSP] = {0, 0, 0, 0};
        if (i < tile_hi) {
            const uint4 a = *reinterpret_cast<const uint4*>(tile_nhdr + i), b = *reinterpret_cast<const uint4*>(tile_head + i),
                        c = *reinterpret_cast<const uint4*>(tile_pre + i), d = *reinterpret_cast<const uint4*>(tile_post + i),
                        e = *reinterpret_cast<const uint4*>(tile_inner + i);
            const uchar4 k = *reinterpret_cast<const uchar4*>(tile_key + i);
            nh[0] = a.x; nh[1] = a.y; nh[2] = a.z; nh[3] = a.w;  hd[0] = b.x; hd[1] = b.y; hd[2] = b.z; hd[3] = b.w;
            pr[0] = c.x; pr[1] = c.y; pr[2] = c.z; pr[3] = c.w;  po[0] = d.x; po[1] = d.y; po[2] = d.z; po[3] = d.w;
            in[0] = e.x; in[1] = e.y; in[2] = e.z; in[3] = e.w;  ky[0] = k.x; ky[1] = k.y; ky[2] = k.z; ky[3] = k.w;
#pragma unroll
            for (int j = 0; j < kSP; ++j)
                if (i + j >= tile_hi) { nh[j] = hd[j] = pr[j] = po[j] = in[j] = ky[j] = 0; }   // beyond the range: neutral
        }
        // 1. records and line state
        uint32_t sum = 0, key = 0;
#pragma unroll
        for (int j = 0; j < kSP; ++j) { sum += nh[j]; if (ky[j]) key = ky[j]; }
        uint32_t total, last;
        unsigned long long run = rec_c + block_excl_sum<uint32_t>(sum, reinterpret_cast<uint32_t*>(sm), &total);
        uint32_t rk = block_excl_last(key, reinterpret_cast<uint32_t*>(sm), &last);
        if (!rk) rk = key_c;
        uint32_t recb[kSP], ch[kSP];
        bool f = false;
        unsigned long long v = 0;
#pragma unroll
        for (int j = 0; j < kSP; ++j) {
            recb[j] = (uint32_t)run;
            ch[j] = rk == 2u;
            // bases before the tile's first header: none of them counts before the first record of the file (F:153)
            pr[j] = run ? (rk == 2u ? 0u : hd[j]) + pr[j] : 0u;
            if (nh[j]) { f = true; v = po[j]; } else v += pr[j];
            run += nh[j];
            if (ky[j]) rk = ky[j];
        }
        // 2. bases of the open record before every tile (segmented by headers), and what the tile's closed records take
        bool rb;
        unsigned long long bases = block_excl_seg<unsigned long long>(f, v, sm, smf, &rb);
        if (!rb) bases += base_c;
        unsigned long long bi[kSP], ta[kSP], taken = 0;
#pragma unroll
        for (int j = 0; j < kSP; ++j) {
            bi[j] = bases;
            ta[j] = 0;
            if (nh[j]) {
                ta[j] = (recb[j] ? align128(bases + pr[j] + 1ull) : 0ull) + in[j];
                bases = po[j];
            } else bases += pr[j];
            taken += ta[j];
        }
        if (threadIdx.x == kST - 1) s_bases = bases;
        // 3. packed offset of the record open at every tile
        unsigned long long all;
        unsigned long long off = off_c + block_excl_sum<unsigned long long>(taken, sm, &all);   // (its barriers publish s_bases)
        if (i < tile_hi) {
            unsigned long long oo[kSP];
#pragma unroll
            for (int j = 0; j < kSP; ++j) { oo[j] = off; off += ta[j]; }
            *reinterpret_cast<uint4*>(tile_rec_base + i) = make_uint4(recb[0], recb[1], recb[2], recb[3]);
            *reinterpret_cast<uchar4*>(tile_carry_hdr + i) = make_uchar4((uint8_t)ch[0], (uint8_t)ch[1], (uint8_t)ch[2], (uint8_t)ch[3]);
            *reinterpret_cast<ulonglong2*>(tile_base_in + i) = make_ulonglong2(bi[0], bi[1]);
            *reinterpret_cast<ulonglong2*>(tile_base_in + i + 2) = make_ulonglong2(bi[2], bi[3]);
            *reinterpret_cast<ulonglong2*>(tile_open_off + i) = make_ulonglong2(oo[0], oo[1]);
            *reinterpret_cast<ulonglong2*>(tile_open_off + i + 2) = make_ulonglong2(oo[2], oo[3]);
        }
        rec_c += total;
        if (last) key_c = last;
        base_c = s_bases;
        off_c += all;
        __syncthreads();                                    // s_bases is rewritten by the next batch
    }
    if (threadIdx.x == 0) {
        const unsigned long long n_rec = rec_c;
        const unsigned long long pos_hi = n_rec ? off_c + base_c : 0ull;                   // first base not written yet
        const unsigned long long padded = (n_rec ? align128(pos_hi + 1ull) : 0ull) + 128ull;
        counters[kCtrRecords] = n_rec;
        counters[kCtrKeyCarry] = key_c;
        counters[kCtrBaseCarry] = base_c;
        counters[kCtrOffCarry] = off_c;
        const unsigned long long w_lo = counters[kLayCounted];
        unsigned long long w_hi = w_lo;
        if (n_rec > rec_cap || padded > plane_cap || counters[kCtrOverflow]) {
            counters[kCtrOverflow] = 1ull;
        } else {
            if (final) { w_hi = padded / 32ull - 1ull; counters[kLayPaddedLen] = padded; }
            else if (count_now && (pos_hi >> 5) >= 1ull) w_hi = max(w_lo, (pos_hi >> 5) - 1ull);
            if (!count_now) w_hi = w_lo;
        }
        range_out[0] = w_lo; range_out[1] = w_hi;
        counters[kLayCounted] = w_hi;
    }
}

// ---- pass B: everything else -- planes, record table, padding flags, countN statistics ----------------------------------
__device__ __forceinline__ void flag_invalid(uint32_t* __restrict__ inv, unsigned long long a, unsigned long long b) {   // [a, b), b % 32 == 0
    if (a & 31ull) {
        atomicOr(&inv[a >> 5], 0xffffffffu >> (uint32_t)(a & 31ull));   // shares its word with the record's last bases
        a = (a | 31ull) + 1ull;
    }
    for (; a < b; a += 32ull) inv[a >> 5] = 0xffffffffu;
}

// 2-bit codes of 4 characters (A=0, T=1, G=2, C=3, F:70 order; garbage for anything else), first character in bits 7..6
__device__ __forceinline__ uint32_t codes_of_word(uint32_t x) {
    const uint32_t y = x >> 1;                               // ASCII bits 2..1: A=00 C=01 T=10 G=11
    const uint32_t c = ((y & 0x01010101u) << 1) | ((y ^ (y >> 1)) & 0x01010101u);
    return (c * 0x40100401u) >> 24;
}
__device__ __forceinline__ uint32_t not_acgt_bytes(uint32_t x) {             // bit 7 of every byte that is not one of A, C, G, T
    const uint32_t a = x ^ 0x41414141u, c = x ^ 0x43434343u, g = x ^ 0x47474747u, u = x ^ 0x54545454u;
    const uint32_t m = 0x7F7F7F7Fu;
    return (((a & m) + m) | a) & (((c & m) + m) | c) & (((g & m) + m) | g) & (((u & m) + m) | u) & 0x80808080u;
}

__global__ void __launch_bounds__(kTT)
fasta_pack_kernel(const uint8_t* __restrict__ t, uint64_t n, uint64_t tile0, uint64_t avail, uint64_t n_tiles_total, int final,
                  const uint32_t* __restrict__ tile_nhdr, const uint32_t* __restrict__ tile_rec_base,
                  const uint8_t* __restrict__ tile_carry_hdr, const unsigned long long* __restrict__ tile_base_in,
                  const unsigned long long* __restrict__ tile_open_off, unsigned long long* __restrict__ counters,
                  unsigned long long* __restrict__ rec_hdr_pos, unsigned long long* __restrict__ rec_len,
                  unsigned long long* __restrict__ rec_off, uint64_t rec_cap,
                  uint32_t* __restrict__ codes, uint32_t* __restrict__ inv, uint32_t* __restrict__ low) {
    __shared__ unsigned long long sm[64];
    __shared__ uint32_t smf[32];
    __shared__ uint32_t s_stats[2];
    if (counters[kCtrOverflow]) return;                      // speculative capacities exceeded: nothing to write to (whole grid)
    const int tid = threadIdx.x;
    if (tid < 2) s_stats[tid] = 0;
    const uint64_t tile = tile0 + blockIdx.x;
    const uint64_t i0 = tile * kTile + (uint64_t)tid * 16u;
    const uint4 raw = *reinterpret_cast<const uint4*>(t + i0);
    uint32_t* const ambig = reinterpret_cast<uint32_t*>(counters + kCtrAmbig);
    const Lines L = thread_lines(t, n, i0, raw, prev_byte(t, i0, raw), avail, ambig);
    const ThreadSum s = thread_sum(L);
    const bool f = s.n_hdr != 0u;
    uint32_t hdr_before = 0, pre_def;
    unsigned long long bases_before, off;
    bool in_hdr;
    if (tile_nhdr[tile] == 0u) {                             // no header line in this tile: one record, one running sum
        __shared__ uint32_t s_ball[kTT / 32];
        bool any_start;
        in_hdr = !start_before(L.start != 0u, s_ball, &any_start) && tile_carry_hdr[tile] != 0;      // (also orders s_stats)
        pre_def = (in_hdr ? 0u : s.head) + s.pre;
        uint32_t tot;
        bases_before = tile_base_in[tile] + block_excl_sum<uint32_t>(pre_def, reinterpret_cast<uint32_t*>(sm), &tot);
        off = tile_open_off[tile];
    } else {
        uint32_t tot, last;
        const uint32_t key_before = block_excl_last(s.key, reinterpret_cast<uint32_t*>(sm), &last);  // (also orders s_stats)
        in_hdr = key_before ? key_before == 2u : tile_carry_hdr[tile] != 0;
        pre_def = (in_hdr ? 0u : s.head) + s.pre;
        hdr_before = block_excl_sum<uint32_t>(s.n_hdr, reinterpret_cast<uint32_t*>(sm), &tot);
        bool reset_before;
        const uint32_t carry = block_excl_seg<uint32_t>(f, f ? s.post : pre_def, reinterpret_cast<uint32_t*>(sm), smf, &reset_before);
        bases_before = reset_before ? (unsigned long long)carry : tile_base_in[tile] + carry;
        unsigned long long a = s.inner, all;
        if (f && tile_rec_base[tile] + hdr_before >= 1u) a += align128(bases_before + pre_def + 1ull);
        off = tile_open_off[tile] + block_excl_sum<unsigned long long>(a, sm, &all);
    }
    uint32_t rec = tile_rec_base[tile] + hdr_before;         // records opened before this thread; the open one is rec - 1
    unsigned long long pos = off + bases_before;             // where the thread's first base goes

    uint32_t bad = 0;
    if (!f && rec >= 1u) {
        bad = (flags_to_nibble(not_acgt_bytes(raw.x)) | (flags_to_nibble(not_acgt_bytes(raw.y)) << 4) |
               (flags_to_nibble(not_acgt_bytes(raw.z)) << 8) | (flags_to_nibble(not_acgt_bytes(raw.w)) << 12));
    }
    const int first = L.start ? __ffs(L.start) - 1 : 16;
    const uint32_t emit = L.nonblank & (in_hdr ? ~below(first) : 0xffffu);
    const uint32_t ws_hard = L.ws & ~(L.nl >> 1);            // a blank that is not directly followed by the newline (a '\r' is)
    if (!f && (rec == 0u || ((bad & emit) == 0u && ws_hard == 0u))) {
        // ---- the common thread: part of sequence lines, every base an upper-case A, C, G or T, no blank but newlines ----
        const uint32_t cnt = rec ? __popc(emit) : 0u;
        if (cnt) {
            uint32_t cw = (codes_of_word(raw.x) << 24) | (codes_of_word(raw.y) << 16) | (codes_of_word(raw.z) << 8) | codes_of_word(raw.w);
            for (uint32_t skip = ~emit & 0xffffu; skip;) {   // squeeze the skipped bytes out, last one first
                const int k = 31 - __clz(skip);
                skip &= ~(1u << k);
                const uint32_t hi = k ? cw & (0xffffffffu << (32 - 2 * k)) : 0u;
                const uint32_t lo = k < 15 ? cw & (0xffffffffu >> (2 * k + 2)) : 0u;
                cw = hi | (lo << 2);
            }
            if (cnt < 16u) cw &= ~(0xffffffffu >> (2u * cnt));
            const uint32_t sh = 2u * ((uint32_t)pos & 15u);
            atomicOr(&codes[pos >> 4], cw >> sh);
            if (sh && cnt > 16u - ((uint32_t)pos & 15u)) atomicOr(&codes[(pos >> 4) + 1ull], cw << (32u - sh));
            pos += cnt;
        }
    } else {
        // ---- anything else (a header line, lower case, N, blanks): byte by byte ----------------------------------------------
        unsigned long long cidx = pos >> 4, midx = pos >> 5;
        uint32_t cacc = 0, iacc = 0, lacc = 0, non_upper = 0, lower = 0;
        auto flush_codes = [&]() { if (cacc) atomicOr(&codes[cidx], cacc); cacc = 0; };
        auto flush_masks = [&]() {
            if (iacc) atomicOr(&inv[midx], iacc);
            if (lacc) atomicOr(&low[midx], lacc);
            iacc = 0; lacc = 0;
        };
#pragma unroll 1
        for (int k = 0; k < 16; ++k) {
            if ((L.start >> k) & 1u) {
                const bool h = (L.hdr >> k) & 1u;
                if (h) {                                     // a record begins: the open one (if any) is complete
                    flush_codes(); flush_masks();
                    unsigned long long next = 0;
                    if (rec >= 1u) {
                        const unsigned long long len = pos - off;
                        next = off + align128(len + 1ull);
                        if (rec - 1u < rec_cap) rec_len[rec - 1u] = len;
                        flag_invalid(inv, pos, next);        // >= 1 padding base after every record
                    }
                    ++rec;
                    if (rec - 1u < rec_cap) { rec_hdr_pos[rec - 1u] = i0 + k; rec_off[rec - 1u] = next; }
                    off = pos = next;
                    cidx = pos >> 4; midx = pos >> 5;
                }
                in_hdr = h;
            }
            const uint32_t b = byte_of(raw, k);
            const uint32_t c = class_of(b);
            if (c == 9u && !in_hdr && rec >= 1u && b != '\n') {
                // Whitespace in a sequence line: harmless at the ends (the reference strips them, F:149 -- every '\r' of a
                // CRLF file lands here and is cleared by its two neighbours), refused INSIDE the line, where the
                // reference keeps it as a character of the sequence (same rule as frisk_b200_fasta_scan).
                bool before = false, after = false;
                uint64_t p = i0 + k;
                int q = 0;
                for (; q < 4096 && p > 0; ++q) {
                    const uint32_t x = t[--p];
                    if (x == '\n') break;
                    if (class_of(x) != 9u) { before = true; break; }
                }
                if (q == 4096) before = true;                // a whitespace run this long is not a line ending
                p = i0 + k;
                for (q = 0; q < 4096 && p + 1 < n; ++q) {
                    if (p + 1 >= avail) { *ambig = 1u; break; }             // the rest of the line is not on the device yet
                    const uint32_t x = t[++p];
                    if (x == '\n') break;
                    if (class_of(x) != 9u) { after = true; break; }
                }
                if (q == 4096) after = true;
                if (before && after) counters[kCtrWhitespace] = 1ull;
            }
            if (!in_hdr && c != 9u && rec >= 1u) {
                if ((pos >> 4) != cidx) { flush_codes(); cidx = pos >> 4; }
                if ((pos >> 5) != midx) { flush_masks(); midx = pos >> 5; }
                const uint32_t b32 = 0x80000000u >> ((uint32_t)pos & 31u);
                if (c < 8u) cacc |= (c & 3u) << (30u - 2u * ((uint32_t)pos & 15u)); else iacc |= b32;
                if ((c >= 4u) & (c < 8u)) lacc |= b32;
                non_upper += c >= 4u;
                lower += (c >= 4u) & (c < 8u);
                ++pos;
            }
        }
        flush_codes(); flush_masks();
        if (non_upper) atomicAdd(&s_stats[0], non_upper);
        if (lower) atomicAdd(&s_stats[1], lower);
    }
    if (final && tile == n_tiles_total - 1 && tid == kTT - 1) {             // the text ends here: the open record closes
        unsigned long long end = 0;
        if (rec >= 1u) {
            const unsigned long long len = pos - off;
            if (rec - 1u < rec_cap) rec_len[rec - 1u] = len;
            end = off + align128(len + 1ull);
            flag_invalid(inv, pos, end + 128ull);            // + the >= 128 trailing bases the kernels look ahead into
        } else flag_invalid(inv, 0ull, 128ull);
    }
    __syncthreads();
    if (tid == 0) {
        if (s_stats[0]) atomicAdd(&counters[kCtrNonUpper], (unsigned long long)s_stats[0]);
        if (s_stats[1]) atomicAdd(&counters[kCtrLower], (unsigned long long)s_stats[1]);
    }
}

// ---- names of a BGZF open: the text stays on the device, so the header lines are gathered into one buffer ----------------
// line_len[r]: bytes of record r's header line from hdr_pos[r], its newline included (none at the end of the text)
__global__ void header_len_kernel(const uint8_t* __restrict__ t, uint64_t n, const unsigned long long* __restrict__ hdr_pos,
                                  uint64_t n_rec, unsigned long long* __restrict__ line_len) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rec) return;
    uint64_t i = hdr_pos[r];
    while (i < n && t[i] != '\n') ++i;
    line_len[r] = (i < n ? i + 1 : n) - hdr_pos[r];
}

// in place: line_len[0..n_rec) -> exclusive prefix sum, line_len[n_rec] = total (one CTA of kST threads)
__global__ void __launch_bounds__(kST) header_scan_kernel(unsigned long long* __restrict__ v, uint64_t n_rec) {
    __shared__ unsigned long long sm[64];
    unsigned long long carry = 0;
    for (uint64_t b0 = 0; b0 < n_rec; b0 += kST) {
        const uint64_t i = b0 + threadIdx.x;
        const unsigned long long x = i < n_rec ? v[i] : 0ull;
        unsigned long long total;
        const unsigned long long e = block_excl_sum<unsigned long long>(x, sm, &total);
        if (i < n_rec) v[i] = carry + e;
        carry += total;
    }
    if (threadIdx.x == 0) v[n_rec] = carry;
}

__global__ void header_gather_kernel(const uint8_t* __restrict__ t, const unsigned long long* __restrict__ hdr_pos,
                                     const unsigned long long* __restrict__ line_off, uint64_t n_rec, uint8_t* __restrict__ out) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rec) return;
    const uint64_t a = hdr_pos[r], o = line_off[r], len = line_off[r + 1] - o;
    for (uint64_t k = 0; k < len; ++k) out[o + k] = t[a + k];
}

}  // namespace

struct frisk_b200_fasta {
    uint64_t n = 0, n_tiles = 0, n_rec = 0, padded_len = 128;
    uint64_t stats[3] = {0, 0, 0};
    uint8_t* d_text = nullptr;
    uint32_t *d_nhdr = nullptr, *d_head = nullptr, *d_pre = nullptr, *d_post = nullptr, *d_inner = nullptr, *d_rec_base = nullptr;
    uint8_t *d_key = nullptr, *d_carry = nullptr;
    unsigned long long *d_base_in = nullptr, *d_open_off = nullptr, *d_hdr_pos = nullptr, *d_len = nullptr, *d_scaf_off = nullptr,
                       *d_counters = nullptr;
    uint32_t *d_codes = nullptr, *d_inv = nullptr, *d_low = nullptr;     // the planes, built by the open and owned by the handle
    void *d_scan_slab = nullptr, *d_out_slab = nullptr;                  // what the pointers above (but d_text) are carved from
    uint64_t rec_cap = 0;                                                // entries of the device record table
    bool streamed = false;                                               // opened on the chunked, speculatively sized path
    bool device_text = false;                                            // opened from BGZF or gzip: names index name_text
    void* d_gz_slab = nullptr;                                           // BGZF: compressed bytes, block table, status words
    std::vector<uint64_t> name_off, seq_len, scaf_off, hdr_pos;
    std::vector<uint32_t> name_len;
    std::vector<char> name_text;                                         // BGZF / gzip: the header lines, one after the other
};

namespace {
int free_all(frisk_b200_fasta* h, cudaStream_t st) {
    void* ptrs[] = {h->d_text, h->d_scan_slab, h->d_out_slab, h->d_gz_slab};
    for (void* p : ptrs)
        if (p) FRISK_CK(cudaFreeAsync(p, st));
    h->d_text = nullptr; h->d_scan_slab = h->d_out_slab = h->d_gz_slab = nullptr;
    h->d_nhdr = h->d_head = h->d_pre = h->d_post = h->d_inner = h->d_rec_base = nullptr;
    h->d_key = h->d_carry = nullptr;
    h->d_base_in = h->d_open_off = h->d_hdr_pos = h->d_len = h->d_scaf_off = h->d_counters = nullptr;
    h->d_codes = h->d_inv = h->d_low = nullptr;
    return FRISK_OK;
}

// carve `bytes` (rounded up to 256) off a slab
template <typename T>
void carve(char*& cursor, T*& out, uint64_t bytes) {
    out = reinterpret_cast<T*>(cursor);
    cursor += (bytes + 255) & ~255ull;
}

// ---- the upload lane: text chunks travel on a second stream while the passes of the previous chunk run -------------------
constexpr int kMaxChunks = 48;
constexpr uint64_t kMinChunkTiles = 1400;           // 5.6 MiB of text per chunk at least (see the chunk plan in open_impl)
constexpr int kRetryExact = -1000;                  // internal: the chunked / speculative open could not decide, open again
constexpr uint64_t kFirstFetch = 4096;              // records read back with the counters (one synchronisation when R <= this)

struct UploadLane {
    cudaStream_t copy = nullptr;
    cudaEvent_t ready = nullptr, done[kMaxChunks] = {};
    std::mutex mu;                                   // one open at a time per device: the events above are shared
    unsigned long long* stage = nullptr;             // page-locked landing zone of the counters + the first kFirstFetch records
};
std::mutex g_lane_mu;
std::atomic<uint64_t> g_open_stats[2];
UploadLane g_lane[64];

int upload_lane(UploadLane** out) {
    int dev = 0;
    FRISK_CK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return FRISK_E_UNSUPPORTED;
    std::lock_guard<std::mutex> lk(g_lane_mu);
    UploadLane& l = g_lane[dev];
    if (!l.copy) {
        FRISK_CK(cudaStreamCreateWithFlags(&l.copy, cudaStreamNonBlocking));
        FRISK_CK(cudaEventCreateWithFlags(&l.ready, cudaEventDisableTiming));
        for (auto& e : l.done) FRISK_CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        FRISK_CK(cudaHostAlloc((void**)&l.stage, (2 * kFirstFetch + kCtrCount + 1) * 8, cudaHostAllocDefault));
    }
    *out = &l;
    return FRISK_OK;
}

// What an open reads: a host text, a BGZF buffer with its block table, or a gzip member (the text is inflated on the device).
struct Source {
    const char* text = nullptr;           // host text (nullptr for BGZF and gzip)
    uint64_t n = 0;                       // text bytes (BGZF, gzip: inflated)
    bool bgzf = false, gzip = false;
    const uint8_t* gz = nullptr;
    uint64_t gz_n = 0, n_blocks = 0;
    std::vector<uint64_t> table;          // per block: comp_off, text_off (8 bytes each), comp_len, crc (4 bytes each)
    uint8_t* d_ready = nullptr;           // gzip, the exact re-open: the text inflated already (the handle takes it)
    bool device() const { return bgzf || gzip; }   // the text exists on the device only
};

// the text buffer of an open: kTile-padded, '\n' behind the text
int alloc_text(uint64_t n, cudaStream_t st, uint8_t** out) {
    const uint64_t padded_text = (n + kTile - 1) / kTile * kTile + 16;
    FRISK_CK(cudaMallocAsync((void**)out, padded_text, st));
    FRISK_CK(cudaMemsetAsync(*out + n, '\n', padded_text - n, st));
    return FRISK_OK;
}

// gzip: the member goes up and is inflated into a text buffer of its own (src->d_ready)
int gzip_source(const char* gz, uint64_t n, cudaStream_t st, Source* src) {
    src->gzip = true;
    uint8_t* d_gz = nullptr;
    FRISK_CK(cudaMallocAsync((void**)&d_gz, n ? n : 1, st));
    auto alloc = [&](uint64_t len, uint8_t** out) -> int {
        *out = nullptr;
        if (!len) return FRISK_OK;                        // no text: the open's empty path
        const int rc = alloc_text(len, st, out);
        src->d_ready = *out;
        return rc;
    };
    const cudaError_t e = cudaMemcpyAsync(d_gz, gz, n, cudaMemcpyHostToDevice, st);
    int rc = e == cudaSuccess ? frisk_internal::gzip_inflate(d_gz, reinterpret_cast<const uint8_t*>(gz), n, alloc, &src->n, nullptr, st)
                              : frisk_internal::cuda_fail(e, "cudaMemcpyAsync(d_gz)");
    cudaFreeAsync(d_gz, st);                              // (every exit; a failed text buffer is freed by open_handle)
    return rc;
}

int make_source(const char* text, uint64_t n, frisk_internal::TextFormat fmt, cudaStream_t st, Source* src) {
    if (fmt == frisk_internal::kFmtGzip) return gzip_source(text, n, st, src);
    if (fmt != frisk_internal::kFmtBgzf) { src->text = text; src->n = n; return FRISK_OK; }
    src->bgzf = true;
    src->gz = reinterpret_cast<const uint8_t*>(text);
    src->gz_n = n;
    uint64_t nb = 0, tl = 0;
    int rc = frisk_b200_bgzf_blocks(src->gz, n, 0, nullptr, nullptr, nullptr, nullptr, &nb, &tl);
    if (rc) return rc;
    src->table.assign(nb * 3, 0);
    uint64_t* const t = src->table.data();
    uint32_t* const t32 = reinterpret_cast<uint32_t*>(t + 2 * nb);
    if ((rc = frisk_b200_bgzf_blocks(src->gz, n, nb, t, t32, t32 + nb, t + nb, &nb, &tl))) return rc;
    src->n_blocks = nb;
    src->n = tl;
    return FRISK_OK;
}

// BGZF: compressed bytes and block table up on `copy`, every member inflated into h->d_text behind them.  The status words
// and the "some member failed" word stay in h->d_gz_slab until the open has read that word back.
int bgzf_upload_inflate(frisk_b200_fasta* h, const Source& src, cudaStream_t alloc_st, cudaStream_t copy, unsigned int** d_any_bad) {
    const uint64_t nb = src.n_blocks;
    const uint64_t gz_bytes = (src.gz_n + 255) & ~255ull, tab_bytes = nb * 24;
    FRISK_CK(cudaMallocAsync(&h->d_gz_slab, gz_bytes + tab_bytes + nb * 4 + 256, alloc_st));
    char* const base = (char*)h->d_gz_slab;
    const uint64_t* const tab = (const uint64_t*)(base + gz_bytes);
    uint32_t* const status = (uint32_t*)(base + gz_bytes + tab_bytes);
    *d_any_bad = (unsigned int*)(status + nb);
    FRISK_CK(cudaMemsetAsync(*d_any_bad, 0, 4, alloc_st));
    cudaEvent_t ready;                                                  // (the slab exists in stream order)
    FRISK_CK(cudaEventCreateWithFlags(&ready, cudaEventDisableTiming));
    FRISK_CK(cudaEventRecord(ready, alloc_st));
    FRISK_CK(cudaStreamWaitEvent(copy, ready, 0));
    FRISK_CK(cudaEventDestroy(ready));
    FRISK_CK(cudaMemcpyAsync(base, src.gz, src.gz_n, cudaMemcpyHostToDevice, copy));
    FRISK_CK(cudaMemcpyAsync((void*)tab, src.table.data(), tab_bytes, cudaMemcpyHostToDevice, copy));
    const uint32_t* const t32 = (const uint32_t*)(tab + 2 * nb);
    return frisk_internal::bgzf_inflate((const uint8_t*)base, tab, t32, t32 + nb, tab + nb, nb, src.n, h->d_text, status, *d_any_bad, copy);
}

// The names of a BGZF handle: the header lines (hdr_pos[r] to their newline) are gathered on the device into one buffer that
// comes back in one copy; parse_header_name then reads it exactly as it reads the text of a text open.
int gather_names(frisk_b200_fasta* h, cudaStream_t st) {
    const uint64_t R = h->n_rec;
    h->name_text.clear();
    if (!R) return FRISK_OK;
    unsigned long long* d_off = nullptr;
    FRISK_CK(cudaMallocAsync((void**)&d_off, (R + 1) * 8, st));
    const unsigned grid = (unsigned)((R + 255) / 256);
    header_len_kernel<<<grid, 256, 0, st>>>(h->d_text, h->n, h->d_hdr_pos, R, d_off);
    header_scan_kernel<<<1, kST, 0, st>>>(d_off, R);
    FRISK_CK(cudaGetLastError());
    std::vector<uint64_t> off(R + 1);
    FRISK_CK(cudaMemcpyAsync(off.data(), d_off, (R + 1) * 8, cudaMemcpyDeviceToHost, st));
    FRISK_CK(cudaStreamSynchronize(st));
    const uint64_t total = off[R];
    uint8_t* d_lines = nullptr;
    FRISK_CK(cudaMallocAsync((void**)&d_lines, total + 1, st));
    header_gather_kernel<<<grid, 256, 0, st>>>(h->d_text, h->d_hdr_pos, d_off, R, d_lines);
    FRISK_CK(cudaGetLastError());
    h->name_text.resize(total);
    FRISK_CK(cudaMemcpyAsync(h->name_text.data(), d_lines, total, cudaMemcpyDeviceToHost, st));
    FRISK_CK(cudaFreeAsync(d_lines, st));
    FRISK_CK(cudaFreeAsync(d_off, st));
    FRISK_CK(cudaStreamSynchronize(st));
    const unsigned char* const t = reinterpret_cast<const unsigned char*>(h->name_text.data());
    for (uint64_t r = 0; r < R; ++r)
        if (!frisk_internal::parse_header_name(t, total, off[r], &h->name_off[r], &h->name_len[r])) return FRISK_E_FORMAT;
    return FRISK_OK;
}

// The open: text up, tokenised, laid out and packed.
// exact = false: the text goes up in chunks on a second stream and every chunk runs its three passes (summary, tile scan,
//   pack) while the next one is on the bus; record table and planes are sized by a guess (one record per 64 bytes of text +
//   4096 for the table; text bytes + 256 bases per KiB of text + 1 M bases for the planes), so the host synchronises once,
//   behind the last chunk's pack.  A line decision that needs a byte of a later chunk, or a text that outgrows the guesses,
//   returns kRetryExact.
// exact = true: one copy; summary + tile scan give the record count and the layout's length, the host reads them (one more
//   synchronisation), allocates exactly and runs the pack pass.  Cannot fail that way.
// sink (nullable, !exact only): sink->on_range is handed the plane words that became final with every chunk.
// BGZF source: the compressed bytes go up on the upload lane in one copy and one inflate launch fills the text buffer; the
// passes of every chunk wait on it (the whole text is there, so no line decision needs a later chunk), and the text is one
// chunk unless ingest_chunk_tiles asks for more.  The exact re-open takes over the text the first attempt inflated.
int open_impl(frisk_b200_fasta* h, const Source& src, cudaStream_t st, bool exact, frisk_internal::IngestSink* sink) {
    int rc = frisk_internal::pool_ready();
    if (rc) return rc;
    if (exact) sink = nullptr;
    const char* const text = src.text;
    const uint64_t n = src.n;
    h->n = n;
    h->device_text = src.device();
    unsigned int* d_any_bad = nullptr;                                  // BGZF: some member failed to inflate
    h->n_tiles = n ? (n + kTile - 1) / kTile : 0;
    if (h->n_tiles > 0x7fffffffull) return FRISK_E_UNSUPPORTED;         // 8 TB of text per call
    const uint64_t T = h->n_tiles;
    UploadLane* lane = nullptr;
    if ((rc = upload_lane(&lane))) return rc;
    std::lock_guard<std::mutex> one_open(lane->mu);
    constexpr size_t kCtrWords = kCtrCount + (size_t)kRangeSlots * kMaxChunks;
    const uint64_t Tp = (T + kSP - 1) / kSP * kSP;                      // the tile scan loads vectors of kSP tiles
    auto alloc_scan = [&]() -> int {   // one allocation for the counters and everything per tile
        const uint64_t bytes = 256 + kCtrWords * 8 + 6 * (Tp * 4 + 256) + 2 * (Tp + 256) + 2 * (Tp * 8 + 256);
        FRISK_CK(cudaMallocAsync(&h->d_scan_slab, bytes, st));
        char* cur = (char*)h->d_scan_slab;
        carve(cur, h->d_counters, kCtrWords * 8);
        carve(cur, h->d_nhdr, Tp * 4); carve(cur, h->d_head, Tp * 4); carve(cur, h->d_pre, Tp * 4);
        carve(cur, h->d_post, Tp * 4); carve(cur, h->d_inner, Tp * 4); carve(cur, h->d_rec_base, Tp * 4);
        carve(cur, h->d_key, Tp); carve(cur, h->d_carry, Tp);
        carve(cur, h->d_base_in, Tp * 8); carve(cur, h->d_open_off, Tp * 8);
        FRISK_CK(cudaMemsetAsync(h->d_counters, 0, kCtrWords * 8, st));
        return FRISK_OK;
    };
    uint64_t rec_cap = 0, plane_cap = 0;
    auto alloc_out = [&](uint64_t R, uint64_t P) -> int {              // record table of R entries, planes of P bases (zeroed)
        rec_cap = R; plane_cap = P;
        h->rec_cap = R;
        FRISK_CK(cudaMallocAsync(&h->d_out_slab, 3 * (R * 8 + 256) + P / 2 + 3 * 256, st));
        char* cur = (char*)h->d_out_slab;
        carve(cur, h->d_codes, P / 4); carve(cur, h->d_inv, P / 8); carve(cur, h->d_low, P / 8);
        FRISK_CK(cudaMemsetAsync(h->d_codes, 0, (size_t)(cur - (char*)h->d_codes), st));
        carve(cur, h->d_hdr_pos, R * 8); carve(cur, h->d_len, R * 8); carve(cur, h->d_scaf_off, R * 8);
        return FRISK_OK;
    };
    unsigned long long ctr[kCtrCount] = {};
    if (!T) {                                                           // no text: no record, 128 invalid bases
        if ((rc = alloc_scan())) return rc;
        if ((rc = alloc_out(1, 128))) return rc;
        FRISK_CK(cudaMemsetAsync(h->d_inv, 0xff, 128 / 8, st));
        h->padded_len = 128;
        if (src.n_blocks) {                                             // empty members only: still checked
            if ((rc = bgzf_upload_inflate(h, src, st, st, &d_any_bad))) return rc;
            if (sink && sink->uploaded_mark) FRISK_CK(cudaEventRecord(sink->uploaded_mark, st));
            unsigned int bad = 0;
            FRISK_CK(cudaMemcpyAsync(&bad, d_any_bad, 4, cudaMemcpyDeviceToHost, st));
            FRISK_CK(cudaStreamSynchronize(st));
            if (bad) return FRISK_E_FORMAT;
        } else if (src.gzip && sink && sink->uploaded_mark) {          // (inflated before the open)
            FRISK_CK(cudaEventRecord(sink->uploaded_mark, st));
        }
    } else {
        if (src.d_ready) h->d_text = src.d_ready;                      // (its padding is in place)
        else if ((rc = alloc_text(n, st, &h->d_text))) return rc;
        // Chunk plan (tile bounds, multiples of kSP): equal chunks of >= 1400 tiles (5.6 MiB; ingest_chunk_tiles overrides), at most
        // kMaxChunks.  Measured on C2 (40.8 MB, 52 GB/s over PCIe): beside a running H2D copy the three passes + count of a
        // chunk take about as long as the chunk's copy, and every launch of a short chunk costs ~10 us whatever its size, so
        // shorter chunks at the end do not shorten what is left after the last byte (0.12 ms with 3..8 chunks, more with 16);
        // counting every second chunk halves the count launches' fixed cost (128 KiB table per CTA zeroed, stored, reduced).
        // (Cutting the last chunk once more, 3 : 1, with a count of its own for the first part: +0.02 ms.)
        uint64_t bound[kMaxChunks + 1];
        bool count_at[kMaxChunks] = {};
        int n_chunks = 1;
        bound[0] = 0;
        if (!exact) {
            auto round_sp = [](uint64_t v) { return (v + kSP - 1) / kSP * kSP; };
            const uint64_t min_tiles = frisk_internal::g_ingest_chunk_tiles > 0 ? (uint64_t)frisk_internal::g_ingest_chunk_tiles : kMinChunkTiles;
            const uint64_t want = src.device() && frisk_internal::g_ingest_chunk_tiles <= 0
                                      ? 1 : std::max<uint64_t>(1, std::min<uint64_t>(kMaxChunks, T / min_tiles));
            const uint64_t per = round_sp((T + want - 1) / want);
            n_chunks = 0;
            for (uint64_t t0 = 0; t0 < T; t0 += per) bound[++n_chunks] = std::min<uint64_t>(t0 + per, T);
            for (int c = 0; c < n_chunks; ++c) count_at[c] = n_chunks <= 4 || (c & 1);
        }
        if (n_chunks == 1) bound[1] = T;
        bound[n_chunks] = T;
        count_at[n_chunks - 1] = true;
        const int last_chunk = n_chunks - 1;
        FRISK_CK(cudaEventRecord(lane->ready, st));                     // the text buffer exists (stream-ordered allocation)
        FRISK_CK(cudaStreamWaitEvent(lane->copy, lane->ready, 0));
        // FRISK_INGEST_TRACE=1: per-chunk event times (ms since the open began) on stderr -- diagnostic, costs a synchronisation
        static const bool trace = getenv("FRISK_INGEST_TRACE") != nullptr;
        std::vector<cudaEvent_t> tev;
        auto tmark = [&](cudaStream_t s2) {
            if (!trace) return;
            cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, s2); tev.push_back(e);
        };
        tmark(st);
        auto issue_copy = [&](int c) -> int {
            if (src.device()) return FRISK_OK;                          // (inflated already or below, all chunks at once)
            const uint64_t b0 = bound[c] * kTile, b1 = std::min<uint64_t>(bound[c + 1] * kTile, n);
            FRISK_CK(cudaMemcpyAsync(h->d_text + b0, text + b0, b1 - b0, cudaMemcpyHostToDevice, lane->copy));
            FRISK_CK(cudaEventRecord(lane->done[c], lane->copy));
            if (c == last_chunk && sink && sink->uploaded_mark) FRISK_CK(cudaEventRecord(sink->uploaded_mark, lane->copy));
            return FRISK_OK;
        };
        // page-locked text: every copy is queued before anything else is set up (the first byte leaves ~20 us earlier);
        // pageable text: a copy returns when its chunk is staged, so each one is issued just before its chunk's passes
        cudaPointerAttributes pa{};
        const bool pinned = !src.device() && cudaPointerGetAttributes(&pa, text) == cudaSuccess && pa.type == cudaMemoryTypeHost;
        cudaGetLastError();
        if (src.device()) {
            if (!src.d_ready && (rc = bgzf_upload_inflate(h, src, st, lane->copy, &d_any_bad))) return rc;
            for (int c = 0; c <= last_chunk; ++c) FRISK_CK(cudaEventRecord(lane->done[c], lane->copy));
            if (sink && sink->uploaded_mark) FRISK_CK(cudaEventRecord(sink->uploaded_mark, lane->copy));
        }
        if (pinned && !trace)
            for (int c = 0; c <= last_chunk; ++c)
                if ((rc = issue_copy(c))) return rc;
        if ((rc = alloc_scan())) return rc;
        if (!exact && (rc = alloc_out(n / 64 + 4096, ((n + 127) & ~127ull) + 256ull * (n / 1024 + 4096) + 256))) return rc;
        auto pack_pass = [&](uint64_t t0, uint64_t t1, uint64_t avail, bool final) {
            fasta_pack_kernel<<<(unsigned)(t1 - t0), kTT, 0, st>>>(h->d_text, n, t0, avail, T, (int)final, h->d_nhdr, h->d_rec_base,
                                                                    h->d_carry, h->d_base_in, h->d_open_off, h->d_counters, h->d_hdr_pos,
                                                                    h->d_len, h->d_scaf_off, rec_cap, h->d_codes, h->d_inv, h->d_low);
        };
        uint64_t counted_from = 0;
        for (int c = 0; c <= last_chunk; ++c) {
            const uint64_t t0 = bound[c], t1 = bound[c + 1];
            const uint64_t b1 = std::min<uint64_t>(t1 * kTile, n);
            const uint64_t avail = src.device() ? n : b1;               // bytes on the device when the chunk's passes run
            const bool final = c == last_chunk;
            if (!pinned || trace) {
                if ((rc = issue_copy(c))) return rc;
                tmark(lane->copy);
            }
            FRISK_CK(cudaStreamWaitEvent(st, lane->done[c], 0));
            unsigned long long* const d_range = h->d_counters + kCtrCount + (size_t)kRangeSlots * c;
            const bool count_now = sink && sink->on_range && count_at[c];
            fasta_summary_kernel<<<(unsigned)(t1 - t0), kTT, 0, st>>>(h->d_text, n, t0, avail, h->d_counters, h->d_nhdr, h->d_key, h->d_head,
                                                                       h->d_pre, h->d_post, h->d_inner);
            fasta_tilescan_kernel<<<1, kST, 0, st>>>(h->d_nhdr, h->d_key, h->d_head, h->d_pre, h->d_post, h->d_inner, t0, t1, h->d_rec_base,
                                                     h->d_carry, h->d_base_in, h->d_open_off, h->d_counters, d_range,
                                                     exact ? ~0ull : rec_cap, exact ? ~0ull : plane_cap, (int)count_now, (int)final);
            tmark(st);
            if (!exact) pack_pass(t0, t1, avail, final);
            tmark(st);
            FRISK_CK(cudaGetLastError());
            if (final && !exact) {                                      // the record table is complete: the host can have it now,
                FRISK_CK(cudaEventRecord(lane->ready, st));             // while the last chunk is still being counted
                FRISK_CK(cudaStreamWaitEvent(lane->copy, lane->ready, 0));
            }
            if (count_now) {
                if ((rc = sink->on_range(h->d_codes, h->d_inv, h->d_low, d_range, ((b1 - counted_from) >> 5) + 8, st))) return rc;
                counted_from = b1;
            }
            if (final && sink && sink->on_complete && (rc = sink->on_complete(h, st))) return rc;
            tmark(st);
        }
        if (trace) {
            cudaStreamSynchronize(st); cudaStreamSynchronize(lane->copy);
            fprintf(stderr, "ingest trace (%d chunks): chunk [tiles] copied | summary+scan | pack | count  (ms)\n", n_chunks);
            for (int c = 0; c <= last_chunk; ++c) {
                float t[4];
                for (int j = 0; j < 4; ++j) cudaEventElapsedTime(&t[j], tev[0], tev[1 + 4 * c + j]);
                fprintf(stderr, "  %2d [%6llu] %.3f | %.3f | %.3f | %.3f\n", c, (unsigned long long)(bound[c + 1] - bound[c]), t[0], t[1], t[2], t[3]);
            }
            for (auto e : tev) cudaEventDestroy(e);
        }
        cudaStream_t back = lane->copy;                                 // the stream the record table comes back on
        if (exact) {
            FRISK_CK(cudaMemcpyAsync(ctr, h->d_counters, kCtrCount * 8, cudaMemcpyDeviceToHost, st));
            FRISK_CK(cudaStreamSynchronize(st));
            if ((rc = alloc_out(ctr[kCtrRecords] ? ctr[kCtrRecords] : 1, ctr[kLayPaddedLen]))) return rc;
            pack_pass(0, T, n, true);
            FRISK_CK(cudaGetLastError());
            back = st;
        }
        // counters and the first records land in page-locked memory (a pageable destination makes every copy a blocking,
        // staged one): three copies queued, one synchronisation
        const uint64_t first = std::min<uint64_t>(rec_cap, kFirstFetch);
        unsigned long long* const sg = lane->stage;
        FRISK_CK(cudaMemcpyAsync(sg, h->d_len, first * 8, cudaMemcpyDeviceToHost, back));
        FRISK_CK(cudaMemcpyAsync(sg + kFirstFetch, h->d_hdr_pos, first * 8, cudaMemcpyDeviceToHost, back));
        FRISK_CK(cudaMemcpyAsync(sg + 2 * kFirstFetch, h->d_counters, kCtrCount * 8, cudaMemcpyDeviceToHost, back));
        sg[2 * kFirstFetch + kCtrCount] = 0;
        if (d_any_bad) FRISK_CK(cudaMemcpyAsync(sg + 2 * kFirstFetch + kCtrCount, d_any_bad, 4, cudaMemcpyDeviceToHost, back));
        FRISK_CK(cudaStreamSynchronize(back));
        memcpy(ctr, sg + 2 * kFirstFetch, kCtrCount * 8);
        if (sg[2 * kFirstFetch + kCtrCount]) return FRISK_E_FORMAT;    // a BGZF member is not valid deflate or fails its CRC
        if (!exact && (ctr[kCtrAmbig] || ctr[kCtrOverflow])) return kRetryExact;
        if (ctr[kCtrWhitespace]) return FRISK_E_FORMAT;                // whitespace inside a sequence line
        const uint64_t n_rec = ctr[kCtrRecords];
        h->n_rec = n_rec;
        h->seq_len.resize(n_rec);
        h->hdr_pos.resize(n_rec);
        memcpy(h->seq_len.data(), sg, std::min<uint64_t>(first, n_rec) * 8);
        memcpy(h->hdr_pos.data(), sg + kFirstFetch, std::min<uint64_t>(first, n_rec) * 8);
        if (n_rec > first) {
            FRISK_CK(cudaMemcpyAsync(h->seq_len.data() + first, h->d_len + first, (n_rec - first) * 8, cudaMemcpyDeviceToHost, back));
            FRISK_CK(cudaMemcpyAsync(h->hdr_pos.data() + first, h->d_hdr_pos + first, (n_rec - first) * 8, cudaMemcpyDeviceToHost, back));
            FRISK_CK(cudaStreamSynchronize(back));
        }
        h->stats[1] = ctr[kCtrNonUpper];
        h->stats[2] = ctr[kCtrLower];
        h->padded_len = ctr[kLayPaddedLen];                            // (checked against the host's layout below)
    }
    // names (F:156) and the 128-base aligned layout
    const uint64_t R = h->n_rec;
    h->name_off.resize(R); h->name_len.resize(R); h->scaf_off.resize(R);
    if (src.device()) {
        if (h->d_gz_slab) FRISK_CK(cudaFreeAsync(h->d_gz_slab, st));    // (the inflate is behind the synchronisation above)
        h->d_gz_slab = nullptr;
        // beside the tail run_fasta may have queued on `st`: on the upload lane, which follows the last chunk's pack
        if ((rc = gather_names(h, exact || !T ? st : lane->copy))) return rc;
    } else {
        const unsigned char* tt = reinterpret_cast<const unsigned char*>(text);
        for (uint64_t r = 0; r < R; ++r)
            if (!frisk_internal::parse_header_name(tt, n, h->hdr_pos[r], &h->name_off[r], &h->name_len[r])) return FRISK_E_FORMAT;
    }
    uint64_t total = 0;
    for (uint64_t r = 0; r < R; ++r) total += h->seq_len[r];
    h->stats[0] = total;
    const uint64_t device_padded = h->padded_len;
    rc = frisk_b200_pack_layout(h->seq_len.data(), R, h->scaf_off.data(), &h->padded_len);
    if (rc) return rc;
    if (device_padded != h->padded_len) return exact ? FRISK_E_CUDA : kRetryExact;   // (cannot happen: both sides apply one rule)
    if (sink) sink->counted = (bool)sink->on_range;
    h->streamed = !exact;
    return FRISK_OK;
}

// open with retry
int open_any(frisk_b200_fasta* h, Source& src, cudaStream_t st, frisk_internal::IngestSink* sink) {
    const bool exact = frisk_internal::g_ingest_exact != 0;
    if (sink) sink->counted = false;
    int rc = open_impl(h, src, st, exact, sink);
    if (rc == FRISK_OK && !exact) g_open_stats[0].fetch_add(1);
    if (rc == kRetryExact) {
        g_open_stats[1].fetch_add(1);
        FRISK_CK(cudaStreamSynchronize(st));                            // (the abandoned attempt's work targets what is freed next)
        if (sink && sink->abandon && (rc = sink->abandon(st))) return rc;
        if (src.device()) { src.d_ready = h->d_text; h->d_text = nullptr; }   // inflated once: the re-open keeps the text
        if ((rc = free_all(h, st))) return rc;
        *h = frisk_b200_fasta();
        rc = open_impl(h, src, st, true, nullptr);
        if (!h->d_text && src.d_ready) FRISK_CK(cudaFreeAsync(src.d_ready, st));   // (not taken over)
        src.d_ready = nullptr;
        if (sink) sink->counted = false;
    }
    return rc;
}

// the public opens and the one-call path: block table (BGZF) or inflate (gzip), open with retry; no handle on failure
int open_handle(const char* text, uint64_t n, frisk_internal::TextFormat fmt, cudaStream_t st, frisk_internal::IngestSink* sink,
                frisk_b200_fasta** out) {
    *out = nullptr;
    frisk_b200_fasta* h = new (std::nothrow) frisk_b200_fasta();
    if (!h) return FRISK_E_INVALID;
    int rc;
    if (fmt == frisk_internal::kFmt2bit) {                // planes decoded by frisk_twobit.cu, handle made by fasta_adopt
        delete h;
        try {
            return frisk_internal::twobit_open(text, n, st, sink, out);
        } catch (...) {
            return FRISK_E_CAPACITY;
        }
    }
    Source src;
    try {                                                 // std::bad_alloc of the record table: nothing crosses the ABI
        rc = make_source(text, n, fmt, st, &src);
        if (!rc) rc = open_any(h, src, st, sink);
    } catch (...) {
        rc = FRISK_E_CAPACITY;
    }
    if (src.d_ready && h->d_text != src.d_ready) cudaFreeAsync(src.d_ready, st);   // gzip: a text the handle did not take
    if (rc) {
        free_all(h, st);
        delete h;
        return rc;
    }
    *out = h;
    return FRISK_OK;
}

// frisk_b200_fasta_open, _open_bgzf and _open_gzip
int open_public(const char* text, uint64_t n, frisk_internal::TextFormat fmt, void* stream, frisk_b200_fasta** out, uint64_t* n_records,
                uint64_t* padded_len, uint64_t stats[3]) {
    if (!out || (!text && n)) return FRISK_E_INVALID;
    *out = nullptr;
    if (frisk_b200_device_count() <= 0) return FRISK_E_NO_DEVICE;
    frisk_b200_fasta* h = nullptr;
    const int rc = open_handle(text, n, fmt, (cudaStream_t)stream, nullptr, &h);
    if (rc) return rc;
    if (n_records) *n_records = h->n_rec;
    if (padded_len) *padded_len = h->padded_len;
    if (stats) { stats[0] = h->stats[0]; stats[1] = h->stats[1]; stats[2] = h->stats[2]; }
    *out = h;
    return FRISK_OK;
}

// fasta_adopt behind the take-over: on_range over every word, the counters back on the upload lane beside on_complete's work
int adopt_finish(frisk_b200_fasta* h, cudaStream_t st, frisk_internal::IngestSink* sink) {
    UploadLane* lane = nullptr;
    int rc = upload_lane(&lane);
    if (rc) return rc;
    std::lock_guard<std::mutex> one_open(lane->mu);
    FRISK_CK(cudaEventRecord(lane->ready, st));                         // the planes and counters are final here
    FRISK_CK(cudaStreamWaitEvent(lane->copy, lane->ready, 0));
    FRISK_CK(cudaMemcpyAsync(lane->stage, h->d_counters, frisk_internal::kIngestCounters * 8, cudaMemcpyDeviceToHost, lane->copy));
    if (sink && sink->on_range &&
        (rc = sink->on_range(h->d_codes, h->d_inv, h->d_low, h->d_counters + frisk_internal::kIngestRange, h->padded_len / 32, st)))
        return rc;
    if (sink && sink->on_complete && (rc = sink->on_complete(h, st))) return rc;
    FRISK_CK(cudaStreamSynchronize(lane->copy));
    h->stats[1] = lane->stage[kCtrNonUpper];
    h->stats[2] = lane->stage[kCtrLower];
    if (sink) sink->counted = (bool)sink->on_range;
    return FRISK_OK;
}
}  // namespace

int frisk_internal::fasta_adopt(AdoptedGenome& g, cudaStream_t st, IngestSink* sink, frisk_b200_fasta** out) {
    *out = nullptr;
    if (sink) sink->counted = false;
    frisk_b200_fasta* h = new (std::nothrow) frisk_b200_fasta();
    if (!h) {
        cudaFreeAsync(g.d_slab, st);
        return FRISK_E_CAPACITY;
    }
    h->d_out_slab = g.d_slab;
    g.d_slab = nullptr;
    h->d_codes = g.d_codes; h->d_inv = g.d_inv; h->d_low = g.d_low;
    h->d_len = g.d_len; h->d_scaf_off = g.d_scaf_off; h->d_counters = g.d_counters;
    h->rec_cap = g.rec_cap;
    h->n_rec = g.seq_len.size();
    h->padded_len = g.padded_len;
    h->stats[0] = g.total;
    h->name_off = std::move(g.name_off); h->name_len = std::move(g.name_len);
    h->seq_len = std::move(g.seq_len); h->scaf_off = std::move(g.scaf_off);
    h->name_text = std::move(g.name_text);
    h->device_text = true;                                             // the names index the handle's buffer
    h->streamed = true;                                                // what on_complete queued ran on the final table
    const int rc = adopt_finish(h, st, sink);
    if (rc) {
        free_all(h, st);
        delete h;
        return rc;
    }
    *out = h;
    return FRISK_OK;
}

bool frisk_internal::fasta_open_was_streamed(const frisk_b200_fasta* h) { return h && h->streamed; }

int frisk_internal::fasta_open_planes(const char* text, uint64_t n, TextFormat fmt, cudaStream_t st, IngestSink* sink,
                                      frisk_b200_fasta** out) {
    if (!out || !sink || (!text && n)) return FRISK_E_INVALID;
    return open_handle(text, n, fmt, st, sink, out);
}

int frisk_internal::fasta_device_table(const frisk_b200_fasta* h, const unsigned long long** d_len, const unsigned long long** d_scaf_off,
                                       const unsigned long long** d_counters, uint64_t* rec_cap, const uint32_t** d_codes,
                                       const uint32_t** d_inv, const uint32_t** d_low) {
    if (!h || !h->d_counters || !h->d_len || !h->d_codes) return FRISK_E_INVALID;
    *d_len = h->d_len; *d_scaf_off = h->d_scaf_off; *d_counters = h->d_counters; *rec_cap = h->rec_cap;
    *d_codes = h->d_codes; *d_inv = h->d_inv; *d_low = h->d_low;
    return FRISK_OK;
}

extern "C" {

int frisk_b200_fasta_info(const frisk_b200_fasta* h, uint64_t* n_records, uint64_t* padded_len, uint64_t stats[3]) {
    if (!h) return FRISK_E_INVALID;
    if (n_records) *n_records = h->n_rec;
    if (padded_len) *padded_len = h->padded_len;
    if (stats) { stats[0] = h->stats[0]; stats[1] = h->stats[1]; stats[2] = h->stats[2]; }
    return FRISK_OK;
}

int frisk_b200_fasta_open(const char* text, uint64_t n, void* stream, frisk_b200_fasta** out, uint64_t* n_records,
                          uint64_t* padded_len, uint64_t stats[3]) {
    return open_public(text, n, frisk_internal::kFmtText, stream, out, n_records, padded_len, stats);
}

int frisk_b200_fasta_open_bgzf(const char* gz, uint64_t n, void* stream, frisk_b200_fasta** out, uint64_t* n_records,
                               uint64_t* padded_len, uint64_t stats[3]) {
    return open_public(gz, n, frisk_internal::kFmtBgzf, stream, out, n_records, padded_len, stats);
}

int frisk_b200_fasta_open_gzip(const char* gz, uint64_t n, void* stream, frisk_b200_fasta** out, uint64_t* n_records,
                               uint64_t* padded_len, uint64_t stats[3]) {
    return open_public(gz, n, frisk_internal::kFmtGzip, stream, out, n_records, padded_len, stats);
}

int frisk_b200_fasta_open_2bit(const char* buf, uint64_t n, void* stream, frisk_b200_fasta** out, uint64_t* n_records,
                               uint64_t* padded_len, uint64_t stats[3]) {
    return open_public(buf, n, frisk_internal::kFmt2bit, stream, out, n_records, padded_len, stats);
}

int frisk_b200_fasta_name_text(const frisk_b200_fasta* h, const char** text, uint64_t* n) {
    if (!h || !text || !n) return FRISK_E_INVALID;
    *text = h->device_text ? h->name_text.data() : nullptr;
    *n = h->device_text ? h->name_text.size() : 0;
    return FRISK_OK;
}

int frisk_b200_fasta_records(const frisk_b200_fasta* h, uint64_t* name_off, uint32_t* name_len, uint64_t* seq_len,
                             uint64_t* scaf_off) {
    if (!h) return FRISK_E_INVALID;
    const size_t R = (size_t)h->n_rec;
    if (name_off && R) memcpy(name_off, h->name_off.data(), R * 8);
    if (name_len && R) memcpy(name_len, h->name_len.data(), R * 4);
    if (seq_len && R) memcpy(seq_len, h->seq_len.data(), R * 8);
    if (scaf_off && R) memcpy(scaf_off, h->scaf_off.data(), R * 8);
    return FRISK_OK;
}

int frisk_b200_fasta_pack(frisk_b200_fasta* h, uint32_t* d_codes, uint32_t* d_inv, uint32_t* d_low, void* stream) {
    if (!h || !d_codes || !d_inv || !h->d_codes) return FRISK_E_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    const uint64_t P = h->padded_len;                                   // the planes exist since the open: hand out copies
    FRISK_CK(cudaMemcpyAsync(d_codes, h->d_codes, P / 4, cudaMemcpyDeviceToDevice, st));
    FRISK_CK(cudaMemcpyAsync(d_inv, h->d_inv, P / 8, cudaMemcpyDeviceToDevice, st));
    if (d_low) FRISK_CK(cudaMemcpyAsync(d_low, h->d_low, P / 8, cudaMemcpyDeviceToDevice, st));
    return FRISK_OK;
}

int frisk_b200_fasta_planes(const frisk_b200_fasta* h, const uint32_t** d_codes, const uint32_t** d_inv, const uint32_t** d_low) {
    if (!h || !h->d_codes) return FRISK_E_INVALID;
    if (d_codes) *d_codes = h->d_codes;
    if (d_inv) *d_inv = h->d_inv;
    if (d_low) *d_low = h->stats[2] ? h->d_low : nullptr;            // no lower-case base: no plane (as frisk_b200_pack reports it)
    return FRISK_OK;
}

int frisk_b200_fasta_open_stats(uint64_t out[2]) {
    if (!out) return FRISK_E_INVALID;
    out[0] = g_open_stats[0].load();
    out[1] = g_open_stats[1].load();
    return FRISK_OK;
}

int frisk_b200_fasta_close(frisk_b200_fasta* h, void* stream) {
    if (!h) return FRISK_OK;
    const int rc = free_all(h, (cudaStream_t)stream);
    delete h;
    return rc;
}

}  // extern "C"
