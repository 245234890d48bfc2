// frisk_b200 BGZF inflate: blocked gzip (the format bgzip writes and samtools faidx requires) in, text out, on the GPU.
//
// A BGZF file is a series of gzip members of at most 64 KiB each, compressed and inflated.  Every member carries its own
// compressed size in the header (the "BC" extra subfield) and its CRC32 and inflated size in the trailer, so one host pass
// that hops from header to header (frisk_b200_bgzf_blocks) gives every member's input range and output offset before
// anything is decoded, and every member can be inflated by a decoder of its own.
//
// One warp per member (bgzf_inflate_kernel).  Huffman decoding is a serial bit chain, so lane 0 decodes a batch of up to
// kMaxTok tokens (literal, or length + distance) with lookup tables in shared memory; the warp then materialises the batch:
// a prefix sum of the token lengths gives every token's place, the lanes copy the batch's bytes out of a shared-memory
// history ring that holds deflate's whole 32 KiB window, and the same bytes go to the output as coalesced stores.  A match
// whose source overlaps the batch's own output is copied after the rest, in token order.  When the member is done, each
// lane computes the CRC32 of a slice of its output and lane 0 folds the 32 partial CRCs with x^(8n) mod P.
//
// The bit reader, the table construction and the token decoder are __host__ __device__ (struct Inflater, decode_batch):
// frisk_b200_bgzf_inflate_host runs the same code on the CPU, so that the decoder's logic and its bounds checks are tested
// on machines without a GPU.  No user path calls it.
//
// Safety: every read is bounded by the member's compressed length (bytes past it read as zero and the overrun is an
// error), every write by its inflated size, and every loop by input bits or output bytes.  Malformed input sets the
// member's status word (kSt*) and is never scored.
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <memory>
#include <new>

#include "../../include/frisk_b200.h"
#include "frisk_internal.h"

#define FRISK_HD __host__ __device__ __forceinline__

namespace {

constexpr uint32_t kWindow = 32768;          // deflate's longest distance
constexpr uint32_t kBatchBytes = 4096;       // output bytes of one batch at most
constexpr uint32_t kRing = kWindow + kBatchBytes;   // every source of a batch survives the batch's own writes
constexpr uint32_t kInBuf = 2048;            // staged compressed bytes (a batch reads < 200, a block header < 600)
constexpr int kMaxTok = 32;
constexpr int kLitBits = 10, kDistBits = 8;  // primary lookup tables; longer codes take the canonical walk
constexpr uint32_t kMaxIsize = 65536;

// per-member status (0 = inflated, size and CRC32 match)
enum : uint32_t {
    kStOk = 0,
    kStBlockType = 1,      // BTYPE 3
    kStBadCode = 2,        // over-subscribed or (where zlib refuses it) incomplete code, too many length/distance codes,
                           // a repeat with no previous length, a code-length run past the end, no end-of-block code
    kStBadSymbol = 3,      // a code that is not in the table, litlen 286/287, distance 30/31
    kStDistance = 4,       // a distance before the member's first byte
    kStStored = 5,         // stored LEN != ~NLEN
    kStOutput = 6,         // output beyond ISIZE
    kStInput = 7,          // the deflate stream runs past the member's payload, or ends before its last byte
    kStSize = 8,           // fewer bytes than ISIZE
    kStCrc = 9,            // CRC32 mismatch
    kStTable = 10,         // block table inconsistent (ISIZE > 64 KiB, output past text_len)
};

enum : int { kPhHeader = 0, kPhHuff = 1, kPhStored = 2, kPhDone = 3 };

// base | extra bits << 16 of the length symbols 257..285 and the distance symbols 0..29
#define FRISK_LEN_CODES                                                                                                   \
    {3, 4, 5, 6, 7, 8, 9, 10, 11 | 1 << 16, 13 | 1 << 16, 15 | 1 << 16, 17 | 1 << 16, 19 | 2 << 16, 23 | 2 << 16,         \
     27 | 2 << 16, 31 | 2 << 16, 35 | 3 << 16, 43 | 3 << 16, 51 | 3 << 16, 59 | 3 << 16, 67 | 4 << 16, 83 | 4 << 16,     \
     99 | 4 << 16, 115 | 4 << 16, 131 | 5 << 16, 163 | 5 << 16, 195 | 5 << 16, 227 | 5 << 16, 258}
#define FRISK_DIST_CODES                                                                                                  \
    {1, 2, 3, 4, 5 | 1 << 16, 7 | 1 << 16, 9 | 2 << 16, 13 | 2 << 16, 17 | 3 << 16, 25 | 3 << 16, 33 | 4 << 16,         \
     49 | 4 << 16, 65 | 5 << 16, 97 | 5 << 16, 129 | 6 << 16, 193 | 6 << 16, 257 | 7 << 16, 385 | 7 << 16,             \
     513 | 8 << 16, 769 | 8 << 16, 1025 | 9 << 16, 1537 | 9 << 16, 2049 | 10 << 16, 3073 | 10 << 16, 4097 | 11 << 16,   \
     6145 | 11 << 16, 8193 | 12 << 16, 12289 | 12 << 16, 16385 | 13 << 16, 24577 | 13 << 16}
__constant__ uint32_t c_len_code[29] = FRISK_LEN_CODES;
__constant__ uint32_t c_dist_code[30] = FRISK_DIST_CODES;
#ifndef __CUDA_ARCH__
const uint32_t h_len_code[29] = FRISK_LEN_CODES;
const uint32_t h_dist_code[30] = FRISK_DIST_CODES;
#endif

FRISK_HD uint32_t len_code(int i) {
#ifdef __CUDA_ARCH__
    return c_len_code[i];
#else
    return h_len_code[i];
#endif
}
FRISK_HD uint32_t dist_code(int i) {
#ifdef __CUDA_ARCH__
    return c_dist_code[i];
#else
    return h_dist_code[i];
#endif
}

// A decoder's shared memory (42.7 KB: five decoders fit an SM).  The ring doubles as the CRC table once decoding is done.
struct Inflater {
    uint8_t ring[kRing];                     // output position p lives at ring[p % kRing]
    uint8_t in[kInBuf];                      // compressed byte x lives at in[x % kInBuf]
    uint16_t lit_fast[1 << kLitBits];        // symbol | length << 9 for codes <= kLitBits; 0: canonical walk
    uint16_t dist_fast[1 << kDistBits];
    uint16_t lit_count[16], dist_count[16];  // codes of every length
    uint16_t lit_sym[288], dist_sym[32];     // symbols in canonical order
    uint8_t lens[288 + 32];                  // code lengths of a dynamic block
    uint32_t tok[kMaxTok];                   // distance << 16 | length (distance 0: a literal, the byte in the low bits)
    uint32_t tok_pos[kMaxTok + 1];           // the batch's exclusive prefix sum of token lengths
};

// lane 0's registers
struct Dec {
    uint64_t bb;          // bit buffer, next bit in bit 0
    uint32_t bc;          // bits in bb
    uint32_t pos;         // next compressed byte to load into bb
    uint32_t len;         // compressed bytes of the member
    uint32_t isize, out;  // bytes promised by the trailer / produced so far
    uint32_t stored_left;
    int phase;
    bool last;            // the block being decoded has BFINAL set
    uint32_t status;
};

FRISK_HD void dec_init(Dec& d, uint32_t len, uint32_t isize) {
    d.bb = 0; d.bc = 0; d.pos = 0; d.len = len; d.isize = isize; d.out = 0; d.stored_left = 0;
    d.phase = kPhHeader; d.last = false; d.status = kStOk;
}

// fills bb to >= 57 bits; bytes past the payload read as zero (bits_overrun catches their use)
FRISK_HD void refill(const Inflater& S, Dec& d) {
    while (d.bc <= 56) {
        const uint64_t x = d.pos < d.len ? S.in[d.pos % kInBuf] : 0u;
        d.bb |= x << d.bc;
        d.bc += 8;
        ++d.pos;
    }
}
FRISK_HD uint32_t bits(Dec& d, uint32_t n) {     // n <= 32, bb holds them
    const uint32_t v = (uint32_t)(d.bb & ((1ull << n) - 1ull));
    d.bb >>= n;
    d.bc -= n;
    return v;
}
FRISK_HD bool bits_overrun(const Dec& d) { return (uint64_t)d.pos * 8u - d.bc > (uint64_t)d.len * 8u; }

// Canonical code from lengths (as zlib's inflate_table decides): counts, symbols in canonical order, primary table.
// kind 0: code-length code (an incomplete code is refused), 1: litlen / distance (incomplete only with one code of length 1,
// an empty code is accepted and fails when used).  Returns false for a code zlib refuses.
FRISK_HD bool build_code(const uint8_t* lens, int n, uint16_t* count, uint16_t* sym, uint16_t* fast, int fast_bits, int kind) {
    for (int l = 0; l < 16; ++l) count[l] = 0;
    for (int s = 0; s < n; ++s) ++count[lens[s]];
    count[0] = 0;
    int left = 1, max = 0;
    for (int l = 1; l < 16; ++l) {
        left <<= 1;
        left -= count[l];
        if (left < 0) return false;                      // over-subscribed
        if (count[l]) max = l;
    }
    if (left > 0 && max != 0 && (kind == 0 || max != 1)) return false;   // incomplete
    uint16_t offs[16];
    offs[1] = 0;
    for (int l = 1; l < 15; ++l) offs[l + 1] = offs[l] + count[l];
    for (int s = 0; s < n; ++s)
        if (lens[s]) sym[offs[lens[s]]++] = (uint16_t)s;
    if (fast) {
        const int size = 1 << fast_bits;
        for (int i = 0; i < size; ++i) fast[i] = 0;
        uint32_t code = 0;
        int idx = 0;
        for (int l = 1; l <= fast_bits; ++l) {           // codes of length l: consecutive, in canonical symbol order
            for (int k = 0; k < count[l]; ++k, ++idx, ++code) {
                uint32_t rev = 0;                         // deflate sends codes most significant bit first
                for (int b = 0; b < l; ++b) rev |= ((code >> b) & 1u) << (l - 1 - b);
                for (uint32_t f = rev; f < (uint32_t)size; f += 1u << l) fast[f] = (uint16_t)(sym[idx] | (l << 9));
            }
            code <<= 1;
        }
    }
    return true;
}

// one symbol; -1 if the bits are no code of the table
FRISK_HD int decode_sym(Dec& d, const uint16_t* count, const uint16_t* sym, const uint16_t* fast, int fast_bits) {
    if (fast) {
        const uint16_t e = fast[d.bb & ((1u << fast_bits) - 1u)];
        if (e >> 9) {
            bits(d, e >> 9);
            return e & 511;
        }
    }
    int code = 0, first = 0, index = 0;                  // canonical walk, one bit at a time (puff's decode)
    for (int l = 1; l < 16; ++l) {
        code |= (int)((d.bb >> (l - 1)) & 1u);
        const int c = count[l];
        if (code - c < first) {
            bits(d, l);
            return sym[index + (code - first)];
        }
        index += c;
        first = (first + c) << 1;
        code <<= 1;
    }
    return -1;
}

FRISK_HD uint32_t fail(Dec& d, uint32_t st) {
    d.status = st;
    d.phase = kPhDone;
    return st;
}

// a block header: BFINAL, BTYPE, and the stored length or the Huffman tables
FRISK_HD void block_header(Inflater& S, Dec& d) {
    refill(S, d);
    d.last = bits(d, 1) != 0u;
    const uint32_t type = bits(d, 2);
    if (type == 0) {
        bits(d, d.bc & 7u);                               // to the byte boundary
        const uint32_t ln = bits(d, 16), nln = bits(d, 16);
        if (ln != (~nln & 0xffffu)) { fail(d, kStStored); return; }
        if (ln > d.isize - d.out) { fail(d, kStOutput); return; }
        d.stored_left = ln;
        d.phase = kPhStored;
    } else if (type == 1) {
        for (int s = 0; s < 288; ++s) S.lens[s] = s < 144 ? 8 : (s < 256 ? 9 : (s < 280 ? 7 : 8));
        for (int s = 0; s < 32; ++s) S.lens[288 + s] = 5;      // 30 and 31 have codes; decoding them is an error
        build_code(S.lens, 288, S.lit_count, S.lit_sym, S.lit_fast, kLitBits, 1);
        build_code(S.lens + 288, 32, S.dist_count, S.dist_sym, S.dist_fast, kDistBits, 1);
        d.phase = kPhHuff;
    } else if (type == 2) {
        const int nlen = (int)bits(d, 5) + 257, ndist = (int)bits(d, 5) + 1, ncode = (int)bits(d, 4) + 4;
        if (nlen > 286 || ndist > 30) { fail(d, kStBadCode); return; }
        constexpr uint8_t order[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
        uint8_t cl[19];
        for (int i = 0; i < 19; ++i) cl[i] = 0;
        refill(S, d);
        for (int i = 0; i < ncode; ++i) cl[order[i]] = (uint8_t)bits(d, 3);
        uint16_t cl_count[16], cl_sym[19];
        if (!build_code(cl, 19, cl_count, cl_sym, nullptr, 0, 0)) { fail(d, kStBadCode); return; }
        int i = 0;
        while (i < nlen + ndist) {                        // every step writes >= 1 length
            refill(S, d);
            if (bits_overrun(d)) { fail(d, kStInput); return; }
            const int s = decode_sym(d, cl_count, cl_sym, nullptr, 0);
            if (s < 0) { fail(d, kStBadCode); return; }
            if (s < 16) { S.lens[i++] = (uint8_t)s; continue; }
            uint8_t v = 0;
            int rep;
            if (s == 16) {
                if (i == 0) { fail(d, kStBadCode); return; }     // a repeat with no previous length
                v = S.lens[i - 1];
                rep = 3 + (int)bits(d, 2);
            } else if (s == 17) rep = 3 + (int)bits(d, 3);
            else rep = 11 + (int)bits(d, 7);
            if (i + rep > nlen + ndist) { fail(d, kStBadCode); return; }
            while (rep--) S.lens[i++] = v;
        }
        if (bits_overrun(d)) { fail(d, kStInput); return; }
        if (S.lens[256] == 0) { fail(d, kStBadCode); return; }     // no end-of-block code
        // (the distance lengths move behind the 288 litlen slots; nlen <= 286 keeps the copy from overlapping itself)
        for (int k = ndist - 1; k >= 0; --k) S.lens[288 + k] = S.lens[nlen + k];
        for (int k = nlen; k < 288; ++k) S.lens[k] = 0;
        if (!build_code(S.lens, 288, S.lit_count, S.lit_sym, S.lit_fast, kLitBits, 1) ||
            !build_code(S.lens + 288, ndist, S.dist_count, S.dist_sym, S.dist_fast, kDistBits, 1)) {
            fail(d, kStBadCode);
            return;
        }
        d.phase = kPhHuff;
    } else {
        fail(d, kStBlockType);
    }
}

// Lane 0's part: decode the next batch into S.tok (a block header first when one is due).  Returns the number of tokens;
// sets d.phase to kPhDone at the end of the member or on an error (d.status).  Consumes input bits whenever it returns
// with the member unfinished, so that the caller's loop is bounded by the member's bits.
FRISK_HD int decode_batch(Inflater& S, Dec& d) {
    if (d.phase == kPhHeader) {
        block_header(S, d);
        if (d.phase == kPhDone) return 0;
        if (bits_overrun(d)) { fail(d, kStInput); return 0; }
    }
    int nt = 0;
    uint32_t bytes = 0;
    while (nt < kMaxTok && bytes + 258u <= kBatchBytes) {
        refill(S, d);
        if (d.phase == kPhStored) {
            if (d.stored_left == 0) { d.phase = kPhHeader; break; }
            S.tok[nt++] = bits(d, 8);
            ++bytes;
            ++d.out;
            --d.stored_left;
            continue;
        }
        const int s = decode_sym(d, S.lit_count, S.lit_sym, S.lit_fast, kLitBits);
        if (s < 0 || s > 285) { fail(d, kStBadSymbol); break; }
        if (s < 256) {
            if (d.out >= d.isize) { fail(d, kStOutput); break; }
            S.tok[nt++] = (uint32_t)s;
            ++bytes;
            ++d.out;
        } else if (s == 256) {
            d.phase = kPhHeader;
            break;
        } else {
            const uint32_t lc = len_code(s - 257);
            const uint32_t ln = (lc & 0xffffu) + bits(d, lc >> 16);
            const int ds = decode_sym(d, S.dist_count, S.dist_sym, S.dist_fast, kDistBits);
            if (ds < 0 || ds > 29) { fail(d, kStBadSymbol); break; }
            const uint32_t dc = dist_code(ds);
            const uint32_t dist = (dc & 0xffffu) + bits(d, dc >> 16);
            if (dist > d.out) { fail(d, kStDistance); break; }
            if (ln > d.isize - d.out) { fail(d, kStOutput); break; }
            S.tok[nt++] = dist << 16 | ln;
            bytes += ln;
            d.out += ln;
        }
        if (bits_overrun(d)) { fail(d, kStInput); break; }
    }
    if (d.status == kStOk && bits_overrun(d)) fail(d, kStInput);
    if (d.status == kStOk && d.phase == kPhHeader && d.last) {
        d.phase = kPhDone;                                 // the final block ended: the payload must end in this byte
        const uint64_t used = (uint64_t)d.pos * 8u - d.bc;
        if ((used + 7u) / 8u != d.len) fail(d, kStInput);
        else if (d.out != d.isize) fail(d, kStSize);
    }
    return nt;
}

FRISK_HD uint32_t tok_len(uint32_t t) { return (t >> 16) ? (t & 0xffffu) : 1u; }

// ---- CRC32 (zlib's polynomial) and the fold of partial CRCs ---------------------------------------------------------------
constexpr uint32_t kPoly = 0xedb88320u;

FRISK_HD uint32_t crc_table_entry(uint32_t i) {
    uint32_t c = i;
    for (int k = 0; k < 8; ++k) c = (c & 1u) ? (c >> 1) ^ kPoly : c >> 1;
    return c;
}
FRISK_HD uint32_t crc_bytes(const uint32_t* table, uint32_t crc, const uint8_t* p, uint32_t n) {
    crc = ~crc;
    for (uint32_t i = 0; i < n; ++i) crc = table[(crc ^ p[i]) & 0xffu] ^ (crc >> 8);
    return ~crc;
}
// a(x) b(x) mod P, bit-reflected
FRISK_HD uint32_t multmodp(uint32_t a, uint32_t b) {
    uint32_t p = 0;
    for (int i = 0; i < 32; ++i) {
        if (a & (0x80000000u >> i)) p ^= b;
        b = (b & 1u) ? (b >> 1) ^ kPoly : b >> 1;
    }
    return p;
}
// x^(8n) mod P
FRISK_HD uint32_t x8nmodp(uint32_t n) {
    uint32_t t = 1u << 30;                                // x^1
    for (int k = 0; k < 3; ++k) t = multmodp(t, t);       // x^8
    uint32_t p = 1u << 31;                                // x^0
    for (; n; n >>= 1) {
        if (n & 1u) p = multmodp(t, p);
        t = multmodp(t, t);
    }
    return p;
}
FRISK_HD uint32_t umin(uint32_t a, uint32_t b) { return a < b ? a : b; }
// slice i of 32 of n bytes: ceil(n / 32) bytes each, fewer (or none) at the end
FRISK_HD void crc_slice(uint32_t n, int i, uint32_t* lo, uint32_t* len) {
    const uint32_t per = (n + 31u) / 32u;
    *lo = umin(n, (uint32_t)i * per);
    *len = umin(n, (uint32_t)(i + 1) * per) - *lo;
}
// CRC32 of n bytes from the CRCs of its 32 slices: crc(A B) = crc(A) x^(8 |B|) + crc(B) mod P
FRISK_HD uint32_t fold_crcs(const uint32_t* part, uint32_t n) {
    const uint32_t per = (n + 31u) / 32u, shift = x8nmodp(per);
    uint32_t acc = part[0];
    for (int i = 1; i < 32; ++i) {
        uint32_t lo, len;
        crc_slice(n, i, &lo, &len);
        if (len) acc = multmodp(len == per ? shift : x8nmodp(len), acc) ^ part[i];
    }
    return acc;
}

// ---- the kernel: one warp per member --------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32)
bgzf_inflate_kernel(const uint8_t* __restrict__ gz, const uint64_t* __restrict__ comp_off, const uint32_t* __restrict__ comp_len,
                    const uint32_t* __restrict__ crc, const uint64_t* __restrict__ text_off, uint64_t n_blocks, uint64_t text_len,
                    uint8_t* __restrict__ text, uint32_t* __restrict__ status, unsigned int* __restrict__ any_bad) {
    __shared__ Inflater S;
    __shared__ uint32_t s_part[32];
    const uint64_t b = blockIdx.x;
    const int lane = threadIdx.x;
    const uint64_t t0 = text_off[b], t1 = b + 1 < n_blocks ? text_off[b + 1] : text_len;
    if (t1 < t0 || t1 > text_len || t1 - t0 > kMaxIsize) {
        if (lane == 0) { status[b] = kStTable; if (any_bad) atomicOr(any_bad, 1u); }
        return;
    }
    const uint32_t isize = (uint32_t)(t1 - t0), len = comp_len[b];
    const uint8_t* const src = gz + comp_off[b];
    uint8_t* const dst = text + t0;
    Dec d;
    dec_init(d, len, isize);
    uint32_t fill_hi = 0, done = 0, st = kStOk;
    while (true) {                                        // every pass consumes input bits (decode_batch) or ends
        // stage the compressed bytes lane 0 can reach in this batch
        const uint32_t pos = __shfl_sync(0xffffffffu, d.pos, 0);
        const uint32_t want = umin(len, pos + kInBuf);
        for (uint32_t x = fill_hi + lane; x < want; x += 32) S.in[x % kInBuf] = src[x];
        fill_hi = fill_hi > want ? fill_hi : want;
        __syncwarp();
        int nt = 0;
        if (lane == 0) nt = decode_batch(S, d);
        nt = __shfl_sync(0xffffffffu, nt, 0);
        const int phase = __shfl_sync(0xffffffffu, d.phase, 0);
        st = __shfl_sync(0xffffffffu, d.status, 0);
        __syncwarp();
        // materialise: place of every token, then the bytes whose sources precede the batch, then the rest in order
        const uint32_t tk = lane < nt ? S.tok[lane] : 0u;
        const uint32_t tl = lane < nt ? tok_len(tk) : 0u;
        uint32_t incl = tl;
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += y;
        }
        const uint32_t excl = incl - tl, total = __shfl_sync(0xffffffffu, incl, 31);
        const uint32_t dist = tk >> 16;
        const bool dep = lane < nt && dist != 0u && excl + umin(dist, tl) > dist;   // source reaches into this batch
        const uint32_t dep_mask = __ballot_sync(0xffffffffu, dep);
        S.tok_pos[lane] = excl;
        if (lane == 0) S.tok_pos[nt] = total;
        __syncwarp();
        for (uint32_t i = lane; i < total; i += 32) {
            int lo = 0, hi = nt - 1;                      // the token holding byte i
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (S.tok_pos[mid] <= i) lo = mid; else hi = mid - 1;
            }
            if ((dep_mask >> lo) & 1u) continue;
            // byte j of a copy repeats byte j % ds of its source: only bytes before the token are read, even when the copy
            // overlaps itself (ds < length; such a token is independent only at the start of the batch)
            const uint32_t t = S.tok[lo], ds = t >> 16, p = done + i, j = i - S.tok_pos[lo];
            const uint8_t v = ds ? S.ring[(p - j - ds + (j < ds ? j : j % ds)) % kRing] : (uint8_t)t;
            S.ring[p % kRing] = v;
            dst[p] = v;
        }
        __syncwarp();
        for (uint32_t m = dep_mask; m; m &= m - 1u) {
            const int j = __ffs(m) - 1;
            const uint32_t t = S.tok[j], ds = t >> 16, l = t & 0xffffu, p0 = done + S.tok_pos[j];
            for (uint32_t i = lane; i < l; i += 32) {     // byte i of a copy with distance ds repeats byte i % ds of its source
                const uint32_t v = S.ring[(p0 - ds + (i < ds ? i : i % ds)) % kRing];
                S.ring[(p0 + i) % kRing] = v;
                dst[p0 + i] = (uint8_t)v;
            }
            __syncwarp();
        }
        done += total;
        if (st != kStOk || phase == kPhDone) break;
    }
    if (st == kStOk) {
        // CRC32: the ring's first KiB becomes the table, every lane takes a slice of the output (written by this warp)
        uint32_t* const table = reinterpret_cast<uint32_t*>(S.ring);
        for (uint32_t i = lane; i < 256; i += 32) table[i] = crc_table_entry(i);
        __syncwarp();
        uint32_t lo, n;
        crc_slice(isize, lane, &lo, &n);
        s_part[lane] = crc_bytes(table, 0u, dst + lo, n);
        __syncwarp();
        if (lane == 0 && fold_crcs(s_part, isize) != crc[b]) st = kStCrc;
    }
    if (lane == 0) {
        status[b] = st;
        if (st != kStOk && any_bad) atomicOr(any_bad, 1u);
    }
}

int check_table_args(const void* gz, const void* comp_off, const void* comp_len, const void* crc, const void* text_off,
                     uint64_t n_blocks, uint64_t text_len, const void* text, const void* status) {
    if (n_blocks && (!gz || !comp_off || !comp_len || !crc || !text_off || !status)) return FRISK_E_INVALID;
    if (text_len && !text) return FRISK_E_INVALID;
    if (n_blocks > 0x7fffffffull) return FRISK_E_UNSUPPORTED;
    return FRISK_OK;
}

FRISK_HD uint32_t rd16(const uint8_t* p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8; }
FRISK_HD uint32_t rd32(const uint8_t* p) { return rd16(p) | rd16(p + 2) << 16; }

}  // namespace

int frisk_internal::bgzf_inflate(const uint8_t* d_gz, const uint64_t* d_comp_off, const uint32_t* d_comp_len, const uint32_t* d_crc,
                                 const uint64_t* d_text_off, uint64_t n_blocks, uint64_t text_len, uint8_t* d_text,
                                 uint32_t* d_block_status, unsigned int* d_any_bad, cudaStream_t st) {
    if (!n_blocks) return FRISK_OK;
    bgzf_inflate_kernel<<<(unsigned)n_blocks, 32, 0, st>>>(d_gz, d_comp_off, d_comp_len, d_crc, d_text_off, n_blocks, text_len, d_text,
                                                           d_block_status, d_any_bad);
    FRISK_CK(cudaGetLastError());
    return FRISK_OK;
}

extern "C" {

int frisk_b200_bgzf_blocks(const uint8_t* gz, uint64_t n, uint64_t cap, uint64_t* comp_off, uint32_t* comp_len, uint32_t* crc,
                           uint64_t* text_off, uint64_t* n_blocks, uint64_t* text_len) {
    if (!n_blocks || !text_len || (!gz && n)) return FRISK_E_INVALID;
    const bool store = comp_off || comp_len || crc || text_off;
    uint64_t pos = 0, nb = 0, total = 0;
    while (pos < n) {
        const uint8_t* const p = gz + pos;
        const uint64_t avail = n - pos;
        if (avail < 12 || p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || p[3] != 4) return FRISK_E_FORMAT;
        const uint64_t xlen = rd16(p + 10);
        if (12 + xlen > avail) return FRISK_E_FORMAT;
        int64_t bsize = -1;
        for (uint64_t q = 12; q < 12 + xlen;) {             // the extra subfields: SI1 SI2 SLEN data; BC may be anywhere
            if (12 + xlen - q < 4) return FRISK_E_FORMAT;
            const uint64_t slen = rd16(p + q + 2);
            if (slen > 12 + xlen - q - 4) return FRISK_E_FORMAT;
            if (p[q] == 'B' && p[q + 1] == 'C') {
                if (slen != 2 || bsize >= 0) return FRISK_E_FORMAT;
                bsize = rd16(p + q + 4);
            }
            q += 4 + slen;
        }
        if (bsize < 0) return FRISK_E_FORMAT;
        const uint64_t size = (uint64_t)bsize + 1;          // BSIZE: the member's length minus one
        if (size > avail || size < 12 + xlen + 8) return FRISK_E_FORMAT;
        const uint32_t isize = rd32(p + size - 4);
        if (isize > kMaxIsize) return FRISK_E_FORMAT;
        if (store && nb < cap) {
            if (comp_off) comp_off[nb] = pos + 12 + xlen;
            if (comp_len) comp_len[nb] = (uint32_t)(size - 12 - xlen - 8);
            if (crc) crc[nb] = rd32(p + size - 8);
            if (text_off) text_off[nb] = total;
        }
        ++nb;
        total += isize;
        pos += size;
    }
    *n_blocks = nb;
    *text_len = total;
    return nb > cap && store ? FRISK_E_CAPACITY : FRISK_OK;
}

int frisk_b200_bgzf_inflate(const uint8_t* d_gz, const uint64_t* d_comp_off, const uint32_t* d_comp_len, const uint32_t* d_crc,
                            const uint64_t* d_text_off, uint64_t n_blocks, uint64_t text_len, uint8_t* d_text, uint32_t* d_block_status,
                            void* stream) {
    int rc = check_table_args(d_gz, d_comp_off, d_comp_len, d_crc, d_text_off, n_blocks, text_len, d_text, d_block_status);
    if (rc) return rc;
    if (frisk_b200_device_count() <= 0) return FRISK_E_NO_DEVICE;
    return frisk_internal::bgzf_inflate(d_gz, d_comp_off, d_comp_len, d_crc, d_text_off, n_blocks, text_len, d_text, d_block_status,
                                        nullptr, (cudaStream_t)stream);
}

int frisk_b200_bgzf_inflate_host(const uint8_t* gz, const uint64_t* comp_off, const uint32_t* comp_len, const uint32_t* crc,
                                 const uint64_t* text_off, uint64_t n_blocks, uint64_t text_len, uint8_t* text, uint32_t* block_status,
                                 void* stream) {
    (void)stream;
    int rc = check_table_args(gz, comp_off, comp_len, crc, text_off, n_blocks, text_len, text, block_status);
    if (rc) return rc;
    std::unique_ptr<Inflater> S(new (std::nothrow) Inflater());
    if (!S) return FRISK_E_CAPACITY;
    uint32_t table[256];
    for (uint32_t i = 0; i < 256; ++i) table[i] = crc_table_entry(i);
    bool bad = false;
    for (uint64_t b = 0; b < n_blocks; ++b) {
        const uint64_t t0 = text_off[b], t1 = b + 1 < n_blocks ? text_off[b + 1] : text_len;
        uint32_t st = kStOk;
        if (t1 < t0 || t1 > text_len || t1 - t0 > kMaxIsize) st = kStTable;
        if (st == kStOk) {
            const uint32_t isize = (uint32_t)(t1 - t0), len = comp_len[b];
            const uint8_t* const src = gz + comp_off[b];
            uint8_t* const dst = text + t0;
            Dec d;
            dec_init(d, len, isize);
            uint32_t fill_hi = 0, done = 0;
            while (true) {                                // the kernel's loop, one lane
                const uint32_t want = std::min(len, d.pos + kInBuf);
                for (uint32_t x = fill_hi; x < want; ++x) S->in[x % kInBuf] = src[x];
                fill_hi = std::max(fill_hi, want);
                const int nt = decode_batch(*S, d);
                for (int j = 0; j < nt; ++j) {            // tokens in order, bytes in order
                    const uint32_t t = S->tok[j], ds = t >> 16, l = tok_len(t);
                    for (uint32_t i = 0; i < l; ++i, ++done) {
                        const uint8_t v = ds ? S->ring[(done - ds) % kRing] : (uint8_t)t;
                        S->ring[done % kRing] = v;
                        dst[done] = v;
                    }
                }
                if (d.status != kStOk || d.phase == kPhDone) break;
            }
            st = d.status;
            if (st == kStOk) {                            // the kernel's CRC: 32 slices folded
                uint32_t part[32];
                for (int i = 0; i < 32; ++i) {
                    uint32_t lo, n;
                    crc_slice(isize, i, &lo, &n);
                    part[i] = crc_bytes(table, 0u, dst + lo, n);
                }
                if (fold_crcs(part, isize) != crc[b]) st = kStCrc;
            }
        }
        block_status[b] = st;
        bad = bad || st != kStOk;
    }
    return bad ? FRISK_E_FORMAT : FRISK_OK;
}

}  // extern "C"
