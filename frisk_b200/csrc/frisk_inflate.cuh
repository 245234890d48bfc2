// frisk_b200 deflate decoder (RFC 1951), shared by the BGZF inflate (frisk_bgzf.cu) and the gzip inflate (frisk_gzip.cu).
//
// The bit reader, the table construction, the token decoder and the CRC32 helpers are __host__ __device__, so the
// *_inflate_host entry points run the very code the kernels run.  A decoder state `St` holds the staged compressed bytes
// (in[x % kInBuf]), the Huffman tables and the token batch; each kernel keeps its own output side (frisk_bgzf.cu: a byte
// history ring in shared memory, frisk_gzip.cu: 16-bit symbols in global scratch).
//
// decode_batch<false> decodes one whole member (its length and ISIZE known).  decode_batch<true> is the speculative form
// of frisk_gzip.cu: the decoder may start at any block header of one long stream, a distance may reach `ctx` bytes before
// its first byte, it stops at the first block boundary at or after bit `stop`, and the caller bounds the output.
//
// Safety: every read is bounded by Dec::len (bytes past it read as zero and their use is kStInput), every loop by input
// bits or output bytes; malformed input sets Dec::status and never faults.
#ifndef FRISK_INFLATE_CUH
#define FRISK_INFLATE_CUH

#include <cuda_runtime.h>
#include <stdint.h>

#define FRISK_HD __host__ __device__ __forceinline__

namespace {

constexpr uint32_t kWindow = 32768;          // deflate's longest distance
constexpr uint32_t kBatchBytes = 4096;       // output bytes of one batch at most
constexpr uint32_t kInBuf = 2048;            // staged compressed bytes (a batch reads < 200, a block header < 600)
constexpr int kMaxTok = 32;
constexpr int kLitBits = 10, kDistBits = 8;  // primary lookup tables; longer codes take the canonical walk

// decoder status (0 = decoded; for a BGZF member: size and CRC32 match too)
enum : uint32_t {
    kStOk = 0,
    kStBlockType = 1,      // BTYPE 3
    kStBadCode = 2,        // over-subscribed or (where zlib refuses it) incomplete code, too many length/distance codes,
                           // a repeat with no previous length, a code-length run past the end, no end-of-block code
    kStBadSymbol = 3,      // a code that is not in the table, litlen 286/287, distance 30/31
    kStDistance = 4,       // a distance before the first byte the decoder may reach
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
// decode_batch<true>: a decoder started at a block header inside one long stream
struct SpecDec : Dec {
    uint64_t stop;        // end at the first block boundary at or after this bit (counted like pos * 8 - bc)
    uint32_t ctx;         // bytes before the first output byte a distance may reach (0 or kWindow)
};

FRISK_HD void dec_init(Dec& d, uint32_t len, uint32_t isize) {
    d.bb = 0; d.bc = 0; d.pos = 0; d.len = len; d.isize = isize; d.out = 0; d.stored_left = 0;
    d.phase = kPhHeader; d.last = false; d.status = kStOk;
}

// fills bb to >= 57 bits; bytes past the payload read as zero (bits_overrun catches their use)
template <class St>
FRISK_HD void refill(const St& S, Dec& d) {
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

// the rest of a dynamic block's header (after BFINAL and BTYPE): code lengths and the litlen / distance codes in S.
// d.phase becomes kPhHuff, or kPhDone with d.status set.  (The boundary search of frisk_gzip.cu runs it at every bit offset
// it tests, with a state whose fast tables are null.)
template <class St>
FRISK_HD void dynamic_header(St& S, Dec& d) {
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
}

// a block header: BFINAL, BTYPE, and the stored length or the Huffman tables
template <class St>
FRISK_HD void block_header(St& S, Dec& d) {
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
        dynamic_header(S, d);
    } else {
        fail(d, kStBlockType);
    }
}

// Lane 0's part: decode the next batch into S.tok (a block header first when one is due).  Returns the number of tokens;
// sets d.phase to kPhDone at the end of the member or on an error (d.status).  Consumes input bits whenever it returns
// with the member unfinished, so that the caller's loop is bounded by the member's bits.
// kSpec (D = SpecDec): no member end to check; ends at a block boundary at or after d.stop too, and a distance may reach
// d.ctx bytes before the first output byte.
template <bool kSpec = false, class St, class D>
FRISK_HD int decode_batch(St& S, D& d) {
    if (d.phase == kPhHeader) {
        if constexpr (kSpec) {
            if ((uint64_t)d.pos * 8u - d.bc >= d.stop) { d.phase = kPhDone; return 0; }
        }
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
            if constexpr (kSpec) {
                if ((uint64_t)dist > (uint64_t)d.out + d.ctx) { fail(d, kStDistance); break; }
            } else {
                if (dist > d.out) { fail(d, kStDistance); break; }
            }
            if (ln > d.isize - d.out) { fail(d, kStOutput); break; }
            S.tok[nt++] = dist << 16 | ln;
            bytes += ln;
            d.out += ln;
        }
        if (bits_overrun(d)) { fail(d, kStInput); break; }
    }
    if (d.status == kStOk && bits_overrun(d)) fail(d, kStInput);
    if (d.status == kStOk && d.phase == kPhHeader && d.last) {
        d.phase = kPhDone;                                 // the final block ended
        if constexpr (!kSpec) {                            // a member's payload must end in this byte
            const uint64_t used = (uint64_t)d.pos * 8u - d.bc;
            if ((used + 7u) / 8u != d.len) fail(d, kStInput);
            else if (d.out != d.isize) fail(d, kStSize);
        }
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

FRISK_HD uint32_t rd16(const uint8_t* p) { return (uint32_t)p[0] | (uint32_t)p[1] << 8; }
FRISK_HD uint32_t rd32(const uint8_t* p) { return rd16(p) | rd16(p + 2) << 16; }

}  // namespace

#endif
