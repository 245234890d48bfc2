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
// The bit reader, the table construction and the token decoder (frisk_inflate.cuh, shared with frisk_gzip.cu) are
// __host__ __device__: frisk_b200_bgzf_inflate_host runs the same code on the CPU, so that the decoder's logic and its
// bounds checks are tested on machines without a GPU.  No user path calls it.
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
#include "frisk_inflate.cuh"
#include "frisk_internal.h"

namespace {

constexpr uint32_t kRing = kWindow + kBatchBytes;   // every source of a batch survives the batch's own writes
constexpr uint32_t kMaxIsize = 65536;

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
