// frisk_b200 gzip inflate: one plain gzip member (gzip, pigz; NCBI, Ensembl and UCSC .fa.gz) in, text out, on the GPU.
//
// A gzip member is one deflate stream: block starts are neither byte-aligned nor indexed, and a match may reach 32 KiB
// back into text another decoder has not produced yet.  So the stream is inflated in two passes, as pugz does
// (Kerbiriou & Chikhi, 2019):
//
// 1. Plan.  Nominal chunk starts every C compressed bytes (kChunkBytes; option "gzip_chunk_bytes").  For each nominal
//    start but the first, one warp tests 32 consecutive bit offsets at a time for a fully valid dynamic block header
//    (gzip_search_kernel); the first hit before the next nominal start is the chunk's start.  A window with no hit merges
//    into its predecessor.  Chunk 0 starts at the first payload bit and is exact.
// 2. Speculative decode, one warp per chunk (gzip_decode_kernel, the decoder of frisk_inflate.cuh): whole blocks from the
//    chunk's start to the first block boundary at or after the next chunk's start, or to the end of the final block.  The
//    output is 16-bit symbols in global scratch: 0..255 a byte, 256 + p byte p of the 32 KiB before the chunk (a match that
//    reaches before the chunk's first byte; copies of such symbols propagate them).  History is read back from the same
//    scratch, so a decoder needs little shared memory: cuobjdump lists 6,916 bytes for gzip_decode_kernel, 7,940 with the
//    1 KiB the runtime reserves per CTA, so 29 decoders fit an SM's 228 KiB.  The first pass's scratch holds kSymPerByte
//    symbols per compressed byte (16 bytes of device memory per compressed byte: ~14 GB for a 900 MB .gz); a chunk that
//    outgrows it keeps decoding to learn its length and end.
// 3. Join (host, after one read-back of the chunk results): walking from chunk 0, chunk i + 1 is accepted only if chunk i
//    decoded OK and ended exactly where chunk i + 1 started.  A chunk that is not accepted is decoded again from its
//    predecessor's end (one launch for every such chunk whose predecessor decoded OK), until the chain reaches the final
//    block.  A decode from a false start is discarded, never used; speculation only decides how much runs in parallel.
//    Chunks of the chain that outgrew their scratch are decoded once more into exact scratch.
// 4. Resolve: text offsets from the chunk lengths; every literal symbol, in parallel (gzip_literal_kernel); the
//    placeholders of the last 32 KiB of every chunk in chain order (gzip_context_kernel, the one serial step: they read the
//    text before their chunk); then every chunk's other placeholders in parallel with its CRC32 (gzip_translate_kernel);
//    the host folds the chunk CRCs with x^(8n) and checks CRC32 and ISIZE.
//
// frisk_b200_gzip_inflate_host runs the same plan, joins and repairs on the CPU with the same decoder (test
// infrastructure, like frisk_b200_bgzf_inflate_host): same text, same stats.
//
// Safety: every read is bounded by the payload, every write by the chunk's scratch or the text length, every loop by input
// bits; malformed input ends in a status word and FRISK_E_FORMAT, never a fault.
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <functional>
#include <memory>
#include <new>
#include <vector>

#include "../../include/frisk_b200.h"
#include "frisk_inflate.cuh"
#include "frisk_internal.h"

int frisk_internal::g_gzip_chunk_bytes = 0;

namespace {

// Default chunk: below the compressed size of a zlib block on FASTA (22.7 KB at level 1 .. 29 KB at level 9), so every
// block boundary can start a chunk; a smaller C only adds windows that merge.
constexpr uint64_t kChunkBytes = 16384;
constexpr uint32_t kSymPerByte = 8;                    // scratch symbols per compressed byte of a chunk's span
constexpr uint32_t kSymSlack = 4096;
constexpr uint64_t kMaxCap = 1ull << 30;               // first-pass scratch of one chunk at most (symbols)
constexpr uint64_t kMaxSpan = 1ull << 31;              // compressed bytes one decoder may read (its bit counts stay 32-bit)
constexpr uint32_t kSpecIsize = 0xffff0000u;           // a chunk's text stays below 4 GiB
constexpr uint64_t kNone = ~0ull;
// The boundary search splits windows into sub-windows of one warp each until about kSearchWarps warps run, with at
// least kSubBytes per sub-window.  One warp per 16 KiB window leaves most of the GPU idle on a 40 MB genome (~5 warps per
// SM for C2's 772 windows), while on a 1 GB genome the windows alone fill it and extra sub-windows only add scanning.
constexpr uint64_t kSubBytes = 1024, kSearchWarps = 8192;
constexpr int kNeedMore = -1;                          // the header runs past the bytes seen so far

// one chunk's decode: in = start, stop, sym, cap, ctx; out = end, len, status, final
struct GzChunk {
    uint64_t start, stop;     // bits from the payload's first bit
    uint64_t end;             // the bit after the last block decoded
    uint16_t* sym;            // scratch (device memory for the kernel)
    uint32_t cap, ctx;        // symbols sym holds; bytes before the chunk a distance may reach (0: chunk 0)
    uint32_t len, status;     // symbols produced (counted past cap too); kSt*
    uint32_t final_, pad;     // the final block ended this decode
};

// a chunk of the chain, for the resolve
struct ChainRef {
    const uint16_t* sym;
    uint64_t text_off;
    uint32_t len, pad;
};

// a decoder's shared memory: Inflater (frisk_bgzf.cu) without the history ring
struct GzInflater {
    uint8_t in[kInBuf];
    uint16_t lit_fast[1 << kLitBits];
    uint16_t dist_fast[1 << kDistBits];
    uint16_t lit_count[16], dist_count[16];
    uint16_t lit_sym[288], dist_sym[32];
    uint8_t lens[288 + 32];
    uint32_t tok[kMaxTok];
    uint32_t tok_pos[kMaxTok + 1];
};

// one lane's boundary test: the tables are built without their fast lookups (counts and symbols decide validity)
struct Probe {
    const uint8_t* in;        // the payload from the tested bit's byte; Dec::len <= kInBuf keeps in[pos % kInBuf] == in[pos]
    uint8_t lens[288 + 32];
    uint16_t lit_count[16], dist_count[16];
    uint16_t lit_sym[288], dist_sym[32];
    static constexpr uint16_t* lit_fast = nullptr;
    static constexpr uint16_t* dist_fast = nullptr;
};

// a valid dynamic block header (BTYPE 2, HLIT / HDIST in range, complete code-length code, lengths that decode, an
// end-of-block code, litlen and distance codes build_code accepts) starts at payload bit `bit` (< P * 8)
FRISK_HD bool dynamic_at(const uint8_t* pay, uint64_t P, uint64_t bit, Probe& S) {
    const uint64_t base = bit >> 3;
    S.in = pay + base;
    Dec d;
    dec_init(d, (uint32_t)(P - base < kInBuf ? P - base : kInBuf), 0);
    refill(S, d);
    bits(d, (uint32_t)(bit & 7u));
    bits(d, 1);
    if (bits(d, 2) != 2u) return false;
    dynamic_header(S, d);
    return d.phase == kPhHuff;
}

// symbol of output position s of a chunk (s < 0: a placeholder for the context)
FRISK_HD uint16_t sym_at(const uint16_t* out, uint32_t cap, int64_t s) {
    if (s < 0) return (uint16_t)(256 + (int64_t)kWindow + s);
    return s < (int64_t)cap ? out[s] : (uint16_t)0;
}

// byte of symbol v at text offset off of a chunk; *bad when a placeholder reaches before the text
FRISK_HD uint8_t sym_byte(uint16_t v, const uint8_t* text, uint64_t off, bool* bad) {
    if (v < 256) return (uint8_t)v;
    const uint64_t q = v - 256u;
    if (off + q < kWindow) { *bad = true; return 0; }
    return text[off - kWindow + q];
}

FRISK_HD void spec_init(SpecDec& d, const GzChunk& J, uint64_t P, uint64_t* base) {
    *base = J.start >> 3;
    const uint64_t avail = *base < P ? P - *base : 0;
    dec_init(d, (uint32_t)(avail < kMaxSpan ? avail : kMaxSpan), kSpecIsize);
    d.stop = J.stop >= *base * 8u ? J.stop - *base * 8u : 0;
    d.ctx = J.ctx;
}

// ---- kernels ---------------------------------------------------------------------------------------------------------------
// sub-window s of window k + 1 (width C, n_sub sub-windows of `sub` bytes): cand[k * n_sub + s] = its first dynamic block
// header, or kNone.  (A window's candidate is the first hit of its sub-windows: the bit a scan of the whole window finds.)
__global__ void __launch_bounds__(32) gzip_search_kernel(const uint8_t* __restrict__ pay, uint64_t P, uint64_t C, uint64_t n_sub,
                                                         uint64_t* __restrict__ cand) {
    const uint64_t k = blockIdx.x / n_sub + 1, s = blockIdx.x % n_sub, sub = (C + n_sub - 1) / n_sub;
    uint64_t hi = (k + 1) * C < P ? (k + 1) * C : P;
    if (k * C + (s + 1) * sub < hi) hi = k * C + (s + 1) * sub;
    const uint64_t lo = (k * C + s * sub) * 8u;
    hi *= 8u;
    const int lane = threadIdx.x;
    Probe S;
    for (uint64_t b0 = lo; b0 < hi; b0 += 32) {
        const uint64_t bit = b0 + lane;
        const unsigned m = __ballot_sync(0xffffffffu, bit < hi && dynamic_at(pay, P, bit, S));
        if (m) {
            if (lane == 0) cand[blockIdx.x] = b0 + __ffs(m) - 1;
            return;
        }
    }
    if (lane == 0) cand[blockIdx.x] = kNone;
}

// one warp per chunk: lane 0 decodes batches of tokens, the warp writes their symbols (the materialisation of
// bgzf_inflate_kernel, with the history read back from the chunk's scratch instead of a ring)
__global__ void __launch_bounds__(32) gzip_decode_kernel(const uint8_t* __restrict__ pay, uint64_t P, GzChunk* __restrict__ jobs) {
    __shared__ GzInflater S;
    GzChunk& J = jobs[blockIdx.x];
    const int lane = threadIdx.x;
    uint16_t* const out = J.sym;
    const uint32_t cap = J.cap;
    SpecDec d;
    uint64_t base;
    spec_init(d, J, P, &base);
    const uint8_t* const src = pay + base;
    const uint32_t span = d.len;
    uint32_t fill_hi = 0, done = 0;
    bool primed = false;
    while (true) {                                        // every pass consumes input bits (decode_batch) or ends
        const uint32_t pos = __shfl_sync(0xffffffffu, d.pos, 0);
        const uint32_t want = umin(span, pos + kInBuf);
        for (uint32_t x = fill_hi + lane; x < want; x += 32) S.in[x % kInBuf] = src[x];
        fill_hi = fill_hi > want ? fill_hi : want;
        __syncwarp();
        int nt = 0;
        if (lane == 0) {
            if (!primed) { refill(S, d); bits(d, (uint32_t)(J.start & 7u)); }
            nt = decode_batch<true>(S, d);
        }
        primed = true;
        nt = __shfl_sync(0xffffffffu, nt, 0);
        const int phase = __shfl_sync(0xffffffffu, d.phase, 0);
        const uint32_t st = __shfl_sync(0xffffffffu, d.status, 0);
        __syncwarp();
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
            int lo = 0, hi = nt - 1;                      // the token holding symbol i
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (S.tok_pos[mid] <= i) lo = mid; else hi = mid - 1;
            }
            if ((dep_mask >> lo) & 1u) continue;
            const uint32_t t = S.tok[lo], ds = t >> 16, p = done + i, j = i - S.tok_pos[lo];
            const uint16_t v = ds ? sym_at(out, cap, (int64_t)p - j - ds + (j < ds ? j : j % ds)) : (uint16_t)t;
            if (p < cap) out[p] = v;
        }
        __syncwarp();
        for (uint32_t m = dep_mask; m; m &= m - 1u) {
            const int j = __ffs(m) - 1;
            const uint32_t t = S.tok[j], ds = t >> 16, l = t & 0xffffu, p0 = done + S.tok_pos[j];
            for (uint32_t i = lane; i < l; i += 32) {
                const uint16_t v = sym_at(out, cap, (int64_t)p0 - ds + (i < ds ? i : i % ds));
                if (p0 + i < cap) out[p0 + i] = v;
            }
            __syncwarp();
        }
        done += total;
        if (st != kStOk || phase == kPhDone) break;
    }
    if (lane == 0) {
        J.end = base * 8u + ((uint64_t)d.pos * 8u - d.bc);
        J.len = d.out;
        J.status = d.status;
        J.final_ = d.status == kStOk && d.last;
    }
}

// one CTA per chunk: every literal symbol
__global__ void __launch_bounds__(256) gzip_literal_kernel(const ChainRef* __restrict__ ch, uint8_t* __restrict__ text) {
    const ChainRef c = ch[blockIdx.x];
    for (uint32_t k = threadIdx.x; k < c.len; k += blockDim.x) {
        const uint16_t v = c.sym[k];
        if (v < 256) text[c.text_off + k] = (uint8_t)v;
    }
}

// the serial step: the placeholders of the last 32 KiB of every chunk, in chain order (each reads only text before its
// chunk, complete once the chunks before it are done); 32 symbols per thread, all loaded before any is resolved
constexpr int kCtxThreads = 1024, kCtxPer = (int)kWindow / kCtxThreads;
__global__ void __launch_bounds__(kCtxThreads) gzip_context_kernel(const ChainRef* __restrict__ ch, uint64_t n,
                                                                   uint8_t* __restrict__ text, unsigned int* __restrict__ bad) {
    bool b = false;
    for (uint64_t i = 0; i < n; ++i) {
        const ChainRef c = ch[i];
        const uint32_t lo = c.len > kWindow ? c.len - kWindow : 0u;
        uint16_t v[kCtxPer];
#pragma unroll
        for (int r = 0; r < kCtxPer; ++r) {
            const uint32_t k = lo + r * kCtxThreads + threadIdx.x;
            v[r] = k < c.len ? c.sym[k] : (uint16_t)0;
        }
#pragma unroll
        for (int r = 0; r < kCtxPer; ++r)
            if (v[r] >= 256) text[c.text_off + lo + r * kCtxThreads + threadIdx.x] = sym_byte(v[r], text, c.text_off, &b);
        __syncthreads();
    }
    if (b) atomicOr(bad, 1u);
}

// one CTA per chunk: the placeholders before its last 32 KiB, then its CRC32 (warp 0, 32 slices folded)
__global__ void __launch_bounds__(256) gzip_translate_kernel(const ChainRef* __restrict__ ch, uint8_t* __restrict__ text,
                                                             uint32_t* __restrict__ crc, unsigned int* __restrict__ bad) {
    __shared__ uint32_t table[256];
    __shared__ uint32_t part[32];
    const ChainRef c = ch[blockIdx.x];
    const uint32_t hi = c.len > kWindow ? c.len - kWindow : 0u;
    bool b = false;
    for (uint32_t k = threadIdx.x; k < hi; k += blockDim.x) {
        const uint16_t v = c.sym[k];
        if (v >= 256) text[c.text_off + k] = sym_byte(v, text, c.text_off, &b);
    }
    if (b) atomicOr(bad, 1u);
    table[threadIdx.x] = crc_table_entry(threadIdx.x);
    __syncthreads();
    if (threadIdx.x < 32) {
        uint32_t lo, n;
        crc_slice(c.len, threadIdx.x, &lo, &n);
        part[threadIdx.x] = crc_bytes(table, 0u, text + c.text_off + lo, n);
        __syncwarp();
        if (threadIdx.x == 0) crc[blockIdx.x] = fold_crcs(part, c.len);
    }
}

// ---- the header -------------------------------------------------------------------------------------------------------------
// m of the member's n bytes at p: FRISK_OK and the payload's offset, FRISK_E_FORMAT, or kNeedMore (m < n and the header
// reaches past m).  CM 8; FTEXT, FHCRC (checked), FEXTRA, FNAME, FCOMMENT; reserved flag bits are FRISK_E_FORMAT.  At least
// one payload byte and the 8-byte trailer must follow.
int parse_header(const uint8_t* p, uint64_t m, uint64_t n, uint64_t* off) {
    const int short_rc = m < n ? kNeedMore : FRISK_E_FORMAT;
    if (m < 10) return short_rc;
    if (p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || (p[3] & 0xe0)) return FRISK_E_FORMAT;
    const uint8_t flg = p[3];
    uint64_t q = 10;
    if (flg & 4) {
        if (q + 2 > m) return short_rc;
        q += 2 + rd16(p + q);
    }
    for (int f = 8; f <= 16; f <<= 1) {                   // FNAME, FCOMMENT: zero-terminated
        if (!(flg & f)) continue;
        while (q < m && p[q]) ++q;
        if (q >= m) return short_rc;
        ++q;
    }
    if (flg & 2) {
        if (q + 2 > m) return short_rc;
        uint32_t table[256];
        for (uint32_t i = 0; i < 256; ++i) table[i] = crc_table_entry(i);
        uint32_t crc = 0;
        for (uint64_t a = 0; a < q; a += 0x40000000u) crc = crc_bytes(table, crc, p + a, (uint32_t)std::min<uint64_t>(q - a, 0x40000000u));
        if ((crc & 0xffffu) != rd16(p + q)) return FRISK_E_FORMAT;
        q += 2;
    }
    if (q + 9 > n) return FRISK_E_FORMAT;
    *off = q;
    return FRISK_OK;
}

// ---- the two places the passes run ------------------------------------------------------------------------------------------
struct Backend {
    virtual ~Backend() {}
    virtual int read(uint64_t off, uint64_t len, uint8_t* dst) = 0;                 // member bytes to the host
    virtual int search(uint64_t hdr, uint64_t P, uint64_t C, uint64_t K, std::vector<uint64_t>& cand) = 0;   // windows 1..K-1
    virtual int scratch(uint64_t syms, uint16_t** out) = 0;                          // owned by the backend
    virtual int decode(uint64_t hdr, uint64_t P, std::vector<GzChunk>& jobs) = 0;
    virtual int resolve(const std::vector<ChainRef>& chain, uint8_t* text, std::vector<uint32_t>& crc, bool* bad) = 0;
};

struct HostBackend : Backend {
    const uint8_t* gz;
    std::vector<std::unique_ptr<uint16_t[]>> bufs;
    explicit HostBackend(const uint8_t* g) : gz(g) {}
    int read(uint64_t off, uint64_t len, uint8_t* dst) override {
        memcpy(dst, gz + off, len);
        return FRISK_OK;
    }
    int search(uint64_t hdr, uint64_t P, uint64_t C, uint64_t K, std::vector<uint64_t>& cand) override {
        std::unique_ptr<Probe> S(new (std::nothrow) Probe());
        if (!S) return FRISK_E_CAPACITY;
        for (uint64_t k = 1; k < K; ++k) {
            const uint64_t hi = std::min<uint64_t>((k + 1) * C, P) * 8u;
            cand[k - 1] = kNone;
            for (uint64_t bit = k * C * 8u; bit < hi; ++bit)
                if (dynamic_at(gz + hdr, P, bit, *S)) { cand[k - 1] = bit; break; }
        }
        return FRISK_OK;
    }
    int scratch(uint64_t syms, uint16_t** out) override {
        bufs.emplace_back(new (std::nothrow) uint16_t[syms ? syms : 1]);
        *out = bufs.back().get();
        return *out ? FRISK_OK : FRISK_E_CAPACITY;
    }
    int decode(uint64_t hdr, uint64_t P, std::vector<GzChunk>& jobs) override {
        std::unique_ptr<GzInflater> S(new (std::nothrow) GzInflater());
        if (!S) return FRISK_E_CAPACITY;
        for (GzChunk& J : jobs) {                         // the kernel's loop, one lane, symbols in order
            SpecDec d;
            uint64_t base;
            spec_init(d, J, P, &base);
            const uint8_t* const src = gz + hdr + base;
            uint32_t fill_hi = 0, done = 0;
            bool primed = false;
            while (true) {
                const uint32_t want = std::min(d.len, d.pos + kInBuf);
                for (uint32_t x = fill_hi; x < want; ++x) S->in[x % kInBuf] = src[x];
                fill_hi = std::max(fill_hi, want);
                if (!primed) { refill(*S, d); bits(d, (uint32_t)(J.start & 7u)); primed = true; }
                const int nt = decode_batch<true>(*S, d);
                for (int t = 0; t < nt; ++t) {
                    const uint32_t tk = S->tok[t], ds = tk >> 16, l = tok_len(tk);
                    for (uint32_t i = 0; i < l; ++i, ++done) {
                        const uint16_t v = ds ? sym_at(J.sym, J.cap, (int64_t)done - ds) : (uint16_t)tk;
                        if (done < J.cap) J.sym[done] = v;
                    }
                }
                if (d.status != kStOk || d.phase == kPhDone) break;
            }
            J.end = base * 8u + ((uint64_t)d.pos * 8u - d.bc);
            J.len = d.out;
            J.status = d.status;
            J.final_ = d.status == kStOk && d.last;
        }
        return FRISK_OK;
    }
    int resolve(const std::vector<ChainRef>& chain, uint8_t* text, std::vector<uint32_t>& crc, bool* bad) override {
        uint32_t table[256];
        for (uint32_t i = 0; i < 256; ++i) table[i] = crc_table_entry(i);
        for (size_t i = 0; i < chain.size(); ++i) {       // in chain order, every symbol: the context is always there
            const ChainRef& c = chain[i];
            for (uint32_t k = 0; k < c.len; ++k) text[c.text_off + k] = sym_byte(c.sym[k], text, c.text_off, bad);
            uint32_t part[32];
            for (int s = 0; s < 32; ++s) {
                uint32_t lo, n;
                crc_slice(c.len, s, &lo, &n);
                part[s] = crc_bytes(table, 0u, text + c.text_off + lo, n);
            }
            crc[i] = fold_crcs(part, c.len);
        }
        return FRISK_OK;
    }
};

struct DeviceBackend : Backend {
    const uint8_t* d_gz;
    const uint8_t* h_gz;      // nullable: the caller's host copy of the member
    cudaStream_t st;
    std::vector<void*> bufs;
    DeviceBackend(const uint8_t* d, const uint8_t* h, cudaStream_t s) : d_gz(d), h_gz(h), st(s) {}
    ~DeviceBackend() override {
        for (void* p : bufs) cudaFreeAsync(p, st);
    }
    int alloc(uint64_t bytes, void** out) {
        FRISK_CK(cudaMallocAsync(out, bytes ? bytes : 1, st));
        bufs.push_back(*out);
        return FRISK_OK;
    }
    int read(uint64_t off, uint64_t len, uint8_t* dst) override {
        if (h_gz) { memcpy(dst, h_gz + off, len); return FRISK_OK; }
        FRISK_CK(cudaMemcpyAsync(dst, d_gz + off, len, cudaMemcpyDeviceToHost, st));
        FRISK_CK(cudaStreamSynchronize(st));
        return FRISK_OK;
    }
    int search(uint64_t hdr, uint64_t P, uint64_t C, uint64_t K, std::vector<uint64_t>& cand) override {
        if (K < 2) return FRISK_OK;
        const uint64_t S = std::max<uint64_t>(1, std::min<uint64_t>((C + kSubBytes - 1) / kSubBytes, kSearchWarps / (K - 1)));
        if ((K - 1) * S > 0x7fffffffull) return FRISK_E_UNSUPPORTED;
        void* d_cand;
        int rc = alloc((K - 1) * S * 8, &d_cand);
        if (rc) return rc;
        gzip_search_kernel<<<(unsigned)((K - 1) * S), 32, 0, st>>>(d_gz + hdr, P, C, S, (uint64_t*)d_cand);
        FRISK_CK(cudaGetLastError());
        std::vector<uint64_t> sub((K - 1) * S);
        FRISK_CK(cudaMemcpyAsync(sub.data(), d_cand, sub.size() * 8, cudaMemcpyDeviceToHost, st));
        FRISK_CK(cudaStreamSynchronize(st));
        for (uint64_t k = 0; k + 1 < K; ++k)
            for (uint64_t s = S; s-- > 0;)
                if (sub[k * S + s] != kNone) cand[k] = sub[k * S + s];
        return FRISK_OK;
    }
    int scratch(uint64_t syms, uint16_t** out) override { return alloc(syms * 2, (void**)out); }
    int decode(uint64_t hdr, uint64_t P, std::vector<GzChunk>& jobs) override {
        if (jobs.empty()) return FRISK_OK;
        if (jobs.size() > 0x7fffffffull) return FRISK_E_UNSUPPORTED;
        const size_t bytes = jobs.size() * sizeof(GzChunk);
        GzChunk* d_jobs;
        int rc = alloc(bytes, (void**)&d_jobs);           // (freed with the other buffers, on every exit)
        if (rc) return rc;
        FRISK_CK(cudaMemcpyAsync(d_jobs, jobs.data(), bytes, cudaMemcpyHostToDevice, st));
        gzip_decode_kernel<<<(unsigned)jobs.size(), 32, 0, st>>>(d_gz + hdr, P, d_jobs);
        FRISK_CK(cudaGetLastError());
        FRISK_CK(cudaMemcpyAsync(jobs.data(), d_jobs, bytes, cudaMemcpyDeviceToHost, st));
        FRISK_CK(cudaStreamSynchronize(st));
        return FRISK_OK;
    }
    int resolve(const std::vector<ChainRef>& chain, uint8_t* text, std::vector<uint32_t>& crc, bool* bad) override {
        const uint64_t n = chain.size();
        if (n > 0x7fffffffull) return FRISK_E_UNSUPPORTED;
        void* d;                                          // chain | CRCs | bad word
        const uint64_t ref_bytes = n * sizeof(ChainRef);
        int rc = alloc(ref_bytes + n * 4 + 4, &d);
        if (rc) return rc;
        ChainRef* const d_ch = (ChainRef*)d;
        uint32_t* const d_crc = (uint32_t*)((char*)d + ref_bytes);
        unsigned int* const d_bad = (unsigned int*)(d_crc + n);
        FRISK_CK(cudaMemcpyAsync(d_ch, chain.data(), ref_bytes, cudaMemcpyHostToDevice, st));
        FRISK_CK(cudaMemsetAsync(d_bad, 0, 4, st));
        gzip_literal_kernel<<<(unsigned)n, 256, 0, st>>>(d_ch, text);
        gzip_context_kernel<<<1, kCtxThreads, 0, st>>>(d_ch, n, text, d_bad);
        gzip_translate_kernel<<<(unsigned)n, 256, 0, st>>>(d_ch, text, d_crc, d_bad);
        FRISK_CK(cudaGetLastError());
        unsigned int b = 0;
        FRISK_CK(cudaMemcpyAsync(crc.data(), d_crc, n * 4, cudaMemcpyDeviceToHost, st));
        FRISK_CK(cudaMemcpyAsync(&b, d_bad, 4, cudaMemcpyDeviceToHost, st));
        FRISK_CK(cudaStreamSynchronize(st));
        *bad = b != 0;
        return FRISK_OK;
    }
};

// a chain chunk's failure: a chunk of 4 GiB of text or more, or one decoder's 2 GiB input window, is unsupported
int chunk_error(const GzChunk& c, uint64_t P) {
    if (c.status == kStOutput) return FRISK_E_UNSUPPORTED;
    if (c.status == kStInput && P - std::min(P, c.start >> 3) > kMaxSpan) return FRISK_E_UNSUPPORTED;
    return FRISK_E_FORMAT;
}

// the whole inflate; alloc_text(text_len, &text) is called once the length is known and before anything is written
int inflate(Backend& B, uint64_t n, const std::function<int(uint64_t, uint8_t**)>& alloc_text, uint64_t* text_len, uint64_t stats[4]) {
    // header (read in growing pieces: FEXTRA, FNAME and FCOMMENT may be long)
    uint64_t hdr = 0;
    std::vector<uint8_t> head;
    int rc = kNeedMore;
    for (uint64_t m = std::min<uint64_t>(n, 65536); rc == kNeedMore; m = std::min<uint64_t>(n, 2 * m)) {
        head.resize(m);
        if ((rc = B.read(0, m, head.data()))) return rc;
        rc = parse_header(head.data(), m, n, &hdr);
    }
    if (rc) return rc;
    const uint64_t P = n - 8 - hdr;                       // the stream's bytes at most (a trailer follows it)
    // plan: chunk 0 at bit 0, then the first dynamic block header of every window that has one
    const uint64_t C = frisk_internal::g_gzip_chunk_bytes > 0 ? (uint64_t)frisk_internal::g_gzip_chunk_bytes : kChunkBytes;
    const uint64_t K = (P + C - 1) / C;
    std::vector<uint64_t> cand(K > 1 ? K - 1 : 0, kNone);
    if ((rc = B.search(hdr, P, C, K, cand))) return rc;
    std::vector<GzChunk> ch(1);
    for (uint64_t c : cand)
        if (c != kNone) ch.emplace_back().start = c;
    const size_t N = ch.size();
    uint64_t total = 0;
    for (size_t i = 0; i < N; ++i) {
        GzChunk& c = ch[i];
        c.stop = i + 1 < N ? ch[i + 1].start : kNone;
        const uint64_t span = (i + 1 < N ? (c.stop + 7) / 8 : P) - c.start / 8;
        c.cap = (uint32_t)std::min<uint64_t>(kSymPerByte * span + kSymSlack, kMaxCap);
        c.ctx = i ? kWindow : 0u;
        total += c.cap;
    }
    uint16_t* scratch = nullptr;
    if ((rc = B.scratch(total, &scratch))) return rc;
    for (GzChunk& c : ch) { c.sym = scratch; scratch += c.cap; }
    // speculative decode, then joins and repairs until the chain reaches the final block
    if ((rc = B.decode(hdr, P, ch))) return rc;
    std::vector<bool> repaired(N, false);
    uint64_t n_repaired = 0;
    size_t last = 0;
    while (true) {
        size_t f = 0;
        uint64_t pos = 0;
        bool complete = false;
        for (; f < N; ++f) {
            const GzChunk& c = ch[f];
            if (c.start != pos) break;                    // f starts where its predecessor did not end
            if (c.status != kStOk) return chunk_error(c, P);
            if (c.final_) { complete = true; break; }
            pos = c.end;
        }
        if (complete) { last = f; break; }
        if (f == N) return FRISK_E_FORMAT;                // (the last chunk has no stop: not reached)
        // f from its predecessor's true end, and every later chunk whose predecessor decoded OK to somewhere else
        std::vector<GzChunk> jobs;
        std::vector<size_t> idx;
        for (size_t k = f; k < N; ++k) {
            const GzChunk& p = ch[k - 1];
            const bool pred_redone = !idx.empty() && idx.back() == k - 1;
            if (k > f && (pred_redone || p.status != kStOk || p.final_ || p.end == ch[k].start)) continue;
            GzChunk j = ch[k];
            j.start = p.end;
            jobs.push_back(j);
            idx.push_back(k);
        }
        if ((rc = B.decode(hdr, P, jobs))) return rc;
        for (size_t q = 0; q < idx.size(); ++q) { ch[idx[q]] = jobs[q]; repaired[idx[q]] = true; }
        n_repaired += idx.size();
    }
    // chain chunks that outgrew their scratch: once more, into exact scratch
    std::vector<GzChunk> over;
    std::vector<size_t> over_idx;
    uint64_t over_total = 0;
    for (size_t i = 0; i <= last; ++i)
        if (ch[i].len > ch[i].cap) { over.push_back(ch[i]); over_idx.push_back(i); over_total += ch[i].len; }
    if (!over.empty()) {
        if ((rc = B.scratch(over_total, &scratch))) return rc;
        for (GzChunk& c : over) { c.sym = scratch; c.cap = c.len; scratch += c.len; }
        if ((rc = B.decode(hdr, P, over))) return rc;
        for (size_t q = 0; q < over.size(); ++q) {
            const GzChunk& a = ch[over_idx[q]];
            const GzChunk& b = over[q];
            if (b.status != kStOk || b.end != a.end || b.len != a.len || b.final_ != a.final_) return FRISK_E_FORMAT;
            ch[over_idx[q]] = b;
        }
    }
    // the trailer behind the final block; nothing may follow it but another member (not supported here)
    uint64_t t = 0;
    std::vector<ChainRef> chain(last + 1);
    for (size_t i = 0; i <= last; ++i) { chain[i] = ChainRef{ch[i].sym, t, ch[i].len, 0}; t += ch[i].len; }
    const uint64_t E = hdr + (ch[last].end + 7) / 8;
    if (E + 8 > n) return FRISK_E_FORMAT;
    uint8_t tr[11] = {};
    const uint64_t after = n - E - 8;
    if ((rc = B.read(E, 8 + std::min<uint64_t>(after, 3), tr))) return rc;
    if (after) return after >= 10 && tr[8] == 0x1f && tr[9] == 0x8b && tr[10] == 8 ? FRISK_E_UNSUPPORTED : FRISK_E_FORMAT;
    if (rd32(tr + 4) != (uint32_t)t) return FRISK_E_FORMAT;
    if (stats) {
        uint64_t first = 0;
        for (size_t i = 1; i <= last; ++i) first += !repaired[i];
        stats[0] = N; stats[1] = first; stats[2] = n_repaired; stats[3] = over.size();
    }
    *text_len = t;
    uint8_t* text = nullptr;
    if ((rc = alloc_text(t, &text))) return rc;
    std::vector<uint32_t> crc(last + 1);
    bool bad = false;
    if ((rc = B.resolve(chain, text, crc, &bad))) return rc;
    if (bad) return FRISK_E_FORMAT;                       // a match before the first byte of the text
    uint32_t acc = 0;
    for (size_t i = 0; i <= last; ++i)
        if (chain[i].len) acc = multmodp(x8nmodp(chain[i].len), acc) ^ crc[i];
    return acc == rd32(tr) ? FRISK_OK : FRISK_E_FORMAT;
}

}  // namespace

int frisk_internal::gzip_inflate(const uint8_t* d_gz, const uint8_t* h_gz, uint64_t n,
                                 const std::function<int(uint64_t, uint8_t**)>& alloc_text, uint64_t* text_len, uint64_t stats[4],
                                 cudaStream_t st) {
    int rc = pool_ready();
    if (rc) return rc;
    DeviceBackend B(d_gz, h_gz, st);
    rc = inflate(B, n, alloc_text, text_len, stats);
    if (rc) {                                             // nothing of a failed call stays queued
        cudaStreamSynchronize(st);
        cudaGetLastError();
    }
    return rc;
}

extern "C" {

int frisk_b200_gzip_member(const uint8_t* gz, uint64_t n, uint64_t* payload_off, uint64_t* payload_len, uint32_t* crc,
                           uint32_t* isize) {
    if (!gz && n) return FRISK_E_INVALID;
    uint64_t off = 0;
    const int rc = parse_header(gz, n, n, &off);
    if (rc) return rc;
    if (payload_off) *payload_off = off;
    if (payload_len) *payload_len = n - 8 - off;
    if (crc) *crc = rd32(gz + n - 8);
    if (isize) *isize = rd32(gz + n - 4);
    return FRISK_OK;
}

int frisk_b200_gzip_inflate(const uint8_t* d_gz, uint64_t n, uint8_t* d_text, uint64_t text_cap, uint64_t* text_len,
                            uint64_t stats[4], void* stream) {
    if (!text_len || (!d_gz && n) || (!d_text && text_cap)) return FRISK_E_INVALID;
    if (frisk_b200_device_count() <= 0) return FRISK_E_NO_DEVICE;
    auto alloc = [&](uint64_t len, uint8_t** out) { *out = d_text; return len > text_cap ? FRISK_E_CAPACITY : FRISK_OK; };
    return frisk_internal::gzip_inflate(d_gz, nullptr, n, alloc, text_len, stats, (cudaStream_t)stream);
}

int frisk_b200_gzip_inflate_host(const uint8_t* gz, uint64_t n, uint8_t* text, uint64_t text_cap, uint64_t* text_len,
                                 uint64_t stats[4], void* stream) {
    (void)stream;
    if (!text_len || (!gz && n) || (!text && text_cap)) return FRISK_E_INVALID;
    HostBackend B(gz);
    auto alloc = [&](uint64_t len, uint8_t** out) { *out = text; return len > text_cap ? FRISK_E_CAPACITY : FRISK_OK; };
    try {
        return inflate(B, n, alloc, text_len, stats);
    } catch (...) {                                       // std::bad_alloc of the plan: nothing crosses the ABI
        return FRISK_E_CAPACITY;
    }
}

}  // extern "C"
