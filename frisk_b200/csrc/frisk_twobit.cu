// frisk_b200 UCSC .2bit input: the packed bases, N blocks and soft-mask blocks of a twoBit file (versions 0 and 1, either
// byte order) decoded straight into the planes, bit for bit what frisk_b200_fasta_scan + frisk_b200_pack make of the same
// genome as FASTA (N blocks: every non-ACGT character; mask blocks: lower case).  Nothing is tokenised:
//   host      the parser checks every offset, count and length against the buffer before it reads, and produces the record
//             table (lengths, frisk_b200_pack_layout offsets, file offset of each record's packed DNA), the names, and one
//             run table of N and mask blocks in absolute plane coordinates with an exclusive scan of the 32-base plane
//             words each run touches
//   device    one copy of the file; twobit_runs_kernel gives one thread to each (run, word) item (a 3 Mbp N run is 94 K
//             threads, not one) and ORs the run's bits into inv (N) or low (mask); twobit_decode_kernel gives one thread to
//             each 32-base word: 8 source bytes remapped from T,C,A,G = 0..3 to the planes' A,T,G,C = 0..3 and byte-reversed,
//             codes cleared under inv, padding beyond the record ORed into inv, low = mask & ~inv, and the popcounts of inv
//             and low summed into the countN statistics
// frisk_b200_2bit_unpack_host runs the same plan, with the same per-word code, on the CPU.  The handle of a device open is
// made by frisk_ingest.cu's fasta_adopt, which hands the planes to the one-call path's count and device-only tail.
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <vector>

#include "../../include/frisk_b200.h"
#include "frisk_internal.h"

namespace {

constexpr uint32_t kSignature = 0x1A412743u;
constexpr uint64_t kMaskRun = 1ull << 63;          // run table: bit 63 of a run's start marks a mask block (else N)
constexpr int kTB = 256;                           // threads per block of both kernels

// ---- the parse ----------------------------------------------------------------------------------------------------------
struct Reader {
    const uint8_t* b;
    uint64_t n;
    bool swap;
    bool u32(uint64_t at, uint32_t* v) const {
        if (at > n || n - at < 4) return false;
        uint32_t x;
        memcpy(&x, b + at, 4);
        *v = swap ? __builtin_bswap32(x) : x;
        return true;
    }
    bool u64(uint64_t at, uint64_t* v) const {
        if (at > n || n - at < 8) return false;
        uint64_t x;
        memcpy(&x, b + at, 8);
        *v = swap ? __builtin_bswap64(x) : x;
        return true;
    }
};

struct Plan {
    std::vector<uint64_t> name_off, seq_len, dna_off, scaf_off;   // name_off: into the file
    std::vector<uint32_t> name_len;
    uint64_t total = 0, padded_len = 128;
    // runs: [start | kMaskRun, end) in absolute plane bases; scan[k] = plane words touched by runs before k (n_runs + 1)
    std::vector<uint64_t> run_a, run_b, scan;
};

// Header, index and record headers; with runs, the layout and the run table too.  FRISK_E_FORMAT for anything the format
// does not allow, before a byte beyond the buffer is read.
int parse(const uint8_t* buf, uint64_t n, bool runs, Plan* p) {
    if (!buf || n < 16) return FRISK_E_FORMAT;
    uint32_t sig;
    memcpy(&sig, buf, 4);
    Reader r{buf, n, false};
    if (sig != kSignature) {
        if (__builtin_bswap32(sig) != kSignature) return FRISK_E_FORMAT;
        r.swap = true;
    }
    uint32_t version = 0, count = 0;
    r.u32(4, &version);
    r.u32(8, &count);
    if (version > 1) return FRISK_E_FORMAT;
    uint64_t at = 16;
    std::vector<uint64_t> rec_off;
    for (uint32_t i = 0; i < count; ++i) {
        if (at >= n) return FRISK_E_FORMAT;
        const uint32_t ns = buf[at];
        if (ns == 0) return FRISK_E_FORMAT;                             // an empty name (the reference raises IndexError, F:156)
        if (n - at - 1 < ns) return FRISK_E_FORMAT;
        p->name_off.push_back(at + 1);
        p->name_len.push_back(ns);
        at += 1 + ns;
        uint64_t off;
        if (version == 0) {
            uint32_t o32;
            if (!r.u32(at, &o32)) return FRISK_E_FORMAT;
            off = o32;
            at += 4;
        } else {
            if (!r.u64(at, &off)) return FRISK_E_FORMAT;
            at += 8;
        }
        rec_off.push_back(off);
    }
    const uint64_t R = count;
    p->seq_len.resize(R);
    p->dna_off.resize(R);
    for (uint64_t i = 0; i < R; ++i) {                                 // records: sizes and bounds
        uint64_t q = rec_off[i];
        uint32_t dna = 0, nb = 0, mb = 0;
        if (!r.u32(q, &dna) || !r.u32(q + 4, &nb)) return FRISK_E_FORMAT;
        q += 8;
        if ((n - q) / 8 < nb) return FRISK_E_FORMAT;                  // (q <= n: the reads above succeeded)
        const uint64_t n_starts = q;
        q += 8ull * nb;
        if (!r.u32(q, &mb)) return FRISK_E_FORMAT;
        q += 4;
        if ((n - q) / 8 < mb) return FRISK_E_FORMAT;
        const uint64_t m_starts = q;
        q += 8ull * mb;
        uint32_t reserved = 0;
        if (!r.u32(q, &reserved)) return FRISK_E_FORMAT;
        q += 4;
        const uint64_t bytes = ((uint64_t)dna + 3) / 4;
        if (n - q < bytes) return FRISK_E_FORMAT;
        p->seq_len[i] = dna;
        p->dna_off[i] = q;
        p->total += dna;
        for (int kind = 0; kind < 2; ++kind) {                         // blocks: inside the sequence, zero-size ones ignored
            const uint64_t s0 = kind ? m_starts : n_starts;
            const uint32_t cnt = kind ? mb : nb;
            for (uint32_t k = 0; k < cnt; ++k) {
                uint32_t st = 0, sz = 0;
                r.u32(s0 + 4ull * k, &st);
                r.u32(s0 + 4ull * cnt + 4ull * k, &sz);
                if ((uint64_t)st + sz > dna) return FRISK_E_FORMAT;
            }
        }
    }
    if (!runs) return FRISK_OK;
    p->scaf_off.resize(R);
    int rc = frisk_b200_pack_layout(p->seq_len.data(), R, p->scaf_off.data(), &p->padded_len);
    if (rc) return rc;
    p->scan.push_back(0);
    for (uint64_t i = 0; i < R; ++i) {
        uint64_t q = rec_off[i] + 4;
        uint32_t nb = 0, mb = 0;
        r.u32(q, &nb);
        const uint64_t n_starts = q + 4;
        r.u32(n_starts + 8ull * nb, &mb);
        const uint64_t m_starts = n_starts + 8ull * nb + 4;
        for (int kind = 0; kind < 2; ++kind) {
            const uint64_t s0 = kind ? m_starts : n_starts;
            const uint32_t cnt = kind ? mb : nb;
            for (uint32_t k = 0; k < cnt; ++k) {
                uint32_t st = 0, sz = 0;
                r.u32(s0 + 4ull * k, &st);
                r.u32(s0 + 4ull * cnt + 4ull * k, &sz);
                if (!sz) continue;
                const uint64_t a = p->scaf_off[i] + st, b = a + sz;
                p->run_a.push_back(a | (kind ? kMaskRun : 0ull));
                p->run_b.push_back(b);
                p->scan.push_back(p->scan.back() + ((b - 1) >> 5) - (a >> 5) + 1);
            }
        }
    }
    return FRISK_OK;
}

// ---- per-item and per-word work, shared by the kernels and the host decoder ---------------------------------------------
// bits of run [a, b) in plane word `word`
__host__ __device__ __forceinline__ uint32_t run_bits(uint64_t a, uint64_t b, uint64_t word) {
    const uint64_t w0 = word << 5;
    const uint32_t s = (uint32_t)((a > w0 ? a : w0) - w0), e = (uint32_t)((b < w0 + 32 ? b : w0 + 32) - w0);
    return (0xffffffffu >> s) & (e == 32 ? 0xffffffffu : ~(0xffffffffu >> e));
}

// the run and word of item i: run k with scan[k] <= i < scan[k + 1]
__host__ __device__ __forceinline__ void run_item(const uint64_t* scan, uint64_t n_runs, const uint64_t* run_a, uint64_t i,
                                                  uint64_t* k_out, uint64_t* word) {
    uint64_t lo = 0, hi = n_runs;                                       // scan[lo] <= i < scan[hi]
    while (hi - lo > 1) {
        const uint64_t mid = (lo + hi) >> 1;
        if (scan[mid] <= i) lo = mid; else hi = mid;
    }
    *k_out = lo;
    *word = ((run_a[lo] & ~kMaskRun) >> 5) + (i - scan[lo]);
}

__host__ __device__ __forceinline__ uint32_t bswap32(uint32_t x) {
    return (x >> 24) | ((x >> 8) & 0xff00u) | ((x << 8) & 0xff0000u) | (x << 24);
}
// four bases of a twoBit byte (T=0, C=1, A=2, G=3) in the planes' codes (A=0, T=1, G=2, C=3): hi = old lo, lo = ~old hi
__host__ __device__ __forceinline__ uint32_t remap(uint32_t x) {
    return ((x & 0x55555555u) << 1) | ((~x & 0xAAAAAAAAu) >> 1);
}
// 16 mask bits (bit 15 - j = base j) -> the two code bits of every base (bits 31 - 2j, 30 - 2j)
__host__ __device__ __forceinline__ uint32_t spread16(uint32_t x) {
    x = (x | (x << 8)) & 0x00FF00FFu;
    x = (x | (x << 4)) & 0x0F0F0F0Fu;
    x = (x | (x << 2)) & 0x33333333u;
    x = (x | (x << 1)) & 0x55555555u;
    return x | (x << 1);
}

struct Word { uint32_t c0, c1, inv, low; };
// One 32-base plane word: its first base is base p0 of a record of `len` bases; src_lo / src_hi are the 8 file bytes of
// bases p0 .. p0 + 31 as little-endian words (ignored where p0 >= len); runs_inv / runs_low: what the run expansion set.
__host__ __device__ __forceinline__ Word decode_word(uint32_t src_lo, uint32_t src_hi, uint64_t p0, uint64_t len, uint32_t runs_inv,
                                                     uint32_t runs_low) {
    const uint64_t v = len > p0 ? (len - p0 < 32 ? len - p0 : 32) : 0;      // data bases in the word, padding behind them
    const uint32_t iv = runs_inv | (v == 32 ? 0u : 0xffffffffu >> v);
    Word o;
    o.c0 = remap(bswap32(src_lo)) & ~spread16(iv >> 16);
    o.c1 = remap(bswap32(src_hi)) & ~spread16(iv & 0xffffu);
    o.inv = iv;
    o.low = runs_low & ~iv;
    return o;
}

// record of plane base `pos`: the last r with scaf_off[r] <= pos (R >= 1)
__host__ __device__ __forceinline__ uint64_t record_of(const uint64_t* scaf_off, uint64_t R, uint64_t pos) {
    uint64_t lo = 0, hi = R;
    while (hi - lo > 1) {
        const uint64_t mid = (lo + hi) >> 1;
        if (scaf_off[mid] <= pos) lo = mid; else hi = mid;
    }
    return lo;
}

// ---- kernels --------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kTB)
twobit_runs_kernel(const uint64_t* __restrict__ run_a, const uint64_t* __restrict__ run_b, const uint64_t* __restrict__ scan,
                   uint64_t n_runs, uint32_t* __restrict__ inv, uint32_t* __restrict__ low) {
    const uint64_t items = scan[n_runs];
    for (uint64_t i = (uint64_t)blockIdx.x * kTB + threadIdx.x; i < items; i += (uint64_t)gridDim.x * kTB) {
        uint64_t k, word;
        run_item(scan, n_runs, run_a, i, &k, &word);
        const uint64_t a = run_a[k];
        const uint32_t bits = run_bits(a & ~kMaskRun, run_b[k], word);
        uint32_t* const plane = (a & kMaskRun) ? low : inv;
        if (bits == 0xffffffffu) plane[word] = bits;                   // (whatever else lands there, the word ends all ones)
        else atomicOr(&plane[word], bits);
    }
}

// counters[ctr_non_upper] starts at -(padded_len - totalLen): the padding bits of inv are taken off the popcount in advance
__global__ void __launch_bounds__(kTB)
twobit_decode_kernel(const uint8_t* __restrict__ file, const uint64_t* __restrict__ dna_off, const unsigned long long* __restrict__ len,
                     const unsigned long long* __restrict__ scaf_off, uint64_t R, uint64_t n_words, uint32_t* __restrict__ codes,
                     uint32_t* __restrict__ inv, uint32_t* __restrict__ low, unsigned long long* __restrict__ counters,
                     int ctr_non_upper, int ctr_lower) {
    __shared__ uint32_t s_sum[2][kTB / 32];
    uint32_t n_inv = 0, n_low = 0;                                     // (< 2^32: a thread covers far fewer than 2^27 words)
    for (uint64_t w = (uint64_t)blockIdx.x * kTB + threadIdx.x; w < n_words; w += (uint64_t)gridDim.x * kTB) {
        const uint64_t pos = w << 5;
        uint64_t p0 = 0, rl = 0;
        uint32_t lo = 0, hi = 0;
        if (R) {
            const uint64_t r = record_of(reinterpret_cast<const uint64_t*>(scaf_off), R, pos);
            p0 = pos - scaf_off[r];
            rl = len[r];
            if (p0 < rl) {                                              // bytes dna_off + p0/4 .. + 7, byte- but not word-aligned
                const uint64_t at = dna_off[r] + (p0 >> 2);
                const uint32_t* q = reinterpret_cast<const uint32_t*>(file + (at & ~3ull));
                const uint32_t sh = 8u * (uint32_t)(at & 3u), x0 = q[0], x1 = q[1], x2 = q[2];
                lo = __funnelshift_r(x0, x1, sh);
                hi = __funnelshift_r(x1, x2, sh);
            }
        }
        const Word o = decode_word(lo, hi, p0, rl, inv[w], low[w]);
        *reinterpret_cast<uint2*>(codes + 2 * w) = make_uint2(o.c0, o.c1);
        inv[w] = o.inv;
        low[w] = o.low;
        n_inv += __popc(o.inv);
        n_low += __popc(o.low);
    }
    n_inv = __reduce_add_sync(0xffffffffu, n_inv);
    n_low = __reduce_add_sync(0xffffffffu, n_low);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { s_sum[0][warp] = n_inv; s_sum[1][warp] = n_low; }
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long a = 0, b = 0;
        for (int k = 0; k < kTB / 32; ++k) { a += s_sum[0][k]; b += s_sum[1][k]; }
        if (a + b) atomicAdd(&counters[ctr_non_upper], a + b);         // nnTotal = |N| + nLower
        if (b) atomicAdd(&counters[ctr_lower], b);
    }
}

// ---- the device open -------------------------------------------------------------------------------------------------------
template <typename T>
void carve(char*& cursor, T*& out, uint64_t bytes) {
    out = reinterpret_cast<T*>(cursor);
    cursor += (bytes + 255) & ~255ull;
}

int grid_for(uint64_t items) {
    const uint64_t per_sm = 8;                                          // resident blocks of 256 threads asked for per SM
    const uint64_t cap = std::max<uint64_t>(1, (uint64_t)frisk_internal::sm_count_cached() * per_sm);
    return (int)std::max<uint64_t>(1, std::min<uint64_t>((items + kTB - 1) / kTB, cap));
}

}  // namespace

int frisk_internal::twobit_open(const char* buf, uint64_t n, cudaStream_t st, IngestSink* sink, frisk_b200_fasta** out) {
    *out = nullptr;
    int rc = pool_ready();
    if (rc) return rc;
    Plan p;
    const uint8_t* const b = reinterpret_cast<const uint8_t*>(buf);
    if ((rc = parse(b, n, true, &p))) return rc;
    const uint64_t R = p.seq_len.size(), P = p.padded_len, W = P / 32, n_runs = p.run_a.size();
    const uint64_t rec_cap = std::max<uint64_t>(R, 1);

    // what the handle keeps: counters, record table, planes (inv and low side by side: one memset)
    AdoptedGenome g;
    char* cur = nullptr;
    const uint64_t slab_bytes = kIngestCounters * 8 + 2 * (rec_cap * 8) + P / 4 + 2 * (P / 8) + 5 * 256;
    FRISK_CK(cudaMallocAsync(&g.d_slab, slab_bytes, st));
    cur = (char*)g.d_slab;
    carve(cur, g.d_counters, kIngestCounters * 8);
    carve(cur, g.d_len, rec_cap * 8);
    carve(cur, g.d_scaf_off, rec_cap * 8);
    carve(cur, g.d_codes, P / 4);
    carve(cur, g.d_inv, P / 8);
    g.d_low = g.d_inv + W;                                              // (P / 8 is a multiple of 16 bytes)
    // what is freed behind the decode: the file (+ slack for the decode's aligned loads), packed-DNA offsets, run table
    void* scratch = nullptr;
    const uint64_t file_bytes = (n + 16 + 255) & ~255ull;
    const uint64_t tab_words = rec_cap + 2 * n_runs + n_runs + 1;
    auto fail = [&](int code) {
        if (scratch) cudaFreeAsync(scratch, st);
        cudaFreeAsync(g.d_slab, st);
        return code;
    };
    cudaError_t e = cudaMallocAsync(&scratch, file_bytes + tab_words * 8, st);
    if (e != cudaSuccess) { scratch = nullptr; return fail(cuda_fail(e, "cudaMallocAsync(2bit scratch)")); }
    uint8_t* const d_file = (uint8_t*)scratch;
    uint64_t* const d_tab = (uint64_t*)(d_file + file_bytes);
    uint64_t *d_dna_off = d_tab, *d_run_a = d_tab + rec_cap, *d_run_b = d_run_a + n_runs, *d_scan = d_run_b + n_runs;

    std::vector<unsigned long long> head(kIngestCounters + 2 * rec_cap, 0ull);   // counters, lengths, offsets
    head[kIngestRecords] = R;
    head[kIngestNonUpper] = 0ull - (unsigned long long)(P - p.total);
    head[kIngestRange] = 0;
    head[kIngestRange + 1] = W - 1;                                    // on_range: every word but the last (look-ahead only)
    std::vector<uint64_t> tab(tab_words, 0);
    for (uint64_t r = 0; r < R; ++r) {
        head[kIngestCounters + r] = p.seq_len[r];
        head[kIngestCounters + rec_cap + r] = p.scaf_off[r];
        tab[r] = p.dna_off[r];
    }
    std::copy(p.run_a.begin(), p.run_a.end(), tab.begin() + rec_cap);
    std::copy(p.run_b.begin(), p.run_b.end(), tab.begin() + rec_cap + n_runs);
    std::copy(p.scan.begin(), p.scan.end(), tab.begin() + rec_cap + 2 * n_runs);
    auto queue = [&]() -> int {
        FRISK_CK(cudaMemsetAsync(g.d_inv, 0, P / 4, st));
        FRISK_CK(cudaMemsetAsync(d_file + n, 0, 16, st));
        FRISK_CK(cudaMemcpyAsync(g.d_counters, head.data(), kIngestCounters * 8, cudaMemcpyHostToDevice, st));
        FRISK_CK(cudaMemcpyAsync(g.d_len, head.data() + kIngestCounters, rec_cap * 8, cudaMemcpyHostToDevice, st));
        FRISK_CK(cudaMemcpyAsync(g.d_scaf_off, head.data() + kIngestCounters + rec_cap, rec_cap * 8, cudaMemcpyHostToDevice, st));
        FRISK_CK(cudaMemcpyAsync(d_tab, tab.data(), tab_words * 8, cudaMemcpyHostToDevice, st));
        if (n_runs) {
            twobit_runs_kernel<<<grid_for(p.scan.back()), kTB, 0, st>>>(d_run_a, d_run_b, d_scan, n_runs, g.d_inv, g.d_low);
            FRISK_CK(cudaGetLastError());
        }
        FRISK_CK(cudaMemcpyAsync(d_file, b, n, cudaMemcpyHostToDevice, st));
        twobit_decode_kernel<<<grid_for(W), kTB, 0, st>>>(d_file, d_dna_off, g.d_len, g.d_scaf_off, R, W, g.d_codes, g.d_inv, g.d_low,
                                                          g.d_counters, kIngestNonUpper, kIngestLower);
        FRISK_CK(cudaGetLastError());
        if (sink && sink->uploaded_mark) FRISK_CK(cudaEventRecord(sink->uploaded_mark, st));   // file uploaded and decoded
        return FRISK_OK;
    };
    if ((rc = queue())) return fail(rc);
    e = cudaFreeAsync(scratch, st);                                     // stream-ordered: behind the decode
    scratch = nullptr;
    if (e != cudaSuccess) return fail(cuda_fail(e, "cudaFreeAsync(2bit scratch)"));
    g.padded_len = P;
    g.rec_cap = rec_cap;
    g.total = p.total;
    g.seq_len = std::move(p.seq_len);
    g.scaf_off = std::move(p.scaf_off);
    g.name_off.resize(R);
    g.name_len = std::move(p.name_len);
    uint64_t total_names = 0;
    for (uint64_t r = 0; r < R; ++r) total_names += g.name_len[r];
    g.name_text.resize(total_names);
    for (uint64_t r = 0, o = 0; r < R; ++r) {
        memcpy(g.name_text.data() + o, buf + p.name_off[r], g.name_len[r]);
        g.name_off[r] = o;
        o += g.name_len[r];
    }
    return fasta_adopt(g, st, sink, out);
}

extern "C" {

int frisk_b200_2bit_records(const uint8_t* buf, uint64_t n, uint64_t cap, uint64_t* name_off, uint32_t* name_len, uint64_t* seq_len,
                            uint64_t* n_records, uint64_t* bases) {
    if (!n_records || (!buf && n)) return FRISK_E_INVALID;
    Plan p;
    int rc;
    try {
        rc = parse(buf, n, false, &p);
    } catch (...) {
        return FRISK_E_CAPACITY;
    }
    if (rc) return rc;
    const uint64_t R = p.seq_len.size();
    *n_records = R;
    if (bases) *bases = p.total;
    if (R > cap && (name_off || name_len || seq_len)) return FRISK_E_CAPACITY;
    for (uint64_t r = 0; r < R; ++r) {
        if (name_off) name_off[r] = p.name_off[r];
        if (name_len) name_len[r] = p.name_len[r];
        if (seq_len) seq_len[r] = p.seq_len[r];
    }
    return FRISK_OK;
}

int frisk_b200_2bit_unpack_host(const uint8_t* buf, uint64_t n, uint64_t padded_len, uint32_t* codes, uint32_t* inv, uint32_t* low,
                                uint64_t stats[3]) {
    if (!codes || !inv || !stats || (!buf && n)) return FRISK_E_INVALID;
    Plan p;
    int rc;
    try {
        rc = parse(buf, n, true, &p);
        if (rc) return rc;
        if (padded_len != p.padded_len) return FRISK_E_INVALID;
        const uint64_t W = padded_len / 32, R = p.seq_len.size(), n_runs = p.run_a.size();
        std::vector<uint32_t> mask(W, 0);
        memset(inv, 0, W * 4);
        for (uint64_t i = 0; i < p.scan.back(); ++i) {                 // the run expansion, one (run, word) item at a time
            uint64_t k, word;
            run_item(p.scan.data(), n_runs, p.run_a.data(), i, &k, &word);
            const uint64_t a = p.run_a[k];
            ((a & kMaskRun) ? mask.data() : inv)[word] |= run_bits(a & ~kMaskRun, p.run_b[k], word);
        }
        stats[0] = p.total; stats[1] = 0; stats[2] = 0;
        uint64_t n_inv = 0;
        for (uint64_t w = 0; w < W; ++w) {                             // the decode, one 32-base word at a time
            uint64_t p0 = 0, rl = 0;
            uint32_t src[2] = {0, 0};
            if (R) {
                const uint64_t r = record_of(p.scaf_off.data(), R, w << 5);
                p0 = (w << 5) - p.scaf_off[r];
                rl = p.seq_len[r];
                if (p0 < rl) {
                    const uint64_t at = p.dna_off[r] + (p0 >> 2);
                    memcpy(src, buf + at, (size_t)std::min<uint64_t>(8, n - at));
                }
            }
            const Word o = decode_word(src[0], src[1], p0, rl, inv[w], mask[w]);
            codes[2 * w] = o.c0; codes[2 * w + 1] = o.c1;
            inv[w] = o.inv;
            mask[w] = o.low;
            n_inv += (uint64_t)__builtin_popcount(o.inv);
            stats[2] += (uint64_t)__builtin_popcount(o.low);
        }
        stats[1] = n_inv - (padded_len - p.total) + stats[2];
        if (low) memcpy(low, mask.data(), W * 4);
        else if (stats[2]) return FRISK_E_FORMAT;                      // (as frisk_b200_pack: lower case but no plane for it)
    } catch (...) {
        return FRISK_E_CAPACITY;
    }
    return FRISK_OK;
}

}  // extern "C"
