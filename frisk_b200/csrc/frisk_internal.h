// Shared by the translation units of libfrisk_b200.so; not part of the C ABI.
#ifndef FRISK_INTERNAL_H
#define FRISK_INTERNAL_H

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <functional>
#include <vector>

struct frisk_b200_fasta;

#define FRISK_CK(call)                                                        \
    do {                                                                      \
        cudaError_t e_ = (call);                                              \
        if (e_ != cudaSuccess) return frisk_internal::cuda_fail(e_, #call);   \
    } while (0)

namespace frisk_internal {

// records the CUDA error text for frisk_b200_last_cuda_error() and returns FRISK_E_CUDA
int cuda_fail(cudaError_t e, const char* what);

// once per device: let the default memory pool keep up to 32 GiB of freed cudaMallocAsync scratch (frisk_common.cu says why)
int pool_ready();
extern int g_ingest_exact, g_ingest_chunk_tiles;   // frisk_ingest.cu; set through frisk_b200_set_option

// Streamed FASTA open that also builds the planes (frisk_ingest.cu; used by frisk_b200_run_fasta).  While the text is
// still arriving, on_range (optional) is handed the plane words [d_word_range[0], d_word_range[1]) -- a DEVICE-side range --
// that became final: the caller counts them.  If the streamed attempt has to be abandoned (see frisk_b200_fasta_open),
// abandon() undoes what on_range accumulated, the text is opened and packed in one piece, and counted stays false.
struct IngestSink {
    std::function<int(const uint32_t* codes, const uint32_t* inv, const uint32_t* low, const unsigned long long* d_word_range,
                      uint64_t words_hint, cudaStream_t st)> on_range;
    std::function<int(cudaStream_t st)> abandon;
    // called once the last chunk's passes (and its on_range) are queued: the record table and the planes are complete in
    // stream order, the host has not seen anything yet -- whatever only needs DEVICE-side results can be queued here
    std::function<int(frisk_b200_fasta* h, cudaStream_t st)> on_complete;
    cudaEvent_t uploaded_mark = nullptr;     // recorded behind the last text chunk's copy
    bool counted = false;                    // out: on_range saw every word of [0, padded_len / 32 - 1)
};
// the device side of a handle's record table, for on_complete: lengths, offsets, capacity, and the ingest's counters
// (records at [kIngestRecords], non-upper-case bases at [kIngestNonUpper], lower-case acgt at [kIngestLower], "capacities
// exceeded" at [kIngestOverflow]; an adopted handle's {first, last} word of on_range at [kIngestRange]; kIngestCounters words)
enum { kIngestRecords = 0, kIngestNonUpper = 1, kIngestLower = 2, kIngestOverflow = 5, kIngestRange = 12, kIngestCounters = 14 };
bool fasta_open_was_streamed(const frisk_b200_fasta* h);     // false: the handle comes from the exact re-open
int fasta_device_table(const frisk_b200_fasta* h, const unsigned long long** d_len, const unsigned long long** d_scaf_off,
                       const unsigned long long** d_counters, uint64_t* rec_cap, const uint32_t** d_codes, const uint32_t** d_inv,
                       const uint32_t** d_low);
// what the bytes handed to an open are: the text, a BGZF buffer (frisk_b200_fasta_open_bgzf), one gzip member
// (frisk_b200_fasta_open_gzip) -- compressed input is inflated on the device into the text buffer -- or a UCSC .2bit file
// (frisk_b200_fasta_open_2bit), decoded on the device straight into the planes
enum TextFormat : int { kFmtText = 0, kFmtBgzf = 1, kFmtGzip = 2, kFmt2bit = 3 };
int fasta_open_planes(const char* text, uint64_t n, TextFormat fmt, cudaStream_t st, IngestSink* sink, frisk_b200_fasta** out);
// A genome whose record table and planes were built in device memory by an open other than the text ingest (frisk_twobit.cu).
// d_slab is one stream-ordered allocation holding every d_ pointer; d_counters has kIngestCounters words, with the records,
// overflow (0) and on_range's word range set, and nnTotal / lower-case counts that are final once the work queued on the
// open's stream is done.  Names index name_text.
struct AdoptedGenome {
    void* d_slab = nullptr;
    uint32_t *d_codes = nullptr, *d_inv = nullptr, *d_low = nullptr;
    unsigned long long *d_len = nullptr, *d_scaf_off = nullptr, *d_counters = nullptr;
    uint64_t rec_cap = 0, padded_len = 0, total = 0;
    std::vector<uint64_t> name_off, seq_len, scaf_off;
    std::vector<uint32_t> name_len;
    std::vector<char> name_text;
};
// frisk_ingest.cu: a handle takes g over (its slab is freed with the handle, or here on failure) and does what the text open
// does behind its last chunk: the planes go to sink->on_range (every word), the counters come back, sink->on_complete runs.
int fasta_adopt(AdoptedGenome& g, cudaStream_t st, IngestSink* sink, frisk_b200_fasta** out);
// frisk_twobit.cu: the open of a .2bit file (kFmt2bit)
int twobit_open(const char* buf, uint64_t n, cudaStream_t st, IngestSink* sink, frisk_b200_fasta** out);
// frisk_b200_bgzf_inflate's kernel (frisk_bgzf.cu); d_any_bad (nullable) receives a non-zero word when a member fails
int bgzf_inflate(const uint8_t* d_gz, const uint64_t* d_comp_off, const uint32_t* d_comp_len, const uint32_t* d_crc,
                 const uint64_t* d_text_off, uint64_t n_blocks, uint64_t text_len, uint8_t* d_text, uint32_t* d_block_status,
                 unsigned int* d_any_bad, cudaStream_t st);
// frisk_b200_gzip_inflate (frisk_gzip.cu) with the text buffer from alloc_text(text_len, &d_text), called once the length
// is known; h_gz (nullable) is a host copy of the member, read instead of d_gz for the header and trailer.  Synchronises st.
extern int g_gzip_chunk_bytes;                     // compressed bytes per nominal chunk (0 = default); frisk_b200_set_option
int gzip_inflate(const uint8_t* d_gz, const uint8_t* h_gz, uint64_t n, const std::function<int(uint64_t, uint8_t**)>& alloc_text,
                 uint64_t* text_len, uint64_t stats[4], cudaStream_t st);
// background count of a word range that lives in device memory (frisk_tables.cu); kmax <= FRISK_B200_FAST_K
int background_device_range(const uint32_t* codes, const uint32_t* inv, const uint32_t* low, const unsigned long long* d_word_range,
                            uint64_t words_hint, int kmax, int mask_host, uint64_t* fwd, cudaStream_t st);

// frisk_b200_windows on the device (frisk_windows.cu): window list, window count and genome space from a record table in
// device memory; d_n_rec / d_bad / d_non_upper point into the ingest's counters.  d_win_off == nullptr: count / space only.
int windows_device(const unsigned long long* d_len, const unsigned long long* d_scaf_off, const unsigned long long* d_n_rec,
                   const unsigned long long* d_bad, const unsigned long long* d_non_upper, uint64_t rec_cap, int w, int step,
                   int scaffolds_all, uint64_t cap, unsigned long long* d_first, unsigned long long* d_win_off, uint32_t* d_win_len,
                   unsigned long long* d_n_win, long long* d_space, cudaStream_t st);

// FASTA header rule of the reference (F:156): name = line.strip().strip('>').split()[0].
// The line starts at `line_start`; returns false for an empty name (the reference raises IndexError).
bool parse_header_name(const unsigned char* t, uint64_t n, uint64_t line_start, uint64_t* name_off, uint32_t* name_len);

// general path (frisk_general.cu): run-time K up to FRISK_B200_MAX_K, windows of any length
int general_background(const uint32_t* codes, const uint32_t* inv, const uint32_t* low, uint64_t w_lo, uint64_t w_hi, int K,
                       int mask_host, uint64_t* fwd, cudaStream_t st);
int general_finalize(const uint64_t* fwd, int K, int symmetric, uint64_t* tables, uint64_t* valid, cudaStream_t st);
int general_genome_ivom(const uint64_t* tables, int kmin, int K, int64_t space, double* ig, cudaStream_t st);
int general_score(const uint32_t* codes, const uint32_t* inv, const uint32_t* low, const uint64_t* win_off,
                  const uint32_t* win_len, uint64_t n_win, uint32_t max_len, const double* ig, int kmin, int K, int want_rip,
                  double* rows, uint32_t* status, uint16_t* dump, cudaStream_t st, const uint32_t* redo_src = nullptr,
                  int grid_cap = 0);

// FRISK_E_INVALID unless 1 <= kmin <= kmax; FRISK_E_UNSUPPORTED for kmax > FRISK_B200_MAX_K
int check_k(int kmin, int kmax);

// `return expr;` with the run-time kmax as the compile-time constant K (1..8); FRISK_E_UNSUPPORTED for any other kmax
#define DISPATCH_K(kmax, expr)                      \
    switch (kmax) {                                 \
        case 1: { constexpr int K = 1; return expr; } \
        case 2: { constexpr int K = 2; return expr; } \
        case 3: { constexpr int K = 3; return expr; } \
        case 4: { constexpr int K = 4; return expr; } \
        case 5: { constexpr int K = 5; return expr; } \
        case 6: { constexpr int K = 6; return expr; } \
        case 7: { constexpr int K = 7; return expr; } \
        case 8: { constexpr int K = 8; return expr; } \
        default: return FRISK_E_UNSUPPORTED;        \
    }

// most ranks a sharded finalize sums over (frisk_b200_finalize_ivom, frisk_b200_run_host_peers)
constexpr int kMaxPeers = 16;
// frisk_b200_finalize_ivom without its argument checks (the run paths of frisk_run.cu have made them).  space_dev
// (nullable, single GPU, kmax <= FRISK_B200_FAST_K): the genome space in device memory, read in place of `space`.
int finalize_ivom(const uint64_t* d_fwd, const uint64_t* const* d_fwd_peers, uint64_t* const* d_flag_peers, int rank, int world,
                  uint64_t epoch, int kmin, int kmax, int64_t space, const long long* space_dev, uint64_t* tables, uint64_t* valid,
                  double* ig, cudaStream_t st);

// Longest window the shared-memory window kernels hold: an 8,192-base buffer less 6 bases of look-ahead.
constexpr uint32_t kSmemMaxWindow = 8186u;

// The window kernels of frisk_b200_score and how one of them is instantiated for a call.  plan_score (frisk_score.cu)
// is the one place that chooses them, from (kmin, kmax, longest window, dump) and the kernel forced through
// frisk_b200_set_option.  variant: ROUNDS of the bucketed and direct kernels or PP of the nibble and extension kernels,
// positions per thread from the longest window (window_variant).  dump / allk pick the <DUMP, ALLK> instantiation.
enum class WinKernel { Small, Nibble, Direct, Bucket, Dense, NibbleExt, General };
struct WinPlan {
    WinKernel kind;
    int variant;
    bool dump, allk;
};
int plan_score(int kmin, int kmax, uint32_t max_win_len, bool dump, WinPlan* out);
int window_variant(WinKernel kind, uint32_t max_win_len);
// the instantiation of a window kernel template <..., DUMP, ALLK> a plan runs: the table dump and kmin > 1 share the generic
// <..., DUMP, false> one, the production default (no dump, kmin 1) has its own
#define FRISK_WIN_INSTANCE(p, kern, ...)                                                                      \
    ((p).dump ? (const void*)kern<__VA_ARGS__, true, false>                                                   \
              : ((p).allk ? (const void*)kern<__VA_ARGS__, false, true> : (const void*)kern<__VA_ARGS__, false, false>))

// How a persistent window kernel is launched: each CTA walks windows until none are left, grid = min(SMs x resident CTAs
// per SM, windows).  max_carveout: ask for the whole shared-memory carve-out instead of leaving the L1 / shared split to
// the driver's per-launch heuristic (a smaller split silently costs a CTA per SM).
struct LaunchShape {
    const void* fn;
    int threads;
    size_t smem;
    bool max_carveout;
};
// resident CTAs per SM of `s` on the current device; sets its attributes first (once per device, kernel and smem, cached)
int ctas_per_sm(const LaunchShape& s, int* out);
// one persistent launch of `s`; args as for cudaLaunchKernel
int launch_persistent(const LaunchShape& s, uint64_t n_win, void** args, cudaStream_t st);
int sm_count_cached();     // multiprocessors of the current device (0: none)

// The hand-over of the nibble, direct and extension kernels: the windows they cannot finish exactly are marked kRowRedo
// and re-done by a second launch behind them on the same stream.  body(redo) queues both launches.  The marks go into
// `status` when that is device memory, otherwise into stream-ordered scratch: when `status` is a pinned host buffer
// written over PCIe the second launch must not read its marks back across the bus one window at a time, and the k sweep
// (status == nullptr) has eight status arrays.  zero: the window count lives in device memory, so n_win is only the
// capacity and the second launch walks all of it -- scratch is used and cleared, marks beyond the real count read
// "nothing to redo".  The scratch is freed behind body's launches on every path.
constexpr uint32_t kRowRedo = 0x80000000u;
template <typename F>
int with_redo_marks(uint32_t* status, uint64_t n_win, bool zero, cudaStream_t st, F body) {
    uint32_t* scratch = nullptr;
    cudaPointerAttributes pa{};
    if (zero || !status || cudaPointerGetAttributes(&pa, status) != cudaSuccess || pa.type != cudaMemoryTypeDevice) {
        cudaGetLastError();                                  // a host pointer makes the query itself report an error
        int rc = pool_ready();
        if (rc) return rc;
        FRISK_CK(cudaMallocAsync((void**)&scratch, n_win * sizeof(uint32_t), st));
    }
    int rc = FRISK_OK;
    if (zero) {
        const cudaError_t e = cudaMemsetAsync(scratch, 0, n_win * sizeof(uint32_t), st);
        if (e != cudaSuccess) rc = cuda_fail(e, "cudaMemsetAsync(redo scratch)");
    }
    if (!rc) rc = body(scratch ? scratch : status);
    if (scratch) {                                           // stream-ordered: behind body's launches
        const cudaError_t e = cudaFreeAsync(scratch, st);
        if (!rc && e != cudaSuccess) return cuda_fail(e, "cudaFreeAsync(redo scratch)");
    }
    return rc;
}

// A *_shape function expects a K its kernel serves (a plan only picks a kernel for those); a score_* entry refuses any
// other K with FRISK_E_UNSUPPORTED.
//
// small-K kernel (frisk_small.cu): kmax 1..6, windows <= 65,535 bases.  redo_src: only the windows marked kRowRedo there.
LaunchShape small_shape(const WinPlan& p, int K);
int score_small(const WinPlan& p, const uint32_t* codes, const uint32_t* inv, const uint32_t* low, const uint64_t* win_off,
                const uint32_t* win_len, uint64_t n_win, const double* ig, int kmin, int K, int want_rip, double* rows,
                uint32_t* status, uint16_t* dump, cudaStream_t st, const uint32_t* redo_src = nullptr);
// bucketed kernel (frisk_bucket.cu): kmax 4..8, windows <= kSmemMaxWindow bases; its buffer is sized by max_len
LaunchShape bucket_shape(const WinPlan& p, int K, uint32_t max_len);
int score_bucket(const WinPlan& p, const uint32_t* codes, const uint32_t* inv, const uint32_t* low, const uint64_t* win_off,
                 const uint32_t* win_len, uint64_t n_win, uint32_t max_len, const double* ig, int kmin, int K, int want_rip,
                 double* rows, uint32_t* status, uint16_t* dump, cudaStream_t st, const uint32_t* redo_src = nullptr);
// The hand-over target of the direct and nibble kernels and of the k sweep (frisk_score.cu): the windows marked kRowRedo
// in redo_src, re-done on the small-K kernel for K <= 3 and on the bucketed kernel for K >= 4.
int score_bucket_redo(const uint32_t* codes, const uint32_t* inv, const uint32_t* low, const uint64_t* win_off,
                      const uint32_t* win_len, uint64_t n_win, uint32_t max_len, const double* ig, int kmin, int K, int want_rip,
                      double* rows, uint32_t* status, uint16_t* dump, const uint32_t* redo_src, cudaStream_t st);
// dense-table kernel (frisk_dense.cu): kmax 1..8, windows <= 65,535 bases; one CTA of dense_shape(K).threads per SM
LaunchShape dense_shape(int K);
int score_dense(const uint32_t* codes, const uint32_t* inv, const uint32_t* low, const uint64_t* win_off, const uint32_t* win_len,
                uint64_t n_win, uint32_t max_len, const double* ig, int kmin, int K, int want_rip, double* rows, uint32_t* status,
                uint16_t* dump, cudaStream_t st);

// kmax 9..12, windows <= kSmemMaxWindow bases (frisk_nibble_ext.cu): orders 1..8 as in the kmax-8 nibble kernel, orders
// 9..K from the observation that an 8-mer seen once has only unique extensions (the few repeated ones go through a
// shared-memory hash table).  What it cannot hold is re-done by general_score behind it.
LaunchShape ext_shape(const WinPlan& p);
int score_nibble_ext(const WinPlan& p, const uint32_t* codes, const uint32_t* inv, const uint32_t* low, const uint64_t* win_off,
                     const uint32_t* win_len, uint64_t n_win, uint32_t max_len, const double* ig, int kmin, int K, int want_rip,
                     double* rows, uint32_t* status, cudaStream_t st);

// direct score kernel (frisk_direct.cu): kmax 7, 8 and windows <= kSmemMaxWindow bases.  Windows it cannot finish exactly
// (a K-mer seen 256+ times, more than 64 N-boundary words) are re-done by score_bucket_redo.
LaunchShape direct_shape(const WinPlan& p, int K);
int score_direct(const WinPlan& p, const uint32_t* codes, const uint32_t* inv, const uint32_t* low, const uint64_t* win_off,
                 const uint32_t* win_len, uint64_t n_win, uint32_t max_len, const double* ig, int kmin, int K, int want_rip,
                 double* rows, uint32_t* status, uint16_t* dump, cudaStream_t st);

// nibble score kernel (frisk_nibble.cu): kmax 7, 8 and windows <= kSmemMaxWindow bases; one 4-bit counter per K-mer, one
// atomic per position, the first occurrence of a K-mer scores it.  Windows with a K-mer seen 16+ times (or more than 64
// N-boundary words) are re-done by the bucketed kernel, exactly like the direct kernel's hand-over.  n_win_dev: the window
// count in device memory, n_win its capacity.  It reads ig through a (K+1)-mer pair table it builds in stream-ordered scratch
// before its launch (frisk_nibble.cu); the hand-over reads ig itself.
LaunchShape nibble_shape(const WinPlan& p, int K);
int score_nibble(const WinPlan& p, const uint32_t* codes, const uint32_t* inv, const uint32_t* low, const uint64_t* win_off,
                 const uint32_t* win_len, uint64_t n_win, uint32_t max_len, const double* ig, int kmin, int K, int want_rip,
                 double* rows, uint32_t* status, uint16_t* dump, cudaStream_t st, const unsigned long long* n_win_dev = nullptr);
// the k sweep (BASELINE config C3): rows of kmax' = 1..8, kmin 1, from one pass over every window; ig / rows / status are
// HOST arrays of 8 device pointers
int score_sweep(const uint32_t* codes, const uint32_t* inv, const uint32_t* low, const uint64_t* win_off, const uint32_t* win_len,
                uint64_t n_win, uint32_t max_len, const double* const* ig, int want_rip, double* const* rows,
                uint32_t* const* status, cudaStream_t st);

}  // namespace frisk_internal

#endif
