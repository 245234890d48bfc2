/*
 * frisk_b200 -- C ABI of the B200-native frisk hot path (k-mer background tables + per-window
 * IVOM/KLD scoring).  Plain pointers and sizes only; no C++/torch types cross this boundary.
 *
 * The reference (Adamtaranto/frisk) has no FFI of its own: its hot path is a set of Python
 * functions called from main() (frisk/__init__.py, "F:" below).  Every entry point here names
 * the reference code it replaces; INTEGRATION.md shows the ctypes binding a frisk maintainer
 * would add.  Conventions:
 *   - return 0 on success, a negative FRISK_E_* code otherwise (never throws, never exits);
 *     frisk_b200_strerror() explains a code, frisk_b200_last_cuda_error() the CUDA detail;
 *   - "d_" pointers are device memory owned by the caller (e.g. torch tensors' data_ptr());
 *     the library never frees caller memory;
 *   - `stream` is a cudaStream_t passed as void*; device entry points only enqueue work on it;
 *   - k-mer table index = base-4 number, digits A=0,T=1,G=2,C=3, first base most significant:
 *     exactly the key order of the reference's dict tables (F:70, F:253-274).
 *
 * Packed sequence layout ("planes"), shared by host and device:
 *   codes: uint32 words, 16 bases/word, base j of a word in bits [31-2j, 30-2j] (big-endian),
 *          invalid bases coded 0;
 *   inv  : uint32 words, 32 bases/word, base j at bit 31-j; 1 = not one of ACGTacgt (or padding);
 *   low  : same layout; 1 = lower-case acgt (soft-masked).  May be NULL when the input has none.
 *   Scaffold i starts at base offset scaf_off[i] (a multiple of 128) and is followed by >= 1
 *   padding base; padded_len is a multiple of 128 and includes >= 128 trailing padding bases.
 *   codes has padded_len/16 words, inv/low padded_len/32 words.
 */
#ifndef FRISK_B200_H
#define FRISK_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FRISK_B200_ABI_VERSION 2              /* 2: round 2 -- run_fasta, fasta handles own their planes, score sweep, timing mark 5 */
#define FRISK_B200_MAX_K 12              /* largest supported --maxWordSize (K <= 8: shared-memory kernels; 9..12: general path) */
#define FRISK_B200_FAST_K 8              /* ... served by the tuned shared-memory kernels */
#define FRISK_B200_MAX_WINDOW 0x7fffffff /* largest window length (<= 65,535: shared-memory kernels; longer: general path) */

enum {
    FRISK_OK = 0,
    FRISK_E_INVALID = -1,     /* bad argument (null pointer, kmin > kmax, ...) */
    FRISK_E_UNSUPPORTED = -2, /* kmax > FRISK_B200_MAX_K, window longer than FRISK_B200_MAX_WINDOW, > 2^32-1 windows */
    FRISK_E_CUDA = -3,        /* a CUDA call failed; see frisk_b200_last_cuda_error() */
    FRISK_E_NO_DEVICE = -4,   /* no CUDA device: there is deliberately no CPU fallback */
    FRISK_E_CAPACITY = -5,    /* an output array is too small; the required count is still reported */
    FRISK_E_FORMAT = -6       /* malformed FASTA */
};

/* Per-window status bits written by frisk_b200_score (0 = a normal row). */
#define FRISK_ROW_KLD_ZERODIV 1u /* the reference would raise ZeroDivisionError in IvomBuild (F:401-437) */
#define FRISK_ROW_GC_ZERODIV 2u  /* ... in calcGC (F:136): no upper-case base in the window */
#define FRISK_ROW_LOG_DOMAIN 4u  /* ... ValueError in KLD's math.log (F:470) */
#define FRISK_ROW_EXCLUDED 8u    /* dropped by the >= 30 % unresolved rule (F:213, F:238): not a row */

const char *frisk_b200_strerror(int code);
const char *frisk_b200_last_cuda_error(void);
int frisk_b200_abi_version(void);
/* Number of CUDA devices visible (0 when none / no driver). */
int frisk_b200_device_count(void);

/* Number of table entries for orders kmin..kmax: sum 4^k (F:267-274 rangeMaps). */
uint64_t frisk_b200_table_size(int kmin, int kmax);

/* ------------------------------------------------------------------ host side: ingest (F:139-164, F:106-118)
 *
 * frisk_b200_fasta_scan: one pass over FASTA text, replaces iterFasta's record splitting
 * (F:148-163).  Record i has its name at text[name_off[i] .. name_off[i]+name_len[i]) (first
 * whitespace token after stripping '>' characters, F:156), its sequence lines inside
 * text[body_off[i] .. body_end[i]) and seq_len[i] characters after the line ends are stripped.  Whitespace INSIDE a
 * sequence line -- which the reference keeps as a character of the sequence (F:149 strips only the ends) and real
 * FASTA never has -- is refused with FRISK_E_FORMAT, here and in frisk_b200_fasta_open, instead of silently shifting
 * every coordinate behind it.
 * Outputs may be NULL to only count.  *n_records always receives the record count;
 * FRISK_E_CAPACITY if cap is too small.
 */
int frisk_b200_fasta_scan(const char *text, uint64_t n, uint64_t cap, uint64_t *name_off, uint32_t *name_len,
                          uint64_t *body_off, uint64_t *body_end, uint64_t *seq_len, uint64_t *n_records);

/* Layout of n scaffolds of the given lengths: fills scaf_off[n] and *padded_len. */
int frisk_b200_pack_layout(const uint64_t *scaf_len, uint64_t n, uint64_t *scaf_off, uint64_t *padded_len);

/*
 * frisk_b200_pack: 2-bit pack scaffolds into the planes (host buffers, ideally pinned).
 * Scaffold i's characters are src[src_off[i] .. src_end[i]) with ASCII whitespace skipped (so a
 * FASTA body can be packed in place); exactly scaf_len[i] non-space characters are expected
 * (FRISK_E_FORMAT otherwise).  low may be NULL only if the caller knows there is no lower case
 * (then *n_lower reports how many were seen and FRISK_E_FORMAT is returned if any).
 * stats[0] = totalLen (F:323), stats[1] = nnTotal: characters that are not upper-case ATGC
 * (F:106-118 countN, case-sensitive), stats[2] = number of lower-case acgt.
 * threads <= 0 means "all hardware threads".
 */
int frisk_b200_pack(const char *src, const uint64_t *src_off, const uint64_t *src_end, const uint64_t *scaf_len,
                    const uint64_t *scaf_off, uint64_t n, uint64_t padded_len, uint32_t *codes, uint32_t *inv,
                    uint32_t *low, uint64_t stats[3], int threads);

/*
 * frisk_b200_windows: candidate windows per crawlGenome (F:194-251) WITHOUT the 30 % filter
 * (the score kernel applies it and flags FRISK_ROW_EXCLUDED, so no second pass over the bases is
 * needed): minimum-size rule (F:211, F:222), j = 0, step, ... (F:228), tail jump-back and its
 * sticky coordinates (F:230-232, F:243), 1-based inclusive coords (F:245), --scaffoldsAll rescue
 * (F:211-221).  win_off is the absolute base offset in the packed planes.  Arrays may be NULL to
 * only count; *n_windows always receives the count.
 */
int frisk_b200_windows(const uint64_t *scaf_len, const uint64_t *scaf_off, uint64_t n_scaf, int w, int step,
                       int scaffolds_all, uint64_t cap, uint64_t *win_off, uint32_t *win_len, uint32_t *win_scaf,
                       int64_t *win_start, int64_t *win_stop, uint64_t *n_windows);

/*
 * frisk_b200_format_rows (host, threads): the body of the reference's raw_window_scores.bed (F:1493):
 * per row "name \t start \t stop \t v0 ... \n" with the first n_values (2: windowKLD, GC; 5: + PI, SI,
 * CRI) of the row's five doubles, every float written exactly as Python 3's str(float) writes it
 * (shortest round-trip digits, "1e-05"-style exponents, "nan"/"inf", ".0" on integral values).
 * Row i's name is names[name_off[row_name[i]] ..+ name_len[row_name[i]]).  out == NULL only
 * reports *n_bytes; FRISK_E_CAPACITY if cap is too small.  A 1.2 M-row table takes seconds in a
 * Python loop and tens of milliseconds here.
 */
int frisk_b200_format_rows(const char *names, const uint64_t *name_off, const uint32_t *name_len,
                           const uint32_t *row_name, const int64_t *start, const int64_t *stop, const double *rows,
                           uint64_t n_rows, int n_values, char *out, uint64_t cap, uint64_t *n_bytes, int threads);

/*
 * Host helpers of the 2-state HMM segmentation (F:1536-1548) for installations without hmmlearn: a
 * deterministic 1-D, 2-state Gaussian HMM.  frisk_b200_hmm2_fit: Baum-Welch from uniform start/transition
 * probabilities, means = means of the lower/upper half of the sorted data, variances = data variance +
 * min_covar; at most n_iter iterations, stops when the log-likelihood gains less than tol.  trans is
 * row-major [from][to].  frisk_b200_hmm2_viterbi: the most likely state path (0/1 per observation).
 */
int frisk_b200_hmm2_fit(const double *x, uint64_t n, int n_iter, double tol, double min_covar, double start[2],
                        double trans[4], double mean[2], double var[2]);
int frisk_b200_hmm2_viterbi(const double *x, uint64_t n, const double start[2], const double trans[4],
                            const double mean[2], const double var[2], int32_t *path);

/* ------------------------------------------------------------------ device side
 *
 * frisk_b200_background: forward-strand k-mer counts of the packed bases [first_base, last_base)
 * (multiples of 32) -- the counting half of computeKmers(genomeMode=True), F:321-351.  ADDS into
 * d_fwd, a uint64 array of frisk_b200_table_size(1, kmax) entries (orders 1..kmax concatenated):
 * order kmax holds the count of every position whose kmax-word is valid, order x < kmax only the
 * positions whose longest valid word has length exactly x (scaffold ends, N boundaries).
 * frisk_b200_finalize_tables turns this into the reference's tables.  mask_host != 0 drops words
 * containing lower-case bases (--maskHost, F:336).  Zero d_fwd before the first call; ranks of a
 * multi-GPU job sum their d_fwd (one allreduce) before finalising.
 */
int frisk_b200_background(const uint32_t *d_codes, const uint32_t *d_inv, const uint32_t *d_low, uint64_t first_base,
                          uint64_t last_base, int kmax, int mask_host, uint64_t *d_fwd, void *stream);

/*
 * frisk_b200_finalize_tables: F_x = full forward count of order x (marginals of order x+1 plus
 * the short-word counts in d_fwd).  symmetric != 0 (genomeMode or sym, F:350): d_tables[x][kmer]
 * = F_x[kmer] + F_x[revcomp(kmer)] -- bit-identical to the reference's "+1 word, +1
 * revComplement(word)" (F:348-351); symmetric == 0: d_tables = F (window mode, F:1480).
 * d_tables has frisk_b200_table_size(1, kmax) entries.  d_valid_kmax (1 uint64, nullable)
 * receives the number of valid forward kmax-words; exMax (F:344) = sum_i max(0, len_i-kmax+1) - that.
 */
int frisk_b200_finalize_tables(const uint64_t *d_fwd, int kmax, int symmetric, uint64_t *d_tables,
                               uint64_t *d_valid_kmax, void *stream);

/*
 * frisk_b200_finalize_tables_peers: multi-GPU frisk_b200_finalize_tables with the all-reduce of the
 * counters FUSED in: d_fwd_peers is a HOST array of `world` device pointers, the counter buffer of
 * every rank as mapped into this process (NVLink peer mappings, e.g. the buffer_ptrs of a torch
 * symmetric-memory allocation); the kernels read and sum them directly, so no collective and no
 * staging copy sits between the background count and the finalised tables.
 * Synchronisation between the GPUs is folded into the first kernel: d_flag_peers (host array of
 * `world` device pointers, NULLable) names, per rank, an array of `world` uint64 flags in that rank's
 * peer-mapped memory, zero before the first call; `epoch` must be 1, 2, 3, ... on successive calls (the
 * same sequence on every rank).  Rank r posts `epoch` into flags[q][r] of every peer q and waits for
 * flags[r][*] >= epoch (a peer that never arrives traps the kernel after ~10 s instead of hanging).
 * With d_flag_peers == NULL the caller must have put its own cross-GPU barrier on `stream` after its
 * frisk_b200_background calls.  Either way a counter buffer must not be rewritten before the call after
 * next (alternate between two buffers).  kmax <= 8, world <= 16; FRISK_E_UNSUPPORTED otherwise (use an
 * all-reduce then).
 */
int frisk_b200_finalize_tables_peers(const uint64_t *const *d_fwd_peers, uint64_t *const *d_flag_peers, int rank,
                                     int world, uint64_t epoch, int kmax, int symmetric, uint64_t *d_tables,
                                     uint64_t *d_valid_kmax, void *stream);

/*
 * frisk_b200_finalize_ivom: frisk_b200_finalize_tables (symmetric) + frisk_b200_genome_ivom as ONE
 * cooperative launch (grid-wide barriers instead of five launch boundaries).  world == 0: the counters
 * are d_fwd; world > 0: they are summed from d_fwd_peers exactly as frisk_b200_finalize_tables_peers does
 * (flags / rank / epoch as there).  kmax 9..12: falls back to the separate general-path launches
 * (single GPU only).
 */
int frisk_b200_finalize_ivom(const uint64_t *d_fwd, const uint64_t *const *d_fwd_peers, uint64_t *const *d_flag_peers,
                             int rank, int world, uint64_t epoch, int kmin, int kmax, int64_t genome_space,
                             uint64_t *d_tables, uint64_t *d_valid_kmax, double *d_ig, void *stream);

/*
 * frisk_b200_genome_ivom: for every kmax-mer, the un-normalised genome IVOM value of
 * IvomBuild(isGenomeIVOM=True) (F:411-450) and its log2, as pairs of doubles (4^kmax pairs).
 * It depends only on the genome tables, so it is computed once instead of once per window.
 * genome_space = totalLen - nnTotal (F:379).  An entry whose reference evaluation would raise
 * ZeroDivisionError is NaN.
 */
int frisk_b200_genome_ivom(const uint64_t *d_tables, int kmin, int kmax, int64_t genome_space, double *d_ig,
                           void *stream);

/*
 * frisk_b200_score: the per-window loop of main() (F:1478-1494): window k-mer tables
 * (computeKmers, forward strand, upper-cased, F:1480), IvomBuild x2 + KLD (F:1481-1483), calcGC
 * (F:1484) and calcRIP (F:1486), fused in one kernel; window tables live only in shared memory.
 * d_rows: n_win x 5 doubles {windowKLD, GC, PI, SI, CRI} (PI/SI/CRI NaN unless want_rip and
 * kmin <= 2 <= kmax).  d_status: n_win FRISK_ROW_* words.  d_dump (nullable, tests only):
 * n_win x frisk_b200_table_size(1,kmax) uint16 window tables, orders 1..kmax.
 * max_win_len: the largest win_len (<= FRISK_B200_MAX_WINDOW).  kmax <= 8 and windows <= 65,535 bases
 * run in the shared-memory kernels, kmax 9..12 on windows <= 8,186 bases (without d_dump) in the extension kernel,
 * anything else in the general kernel (frisk_general.cu); same results.  frisk_b200_score_kernel_name names the kernel.
 */
int frisk_b200_score(const uint32_t *d_codes, const uint32_t *d_inv, const uint32_t *d_low,
                     const uint64_t *d_win_off, const uint32_t *d_win_len, uint64_t n_win, uint32_t max_win_len,
                     const double *d_ig, int kmin, int kmax, int want_rip, double *d_rows, uint32_t *d_status,
                     uint16_t *d_dump, void *stream);

/*
 * Strand-symmetric composition vectors of sequence regions, in batch: what the reference builds per
 * anomalous window for its PCA / t-SNE stage with computeKmers(pcaMode=True, sym=True) (F:1576-1578),
 * scrubMirrors (F:797-811) and flattenKmerMap(prop=True) (F:813-831).  For every order k = kmin..kmax
 * (<= 7; the reference's default is 1..6) and every k-mer that comes first of its {k-mer, reverse
 * complement} pair in table order: (count + count of the reverse complement) / (sum of that over the
 * kept k-mers of the order).  Regions are upper-cased like windows (soft-masked bases count).
 * frisk_b200_feature_slots (host): slot[sum 4^k entries, orders 1..kmax] = position of the k-mer in
 * the vector or -1; *n_features = vector length.  frisk_b200_region_features: d_out[n_regions][n_features];
 * an order without any valid word gives NaN (the reference raises ZeroDivisionError, F:824).
 */
int frisk_b200_feature_slots(int kmin, int kmax, int32_t *slot, uint64_t *n_features);
int frisk_b200_region_features(const uint32_t *d_codes, const uint32_t *d_inv, const uint64_t *d_reg_off,
                               const uint32_t *d_reg_len, uint64_t n_regions, int kmin, int kmax, const int32_t *d_slot,
                               uint64_t n_features, double *d_out, void *stream);

/* How frisk_b200_score would run the default (kmin = 1, no dump) configuration on the current device:
 * resident CTAs per SM and threads per CTA of the window kernel it selects, a forced one included (diagnostic;
 * bench.py reports it). */
int frisk_b200_score_occupancy(int kmax, uint32_t max_win_len, int *ctas_per_sm, int *threads_per_cta);

/* Tuning/test switches (0 = default behaviour).  "force_dense_kernel", "force_bucket_kernel", "force_direct_kernel",
 * "force_nibble_kernel" and "force_general_kernel" = 1 make frisk_b200_score run that window kernel wherever it can:
 * dense-table (the kernel for windows of 8,187..65,535 bases) for kmax <= 8; bucketed for kmax 4..8 and direct or nibble
 * for kmax 7 and 8, on windows <= 8,186 bases; general (global-memory, run-time K) for everything.  Elsewhere the default
 * choice stands (kmax 9..12 keep the extension kernel unless the general one is forced).  One kernel is forced at a time:
 * the last switch set to 1 wins, and setting a switch to 0 clears it only if it is the one in force.  Every entry point
 * that scores windows honours it, and all of them produce the same rows (tests/test_gpu_parity.py).
 * "ingest_exact_open" = 1 makes frisk_b200_fasta_open copy the text in one piece and count the records before it
 * allocates the record table (the fallback of the default chunked open); "ingest_chunk_tiles" = t lets texts of
 * 2t or more 4096-byte tiles be uploaded in chunks (default 512: 2 MiB per chunk, at most 8 chunks).  Same genome
 * either way (tests/test_ingest_gpu.py).  "gzip_chunk_bytes" = c places the gzip inflate's nominal chunk starts every c
 * compressed bytes (0: default); same text either way. */
int frisk_b200_set_option(const char *name, int value);

/*
 * frisk_b200_kld: KLD(GenomeIVOM, windowIVOM) (F:459-472) of two normalised IVOM vectors of n
 * doubles in the same k-mer order: sum w*log2(w/G), terms with G == 0 skipped; *d_out gets the
 * sum.  Serves the dict-level compatibility API; frisk_b200_score fuses the same computation.
 */
int frisk_b200_kld(const double *d_genome_ivom, const double *d_window_ivom, uint64_t n, double *d_out, void *stream);

/*
 * frisk_b200_run_host: the whole path from HOST buffers: H2D of the packed planes and window
 * list, background + finalize + genome IVOM + score, D2H of rows/status/tables.  Query planes are
 * scored against the host planes' background (pass the same planes for the default -Q == -H).
 * All host pointers should be pinned for the copies to be asynchronous.  Device workspace is
 * cached per device between calls.  tables_out: frisk_b200_table_size(1,kmax) uint64 (nullable);
 * valid_kmax_out: 1 uint64 (nullable).  Synchronises `stream` before returning.
 */
int frisk_b200_run_host(const uint32_t *h_codes, const uint32_t *h_inv, const uint32_t *h_low, uint64_t h_padded_len,
                        const uint32_t *q_codes, const uint32_t *q_inv, const uint32_t *q_low, uint64_t q_padded_len,
                        const uint64_t *win_off, const uint32_t *win_len, uint64_t n_win, uint32_t max_win_len,
                        int kmin, int kmax, int mask_host, int want_rip, int64_t genome_space, double *rows_out,
                        uint32_t *status_out, uint64_t *tables_out, uint64_t *valid_kmax_out, void *stream);

/*
 * Sparse form of a 1-bit plane: its non-zero 32-base words as (word index, word) pairs.  Assemblies
 * have few unresolved bases, so the invalid plane -- a third of the packed bytes -- is nearly all
 * zeros; frisk_b200_run_host_sparse uploads the pairs instead and expands them on the device, which
 * takes that third off the PCIe transfer.  frisk_b200_plane_sparse (host) extracts the pairs: arrays
 * may be NULL to only count; *n_nonzero always receives the count; FRISK_E_CAPACITY if cap is too small.
 * Planes of up to 2^32 words (137 Gbases).
 */
int frisk_b200_plane_sparse(const uint32_t *plane, uint64_t n_words, uint64_t cap, uint32_t *idx, uint32_t *val,
                            uint64_t *n_nonzero);
int frisk_b200_run_host_sparse(const uint32_t *h_codes, const uint32_t *h_inv_idx, const uint32_t *h_inv_val,
                               uint64_t h_inv_n, const uint32_t *h_low, uint64_t h_padded_len, const uint32_t *q_codes,
                               const uint32_t *q_inv_idx, const uint32_t *q_inv_val, uint64_t q_inv_n,
                               const uint32_t *q_low, uint64_t q_padded_len, const uint64_t *win_off,
                               const uint32_t *win_len, uint64_t n_win, uint32_t max_win_len, int kmin, int kmax,
                               int mask_host, int want_rip, int64_t genome_space, double *rows_out, uint32_t *status_out,
                               uint64_t *tables_out, uint64_t *valid_kmax_out, void *stream);

/*
 * frisk_b200_run_host_peers: one rank's share of a multi-GPU run in one call -- frisk_b200_run_host_sparse
 * for this rank's scaffolds (query == host shard) with the exchange of the counters fused in
 * (frisk_b200_finalize_tables_peers: d_fwd_local is this rank's counter buffer for this call, one of the
 * d_fwd_peers; flags / rank / world / epoch as there).  genome_space is the GLOBAL totalLen - nnTotal.
 * tables_out / valid_kmax_out are global.  Every rank must make the call; kmax <= 8.
 */
int frisk_b200_run_host_peers(const uint32_t *h_codes, const uint32_t *h_inv_idx, const uint32_t *h_inv_val,
                              uint64_t h_inv_n, const uint32_t *h_low, uint64_t h_padded_len, const uint64_t *win_off,
                              const uint32_t *win_len, uint64_t n_win, uint32_t max_win_len, int kmin, int kmax,
                              int mask_host, int want_rip, int64_t genome_space, uint64_t *d_fwd_local,
                              const uint64_t *const *d_fwd_peers, uint64_t *const *d_flag_peers, int rank, int world,
                              uint64_t epoch, double *rows_out, uint32_t *status_out, uint64_t *tables_out,
                              uint64_t *valid_kmax_out, void *stream);

/*
 * frisk_b200_run_resident: frisk_b200_run_host for planes that are already in device memory (e.g.
 * written by frisk_b200_fasta_pack): no plane upload; the window list still comes from, and the
 * results still go to, host memory.
 */
int frisk_b200_run_resident(const uint32_t *d_h_codes, const uint32_t *d_h_inv, const uint32_t *d_h_low,
                            uint64_t h_padded_len, const uint32_t *d_q_codes, const uint32_t *d_q_inv,
                            const uint32_t *d_q_low, uint64_t q_padded_len, const uint64_t *win_off,
                            const uint32_t *win_len, uint64_t n_win, uint32_t max_win_len, int kmin, int kmax,
                            int mask_host, int want_rip, int64_t genome_space, double *rows_out, uint32_t *status_out,
                            uint64_t *tables_out, uint64_t *valid_kmax_out, void *stream);

/* ------------------------------------------------------------------ device-side FASTA ingest
 *
 * The GPU replacement of iterFasta (F:139-164) + countN (F:106-118): the raw FASTA text is copied
 * to the device once and tokenised, measured and 2-bit packed there (frisk_ingest.cu); the planes
 * are bit-identical to those of frisk_b200_fasta_scan + frisk_b200_pack_layout + frisk_b200_pack.
 *
 * frisk_b200_fasta_open: H2D of text[0..n) (asynchronous when `text` is pinned), record detection
 * and per-record lengths on the device, names (F:156) and the packed layout on the host.  Texts of
 * 4 MiB and more go up in <= 8 chunks on a second stream, each chunk tokenised while the next is on
 * the bus; the record table is sized by a guess (n/64 + 4096 records) so that the call synchronises
 * once.  A text the chunked pass cannot decide (a blank run across a chunk boundary, more records than
 * the guess) is opened again in one piece with the records counted first -- same result, reported by
 * frisk_b200_fasta_open_stats (out[0] opens that completed chunked/speculative, out[1] opens that were
 * redone exactly; process-wide).  Blocks until the record table is known.  *n_records, *padded_len and stats[3] (totalLen, nnTotal,
 * number of lower-case acgt -- as frisk_b200_pack) describe the result; the caller then allocates
 * the planes (padded_len/16 and padded_len/32 uint32 words) and calls frisk_b200_fasta_pack, which
 * only enqueues work on `stream`.  frisk_b200_fasta_records copies the record table (any pointer
 * may be NULL); name_off/name_len index into `text`.  frisk_b200_fasta_close releases the device
 * copy of the text (stream-ordered) and the handle.  Use one stream for all calls on a handle.
 * FRISK_E_FORMAT: a header line without a name (the reference raises IndexError, F:156).
 */
typedef struct frisk_b200_fasta frisk_b200_fasta;
int frisk_b200_fasta_open(const char *text, uint64_t n, void *stream, frisk_b200_fasta **out, uint64_t *n_records,
                          uint64_t *padded_len, uint64_t stats[3]);
int frisk_b200_fasta_records(const frisk_b200_fasta *h, uint64_t *name_off, uint32_t *name_len, uint64_t *seq_len,
                             uint64_t *scaf_off);
int frisk_b200_fasta_pack(frisk_b200_fasta *h, uint32_t *d_codes, uint32_t *d_inv, uint32_t *d_low, void *stream);
int frisk_b200_fasta_close(frisk_b200_fasta *h, void *stream);
int frisk_b200_fasta_open_stats(uint64_t out[2]);

/* frisk_b200_run_fasta: FASTA text in, rows out, ONE call -- the reference's stages 2+3 (F:1442, F:1478-1494) including
 * its three passes over the file (F:170, F:203, F:297).  h_text is the genome the background is counted on (--hostSeq,
 * or the query itself), q_text the genome whose windows are scored (NULL, or the same pointer and size: the same genome).
 * The text goes up in chunks; each chunk is tokenised, laid out, packed and (kmax <= 8) counted on the device while the next
 * chunk is on the bus.  With kmax 7 or 8 and windows of <= 8,186 bases nothing behind the last chunk waits for the host:
 * genome space, window list (frisk_b200_windows' windows for w, step, scaffolds_all) and window count are produced on the
 * device, and tables -> IVOM -> window kernel are queued before the host has seen the record table, which it reads (names,
 * FRISK_E_FORMAT) while the window kernel runs.  Otherwise the record table comes back once, as soon as the last chunk is
 * packed, and windows and launches happen on the host while that chunk is still being counted.  rows_out / status_out have room for rows_cap windows (pinned buffers are
 * written by the kernel directly); *n_win_out always receives the number of windows.
 * *host_out / *query_out (query_out: NULL when the genomes are the same) are handles as of frisk_b200_fasta_open whose PLANES
 * exist and belong to the handle (frisk_b200_fasta_planes; padded_len etc. from frisk_b200_fasta_info, the record table
 * from frisk_b200_fasta_records) until frisk_b200_fasta_close.
 * FRISK_E_CAPACITY: more windows than rows_cap -- nothing was scored, but the handles are valid: allocate *n_win_out rows and
 * call frisk_b200_run_resident on their planes.  Any other error: no handle is returned.  Blocks until the rows are on the
 * host.  Stage times: frisk_b200_last_run_timing (ms[0] = text uploaded, ms[1] = tokenised + packed + counted). */
int frisk_b200_run_fasta(const char *h_text, uint64_t h_n, const char *q_text, uint64_t q_n, int w, int step,
                         int scaffolds_all, int kmin, int kmax, int mask_host, int want_rip, uint64_t rows_cap,
                         double *rows_out, uint32_t *status_out, uint64_t *tables_out, uint64_t *valid_kmax_out,
                         uint64_t *n_win_out, frisk_b200_fasta **host_out, frisk_b200_fasta **query_out, void *stream);
/* frisk_b200_windows_device: the window list of frisk_b200_windows (same windows, same order) from a record table that
 * lives in DEVICE memory, written to device memory; *d_n_windows receives the count (windows beyond `cap` are not
 * written), *d_genome_space (nullable) the sum of the lengths.  What frisk_b200_run_fasta does between the ingest and the
 * window kernel, exposed for tests. */
int frisk_b200_windows_device(const uint64_t *d_scaf_len, const uint64_t *d_scaf_off, uint64_t n_scaf, int w, int step,
                              int scaffolds_all, uint64_t cap, uint64_t *d_win_off, uint32_t *d_win_len,
                              uint64_t *d_n_windows, int64_t *d_genome_space, void *stream);
int frisk_b200_fasta_info(const frisk_b200_fasta *h, uint64_t *n_records, uint64_t *padded_len, uint64_t stats[3]);
int frisk_b200_fasta_planes(const frisk_b200_fasta *h, const uint32_t **d_codes, const uint32_t **d_inv,
                            const uint32_t **d_low);

/* ------------------------------------------------------------------ BGZF-compressed FASTA (frisk_bgzf.cu)
 *
 * BGZF (bgzip, `samtools faidx`) is a series of gzip members of <= 64 KiB each; every member's header gives its
 * compressed size and its trailer the CRC32 and inflated size, so every member is inflated on the device by a decoder of
 * its own, straight into the ingest's text buffer.  A single-member .gz (gzip, pigz) is not BGZF: it is FRISK_E_FORMAT
 * here and goes to the gzip entry points below.
 *
 * frisk_b200_bgzf_blocks: the block table of a BGZF buffer, from the headers and trailers alone.  comp_off / comp_len: the
 * raw deflate payload of every member; crc: the CRC32 of its trailer; text_off: the exclusive prefix sum of the inflated
 * sizes; *text_len their sum.  Every member must be a BGZF block (1f 8b, CM 8, FLG 4, a "BC" subfield of SLEN 2 among the
 * extra subfields, BSIZE inside the buffer, ISIZE <= 65,536); empty members (the EOF marker) may appear anywhere.
 * Anything else, trailing bytes included: FRISK_E_FORMAT.  Arrays may be NULL to count only (as frisk_b200_fasta_scan);
 * *n_blocks always receives the count; FRISK_E_CAPACITY if cap is too small.
 *
 * frisk_b200_bgzf_inflate: inflates every member of the table into d_text[text_off[b] ..] (exactly text_len bytes are
 * written; nothing beyond), one warp per member, and checks each member's size and CRC32 (the CRCs come from the block
 * table).  Full RFC 1951 (stored, fixed and dynamic Huffman blocks).  Malformed input never faults: d_block_status[b] != 0
 * marks a member that is not valid deflate, does not fit its ISIZE or fails its CRC; the caller reads the status words
 * behind the stream's work and treats any non-zero one as FRISK_E_FORMAT.  Only enqueues work on `stream`.
 * frisk_b200_bgzf_inflate_host: the same decoder run on the CPU over host arrays (test infrastructure: no user path calls it);
 * returns FRISK_E_FORMAT itself when a status word is non-zero.  `stream` is unused.
 *
 * frisk_b200_fasta_open_bgzf / frisk_b200_run_fasta_bgzf: frisk_b200_fasta_open / frisk_b200_run_fasta with BGZF buffers in
 * place of the texts, same arguments and results: the compressed bytes go up, are inflated into the ingest's text buffer
 * and are tokenised and packed there.  The inflated text never reaches the host, so the names of a BGZF handle index into
 * a buffer the handle owns: frisk_b200_fasta_name_text gives it (NULL / 0 for a handle opened from text, whose names index
 * the caller's text).  ms[0] of frisk_b200_last_run_timing is "compressed bytes uploaded and inflated". */
int frisk_b200_bgzf_blocks(const uint8_t *gz, uint64_t n, uint64_t cap, uint64_t *comp_off, uint32_t *comp_len,
                           uint32_t *crc, uint64_t *text_off, uint64_t *n_blocks, uint64_t *text_len);
int frisk_b200_bgzf_inflate(const uint8_t *d_gz, const uint64_t *d_comp_off, const uint32_t *d_comp_len,
                            const uint32_t *d_crc, const uint64_t *d_text_off, uint64_t n_blocks, uint64_t text_len,
                            uint8_t *d_text, uint32_t *d_block_status, void *stream);
int frisk_b200_bgzf_inflate_host(const uint8_t *gz, const uint64_t *comp_off, const uint32_t *comp_len, const uint32_t *crc,
                                 const uint64_t *text_off, uint64_t n_blocks, uint64_t text_len, uint8_t *text,
                                 uint32_t *block_status, void *stream);
int frisk_b200_fasta_open_bgzf(const char *gz, uint64_t n, void *stream, frisk_b200_fasta **out, uint64_t *n_records,
                               uint64_t *padded_len, uint64_t stats[3]);
int frisk_b200_run_fasta_bgzf(const char *h_gz, uint64_t h_n, const char *q_gz, uint64_t q_n, int w, int step,
                              int scaffolds_all, int kmin, int kmax, int mask_host, int want_rip, uint64_t rows_cap,
                              double *rows_out, uint32_t *status_out, uint64_t *tables_out, uint64_t *valid_kmax_out,
                              uint64_t *n_win_out, frisk_b200_fasta **host_out, frisk_b200_fasta **query_out, void *stream);
int frisk_b200_fasta_name_text(const frisk_b200_fasta *h, const char **text, uint64_t *n);

/* ------------------------------------------------------------------ gzip-compressed FASTA (frisk_gzip.cu)
 *
 * One plain gzip member (gzip, pigz, NCBI / Ensembl / UCSC .fa.gz) is one deflate stream, inflated on the device in two
 * passes: decoders start at block boundaries found by a search for valid dynamic block headers, every C compressed bytes,
 * and write matches that reach before their chunk as placeholders; the host accepts a chunk only where its predecessor
 * ended exactly at its start and decodes the others again from there; the placeholders are then resolved in chunk order.
 * A file without dynamic blocks (level 0, Z_FIXED) is one chunk.  "gzip_chunk_bytes" (frisk_b200_set_option) sets C
 * (0: the default, 16 KiB).  Device memory: besides the member and the text, the first pass takes about 16 bytes of
 * scratch per compressed byte (16-bit symbols, 8 per compressed byte), about 14 GB for a 900 MB .gz.
 *
 * frisk_b200_gzip_member: the header of the member at gz (1f 8b, CM 8; FTEXT, FHCRC (checked), FEXTRA, FNAME, FCOMMENT;
 * reserved flag bits are FRISK_E_FORMAT): the deflate payload's offset and length up to the last 8 bytes, and the CRC32 and
 * ISIZE of those last 8 bytes (the trailer of a single-member file).  Any pointer but gz may be NULL.
 *
 * frisk_b200_gzip_inflate: inflates the member in d_gz[0, n) (device memory) into d_text.  Synchronises `stream`.
 * *text_len receives the text's length (exact: no ISIZE guess; ISIZE must equal it mod 2^32); FRISK_E_CAPACITY, with
 * *text_len set, when text_cap is smaller.  stats (nullable): {chunks, joins accepted on the first pass, chunks decoded
 * again from their predecessor's end, chain chunks decoded again because their scratch was too small}.  Not valid
 * deflate, a CRC32 or ISIZE mismatch, truncation or trailing bytes: FRISK_E_FORMAT.  Another gzip member after the
 * trailer (a multi-member file): FRISK_E_UNSUPPORTED (the Python layer then inflates on the host); so are chunks of 4 GiB
 * of text or more.  Malformed input never faults and leaves no CUDA error behind.
 * frisk_b200_gzip_inflate_host: the same plan, joins and repairs run on the CPU over host memory (test infrastructure: no
 * user path calls it); same text, same stats, same return codes.  `stream` is unused.
 *
 * frisk_b200_fasta_open_gzip / frisk_b200_run_fasta_gzip: frisk_b200_fasta_open / frisk_b200_run_fasta with one gzip member
 * in place of the texts, same arguments and results, as the _bgzf pair: the member goes up and is inflated into the
 * ingest's text buffer; the names come from frisk_b200_fasta_name_text; ms[0] of frisk_b200_last_run_timing is
 * "compressed bytes uploaded and inflated". */
int frisk_b200_gzip_member(const uint8_t *gz, uint64_t n, uint64_t *payload_off, uint64_t *payload_len, uint32_t *crc,
                           uint32_t *isize);
int frisk_b200_gzip_inflate(const uint8_t *d_gz, uint64_t n, uint8_t *d_text, uint64_t text_cap, uint64_t *text_len,
                            uint64_t stats[4], void *stream);
int frisk_b200_gzip_inflate_host(const uint8_t *gz, uint64_t n, uint8_t *text, uint64_t text_cap, uint64_t *text_len,
                                 uint64_t stats[4], void *stream);
int frisk_b200_fasta_open_gzip(const char *gz, uint64_t n, void *stream, frisk_b200_fasta **out, uint64_t *n_records,
                               uint64_t *padded_len, uint64_t stats[3]);
int frisk_b200_run_fasta_gzip(const char *h_gz, uint64_t h_n, const char *q_gz, uint64_t q_n, int w, int step,
                              int scaffolds_all, int kmin, int kmax, int mask_host, int want_rip, uint64_t rows_cap,
                              double *rows_out, uint32_t *status_out, uint64_t *tables_out, uint64_t *valid_kmax_out,
                              uint64_t *n_win_out, frisk_b200_fasta **host_out, frisk_b200_fasta **query_out, void *stream);

/* ------------------------------------------------------------------ UCSC .2bit genomes (frisk_twobit.cu)
 *
 * A twoBit file (UCSC hg38.2bit, faToTwoBit; versions 0 and 1, either byte order: a signature that reads 0x4327411A means
 * every integer of the file is byte-swapped) holds 2-bit bases, N blocks and soft-mask blocks: exactly what the planes hold.
 * Every non-ACGT character of a FASTA is an N there and every lower-case character lies in a mask block, so a .2bit file and
 * its FASTA give the same records, planes, tables and rows, bit for bit.  Nothing is tokenised: the bases are remapped and
 * realigned to the 128-base layout, the blocks expanded into the invalid and lower-case planes (N blocks: invalid, code 0;
 * mask blocks minus N blocks: lower case).  The name of a record is its index name, verbatim.
 *
 * frisk_b200_2bit_records: parses and checks the whole file on the host: header, index and record headers, every block
 * inside its sequence (zero-size blocks are ignored; blocks may overlap and come in any order), the packed bases inside the
 * buffer.  A bad signature, a version other than 0 or 1, an empty name, an offset, count or length that reaches beyond the
 * buffer, or a block beyond its sequence: FRISK_E_FORMAT, before any byte beyond the buffer is read.  name_off / name_len:
 * the index names in buf; seq_len: dnaSize; *bases (nullable): their sum.  Arrays may be NULL to count only; *n_records
 * always receives the count; FRISK_E_CAPACITY if cap is too small.
 *
 * frisk_b200_2bit_unpack_host: the planes of the file on the CPU, with the device path's plan and per-word code (test
 * infrastructure, and the producer of host planes).  padded_len must be frisk_b200_pack_layout's for the record lengths
 * (FRISK_E_INVALID otherwise); codes / inv / low as frisk_b200_pack (low may be NULL when the file has no mask bases,
 * FRISK_E_FORMAT if it has some); stats[3] as frisk_b200_pack (totalLen, nnTotal, lower-case acgt).
 *
 * frisk_b200_fasta_open_2bit / frisk_b200_run_2bit: frisk_b200_fasta_open / frisk_b200_run_fasta with .2bit files in place of
 * the texts, same arguments and results.  The file goes up in one copy and is decoded into planes the handle owns; the names
 * come from frisk_b200_fasta_name_text; with kmax 7 or 8 and windows of <= 8,186 bases the one-call path takes the
 * device-only tail as text does.  ms[0] of frisk_b200_last_run_timing is "file uploaded and decoded". */
int frisk_b200_2bit_records(const uint8_t *buf, uint64_t n, uint64_t cap, uint64_t *name_off, uint32_t *name_len,
                            uint64_t *seq_len, uint64_t *n_records, uint64_t *bases);
int frisk_b200_2bit_unpack_host(const uint8_t *buf, uint64_t n, uint64_t padded_len, uint32_t *codes, uint32_t *inv,
                                uint32_t *low, uint64_t stats[3]);
int frisk_b200_fasta_open_2bit(const char *buf, uint64_t n, void *stream, frisk_b200_fasta **out, uint64_t *n_records,
                               uint64_t *padded_len, uint64_t stats[3]);
int frisk_b200_run_2bit(const char *h_2bit, uint64_t h_n, const char *q_2bit, uint64_t q_n, int w, int step,
                        int scaffolds_all, int kmin, int kmax, int mask_host, int want_rip, uint64_t rows_cap,
                        double *rows_out, uint32_t *status_out, uint64_t *tables_out, uint64_t *valid_kmax_out,
                        uint64_t *n_win_out, frisk_b200_fasta **host_out, frisk_b200_fasta **query_out, void *stream);

/* Stage times (ms since the start of the call) of the last frisk_b200_run_host / _sparse / _peers / _run_resident call
 * on the current device, from CUDA events recorded on the call's own streams: ms[0] planes uploaded, ms[1] background
 * counted, ms[2] tables + genome IVOM finalised (multi-GPU: includes the wait for the peers' counters), ms[3] window
 * kernel(s) done, ms[4] results on the host, ms[5] the moment the window kernel could start (its inputs done, its launch on the device).  -1 for a mark the call did not set.  *n = values written. */
int frisk_b200_last_run_timing(float *ms, int cap, int *n);

/* The k sweep of BASELINE config C3 in ONE launch: rows for kmax' = 1..8 (kmin 1: eight reference runs `-m 1 -k k'`,
 * F:1197-1206 / F:1478-1494) of every window from one pass over it.  d_ig / d_rows / d_status are HOST arrays of 8
 * device pointers: the genome IVOM table (frisk_b200_genome_ivom with kmin 1, kmax k'), the rows [n_win][5] and the
 * status words of kmax' = index + 1.  kmax must be 8 and windows at most 8,186 bases (FRISK_E_UNSUPPORTED otherwise:
 * call frisk_b200_score per kmax').  PI / SI / CRI are NaN for kmax' = 1, as in the reference (F:1467). */
int frisk_b200_score_sweep(const uint32_t *d_codes, const uint32_t *d_inv, const uint32_t *d_low, const uint64_t *d_win_off,
                           const uint32_t *d_win_len, uint64_t n_win, uint32_t max_win_len, const double *const *d_ig,
                           int kmax, int want_rip, double *const *d_rows, uint32_t *const *d_status, void *stream);

/* The window kernel frisk_b200_score launches for (kmin, kmax, longest window), spelled as profilers print it
 * (e.g. "score_windows_nibble_kernel<8, 20, 0, 1>"): labels of profiles and bench lines come from the launcher's own
 * selection, honouring frisk_b200_set_option. */
int frisk_b200_score_kernel_name(int kmin, int kmax, uint32_t max_win_len, char *buf, uint64_t cap);

/* Free the cached device workspace of frisk_b200_run_host on the current device. */
int frisk_b200_release_workspace(void);

/* Plain device memory (cudaMalloc / cudaFree) and device selection, so that a caller without a GPU array
 * library of its own -- the CLI: importing PyTorch costs more than the whole run -- can own its planes. */
int frisk_b200_device_alloc(void **ptr, uint64_t bytes);
int frisk_b200_device_free(void *ptr);
int frisk_b200_set_device(int index);

/* Pinned host memory helpers (cudaHostAlloc / cudaFreeHost) so Python can build pinned planes. */
int frisk_b200_host_alloc(void **ptr, uint64_t bytes);
int frisk_b200_host_free(void *ptr);

/* Shared-memory atomic micro-benchmark used for the smem-atomic roofline (BASELINE.md section 4):
 * every thread of `blocks` x 1024 threads issues `iters` u32 atomicAdd's on a 64 KiB shared table
 * with (mode 0) conflict-free, (mode 1) uniformly random, (mode 2) single-address indices.
 * *ms receives the kernel time; updates = blocks*1024*iters. */
int frisk_b200_bench_smem_atomics(int blocks, int iters, int mode, float *ms, void *stream);

/* Two more roofline denominators of the window kernels, measured on the GPU at hand (frisk_bench.cu):
 * _l2_gather: `blocks` x 256 threads each issue `iters` (multiple of 4) 16-byte loads from an L2-resident table of
 *   `table_bytes` (power of two; 1 MiB = the genome-IVOM table of kmax 8).  mode 0: every lane an independent random
 *   entry; mode 1: a warp's lanes read increasing entries with random gaps (the sorted epilogue's pattern); mode 2: mode 0
 *   as 16-byte cp.async into shared memory; mode 3: mode 0 with 8-byte entries; mode 4: mode 0 as 16-byte cp.async.bulk
 *   copies (the TMA engine) completing on an mbarrier; mode 5: as TMA tile::gather4 loads (4 rows per instruction; the
 *   gathered data is verified: FRISK_E_UNSUPPORTED = never completed, FRISK_E_FORMAT = wrong data); mode 7: mode 0 with
 *   32-byte entries, each read by one 256-bit load.  gathers = blocks*256*iters.
 * _smem_loads: `blocks` x 256 threads each issue `iters` random loads of `elem_bytes` (4, 8 or 16) from a 32 KiB
 *   shared-memory table (bank-conflicted reads).  loads = blocks*256*iters. */
int frisk_b200_bench_l2_gather(int blocks, int iters, uint64_t table_bytes, int mode, float *ms, void *stream);
int frisk_b200_bench_smem_loads(int blocks, int iters, int elem_bytes, float *ms, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* FRISK_B200_H */
