// frisk_b200 one-call run paths: host planes, resident planes, FASTA text or a .2bit file in, rows out, in one C call
// (frisk_b200_run_host / _sparse / _peers, frisk_b200_run_resident, frisk_b200_run_fasta / _bgzf / _gzip, frisk_b200_run_2bit).  Every path enters and
// leaves through RunCall (device lock, stage marks, error drain), finalises through queue_tables and ends in results.  The
// per-device state they share lives here too: the workspace, the copy stream, the stage marks and the window staging.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <chrono>
#include <functional>
#include <mutex>
#include <vector>

#include "../../include/frisk_b200.h"
#include "frisk_internal.h"

namespace {
using frisk_internal::WinKernel;
using frisk_internal::WinPlan;
#define CK(call) FRISK_CK(call)

// Workspace slots: device buffers cached per device between calls, grown on demand.  Each slot is its own allocation and
// holds the same thing on every path, with one exception: kWsWinOff holds the window offsets of the host tails (their
// lengths right behind them when the two arrive as one host block, otherwise in kWsWinLen), but rows_cap offsets followed
// by rows_cap lengths in the FASTA device tail.
enum WsSlot {
    kWsHostCodes = 0, kWsHostInv, kWsHostLow,        // planes of the host genome (frisk_b200_run_host*)
    kWsQueryCodes, kWsQueryInv, kWsQueryLow,         // planes of a separate query genome
    kWsFwd,                                          // forward counters (+ 1 word)
    kWsTables, kWsIvom,                              // finalised tables + valid count; genome IVOM table
    kWsWinOff, kWsWinLen,                            // window list
    kWsRows, kWsStatus,                              // rows and status when the caller's buffers are not pinned
    kWsHostInvIdx = 15, kWsHostInvVal,               // sparse invalid plane of the host genome: word indices, words
    kWsQueryInvIdx, kWsQueryInvVal,                  // ... of the query genome
    kWsFirst,                                        // FASTA device tail: first window of each record
    kWsScalars,                                      // FASTA device tail: [window count, genome space]
    kWsSlots
};
struct Workspace {
    void* buf[kWsSlots] = {};
    size_t cap[kWsSlots] = {};
};
Workspace g_ws[64];
std::mutex g_run_mu[64];     // the run paths share the workspace, copy stream and marks: one call at a time per device

int ws_get(WsSlot slot, size_t bytes, void** out) {
    int dev = 0;
    CK(cudaGetDevice(&dev));
    Workspace& w = g_ws[dev & 63];
    if (w.cap[slot] < bytes) {
        if (w.buf[slot]) CK(cudaFree(w.buf[slot]));
        w.buf[slot] = nullptr; w.cap[slot] = 0;
        size_t want = bytes + bytes / 8 + 256;
        CK(cudaMalloc(&w.buf[slot], want));
        w.cap[slot] = want;
    }
    *out = w.buf[slot];
    return FRISK_OK;
}

// per-device copy stream and its events (uploads overlap the background count, the tables go back beside the window kernel)
constexpr int kMaxChunks = 16;
struct CopyCtx {
    cudaStream_t copy = nullptr;
    cudaEvent_t chunk[kMaxChunks] = {};   // a chunk of the host planes has landed
    cudaEvent_t join = nullptr;           // the copy stream starts behind the work queued on the caller's stream so far
    cudaEvent_t windows = nullptr;        // the window list has landed
    cudaEvent_t tables = nullptr;         // the tables are final
};
CopyCtx g_copy[64];

int copy_ctx(CopyCtx** out) {
    int dev = 0;
    CK(cudaGetDevice(&dev));
    CopyCtx& c = g_copy[dev & 63];
    if (!c.copy) {
        CK(cudaStreamCreateWithFlags(&c.copy, cudaStreamNonBlocking));
        for (auto& e : c.chunk) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        for (cudaEvent_t* e : {&c.join, &c.windows, &c.tables}) CK(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
    }
    *out = &c;
    return FRISK_OK;
}

// Stage marks of the last run call on a device (frisk_b200_last_run_timing): timing-enabled events recorded on the call's
// streams; reading them back costs nothing on the data path.
enum { kTmStart = 0, kTmUploaded, kTmCounted, kTmFinalised, kTmScored, kTmEnd, kTmScoreStart, kTmCount };
struct RunMarks {
    cudaEvent_t ev[kTmCount] = {};
    bool have[kTmCount] = {};
    bool ready = false;
};
RunMarks g_marks[64];
int run_marks(RunMarks** out) {
    int dev = 0;
    CK(cudaGetDevice(&dev));
    RunMarks& m = g_marks[dev & 63];
    if (!m.ready) {
        for (auto& e : m.ev) CK(cudaEventCreate(&e));
        m.ready = true;
    }
    for (auto& h : m.have) h = false;
    *out = &m;
    return FRISK_OK;
}
int mark(RunMarks* m, int which, cudaStream_t st) {
    CK(cudaEventRecord(m->ev[which], st));
    m->have[which] = true;
    return FRISK_OK;
}

// FRISK_RUN_TRACE=1: host-side timeline of a one-call run on stderr (microseconds since the first stamp)
struct HostTrace {
    bool on = getenv("FRISK_RUN_TRACE") != nullptr;
    std::chrono::steady_clock::time_point t0;
    char buf[512]; int len = 0; bool started = false;
    void stamp(const char* what) {
        if (!on) return;
        const auto now = std::chrono::steady_clock::now();
        if (!started) { t0 = now; started = true; }
        len += snprintf(buf + len, sizeof(buf) - (size_t)len, " %s=%.1f", what, std::chrono::duration<double, std::micro>(now - t0).count());
    }
    void flush() { if (on && len) fprintf(stderr, "host trace (us):%s\n", buf); len = 0; started = false; }
};
thread_local HostTrace g_trace;

// One run call on the current device.  enter(): the device's run lock, the copy stream (with_copy), the stage marks, and
// kTmStart on the caller's stream.  leave(rc): once entered, a failure may leave copies and kernels queued that still
// target the caller's buffers -- drain both streams before control, and with it the right to free those buffers, goes
// back, and clear the error.
struct RunCall {
    std::unique_lock<std::mutex> lock;
    int dev = 0;
    cudaStream_t st = nullptr;
    CopyCtx* cc = nullptr;       // nullptr: everything runs on `st` (frisk_b200_run_resident)
    RunMarks* tm = nullptr;

    int enter(void* stream, bool with_copy) {
        if (frisk_b200_device_count() <= 0) return FRISK_E_NO_DEVICE;
        CK(cudaGetDevice(&dev));
        lock = std::unique_lock<std::mutex>(g_run_mu[dev & 63]);
        st = (cudaStream_t)stream;
        int rc;
        if (with_copy && (rc = copy_ctx(&cc))) return rc;
        if ((rc = run_marks(&tm))) return rc;
        return mark(tm, kTmStart, st);
    }
    int leave(int rc) {
        if (rc != FRISK_OK && lock.owns_lock()) {
            cudaStreamSynchronize(st);
            if (cc) cudaStreamSynchronize(cc->copy);
            cudaGetLastError();
        }
        return rc;
    }
};

// What a run computes and where it goes: the caller's result buffers (tables and valid nullable)
struct Job {
    int kmin, kmax, mask_host, want_rip;
    double* rows;
    uint32_t* status;
    uint64_t* tables;
    uint64_t* valid;
};
struct WindowList {
    const uint64_t* off;
    const uint32_t* len;
    uint64_t n;
    uint32_t max_len;
};
struct Planes {                  // one genome's planes in device memory
    const uint32_t *codes, *inv, *low;
    uint64_t padded_len;
};
// multi-GPU: where the other ranks' counters are (frisk_b200_finalize_ivom); world == 0: single GPU
struct PeerArgs {
    uint64_t* d_fwd_local = nullptr;
    const uint64_t* const* d_fwd_peers = nullptr;
    uint64_t* const* d_flag_peers = nullptr;
    int rank = 0, world = 0;
    uint64_t epoch = 0;
};

size_t table_words(int kmax) { return (size_t)frisk_b200_table_size(1, kmax); }
size_t ivom_bytes(int kmax) { return (size_t)16 << (2 * kmax); }

// The checks of a run from planes, before anything touches a device: the planes are there and padded to whole 128-base
// tiles, kmin / kmax, and every window lies inside the query planes -- the window list is host memory here, and a window
// outside the planes would be an illegal-address fault (and a sticky context error) in the window kernel: O(n), ~1 ns
// per window.
int check_plane_run(bool planes, uint64_t h_padded_len, uint64_t q_padded_len, const WindowList& wins, const Job& j) {
    if (!planes || (h_padded_len & 127) || (q_padded_len & 127) || h_padded_len < 128 || q_padded_len < 128) return FRISK_E_INVALID;
    if (wins.n && (!wins.off || !wins.len || !j.rows || !j.status)) return FRISK_E_INVALID;
    int rc = frisk_internal::check_k(j.kmin, j.kmax);
    if (rc) return rc;
    for (uint64_t i = 0; i < wins.n; ++i) {
        const uint64_t l = wins.len[i];
        if (l == 0 || l > wins.max_len || wins.off[i] > q_padded_len || l > q_padded_len - wins.off[i]) return FRISK_E_INVALID;
    }
    return FRISK_OK;
}

// Where the window kernel writes n rows and their status: straight into the caller's buffers when both are page-locked
// host memory with a device view (40 + 4 bytes per window, posted PCIe writes while it runs, no download behind it; a
// pageable pointer makes the query itself report an error, which is cleared), else into workspace rows that results downloads.
struct Rows {
    double* rows;
    uint32_t* status;
    bool direct;
};
int rows_for(uint64_t n, const Job& j, Rows* r) {
    cudaPointerAttributes pa_rows{}, pa_stat{};
    r->direct = cudaPointerGetAttributes(&pa_rows, j.rows) == cudaSuccess && pa_rows.type == cudaMemoryTypeHost &&
                cudaPointerGetAttributes(&pa_stat, j.status) == cudaSuccess && pa_stat.type == cudaMemoryTypeHost &&
                pa_rows.devicePointer && pa_stat.devicePointer;
    cudaGetLastError();
    if (r->direct) {
        r->rows = (double*)pa_rows.devicePointer;
        r->status = (uint32_t*)pa_stat.devicePointer;
        return FRISK_OK;
    }
    int rc;
    if ((rc = ws_get(kWsRows, n * 40, (void**)&r->rows))) return rc;
    return ws_get(kWsStatus, n * 4, (void**)&r->status);
}

// The tables step: the counters in dfwd (this GPU's, or summed over the peers') become the tables (kWsTables) and the
// genome IVOM table (kWsIvom) on stream s; kTmFinalised.  With a copy stream the tables and the valid count go back on it
// right away, beside the window kernel instead of behind it; without one the results step brings them.  space_dev
// (nullable): the genome space in device memory, in place of `space`.
int queue_tables(RunCall& c, const PeerArgs& peers, const void* dfwd, const Job& j, int64_t space, const long long* space_dev,
                 void* dtab, void* dig, cudaStream_t s) {
    const size_t tsz = table_words(j.kmax);
    uint64_t* dvalid = (uint64_t*)dtab + tsz;
    int rc = frisk_internal::finalize_ivom((const uint64_t*)dfwd, peers.d_fwd_peers, peers.d_flag_peers, peers.rank, peers.world,
                                           peers.epoch, j.kmin, j.kmax, space, space_dev, (uint64_t*)dtab, dvalid, (double*)dig, s);
    if (rc) return rc;
    if ((rc = mark(c.tm, kTmFinalised, s))) return rc;
    if (c.cc) {
        CK(cudaEventRecord(c.cc->tables, s));
        CK(cudaStreamWaitEvent(c.cc->copy, c.cc->tables, 0));
        if (j.tables) CK(cudaMemcpyAsync(j.tables, dtab, tsz * 8, cudaMemcpyDeviceToHost, c.cc->copy));
        if (j.valid) CK(cudaMemcpyAsync(j.valid, dvalid, 8, cudaMemcpyDeviceToHost, c.cc->copy));
    }
    return FRISK_OK;
}

// The results step, on the caller's stream: n rows and their status unless the window kernel wrote them through pinned
// views, the tables unless they went back on the copy stream, then `extra` bytes from d_extra (if any); kTmEnd; wait for
// the caller's stream, then the copy stream.
int results(RunCall& c, uint64_t n, const Rows& r, const Job& j, const void* dtab, const void* d_extra = nullptr,
            void* h_extra = nullptr, size_t extra = 0) {
    if (n && !r.direct) {
        CK(cudaMemcpyAsync(j.rows, r.rows, n * 40, cudaMemcpyDeviceToHost, c.st));
        CK(cudaMemcpyAsync(j.status, r.status, n * 4, cudaMemcpyDeviceToHost, c.st));
    }
    const size_t tsz = table_words(j.kmax);
    if (!c.cc && j.tables) CK(cudaMemcpyAsync(j.tables, dtab, tsz * 8, cudaMemcpyDeviceToHost, c.st));
    if (!c.cc && j.valid) CK(cudaMemcpyAsync(j.valid, (const uint64_t*)dtab + tsz, 8, cudaMemcpyDeviceToHost, c.st));
    if (extra) CK(cudaMemcpyAsync(h_extra, d_extra, extra, cudaMemcpyDeviceToHost, c.st));
    int rc;
    if ((rc = mark(c.tm, kTmEnd, c.st))) return rc;
    CK(cudaStreamSynchronize(c.st));
    if (c.cc) CK(cudaStreamSynchronize(c.cc->copy));
    g_trace.stamp("done");
    g_trace.flush();
    return FRISK_OK;
}

// the window list of frisk_b200_run_fasta's host tail, produced by the caller after the tables' finalisation is queued (the
// host derives the windows while the device is still counting)
typedef std::function<int(WindowList* wins)> LateWindows;

// Everything after the planes are on the device (or on their way, on the copy stream): [background count unless
// `counted`], tables, window list, window kernel, results.
int run_tail(RunCall& c, const PeerArgs& peers, const Planes& h, bool counted, const Planes& q, WindowList wins, const Job& j,
             int64_t space, void* dfwd, const LateWindows* late = nullptr) {
    const size_t tsz = table_words(j.kmax);
    void *dtab = nullptr, *dig = nullptr, *dwo = nullptr, *dwl = nullptr;
    Rows r{};
    int rc;
    if ((rc = ws_get(kWsTables, (tsz + 1) * 8, &dtab))) return rc;
    if ((rc = ws_get(kWsIvom, ivom_bytes(j.kmax), &dig))) return rc;
    auto upload_windows = [&]() -> int {
        if (wins.n) {
            int rc2;
            // (offsets and lengths in one host block -- frisk_b200_run_fasta's staging -- travel as one copy)
            const bool one_block = (const void*)wins.len == (const void*)(wins.off + wins.n);
            if ((rc2 = ws_get(kWsWinOff, one_block ? wins.n * 12 : wins.n * 8, &dwo))) return rc2;
            if (one_block) dwl = (char*)dwo + wins.n * 8;
            else if ((rc2 = ws_get(kWsWinLen, wins.n * 4, &dwl))) return rc2;
            if ((rc2 = rows_for(wins.n, j, &r))) return rc2;
            // the window list rides behind the planes -- but a late one goes on the compute stream: the copy stream is busy
            // bringing the tables back by then, and the window kernel would wait 0.03 ms for its 190 KB behind them
            cudaStream_t up = (c.cc && !late) ? c.cc->copy : c.st;
            if (one_block) CK(cudaMemcpyAsync(dwo, wins.off, wins.n * 12, cudaMemcpyHostToDevice, up));
            else {
                CK(cudaMemcpyAsync(dwo, wins.off, wins.n * 8, cudaMemcpyHostToDevice, up));
                CK(cudaMemcpyAsync(dwl, wins.len, wins.n * 4, cudaMemcpyHostToDevice, up));
            }
        }
        if (c.cc) CK(cudaEventRecord(c.cc->windows, c.cc->copy));
        return FRISK_OK;
    };
    if (!late && (rc = upload_windows())) return rc;
    if (!counted) {
        CK(cudaMemsetAsync(dfwd, 0, (tsz + 1) * 8, c.st));
        // the last 32-base word is padding by construction and is only ever read as look-ahead
        rc = frisk_b200_background(h.codes, h.inv, h.low, 0, h.padded_len - 32, j.kmax, j.mask_host, (uint64_t*)dfwd, c.st);
        if (rc) return rc;
        if ((rc = mark(c.tm, kTmCounted, c.st))) return rc;
    }
    if ((rc = queue_tables(c, peers, dfwd, j, space, nullptr, dtab, dig, c.st))) return rc;
    g_trace.stamp("finalize_queued");
    if (late) {
        if ((rc = (*late)(&wins))) return rc;
        g_trace.stamp("windows");
        if ((rc = upload_windows())) return rc;
        g_trace.stamp("windows_queued");
    }
    if (c.cc) CK(cudaStreamWaitEvent(c.st, c.cc->windows, 0));
    if (wins.n) {
        if ((rc = mark(c.tm, kTmScoreStart, c.st))) return rc;
        rc = frisk_b200_score(q.codes, q.inv, q.low, (const uint64_t*)dwo, (const uint32_t*)dwl, wins.n, wins.max_len,
                              (const double*)dig, j.kmin, j.kmax, j.want_rip, r.rows, r.status, nullptr, c.st);
        if (rc) return rc;
        g_trace.stamp("score_queued");
        if ((rc = mark(c.tm, kTmScored, c.st))) return rc;
    }
    return results(c, wins.n, r, j, dtab);
}

// ---- planes in host memory (frisk_b200_run_host / _sparse / _peers) ---------------------------------------------------

// One genome's planes in host memory; the invalid plane either dense or as its non-zero words.
struct HostPlanes {
    const uint32_t* codes;
    const uint32_t* inv;            // dense (padded_len / 32 words) or nullptr
    const uint32_t* inv_idx;        // sparse: word indices ...
    const uint32_t* inv_val;        // ... and the words
    uint64_t inv_n;
    const uint32_t* low;            // nullable
    uint64_t padded_len;
};

__global__ void __launch_bounds__(256)
plane_scatter_kernel(const uint32_t* __restrict__ idx, const uint32_t* __restrict__ val, uint64_t n, uint32_t* __restrict__ plane) {
    const uint64_t i = (uint64_t)blockIdx.x * 256u + threadIdx.x;
    if (i < n) plane[idx[i]] = val[i];
}

// invalid plane of `hp` -> d_inv on stream s (sparse: zero fill + pairs + scatter)
int upload_inv(const HostPlanes& hp, void* d_inv, WsSlot slot_idx, WsSlot slot_val, cudaStream_t s) {
    if (hp.inv) return FRISK_OK;                      // dense: goes up with the code chunks
    CK(cudaMemsetAsync(d_inv, 0, hp.padded_len / 8, s));
    if (hp.inv_n) {
        void *di, *dv;
        int rc;
        if ((rc = ws_get(slot_idx, hp.inv_n * 4, &di))) return rc;
        if ((rc = ws_get(slot_val, hp.inv_n * 4, &dv))) return rc;
        CK(cudaMemcpyAsync(di, hp.inv_idx, hp.inv_n * 4, cudaMemcpyHostToDevice, s));
        CK(cudaMemcpyAsync(dv, hp.inv_val, hp.inv_n * 4, cudaMemcpyHostToDevice, s));
        plane_scatter_kernel<<<(unsigned)((hp.inv_n + 255) / 256), 256, 0, s>>>((const uint32_t*)di, (const uint32_t*)dv, hp.inv_n,
                                                                               (uint32_t*)d_inv);
        CK(cudaGetLastError());
    }
    return FRISK_OK;
}

int run_host_body(RunCall& c, const PeerArgs& peers, const HostPlanes& h, const HostPlanes& q, bool same, const WindowList& wins,
                  const Job& j, int64_t space) {
    const uint64_t h_padded_len = h.padded_len, q_padded_len = q.padded_len;
    const size_t tsz = table_words(j.kmax);
    CopyCtx* const cc = c.cc;
    void *dhc, *dhi, *dhl = nullptr, *dqc, *dqi, *dql = nullptr, *dfwd;
    int rc;
    if ((rc = ws_get(kWsHostCodes, h_padded_len / 4, &dhc))) return rc;
    if ((rc = ws_get(kWsHostInv, h_padded_len / 8, &dhi))) return rc;
    if (h.low && (rc = ws_get(kWsHostLow, h_padded_len / 8, &dhl))) return rc;
    if (peers.world) {
        dfwd = peers.d_fwd_local;                     // this rank's counters live where the peers can read them
        CK(cudaMemsetAsync(dfwd, 0, tsz * 8, c.st));
    } else {
        if ((rc = ws_get(kWsFwd, (tsz + 1) * 8, &dfwd))) return rc;
        CK(cudaMemsetAsync(dfwd, 0, (tsz + 1) * 8, c.st));
    }
    // The planes go up in chunks on the copy stream; the background count of a chunk starts as soon
    // as the chunk has landed (it stops 128 bases short of the chunk's end: the kernel looks ahead),
    // so only the last chunk's count is not hidden behind PCIe.
    CK(cudaEventRecord(cc->join, c.st));
    CK(cudaStreamWaitEvent(cc->copy, cc->join, 0));                  // order behind earlier work on `stream`
    // sparse invalid plane: zero fill + pairs + scatter on the COMPUTE stream, behind the first code chunk's transfer
    // (on the copy stream they would delay that chunk by four small operations); the counts on `st` follow in order
    if ((rc = upload_inv(h, dhi, kWsHostInvIdx, kWsHostInvVal, c.st))) return rc;
    // Chunk plan: equal chunks of <= 64 M bases.  Measured on C2 (40 Mbp, profiles/r02_upload_plans.txt): one chunk -- upload,
    // then one count of 0.07 ms -- beats every split (2 chunks +0.02 ms, 3 chunks +0.04..0.1 ms): a count that runs beside
    // the copy takes about twice as long, every extra copy and count launch has a fixed cost, and the whole count is short
    // next to the upload.  Genomes of hundreds of Mbp and more keep the split: there the last chunk's count is what shows.
    // (One chunk wins also when eight ranks share the host's H2D bandwidth and the upload takes twice as long, profiles/
    // r02_pcie_contention_8gpu.json: two chunks measured 0.50 ms to the end of the count against 0.48 for one.)
    int n_parts = (int)((h_padded_len + (64ull << 20) - 1) / (64ull << 20));
    if (n_parts > kMaxChunks - 1) n_parts = kMaxChunks - 1;
    if (n_parts < 1) n_parts = 1;
    uint64_t bounds[kMaxChunks + 1];
    uint64_t n_chunks = 0;
    bounds[0] = 0;
    for (int i = 1; i <= n_parts; ++i) {
        uint64_t b = i == n_parts ? h_padded_len : ((h_padded_len / (uint64_t)n_parts) * (uint64_t)i + 127) & ~127ull;
        if (b > h_padded_len) b = h_padded_len;
        if (b > bounds[n_chunks]) bounds[++n_chunks] = b;
    }
    uint64_t counted = 0;
    for (uint64_t k = 0; k < n_chunks; ++k) {
        const uint64_t b0 = bounds[k], b1 = bounds[k + 1];
        if (b0 >= b1) continue;
        CK(cudaMemcpyAsync((char*)dhc + b0 / 4, (const char*)h.codes + b0 / 4, (b1 - b0) / 4, cudaMemcpyHostToDevice, cc->copy));
        if (h.inv) CK(cudaMemcpyAsync((char*)dhi + b0 / 8, (const char*)h.inv + b0 / 8, (b1 - b0) / 8, cudaMemcpyHostToDevice, cc->copy));
        if (h.low) CK(cudaMemcpyAsync((char*)dhl + b0 / 8, (const char*)h.low + b0 / 8, (b1 - b0) / 8, cudaMemcpyHostToDevice, cc->copy));
        CK(cudaEventRecord(cc->chunk[k], cc->copy));
        CK(cudaStreamWaitEvent(c.st, cc->chunk[k], 0));
        const uint64_t upto = (b1 == h_padded_len) ? h_padded_len - 32 : b1 - 128;
        if (upto > counted) {
            rc = frisk_b200_background((const uint32_t*)dhc, (const uint32_t*)dhi, (const uint32_t*)dhl, counted, upto, j.kmax,
                                       j.mask_host, (uint64_t*)dfwd, c.st);
            if (rc) return rc;
            counted = upto;
        }
    }
    if ((rc = mark(c.tm, kTmUploaded, cc->copy))) return rc;
    if ((rc = mark(c.tm, kTmCounted, c.st))) return rc;
    if (same) { dqc = dhc; dqi = dhi; dql = dhl; }
    else {
        if ((rc = ws_get(kWsQueryCodes, q_padded_len / 4, &dqc))) return rc;
        if ((rc = ws_get(kWsQueryInv, q_padded_len / 8, &dqi))) return rc;
        if (q.low && (rc = ws_get(kWsQueryLow, q_padded_len / 8, &dql))) return rc;
        CK(cudaMemcpyAsync(dqc, q.codes, q_padded_len / 4, cudaMemcpyHostToDevice, cc->copy));
        if (q.inv) CK(cudaMemcpyAsync(dqi, q.inv, q_padded_len / 8, cudaMemcpyHostToDevice, cc->copy));
        else if ((rc = upload_inv(q, dqi, kWsQueryInvIdx, kWsQueryInvVal, cc->copy))) return rc;
        if (q.low) CK(cudaMemcpyAsync(dql, q.low, q_padded_len / 8, cudaMemcpyHostToDevice, cc->copy));
    }
    return run_tail(c, peers, Planes{(const uint32_t*)dhc, (const uint32_t*)dhi, (const uint32_t*)dhl, h_padded_len}, true,
                    Planes{(const uint32_t*)dqc, (const uint32_t*)dqi, (const uint32_t*)dql, q_padded_len}, wins, j, space, dfwd);
}

int run_host_any(const PeerArgs& peers, const HostPlanes& h, const HostPlanes& q, bool same, const WindowList& wins, const Job& j,
                 int64_t space, void* stream) {
    const bool planes = h.codes && q.codes && (h.inv || h.inv_idx || !h.inv_n) && (q.inv || q.inv_idx || !q.inv_n);
    int rc = check_plane_run(planes, h.padded_len, q.padded_len, wins, j);
    if (rc) return rc;
    RunCall c;
    if (!(rc = c.enter(stream, true))) rc = run_host_body(c, peers, h, q, same, wins, j, space);
    return c.leave(rc);
}

// ---- FASTA text in, rows out, one call -------------------------------------------------------------------------------
// The text goes up in chunks; each chunk is tokenised, laid out, packed and (kmax <= 8) counted on the device while the
// next one is on the bus (frisk_ingest.cu).  The host sees the record table as soon as the last chunk is tokenised, derives
// names and windows while that chunk is still being packed and counted, and queues tables -> IVOM -> window kernel behind it.
struct HostStage { void* p = nullptr; size_t cap = 0; };
HostStage g_stage[64][2];        // pinned staging of the window list (off, len), grown on demand

int stage_get(int dev, int slot, size_t bytes, void** out) {
    HostStage& s = g_stage[dev & 63][slot];
    if (s.cap < bytes) {
        if (s.p) CK(cudaFreeHost(s.p));
        s.p = nullptr; s.cap = 0;
        const size_t want = bytes + bytes / 2 + 4096;
        CK(cudaHostAlloc(&s.p, want, cudaHostAllocDefault));
        s.cap = want;
    }
    *out = s.p;
    return FRISK_OK;
}

// fmt: h_text / q_text are texts, BGZF buffers or gzip members (the last two inflated on the device by the ingest), or .2bit
// files (decoded on the device into the planes by frisk_twobit.cu)
int run_fasta_body(RunCall& c, const char* h_text, uint64_t h_n, const char* q_text, uint64_t q_n, frisk_internal::TextFormat fmt,
                   int w, int step, int scaffolds_all, const Job& j, uint64_t rows_cap, uint64_t* n_win_out,
                   frisk_b200_fasta** host_out, frisk_b200_fasta** query_out) {
    const int kmin = j.kmin, kmax = j.kmax;
    const size_t tsz = table_words(kmax);
    void* dfwd;
    int rc;
    if ((rc = ws_get(kWsFwd, (tsz + 1) * 8, &dfwd))) return rc;
    CK(cudaMemsetAsync(dfwd, 0, (tsz + 1) * 8, c.st));

    frisk_internal::IngestSink sink;
    if (kmax <= FRISK_B200_FAST_K)
        sink.on_range = [&](const uint32_t* cd, const uint32_t* i, const uint32_t* l, const unsigned long long* d_range,
                            uint64_t hint, cudaStream_t s2) {
            return frisk_internal::background_device_range(cd, i, l, d_range, hint, kmax, j.mask_host, (uint64_t*)dfwd, s2);
        };
    sink.abandon = [&](cudaStream_t s2) {
        CK(cudaMemsetAsync(dfwd, 0, (tsz + 1) * 8, s2));
        return (int)FRISK_OK;
    };
    sink.uploaded_mark = c.tm->ev[kTmUploaded];
    const bool same = !q_text || (q_text == h_text && q_n == h_n);

    // ---- the device-only tail: with the nibble kernel (kmax 7, 8; windows <= 8,186 bases) everything behind the ingest is queued
    // from inside the open, before the host has seen the record table -- genome space and window list by frisk_windows.cu,
    // the window count read by the window kernel from device memory -- so that no launch waits for the host.  If the
    // streamed open has to be redone (sink.counted comes back false), what was queued here ran on provisional data into
    // the caller's row buffers (inside their capacity) and is simply done again by the host-driven tail below.
    const double min_size = (double)w + (((double)w * 0.75) - (double)step);
    const uint32_t len_bound = (uint32_t)std::min<double>(4.0e9, std::max<double>((double)w, scaffolds_all ? min_size : 0.0));
    WinPlan tail_plan;
    const bool dev_tail = rows_cap > 0 && rows_cap <= 0xffffffffull && (uint64_t)w <= FRISK_B200_MAX_WINDOW &&
                          frisk_internal::plan_score(kmin, kmax, len_bound, false, &tail_plan) == FRISK_OK &&
                          tail_plan.kind == WinKernel::Nibble;
    void *dtab = nullptr, *dig = nullptr, *dwin = nullptr, *dfirst = nullptr, *dscal = nullptr;
    Rows r{};
    bool tail_queued = false;
    if (dev_tail) {
        if ((rc = ws_get(kWsTables, (tsz + 1) * 8, &dtab))) return rc;
        if ((rc = ws_get(kWsIvom, ivom_bytes(kmax), &dig))) return rc;
        if ((rc = ws_get(kWsWinOff, rows_cap * 12, &dwin))) return rc;
        if ((rc = ws_get(kWsScalars, 64, &dscal))) return rc;
        if ((rc = rows_for(rows_cap, j, &r))) return rc;
    }
    unsigned long long* const scal = (unsigned long long*)dscal;
    const uint32_t* win_codes[3] = {nullptr, nullptr, nullptr};      // planes of the genome whose windows are scored
    auto queue_windows = [&](frisk_b200_fasta* h, bool with_space, cudaStream_t s2) -> int {
        const unsigned long long *d_len, *d_off, *d_ctr;
        uint64_t rec_cap = 0;
        int rc2;
        if ((rc2 = frisk_internal::fasta_device_table(h, &d_len, &d_off, &d_ctr, &rec_cap, &win_codes[0], &win_codes[1], &win_codes[2])))
            return rc2;
        if ((rc2 = ws_get(kWsFirst, (rec_cap + 2) * 8, &dfirst))) return rc2;
        return frisk_internal::windows_device(d_len, d_off, d_ctr + frisk_internal::kIngestRecords, d_ctr + frisk_internal::kIngestOverflow,
                                              d_ctr + frisk_internal::kIngestNonUpper, rec_cap, w, step, scaffolds_all, rows_cap,
                                              (unsigned long long*)dfirst, (unsigned long long*)dwin,
                                              (uint32_t*)((unsigned long long*)dwin + rows_cap), scal,
                                              with_space ? (long long*)(scal + 1) : nullptr, s2);
    };
    auto queue_score = [&](cudaStream_t s2) -> int {
        int rc2;
        if ((rc2 = mark(c.tm, kTmScoreStart, s2))) return rc2;
        rc2 = frisk_internal::score_nibble(tail_plan, win_codes[0], win_codes[1], win_codes[2], (const uint64_t*)dwin,
                                           (const uint32_t*)((unsigned long long*)dwin + rows_cap), rows_cap, len_bound, (const double*)dig,
                                           kmin, kmax, j.want_rip && kmin <= 2 && kmax >= 2 /* as frisk_b200_score: RIP needs orders 1 and 2 */,
                                           r.rows, r.status, nullptr, s2, scal);
        if (rc2) return rc2;
        tail_queued = true;
        return mark(c.tm, kTmScored, s2);
    };
    if (dev_tail)
        sink.on_complete = [&](frisk_b200_fasta* h, cudaStream_t s2) -> int {
            int rc2;
            if ((rc2 = mark(c.tm, kTmCounted, s2))) return rc2;
            // genome space of the host genome (and, when it is the scored genome too, its window list), tables, IVOM, score
            if ((rc2 = queue_windows(h, true, s2))) return rc2;
            if ((rc2 = queue_tables(c, PeerArgs(), dfwd, j, 0, (const long long*)(scal + 1), dtab, dig, s2))) return rc2;
            return same ? queue_score(s2) : FRISK_OK;
        };
    g_trace.stamp("call");
    if ((rc = frisk_internal::fasta_open_planes(h_text, h_n, fmt, c.st, &sink, host_out))) return rc;
    g_trace.stamp("open_returned");
    c.tm->have[kTmUploaded] = h_n > 0;                              // (recorded behind the last text chunk)
    const bool counted = sink.counted;
    bool tail_ok = dev_tail && counted && (tail_queued || !same);   // (an exact re-open leaves counted == false)
    if (!tail_ok) c.tm->have[kTmFinalised] = c.tm->have[kTmScoreStart] = c.tm->have[kTmScored] = false;
    if (counted && !dev_tail && (rc = mark(c.tm, kTmCounted, c.st))) return rc;
    frisk_b200_fasta* hh = *host_out;
    frisk_b200_fasta* qh = hh;
    if (!same) {
        frisk_internal::IngestSink qsink;                            // planes only: nothing of the query is counted
        bool q_queued = false;
        if (tail_ok)
            qsink.on_complete = [&](frisk_b200_fasta* h, cudaStream_t s2) -> int {
                int rc2;
                if ((rc2 = queue_windows(h, false, s2))) return rc2;
                if ((rc2 = queue_score(s2))) return rc2;
                q_queued = true;
                return FRISK_OK;
            };
        qsink.counted = false;
        if ((rc = frisk_internal::fasta_open_planes(q_text, q_n, fmt, c.st, &qsink, query_out))) return rc;
        qh = *query_out;
        // (qsink has no on_range, so `counted` says nothing: a query that was re-opened exactly has a handle without the
        // speculative table the hook used -- detect it by the hook not having run or the open statistics)
        tail_ok = tail_ok && q_queued && frisk_internal::fasta_open_was_streamed(qh);
    }
    uint64_t h_rec = 0, h_padded = 0, h_stats[3], q_rec = 0, q_padded = 0, q_stats[3];
    if ((rc = frisk_b200_fasta_info(hh, &h_rec, &h_padded, h_stats))) return rc;
    if ((rc = frisk_b200_fasta_info(qh, &q_rec, &q_padded, q_stats))) return rc;
    const uint32_t *dhc, *dhi, *dhl, *dqc, *dqi, *dql;
    if ((rc = frisk_b200_fasta_planes(hh, &dhc, &dhi, &dhl))) return rc;
    if ((rc = frisk_b200_fasta_planes(qh, &dqc, &dqi, &dql))) return rc;
    const int64_t space = (int64_t)h_stats[0] - (int64_t)h_stats[1];

    if (tail_ok) {
        // everything is queued: bring the rows and the [window count, genome space] back, wait, check the capacity
        void* h_scal = nullptr;
        if ((rc = stage_get(c.dev, 1, 64, &h_scal))) return rc;
        if ((rc = results(c, rows_cap, r, j, dtab, dscal, h_scal, 16))) return rc;
        const uint64_t n_win = ((const uint64_t*)h_scal)[0];
        if (n_win_out) *n_win_out = n_win;
        if ((int64_t)((const uint64_t*)h_scal)[1] != space) return FRISK_E_CUDA;   // (cannot happen)
        return n_win > rows_cap ? FRISK_E_CAPACITY : FRISK_OK;
    }
    // windows of the query (F:194-251), into pinned staging -- produced once the tables' finalisation is queued
    const LateWindows late = [&](WindowList* wins) -> int {
        int rc2;
        std::vector<uint64_t> seq_len((size_t)q_rec), scaf_off((size_t)q_rec);
        if ((rc2 = frisk_b200_fasta_records(qh, nullptr, nullptr, seq_len.data(), scaf_off.data()))) return rc2;
        void *wo = nullptr, *wl = nullptr;
        if ((rc2 = stage_get(c.dev, 0, (rows_cap + 1) * 12, &wo))) return rc2;
        if ((rc2 = stage_get(c.dev, 1, (rows_cap + 1) * 4, &wl))) return rc2;
        uint64_t nw = 0;
        rc2 = frisk_b200_windows(seq_len.data(), scaf_off.data(), q_rec, w, step, scaffolds_all, rows_cap, (uint64_t*)wo, (uint32_t*)wl,
                                 nullptr, nullptr, nullptr, &nw);
        if (n_win_out) *n_win_out = nw;
        if (rc2) return rc2;                                         // (FRISK_E_CAPACITY: more windows than rows_cap)
        uint32_t mx = 0;
        uint32_t* const packed = (uint32_t*)((uint64_t*)wo + nw);    // the lengths move right behind the offsets: one H2D copy
        for (uint64_t i = 0; i < nw; ++i) {
            const uint32_t l = ((const uint32_t*)wl)[i];
            packed[i] = l;
            mx = l > mx ? l : mx;
        }
        *wins = {(const uint64_t*)wo, packed, nw, mx};
        return FRISK_OK;
    };
    CK(cudaEventRecord(c.cc->join, c.st));                          // the copy stream joins behind the ingest
    CK(cudaStreamWaitEvent(c.cc->copy, c.cc->join, 0));
    return run_tail(c, PeerArgs(), Planes{dhc, dhi, dhl, h_padded}, counted, Planes{dqc, dqi, dql, q_padded}, {}, j, space, dfwd,
                    &late);
}

// frisk_b200_run_fasta, _run_fasta_bgzf, _run_fasta_gzip and _run_2bit
int run_fasta_any(const char* h_text, uint64_t h_n, const char* q_text, uint64_t q_n, frisk_internal::TextFormat fmt, int w, int step,
                  int scaffolds_all, int kmin, int kmax, int mask_host, int want_rip, uint64_t rows_cap, double* rows_out,
                  uint32_t* status_out, uint64_t* tables_out, uint64_t* valid_kmax_out, uint64_t* n_win_out,
                  frisk_b200_fasta** host_out, frisk_b200_fasta** query_out, void* stream) {
    if (!host_out || !query_out || (!h_text && h_n) || (!q_text && q_n) || (rows_cap && (!rows_out || !status_out)))
        return FRISK_E_INVALID;
    *host_out = *query_out = nullptr;
    if (n_win_out) *n_win_out = 0;
    int rc = frisk_internal::check_k(kmin, kmax);
    if (rc) return rc;
    if (w < 1 || step < 1) return FRISK_E_INVALID;
    const Job j{kmin, kmax, mask_host, want_rip, rows_out, status_out, tables_out, valid_kmax_out};
    RunCall c;
    bool threw = false;
    if (!(rc = c.enter(stream, true))) {
        try {
            rc = run_fasta_body(c, h_text, h_n, q_text, q_n, fmt, w, step, scaffolds_all, j, rows_cap, n_win_out, host_out, query_out);
        } catch (...) {
            rc = FRISK_E_CAPACITY;
            threw = true;
        }
    }
    if (c.leave(rc) != FRISK_OK && (rc != FRISK_E_CAPACITY || threw)) {   // (too few rows: the handles stay, with their planes)
        if (*query_out) frisk_b200_fasta_close(*query_out, c.st);
        if (*host_out) frisk_b200_fasta_close(*host_out, c.st);
        *host_out = *query_out = nullptr;
    }
    return rc;
}

}  // namespace

int frisk_b200_run_host(const uint32_t* h_codes, const uint32_t* h_inv, const uint32_t* h_low, uint64_t h_padded_len,
                        const uint32_t* q_codes, const uint32_t* q_inv, const uint32_t* q_low, uint64_t q_padded_len,
                        const uint64_t* win_off, const uint32_t* win_len, uint64_t n_win, uint32_t max_win_len,
                        int kmin, int kmax, int mask_host, int want_rip, int64_t genome_space, double* rows_out,
                        uint32_t* status_out, uint64_t* tables_out, uint64_t* valid_kmax_out, void* stream) {
    if (!h_inv || !q_inv) return FRISK_E_INVALID;
    const HostPlanes h{h_codes, h_inv, nullptr, nullptr, 0, h_low, h_padded_len};
    const HostPlanes q{q_codes, q_inv, nullptr, nullptr, 0, q_low, q_padded_len};
    const bool same = (h_codes == q_codes) && (h_inv == q_inv) && (h_padded_len == q_padded_len);
    return run_host_any(PeerArgs(), h, q, same, {win_off, win_len, n_win, max_win_len},
                        {kmin, kmax, mask_host, want_rip, rows_out, status_out, tables_out, valid_kmax_out}, genome_space, stream);
}

int frisk_b200_run_host_sparse(const uint32_t* h_codes, const uint32_t* h_inv_idx, const uint32_t* h_inv_val, uint64_t h_inv_n,
                               const uint32_t* h_low, uint64_t h_padded_len, const uint32_t* q_codes,
                               const uint32_t* q_inv_idx, const uint32_t* q_inv_val, uint64_t q_inv_n, const uint32_t* q_low,
                               uint64_t q_padded_len, const uint64_t* win_off, const uint32_t* win_len, uint64_t n_win,
                               uint32_t max_win_len, int kmin, int kmax, int mask_host, int want_rip, int64_t genome_space,
                               double* rows_out, uint32_t* status_out, uint64_t* tables_out, uint64_t* valid_kmax_out,
                               void* stream) {
    if ((h_inv_n && (!h_inv_idx || !h_inv_val)) || (q_inv_n && (!q_inv_idx || !q_inv_val))) return FRISK_E_INVALID;
    if (h_padded_len / 32 > 0xffffffffull || q_padded_len / 32 > 0xffffffffull) return FRISK_E_UNSUPPORTED;   // 32-bit word indices
    const HostPlanes h{h_codes, nullptr, h_inv_idx, h_inv_val, h_inv_n, h_low, h_padded_len};
    const HostPlanes q{q_codes, nullptr, q_inv_idx, q_inv_val, q_inv_n, q_low, q_padded_len};
    const bool same = (h_codes == q_codes) && (h_inv_idx == q_inv_idx) && (h_inv_n == q_inv_n) && (h_padded_len == q_padded_len);
    return run_host_any(PeerArgs(), h, q, same, {win_off, win_len, n_win, max_win_len},
                        {kmin, kmax, mask_host, want_rip, rows_out, status_out, tables_out, valid_kmax_out}, genome_space, stream);
}

int frisk_b200_run_host_peers(const uint32_t* h_codes, const uint32_t* h_inv_idx, const uint32_t* h_inv_val, uint64_t h_inv_n,
                              const uint32_t* h_low, uint64_t h_padded_len, const uint64_t* win_off, const uint32_t* win_len,
                              uint64_t n_win, uint32_t max_win_len, int kmin, int kmax, int mask_host, int want_rip,
                              int64_t genome_space, uint64_t* d_fwd_local, const uint64_t* const* d_fwd_peers,
                              uint64_t* const* d_flag_peers, int rank, int world, uint64_t epoch, double* rows_out,
                              uint32_t* status_out, uint64_t* tables_out, uint64_t* valid_kmax_out, void* stream) {
    if ((h_inv_n && (!h_inv_idx || !h_inv_val)) || world < 1 || rank < 0 || rank >= world || !d_fwd_local || !d_fwd_peers ||
        !d_flag_peers || epoch == 0)
        return FRISK_E_INVALID;
    if (h_padded_len / 32 > 0xffffffffull || kmax > FRISK_B200_FAST_K || world > frisk_internal::kMaxPeers) return FRISK_E_UNSUPPORTED;
    const HostPlanes h{h_codes, nullptr, h_inv_idx, h_inv_val, h_inv_n, h_low, h_padded_len};
    return run_host_any({d_fwd_local, d_fwd_peers, d_flag_peers, rank, world, epoch}, h, h, true, {win_off, win_len, n_win, max_win_len},
                        {kmin, kmax, mask_host, want_rip, rows_out, status_out, tables_out, valid_kmax_out}, genome_space, stream);
}

int frisk_b200_run_resident(const uint32_t* d_h_codes, const uint32_t* d_h_inv, const uint32_t* d_h_low,
                            uint64_t h_padded_len, const uint32_t* d_q_codes, const uint32_t* d_q_inv,
                            const uint32_t* d_q_low, uint64_t q_padded_len, const uint64_t* win_off,
                            const uint32_t* win_len, uint64_t n_win, uint32_t max_win_len, int kmin, int kmax,
                            int mask_host, int want_rip, int64_t genome_space, double* rows_out, uint32_t* status_out,
                            uint64_t* tables_out, uint64_t* valid_kmax_out, void* stream) {
    const WindowList wins{win_off, win_len, n_win, max_win_len};
    const Job j{kmin, kmax, mask_host, want_rip, rows_out, status_out, tables_out, valid_kmax_out};
    int rc = check_plane_run(d_h_codes && d_h_inv && d_q_codes && d_q_inv, h_padded_len, q_padded_len, wins, j);
    if (rc) return rc;
    RunCall c;
    void* dfwd;
    if (!(rc = c.enter(stream, false)) && !(rc = ws_get(kWsFwd, (table_words(kmax) + 1) * 8, &dfwd)))
        rc = run_tail(c, PeerArgs(), Planes{d_h_codes, d_h_inv, d_h_low, h_padded_len}, false,
                      Planes{d_q_codes, d_q_inv, d_q_low, q_padded_len}, wins, j, genome_space, dfwd);
    return c.leave(rc);
}

int frisk_b200_run_fasta(const char* h_text, uint64_t h_n, const char* q_text, uint64_t q_n, int w, int step, int scaffolds_all,
                         int kmin, int kmax, int mask_host, int want_rip, uint64_t rows_cap, double* rows_out,
                         uint32_t* status_out, uint64_t* tables_out, uint64_t* valid_kmax_out, uint64_t* n_win_out,
                         frisk_b200_fasta** host_out, frisk_b200_fasta** query_out, void* stream) {
    return run_fasta_any(h_text, h_n, q_text, q_n, frisk_internal::kFmtText, w, step, scaffolds_all, kmin, kmax, mask_host, want_rip, rows_cap, rows_out,
                         status_out, tables_out, valid_kmax_out, n_win_out, host_out, query_out, stream);
}

int frisk_b200_run_fasta_bgzf(const char* h_gz, uint64_t h_n, const char* q_gz, uint64_t q_n, int w, int step, int scaffolds_all,
                              int kmin, int kmax, int mask_host, int want_rip, uint64_t rows_cap, double* rows_out,
                              uint32_t* status_out, uint64_t* tables_out, uint64_t* valid_kmax_out, uint64_t* n_win_out,
                              frisk_b200_fasta** host_out, frisk_b200_fasta** query_out, void* stream) {
    return run_fasta_any(h_gz, h_n, q_gz, q_n, frisk_internal::kFmtBgzf, w, step, scaffolds_all, kmin, kmax, mask_host, want_rip,
                         rows_cap, rows_out, status_out, tables_out, valid_kmax_out, n_win_out, host_out, query_out, stream);
}

int frisk_b200_run_fasta_gzip(const char* h_gz, uint64_t h_n, const char* q_gz, uint64_t q_n, int w, int step, int scaffolds_all,
                              int kmin, int kmax, int mask_host, int want_rip, uint64_t rows_cap, double* rows_out,
                              uint32_t* status_out, uint64_t* tables_out, uint64_t* valid_kmax_out, uint64_t* n_win_out,
                              frisk_b200_fasta** host_out, frisk_b200_fasta** query_out, void* stream) {
    return run_fasta_any(h_gz, h_n, q_gz, q_n, frisk_internal::kFmtGzip, w, step, scaffolds_all, kmin, kmax, mask_host, want_rip,
                         rows_cap, rows_out, status_out, tables_out, valid_kmax_out, n_win_out, host_out, query_out, stream);
}

int frisk_b200_run_2bit(const char* h_2bit, uint64_t h_n, const char* q_2bit, uint64_t q_n, int w, int step, int scaffolds_all,
                        int kmin, int kmax, int mask_host, int want_rip, uint64_t rows_cap, double* rows_out, uint32_t* status_out,
                        uint64_t* tables_out, uint64_t* valid_kmax_out, uint64_t* n_win_out, frisk_b200_fasta** host_out,
                        frisk_b200_fasta** query_out, void* stream) {
    return run_fasta_any(h_2bit, h_n, q_2bit, q_n, frisk_internal::kFmt2bit, w, step, scaffolds_all, kmin, kmax, mask_host, want_rip,
                         rows_cap, rows_out, status_out, tables_out, valid_kmax_out, n_win_out, host_out, query_out, stream);
}

// Stage times (ms) of the last frisk_b200_run_* call on the current device,
// from events recorded on its streams: [0] upload of the planes finished, [1] background count finished, [2] tables
// finalised + genome IVOM table (multi-GPU: includes the wait for the peers' counters), [3] window kernel(s) finished,
// [4] results on the host -- each since the start of the call -- and [5] the moment the window kernel could start
// (everything it waits for is done and its launch has reached the device).  A mark the call did not set
// (run_resident has no upload) reads -1.
int frisk_b200_last_run_timing(float* ms, int cap, int* n) {
    if (!ms || cap < 1) return FRISK_E_INVALID;
    int dev = 0;
    CK(cudaGetDevice(&dev));
    RunMarks& m = g_marks[dev & 63];
    if (!m.ready || !m.have[kTmStart] || !m.have[kTmEnd]) return FRISK_E_INVALID;
    CK(cudaEventSynchronize(m.ev[kTmEnd]));
    const int order[6] = {kTmUploaded, kTmCounted, kTmFinalised, kTmScored, kTmEnd, kTmScoreStart};
    int k = 0;
    for (; k < 6 && k < cap; ++k) {
        ms[k] = -1.0f;
        if (!m.have[order[k]]) continue;
        if (order[k] == kTmUploaded) CK(cudaEventSynchronize(m.ev[kTmUploaded]));
        CK(cudaEventElapsedTime(&ms[k], m.ev[kTmStart], m.ev[order[k]]));
    }
    if (n) *n = k;
    return FRISK_OK;
}

int frisk_b200_release_workspace(void) {
    int dev = 0;
    CK(cudaGetDevice(&dev));
    Workspace& w = g_ws[dev & 63];
    for (int i = 0; i < kWsSlots; ++i) {
        if (w.buf[i]) CK(cudaFree(w.buf[i]));
        w.buf[i] = nullptr; w.cap[i] = 0;
    }
    return FRISK_OK;
}
