// C ABI of the engine (include/rssync_b200.h): problem state, host->device staging, kernel
// launches, and the host-side control loop of Sync.  Everything numerical on the hot path runs
// in engine.cu; this file holds what the reference keeps in OptData / SyncProblemPrivate
// (core_private.hpp:15-61) plus the solver's irregular iteration control, which stays on the
// host (Backtrack, backtrack.cpp:3-13; momentum loop, core_private.cpp:298-331).
#include "rssync_b200.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <unordered_set>
#include <utility>
#include <vector>
#if defined(__x86_64__)
#include <immintrin.h>
#endif
#if defined(__linux__)
#include <pthread.h>
#include <sched.h>
#endif
#ifndef RSSYNC_STAGE_DEFAULT
#define RSSYNC_STAGE_DEFAULT 2  // staging copy: 0 scalar, 1 AVX2, 2 AVX2 with non-temporal stores
#endif

#include <nvtx3/nvToolsExt.h>  // header-only; a no-op unless a profiler is attached

#include "engine.h"
#include "host_ingest.h"
#include "nccl_dyn.h"
#include "rng.h"
#include "spec_trig.h"

using rs::FrameDesc;

namespace {

#define CUDA_TRY(p, expr)                                                                 \
    do {                                                                                  \
        cudaError_t e__ = (expr);                                                         \
        if (e__ != cudaSuccess) {                                                         \
            (p)->err = std::string("CUDA error: ") + cudaGetErrorString(e__) + " at " #expr; \
            return RSSYNC_E_CUDA;                                                         \
        }                                                                                 \
    } while (0)

// growable device buffer
template <class T>
struct DevBuf {
    T* ptr = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        size_t want = std::max(n, cap * 2);
        cudaError_t e = cudaMalloc((void**)&ptr, want * sizeof(T));
        cap = (e == cudaSuccess) ? want : 0;
        return e;
    }
    // grow to at least n elements keeping the first `keep` (device-to-device copy on `st`)
    cudaError_t grow(size_t n, size_t keep, cudaStream_t st) {
        if (n <= cap) return cudaSuccess;
        size_t want = std::max(n, cap * 2);
        T* np = nullptr;
        cudaError_t e = cudaMalloc((void**)&np, want * sizeof(T));
        if (e != cudaSuccess) return e;
        if (ptr && keep) e = cudaMemcpyAsync(np, ptr, std::min(keep, cap) * sizeof(T), cudaMemcpyDeviceToDevice, st);
        if (e == cudaSuccess && ptr) {
            e = cudaStreamSynchronize(st);
            cudaFree(ptr);
        }
        ptr = np;
        cap = want;
        return e;
    }
    void release() {
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        cap = 0;
    }
};

// growable pinned host buffer
template <class T>
struct PinBuf {
    T* ptr = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t n, size_t keep = 0) {
        if (n <= cap) return cudaSuccess;
        size_t want = std::max(n, cap * 2);
        T* np = nullptr;
        cudaError_t e = cudaHostAlloc((void**)&np, want * sizeof(T), cudaHostAllocDefault);
        if (e != cudaSuccess) return e;
        if (ptr && keep) std::memcpy(np, ptr, std::min(keep, cap) * sizeof(T));
        if (ptr) cudaFreeHost(ptr);
        ptr = np;
        cap = want;
        return cudaSuccess;
    }
    void release() {
        if (ptr) cudaFreeHost(ptr);
        ptr = nullptr;
        cap = 0;
    }
};

// RSSYNC_DEBUG_TIMING=1: wall-clock marks of the host-side ingest on stderr
// NVTX range around a C-ABI call: the calls show up by name on a profiler's timeline (SURVEY section 5)
struct NvtxRange {
    explicit NvtxRange(const char* name) { nvtxRangePushA(name); }
    ~NvtxRange() { nvtxRangePop(); }
    NvtxRange(const NvtxRange&) = delete;
    NvtxRange& operator=(const NvtxRange&) = delete;
};
#define RS_NVTX_RANGE() NvtxRange nvtx_range_(__func__)

struct DebugTimer {
    bool on;
    std::chrono::steady_clock::time_point t0;
    const char* who;
    explicit DebugTimer(const char* w) : on(std::getenv("RSSYNC_DEBUG_TIMING") != nullptr), t0(std::chrono::steady_clock::now()), who(w) {}
    void mark(const char* what) {
        if (!on) return;
        const auto t = std::chrono::steady_clock::now();
        std::fprintf(stderr, "[%s] %s +%.3f ms\n", who, what, std::chrono::duration<double, std::milli>(t - t0).count());
        t0 = t;
    }
};

bool all_finite(const double* p, size_t n) {
    for (size_t i = 0; i < n; ++i)
        if (!std::isfinite(p[i])) return false;
    return true;
}

}  // namespace

namespace {
struct SyncPointState {
    double delay = 0.0, v = 0.0, center = 0.0, radius = 0.0;
    int converge = 0;
    bool done = false;
};
// One lane of the Sync batch driver (sync_batch_impl): a contiguous group of syncpoints with its
// own stream, device scratch and pinned I/O blocks.
struct SyncLane {
    enum Phase { Running, MoreTrials, Final, Done };
    int n_eval = 10;  // Backtrack trial points evaluated speculatively per iteration (see sync_lane_step)
    cudaStream_t stream = nullptr;
    cudaEvent_t ev = nullptr;
    int s0 = 0, n = 0, t0 = 0, T = 0, iters = 0;
    Phase phase = Done;
    DevBuf<rs::SyncTask> d_tasks;
    DevBuf<int> d_sp_begin, d_lbfgs_stats;
    DevBuf<double> d_m, d_k, d_task_scratch, d_trial_delay, d_in, d_out;
    DevBuf<uint64_t> d_sp_callno;
    PinBuf<double> h_in, h_out;
    size_t in_doubles = 0, out_doubles = 0;
    rs::SyncBatchDev b{};
    std::vector<SyncPointState> st;
    std::vector<int> h_stats, local_sp, sp_frames;  // sp_frames[s]: frames (tasks) of syncpoint s
    const unsigned char* h_active = nullptr;
    bool many_tasks = false;  // which build of the L-BFGS kernel the lane launches (engine.cu LbfgsCfg)
    // one outer iteration (copy in, four kernels, copy out) as an instantiated CUDA graph; valid as
    // long as every captured argument (graph_key) is unchanged, which holds across chained Sync calls
    cudaGraphExec_t graph_exec = nullptr;
    std::vector<unsigned char> graph_key;
    unsigned char* active_dev() const { return reinterpret_cast<unsigned char*>(d_in.ptr + 2 * (size_t)n); }
    unsigned long long* evals_dev() const { return reinterpret_cast<unsigned long long*>(d_out.ptr + out_doubles - 1); }
    void release() {
        d_tasks.release(); d_sp_begin.release(); d_lbfgs_stats.release(); d_m.release(); d_k.release();
        d_task_scratch.release(); d_trial_delay.release(); d_in.release(); d_out.release();
        d_sp_callno.release(); h_in.release(); h_out.release();
        if (graph_exec) cudaGraphExecDestroy(graph_exec);
        graph_exec = nullptr;
        if (ev) cudaEventDestroy(ev);
        if (stream) cudaStreamDestroy(stream);
        ev = nullptr;
        stream = nullptr;
    }
};

}  // namespace

struct rssync_problem {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::string err;

    // gyro spline (OptData::quats, quats_start, sample_rate)
    // pinned staging of one SetGyroQuaternions call: the samples (nq x 4), and the eliminated spline
    // system the worker builds from them, rhs (nq x 4) and diag (nq); one async copy, then the
    // records are finished on the device (launch_spline_finish)
    PinBuf<double> h_gyro;
    DevBuf<double> d_gyro;
    double q0 = 0.0, sr = 0.0;
    size_t nq = 0;
    bool gyro_dirty = false;
    bool gyro_on_device = false;  // the pending gyro was built from device-side inputs (no 9-double upload)
    // The spline coefficient solve (4 sequential recurrences, ~2.5 ms per minute of 1 kHz gyro) runs
    // on a worker thread so that it overlaps the caller's SetTrackResult calls; it is joined by the
    // first thing that needs the records.
    std::thread gyro_worker;
    // the worker also starts the records' host->device copy on its own stream as soon as they are
    // built; the problem's stream waits for ev_gyro before the first kernel that reads them
    cudaStream_t gyro_stream = nullptr;
    cudaEvent_t ev_gyro = nullptr;
    cudaError_t gyro_copy_err = cudaSuccess;  // written by the worker, read after join
    // eager host->device copies issued by the bulk track ingest; host writes to the pinned arena
    // wait for them
    cudaEvent_t ev_arena = nullptr;
    bool arena_copy_pending = false;
    // a foreign stream still reading the device state (rssync_note_reader: a replication in flight)
    cudaEvent_t ev_reader = nullptr;
    bool reader_pending = false;
    // The bulk ingest runs on its own stream, one event per chunk of frames: a PreSync grid that
    // follows evaluates the frames of a chunk as soon as that chunk has landed instead of waiting
    // for the whole upload (the upload of C2 takes 2 ms at the 24 GB/s this host's PCIe delivers,
    // the grid 4.5 ms).  in_flight lists the arena ranges (in rays) still being written, in stream
    // order; anything else that touches the arena waits for all of them first.
    struct InFlight {
        size_t lo, hi;
        cudaEvent_t ev;
        bool foreign = false;  // delivered, or sent on, by a collective's kernel (rssync_expect_chunk / _stream_wait_chunk)
    };
    cudaStream_t copy_stream = nullptr;
    cudaStream_t repl_stream = nullptr;  // multi-device problems: the replication's collectives
    static constexpr int kGridStreams = 3;  // side streams of a chunk-by-chunk PreSync grid
    cudaStream_t grid_stream[kGridStreams] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_grid[kGridStreams] = {nullptr, nullptr, nullptr};
    std::vector<InFlight> in_flight;
    std::vector<cudaEvent_t> ev_pool;
    cudaEvent_t ev_order = nullptr;
    DevBuf<double> d_rec;

    // ray arena (DeviceData::rays): frames appended in arrival order, each padded to a multiple of
    // 32 rays; every group of 32 rays is one 2 KB tile [8 fields][32 rays] of doubles (fields ts_a,
    // ts_b, ra.xyz, rb.xyz), so a frame is one contiguous run of tiles (one TMA bulk copy) and a
    // warp's field loads are full coalesced 256-byte rows.  Inside a frame the rays are stored
    // sorted by ts_a, so the 32 lanes of a warp hit one or two spline records per load instead of
    // ~11 (the rolling-shutter readout spans ~11 gyro samples); `orig` maps a stored ray back to
    // the caller's index and `pos` is its inverse (the estimator's random draws index the caller's
    // order).
    PinBuf<double> h_rays;
    DevBuf<double> d_rays;
    PinBuf<int32_t> h_orig, h_pos;
    DevBuf<int32_t> d_orig, d_pos;
    size_t used = 0, garbage = 0;
    // arena ranges [first, last) (in rays) whose pinned host copy is newer than the device's; frames
    // ingested on the device (rssync_set_track_pixels) never appear here, so the device arena is
    // the one complete copy and grows with its contents preserved
    std::vector<std::pair<size_t, size_t>> pending;
    size_t dev_used = 0;  // extent of the device arena holding data
    std::map<int64_t, FrameDesc> frames;  // OptData::frame_data
    // callers set frames in ascending order, mostly: the node after the one placed last is tried
    // before a tree search (map iterators survive insertions; frames are never erased one by one)
    std::map<int64_t, FrameDesc>::iterator place_hint;
    bool place_hint_valid = false;
    size_t total_rays = 0;

    uint64_t seed = 100, call_no = 0;
    bool simplified = false;  // rssync_set_loss_mode
    // device-side gyro ingest (variable-rate SetGyroQuaternions, orientation search): inputs,
    // per-variant intermediates, and the spline elimination factors of the most recent track length
    DevBuf<int64_t> d_var_ts;
    DevBuf<double> d_var_in, d_var_q, d_var_y, d_var_rhs, d_var_rec, d_var_prefix, d_elim;
    DevBuf<unsigned char> d_var_orients;
    DevBuf<unsigned> d_var_flags;  // the resampling's non-finite flags (one per variant)
    size_t elim_n = 0;

    // ---- several GPUs behind one problem (rssync_create_multi) -----------------------------------
    // The problem the caller holds is the PRIMARY: it takes every Set* call and holds the one
    // complete copy of the inputs.  replicas[i] live on the other devices; before a compute call
    // they receive the primary's finished device state (ray arena, orig / pos planes, spline
    // records) by ncclBroadcast over NVLink -- `version` counts the primary's input changes,
    // `synced_version` is the one a replica holds.  comms[0] is the primary's communicator.
    std::vector<rssync_problem*> replicas;
    std::vector<void*> comms;
    bool is_replica = false, owns_stream = false;
    bool force_single = false;  // the primary works alone (inside a call that has sharded the work itself)
    uint64_t version = 0, synced_version = 0;
    DevBuf<unsigned char> d_gather;   // G slices of {costs of the rank's delays, 2 flag words}
    PinBuf<unsigned char> h_gather;
    uint64_t nccl_calls = 0, broadcast_bytes = 0;

    // Grid scratch of every PreSync entry point: frame tables (the readout search's one per readout),
    // delays, per-task costs, the loss curves and their flag words (2 per curve).  d_pixframes holds the
    // PixelFrame records of set_readout and of the readout search.  One set
    // serves all calls because each buffer is written and read only on `stream`: a call's use of it is
    // ordered after the previous call's, and every call that reads a result back synchronises that
    // stream before it returns.
    DevBuf<FrameDesc> d_frames;
    DevBuf<double> d_delays, d_framecost, d_costs;
    DevBuf<unsigned> d_flags;
    DevBuf<rs::PixelFrame> d_pixframes;
    DevBuf<uint64_t> d_frame_call;
    DevBuf<int> d_win_begin;
    // staging of the bulk ingests
    DevBuf<double> d_stage;
    PinBuf<double> h_stage;
    // sync: per-lane scratch (sync_batch_impl)
    std::vector<SyncLane> lanes;
    cudaEvent_t ev_sync_ready = nullptr;
    DevBuf<double> d_probe;

    // rolling-shutter re-timing (rssync_readout_search, rssync_set_readout).  A frame ingested from pixels
    // keeps its two frame timestamps here and, in d_rowq (2 doubles per arena ray, the caller's ray
    // order), y_a / rows and y_b / rows of every ray; a frame placed by any other form since, and every
    // frame of an adopted state, has no entry.  d_rowq is allocated by the first pixels ingest.
    std::unordered_map<int64_t, std::pair<double, double>> retime;
    DevBuf<double> d_rowq;
    // A multi-device problem sends `retime` and d_rowq to its replicas only for a readout search:
    // rowq_version counts the changes of either (and moves of the plane), rowq_synced is the one a replica
    // holds.  adopted_version: the `version` rssync_adopt_state left, which rssync_adopt_row_fractions
    // requires to be current (no input set since).
    uint64_t rowq_version = 0, rowq_synced = 0, adopted_version = ~0ull;
    // re-timing scratch: the readout search's arena of the selected frames, and the frames' row extremes
    // (4 doubles per frame)
    DevBuf<double> d_rt_rays, d_rt_ext;
    DevBuf<int32_t> d_rt_orig, d_rt_pos;
    // rssync_track_frames_device: image pyramids, the compacted pairs and the tracked positions when the
    // caller takes none (6 doubles per point), the kept offsets, the statuses, the non-finite-query flag
    DevBuf<float> d_trk_pyr;
    DevBuf<double> d_trk_pts;
    DevBuf<int64_t> d_trk_at;
    DevBuf<uint8_t> d_trk_status;
    DevBuf<unsigned> d_trk_flag;
    PinBuf<unsigned> h_trk_flag;
    // rssync_track_frames_ex_device's selection: cell keys, picks and pick counts of a chunk; the
    // selected offsets read back
    DevBuf<unsigned long long> d_trk_keys;
    DevBuf<uint32_t> d_trk_picks;
    DevBuf<int32_t> d_trk_count;
    PinBuf<int64_t> h_trk_qat;
    // rssync_track_frames_masked_device: the eligibility planes (one, or one per pyramid slot)
    DevBuf<uint8_t> d_trk_elig;

    std::vector<std::pair<double, int32_t>> sort_scratch;
    std::vector<double> trace_delay, trace_step;
    uint64_t h2d = 0, d2h = 0, sync_outer = 0, sync_evals = 0;
    // evaluation accounting of the most recent Sync / Sync batch, in (syncpoint, frame) tasks:
    // problem-matrix builds, objective evaluations outside L-BFGS (x0, x0 -/+ h, Backtrack's trial
    // points, the final objective), estimator runs of the initialisation (200 hypotheses each), and
    // the outer iterations summed over syncpoints
    uint64_t sync_row_builds = 0, sync_loss_evals = 0, sync_init_tasks = 0, sync_outer_total = 0;
    uint64_t sync_trial_hist[16] = {0};  // index of the Backtrack trial point accepted (kTrials: none), since creation
    bool kernel_timing = false;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    double last_grid_ms = 0.0;
    uint64_t grid_tasks = 0, grid_exact_tasks = 0;

    rs::DeviceData device_data() const {
        rs::DeviceData dd;
        dd.rec = d_rec.ptr;
        dd.nq = (int)nq;
        dd.q0 = q0;
        dd.sr = sr;
        dd.rays = d_rays.ptr;
        dd.orig = d_orig.ptr;
        dd.pos = d_pos.ptr;
        return dd;
    }
};

namespace {

int h2d(rssync_problem* p, void* dst, const void* src, size_t bytes) {
    if (!bytes) return RSSYNC_OK;
    CUDA_TRY(p, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, p->stream));
    p->h2d += bytes;
    return RSSYNC_OK;
}
int d2h(rssync_problem* p, void* dst, const void* src, size_t bytes) {
    if (!bytes) return RSSYNC_OK;
    CUDA_TRY(p, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, p->stream));
    p->d2h += bytes;
    return RSSYNC_OK;
}

void join_gyro(rssync_problem* p) {
    if (p->gyro_worker.joinable()) p->gyro_worker.join();
}
// a replication still reading this problem's device state on a foreign stream (rssync_note_reader)
int wait_reader(rssync_problem* p) {
    if (p->reader_pending) {
        CUDA_TRY(p, cudaEventSynchronize(p->ev_reader));
        p->reader_pending = false;
    }
    return RSSYNC_OK;
}
int wait_arena_copies(rssync_problem* p) {
    if (p->arena_copy_pending) {
        CUDA_TRY(p, cudaEventSynchronize(p->ev_arena));
        p->arena_copy_pending = false;
    }
    return wait_reader(p);
}

// the problem's stream waits (on the device) for every bulk-ingest chunk still in flight
int wait_in_flight(rssync_problem* p, size_t upto = (size_t)-1) {
    size_t n = std::min(upto, p->in_flight.size());
    if (n == 0) return RSSYNC_OK;
    // the chunks were queued on one stream: the last event covers the earlier ones
    CUDA_TRY(p, cudaStreamWaitEvent(p->stream, p->in_flight[n - 1].ev, 0));
    for (size_t i = 0; i < n; ++i) p->ev_pool.push_back(p->in_flight[i].ev);
    p->in_flight.erase(p->in_flight.begin(), p->in_flight.begin() + (long)n);
    return RSSYNC_OK;
}
// host-side: nothing of the bulk ingest is running any more
int drain_in_flight(rssync_problem* p) {
    if (p->copy_stream) CUDA_TRY(p, cudaStreamSynchronize(p->copy_stream));
    for (const auto& f : p->in_flight) p->ev_pool.push_back(f.ev);
    p->in_flight.clear();
    return RSSYNC_OK;
}

// device arena large enough for `used` rays, contents preserved
int reserve_device_arena(rssync_problem* p, size_t at_least = 0) {
    const size_t want = std::max(std::max(p->used, p->h_orig.cap), at_least);
    if (want > p->d_orig.cap || want * 8 > p->d_rays.cap)  // growing moves the arena
        if (int rc = drain_in_flight(p)) return rc;
    CUDA_TRY(p, p->d_rays.grow(want * 8, p->dev_used * 8, p->stream));
    CUDA_TRY(p, p->d_orig.grow(want, p->dev_used, p->stream));
    CUDA_TRY(p, p->d_pos.grow(want, p->dev_used, p->stream));
    return RSSYNC_OK;
}
int upload_arena_range(rssync_problem* p, size_t a, size_t b) {
    if (int rc = h2d(p, p->d_rays.ptr + a * 8, p->h_rays.ptr + a * 8, (b - a) * 8 * sizeof(double))) return rc;
    if (int rc = h2d(p, p->d_orig.ptr + a, p->h_orig.ptr + a, (b - a) * sizeof(int32_t))) return rc;
    if (int rc = h2d(p, p->d_pos.ptr + a, p->h_pos.ptr + a, (b - a) * sizeof(int32_t))) return rc;
    p->dev_used = std::max(p->dev_used, b);
    return RSSYNC_OK;
}
void add_pending(rssync_problem* p, size_t a, size_t b) {
    if (!p->pending.empty() && p->pending.back().second == a) p->pending.back().second = b;
    else p->pending.emplace_back(a, b);
}

// keep_in_flight: the caller (the PreSync grid) orders itself against the bulk-ingest chunks
int flush(rssync_problem* p, bool keep_in_flight = false) {
    DebugTimer tm("flush");
    CUDA_TRY(p, cudaSetDevice(p->device));
    join_gyro(p);
    tm.mark("join gyro");
    if (p->gyro_dirty) {  // the worker queued the copy and the finishing kernel on gyro_stream
        CUDA_TRY(p, p->gyro_copy_err);
        CUDA_TRY(p, cudaStreamWaitEvent(p->stream, p->ev_gyro, 0));
        if (!p->gyro_on_device) p->h2d += p->nq * 9 * sizeof(double);
        p->gyro_on_device = false;
        p->gyro_dirty = false;
    }
    // frames set one by one after a bulk ingest are newer than it: their upload follows it
    if (!keep_in_flight || !p->pending.empty())
        if (int rc = wait_in_flight(p)) return rc;
    if (!p->pending.empty()) {
        if (int rc = reserve_device_arena(p)) return rc;
        for (const auto& r : p->pending)
            if (int rc = upload_arena_range(p, r.first, r.second)) return rc;
        p->pending.clear();
    }
    return RSSYNC_OK;
}

// The start of a bulk ingest on the problem's stream (every form but the chunked rssync_set_track_batch):
// an earlier call's staging block is free again, and the ingest follows everything that writes the arena.
// Frames set one by one before this call are older than it: their upload goes first.
int begin_ingest(rssync_problem* p) {
    CUDA_TRY(p, cudaSetDevice(p->device));
    if (int rc = wait_arena_copies(p)) return rc;
    return p->pending.empty() ? wait_in_flight(p) : flush(p);
}

// frames with begin <= id < end_exclusive, ascending id
int select_frames(rssync_problem* p, int64_t begin, int64_t end_exclusive,
                  std::vector<FrameDesc>& out, int& max_n, const char* who) {
    out.clear();
    max_n = 0;
    for (auto it = p->frames.lower_bound(begin); it != p->frames.end() && it->first < end_exclusive; ++it) {
        const FrameDesc& fd = it->second;
        if (fd.n < 2) {
            p->err = std::string(who) + ": frame " + std::to_string(fd.id) + " has fewer than 2 rays";
            return RSSYNC_E_INVALID;
        }
        out.push_back(fd);
        max_n = std::max(max_n, (int)fd.n);
    }
    return RSSYNC_OK;
}

// ---- steps shared by the PreSync entry points ---------------------------------------------------
int check_search_window(rssync_problem* p, double initial, double step, double radius) {
    if (!(step > 0) || !std::isfinite(radius) || !std::isfinite(initial)) {
        p->err = "pre-sync: search_step must be > 0 and the search window finite";
        return RSSYNC_E_INVALID;
    }
    return RSSYNC_OK;
}

// the delay grid of a PreSync search (core_private.cpp:69-70)
int presync_delay_grid(rssync_problem* p, double initial, double step, double radius, std::vector<double>& delays) {
    if (int rc = check_search_window(p, initial, step, radius)) return rc;
    const int D = rssync_presync_delays(initial, step, radius, nullptr, 0);
    if (D <= 0 || D > (1 << 28)) { p->err = "pre-sync: empty or oversized delay grid"; return RSSYNC_E_INVALID; }
    delays.resize((size_t)D);
    rssync_presync_delays(initial, step, radius, delays.data(), D);
    return RSSYNC_OK;
}

// DESIGN §0: a grid holds at most 2^34 (frame, delay) tasks, so that every task index stays in range
int check_grid_size(rssync_problem* p, long long F, long long D) {
    if (F * D > (1LL << 34)) { p->err = "pre-sync: grid too large"; return RSSYNC_E_INVALID; }
    return RSSYNC_OK;
}

// A grid's inputs and scratch on the device: `n_frames` frame records (one table of F frames, or one per
// curve) in d_frames, the D delays in d_delays, the per-task costs, and `curves` loss curves with their
// flag words (zeroed) in d_costs / d_flags.  Without frames no grid runs and nothing is uploaded.
int stage_grid(rssync_problem* p, const FrameDesc* frames, size_t n_frames, int F, const double* delays, int D,
               int curves) {
    CUDA_TRY(p, p->d_frames.reserve(std::max<size_t>(n_frames, 1)));
    CUDA_TRY(p, p->d_delays.reserve((size_t)D));
    CUDA_TRY(p, p->d_framecost.reserve((size_t)std::max(F, 1) * D));
    CUDA_TRY(p, p->d_costs.reserve((size_t)curves * D));
    CUDA_TRY(p, p->d_flags.reserve((size_t)curves * 2));
    CUDA_TRY(p, cudaMemsetAsync(p->d_flags.ptr, 0, (size_t)curves * 2 * sizeof(unsigned), p->stream));
    if (F == 0) return RSSYNC_OK;
    if (int rc = h2d(p, p->d_frames.ptr, frames, sizeof(FrameDesc) * n_frames)) return rc;
    return h2d(p, p->d_delays.ptr, delays, sizeof(double) * D);
}

// max_chunk of a grid over these frames (rs::presync_max_chunk)
int grid_max_chunk(const FrameDesc* frames, int F, const double* delays, int D, double sr, int max_n) {
    double span = 0.0;
    for (int f = 0; f < F; ++f) span = std::max(span, frames[f].ts_hi - frames[f].ts_lo);
    return rs::presync_max_chunk(delays, D, span, sr, max_n);
}

// the RNG call numbers of n calls: the caller's, or the next n of the problem's counter (which the
// caller advances)
std::vector<uint64_t> call_numbers(const rssync_problem* p, const uint64_t* call_nos, int n) {
    std::vector<uint64_t> calls((size_t)n);
    for (int i = 0; i < n; ++i) calls[(size_t)i] = call_nos ? call_nos[i] : p->call_no + (uint64_t)i;
    return calls;
}

const char* presync_panic_text(unsigned fl) {  // core_private.cpp:76-83
    return (fl & rs::kFlagP)   ? "pre-sync: non-finite numbers in P"
           : (fl & rs::kFlagM) ? "pre-sync: non-finite numbers in M"
           : (fl & rs::kFlagR) ? "pre-sync: non-finite r"
                               : "pre-sync: non-finite rho";
}

// std::min_element over (cost, delay) pairs, core_private.cpp:89
void curve_argmin(const double* costs, const double* delays, int D, double* cost, double* delay) {
    int best = 0;
    for (int d = 1; d < D; ++d)
        if (costs[d] < costs[best] || (costs[d] == costs[best] && delays[d] < delays[best])) best = d;
    *cost = costs[best];
    *delay = delays[best];
}

// a failed device-side assertion of an RS_CHECKED build on the current device
int check_device_assert(rssync_problem* p) {
    if (const int line = rs::checked_assert_line()) {
        p->err = "device-side assertion failed at engine.cu:" + std::to_string(line);
        return RSSYNC_E_CUDA;
    }
    return RSSYNC_OK;
}

// the end of a call's work on `st`: launch errors, the wait, device-side assertions
int finish_stream(rssync_problem* p, cudaStream_t st) {
    CUDA_TRY(p, cudaGetLastError());
    CUDA_TRY(p, cudaStreamSynchronize(st));
    return check_device_assert(p);
}

// SetGyroQuaternions' spline build (ndspline::make, core_private.cpp:139 / :189) for the `count`
// samples already copied to the head of the pinned staging block: a worker thread eliminates the
// tridiagonal system (sequential, host_ingest.cpp), then queues the copy of samples + system and the
// kernel that finishes the records on gyro_stream.  The caller's thread goes on ingesting tracks.
int start_gyro_worker(rssync_problem* p, size_t count) {
    CUDA_TRY(p, p->d_rec.reserve(count * 16));
    CUDA_TRY(p, p->d_gyro.reserve(count * 9));
    if (!p->gyro_stream) CUDA_TRY(p, cudaStreamCreateWithFlags(&p->gyro_stream, cudaStreamNonBlocking));
    if (!p->ev_gyro) CUDA_TRY(p, cudaEventCreateWithFlags(&p->ev_gyro, cudaEventDisableTiming));
    double* h = p->h_gyro.ptr;
    double* d = p->d_gyro.ptr;
    double* d_rec = p->d_rec.ptr;
    p->gyro_worker = std::thread([=]() {
        rs::build_spline_system(h, count, h + 4 * count, h + 8 * count);
        cudaError_t e = cudaSetDevice(p->device);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d, h, count * 9 * sizeof(double), cudaMemcpyHostToDevice, p->gyro_stream);
        if (e == cudaSuccess) {
            rs::launch_spline_finish(d, d + 4 * count, d + 8 * count, (int)count, d_rec, p->gyro_stream);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaEventRecord(p->ev_gyro, p->gyro_stream);
        p->gyro_copy_err = e;
    });
    return RSSYNC_OK;
}

// the spline system's elimination factors for n knots on the device: d_elim = {f_down[n], f_up[n], diag[n]}
int upload_elimination(rssync_problem* p, size_t n, cudaStream_t st) {
    if (p->elim_n == n && p->d_elim.ptr) return RSSYNC_OK;
    const std::shared_ptr<const rs::SplineElimination> se = rs::spline_elimination(n);
    CUDA_TRY(p, cudaStreamSynchronize(st));  // (a reallocation must not pull the buffer from under a running kernel)
    CUDA_TRY(p, p->d_elim.reserve(3 * n));
    CUDA_TRY(p, cudaMemcpyAsync(p->d_elim.ptr, se->f_down.data(), n * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(p, cudaMemcpyAsync(p->d_elim.ptr + n, se->f_up.data(), n * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(p, cudaMemcpyAsync(p->d_elim.ptr + 2 * n, se->diag.data(), n * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(p, cudaStreamSynchronize(st));  // the host vectors may go away with the cache entry
    p->h2d += 3 * n * sizeof(double);
    p->elim_n = n;
    return RSSYNC_OK;
}

int require_gyro(rssync_problem* p, const char* who) {
    if (p->nq < 2) {
        p->err = std::string(who) + ": gyro quaternions have not been set";
        return RSSYNC_E_STATE;
    }
    return RSSYNC_OK;
}

int multi_presync_grid(rssync_problem* p, int64_t fb, int64_t fe, const double* delays, int n,
                       uint64_t stream_id, uint64_t call_no, uint64_t idx_base, double* costs,
                       unsigned* flags_out);
bool is_multi(const rssync_problem* p) { return !p->replicas.empty() && !p->force_single; }

void parallel_copy(void* dst, const void* src, size_t bytes);  // worker pool, below

int spare_sms_for_collectives() {
    static const int n = [] {
        const char* e = std::getenv("RSSYNC_SPARE_SMS");
        return e ? std::max(0, std::atoi(e)) : 0;  // measured on 2 and 8 GPUs: 8 spare SMs cost 3 % of the grid and gain nothing
    }();
    return n;
}

// The kernel launches of one PreSync grid over the frames `sel` (already in p->d_frames) and the n
// delays in p->d_delays, into p->d_framecost; the per-delay reduction is the caller's.
int enqueue_grid_kernels(rssync_problem* p, const std::vector<FrameDesc>& sel, int max_n, int n, uint64_t stream_id,
                         uint64_t call_no, uint64_t idx_base, unsigned* d_flags, int max_chunk, bool timed,
                         size_t* n_launches, int* n_waited) {
    const int F = (int)sel.size();
    // Frames still being uploaded by a bulk ingest: cut the frame list into runs by the ingest chunk
    // they wait for, and launch each run behind that chunk's event, so the grid works on the first
    // chunks while the last ones are on the bus.  (Frame costs do not depend on how frames are
    // grouped into launches.)  dep[f] = 1 + index of the last in-flight chunk overlapping frame f.
    std::vector<int> run_end, run_dep;
    if (!p->in_flight.empty()) {
        int cur = -1;
        for (int f = 0; f < F; ++f) {
            const size_t a = (size_t)sel[f].off, b = a + (size_t)(sel[f].n + 31) / 32 * 32;
            int dep = 0;
            for (size_t k = p->in_flight.size(); k-- > 0;)
                if (a < p->in_flight[k].hi && p->in_flight[k].lo < b) { dep = (int)k + 1; break; }
            dep = std::max(dep, cur < 0 ? 0 : run_dep.back());  // events complete in order: keep runs monotone
            if (dep != cur) {
                if (cur >= 0) run_end.push_back(f);
                run_dep.push_back(dep);
                cur = dep;
            }
        }
        run_end.push_back(F);
        if (run_end.size() > 16) { run_end.assign(1, F); run_dep.assign(1, (int)p->in_flight.size()); }
    } else {
        run_end.assign(1, F);
        run_dep.assign(1, 0);
    }
    const rs::DeviceData dd = p->device_data();
    if (timed) CUDA_TRY(p, cudaEventRecord(p->ev0, p->stream));
    int f0 = 0, waited = 0;
    if (run_end.size() == 1) {
        if (run_dep[0] > 0) {
            CUDA_TRY(p, cudaStreamWaitEvent(p->stream, p->in_flight[(size_t)run_dep[0] - 1].ev, 0));
            waited = run_dep[0];
        }
        rs::launch_presync_tasks(dd, p->d_frames.ptr, F, max_n, p->d_delays.ptr, n, p->seed, stream_id, call_no,
                                 idx_base, p->d_framecost.ptr, F, d_flags, p->stream, nullptr, max_chunk, p->simplified);
    } else {
        // The runs go round-robin to a few side streams: kernels of one stream run one after the
        // other, so a single stream would leave the tail of every run (its last blocks) unshared;
        // from neighbouring streams the next run's blocks move in as the previous run's retire.
        for (int k = 0; k < rssync_problem::kGridStreams; ++k) {
            if (!p->grid_stream[k]) CUDA_TRY(p, cudaStreamCreateWithFlags(&p->grid_stream[k], cudaStreamNonBlocking));
            if (!p->ev_grid[k]) CUDA_TRY(p, cudaEventCreateWithFlags(&p->ev_grid[k], cudaEventDisableTiming));
        }
        if (!p->ev_order) CUDA_TRY(p, cudaEventCreateWithFlags(&p->ev_order, cudaEventDisableTiming));
        CUDA_TRY(p, cudaEventRecord(p->ev_order, p->stream));  // frame table, delays, gyro records
        for (size_t r = 0; r < run_end.size(); ++r) {
            cudaStream_t gs = p->grid_stream[r % rssync_problem::kGridStreams];
            if (r < (size_t)rssync_problem::kGridStreams) CUDA_TRY(p, cudaStreamWaitEvent(gs, p->ev_order, 0));
            if (run_dep[r] > 0) {
                CUDA_TRY(p, cudaStreamWaitEvent(gs, p->in_flight[(size_t)run_dep[r] - 1].ev, 0));
                waited = std::max(waited, run_dep[r]);
            }
            // A run that is followed by chunks a collective still has to deliver can leave a few SMs
            // free (RSSYNC_SPARE_SMS; default 0): the grid's blocks are persistent and fill the device,
            // and the collective's kernel for the next chunks starts while this run is resident.
            // Measured (r02, 2 and 8 GPUs): the collectives are not held up in practice.
            int spare = 0;
            for (size_t k = (size_t)run_dep[r]; k < p->in_flight.size(); ++k)
                if (p->in_flight[k].foreign) spare = spare_sms_for_collectives();
            rs::launch_presync_tasks(dd, p->d_frames.ptr + f0, run_end[r] - f0, max_n, p->d_delays.ptr, n, p->seed,
                                     stream_id, call_no, idx_base, p->d_framecost.ptr + f0, F, d_flags, gs,
                                     nullptr, max_chunk, p->simplified, spare);
            f0 = run_end[r];
        }
        for (int k = 0; k < rssync_problem::kGridStreams; ++k) {
            CUDA_TRY(p, cudaEventRecord(p->ev_grid[k], p->grid_stream[k]));
            CUDA_TRY(p, cudaStreamWaitEvent(p->stream, p->ev_grid[k], 0));
        }
    }
    if (timed) CUDA_TRY(p, cudaEventRecord(p->ev1, p->stream));
    if (n_launches) *n_launches = run_end.size();
    if (n_waited) *n_waited = waited;
    // the chunks this call waited for are done with; later ones (frames outside this call) stay
    for (int k = 0; k < waited; ++k) p->ev_pool.push_back(p->in_flight[(size_t)k].ev);
    p->in_flight.erase(p->in_flight.begin(), p->in_flight.begin() + waited);
    return RSSYNC_OK;
}

// The opening of a grid over one frame range (presync_grid_impl, multi_presync_grid): the checks, the
// frame selection and the flush.  `sel` comes back empty when the call is complete: no delays, or no
// frames, where the reference sums over none (cost 0 for every delay).
int grid_prologue(rssync_problem* p, int64_t fb, int64_t fe, int n, double* costs, unsigned* flags_out,
                  std::vector<FrameDesc>& sel, int& max_n) {
    if (int rc = require_gyro(p, "pre-sync")) return rc;
    if (n < 0) { p->err = "pre-sync: negative delay count"; return RSSYNC_E_INVALID; }
    if (flags_out) *flags_out = 0;
    sel.clear();
    if (n == 0) return RSSYNC_OK;
    if (int rc = select_frames(p, fb, fe, sel, max_n, "pre-sync")) return rc;
    if (int rc = flush(p, /*keep_in_flight=*/true)) return rc;
    if (sel.empty()) std::fill(costs, costs + n, 0.0);
    return check_grid_size(p, (long long)sel.size(), n);
}

// the statistics of a finished grid over one frame range
void note_grid(rssync_problem* p, int F, int n, uint64_t exact_tasks) {
    p->grid_tasks = (uint64_t)F * (uint64_t)n;
    p->grid_exact_tasks = exact_tasks;
    if (p->kernel_timing) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, p->ev0, p->ev1) == cudaSuccess) p->last_grid_ms = ms;
    }
}

int presync_grid_impl(rssync_problem* p, int64_t fb, int64_t fe, const double* delays, int n,
                      uint64_t stream_id, uint64_t call_no, uint64_t idx_base, double* costs,
                      unsigned* flags_out) {
    if (is_multi(p)) return multi_presync_grid(p, fb, fe, delays, n, stream_id, call_no, idx_base, costs, flags_out);
    DebugTimer tm("presync_grid");
    std::vector<FrameDesc> sel;
    int max_n = 0;
    if (int rc = grid_prologue(p, fb, fe, n, costs, flags_out, sel, max_n)) return rc;
    if (sel.empty()) return RSSYNC_OK;
    tm.mark("checks and flush");
    const int F = (int)sel.size();
    const int max_chunk = grid_max_chunk(sel.data(), F, delays, n, p->sr, max_n);
    if (int rc = stage_grid(p, sel.data(), sel.size(), F, delays, n, 1)) return rc;
    size_t n_launches = 0;
    int waited = 0;
    if (int rc = enqueue_grid_kernels(p, sel, max_n, n, stream_id, call_no, idx_base, p->d_flags.ptr, max_chunk,
                                      p->kernel_timing, &n_launches, &waited))
        return rc;
    rs::launch_presync_reduce(p->d_framecost.ptr, F, n, p->d_costs.ptr, p->stream);
    if (tm.on) std::fprintf(stderr, "[presync_grid] %zu launch(es) behind %d in-flight chunk(s)\n", n_launches, waited);
    tm.mark("launch");
    unsigned flags[2] = {0, 0};
    if (int rc = d2h(p, costs, p->d_costs.ptr, sizeof(double) * n)) return rc;
    if (int rc = d2h(p, flags, p->d_flags.ptr, 2 * sizeof(unsigned))) return rc;
    if (int rc = finish_stream(p, p->stream)) return rc;
    tm.mark("wait for the device");
    note_grid(p, F, n, flags[1]);
    if (flags_out) *flags_out = flags[0];
    return RSSYNC_OK;
}

// ---- Sync: host control loop over a batch of syncpoints ---------------------------------------
// The outer loop of Sync (core_private.cpp:298-331) stays on the host: per iteration one launch
// sequence (L-BFGS of every frame + objective at x0, x0 -/+ h; the per-syncpoint sums, which also
// form Backtrack's trial points on the device; the trial losses; their sums) and one read-back.
// A frame whose L-BFGS runs to its 200-iteration cap takes ~0.3 ms of dependent scalar FP64 work on
// one warp against ~20 us for the typical frame, and every syncpoint needs all of its frames before
// it can step.  Syncpoints are independent of each other, so the batch is cut into LANES
// (contiguous groups of syncpoints), each with its own stream, scratch and pinned I/O blocks; one
// host thread drives all lanes as state machines and polls their events, so a lane waiting for a
// straggler does not hold up the others and their kernels overlap on the device.  The result of a
// syncpoint does not depend on the lane it runs in.
constexpr int kTrials = 10;  // Backtrack max_iterations, core_private.cpp:226

int sync_lane_count(int n) {
    static const int cfg = [] {
        const char* e = std::getenv("RSSYNC_SYNC_LANES");
        const int v = e ? std::atoi(e) : 0;
        return v > 0 ? v : 8;
    }();
    return std::max(1, std::min(n, cfg));
}

// stream-ordered setup of one lane: buffers, task upload, GuessMotion / GuessK (:218-223)
int sync_lane_begin(rssync_problem* p, SyncLane& L, const rs::DeviceData& dd, const std::vector<rs::SyncTask>& tasks,
                    const std::vector<int>& sp_begin, const std::vector<uint64_t>& callno, int max_n,
                    const double* initial, bool dbg) {
    const int n = L.n, T = L.T;
    if (!L.stream) CUDA_TRY(p, cudaStreamCreateWithFlags(&L.stream, cudaStreamNonBlocking));
    if (!L.ev) CUDA_TRY(p, cudaEventCreateWithFlags(&L.ev, cudaEventDisableTiming));
    CUDA_TRY(p, L.d_tasks.reserve(std::max(T, 1)));
    CUDA_TRY(p, L.d_sp_begin.reserve(n + 1));
    CUDA_TRY(p, L.d_m.reserve((size_t)std::max(T, 1) * 3));
    CUDA_TRY(p, L.d_k.reserve(std::max(T, 1)));
    CUDA_TRY(p, L.d_task_scratch.reserve((size_t)std::max(T, 1) * kTrials));
    CUDA_TRY(p, L.d_lbfgs_stats.reserve((size_t)std::max(T, 1) * 2));
    CUDA_TRY(p, L.d_sp_callno.reserve(n));
    CUDA_TRY(p, L.d_trial_delay.reserve((size_t)n * kTrials));
    // per-iteration traffic: one pinned block each way (one async copy in, one out)
    //   in : delay[n], x0[n] (doubles), active[n] (bytes); host block 0 serves the iterations (it
    //        is rewritten only after the previous iteration's event), block 1 the initialisation
    //   out: v[n], g[n], trial losses[n x kTrials] (doubles), objective evaluations so far (u64)
    L.in_doubles = 2 * (size_t)n + ((size_t)n + 7) / 8 + 1;  // + the number of trial points to evaluate
    L.out_doubles = (2 + (size_t)kTrials) * n + 1;
    CUDA_TRY(p, L.d_in.reserve(L.in_doubles));
    CUDA_TRY(p, L.h_in.reserve(2 * L.in_doubles));
    CUDA_TRY(p, L.d_out.reserve(L.out_doubles));
    CUDA_TRY(p, L.h_out.reserve(L.out_doubles));
    // everything queued on the problem's stream so far (gyro records, ray arena) precedes this lane
    CUDA_TRY(p, cudaStreamWaitEvent(L.stream, p->ev_sync_ready, 0));
    CUDA_TRY(p, cudaMemcpyAsync(L.d_tasks.ptr, tasks.data() + L.t0, sizeof(rs::SyncTask) * T, cudaMemcpyHostToDevice, L.stream));
    CUDA_TRY(p, cudaMemcpyAsync(L.d_sp_begin.ptr, sp_begin.data(), sizeof(int) * (n + 1), cudaMemcpyHostToDevice, L.stream));
    CUDA_TRY(p, cudaMemcpyAsync(L.d_sp_callno.ptr, callno.data() + L.s0, sizeof(uint64_t) * n, cudaMemcpyHostToDevice, L.stream));
    p->h2d += sizeof(rs::SyncTask) * T + sizeof(int) * (n + 1) + sizeof(uint64_t) * n;
    CUDA_TRY(p, cudaMemsetAsync(L.evals_dev(), 0, sizeof(unsigned long long), L.stream));
    L.b.tasks = L.d_tasks.ptr;
    L.b.T = T;
    L.b.max_n = max_n;
    L.b.sp_begin = L.d_sp_begin.ptr;
    L.b.S = n;
    L.b.m = L.d_m.ptr;
    L.b.k = L.d_k.ptr;
    L.b.simplified = p->simplified ? 1 : 0;
    L.st.assign(n, SyncPointState());
    L.iters = 0;
    L.phase = SyncLane::Running;
    if (dbg) L.h_stats.resize((size_t)std::max(T, 1) * 2);
    double* hd = L.h_in.ptr + L.in_doubles;  // host block 1: the iterations use block 0
    for (int s = 0; s < n; ++s) {
        L.st[s].delay = initial[L.s0 + s];
        hd[s] = L.st[s].delay;
        hd[n + s] = L.st[s].delay;
        reinterpret_cast<unsigned char*>(hd + 2 * n)[s] = 1;
    }
    L.n_eval = kTrials;
    hd[L.in_doubles - 1] = (double)kTrials;
    CUDA_TRY(p, cudaMemcpyAsync(L.d_in.ptr, hd, L.in_doubles * sizeof(double), cudaMemcpyHostToDevice, L.stream));
    p->h2d += L.in_doubles * sizeof(double);
    rs::launch_sync_init(dd, L.b, L.d_in.ptr, L.d_sp_callno.ptr, L.active_dev(), p->seed, L.stream);
    CUDA_TRY(p, cudaGetLastError());
    return RSSYNC_OK;
}

// the launch sequence of one outer iteration on the lane's stream (also what the graph captures)
int sync_lane_enqueue_iteration(rssync_problem* p, SyncLane& L, const rs::DeviceData& dd, bool dbg) {
    const int n = L.n;
    double* d_delay = L.d_in.ptr;
    double* d_x0 = d_delay + n;
    CUDA_TRY(p, cudaMemcpyAsync(L.d_in.ptr, L.h_in.ptr, L.in_doubles * sizeof(double), cudaMemcpyHostToDevice, L.stream));
    // do_opt_motion (:262-296) + f_and_grad at x0 (:228-240), then Backtrack::Step
    // (backtrack.cpp:3-13): all trial points x0 - t g are known once the gradient is, so the
    // device forms them and evaluates them in one launch; the host takes the first that passes.
    rs::launch_sync_motion_fgrad(dd, L.b, d_delay, d_x0, L.active_dev(), L.d_task_scratch.ptr, L.d_out.ptr,
                                 L.d_out.ptr + n, L.d_trial_delay.ptr, kTrials,
                                 dbg ? L.d_lbfgs_stats.ptr : nullptr, L.evals_dev(), L.many_tasks, L.stream);
    if (dbg)
        CUDA_TRY(p, cudaMemcpyAsync(L.h_stats.data(), L.d_lbfgs_stats.ptr, sizeof(int) * 2 * L.T, cudaMemcpyDeviceToHost, L.stream));
    rs::launch_sync_trials(dd, L.b, L.d_trial_delay.ptr, kTrials, L.active_dev(), L.d_task_scratch.ptr,
                           L.d_out.ptr + 2 * n, L.stream, L.d_in.ptr + L.in_doubles - 1);
    CUDA_TRY(p, cudaGetLastError());
    CUDA_TRY(p, cudaMemcpyAsync(L.h_out.ptr, L.d_out.ptr, L.out_doubles * sizeof(double), cudaMemcpyDeviceToHost, L.stream));
    return RSSYNC_OK;
}

// Backtrack got further than the trial points evaluated speculatively: evaluate all of them for the
// lane (same gradient, same trial delays -- they are still on the device) and read them back
int sync_lane_more_trials(rssync_problem* p, SyncLane& L, const rs::DeviceData& dd) {
    const int n = L.n;
    rs::launch_sync_trials(dd, L.b, L.d_trial_delay.ptr, kTrials, L.active_dev(), L.d_task_scratch.ptr,
                           L.d_out.ptr + 2 * n, L.stream);
    CUDA_TRY(p, cudaGetLastError());
    CUDA_TRY(p, cudaMemcpyAsync(L.h_out.ptr, L.d_out.ptr, L.out_doubles * sizeof(double), cudaMemcpyDeviceToHost, L.stream));
    CUDA_TRY(p, cudaEventRecord(L.ev, L.stream));
    p->d2h += L.out_doubles * sizeof(double);
    uint64_t tasks = 0;
    for (int s = 0; s < n; ++s)
        if (L.h_active[s]) tasks += (uint64_t)L.sp_frames[(size_t)s];
    p->sync_row_builds += tasks * (uint64_t)(kTrials - L.n_eval);  // (the kernel recomputes the first ones too;
    p->sync_loss_evals += tasks * (uint64_t)(kTrials - L.n_eval);  //  only the new ones are counted as work)
    L.n_eval = kTrials;
    L.phase = SyncLane::MoreTrials;
    return RSSYNC_OK;
}

// queue one outer iteration of the lane (or, when all its syncpoints are done, the final objective)
int sync_lane_launch(rssync_problem* p, SyncLane& L, const rs::DeviceData& dd, bool dbg) {
    static const bool use_graphs = std::getenv("RSSYNC_NO_GRAPHS") == nullptr;
    const int n = L.n;
    double* hd = L.h_in.ptr;
    unsigned char* ha = reinterpret_cast<unsigned char*>(hd + 2 * n);
    int n_active = 0;
    for (int s = 0; s < n; ++s) {
        ha[s] = L.st[s].done ? 0 : 1;
        n_active += ha[s];
        hd[s] = L.st[s].delay;
        hd[n + s] = L.st[s].delay - .3 * L.st[s].v;  // x0 = delay - delay_b * v, :299 (delay_b :260)
    }
    hd[L.in_doubles - 1] = (double)L.n_eval;
    L.h_active = ha;
    const bool finish = n_active == 0 || L.iters >= 400;  // :309
    if (!finish) {
        uint64_t tasks = 0;
        for (int s = 0; s < n; ++s)
            if (ha[s]) tasks += (uint64_t)L.sp_frames[(size_t)s];
        p->sync_row_builds += tasks * (uint64_t)((p->simplified ? 3 : 4) + L.n_eval);  // at the delay (L-BFGS), x0, x0 -/+ h, the trial points
        p->sync_loss_evals += tasks * (uint64_t)(3 + L.n_eval);
        p->sync_outer_total += (uint64_t)n_active;
    } else {
        p->sync_row_builds += (uint64_t)L.T;  // the final objective (:333)
        p->sync_loss_evals += (uint64_t)L.T;
    }
    if (finish) {
        // {simple_objective(gyro_delay), gyro_delay}  (:333)
        for (int s = 0; s < n; ++s) ha[s] = 1;
        CUDA_TRY(p, cudaMemcpyAsync(L.d_in.ptr, hd, L.in_doubles * sizeof(double), cudaMemcpyHostToDevice, L.stream));
        rs::launch_sync_trials(dd, L.b, L.d_in.ptr, 1, L.active_dev(), L.d_task_scratch.ptr, L.d_out.ptr + 2 * n, L.stream);
        CUDA_TRY(p, cudaGetLastError());
        CUDA_TRY(p, cudaMemcpyAsync(L.h_out.ptr, L.d_out.ptr, L.out_doubles * sizeof(double), cudaMemcpyDeviceToHost, L.stream));
        L.phase = SyncLane::Final;
    } else {
        L.iters++;
        // every argument the iteration's launches capture
        struct Key {
            rs::DeviceData dd;
            rs::SyncBatchDev b;
            const void* ptr[8];
            size_t in_doubles, out_doubles, many_tasks;
        } key;
        std::memset(&key, 0, sizeof(key));
        key.dd = dd;
        key.b = L.b;
        const void* ptrs[8] = {L.d_in.ptr, L.d_out.ptr, L.d_task_scratch.ptr, L.d_trial_delay.ptr,
                               L.h_in.ptr, L.h_out.ptr, L.stream, nullptr};
        std::memcpy(key.ptr, ptrs, sizeof(ptrs));
        key.in_doubles = L.in_doubles;
        key.out_doubles = L.out_doubles;
        key.many_tasks = L.many_tasks ? 1 : 0;
        const bool key_ok = L.graph_exec && L.graph_key.size() == sizeof(key) &&
                            std::memcmp(L.graph_key.data(), &key, sizeof(key)) == 0;
        if (!use_graphs || dbg || (!key_ok && L.iters == 1)) {
            // plain launches: debugging, and the first iteration of a new configuration (it also
            // performs the launchers' one-time attribute / occupancy calls outside any capture)
            if (int rc = sync_lane_enqueue_iteration(p, L, dd, dbg)) return rc;
        } else {
            if (!key_ok) {
                if (L.graph_exec) { cudaGraphExecDestroy(L.graph_exec); L.graph_exec = nullptr; }
                cudaGraph_t graph = nullptr;
                CUDA_TRY(p, cudaStreamBeginCapture(L.stream, cudaStreamCaptureModeThreadLocal));
                const int rc = sync_lane_enqueue_iteration(p, L, dd, false);
                const cudaError_t e = cudaStreamEndCapture(L.stream, &graph);
                rs::count_launches((uint64_t)-4);  // the launchers counted kernels that were only captured
                if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
                CUDA_TRY(p, e);
                const cudaError_t ei = cudaGraphInstantiate(&L.graph_exec, graph, 0);
                cudaGraphDestroy(graph);
                CUDA_TRY(p, ei);
                L.graph_key.assign(reinterpret_cast<unsigned char*>(&key), reinterpret_cast<unsigned char*>(&key) + sizeof(key));
            }
            CUDA_TRY(p, cudaGraphLaunch(L.graph_exec, L.stream));
            rs::count_launches(4);
        }
    }
    p->h2d += L.in_doubles * sizeof(double);
    p->d2h += L.out_doubles * sizeof(double);
    CUDA_TRY(p, cudaEventRecord(L.ev, L.stream));
    return RSSYNC_OK;
}

// host half of one outer iteration: Backtrack's acceptance test, momentum, stopping rules.
// Backtrack::Step (backtrack.cpp:3-13) takes the FIRST of the trial points t = 1e-3, 1e-4, ... that
// satisfies the Armijo condition.  All ten are known once the gradient is, so the device evaluates
// them without a host round trip -- but only the first n_eval of them: Backtrack stops at the same
// index iteration after iteration (the fourth on GoPro-shaped data: the gradient is ~1e3 1/s, so
// the first three steps overshoot by orders of magnitude), and every trial point costs a problem
// matrix per frame.  n_eval follows the index last accepted (+ 2); returns false when no evaluated
// point passed and points remain, in which case the caller has the rest evaluated and calls again.
bool sync_lane_step(rssync_problem* p, SyncLane& L, bool record_trace, bool dbg) {
    const int n = L.n;
    const double* h_v = L.h_out.ptr;
    const double* h_g = h_v + n;
    const double* h_trial_out = h_g + n;
    if (dbg) {
        int max_ev = 0, max_it = 0;
        for (int t = 0; t < L.T; ++t)
            if (L.h_active[L.local_sp[t]]) {
                max_ev = std::max(max_ev, L.h_stats[2 * t + 1]);
                max_it = std::max(max_it, L.h_stats[2 * t]);
            }
        std::fprintf(stderr, "sync lane %d it %d: L-BFGS max iters %d, max evals %d\n", L.s0, L.iters, max_it, max_ev);
    }
    const double delay_b = .3;  // :260
    if (L.n_eval < kTrials)  // does every syncpoint's Backtrack end inside what was evaluated?
        for (int s = 0; s < n; ++s) {
            if (L.st[s].done) continue;
            const double v = h_v[s], g = h_g[s], mm = g * g;
            double t = 1e-3;
            bool found = false;
            for (int i = 0; i < L.n_eval && !found; ++i) {
                found = v - h_trial_out[(size_t)s * kTrials + i] >= t * 2e-4 * mm;
                t *= .1;
            }
            if (!found) return false;
        }
    int furthest = 0;
    for (int s = 0; s < n; ++s) {
        SyncPointState& st = L.st[s];
        if (st.done) continue;
        const double v = h_v[s], g = h_g[s];
        const double mm = g * g;
        double t = 1e-3;
        int accepted = kTrials;
        for (int i = 0; i < L.n_eval; ++i) {
            const double v1 = h_trial_out[(size_t)s * kTrials + i];
            if (v - v1 >= t * 2e-4 * mm) { accepted = i; break; }
            t *= .1;
        }
        // (none passed among all ten: t has been multiplied ten times, backtrack.cpp:9-12 returns that step)
        p->sync_trial_hist[accepted]++;
        furthest = std::max(furthest, accepted);
        const double step = -t * g;
        st.v = delay_b * st.v + step;  // :301
        st.delay += st.v;              // :302
        const double step_size = std::fabs(step);
        if (record_trace && L.s0 + s == 0) {
            p->trace_delay.push_back(st.delay);
            p->trace_step.push_back(step_size);
        }
        if (step_size < 1e-4) st.converge++; else st.converge = 0;  // :316-320
        if (st.converge > 5) st.done = true;                        // :322
        if (std::fabs(st.delay - st.center) > st.radius) st.done = true;  // :326
    }
    static const bool all_trials = std::getenv("RSSYNC_ALL_TRIALS") != nullptr;
    L.n_eval = all_trials ? kTrials : std::min(kTrials, std::max(2, furthest + 2));
    return true;
}

int sync_batch_impl(rssync_problem* p, int n, const double* initial, const int64_t* fb,
                    const int64_t* fe, const double* center, const double* radius, double* out_cost,
                    double* out_delay, bool record_trace, const uint64_t* call_nos = nullptr) {
    if (int rc = require_gyro(p, "sync")) return rc;
    if (n <= 0) return RSSYNC_OK;
    // tasks: frames frame_begin <= f <= frame_end, INCLUSIVE (core_private.cpp:219)
    std::vector<rs::SyncTask> tasks;
    std::vector<int> sp_first(n + 1, 0);
    std::vector<int> sp_max_n(n, 0);
    std::vector<FrameDesc> sel;
    for (int s = 0; s < n; ++s) {
        if (fe[s] == INT64_MAX) { p->err = "sync: frame_end out of range"; return RSSYNC_E_INVALID; }
        if (int rc = select_frames(p, fb[s], fe[s] + 1, sel, sp_max_n[s], "sync")) return rc;
        for (const FrameDesc& fd : sel) tasks.push_back(rs::SyncTask{fd, s, 0});
        sp_first[s + 1] = (int)tasks.size();
    }
    if (int rc = flush(p)) return rc;
    const std::vector<uint64_t> callno = call_numbers(p, call_nos, n);
    if (!call_nos) p->call_no += (uint64_t)n;
    static const bool dbg = std::getenv("RSSYNC_DEBUG_SYNC") != nullptr;
    if (record_trace) { p->trace_delay.clear(); p->trace_step.clear(); }
    p->sync_outer = 0;
    p->sync_evals = 0;
    p->sync_row_builds = p->sync_loss_evals = p->sync_outer_total = 0;
    p->sync_init_tasks = p->simplified ? 0 : (uint64_t)tasks.size();
    p->sync_row_builds += (uint64_t)tasks.size();  // GuessMotion / GuessK build the rows once (:125-133 builds them twice)

    if (!p->ev_sync_ready) CUDA_TRY(p, cudaEventCreateWithFlags(&p->ev_sync_ready, cudaEventDisableTiming));
    CUDA_TRY(p, cudaEventRecord(p->ev_sync_ready, p->stream));
    const rs::DeviceData dd = p->device_data();
    const int G = sync_lane_count(n);
    if ((int)p->lanes.size() < G) p->lanes.resize(G);
    // A small batch is bound by the latency of its slowest frames, a large one by throughput: past
    // ~3 000 frame tasks (two waves of the large-block build on 148 SMs) the small-block build wins.
    // RSSYNC_LBFGS_BLOCKS=small|large overrides (tests run both).
    bool many_tasks = tasks.size() >= 3000;
    if (const char* e = std::getenv("RSSYNC_LBFGS_BLOCKS")) many_tasks = e[0] == 's';
    std::vector<std::vector<int>> lane_sp_begin(G);
    for (int g = 0; g < G; ++g) {
        SyncLane& L = p->lanes[g];
        L.many_tasks = many_tasks;
        L.s0 = (int)((long long)n * g / G);
        L.n = (int)((long long)n * (g + 1) / G) - L.s0;
        L.t0 = sp_first[L.s0];
        L.T = sp_first[L.s0 + L.n] - L.t0;
        int max_n = 0;
        lane_sp_begin[g].resize(L.n + 1);
        for (int s = 0; s <= L.n; ++s) lane_sp_begin[g][s] = sp_first[L.s0 + s] - L.t0;
        L.sp_frames.resize((size_t)L.n);
        for (int s = 0; s < L.n; ++s) L.sp_frames[(size_t)s] = sp_first[L.s0 + s + 1] - sp_first[L.s0 + s];
        for (int s = 0; s < L.n; ++s) max_n = std::max(max_n, sp_max_n[L.s0 + s]);
        L.local_sp.resize(L.T);
        for (int t = 0; t < L.T; ++t) {
            tasks[L.t0 + t].sp -= L.s0;  // syncpoint index inside the lane
            L.local_sp[t] = tasks[L.t0 + t].sp;
        }
        if (int rc = sync_lane_begin(p, L, dd, tasks, lane_sp_begin[g], callno, max_n, initial, dbg)) return rc;
        for (int s = 0; s < L.n; ++s) {
            L.st[s].center = center[L.s0 + s];
            L.st[s].radius = radius[L.s0 + s];
        }
        if (int rc = sync_lane_launch(p, L, dd, dbg)) return rc;
    }
    // drive the lanes: whichever has its iteration back on the host steps and is relaunched
    int running = G;
    while (running > 0) {
        bool progressed = false;
        for (int g = 0; g < G; ++g) {
            SyncLane& L = p->lanes[g];
            if (L.phase == SyncLane::Done) continue;
            const cudaError_t q = cudaEventQuery(L.ev);
            if (q == cudaErrorNotReady) continue;
            CUDA_TRY(p, q);
            progressed = true;
            if (L.phase == SyncLane::Final) {
                const double* h_cost = L.h_out.ptr + 2 * L.n;
                for (int s = 0; s < L.n; ++s) {
                    const bool empty = lane_sp_begin[g][s + 1] == lane_sp_begin[g][s];
                    out_cost[L.s0 + s] = empty ? 0.0 : h_cost[s];
                    out_delay[L.s0 + s] = L.st[s].delay;
                }
                p->sync_evals += (uint64_t)*reinterpret_cast<const unsigned long long*>(L.h_out.ptr + L.out_doubles - 1);
                p->sync_outer = std::max<uint64_t>(p->sync_outer, (uint64_t)L.iters);
                L.phase = SyncLane::Done;
                --running;
                continue;
            }
            if (!sync_lane_step(p, L, record_trace, dbg)) {
                if (int rc = sync_lane_more_trials(p, L, dd)) return rc;
                continue;
            }
            L.phase = SyncLane::Running;
            if (int rc = sync_lane_launch(p, L, dd, dbg)) return rc;
        }
        if (!progressed) std::this_thread::yield();
    }
    if (int rc = check_device_assert(p)) return rc;
    if (dbg) {
        std::fprintf(stderr, "sync: Backtrack trial accepted (cumulative):");
        for (int i = 0; i <= kTrials; ++i) std::fprintf(stderr, " %llu", (unsigned long long)p->sync_trial_hist[i]);
        std::fprintf(stderr, "\n");
    }
    return RSSYNC_OK;
}

// ---- several GPUs behind one problem ------------------------------------------------------------
// The path shards by independent units (SURVEY 8e): PreSync / DebugPreSync by offset range -- the
// RNG is keyed by the GLOBAL offset index, every frame's reduction stays on one device, so the
// sharded curve is bit-identical to one GPU's -- Sync and the windowed PreSync by syncpoint, the
// orientation search by variant.  Exchanges: one grouped ncclBroadcast of the finished device state
// whenever the inputs changed, and ONE ncclAllGather of the loss-curve slices per grid call, on
// device buffers.  Sync's per-syncpoint results are produced by the host-side control loop of each
// device's driver thread, i.e. they are born on the host: they are assembled there, no collective.
#define NCCL_TRY(p, expr)                                                                        \
    do {                                                                                         \
        int r__ = (expr);                                                                        \
        if (r__ != 0) {                                                                          \
            (p)->err = std::string("NCCL error: ") + rs::Nccl::get()->GetErrorString(r__) + " at " #expr; \
            return RSSYNC_E_CUDA;                                                                \
        }                                                                                        \
    } while (0)

struct DeviceGuard {  // restores the calling thread's current device
    int prev = 0;
    DeviceGuard() { cudaGetDevice(&prev); }
    ~DeviceGuard() { cudaSetDevice(prev); }
};
inline int n_ranks(const rssync_problem* p) { return 1 + (int)p->replicas.size(); }
inline rssync_problem* rank_problem(rssync_problem* p, int i) { return i == 0 ? p : p->replicas[(size_t)i - 1]; }

// bring every replica up to the primary's inputs
// The pieces a replication sends, covering the whole arena [0, rays): first whatever no chunk in
// flight covers (k_last = -1: it is on the device already -- an ingest that had to grow the arena
// waited for its first chunks, frames set one by one were uploaded by the flush), then the chunks in
// flight (stream order), consecutive ones together in at most `groups` pieces, each to be sent once
// its last chunk (k_last) has landed.  More than 16 pieces (scattered updates): one piece, sent last.
struct ReplicationPiece { int k_last; size_t lo, hi; };
std::vector<ReplicationPiece> plan_replication(const std::vector<std::pair<size_t, size_t>>& flying, size_t rays,
                                               size_t groups) {
    std::vector<ReplicationPiece> pieces;
    const size_t nfl = flying.size();
    {
        std::vector<std::pair<size_t, size_t>> busy = flying;
        std::sort(busy.begin(), busy.end());
        size_t at = 0;
        for (const auto& b : busy) {
            if (b.first > at) pieces.push_back(ReplicationPiece{-1, at, b.first});
            at = std::max(at, b.second);
        }
        if (rays > at) pieces.push_back(ReplicationPiece{-1, at, rays});
    }
    const size_t n_groups = std::min<size_t>(nfl, groups);
    for (size_t g = 0; g < n_groups; ++g) {
        const size_t a = nfl * g / n_groups, b = nfl * (g + 1) / n_groups;
        ReplicationPiece pc{(int)b - 1, flying[a].first, flying[a].second};
        for (size_t k = a; k < b; ++k) {
            pc.lo = std::min(pc.lo, flying[k].first);
            pc.hi = std::max(pc.hi, flying[k].second);
        }
        if (pc.lo < pc.hi) pieces.push_back(pc);
    }
    if (pieces.size() > 16) pieces.assign(1, ReplicationPiece{(int)nfl - 1, 0, rays});
    return pieces;
}

int multi_replicate(rssync_problem* p) {
    RS_NVTX_RANGE();
    bool stale = false;
    for (const rssync_problem* r : p->replicas) stale = stale || r->synced_version != p->version;
    if (!stale) return RSSYNC_OK;
    // Device 0 holds everything.  A bulk SetTrackResult may still be on its way there, chunk by chunk:
    // the chunks are sent on in a few pieces, each as soon as it has landed, on streams of their own,
    // and every replica is told which arena ranges are still coming (rssync_expect_chunk) -- its grid
    // then starts on the first frames while the last are on the bus, as the primary's does.
    if (int rc = flush(p, /*keep_in_flight=*/true)) return rc;
    const rs::Nccl* nc = rs::Nccl::get();
    DeviceGuard guard;
    const size_t rays = p->dev_used;
    std::vector<std::pair<size_t, size_t>> flying;
    for (const auto& f : p->in_flight) flying.emplace_back(f.lo, f.hi);
    const std::vector<ReplicationPiece> pieces = plan_replication(flying, rays, 4);
    using Piece = ReplicationPiece;
    for (rssync_problem* r : p->replicas) {
        cudaSetDevice(r->device);
        r->frames = p->frames;
        r->q0 = p->q0; r->sr = p->sr; r->nq = p->nq;
        r->used = p->used; r->dev_used = p->dev_used; r->total_rays = p->total_rays; r->garbage = p->garbage;
        r->seed = p->seed;
        r->simplified = p->simplified;
        cudaError_t e = cudaStreamSynchronize(r->stream);  // nothing of an earlier call still reads the buffers
        if (e == cudaSuccess && r->repl_stream) e = cudaStreamSynchronize(r->repl_stream);
        for (const auto& f : r->in_flight) r->ev_pool.push_back(f.ev);
        r->in_flight.clear();
        if (e == cudaSuccess) e = r->d_rays.reserve(std::max<size_t>(rays, 1) * 8);
        if (e == cudaSuccess) e = r->d_orig.reserve(std::max<size_t>(rays, 1));
        if (e == cudaSuccess) e = r->d_pos.reserve(std::max<size_t>(rays, 1));
        if (e == cudaSuccess) e = r->d_rec.reserve(std::max<size_t>(p->nq, 1) * 16);
        if (e != cudaSuccess) {
            p->err = std::string("CUDA error on device ") + std::to_string(r->device) + ": " + cudaGetErrorString(e);
            return RSSYNC_E_CUDA;
        }
    }
    for (int i = 0; i < n_ranks(p); ++i) {
        rssync_problem* q = rank_problem(p, i);
        cudaSetDevice(q->device);
        if (!q->repl_stream) CUDA_TRY(p, cudaStreamCreateWithFlags(&q->repl_stream, cudaStreamNonBlocking));
    }
    // the primary's sending stream follows what its own stream holds (spline records, frames set one by one)
    if (int rc = rssync_stream_wait_chunk(p, -1, p->repl_stream)) return rc;
    auto broadcast = [&](const Piece* pc) -> int {  // pc == nullptr: the spline records
        NCCL_TRY(p, nc->GroupStart());
        for (int i = 0; i < n_ranks(p); ++i) {
            rssync_problem* q = rank_problem(p, i);
            cudaSetDevice(q->device);
            void* comm = p->comms[(size_t)i];
            if (!pc) {
                NCCL_TRY(p, nc->Broadcast(q->d_rec.ptr, q->d_rec.ptr, p->nq * 16 * sizeof(double), rs::Nccl::kChar, 0, comm, q->repl_stream));
                continue;
            }
            const size_t lo = pc->lo, n = pc->hi - pc->lo;
            NCCL_TRY(p, nc->Broadcast(q->d_rays.ptr + lo * 8, q->d_rays.ptr + lo * 8, n * 8 * sizeof(double), rs::Nccl::kChar, 0, comm, q->repl_stream));
            NCCL_TRY(p, nc->Broadcast(q->d_orig.ptr + lo, q->d_orig.ptr + lo, n * sizeof(int32_t), rs::Nccl::kChar, 0, comm, q->repl_stream));
            NCCL_TRY(p, nc->Broadcast(q->d_pos.ptr + lo, q->d_pos.ptr + lo, n * sizeof(int32_t), rs::Nccl::kChar, 0, comm, q->repl_stream));
        }
        NCCL_TRY(p, nc->GroupEnd());
        p->nccl_calls += 1;
        for (rssync_problem* r : p->replicas)
            if (int rc = rssync_expect_chunk(r, pc ? pc->lo : 0, pc ? pc->hi : rays, r->repl_stream)) {
                p->err = r->err;
                return rc;
            }
        return RSSYNC_OK;
    };
    if (p->nq)
        if (int rc = broadcast(nullptr)) return rc;  // every frame waits at least for the records
    for (const Piece& pc : pieces) {
        if (pc.k_last >= 0)
            if (int rc = rssync_stream_wait_chunk(p, pc.k_last, p->repl_stream)) return rc;
        if (int rc = broadcast(&pc)) return rc;
    }
    if (int rc = rssync_note_reader(p, p->repl_stream)) return rc;  // the next Set* call waits for these sends
    for (rssync_problem* r : p->replicas) r->synced_version = p->version;
    p->broadcast_bytes += p->nq * 16 * sizeof(double);
    for (const Piece& pc : pieces) p->broadcast_bytes += (pc.hi - pc.lo) * (8 * sizeof(double) + 2 * sizeof(int32_t));
    return RSSYNC_OK;
}

// one rank's share of a grid: kernel + per-delay reduction into d_costs_dst (device), flags into
// d_flags_dst (2 words, device); nothing is copied back and nothing is waited for
int grid_enqueue_rank(rssync_problem* q, const std::vector<FrameDesc>& sel, int max_n, const double* delays,
                      int cnt, uint64_t stream_id, uint64_t call_no, uint64_t idx_base, int max_chunk,
                      double* d_costs_dst, unsigned* d_flags_dst, bool timed) {
    const int F = (int)sel.size();
    CUDA_TRY(q, cudaMemsetAsync(d_flags_dst, 0, 2 * sizeof(unsigned), q->stream));
    if (cnt <= 0) return RSSYNC_OK;
    CUDA_TRY(q, q->d_frames.reserve(F));
    CUDA_TRY(q, q->d_delays.reserve(cnt));
    CUDA_TRY(q, q->d_framecost.reserve((size_t)F * cnt));
    if (int rc = h2d(q, q->d_frames.ptr, sel.data(), sizeof(FrameDesc) * F)) return rc;
    if (int rc = h2d(q, q->d_delays.ptr, delays, sizeof(double) * cnt)) return rc;
    if (int rc = enqueue_grid_kernels(q, sel, max_n, cnt, stream_id, call_no, idx_base, d_flags_dst, max_chunk, timed,
                                      nullptr, nullptr))
        return rc;
    rs::launch_presync_reduce(q->d_framecost.ptr, F, cnt, d_costs_dst, q->stream);
    CUDA_TRY(q, cudaGetLastError());
    return RSSYNC_OK;
}

int multi_presync_grid(rssync_problem* p, int64_t fb, int64_t fe, const double* delays, int n,
                       uint64_t stream_id, uint64_t call_no, uint64_t idx_base, double* costs,
                       unsigned* flags_out) {
    std::vector<FrameDesc> sel;
    int max_n = 0;
    if (int rc = grid_prologue(p, fb, fe, n, costs, flags_out, sel, max_n)) return rc;
    if (sel.empty()) return RSSYNC_OK;
    const int F = (int)sel.size();
    if (int rc = multi_replicate(p)) return rc;
    static const bool dbg_sync = std::getenv("RSSYNC_DEBUG_MULTI") != nullptr;
    auto dbg_check = [&](const char* what) {
        if (!dbg_sync) return;
        for (int i = 0; i < n_ranks(p); ++i) {
            cudaSetDevice(rank_problem(p, i)->device);
            const cudaError_t e = cudaDeviceSynchronize();
            std::fprintf(stderr, "[multi] %s: device %d: %s (in flight %zu)\n", what, rank_problem(p, i)->device,
                         cudaGetErrorString(e), rank_problem(p, i)->in_flight.size());
        }
    };
    dbg_check("after replicate");
    const int max_chunk = grid_max_chunk(sel.data(), F, delays, n, p->sr, max_n);
    const rs::Nccl* nc = rs::Nccl::get();
    const int G = n_ranks(p);
    const int per = (n + G - 1) / G;  // delays per rank (the last ranks may hold fewer, or none)
    const size_t slice = (size_t)per * sizeof(double) + 2 * sizeof(unsigned);
    DeviceGuard guard;
    for (int i = 0; i < G; ++i) {
        rssync_problem* q = rank_problem(p, i);
        cudaSetDevice(q->device);
        const cudaError_t e = q->d_gather.reserve(slice * G);
        if (e != cudaSuccess) { p->err = std::string("CUDA error: ") + cudaGetErrorString(e); return RSSYNC_E_CUDA; }
        const int lo = std::min(n, i * per), cnt = std::min(per, n - lo);
        unsigned char* mine = q->d_gather.ptr + slice * i;
        const int rc = grid_enqueue_rank(q, sel, max_n, delays + lo, cnt, stream_id, call_no, idx_base + (uint64_t)lo,
                                         max_chunk, reinterpret_cast<double*>(mine),
                                         reinterpret_cast<unsigned*>(mine + (size_t)per * sizeof(double)),
                                         i == 0 && p->kernel_timing);
        if (rc) { if (q != p) p->err = q->err; return rc; }
        dbg_check("after a rank's grid");
    }
    // the one exchange of the call: every rank's slice {costs, flags} to every rank, in place
    NCCL_TRY(p, nc->GroupStart());
    for (int i = 0; i < G; ++i) {
        rssync_problem* q = rank_problem(p, i);
        cudaSetDevice(q->device);
        NCCL_TRY(p, nc->AllGather(q->d_gather.ptr + slice * i, q->d_gather.ptr, slice, rs::Nccl::kChar, p->comms[(size_t)i], q->stream));
    }
    NCCL_TRY(p, nc->GroupEnd());
    p->nccl_calls += 1;
    cudaSetDevice(p->device);
    CUDA_TRY(p, p->h_gather.reserve(slice * G));
    if (int rc = d2h(p, p->h_gather.ptr, p->d_gather.ptr, slice * G)) return rc;
    CUDA_TRY(p, cudaStreamSynchronize(p->stream));
    // the gather waited for every rank's grid; the primary's device is checked last and stays current
    for (int i = G; i-- > 0;) {
        cudaSetDevice(rank_problem(p, i)->device);
        if (int rc = check_device_assert(p)) return rc;
    }
    unsigned flags = 0;
    uint64_t exact = 0;
    for (int i = 0; i < G; ++i) {
        const int lo = std::min(n, i * per), cnt = std::min(per, n - lo);
        const unsigned char* sl = p->h_gather.ptr + slice * i;
        if (cnt > 0) std::memcpy(costs + lo, sl, sizeof(double) * (size_t)cnt);
        unsigned fl[2];
        std::memcpy(fl, sl + (size_t)per * sizeof(double), sizeof(fl));
        flags |= fl[0];
        exact += fl[1];
    }
    note_grid(p, F, n, exact);
    if (flags_out) *flags_out = flags;
    return RSSYNC_OK;
}

// run fn(rank, problem, lo, cnt) for every rank's contiguous share of n units, the primary's in the
// calling thread and each replica's in a thread of its own (the Sync driver is a host-side loop per
// device); primary_last: the primary takes the LAST share instead of the first
int multi_for_each_shard(rssync_problem* p, int n, bool primary_last,
                         const std::function<int(rssync_problem*, int, int)>& fn) {
    const int G = n_ranks(p);
    std::vector<int> rcs((size_t)G, RSSYNC_OK);
    std::vector<std::thread> th;
    auto share = [&](int i, int& lo, int& cnt) {
        const int k = primary_last ? (i == 0 ? G - 1 : i - 1) : i;  // position of rank i's share
        lo = (int)((long long)n * k / G);
        cnt = (int)((long long)n * (k + 1) / G) - lo;
    };
    for (int i = 1; i < G; ++i) {
        int lo, cnt;
        share(i, lo, cnt);
        if (cnt == 0) continue;
        rssync_problem* q = rank_problem(p, i);
        th.emplace_back([&, q, i, lo, cnt]() {
            cudaSetDevice(q->device);
            rcs[(size_t)i] = fn(q, lo, cnt);
        });
    }
    int lo, cnt;
    share(0, lo, cnt);
    p->force_single = true;
    if (cnt) rcs[0] = fn(p, lo, cnt);
    p->force_single = false;
    for (auto& t : th) t.join();
    for (int i = 0; i < G; ++i)
        if (rcs[(size_t)i]) {
            if (i) p->err = rank_problem(p, i)->err;
            return rcs[(size_t)i];
        }
    return RSSYNC_OK;
}

int multi_sync_batch(rssync_problem* p, int n, const double* initial, const int64_t* fb, const int64_t* fe,
                     const double* center, const double* radius, double* out_cost, double* out_delay,
                     const uint64_t* call_nos) {
    if (int rc = require_gyro(p, "sync")) return rc;
    if (int rc = multi_replicate(p)) return rc;
    const std::vector<uint64_t> callno = call_numbers(p, call_nos, n);
    if (!call_nos) p->call_no += (uint64_t)n;
    for (int i = 0; i < n_ranks(p); ++i) {
        rssync_problem* q = rank_problem(p, i);
        q->sync_outer = q->sync_evals = q->sync_row_builds = q->sync_loss_evals = q->sync_init_tasks = q->sync_outer_total = 0;
    }
    const int rc = multi_for_each_shard(p, n, false, [&](rssync_problem* q, int lo, int cnt) {
        return sync_batch_impl(q, cnt, initial + lo, fb + lo, fe + lo, center + lo, radius + lo, out_cost + lo,
                               out_delay + lo, false, callno.data() + lo);
    });
    uint64_t outer = 0, evals = 0, acc[4] = {0, 0, 0, 0};
    for (int i = 0; i < n_ranks(p); ++i) {
        const rssync_problem* q = rank_problem(p, i);
        outer = std::max(outer, q->sync_outer);
        evals += q->sync_evals;
        acc[0] += q->sync_row_builds; acc[1] += q->sync_loss_evals; acc[2] += q->sync_init_tasks; acc[3] += q->sync_outer_total;
    }
    p->sync_outer = outer;
    p->sync_evals = evals;
    p->sync_row_builds = acc[0]; p->sync_loss_evals = acc[1]; p->sync_init_tasks = acc[2]; p->sync_outer_total = acc[3];
    return rc;
}

}  // namespace

// =============================================================================================
extern "C" {

int rssync_create(rssync_problem** out) {
    if (!out) return RSSYNC_E_INVALID;
    *out = nullptr;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return RSSYNC_E_CUDA;
    int cc_major = 0;
    if (cudaDeviceGetAttribute(&cc_major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess)
        return RSSYNC_E_CUDA;
    rssync_problem* p = new rssync_problem();
    p->device = dev;
    *out = p;
    rs::checked_assert_line();  // (arms the device-side assertions of an RS_CHECKED build)
    if (cc_major < 10) {
        p->err = "rssync_b200 needs an sm_100a (Blackwell B200) device; there is no CPU or other-GPU fallback";
        return RSSYNC_E_CUDA;
    }
    return RSSYNC_OK;
}

int rssync_create_multi(const int* devices, int n_devices, rssync_problem** out) {
    if (!out) return RSSYNC_E_INVALID;
    *out = nullptr;
    if (!devices || n_devices < 1) return RSSYNC_E_INVALID;
    for (int i = 0; i < n_devices; ++i)
        for (int j = 0; j < i; ++j)
            if (devices[i] == devices[j]) return RSSYNC_E_INVALID;
    if (cudaSetDevice(devices[0]) != cudaSuccess) return RSSYNC_E_CUDA;
    int rc = rssync_create(out);
    rssync_problem* p = *out;
    if (rc != RSSYNC_OK || n_devices == 1) return rc;
    const rs::Nccl* nc = rs::Nccl::get();
    if (!nc) {
        p->err = "rssync_create_multi: libnccl.so.2 could not be loaded (needed for more than one device)";
        return RSSYNC_E_CUDA;
    }
    for (int i = 1; i < n_devices; ++i) {
        rssync_problem* r = nullptr;
        if (cudaSetDevice(devices[i]) != cudaSuccess) rc = RSSYNC_E_CUDA;
        if (rc == RSSYNC_OK) rc = rssync_create(&r);
        if (rc == RSSYNC_OK && cudaStreamCreateWithFlags(&r->stream, cudaStreamNonBlocking) != cudaSuccess) rc = RSSYNC_E_CUDA;
        if (rc != RSSYNC_OK) {
            p->err = r && !r->err.empty() ? r->err : std::string("rssync_create_multi: device ") + std::to_string(devices[i]) + " is not usable";
            if (r) rssync_destroy(r);
            cudaSetDevice(devices[0]);
            return rc;
        }
        r->is_replica = true;
        r->owns_stream = true;
        r->synced_version = ~0ull;
        r->rowq_synced = ~0ull;
        p->replicas.push_back(r);
    }
    p->comms.assign((size_t)n_devices, nullptr);
    const int nr = nc->CommInitAll(p->comms.data(), n_devices, devices);
    cudaSetDevice(devices[0]);
    if (nr != 0) {
        p->err = std::string("NCCL error: ") + nc->GetErrorString(nr) + " at ncclCommInitAll";
        p->comms.clear();
        return RSSYNC_E_CUDA;
    }
    return RSSYNC_OK;
}

int rssync_device_count(const rssync_problem* p) { return p ? 1 + (int)p->replicas.size() : 0; }

void rssync_destroy(rssync_problem* p) {
    if (!p) return;
    if (!p->replicas.empty() || !p->comms.empty()) {
        int prev = 0;
        cudaGetDevice(&prev);
        const rs::Nccl* nc = rs::Nccl::get();
        for (size_t i = 0; i <= p->replicas.size(); ++i) {  // no collective still queued when the communicators go
            rssync_problem* q = i == 0 ? p : p->replicas[i - 1];
            cudaSetDevice(q->device);
            if (q->repl_stream) cudaStreamSynchronize(q->repl_stream);
            cudaStreamSynchronize(q->stream);
        }
        for (size_t i = 0; i < p->comms.size(); ++i)
            if (nc && p->comms[i]) {
                cudaSetDevice(i == 0 ? p->device : p->replicas[i - 1]->device);
                nc->CommDestroy(p->comms[i]);
            }
        for (rssync_problem* r : p->replicas) rssync_destroy(r);
        p->replicas.clear();
        p->comms.clear();
        cudaSetDevice(prev);
    }
    cudaSetDevice(p->device);
    join_gyro(p);
    if (p->arena_copy_pending) cudaEventSynchronize(p->ev_arena);
    if (p->ev_arena) cudaEventDestroy(p->ev_arena);
    if (p->ev_reader) cudaEventDestroy(p->ev_reader);
    if (p->copy_stream) { cudaStreamSynchronize(p->copy_stream); cudaStreamDestroy(p->copy_stream); }
    if (p->repl_stream) { cudaStreamSynchronize(p->repl_stream); cudaStreamDestroy(p->repl_stream); }
    for (const auto& fl : p->in_flight) cudaEventDestroy(fl.ev);
    for (cudaEvent_t e : p->ev_pool) cudaEventDestroy(e);
    if (p->ev_order) cudaEventDestroy(p->ev_order);
    for (int k = 0; k < rssync_problem::kGridStreams; ++k) {
        if (p->grid_stream[k]) cudaStreamDestroy(p->grid_stream[k]);
        if (p->ev_grid[k]) cudaEventDestroy(p->ev_grid[k]);
    }
    if (p->gyro_stream) { cudaStreamSynchronize(p->gyro_stream); cudaStreamDestroy(p->gyro_stream); }
    if (p->ev_gyro) cudaEventDestroy(p->ev_gyro);
    p->d_rec.release();
    p->h_gyro.release();
    p->d_gyro.release();
    p->h_rays.release(); p->d_rays.release();
    p->h_orig.release(); p->d_orig.release();
    p->h_pos.release(); p->d_pos.release();
    p->d_frames.release(); p->d_delays.release(); p->d_framecost.release(); p->d_costs.release();
    p->d_frame_call.release(); p->d_win_begin.release();
    p->d_pixframes.release(); p->d_stage.release();
    p->d_flags.release(); p->h_stage.release(); p->d_probe.release();
    p->d_gather.release(); p->h_gather.release();
    p->d_var_ts.release(); p->d_var_in.release(); p->d_var_q.release(); p->d_var_y.release(); p->d_var_rhs.release();
    p->d_var_rec.release(); p->d_var_prefix.release(); p->d_elim.release();
    p->d_var_orients.release(); p->d_var_flags.release();
    p->d_rowq.release(); p->d_rt_rays.release(); p->d_rt_ext.release(); p->d_rt_orig.release(); p->d_rt_pos.release();
    p->d_trk_pyr.release(); p->d_trk_pts.release(); p->d_trk_at.release(); p->d_trk_status.release();
    p->d_trk_flag.release(); p->h_trk_flag.release();
    p->d_trk_keys.release(); p->d_trk_picks.release(); p->d_trk_count.release(); p->h_trk_qat.release();
    if (p->owns_stream && p->stream) { cudaStreamSynchronize(p->stream); cudaStreamDestroy(p->stream); }
    for (SyncLane& L : p->lanes) L.release();
    if (p->ev_sync_ready) cudaEventDestroy(p->ev_sync_ready);
    if (p->ev0) cudaEventDestroy(p->ev0);
    if (p->ev1) cudaEventDestroy(p->ev1);
    delete p;
}

const char* rssync_last_error(const rssync_problem* p) { return p ? p->err.c_str() : "null problem"; }

int rssync_set_gyro_fixed(rssync_problem* p, const double* quats, size_t count, double sample_rate,
                          double first_timestamp) {
    RS_NVTX_RANGE();
    if (!p || !quats) return RSSYNC_E_INVALID;
    if (count < 2) { p->err = "set-gyro-quaternions: need at least 2 samples"; return RSSYNC_E_INVALID; }
    if (count > (size_t)INT32_MAX) { p->err = "set-gyro-quaternions: too many samples"; return RSSYNC_E_INVALID; }
    join_gyro(p);
    p->version++;
    p->sr = sample_rate;       // core_private.cpp:137
    p->q0 = first_timestamp;   // :138
    cudaSetDevice(p->device);
    if (int rc = wait_reader(p)) return rc;
    if (p->gyro_dirty == false && p->nq) CUDA_TRY(p, cudaStreamSynchronize(p->stream));  // records in flight
    if (p->gyro_stream) CUDA_TRY(p, cudaStreamSynchronize(p->gyro_stream));  // a copy never waited for
    CUDA_TRY(p, p->h_gyro.reserve(count * 9));
    parallel_copy(p->h_gyro.ptr, quats, 4 * count * sizeof(double));  // the caller's buffer is only borrowed
    p->nq = count;
    p->gyro_dirty = true;
    p->gyro_on_device = false;
    return start_gyro_worker(p, count);  // :139
}

int rssync_set_gyro_var(rssync_problem* p, const int64_t* ts, const double* quats, size_t count) {
    RS_NVTX_RANGE();
    if (!p || !ts || !quats) return RSSYNC_E_INVALID;
    rs::ResamplePlan plan;
    const rs::IngestStatus s = rs::plan_variable_rate(ts, count, plan, p->err);  // core_private.cpp:146-164
    if (s == rs::IngestStatus::Invalid) return RSSYNC_E_INVALID;
    if (s == rs::IngestStatus::NonFinite) return RSSYNC_E_NONFINITE;
    if (s == rs::IngestStatus::OutOfOrder) return RSSYNC_E_ORDER;
    if (count > (size_t)INT32_MAX) { p->err = "set-gyro-quaternions: too many samples"; return RSSYNC_E_INVALID; }
    join_gyro(p);
    cudaSetDevice(p->device);
    if (int rc = wait_reader(p)) return rc;
    if (p->gyro_dirty == false && p->nq) CUDA_TRY(p, cudaStreamSynchronize(p->stream));
    if (!p->gyro_stream) CUDA_TRY(p, cudaStreamCreateWithFlags(&p->gyro_stream, cudaStreamNonBlocking));
    if (!p->ev_gyro) CUDA_TRY(p, cudaEventCreateWithFlags(&p->ev_gyro, cudaEventDisableTiming));
    CUDA_TRY(p, cudaStreamSynchronize(p->gyro_stream));
    // The per-sample half (:166-182: lower_bound + slerp), the elimination sweeps of the spline system
    // and the record build all run on the device, on the gyro stream; the call waits only for the
    // resampling's non-finite flag, which the reference reports here (:180-181).
    const size_t nq = plan.n_out;
    cudaStream_t gs = p->gyro_stream;
    CUDA_TRY(p, p->d_var_ts.reserve(count));
    CUDA_TRY(p, p->d_var_in.reserve(count * 4));
    CUDA_TRY(p, p->d_gyro.reserve(nq * 9));
    CUDA_TRY(p, p->d_var_flags.reserve(1));
    CUDA_TRY(p, cudaMemcpyAsync(p->d_var_ts.ptr, ts, count * sizeof(int64_t), cudaMemcpyHostToDevice, gs));
    CUDA_TRY(p, cudaMemcpyAsync(p->d_var_in.ptr, quats, count * 4 * sizeof(double), cudaMemcpyHostToDevice, gs));
    CUDA_TRY(p, cudaMemsetAsync(p->d_var_flags.ptr, 0, sizeof(unsigned), gs));
    rs::launch_gyro_resample(p->d_var_ts.ptr, (int)count, p->d_var_in.ptr, 1, plan.tick0, plan.rate_hz, (int)nq,
                             p->d_gyro.ptr, p->d_var_flags.ptr, gs);
    unsigned bad = 0;
    CUDA_TRY(p, cudaMemcpyAsync(&bad, p->d_var_flags.ptr, sizeof(unsigned), cudaMemcpyDeviceToHost, gs));
    if (int rc = upload_elimination(p, nq, gs)) return rc;
    CUDA_TRY(p, cudaMemcpyAsync(p->d_gyro.ptr + 8 * nq, p->d_elim.ptr + 2 * nq, nq * sizeof(double), cudaMemcpyDeviceToDevice, gs));
    CUDA_TRY(p, cudaStreamSynchronize(gs));
    p->h2d += count * (sizeof(int64_t) + 4 * sizeof(double));
    if (bad) { p->err = "set-gyro-quaternions: non-finite sample after interpolation"; return RSSYNC_E_NONFINITE; }
    p->version++;
    p->sr = plan.sample_rate;        // :183
    p->q0 = plan.first_timestamp;    // :184
    p->nq = nq;
    CUDA_TRY(p, p->d_rec.reserve(nq * 16));
    rs::launch_spline_chains(p->d_gyro.ptr, p->d_elim.ptr, p->d_elim.ptr + nq, (int)nq, 1, p->d_gyro.ptr + 4 * nq, gs);
    rs::launch_spline_finish(p->d_gyro.ptr, p->d_gyro.ptr + 4 * nq, p->d_gyro.ptr + 8 * nq, (int)nq, p->d_rec.ptr, gs);  // :189
    CUDA_TRY(p, cudaGetLastError());
    CUDA_TRY(p, cudaEventRecord(p->ev_gyro, gs));
    p->gyro_copy_err = cudaSuccess;
    p->gyro_dirty = true;  // the next compute call makes its stream wait for ev_gyro
    p->gyro_on_device = true;
    return RSSYNC_OK;
}

}  // extern "C"

namespace {

// SetTrackResult's error texts.  The non-finite ones are the reference's panic texts, indexed in its
// order of checks (core_private.cpp:199-202); the pixels forms report points_a / points_b as rays_a /
// rays_b.
const char* const kMsgNullBuffer = "set-track-result: null buffer";
const char* const kMsgTooManyRays = "set-track-result: more than 512 rays in one frame is not supported";
enum { kRaysA, kRaysB, kTsA, kTsB };
const char* const kMsgNonFinite[4] = {
    "set-track-result: non-finite numbers in rays_a", "set-track-result: non-finite numbers in rays_b",
    "set-track-result: non-finite numbers in ts_a", "set-track-result: non-finite numbers in ts_b"};

// SetTrackResult, stage 1: the reference's panic conditions, in its order (core_private.cpp:199-202)
int validate_track(const double* ts_a, const double* ts_b, const double* rays_a, const double* rays_b,
                   size_t count, const char** msg) {
    if (count && (!ts_a || !ts_b || !rays_a || !rays_b)) { *msg = kMsgNullBuffer; return RSSYNC_E_INVALID; }
    if (count > (size_t)rs::kMaxRaysPerFrame) { *msg = kMsgTooManyRays; return RSSYNC_E_INVALID; }
    if (!all_finite(rays_a, 3 * count)) { *msg = kMsgNonFinite[kRaysA]; return RSSYNC_E_NONFINITE; }
    if (!all_finite(rays_b, 3 * count)) { *msg = kMsgNonFinite[kRaysB]; return RSSYNC_E_NONFINITE; }
    if (!all_finite(ts_a, count)) { *msg = kMsgNonFinite[kTsA]; return RSSYNC_E_NONFINITE; }
    if (!all_finite(ts_b, count)) { *msg = kMsgNonFinite[kTsB]; return RSSYNC_E_NONFINITE; }
    return RSSYNC_OK;
}

// copy n doubles, report whether all are finite, and fold them into [lo, hi] when asked to:
// x * 0.0 is +-0 for finite x and NaN otherwise, so one accumulator carries the check
inline bool copy_checked_scalar(double* dst, const double* src, size_t n, double* lo, double* hi) {
    double acc = 0.0, l = lo ? *lo : 0.0, h = hi ? *hi : 0.0;
    for (size_t i = 0; i < n; ++i) {
        const double v = src[i];
        dst[i] = v;
        acc += v * 0.0;
        if (lo) { l = v < l ? v : l; h = v > h ? v : h; }
    }
    if (lo) { *lo = l; *hi = h; }
    return acc == 0.0;
}
#if defined(__x86_64__)
// The same with four doubles per instruction (the scalar form is a floating-point reduction, which the
// compiler may not vectorise).  NT: non-temporal stores -- the staging buffer is written once and read
// next by the copy engine, so the lines need not be fetched for ownership nor kept in the cache.
template <bool NT>
__attribute__((target("avx2"))) bool copy_checked_avx2(double* dst, const double* src, size_t n, double* lo, double* hi) {
    double acc = 0.0, l = lo ? *lo : 0.0, h = hi ? *hi : 0.0;
    size_t i = 0;
    for (; i < n && (reinterpret_cast<uintptr_t>(dst + i) & 31); ++i) {
        const double v = src[i];
        dst[i] = v;
        acc += v * 0.0;
        l = v < l ? v : l;
        h = v > h ? v : h;
    }
    __m256d va = _mm256_setzero_pd(), vl = _mm256_set1_pd(l), vh = _mm256_set1_pd(h);
    const __m256d zero = _mm256_setzero_pd();
    for (; i + 4 <= n; i += 4) {
        const __m256d v = _mm256_loadu_pd(src + i);
        if (NT) _mm256_stream_pd(dst + i, v);
        else _mm256_store_pd(dst + i, v);
        va = _mm256_add_pd(va, _mm256_mul_pd(v, zero));
        vl = _mm256_min_pd(v, vl);  // v < vl ? v : vl, as the scalar form
        vh = _mm256_max_pd(v, vh);
    }
    double ta[4], tl[4], th[4];
    _mm256_storeu_pd(ta, va);
    _mm256_storeu_pd(tl, vl);
    _mm256_storeu_pd(th, vh);
    for (int k = 0; k < 4; ++k) {
        acc += ta[k];
        l = tl[k] < l ? tl[k] : l;
        h = th[k] > h ? th[k] : h;
    }
    for (; i < n; ++i) {
        const double v = src[i];
        dst[i] = v;
        acc += v * 0.0;
        l = v < l ? v : l;
        h = v > h ? v : h;
    }
    if (NT) _mm_sfence();  // the stores are globally visible before the copy engine is pointed at them
    if (lo) { *lo = l; *hi = h; }
    return acc == 0.0;
}
#endif
inline bool copy_checked(double* dst, const double* src, size_t n, double* lo, double* hi) {
#if defined(__x86_64__)
    // RSSYNC_STAGE = scalar | avx2 | nt (measurement knob)
    static const int mode = [] {
        if (!__builtin_cpu_supports("avx2")) return 0;
        const char* e = std::getenv("RSSYNC_STAGE");
        if (!e) return RSSYNC_STAGE_DEFAULT;
        return e[0] == 's' ? 0 : e[0] == 'a' ? 1 : 2;
    }();
    if (mode == 1) return copy_checked_avx2<false>(dst, src, n, lo, hi);
    if (mode == 2) return copy_checked_avx2<true>(dst, src, n, lo, hi);
#endif
    return copy_checked_scalar(dst, src, n, lo, hi);
}

// SetTrackResult, stage 1 of the bulk form: validate_track fused with the copy into the staging
// buffers and with the frame's timestamp bounds (one pass over the caller's data)
int stage_track(const double* ts_a, const double* ts_b, const double* rays_a, const double* rays_b,
                size_t count, double* s_ts_a, double* s_ts_b, double* s_rays_a, double* s_rays_b,
                double& ts_lo, double& ts_hi, const char** msg) {
    if (count && (!ts_a || !ts_b || !rays_a || !rays_b)) { *msg = kMsgNullBuffer; return RSSYNC_E_INVALID; }
    if (count > (size_t)rs::kMaxRaysPerFrame) { *msg = kMsgTooManyRays; return RSSYNC_E_INVALID; }
    double lo = count ? ts_a[0] : 0.0, hi = lo;
    const bool ok_ra = copy_checked(s_rays_a, rays_a, 3 * count, nullptr, nullptr);
    const bool ok_rb = copy_checked(s_rays_b, rays_b, 3 * count, nullptr, nullptr);
    const bool ok_ta = copy_checked(s_ts_a, ts_a, count, &lo, &hi);
    const bool ok_tb = copy_checked(s_ts_b, ts_b, count, &lo, &hi);
    ts_lo = lo;
    ts_hi = hi;
    // the reference's order of checks (core_private.cpp:199-202)
    if (!ok_ra) { *msg = kMsgNonFinite[kRaysA]; return RSSYNC_E_NONFINITE; }
    if (!ok_rb) { *msg = kMsgNonFinite[kRaysB]; return RSSYNC_E_NONFINITE; }
    if (!ok_ta) { *msg = kMsgNonFinite[kTsA]; return RSSYNC_E_NONFINITE; }
    if (!ok_tb) { *msg = kMsgNonFinite[kTsB]; return RSSYNC_E_NONFINITE; }
    return RSSYNC_OK;
}

// stage 2 (serial bookkeeping): where the frame lives in the arena
// host_mirror: the frame is filled on the host (frames set one by one, small batches) and needs its
// range of the pinned mirror of the arena; a bulk ingest goes through its own staging buffer instead
int place_track(rssync_problem* p, int64_t frame, size_t count, FrameDesc** fd_out, bool host_mirror = true) {
    const size_t padded = (count + 31) / 32 * 32;
    size_t off;
    auto it = p->frames.end();
    if (p->place_hint_valid) {
        auto nx = std::next(p->place_hint);
        if (nx != p->frames.end() && nx->first == frame) it = nx;
    }
    auto pos = it;  // where a new node goes
    if (it == p->frames.end()) {
        pos = p->frames.lower_bound(frame);
        if (pos != p->frames.end() && pos->first == frame) it = pos;
    }
    if (it != p->frames.end() && (size_t)((it->second.n + 31) / 32 * 32) == padded) {
        off = (size_t)it->second.off;  // replace in place
        p->total_rays -= (size_t)it->second.n;
    } else {
        if (it != p->frames.end()) {
            p->garbage += (size_t)(it->second.n + 31) / 32 * 32;
            p->total_rays -= (size_t)it->second.n;
        }
        off = p->used;
        if (off + padded > (size_t)INT32_MAX) { p->err = "set-track-result: ray arena full"; return RSSYNC_E_INVALID; }
        p->used = off + padded;
    }
    if (host_mirror && off + padded > p->h_orig.cap) {  // (also a frame replaced in place that came in bulk)
        const size_t want = std::max<size_t>(std::max(off + padded, p->used), std::max<size_t>(p->h_orig.cap * 2, 1u << 16));
        cudaSetDevice(p->device);
        CUDA_TRY(p, p->h_rays.reserve(want * 8, p->used * 8));
        CUDA_TRY(p, p->h_orig.reserve(want, p->used));
        CUDA_TRY(p, p->h_pos.reserve(want, p->used));
    }
    if (it == p->frames.end()) it = p->frames.emplace_hint(pos, frame, FrameDesc{});
    if (!p->retime.empty()) p->retime.erase(frame);  // the pixels forms enter it again after placing
    p->rowq_version++;
    FrameDesc& fd = it->second;  // map nodes are stable: fill_track completes ts_lo / ts_hi
    fd = FrameDesc{frame, (int32_t)off, (int32_t)count, 0.0, 0.0};
    p->total_rays += count;
    p->place_hint = it;
    p->place_hint_valid = true;
    *fd_out = &fd;
    return RSSYNC_OK;
}

// stage 3 (thread-safe, disjoint arena ranges): sort by ts_a, transpose AoS -> [8][32] tiles
void fill_track(rssync_problem* p, FrameDesc* fd, const double* ts_a, const double* ts_b,
                const double* rays_a, const double* rays_b, size_t count,
                std::vector<std::pair<double, int32_t>>& scratch) {
    const size_t off = (size_t)fd->off;
    const size_t padded = (count + 31) / 32 * 32;
    double* tiles = p->h_rays.ptr + off * 8;
    int32_t* og = p->h_orig.ptr + off;
    int32_t* ps = p->h_pos.ptr + off;
    scratch.resize(count);
    for (size_t i = 0; i < count; ++i) scratch[i] = {ts_a[i], (int32_t)i};
    std::sort(scratch.begin(), scratch.end());  // (ts_a, index): ties keep the caller's order
    double lo = count ? ts_a[0] : 0.0, hi = lo;
    for (size_t j = 0; j < padded; ++j) {
        double* t = tiles + (j >> 5) * 256 + (j & 31);
        if (j < count) {
            const size_t i = (size_t)scratch[j].second;
            og[j] = (int32_t)i;
            ps[i] = (int32_t)j;
            t[0] = ts_a[i];
            t[32] = ts_b[i];
            t[64] = rays_a[3 * i]; t[96] = rays_a[3 * i + 1]; t[128] = rays_a[3 * i + 2];
            t[160] = rays_b[3 * i]; t[192] = rays_b[3 * i + 1]; t[224] = rays_b[3 * i + 2];
            lo = std::min(lo, std::min(ts_a[i], ts_b[i]));
            hi = std::max(hi, std::max(ts_a[i], ts_b[i]));
        } else {  // padding lanes: finite, masked out by n
            og[j] = (int32_t)j;
            ps[j] = (int32_t)j;
            t[0] = count ? ts_a[(size_t)scratch[count - 1].second] : 0.0;
            t[32] = count ? ts_b[(size_t)scratch[count - 1].second] : 0.0;
            for (int c = 2; c < 8; ++c) t[c * 32] = 0.0;
        }
    }
    fd->ts_lo = lo;
    fd->ts_hi = hi;
}

// Persistent host worker pool for the bulk ingest (validation, sort + transpose).  Creating
// std::threads per call costs ~30 us each, which is milliseconds per batch at 16 threads x several
// parallel regions; the pool's threads sleep on a condition variable between regions.
// Cores this process may use: RSSYNC_HOST_THREADS when set (one process per GPU shares the host with
// its siblings, and an oversubscribed pool that spins between regions is worse than a small one),
// else all of them.
unsigned host_cores() {
    if (const char* e = std::getenv("RSSYNC_HOST_THREADS")) {
        const int v = std::atoi(e);
        if (v > 0) return (unsigned)v;
    }
    const unsigned hw = std::thread::hardware_concurrency();
    return hw ? hw : 1;
}

// CPUs of the NUMA node the calling thread runs on (empty: one node, or unknown).  The staging copy
// is bound by host memory bandwidth; on a two-socket host, workers on the other socket would pull
// the caller's buffers and push the pinned staging buffer across the inter-socket link.
std::vector<int> numa_local_cpus() {
#if defined(__linux__)
    if (std::getenv("RSSYNC_NO_NUMA_PIN")) return {};
    const int cpu = sched_getcpu();
    if (cpu < 0) return {};
    std::vector<int> local;
    int nodes = 0;
    for (int node = 0; node < 64; ++node) {
        char path[96];
        std::snprintf(path, sizeof(path), "/sys/devices/system/node/node%d/cpulist", node);
        FILE* f = std::fopen(path, "r");
        if (!f) break;
        ++nodes;
        std::vector<int> cpus;
        int a = 0, b = 0;
        for (;;) {
            if (std::fscanf(f, "%d", &a) != 1) break;
            b = a;
            int c = std::fgetc(f);
            if (c == '-') {
                if (std::fscanf(f, "%d", &b) != 1) break;
                c = std::fgetc(f);
            }
            for (int k = a; k <= b; ++k) cpus.push_back(k);
            if (c != ',') break;
        }
        std::fclose(f);
        if (std::find(cpus.begin(), cpus.end(), cpu) != cpus.end()) local = cpus;
    }
    if (nodes < 2) return {};
    cpu_set_t allowed;
    CPU_ZERO(&allowed);
    if (sched_getaffinity(0, sizeof(allowed), &allowed) == 0) {
        std::vector<int> keep;
        for (int c : local)
            if (c < CPU_SETSIZE && CPU_ISSET(c, &allowed)) keep.push_back(c);
        local.swap(keep);
    }
    return local.size() >= 4 ? local : std::vector<int>{};
#else
    return {};
#endif
}

class WorkerPool {
public:
    static WorkerPool& get() {
        static WorkerPool pool;
        return pool;
    }
    size_t size() const { return threads_.size() + 1; }
    // fn(i, t) for i in [0, n), t = worker index; blocks of `grain` items are handed out dynamically
    void run(size_t n, const std::function<void(size_t, size_t)>& fn, size_t grain = 16) {
        if (n == 0) return;
        {
            std::lock_guard<std::mutex> lk(m_);
            fn_ = &fn;
            n_ = n;
            grain_ = grain ? grain : 1;
            next_.store(0);
            pending_.store(threads_.size());
            generation_.fetch_add(1, std::memory_order_release);
        }
        cv_.notify_all();
        work(0);
        // the regions of one ingest call follow each other within microseconds: spin briefly before
        // sleeping (a condition-variable wake-up costs 30-50 us, six regions per call)
        if (!spin_until([&] { return pending_.load(std::memory_order_acquire) == 0; })) {
            std::unique_lock<std::mutex> lk(m_);
            done_.wait(lk, [&] { return pending_.load() == 0; });
        }
        fn_ = nullptr;
    }

private:
    template <class Pred>
    static bool spin_until(Pred&& pred) {
        const auto t0 = std::chrono::steady_clock::now();
        for (int i = 0;; ++i) {
            if (pred()) return true;
            if ((i & 63) == 63 && std::chrono::steady_clock::now() - t0 > std::chrono::microseconds(150)) return false;
#if defined(__x86_64__) || defined(__i386__)
            __builtin_ia32_pause();
#endif
        }
    }
    WorkerPool() {
        // one core is left to the gyro worker thread, which runs beside the track ingest
        const std::vector<int> local = numa_local_cpus();
        const unsigned hw = local.empty() ? host_cores() : std::min<unsigned>(host_cores(), (unsigned)local.size());
        const size_t n = std::min<size_t>(hw > 2 ? hw - 1 : 1, 16);
        for (size_t t = 1; t < n; ++t)
            threads_.emplace_back([this, t, local]() {
#if defined(__linux__)
                if (!local.empty()) {  // stay on the caller's NUMA node
                    cpu_set_t set;
                    CPU_ZERO(&set);
                    for (int c : local)
                        if (c < CPU_SETSIZE) CPU_SET(c, &set);
                    pthread_setaffinity_np(pthread_self(), sizeof(set), &set);
                }
#endif
                uint64_t seen = 0;
                for (;;) {
                    if (!spin_until([&] { return generation_.load(std::memory_order_acquire) != seen || stop_.load(); })) {
                        std::unique_lock<std::mutex> lk(m_);
                        cv_.wait(lk, [&] { return generation_.load() != seen || stop_.load(); });
                    }
                    if (stop_.load()) return;
                    seen = generation_.load(std::memory_order_acquire);
                    work(t);
                    if (pending_.fetch_sub(1, std::memory_order_acq_rel) == 1) {
                        std::lock_guard<std::mutex> lk(m_);
                        done_.notify_one();
                    }
                }
            });
    }
    ~WorkerPool() {
        {
            std::lock_guard<std::mutex> lk(m_);
            stop_.store(true);
        }
        cv_.notify_all();
        for (auto& th : threads_) th.join();
    }
    void work(size_t t) {
        for (;;) {
            const size_t lo = next_.fetch_add(grain_);
            if (lo >= n_) break;
            for (size_t i = lo; i < std::min(n_, lo + grain_); ++i) (*fn_)(i, t);
        }
    }
    std::vector<std::thread> threads_;
    std::mutex m_;
    std::condition_variable cv_, done_;
    const std::function<void(size_t, size_t)>* fn_ = nullptr;
    size_t n_ = 0, grain_ = 16;
    std::atomic<size_t> next_{0}, pending_{0};
    std::atomic<uint64_t> generation_{0};
    std::atomic<bool> stop_{false};
};

}  // namespace
namespace {
void parallel_copy(void* dst, const void* src, size_t bytes) {
    constexpr size_t kPiece = 128 * 1024;
    if (bytes < 4 * kPiece) {
        std::memcpy(dst, src, bytes);
        return;
    }
    const size_t pieces = (bytes + kPiece - 1) / kPiece;
    WorkerPool::get().run(pieces, [&](size_t i, size_t) {
        const size_t a = i * kPiece, b = std::min(bytes, a + kPiece);
        std::memcpy(static_cast<char*>(dst) + a, static_cast<const char*>(src) + a, b - a);
    }, 1);
}

void parallel_frames(size_t n, const std::function<void(size_t, size_t)>& fn) {
    if (n < 64) {
        for (size_t i = 0; i < n; ++i) fn(i, 0);
        return;
    }
    WorkerPool::get().run(n, fn);
}

}  // namespace

extern "C" {

int rssync_set_track(rssync_problem* p, int64_t frame, const double* ts_a, const double* ts_b,
                     const double* rays_a, const double* rays_b, size_t count) {
    if (!p) return RSSYNC_E_INVALID;
    const char* msg = nullptr;
    if (int rc = validate_track(ts_a, ts_b, rays_a, rays_b, count, &msg)) { p->err = msg; return rc; }
    if (int rc = wait_arena_copies(p)) return rc;
    p->version++;
    FrameDesc* fd = nullptr;
    if (int rc = place_track(p, frame, count, &fd)) return rc;
    fill_track(p, fd, ts_a, ts_b, rays_a, rays_b, count, p->sort_scratch);
    add_pending(p, (size_t)fd->off, (size_t)fd->off + (count + 31) / 32 * 32);
    return RSSYNC_OK;
}

// Bulk ingest: same result as n_frames rssync_set_track calls (frames after a failing one are
// not applied), with validation and the sort/transpose spread over host threads.
int rssync_set_track_batch(rssync_problem* p, size_t n_frames, const int64_t* frames,
                           const size_t* counts, const double* ts_a, const double* ts_b,
                           const double* rays_a, const double* rays_b) {
    RS_NVTX_RANGE();
    if (!p || (n_frames && (!frames || !counts))) return RSSYNC_E_INVALID;
    p->version++;
    DebugTimer tm("set_track_batch");
    std::vector<size_t> at(n_frames + 1, 0);
    for (size_t i = 0; i < n_frames; ++i) at[i + 1] = at[i] + counts[i];
    std::vector<int> rc(n_frames, 0);
    std::vector<const char*> msg(n_frames, nullptr);
    // A frame id that appears twice in one batch: the blocks of one ingest launch would write the same
    // arena range concurrently.  The contract is n_frames SetTrackResult calls in order (the last one
    // wins, the reference's map semantics), which the frame-by-frame path below gives by construction.
    bool has_duplicates = false;
    if (n_frames >= 64) {
        std::vector<int64_t> ids(frames, frames + n_frames);
        std::sort(ids.begin(), ids.end());
        has_duplicates = std::adjacent_find(ids.begin(), ids.end()) != ids.end();
    }
    if (n_frames >= 64 && !has_duplicates) {
        // Large batch: the sort by ts_a and the transpose into tiles run on the device
        // (ingest_rays_kernel).  The host makes ONE pass over the caller's buffers: each value is
        // checked (the reference's panic conditions, core_private.cpp:199-202) while it is copied
        // into pinned staging memory, and the per-frame timestamp bounds are taken on the way.
        // Each eighth of the batch (RSSYNC_INGEST_CHUNKS) is placed, copied to the device and ingested as soon as it is
        // staged, overlapping the staging of the next.
        cudaSetDevice(p->device);
        if (int r = wait_arena_copies(p)) return r;
        if (int r = drain_in_flight(p)) return r;  // an earlier bulk call's chunks: all done by now
        if (!p->copy_stream) CUDA_TRY(p, cudaStreamCreateWithFlags(&p->copy_stream, cudaStreamNonBlocking));
        if (!p->ev_order) CUDA_TRY(p, cudaEventCreateWithFlags(&p->ev_order, cudaEventDisableTiming));
        // frames set one by one before this call are older than it: their upload goes first
        if (!p->pending.empty())
            if (int r = flush(p)) return r;
        // the ingest stream follows whatever the problem's stream has queued on the arena
        CUDA_TRY(p, cudaEventRecord(p->ev_order, p->stream));
        CUDA_TRY(p, cudaStreamWaitEvent(p->copy_stream, p->ev_order, 0));
        cudaStream_t cs = p->copy_stream;
        const size_t total = at[n_frames];
        // staging layout, per chunk and contiguous so that a chunk is ONE host->device copy:
        //   [frame records: 4 doubles (one PixelFrame) per frame][ts_a n][ts_b n][rays_a 3n][rays_b 3n]
        const size_t stage_doubles = 8 * total + 4 * n_frames + 1;
        CUDA_TRY(p, p->h_stage.reserve(stage_doubles));
        CUDA_TRY(p, p->d_stage.reserve(stage_doubles));
        if (!p->ev_arena) CUDA_TRY(p, cudaEventCreateWithFlags(&p->ev_arena, cudaEventDisableTiming));
        std::vector<double> lo_ts(n_frames), hi_ts(n_frames);
        // room for what this batch appends at the end of the arena: every frame that is new or changes
        // its padded size (the others are replaced in place) -- reserved up front, because growing
        // the arena moves it, which has to wait for the chunks already in flight
        size_t padded_new = 0;
        {
            auto it = p->frames.begin();
            for (size_t i = 0; i < n_frames; ++i) {
                const size_t padded = (counts[i] + 31) / 32 * 32;
                if (it == p->frames.end() || it->first != frames[i]) it = p->frames.find(frames[i]);
                const bool in_place = it != p->frames.end() && (size_t)((it->second.n + 31) / 32 * 32) == padded;
                if (!in_place) padded_new += padded;
                if (it != p->frames.end()) ++it;  // batches mostly come in frame order
            }
        }
        if (int r = reserve_device_arena(p, p->used + padded_new)) return r;
        tm.mark("reserve");
        double* hs = p->h_stage.ptr;
        double* ds = p->d_stage.ptr;
        static const size_t n_chunks = [] {
            const char* e = std::getenv("RSSYNC_INGEST_CHUNKS");
            const int v = e ? std::atoi(e) : 0;
            return (size_t)(v > 0 ? v : 8);
        }();
        size_t n_ok = n_frames;
        for (size_t c = 0; c < n_chunks && n_ok == n_frames; ++c) {
            const size_t lo = n_frames * c / n_chunks, hi = n_frames * (c + 1) / n_chunks;
            if (lo == hi) continue;
            const size_t a0 = at[lo], n = at[hi] - at[lo];          // the chunk's rays
            const size_t base = 8 * a0 + 4 * lo;                     // its block in the staging buffers
            double* h_rec = hs + base;                               // frame records
            double* h_tsa = h_rec + 4 * (hi - lo);
            double* h_tsb = h_tsa + n;
            double* h_ra = h_tsb + n;
            double* h_rb = h_ra + 3 * n;
            parallel_frames(hi - lo, [&](size_t k, size_t) {
                const size_t i = lo + k, cnt = counts[i], l = at[i] - a0;
                rc[i] = stage_track(ts_a + at[i], ts_b + at[i], rays_a + 3 * at[i], rays_b + 3 * at[i], cnt, h_tsa + l,
                                    h_tsb + l, h_ra + 3 * l, h_rb + 3 * l, lo_ts[i], hi_ts[i], &msg[i]);
            });
            tm.mark("stage + validate chunk");
            size_t end = hi;
            for (size_t i = lo; i < hi; ++i)
                if (rc[i]) { end = i; n_ok = i; break; }
            rssync_problem::InFlight fl{(size_t)-1, 0, nullptr, false};
            rs::PixelFrame* pf = reinterpret_cast<rs::PixelFrame*>(h_rec);
            for (size_t i = lo; i < end; ++i) {
                FrameDesc* fd = nullptr;
                if (int r = place_track(p, frames[i], counts[i], &fd, /*host_mirror=*/false)) return r;
                fd->ts_lo = lo_ts[i];
                fd->ts_hi = hi_ts[i];
                pf[i - lo] = rs::PixelFrame{fd->off, fd->n, (int64_t)(at[i] - a0), 0.0, 0.0};
                // the arena range this chunk writes
                fl.lo = std::min(fl.lo, (size_t)fd->off);
                fl.hi = std::max(fl.hi, (size_t)fd->off + (counts[i] + 31) / 32 * 32);
            }
            if (end == lo) break;
            if (int r = reserve_device_arena(p)) return r;
            tm.mark("place chunk");
            const size_t block = 4 * (hi - lo) + 8 * n;  // doubles
            p->h2d += block * sizeof(double);
            CUDA_TRY(p, cudaMemcpyAsync(ds + base, hs + base, block * sizeof(double), cudaMemcpyHostToDevice, cs));
            double* d_rec = ds + base;
            double* d_tsa = d_rec + 4 * (hi - lo);
            rs::launch_ingest_rays(reinterpret_cast<const rs::PixelFrame*>(d_rec), (int)(end - lo), d_tsa, d_tsa + n,
                                   d_tsa + 2 * n, d_tsa + 5 * n, p->d_rays.ptr, p->d_orig.ptr, p->d_pos.ptr, cs);
            CUDA_TRY(p, cudaGetLastError());
            p->dev_used = std::max(p->dev_used, p->used);  // a later growth of the arena keeps this chunk
            // the event that says the chunk's arena range has been written
            if (p->ev_pool.empty()) {
                CUDA_TRY(p, cudaEventCreateWithFlags(&fl.ev, cudaEventDisableTiming));
            } else {
                fl.ev = p->ev_pool.back();
                p->ev_pool.pop_back();
            }
            CUDA_TRY(p, cudaEventRecord(fl.ev, cs));
            p->in_flight.push_back(fl);
            tm.mark("enqueue chunk");
        }
        // the staging buffers are reused by the next ingest call, which waits for this event
        CUDA_TRY(p, cudaEventRecord(p->ev_arena, cs));
        p->arena_copy_pending = true;
        if (n_ok < n_frames) { p->err = msg[n_ok]; return rc[n_ok]; }
        return RSSYNC_OK;
    }
    size_t n_ok = n_frames;
    for (size_t i = 0; i < n_frames; ++i) {
        rc[i] = validate_track(ts_a + at[i], ts_b + at[i], rays_a + 3 * at[i], rays_b + 3 * at[i], counts[i], &msg[i]);
        if (rc[i]) { n_ok = i; break; }
    }
    if (int r = wait_arena_copies(p)) return r;
    std::vector<std::pair<double, int32_t>> scratch;
    for (size_t i = 0; i < n_ok; ++i) {
        FrameDesc* fd = nullptr;
        if (int r = place_track(p, frames[i], counts[i], &fd)) return r;
        fill_track(p, fd, ts_a + at[i], ts_b + at[i], rays_a + 3 * at[i], rays_b + 3 * at[i], counts[i], scratch);
        add_pending(p, (size_t)fd->off, (size_t)fd->off + (counts[i] + 31) / 32 * 32);
    }
    if (n_ok < n_frames) { p->err = msg[n_ok]; return rc[n_ok]; }
    return RSSYNC_OK;
}

}  // extern "C"

namespace {

// at = offsets of the frames' rays in the concatenated per-ray buffers (n_frames + 1 entries)
int frame_offsets(rssync_problem* p, size_t n_frames, const size_t* counts, std::vector<size_t>& at) {
    at.assign(n_frames + 1, 0);
    for (size_t i = 0; i < n_frames; ++i) {
        if (counts[i] > (size_t)rs::kMaxRaysPerFrame) { p->err = kMsgTooManyRays; return RSSYNC_E_INVALID; }
        at[i + 1] = at[i] + counts[i];
    }
    return RSSYNC_OK;
}

// Upper bounds of |theta (1 + k1 theta^2 + .. + k4 theta^8)| and of its derivative over [0, pi/2], where
// undistort_point (engine.cu) keeps its Newton iterates: while both are finite, so are the iterates (a
// derivative of exactly 0 aside).  Twice the bounds are checked, headroom for the roundings of both sides.
bool lens_polynomial_bounded(const rssync_lens& l) {
    const double h = 1.5707963267948966, h2 = h * h;
    const double a1 = std::fabs(l.k1), a2 = std::fabs(l.k2), a3 = std::fabs(l.k3), a4 = std::fabs(l.k4);
    const double f = h * (1.0 + h2 * (a1 + h2 * (a2 + h2 * (a3 + h2 * a4))));
    const double df = 1.0 + h2 * (3.0 * a1 + h2 * (5.0 * a2 + h2 * (7.0 * a3 + h2 * 9.0 * a4)));
    return std::isfinite(2.0 * f) && std::isfinite(2.0 * df);
}

// n points (x, y) are finite, and so are undistort_point's x_ = (px - cx) / fx, y_ and theta_^2 = x_^2 + y_^2
// (engine.cu): a finite pixel far enough out for the focal length is not, and would give a NaN ray
bool points_ok(const double* pts, size_t n, const rssync_lens& l) {
    if (!all_finite(pts, 2 * n)) return false;
    for (size_t k = 0; k < n; ++k) {
        const double x_ = (pts[2 * k] - l.cx) / l.fx, y_ = (pts[2 * k + 1] - l.cy) / l.fy;
        if (!std::isfinite(x_ * x_ + y_ * y_)) return false;
    }
    return true;
}

// the pixels forms' lens profile, image height and counts
int check_pixel_args(rssync_problem* p, size_t n_frames, const size_t* counts, const rssync_lens* lens,
                     double image_rows, std::vector<size_t>& at) {
    const double lv[9] = {lens->readout, lens->fx, lens->fy, lens->cx, lens->cy, lens->k1, lens->k2, lens->k3, lens->k4};
    if (!all_finite(lv, 9) || !(image_rows > 0) || !std::isfinite(image_rows) || lens->fx == 0 || lens->fy == 0 ||
        !lens_polynomial_bounded(*lens)) {
        p->err = "set-track-pixels: bad lens profile or image height";
        return RSSYNC_E_INVALID;
    }
    return frame_offsets(p, n_frames, counts, at);
}

rs::LensDev lens_dev(const rssync_lens& l) {
    return rs::LensDev{l.readout, l.fx, l.fy, l.cx, l.cy, l.k1, l.k2, l.k3, l.k4};
}

// the pixels forms' per-frame timestamps, checked before any point
int check_frame_ts(rssync_problem* p, size_t n_frames, const double* frame_ts_a, const double* frame_ts_b) {
    if (!all_finite(frame_ts_a, n_frames)) { p->err = kMsgNonFinite[kTsA]; return RSSYNC_E_NONFINITE; }
    if (!all_finite(frame_ts_b, n_frames)) { p->err = kMsgNonFinite[kTsB]; return RSSYNC_E_NONFINITE; }
    return RSSYNC_OK;
}

// The per-ray buffers of a *_device call: device (or managed) memory of the problem's device.  A plain
// host pointer is reported as unregistered memory.
int check_device_buffers(rssync_problem* p, std::initializer_list<const double*> bufs, size_t total) {
    if (!total) return RSSYNC_OK;
    for (const double* b : bufs) {
        if (!b) { p->err = kMsgNullBuffer; return RSSYNC_E_INVALID; }
        cudaPointerAttributes attr{};
        const cudaError_t e = cudaPointerGetAttributes(&attr, b);
        if (e != cudaSuccess) cudaGetLastError();  // (clears the error)
        if (e != cudaSuccess || (attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged) ||
            attr.device != p->device) {
            p->err = "set-track-result: a per-ray buffer is not device memory of the problem's device";
            return RSSYNC_E_INVALID;
        }
    }
    return RSSYNC_OK;
}

// The device forms' per-call blocks, in the pinned h_stage and (mirrored) in d_stage, in doubles:
//   [at: n + 1 int64][frame_ts: 2n][info: 3n (rs::StageInfo)][records: 4n (rs::PixelFrame)]
// followed on the device by the staged per-ray data.  Per frame 8 bytes go up before the check, 24
// come back, 32 go up after the placement (pixels form: 16 more up, the frame timestamps).
struct DeviceStaging {
    int64_t* h_at;
    double* h_fts;
    rs::StageInfo* h_info;
    rs::PixelFrame* h_rec;
    int64_t* d_at;
    double* d_fts;
    rs::StageInfo* d_info;
    rs::PixelFrame* d_rec;
    double* d_data;
};

// Before the check-and-stage kernel of a device form: order the problem's stream behind everything
// that writes the arena (as the host forms do) and behind the work the caller has queued on `stream`,
// and upload the frame offsets (and the pixels form's frame timestamps).
int begin_device_staging(rssync_problem* p, const std::vector<size_t>& at, size_t data_doubles,
                         const double* frame_ts_a, const double* frame_ts_b, void* stream, DeviceStaging& s) {
    const size_t n = at.size() - 1;
    if (int rc = begin_ingest(p)) return rc;
    const size_t block = 10 * n + 1;
    CUDA_TRY(p, p->h_stage.reserve(block));
    CUDA_TRY(p, p->d_stage.reserve(block + data_doubles));
    double* h = p->h_stage.ptr;
    double* d = p->d_stage.ptr;
    s = DeviceStaging{reinterpret_cast<int64_t*>(h), h + n + 1, reinterpret_cast<rs::StageInfo*>(h + 3 * n + 1),
                      reinterpret_cast<rs::PixelFrame*>(h + 6 * n + 1), reinterpret_cast<int64_t*>(d), d + n + 1,
                      reinterpret_cast<rs::StageInfo*>(d + 3 * n + 1), reinterpret_cast<rs::PixelFrame*>(d + 6 * n + 1),
                      d + block};
    for (size_t i = 0; i <= n; ++i) s.h_at[i] = (int64_t)at[i];
    if (int rc = h2d(p, s.d_at, s.h_at, (n + 1) * sizeof(int64_t))) return rc;
    if (frame_ts_a) {
        for (size_t i = 0; i < n; ++i) {
            s.h_fts[2 * i] = frame_ts_a[i];
            s.h_fts[2 * i + 1] = frame_ts_b[i];
        }
        if (int rc = h2d(p, s.d_fts, s.h_fts, 2 * n * sizeof(double))) return rc;
    }
    if (!p->ev_order) CUDA_TRY(p, cudaEventCreateWithFlags(&p->ev_order, cudaEventDisableTiming));
    CUDA_TRY(p, cudaEventRecord(p->ev_order, static_cast<cudaStream_t>(stream)));
    CUDA_TRY(p, cudaStreamWaitEvent(p->stream, p->ev_order, 0));
    return RSSYNC_OK;
}

// After the kernel: the per-frame verdicts come back (the one round trip of a device form).  Once
// this returns nothing reads the caller's buffers any more.
int read_stage_info(rssync_problem* p, size_t n, const DeviceStaging& s) {
    if (int rc = d2h(p, s.h_info, s.d_info, n * sizeof(rs::StageInfo))) return rc;
    return finish_stream(p, p->stream);
}

// After the ingest kernel: the arena holds the frames; the next call that reuses the staging blocks
// waits for this point of the problem's stream
int end_device_ingest(rssync_problem* p) {
    CUDA_TRY(p, cudaGetLastError());
    p->dev_used = std::max(p->dev_used, p->used);
    if (!p->ev_arena) CUDA_TRY(p, cudaEventCreateWithFlags(&p->ev_arena, cudaEventDisableTiming));
    CUDA_TRY(p, cudaEventRecord(p->ev_arena, p->stream));
    p->arena_copy_pending = true;
    return RSSYNC_OK;
}

// The row-fraction plane of the pixels forms, as large as the device arena (contents kept)
int reserve_rowq(rssync_problem* p) {
    CUDA_TRY(p, p->d_rowq.grow(2 * std::max<size_t>(p->d_orig.cap, 1), 2 * p->dev_used, p->stream));
    p->rowq_version++;
    return RSSYNC_OK;
}

// The bulk ingests on the problem's stream, once the first n frames have passed their checks: place the
// last occurrence of each frame id among them (an ingest block per occurrence would write the same arena
// range twice; the last one wins, as with rssync_set_track calls in order), fill its ingest record
// (rec[0..k)) and make room in the device arena.  at: the frames' offsets in the staged data; info: their
// timestamp bounds.  frame_ts_a / frame_ts_b (pixels and row-fractions forms, else null): the frames keep
// them for re-timing, and the row-fraction plane grows with the arena.
int place_frames(rssync_problem* p, size_t n, const int64_t* frames, const std::vector<size_t>& at,
                 const rs::StageInfo* info, const double* frame_ts_a, const double* frame_ts_b, rs::PixelFrame* rec,
                 size_t& k) {
    std::vector<char> last(n, 1);
    if (std::adjacent_find(frames, frames + n, std::greater_equal<int64_t>()) != frames + n) {  // not ascending
        std::unordered_set<int64_t> seen;
        for (size_t i = n; i-- > 0;) last[i] = seen.insert(frames[i]).second;
    }
    p->version++;
    k = 0;
    for (size_t i = 0; i < n; ++i) {
        if (!last[i]) continue;
        FrameDesc* fd = nullptr;
        if (int rc = place_track(p, frames[i], at[i + 1] - at[i], &fd, /*host_mirror=*/false)) return rc;
        fd->ts_lo = info[i].lo;
        fd->ts_hi = info[i].hi;
        rec[k++] = rs::PixelFrame{fd->off, fd->n, (int64_t)at[i], frame_ts_a ? frame_ts_a[i] : 0.0,
                                  frame_ts_a ? frame_ts_b[i] : 0.0};
        if (frame_ts_a) p->retime[frames[i]] = {frame_ts_a[i], frame_ts_b[i]};
    }
    if (int rc = reserve_device_arena(p)) return rc;
    return frame_ts_a ? reserve_rowq(p) : RSSYNC_OK;
}

// the first of n frames whose check found a non-finite value (n: none)
size_t first_bad(const rs::StageInfo* info, size_t n) {
    size_t i = 0;
    while (i < n && !info[i].bad) ++i;
    return i;
}
// such a frame fails the call with the text of its first source buffer holding the value
int fail_nonfinite(rssync_problem* p, const rs::StageInfo& info) {
    p->err = kMsgNonFinite[__builtin_ctz(info.bad)];
    return RSSYNC_E_NONFINITE;
}

// A plane that covers the whole device arena: frames a rays form appended since the last row fractions
// have grown the arena but not the plane (their rays have no row fractions; the bytes only have to exist)
int rowq_cover_arena(rssync_problem* p) {
    if (2 * p->dev_used <= p->d_rowq.cap) return RSSYNC_OK;
    if (int rc = wait_reader(p)) return rc;  // a replication still reading the old plane
    return reserve_rowq(p);
}

// The row fractions to every replica whose copy is stale: the re-timing table on the host, the plane
// (2 doubles per arena ray) as ONE grouped ncclBroadcast of [0, 2 dev_used) doubles on the replication
// streams, behind the arena's replication (multi_replicate, called first), announced to each replica as
// an arena range in flight so that its re-timing waits for it.  Only the readout search reads them.
int multi_replicate_row_fractions(rssync_problem* p) {
    RS_NVTX_RANGE();
    bool stale = false;
    for (const rssync_problem* r : p->replicas) stale = stale || r->rowq_synced != p->rowq_version;
    if (!stale) return RSSYNC_OK;
    const bool plane = !p->retime.empty();
    if (plane)
        if (int rc = rowq_cover_arena(p)) return rc;
    const size_t rays = p->dev_used;
    DeviceGuard guard;
    for (rssync_problem* r : p->replicas) {
        cudaSetDevice(r->device);
        r->retime = p->retime;
        cudaError_t e = cudaStreamSynchronize(r->stream);  // no earlier search still reads the old plane
        if (e == cudaSuccess && r->repl_stream) e = cudaStreamSynchronize(r->repl_stream);
        if (e == cudaSuccess && plane) e = r->d_rowq.reserve(2 * std::max<size_t>(rays, 1));
        if (e == cudaSuccess && !r->repl_stream) e = cudaStreamCreateWithFlags(&r->repl_stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) {
            p->err = std::string("CUDA error on device ") + std::to_string(r->device) + ": " + cudaGetErrorString(e);
            return RSSYNC_E_CUDA;
        }
    }
    if (plane && rays) {
        cudaSetDevice(p->device);
        if (!p->repl_stream) CUDA_TRY(p, cudaStreamCreateWithFlags(&p->repl_stream, cudaStreamNonBlocking));
        if (int rc = rssync_stream_wait_chunk(p, -1, p->repl_stream)) return rc;  // the plane as the ingests left it
        const rs::Nccl* nc = rs::Nccl::get();
        NCCL_TRY(p, nc->GroupStart());
        for (int i = 0; i < n_ranks(p); ++i) {
            rssync_problem* q = rank_problem(p, i);
            cudaSetDevice(q->device);
            NCCL_TRY(p, nc->Broadcast(q->d_rowq.ptr, q->d_rowq.ptr, 2 * rays * sizeof(double), rs::Nccl::kChar, 0,
                                      p->comms[(size_t)i], q->repl_stream));
        }
        NCCL_TRY(p, nc->GroupEnd());
        p->nccl_calls += 1;
        p->broadcast_bytes += 2 * rays * sizeof(double);
        for (rssync_problem* r : p->replicas)
            if (int rc = rssync_expect_chunk(r, 0, rays, r->repl_stream)) {
                p->err = r->err;
                return rc;
            }
        if (int rc = rssync_note_reader(p, p->repl_stream)) return rc;  // the next ingest waits for this send
    }
    for (rssync_problem* r : p->replicas) r->rowq_synced = p->rowq_version;
    return RSSYNC_OK;
}

}  // namespace

extern "C" {

// Bulk SetTrackResult from device memory.  The check, the timestamp bounds and the copy into the
// staging buffer run on the device (stage_tracks_kernel), the sort and transpose in the same ingest
// kernel as the host form's.  Frames before the first one holding a non-finite value are applied;
// of a frame id given more than once among them, the last occurrence (n_frames rssync_set_track
// calls in order).
int rssync_set_track_batch_device(rssync_problem* p, size_t n_frames, const int64_t* frames,
                                  const size_t* counts, const double* ts_a, const double* ts_b,
                                  const double* rays_a, const double* rays_b, void* stream) {
    RS_NVTX_RANGE();
    if (!p || (n_frames && (!frames || !counts)) || n_frames > (size_t)INT32_MAX) return RSSYNC_E_INVALID;
    std::vector<size_t> at;
    if (int rc = frame_offsets(p, n_frames, counts, at)) return rc;
    const size_t total = at[n_frames];
    if (int rc = check_device_buffers(p, {rays_a, rays_b, ts_a, ts_b}, total)) return rc;
    if (n_frames == 0) return RSSYNC_OK;
    DeviceStaging s;
    if (int rc = begin_device_staging(p, at, 8 * total, nullptr, nullptr, stream, s)) return rc;
    rs::launch_stage_rays(s.d_at, (int)n_frames, (int64_t)total, rays_a, rays_b, ts_a, ts_b, s.d_data, s.d_info,
                          p->stream);
    if (int rc = read_stage_info(p, n_frames, s)) return rc;
    const size_t n_ok = first_bad(s.h_info, n_frames);
    size_t k = 0;
    if (int rc = place_frames(p, n_ok, frames, at, s.h_info, nullptr, nullptr, s.h_rec, k)) return rc;
    if (k) {
        if (int rc = h2d(p, s.d_rec, s.h_rec, k * sizeof(rs::PixelFrame))) return rc;
        rs::launch_ingest_rays(s.d_rec, (int)k, s.d_data, s.d_data + total, s.d_data + 2 * total, s.d_data + 5 * total,
                               p->d_rays.ptr, p->d_orig.ptr, p->d_pos.ptr, p->stream);
        if (int rc = end_device_ingest(p)) return rc;
    }
    return n_ok < n_frames ? fail_nonfinite(p, s.h_info[n_ok]) : RSSYNC_OK;
}

// The per-frame tail of track_frames (core_testcode.cpp:134-161) on the device: pixel pairs in,
// rays + rolling-shutter timestamps straight into the device arena (no host sort / transpose, half
// the host->device bytes of the ray form).  One pass on the worker pool checks every frame while it copies
// it into the pinned staging block and takes its timestamp bounds, then one upload and one ingest launch.
// Staging block, in doubles: [records: 4 per frame][points_a 2n][points_b 2n].
int rssync_set_track_pixels(rssync_problem* p, size_t n_frames, const int64_t* frames, const size_t* counts,
                            const double* frame_ts_a, const double* frame_ts_b, const double* points_a,
                            const double* points_b, const rssync_lens* lens, double image_rows) {
    RS_NVTX_RANGE();
    if (!p) return RSSYNC_E_INVALID;
    if (n_frames == 0) return RSSYNC_OK;
    if (!frames || !counts || !frame_ts_a || !frame_ts_b || !points_a || !points_b || !lens) return RSSYNC_E_INVALID;
    std::vector<size_t> at;
    if (int rc = check_pixel_args(p, n_frames, counts, lens, image_rows, at)) return rc;
    const size_t total = at[n_frames];
    if (int rc = check_frame_ts(p, n_frames, frame_ts_a, frame_ts_b)) return rc;
    if (int rc = begin_ingest(p)) return rc;
    const size_t block = 4 * n_frames + 4 * total;
    CUDA_TRY(p, p->h_stage.reserve(block + 1));
    double* h_pa = p->h_stage.ptr + 4 * n_frames;
    double* h_pb = h_pa + 2 * total;
    // per frame (worker pool): validate, copy into the pinned staging block, timestamp bounds with
    // the device's expression (core_testcode.cpp:144-145)
    std::vector<rs::StageInfo> info(n_frames, rs::StageInfo{0u, 0u, 0.0, 0.0});
    parallel_frames(n_frames, [&](size_t i, size_t) {
        const double* a = points_a + 2 * at[i];
        const double* b = points_b + 2 * at[i];
        const size_t n = counts[i];
        if (!points_ok(a, n, *lens)) { info[i].bad = 1u << kRaysA; return; }
        if (!points_ok(b, n, *lens)) { info[i].bad = 1u << kRaysB; return; }
        std::memcpy(h_pa + 2 * at[i], a, 2 * n * sizeof(double));
        std::memcpy(h_pb + 2 * at[i], b, 2 * n * sizeof(double));
        double l = 0.0, h = 0.0;
        for (size_t k = 0; k < n; ++k) {
            const double ta = frame_ts_a[i] + lens->readout * (a[2 * k + 1] / image_rows);
            const double tb = frame_ts_b[i] + lens->readout * (b[2 * k + 1] / image_rows);
            if (k == 0) { l = std::min(ta, tb); h = std::max(ta, tb); }
            l = std::min(l, std::min(ta, tb));
            h = std::max(h, std::max(ta, tb));
        }
        info[i].lo = l;
        info[i].hi = h;
    });
    if (const size_t i = first_bad(info.data(), n_frames); i < n_frames) return fail_nonfinite(p, info[i]);
    rs::PixelFrame* rec = reinterpret_cast<rs::PixelFrame*>(p->h_stage.ptr);
    size_t k = 0;
    if (int rc = place_frames(p, n_frames, frames, at, info.data(), frame_ts_a, frame_ts_b, rec, k)) return rc;
    CUDA_TRY(p, p->d_stage.reserve(block + 1));
    if (int rc = h2d(p, p->d_stage.ptr, p->h_stage.ptr, block * sizeof(double))) return rc;
    const double* d_pa = p->d_stage.ptr + 4 * n_frames;
    rs::launch_ingest_pixels(reinterpret_cast<const rs::PixelFrame*>(p->d_stage.ptr), (int)k, d_pa, d_pa + 2 * total,
                             lens_dev(*lens), image_rows, p->d_rays.ptr, p->d_orig.ptr, p->d_pos.ptr, p->d_rowq.ptr,
                             p->stream);
    return end_device_ingest(p);
}

}  // extern "C"

namespace {

// The device pixels forms once the per-frame verdicts are back (read_stage_info): the first frame holding a
// non-finite value fails the call before anything is placed, else the frames are placed and their points,
// staged at the offsets `at` of `total` points per side, ingested.
int ingest_staged_pixels(rssync_problem* p, size_t n_frames, const int64_t* frames, const std::vector<size_t>& at,
                         size_t total, const double* frame_ts_a, const double* frame_ts_b, const rs::LensDev& L,
                         double image_rows, const DeviceStaging& s) {
    if (const size_t i = first_bad(s.h_info, n_frames); i < n_frames) return fail_nonfinite(p, s.h_info[i]);
    size_t k = 0;
    if (int rc = place_frames(p, n_frames, frames, at, s.h_info, frame_ts_a, frame_ts_b, s.h_rec, k)) return rc;
    if (int rc = h2d(p, s.d_rec, s.h_rec, k * sizeof(rs::PixelFrame))) return rc;
    rs::launch_ingest_pixels(s.d_rec, (int)k, s.d_data, s.d_data + 2 * total, L, image_rows, p->d_rays.ptr,
                             p->d_orig.ptr, p->d_pos.ptr, p->d_rowq.ptr, p->stream);
    return end_device_ingest(p);
}

// The buffers of rssync_track_frames_device: device (or managed) memory of the problem's device, as
// check_device_buffers requires of per-ray buffers
int check_device_pointer(rssync_problem* p, const void* b, const char* what) {
    cudaPointerAttributes attr{};
    const cudaError_t e = b ? cudaPointerGetAttributes(&attr, b) : cudaErrorInvalidValue;
    if (e != cudaSuccess) cudaGetLastError();  // (clears the error)
    if (e != cudaSuccess || (attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged) ||
        attr.device != p->device) {
        p->err = std::string("track-frames: ") + what + " is not device memory of the problem's device";
        return RSSYNC_E_INVALID;
    }
    return RSSYNC_OK;
}

// the tracker's scratch budget: the pyramids of as many images as fit are alive at once
constexpr size_t kTrackScratchBytes = size_t(256) << 20;

// the outputs of rssync_track_frames_ex_device (each may be null)
struct TrackOutputs {
    double* points;
    size_t* counts;
    double* tracked;
    uint8_t* status;
    double* fb;
};

// The body of the tracking entry points once their null checks have passed.  opt null: the plain form
// (caller's points, no backward pass, no options checked).  sample: bytes per sample of the planes, 1
// (uint8) or 2 (uint16, level 0 = v * 2^-shift).  mask null: no mask.
int track_frames(rssync_problem* p, size_t n_frames, const int64_t* frames, const size_t* counts,
                 const double* image_ts, const double* points, const void* images, size_t pitch, int width,
                 int height, const rssync_lens* lens, const rssync_track_params* params,
                 const rssync_track_options* opt, const TrackOutputs& out, void* stream, int sample = 1,
                 int shift = 0, const rssync_track_mask* mask = nullptr) {
    const rssync_track_params tp = params ? *params : rssync_track_params{3, 21, 30, 0.01, 1e-4};
    if (tp.levels < 1 || tp.levels > 6 || tp.window < 5 || tp.window > 63 || tp.window % 2 == 0 || tp.max_iters < 1 ||
        tp.max_iters > 100 || !(tp.epsilon >= 0.0) || !std::isfinite(tp.epsilon) || !(tp.min_eig >= 0.0) ||
        !std::isfinite(tp.min_eig)) {
        p->err = "track-frames: parameters out of range";
        return RSSYNC_E_INVALID;
    }
    const bool select = opt && !points;
    if (opt && (opt->cell < 16 || opt->cell > 128 || (opt->block != 3 && opt->block != 5 && opt->block != 7) ||
                !(opt->quality > 0.0 && opt->quality <= 1.0) || opt->max_points < 1 ||
                opt->max_points > rs::kMaxRaysPerFrame || !(opt->fb_max >= 0.0))) {
        p->err = "track-frames: options out of range";
        return RSSYNC_E_INVALID;
    }
    const int64_t min_side = (int64_t)tp.window << (tp.levels - 1);
    if (width < min_side || height < min_side || pitch < (size_t)width) {
        p->err = "track-frames: image smaller than window * 2^(levels - 1), or pitch below width";
        return RSSYNC_E_INVALID;
    }
    if (sample == 2) {
        if (shift < 0 || shift > 8) {
            p->err = "track-frames: shift outside 0..8";
            return RSSYNC_E_INVALID;
        }
        if (reinterpret_cast<uintptr_t>(images) % 2 || pitch % 2 || pitch < 2 * (size_t)width) {
            p->err = "track-frames: 16-bit images need a 2-byte aligned address and an even pitch >= 2 * width bytes";
            return RSSYNC_E_INVALID;
        }
    }
    rs::TrackSelect sel{};
    if (select) {
        sel.cell = opt->cell;
        sel.block = opt->block;
        sel.max_points = opt->max_points;
        sel.quality = (float)opt->quality;
        sel.cells_x = (width + opt->cell - 1) / opt->cell;
        sel.cells_y = (height + opt->cell - 1) / opt->cell;
        const int min_sel = 2 * (opt->block / 2 + 2) + 1;
        if (width < min_sel || height < min_sel) {
            p->err = "track-frames: image smaller than 2 * (block / 2 + 2) + 1 for the selection";
            return RSSYNC_E_INVALID;
        }
        if ((int64_t)sel.cells_x * sel.cells_y > 65536) {
            p->err = "track-frames: more than 65536 selection cells per image";
            return RSSYNC_E_INVALID;
        }
    }
    // selection: every frame is sized for max_points points until the device has chosen them
    const std::vector<size_t> bound(select ? n_frames : 0, select ? (size_t)opt->max_points : 0);
    std::vector<size_t> at;
    if (int rc = check_pixel_args(p, n_frames, select ? bound.data() : counts, lens, (double)height, at)) return rc;
    const size_t total = at[n_frames];
    if (int rc = check_device_pointer(p, images, "images")) return rc;
    if (total && !select)
        if (int rc = check_device_pointer(p, points, "points")) return rc;
    for (void* o : {(void*)out.points, (void*)out.tracked, (void*)out.status, (void*)out.fb})
        if (o && total)
            if (int rc = check_device_pointer(p, o, "an output buffer")) return rc;
    if (mask) {
        if (int rc = check_device_pointer(p, mask->mask, "mask")) return rc;
        const char* bad = mask->pitch < (size_t)width ? "track-frames: mask pitch below width"
                          : mask->margin < 0 || mask->margin > rs::kTrackMaxMargin
                              ? "track-frames: mask margin outside 0..63"
                          : mask->image_stride && mask->image_stride / mask->pitch < (size_t)height
                              ? "track-frames: mask image_stride below height * pitch"
                              : nullptr;
        if (bad) {
            p->err = bad;
            return RSSYNC_E_INVALID;
        }
    }
    if (int rc = check_frame_ts(p, n_frames, image_ts, image_ts + 1)) return rc;

    const size_t per_image = rs::track_pyramid_floats(width, height, tp.levels);
    const size_t n_images = n_frames + 1;
    const size_t plane = (size_t)width * height;
    const bool mask_per_image = mask && mask->image_stride;
    // bytes of one slot: its pyramid, the selection's scratch and a per-image mask's eligibility plane
    const size_t n_cells = (size_t)sel.cells_x * sel.cells_y;
    const size_t bytes = 4 * per_image + (select ? 8 * n_cells + 4 * (size_t)sel.max_points + 4 : 0) +
                         (mask_per_image ? plane : 0);
    size_t slots = bytes ? std::min(n_images, std::max<size_t>(2, kTrackScratchBytes / bytes)) : n_images;
    if (select) slots = std::min(slots, size_t(65536));
    if (mask_per_image) slots = std::min(slots, size_t(65535));  // (the erosion's grid.z)
    const double fb_max = opt ? opt->fb_max : 0.0;
    CUDA_TRY(p, cudaSetDevice(p->device));
    CUDA_TRY(p, p->d_trk_pyr.reserve(std::max<size_t>(1, slots * per_image)));
    // compacted a, b (4 per point), tracked (2 per point), selected points (2 per point)
    CUDA_TRY(p, p->d_trk_pts.reserve((select ? 8 : 6) * total + 1));
    CUDA_TRY(p, p->d_trk_at.reserve(n_frames + 1));
    CUDA_TRY(p, p->d_trk_status.reserve(total + 1));
    CUDA_TRY(p, p->d_trk_flag.reserve(1));
    CUDA_TRY(p, p->h_trk_flag.reserve(1));
    if (select) {
        CUDA_TRY(p, p->d_trk_keys.reserve(slots * n_cells));
        CUDA_TRY(p, p->d_trk_picks.reserve(slots * sel.max_points));
        CUDA_TRY(p, p->d_trk_count.reserve(slots));
        CUDA_TRY(p, p->h_trk_qat.reserve(n_frames + 1));
        sel.d_keys = p->d_trk_keys.ptr;
        sel.d_picks = p->d_trk_picks.ptr;
        sel.d_count = p->d_trk_count.ptr;
    }
    rs::TrackMask tm{};
    if (mask) {
        CUDA_TRY(p, p->d_trk_elig.reserve((mask_per_image ? slots : 1) * plane));
        tm = rs::TrackMask{mask->mask, (int64_t)mask->pitch, (int64_t)mask->image_stride, mask->margin,
                           p->d_trk_elig.ptr};
    }
    double* d_a = p->d_trk_pts.ptr;
    double* d_b = d_a + 2 * total;
    double* d_tracked = out.tracked ? out.tracked : d_b + 2 * total;
    double* d_points = select ? (out.points ? out.points : d_b + 4 * total) : const_cast<double*>(points);
    uint8_t* d_status = out.status ? out.status : p->d_trk_status.ptr;
    int64_t* d_kept_at = p->d_trk_at.ptr;
    std::vector<int64_t> q_at(at.begin(), at.end());
    const rs::TrackImages im{static_cast<const uint8_t*>(images), (int64_t)pitch, width, height, tp.levels,
                             tp.window, tp.max_iters, (float)tp.epsilon, (float)tp.min_eig, (uint8_t)sample,
                             (uint8_t)shift};
    const rs::TrackExtra ex{select ? &sel : nullptr, fb_max, out.fb, mask ? &tm : nullptr};
    // s.d_at holds the query offsets (in selection mode the bound, overwritten on the device by the selected
    // offsets); the compacted pairs are staged at the kept offsets, which s.h_at receives
    DeviceStaging s;
    if (int rc = begin_device_staging(p, at, 4 * total, image_ts, image_ts + 1, stream, s)) return rc;
    CUDA_TRY(p, cudaMemsetAsync(p->d_trk_flag.ptr, 0, sizeof(unsigned), p->stream));
    if (out.fb && total) CUDA_TRY(p, cudaMemsetAsync(out.fb, 0xff, total * sizeof(double), p->stream));
    if (out.points && total && !select)
        CUDA_TRY(p, cudaMemcpyAsync(out.points, points, 2 * total * sizeof(double), cudaMemcpyDeviceToDevice,
                                    p->stream));
    rs::launch_track_frames(im, (int)n_frames, select ? nullptr : q_at.data(), s.d_at, d_points, p->d_trk_pyr.ptr,
                            (int)slots, d_tracked, d_status, p->d_trk_flag.ptr, ex, p->stream);
    rs::launch_track_compact(s.d_at, (int)n_frames, d_points, d_tracked, d_status, d_a, d_b, d_kept_at, p->stream);
    if (int rc = d2h(p, s.h_at, d_kept_at, (n_frames + 1) * sizeof(int64_t))) return rc;
    if (int rc = d2h(p, p->h_trk_flag.ptr, p->d_trk_flag.ptr, sizeof(unsigned))) return rc;
    if (select)
        if (int rc = d2h(p, p->h_trk_qat.ptr, s.d_at, (n_frames + 1) * sizeof(int64_t))) return rc;
    const rs::LensDev L = lens_dev(*lens);
    rs::launch_stage_points(d_kept_at, s.d_fts, (int)n_frames, (int64_t)total, d_a, d_b, L, (double)height, s.d_data,
                            s.d_info, p->stream);
    if (int rc = read_stage_info(p, n_frames, s)) return rc;
    if (*p->h_trk_flag.ptr) {
        p->err = kMsgNonFinite[kRaysA];
        return RSSYNC_E_NONFINITE;
    }
    if (out.counts)
        for (size_t i = 0; i < n_frames; ++i)
            out.counts[i] = select ? (size_t)(p->h_trk_qat.ptr[i + 1] - p->h_trk_qat.ptr[i]) : counts[i];
    for (size_t i = 0; i <= n_frames; ++i) at[i] = (size_t)s.h_at[i];
    return ingest_staged_pixels(p, n_frames, frames, at, total, image_ts, image_ts + 1, L, (double)height, s);
}

// The ex entry points (rssync_track_frames_ex_device, rssync_track_frames16_device,
// rssync_track_frames_masked_device): their null checks and default options, then track_frames
int track_frames_ex(rssync_problem* p, size_t n_frames, const int64_t* frames, const size_t* counts,
                    const double* image_ts, const double* points, const void* images, size_t pitch, int width,
                    int height, const rssync_lens* lens, const rssync_track_params* params,
                    const rssync_track_options* options, const TrackOutputs& out, void* stream, int sample,
                    int shift, const rssync_track_mask* mask = nullptr) {
    if (!p) return RSSYNC_E_INVALID;
    if (n_frames == 0) return RSSYNC_OK;
    if (!frames || !image_ts || !lens || n_frames > (size_t)INT32_MAX - 1) return RSSYNC_E_INVALID;
    if (!points != !counts) {
        p->err = "track-frames: points and counts must both be given or both be NULL";
        return RSSYNC_E_INVALID;
    }
    const rssync_track_options opt = options ? *options : rssync_track_options{128, 5, 0.01, 512, 1.0};
    return track_frames(p, n_frames, frames, counts, image_ts, points, images, pitch, width, height, lens, params,
                        &opt, out, stream, sample, shift, mask);
}

}  // namespace

extern "C" {

// rssync_set_track_pixels with the points in device memory: the check, the timestamp bounds and the
// copy into the staging buffer run on the device (stage_tracks_kernel).  As in the host form,
// everything is checked before anything is placed.
int rssync_set_track_pixels_device(rssync_problem* p, size_t n_frames, const int64_t* frames,
                                   const size_t* counts, const double* frame_ts_a, const double* frame_ts_b,
                                   const double* points_a, const double* points_b, const rssync_lens* lens,
                                   double image_rows, void* stream) {
    RS_NVTX_RANGE();
    if (!p) return RSSYNC_E_INVALID;
    if (n_frames == 0) return RSSYNC_OK;
    if (!frames || !counts || !frame_ts_a || !frame_ts_b || !lens || n_frames > (size_t)INT32_MAX)
        return RSSYNC_E_INVALID;
    std::vector<size_t> at;
    if (int rc = check_pixel_args(p, n_frames, counts, lens, image_rows, at)) return rc;
    const size_t total = at[n_frames];
    if (int rc = check_device_buffers(p, {points_a, points_b}, total)) return rc;
    if (int rc = check_frame_ts(p, n_frames, frame_ts_a, frame_ts_b)) return rc;
    DeviceStaging s;
    if (int rc = begin_device_staging(p, at, 4 * total, frame_ts_a, frame_ts_b, stream, s)) return rc;
    const rs::LensDev L = lens_dev(*lens);
    rs::launch_stage_points(s.d_at, s.d_fts, (int)n_frames, (int64_t)total, points_a, points_b, L, image_rows,
                            s.d_data, s.d_info, p->stream);
    if (int rc = read_stage_info(p, n_frames, s)) return rc;
    return ingest_staged_pixels(p, n_frames, frames, at, total, frame_ts_a, frame_ts_b, L, image_rows, s);
}

// Sparse pyramidal Lucas-Kanade from image i to image i + 1 of the caller's luma planes, then the kept
// pairs through rssync_set_track_pixels_device's ingest (ingest_staged_pixels), compacted on the device.
int rssync_track_frames_device(rssync_problem* p, size_t n_frames, const int64_t* frames, const size_t* counts,
                               const double* image_ts, const double* points, const uint8_t* images, size_t pitch,
                               int width, int height, const rssync_lens* lens, const rssync_track_params* params,
                               double* tracked_out, uint8_t* status_out, void* stream) {
    RS_NVTX_RANGE();
    if (!p) return RSSYNC_E_INVALID;
    if (n_frames == 0) return RSSYNC_OK;
    if (!frames || !counts || !image_ts || !lens || n_frames > (size_t)INT32_MAX - 1) return RSSYNC_E_INVALID;
    return track_frames(p, n_frames, frames, counts, image_ts, points, images, pitch, width, height, lens, params,
                        nullptr, TrackOutputs{nullptr, nullptr, tracked_out, status_out, nullptr}, stream);
}

// rssync_track_frames_device with the points selected on the device (points and counts NULL) and the
// forward-backward check
int rssync_track_frames_ex_device(rssync_problem* p, size_t n_frames, const int64_t* frames, const size_t* counts,
                                  const double* image_ts, const double* points, const uint8_t* images, size_t pitch,
                                  int width, int height, const rssync_lens* lens, const rssync_track_params* params,
                                  const rssync_track_options* options, double* points_out, size_t* counts_out,
                                  double* tracked_out, uint8_t* status_out, double* fb_out, void* stream) {
    RS_NVTX_RANGE();
    return track_frames_ex(p, n_frames, frames, counts, image_ts, points, images, pitch, width, height, lens, params,
                           options, TrackOutputs{points_out, counts_out, tracked_out, status_out, fb_out}, stream, 1,
                           0);
}

// rssync_track_frames_ex_device on 16-bit planes: level 0 is (float)v * 2^-shift
int rssync_track_frames16_device(rssync_problem* p, size_t n_frames, const int64_t* frames, const size_t* counts,
                                 const double* image_ts, const double* points, const uint16_t* images, size_t pitch,
                                 int width, int height, int shift, const rssync_lens* lens,
                                 const rssync_track_params* params, const rssync_track_options* options,
                                 double* points_out, size_t* counts_out, double* tracked_out, uint8_t* status_out,
                                 double* fb_out, void* stream) {
    RS_NVTX_RANGE();
    return track_frames_ex(p, n_frames, frames, counts, image_ts, points, images, pitch, width, height, lens, params,
                           options, TrackOutputs{points_out, counts_out, tracked_out, status_out, fb_out}, stream, 2,
                           shift);
}

// rssync_track_frames_ex_device (sample_bytes 1) or rssync_track_frames16_device (sample_bytes 2) with the
// caller's mask: selection takes eligible candidates only, and points kept forward off the eligible region get
// status 3 and are not ingested
int rssync_track_frames_masked_device(rssync_problem* p, size_t n_frames, const int64_t* frames, const size_t* counts,
                                      const double* image_ts, const double* points, const void* images, size_t pitch,
                                      int width, int height, int sample_bytes, int shift,
                                      const rssync_track_mask* mask, const rssync_lens* lens,
                                      const rssync_track_params* params, const rssync_track_options* options,
                                      double* points_out, size_t* counts_out, double* tracked_out,
                                      uint8_t* status_out, double* fb_out, void* stream) {
    RS_NVTX_RANGE();
    if (p && n_frames && (sample_bytes < 1 || sample_bytes > 2 || (sample_bytes == 1 && shift != 0))) {
        p->err = "track-frames: sample_bytes must be 1 or 2, and shift 0 with 1-byte samples";
        return RSSYNC_E_INVALID;
    }
    return track_frames_ex(p, n_frames, frames, counts, image_ts, points, images, pitch, width, height, lens, params,
                           options, TrackOutputs{points_out, counts_out, tracked_out, status_out, fb_out}, stream,
                           sample_bytes, shift, mask);
}

}  // extern "C"

namespace {

const char* const kMsgRowFractionsNull = "set-track-row-fractions: null argument";

// the row-fractions forms' counts and readout
int check_row_fraction_args(rssync_problem* p, size_t n_frames, const size_t* counts, double readout,
                            std::vector<size_t>& at) {
    if (int rc = frame_offsets(p, n_frames, counts, at)) return rc;
    if (!std::isfinite(readout)) {
        p->err = "set-track-row-fractions: non-finite readout";
        return RSSYNC_E_INVALID;
    }
    return RSSYNC_OK;
}

}  // namespace

extern "C" {

// SetTrackResult with the rolling-shutter timestamps formed from the caller's row fractions.  Like
// rssync_set_track_pixels: one pass on the worker pool checks every frame while it copies it into the
// pinned staging block and takes its timestamp bounds, then one upload and one ingest launch.  Staging
// block, in doubles: [records: 4 per frame][frac_a n][frac_b n][rays_a 3n][rays_b 3n], the part after the
// records in ingest_rays_kernel's layout.
int rssync_set_track_row_fractions(rssync_problem* p, size_t n_frames, const int64_t* frames, const size_t* counts,
                                   const double* frame_ts_a, const double* frame_ts_b, const double* frac_a,
                                   const double* frac_b, const double* rays_a, const double* rays_b,
                                   double readout) {
    RS_NVTX_RANGE();
    if (!p) return RSSYNC_E_INVALID;
    if (n_frames == 0) return RSSYNC_OK;
    if (!frames || !counts || !frame_ts_a || !frame_ts_b || !frac_a || !frac_b || !rays_a || !rays_b ||
        n_frames > (size_t)INT32_MAX) {
        p->err = kMsgRowFractionsNull;
        return RSSYNC_E_INVALID;
    }
    std::vector<size_t> at;
    if (int rc = check_row_fraction_args(p, n_frames, counts, readout, at)) return rc;
    const size_t total = at[n_frames];
    if (int rc = check_frame_ts(p, n_frames, frame_ts_a, frame_ts_b)) return rc;
    if (int rc = begin_ingest(p)) return rc;
    const size_t block = 4 * n_frames + 8 * total;
    CUDA_TRY(p, p->h_stage.reserve(block + 1));
    double* h_fa = p->h_stage.ptr + 4 * n_frames;
    double* h_fb = h_fa + total;
    double* h_ra = h_fb + total;
    double* h_rb = h_ra + 3 * total;
    std::vector<rs::StageInfo> info(n_frames);
    parallel_frames(n_frames, [&](size_t i, size_t) {
        const size_t a0 = at[i], n = counts[i];
        const bool ok_ra = copy_checked(h_ra + 3 * a0, rays_a + 3 * a0, 3 * n, nullptr, nullptr);
        const bool ok_rb = copy_checked(h_rb + 3 * a0, rays_b + 3 * a0, 3 * n, nullptr, nullptr);
        const double fa = frame_ts_a[i], fb = frame_ts_b[i];
        bool ok_ta = true, ok_tb = true;
        double l = 0.0, h = 0.0;
        for (size_t k = 0; k < n; ++k) {
            const double qa = frac_a[a0 + k], qb = frac_b[a0 + k];
            h_fa[a0 + k] = qa;
            h_fb[a0 + k] = qb;
            // ingest_rays_kernel's expression (host code is built without contraction); a non-finite q
            // gives a non-finite timestamp, since the readout is finite
            const double ta = fa + readout * qa, tb = fb + readout * qb;
            ok_ta = ok_ta && std::isfinite(ta);
            ok_tb = ok_tb && std::isfinite(tb);
            if (k == 0) l = h = ta;
            l = ta < l ? ta : l;
            h = ta > h ? ta : h;
            l = tb < l ? tb : l;
            h = tb > h ? tb : h;
        }
        // bit b: source buffer b (kRaysA .. kTsB) holds a non-finite value, as StageInfo::bad
        const unsigned bad = (!ok_ra << kRaysA) | (!ok_rb << kRaysB) | (!ok_ta << kTsA) | (!ok_tb << kTsB);
        info[i] = rs::StageInfo{bad, 0u, l, h};
    });
    if (const size_t i = first_bad(info.data(), n_frames); i < n_frames) return fail_nonfinite(p, info[i]);
    rs::PixelFrame* rec = reinterpret_cast<rs::PixelFrame*>(p->h_stage.ptr);
    size_t k = 0;
    if (int rc = place_frames(p, n_frames, frames, at, info.data(), frame_ts_a, frame_ts_b, rec, k)) return rc;
    CUDA_TRY(p, p->d_stage.reserve(block + 1));
    if (int rc = h2d(p, p->d_stage.ptr, p->h_stage.ptr, block * sizeof(double))) return rc;
    const double* d_fa = p->d_stage.ptr + 4 * n_frames;
    rs::launch_ingest_row_fractions(reinterpret_cast<const rs::PixelFrame*>(p->d_stage.ptr), (int)k, d_fa,
                                    d_fa + total, d_fa + 2 * total, d_fa + 5 * total, readout, p->d_rays.ptr,
                                    p->d_orig.ptr, p->d_pos.ptr, p->d_rowq.ptr, p->stream);
    return end_device_ingest(p);
}

// rssync_set_track_row_fractions with the per-ray buffers in device memory: the check, the timestamp
// bounds and the copy into the staging buffer run on the device (stage_tracks_kernel); as in the host
// form, everything is checked before anything is placed.
int rssync_set_track_row_fractions_device(rssync_problem* p, size_t n_frames, const int64_t* frames,
                                          const size_t* counts, const double* frame_ts_a, const double* frame_ts_b,
                                          const double* frac_a, const double* frac_b, const double* rays_a,
                                          const double* rays_b, double readout, void* stream) {
    RS_NVTX_RANGE();
    if (!p) return RSSYNC_E_INVALID;
    if (n_frames == 0) return RSSYNC_OK;
    if (!frames || !counts || !frame_ts_a || !frame_ts_b || n_frames > (size_t)INT32_MAX) {
        p->err = kMsgRowFractionsNull;
        return RSSYNC_E_INVALID;
    }
    std::vector<size_t> at;
    if (int rc = check_row_fraction_args(p, n_frames, counts, readout, at)) return rc;
    const size_t total = at[n_frames];
    if (int rc = check_device_buffers(p, {frac_a, frac_b, rays_a, rays_b}, total)) return rc;
    if (int rc = check_frame_ts(p, n_frames, frame_ts_a, frame_ts_b)) return rc;
    DeviceStaging s;
    if (int rc = begin_device_staging(p, at, 8 * total, frame_ts_a, frame_ts_b, stream, s)) return rc;
    rs::launch_stage_row_fractions(s.d_at, s.d_fts, (int)n_frames, (int64_t)total, rays_a, rays_b, frac_a, frac_b,
                                   readout, s.d_data, s.d_info, p->stream);
    if (int rc = read_stage_info(p, n_frames, s)) return rc;
    if (const size_t i = first_bad(s.h_info, n_frames); i < n_frames) return fail_nonfinite(p, s.h_info[i]);
    size_t k = 0;
    if (int rc = place_frames(p, n_frames, frames, at, s.h_info, frame_ts_a, frame_ts_b, s.h_rec, k)) return rc;
    if (int rc = h2d(p, s.d_rec, s.h_rec, k * sizeof(rs::PixelFrame))) return rc;
    rs::launch_ingest_row_fractions(s.d_rec, (int)k, s.d_data, s.d_data + total, s.d_data + 2 * total,
                                    s.d_data + 5 * total, readout, p->d_rays.ptr, p->d_orig.ptr, p->d_pos.ptr,
                                    p->d_rowq.ptr, p->stream);
    return end_device_ingest(p);
}

int rssync_set_kernel_timing(rssync_problem* p, int enabled) {
    if (!p) return RSSYNC_E_INVALID;
    if (enabled && !p->ev0) {
        CUDA_TRY(p, cudaSetDevice(p->device));
        CUDA_TRY(p, cudaEventCreate(&p->ev0));
        CUDA_TRY(p, cudaEventCreate(&p->ev1));
    }
    p->kernel_timing = enabled != 0;
    return RSSYNC_OK;
}

int rssync_presync_delays(double initial, double step, double radius, double* out, int cap) {
    int n = 0;
    for (double d = initial - radius; d < initial + radius; d += step) {  // core_private.cpp:69-70
        if (out && n < cap) out[n] = d;
        if (++n > (1 << 28)) break;
    }
    return n;
}

int rssync_presync(rssync_problem* p, double initial, int64_t fb, int64_t fe, double step,
                   double radius, double* out_cost, double* out_delay) {
    RS_NVTX_RANGE();
    if (!p || !out_cost || !out_delay) return RSSYNC_E_INVALID;
    std::vector<double> delays;
    if (int rc = presync_delay_grid(p, initial, step, radius, delays)) return rc;
    const int n = (int)delays.size();
    std::vector<double> costs((size_t)n);
    const uint64_t call = p->call_no++;
    unsigned flags = 0;
    if (int rc = presync_grid_impl(p, fb, fe, delays.data(), n, rs::kStreamPreSync, call, 0, costs.data(), &flags))
        return rc;
    if (flags) { p->err = presync_panic_text(flags); return RSSYNC_E_NONFINITE; }
    curve_argmin(costs.data(), delays.data(), n, out_cost, out_delay);
    return RSSYNC_OK;
}

// n PreSync calls over n frame windows with one shared delay grid, evaluated as ONE grid launch
// (the syncpoint loop of core_testcode.cpp:303-312 issues them one by one).  Result i equals the
// i-th of n consecutive rssync_presync calls; call_nos (or the problem's counter) key the RNG.
int rssync_presync_windows(rssync_problem* p, int n, double initial, const int64_t* fb, const int64_t* fe,
                           double step, double radius, const uint64_t* call_nos, double* out_cost,
                           double* out_delay) {
    RS_NVTX_RANGE();
    if (!p || n < 0) return RSSYNC_E_INVALID;
    if (n == 0) return RSSYNC_OK;
    if (!fb || !fe || !out_cost || !out_delay) return RSSYNC_E_INVALID;
    if (int rc = require_gyro(p, "pre-sync")) return rc;
    std::vector<double> delays;
    if (int rc = presync_delay_grid(p, initial, step, radius, delays)) return rc;
    const int D = (int)delays.size();
    const std::vector<uint64_t> calls = call_numbers(p, call_nos, n);
    if (is_multi(p) && n > 1) {  // windows are independent: shard them, explicit call numbers
        if (int rc = multi_replicate(p)) return rc;
        if (!call_nos) p->call_no += (uint64_t)n;
        return multi_for_each_shard(p, n, false, [&](rssync_problem* q, int lo, int cnt) {
            return rssync_presync_windows(q, cnt, initial, fb + lo, fe + lo, step, radius, calls.data() + lo,
                                          out_cost + lo, out_delay + lo);
        });
    }
    std::vector<FrameDesc> all, sel;
    std::vector<uint64_t> fcall;
    std::vector<int> wbeg(n + 1, 0);
    int max_n = 0;
    for (int i = 0; i < n; ++i) {
        int mn = 0;
        if (int rc = select_frames(p, fb[i], fe[i], sel, mn, "pre-sync")) return rc;
        max_n = std::max(max_n, mn);
        for (const FrameDesc& fd : sel) { all.push_back(fd); fcall.push_back(calls[(size_t)i]); }
        wbeg[i + 1] = (int)all.size();
    }
    if (!call_nos) p->call_no += (uint64_t)n;
    if (int rc = flush(p)) return rc;
    const int F = (int)all.size();
    std::vector<double> costs((size_t)n * D, 0.0);
    unsigned flags[2] = {0, 0};
    if (F > 0) {
        if (int rc = check_grid_size(p, F, D)) return rc;
        const int max_chunk = grid_max_chunk(all.data(), F, delays.data(), D, p->sr, max_n);
        if (int rc = stage_grid(p, all.data(), all.size(), F, delays.data(), D, n)) return rc;
        CUDA_TRY(p, p->d_frame_call.reserve(F));
        CUDA_TRY(p, p->d_win_begin.reserve(n + 1));
        if (int rc = h2d(p, p->d_frame_call.ptr, fcall.data(), sizeof(uint64_t) * F)) return rc;
        if (int rc = h2d(p, p->d_win_begin.ptr, wbeg.data(), sizeof(int) * (n + 1))) return rc;
        rs::launch_presync_grid(p->device_data(), p->d_frames.ptr, F, max_n, p->d_delays.ptr, D, p->seed,
                                rs::kStreamPreSync, 0, 0, p->d_framecost.ptr, p->d_costs.ptr, p->d_flags.ptr,
                                p->stream, max_chunk, p->simplified, p->d_frame_call.ptr, p->d_win_begin.ptr, n);
        if (int rc = d2h(p, costs.data(), p->d_costs.ptr, sizeof(double) * n * D)) return rc;
        if (int rc = d2h(p, flags, p->d_flags.ptr, 2 * sizeof(unsigned))) return rc;
        if (int rc = finish_stream(p, p->stream)) return rc;
        p->grid_tasks = (uint64_t)F * (uint64_t)D;
        p->grid_exact_tasks = flags[1];
    }
    if (flags[0]) { p->err = presync_panic_text(flags[0]); return RSSYNC_E_NONFINITE; }
    for (int i = 0; i < n; ++i) curve_argmin(&costs[(size_t)i * D], delays.data(), D, &out_cost[i], &out_delay[i]);
    return RSSYNC_OK;
}

int rssync_debug_presync(rssync_problem* p, double initial, int64_t fb, int64_t fe, double radius,
                         double* delays, double* costs, int point_count) {
    RS_NVTX_RANGE();
    if (!p || (point_count > 0 && (!delays || !costs))) return RSSYNC_E_INVALID;
    if (point_count <= 0) return RSSYNC_OK;
    for (int i = 0; i < point_count; ++i)
        delays[i] = initial - radius + 2 * radius * i / (point_count - 1);  // core_private.cpp:345
    const uint64_t call = p->call_no++;
    return presync_grid_impl(p, fb, fe, delays, point_count, rs::kStreamDebugPreSync, call, 0, costs, nullptr);
}

int rssync_presync_grid(rssync_problem* p, int64_t fb, int64_t fe, const double* delays, int n,
                        int stream, uint64_t call_no, uint64_t idx_base, double* costs,
                        unsigned* nonfinite_flags) {
    RS_NVTX_RANGE();
    if (!p || (n > 0 && (!delays || !costs))) return RSSYNC_E_INVALID;
    return presync_grid_impl(p, fb, fe, delays, n, (uint64_t)stream, call_no, idx_base, costs, nonfinite_flags);
}

int rssync_integrate_gyro(const double* timestamps_s, const double* gyro_xyz, size_t count,
                          const char* orientation, double* quats_out) {
    if (count && (!timestamps_s || !gyro_xyz || !quats_out)) return RSSYNC_E_INVALID;
    double m[9];
    if (!rs::parse_orientation(orientation, m)) return RSSYNC_E_INVALID;
    rs::integrate_gyro(timestamps_s, gyro_xyz, count, m, quats_out);
    return RSSYNC_OK;
}

int rssync_integrate_gyro_matrix(const double* timestamps_s, const double* gyro_xyz, size_t count,
                                 const double* matrix, double* quats_out) {
    if (count && (!timestamps_s || !gyro_xyz || !quats_out)) return RSSYNC_E_INVALID;
    double m[9] = {1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0};
    if (matrix) std::memcpy(m, matrix, sizeof(m));
    if (!all_finite(m, 9)) return RSSYNC_E_INVALID;
    rs::integrate_gyro(timestamps_s, gyro_xyz, count, m, quats_out);
    return RSSYNC_OK;
}

}  // extern "C"

namespace {

// The frame windows of a windowed search (W >= 1): every window's frames, concatenated in window order
// (a frame in several windows appears once per window), the window starts into that list, and the
// largest frame.  All windows are checked, in window order, before anything runs; `check` (optional)
// is a search's own check of a window's frames.
struct SearchWindows {
    std::vector<FrameDesc> frames;
    std::vector<int> begin;  // W + 1 offsets into frames
    int max_n = 0;

    int select(rssync_problem* p, int W, const int64_t* fb, const int64_t* fe,
               const std::function<int(const std::vector<FrameDesc>&)>& check = nullptr) {
        frames.clear();
        begin.assign(1, 0);
        std::vector<FrameDesc> sel;
        for (int w = 0; w < W; ++w) {
            int mn = 0;
            if (int rc = select_frames(p, fb[w], fe[w], sel, mn, "pre-sync")) return rc;
            if (check)
                if (int rc = check(sel)) return rc;
            max_n = std::max(max_n, mn);
            frames.insert(frames.end(), sel.begin(), sel.end());
            begin.push_back((int)frames.size());
        }
        return RSSYNC_OK;
    }
    int F() const { return (int)frames.size(); }
    int W() const { return (int)begin.size() - 1; }

    // the RNG call number of every listed frame for candidate j: calls[j W + its window]
    std::vector<uint64_t> frame_calls(const std::vector<uint64_t>& calls, int n) const {
        std::vector<uint64_t> fc((size_t)n * F());
        for (int j = 0; j < n; ++j)
            for (int w = 0; w < W(); ++w)
                for (int f = begin[(size_t)w]; f < begin[(size_t)w + 1]; ++f)
                    fc[(size_t)j * F() + f] = calls[(size_t)j * W() + w];
        return fc;
    }
};

// Checks shared by the windowed searches: counts and window buffers.  `who` names the search.
int check_search_counts(rssync_problem* p, int n, int W, const int64_t* fb, const int64_t* fe, const char* who) {
    if (n < 0 || W < 0) { p->err = std::string(who) + ": negative candidate or window count"; return RSSYNC_E_INVALID; }
    if ((long long)n * W > INT32_MAX) { p->err = std::string(who) + ": too many candidate windows"; return RSSYNC_E_INVALID; }
    if (n > 0 && W > 0 && (!fb || !fe)) { p->err = std::string(who) + ": null window buffer"; return RSSYNC_E_INVALID; }
    return RSSYNC_OK;
}

// For candidate grids with more than one window: the per-frame call numbers of all n candidates and the
// window starts, on the device (rssync_presync_windows' arrays).  One window needs neither.
int stage_windows(rssync_problem* p, const SearchWindows& win, const std::vector<uint64_t>& calls, int n) {
    if (win.W() == 1 || win.F() == 0) return RSSYNC_OK;
    const std::vector<uint64_t> fcall = win.frame_calls(calls, n);
    CUDA_TRY(p, p->d_frame_call.reserve(fcall.size()));
    CUDA_TRY(p, p->d_win_begin.reserve(win.begin.size()));
    if (int rc = h2d(p, p->d_frame_call.ptr, fcall.data(), sizeof(uint64_t) * fcall.size())) return rc;
    return h2d(p, p->d_win_begin.ptr, win.begin.data(), sizeof(int) * win.begin.size());
}

// candidate j's grid over the windows: one window is a plain grid, several are rssync_presync_windows'
// multi-window grid with the per-frame call numbers staged by stage_windows
void launch_candidate_grid(rssync_problem* p, const rs::DeviceData& dd, const SearchWindows& win, int j,
                           const FrameDesc* d_frames, const double* d_delays, int D, uint64_t call, int max_chunk,
                           cudaStream_t st) {
    const int F = win.F(), W = win.W();
    rs::launch_presync_grid(dd, d_frames, F, win.max_n, d_delays, D, p->seed, rs::kStreamPreSync, call, 0,
                            p->d_framecost.ptr, p->d_costs.ptr + (size_t)j * W * D, p->d_flags.ptr + 2 * (size_t)j, st,
                            max_chunk, p->simplified, W > 1 ? p->d_frame_call.ptr + (size_t)j * F : nullptr,
                            W > 1 ? p->d_win_begin.ptr : nullptr, W);
}

// candidate j's W results from the curves (n x W x D)
void candidate_results(int j, int W, const std::vector<double>& costs, const std::vector<double>& delays,
                       double* out_cost, double* out_delay, double* out_curves) {
    const int D = (int)delays.size();
    for (int w = 0; w < W; ++w) {
        const size_t r = (size_t)j * W + w;
        curve_argmin(&costs[r * D], delays.data(), D, &out_cost[r], &out_delay[r]);
        if (out_curves) std::memcpy(out_curves + r * D, &costs[r * D], sizeof(double) * D);
    }
}

// The axis mappings of a gyro-variant search: gyro_orientation strings (the orientation search) or 3x3
// row-major matrices (the rotation search).  The search turns either into matrices at the same step.
struct GyroVariants {
    const char* const* strings;
    const double* matrices;

    GyroVariants from(int lo) const {
        return {strings ? strings + lo : nullptr, matrices ? matrices + 9 * (size_t)lo : nullptr};
    }
    int to_matrices(rssync_problem* p, int n, std::vector<double>& m) const {
        m.resize((size_t)n * 9);
        if (!strings) {
            std::copy(matrices, matrices + (size_t)n * 9, m.begin());
            return RSSYNC_OK;
        }
        for (int k = 0; k < n; ++k)
            if (!rs::parse_orientation(strings[k], &m[(size_t)k * 9])) {
                p->err = std::string("orientation-search: malformed gyro_orientation '") +
                         (strings[k] ? strings[k] : "(null)") + "'";
                return RSSYNC_E_INVALID;
            }
        return RSSYNC_OK;
    }
};

// The orientation search of core_testcode.cpp:184-233, for any axis mappings: for every variant,
// integrate the raw gyro (optdata_fill_gyro, :37-53) under its mapping, ingest it through the
// variable-rate SetGyroQuaternions and run PreSync over each of the W frame windows [fb[w], fe[w]) -- one
// loss grid per variant over all windows.  Results are n x W, variant-major; out_curves (n x W x D or
// null): every variant's cost curve per window.
int gyro_variant_search(rssync_problem* p, const double* timestamps_s, const double* gyro_xyz, size_t count,
                        const GyroVariants& variants, int n_orient, double initial_delay, int W, const int64_t* fb,
                        const int64_t* fe, double step, double radius, const uint64_t* call_nos, double* out_cost,
                        double* out_delay, double* out_curves) {
    if (!p || n_orient < 0) return RSSYNC_E_INVALID;
    if (int rc = check_search_counts(p, n_orient, W, fb, fe, "rotation-search")) return rc;
    if (n_orient == 0 || W == 0) return RSSYNC_OK;
    if (!timestamps_s || !gyro_xyz || (!variants.strings && !variants.matrices) || !out_cost || !out_delay)
        return RSSYNC_E_INVALID;
    const int nw = n_orient * W;
    if (is_multi(p) && n_orient > 1) {
        // variants are independent: shard them.  Every device sets its own gyro per variant, so the
        // replicas' inputs are stale afterwards; the primary takes the LAST share, which leaves it
        // holding the last variant's gyro as the single-device search does.
        if (int rc = multi_replicate(p)) return rc;
        const std::vector<uint64_t> callno = call_numbers(p, call_nos, nw);
        // curve rows per variant and window (a window the shards reject leaves no curves to place)
        const size_t D = out_curves && step > 0 && std::isfinite(initial_delay) && std::isfinite(radius)
                             ? (size_t)std::max(0, rssync_presync_delays(initial_delay, step, radius, nullptr, 0))
                             : 0;
        const int rc = multi_for_each_shard(p, n_orient, true, [&](rssync_problem* q, int lo, int cnt) {
            const size_t r = (size_t)lo * W;
            return gyro_variant_search(q, timestamps_s, gyro_xyz, count, variants.from(lo), cnt, initial_delay, W,
                                       fb, fe, step, radius, callno.data() + r, out_cost + r, out_delay + r,
                                       out_curves ? out_curves + r * D : nullptr);
        });
        if (!call_nos) p->call_no += (uint64_t)nw;
        for (rssync_problem* r : p->replicas) r->synced_version = ~0ull;
        return rc;
    }
    // Single device.  Everything per variant runs on the device: integration (blocked scan),
    // resampling onto the uniform grid, the spline system's sweeps, the record build, the loss grid.
    // The host prepares what does not depend on the variant -- the microsecond timestamps
    // (core_testcode.cpp:47-50), the resampling plan, the frame table, the delay grid -- queues the whole
    // search and reads all curves back at the end.
    if (count < 2 || count > (size_t)INT32_MAX) { p->err = "set-gyro-quaternions: need at least 2 samples"; return RSSYNC_E_INVALID; }
    if (int rc = check_search_window(p, initial_delay, step, radius)) return rc;
    std::vector<double> mats;
    if (int rc = variants.to_matrices(p, n_orient, mats)) return rc;
    std::vector<int64_t> ts_us(count);
    for (size_t i = 0; i < count; ++i) ts_us[i] = (int64_t)(timestamps_s[i] * 1000000);  // :47-50
    rs::ResamplePlan plan;
    {
        const rs::IngestStatus st = rs::plan_variable_rate(ts_us.data(), count, plan, p->err);
        if (st != rs::IngestStatus::Ok)
            return st == rs::IngestStatus::NonFinite ? RSSYNC_E_NONFINITE
                   : st == rs::IngestStatus::OutOfOrder ? RSSYNC_E_ORDER : RSSYNC_E_INVALID;
    }
    std::vector<double> delays;
    if (int rc = presync_delay_grid(p, initial_delay, step, radius, delays)) return rc;
    const int D = (int)delays.size();
    SearchWindows win;
    if (int rc = win.select(p, W, fb, fe)) return rc;
    const int F = win.F();
    if (int rc = check_grid_size(p, F, D)) return rc;
    const std::vector<uint64_t> calls = call_numbers(p, call_nos, nw);
    join_gyro(p);
    if (int rc = flush(p)) return rc;  // the tracks, and whatever gyro was pending
    cudaSetDevice(p->device);
    cudaStream_t st = p->stream;
    // the variants' spline records overwrite the problem's own: not before a replication still reading them
    if (p->reader_pending) CUDA_TRY(p, cudaStreamWaitEvent(st, p->ev_reader, 0));
    const size_t nq = plan.n_out, n = count;
    // variants per pass: bounded by ~2 GB of intermediates
    const size_t per_var = (n * 4 + nq * (4 + 4 + 16)) * sizeof(double);
    const int G = (int)std::max<size_t>(1, std::min<size_t>((size_t)n_orient, (size_t(2) << 30) / std::max<size_t>(per_var, 1)));
    CUDA_TRY(p, p->d_var_ts.reserve(n));
    CUDA_TRY(p, p->d_var_in.reserve(n * 4));  // timestamps (n) and raw gyro (3 n), seconds / rad/s
    CUDA_TRY(p, p->d_var_q.reserve((size_t)G * n * 4));
    CUDA_TRY(p, p->d_var_y.reserve((size_t)G * nq * 4));
    CUDA_TRY(p, p->d_var_rhs.reserve((size_t)G * nq * 4));
    CUDA_TRY(p, p->d_var_rec.reserve((size_t)G * nq * 16));
    CUDA_TRY(p, p->d_var_prefix.reserve(rs::gyro_prefix_doubles((int)n, G)));
    CUDA_TRY(p, p->d_var_orients.reserve(rs::gyro_orient_bytes(G)));
    CUDA_TRY(p, p->d_var_flags.reserve((size_t)n_orient));
    CUDA_TRY(p, cudaMemcpyAsync(p->d_var_ts.ptr, ts_us.data(), n * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    CUDA_TRY(p, cudaMemcpyAsync(p->d_var_in.ptr, timestamps_s, n * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(p, cudaMemcpyAsync(p->d_var_in.ptr + n, gyro_xyz, 3 * n * sizeof(double), cudaMemcpyHostToDevice, st));
    CUDA_TRY(p, cudaMemsetAsync(p->d_var_flags.ptr, 0, (size_t)n_orient * sizeof(unsigned), st));
    p->h2d += n * (sizeof(int64_t) + 4 * sizeof(double));
    if (int rc = stage_grid(p, win.frames.data(), win.frames.size(), F, delays.data(), D, nw)) return rc;
    if (int rc = stage_windows(p, win, calls, n_orient)) return rc;
    if (int rc = upload_elimination(p, nq, st)) return rc;
    const int max_chunk = grid_max_chunk(win.frames.data(), F, delays.data(), D, plan.sample_rate, win.max_n);
    rs::DeviceData dd = p->device_data();
    dd.nq = (int)nq;
    dd.q0 = plan.first_timestamp;
    dd.sr = plan.sample_rate;
    for (int k0 = 0; k0 < n_orient; k0 += G) {
        const int g = std::min(G, n_orient - k0);
        rs::launch_gyro_integrate(p->d_var_in.ptr, p->d_var_in.ptr + n, (int)n, &mats[(size_t)k0 * 9], g, p->d_var_orients.ptr,
                                  p->d_var_q.ptr, p->d_var_prefix.ptr, st);
        rs::launch_gyro_resample(p->d_var_ts.ptr, (int)n, p->d_var_q.ptr, g, plan.tick0, plan.rate_hz, (int)nq,
                                 p->d_var_y.ptr, p->d_var_flags.ptr + k0, st);
        rs::launch_spline_chains(p->d_var_y.ptr, p->d_elim.ptr, p->d_elim.ptr + nq, (int)nq, g, p->d_var_rhs.ptr, st);
        for (int v = 0; v < g; ++v) {
            double* rec = p->d_var_rec.ptr + (size_t)v * nq * 16;
            rs::launch_spline_finish(p->d_var_y.ptr + (size_t)v * nq * 4, p->d_var_rhs.ptr + (size_t)v * nq * 4,
                                     p->d_elim.ptr + 2 * nq, (int)nq, rec, st);
            if (F > 0) {
                dd.rec = rec;
                launch_candidate_grid(p, dd, win, k0 + v, p->d_frames.ptr, p->d_delays.ptr, D,
                                      calls[(size_t)(k0 + v) * W], max_chunk, st);
            }
        }
        CUDA_TRY(p, cudaGetLastError());
        if (k0 + g >= n_orient) {  // the problem is left holding the last variant's gyro
            CUDA_TRY(p, p->d_rec.reserve(nq * 16));
            CUDA_TRY(p, cudaMemcpyAsync(p->d_rec.ptr, p->d_var_rec.ptr + (size_t)(g - 1) * nq * 16, nq * 16 * sizeof(double),
                                        cudaMemcpyDeviceToDevice, st));
        }
    }
    std::vector<double> costs((size_t)nw * D, 0.0);
    std::vector<unsigned> resampled((size_t)n_orient, 0u), flags((size_t)n_orient * 2, 0u);
    if (F > 0)
        if (int rc = d2h(p, costs.data(), p->d_costs.ptr, costs.size() * sizeof(double))) return rc;
    if (int rc = d2h(p, resampled.data(), p->d_var_flags.ptr, resampled.size() * sizeof(unsigned))) return rc;
    if (int rc = d2h(p, flags.data(), p->d_flags.ptr, flags.size() * sizeof(unsigned))) return rc;
    if (int rc = finish_stream(p, st)) return rc;
    p->version++;
    p->sr = plan.sample_rate;
    p->q0 = plan.first_timestamp;
    p->nq = nq;
    p->gyro_dirty = false;
    if (!call_nos) p->call_no += (uint64_t)nw;
    p->grid_tasks = (uint64_t)F * (uint64_t)D;
    for (int k = 0; k < n_orient; ++k) {
        if (resampled[(size_t)k]) { p->err = "set-gyro-quaternions: non-finite sample after interpolation"; return RSSYNC_E_NONFINITE; }
        if (const unsigned fl = flags[2 * (size_t)k]) { p->err = presync_panic_text(fl); return RSSYNC_E_NONFINITE; }
        candidate_results(k, W, costs, delays, out_cost, out_delay, out_curves);
    }
    return RSSYNC_OK;
}

}  // namespace

extern "C" {

// The orientation search of core_testcode.cpp:184-233 over gyro_orientation strings.  The per-variant work
// (integration, resampling, spline elimination, records) and the loss grids run back to back on the device.
int rssync_orientation_search(rssync_problem* p, const double* timestamps_s, const double* gyro_xyz,
                              size_t count, const char* const* orientations, int n_orient,
                              double initial_delay, int64_t fb, int64_t fe, double step, double radius,
                              double* out_cost, double* out_delay) {
    return rssync_orientation_search_ex(p, timestamps_s, gyro_xyz, count, orientations, n_orient, initial_delay,
                                        fb, fe, step, radius, nullptr, out_cost, out_delay);
}

int rssync_orientation_search_ex(rssync_problem* p, const double* timestamps_s, const double* gyro_xyz,
                                 size_t count, const char* const* orientations, int n_orient,
                                 double initial_delay, int64_t fb, int64_t fe, double step, double radius,
                                 const uint64_t* call_nos, double* out_cost, double* out_delay) {
    RS_NVTX_RANGE();
    return gyro_variant_search(p, timestamps_s, gyro_xyz, count, GyroVariants{orientations, nullptr}, n_orient,
                               initial_delay, 1, &fb, &fe, step, radius, call_nos, out_cost, out_delay, nullptr);
}

}  // extern "C"

namespace {

// The rotation search over W windows (W = 1: rssync_rotation_search)
int rotation_search_impl(rssync_problem* p, const double* timestamps_s, const double* gyro_xyz, size_t count,
                         const double* matrices, int n_rot, int W, const int64_t* fb, const int64_t* fe,
                         double initial_delay, double step, double radius, const uint64_t* call_nos,
                         double* out_cost, double* out_delay, double* out_curves) {
    if (!p || n_rot < 0) return RSSYNC_E_INVALID;
    if (int rc = check_search_counts(p, n_rot, W, fb, fe, "rotation-search")) return rc;
    if (n_rot == 0 || W == 0) return RSSYNC_OK;
    if (!matrices) return RSSYNC_E_INVALID;
    for (int i = 0; i < n_rot; ++i)
        if (!all_finite(matrices + (size_t)i * 9, 9)) {
            p->err = "rotation-search: matrix " + std::to_string(i) + " has a non-finite entry";
            return RSSYNC_E_INVALID;
        }
    return gyro_variant_search(p, timestamps_s, gyro_xyz, count, GyroVariants{nullptr, matrices}, n_rot,
                               initial_delay, W, fb, fe, step, radius, call_nos, out_cost, out_delay, out_curves);
}

}  // namespace

extern "C" {

// The same search over arbitrary 3x3 gyro axis mappings, e.g. candidate camera mount rotations
int rssync_rotation_search(rssync_problem* p, const double* timestamps_s, const double* gyro_xyz, size_t count,
                           const double* matrices, int n_rot, double initial_delay, int64_t fb, int64_t fe,
                           double step, double radius, const uint64_t* call_nos, double* out_cost,
                           double* out_delay, double* out_curves) {
    RS_NVTX_RANGE();
    return rotation_search_impl(p, timestamps_s, gyro_xyz, count, matrices, n_rot, 1, &fb, &fe, initial_delay, step,
                                radius, call_nos, out_cost, out_delay, out_curves);
}

int rssync_rotation_search_windows(rssync_problem* p, const double* timestamps_s, const double* gyro_xyz,
                                   size_t count, const double* matrices, int n_rot, int n_windows,
                                   const int64_t* fb, const int64_t* fe, double initial_delay, double step,
                                   double radius, const uint64_t* call_nos, double* out_cost, double* out_delay,
                                   double* out_curves) {
    RS_NVTX_RANGE();
    return rotation_search_impl(p, timestamps_s, gyro_xyz, count, matrices, n_rot, n_windows, fb, fe, initial_delay,
                                step, radius, call_nos, out_cost, out_delay, out_curves);
}

}  // extern "C"

namespace {

int check_readouts(rssync_problem* p, const double* readouts, int n, const char* who) {
    if (!all_finite(readouts, (size_t)n)) {
        p->err = std::string(who) + ": readout must be finite";
        return RSSYNC_E_INVALID;
    }
    return RSSYNC_OK;
}

// every frame of `sel` can be re-timed: it was ingested from pixels or row fractions and not overwritten since
int require_retime(rssync_problem* p, const std::vector<FrameDesc>& sel, const char* who) {
    for (const FrameDesc& fd : sel)
        if (!p->retime.count(fd.id)) {
            p->err = std::string(who) + ": frame " + std::to_string(fd.id) +
                     " has no row fractions to re-time (it was not ingested by a pixels or row-fractions form,"
                     " or was overwritten or adopted since)";
            return RSSYNC_E_STATE;
        }
    return RSSYNC_OK;
}

// The re-timing records of `sel`: source offset and frame timestamps, destination offset `dst[f]`
std::vector<rs::PixelFrame> retime_records(const rssync_problem* p, const std::vector<FrameDesc>& sel,
                                           const std::vector<int32_t>& dst) {
    std::vector<rs::PixelFrame> rec(sel.size());
    for (size_t f = 0; f < sel.size(); ++f) {
        const std::pair<double, double>& ts = p->retime.at(sel[f].id);
        rec[f] = rs::PixelFrame{dst[f], sel[f].n, (int64_t)sel[f].off, ts.first, ts.second};
    }
    return rec;
}

// A frame's timestamp bounds at readout r from its row-fraction extremes e = {min q_a, max q_a, min q_b,
// max q_b}.  fl(ts + fl(r q)) is monotone in q -- non-decreasing for r >= 0, non-increasing for r < 0 --
// so the smallest and largest timestamps are among the four ends, and these are the values a re-ingest's
// bounds (the min / max over every ray) take.
void retimed_bounds(const rs::PixelFrame& f, const double* e, double r, double& lo, double& hi) {
    if (f.n == 0) { lo = hi = 0.0; return; }
    const double a0 = f.ts_a + r * e[0], a1 = f.ts_a + r * e[1];
    const double b0 = f.ts_b + r * e[2], b1 = f.ts_b + r * e[3];
    lo = std::min(std::min(a0, a1), std::min(b0, b1));
    hi = std::max(std::max(a0, a1), std::max(b0, b1));
}

// PreSync at n rolling-shutter readouts over W frame windows without re-ingesting: the union of the
// windows' frames is re-timed into a scratch arena (retime_frames_kernel) and one loss grid over all
// windows runs on it, per readout, back to back on the problem's stream; one read-back at the end.  The
// problem's own arena, frame table and gyro are not touched.  A multi-device problem shards the readouts
// over its devices, as the orientation search does its variants.
int readout_search_impl(rssync_problem* p, const double* readouts, int n, int W, const int64_t* fb,
                        const int64_t* fe, double initial, double step, double radius, const uint64_t* call_nos,
                        double* out_cost, double* out_delay, double* out_curves) {
    if (!p) return RSSYNC_E_INVALID;
    if (int rc = check_search_counts(p, n, W, fb, fe, "readout-search")) return rc;
    if (n == 0 || W == 0) return RSSYNC_OK;
    if (!readouts || !out_cost || !out_delay) { p->err = "readout-search: null buffer"; return RSSYNC_E_INVALID; }
    if (int rc = check_readouts(p, readouts, n, "readout-search")) return rc;
    if (int rc = require_gyro(p, "pre-sync")) return rc;
    std::vector<double> delays;
    if (int rc = presync_delay_grid(p, initial, step, radius, delays)) return rc;
    const int D = (int)delays.size();
    SearchWindows win;
    if (int rc = win.select(p, W, fb, fe, [p](const std::vector<FrameDesc>& sel) {
            return require_retime(p, sel, "readout-search");
        }))
        return rc;
    const int F = win.F(), nw = n * W;
    if (int rc = check_grid_size(p, F, D)) return rc;
    const std::vector<uint64_t> calls = call_numbers(p, call_nos, nw);
    if (!call_nos) p->call_no += (uint64_t)nw;
    if (is_multi(p) && n > 1) {
        // readouts are independent: shard them, explicit call numbers.  Every device re-times into its
        // own scratch arena and leaves its inputs alone, so no replica is stale afterwards.  Rank order
        // is readout order: of several failing readouts, the first one's error is reported.
        if (int rc = multi_replicate(p)) return rc;
        if (int rc = multi_replicate_row_fractions(p)) return rc;
        const int rc = multi_for_each_shard(p, n, false, [&](rssync_problem* q, int lo, int cnt) {
            const size_t r = (size_t)lo * W;
            return readout_search_impl(q, readouts + lo, cnt, W, fb, fe, initial, step, radius, calls.data() + r,
                                       out_cost + r, out_delay + r, out_curves ? out_curves + r * D : nullptr);
        });
        if (F > 0 && (rc == RSSYNC_OK || rc == RSSYNC_E_NONFINITE)) {  // the statistics of the last readout's grid
            const rssync_problem* last = rank_problem(p, n_ranks(p) - 1);
            p->grid_tasks = last->grid_tasks;
            p->grid_exact_tasks = last->grid_exact_tasks;
        }
        return rc;
    }
    CUDA_TRY(p, cudaSetDevice(p->device));
    if (int rc = flush(p)) return rc;  // pending gyro and tracks; ordered behind ingests in flight
    std::vector<double> costs((size_t)nw * D, 0.0);  // no frames: the reference sums over none
    std::vector<unsigned> flags((size_t)n * 2, 0u);
    if (F > 0) {
        cudaStream_t st = p->stream;
        // the scratch arena holds the union of the windows' frames back to back; uidx[f]: listed frame f's
        // place in the union
        std::vector<FrameDesc> sel;
        std::vector<int> uidx((size_t)F);
        {
            std::unordered_map<int64_t, int> at;
            for (int f = 0; f < F; ++f) {
                const auto ins = at.emplace(win.frames[(size_t)f].id, (int)sel.size());
                if (ins.second) sel.push_back(win.frames[(size_t)f]);
                uidx[(size_t)f] = ins.first->second;
            }
        }
        const int U = (int)sel.size();
        std::vector<int32_t> dst((size_t)U);
        size_t rays = 0;
        for (int u = 0; u < U; ++u) {
            dst[(size_t)u] = (int32_t)rays;
            rays += (size_t)(sel[(size_t)u].n + 31) / 32 * 32;
        }
        const std::vector<rs::PixelFrame> rec = retime_records(p, sel, dst);
        CUDA_TRY(p, p->d_rt_rays.reserve(rays * 8));
        CUDA_TRY(p, p->d_rt_orig.reserve(rays));
        CUDA_TRY(p, p->d_rt_pos.reserve(rays));
        CUDA_TRY(p, p->d_pixframes.reserve((size_t)U));
        CUDA_TRY(p, p->d_rt_ext.reserve((size_t)U * 4));
        if (int rc = h2d(p, p->d_pixframes.ptr, rec.data(), sizeof(rs::PixelFrame) * U)) return rc;
        // the first readout's re-time also reports each frame's row extremes, from which the host takes
        // every readout's frame bounds (the frame tables and the grids' staging windows)
        rs::launch_retime_frames(p->d_pixframes.ptr, U, p->d_rays.ptr, p->d_orig.ptr, p->d_rowq.ptr, readouts[0],
                                 p->d_rt_rays.ptr, p->d_rt_orig.ptr, p->d_rt_pos.ptr, p->d_rt_ext.ptr, st);
        std::vector<double> ext((size_t)U * 4);
        if (int rc = d2h(p, ext.data(), p->d_rt_ext.ptr, ext.size() * sizeof(double))) return rc;
        if (int rc = finish_stream(p, st)) return rc;
        std::vector<FrameDesc> tables((size_t)n * F);
        std::vector<int> max_chunk((size_t)n);
        for (int j = 0; j < n; ++j) {
            FrameDesc* table = &tables[(size_t)j * F];
            for (int f = 0; f < F; ++f) {
                const size_t u = (size_t)uidx[(size_t)f];
                table[f] = FrameDesc{sel[u].id, dst[u], sel[u].n, 0.0, 0.0};
                retimed_bounds(rec[u], &ext[u * 4], readouts[j], table[f].ts_lo, table[f].ts_hi);
            }
            max_chunk[(size_t)j] = grid_max_chunk(table, F, delays.data(), D, p->sr, win.max_n);
        }
        if (int rc = stage_grid(p, tables.data(), tables.size(), F, delays.data(), D, nw)) return rc;
        if (int rc = stage_windows(p, win, calls, n)) return rc;
        rs::DeviceData dd = p->device_data();
        dd.rays = p->d_rt_rays.ptr;
        dd.orig = p->d_rt_orig.ptr;
        dd.pos = p->d_rt_pos.ptr;
        for (int j = 0; j < n; ++j) {
            if (j > 0)
                rs::launch_retime_frames(p->d_pixframes.ptr, U, p->d_rays.ptr, p->d_orig.ptr, p->d_rowq.ptr, readouts[j],
                                         p->d_rt_rays.ptr, p->d_rt_orig.ptr, p->d_rt_pos.ptr, nullptr, st);
            launch_candidate_grid(p, dd, win, j, p->d_frames.ptr + (size_t)j * F, p->d_delays.ptr, D,
                                  calls[(size_t)j * W], max_chunk[(size_t)j], st);
        }
        if (int rc = d2h(p, costs.data(), p->d_costs.ptr, costs.size() * sizeof(double))) return rc;
        if (int rc = d2h(p, flags.data(), p->d_flags.ptr, flags.size() * sizeof(unsigned))) return rc;
        if (int rc = finish_stream(p, st)) return rc;
        p->grid_tasks = (uint64_t)F * (uint64_t)D;
        p->grid_exact_tasks = flags[(size_t)n * 2 - 1];
    }
    for (int j = 0; j < n; ++j) {
        if (const unsigned fl = flags[2 * (size_t)j]) { p->err = presync_panic_text(fl); return RSSYNC_E_NONFINITE; }
        candidate_results(j, W, costs, delays, out_cost, out_delay, out_curves);
    }
    return RSSYNC_OK;
}

}  // namespace

extern "C" {

int rssync_readout_search(rssync_problem* p, const double* readouts, int n_readouts, double initial,
                          int64_t fb, int64_t fe, double step, double radius, const uint64_t* call_nos,
                          double* out_cost, double* out_delay, double* out_curves) {
    RS_NVTX_RANGE();
    if (p && n_readouts < 0) { p->err = "readout-search: negative readout count"; return RSSYNC_E_INVALID; }
    return readout_search_impl(p, readouts, n_readouts, 1, &fb, &fe, initial, step, radius, call_nos, out_cost,
                               out_delay, out_curves);
}

int rssync_readout_search_windows(rssync_problem* p, const double* readouts, int n_readouts, int n_windows,
                                  const int64_t* fb, const int64_t* fe, double initial, double step, double radius,
                                  const uint64_t* call_nos, double* out_cost, double* out_delay,
                                  double* out_curves) {
    RS_NVTX_RANGE();
    return readout_search_impl(p, readouts, n_readouts, n_windows, fb, fe, initial, step, radius, call_nos, out_cost,
                               out_delay, out_curves);
}

// Re-time the pixel frames of [fb, fe) in place at `readout`: afterwards the problem holds what ingesting
// them with lens.readout = readout would have produced (tiles, orig / pos, frame table).
int rssync_set_readout(rssync_problem* p, double readout, int64_t fb, int64_t fe) {
    RS_NVTX_RANGE();
    if (!p) return RSSYNC_E_INVALID;
    if (int rc = check_readouts(p, &readout, 1, "set-readout")) return rc;
    std::vector<FrameDesc> sel;
    for (auto it = p->frames.lower_bound(fb); it != p->frames.end() && it->first < fe; ++it) sel.push_back(it->second);
    if (int rc = require_retime(p, sel, "set-readout")) return rc;
    if (sel.empty()) return RSSYNC_OK;
    const int F = (int)sel.size();
    CUDA_TRY(p, cudaSetDevice(p->device));
    if (int rc = wait_arena_copies(p)) return rc;  // a replication still reading the arena, the staging block
    if (int rc = flush(p)) return rc;              // uploads and ingests in flight land first
    p->version++;
    std::vector<int32_t> dst((size_t)F);
    for (int f = 0; f < F; ++f) dst[(size_t)f] = sel[(size_t)f].off;
    const std::vector<rs::PixelFrame> rec = retime_records(p, sel, dst);
    CUDA_TRY(p, p->d_pixframes.reserve((size_t)F));
    CUDA_TRY(p, p->d_rt_ext.reserve((size_t)F * 4));
    if (int rc = h2d(p, p->d_pixframes.ptr, rec.data(), sizeof(rs::PixelFrame) * F)) return rc;
    rs::launch_retime_frames(p->d_pixframes.ptr, F, p->d_rays.ptr, p->d_orig.ptr, p->d_rowq.ptr, readout,
                             p->d_rays.ptr, p->d_orig.ptr, p->d_pos.ptr, p->d_rt_ext.ptr, p->stream);
    std::vector<double> ext((size_t)F * 4);
    if (int rc = d2h(p, ext.data(), p->d_rt_ext.ptr, ext.size() * sizeof(double))) return rc;
    if (int rc = finish_stream(p, p->stream)) return rc;
    for (int f = 0; f < F; ++f) {
        FrameDesc& fd = p->frames.at(sel[(size_t)f].id);
        retimed_bounds(rec[(size_t)f], &ext[(size_t)f * 4], readout, fd.ts_lo, fd.ts_hi);
    }
    return RSSYNC_OK;
}

int rssync_sync(rssync_problem* p, double initial, int64_t fb, int64_t fe, double center,
                double radius, double* out_cost, double* out_delay) {
    RS_NVTX_RANGE();
    if (!p || !out_cost || !out_delay) return RSSYNC_E_INVALID;
    // one syncpoint is one unit of work: it runs on the primary device ("replicas only" at this granularity)
    return sync_batch_impl(p, 1, &initial, &fb, &fe, &center, &radius, out_cost, out_delay, true);
}

int rssync_sync_batch(rssync_problem* p, int n, const double* initial, const int64_t* fb,
                      const int64_t* fe, const double* center, const double* radius,
                      double* out_cost, double* out_delay) {
    if (!p || n < 0) return RSSYNC_E_INVALID;
    if (n && (!initial || !fb || !fe || !center || !radius || !out_cost || !out_delay)) return RSSYNC_E_INVALID;
    if (is_multi(p) && n > 1) return multi_sync_batch(p, n, initial, fb, fe, center, radius, out_cost, out_delay, nullptr);
    return sync_batch_impl(p, n, initial, fb, fe, center, radius, out_cost, out_delay, false);
}

int rssync_sync_batch_ex(rssync_problem* p, int n, const double* initial, const int64_t* fb,
                         const int64_t* fe, const double* center, const double* radius,
                         const uint64_t* call_nos, double* out_cost, double* out_delay) {
    RS_NVTX_RANGE();
    if (!p || n < 0) return RSSYNC_E_INVALID;
    if (n && (!initial || !fb || !fe || !center || !radius || !out_cost || !out_delay)) return RSSYNC_E_INVALID;
    if (is_multi(p) && n > 1) return multi_sync_batch(p, n, initial, fb, fe, center, radius, out_cost, out_delay, call_nos);
    return sync_batch_impl(p, n, initial, fb, fe, center, radius, out_cost, out_delay, false, call_nos);
}

int rssync_last_sync_trace(const rssync_problem* p, double* delays, double* steps, int cap) {
    if (!p) return 0;
    int n = (int)std::min<size_t>(p->trace_delay.size(), (size_t)std::max(cap, 0));
    for (int i = 0; i < n; ++i) {
        if (delays) delays[i] = p->trace_delay[i];
        if (steps) steps[i] = p->trace_step[i];
    }
    return (delays || steps) ? n : (int)p->trace_delay.size();
}

int rssync_set_rng(rssync_problem* p, uint64_t seed, uint64_t call_no) {
    if (!p) return RSSYNC_E_INVALID;
    p->seed = seed;
    p->call_no = call_no;
    for (rssync_problem* r : p->replicas) r->seed = seed;
    return RSSYNC_OK;
}
uint64_t rssync_call_counter(const rssync_problem* p) { return p ? p->call_no : 0; }

int rssync_set_loss_mode(rssync_problem* p, int mode) {
    if (!p || (mode != RSSYNC_LOSS_FULL && mode != RSSYNC_LOSS_SIMPLIFIED)) return RSSYNC_E_INVALID;
    p->simplified = mode == RSSYNC_LOSS_SIMPLIFIED;
    for (rssync_problem* r : p->replicas) r->simplified = p->simplified;
    return RSSYNC_OK;
}

int rssync_set_stream(rssync_problem* p, void* s) {
    if (!p) return RSSYNC_E_INVALID;
    p->stream = (cudaStream_t)s;
    return RSSYNC_OK;
}

int rssync_flush(rssync_problem* p) {
    RS_NVTX_RANGE();
    if (!p) return RSSYNC_E_INVALID;
    if (int rc = flush(p)) return rc;
    CUDA_TRY(p, cudaStreamSynchronize(p->stream));
    return RSSYNC_OK;
}

int rssync_frame_table(const rssync_problem* p, rssync_frame_desc* out, size_t cap) {
    if (!p) return 0;
    size_t i = 0;
    for (const auto& kv : p->frames) {
        if (out && i < cap) {
            const FrameDesc& fd = kv.second;
            out[i] = rssync_frame_desc{fd.id, fd.off, fd.n, fd.ts_lo, fd.ts_hi};
        }
        ++i;
    }
    return (int)i;
}

int rssync_device_state(rssync_problem* p, rssync_device_state_t* out) {
    RS_NVTX_RANGE();
    if (!p || !out) return RSSYNC_E_INVALID;
    if (int rc = flush(p)) return rc;
    CUDA_TRY(p, cudaStreamSynchronize(p->stream));
    out->rays = p->d_rays.ptr;
    out->orig = p->d_orig.ptr;
    out->pos = p->d_pos.ptr;
    out->spline_records = p->d_rec.ptr;
    out->arena_rays = p->dev_used;
    out->gyro_samples = p->nq;
    out->sample_rate = p->sr;
    out->first_timestamp = p->q0;
    return RSSYNC_OK;
}

int rssync_device_state_pipelined(rssync_problem* p, rssync_device_state_t* out, size_t* chunk_lo, size_t* chunk_hi,
                                  size_t cap, size_t* n_chunks) {
    if (!p || !out || !n_chunks || (cap && (!chunk_lo || !chunk_hi))) return RSSYNC_E_INVALID;
    if (int rc = flush(p, /*keep_in_flight=*/true)) return rc;  // no host synchronisation with the device
    out->rays = p->d_rays.ptr;
    out->orig = p->d_orig.ptr;
    out->pos = p->d_pos.ptr;
    out->spline_records = p->d_rec.ptr;
    out->arena_rays = p->dev_used;
    out->gyro_samples = p->nq;
    out->sample_rate = p->sr;
    out->first_timestamp = p->q0;
    *n_chunks = p->in_flight.size();
    for (size_t k = 0; k < p->in_flight.size() && k < cap; ++k) {
        chunk_lo[k] = p->in_flight[k].lo;
        chunk_hi[k] = p->in_flight[k].hi;
    }
    return RSSYNC_OK;
}

int rssync_stream_wait_chunk(rssync_problem* p, int k, void* stream) {
    if (!p) return RSSYNC_E_INVALID;
    CUDA_TRY(p, cudaSetDevice(p->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (k < 0) {  // whatever the problem's stream holds now (spline records, frames set one by one)
        if (!p->ev_order) CUDA_TRY(p, cudaEventCreateWithFlags(&p->ev_order, cudaEventDisableTiming));
        CUDA_TRY(p, cudaEventRecord(p->ev_order, p->stream));
        CUDA_TRY(p, cudaStreamWaitEvent(st, p->ev_order, 0));
        return RSSYNC_OK;
    }
    if ((size_t)k >= p->in_flight.size()) { p->err = "stream-wait-chunk: no such chunk in flight"; return RSSYNC_E_INVALID; }
    CUDA_TRY(p, cudaStreamWaitEvent(st, p->in_flight[(size_t)k].ev, 0));
    p->in_flight[(size_t)k].foreign = true;  // a collective's kernel will send this chunk on: see enqueue_grid_kernels
    return RSSYNC_OK;
}

int rssync_expect_chunk(rssync_problem* p, size_t lo, size_t hi, void* stream) {
    if (!p || lo > hi) return RSSYNC_E_INVALID;
    CUDA_TRY(p, cudaSetDevice(p->device));
    rssync_problem::InFlight fl{lo, hi, nullptr, true};
    if (p->ev_pool.empty()) {
        CUDA_TRY(p, cudaEventCreateWithFlags(&fl.ev, cudaEventDisableTiming));
    } else {
        fl.ev = p->ev_pool.back();
        p->ev_pool.pop_back();
    }
    CUDA_TRY(p, cudaEventRecord(fl.ev, static_cast<cudaStream_t>(stream)));
    p->in_flight.push_back(fl);
    return RSSYNC_OK;
}

int rssync_note_reader(rssync_problem* p, void* stream) {
    if (!p) return RSSYNC_E_INVALID;
    CUDA_TRY(p, cudaSetDevice(p->device));
    if (!p->ev_reader) CUDA_TRY(p, cudaEventCreateWithFlags(&p->ev_reader, cudaEventDisableTiming));
    CUDA_TRY(p, cudaEventRecord(p->ev_reader, static_cast<cudaStream_t>(stream)));
    p->reader_pending = true;
    return RSSYNC_OK;
}

int rssync_adopt_state(rssync_problem* p, const rssync_frame_desc* frames, size_t n_frames, size_t arena_rays,
                       size_t gyro_samples, double sample_rate, double first_timestamp) {
    RS_NVTX_RANGE();
    if (!p || (n_frames && !frames)) return RSSYNC_E_INVALID;
    if (gyro_samples > (size_t)INT32_MAX || arena_rays > (size_t)INT32_MAX) { p->err = "adopt-state: too large"; return RSSYNC_E_INVALID; }
    join_gyro(p);
    cudaSetDevice(p->device);
    if (int rc = drain_in_flight(p)) return rc;
    if (int rc = wait_arena_copies(p)) return rc;
    CUDA_TRY(p, cudaStreamSynchronize(p->stream));
    if (p->gyro_stream) CUDA_TRY(p, cudaStreamSynchronize(p->gyro_stream));
    p->version++;
    p->pending.clear();
    p->gyro_dirty = false;
    p->retime.clear();  // an adopted arena comes without row fractions (rssync_adopt_row_fractions adds them)
    p->rowq_version++;
    // the same table as last time (a caller replicating fresh data of an unchanged frame set): keep the map
    bool same = p->frames.size() == n_frames;
    if (same) {
        size_t i = 0;
        for (auto it = p->frames.begin(); it != p->frames.end() && same; ++it, ++i) {
            const FrameDesc& a = it->second;
            const rssync_frame_desc& b = frames[i];
            same = a.id == b.id && a.off == b.off && a.n == b.n && a.ts_lo == b.ts_lo && a.ts_hi == b.ts_hi;
        }
    }
    if (!same) {
    p->frames.clear();
    p->place_hint_valid = false;
    p->total_rays = 0;
    for (size_t i = 0; i < n_frames; ++i) {
        const rssync_frame_desc& f = frames[i];
        if (f.n < 0 || f.n > rs::kMaxRaysPerFrame || f.off < 0 || (f.off & 31) ||
            (size_t)f.off + (size_t)(f.n + 31) / 32 * 32 > arena_rays) {
            p->err = "adopt-state: frame outside the arena";
            return RSSYNC_E_INVALID;
        }
        p->frames[f.id] = FrameDesc{f.id, f.off, f.n, f.ts_lo, f.ts_hi};
        p->total_rays += (size_t)f.n;
    }
    }
    p->used = p->dev_used = arena_rays;
    p->garbage = 0;
    p->nq = gyro_samples;
    p->sr = sample_rate;
    p->q0 = first_timestamp;
    CUDA_TRY(p, p->d_rays.reserve(std::max<size_t>(arena_rays, 1) * 8));
    CUDA_TRY(p, p->d_orig.reserve(std::max<size_t>(arena_rays, 1)));
    CUDA_TRY(p, p->d_pos.reserve(std::max<size_t>(arena_rays, 1)));
    CUDA_TRY(p, p->d_rec.reserve(std::max<size_t>(gyro_samples, 1) * 16));
    // the pinned host mirror belongs to frames set one by one; an adopted arena has none
    p->adopted_version = p->version;
    return RSSYNC_OK;
}

int rssync_retime_table(const rssync_problem* p, rssync_retime_desc* out, size_t cap) {
    if (!p) return 0;
    std::vector<int64_t> ids;
    ids.reserve(p->retime.size());
    for (const auto& kv : p->retime) ids.push_back(kv.first);
    std::sort(ids.begin(), ids.end());
    for (size_t i = 0; out && i < ids.size() && i < cap; ++i) {
        const std::pair<double, double>& ts = p->retime.at(ids[i]);
        out[i] = rssync_retime_desc{ids[i], ts.first, ts.second};
    }
    return (int)ids.size();
}

int rssync_row_fraction_plane(rssync_problem* p, double** plane, size_t* n_doubles) {
    RS_NVTX_RANGE();
    if (!p || !plane || !n_doubles) return RSSYNC_E_INVALID;
    *plane = nullptr;
    *n_doubles = 0;
    if (int rc = flush(p)) return rc;
    CUDA_TRY(p, cudaStreamSynchronize(p->stream));
    if (p->retime.empty()) return RSSYNC_OK;
    if (int rc = rowq_cover_arena(p)) return rc;
    *plane = p->d_rowq.ptr;
    *n_doubles = 2 * p->dev_used;
    return RSSYNC_OK;
}

int rssync_adopt_row_fractions(rssync_problem* p, const rssync_retime_desc* frames, size_t n) {
    RS_NVTX_RANGE();
    if (!p) return RSSYNC_E_INVALID;
    if (p->adopted_version != p->version) {
        p->err = "adopt-row-fractions: the problem's state must come from rssync_adopt_state, with no input set since";
        return RSSYNC_E_STATE;
    }
    if (n && !frames) { p->err = "adopt-row-fractions: null argument"; return RSSYNC_E_INVALID; }
    std::unordered_map<int64_t, std::pair<double, double>> table;
    table.reserve(n);
    for (size_t i = 0; i < n; ++i) {
        const rssync_retime_desc& f = frames[i];
        const std::string which = "adopt-row-fractions: frame " + std::to_string(f.id);
        if (!p->frames.count(f.id)) { p->err = which + " is not in the adopted frame table"; return RSSYNC_E_INVALID; }
        if (!std::isfinite(f.frame_ts_a) || !std::isfinite(f.frame_ts_b)) {
            p->err = which + " has a non-finite frame timestamp";
            return RSSYNC_E_INVALID;
        }
        if (!table.emplace(f.id, std::make_pair(f.frame_ts_a, f.frame_ts_b)).second) {
            p->err = which + " is given more than once";
            return RSSYNC_E_INVALID;
        }
    }
    CUDA_TRY(p, cudaSetDevice(p->device));
    if (int rc = wait_reader(p)) return rc;
    CUDA_TRY(p, cudaStreamSynchronize(p->stream));  // no re-timing still reads the plane
    if (n) CUDA_TRY(p, p->d_rowq.reserve(2 * std::max<size_t>(p->dev_used, 1)));
    p->retime.swap(table);
    p->rowq_version++;
    return RSSYNC_OK;
}

int rssync_get_stats(const rssync_problem* p, rssync_stats* out) {
    if (!p || !out) return RSSYNC_E_INVALID;
    out->kernel_launches = rs::launch_count();
    out->h2d_bytes = p->h2d;
    out->d2h_bytes = p->d2h;
    out->frames = p->frames.size();
    out->rays = p->total_rays;
    out->gyro_samples = p->nq;
    out->sync_outer_iters = p->sync_outer;
    out->sync_lbfgs_evals = p->sync_evals;
    out->last_grid_kernel_ms = p->last_grid_ms;
    out->last_grid_tasks = p->grid_tasks;
    out->last_grid_exact_tasks = p->grid_exact_tasks;
    out->sync_row_builds = p->sync_row_builds;
    out->sync_loss_evals = p->sync_loss_evals;
    out->sync_init_tasks = p->sync_init_tasks;
    out->sync_outer_total = p->sync_outer_total;
    out->nccl_calls = p->nccl_calls;
    out->broadcast_bytes = p->broadcast_bytes;
    return RSSYNC_OK;
}

int rssync_measure_fp64_peak(double* tflops) {
    if (!tflops) return RSSYNC_E_INVALID;
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return RSSYNC_E_CUDA;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    double* sink = nullptr;
    if (cudaMalloc((void**)&sink, 8) != cudaSuccess) return RSSYNC_E_CUDA;
    const int blocks = sms * 8, threads = 256, iters = 1 << 16;
    double best = 0.0;
    for (int rep = 0; rep < 3; ++rep) {
        float ms = rs::run_fp64_peak(blocks, threads, iters, sink, nullptr);
        double flops = 2.0 * 8.0 * (double)iters * (double)blocks * (double)threads;
        if (ms > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    cudaFree(sink);
    if (cudaGetLastError() != cudaSuccess) return RSSYNC_E_CUDA;
    *tflops = best;
    return RSSYNC_OK;
}

// ---- probes -----------------------------------------------------------------------------------
int rssync_probe_gyro(const rssync_problem* p, double* sample_rate, double* first_timestamp,
                      size_t* count, double* rec) {
    if (!p) return RSSYNC_E_INVALID;
    if (sample_rate) *sample_rate = p->sr;
    if (first_timestamp) *first_timestamp = p->q0;
    if (count) *count = p->nq;
    if (rec && p->nq) {  // read the finished records back, out of the device's swizzled group order
        rssync_problem* q = const_cast<rssync_problem*>(p);
        if (int rc = flush(q)) return rc;
        std::vector<double> tmp(p->nq * 16);
        if (int rc = d2h(q, tmp.data(), p->d_rec.ptr, tmp.size() * sizeof(double))) return rc;
        CUDA_TRY(q, cudaStreamSynchronize(p->stream));
        for (size_t i = 0; i < p->nq; ++i)
            for (size_t j = 0; j < 16; ++j) rec[i * 16 + j] = tmp[i * 16 + (j ^ ((i & 3) * 4))];
    }
    return RSSYNC_OK;
}

int rssync_probe_spline_system(const double* quats, size_t count, double* rhs, double* diag) {
    if (!quats || !rhs || !diag || count < 2) return RSSYNC_E_INVALID;
    rs::build_spline_system(quats, count, rhs, diag);
    return RSSYNC_OK;
}

static int probe_frame(rssync_problem* p, int64_t frame, FrameDesc& fd) {
    if (int rc = require_gyro(p, "probe")) return rc;
    auto it = p->frames.find(frame);
    if (it == p->frames.end()) { p->err = "probe: no such frame"; return RSSYNC_E_INVALID; }
    fd = it->second;
    if (fd.n < 2) { p->err = "probe: frame has fewer than 2 rays"; return RSSYNC_E_INVALID; }
    return flush(p);
}

int rssync_probe_problem_matrix(rssync_problem* p, int64_t frame, double delay, double* rows) {
    if (!p || !rows) return RSSYNC_E_INVALID;
    FrameDesc fd;
    if (int rc = probe_frame(p, frame, fd)) return rc;
    CUDA_TRY(p, p->d_probe.reserve((size_t)fd.n * 3));
    rs::launch_probe_problem_matrix(p->device_data(), fd, delay, p->d_probe.ptr, p->stream);
    if (int rc = d2h(p, rows, p->d_probe.ptr, sizeof(double) * 3 * fd.n)) return rc;
    CUDA_TRY(p, cudaStreamSynchronize(p->stream));
    return RSSYNC_OK;
}

int rssync_probe_guess_motion_ex(rssync_problem* p, int64_t frame, double delay, int iters, int stream,
                                 uint64_t call_no, uint64_t offset_index, int mode, double* m3,
                                 double* k, int* used_exact) {
    if (!p || !m3) return RSSYNC_E_INVALID;
    FrameDesc fd;
    if (int rc = probe_frame(p, frame, fd)) return rc;
    CUDA_TRY(p, p->d_probe.reserve(8));
    CUDA_TRY(p, cudaMemsetAsync(p->d_probe.ptr + 4, 0, sizeof(double), p->stream));
    rs::launch_probe_guess(p->device_data(), fd, delay, iters,
                           rs::rng_prefix(p->seed, (uint64_t)stream, call_no, offset_index), mode,
                           p->d_probe.ptr, reinterpret_cast<unsigned*>(p->d_probe.ptr + 4), p->stream);
    double out[5];
    if (int rc = d2h(p, out, p->d_probe.ptr, sizeof(out))) return rc;
    CUDA_TRY(p, cudaStreamSynchronize(p->stream));
    m3[0] = out[0]; m3[1] = out[1]; m3[2] = out[2];
    if (k) *k = out[3];
    if (used_exact) {
        unsigned c;
        std::memcpy(&c, &out[4], sizeof(c));
        *used_exact = (int)c;
    }
    return RSSYNC_OK;
}

int rssync_probe_guess_motion(rssync_problem* p, int64_t frame, double delay, int iters, int stream,
                              uint64_t call_no, uint64_t offset_index, double* m3, double* k) {
    return rssync_probe_guess_motion_ex(p, frame, delay, iters, stream, call_no, offset_index, 0, m3, k,
                                        nullptr);
}

int rssync_probe_loss(rssync_problem* p, int64_t frame, double delay, const double* m3, double k,
                      double* loss3, double* loss5, double* grad3) {
    if (!p || !m3) return RSSYNC_E_INVALID;
    FrameDesc fd;
    if (int rc = probe_frame(p, frame, fd)) return rc;
    CUDA_TRY(p, p->d_probe.reserve(16));
    if (int rc = h2d(p, p->d_probe.ptr + 8, m3, 3 * sizeof(double))) return rc;
    rs::launch_probe_loss(p->device_data(), fd, delay, p->d_probe.ptr + 8, k, p->d_probe.ptr, p->stream);
    double out[5];
    if (int rc = d2h(p, out, p->d_probe.ptr, sizeof(out))) return rc;
    CUDA_TRY(p, cudaStreamSynchronize(p->stream));
    if (loss3) *loss3 = out[0];
    if (loss5) *loss5 = out[1];
    if (grad3) { grad3[0] = out[2]; grad3[1] = out[3]; grad3[2] = out[4]; }
    return RSSYNC_OK;
}

int rssync_probe_lbfgs(rssync_problem* p, int64_t frame, double delay, double* m3, double k, double* f,
                       int* iters, int* evals) {
    if (!p || !m3) return RSSYNC_E_INVALID;
    FrameDesc fd;
    if (int rc = probe_frame(p, frame, fd)) return rc;
    CUDA_TRY(p, p->d_probe.reserve(16));
    if (int rc = h2d(p, p->d_probe.ptr, m3, 3 * sizeof(double))) return rc;
    rs::launch_probe_lbfgs(p->device_data(), fd, delay, p->d_probe.ptr, k, p->d_probe.ptr + 4,
                           (int*)(p->d_probe.ptr + 8), p->stream);
    double out[5];
    int st[2];
    if (int rc = d2h(p, out, p->d_probe.ptr, sizeof(out))) return rc;
    if (int rc = d2h(p, st, p->d_probe.ptr + 8, sizeof(st))) return rc;
    CUDA_TRY(p, cudaStreamSynchronize(p->stream));
    m3[0] = out[0]; m3[1] = out[1]; m3[2] = out[2];
    if (f) *f = out[4];
    if (iters) *iters = st[0];
    if (evals) *evals = st[1];
    return RSSYNC_OK;
}

int rssync_probe_replication_plan(const size_t* lo, const size_t* hi, size_t n, size_t arena_rays, size_t groups,
                                  int* k_last, size_t* piece_lo, size_t* piece_hi, size_t cap) {
    if ((n && (!lo || !hi)) || groups == 0 || (cap && (!k_last || !piece_lo || !piece_hi))) return -1;
    std::vector<std::pair<size_t, size_t>> flying;
    for (size_t k = 0; k < n; ++k) flying.emplace_back(lo[k], hi[k]);
    const std::vector<ReplicationPiece> pieces = plan_replication(flying, arena_rays, groups);
    for (size_t i = 0; i < pieces.size() && i < cap; ++i) {
        k_last[i] = pieces[i].k_last;
        piece_lo[i] = pieces[i].lo;
        piece_hi[i] = pieces[i].hi;
    }
    return (int)pieces.size();
}

int rssync_probe_stage_copy(const double* src, size_t n, int mode, double* dst, double* lo, double* hi,
                            int* all_finite_out) {
    if (!src || !dst || !all_finite_out || (lo == nullptr) != (hi == nullptr)) return RSSYNC_E_INVALID;
    bool ok;
#if defined(__x86_64__)
    if (mode != 0 && !__builtin_cpu_supports("avx2")) return RSSYNC_E_INVALID;
    if (mode == 1) ok = copy_checked_avx2<false>(dst, src, n, lo, hi);
    else if (mode == 2) ok = copy_checked_avx2<true>(dst, src, n, lo, hi);
    else
#else
    if (mode != 0) return RSSYNC_E_INVALID;
#endif
        ok = copy_checked_scalar(dst, src, n, lo, hi);
    *all_finite_out = ok ? 1 : 0;
    return RSSYNC_OK;
}

int rssync_probe_spec_trig(const double* x, int n, int which, int on_device, double* out) {
    if (n <= 0) return RSSYNC_OK;
    if (!x || !out || which < 0 || which > 2) return RSSYNC_E_INVALID;
    if (!on_device) {
        for (int i = 0; i < n; ++i) out[i] = which == 0 ? rs::spec_sin(x[i]) : which == 1 ? rs::spec_cos(x[i]) : rs::spec_acos(x[i]);
        return RSSYNC_OK;
    }
    double *dx = nullptr, *dy = nullptr;
    if (cudaMalloc((void**)&dx, sizeof(double) * n) != cudaSuccess) return RSSYNC_E_CUDA;
    if (cudaMalloc((void**)&dy, sizeof(double) * n) != cudaSuccess) { cudaFree(dx); return RSSYNC_E_CUDA; }
    cudaMemcpy(dx, x, sizeof(double) * n, cudaMemcpyHostToDevice);
    rs::launch_probe_trig(dx, n, which, dy, nullptr);
    cudaError_t e = cudaMemcpy(out, dy, sizeof(double) * n, cudaMemcpyDeviceToHost);
    cudaFree(dx);
    cudaFree(dy);
    return e == cudaSuccess ? RSSYNC_OK : RSSYNC_E_CUDA;
}

int rssync_probe_log1p(const double* x, int n, double* out) {
    if (n <= 0) return RSSYNC_OK;
    double *dx = nullptr, *dy = nullptr;
    if (cudaMalloc((void**)&dx, sizeof(double) * n) != cudaSuccess) return RSSYNC_E_CUDA;
    if (cudaMalloc((void**)&dy, sizeof(double) * n) != cudaSuccess) { cudaFree(dx); return RSSYNC_E_CUDA; }
    cudaMemcpy(dx, x, sizeof(double) * n, cudaMemcpyHostToDevice);
    rs::launch_probe_log1p(dx, n, dy, nullptr);
    cudaError_t e = cudaMemcpy(out, dy, sizeof(double) * n, cudaMemcpyDeviceToHost);
    cudaFree(dx);
    cudaFree(dy);
    return e == cudaSuccess ? RSSYNC_OK : RSSYNC_E_CUDA;
}

}  // extern "C"
