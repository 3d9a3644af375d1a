// Internal interface between the host side of the engine (capi.cpp, sync_solver.cpp) and the
// sm_100a kernels (engine.cu).  Not part of the public boundary (include/rssync_b200.h is).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace rs {

constexpr int kMaxRaysPerFrame = 512;  // 16 slots x 32 lanes (one warp per frame task)
constexpr double kNumericDiffStep = 1e-6;  // FrameState::kNumericDiffStep, core_private.hpp:38

// One tracked frame inside the device arena (FrameData, core_private.hpp:8-13).
struct FrameDesc {
    int64_t id;   // caller's frame number (also an RNG key component)
    int32_t off;  // index of the frame's first ray in the arena (multiple of 32)
    int32_t n;    // rays in the frame
    double ts_lo, ts_hi;  // smallest / largest of the frame's ts_a, ts_b (bounds the spline window)
};

// Read-only device state shared by all kernels (OptData, core_private.hpp:15-22).
struct DeviceData {
    const double* rec;  // gyro spline: nq records of {y[4], b[4], c[4], d[4]}
    int nq;
    double q0, sr;      // quats_start, sample_rate
    // ray arena: one 2 KB tile [8 fields][32 rays] of doubles per group of 32 rays; fields ts_a,
    // ts_b, ra.x, ra.y, ra.z, rb.x, rb.y, rb.z.  Ray i of the arena is rays[(i/32)*256 + f*32 + i%32].
    const double* rays;
    const int32_t* orig;  // caller's index of each stored ray (rays are stored sorted by ts_a)
    const int32_t* pos;   // inverse of orig inside each frame: storage slot of caller's ray i
};

enum RngStream : uint64_t { kStreamPreSync = 1, kStreamDebugPreSync = 2, kStreamSyncInit = 3 };

// flags written by the PreSync kernel (panic conditions of core_private.cpp:76-83)
enum : unsigned { kFlagP = 1u, kFlagM = 2u, kFlagR = 4u, kFlagRho = 8u };

// ---- PreSync / DebugPreSync grid: cost[d] = sum_f framecost(d, f) -----------------------------
// d_framecost: D x F scratch; d_costs: D outputs; d_flags: 2 words {panic flags, tasks whose
// translation estimate needed the exact binary64 estimator}.  All pointers are device pointers.
void launch_presync_grid(const DeviceData& dd, const FrameDesc* d_frames, int F, int max_n,
                         const double* d_delays, int D, uint64_t seed, uint64_t stream,
                         uint64_t call_no, uint64_t idx_base, double* d_framecost, double* d_costs,
                         unsigned* d_flags, cudaStream_t st, int max_chunk, bool simplified,
                         // several windows in one grid: the F frames are the windows' frames
                         // concatenated, frame f belongs to the call d_frame_call_no[f], window w
                         // covers frames [d_win_begin[w], d_win_begin[w+1]); d_costs is W x D
                         const uint64_t* d_frame_call_no = nullptr, const int* d_win_begin = nullptr,
                         int n_windows = 0);

// How many consecutive delays of the (host copy of the) delay list one work unit of the grid kernel
// may hold so that the spline window of any frame whose timestamps span at most frame_span_s seconds
// fits the kernel's staging buffer.  Host-side helper; pass the result as max_chunk.
int presync_max_chunk(const double* h_delays, int D, double frame_span_s, double sample_rate, int max_n);

// The two halves of launch_presync_grid, for callers that evaluate the frames in several launches
// (capi.cpp runs the frames of each upload chunk as soon as that chunk has landed): the task kernel
// over F frames writes framecost[d * cost_stride + f] for f in [0, F) -- pass d_framecost offset by
// the sub-range's first frame and the whole grid's frame count as cost_stride -- and the reduction
// sums the whole D x F scratch.
void launch_presync_tasks(const DeviceData& dd, const FrameDesc* d_frames, int F, int max_n,
                          const double* d_delays, int D, uint64_t seed, uint64_t stream, uint64_t call_no,
                          uint64_t idx_base, double* d_framecost, int cost_stride, unsigned* d_flags,
                          cudaStream_t st, const uint64_t* d_frame_call_no = nullptr, int max_chunk = 0,
                          bool simplified = false, int spare_sms = 0);  // spare_sms: SMs this launch leaves free
void launch_presync_reduce(const double* d_framecost, int F, int D, double* d_costs, cudaStream_t st,
                           const int* d_win_begin = nullptr, int n_windows = 0);

// ---- Sync: batched over syncpoints; tasks = (syncpoint, frame) --------------------------------
struct SyncTask {
    FrameDesc fd;
    int32_t sp;   // syncpoint index inside the batch
    int32_t pad;
};
struct SyncBatchDev {
    const SyncTask* tasks;  // T tasks, grouped by syncpoint
    int T;
    int max_n;
    const int* sp_begin;    // S+1 offsets into tasks
    int S;
    double* m;              // T x 3 translation directions (FrameState::motion_vec)
    double* k;              // T   (FrameState::var_k)
    int simplified;         // simplified (no-translation) loss mode: residual = |row|, m unused
};
// GuessMotion + GuessK at sp_delay[sp] (core_private.cpp:125-133, 218-223)
void launch_sync_init(const DeviceData& dd, const SyncBatchDev& b, const double* d_sp_delay,
                      const uint64_t* d_sp_callno, const unsigned char* d_sp_active, uint64_t seed,
                      cudaStream_t st);
// do_opt_motion (:262-296) at sp_delay, then Loss5 value at sp_x0 and Loss3 at sp_x0 -/+ h
// (f_and_grad, :228-240); reduced per syncpoint into out_v[sp], out_g[sp], and the ntrial trial
// points of Backtrack::Step (backtrack.cpp:5-12), x0 - t g with t = 1e-3, 1e-4, ..., into
// d_trial_delay[sp * ntrial + i].  *d_evals_total accumulates the objective evaluations.
void launch_sync_motion_fgrad(const DeviceData& dd, const SyncBatchDev& b, const double* d_sp_delay,
                              const double* d_sp_x0, const unsigned char* d_sp_active,
                              double* d_task_scratch /* T x 3 */, double* d_out_v, double* d_out_g,
                              double* d_trial_delay /* S x ntrial */, int ntrial,
                              int* d_lbfgs_stats /* T x 2 or null */,
                              unsigned long long* d_evals_total /* or null */,
                              bool many_tasks /* the batch has many more tasks than the device has warp
                                                 slots: use the small-block, register-capped build */,
                              cudaStream_t st);
// Loss3 summed per syncpoint at ntrial delays per syncpoint (simple_objective, :242-252)
// d_n_eval (device, optional): only the first (int)*d_n_eval of the ntrial points are evaluated
void launch_sync_trials(const DeviceData& dd, const SyncBatchDev& b, const double* d_trial_delay,
                        int ntrial, const unsigned char* d_sp_active,
                        double* d_task_scratch /* T x ntrial */, double* d_out /* S x ntrial */,
                        cudaStream_t st, const double* d_n_eval = nullptr);

// ---- gyro spline: finish the records on the device (host_ingest.h build_spline_system) ---------
// d_quats: n x 4 samples; d_rhs: n x 4, d_diag: n (the eliminated system); d_rec: n records of 16
// doubles in the layout of DeviceData::rec.  n >= 2.
void launch_spline_finish(const double* d_quats, const double* d_rhs, const double* d_diag, int n,
                          double* d_rec, cudaStream_t st);

// ---- gyro ingest on the device (K8, engine.cu) ---------------------------------------------------
// optdata_fill_gyro (core_testcode.cpp:37-53) for n_var gyro axis mappings: d_ts (n doubles, seconds),
// d_gyro (n x 3), h_matrices (9 per variant: the 3x3 row-major mapping of gyro_scan.h) -> d_quats
// (n_var x n x 4).  d_orients: gyro_orient_bytes(n_var) bytes, d_prefix: gyro_prefix_doubles(n, n_var)
// doubles of device scratch.
void launch_gyro_integrate(const double* d_ts, const double* d_gyro, int n, const double* h_matrices, int n_var,
                           void* d_orients, double* d_quats, double* d_prefix, cudaStream_t st);
size_t gyro_orient_bytes(int n_var);
size_t gyro_prefix_doubles(int n, int n_var);
// the per-sample half of the variable-rate SetGyroQuaternions (core_private.cpp:166-182): d_quats
// (n_var x count x 4) at timestamps d_ts_us (count) -> d_out (n_var x n_out x 4) on the grid
// 1e6 (tick0 + j) / rate_hz; d_nonfinite[v] is set when variant v produced a non-finite sample
void launch_gyro_resample(const int64_t* d_ts_us, int count, const double* d_quats, int n_var, uint64_t tick0,
                          unsigned rate_hz, int n_out, double* d_out, unsigned* d_nonfinite, cudaStream_t st);
// the two elimination sweeps of the spline system (minispline.cpp:22-32) for n_var tracks of n
// samples: d_y (n_var x n x 4) -> d_rhs (n_var x n x 4); d_f_down / d_f_up: the factors of
// spline_elimination(n) (host_ingest.h)
void launch_spline_chains(const double* d_y, const double* d_f_down, const double* d_f_up, int n, int n_var,
                          double* d_rhs, cudaStream_t st);
void launch_probe_trig(const double* d_x, int n, int which, double* d_out, cudaStream_t st);

// ---- pixel -> ray front end (track_frames' per-frame tail, core_testcode.cpp:134-161) --------
struct LensDev {  // Lens, core_testcode.cpp:55-61
    double ro, fx, fy, cx, cy, k1, k2, k3, k4;
};
struct PixelFrame {
    int32_t off;     // frame's first ray in the arena
    int32_t n;       // points in the frame
    int64_t src;     // index of the frame's first point in the pixel buffers
    double ts_a, ts_b;  // start-of-exposure timestamps of the two frames, seconds
};
// One block per frame: undistort both points of every pair (lens_undistort_point, :63-95),
// rolling-shutter timestamps (:144-145), unit rays (:153-154), sort by ts_a (ties keep the caller's
// order) and write the frame's tiles and orig / pos planes straight into the device arena.
// d_rowq: the row-fraction plane, 2 doubles per arena ray; ray i of a frame (caller's order) gets
// {y_a / image_rows, y_b / image_rows}, the factors of the readout in the timestamps.
void launch_ingest_pixels(const PixelFrame* d_frames, int n_frames, const double* d_points_a,
                          const double* d_points_b, LensDev lens, double image_rows, double* d_rays,
                          int32_t* d_orig, int32_t* d_pos, double* d_rowq, cudaStream_t st);
// Re-time frames ingested from pixels at another readout: one block per frame reads the frame's tiles
// and orig plane at PixelFrame::src of (d_src_rays, d_src_orig) and its row fractions d_rowq[2 (src +
// i) ..], recomputes ts = frame_ts + readout * q (ingest_pixels_kernel's expression; PixelFrame::ts_a /
// ts_b are the frame timestamps), sorts by (ts_a, caller index) and writes tiles and orig / pos at
// PixelFrame::off of (d_rays, d_orig, d_pos) -- which may be the source arena itself.  d_ext (4 doubles
// per frame, or null): min q_a, max q_a, min q_b, max q_b of the frame (+inf, -inf for no rays).
void launch_retime_frames(const PixelFrame* d_frames, int n_frames, const double* d_src_rays,
                          const int32_t* d_src_orig, const double* d_rowq, double readout, double* d_rays,
                          int32_t* d_orig, int32_t* d_pos, double* d_ext, cudaStream_t st);

// SetTrackResult for a batch of frames with the sort + transpose on the device: the callers' buffers
// (ts_a, ts_b: n doubles; rays_a, rays_b: n x 3 doubles, concatenated over frames) are staged as they
// are; one block per frame sorts by (ts_a, caller index) and writes tiles + orig / pos planes.
// PixelFrame::src is the index of the frame's first ray in the staged buffers; ts_a / ts_b unused.
void launch_ingest_rays(const PixelFrame* d_frames, int n_frames, const double* d_ts_a,
                        const double* d_ts_b, const double* d_rays_a, const double* d_rays_b,
                        double* d_rays, int32_t* d_orig, int32_t* d_pos, cudaStream_t st);
// The same with row fractions in place of the timestamps (d_frac_a / d_frac_b: 1 double per ray): ray i
// gets ts = PixelFrame::ts_a + readout * frac_a[i] (ts_b alike), ingest_pixels_kernel's expression, and
// d_rowq its {frac_a, frac_b} as launch_ingest_pixels writes them.
void launch_ingest_row_fractions(const PixelFrame* d_frames, int n_frames, const double* d_frac_a,
                                 const double* d_frac_b, const double* d_rays_a, const double* d_rays_b,
                                 double readout, double* d_rays, int32_t* d_orig, int32_t* d_pos, double* d_rowq,
                                 cudaStream_t st);

// ---- track buffers the caller holds in device memory (rssync_set_track_*_device) ---------------
// What the check-and-stage kernel reports per frame; the host reads these back and places the frames.
struct StageInfo {
    uint32_t bad;  // bit b set: source buffer b of the frame holds a NaN or an infinity
    uint32_t pad;
    double lo, hi;  // smallest / largest timestamp of the frame (0, 0 for a frame without rays)
};
// One block per frame reads the frame's segment of every per-ray buffer once, copies it into the
// staging buffer at the same offsets (the layout launch_ingest_rays / launch_ingest_pixels read) and
// writes info[f].  d_at: n_frames + 1 offsets (in rays) of the frames in the buffers.
// Rays form: src = {rays_a, rays_b, ts_a, ts_b} (3, 3, 1, 1 doubles per ray), the reference's order of
// checks; d_stage holds ts_a, ts_b, rays_a, rays_b of `total` rays back to back; lo / hi over ts_a, ts_b.
void launch_stage_rays(const int64_t* d_at, int n_frames, int64_t total, const double* rays_a,
                       const double* rays_b, const double* ts_a, const double* ts_b, double* d_stage,
                       StageInfo* d_info, cudaStream_t st);
// Pixels form: src = {points_a, points_b} (2 doubles per point); d_stage holds points_a, points_b;
// lo / hi over frame_ts + lens.ro * (y / rows), the expression ingest_pixels_kernel uses.  Bit b is
// also set when a point's (p - c) / f or its squared norm is not finite (undistort_point's x_, y_,
// theta_).  d_frame_ts: ts_a, ts_b of each frame (2 per frame).
void launch_stage_points(const int64_t* d_at, const double* d_frame_ts, int n_frames, int64_t total,
                         const double* points_a, const double* points_b, const LensDev& lens, double rows,
                         double* d_stage, StageInfo* d_info, cudaStream_t st);
// Row-fractions form: src = {rays_a, rays_b, frac_a, frac_b} (3, 3, 1, 1 doubles per ray); d_stage holds
// frac_a, frac_b, rays_a, rays_b (the rays form's layout, fractions in the ts slots); bit 2 / 3 is also
// set when frame_ts + readout * frac is not finite; lo / hi over those timestamps.
void launch_stage_row_fractions(const int64_t* d_at, const double* d_frame_ts, int n_frames, int64_t total,
                                const double* rays_a, const double* rays_b, const double* frac_a,
                                const double* frac_b, double readout, double* d_stage, StageInfo* d_info,
                                cudaStream_t st);

// ---- sparse pyramidal Lucas-Kanade between decoded frames (rssync_track_frames_device) -----------
// The arithmetic is the contract stated at rssync_track_frames_device in include/rssync_b200.h.
constexpr int kTrackMaxLevels = 6;
struct TrackImages {
    const uint8_t* img0;  // n_frames + 1 luma planes: row y of image j at img0 + (j * h0 + y) * pitch0 bytes
    int64_t pitch0;
    int w0, h0;
    int levels, window, max_iters;
    float epsilon, min_eig;
    uint8_t sample;  // bytes per sample: 1 (uint8_t, level 0 = (float)v) or 2 (uint16_t)
    uint8_t shift;   // 16-bit samples: level 0 = (float)v * 2^-shift, shift 0..8
};
// floats of one image's pyramid levels 1 .. levels - 1
size_t track_pyramid_floats(int w0, int h0, int levels);
// The kept pairs, frame by frame in the query order: d_out_a / d_out_b at the kept offsets d_kept_at
// (n_frames + 1, written here), the layout launch_stage_points reads.
void launch_track_compact(const int64_t* d_q_at, int n_frames, const double* d_points, const double* d_tracked,
                          const uint8_t* d_status, double* d_out_a, double* d_out_b, int64_t* d_kept_at,
                          cudaStream_t st);

// ---- point selection and the forward-backward check (rssync_track_frames_ex_device) -------------
// The selection contract is stated at rssync_track_frames_ex_device in include/rssync_b200.h.
struct TrackSelect {
    int cell, block, max_points;
    float quality;
    int cells_x, cells_y;  // cells per row and column of an image
    unsigned long long* d_keys;  // scratch: one key per (cell, image) of a chunk, slots * cells_x * cells_y
    uint32_t* d_picks;           // scratch: per frame of a chunk, max_points pixel indices y * w + x
    int32_t* d_count;            // scratch: per frame of a chunk, the number of picks
};
// ---- the caller's mask (rssync_track_frames_masked_device) ---------------------------------------
// The contract is stated at rssync_track_frames_masked_device in include/rssync_b200.h.  Row y of image j's
// mask at mask + j * image_stride + y * pitch bytes (image_stride 0: one mask for every image).  The mask is
// eroded by a (2 margin + 1)^2 square into eligibility planes of w0 * h0 bytes in d_elig: one plane when
// image_stride is 0, else one per pyramid slot (image j in slot j % slots, eroded with its pyramid).
constexpr int kTrackMaxMargin = 63;
struct TrackMask {
    const uint8_t* mask;
    int64_t pitch, image_stride;
    int margin;
    uint8_t* d_elig;
};
// Options of launch_track_frames beyond forward tracking.  sel null: the query points are the
// caller's (h_q_at known); otherwise the points of frame i are selected on image i into d_points (which
// holds n_frames * max_points points) and d_q_at (written here, from d_q_at[0] = 0).  fb_max > 0: every
// point kept forward is tracked back, its distance written to d_fb and its status set to 2 when the
// backward pass loses it or the distance exceeds fb_max.  mask null: no mask.
struct TrackExtra {
    const TrackSelect* sel;
    double fb_max;
    double* d_fb;
    const TrackMask* mask;
};
// Shared memory of one select_cells_kernel block staging `sample`-byte pixels
size_t track_select_smem(int cell, int block, int sample);
// Tracks every query point of frame i (d_points[2 d_q_at[i] ..], host copy h_q_at) from image i to
// image i + 1, for i in [0, n_frames).  The pyramids of `slots` (>= 2) images live in d_pyr at once
// (slots * track_pyramid_floats floats): the images are processed in chunks, image j in slot j % slots,
// each pyramid built once.  Per point: d_tracked (2 doubles) and d_status (1 = kept); *d_flag gets bit 0
// when a query point is not finite.  ex: selection, the backward pass and the mask (TrackExtra); with
// ex.sel and ex.mask null and ex.fb_max 0 the launches are the forward tracker's alone.  With a mask the
// selection takes eligible candidates only, and a point the forward pass keeps gets status 3 instead of 1
// when its query or tracked position is not eligible.  im.sample picks the kernels' pixel type.
void launch_track_frames(const TrackImages& im, int n_frames, const int64_t* h_q_at, int64_t* d_q_at,
                         double* d_points, float* d_pyr, int slots, double* d_tracked, uint8_t* d_status,
                         unsigned* d_flag, const TrackExtra& ex, cudaStream_t st);

// ---- stage probes (tests only) ---------------------------------------------------------------
void launch_probe_problem_matrix(const DeviceData& dd, FrameDesc fd, double delay, double* d_P,
                                 cudaStream_t st);
void launch_probe_log1p(const double* d_x, int n, double* d_out, cudaStream_t st);
void launch_probe_loss(const DeviceData& dd, FrameDesc fd, double delay, const double* d_m, double k,
                       double* d_out /* loss3, loss5, g0,g1,g2 */, cudaStream_t st);
void launch_probe_lbfgs(const DeviceData& dd, FrameDesc fd, double delay, double* d_m, double k,
                        double* d_f, int* d_stats, cudaStream_t st);
// mode 0: the product path (fp32 tournament, exact estimator when it cannot certify the winner);
// mode 2: the exact binary64 estimator only.  *d_n_exact is incremented when the exact one ran.
void launch_probe_guess(const DeviceData& dd, FrameDesc fd, double delay, int iters, uint64_t key_prefix,
                        int mode, double* d_mk /* m[3], k */, unsigned* d_n_exact, cudaStream_t st);

// FP64 FMA peak microbenchmark: returns elapsed ms for `iters` x 8 dependent-chain FMAs per thread
float run_fp64_peak(int blocks, int threads, int iters, double* d_sink, cudaStream_t st);

// RS_CHECKED builds: source line (engine.cu) of the first failed device-side assertion on the current
// device, 0 if none; the first call on a device arms the checks.  Always 0 in regular builds.
int checked_assert_line();

// bookkeeping for gpu_launches reporting
uint64_t launch_count();
// kernels launched through a replayed CUDA graph (the launchers only run at capture time)
void count_launches(uint64_t n);

}  // namespace rs
