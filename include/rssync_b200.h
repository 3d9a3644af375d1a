/* rssync_b200.h — C ABI of the B200-native rs-sync synchronisation loss engine.
 *
 * This is the drop-in boundary: plain pointers and sizes, `int` status codes, no C++ or torch
 * types.  Each entry point names the member of the reference's ISyncProblem interface
 * (src/core/public/rssync.h in VladimirP1/rs-sync) that it replaces; argument meaning, units
 * (seconds unless the name ends in _us) and buffer layouts are the reference's:
 *   quaternions  count x 4 doubles, (w,x,y,z) per sample
 *   rays         count x 3 doubles, xyz interleaved unit vectors
 *   ts_a / ts_b  count doubles, camera-clock seconds incl. the rolling-shutter row offset
 * Input buffers are borrowed for the duration of the call only (they are copied).
 *
 * Every function returns RSSYNC_OK (0) or an error code; rssync_last_error() gives the message
 * (for the panic conditions it is the reference's panic.txt text, core_private.cpp:76-83,
 * 159-162, 180-188, 199-202).  There is no CPU fallback: if no CUDA device is usable the calls
 * fail with RSSYNC_E_CUDA.
 *
 * The C++ class in include/rssync.h (ISyncProblem / CreateSyncProblem, same vtable layout as the
 * reference) is a thin veneer over this ABI and maps a non-zero status to the reference's
 * panic convention (write ./panic.txt, exit(1)).
 */
#ifndef RSSYNC_B200_H
#define RSSYNC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rssync_problem rssync_problem;

enum {
    RSSYNC_OK = 0,
    RSSYNC_E_INVALID = 1,   /* bad argument / unsupported shape                          */
    RSSYNC_E_NONFINITE = 2, /* a reference panic condition: non-finite data              */
    RSSYNC_E_ORDER = 3,     /* a reference panic condition: timestamps out of order      */
    RSSYNC_E_STATE = 4,     /* call protocol violated (e.g. PreSync before gyro is set)  */
    RSSYNC_E_CUDA = 5       /* CUDA runtime / device failure                             */
};

/* CreateSyncProblem()            rssync.h:31.  Uses the calling thread's current CUDA device. */
int rssync_create(rssync_problem** out);
/* The same problem spread over n_devices GPUs of this process (the "device-count option" of the
 * batch extensions; the reference is a single shared-memory process, src/core/core_private.cpp).
 * devices[0] is the primary: it takes every Set* call and holds the one complete copy of the inputs;
 * the other devices receive the finished device state (ray arena, spline records) by ncclBroadcast
 * over NVLink when a compute call finds them stale.  PreSync / DebugPreSync / rssync_presync_grid
 * shard the delay grid by offset range (one ncclAllGather of the curve slices per call),
 * rssync_sync_batch* / rssync_presync_windows shard by syncpoint, rssync_orientation_search* and
 * rssync_rotation_search by variant, rssync_readout_search by readout (results assembled on the host,
 * where the solver's control loop produces them); every
 * result is bit-identical to the single-device one.  A single rssync_sync call runs on devices[0].
 * NCCL (libnccl.so.2) is loaded at run time, only by this call and only when n_devices > 1.
 * Leaves devices[0] the calling thread's current device. */
int rssync_create_multi(const int* devices, int n_devices, rssync_problem** out);
/* number of devices the problem spans (1 for rssync_create) */
int rssync_device_count(const rssync_problem* p);
/* ISyncProblem::~ISyncProblem()  rssync.h:11 */
void rssync_destroy(rssync_problem* p);
const char* rssync_last_error(const rssync_problem* p);

/* SetGyroQuaternions(const double*, size_t, double, double)        rssync.h:13-14 */
int rssync_set_gyro_fixed(rssync_problem* p, const double* quats, size_t count, double sample_rate,
                          double first_timestamp);
/* SetGyroQuaternions(const int64_t*, const double*, size_t)        rssync.h:15-16 */
int rssync_set_gyro_var(rssync_problem* p, const int64_t* timestamps_us, const double* quats,
                        size_t count);
/* SetTrackResult(...)                                              rssync.h:17-18 */
int rssync_set_track(rssync_problem* p, int64_t frame, const double* ts_a, const double* ts_b,
                     const double* rays_a, const double* rays_b, size_t count);
/* Bulk form of SetTrackResult: n_frames frames in one call.  counts[i] rays for frames[i]; the
 * ts / ray buffers are the per-frame buffers concatenated in order.  Equivalent to n_frames
 * rssync_set_track calls. */
int rssync_set_track_batch(rssync_problem* p, size_t n_frames, const int64_t* frames,
                           const size_t* counts, const double* ts_a, const double* ts_b,
                           const double* rays_a, const double* rays_b);
/* Lens profile: Lens (core_testcode.cpp:55-61), the numbers of one line of the lens file
 * `<name> <readout_s> fx fy cx cy k1 k2 k3 k4` (README.md:52-60, lens_load :164-181). */
typedef struct rssync_lens {
    double readout, fx, fy, cx, cy, k1, k2, k3, k4;
} rssync_lens;
/* The per-frame tail of track_frames (core_testcode.cpp:134-161) followed by SetTrackResult, for
 * n_frames frames, computed on the device: points_a / points_b are the tracked pixel pairs
 * (sum(counts) x 2 doubles, x then y), frame_ts_a / frame_ts_b the two frames' timestamps in
 * seconds (cur_ts / 1000, next_ts / 1000).  Per pair: lens_undistort_point (:63-95) on both points,
 * ts = frame_ts + readout * (y / image_rows) (:144-145), unit rays (x', y', 1) / |.| (:147-154).
 * Equivalent to computing those on the host and calling rssync_set_track for each frame, up to
 * the rounding of tan / cos (CUDA's instead of libm's, <= 2 ulp).
 * Rejected before anything is applied: a lens with a non-finite field, fx or fy = 0, or k1..k4 so
 * large that a bound of |theta (1 + k1 theta^2 + .. + k4 theta^8)| or of its derivative over
 * [0, pi/2] overflows, and a non-finite or non-positive image_rows (RSSYNC_E_INVALID, "bad lens profile
 * or image height"); a non-finite frame timestamp, and a point that is not finite or whose
 * (x - cx) / fx, (y - cy) / fy or their squared norm is not (RSSYNC_E_NONFINITE, reported as the
 * ray buffer of its side: "non-finite numbers in rays_a" for points_a).  Either would give NaN rays. */
int rssync_set_track_pixels(rssync_problem* p, size_t n_frames, const int64_t* frames,
                            const size_t* counts, const double* frame_ts_a, const double* frame_ts_b,
                            const double* points_a, const double* points_b, const rssync_lens* lens,
                            double image_rows);
/* rssync_set_track_batch with the per-ray buffers in device memory of the problem's (primary) device.
 * frames / counts stay host arrays. `stream` (a cudaStream_t, may be NULL = legacy default) is the
 * stream on which the caller produced the buffers: the library orders its reads after the work queued
 * there, and has finished reading the buffers when the call returns, so the caller may overwrite or
 * free them right afterwards (the reference's borrow contract, rssync.h:15-17).
 * Results are bit-identical to rssync_set_track_batch on the same values.  A frame id given more than
 * once: the last occurrence wins.  The first frame holding a non-finite value fails the call with the
 * host form's code and message; the frames before it are applied, the others are not.  A count above
 * 512, a null buffer with rays to read, or a buffer that is not device (or managed) memory of the
 * problem's device: RSSYNC_E_INVALID, nothing applied.  The buffers need 8-byte alignment only. */
int rssync_set_track_batch_device(rssync_problem* p, size_t n_frames, const int64_t* frames,
                                  const size_t* counts, const double* ts_a, const double* ts_b,
                                  const double* rays_a, const double* rays_b, void* stream);
/* rssync_set_track_pixels with points_a / points_b in device memory; frames, counts, frame_ts_a,
 * frame_ts_b and lens stay on the host. Same ordering / borrow contract.  As in the host form,
 * everything is checked (frame timestamps first, then the points in frame order) before anything is
 * applied; results are bit-identical to it. */
int rssync_set_track_pixels_device(rssync_problem* p, size_t n_frames, const int64_t* frames,
                                   const size_t* counts, const double* frame_ts_a,
                                   const double* frame_ts_b, const double* points_a,
                                   const double* points_b, const rssync_lens* lens,
                                   double image_rows, void* stream);
/* SetTrackResult for n_frames frames whose rays the caller computed (any camera model), with the
 * rolling-shutter timestamps formed here from per-ray row fractions.  Ray k of frame i gets
 * ts_a = frame_ts_a[i] + readout * frac_a[k] (ts_b alike): one multiply and one add, not contracted,
 * the expression of the pixels forms with the caller's fraction in place of y / image_rows.  The fraction
 * is usually y / image_rows; any finite value is accepted (x / width for a sensor read along columns).
 * counts / frames and the per-ray buffers use rssync_set_track_batch's layouts: frac_a / frac_b 1 double
 * per ray, rays_a / rays_b 3, concatenated in `frames` order.
 * Afterwards the problem holds, byte for byte, what rssync_set_track_batch with those timestamps gives
 * (frame table, arena tiles, orig / pos) and every later call returns what it would return on that
 * problem.  The frames also keep their row fractions and frame timestamps, so rssync_readout_search and
 * rssync_set_readout accept them, alone or beside pixel-ingested frames; a frame that a rays form or an
 * adoption overwrites later loses them.  A frame id given more than once: the last occurrence wins.
 * Everything is checked before anything is applied: a null argument, a count above 512 or a non-finite
 * readout: RSSYNC_E_INVALID; then non-finite frame timestamps (as rssync_set_track_pixels); then, frame
 * by frame, the first frame holding a non-finite value fails with rssync_set_track_batch's code and
 * message for rays_a, rays_b, ts_a, ts_b in that order, where a non-finite fraction, or a timestamp that
 * overflows, counts as a non-finite ts. */
int rssync_set_track_row_fractions(rssync_problem* p, size_t n_frames, const int64_t* frames,
                                   const size_t* counts, const double* frame_ts_a, const double* frame_ts_b,
                                   const double* frac_a, const double* frac_b,
                                   const double* rays_a, const double* rays_b, double readout);
/* The same with frac_a / frac_b / rays_a / rays_b in device memory of the problem's (primary) device;
 * frames, counts and the frame timestamps stay on the host.  Same ordering / borrow contract as
 * rssync_set_track_batch_device; a per-ray buffer that is not device (or managed) memory of the
 * problem's device: RSSYNC_E_INVALID.  Results are bit-identical to the host form. */
int rssync_set_track_row_fractions_device(rssync_problem* p, size_t n_frames, const int64_t* frames,
                                          const size_t* counts, const double* frame_ts_a,
                                          const double* frame_ts_b, const double* frac_a,
                                          const double* frac_b, const double* rays_a, const double* rays_b,
                                          double readout, void* stream);
/* PreSync(initial_delay, frame_begin, frame_end, search_step, search_radius) -> {cost, delay}
 *                                                                  rssync.h:19-21 */
int rssync_presync(rssync_problem* p, double initial_delay, int64_t frame_begin, int64_t frame_end,
                   double search_step, double search_radius, double* out_cost, double* out_delay);
/* Sync(initial_delay, frame_begin, frame_end, search_center, search_radius) -> {cost, delay}
 *                                                                  rssync.h:22-24 */
int rssync_sync(rssync_problem* p, double initial_delay, int64_t frame_begin, int64_t frame_end,
                double search_center, double search_radius, double* out_cost, double* out_delay);
/* DebugPreSync(initial_delay, frame_begin, frame_end, search_radius, delays, costs, point_count)
 *                                                                  rssync.h:26-28 */
int rssync_debug_presync(rssync_problem* p, double initial_delay, int64_t frame_begin,
                         int64_t frame_end, double search_radius, double* delays, double* costs,
                         int point_count);

/* ---- extensions (no counterpart in the reference interface) ------------------------------- */

/* Loss curve on an arbitrary delay list over frames [frame_begin, frame_end): the body of
 * pre_sync's outer loop (core_private.cpp:69-88).  offset_index_base is the index of delays[0]
 * in the caller's full grid (it keys the RNG), so a grid can be sharded across processes/GPUs
 * and still reproduce the single-GPU curve bit for bit.  stream: 1 = PreSync, 2 = DebugPreSync.
 * Does not advance the call counter. */
int rssync_presync_grid(rssync_problem* p, int64_t frame_begin, int64_t frame_end,
                        const double* delays, int n, int stream, uint64_t call_no,
                        uint64_t offset_index_base, double* costs, unsigned* nonfinite_flags);
/* n PreSync calls — frame windows [frame_begin[i], frame_end[i]), one shared (initial_delay,
 * search_step, search_radius) — evaluated as one grid launch; the syncpoint loop of
 * core_testcode.cpp:303-312 issues them one by one.  Result i equals the i-th of n consecutive
 * rssync_presync calls.  call_nos[i] keys the RNG of window i; NULL = consecutive values of the
 * problem's counter, which then advances by n. */
int rssync_presync_windows(rssync_problem* p, int n, double initial_delay, const int64_t* frame_begin,
                           const int64_t* frame_end, double search_step, double search_radius,
                           const uint64_t* call_nos, double* out_cost, double* out_delay);
/* pre_sync's delay grid (core_private.cpp:69-70, floating-point accumulation included).
 * Returns the number of points; fills at most `cap` of them. */
int rssync_presync_delays(double initial_delay, double search_step, double search_radius,
                          double* out, int cap);

/* n independent Sync calls advanced side by side on the device (lanes of syncpoints); result i
 * equals what the i-th of n consecutive rssync_sync calls would return. */
int rssync_sync_batch(rssync_problem* p, int n, const double* initial_delay,
                      const int64_t* frame_begin, const int64_t* frame_end,
                      const double* search_center, const double* search_radius, double* out_cost,
                      double* out_delay);
/* Same, with an explicit RNG call number per syncpoint (call_nos[i]) instead of consecutive values
 * of the problem's counter, which is left untouched: lets several processes / GPUs each run a
 * subset of a syncpoint list and reproduce exactly what one process would have computed. */
int rssync_sync_batch_ex(rssync_problem* p, int n, const double* initial_delay,
                         const int64_t* frame_begin, const int64_t* frame_end,
                         const double* search_center, const double* search_radius,
                         const uint64_t* call_nos, double* out_cost, double* out_delay);
/* Per-iteration record of the most recent rssync_sync call (delay after the step, |step|), the
 * two numbers the reference prints to stderr (core_private.cpp:330).  Returns entries written. */
int rssync_last_sync_trace(const rssync_problem* p, double* delays, double* steps, int cap);

/* The caller-side step before SetGyroQuaternions, optdata_fill_gyro (core_testcode.cpp:37-53):
 * q_0 = identity, q_i = normalise(quat_from_aa(w_i (t_i - t_{i-1})) (x) q_{i-1}).  gyro_xyz: count x 3
 * rad/s; timestamps in seconds; quats_out: count x 4 (w,x,y,z).  orientation: a gyro_orientation
 * string of the reference's config (core_testcode.cpp:186-190) or NULL for "XYZ"; character i names
 * the input axis routed to output axis i, lower case flips its sign.  (The reference delegates
 * this mapping to the third-party telemetry-parser crate; the convention here is ours.)  Host code;
 * the orientation search runs the same arithmetic on the device.  Order of operations (part of the
 * arithmetic contract, because every step normalises): the recurrence runs inside blocks of 512
 * samples from the identity, the blocks are chained through their last values, and every sample is
 * its block-local value times its block's prefix, normalised; sin / cos are the contract's
 * (csrc/spec_trig.h).  Differs from one sequential recurrence with libm by rounding only. */
int rssync_integrate_gyro(const double* timestamps_s, const double* gyro_xyz, size_t count,
                          const char* orientation, double* quats_out);
/* rssync_integrate_gyro with the axis mapping given as a 3x3 row-major matrix M (NULL = identity):
 * w = M g per sample, then the same blocked integration.  Arithmetic of w (part of the contract):
 * w_c = sum over the j with M[c][j] != 0 of M[c][j] g_j -- terms with a zero coefficient are omitted,
 * the first kept term is the product, the others are added left to right, without contraction --
 * and w_c = +0.0 when row c is zero; then a_c = w_c dt.  A gyro_orientation string is the signed
 * permutation matrix with M[i][src] = +-1 for its character i, and under this rule it gives the string's
 * bits exactly (signs of zeros and a NaN or inf on an axis it does not read included):
 * rssync_integrate_gyro(s) == rssync_integrate_gyro_matrix(matrix of s).  Any finite matrix is
 * accepted (a rotation is the usual case; a diagonal models a gyro gain error); a non-finite entry
 * gives RSSYNC_E_INVALID.  Host code; the searches run the same arithmetic on the device. */
int rssync_integrate_gyro_matrix(const double* timestamps_s, const double* gyro_xyz, size_t count,
                                 const double* matrix, double* quats_out);
/* The orientation search the reference keeps commented out in core_testcode.cpp:184-233 (README.md:
 * 47-48, guess_orient): for each of n_orient gyro_orientation strings, integrate the raw gyro,
 * ingest it through the variable-rate SetGyroQuaternions (timestamps truncated to integer
 * microseconds, :47-50) and run PreSync(initial_delay, frame_begin, frame_end, step, radius).
 * out_cost[i], out_delay[i] = the i-th PreSync result; sort by cost to rank the variants (:226).
 * Equivalent to that sequence of calls on this problem, RNG call counter included; the problem
 * is left holding the last variant's gyro. */
int rssync_orientation_search(rssync_problem* p, const double* timestamps_s, const double* gyro_xyz,
                              size_t count, const char* const* orientations, int n_orient,
                              double initial_delay, int64_t frame_begin, int64_t frame_end,
                              double search_step, double search_radius, double* out_cost,
                              double* out_delay);
/* The same with the RNG call number of every variant given explicitly (call_nos[i] keys variant i's
 * PreSync; the problem's counter is left as it was), so that a subset of the variants evaluated on
 * another GPU reproduces the single-process search; call_nos == NULL: as above. */
int rssync_orientation_search_ex(rssync_problem* p, const double* timestamps_s, const double* gyro_xyz,
                                 size_t count, const char* const* orientations, int n_orient,
                                 double initial_delay, int64_t frame_begin, int64_t frame_end,
                                 double search_step, double search_radius, const uint64_t* call_nos,
                                 double* out_cost, double* out_delay);
/* The orientation search over n_rot arbitrary axis mappings (n_rot x 9, 3x3 row-major each) in place
 * of the strings: a search over camera mount rotations (a camera tilted against the gyro that logs it).
 * Result i equals rssync_integrate_gyro_matrix(matrices + 9 i) -> rssync_set_gyro_var (timestamps
 * truncated to integer microseconds) -> rssync_presync keyed by call_nos[i] (NULL: the counter, which
 * advances by n_rot).  out_curves (n_rot x D or NULL): row i = that PreSync's cost over
 * rssync_presync_delays(initial_delay, search_step, search_radius).  The problem is left holding the
 * last variant's gyro.  A non-finite matrix entry gives RSSYNC_E_INVALID ("rotation-search: matrix <i>
 * has a non-finite entry") before anything is done: the counter and the gyro are left as they were.
 * matrices == NULL with n_rot > 0: RSSYNC_E_INVALID.  Otherwise it behaves as rssync_orientation_search_ex,
 * errors and multi-device sharding by variant included. */
int rssync_rotation_search(rssync_problem* p, const double* timestamps_s, const double* gyro_xyz,
                           size_t count, const double* matrices, int n_rot, double initial_delay,
                           int64_t frame_begin, int64_t frame_end, double search_step,
                           double search_radius, const uint64_t* call_nos, double* out_cost,
                           double* out_delay, double* out_curves);

/* Rolling-shutter readout search: PreSync(initial_delay, frame_begin, frame_end, search_step, search_radius)
 * at each of n_readouts candidate readouts (seconds, as rssync_lens.readout), without re-ingesting.  Every
 * frame in [frame_begin, frame_end) must have been ingested by rssync_set_track_pixels(_device) or
 * rssync_set_track_row_fractions(_device) and not been overwritten by a rays form or adopted since (else
 * RSSYNC_E_STATE naming the frame): those keep the row fraction of every ray (y / image_rows, or the
 * caller's) on the device and their frame timestamps on the host.  Result j equals, bit for bit,
 * rssync_presync on a problem that ingested the same input (pixels, lens and image rows, or rays and row
 * fractions) and frame timestamps with readout = readouts[j], keyed by RNG call number call_nos[j] (NULL: consecutive
 * values of the problem's counter, which then advances by n_readouts); out_curves (n_readouts x D, or
 * NULL) row j is that call's cost over rssync_presync_delays(initial_delay, search_step, search_radius).
 * The problem's arena, frame table and gyro are left as they are.  A non-finite readout or n_readouts < 0:
 * RSSYNC_E_INVALID; n_readouts == 0: nothing done.  Otherwise rssync_presync's errors.  A multi-device
 * problem (n_readouts > 1) shards the readouts: every check runs on devices[0] first, then each device
 * runs a contiguous share of them on its own scratch arena.  The row fractions (the plane and the
 * re-timing table) reach the other devices by one grouped ncclBroadcast, sent only by a search that
 * finds their copy stale (after an ingest, an overwrite, arena growth or an adoption).  Results, errors,
 * the counter and the grid statistics equal the single-device search's. */
int rssync_readout_search(rssync_problem* p, const double* readouts, int n_readouts, double initial_delay,
                          int64_t frame_begin, int64_t frame_end, double search_step, double search_radius,
                          const uint64_t* call_nos, double* out_cost, double* out_delay, double* out_curves);
/* Apply a readout: re-time the frames of [frame_begin, frame_end), ingested from pixels or row fractions,
 * in place, so that the problem holds, byte for byte, what ingesting them with readout = readout gives
 * (arena tiles, orig / pos, frame table) and every later call returns what it would return on that
 * problem.  Frames ingested later use the readout of their own call.  Errors as rssync_readout_search's.
 * A multi-device problem re-times on devices[0]; the other devices receive the arena at the next compute
 * call, as after any Set* call. */
int rssync_set_readout(rssync_problem* p, double readout, int64_t frame_begin, int64_t frame_end);

/* Pinned RNG of the randomised translation estimator (replaces the reference's
 * random_device-seeded mt19937, inline_utils.hpp:13-17).  Default seed 100, call counter 0; the
 * counter advances by one per PreSync / DebugPreSync / Sync call. */
int rssync_set_rng(rssync_problem* p, uint64_t seed, uint64_t call_no);
uint64_t rssync_call_counter(const rssync_problem* p);

/* Loss mode.  RSSYNC_LOSS_FULL (default) is the reference's loss.  RSSYNC_LOSS_SIMPLIFIED is the
 * "simplified" variant of the thesis (pdf-p.27-28, section 2.11: the robust loss with the
 * translation vector removed, a 1-D problem in the delay; no code for it in the reference
 * checkout, so the definition is this engine's): the residual of a ray pair is |ar x br| itself
 * -- the de-rotated rays of a purely rotating camera coincide -- instead of its component along
 * the per-frame translation direction.  With r_i = |P_i| (P = opt_compute_problem's rows):
 *   PreSync / DebugPreSync, per (delay, frame): k = clamp(100 / |r|_2, 10, 1000),
 *       cost = sqrt(sum_i sqrt(log1p((r_i k)^2)))   (the aggregation of core_private.cpp:79-85);
 *   Sync: k per frame from the initial delay, objective sum_frames sum_i log1p((r_i k)^2), the same
 *       central-difference gradient, Backtrack and momentum loop (core_private.cpp:298-331); no
 *       translation estimator, no per-frame L-BFGS, no random numbers.
 * Faster (no estimator); loses accuracy on translation-heavy footage (thesis Fig. 9-10). */
enum { RSSYNC_LOSS_FULL = 0, RSSYNC_LOSS_SIMPLIFIED = 1 };
int rssync_set_loss_mode(rssync_problem* p, int mode);

/* Run the problem's kernels on the given cudaStream_t (default: the legacy default stream). */
int rssync_set_stream(rssync_problem* p, void* cuda_stream);
/* Record CUDA events around the PreSync grid kernel so rssync_get_stats can report its device
 * time (default off). */
int rssync_set_kernel_timing(rssync_problem* p, int enabled);
/* Push any pending host-side ray / gyro data to the device now (otherwise done lazily by the
 * first compute call). */
int rssync_flush(rssync_problem* p);

typedef struct rssync_stats {
    uint64_t kernel_launches;  /* kernels launched by this library (process-wide)              */
    uint64_t h2d_bytes;        /* bytes copied host->device by this problem                     */
    uint64_t d2h_bytes;        /* bytes copied device->host by this problem                     */
    uint64_t frames;           /* frames currently held                                         */
    uint64_t rays;             /* rays currently held                                           */
    uint64_t gyro_samples;     /* samples of the (resampled) gyro track                         */
    uint64_t sync_outer_iters; /* outer iterations of the most recent Sync / Sync batch         */
    uint64_t sync_lbfgs_evals; /* objective evaluations inside L-BFGS, most recent Sync / batch */
    double last_grid_kernel_ms; /* device time of the most recent PreSync grid kernel (CUDA events
                                   on the problem's stream), 0 if timing is off                  */
    uint64_t last_grid_tasks;       /* (delay, frame) tasks of the most recent PreSync grid      */
    uint64_t last_grid_exact_tasks; /* of those, tasks whose translation estimate was redone by
                                       the exact binary64 estimator (fp32 tournament undecided) */
    /* evaluation accounting of the most recent Sync / Sync batch (SURVEY 8d "Algorithmic work for
     * Sync"), in (syncpoint, frame) tasks: */
    uint64_t sync_row_builds;   /* problem-matrix builds (opt_compute_problem, core_private.cpp:15-32) */
    uint64_t sync_loss_evals;   /* objective evaluations outside L-BFGS: x0, x0 -/+ h, Backtrack's
                                   trial points, the final objective                               */
    uint64_t sync_init_tasks;   /* estimator runs of the initialisation, 200 hypotheses each (:127)  */
    uint64_t sync_outer_total;  /* outer iterations summed over the batch's syncpoints             */
    uint64_t nccl_calls;        /* collectives (grouped calls) issued by a multi-device problem     */
    uint64_t broadcast_bytes;   /* bytes per replica replicated from the primary so far             */
} rssync_stats;
int rssync_get_stats(const rssync_problem* p, rssync_stats* out);

/* ---- moving a problem's finished device state (replication without re-ingesting) ---------
 * A problem that has ingested its inputs holds, on its device: the ray arena (arena_rays x 8
 * doubles in 2 KB tiles), the orig / pos planes (arena_rays int32 each) and the spline records
 * (gyro_samples x 16 doubles).  rssync_device_state flushes pending host data and returns those
 * device pointers and sizes; rssync_frame_table returns the host-side frame table (returns the
 * number of frames; fills at most cap); rssync_adopt_state prepares ANOTHER problem (other GPU or
 * other process) to hold a copy: it registers the frame table and sizes and allocates the buffers,
 * whose pointers rssync_device_state then returns for the caller to fill by whatever transport
 * it has (ncclBroadcast over NVLink in bench.py; rssync_create_multi does the same internally).
 * Results of the adopting problem equal the source's bit for bit.  An adopted state comes without row
 * fractions: rssync_readout_search / rssync_set_readout need them too (rssync_adopt_row_fractions). */
typedef struct rssync_frame_desc {
    int64_t id;
    int32_t off, n;
    double ts_lo, ts_hi;
} rssync_frame_desc;
typedef struct rssync_device_state_t {
    void* rays;
    void* orig;
    void* pos;
    void* spline_records;
    size_t arena_rays, gyro_samples;
    double sample_rate, first_timestamp;
} rssync_device_state_t;
int rssync_frame_table(const rssync_problem* p, rssync_frame_desc* out, size_t cap);
int rssync_device_state(rssync_problem* p, rssync_device_state_t* out);
int rssync_adopt_state(rssync_problem* p, const rssync_frame_desc* frames, size_t n_frames,
                       size_t arena_rays, size_t gyro_samples, double sample_rate,
                       double first_timestamp);

/* The row fractions of an adopted state, so that the adopting problem can run rssync_readout_search and
 * rssync_set_readout too.  The same three steps as above:
 * rssync_retime_table (host only): the frames that hold row fractions, ascending id, with their frame
 *   timestamps; returns their number, fills at most cap.
 * rssync_row_fraction_plane: flushes like rssync_device_state, then *plane = the row-fraction plane
 *   (2 doubles per arena ray, indexed by arena offset like the arena; *n_doubles = 2 * arena_rays),
 *   NULL / 0 when no frame holds row fractions.
 * rssync_adopt_row_fractions: on a problem whose state came from rssync_adopt_state with no Set* call
 *   since (else RSSYNC_E_STATE), registers the table and allocates the plane.  An id not in the adopted
 *   frame table, an id given twice, a non-finite timestamp or frames == NULL with n > 0:
 *   RSSYNC_E_INVALID, the problem unchanged.  The caller then fills the plane through
 *   rssync_row_fraction_plane and announces the stream that writes it with
 *   rssync_expect_chunk(p, 0, arena_rays, stream): the re-timing waits for it.  A later
 *   rssync_adopt_state, or a rays form overwriting a frame, drops the frame's row fractions. */
typedef struct rssync_retime_desc {
    int64_t id;
    double frame_ts_a, frame_ts_b;
} rssync_retime_desc;
int rssync_retime_table(const rssync_problem* p, rssync_retime_desc* out, size_t cap);
int rssync_row_fraction_plane(rssync_problem* p, double** plane, size_t* n_doubles);
int rssync_adopt_row_fractions(rssync_problem* p, const rssync_retime_desc* frames, size_t n);

/* Pipelined form of the same, for a source that has just taken a bulk SetTrackResult whose chunks are
 * still on their way to its device.  rssync_device_state_pipelined returns the pointers WITHOUT
 * waiting for the device, plus the arena ranges [lo, hi) (in rays) of the ingest chunks in flight
 * (n_chunks of them; at most cap are written).  rssync_stream_wait_chunk makes `stream` (a
 * cudaStream_t of the caller) wait for chunk k to have landed (k = -1: for everything queued on the
 * problem's own stream so far, i.e. the spline records and frames set one by one), so the caller can
 * send each chunk on as soon as it is there.  On the receiving side, rssync_expect_chunk tells the
 * adopting problem that the arena range [lo, hi) is being written by work queued on `stream`: a
 * PreSync grid that follows evaluates each frame as soon as the chunks covering it have arrived, as
 * it does behind its own ingest.  rssync_note_reader: work queued on `stream` still reads this
 * problem's device state; the next Set* call waits for it before overwriting anything. */
int rssync_device_state_pipelined(rssync_problem* p, rssync_device_state_t* out, size_t* chunk_lo,
                                  size_t* chunk_hi, size_t cap, size_t* n_chunks);
int rssync_stream_wait_chunk(rssync_problem* p, int k, void* stream);
int rssync_expect_chunk(rssync_problem* p, size_t lo, size_t hi, void* stream);
int rssync_note_reader(rssync_problem* p, void* stream);

/* FP64 FMA throughput of the current device in TFLOP/s (FMA = 2 flop): the measured denominator
 * of the FP64 roofline. */
int rssync_measure_fp64_peak(double* tflops);

/* ---- stage probes: expose intermediate results of the device path for parity tests -------- */
int rssync_probe_gyro(const rssync_problem* p, double* sample_rate, double* first_timestamp,
                      size_t* count, double* spline_records /* count*16 or NULL */);
/* Host-only (no device needed): the eliminated tridiagonal system of the natural cubic spline through
 * `count` quaternions (count x 4), as SetGyroQuaternions builds it before the records are finished
 * on the device: rhs (count x 4) and diag (count); c = rhs / diag (minispline.cpp:3-34). */
int rssync_probe_spline_system(const double* quats, size_t count, double* rhs, double* diag);
int rssync_probe_problem_matrix(rssync_problem* p, int64_t frame, double delay, double* rows);
int rssync_probe_guess_motion(rssync_problem* p, int64_t frame, double delay, int iters, int stream,
                              uint64_t call_no, uint64_t offset_index, double* m3, double* k);
/* mode 0: the product path (fp32 tournament + exact estimator when undecided); mode 2: exact
 * binary64 estimator only.  *used_exact = 1 when the exact estimator ran. */
int rssync_probe_guess_motion_ex(rssync_problem* p, int64_t frame, double delay, int iters,
                                 int stream, uint64_t call_no, uint64_t offset_index, int mode,
                                 double* m3, double* k, int* used_exact);
int rssync_probe_loss(rssync_problem* p, int64_t frame, double delay, const double* m3, double k,
                      double* loss3, double* loss5, double* grad3);
int rssync_probe_lbfgs(rssync_problem* p, int64_t frame, double delay, double* m3, double k,
                       double* f, int* iters, int* evals);
int rssync_probe_log1p(const double* x, int n, double* out);
/* Host-only: the pieces a multi-device problem's replication sends for n ingest chunks in flight
 * ([lo, hi) arena ranges in stream order) over an arena of arena_rays, grouped into at most `groups`
 * pieces behind whatever is already on the device (k_last = -1).  Returns the number of pieces
 * (at most cap are written), -1 on bad arguments. */
int rssync_probe_replication_plan(const size_t* lo, const size_t* hi, size_t n, size_t arena_rays,
                                  size_t groups, int* k_last, size_t* piece_lo, size_t* piece_hi,
                                  size_t cap);

/* Host-only: the checked staging copy of the bulk SetTrackResult (n doubles src -> dst; *all_finite = 0
 * when a value is NaN or infinite; [*lo, *hi] widened to the values when both are given), in one of
 * its three forms: mode 0 scalar, 1 AVX2, 2 AVX2 with non-temporal stores.  The forms are
 * interchangeable bit for bit (tests). */
int rssync_probe_stage_copy(const double* src, size_t n, int mode, double* dst, double* lo, double* hi,
                            int* all_finite);

/* sin (which = 0), cos (1), acos (2) of the arithmetic contract (csrc/spec_trig.h), evaluated by the
 * library's host code (on_device = 0, no GPU needed) or by a kernel */
int rssync_probe_spec_trig(const double* x, int n, int which, int on_device, double* out);

#ifdef __cplusplus
}
#endif
#endif /* RSSYNC_B200_H */
