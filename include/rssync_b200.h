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
 * rssync_rotation_search(_windows) by variant, rssync_readout_search(_windows) by readout (results
 * assembled on the host,
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
 * ray buffer of its side: "non-finite numbers in rays_a" for points_a).  Either would give NaN rays.
 * A frame id given more than once: the last occurrence wins. */
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
/* Parameters of rssync_track_frames_device (NULL there = the defaults shown). */
typedef struct rssync_track_params {
    int levels;     /* pyramid levels, 1..6 (default 3) */
    int window;     /* odd window side in pixels, 5..63 (default 21) */
    int max_iters;  /* LK iterations per level, 1..100 (default 30) */
    double epsilon; /* stop when |delta| < epsilon px (default 0.01) */
    double min_eig; /* lost when the minimum eigenvalue of G / window^2 < this (default 1e-4) */
} rssync_track_params;
/* Track points between decoded frames on the device, then ingest the pairs (the first half of
 * track_frames, core_testcode.cpp:97-162, with sparse pyramidal Lucas-Kanade in place of dense flow).
 * images: n_frames + 1 8-bit luma planes in device (or managed) memory of the problem's (primary)
 * device, `height` rows of `pitch` bytes each (pitch >= width), planes back to back: row y of image j
 * starts at images + (j * height + y) * pitch (an NV12 Y plane as decoded, a strided uint8 tensor).
 * Frame i (id frames[i]) pairs image i (timestamp image_ts[i], seconds) with image i + 1
 * (image_ts[i + 1]); points (device, sum(counts) x 2 doubles, x then y, frames concatenated) are its query
 * points on image i.  A clip goes in batches that overlap by one image.
 * Every point is tracked from image i to image i + 1.  The kept points then give exactly, byte for byte,
 * what rssync_set_track_pixels_device gives with points_a = the kept query points, points_b = their
 * tracked positions, counts = the kept counts (a frame may keep 0), frame_ts_a / frame_ts_b =
 * image_ts[i] / image_ts[i + 1] and image_rows = height: frame table, arena, row fractions and re-timing
 * table, so rssync_readout_search(_windows) and rssync_set_readout accept the frames.  The call counter
 * and the gyro are untouched.
 * A point is lost (status 0, not ingested) when it starts or ends outside [0, width - 1] x [0, height - 1],
 * when the minimum-eigenvalue test fails at any level, or when an update is not finite.  tracked_out
 * (sum(counts) x 2) and status_out (sum(counts) bytes), device memory or NULL, receive every point's
 * position and status; a point lost before its last level has ended gets NaN.
 * Algorithm (float32 throughout, evaluated in the order written; a sum over a window: lane k of a warp
 * adds the pixels t = k, k + 32, ... of the row-major window in that order, then the 32 partials are
 * combined by the butterfly xor 16, 8, 4, 2, 1):
 *  - Pyramid: level 0 is the plane as given.  Level l + 1 has size ((w + 1) / 2, (h + 1) / 2); its pixel
 *    (X, Y) is the [1 4 6 4 1] / 16 blur of level l at (2X, 2Y) with BORDER_REFLECT_101: per row
 *    r = (s[-2] + s[2]) + 4 (s[-1] + s[1]) + 6 s[0], then the same over the rows r, times 1/256
 *    (cv2.pyrDown of float32 input).  Images are processed in chunks whose pyramids fit 256 MiB of
 *    scratch (at least 2 images): max(2, floor(2^26 / floats of levels 1..levels-1 of one image)); each
 *    image's pyramid is built once; the chunks change no result.
 *  - A level is read at integer (x, y) clamped to the level (the nearest edge pixel), and at sub-pixel
 *    (x0 + ax, y0 + ay), x0 = floor: (1 - ay)((1 - ax) I00 + ax I01) + ay((1 - ax) I10 + ax I11).
 *  - LK (Bouguet), coarse to fine, guess g = 0 at level levels - 1, g = 2 (g + v) going down a level.
 *    At level l the query point is p = (float)q * 2^-l.  Side a: the (window + 2)^2 samples A at p + (dx, dy),
 *    |dx|, |dy| <= window / 2 + 1; gradients over the window: Ix = (3 (A[-1][+1] - A[-1][-1]) +
 *    10 (A[0][+1] - A[0][-1]) + 3 (A[+1][+1] - A[+1][-1])) / 32, Iy alike with rows and columns swapped;
 *    G = [sum Ix^2, sum Ix Iy; ., sum Iy^2].  Lost unless ((gxx + gyy) - sqrt((gxx - gyy)^2 +
 *    4 gxy^2)) / (2 window^2) >= min_eig.  Then, from v = 0, up to max_iters times: b = sum (A - B) [Ix, Iy]
 *    with B the side-b samples at p + g + v + (dx, dy), delta = G^-1 b = ((gyy bx - gxy by) / det,
 *    (gxx by - gxy bx) / det), det = gxx gyy - gxy^2; lost if delta is not finite; v += delta; stop when
 *    |delta|^2 < epsilon^2.  The tracked position is q + (double)(g + v) of level 0.
 * Checked before anything is applied: RSSYNC_E_INVALID for images / points (or a non-NULL output) that are
 * not device memory of the problem's device, pitch < width, width or height below window * 2^(levels - 1),
 * params out of range, a count above 512, and the lens / image-height checks of the pixels forms;
 * RSSYNC_E_NONFINITE for a non-finite image_ts (reported as the pixels forms report frame timestamps, with
 * image_ts[0..n_frames) the a side) and a non-finite query point ("non-finite numbers in rays_a").
 * Ordering and borrowing as in the other _device forms: reads are ordered after `stream`, and the library
 * has finished with images and points when the call returns.  A multi-device problem ingests on its
 * primary; the replicas receive the arena at the next compute call.  A frame id given more than once: the last
 * occurrence wins (its kept pairs are ingested; tracked_out and status_out still cover every point). */
int rssync_track_frames_device(rssync_problem* p, size_t n_frames, const int64_t* frames, const size_t* counts,
                               const double* image_ts, const double* points, const uint8_t* images, size_t pitch,
                               int width, int height, const rssync_lens* lens, const rssync_track_params* params,
                               double* tracked_out, uint8_t* status_out, void* stream);
/* Options of rssync_track_frames_ex_device (NULL there = the defaults shown). */
typedef struct rssync_track_options {
    int cell;          /* selection cell side in px, 16..128 (default 128) */
    int block;         /* structure-tensor window side, 3, 5 or 7 (default 5) */
    double quality;    /* keep a cell's pick only if score >= quality * image max, (0, 1] (default 0.01) */
    int max_points;    /* per frame when selecting, 1..512 (default 512) */
    double fb_max;     /* forward-backward threshold in px, >= 0; 0 = no backward pass (default 1.0) */
} rssync_track_options;
/* rssync_track_frames_device with two more steps: the query points may be chosen on the device, and
 * every point kept forward may be tracked back and rejected when it does not return.
 * points and counts both non-NULL: the caller's query points, as in rssync_track_frames_device.  Both
 * NULL: the points of frame i are selected on image i (below).  Only one NULL: RSSYNC_E_INVALID.
 * Outputs, each may be NULL, hold sum(counts) points, frames concatenated (in selection mode size the
 * device buffers for n_frames * max_points): points_out (device, 2 doubles per point: the query points),
 * counts_out (host, n_frames), tracked_out (device, 2 doubles), status_out (device, 1 byte) and fb_out
 * (device, 1 double).  counts_out comes back in the ingest's one round trip.
 * Status: 0 lost (as in rssync_track_frames_device), 1 kept and ingested, 2 tracked forward but rejected
 * by the backward check (tracked_out holds the forward position).  fb_out: the forward-backward distance
 * of each point the backward pass kept, NaN for every other point.
 * The kept points (status 1) give exactly what rssync_set_track_pixels_device gives on them, as stated at
 * rssync_track_frames_device; a frame whose points are all lost or rejected is ingested with 0 rays.
 * With the caller's points and fb_max = 0 the call equals rssync_track_frames_device.
 * Selection (float32, evaluated in the order written, no contraction; I = (float)plane[y][x]; reads
 * outside the image use BORDER_REFLECT_101, though no candidate's score or its neighbours' reach one):
 *  - Gradients (3 x 3 Sobel): dx = (((I[y-1][x+1] - I[y-1][x-1]) + 2 (I[y][x+1] - I[y][x-1])) +
 *    (I[y+1][x+1] - I[y+1][x-1])) * s, dy the same with rows and columns swapped,
 *    s = (float)(1.0 / (4 block 255)).
 *  - Sxx, Sxy, Syy: block x block sums of dx dx, dx dy, dy dy, each row summed left to right first, then
 *    the row sums top to bottom.  Score: (a + c) - sqrt((a - c)^2 + b^2), a = 0.5 Sxx, c = 0.5 Syy,
 *    b = Sxy (cv2.cornerMinEigenVal(img, block, 3)).
 *  - Candidate: x in [m, w - 1 - m], y in [m, h - 1 - m] with m = block / 2 + 2, score > 0, and score >=
 *    each of its 8 neighbours' scores.
 *  - Cells: cell x cell squares from (0, 0), the last row and column may be partial.  A cell's pick is
 *    its candidate of greatest score, a tie going to the smallest y w + x.  This cell rule stands in for
 *    cv2.goodFeaturesToTrack's greedy minDistance, which is sequential.
 *  - Threshold: M is the greatest pick score of the image; a pick is kept iff score >= (float)quality M.
 *    When more than max_points picks are kept, those with the greatest score stay, a tie going to the
 *    smaller cell index (row-major).
 *  - The points: the kept picks in ascending row-major cell order, ((double)x, (double)y).
 * Forward-backward (fb_max > 0): for a point q kept forward at t, the tracker above runs from image i + 1
 * to image i with query t, giving u (or losing the point); fb = sqrt((u.x - q.x)^2 + (u.y - q.y)^2) in
 * double; status 2 when u is lost or !(fb <= fb_max), else 1.  fb_max = 0 skips the backward pass.
 * Checked before anything is applied, besides the checks of rssync_track_frames_device: RSSYNC_E_INVALID
 * for an option out of range, in selection mode width or height below 2 (block / 2 + 2) + 1 or more than
 * 65536 cells per image, and outputs that are neither NULL nor device memory of the problem's device. */
int rssync_track_frames_ex_device(rssync_problem* p, size_t n_frames, const int64_t* frames, const size_t* counts,
                                  const double* image_ts, const double* points, const uint8_t* images, size_t pitch,
                                  int width, int height, const rssync_lens* lens, const rssync_track_params* params,
                                  const rssync_track_options* options, double* points_out, size_t* counts_out,
                                  double* tracked_out, uint8_t* status_out, double* fb_out, void* stream);
/* rssync_track_frames_ex_device on 16-bit luma planes (P010 / P016, 10- or 12-bit decoder output).
 * images: n_frames + 1 planes of uint16_t samples, `height` rows of `pitch` BYTES each, row y of image j at
 * (const uint8_t*)images + (j * height + y) * pitch.  The one difference from rssync_track_frames_ex_device:
 * the level-0 intensity is I = (float)v * 2^-shift, v the 16-bit sample, in place of (float)plane[y][x]
 * (pyramid, bilinear reads, LK and selection).  shift 0..8: 8 for P010 / P016 (sample in the most
 * significant bits), 2 for 10-bit and 4 for 12-bit samples in the least significant bits; with the right
 * shift intensities span [0, 256), so min_eig, quality and the Sobel scale keep their 8-bit meaning.  Every
 * other word of the contract above stands as written: statuses, outputs, the ingest identity with
 * rssync_set_track_pixels_device, ordering and borrowing, multi-device behaviour.
 * Identities: v < 2^16 is exact in float32 and the scaling by a power of two is exact, so for an 8-bit
 * plane P and any shift, the 16-bit plane v = P << shift gives byte for byte what
 * rssync_track_frames_ex_device gives on P (every output, frame table, arena, row fractions and re-timing
 * table); likewise a P010 plane (x << 6, shift 8) gives what the LSB-aligned plane x gives with shift 2.
 * There is no 16-bit form of rssync_track_frames_device: with the caller's points and fb_max = 0 this call
 * equals it.
 * Checked before anything is applied, besides the checks of rssync_track_frames_ex_device: RSSYNC_E_INVALID
 * for shift outside 0..8, images not 2-byte aligned, and an odd pitch or pitch < 2 width. */
int rssync_track_frames16_device(rssync_problem* p, size_t n_frames, const int64_t* frames, const size_t* counts,
                                 const double* image_ts, const double* points, const uint16_t* images,
                                 size_t pitch /* bytes */, int width, int height, int shift,
                                 const rssync_lens* lens, const rssync_track_params* params,
                                 const rssync_track_options* options, double* points_out, size_t* counts_out,
                                 double* tracked_out, uint8_t* status_out, double* fb_out, void* stream);
/* The caller's mask of rssync_track_frames_masked_device: row y of image j's mask at
 * mask + j * image_stride + y * pitch bytes. */
typedef struct rssync_track_mask {
    const uint8_t* mask;  /* device memory of the problem's device; nonzero = a point may lie here */
    size_t pitch;         /* bytes per mask row, >= width */
    size_t image_stride;  /* bytes from image j's mask to image j + 1's; 0 = one mask for all n_frames + 1 images */
    int margin;           /* px, 0..63 */
} rssync_track_mask;
/* rssync_track_frames_ex_device (sample_bytes 1, shift 0) or rssync_track_frames16_device (sample_bytes 2,
 * shift 0..8) that keeps points out of the regions the caller's mask excludes: burned-in overlays, parts of
 * the rig in view, independently moving objects.  images, pitch (bytes) and every other argument as there.
 *  - Eligibility: pixel (x, y) of image j is eligible iff every mask pixel (x', y') of image j with
 *    |x' - x| <= margin and |y' - y| <= margin that lies inside the image is nonzero; pixels outside the
 *    image count as usable (cv2.erode of (mask != 0) by a (2 margin + 1)^2 square, default border).  A
 *    position (x, y) in double is looked up at its nearest pixel (floor(x + 0.5), floor(y + 0.5)).  The
 *    margin keeps the level-0 structure-tensor block and LK window of a point off the excluded region (the
 *    side-a patch is window / 2 + 1 px); it is not scaled per pyramid level.
 *  - Selection: a candidate must also be eligible on image i; the rest of the selection contract applies to
 *    eligible candidates only (a cell's pick, the maximum M behind the quality threshold, the max_points
 *    cut), and a cell without an eligible candidate has no pick.
 *  - Status 3 (masked): a point gets status 3 exactly where the unmasked forward tracker gives status 1 and
 *    its query point is not eligible on image i or its tracked position is not eligible on image i + 1.
 *    tracked_out holds the forward position; a status-3 point takes no part in the backward pass, its fb_out
 *    is NaN, and it is not ingested.
 * Identities: mask == NULL gives byte for byte what rssync_track_frames_ex_device (sample_bytes 1) or
 * rssync_track_frames16_device (sample_bytes 2) gives: every output, frame table, arena, row fractions and
 * re-timing table; so does a mask that is nonzero everywhere, for any margin.  On the caller's points,
 * tracked_out equals the unmasked call's and the statuses differ only as 1 -> 3.  The kept points (status 1)
 * give exactly what rssync_set_track_pixels_device gives on them, as stated at rssync_track_frames_device.
 * A shared mask is eroded once per call; per-image masks are eroded with the pyramids, and their planes
 * (width * height bytes per image) count against the 256 MiB of chunk scratch; the chunks change no result.
 * Multi-device problems: the mask lies on the primary, which ingests, as for the other tracking forms.
 * Checked before anything is applied, besides the checks of rssync_track_frames_ex_device /
 * rssync_track_frames16_device: RSSYNC_E_INVALID for sample_bytes other than 1 or 2, a nonzero shift with
 * sample_bytes 1, a mask buffer that is not device memory of the problem's device, mask pitch < width, margin
 * outside 0..63, and a nonzero image_stride below height * pitch. */
int rssync_track_frames_masked_device(rssync_problem* p, size_t n_frames, const int64_t* frames,
                                      const size_t* counts, const double* image_ts, const double* points,
                                      const void* images, size_t pitch /* bytes */, int width, int height,
                                      int sample_bytes /* 1 or 2 */, int shift, const rssync_track_mask* mask,
                                      const rssync_lens* lens, const rssync_track_params* params,
                                      const rssync_track_options* options, double* points_out, size_t* counts_out,
                                      double* tracked_out, uint8_t* status_out, double* fb_out, void* stream);
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
/* rssync_rotation_search over n_windows frame windows [frame_begin[w], frame_end[w]) at once, each with
 * its own delay argmin.  Entry [j][w] (j W + w, W = n_windows) of out_cost / out_delay (n_rot x W) equals,
 * bit for bit, rssync_integrate_gyro_matrix(matrices + 9 j) -> rssync_set_gyro_var -> rssync_presync(
 * initial_delay, frame_begin[w], frame_end[w], search_step, search_radius) keyed by call_nos[j W + w]
 * (NULL: consecutive values of the counter in that order, which advances by n_rot W).  out_curves
 * (n_rot x W x D, or NULL): row [j][w] is that call's cost over rssync_presync_delays(...); the delay grid
 * is shared by all windows, so a clip whose delay drifts needs a radius that covers the drift.  Windows
 * may overlap or be empty (cost 0 at every delay, as rssync_presync on no frames).  Score a candidate by
 * the sum of its row, out_cost[j W + 0 .. W): each window sees about one delay, and the sum averages the
 * windows' tracking noise.  Per variant, one integration and one loss grid over all windows run.  For the
 * 48 gyro_orientation strings, pass the matrices of the strings (rssync_integrate_gyro_matrix's "matrix
 * of s", Python's orientation_matrix(s)): they integrate to the strings' bits exactly.  Errors: negative
 * counts, n_rot W above INT32_MAX, or a null window buffer (with n_rot, W > 0): RSSYNC_E_INVALID before
 * anything is done; n_rot == 0 or W == 0: nothing done; then rssync_rotation_search's errors, checked over
 * the windows in order.  A non-finite value found on the device fails the first such variant in order,
 * with the message of its grid's flags over all its windows (the first failing window's message when its
 * windows fail alike, as a non-finite gyro or ray makes them).  The problem is left holding the last
 * variant's gyro, the grid statistics are those of the last variant's grid, and a multi-device problem
 * shards by variant as rssync_rotation_search does. */
int rssync_rotation_search_windows(rssync_problem* p, const double* timestamps_s, const double* gyro_xyz,
                                   size_t count, const double* matrices, int n_rot, int n_windows,
                                   const int64_t* frame_begin, const int64_t* frame_end, double initial_delay,
                                   double search_step, double search_radius, const uint64_t* call_nos,
                                   double* out_cost, double* out_delay, double* out_curves);

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
/* rssync_readout_search over n_windows frame windows [frame_begin[w], frame_end[w]) at once, each with its
 * own delay argmin.  Entry [j][w] (j W + w, W = n_windows) of out_cost / out_delay (n_readouts x W) equals,
 * bit for bit, rssync_presync(initial_delay, frame_begin[w], frame_end[w], search_step, search_radius) on
 * a problem that ingested the same input with readout = readouts[j], keyed by call_nos[j W + w] (NULL:
 * consecutive values of the counter in that order, which advances by n_readouts W).  out_curves
 * (n_readouts x W x D, or NULL) as in rssync_rotation_search_windows; the delay grid is shared by all
 * windows.  Windows may overlap or be empty.  Score a readout by the sum of its row.  Per readout, the
 * union of the windows' frames is re-timed once and one loss grid over all windows runs.  Errors:
 * negative counts, n_readouts W above INT32_MAX, a null buffer or a non-finite readout: RSSYNC_E_INVALID;
 * a frame without row fractions: RSSYNC_E_STATE naming the first such frame in window order; both before
 * anything is done.  n_readouts == 0 or W == 0: nothing done.  A non-finite value found on the device
 * fails the first such readout in order, with the message of its grid's flags over all its windows (as
 * in rssync_rotation_search_windows).  The arena, frame table and gyro are left as they are, the grid
 * statistics are those of the last readout's grid, and a multi-device problem shards by readout as
 * rssync_readout_search does. */
int rssync_readout_search_windows(rssync_problem* p, const double* readouts, int n_readouts, int n_windows,
                                  const int64_t* frame_begin, const int64_t* frame_end, double initial_delay,
                                  double search_step, double search_radius, const uint64_t* call_nos,
                                  double* out_cost, double* out_delay, double* out_curves);
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
