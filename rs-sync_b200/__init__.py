"""rs-sync_b200 — B200-native synchronisation loss engine behind rs-sync's ISyncProblem API.

Python host-side mirror of the reference interface (src/core/public/rssync.h:9-31 of
VladimirP1/rs-sync) over the C ABI in include/rssync_b200.h.  The numerical work runs in
hand-written sm_100a kernels inside lib/librssync_b200.so; this module only marshals buffers.
There is no CPU fallback: if the library is missing or no B200 is present the calls raise.

The directory name contains a hyphen, so import it with
    importlib.import_module("rs-sync_b200")
"""
from __future__ import annotations

import collections
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# RSSYNC_B200_LIB selects an alternative build of the same library (kernel tuning experiments)
LIB_PATH = os.environ.get("RSSYNC_B200_LIB") or os.path.join(_HERE, "lib", "librssync_b200.so")

c_double_p = C.POINTER(C.c_double)
c_i64_p = C.POINTER(C.c_int64)

OK, E_INVALID, E_NONFINITE, E_ORDER, E_STATE, E_CUDA = range(6)
STREAM_PRESYNC, STREAM_DEBUG, STREAM_SYNCINIT = 1, 2, 3

# every symbol include/rssync_b200.h declares (checked by tests/test_abi.py)
C_ABI_SYMBOLS = [
    "rssync_create", "rssync_destroy", "rssync_last_error", "rssync_set_gyro_fixed",
    "rssync_set_gyro_var", "rssync_set_track", "rssync_presync", "rssync_sync",
    "rssync_debug_presync", "rssync_presync_grid", "rssync_presync_delays", "rssync_sync_batch",
    "rssync_last_sync_trace", "rssync_set_rng", "rssync_call_counter", "rssync_set_stream",
    "rssync_flush", "rssync_get_stats", "rssync_measure_fp64_peak", "rssync_probe_gyro", "rssync_probe_spline_system",
    "rssync_probe_problem_matrix", "rssync_probe_guess_motion", "rssync_probe_loss",
    "rssync_probe_lbfgs", "rssync_probe_log1p", "rssync_set_track_batch", "rssync_set_kernel_timing",
    "rssync_sync_batch_ex", "rssync_probe_guess_motion_ex", "rssync_integrate_gyro",
    "rssync_orientation_search", "rssync_orientation_search_ex", "rssync_presync_windows", "rssync_set_track_pixels",
    "rssync_create_multi", "rssync_device_count", "rssync_frame_table", "rssync_device_state", "rssync_adopt_state",
    "rssync_device_state_pipelined", "rssync_stream_wait_chunk", "rssync_expect_chunk", "rssync_note_reader",
    "rssync_probe_stage_copy", "rssync_probe_replication_plan",
    "rssync_set_loss_mode", "rssync_probe_spec_trig",
    "rssync_set_track_batch_device", "rssync_set_track_pixels_device",
    "rssync_readout_search", "rssync_set_readout", "rssync_integrate_gyro_matrix", "rssync_rotation_search",
    "rssync_set_track_row_fractions", "rssync_set_track_row_fractions_device",
    "rssync_retime_table", "rssync_row_fraction_plane", "rssync_adopt_row_fractions",
    "rssync_readout_search_windows", "rssync_rotation_search_windows", "rssync_track_frames_device",
    "rssync_track_frames_ex_device", "rssync_track_frames16_device", "rssync_track_frames_masked_device",
]
# Itanium-ABI symbols of the C++ drop-in face (same set the reference's librssync_core exports)
CXX_ABI_SYMBOLS = [
    "_Z17CreateSyncProblemv", "_ZN12ISyncProblemD0Ev", "_ZN12ISyncProblemD1Ev",
    "_ZN12ISyncProblemD2Ev", "_ZTV12ISyncProblem", "_ZTI12ISyncProblem", "_ZTS12ISyncProblem",
]


class Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "kernel_launches", "h2d_bytes", "d2h_bytes", "frames", "rays", "gyro_samples",
        "sync_outer_iters", "sync_lbfgs_evals")] + [("last_grid_kernel_ms", C.c_double),
                                                     ("last_grid_tasks", C.c_uint64),
                                                     ("last_grid_exact_tasks", C.c_uint64)] + [
        (n, C.c_uint64) for n in ("sync_row_builds", "sync_loss_evals", "sync_init_tasks", "sync_outer_total",
                                  "nccl_calls", "broadcast_bytes")]


class FrameDesc(C.Structure):
    """rssync_frame_desc: one tracked frame inside the device arena"""
    _fields_ = [("id", C.c_int64), ("off", C.c_int32), ("n", C.c_int32), ("ts_lo", C.c_double), ("ts_hi", C.c_double)]


class DeviceState(C.Structure):
    """rssync_device_state_t: device pointers and sizes of a problem's finished inputs"""
    _fields_ = [("rays", C.c_void_p), ("orig", C.c_void_p), ("pos", C.c_void_p), ("spline_records", C.c_void_p),
                ("arena_rays", C.c_size_t), ("gyro_samples", C.c_size_t), ("sample_rate", C.c_double),
                ("first_timestamp", C.c_double)]


class RetimeDesc(C.Structure):
    """rssync_retime_desc: a frame that holds row fractions, and its two frame timestamps"""
    _fields_ = [("id", C.c_int64), ("frame_ts_a", C.c_double), ("frame_ts_b", C.c_double)]


RETIME_DTYPE = np.dtype([("id", "<i8"), ("frame_ts_a", "<f8"), ("frame_ts_b", "<f8")])


class Lens(C.Structure):
    """rssync_lens: readout_s fx fy cx cy k1 k2 k3 k4 (one line of the reference's lens file)"""
    _fields_ = [(n, C.c_double) for n in ("readout", "fx", "fy", "cx", "cy", "k1", "k2", "k3", "k4")]


class TrackParams(C.Structure):
    """rssync_track_params: the pyramidal Lucas-Kanade tracker's settings (track_frames)"""
    _fields_ = [("levels", C.c_int), ("window", C.c_int), ("max_iters", C.c_int), ("epsilon", C.c_double),
                ("min_eig", C.c_double)]

    def __init__(self, levels=3, window=21, max_iters=30, epsilon=0.01, min_eig=1e-4):
        super().__init__(levels, window, max_iters, epsilon, min_eig)


class TrackOptions(C.Structure):
    """rssync_track_options: point selection and the forward-backward check (track_frames_ex)"""
    _fields_ = [("cell", C.c_int), ("block", C.c_int), ("quality", C.c_double), ("max_points", C.c_int),
                ("fb_max", C.c_double)]

    def __init__(self, cell=128, block=5, quality=0.01, max_points=512, fb_max=1.0):
        super().__init__(cell, block, quality, max_points, fb_max)


class TrackMask(C.Structure):
    """rssync_track_mask: the caller's mask of track_frames_ex (mask=)"""
    _fields_ = [("mask", C.c_void_p), ("pitch", C.c_size_t), ("image_stride", C.c_size_t), ("margin", C.c_int)]


TrackResult = collections.namedtuple("TrackResult", "points counts tracked status fb_error")
TrackResult.__doc__ = """The result of SyncProblem.track_frames_ex: query points, counts per frame, tracked positions,
statuses and forward-backward distances.  Status: 0 lost, 1 kept and ingested, 2 rejected by the backward check,
3 masked (kept by the forward tracker, but its query point or tracked position lies off the eligible region of the
mask: not ingested, no backward pass, fb_error NaN)."""


def grid_points(width, height, step):
    """The query grid of the reference's front end: every `step` pixels in x and y, as an (n, 2) float64 array,
    x fastest.  Origin (this engine's choice; the reference's exact offsets are not known here): the grid is
    centred, its first point at ((width - 1 - step * (nx - 1)) / 2, likewise in y) with nx = (width - 1) // step
    + 1 points per row, so the margins to both edges are equal."""
    if step <= 0 or width < 1 or height < 1:
        raise ValueError("grid_points: width, height and step must be positive")
    nx, ny = (int(width) - 1) // int(step) + 1, (int(height) - 1) // int(step) + 1
    x0, y0 = (width - 1 - step * (nx - 1)) / 2.0, (height - 1 - step * (ny - 1)) / 2.0
    gy, gx = np.meshgrid(y0 + step * np.arange(ny, dtype=np.float64), x0 + step * np.arange(nx, dtype=np.float64),
                         indexing="ij")
    return np.ascontiguousarray(np.stack([gx.ravel(), gy.ravel()], axis=-1))


class RsSyncError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"rssync status {code}: {message}")
        self.code = code
        self.message = message


_lib = None


def load_library():
    """dlopen the engine.  Fails loudly if it was not built (run `make lib` / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: build it with `make lib`; there is no fallback path")
    L = C.CDLL(LIB_PATH)
    P = C.c_void_p
    L.rssync_create.argtypes = [C.POINTER(P)]
    L.rssync_create_multi.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(P)]
    L.rssync_device_count.argtypes = [P]
    L.rssync_frame_table.argtypes = [P, C.POINTER(FrameDesc), C.c_size_t]
    L.rssync_device_state.argtypes = [P, C.POINTER(DeviceState)]
    L.rssync_adopt_state.argtypes = [P, C.POINTER(FrameDesc), C.c_size_t, C.c_size_t, C.c_size_t, C.c_double, C.c_double]
    L.rssync_retime_table.argtypes = [P, C.POINTER(RetimeDesc), C.c_size_t]
    L.rssync_row_fraction_plane.argtypes = [P, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
    L.rssync_adopt_row_fractions.argtypes = [P, C.POINTER(RetimeDesc), C.c_size_t]
    L.rssync_device_state_pipelined.argtypes = [P, C.POINTER(DeviceState), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t),
                                                C.c_size_t, C.POINTER(C.c_size_t)]
    L.rssync_stream_wait_chunk.argtypes = [P, C.c_int, C.c_void_p]
    L.rssync_expect_chunk.argtypes = [P, C.c_size_t, C.c_size_t, C.c_void_p]
    L.rssync_note_reader.argtypes = [P, C.c_void_p]
    L.rssync_probe_replication_plan.argtypes = [C.POINTER(C.c_size_t), C.POINTER(C.c_size_t), C.c_size_t, C.c_size_t,
                                                C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_size_t),
                                                C.POINTER(C.c_size_t), C.c_size_t]
    L.rssync_probe_stage_copy.argtypes = [C.POINTER(C.c_double), C.c_size_t, C.c_int, C.POINTER(C.c_double),
                                          C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int)]
    L.rssync_destroy.argtypes = [P]
    L.rssync_destroy.restype = None
    L.rssync_last_error.argtypes = [P]
    L.rssync_last_error.restype = C.c_char_p
    L.rssync_set_gyro_fixed.argtypes = [P, c_double_p, C.c_size_t, C.c_double, C.c_double]
    L.rssync_set_gyro_var.argtypes = [P, c_i64_p, c_double_p, C.c_size_t]
    L.rssync_set_track.argtypes = [P, C.c_int64, c_double_p, c_double_p, c_double_p, c_double_p, C.c_size_t]
    L.rssync_set_track_batch.argtypes = [P, C.c_size_t, c_i64_p, C.POINTER(C.c_size_t), c_double_p, c_double_p,
                                         c_double_p, c_double_p]
    L.rssync_set_kernel_timing.argtypes = [P, C.c_int]
    L.rssync_set_track_pixels.argtypes = [P, C.c_size_t, c_i64_p, C.POINTER(C.c_size_t), c_double_p, c_double_p,
                                          c_double_p, c_double_p, C.POINTER(Lens), C.c_double]
    # the per-ray buffers of the *_device forms are device addresses, passed as c_void_p
    L.rssync_set_track_batch_device.argtypes = [P, C.c_size_t, c_i64_p, C.POINTER(C.c_size_t), P, P, P, P, P]
    L.rssync_set_track_pixels_device.argtypes = [P, C.c_size_t, c_i64_p, C.POINTER(C.c_size_t), c_double_p,
                                                 c_double_p, P, P, C.POINTER(Lens), C.c_double, P]
    L.rssync_set_track_row_fractions.argtypes = [P, C.c_size_t, c_i64_p, C.POINTER(C.c_size_t), c_double_p,
                                                 c_double_p, c_double_p, c_double_p, c_double_p, c_double_p,
                                                 C.c_double]
    L.rssync_set_track_row_fractions_device.argtypes = [P, C.c_size_t, c_i64_p, C.POINTER(C.c_size_t), c_double_p,
                                                        c_double_p, P, P, P, P, C.c_double, P]
    L.rssync_track_frames_device.argtypes = [P, C.c_size_t, c_i64_p, C.POINTER(C.c_size_t), c_double_p, P, P,
                                             C.c_size_t, C.c_int, C.c_int, C.POINTER(Lens), C.POINTER(TrackParams),
                                             P, P, P]
    L.rssync_track_frames_ex_device.argtypes = [P, C.c_size_t, c_i64_p, C.POINTER(C.c_size_t), c_double_p, P, P,
                                                C.c_size_t, C.c_int, C.c_int, C.POINTER(Lens),
                                                C.POINTER(TrackParams), C.POINTER(TrackOptions), P,
                                                C.POINTER(C.c_size_t), P, P, P, P]
    L.rssync_track_frames16_device.argtypes = [P, C.c_size_t, c_i64_p, C.POINTER(C.c_size_t), c_double_p, P, P,
                                               C.c_size_t, C.c_int, C.c_int, C.c_int, C.POINTER(Lens),
                                               C.POINTER(TrackParams), C.POINTER(TrackOptions), P,
                                               C.POINTER(C.c_size_t), P, P, P, P]
    L.rssync_track_frames_masked_device.argtypes = [P, C.c_size_t, c_i64_p, C.POINTER(C.c_size_t), c_double_p, P,
                                                    P, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int,
                                                    C.POINTER(TrackMask), C.POINTER(Lens), C.POINTER(TrackParams),
                                                    C.POINTER(TrackOptions), P, C.POINTER(C.c_size_t), P, P, P, P]
    L.rssync_presync.argtypes = [P, C.c_double, C.c_int64, C.c_int64, C.c_double, C.c_double, c_double_p, c_double_p]
    L.rssync_sync.argtypes = [P, C.c_double, C.c_int64, C.c_int64, C.c_double, C.c_double, c_double_p, c_double_p]
    L.rssync_debug_presync.argtypes = [P, C.c_double, C.c_int64, C.c_int64, C.c_double, c_double_p, c_double_p, C.c_int]
    L.rssync_presync_grid.argtypes = [P, C.c_int64, C.c_int64, c_double_p, C.c_int, C.c_int, C.c_uint64,
                                      C.c_uint64, c_double_p, C.POINTER(C.c_uint)]
    L.rssync_presync_delays.argtypes = [C.c_double, C.c_double, C.c_double, c_double_p, C.c_int]
    L.rssync_presync_windows.argtypes = [P, C.c_int, C.c_double, c_i64_p, c_i64_p, C.c_double, C.c_double,
                                         C.POINTER(C.c_uint64), c_double_p, c_double_p]
    L.rssync_sync_batch.argtypes = [P, C.c_int, c_double_p, c_i64_p, c_i64_p, c_double_p, c_double_p,
                                    c_double_p, c_double_p]
    L.rssync_sync_batch_ex.argtypes = [P, C.c_int, c_double_p, c_i64_p, c_i64_p, c_double_p, c_double_p,
                                       C.POINTER(C.c_uint64), c_double_p, c_double_p]
    L.rssync_last_sync_trace.argtypes = [P, c_double_p, c_double_p, C.c_int]
    L.rssync_set_rng.argtypes = [P, C.c_uint64, C.c_uint64]
    L.rssync_set_loss_mode.argtypes = [P, C.c_int]
    L.rssync_call_counter.argtypes = [P]
    L.rssync_call_counter.restype = C.c_uint64
    L.rssync_set_stream.argtypes = [P, C.c_void_p]
    L.rssync_flush.argtypes = [P]
    L.rssync_get_stats.argtypes = [P, C.POINTER(Stats)]
    L.rssync_measure_fp64_peak.argtypes = [c_double_p]
    L.rssync_probe_gyro.argtypes = [P, c_double_p, c_double_p, C.POINTER(C.c_size_t), c_double_p]
    L.rssync_probe_spline_system.argtypes = [c_double_p, C.c_size_t, c_double_p, c_double_p]
    L.rssync_probe_problem_matrix.argtypes = [P, C.c_int64, C.c_double, c_double_p]
    L.rssync_probe_guess_motion.argtypes = [P, C.c_int64, C.c_double, C.c_int, C.c_int, C.c_uint64,
                                            C.c_uint64, c_double_p, c_double_p]
    L.rssync_probe_guess_motion_ex.argtypes = [P, C.c_int64, C.c_double, C.c_int, C.c_int, C.c_uint64,
                                               C.c_uint64, C.c_int, c_double_p, c_double_p,
                                               C.POINTER(C.c_int)]
    L.rssync_probe_loss.argtypes = [P, C.c_int64, C.c_double, c_double_p, C.c_double, c_double_p,
                                    c_double_p, c_double_p]
    L.rssync_probe_lbfgs.argtypes = [P, C.c_int64, C.c_double, c_double_p, C.c_double, c_double_p,
                                     C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.rssync_probe_log1p.argtypes = [c_double_p, C.c_int, c_double_p]
    L.rssync_probe_spec_trig.argtypes = [c_double_p, C.c_int, C.c_int, C.c_int, c_double_p]
    L.rssync_integrate_gyro.argtypes = [c_double_p, c_double_p, C.c_size_t, C.c_char_p, c_double_p]
    L.rssync_orientation_search.argtypes = [P, c_double_p, c_double_p, C.c_size_t, C.POINTER(C.c_char_p),
                                            C.c_int, C.c_double, C.c_int64, C.c_int64, C.c_double,
                                            C.c_double, c_double_p, c_double_p]
    L.rssync_orientation_search_ex.argtypes = [P, c_double_p, c_double_p, C.c_size_t, C.POINTER(C.c_char_p),
                                               C.c_int, C.c_double, C.c_int64, C.c_int64, C.c_double,
                                               C.c_double, C.POINTER(C.c_uint64), c_double_p, c_double_p]
    L.rssync_readout_search.argtypes = [P, c_double_p, C.c_int, C.c_double, C.c_int64, C.c_int64, C.c_double,
                                        C.c_double, C.POINTER(C.c_uint64), c_double_p, c_double_p, c_double_p]
    L.rssync_set_readout.argtypes = [P, C.c_double, C.c_int64, C.c_int64]
    L.rssync_integrate_gyro_matrix.argtypes = [c_double_p, c_double_p, C.c_size_t, c_double_p, c_double_p]
    L.rssync_rotation_search.argtypes = [P, c_double_p, c_double_p, C.c_size_t, c_double_p, C.c_int, C.c_double,
                                         C.c_int64, C.c_int64, C.c_double, C.c_double, C.POINTER(C.c_uint64),
                                         c_double_p, c_double_p, c_double_p]
    L.rssync_readout_search_windows.argtypes = [P, c_double_p, C.c_int, C.c_int, c_i64_p, c_i64_p, C.c_double,
                                                C.c_double, C.c_double, C.POINTER(C.c_uint64), c_double_p,
                                                c_double_p, c_double_p]
    L.rssync_rotation_search_windows.argtypes = [P, c_double_p, c_double_p, C.c_size_t, c_double_p, C.c_int, C.c_int,
                                                 c_i64_p, c_i64_p, C.c_double, C.c_double, C.c_double,
                                                 C.POINTER(C.c_uint64), c_double_p, c_double_p, c_double_p]
    _lib = L
    return L


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _dp(a):
    return a.ctypes.data_as(c_double_p)


def _cuda_tensors(*xs):
    """True when every argument is a torch CUDA tensor, False when none is; a mix raises TypeError.
    Recognises tensors without importing torch, so the package imports without it."""
    on_dev = [getattr(x, "is_cuda", False) is True for x in xs]
    if any(on_dev) and not all(on_dev):
        raise TypeError("per-ray buffers: either all host arrays or all CUDA tensors, not a mix")
    return all(on_dev)


def _device_ptrs(tensors, sizes):
    """device addresses of contiguous float64 CUDA tensors of the given element counts, all on one
    device, and that device's current stream (the one the caller produced them on)"""
    import torch
    dev = tensors[0].device
    for t, n in zip(tensors, sizes):
        if t.dtype != torch.float64:
            raise TypeError(f"per-ray CUDA tensors must be float64, got {t.dtype}")
        if not t.is_contiguous():
            raise ValueError("per-ray CUDA tensors must be contiguous")
        if t.device != dev:
            raise ValueError(f"per-ray CUDA tensors on several devices: {dev} and {t.device}")
        if t.numel() != n:
            raise ValueError(f"per-ray CUDA tensor holds {t.numel()} values, the counts give {n}")
    return [C.c_void_p(t.data_ptr() or None) for t in tensors], C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def presync_delays(initial_delay, search_step, search_radius):
    """pre_sync's delay grid (core_private.cpp:69-70), floating-point accumulation included."""
    L = load_library()
    n = L.rssync_presync_delays(initial_delay, search_step, search_radius, None, 0)
    out = np.empty(n)
    L.rssync_presync_delays(initial_delay, search_step, search_radius, _dp(out), n)
    return out


def integrate_gyro(timestamps_s, gyro_xyz, orientation=None, rotation=None):
    """optdata_fill_gyro (core_testcode.cpp:37-53): raw gyro (count x 3 rad/s) -> quaternions (count x 4).
    The gyro axis mapping is a gyro_orientation string (`orientation`) or a 3x3 matrix (`rotation`,
    w = rotation @ g per sample, rssync_integrate_gyro_matrix), not both; neither: as is.  To combine
    them, pass rotation=R @ orientation_matrix(s): the product is exact, the second factor being a
    signed permutation."""
    if orientation is not None and rotation is not None:
        raise ValueError("integrate_gyro: give orientation or rotation, not both")
    ts = _f64(timestamps_s)
    g = _f64(gyro_xyz)
    out = np.empty((ts.shape[0], 4))
    if rotation is not None:
        m = _f64(rotation)
        if m.shape != (3, 3):
            raise ValueError(f"integrate_gyro: rotation must be a 3x3 matrix, got shape {m.shape}")
        rc = load_library().rssync_integrate_gyro_matrix(_dp(ts), _dp(g), ts.shape[0], _dp(m), _dp(out))
        if rc:
            raise RsSyncError(rc, "rotation matrix with a non-finite entry")
        return out
    rc = load_library().rssync_integrate_gyro(_dp(ts), _dp(g), ts.shape[0],
                                              orientation.encode() if orientation else None, _dp(out))
    if rc:
        raise RsSyncError(rc, f"malformed gyro_orientation {orientation!r}")
    return out


def orientation_matrix(orientation):
    """The signed permutation matrix of a gyro_orientation string (None: "XYZ", the identity): row i has
    +1 (upper case) or -1 (lower case) in the column of the input axis that character i names, so that
    integrate_gyro(rotation=orientation_matrix(s)) == integrate_gyro(orientation=s) bit for bit."""
    m = np.zeros((3, 3))
    s = "XYZ" if orientation is None else orientation
    if not isinstance(s, str) or len(s) != 3 or any(ch not in "xyzXYZ" for ch in s):
        raise ValueError(f"malformed gyro_orientation {orientation!r}")
    for i, ch in enumerate(s):
        m[i, "xyz".index(ch.lower())] = 1.0 if ch.isupper() else -1.0
    return m


def rotations_about(axis, angles):
    """(n, 3, 3) right-handed rotation matrices about axis 'x', 'y' or 'z' by each of `angles` (radians)"""
    if axis not in ("x", "y", "z"):
        raise ValueError(f"axis must be 'x', 'y' or 'z', got {axis!r}")
    a = np.asarray(angles, dtype=np.float64).ravel()
    c, s = np.cos(a), np.sin(a)
    i, j = {"x": (1, 2), "y": (2, 0), "z": (0, 1)}[axis]  # the plane the rotation turns, in right-handed order
    out = np.zeros((a.size, 3, 3))
    out[:, 3 - i - j, 3 - i - j] = 1.0
    out[:, i, i] = c
    out[:, j, j] = c
    out[:, i, j] = -s
    out[:, j, i] = s
    return out


def _parabola_vertex(x, costs, what):
    """the vertex of the least-squares parabola through (x[i], costs[i]); `what` names x in the messages"""
    r = np.asarray(x, dtype=np.float64).ravel()
    c = np.asarray(costs, dtype=np.float64).ravel()
    if r.shape != c.shape:
        raise ValueError(f"{r.size} {what} but {c.size} costs")
    if not (np.all(np.isfinite(r)) and np.all(np.isfinite(c))):
        raise ValueError(f"{what} and costs must be finite")
    if np.unique(r).size < 3:
        raise ValueError(f"a parabola needs at least 3 distinct {what}")
    # fit in centred, scaled coordinates: candidates may be milliseconds in seconds, costs are large
    mid, half = 0.5 * (r.max() + r.min()), 0.5 * (r.max() - r.min())
    u = (r - mid) / half
    a, b, _ = np.polyfit(u, c, 2)
    # (a vertex inside the candidates has |b| <= 2 a: the margin only turns rounding noise on a straight
    # line into "not convex")
    if not a > 1e-9 * max(abs(b), float(np.ptp(c))):
        raise ValueError("the least-squares parabola is not convex: no minimum inside the candidates")
    v = mid + half * (-b / (2.0 * a))
    if not (r.min() <= v <= r.max()):
        raise ValueError(f"the parabola's vertex {v!r} lies outside the candidate {what} "
                         f"[{r.min()!r}, {r.max()!r}]")
    return float(v)


def estimate_readout(readouts, costs):
    """The rolling-shutter readout at the vertex of the least-squares parabola through the points
    (readouts[i], costs[i]) -- e.g. a coarse grid of candidates and readout_search's PreSync minima.
    Raises ValueError when there are fewer than 3 distinct candidates, the fit is not convex, or the
    vertex lies outside [min(readouts), max(readouts)]."""
    return _parabola_vertex(readouts, costs, "readouts")


def estimate_angle(angles, costs):
    """The mount angle at the vertex of the least-squares parabola through the points (angles[i],
    costs[i]) -- e.g. candidate rotations about one axis and rotation_search's PreSync minima.  Raises
    ValueError as estimate_readout does."""
    return _parabola_vertex(angles, costs, "angles")


def measure_fp64_peak():
    L = load_library()
    v = C.c_double()
    rc = L.rssync_measure_fp64_peak(C.byref(v))
    if rc != OK:
        raise RsSyncError(rc, "FP64 peak measurement failed (no CUDA device?)")
    return v.value


def probe_spline_system(quats):
    """Host-only: the eliminated spline system (rhs n x 4, diag n) SetGyroQuaternions builds on the host."""
    L = load_library()
    q = _f64(quats).reshape(-1, 4)
    rhs, diag = np.empty_like(q), np.empty(q.shape[0])
    rc = L.rssync_probe_spline_system(_dp(q), q.shape[0], _dp(rhs), _dp(diag))
    if rc != OK:
        raise RsSyncError(rc, "spline system probe failed")
    return rhs, diag


def probe_spec_trig(x, which, on_device=False):
    """the contract's sin / cos / acos (which = "sin" | "cos" | "acos"), host code or a device kernel"""
    L = load_library()
    x = _f64(x)
    out = np.empty_like(x)
    rc = L.rssync_probe_spec_trig(_dp(x), x.size, {"sin": 0, "cos": 1, "acos": 2}[which], 1 if on_device else 0, _dp(out))
    if rc != OK:
        raise RsSyncError(rc, "spec trig probe failed")
    return out


def probe_replication_plan(chunks, arena_rays, groups):
    """host-only: the library's replication pieces [(k_last, lo, hi), ...] for `chunks` in flight"""
    L = load_library()
    n = len(chunks)
    lo = (C.c_size_t * max(n, 1))(*[c[0] for c in chunks])
    hi = (C.c_size_t * max(n, 1))(*[c[1] for c in chunks])
    cap = 64
    k, plo, phi = (C.c_int * cap)(), (C.c_size_t * cap)(), (C.c_size_t * cap)()
    m = L.rssync_probe_replication_plan(lo, hi, n, int(arena_rays), int(groups), k, plo, phi, cap)
    if m < 0 or m > cap:
        raise RsSyncError(E_INVALID, "replication plan probe failed")
    return [(int(k[i]), int(plo[i]), int(phi[i])) for i in range(m)]


def probe_stage_copy(x, mode, bounds=None, misalign=0):
    """host-only: the bulk ingest's checked staging copy of `x` in form `mode` (0 scalar, 1 AVX2, 2 AVX2
    with non-temporal stores); returns (copy, all_finite, lo, hi) -- [lo, hi] starts at `bounds` and is
    widened to the values (None: not tracked).  `misalign`: destination offset in doubles from a
    64-byte boundary."""
    L = load_library()
    x = _f64(x)
    buf = np.zeros(x.size + 16, dtype=np.float64)
    start = (-(buf.ctypes.data // 8) % 8 + misalign) % 8 if misalign else (-(buf.ctypes.data // 8)) % 8
    dst = buf[start:start + x.size]
    ok = C.c_int(0)
    if bounds is None:
        rc = L.rssync_probe_stage_copy(_dp(x), x.size, mode, _dp(dst), None, None, C.byref(ok))
        lo = hi = None
    else:
        lo_c, hi_c = C.c_double(bounds[0]), C.c_double(bounds[1])
        rc = L.rssync_probe_stage_copy(_dp(x), x.size, mode, _dp(dst), C.byref(lo_c), C.byref(hi_c), C.byref(ok))
        lo, hi = lo_c.value, hi_c.value
    if rc != OK:
        raise RsSyncError(rc, "stage copy probe failed (form not supported on this CPU?)")
    return dst.copy(), bool(ok.value), lo, hi


def probe_log1p(x):
    L = load_library()
    x = _f64(x)
    out = np.empty_like(x)
    rc = L.rssync_probe_log1p(_dp(x), x.size, _dp(out))
    if rc != OK:
        raise RsSyncError(rc, "log1p probe failed")
    return out


class SyncProblem:
    """ISyncProblem (rssync.h:9-29): same method names, argument order and return values
    ({cost, delay} pairs).  Errors that make the reference write panic.txt and exit raise
    RsSyncError carrying the same message."""

    def __init__(self, seed=100, devices=None):
        """devices: None = the calling thread's current CUDA device (CreateSyncProblem); a list of
        device ordinals = one problem spread over those GPUs (rssync_create_multi)."""
        self.L = load_library()
        self.h = C.c_void_p()
        if devices is None:
            rc = self.L.rssync_create(C.byref(self.h))
        else:
            arr = (C.c_int * len(devices))(*[int(d) for d in devices])
            rc = self.L.rssync_create_multi(arr, len(devices), C.byref(self.h))
        if rc != OK:
            msg = self.L.rssync_last_error(self.h).decode() if self.h else "no usable CUDA device (no CPU fallback)"
            raise RsSyncError(rc, msg)
        self.L.rssync_set_rng(self.h, seed, 0)
        self.seed = seed

    def close(self):
        if getattr(self, "h", None):
            self.L.rssync_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != OK:
            raise RsSyncError(rc, self.L.rssync_last_error(self.h).decode())

    # ---- reference interface ----------------------------------------------------------------
    def SetGyroQuaternions(self, *args):
        """(data, count, sample_rate, first_timestamp)  rssync.h:13-14, or
        (timestamps_us, quats, count)                 rssync.h:15-16."""
        if len(args) == 4:
            data, count, rate, first = args
            data = _f64(data)
            self._check(self.L.rssync_set_gyro_fixed(self.h, _dp(data), count, rate, first))
        elif len(args) == 3:
            ts, quats, count = args
            ts = np.ascontiguousarray(ts, dtype=np.int64)
            quats = _f64(quats)
            self._check(self.L.rssync_set_gyro_var(self.h, ts.ctypes.data_as(c_i64_p), _dp(quats), count))
        else:
            raise TypeError("SetGyroQuaternions takes 3 or 4 arguments")

    def SetTrackResult(self, frame, ts_a, ts_b, rays_a, rays_b, count):
        a = [_f64(x) for x in (ts_a, ts_b, rays_a, rays_b)]
        self._check(self.L.rssync_set_track(self.h, int(frame), _dp(a[0]), _dp(a[1]), _dp(a[2]), _dp(a[3]), count))

    def PreSync(self, initial_delay, frame_begin, frame_end, search_step, search_radius):
        c, d = C.c_double(), C.c_double()
        self._check(self.L.rssync_presync(self.h, initial_delay, frame_begin, frame_end, search_step,
                                          search_radius, C.byref(c), C.byref(d)))
        return c.value, d.value

    def Sync(self, initial_delay, frame_begin, frame_end, search_center, search_radius):
        c, d = C.c_double(), C.c_double()
        self._check(self.L.rssync_sync(self.h, initial_delay, frame_begin, frame_end, search_center,
                                       search_radius, C.byref(c), C.byref(d)))
        return c.value, d.value

    def DebugPreSync(self, initial_delay, frame_begin, frame_end, search_radius, point_count):
        delays = np.empty(point_count)
        costs = np.empty(point_count)
        self._check(self.L.rssync_debug_presync(self.h, initial_delay, frame_begin, frame_end, search_radius,
                                                _dp(delays), _dp(costs), point_count))
        return delays, costs

    # ---- extensions -------------------------------------------------------------------------
    def set_track_batch(self, frames, counts, ts_a, ts_b, rays_a, rays_b):
        """Bulk SetTrackResult: per-frame buffers concatenated in `frames` order.  ts_a, ts_b, rays_a
        and rays_b may instead all be torch CUDA tensors (contiguous float64, on the problem's device,
        produced on that device's current stream): they are then checked and ingested where they are
        (rssync_set_track_batch_device), with the same results.  frames / counts stay host arrays."""
        frames = np.ascontiguousarray(frames, dtype=np.int64)
        counts = np.ascontiguousarray(counts, dtype=np.uint64)
        fp, cp = frames.ctypes.data_as(c_i64_p), counts.ctypes.data_as(C.POINTER(C.c_size_t))
        if _cuda_tensors(ts_a, ts_b, rays_a, rays_b):
            n = int(counts.sum())
            ptrs, stream = _device_ptrs((ts_a, ts_b, rays_a, rays_b), (n, n, 3 * n, 3 * n))
            self._check(self.L.rssync_set_track_batch_device(self.h, frames.shape[0], fp, cp, *ptrs, stream))
            return
        a = [_f64(x) for x in (ts_a, ts_b, rays_a, rays_b)]
        self._check(self.L.rssync_set_track_batch(self.h, frames.shape[0], fp, cp, _dp(a[0]), _dp(a[1]), _dp(a[2]),
                                                  _dp(a[3])))

    def set_track_pixels(self, frames, counts, frame_ts_a, frame_ts_b, points_a, points_b, lens, image_rows):
        """track_frames' per-frame tail (core_testcode.cpp:134-161) on the device: pixel pairs -> rays.
        points_a / points_b may both be torch CUDA tensors (as in set_track_batch); frames, counts,
        frame_ts_a / frame_ts_b and lens stay on the host."""
        fr = np.ascontiguousarray(frames, dtype=np.int64)
        cn = np.ascontiguousarray(counts, dtype=np.uint64)
        ta, tb = _f64(frame_ts_a), _f64(frame_ts_b)
        lens_c = lens if isinstance(lens, Lens) else Lens(*[float(x) for x in lens])
        args = (self.h, fr.shape[0], fr.ctypes.data_as(c_i64_p), cn.ctypes.data_as(C.POINTER(C.c_size_t)), _dp(ta),
                _dp(tb))
        if _cuda_tensors(points_a, points_b):
            n = int(cn.sum())
            ptrs, stream = _device_ptrs((points_a, points_b), (2 * n, 2 * n))
            self._check(self.L.rssync_set_track_pixels_device(*args, *ptrs, C.byref(lens_c), float(image_rows),
                                                              stream))
            return
        pa, pb = _f64(points_a), _f64(points_b)
        self._check(self.L.rssync_set_track_pixels(*args, _dp(pa), _dp(pb), C.byref(lens_c), float(image_rows)))

    def set_track_row_fractions(self, frames, counts, frame_ts_a, frame_ts_b, frac_a, frac_b, rays_a, rays_b,
                                readout):
        """set_track_batch for rays the caller computed with its own camera model, with the timestamps
        formed here: ts = frame_ts + readout * frac per ray (frac usually y / image_rows).  The frames keep
        their row fractions, so readout_search / set_readout accept them.  frac_a / frac_b (1 value per
        ray) and rays_a / rays_b (3 per ray) may all be torch CUDA tensors (as in set_track_batch);
        frames, counts and frame_ts_a / frame_ts_b stay on the host."""
        fr = np.ascontiguousarray(frames, dtype=np.int64)
        cn = np.ascontiguousarray(counts, dtype=np.uint64)
        ta, tb = _f64(frame_ts_a), _f64(frame_ts_b)
        args = (self.h, fr.shape[0], fr.ctypes.data_as(c_i64_p), cn.ctypes.data_as(C.POINTER(C.c_size_t)), _dp(ta),
                _dp(tb))
        if _cuda_tensors(frac_a, frac_b, rays_a, rays_b):
            n = int(cn.sum())
            ptrs, stream = _device_ptrs((frac_a, frac_b, rays_a, rays_b), (n, n, 3 * n, 3 * n))
            self._check(self.L.rssync_set_track_row_fractions_device(*args, *ptrs, float(readout), stream))
            return
        a = [_f64(x) for x in (frac_a, frac_b, rays_a, rays_b)]
        self._check(self.L.rssync_set_track_row_fractions(*args, *[_dp(x) for x in a], float(readout)))

    def track_frames(self, frames, counts, image_ts, points, images, lens, params=None):
        """Track points between decoded frames on the device and ingest the kept pairs
        (rssync_track_frames_device).  images: CUDA uint8 tensor (n_frames + 1, H, W) whose last dimension is
        contiguous (row pitch = stride(1)); frame i pairs images[i] (image_ts[i]) with images[i + 1];
        points: CUDA float64 tensor (sum(counts), 2), the query points on image i, frames concatenated.
        frames, counts and image_ts stay on the host; params: TrackParams or None (the defaults).  Ordered
        after the current stream of the tensors' device.  Returns (tracked, status): CUDA tensors
        (sum(counts), 2) float64 and (sum(counts),) uint8, every point's tracked position and status
        (1 = kept and ingested)."""
        import torch
        fr = np.ascontiguousarray(frames, dtype=np.int64)
        cn = np.ascontiguousarray(counts, dtype=np.uint64)
        ts = _f64(image_ts)
        n = int(cn.sum())
        if not (getattr(images, "is_cuda", False) and getattr(points, "is_cuda", False)):
            raise TypeError("track_frames: images and points must be CUDA tensors")
        if images.dtype != torch.uint8 or images.dim() != 3 or images.stride(2) != 1:
            raise ValueError("track_frames: images must be a uint8 tensor (n_frames + 1, H, W) with contiguous rows")
        if images.shape[0] != fr.shape[0] + 1 or ts.shape[0] != fr.shape[0] + 1:
            raise ValueError(f"track_frames: {fr.shape[0]} frames need {fr.shape[0] + 1} images and image timestamps, "
                             f"got {images.shape[0]} and {ts.shape[0]}")
        if images.shape[0] > 1 and images.stride(0) != images.shape[1] * images.stride(1):
            raise ValueError("track_frames: the planes must lie back to back (stride(0) = H * stride(1))")
        dev = images.device
        (pp,), stream = _device_ptrs((points,), (2 * n,))
        if points.device != dev:
            raise ValueError(f"track_frames: images on {dev}, points on {points.device}")
        tracked = torch.empty((n, 2), dtype=torch.float64, device=dev)
        status = torch.empty((n,), dtype=torch.uint8, device=dev)
        lens_c = lens if isinstance(lens, Lens) else Lens(*[float(x) for x in lens])
        prm = None if params is None else C.byref(params)
        self._check(self.L.rssync_track_frames_device(
            self.h, fr.shape[0], fr.ctypes.data_as(c_i64_p), cn.ctypes.data_as(C.POINTER(C.c_size_t)), _dp(ts), pp,
            C.c_void_p(images.data_ptr()), images.stride(1), images.shape[2], images.shape[1], C.byref(lens_c), prm,
            C.c_void_p(tracked.data_ptr() if n else None), C.c_void_p(status.data_ptr() if n else None), stream))
        return tracked, status

    def track_frames_ex(self, frames, image_ts, images, lens, params=None, options=None, points=None, counts=None,
                        shift=None, mask=None, mask_margin=None):
        """track_frames with the query points selected on the device (points and counts None) and the
        forward-backward check (rssync_track_frames_ex_device).  images, frames, image_ts, lens and params as in
        track_frames; options: TrackOptions or None (the defaults: 128-px cells, block 5, quality 0.01, 512
        points per frame, fb_max 1 px).  Returns TrackResult(points, counts, tracked, status, fb_error): the
        query points, tracked positions (CUDA float64 (n, 2)), statuses (CUDA uint8 (n,): 0 lost, 1 kept and
        ingested, 2 rejected by the backward check, 3 masked) and forward-backward distances (CUDA float64 (n,),
        NaN where the backward pass did not keep the point or did not run), n = sum(counts); counts: numpy.
        16-bit planes (rssync_track_frames16_device): a torch.uint16 tensor with shift, the intensity being
        sample * 2^-shift: 8 for P010 / P016, 2 for 10-bit and 4 for 12-bit samples in the low bits.  shift
        is required for uint16 and must be None for uint8.
        mask (rssync_track_frames_masked_device): a CUDA bool or uint8 tensor on the images' device with
        contiguous rows, nonzero where points may lie: (H, W) for one mask shared by every image, or
        (n_frames + 1, H, W) for one per image (an expanded tensor, stride(0) = 0, is shared).  The mask is
        eroded by mask_margin px (default params.window // 2 + 1, the level-0 LK patch): selection takes
        eligible candidates only, and a tracked point whose start or end is not eligible gets status 3.  With
        mask None the call is exactly the unmasked one."""
        import torch
        fr = np.ascontiguousarray(frames, dtype=np.int64)
        ts = _f64(image_ts)
        if (points is None) != (counts is None):
            raise ValueError("track_frames_ex: give both points and counts, or neither (selection)")
        if not getattr(images, "is_cuda", False):
            raise TypeError("track_frames_ex: images must be a CUDA tensor")
        wide = images.dtype == torch.uint16
        if not (wide or images.dtype == torch.uint8) or images.dim() != 3 or images.stride(2) != 1:
            raise ValueError("track_frames_ex: images must be a uint8 or uint16 tensor (n_frames + 1, H, W) with "
                             "contiguous rows")
        if wide and shift is None:
            raise ValueError("track_frames_ex: uint16 images need a shift (8 for P010 / P016, 2 for 10-bit and 4 "
                             "for 12-bit samples in the low bits)")
        if not wide and shift is not None:
            raise ValueError("track_frames_ex: shift applies to uint16 images only")
        if images.shape[0] != fr.shape[0] + 1 or ts.shape[0] != fr.shape[0] + 1:
            raise ValueError(f"track_frames_ex: {fr.shape[0]} frames need {fr.shape[0] + 1} images and image "
                             f"timestamps, got {images.shape[0]} and {ts.shape[0]}")
        if images.shape[0] > 1 and images.stride(0) != images.shape[1] * images.stride(1):
            raise ValueError("track_frames_ex: the planes must lie back to back (stride(0) = H * stride(1))")
        dev = images.device
        opt = TrackOptions() if options is None else options
        if points is None:
            cn, pp, cap = None, None, fr.shape[0] * max(int(opt.max_points), 0)
            stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        else:
            cn = np.ascontiguousarray(counts, dtype=np.uint64)
            cap = int(cn.sum())
            if not getattr(points, "is_cuda", False):
                raise TypeError("track_frames_ex: points must be a CUDA tensor")
            if points.device != dev:
                raise ValueError(f"track_frames_ex: images on {dev}, points on {points.device}")
            (pp,), stream = _device_ptrs((points,), (2 * cap,))
        pts_out = torch.empty((cap, 2), dtype=torch.float64, device=dev)
        tracked = torch.empty((cap, 2), dtype=torch.float64, device=dev)
        status = torch.empty((cap,), dtype=torch.uint8, device=dev)
        fb = torch.empty((cap,), dtype=torch.float64, device=dev)
        counts_out = np.zeros(fr.shape[0], dtype=np.uint64)
        lens_c = lens if isinstance(lens, Lens) else Lens(*[float(x) for x in lens])
        prm = None if params is None else C.byref(params)

        def ptr(t):
            return C.c_void_p(t.data_ptr() if cap else None)

        head = (self.h, fr.shape[0], fr.ctypes.data_as(c_i64_p),
                None if cn is None else cn.ctypes.data_as(C.POINTER(C.c_size_t)), _dp(ts), pp,
                C.c_void_p(images.data_ptr()), images.stride(1) * images.element_size(), images.shape[2],
                images.shape[1])
        tail = (C.byref(lens_c), prm, C.byref(opt), ptr(pts_out), counts_out.ctypes.data_as(C.POINTER(C.c_size_t)),
                ptr(tracked), ptr(status), ptr(fb), stream)
        if mask is not None:
            tm = self._track_mask(mask, images, params, mask_margin)
            self._check(self.L.rssync_track_frames_masked_device(*head, 2 if wide else 1, int(shift or 0),
                                                                 C.byref(tm), *tail))
        elif mask_margin is not None:
            raise ValueError("track_frames_ex: mask_margin needs a mask")
        elif wide:
            self._check(self.L.rssync_track_frames16_device(*head, int(shift), *tail))
        else:
            self._check(self.L.rssync_track_frames_ex_device(*head, *tail))
        n = int(counts_out.sum())
        return TrackResult(pts_out[:n], counts_out.astype(np.int64), tracked[:n], status[:n], fb[:n])

    @staticmethod
    def _track_mask(mask, images, params, margin):
        """track_frames_ex's mask tensor as an rssync_track_mask"""
        import torch
        if not getattr(mask, "is_cuda", False) or mask.device != images.device:
            raise ValueError(f"track_frames_ex: the mask must be a CUDA tensor on the images' device {images.device}")
        n, h, w = images.shape
        if mask.dtype not in (torch.bool, torch.uint8) or mask.stride(-1) != 1 or \
                tuple(mask.shape) not in ((h, w), (n, h, w)):
            raise ValueError(f"track_frames_ex: the mask must be a bool or uint8 tensor ({h}, {w}) or ({n}, {h}, {w}) "
                             f"with contiguous rows, got {mask.dtype} {tuple(mask.shape)}")
        if margin is None:
            margin = (TrackParams() if params is None else params).window // 2 + 1
        return TrackMask(mask.data_ptr(), mask.stride(-2), mask.stride(0) if mask.dim() == 3 else 0, int(margin))

    def load(self, w, bulk=False):
        """Feed a synth.Workload the way core_testcode feeds a video (core_testcode.cpp:257-268)."""
        self.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
        n = w.ts_a.shape[1]
        if bulk:
            self.set_track_batch(w.frame_ids, np.full(w.n_frames, n), w.ts_a, w.ts_b, w.rays_a, w.rays_b)
            return self
        for i, fid in enumerate(w.frame_ids):
            self.SetTrackResult(int(fid), w.ts_a[i], w.ts_b[i], w.rays_a[i], w.rays_b[i], n)
        return self

    def orientation_search(self, timestamps_s, gyro_xyz, orientations, initial_delay, frame_begin, frame_end,
                           search_step, search_radius, call_nos=None):
        """core_testcode.cpp:184-233: PreSync under every gyro_orientation variant.  Returns (costs, delays).
        call_nos: explicit RNG call number per variant (the problem's counter is then left alone)."""
        ts = _f64(timestamps_s)
        g = _f64(gyro_xyz)
        n = len(orientations)
        arr = (C.c_char_p * n)(*[o.encode() for o in orientations])
        costs, delays = np.empty(n), np.empty(n)
        cn = None
        if call_nos is not None:
            cn_arr = np.ascontiguousarray(call_nos, dtype=np.uint64)
            assert cn_arr.shape[0] == n
            cn = cn_arr.ctypes.data_as(C.POINTER(C.c_uint64))
        self._check(self.L.rssync_orientation_search_ex(self.h, _dp(ts), _dp(g), ts.shape[0], arr, n, initial_delay,
                                                        frame_begin, frame_end, search_step, search_radius, cn,
                                                        _dp(costs), _dp(delays)))
        return costs, delays

    def rotation_search(self, timestamps_s, gyro_xyz, rotations, initial_delay, frame_begin, frame_end,
                        search_step, search_radius, call_nos=None, curves=False):
        """orientation_search over 3x3 gyro axis mappings (a list of matrices or an (n, 3, 3) array) in
        place of the strings, e.g. candidate camera mount rotations (rssync_rotation_search).  Result i
        equals integrate_gyro(rotation=rotations[i]) -> SetGyroQuaternions (timestamps truncated to
        integer microseconds) -> PreSync.  Returns (costs, delays), plus the n x D cost curves over
        presync_delays(...) when curves=True.  call_nos: explicit RNG call number per matrix (the
        problem's counter is then left alone)."""
        ts = _f64(timestamps_s)
        g = _f64(gyro_xyz)
        m = _f64(rotations)
        if m.size == 0:
            m = m.reshape(0, 3, 3)
        if m.ndim != 3 or m.shape[1:] != (3, 3):
            raise ValueError(f"rotations must be a list of 3x3 matrices or an (n, 3, 3) array, got shape {m.shape}")
        n = m.shape[0]
        costs, delays = np.empty(n), np.empty(n)
        cn = None
        if call_nos is not None:
            cn_arr = np.ascontiguousarray(call_nos, dtype=np.uint64).ravel()
            if cn_arr.shape[0] != n:
                raise ValueError(f"{n} rotations but {cn_arr.shape[0]} call numbers")
            cn = cn_arr.ctypes.data_as(C.POINTER(C.c_uint64))
        cv = None
        if curves:
            D = self.L.rssync_presync_delays(initial_delay, search_step, search_radius, None, 0)
            cv = np.empty((n, max(D, 0)))
        self._check(self.L.rssync_rotation_search(self.h, _dp(ts), _dp(g), ts.shape[0], _dp(m), n, initial_delay,
                                                  frame_begin, frame_end, search_step, search_radius, cn,
                                                  _dp(costs), _dp(delays), _dp(cv) if curves else None))
        return (costs, delays, cv) if curves else (costs, delays)

    def readout_search(self, readouts, initial_delay, frame_begin, frame_end, search_step, search_radius,
                       call_nos=None, curves=False):
        """PreSync at every candidate rolling-shutter readout (seconds) over frames ingested from pixels
        or row fractions, without re-ingesting them (rssync_readout_search).  Returns (costs, delays), plus the n x D cost
        curves over presync_delays(...) when curves=True.  call_nos: explicit RNG call number per readout
        (the problem's counter is then left alone)."""
        r = _f64(readouts).ravel()
        n = r.shape[0]
        costs, delays = np.empty(n), np.empty(n)
        cn = None
        if call_nos is not None:
            cn_arr = np.ascontiguousarray(call_nos, dtype=np.uint64).ravel()
            if cn_arr.shape[0] != n:
                raise ValueError(f"{n} readouts but {cn_arr.shape[0]} call numbers")
            cn = cn_arr.ctypes.data_as(C.POINTER(C.c_uint64))
        cv = None
        if curves:
            D = self.L.rssync_presync_delays(initial_delay, search_step, search_radius, None, 0)
            cv = np.empty((n, max(D, 0)))
        self._check(self.L.rssync_readout_search(self.h, _dp(r), n, initial_delay, frame_begin, frame_end,
                                                 search_step, search_radius, cn, _dp(costs), _dp(delays),
                                                 _dp(cv) if curves else None))
        return (costs, delays, cv) if curves else (costs, delays)

    def _windowed_args(self, n, frame_begin, frame_end, initial_delay, search_step, search_radius, call_nos,
                       curves):
        """the window arrays, call numbers and output buffers of the windowed searches"""
        fb = np.ascontiguousarray(frame_begin, dtype=np.int64).ravel()
        fe = np.ascontiguousarray(frame_end, dtype=np.int64).ravel()
        if fb.shape != fe.shape:
            raise ValueError(f"{fb.shape[0]} window starts but {fe.shape[0]} window ends")
        W = fb.shape[0]
        cn = None
        if call_nos is not None:
            cn_arr = np.ascontiguousarray(call_nos, dtype=np.uint64).ravel()
            if cn_arr.shape[0] != n * W:
                raise ValueError(f"{n} candidates x {W} windows but {cn_arr.shape[0]} call numbers")
            cn = cn_arr
        costs, delays = np.empty((n, W)), np.empty((n, W))
        cv = None
        if curves:
            D = self.L.rssync_presync_delays(initial_delay, search_step, search_radius, None, 0)
            cv = np.empty((n, W, max(D, 0)))
        return fb, fe, cn, costs, delays, cv

    def readout_search_windows(self, readouts, initial_delay, frame_begin, frame_end, search_step, search_radius,
                               call_nos=None, curves=False):
        """readout_search over W frame windows [frame_begin[w], frame_end[w]) at once
        (rssync_readout_search_windows).  Returns (costs, delays) of shape (n, W), plus the (n, W, D) cost
        curves when curves=True; entry [j, w] is PreSync over window w at readout j, keyed by call number
        call_nos[j * W + w] (None: the next n * W values of the problem's counter).  Score the readouts by
        the sum over windows: estimate_readout(readouts, costs.sum(axis=1))."""
        r = _f64(readouts).ravel()
        n = r.shape[0]
        fb, fe, cn, costs, delays, cv = self._windowed_args(n, frame_begin, frame_end, initial_delay, search_step,
                                                            search_radius, call_nos, curves)
        self._check(self.L.rssync_readout_search_windows(
            self.h, _dp(r), n, fb.shape[0], fb.ctypes.data_as(c_i64_p), fe.ctypes.data_as(c_i64_p), initial_delay,
            search_step, search_radius, None if cn is None else cn.ctypes.data_as(C.POINTER(C.c_uint64)),
            _dp(costs), _dp(delays), _dp(cv) if curves else None))
        return (costs, delays, cv) if curves else (costs, delays)

    def rotation_search_windows(self, timestamps_s, gyro_xyz, rotations, initial_delay, frame_begin, frame_end,
                                search_step, search_radius, call_nos=None, curves=False):
        """rotation_search over W frame windows [frame_begin[w], frame_end[w]) at once
        (rssync_rotation_search_windows); shapes and call numbers as in readout_search_windows.  Score the
        rotations by the sum over windows: estimate_angle(angles, costs.sum(axis=1)).  For gyro_orientation
        strings, pass [orientation_matrix(s) for s in strings]."""
        ts = _f64(timestamps_s)
        g = _f64(gyro_xyz)
        m = _f64(rotations)
        if m.size == 0:
            m = m.reshape(0, 3, 3)
        if m.ndim != 3 or m.shape[1:] != (3, 3):
            raise ValueError(f"rotations must be a list of 3x3 matrices or an (n, 3, 3) array, got shape {m.shape}")
        n = m.shape[0]
        fb, fe, cn, costs, delays, cv = self._windowed_args(n, frame_begin, frame_end, initial_delay, search_step,
                                                            search_radius, call_nos, curves)
        self._check(self.L.rssync_rotation_search_windows(
            self.h, _dp(ts), _dp(g), ts.shape[0], _dp(m), n, fb.shape[0], fb.ctypes.data_as(c_i64_p),
            fe.ctypes.data_as(c_i64_p), initial_delay, search_step, search_radius,
            None if cn is None else cn.ctypes.data_as(C.POINTER(C.c_uint64)), _dp(costs), _dp(delays),
            _dp(cv) if curves else None))
        return (costs, delays, cv) if curves else (costs, delays)

    def set_readout(self, readout, frame_begin, frame_end):
        """Re-time the frames of [frame_begin, frame_end), ingested from pixels or row fractions, at
        `readout` (seconds) in place, as if they had been ingested with that readout (rssync_set_readout)."""
        self._check(self.L.rssync_set_readout(self.h, float(readout), int(frame_begin), int(frame_end)))

    def device_count(self):
        return self.L.rssync_device_count(self.h)

    # ---- moving the finished device state (replication without re-ingesting) ----------------
    def frame_table(self):
        """host-side frame table as a numpy structured array (id, off, n, ts_lo, ts_hi)"""
        n = self.L.rssync_frame_table(self.h, None, 0)
        arr = (FrameDesc * max(n, 1))()
        self.L.rssync_frame_table(self.h, arr, n)
        dt = np.dtype([("id", "<i8"), ("off", "<i4"), ("n", "<i4"), ("ts_lo", "<f8"), ("ts_hi", "<f8")])
        return np.frombuffer(bytes(arr), dtype=dt, count=n).copy()

    def device_state(self):
        """flush, then {rays, orig, pos, spline_records: (device pointer, bytes)} + sizes"""
        st = DeviceState()
        self._check(self.L.rssync_device_state(self.h, C.byref(st)))
        return {"rays": (st.rays, st.arena_rays * 64), "orig": (st.orig, st.arena_rays * 4),
                "pos": (st.pos, st.arena_rays * 4), "spline_records": (st.spline_records, st.gyro_samples * 128),
                "arena_rays": st.arena_rays, "gyro_samples": st.gyro_samples, "sample_rate": st.sample_rate,
                "first_timestamp": st.first_timestamp}

    @staticmethod
    def _state_dict(st):
        return {"rays": (st.rays, st.arena_rays * 64), "orig": (st.orig, st.arena_rays * 4),
                "pos": (st.pos, st.arena_rays * 4), "spline_records": (st.spline_records, st.gyro_samples * 128),
                "arena_rays": st.arena_rays, "gyro_samples": st.gyro_samples, "sample_rate": st.sample_rate,
                "first_timestamp": st.first_timestamp}

    def device_state_pipelined(self):
        """device_state() without waiting for the device, plus the arena ranges [(lo, hi), ...] of the
        bulk-ingest chunks still in flight (stream_wait_chunk(k, stream) orders a stream behind chunk k)"""
        st = DeviceState()
        cap = 64
        lo, hi, n = (C.c_size_t * cap)(), (C.c_size_t * cap)(), C.c_size_t(0)
        self._check(self.L.rssync_device_state_pipelined(self.h, C.byref(st), lo, hi, cap, C.byref(n)))
        d = self._state_dict(st)
        if n.value > cap:  # more chunks than we asked for: treat the ingest as one piece
            d["chunks"] = None
        else:
            d["chunks"] = [(int(lo[k]), int(hi[k])) for k in range(n.value)]
        return d

    def stream_wait_chunk(self, k, stream):
        self._check(self.L.rssync_stream_wait_chunk(self.h, int(k), C.c_void_p(int(stream))))

    def expect_chunk(self, lo, hi, stream):
        self._check(self.L.rssync_expect_chunk(self.h, int(lo), int(hi), C.c_void_p(int(stream))))

    def note_reader(self, stream):
        self._check(self.L.rssync_note_reader(self.h, C.c_void_p(int(stream))))

    def adopt_state(self, frame_table, arena_rays, gyro_samples, sample_rate, first_timestamp):
        """prepare this problem to hold a copy of another problem's device state (the buffers are
        allocated here; fill them through device_state()'s pointers)"""
        ft = np.ascontiguousarray(frame_table)
        self._check(self.L.rssync_adopt_state(self.h, ft.ctypes.data_as(C.POINTER(FrameDesc)), ft.shape[0],
                                              int(arena_rays), int(gyro_samples), float(sample_rate),
                                              float(first_timestamp)))

    def retime_table(self):
        """frames that hold row fractions (ascending id) as a numpy structured array (id, frame_ts_a,
        frame_ts_b)"""
        n = self.L.rssync_retime_table(self.h, None, 0)
        arr = (RetimeDesc * max(n, 1))()
        self.L.rssync_retime_table(self.h, arr, n)
        return np.frombuffer(bytes(arr), dtype=RETIME_DTYPE, count=n).copy()

    def row_fraction_plane(self):
        """flush, then (device pointer, bytes) of the row-fraction plane (2 doubles per arena ray);
        (0, 0) when no frame holds row fractions"""
        ptr, n = C.c_void_p(), C.c_size_t(0)
        self._check(self.L.rssync_row_fraction_plane(self.h, C.byref(ptr), C.byref(n)))
        return (ptr.value or 0, n.value * 8)

    def adopt_row_fractions(self, table):
        """after adopt_state: register another problem's retime_table() and allocate the plane (fill it
        through row_fraction_plane(), then expect_chunk(0, arena_rays, stream) for the writing stream)"""
        t = np.ascontiguousarray(table, dtype=RETIME_DTYPE)
        self._check(self.L.rssync_adopt_row_fractions(self.h, t.ctypes.data_as(C.POINTER(RetimeDesc)), t.shape[0]))

    def set_kernel_timing(self, enabled=True):
        self._check(self.L.rssync_set_kernel_timing(self.h, 1 if enabled else 0))

    def set_loss_mode(self, simplified):
        """False: the reference's loss; True: the thesis' simplified (no-translation) variant"""
        self._check(self.L.rssync_set_loss_mode(self.h, 1 if simplified else 0))

    def set_rng(self, seed, call_no=0):
        self._check(self.L.rssync_set_rng(self.h, seed, call_no))
        self.seed = seed

    def call_counter(self):
        return self.L.rssync_call_counter(self.h)

    def set_stream(self, cuda_stream):
        self._check(self.L.rssync_set_stream(self.h, C.c_void_p(cuda_stream)))

    def flush(self):
        self._check(self.L.rssync_flush(self.h))

    def presync_grid(self, frame_begin, frame_end, delays, stream=STREAM_PRESYNC, call_no=0,
                     offset_index_base=0, return_flags=False):
        delays = _f64(delays)
        costs = np.empty(delays.shape[0])
        flags = C.c_uint()
        self._check(self.L.rssync_presync_grid(self.h, frame_begin, frame_end, _dp(delays), delays.shape[0],
                                               stream, call_no, offset_index_base, _dp(costs), C.byref(flags)))
        return (costs, flags.value) if return_flags else costs

    def presync_windows(self, initial_delay, frame_begin, frame_end, search_step, search_radius, call_nos=None):
        """n PreSync calls (one per frame window, shared delay grid) as one grid launch -> (costs, delays)"""
        fb = np.ascontiguousarray(frame_begin, dtype=np.int64)
        fe = np.ascontiguousarray(frame_end, dtype=np.int64)
        n = fb.shape[0]
        cn = None
        if call_nos is not None:
            cn_arr = np.ascontiguousarray(call_nos, dtype=np.uint64)
            cn = cn_arr.ctypes.data_as(C.POINTER(C.c_uint64))
        costs, delays = np.empty(n), np.empty(n)
        self._check(self.L.rssync_presync_windows(self.h, n, initial_delay, fb.ctypes.data_as(c_i64_p),
                                                  fe.ctypes.data_as(c_i64_p), search_step, search_radius, cn,
                                                  _dp(costs), _dp(delays)))
        return costs, delays

    def sync_batch(self, initial_delay, frame_begin, frame_end, search_center, search_radius, call_nos=None):
        ini = _f64(initial_delay)
        n = ini.shape[0]
        fb = np.ascontiguousarray(frame_begin, dtype=np.int64)
        fe = np.ascontiguousarray(frame_end, dtype=np.int64)
        cen = _f64(np.broadcast_to(search_center, (n,)))
        rad = _f64(np.broadcast_to(search_radius, (n,)))
        cost, delay = np.empty(n), np.empty(n)
        if call_nos is not None:
            cn = np.ascontiguousarray(call_nos, dtype=np.uint64)
            self._check(self.L.rssync_sync_batch_ex(
                self.h, n, _dp(ini), fb.ctypes.data_as(c_i64_p), fe.ctypes.data_as(c_i64_p), _dp(cen), _dp(rad),
                cn.ctypes.data_as(C.POINTER(C.c_uint64)), _dp(cost), _dp(delay)))
            return cost, delay
        self._check(self.L.rssync_sync_batch(self.h, n, _dp(ini), fb.ctypes.data_as(c_i64_p),
                                             fe.ctypes.data_as(c_i64_p), _dp(cen), _dp(rad), _dp(cost), _dp(delay)))
        return cost, delay

    def last_sync_trace(self):
        n = self.L.rssync_last_sync_trace(self.h, None, None, 0)
        d, s = np.empty(n), np.empty(n)
        self.L.rssync_last_sync_trace(self.h, _dp(d), _dp(s), n)
        return d, s

    def stats(self):
        s = Stats()
        self._check(self.L.rssync_get_stats(self.h, C.byref(s)))
        return {k: getattr(s, k) for k, _ in Stats._fields_}

    # ---- probes (parity tests) --------------------------------------------------------------
    def probe_gyro(self):
        sr, q0, n = C.c_double(), C.c_double(), C.c_size_t()
        self._check(self.L.rssync_probe_gyro(self.h, C.byref(sr), C.byref(q0), C.byref(n), None))
        rec = np.empty((n.value, 16))
        self._check(self.L.rssync_probe_gyro(self.h, None, None, None, _dp(rec)))
        return sr.value, q0.value, rec

    def probe_problem_matrix(self, frame, delay, n):
        P = np.empty((n, 3))
        self._check(self.L.rssync_probe_problem_matrix(self.h, frame, delay, _dp(P)))
        return P

    def probe_guess_motion(self, frame, delay, iters, stream, call_no, offset_index):
        m = np.empty(3)
        k = C.c_double()
        self._check(self.L.rssync_probe_guess_motion(self.h, frame, delay, iters, stream, call_no, offset_index,
                                                     _dp(m), C.byref(k)))
        return m, k.value

    def probe_guess_motion_ex(self, frame, delay, iters, stream, call_no, offset_index, mode):
        """mode 0: product path, mode 2: exact binary64 estimator.  Returns (m, k, used_exact)."""
        m = np.empty(3)
        k = C.c_double()
        ex = C.c_int()
        self._check(self.L.rssync_probe_guess_motion_ex(self.h, frame, delay, iters, stream, call_no,
                                                        offset_index, mode, _dp(m), C.byref(k), C.byref(ex)))
        return m, k.value, ex.value

    def probe_loss(self, frame, delay, m, k):
        m = _f64(m)
        l3, l5 = C.c_double(), C.c_double()
        g = np.empty(3)
        self._check(self.L.rssync_probe_loss(self.h, frame, delay, _dp(m), k, C.byref(l3), C.byref(l5), _dp(g)))
        return l3.value, l5.value, g

    def probe_lbfgs(self, frame, delay, m, k):
        m = np.array(m, dtype=np.float64)
        f = C.c_double()
        it, ev = C.c_int(), C.c_int()
        self._check(self.L.rssync_probe_lbfgs(self.h, frame, delay, _dp(m), k, C.byref(f), C.byref(it), C.byref(ev)))
        return m, f.value, it.value, ev.value


def CreateSyncProblem(seed=100):
    """CreateSyncProblem(), rssync.h:31."""
    return SyncProblem(seed=seed)
