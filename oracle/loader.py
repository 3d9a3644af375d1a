"""ctypes loader for the CPU oracle (TEST INFRASTRUCTURE ONLY — see oracle/README.md).

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import
this module.  The product package never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

c_double_p = C.POINTER(C.c_double)
c_i64_p = C.POINTER(C.c_int64)


def _dp(a):
    return a.ctypes.data_as(c_double_p)


def _cpu_has_fma():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("flags"):
                    return " fma " in (line + " ")
    except OSError:
        pass
    return False


def build(force=False):
    subprocess.check_call(["make", "-s", "-C", HERE] + (["-B"] if force else []) + ["oracle"])


def lib():
    global _LIB
    if _LIB is not None:
        return _LIB
    name = "liboracle_fma.so" if _cpu_has_fma() else "liboracle_generic.so"
    path = os.path.join(HERE, name)
    if not os.path.exists(path):
        build()
    L = C.CDLL(path)
    L.orc_create.restype = C.c_void_p
    L.orc_last_error.restype = C.c_char_p
    L.orc_last_error.argtypes = [C.c_void_p]
    L.orc_destroy.argtypes = [C.c_void_p]
    L.orc_set_threads.argtypes = [C.c_void_p, C.c_int]
    L.orc_set_rng.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64]
    L.orc_set_loss_mode.argtypes = [C.c_void_p, C.c_int]
    L.orc_set_strict.argtypes = [C.c_void_p, C.c_int, c_i64_p, C.c_int]
    L.orc_call_no.argtypes = [C.c_void_p]
    L.orc_call_no.restype = C.c_uint64
    L.orc_set_gyro_fixed.argtypes = [C.c_void_p, c_double_p, C.c_size_t, C.c_double, C.c_double]
    L.orc_set_gyro_var.argtypes = [C.c_void_p, c_i64_p, c_double_p, C.c_size_t]
    L.orc_set_track.argtypes = [C.c_void_p, C.c_int64, c_double_p, c_double_p, c_double_p, c_double_p, C.c_size_t]
    L.orc_presync_grid.argtypes = [C.c_void_p, C.c_int64, C.c_int64, c_double_p, C.c_int, C.c_uint64,
                                   C.c_uint64, C.c_uint64, c_double_p, c_double_p, C.POINTER(C.c_int)]
    L.orc_presync_delays.argtypes = [C.c_double, C.c_double, C.c_double, c_double_p, C.c_int]
    L.orc_presync.argtypes = [C.c_void_p, C.c_double, C.c_int64, C.c_int64, C.c_double, C.c_double,
                              c_double_p, c_double_p]
    L.orc_debug_presync.argtypes = [C.c_void_p, C.c_double, C.c_int64, C.c_int64, C.c_double,
                                    c_double_p, c_double_p, C.c_int]
    L.orc_sync.argtypes = [C.c_void_p, C.c_double, C.c_int64, C.c_int64, C.c_double, C.c_double,
                           c_double_p, c_double_p]
    L.orc_sync_traced.argtypes = [C.c_void_p, C.c_double, C.c_int64, C.c_int64, C.c_double, C.c_double,
                                  c_double_p, c_double_p, c_double_p, c_double_p, C.c_int,
                                  C.POINTER(C.c_int), C.POINTER(C.c_long)]
    L.orc_gyro_count.argtypes = [C.c_void_p]
    L.orc_gyro_count.restype = C.c_long
    L.orc_gyro_rate.argtypes = [C.c_void_p]
    L.orc_gyro_rate.restype = C.c_double
    L.orc_gyro_start.argtypes = [C.c_void_p]
    L.orc_gyro_start.restype = C.c_double
    L.orc_get_spline.argtypes = [C.c_void_p, c_double_p]
    L.orc_get_resampled.argtypes = [C.c_void_p, c_double_p]
    L.orc_spline_eval.argtypes = [C.c_void_p, c_double_p, C.c_int, c_double_p]
    L.orc_problem_matrix.argtypes = [C.c_void_p, C.c_int64, C.c_double, c_double_p]
    L.orc_guess_motion.argtypes = [C.c_void_p, C.c_int64, C.c_double, C.c_int, C.c_uint64, C.c_uint64,
                                   C.c_uint64, c_double_p, c_double_p]
    L.orc_estimator_trace.argtypes = [C.c_void_p, C.c_int64, C.c_double, C.c_int, C.c_uint64, C.c_uint64,
                                      C.c_uint64, c_double_p, c_double_p, C.POINTER(C.c_int)]
    L.orc_loss3.argtypes =[C.c_void_p, C.c_int64, C.c_double, c_double_p, C.c_double, c_double_p]
    L.orc_loss5.argtypes = [C.c_void_p, C.c_int64, C.c_double, c_double_p, C.c_double, c_double_p, c_double_p]
    L.orc_lbfgs.argtypes = [C.c_void_p, C.c_int64, C.c_double, c_double_p, C.c_double, c_double_p,
                            C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.orc_log1p.argtypes = [c_double_p, C.c_int, c_double_p]
    L.orc_spec_trig.argtypes = [c_double_p, C.c_int, C.c_int, c_double_p]
    L.orc_integrate_gyro.argtypes = [c_double_p, c_double_p, C.c_size_t, C.c_char_p, c_double_p]
    L.orc_slerp.argtypes = [c_double_p, c_double_p, C.c_double, c_double_p]
    L.orc_rng_index.argtypes = [C.c_uint64, C.c_uint64, C.c_uint64, C.c_uint64, C.c_int64, C.c_uint32,
                                C.c_uint32, C.c_uint32]
    L.orc_rng_index.restype = C.c_uint32
    L.orc_ddsum.argtypes = [c_double_p, C.c_int]
    L.orc_ddsum.restype = C.c_double
    _LIB = L
    return L


class OracleError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"oracle status {code}: {msg}")
        self.code = code
        self.message = msg


STREAM_PRESYNC, STREAM_DEBUG, STREAM_SYNCINIT = 1, 2, 3


class OracleProblem:
    """Mirror of ISyncProblem (rssync.h:9-29) over the CPU oracle."""

    def __init__(self, threads=1, seed=100):
        self.L = lib()
        self.h = C.c_void_p(self.L.orc_create())
        self.L.orc_set_threads(self.h, threads)
        self.L.orc_set_rng(self.h, seed, 0)
        self._seed = seed
        self._frames = set()

    def __del__(self):
        try:
            self.L.orc_destroy(self.h)
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise OracleError(rc, self.L.orc_last_error(self.h).decode())

    def set_rng(self, seed, call_no=0):
        self._seed = seed
        self.L.orc_set_rng(self.h, seed, call_no)

    @property
    def seed(self):
        return self._seed

    def call_counter(self):
        self.L.orc_call_no.restype = C.c_uint64
        self.L.orc_call_no.argtypes = [C.c_void_p]
        return int(self.L.orc_call_no(self.h))

    def set_loss_mode(self, simplified):
        """simplified (no-translation) loss mode, see rssync_set_loss_mode"""
        self.L.orc_set_loss_mode(self.h, 1 if simplified else 0)

    def set_threads(self, n):
        self.L.orc_set_threads(self.h, n)

    def set_strict(self, strict=True, frame_order=None):
        """reference-order arithmetic (oracle_strict.hpp); frame_order = the reference's
        unordered_map iteration order, so per-frame sums are accumulated in the same sequence"""
        if frame_order is None:
            self.L.orc_set_strict(self.h, 1 if strict else 0, None, 0)
        else:
            fo = np.ascontiguousarray(frame_order, dtype=np.int64)
            self.L.orc_set_strict(self.h, 1 if strict else 0, fo.ctypes.data_as(c_i64_p), fo.shape[0])

    def SetGyroQuaternions(self, *args):
        if len(args) == 4:
            data, count, rate, first = args
            data = np.ascontiguousarray(data, dtype=np.float64)
            self._check(self.L.orc_set_gyro_fixed(self.h, _dp(data), count, rate, first))
        else:
            ts, quats, count = args
            ts = np.ascontiguousarray(ts, dtype=np.int64)
            quats = np.ascontiguousarray(quats, dtype=np.float64)
            self._check(self.L.orc_set_gyro_var(self.h, ts.ctypes.data_as(c_i64_p), _dp(quats), count))

    def SetTrackResult(self, frame, ts_a, ts_b, rays_a, rays_b, count):
        a = [np.ascontiguousarray(x, dtype=np.float64) for x in (ts_a, ts_b, rays_a, rays_b)]
        self._check(self.L.orc_set_track(self.h, int(frame), _dp(a[0]), _dp(a[1]), _dp(a[2]), _dp(a[3]), count))
        self._frames.add(int(frame))

    def load(self, w):
        self.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
        for i, fid in enumerate(w.frame_ids):
            self.SetTrackResult(int(fid), w.ts_a[i], w.ts_b[i], w.rays_a[i], w.rays_b[i], w.ts_a.shape[1])
        return self

    def load_range(self, w, first_frame, n_frames):
        """gyro + only the frames first_frame .. first_frame + n_frames - 1"""
        self.SetGyroQuaternions(w.quats, w.quats.shape[0], w.gyro_rate, w.gyro_t0)
        for i, fid in enumerate(w.frame_ids):
            if first_frame <= int(fid) < first_frame + n_frames:
                self.SetTrackResult(int(fid), w.ts_a[i], w.ts_b[i], w.rays_a[i], w.rays_b[i], w.ts_a.shape[1])
        return self

    def PreSync(self, initial, fb, fe, step, radius):
        c, d = C.c_double(), C.c_double()
        self._check(self.L.orc_presync(self.h, initial, fb, fe, step, radius, C.byref(c), C.byref(d)))
        return c.value, d.value

    def DebugPreSync(self, initial, fb, fe, radius, point_count):
        delays = np.empty(point_count)
        costs = np.empty(point_count)
        self._check(self.L.orc_debug_presync(self.h, initial, fb, fe, radius, _dp(delays), _dp(costs), point_count))
        return delays, costs

    def Sync(self, initial, fb, fe, center, radius, trace=False):
        c, d = C.c_double(), C.c_double()
        if not trace:
            self._check(self.L.orc_sync(self.h, initial, fb, fe, center, radius, C.byref(c), C.byref(d)))
            return c.value, d.value
        td, ts = np.empty(400), np.empty(400)
        n = C.c_int()
        cnt = (C.c_long * 8)()
        self._check(self.L.orc_sync_traced(self.h, initial, fb, fe, center, radius, C.byref(c), C.byref(d),
                                           _dp(td), _dp(ts), 400, C.byref(n), cnt))
        return c.value, d.value, td[:n.value].copy(), ts[:n.value].copy(), list(cnt)[:5]

    def presync_grid(self, fb, fe, delays, stream=STREAM_PRESYNC, call_no=0, offset_index_base=0,
                     frame_costs=False, idx_base=None):
        if idx_base is None:
            idx_base = offset_index_base
        delays = np.ascontiguousarray(delays, dtype=np.float64)
        n = delays.shape[0]
        costs = np.empty(n)
        flags = C.c_int()
        fc = None
        if frame_costs:
            nf = self.count_frames(fb, fe)
            fc = np.empty((n, nf))
        self._check(self.L.orc_presync_grid(self.h, fb, fe, _dp(delays), n, stream, call_no, idx_base,
                                            _dp(costs), _dp(fc) if fc is not None else None, C.byref(flags)))
        return (costs, fc, flags.value) if frame_costs else costs

    def count_frames(self, fb, fe):
        return sum(1 for f in self._frames if fb <= f < fe)

    def sync_batch(self, initial_delay, frame_begin, frame_end, search_center, search_radius, call_nos=None):
        """n independent Sync calls (the oracle runs them one after another)."""
        n = len(initial_delay)
        cen = np.broadcast_to(search_center, (n,))
        rad = np.broadcast_to(search_radius, (n,))
        cost, delay = np.empty(n), np.empty(n)
        seed = self._seed
        for i in range(n):
            if call_nos is not None:
                self.set_rng(seed, int(call_nos[i]))
            cost[i], delay[i] = self.Sync(float(initial_delay[i]), int(frame_begin[i]), int(frame_end[i]),
                                          float(cen[i]), float(rad[i]))
        return cost, delay

    def problem_matrix(self, frame, delay, n):
        P = np.empty((n, 3))
        self._check(self.L.orc_problem_matrix(self.h, frame, delay, _dp(P)))
        return P

    def guess_motion(self, frame, delay, iters, stream, call_no, offset_idx):
        m = np.empty(3)
        k = C.c_double()
        self._check(self.L.orc_guess_motion(self.h, frame, delay, iters, stream, call_no, offset_idx, _dp(m), C.byref(k)))
        return m, k.value

    def estimator_trace(self, frame, delay, iters, stream, call_no, offset_idx):
        """guess_motion with every hypothesis kept -> (hypotheses (iters, 3), exact quartiles (iters,),
        index of the winner: the first strict minimum)"""
        v = np.empty((iters, 3))
        q = np.empty(iters)
        best = C.c_int()
        self._check(self.L.orc_estimator_trace(self.h, frame, delay, iters, stream, call_no, offset_idx, _dp(v),
                                               _dp(q), C.byref(best)))
        return v, q, best.value

    def loss3(self, frame, delay, m, k):
        m = np.ascontiguousarray(m, dtype=np.float64)
        out = C.c_double()
        self._check(self.L.orc_loss3(self.h, frame, delay, _dp(m), k, C.byref(out)))
        return out.value

    def loss5(self, frame, delay, m, k):
        m = np.ascontiguousarray(m, dtype=np.float64)
        out = C.c_double()
        g = np.empty(3)
        self._check(self.L.orc_loss5(self.h, frame, delay, _dp(m), k, C.byref(out), _dp(g)))
        return out.value, g

    def lbfgs(self, frame, delay, m, k):
        m = np.array(m, dtype=np.float64)
        f = C.c_double()
        it, ev = C.c_int(), C.c_int()
        self._check(self.L.orc_lbfgs(self.h, frame, delay, _dp(m), k, C.byref(f), C.byref(it), C.byref(ev)))
        return m, f.value, it.value, ev.value

    def spline(self):
        n = self.L.orc_gyro_count(self.h)
        rec = np.empty((n, 16))
        self.L.orc_get_spline(self.h, _dp(rec))
        return rec

    def resampled(self):
        n = self.L.orc_gyro_count(self.h)
        q = np.empty((n, 4))
        self.L.orc_get_resampled(self.h, _dp(q))
        return q, self.L.orc_gyro_rate(self.h), self.L.orc_gyro_start(self.h)

    def spline_eval(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        out = np.empty((x.shape[0], 4))
        self.L.orc_spline_eval(self.h, _dp(x), x.shape[0], _dp(out))
        return out


def integrate_gyro(timestamps_s, gyro_xyz, orientation=None):
    """optdata_fill_gyro (core_testcode.cpp:37-53): raw gyro -> orientation quaternions"""
    ts = np.ascontiguousarray(timestamps_s, dtype=np.float64)
    g = np.ascontiguousarray(gyro_xyz, dtype=np.float64)
    out = np.empty((ts.shape[0], 4))
    rc = lib().orc_integrate_gyro(_dp(ts), _dp(g), ts.shape[0], orientation.encode() if orientation else None, _dp(out))
    if rc:
        raise OracleError(rc, "malformed orientation")
    return out


def orientation_search(problem, timestamps_s, gyro_xyz, orientations, initial, fb, fe, step, radius):
    """the loop of core_testcode.cpp:212-224 on an OracleProblem: per variant integrate, ingest through
    the variable-rate SetGyroQuaternions (timestamps truncated to integer microseconds), PreSync"""
    ts = np.ascontiguousarray(timestamps_s, dtype=np.float64)
    ts_us = (ts * 1000000).astype(np.int64)  # :47-50 (truncation)
    out = []
    for o in orientations:
        q = integrate_gyro(ts, gyro_xyz, o)
        problem.SetGyroQuaternions(ts_us, q, len(ts_us))
        out.append(problem.PreSync(initial, fb, fe, step, radius))
    return np.array([c for c, _ in out]), np.array([d for _, d in out])


def presync_delays(initial, step, radius):
    L = lib()
    n = L.orc_presync_delays(initial, step, radius, None, 0)
    out = np.empty(n)
    L.orc_presync_delays(initial, step, radius, _dp(out), n)
    return out


def spec_trig(x, which):
    """the contract's sin / cos / acos as the oracle restates them (oracle/spec_trig.hpp)"""
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.empty_like(x)
    lib().orc_spec_trig(_dp(x), x.size, {"sin": 0, "cos": 1, "acos": 2}[which], _dp(out))
    return out


def log1p(x):
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.empty_like(x)
    lib().orc_log1p(_dp(x), x.size, _dp(out))
    return out
