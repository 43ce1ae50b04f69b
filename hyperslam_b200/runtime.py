"""ctypes binding of libhyperb200.so (include/hyperb200.h) -- the only way Python reaches the hot path.

There is no CPU fallback: constructing a Context without the built library or without a B200
raises.  The oracle under oracle/ is never imported from here.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libhyperb200.so")

PIXEL, INERTIAL, BEARING, MANIFOLD = 0, 1, 2, 3
EVAL_JACOBIANS, EVAL_TRIAL = 1, 2

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


class Options(C.Structure):
    _fields_ = [("device", C.c_int), ("stream", C.c_void_p), ("use_graph", C.c_int), ("reserved", C.c_int),
                ("nccl_comm", C.c_void_p), ("nranks", C.c_int), ("rank", C.c_int)]


class SlideStats(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("knots_dropped", "knots_constant", "landmarks_dropped", "visual_factors_dropped", "inertial_factors_dropped",
                                       "knots", "landmarks", "visual_factors", "inertial_factors")]


SLIDE_DROP_INERTIAL = 1
SLIDE_DROP_POSE = 2


class Iteration(C.Structure):
    _fields_ = [("cost", C.c_double), ("cost_new", C.c_double), ("model_change", C.c_double), ("rho", C.c_double),
                ("radius", C.c_double), ("accepted", C.c_int), ("spd", C.c_int)]


ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p)

EXPORTS = [
    "hb200_create", "hb200_destroy", "hb200_last_error_string", "hb200_synchronize", "hb200_set_spline",
    "hb200_set_bias_splines", "hb200_set_gravity", "hb200_set_cameras", "hb200_set_imu", "hb200_set_landmarks",
    "hb200_set_constant", "hb200_set_options", "hb200_set_pixel_factors", "hb200_set_inertial_factors", "hb200_bind",
    "hb200_get_index_maps", "hb200_evaluate", "hb200_get_pixel_outputs", "hb200_get_inertial_outputs",
    "hb200_factor_evaluate", "hb200_reduced_size", "hb200_build_system", "hb200_get_system", "hb200_solve",
    "hb200_get_delta", "hb200_iterate", "hb200_cost", "hb200_get_state", "hb200_set_allreduce",
    "hb200_system_device_ptr", "hb200_stream", "hb200_launch_count", "hb200_optimize", "hb200_snapshot", "hb200_restore",
    "hb200_profile_iteration", "hb200_interpolate", "hb200_set_bearing_factors", "hb200_set_bearing_loss",
    "hb200_set_pose_sensors", "hb200_set_manifold_factors", "hb200_get_bearing_outputs", "hb200_get_manifold_outputs",
    "hb200_ingest_stereo", "hb200_comm_unique_id", "hb200_comm_init_rank", "hb200_set_nccl_comm", "hb200_peer_handle",
    "hb200_peer_connect", "hb200_peer_disconnect", "hb200_comm_info",
    "hb200_get_bandwidth", "hb200_set_min_bandwidth", "hb200_measure_fp64_peak", "hb200_set_reference_quirks",
    "hb200_append_knots", "hb200_append_landmarks", "hb200_append_pixel_factors", "hb200_append_inertial_factors", "hb200_slide",
    "hb200_window_sizes", "hb200_set_termination", "hb200_get_termination",
    "hb200_append_bearing_factors", "hb200_append_manifold_factors", "hb200_append_stereo_tracks", "hb200_factor_counts",
]

_lib = None


def load_library() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(hyperslam_b200 has no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        lib.hb200_last_error_string.restype = C.c_char_p
        lib.hb200_system_device_ptr.restype = C.c_void_p
        lib.hb200_stream.restype = C.c_void_p
        lib.hb200_launch_count.restype = C.c_longlong
        lib.hb200_launch_count.argtypes = [C.c_void_p]
        lib.hb200_destroy.argtypes = [C.c_void_p]
        lib.hb200_destroy.restype = None
        _lib = lib
    return _lib


class HB200Error(RuntimeError):
    pass


def _d(a):
    return None if a is None else a.ctypes.data_as(_dp)


def _i(a):
    return None if a is None else a.ctypes.data_as(_ip)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


class Context:
    """One sliding-window problem on one GPU (wraps an hb200_ctx)."""

    def __init__(self, device: int = 0, stream: int | None = None, use_graph: bool = True, force_dense: bool = False):
        self.lib = load_library()
        self.h = C.c_void_p()
        opts = Options(device, stream, int(use_graph), int(force_dense), None, 1, 0)
        self._check(self.lib.hb200_create(C.byref(opts), C.byref(self.h)))
        self._cb = None
        self.order = self.K = self.Kbg = self.Kba = self.L = self.Nv = self.Ni = self.Nb = self.Nm = 0
        self.bias_order = 4

    def _check(self, rc: int):
        if rc != 0:
            raise HB200Error(f"hb200 error {rc}: {self.lib.hb200_last_error_string().decode()}")

    def close(self):
        if getattr(self, "h", None) is not None and self.h:
            self.lib.hb200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- state ------------------------------------------------------------------------------
    def set_spline(self, order, knots):
        knots = _f64(knots)
        self.order, self.K = int(order), knots.shape[0]
        self._check(self.lib.hb200_set_spline(self.h, self.order, self.K, _d(knots)))

    def set_bias_splines(self, order, gyro, accel):
        gyro, accel = _f64(gyro), _f64(accel)
        self.bias_order, self.Kbg, self.Kba = int(order), gyro.shape[0], accel.shape[0]
        self._check(self.lib.hb200_set_bias_splines(self.h, int(order), self.Kbg, _d(gyro), self.Kba, _d(accel)))

    def set_gravity(self, g):
        self._check(self.lib.hb200_set_gravity(self.h, _d(_f64(g))))

    def set_cameras(self, cams):
        cams = _f64(cams)
        self._check(self.lib.hb200_set_cameras(self.h, cams.shape[0], _d(cams)))

    def set_imu(self, imu):
        self._check(self.lib.hb200_set_imu(self.h, _d(_f64(imu))))

    def set_landmarks(self, xyz):
        xyz = _f64(xyz)
        self.L = xyz.shape[0]
        self._check(self.lib.hb200_set_landmarks(self.h, self.L, _d(xyz)))

    def set_constant(self, knot_const=None, gravity_const=0, bias_const=0):
        kc = None if knot_const is None else np.ascontiguousarray(knot_const, dtype=np.uint8)
        ptr = None if kc is None else kc.ctypes.data_as(C.POINTER(C.c_ubyte))
        self._check(self.lib.hb200_set_constant(self.h, ptr, int(gravity_const), int(bias_const)))

    def set_options(self, huber_pixel=0.5, imu_loss_scale=1.6e-5, radius=1e4):
        self._check(self.lib.hb200_set_options(self.h, C.c_double(huber_pixel), C.c_double(imu_loss_scale), C.c_double(radius)))

    def set_reference_quirks(self, quirks: int):
        self._check(self.lib.hb200_set_reference_quirks(self.h, int(quirks)))

    def set_pixel_factors(self, stamp, cam, lm, pixel):
        stamp, pixel = _f64(stamp), _f64(pixel)
        cam, lm = np.ascontiguousarray(cam, dtype=np.int32), np.ascontiguousarray(lm, dtype=np.int32)
        self.Nv = stamp.size
        self._check(self.lib.hb200_set_pixel_factors(self.h, self.Nv, _d(stamp), _i(cam), _i(lm), _d(pixel)))

    def set_bearing_factors(self, stamp, cam, lm, bearing, huber=None):
        stamp, bearing = _f64(stamp), _f64(bearing)
        cam, lm = np.ascontiguousarray(cam, dtype=np.int32), np.ascontiguousarray(lm, dtype=np.int32)
        self.Nb = stamp.size
        self._check(self.lib.hb200_set_bearing_factors(self.h, self.Nb, _d(stamp), _i(cam), _i(lm), _d(bearing)))
        if huber is not None:
            self._check(self.lib.hb200_set_bearing_loss(self.h, C.c_double(huber)))

    def set_pose_sensors(self, T_bs):
        T_bs = _f64(T_bs)
        self._check(self.lib.hb200_set_pose_sensors(self.h, T_bs.shape[0], _d(T_bs)))

    def set_manifold_factors(self, stamp, sensor, pose):
        stamp, pose = _f64(stamp), _f64(pose)
        sensor = np.ascontiguousarray(sensor, dtype=np.int32)
        self.Nm = stamp.size
        self._check(self.lib.hb200_set_manifold_factors(self.h, self.Nm, _d(stamp), _i(sensor), _d(pose)))

    def set_inertial_factors(self, stamp, meas):
        stamp, meas = _f64(stamp), _f64(meas)
        self.Ni = stamp.size
        self._check(self.lib.hb200_set_inertial_factors(self.h, self.Ni, _d(stamp), _d(meas)))

    def bind(self) -> int:
        bad = C.c_int(0)
        rc = self.lib.hb200_bind(self.h, C.byref(bad))
        self.num_invalid = bad.value
        self._check(rc)
        return bad.value

    def load_window(self, w, radius=1e4):
        """Upload a hyperslam_b200.synthetic.Window and bind its factors."""
        self.set_spline(w.order, w.knots)
        self.set_bias_splines(w.bias_order, w.gyro_bias, w.accel_bias)
        self.set_gravity(w.gravity)
        self.set_cameras(w.cameras)
        self.set_imu(w.imu)
        self.set_landmarks(w.landmarks)
        self.set_options(w.huber_pixel, w.imu_loss_scale, radius)
        self.set_pixel_factors(w.v_stamp, w.v_cam, w.v_lm, w.v_pixel)
        self.set_inertial_factors(w.i_stamp, w.i_meas)
        self.set_bearing_factors(w.b_stamp, w.b_cam, w.b_lm, w.b_bearing, w.huber_bearing)
        self.set_pose_sensors(w.pose_sensors)
        self.set_manifold_factors(w.m_stamp, w.m_sensor, w.m_pose)
        self.bind()
        self.set_constant(w.knot_const, w.gravity_const, w.bias_const)

    # ---- device-side sliding-window bookkeeping ------------------------------------------------------
    def _refresh_sizes(self, counts=False):
        """counts: also re-read the bearing / pose-prior counts (calls that can change them); Nv = pixel factors."""
        v = [C.c_int(0) for _ in range(4)]
        self._check(self.lib.hb200_window_sizes(self.h, *[C.byref(x) for x in v]))
        self.K, self.L, self.Ni = v[0].value, v[1].value, v[3].value
        if counts:
            n = self.factor_counts()
            self.Nb, self.Nm = n["bearing"], n["manifold"]
        self.Nv = v[2].value - self.Nb

    def factor_counts(self):
        """Factors per kind: dict(pixel, bearing, inertial, manifold)."""
        v = [C.c_int(0) for _ in range(4)]
        self._check(self.lib.hb200_factor_counts(self.h, *[C.byref(x) for x in v]))
        return dict(zip(("pixel", "bearing", "inertial", "manifold"), (x.value for x in v)))

    def append_knots(self, count=1):
        self._check(self.lib.hb200_append_knots(self.h, int(count)))
        self._refresh_sizes()

    def append_landmarks(self, xyz):
        xyz = _f64(xyz).reshape(-1, 3)
        if xyz.shape[0]:
            self._check(self.lib.hb200_append_landmarks(self.h, xyz.shape[0], _d(xyz)))
            self._refresh_sizes()

    def append_pixel_factors(self, stamp, cam, lm, pixel):
        stamp, pixel = _f64(stamp), _f64(pixel)
        cam, lm = np.ascontiguousarray(cam, dtype=np.int32), np.ascontiguousarray(lm, dtype=np.int32)
        if stamp.size:
            self._check(self.lib.hb200_append_pixel_factors(self.h, stamp.size, _d(stamp), _i(cam), _i(lm), _d(pixel)))
            self._refresh_sizes()

    def append_inertial_factors(self, stamp, meas):
        stamp, meas = _f64(stamp), _f64(meas)
        if stamp.size:
            self._check(self.lib.hb200_append_inertial_factors(self.h, stamp.size, _d(stamp), _d(meas)))
            self._refresh_sizes()

    def append_bearing_factors(self, stamp, cam, lm, bearing):
        stamp, bearing = _f64(stamp), _f64(bearing)
        cam, lm = np.ascontiguousarray(cam, dtype=np.int32), np.ascontiguousarray(lm, dtype=np.int32)
        if stamp.size:
            self._check(self.lib.hb200_append_bearing_factors(self.h, stamp.size, _d(stamp), _i(cam), _i(lm), _d(bearing)))
            self._refresh_sizes(counts=True)

    def append_manifold_factors(self, stamp, sensor, pose):
        stamp, pose = _f64(stamp), _f64(pose)
        sensor = np.ascontiguousarray(sensor, dtype=np.int32)
        if stamp.size:
            self._check(self.lib.hb200_append_manifold_factors(self.h, stamp.size, _d(stamp), _i(sensor), _d(pose)))
            self._refresh_sizes(counts=True)

    def append_stereo_tracks(self, stamp, cam0, cam1, px0, px1, landmark):
        """process(VisualTracks): two bearing factors per track; landmark[i] == -1 triangulates and appends a new
        landmark.  Returns every track's landmark slot (new ones take L, L+1, ... in track order)."""
        stamp, px0, px1 = _f64(stamp), _f64(px0), _f64(px1)
        cam0, cam1 = np.ascontiguousarray(cam0, dtype=np.int32), np.ascontiguousarray(cam1, dtype=np.int32)
        landmark = np.ascontiguousarray(landmark, dtype=np.int32)
        out = np.zeros(stamp.size, dtype=np.int32)
        if stamp.size:
            num_new = C.c_int(0)
            self._check(self.lib.hb200_append_stereo_tracks(self.h, stamp.size, _d(stamp), _i(cam0), _i(cam1), _d(px0), _d(px1), _i(landmark),
                                                            _i(out), C.byref(num_new)))
            self._refresh_sizes(counts=True)
        return out

    def slide(self, lower_bound, drop_inertial=True, drop_pose=False):
        st = SlideStats()
        flags = (SLIDE_DROP_INERTIAL if drop_inertial else 0) | (SLIDE_DROP_POSE if drop_pose else 0)
        self._check(self.lib.hb200_slide(self.h, C.c_double(lower_bound), flags, C.byref(st)))
        self._refresh_sizes(counts=self.Nb > 0 or self.Nm > 0)
        return {n: getattr(st, n) for n, _ in SlideStats._fields_}

    def index_maps(self):
        vb = np.zeros(self.Nv, dtype=np.int32)
        ib, ig, ia = (np.zeros(self.Ni, dtype=np.int32) for _ in range(3))
        self._check(self.lib.hb200_get_index_maps(self.h, _i(vb), _i(ib), _i(ig), _i(ia)))
        return vb, ib, ig, ia

    # ---- hot path ---------------------------------------------------------------------------
    def evaluate(self, jacobians=True, trial=False):
        self._check(self.lib.hb200_evaluate(self.h, (EVAL_JACOBIANS if jacobians else 0) | (EVAL_TRIAL if trial else 0)))

    def outputs(self, jacobians=True):
        k, kb = self.order, self.bias_order
        out = dict(v_r=np.zeros((self.Nv, 2)), i_r=np.zeros((self.Ni, 6)))
        if jacobians:
            out.update(v_Jp=np.zeros((self.Nv, 2, 6 * k)), v_Jl=np.zeros((self.Nv, 2, 3)), i_Jp=np.zeros((self.Ni, 6, 6 * k)),
                       i_wg=np.zeros((self.Ni, kb)), i_wa=np.zeros((self.Ni, kb)), i_Jg=np.zeros((self.Ni, 6, 2)))
        self._check(self.lib.hb200_get_pixel_outputs(self.h, _d(out["v_r"]), _d(out.get("v_Jp")), _d(out.get("v_Jl"))))
        self._check(self.lib.hb200_get_inertial_outputs(self.h, _d(out["i_r"]), _d(out.get("i_Jp")), _d(out.get("i_wg")),
                                                        _d(out.get("i_wa")), _d(out.get("i_Jg"))))
        Nb, Nm = self.Nb, self.Nm
        if Nb:
            out["b_r"] = np.zeros(Nb)
            if jacobians:
                out.update(b_Jp=np.zeros((Nb, 6 * k)), b_Jl=np.zeros((Nb, 3)))
            self._check(self.lib.hb200_get_bearing_outputs(self.h, _d(out["b_r"]), _d(out.get("b_Jp")), _d(out.get("b_Jl"))))
        if Nm:
            out["m_r"] = np.zeros((Nm, 6))
            if jacobians:
                out["m_Jp"] = np.zeros((Nm, 6, 6 * k))
            self._check(self.lib.hb200_get_manifold_outputs(self.h, _d(out["m_r"]), _d(out.get("m_Jp"))))
        return out

    def factor_evaluate(self, kind, index, blocks, want_jacobians=True):
        """Ceres-shaped copy-out; blocks = list of 1-D parameter-block arrays in ExteroceptiveCost order."""
        blocks = [_f64(b) for b in blocks]
        nb = len(blocks)
        nr = {PIXEL: 2, INERTIAL: 6, BEARING: 1, MANIFOLD: 6}[kind]
        params = (_dp * nb)(*[_d(b) for b in blocks])
        r = np.zeros(nr)
        if want_jacobians:
            jac = [np.zeros((nr, b.size)) for b in blocks]
            jp = (_dp * nb)(*[_d(j) for j in jac])
        else:
            jac, jp = None, None
        self._check(self.lib.hb200_factor_evaluate(self.h, kind, int(index), params, _d(r), jp))
        return r, jac

    def reduced_size(self):
        return self.lib.hb200_reduced_size(self.h)

    def build_system(self):
        self._check(self.lib.hb200_build_system(self.h))

    def system(self):
        n = self.reduced_size()
        S, b = np.zeros((n, n)), np.zeros(n)
        self._check(self.lib.hb200_get_system(self.h, _d(S), _d(b)))
        return S, b

    def solve(self):
        self._check(self.lib.hb200_solve(self.h))

    def delta(self):
        dp, dl = np.zeros(self.reduced_size()), np.zeros((self.L, 3))
        self._check(self.lib.hb200_get_delta(self.h, _d(dp), _d(dl)))
        return dp, dl

    def iterate(self, iterations=1, records=True):
        rec = (Iteration * max(iterations, 1))()
        self._check(self.lib.hb200_iterate(self.h, int(iterations), rec if records else None))
        if not records:
            return None
        return [dict(cost=r.cost, cost_new=r.cost_new, model_change=r.model_change, rho=r.rho, radius=r.radius,
                     accepted=r.accepted, spd=r.spd) for r in rec[:iterations]]

    def optimize(self, iterations, knots, gyro, accel, gravity, landmarks, records=True):
        """hb200_optimize: host (ideally pinned) float64 arrays, updated in place."""
        rec = (Iteration * max(iterations, 1))()
        self._check(self.lib.hb200_optimize(self.h, int(iterations), _d(knots), _d(gyro), _d(accel), _d(gravity), _d(landmarks),
                                            rec if records else None))
        return [dict(cost=r.cost, cost_new=r.cost_new, rho=r.rho, radius=r.radius, accepted=r.accepted, spd=r.spd)
                for r in rec[:iterations]] if records else None

    def set_termination(self, function_tolerance=1e-6, gradient_tolerance=1e-10, parameter_tolerance=1e-8, min_trust_region_radius=1e-32):
        """Ceres' termination tests (defaults = ceres::Solver::Options defaults); all <= 0 switches them off."""
        self._check(self.lib.hb200_set_termination(self.h, C.c_double(function_tolerance), C.c_double(gradient_tolerance), C.c_double(parameter_tolerance),
                                                   C.c_double(min_trust_region_radius)))

    def termination(self):
        t, n = C.c_int(0), C.c_int(0)
        g, s_, x = C.c_double(0), C.c_double(0), C.c_double(0)
        self._check(self.lib.hb200_get_termination(self.h, C.byref(t), C.byref(n), C.byref(g), C.byref(s_), C.byref(x)))
        return dict(type=t.value, iterations=n.value, gradient_max_norm=g.value, step_norm=s_.value, x_norm=x.value)

    def snapshot(self):
        self._check(self.lib.hb200_snapshot(self.h))

    def restore(self):
        self._check(self.lib.hb200_restore(self.h))

    def profile_iteration(self, reps=5, max_entries=64, evaluate_only=False):
        if evaluate_only:
            reps = -abs(reps)
        names = C.create_string_buffer(32 * max_entries)
        ms = np.zeros(max_entries)
        cnt = C.c_int(0)
        self._check(self.lib.hb200_profile_iteration(self.h, int(reps), max_entries, names, _d(ms), C.byref(cnt)))
        out = []
        for i in range(cnt.value):
            raw = names.raw[32 * i: 32 * (i + 1)]
            out.append((raw.split(b"\0", 1)[0].decode(), float(ms[i])))
        return out

    def cost(self):
        c = C.c_double(0)
        self._check(self.lib.hb200_cost(self.h, C.byref(c)))
        return c.value

    def state(self):
        knots, bg, ba = np.zeros((self.K, 8)), np.zeros((self.Kbg, 4)), np.zeros((self.Kba, 4))
        g, lm = np.zeros(3), np.zeros((self.L, 3))
        self._check(self.lib.hb200_get_state(self.h, _d(knots), _d(bg), _d(ba), _d(g), _d(lm)))
        return dict(knots=knots, gyro_bias=bg, accel_bias=ba, gravity=g, landmarks=lm)

    def interpolate(self, stamps, derivatives=True):
        stamps = _f64(stamps)
        n = stamps.size
        pose = np.zeros((n, 7))
        vel = np.zeros((n, 6)) if derivatives else None
        acc = np.zeros((n, 6)) if derivatives else None
        bad = C.c_int(0)
        self._check(self.lib.hb200_interpolate(self.h, n, _d(stamps), _d(pose), _d(vel), _d(acc), C.byref(bad)))
        return pose, vel, acc, bad.value

    def ingest_stereo(self, stamp, cam0, cam1, px0, px1):
        """Stereo-track ingest (pixels -> bearings + triangulated world landmark at the current state)."""
        stamp, px0, px1 = _f64(stamp), _f64(px0), _f64(px1)
        cam0, cam1 = np.ascontiguousarray(cam0, dtype=np.int32), np.ascontiguousarray(cam1, dtype=np.int32)
        n = stamp.size
        b0, b1, lm = np.zeros((n, 3)), np.zeros((n, 3)), np.zeros((n, 3))
        bad = C.c_int(0)
        self._check(self.lib.hb200_ingest_stereo(self.h, n, _d(stamp), _i(cam0), _i(cam1), _d(px0), _d(px1), _d(b0), _d(b1), _d(lm), C.byref(bad)))
        return b0, b1, lm, bad.value

    def synchronize(self):
        self._check(self.lib.hb200_synchronize(self.h))

    def set_allreduce(self, fn):
        """fn(device_ptr: int, count: int, stream: int) -> int; kept alive by this object."""
        if fn is None:
            self._cb = None
            self._check(self.lib.hb200_set_allreduce(self.h, None, None))
            return
        self._cb = ALLREDUCE_FN(lambda user, ptr, count, stream: int(fn(ptr, count, stream) or 0))
        self._check(self.lib.hb200_set_allreduce(self.h, self._cb, None))

    # ---- multi-GPU: NCCL communicator owned by the library + peer-memory mailbox ------------------
    def comm_unique_id(self) -> bytes:
        buf = C.create_string_buffer(128)
        self._check(self.lib.hb200_comm_unique_id(buf))
        return buf.raw

    def comm_init_rank(self, nranks: int, rank: int, unique_id: bytes):
        self._check(self.lib.hb200_comm_init_rank(self.h, int(nranks), int(rank), C.c_char_p(unique_id)))

    def peer_handle(self) -> bytes:
        buf = C.create_string_buffer(64)
        self._check(self.lib.hb200_peer_handle(self.h, buf))
        return buf.raw

    def peer_connect(self, nranks: int, rank: int, handles: list):
        blob = b"".join(handles)
        assert len(blob) == 64 * nranks
        self._check(self.lib.hb200_peer_connect(self.h, int(nranks), int(rank), C.c_char_p(blob)))

    def measure_fp64_peak(self) -> float:
        v = C.c_double(0)
        self._check(self.lib.hb200_measure_fp64_peak(self.h, C.byref(v)))
        return v.value

    def bandwidth(self) -> int:
        b = C.c_int(0)
        self._check(self.lib.hb200_get_bandwidth(self.h, C.byref(b)))
        return b.value

    def set_min_bandwidth(self, beta: int):
        self._check(self.lib.hb200_set_min_bandwidth(self.h, int(beta)))

    def comm_info(self):
        v = [C.c_int(0) for _ in range(5)]
        pay = C.c_longlong(0)
        self._check(self.lib.hb200_comm_info(self.h, *[C.byref(x) for x in v], C.byref(pay)))
        return dict(nranks=v[0].value, rank=v[1].value, nccl=bool(v[2].value), peer_mailbox=bool(v[3].value), peer_reduce=(v[3].value == 2),
                    graph=bool(v[4].value), payload_doubles=pay.value)

    def connect_torch_distributed(self, dist, peer_mailbox=True, log=lambda m: None):
        """Plumbing only: ships the NCCL unique id and the mailbox handles over an initialised torch.distributed
        group; the communicator itself and every collective on the iteration path live inside the library."""
        world, rank = dist.get_world_size(), dist.get_rank()
        box = [self.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(box, src=0)
        log("unique id shipped")
        self.comm_init_rank(world, rank, box[0])
        log("communicator up")
        if peer_mailbox:
            handles = [None] * world
            dist.all_gather_object(handles, self.peer_handle())
            log("handles gathered")
            try:
                self.peer_connect(world, rank, handles)
                ok = 1
            except HB200Error:
                ok = 0
            flags = [None] * world
            dist.all_gather_object(flags, ok)
            if not all(flags):   # all ranks or none: the exchange is collective
                self._check(self.lib.hb200_peer_disconnect(self.h))
        return self.comm_info()

    def system_device_ptr(self):
        cnt = C.c_longlong(0)
        p = self.lib.hb200_system_device_ptr(self.h, C.byref(cnt))
        return p, cnt.value

    @property
    def stream(self):
        return self.lib.hb200_stream(self.h)

    @property
    def launch_count(self):
        return self.lib.hb200_launch_count(self.h)
