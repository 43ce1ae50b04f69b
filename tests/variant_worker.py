"""Worker for tests/test_gpu_variants.py: one process per runtime-switch variant (the HB200_* switches are read once per
process).  For every window named on the command line it runs one LM iteration through the CUDA graph, copies the
packed reduced system the iteration assembled (hb200_system_device_ptr) and the step, runs three more iterations,
and profiles the launch sequence of one iteration on a fresh context.  Results go to <out>/<window>.npz; the test
makes every assertion.

    python variant_worker.py OUT_DIR WINDOW [WINDOW ...]
"""
import json
import os
import sys
import traceback

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from hyperslam_b200 import synthetic  # noqa: E402

S0 = synthetic.SEED_BASE + 900
SMALL = dict(num_knots=20, num_landmarks=120, num_imu=400)


def _mixed(order):
    return synthetic.make_window(order=order, seed=S0, constant_knots=2, **SMALL)


def _widened(order):
    base = synthetic.make_window(order=order, seed=S0 + 1, constant_knots=2, **SMALL)
    return synthetic.add_bearing_and_pose_factors(base, num_bearing=150, num_pose=40, seed=S0 + 2)


def _ragged():
    """Factors in arbitrary order, one landmark without observations, landmarks seen by a single pixel factor."""
    win = synthetic.make_window(order=4, num_knots=16, num_landmarks=50, num_imu=77, seed=S0 + 3, constant_knots=2)
    rng = np.random.default_rng(5)
    keep = rng.random(win.v_stamp.size) > 0.3
    keep &= win.v_lm != 7
    for lm in (11, 23, 31):                                   # exactly one observation left
        idx = np.nonzero(win.v_lm == lm)[0]
        keep[idx] = False
        keep[idx[1]] = True
    pv = rng.permutation(np.nonzero(keep)[0])
    pi = rng.permutation(win.i_stamp.size)
    win.v_stamp, win.v_cam, win.v_lm, win.v_pixel = (np.ascontiguousarray(a[pv]) for a in (win.v_stamp, win.v_cam, win.v_lm, win.v_pixel))
    win.i_stamp, win.i_meas = np.ascontiguousarray(win.i_stamp[pi]), np.ascontiguousarray(win.i_meas[pi])
    return win


def _track(order=4, num_knots=64, dt=0.025, span_dt=4.4, bias_knots=4, num_landmarks=200, seed=0):
    """Landmark tracks spanning `span_dt` knot intervals (not an integer: the longest track then spans ceil(span_dt) + 1
    knot bases, beta = ceil(span_dt) + order - 1) and `bias_knots` knots in each bias spline (m = 6 bias_knots + 2)."""
    F = 5
    t_valid = (num_knots - order + 1) * dt
    bias_dt = t_valid / (bias_knots - 3) * (1 - 1e-9)
    return synthetic.make_window(order=order, num_knots=num_knots, dt=dt, num_landmarks=num_landmarks, frames_per_landmark=F,
                                 frame_dt=span_dt * dt / (F - 1), num_imu=800, bias_dt=bias_dt, seed=S0 + 10 + seed, constant_knots=2)


def windows(num_sms):
    """name -> window builder.  Each window targets one edge of the kernels or of a size-selected path."""
    merge_pix = (1800 + 63) // 64       # 300 landmarks x 3 frames x 2 cameras
    merge_imu = 64 * (4 * num_sms - merge_pix)
    return {
        "k4": lambda: _mixed(4),
        "k6": lambda: _mixed(6),
        "wide_k4": lambda: _widened(4),
        "wide_k6": lambda: _widened(6),
        # ~1 pixel factor per knot: a 64-factor tile spans far more than 16 knot-table rows; Nv % 64 == 1
        "sparse_pixels": lambda: synthetic.make_window(order=4, num_knots=120, num_landmarks=43, frames_per_landmark=3, num_cameras=1,
                                                       num_imu=2000, seed=S0 + 4, constant_knots=2),
        # inertial factors only: the inertial J^T J is the whole system; bias knots every 0.37 s against knots every 0.1 s
        # cut the per-segment runs into ragged lengths (1 .. 13)
        "inertial_only": lambda: synthetic.make_window(order=4, num_knots=30, num_landmarks=0, num_imu=351, bias_dt=0.37,
                                                       seed=S0 + 5, constant_knots=2),
        "ragged": _ragged,
        # solver selection (band workspace vs 220 KB of shared memory; bcr needs 6 beta <= 48 and m <= 54)
        "smem_in": lambda: _track(num_knots=57, span_dt=1.5, seed=1),          # beta 5, m 26: 219 KB, in shared memory
        "smem_out": lambda: _track(num_knots=58, span_dt=1.5, seed=2),         # beta 5, m 26: 222 KB, bcr
        "beta8": lambda: _track(span_dt=4.4, seed=3),                          # 6 beta = 48: bcr
        "beta9": lambda: _track(span_dt=5.4, seed=4),                          # 6 beta = 54: chunked band solver
        "arrow50": lambda: _track(span_dt=1.5, bias_knots=8, seed=5),          # m = 50: bcr
        "arrow56": lambda: _track(span_dt=1.5, bias_knots=9, seed=6),          # m = 56: chunked band solver
        "beta16": lambda: _track(num_knots=40, span_dt=12.4, seed=7),          # beta 16: no band plan fits, dense
        # size thresholds that need no switch
        "imu_16383": lambda: synthetic.make_window(order=4, num_knots=40, num_landmarks=0, num_imu=16383, seed=S0 + 20, constant_knots=2),
        "imu_16384": lambda: synthetic.make_window(order=4, num_knots=40, num_landmarks=0, num_imu=16384, seed=S0 + 20, constant_knots=2),
        "lm_8191": lambda: synthetic.make_window(order=4, num_knots=40, num_landmarks=8191, frames_per_landmark=1, num_imu=400,
                                                 seed=S0 + 21, constant_knots=2),
        "lm_8192": lambda: synthetic.make_window(order=4, num_knots=40, num_landmarks=8192, frames_per_landmark=1, num_imu=400,
                                                 seed=S0 + 21, constant_knots=2),
        # 4 x SMs CTAs of 64 factors: one merged launch up to there, separate launches above
        "merge_at": lambda: synthetic.make_window(order=4, num_knots=40, num_landmarks=300, frames_per_landmark=3, num_imu=merge_imu,
                                                  seed=S0 + 22, constant_knots=2),
        "merge_over": lambda: synthetic.make_window(order=4, num_knots=40, num_landmarks=300, frames_per_landmark=3, num_imu=merge_imu + 1,
                                                    seed=S0 + 22, constant_knots=2),
    }


def run_window(win, out_path):
    import torch
    from hyperslam_b200 import runtime
    res = {}
    ctx = runtime.Context(0, use_graph=True)
    ctx.load_window(win)
    res["beta"] = ctx.bandwidth()
    recs = ctx.iterate(1)
    ctx.synchronize()
    ptr, count = ctx.system_device_ptr()

    class _Arr:
        __cuda_array_interface__ = dict(shape=(count,), typestr="<f8", data=(ptr, False), version=2)

    res["sys"] = torch.as_tensor(_Arr(), device="cuda").cpu().numpy().copy()
    res["dp"], res["dl"] = ctx.delta()
    recs += ctx.iterate(3)
    for key, val in ctx.state().items():
        res["state_" + key] = val
    res["recs"] = np.array([[r["cost"], r["cost_new"], r["radius"], r["accepted"], r["spd"]] for r in recs])
    ctx.close()
    ctx = runtime.Context(0, use_graph=True)
    ctx.load_window(win)
    labels = sorted({name for name, _ in ctx.profile_iteration(reps=1)})
    ctx.close()
    np.savez(out_path, labels=json.dumps(labels), **res)


def main():
    out, names = sys.argv[1], sys.argv[2:]
    import torch
    num_sms = torch.cuda.get_device_properties(0).multi_processor_count
    wins = windows(num_sms)
    status = {"num_sms": num_sms}
    for name in names:
        try:
            run_window(wins[name](), os.path.join(out, name + ".npz"))
            status[name] = "ok"
        except Exception:  # noqa: BLE001  (reported per window by the test)
            status[name] = traceback.format_exc()[-3000:]
    with open(os.path.join(out, "status.json"), "w") as f:
        json.dump(status, f)


if __name__ == "__main__":
    main()
