"""GPU-vs-oracle parity through the C-ABI (the parity tests proper; need a B200).

Tolerances follow BASELINE.json north_star: bit-exact factor/knot indexing, residuals within
1e-6 relative, Jacobians within 1e-4 relative (we assert far tighter: both paths are FP64).
"""
import numpy as np
import pytest

import oracle_lib as ol
import system_blocks as sb
from hyperslam_b200 import runtime, synthetic

pytestmark = pytest.mark.gpu

R_TOL = 1e-9   # residuals, relative to the largest residual magnitude of the list
J_TOL = 1e-8   # Jacobians, relative to the largest entry of the list


def rel_err(a, b):
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-300))


def make_ctx(win, **kw):
    ctx = runtime.Context(0, **kw)
    ctx.load_window(win)
    return ctx


SMALL = dict(num_knots=20, num_landmarks=120, num_imu=400)
CASES = {
    "k4": dict(order=4, **SMALL),
    "k6": dict(order=6, **SMALL),
    "k4_generic_calib": dict(order=4, generic_calibration=True, **SMALL),
    "k6_generic_calib": dict(order=6, generic_calibration=True, **SMALL),
    "k4_four_cams": dict(order=4, num_cameras=4, num_knots=20, num_landmarks=80, num_imu=100),
    "cfg0_plumbing": dict(order=4, num_knots=8, num_landmarks=0, num_imu=200),
    "pixel_only": dict(order=4, num_knots=20, num_landmarks=100, num_imu=0),
}


@pytest.mark.parametrize("name", list(CASES))
def test_evaluate_parity(built, name):
    win = synthetic.make_window(seed=synthetic.SEED_BASE + 100 + list(CASES).index(name), **CASES[name])
    ow = ol.OracleWindow(win)
    assert ow.bad == 0
    ref = ow.evaluate()
    ctx = make_ctx(win)
    # a2/a4: index maps bit-exact
    for got, exp in zip(ctx.index_maps(), ow.index_maps()):
        assert np.array_equal(got, exp)
    ctx.evaluate(jacobians=True)
    got = ctx.outputs()
    for key in ("v_r", "i_r"):
        if ref[key].size:
            assert rel_err(got[key], ref[key]) < R_TOL, key
    for key in ("v_Jp", "v_Jl", "i_Jp", "i_wg", "i_wa", "i_Jg"):
        if ref[key].size:
            assert rel_err(got[key], ref[key]) < J_TOL, key
    # cost-only path gives the same residuals
    ctx.evaluate(jacobians=False)
    assert abs(ctx.cost() - ow.cost()) <= 1e-10 * abs(ow.cost())
    ctx.close()


def test_unsorted_and_ragged_inputs(built):
    """Factors in arbitrary order, a landmark without observations, ragged track lengths."""
    win = synthetic.make_window(order=4, num_knots=16, num_landmarks=50, num_imu=77, seed=synthetic.SEED_BASE + 300)
    rng = np.random.default_rng(3)
    keep = rng.random(win.v_stamp.size) > 0.3           # ragged tracks
    keep &= win.v_lm != 7                               # landmark 7 loses all observations
    pv = rng.permutation(np.nonzero(keep)[0])
    pi = rng.permutation(win.i_stamp.size)
    win.v_stamp, win.v_cam, win.v_lm, win.v_pixel = (np.ascontiguousarray(a[pv]) for a in (win.v_stamp, win.v_cam, win.v_lm, win.v_pixel))
    win.i_stamp, win.i_meas = np.ascontiguousarray(win.i_stamp[pi]), np.ascontiguousarray(win.i_meas[pi])
    ow = ol.OracleWindow(win)
    ref = ow.evaluate()
    ctx = make_ctx(win)
    for got, exp in zip(ctx.index_maps(), ow.index_maps()):
        assert np.array_equal(got, exp)
    ctx.evaluate()
    got = ctx.outputs()
    for key in ref:
        assert rel_err(got[key], ref[key]) < J_TOL, key
    ctx.build_system()
    S, b = ctx.system()
    o = ow.iterate(apply=False)
    sb.assert_system_close(S, b, o["S"], o["b"], sb.DofLayout.of(win))
    ctx.close()


def test_edge_cases(built):
    win = synthetic.make_window(order=4, num_knots=12, num_landmarks=10, num_imu=10, seed=synthetic.SEED_BASE + 301)
    # stamp outside the valid span is reported, not silently clamped
    bad = synthetic.make_window(order=4, num_knots=12, num_landmarks=10, num_imu=10, seed=synthetic.SEED_BASE + 301)
    bad.i_stamp = bad.i_stamp.copy()
    bad.i_stamp[3] = bad.knots[-1, 7] + 1.0
    ctx = runtime.Context(0)
    with pytest.raises(runtime.HB200Error):
        ctx.load_window(bad)
    assert ctx.num_invalid == 1
    assert ol.OracleWindow(bad).bad == 1
    # stamp exactly on a knot belongs to the segment starting there (lower-inclusive range)
    win.i_stamp = win.i_stamp.copy()
    win.i_stamp[0] = win.knots[1, 7]
    win.i_stamp[1] = np.nextafter(win.knots[2, 7], -np.inf)
    ctx2 = make_ctx(win)
    ow = ol.OracleWindow(win)
    assert np.array_equal(ctx2.index_maps()[1], ow.index_maps()[1])
    assert ctx2.index_maps()[1][0] == 0 and ctx2.index_maps()[1][1] == 0
    # empty factor lists
    empty = synthetic.make_window(order=4, num_knots=12, num_landmarks=0, num_imu=5, seed=1)
    ctx3 = make_ctx(empty)
    ctx3.evaluate()
    assert ctx3.outputs()["v_r"].shape == (0, 2)
    ctx.close(); ctx2.close(); ctx3.close()


@pytest.mark.parametrize("force_dense", [False, True])
@pytest.mark.parametrize("name", ["k4", "k6", "k4_generic_calib", "cfg0_plumbing", "pixel_only"])
def test_system_and_step_parity(built, name, force_dense):
    kw = dict(CASES[name])
    win = synthetic.make_window(seed=synthetic.SEED_BASE + 200, constant_knots=2, **kw)
    ow = ol.OracleWindow(win)
    o = ow.iterate(apply=False)
    ctx = make_ctx(win, force_dense=force_dense)
    ctx.evaluate()
    ctx.build_system()
    S, b = ctx.system()
    sb.assert_system_close(S, b, o["S"], o["b"], sb.DofLayout.of(win))
    ctx.solve()
    dp, dl = ctx.delta()
    # the reduced system is ill-conditioned along gauge directions: compare through the residual
    # of the linear system and directly with a condition-aware tolerance
    res = np.abs(o["S"] @ dp - o["b"]).max() / (np.abs(o["b"]).max() + 1e-300)
    assert res < 1e-7, res
    assert rel_err(dp, o["delta_p"]) < 1e-5
    if dl.size:
        assert rel_err(dl, o["delta_l"]) < 1e-5
    ctx.close()


@pytest.mark.parametrize("use_graph,force_dense", [(True, False), (False, False), (True, True)])
def test_iterate_parity(built, use_graph, force_dense):
    win = synthetic.make_window(order=4, num_knots=20, num_landmarks=150, num_imu=400, seed=synthetic.SEED_BASE + 201, constant_knots=2)
    ow = ol.OracleWindow(win)
    ctx = make_ctx(win, use_graph=use_graph, force_dense=force_dense)
    recs = ctx.iterate(5)
    for it, rec in enumerate(recs):
        o = ow.iterate(apply=True)
        assert rec["spd"] == 1 and o["spd"] == 1
        assert abs(rec["cost"] - o["cost"]) <= 1e-7 * abs(o["cost"]), (it, rec, o["cost"])
        assert abs(rec["cost_new"] - o["cost_new"]) <= 1e-6 * abs(o["cost_new"]), (it, rec, o["cost_new"])
        assert rec["accepted"] == o["accepted"], (it, rec, o["rho"])
        assert abs(rec["radius"] - o["radius"]) <= 1e-4 * o["radius"]
    st, so = ctx.state(), ow.state()
    for key in so:
        assert rel_err(st[key], so[key]) < 1e-6, key
    assert recs[-1]["cost"] < recs[0]["cost"]
    ctx.close()


def test_factor_evaluate_ceres_shape(built):
    """hb200_factor_evaluate == oracle ExteroceptiveCost::Evaluate after manifold projection."""
    win = synthetic.make_window(order=4, num_knots=14, num_landmarks=20, num_imu=30, seed=synthetic.SEED_BASE + 202)
    ctx = make_ctx(win)
    ctx.evaluate()
    vb, ib, ig, ia = ctx.index_maps()
    k, kb = win.order, win.bias_order
    for f in (0, 7, win.v_stamp.size - 1):
        cam = win.cameras[win.v_cam[f]]
        blocks = [win.knots[vb[f] + m] for m in range(k)] + [cam[:7], cam[7:11], cam[11:15], win.landmarks[win.v_lm[f]]]
        r, jac = ctx.factor_evaluate(runtime.PIXEL, f, blocks)
        r_o, jac_o = ol.cost_evaluate(ol.PIXEL, win.v_stamp[f], win.v_pixel[f], np.concatenate(blocks), k=k)
        assert rel_err(r, r_o) < 1e-9
        for m in range(k):
            PJ = ol.manifold_plus_jacobian(ol.M_STATE, blocks[m])
            assert rel_err(jac[m] @ PJ, jac_o[m] @ PJ) < 1e-8
        assert rel_err(jac[k + 3], jac_o[k + 3]) < 1e-8
    for f in (0, 11, win.i_stamp.size - 1):
        imu = win.imu
        blocks = ([win.knots[ib[f] + m] for m in range(k)] + [imu[:7], imu[7:13], imu[13:19], imu[19:28], imu[28:37]]
                  + [win.gyro_bias[ig[f] + m] for m in range(kb)] + [win.accel_bias[ia[f] + m] for m in range(kb)] + [win.gravity])
        r, jac = ctx.factor_evaluate(runtime.INERTIAL, f, blocks)
        r_o, jac_o = ol.cost_evaluate(ol.INERTIAL, win.i_stamp[f], win.i_meas[f], np.concatenate(blocks), k=k)
        assert rel_err(r, r_o) < 1e-9
        for m in range(k):
            PJ = ol.manifold_plus_jacobian(ol.M_STATE, blocks[m])
            assert rel_err(jac[m] @ PJ, jac_o[m] @ PJ) < 1e-8
        for m in range(2 * kb):
            assert rel_err(jac[k + 5 + m], jac_o[k + 5 + m]) < 1e-10
        PJ = ol.manifold_plus_jacobian(ol.M_SPHERE, win.gravity)
        assert rel_err(jac[-1] @ PJ, jac_o[-1] @ PJ) < 1e-8
    ctx.close()


def test_full_size_properties(built):
    """BASELINE config 1 (50 knots, 10k pixel + 2k IMU) at full size: size-independent properties."""
    win = synthetic.make_config(1, constant_knots=2)
    ctx = make_ctx(win)
    ctx.evaluate()
    out = ctx.outputs()
    # (1) rigidly moving every control point by a global rotation-tangent leaves every residual's
    #     rotation Jacobian summing to the Jacobian of a global rotation: sum_m dtheta/dphi_m = I
    #     => translation blocks sum to -F (pixel) ; check partition of unity on translation weights
    k = win.order
    Jp = out["v_Jp"].reshape(-1, 2, k, 6)
    Jl = out["v_Jl"]
    assert np.abs(Jp[..., 3:].sum(axis=2) + Jl).max() < 1e-9 * np.abs(Jl).max()
    # (2) the sample the oracle can finish in seconds agrees
    ow = ol.OracleWindow(win)
    ref = ow.evaluate()
    for key in ref:
        assert rel_err(out[key], ref[key]) < J_TOL, key
    # (3) five LM iterations reduce the cost and stay SPD
    recs = ctx.iterate(5)
    assert all(r["spd"] == 1 for r in recs)
    assert recs[-1]["cost_new"] < 0.6 * recs[0]["cost"]
    ctx.close()


def test_gpu_matches_mpmath_golden(built):
    """CUDA path vs the 80-digit known-answer vectors (independent of the oracle)."""
    import glob
    import json
    import os
    from test_oracle import check_against_golden, window_from_golden
    paths = sorted(glob.glob(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "*.json")))
    assert len(paths) >= 6
    for path in paths:
        with open(path) as f:
            case = json.load(f)
        win = window_from_golden(case)
        ctx = make_ctx(win)
        ctx.evaluate()
        check_against_golden(case, ctx.outputs(), ctx.index_maps())
        ctx.close()


def test_interpolate_matches_oracle_state_evaluate(built):
    for order in (4, 6):
        win = synthetic.make_window(order=order, num_knots=14, num_landmarks=5, num_imu=5, seed=synthetic.SEED_BASE + 400)
        ctx = make_ctx(win)
        left = (order - 1) // 2
        t = np.linspace(win.knots[left, 7], win.knots[14 - order + left, 7], 57, endpoint=False)
        t = np.concatenate([t, [win.knots[-1, 7] + 5.0]])            # one stamp outside the span
        pose, vel, acc, bad = ctx.interpolate(t)
        assert bad == 1 and np.array_equal(pose[-1], [0, 0, 0, 1, 0, 0, 0])
        ow = ol.OracleWindow(win)
        for i in range(t.size - 1):
            j = int(np.searchsorted(win.knots[:, 7], t[i], side="right") - 1) - left
            v, ve, ac, _ = ol.state_evaluate(win.knots[j:j + order], t[i], 2, False)
            assert np.abs(pose[i] - v).max() < 1e-12
            assert np.abs(vel[i] - ve).max() < 1e-9 * max(1.0, np.abs(ve).max())
            assert np.abs(acc[i] - ac).max() < 1e-8 * max(1.0, np.abs(ac).max())
        ctx.close()


# ---- (f) rank 1: bearing + manifold (pose) factors --------------------------------------------------
def widened_window(order, seed_off=0, **kw):
    cfg = dict(order=order, num_knots=20, num_landmarks=120, num_imu=400, constant_knots=2)
    cfg.update(kw)
    base = synthetic.make_window(seed=synthetic.SEED_BASE + 300 + seed_off, **cfg)
    return synthetic.add_bearing_and_pose_factors(base, num_bearing=150, num_pose=40, seed=synthetic.SEED_BASE + 310 + seed_off)


@pytest.mark.parametrize("order", [4, 6])
def test_bearing_and_manifold_evaluate_parity(built, order):
    """VisualBearingEvaluator + AngularMetric and ManifoldEvaluator + ManifoldMetric (reference
    evaluators/bearing.cpp:14-79, manifold.cpp:12-61) against the oracle, next to the pixel / inertial lists."""
    win = widened_window(order)
    ow = ol.OracleWindow(win)
    assert ow.bad == 0
    ref = ow.evaluate()
    ctx = make_ctx(win)
    ctx.evaluate(jacobians=True)
    got = ctx.outputs()
    for key in ("v_r", "i_r", "b_r", "m_r"):
        assert rel_err(got[key], ref[key]) < R_TOL, key
    for key in ("v_Jp", "v_Jl", "i_Jp", "i_wg", "i_wa", "i_Jg", "b_Jp", "b_Jl", "m_Jp"):
        assert rel_err(got[key], ref[key]) < J_TOL, key
    ctx.evaluate(jacobians=False)
    assert abs(ctx.cost() - ow.cost()) <= 1e-10 * abs(ow.cost())
    ctx.close()


@pytest.mark.parametrize("force_dense", [False, True])
@pytest.mark.parametrize("order", [4, 6])
def test_bearing_and_manifold_system_parity(built, order, force_dense):
    win = widened_window(order, seed_off=1)
    ow = ol.OracleWindow(win)
    o = ow.iterate(apply=False)
    ctx = make_ctx(win, force_dense=force_dense)
    ctx.evaluate()
    ctx.build_system()
    S, b = ctx.system()
    sb.assert_system_close(S, b, o["S"], o["b"], sb.DofLayout.of(win))
    ctx.solve()
    dp, dl = ctx.delta()
    res = np.abs(o["S"] @ dp - o["b"]).max() / (np.abs(o["b"]).max() + 1e-300)
    assert res < 1e-7, res
    assert rel_err(dp, o["delta_p"]) < 1e-5
    assert rel_err(dl, o["delta_l"]) < 1e-5
    ctx.close()


@pytest.mark.parametrize("use_graph", [True, False])
def test_bearing_and_manifold_iterate_parity(built, use_graph):
    win = widened_window(4, seed_off=2)
    ow = ol.OracleWindow(win)
    ctx = make_ctx(win, use_graph=use_graph)
    recs = ctx.iterate(5)
    for it, rec in enumerate(recs):
        o = ow.iterate(apply=True)
        assert rec["spd"] == 1 and o["spd"] == 1
        assert abs(rec["cost"] - o["cost"]) <= 1e-7 * abs(o["cost"]), (it, rec, o["cost"])
        assert abs(rec["cost_new"] - o["cost_new"]) <= 1e-6 * abs(o["cost_new"]), (it, rec, o["cost_new"])
        assert rec["accepted"] == o["accepted"], (it, rec, o["rho"])
    st, so = ctx.state(), ow.state()
    for key in so:
        assert rel_err(st[key], so[key]) < 1e-6, key
    assert recs[-1]["cost"] < recs[0]["cost"]
    ctx.close()


def test_bearing_only_and_pose_only_windows(built):
    """Windows holding a single factor family: bearing-only (no pixel factors at all) and pose-only
    (no cameras, landmarks or IMU) bind, evaluate and solve."""
    base = synthetic.make_window(order=4, num_knots=16, num_landmarks=60, num_imu=0, seed=synthetic.SEED_BASE + 320, constant_knots=2)
    win = synthetic.add_bearing_and_pose_factors(base, num_bearing=base.v_stamp.size, num_pose=0)
    assert win.v_stamp.size == 0 and win.b_stamp.size == base.v_stamp.size
    ow = ol.OracleWindow(win)
    ctx = make_ctx(win)
    ctx.evaluate()
    got, ref = ctx.outputs(), ow.evaluate()
    assert rel_err(got["b_r"], ref["b_r"]) < R_TOL and rel_err(got["b_Jp"], ref["b_Jp"]) < J_TOL and rel_err(got["b_Jl"], ref["b_Jl"]) < J_TOL
    rec, o = ctx.iterate(1)[0], ow.iterate()
    assert abs(rec["cost"] - o["cost"]) <= 1e-8 * o["cost"] and abs(rec["cost_new"] - o["cost_new"]) <= 1e-6 * o["cost_new"]
    ctx.close()
    plain = synthetic.make_window(order=6, num_knots=16, num_landmarks=0, num_imu=0, seed=synthetic.SEED_BASE + 321)
    win = synthetic.add_bearing_and_pose_factors(plain, num_bearing=0, num_pose=64)
    ow = ol.OracleWindow(win)
    ctx = make_ctx(win)
    recs = ctx.iterate(3)
    for rec in recs:
        o = ow.iterate()
        assert abs(rec["cost"] - o["cost"]) <= 1e-7 * o["cost"] and rec["accepted"] == o["accepted"]
    assert recs[-1]["cost_new"] < 0.6 * recs[0]["cost"]
    ctx.close()


def test_bearing_and_manifold_factor_evaluate_ceres_shape(built):
    """hb200_factor_evaluate for kinds BEARING / MANIFOLD == oracle ExteroceptiveCost::Evaluate after the
    manifold projection (calibration blocks are constant in the live configuration: zero)."""
    win = widened_window(4, seed_off=3)
    ctx = make_ctx(win)
    ctx.evaluate()
    k = win.order
    left = (k - 1) // 2
    for f in (0, 17, win.b_stamp.size - 1):
        base = int(np.searchsorted(win.knots[:, 7], win.b_stamp[f], side="right") - 1 - left)
        cam = win.cameras[win.b_cam[f]]
        blocks = [win.knots[base + m] for m in range(k)] + [cam[:7], cam[7:11], cam[11:15], win.landmarks[win.b_lm[f]]]
        r, jac = ctx.factor_evaluate(runtime.BEARING, f, blocks)
        r_o, jac_o = ol.cost_evaluate(ol.BEARING, win.b_stamp[f], win.b_bearing[f], np.concatenate(blocks), k=k)
        assert r.shape == (1,) and abs(r[0] - r_o[0]) < 1e-12
        for m in range(k):
            PJ = ol.manifold_plus_jacobian(ol.M_STATE, blocks[m])
            assert rel_err(jac[m] @ PJ, jac_o[m] @ PJ) < 1e-8
        assert rel_err(jac[k + 3], jac_o[k + 3]) < 1e-8
    for f in (0, 9, win.m_stamp.size - 1):
        base = int(np.searchsorted(win.knots[:, 7], win.m_stamp[f], side="right") - 1 - left)
        blocks = [win.knots[base + m] for m in range(k)] + [win.pose_sensors[win.m_sensor[f]]]
        r, jac = ctx.factor_evaluate(runtime.MANIFOLD, f, blocks)
        r_o, jac_o = ol.cost_evaluate(ol.MANIFOLD, win.m_stamp[f], win.m_pose[f], np.concatenate(blocks), k=k)
        assert rel_err(r, r_o) < 1e-9
        for m in range(k):
            PJ = ol.manifold_plus_jacobian(ol.M_STATE, blocks[m])
            assert rel_err(jac[m] @ PJ, jac_o[m] @ PJ) < 1e-8
    ctx.close()


@pytest.mark.parametrize("order,knots", [(4, 140), (6, 96), (4, 64)])
def test_long_windows_band_solver_out_of_shared_memory(built, order, knots):
    """Windows whose band + arrow workspace exceeds shared memory (K = 140 / 96 / 64, beta 5 or 7, m 32 or 26): all
    three select the cyclic-reduction solver (bcr_solve_kernel).  Compared with the dense cooperative Cholesky on the
    same system and with the oracle's step; also through full LM iterations.  The chunked band solver and the other
    solver-selection edges are covered by tests/test_gpu_variants.py."""
    win = synthetic.make_window(order=order, num_knots=knots, num_landmarks=300, num_imu=600, seed=synthetic.SEED_BASE + 600 + knots,
                                constant_knots=2)
    ow = ol.OracleWindow(win)
    o = ow.iterate(apply=False)
    deltas = []
    for force_dense in (False, True):
        ctx = make_ctx(win, force_dense=force_dense)
        ctx.evaluate()
        ctx.build_system()
        ctx.solve()
        dp, dl = ctx.delta()
        res = np.abs(o["S"] @ dp - o["b"]).max() / (np.abs(o["b"]).max() + 1e-300)
        assert res < 1e-7, (force_dense, res)
        assert rel_err(dp, o["delta_p"]) < 1e-5
        assert rel_err(dl, o["delta_l"]) < 1e-5
        deltas.append(dp)
        ctx.close()
    assert rel_err(deltas[0], deltas[1]) < 1e-6
    ctx = make_ctx(win)
    recs = ctx.iterate(3)
    for rec in recs:
        oo = ow.iterate(apply=True)
        assert rec["spd"] == 1 and abs(rec["cost"] - oo["cost"]) <= 1e-7 * oo["cost"] and rec["accepted"] == oo["accepted"]
    ctx.close()
