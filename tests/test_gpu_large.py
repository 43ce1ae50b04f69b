"""Parity at the FULL sizes of BASELINE.json configs 3-5 (indices 2, 3, 4 of `configs`):
  cfg2  order 6, 200 knots, 100 k pixel + 20 k IMU factors (n = 1 226)
  cfg3  4-camera rig, 500 knots, 500 k pixel factors       (n = 3 026)
  cfg4  1 M factors (833 k pixel + 167 k IMU), 500 knots    (n = 3 026)
Every factor's index map, residual and Jacobian, the full reduced system, the LM step and three LM iterations
are compared with the CPU oracle on the same seeded window (the reduced system block by block, tests/system_blocks.py)
-- the chunked (out-of-shared-memory) band solver is the default path at these sizes; cfg2 is repeated with the dense cooperative Cholesky.
"""
import numpy as np
import pytest

import oracle_lib as ol
import system_blocks as sb
from hyperslam_b200 import runtime, synthetic

pytestmark = pytest.mark.gpu


def rel_err(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / (np.abs(np.asarray(b)).max() + 1e-300))


def chunked_rel_err(a, b, rows=65536):
    """max |a - b| / max |b| without a full-size temporary (the 1 M-factor Jacobian arrays are hundreds of MB)."""
    worst, scale = 0.0, 0.0
    for lo in range(0, a.shape[0], rows):
        worst = max(worst, float(np.abs(a[lo:lo + rows] - b[lo:lo + rows]).max()))
        scale = max(scale, float(np.abs(b[lo:lo + rows]).max()))
    return worst / (scale + 1e-300)


@pytest.mark.parametrize("config,force_dense", [(2, False), (2, True), (3, False), (4, False)])
def test_full_size_config_parity(built, config, force_dense):
    win = synthetic.make_config(config, constant_knots=2)
    ow = ol.OracleWindow(win)
    assert ow.bad == 0
    ctx = runtime.Context(0, force_dense=force_dense)
    ctx.load_window(win)
    assert ctx.num_invalid == 0

    # a2 / a4: factor and knot indexing, bit-exact, every factor
    for got, want in zip(ctx.index_maps(), ow.index_maps()):
        assert np.array_equal(got, want)

    # a1 / a3 / a5 / a6: every residual and Jacobian block (north_star: 1e-6 / 1e-4 relative; held to 1e-9 / 1e-8)
    ref = ow.evaluate()
    ctx.evaluate()
    got = ctx.outputs()
    for key, tol in (("v_r", 1e-9), ("i_r", 1e-9), ("v_Jp", 1e-8), ("v_Jl", 1e-8), ("i_Jp", 1e-8), ("i_wg", 1e-12), ("i_wa", 1e-12), ("i_Jg", 1e-8)):
        if ref[key].shape[0]:
            assert chunked_rel_err(got[key], ref[key]) < tol, key
    del ref, got

    # a11: reduced system (landmark Schur complement applied, damped, constant dofs masked) and the LM step
    o = ow.iterate(apply=False)
    ctx.build_system()
    S, b = ctx.system()
    sb.assert_system_close(S, b, o["S"], o["b"], sb.DofLayout.of(win))
    ctx.solve()
    dp, dl = ctx.delta()
    res = np.abs(o["S"] @ dp - o["b"]).max() / (np.abs(o["b"]).max() + 1e-300)
    assert res < 1e-7, res
    assert rel_err(dp, o["delta_p"]) < 1e-5
    assert rel_err(dl, o["delta_l"]) < 1e-5
    del S, o

    # three LM iterations: costs, acceptance, trust region, final state
    recs = ctx.iterate(3)
    for it, rec in enumerate(recs):
        oo = ow.iterate(apply=True, outputs=False)["stats"]
        cost, cost_new, radius, accepted = oo[0], oo[1], oo[4], int(oo[5])
        assert rec["spd"] == 1
        assert abs(rec["cost"] - cost) <= 1e-7 * abs(cost), (it, rec, cost)
        assert abs(rec["cost_new"] - cost_new) <= 1e-6 * abs(cost_new), (it, rec, cost_new)
        assert rec["accepted"] == accepted, (it, rec)
        assert abs(rec["radius"] - radius) <= 1e-4 * radius
    st, so = ctx.state(), ow.state()
    for key in so:
        assert rel_err(st[key], so[key]) < 1e-6, key
    assert recs[-1]["cost"] < recs[0]["cost"]
    ctx.close()
