"""The iteration's own normal equations, for every kernel variant, against the oracle block by block.

`hb200_iterate` fuses the pixel J^T J into the factor kernels and picks the inertial J^T J kernel, the Schur kernel and
the solver by window size; the HB200_* runtime switches (DESIGN.md section 6.1) force the other choices.  Each switch is
read once per process, so every variant runs in its own worker process (tests/variant_worker.py) over the windows
where it changes something.  For each window the test checks:
  * the packed system the iteration assembled (undamped S after the landmark Schur complement, b, diag(J^T J), g,
    cost) against OracleWindow.build_packed(), per block at 1e-9 of the block's own max, exact zeros kept;
  * the same system against the default variant's, per block at 1e-12 (only the order of the atomics differs);
  * the step against the oracle's (linear-system residual 1e-7, delta_p / delta_l 1e-5);
  * four LM records and the final state against the oracle (as test_iterate_parity);
  * that the launches the variant exists for actually ran (hb200_profile_iteration labels).
The device assembles every dof, constant ones included (the solvers mask them), so no row is skipped here.
"""
import functools
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_lib as ol
import system_blocks as sb
import variant_worker as vw

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

MERGED, PIX, IMU = "factor_eval_kernel", "pixel_eval_kernel", "inertial_eval_kernel"
IMU_H, IMU_MMA, PIX_H = "inertial_hessian_kernel", "inertial_hessian_mma_kernel", "pixel_hessian_kernel"
SCHUR, SCHUR_G = "schur_kernel", "schur_group_kernel"
BAND, CHUNKED, BCR, DENSE = "band_solve_kernel", "band_solve_kernel<chunked>", "bcr_solve_kernel", "cholesky_kernel"
SOLVERS = {BAND, CHUNKED, BCR, DENSE}

# window -> (launches of the default iteration, launches it must not contain, block half-bandwidth or None)
WINDOWS = {
    "k4": ({MERGED, IMU_H, SCHUR, BAND}, {PIX, PIX_H}, 5),
    "k6": ({MERGED, IMU_H, SCHUR, BAND}, {PIX, PIX_H}, 7),
    "wide_k4": ({MERGED, IMU_H, SCHUR, BAND, "manifold_hessian_kernel"}, {PIX}, None),
    "wide_k6": ({MERGED, IMU_H, SCHUR, BAND, "manifold_hessian_kernel"}, {PIX}, None),
    "sparse_pixels": ({MERGED, IMU_H, SCHUR, BCR}, {PIX}, 4),
    "inertial_only": ({IMU, IMU_H, BAND}, {SCHUR, MERGED, PIX}, 3),
    "ragged": ({MERGED, IMU_H, SCHUR, BAND}, {PIX}, 5),
    "smem_in": ({BAND}, SOLVERS - {BAND}, 5),
    "smem_out": ({BCR}, SOLVERS - {BCR}, 5),
    "beta8": ({BCR}, SOLVERS - {BCR}, 8),
    "beta9": ({CHUNKED}, SOLVERS - {CHUNKED}, 9),
    "arrow50": ({BCR}, SOLVERS - {BCR}, 5),
    "arrow56": ({CHUNKED}, SOLVERS - {CHUNKED}, 5),
    "beta16": ({DENSE}, SOLVERS - {DENSE}, 16),
    "imu_16383": ({IMU_H}, {IMU_MMA}, 3),
    "imu_16384": ({IMU_MMA}, {IMU_H}, 3),
    "lm_8191": ({SCHUR}, {SCHUR_G}, None),
    "lm_8192": ({SCHUR_G}, {SCHUR}, None),
    "merge_at": ({MERGED, IMU_MMA}, {PIX, IMU}, None),
    "merge_over": ({PIX, IMU, IMU_MMA}, {MERGED}, None),
}

# variant -> (environment, windows, launches that must run, launches that must not)
VARIANTS = {
    "default": ({}, list(WINDOWS), set(), set()),
    "no_merge": ({"HB200_NO_MERGE": "1"}, ["k4", "k6", "wide_k4", "sparse_pixels", "ragged"], {PIX, IMU}, {MERGED}),
    "unfused": ({"HB200_FUSE": "0"}, ["k4", "k6", "wide_k6", "sparse_pixels", "ragged", "merge_over"], {PIX_H}, set()),
    "pix_tiles3": ({"HB200_NO_MERGE": "1", "HB200_PIX_TILES": "3"}, ["k4", "k6", "sparse_pixels", "ragged", "merge_over"], {PIX}, {MERGED, PIX_H}),
    "imu_mma": ({"HB200_IMU_HESS": "1"}, ["k4", "k6", "wide_k4", "inertial_only"], {IMU_MMA}, {IMU_H}),
    "imu_mma16": ({"HB200_IMU_HESS": "1", "HB200_IMU_CH": "16"}, ["k4", "inertial_only", "imu_16383"], {IMU_MMA}, {IMU_H}),
    "imu_scalar": ({"HB200_IMU_HESS": "0"}, ["imu_16384", "merge_at"], {IMU_H}, {IMU_MMA}),
    "schur_group": ({"HB200_SCHUR_GROUP_MIN": "1"}, ["k4", "k6", "wide_k4", "ragged", "sparse_pixels", "beta9"], {SCHUR_G}, {SCHUR}),
    "no_bcr": ({"HB200_NO_BCR": "1"}, ["smem_out", "beta8", "arrow50", "sparse_pixels"], {CHUNKED}, {BCR}),
    "no_fork": ({"HB200_NO_FORK": "1"}, ["k4", "wide_k4", "merge_over"], set(), set()),
    "pdl": ({"HB200_PDL": "1"}, ["k4", "k6", "wide_k4", "merge_at"], set(), set()),
    "imu_min_chunk": ({"HB200_IMU_MIN_CHUNK": "1", "HB200_IMU_CTAS_PER_SM": "1"}, ["k4", "inertial_only", "imu_16384"], set(), set()),
}
CASES = [(v, w) for v, (_, wins, _, _) in VARIANTS.items() for w in wins]

# looser per-block bounds, measured on a B200:
# 8 k single-frame stereo landmarks: each 3x3 V_l is nearly singular along the viewing ray (one stereo pair) and the
# Schur complement removes most of the diagonal pose blocks; measured 1.27e-9 of the block's max
WINDOW_TOLS = {"lm_8191": {("pose", "pose"): 3e-9}, "lm_8192": {("pose", "pose"): 3e-9}}
# against the default variant: the grouped Schur kernel sums W V^-1 W^T in another grouping than schur_kernel; where
# the Schur term cancels most of H (pose blocks on and next to the diagonal) measured up to 2.2e-11 of the block's
# max (sparse_pixels; 3.2e-12 on the mixed windows) and 1.8e-12 of max |b| in the pose rows of b
VARIANT_TOLS = {"schur_group": ({("pose", "pose"): 1e-10}, 1e-11)}

_runs = {}


def worker_run(variant, tmp_root):
    """Run the worker once per variant; returns (status dict, output dir)."""
    if variant not in _runs:
        env_add, wins, _, _ = VARIANTS[variant]
        out = tmp_root / variant
        out.mkdir()
        env = {k: v for k, v in os.environ.items() if not k.startswith("HB200_")}
        env.update(env_add)
        res = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "variant_worker.py"), str(out)] + wins, env=env,
                             capture_output=True, text=True, timeout=900)
        status_path = out / "status.json"
        assert res.returncode == 0 and status_path.exists(), res.stdout[-3000:] + res.stderr[-3000:]
        with open(status_path) as f:
            _runs[variant] = (json.load(f), out)
    return _runs[variant]


@functools.lru_cache(maxsize=None)
def oracle_run(window, num_sms):
    win = vw.windows(num_sms)[window]()
    ow = ol.OracleWindow(win)
    assert ow.bad == 0
    packed = sb.oracle_packed(ow.build_packed(), ow.n)
    first = ow.iterate(apply=True)
    stats = [first["stats"]] + [ow.iterate(apply=True, outputs=False)["stats"] for _ in range(3)]
    return win, packed, first, np.array(stats), ow.state()


def load(variant, window, tmp_root):
    status, out = worker_run(variant, tmp_root)
    assert status[window] == "ok", status[window]
    r = np.load(out / f"{window}.npz")
    return {k: r[k] for k in r.files}, status["num_sms"]


@pytest.fixture(scope="module")
def tmp_root(tmp_path_factory):
    return tmp_path_factory.mktemp("variants")


@pytest.mark.parametrize("variant,window", CASES)
def test_variant_system_step_and_iterations(built, tmp_root, variant, window):
    got, num_sms = load(variant, window, tmp_root)
    win, ref, o, stats, state = oracle_run(window, num_sms)
    lay = sb.DofLayout.of(win)
    K, m = lay.K, lay.n - 6 * lay.K
    beta = int(got["beta"])
    if WINDOWS[window][2] is not None:
        assert beta == WINDOWS[window][2]

    # the launches this variant and this window exist for
    labels = set(json.loads(str(got["labels"])))
    must, never = set(WINDOWS[window][0]) if variant == "default" else set(), set(WINDOWS[window][1]) if variant == "default" else set()
    must |= VARIANTS[variant][2]
    never |= VARIANTS[variant][3]
    assert must <= labels and not (never & labels), (sorted(must - labels), sorted(never & labels), sorted(labels))

    # the iteration's own packed system
    dev = sb.device_packed(got["sys"], K, beta, m)
    found = sb.packed_mismatches(dev, ref, lay, tols=WINDOW_TOLS.get(window))
    assert not found, "\n".join(found)
    if variant != "default":
        base, _ = load("default", window, tmp_root)
        found = sb.packed_mismatches(dev, sb.device_packed(base["sys"], K, int(base["beta"]), m), lay, tol=1e-12, cost_tol=1e-13,
                                     tols=VARIANT_TOLS.get(variant, (None, None))[0], vec_tol=VARIANT_TOLS.get(variant, (None, None))[1],
                                     zeros=ref["S"] == 0)
        assert not found, "vs the default variant:\n" + "\n".join(found)

    # the step solved from it
    dp, dl = got["dp"], got["dl"]
    res = np.abs(o["S"] @ dp - o["b"]).max() / (np.abs(o["b"]).max() + 1e-300)
    assert res < 1e-7, res
    assert sb.rel_err(dp, o["delta_p"]) < 1e-5
    if dl.size:
        assert sb.rel_err(dl, o["delta_l"]) < 1e-5

    # records of four iterations and the final state
    for it, (rec, s) in enumerate(zip(got["recs"], stats)):
        cost, cost_new, radius, accepted, spd = rec
        assert spd == 1 and s[6] == 1, it
        assert abs(cost - s[0]) <= 1e-7 * abs(s[0]), (it, cost, s[0])
        assert abs(cost_new - s[1]) <= 1e-6 * abs(s[1]), (it, cost_new, s[1])
        assert int(accepted) == int(s[5]), (it, s[3])
        assert abs(radius - s[4]) <= 1e-4 * s[4], (it, radius, s[4])
    for key in state:
        if state[key].size:
            assert sb.rel_err(got["state_" + key], state[key]) < 1e-6, key
