"""CPU checks of tests/system_blocks.py (the block-wise reduced-system comparison) and of the windows the GPU variant
tests run on (tests/variant_worker.py), with the oracle alone."""
import numpy as np
import pytest

import oracle_lib as ol
import system_blocks as sb
import variant_worker as vw
from hyperslam_b200 import synthetic


@pytest.fixture(scope="module")
def k4_system():
    """The k4 window of test_system_and_step_parity, its oracle packed system."""
    win = synthetic.make_window(order=4, num_knots=20, num_landmarks=120, num_imu=400, seed=synthetic.SEED_BASE + 200, constant_knots=2)
    ow = ol.OracleWindow(win)
    return sb.DofLayout.of(win), sb.oracle_packed(ow.build_packed(), ow.n)


def block_family(lay, a, b):
    ka, kb = lay.kind_of_dof == sb.KINDS.index(a), lay.kind_of_dof == sb.KINDS.index(b)
    return np.outer(ka, kb) | np.outer(kb, ka)


def test_every_block_perturbed_by_1e7_is_flagged(k4_system):
    lay, ref = k4_system
    S = ref["S"]
    assert not sb.packed_mismatches(ref, ref, lay)
    nb = lay.starts.size
    ends = np.append(lay.starts[1:], lay.n)
    for i in range(nb):
        for j in range(i + 1):
            r, c = slice(lay.starts[i], ends[i]), slice(lay.starts[j], ends[j])
            P = S.copy()
            if np.any(P[r, c] != 0):
                P[r, c] *= 1 + 1e-7
            else:
                P[lay.starts[i], lay.starts[j]] = 1e-30
            P[c, r] = P[r, c].T
            found = sb.matrix_mismatches(P, S, lay)
            assert any(f"S[{lay.name(i)}, {lay.name(j)}]" in f for f in found), (lay.name(i), lay.name(j))


@pytest.mark.parametrize("a,b", [("gyro_bias", "pose"), ("accel_bias", "pose"), ("gyro_bias", "gyro_bias"), ("accel_bias", "accel_bias")])
def test_global_tolerance_misses_bias_blocks(k4_system, a, b):
    """max |S_block| / max |S| of the bias blocks is 1e-9 .. 2e-8 here: a 1e-7 relative error in a whole family passes
    rel_err(S) < 1e-9; the block-wise helper flags it."""
    lay, ref = k4_system
    S = ref["S"]
    P = np.where(block_family(lay, a, b), S * (1 + 1e-7), S)
    assert sb.rel_err(P, S) < 1e-9
    assert sb.matrix_mismatches(P, S, lay)


def test_scaled_gyro_bias_pose_block_passes_global_check(k4_system):
    """The gyro-bias x pose family scaled by 1.3 still passes the global check (6.5e-10); the helper does not."""
    lay, ref = k4_system
    S = ref["S"]
    P = np.where(block_family(lay, "gyro_bias", "pose"), 1.3 * S, S)
    assert sb.rel_err(P, S) < 1e-9
    assert len(sb.matrix_mismatches(P, S, lay)) > 10


@pytest.mark.parametrize("key", ["b", "diagH", "g"])
def test_vector_families_flagged(k4_system, key):
    lay, ref = k4_system
    v = ref[key]
    for k, kind in enumerate(sb.KINDS):
        sel = lay.kind_of_dof == k
        if not np.any(v[sel]):
            continue
        w = v.copy()
        w[sel] *= 1 + 1e-7
        assert any(f"{key}[{kind}]" in f for f in sb.vector_mismatches(w, v, lay, key)), kind
    gyro = lay.kind_of_dof == 1
    w = v.copy()
    w[gyro] *= 1 + 1e-7
    if key == "b":
        assert sb.rel_err(w, v) < 1e-9     # the gyro-bias rows of b sit ~1e-8 below max |b|


def encode_device(S, b_schur, diagH, g, cost, K, beta, m):
    """The device's packed layout (hb200_types.cuh sys_index) written from a dense system."""
    L = sb.sys_layout(K, beta, m)
    buf = np.full(L["total"], np.nan)
    np_, h = L["np"], L["h"]
    for row in range(L["n"]):
        for col in range(row + 1):
            if row < np_:
                c = col // 6
                if row - 6 * c >= h:
                    continue
                buf[(c * h + row - 6 * c) * 6 + col - 6 * c] = S[row, col]
            elif col < np_:
                buf[L["oA"] + (row - np_) * np_ + col] = S[row, col]
            else:
                buf[L["oC"] + (row - np_) * m + col - np_] = S[row, col]
    for off, v in ((L["ob"], b_schur), (L["oD"], diagH), (L["og"], g)):
        buf[off: off + L["n"]] = v
    buf[L["os"]] = cost
    return np.nan_to_num(buf, nan=7.0)   # padding and unused slots hold garbage the decoder must ignore


def test_device_layout_decoder_round_trip(k4_system):
    lay, ref = k4_system
    K, m = lay.K, lay.n - 6 * lay.K
    S = ref["S"]
    pose = np.arange(lay.n) < 6 * K
    dist = np.abs(np.subtract.outer(np.arange(lay.n) // 6, np.arange(lay.n) // 6))
    beta = int(dist[np.outer(pose, pose) & (S != 0)].max())   # the block half-bandwidth the device would choose
    assert beta >= 3
    buf = encode_device(S, ref["b"] + ref["g"], ref["diagH"], ref["g"], ref["cost"], K, beta, m)
    dev = sb.device_packed(buf, K, beta, m)
    assert np.array_equal(dev["S"], np.tril(S) + np.tril(S, -1).T)    # the device keeps the lower triangle
    assert np.array_equal(dev["diagH"], ref["diagH"]) and np.array_equal(dev["g"], ref["g"]) and dev["cost"] == ref["cost"]
    assert not sb.packed_mismatches(dev, ref, lay)


def run_lengths(ib, ig, ia):
    key = np.stack([ib, ig, ia], 1)[np.lexsort((ia, ig, ib))]
    cut = np.nonzero(np.any(np.diff(key, axis=0) != 0, axis=1))[0] + 1
    return np.diff(np.concatenate([[0], cut, [key.shape[0]]]))


def test_variant_windows_hit_their_edges():
    """The windows of tests/test_gpu_variants.py have the shapes their comments claim (B200: 148 SMs)."""
    W = vw.windows(148)

    def maps(name):
        win = W[name]()
        return win, ol.OracleWindow(win).index_maps()

    def beta(win, vb):
        spans = [vb[win.v_lm == l].max() - vb[win.v_lm == l].min() for l in np.unique(win.v_lm)]
        return max(spans) + win.order - 1

    for name, want in (("smem_in", 5), ("smem_out", 5), ("beta8", 8), ("beta9", 9), ("arrow50", 5), ("arrow56", 5), ("beta16", 16)):
        win, (vb, *_) = maps(name)
        assert beta(win, vb) == want, name
    for name, m in (("arrow50", 50), ("arrow56", 56), ("beta8", 26)):
        assert 6 * W[name]().gyro_bias.shape[0] + 2 == m, name
    assert [W[n]().knots.shape[0] for n in ("smem_in", "smem_out")] == [57, 58]

    # sparse pixels: Nv % 64 == 1 and 64-factor tiles (bound order = sorted knot base) spanning > 16 table rows
    win, (vb, *_) = maps("sparse_pixels")
    assert vb.size % 64 == 1
    vs = np.sort(vb)
    assert max(t.max() + win.order - t.min() for t in np.split(vs, np.arange(64, vs.size, 64))) > 16

    # inertial only: runs of equal (knot, gyro, accel) base of ragged lengths, including 1, not multiples of 8 / 12 / 16
    win, (_, ib, ig, ia) = maps("inertial_only")
    assert win.v_stamp.size == 0 and win.landmarks.shape[0] == 0
    lengths = run_lengths(ib, ig, ia)
    hist = np.bincount(lengths)
    assert hist[1] > 0 and np.count_nonzero(hist) >= 8 and np.any(lengths % 4)

    # ragged: a landmark without observations, landmarks with one
    win = W["ragged"]()
    counts = np.bincount(win.v_lm, minlength=win.landmarks.shape[0])
    assert counts[7] == 0 and np.count_nonzero(counts == 1) >= 3
    assert not np.all(np.diff(win.v_stamp) >= 0)

    # size thresholds
    assert [W[n]().i_stamp.size for n in ("imu_16383", "imu_16384")] == [16383, 16384]
    assert [W[n]().landmarks.shape[0] for n in ("lm_8191", "lm_8192")] == [8191, 8192]
    blocks = [(W[n]().v_stamp.size + 63) // 64 + (W[n]().i_stamp.size + 63) // 64 for n in ("merge_at", "merge_over")]
    assert blocks == [4 * 148, 4 * 148 + 1]
