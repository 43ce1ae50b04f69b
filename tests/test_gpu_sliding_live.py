"""Device-side sliding window on the factor set the reference builds live: stereo tracks become two bearing factors
(reference abstract.cpp:243-260, optimizer.cpp:189-210), pose measurements become pose priors (abstract.cpp:266-270),
inertial factors as before.  A 20-frame sequence per spline order runs through hb200_append_knots ->
hb200_append_stereo_tracks -> hb200_append_inertial_factors -> hb200_append_manifold_factors -> hb200_slide and is
checked every frame against

  * a host restatement of the window rules (LiveWindow below: sizes, landmark slots, bit-exact state copies),
  * a twin context rebuilt from the restated lists with hb200_set_* + hb200_bind (bitwise factor outputs, index maps,
    the iteration's packed system per block to 1e-12),
  * the oracle (new landmarks, the cost at the linearisation point).

What these windows do not support is a comparison of the LM step or of the assembled system with the oracle at the
tolerances of tests/test_gpu_sliding.py: the newest landmarks are seen from one stereo pair only, so the reduced system
is ill-conditioned.  Measured on a B200: the iteration's pose blocks deviate from the oracle's by up to 2.4e-7 of the
block's max, trial costs differ by 17-80 % on some frames, and even the twin, whose system agrees to 1e-12, can reject
a step the device-managed context accepts.  The step-level oracle checks of the bookkeeping stay with the
better-conditioned pixel sequence of tests/test_gpu_sliding.py.

The sequence generator, the restatement and the per-frame oracle windows also run without a device
(test_live_sequence_rehearsal_on_the_oracle).
"""
import dataclasses
import re

import numpy as np
import pytest

import oracle_lib as ol
import system_blocks as sb
from hyperslam_b200 import runtime, synthetic

FRAMES = 20
K0 = 14
WIDTH = 9            # state elements behind the newest one that stay variable
TRACK_LEN = 5        # frames a landmark is observed in
NEW_PER_FRAME = 12   # landmarks first seen per frame (~60 tracks per frame once the pipeline is full)
PIXEL_SIGMA = 0.4
POSE_EVERY = 3       # pose priors arrive on every third frame
DROP_INERTIAL, DROP_POSE = runtime.SLIDE_DROP_INERTIAL, runtime.SLIDE_DROP_POSE
# a full hb200_bind orders the visual list differently (a segment's pixel factors ahead of its bearing factors), so the
# per-landmark sums run in another order; with near-singular landmark blocks S reaches 1e16 and the reassociation shows
# at up to 1.5e-10 of a block's max (measured on a B200)
REBIND_TOL = 1e-9


def rel_err(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / (np.abs(np.asarray(b)).max() + 1e-300))


# ---- the sequence ------------------------------------------------------------------------------------------------
class LiveSequence:
    """One state element per frame; per frame the stereo tracks of the landmarks first seen in the last TRACK_LEN frames
    (pixels of the ground truth + PIXEL_SIGMA noise), the IMU samples and (every POSE_EVERY frames) the pose priors
    that fall into the newly valid spline segment."""

    def __init__(self, order, frames=FRAMES, seed=synthetic.SEED_BASE + 4321):
        k, left = order, (order - 1) // 2
        K = K0 + frames + 2
        nseg = K - k + 1
        full = synthetic.make_window(order=k, num_knots=K, num_landmarks=0, num_imu=15 * nseg, seed=seed + order)
        self.full = synthetic.add_bearing_and_pose_factors(full, num_pose=2 * nseg, seed=seed + order + 1)
        self.order, self.frames, self.seed = k, frames, seed + order
        kt = self.full.knots[:, 7]
        ends = [kt[K0 - 1 - (k - 1 - left)]] + [kt[K0 + f - (k - 1 - left)] for f in range(frames)]
        t_pred = np.array([0.5 * (ends[f] + ends[f + 1]) for f in range(frames)])
        truth, cams = self.full.truth, self.full.cameras
        rng = np.random.Generator(np.random.Philox(self.seed + 2))
        first, xyz = [], []
        for f in range(frames):
            seen = t_pred[f:f + TRACK_LEN]
            got = 0
            while got < NEW_PER_FRAME:
                n = 64
                px = np.stack([rng.uniform(200, synthetic.IMAGE_SIZE[0] - 200, n), rng.uniform(150, synthetic.IMAGE_SIZE[1] - 150, n)], -1)
                depth = rng.uniform(2.0, 8.0, n)
                R, p, *_ = synthetic.spline_eval(truth["knots"], k, np.full(n, t_pred[f]))
                c0 = cams[0]
                ray = np.stack([(px[:, 0] - c0[7]) / c0[9], (px[:, 1] - c0[8]) / c0[10], np.ones(n)], -1) * depth[:, None]
                p_b = ray @ synthetic.quat_to_rot(c0[None, :4])[0].T + c0[4:7]
                lm = (R @ p_b[..., None])[..., 0] + p
                ok = np.ones(n, dtype=bool)
                for t in seen:
                    for c in range(2):
                        pix, p_s = synthetic.pixel_model(truth["knots"], k, cams, lm, np.full(n, t), np.full(n, c), np.arange(n))
                        ok &= (p_s[:, 2] > 0.5) & (pix[:, 0] > 10) & (pix[:, 0] < synthetic.IMAGE_SIZE[0] - 10)
                        ok &= (pix[:, 1] > 10) & (pix[:, 1] < synthetic.IMAGE_SIZE[1] - 10)
                take = lm[ok][: NEW_PER_FRAME - got]
                xyz.append(take); first += [f] * take.shape[0]
                got += take.shape[0]
        self.lm_first, self.lm_truth = np.array(first), np.concatenate(xyz)

    def tracks(self, f, t):
        """(global landmark ids, pixel0, pixel1) of frame f observed at stamp t."""
        gids = np.nonzero((self.lm_first <= f) & (f < self.lm_first + TRACK_LEN))[0]
        n = gids.size
        truth, cams = self.full.truth, self.full.cameras
        px0, _ = synthetic.pixel_model(truth["knots"], self.order, cams, self.lm_truth, np.full(n, t), np.zeros(n, dtype=int), gids)
        px1, _ = synthetic.pixel_model(truth["knots"], self.order, cams, self.lm_truth, np.full(n, t), np.ones(n, dtype=int), gids)
        rng = np.random.Generator(np.random.Philox(self.seed + 1000 + f))
        return gids, px0 + rng.normal(0, PIXEL_SIGMA, px0.shape), px1 + rng.normal(0, PIXEL_SIGMA, px1.shape)

    def inertial(self, lo, hi):
        f = self.full
        m = (f.i_stamp >= lo) & (f.i_stamp < hi)
        return f.i_stamp[m], f.i_meas[m]

    def poses(self, lo, hi):
        f = self.full
        m = (f.m_stamp >= lo) & (f.m_stamp < hi)
        return f.m_stamp[m], f.m_sensor[m], f.m_pose[m]


class LiveWindow:
    """The reference's window rules on plain arrays, for pixel, bearing, inertial and pose factors (the test's own
    restatement; lists in arrival order per kind, which is the user order of a device-managed window)."""

    def __init__(self, seq):
        self.full, self.k = seq.full, seq.order
        self.knots = seq.full.knots[:K0].copy()
        self.lm_ids, self.lm_xyz = [], np.zeros((0, 3))
        self.p = dict(stamp=np.zeros(0), cam=np.zeros(0, np.int32), gid=np.zeros(0, np.int64), pixel=np.zeros((0, 2)))
        self.b = dict(stamp=np.zeros(0), cam=np.zeros(0, np.int32), gid=np.zeros(0, np.int64), bearing=np.zeros((0, 3)))
        self.i = dict(stamp=np.zeros(0), meas=np.zeros((0, 6)))
        self.m = dict(stamp=np.zeros(0), sensor=np.zeros(0, np.int32), pose=np.zeros((0, 7)))
        self.knot_const = np.zeros(K0, np.uint8)
        self.knot_const[:2] = 1
        self.gravity_const = 0

    def valid_range(self):
        left = (self.k - 1) // 2
        st = self.knots[:, 7]
        return st[left], st[len(st) - (self.k - 1 - left) - 1]

    def append_knot(self):
        st = self.knots[:, 7]
        new = self.knots[-2].copy()
        self.knots[-1, :7] = self.knots[-2, :7]
        new[7] = st[-1] + (st[-1] - st[-2])
        self.knots = np.vstack([self.knots, new])
        self.knot_const = np.append(self.knot_const, 0).astype(np.uint8)

    def base_of(self, stamps):
        return np.searchsorted(self.knots[:, 7], stamps, side="right") - 1 - (self.k - 1) // 2

    def slots_for(self, gids):
        """landmark_in of hb200_append_stereo_tracks: the window slot, -1 for a landmark the window does not hold."""
        pos = {g: p for p, g in enumerate(self.lm_ids)}
        return np.array([pos.get(g, -1) for g in gids.tolist()], dtype=np.int32)

    def add_landmarks(self, gids, xyz):
        """New landmarks (slots L, L+1, ... in track order); returns every track's slot."""
        new = self.slots_for(gids) == -1
        self.lm_ids += gids[new].tolist()
        self.lm_xyz = np.vstack([self.lm_xyz, xyz[new].reshape(-1, 3)])
        return self.slots_for(gids)

    @staticmethod
    def _cat(lst, part):
        for key in lst:
            lst[key] = np.concatenate([lst[key], part[key]])

    def add_tracks(self, t, gids, b0, b1):   # camera0's factor, then camera1's, per track
        n = gids.size
        self._cat(self.b, dict(stamp=np.full(2 * n, t), cam=np.tile(np.array([0, 1], np.int32), n), gid=np.repeat(gids, 2),
                               bearing=np.stack([b0, b1], 1).reshape(-1, 3)))

    def add_pixels(self, t, gids, px0, px1):
        n = gids.size
        self._cat(self.p, dict(stamp=np.full(2 * n, t), cam=np.tile(np.array([0, 1], np.int32), n), gid=np.repeat(gids, 2),
                               pixel=np.stack([px0, px1], 1).reshape(-1, 2)))

    def add_inertial(self, stamp, meas):
        self._cat(self.i, dict(stamp=stamp, meas=meas))

    def add_poses(self, stamp, sensor, pose):
        self._cat(self.m, dict(stamp=stamp, sensor=sensor.astype(np.int32), pose=pose))

    def slide(self, lower, flags):
        st = self.knots[:, 7]
        ub = int(np.searchsorted(st, lower, side="right"))
        begin, last_const = max(0, ub - 1 - (self.k - 1) // 2), ub - 1
        last = {}
        for lst in (self.p, self.b):
            for g, t in zip(lst["gid"].tolist(), lst["stamp"].tolist()):
                last[g] = max(last.get(g, -np.inf), t)
        keep_lm = [g for g in self.lm_ids if g not in last or last[g] >= lower]
        keep_set = set(keep_lm)
        pm = np.array([g in keep_set for g in self.p["gid"].tolist()], dtype=bool)
        bm = np.array([g in keep_set for g in self.b["gid"].tolist()], dtype=bool)
        ib, mb = self.base_of(self.i["stamp"]), self.base_of(self.m["stamp"])
        im = ~(ib + self.k - 1 <= last_const) if flags & DROP_INERTIAL else np.ones(ib.size, dtype=bool)
        mm = ~(mb + self.k - 1 <= last_const) if flags & DROP_POSE else np.ones(mb.size, dtype=bool)
        mins = [begin]
        for bases, keep in ((self.base_of(self.p["stamp"]), pm), (self.base_of(self.b["stamp"]), bm), (ib, im), (mb, mm)):
            if keep.any():
                mins.append(int(bases[keep].min()))
        shift = max(0, min(min(mins), len(st) - self.k))
        dropped = dict(landmarks=len(self.lm_ids) - len(keep_lm), visual=int((~pm).sum() + (~bm).sum()), inertial=int((~im).sum()),
                       pose=int((~mm).sum()), knots=shift, constant=max(0, ub - shift))
        sel = [p for p, g in enumerate(self.lm_ids) if g in keep_set]
        self.lm_xyz, self.lm_ids = self.lm_xyz[sel], keep_lm
        for lst, keep in ((self.p, pm), (self.b, bm), (self.i, im), (self.m, mm)):
            for key in lst:
                lst[key] = lst[key][keep]
        self.knots = self.knots[shift:]
        self.knot_const = (self.knots[:, 7] <= lower).astype(np.uint8)
        if ub > 0:
            self.gravity_const = 1
        return dropped

    def counts(self):
        return dict(pixel=self.p["stamp"].size, bearing=self.b["stamp"].size, inertial=self.i["stamp"].size, manifold=self.m["stamp"].size)

    def window(self):
        local = self.slots_for
        return dataclasses.replace(
            self.full, knots=self.knots.copy(), landmarks=self.lm_xyz.copy(),
            v_stamp=self.p["stamp"].copy(), v_cam=self.p["cam"].astype(np.int32), v_lm=local(self.p["gid"]), v_pixel=self.p["pixel"].copy(),
            b_stamp=self.b["stamp"].copy(), b_cam=self.b["cam"].astype(np.int32), b_lm=local(self.b["gid"]), b_bearing=self.b["bearing"].copy(),
            i_stamp=self.i["stamp"].copy(), i_meas=self.i["meas"].copy(),
            m_stamp=self.m["stamp"].copy(), m_sensor=self.m["sensor"].astype(np.int32), m_pose=self.m["pose"].copy(),
            knot_const=self.knot_const.copy(), gravity_const=self.gravity_const, truth=None)


def start(seq):
    """Initial window: K0 state elements, the inertial factors and pose priors of its valid range, no landmarks yet."""
    hw = LiveWindow(seq)
    lo, hi = hw.valid_range()
    hw.add_inertial(*seq.inertial(lo, hi))
    hw.add_poses(*seq.poses(lo, hi))
    return hw, hi


def frame_inputs(seq, hw, f, prev_hi):
    """The message of frame f after the new state element: stamp, tracks, IMU samples, pose priors."""
    _, hi = hw.valid_range()
    t = 0.5 * (prev_hi + hi)
    gids, px0, px1 = seq.tracks(f, t)
    imu = seq.inertial(prev_hi, hi)
    poses = seq.poses(prev_hi, hi) if f % POSE_EVERY == 1 else None
    return hi, t, gids, px0, px1, imu, poses


def lower_bound(hw):
    return hw.knots[len(hw.knots) - 1 - WIDTH, 7] + 1e-9


def ingest_oracle(hw, t, px0, px1):
    base = int(hw.base_of(np.array([t]))[0])
    cams = hw.full.cameras
    return ol.ingest_stereo_frame(hw.knots[base:base + hw.k], t, cams[0], cams[1], px0, px1)


def rc_of(err):
    return int(re.match(r"hb200 error (-?\d+)", str(err)).group(1))


# ---- device helpers ----------------------------------------------------------------------------------------------
def device_system(ctx):
    """The packed reduced system the last iteration assembled (read through torch, as tests/variant_worker.py does)."""
    import torch
    ctx.synchronize()
    ptr, count = ctx.system_device_ptr()

    class _Arr:
        __cuda_array_interface__ = dict(shape=(count,), typestr="<f8", data=(ptr, False), version=2)

    return torch.as_tensor(_Arr(), device="cuda").cpu().numpy().copy()


def decode(ctx, buf, win):
    K = win.knots.shape[0]
    m = 3 * win.gyro_bias.shape[0] + 3 * win.accel_bias.shape[0] + 2
    return sb.device_packed(buf, K, ctx.bandwidth(), m)


def assert_outputs_equal(a, b, where):
    assert sorted(a) == sorted(b), where
    for key in a:
        assert a[key].shape == b[key].shape and np.array_equal(a[key], b[key]), (where, key)


def twin(win, radius):
    t = runtime.Context(0)
    t.load_window(win, radius=radius)
    return t


def check_sizes(ctx, stats, hw, dropped, where):
    assert (stats["knots"], stats["landmarks"], stats["visual_factors"], stats["inertial_factors"]) == \
        (len(hw.knots), len(hw.lm_ids), hw.p["stamp"].size + hw.b["stamp"].size, hw.i["stamp"].size), (where, stats, dropped)
    assert (stats["knots_dropped"], stats["knots_constant"], stats["landmarks_dropped"], stats["visual_factors_dropped"], stats["inertial_factors_dropped"]) == \
        (dropped["knots"], dropped["constant"], dropped["landmarks"], dropped["visual"], dropped["inertial"]), (where, stats, dropped)
    assert ctx.factor_counts() == hw.counts(), (where, ctx.factor_counts(), hw.counts())


# ---- 1. the live sequence ----------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("flags", [0, DROP_INERTIAL, DROP_INERTIAL | DROP_POSE])
@pytest.mark.parametrize("order", [4, 6])
def test_live_sequence_matches_restatement_twin_and_oracle(built, order, flags):
    seq = LiveSequence(order)
    hw, prev_hi = start(seq)
    ctx = runtime.Context(0)
    ctx.load_window(hw.window())
    radius = 1e4
    total = dict(landmarks=0, visual=0, inertial=0, pose=0, knots=0)
    for f in range(FRAMES):
        hw.append_knot()
        ctx.append_knots(1)
        prev_hi, t, gids, px0, px1, imu, poses = frame_inputs(seq, hw, f, prev_hi)
        n = gids.size
        assert 10 <= n <= 80
        # the restatement takes the bearings / new landmarks hb200_ingest_stereo computes from the same input
        b0, b1, lm_w, bad = ctx.ingest_stereo(np.full(n, t), np.zeros(n), np.ones(n), px0, px1)
        assert bad == 0
        L_before, lm_in = len(hw.lm_ids), hw.slots_for(gids)
        slots = ctx.append_stereo_tracks(np.full(n, t), np.zeros(n), np.ones(n), px0, px1, lm_in)
        want = hw.add_landmarks(gids, lm_w)
        hw.add_tracks(t, gids, b0, b1)
        assert np.array_equal(slots, want), f
        new = lm_in == -1
        assert np.array_equal(slots[new], L_before + np.arange(new.sum()))
        # new landmarks: the state's pose at the stamp, midpoint triangulation (oracle)
        _, _, lm_o = ingest_oracle(hw, t, px0[new], px1[new])
        assert rel_err(ctx.state()["landmarks"][slots[new]], lm_o) < 1e-9, f
        ctx.append_inertial_factors(*imu)
        hw.add_inertial(*imu)
        if poses is not None and poses[0].size:
            ctx.append_manifold_factors(*poses)
            hw.add_poses(*poses)
        lower = lower_bound(hw)
        stats = ctx.slide(lower, drop_inertial=bool(flags & DROP_INERTIAL), drop_pose=bool(flags & DROP_POSE))
        dropped = hw.slide(lower, flags)
        for key in total:
            total[key] += dropped[key]
        check_sizes(ctx, stats, hw, dropped, f)
        st = ctx.state()
        assert np.array_equal(st["knots"], hw.knots) and np.array_equal(st["landmarks"], hw.lm_xyz), f
        # --- twin context: the restated lists through hb200_set_* + hb200_bind ---
        win = hw.window()
        tw = twin(win, radius)
        ctx.evaluate(jacobians=True)
        tw.evaluate(jacobians=True)
        assert_outputs_equal(ctx.outputs(), tw.outputs(), f)
        for got, ref in zip(ctx.index_maps(), tw.index_maps()):
            assert np.array_equal(got, ref), f
        ow = ol.OracleWindow(win, radius=radius)
        assert ow.bad == 0
        lay = sb.DofLayout.of(win)
        rec = ctx.iterate(1)
        dev = decode(ctx, device_system(ctx), win)
        rec_tw = tw.iterate(1)
        found = sb.packed_mismatches(dev, decode(tw, device_system(tw), win), lay, tol=1e-12, cost_tol=1e-12)
        assert not found, (f, "\n".join(found[:10]))
        tw.close()
        # --- the cost at the linearisation point: the oracle's, the twin's ---
        assert abs(rec[0]["cost"] - ow.cost()) <= 1e-7 * abs(ow.cost()), (f, rec[0], ow.cost())
        assert abs(rec[0]["cost"] - rec_tw[0]["cost"]) <= 1e-12 * abs(rec_tw[0]["cost"]), (f, rec[0], rec_tw[0])
        recs = rec + ctx.iterate(1)   # (the second iteration moves the state on, as the live loop does)
        radius = recs[-1]["radius"]
        st = ctx.state()
        hw.knots, hw.lm_xyz = st["knots"].copy(), st["landmarks"].copy()
        hw.full = dataclasses.replace(hw.full, gyro_bias=st["gyro_bias"].copy(), accel_bias=st["accel_bias"].copy(), gravity=st["gravity"].copy())
    ctx.close()
    assert total["landmarks"] > 50 and total["visual"] > 500, total
    if flags & DROP_POSE:
        assert total["knots"] > 5 and total["pose"] > 0 and total["inertial"] > 100, total
    else:   # kept pose priors (and, without DROP_INERTIAL, inertial factors) keep the leading state elements
        assert total["knots"] == 0 and total["pose"] == 0, total
        assert (total["inertial"] > 100) == bool(flags & DROP_INERTIAL), total


# ---- 2. pixel and stereo-track frames in one window ------------------------------------------------------------------
@pytest.mark.gpu
def test_mixed_pixel_and_stereo_frames(built):
    """Pixel frames (hb200_append_landmarks + hb200_append_pixel_factors) alternate with stereo-track frames.  The
    per-kind copy-out of the slid window serves oracle-shaped factors, and a full hb200_bind from the host mirrors
    reproduces the outputs bitwise and the iteration's system per block to 1e-12."""
    order, flags, frames = 4, DROP_INERTIAL | DROP_POSE, 14
    seq = LiveSequence(order, frames=frames)
    hw, prev_hi = start(seq)
    ctx = runtime.Context(0)
    ctx.load_window(hw.window())
    for f in range(frames):
        hw.append_knot()
        ctx.append_knots(1)
        prev_hi, t, gids, px0, px1, imu, poses = frame_inputs(seq, hw, f, prev_hi)
        n = gids.size
        b0, b1, lm_w, _ = ctx.ingest_stereo(np.full(n, t), np.zeros(n), np.ones(n), px0, px1)
        lm_in = hw.slots_for(gids)
        if f % 2 == 0:
            slots = ctx.append_stereo_tracks(np.full(n, t), np.zeros(n), np.ones(n), px0, px1, lm_in)
            assert np.array_equal(slots, hw.add_landmarks(gids, lm_w))
            hw.add_tracks(t, gids, b0, b1)
        else:
            ctx.append_landmarks(lm_w[lm_in == -1])
            slots = hw.add_landmarks(gids, lm_w)
            ctx.append_pixel_factors(np.full(2 * n, t), np.tile([0, 1], n), np.repeat(slots, 2), np.stack([px0, px1], 1).reshape(-1, 2))
            hw.add_pixels(t, gids, px0, px1)
        ctx.append_inertial_factors(*imu)
        hw.add_inertial(*imu)
        if poses is not None and poses[0].size:
            ctx.append_manifold_factors(*poses)
            hw.add_poses(*poses)
        lower = lower_bound(hw)
        stats = ctx.slide(lower, drop_inertial=True, drop_pose=True)
        check_sizes(ctx, stats, hw, hw.slide(lower, flags), f)
        assert np.array_equal(ctx.state()["knots"], hw.knots) and np.array_equal(ctx.state()["landmarks"], hw.lm_xyz), f
        ctx.iterate(2)
        st = ctx.state()
        hw.knots, hw.lm_xyz = st["knots"].copy(), st["landmarks"].copy()
        hw.full = dataclasses.replace(hw.full, gyro_bias=st["gyro_bias"].copy(), accel_bias=st["accel_bias"].copy(), gravity=st["gravity"].copy())
    win = hw.window()
    assert win.v_stamp.size > 100 and win.b_stamp.size > 100 and win.m_stamp.size > 0
    # --- Ceres-shaped per-factor copy-out (user order = per-kind list order) against the oracle ---
    ctx.evaluate(jacobians=True)
    k, left = win.order, (win.order - 1) // 2
    for kind, okind, stamps, cams_, lms, meas in ((runtime.PIXEL, ol.PIXEL, win.v_stamp, win.v_cam, win.v_lm, win.v_pixel),
                                                  (runtime.BEARING, ol.BEARING, win.b_stamp, win.b_cam, win.b_lm, win.b_bearing)):
        for i in (0, 7, stamps.size // 2, stamps.size - 1):
            base = int(np.searchsorted(win.knots[:, 7], stamps[i], side="right") - 1 - left)
            cam = win.cameras[cams_[i]]
            blocks = [win.knots[base + m] for m in range(k)] + [cam[:7], cam[7:11], cam[11:15], win.landmarks[lms[i]]]
            r, jac = ctx.factor_evaluate(kind, i, blocks)
            r_o, jac_o = ol.cost_evaluate(okind, stamps[i], meas[i], np.concatenate(blocks), k=k)
            assert rel_err(r, r_o) < 1e-9, (kind, i)
            for m in range(k):
                PJ = ol.manifold_plus_jacobian(ol.M_STATE, blocks[m])
                assert rel_err(jac[m] @ PJ, jac_o[m] @ PJ) < 1e-8, (kind, i, m)
            assert rel_err(jac[k + 3], jac_o[k + 3]) < 1e-8, (kind, i)
    # --- a full hb200_bind from the host mirrors reproduces the device-managed window ---
    ctx.snapshot()
    ctx.evaluate(jacobians=True)
    out_a, maps_a = ctx.outputs(), ctx.index_maps()
    ctx.iterate(1)
    sys_a = decode(ctx, device_system(ctx), win)
    ctx.restore()
    ctx.bind()
    ctx.evaluate(jacobians=True)
    assert_outputs_equal(out_a, ctx.outputs(), "rebind")
    for a, b in zip(maps_a, ctx.index_maps()):
        assert np.array_equal(a, b)
    ctx.iterate(1)
    found = sb.packed_mismatches(decode(ctx, device_system(ctx), win), sys_a, sb.DofLayout.of(win), tol=REBIND_TOL, cost_tol=1e-12)
    assert not found, "\n".join(found[:10])
    ctx.close()


# ---- 3. rejected appends ---------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_rejected_appends_leave_the_window_unchanged(built):
    seq = LiveSequence(4, frames=4)
    hw, prev_hi = start(seq)
    ctx = runtime.Context(0)
    ctx.load_window(hw.window())
    last_t = None
    for f in range(3):
        hw.append_knot()
        ctx.append_knots(1)
        prev_hi, t, gids, px0, px1, imu, poses = frame_inputs(seq, hw, f, prev_hi)
        n = gids.size
        ctx.append_stereo_tracks(np.full(n, t), np.zeros(n), np.ones(n), px0, px1, hw.slots_for(gids))
        _, _, lm_w, _ = ctx.ingest_stereo(np.full(n, t), np.zeros(n), np.ones(n), px0, px1)
        hw.add_landmarks(gids, lm_w)
        ctx.append_inertial_factors(*imu)
        last_t = t
    assert ctx.factor_counts()["manifold"] > 0
    lo, hi = hw.valid_range()
    L = ctx.L
    gids, px0, px1 = seq.tracks(2, last_t)
    n = gids.size
    ones, zeros, new = np.ones(n), np.zeros(n), np.full(n, -1)

    def snapshot():
        return (ctx.K, ctx.L, ctx.Nv, ctx.Nb, ctx.Ni, ctx.Nm), ctx.factor_counts(), ctx.state()

    before = snapshot()
    p_stamp, p_meas, p_sensor = hw.full.m_stamp, hw.full.m_pose, hw.full.m_sensor
    cases = [
        (2, lambda: ctx.append_stereo_tracks(np.full(n, hi + 1.0), zeros, ones, px0, px1, new)),              # stamp outside the spline
        (2, lambda: ctx.append_stereo_tracks(np.full(n, last_t), np.full(n, 2), ones, px0, px1, new)),       # camera0 out of range
        (2, lambda: ctx.append_stereo_tracks(np.full(n, last_t), zeros, np.full(n, -1), px0, px1, new)),     # camera1 out of range
        (2, lambda: ctx.append_stereo_tracks(np.full(n, last_t), zeros, ones, px0, px1, np.full(n, -2))),    # landmark_in < -1
        (2, lambda: ctx.append_stereo_tracks(np.full(n, last_t), zeros, ones, px0, px1, np.full(n, L))),     # landmark_in >= L
        (3, lambda: ctx.append_stereo_tracks(np.full(n, last_t - 0.1), zeros, ones, px0, px1, new)),         # arrival order
        (2, lambda: ctx.append_bearing_factors([hi + 1.0], [0], [0], [[0.0, 0.0, 1.0]])),
        (2, lambda: ctx.append_bearing_factors([last_t], [2], [0], [[0.0, 0.0, 1.0]])),
        (2, lambda: ctx.append_bearing_factors([last_t], [0], [L], [[0.0, 0.0, 1.0]])),
        (3, lambda: ctx.append_bearing_factors([last_t - 0.1], [0], [0], [[0.0, 0.0, 1.0]])),
        (2, lambda: ctx.append_manifold_factors([hi + 1.0], [0], p_meas[:1])),
        (2, lambda: ctx.append_manifold_factors([last_t], [p_sensor.max() + 1], p_meas[:1])),
        (3, lambda: ctx.append_manifold_factors([lo], [0], p_meas[:1])),
    ]
    assert p_stamp.size and hw.base_of(np.array([lo]))[0] < hw.base_of(hw.m["stamp"]).max()
    for i, (rc, call) in enumerate(cases):
        with pytest.raises(runtime.HB200Error) as err:
            call()
        assert rc_of(err.value) == rc, (i, str(err.value))
        after = snapshot()
        assert after[0] == before[0] and after[1] == before[1], (i, after[:2], before[:2])
        for key in before[2]:
            assert np.array_equal(after[2][key], before[2][key]), (i, key)
    # the window still works: a valid frame appends, the counts move
    ctx.append_stereo_tracks(np.full(n, last_t), zeros, ones, px0, px1, new)
    assert ctx.L == L + n and ctx.factor_counts()["bearing"] == before[1]["bearing"] + 2 * n
    ctx.close()
    # pose priors without pose sensors
    hw0, _ = start(seq)
    win = dataclasses.replace(hw0.window(), pose_sensors=np.zeros((0, 7)), m_stamp=np.zeros(0), m_sensor=np.zeros(0, np.int32), m_pose=np.zeros((0, 7)))
    ctx = runtime.Context(0)
    ctx.load_window(win)
    with pytest.raises(runtime.HB200Error) as err:
        ctx.append_manifold_factors([lo + 0.05], [0], p_meas[:1])
    assert rc_of(err.value) == -2 and ctx.factor_counts()["manifold"] == 0
    ctx.close()


# ---- 4. the same sequence without a device ---------------------------------------------------------------------------
@pytest.mark.parametrize("order", [4, 6])
def test_live_sequence_rehearsal_on_the_oracle(order):
    """Sequence generator + restatement + per-frame oracle windows of the live test, new landmarks and bearings from
    the oracle's ingest: every window binds (no factor outside the spline) and the flags drop what they should."""
    seq = LiveSequence(order)
    totals = {}
    for flags in (DROP_INERTIAL, DROP_INERTIAL | DROP_POSE):
        hw, prev_hi = start(seq)
        total = dict(landmarks=0, visual=0, inertial=0, pose=0, knots=0)
        for f in range(FRAMES):
            hw.append_knot()
            prev_hi, t, gids, px0, px1, imu, poses = frame_inputs(seq, hw, f, prev_hi)
            assert 10 <= gids.size <= 80
            b0, b1, lm_w = ingest_oracle(hw, t, px0, px1)
            hw.add_landmarks(gids, lm_w)
            hw.add_tracks(t, gids, b0, b1)
            hw.add_inertial(*imu)
            if poses is not None:
                hw.add_poses(*poses)
            dropped = hw.slide(lower_bound(hw), flags)
            for key in total:
                total[key] += dropped[key]
            win = hw.window()
            ow = ol.OracleWindow(win)
            assert ow.bad == 0, f
        totals[flags] = total
    assert totals[DROP_INERTIAL]["knots"] == 0 and totals[DROP_INERTIAL]["pose"] == 0
    assert totals[DROP_INERTIAL | DROP_POSE]["knots"] > 5 and totals[DROP_INERTIAL | DROP_POSE]["pose"] > 0
    for total in totals.values():
        assert total["landmarks"] > 50 and total["inertial"] > 100, total
