"""Per-frame cost of the device-resident sliding window in the reference's live configuration.

Window of ~33 state elements (3.0 s at 0.1 s), one new element per frame, ~150 stereo tracks x 2 cameras per frame
(landmarks observed over 5 frames), 20 IMU samples per frame, then hb200_slide, 5 LM iterations and a read-back of
the state.  Two ways of bringing the tracks in, alternated frame by frame in the same process on two contexts:

  (a) stereo  hb200_append_stereo_tracks (bearings + triangulation + bind on the device, one H2D, one small D2H)
  (b) split   hb200_ingest_stereo -> hb200_append_landmarks -> hb200_append_bearing_factors

Reports median and minimum ms per frame (host clock around the whole frame; every frame ends in the state
read-back, a device synchronise) with the card name and its power limit.

    python tools/sliding_live.py [--frames 240] [--warmup 20]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from hyperslam_b200 import runtime, synthetic  # noqa: E402

K_WINDOW, DT, TRACKS, TRACK_LEN, IMU_PER_FRAME, ITERATIONS = 33, 0.1, 150, 5, 20, 5


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30)
        power = float(out.stdout.strip().splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        power = None
    return name, power


class Sequence:
    """Ground-truth trajectory, IMU samples and stereo tracks; TRACKS / TRACK_LEN new landmarks per frame."""

    def __init__(self, frames, seed=synthetic.SEED_BASE + 9001):
        k = 4
        self.K = K_WINDOW + frames + 4
        self.win = synthetic.make_window(order=k, num_knots=self.K, num_landmarks=0, num_imu=IMU_PER_FRAME * (self.K - k + 1), seed=seed)
        self.rng = np.random.Generator(np.random.Philox(seed + 1))
        self.born = TRACKS // TRACK_LEN
        self.xyz = np.zeros((0, 3))

    def new_landmarks(self, t):
        n, w = self.born, self.win
        c0 = w.cameras[0]
        px = np.stack([self.rng.uniform(250, synthetic.IMAGE_SIZE[0] - 250, n), self.rng.uniform(150, synthetic.IMAGE_SIZE[1] - 150, n)], -1)
        ray = np.stack([(px[:, 0] - c0[7]) / c0[9], (px[:, 1] - c0[8]) / c0[10], np.ones(n)], -1) * self.rng.uniform(3.0, 8.0, (n, 1))
        R, p, *_ = synthetic.spline_eval(w.truth["knots"], w.order, np.full(n, t))
        p_b = ray @ synthetic.quat_to_rot(c0[None, :4])[0].T + c0[4:7]
        self.xyz = np.vstack([self.xyz, (R @ p_b[..., None])[..., 0] + p])

    def tracks(self, f, t):
        """global landmark ids alive at frame f and their noisy pixels in both cameras."""
        while self.xyz.shape[0] < (f + 1) * self.born:
            self.new_landmarks(t)
        lo = max(0, f - TRACK_LEN + 1) * self.born
        gids = np.arange(lo, (f + 1) * self.born)
        n, w = gids.size, self.win
        px0, _ = synthetic.pixel_model(w.truth["knots"], w.order, w.cameras, self.xyz, np.full(n, t), np.zeros(n, dtype=int), gids)
        px1, _ = synthetic.pixel_model(w.truth["knots"], w.order, w.cameras, self.xyz, np.full(n, t), np.ones(n, dtype=int), gids)
        return gids, px0 + self.rng.normal(0, 0.4, px0.shape), px1 + self.rng.normal(0, 0.4, px1.shape)


class Runner:
    """One context fed frame by frame; the caller-side identifier -> slot map lives here, as INTEGRATION.md describes."""

    def __init__(self, seq, variant):
        w, k = seq.win, seq.win.order
        self.seq, self.variant, self.k = seq, variant, k
        stamps = w.knots[:, 7]
        self.hi = stamps[K_WINDOW - 1 - (k - 1 - (k - 1) // 2)]
        lo = stamps[(k - 1) // 2]
        m = (w.i_stamp >= lo) & (w.i_stamp < self.hi)
        import dataclasses
        init = dataclasses.replace(w, knots=w.knots[:K_WINDOW].copy(), landmarks=np.zeros((0, 3)), v_stamp=np.zeros(0), v_cam=np.zeros(0, np.int32),
                                   v_lm=np.zeros(0, np.int32), v_pixel=np.zeros((0, 2)), i_stamp=w.i_stamp[m], i_meas=w.i_meas[m],
                                   knot_const=np.r_[np.ones(2, np.uint8), np.zeros(K_WINDOW - 2, np.uint8)])
        self.ctx = runtime.Context(0)
        self.ctx.load_window(init)
        self.stamps = list(stamps[:K_WINDOW])
        self.window_gids, self.last_t = [], {}

    def frame(self, f):
        ctx, seq = self.ctx, self.seq
        ctx.append_knots(1)
        self.stamps.append(self.stamps[-1] + DT)
        lo, self.hi = self.hi, self.hi + DT
        t = lo + 0.5 * DT
        gids, px0, px1 = seq.tracks(f, t)
        n = gids.size
        slot = {g: s for s, g in enumerate(self.window_gids)}
        lm_in = np.array([slot.get(g, -1) for g in gids.tolist()], dtype=np.int32)
        stamp, c0, c1 = np.full(n, t), np.zeros(n, np.int32), np.ones(n, np.int32)
        if self.variant == "stereo":
            ctx.append_stereo_tracks(stamp, c0, c1, px0, px1, lm_in)
        else:
            b0, b1, lm, _ = ctx.ingest_stereo(stamp, c0, c1, px0, px1)
            new = lm_in == -1
            ctx.append_landmarks(lm[new])
            slots = lm_in.copy()
            slots[new] = len(self.window_gids) + np.arange(new.sum())
            ctx.append_bearing_factors(np.full(2 * n, t), np.tile([0, 1], n), np.repeat(slots, 2), np.stack([b0, b1], 1).reshape(-1, 3))
        self.window_gids += gids[lm_in == -1].tolist()
        for g in gids.tolist():
            self.last_t[g] = t
        w = seq.win
        m = (w.i_stamp >= lo) & (w.i_stamp < self.hi)
        ctx.append_inertial_factors(w.i_stamp[m], w.i_meas[m])
        lower = self.stamps[len(self.stamps) - K_WINDOW] + 1e-9
        st = ctx.slide(lower, drop_inertial=True)
        self.stamps = self.stamps[st["knots_dropped"]:]
        self.window_gids = [g for g in self.window_gids if self.last_t[g] >= lower]
        ctx.iterate(ITERATIONS, records=False)
        state = ctx.state()
        assert state["landmarks"].shape[0] == len(self.window_gids) and state["knots"].shape[0] == len(self.stamps)
        return n


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--frames", type=int, default=240)
    ap.add_argument("--warmup", type=int, default=20)
    args = ap.parse_args()
    name, power = card()
    frames = args.frames + args.warmup
    runners = [Runner(Sequence(frames), v) for v in ("stereo", "split")]
    times = {r.variant: [] for r in runners}
    tracks = []
    for f in range(frames):
        for r in runners:   # alternated frame by frame: both variants see the same machine state
            t0 = time.perf_counter()
            n = r.frame(f)
            dt = (time.perf_counter() - t0) * 1e3
            if f >= args.warmup:
                times[r.variant].append(dt)
        tracks.append(n)
    ctx = runners[0].ctx
    sizes = dict(knots=ctx.K, landmarks=ctx.L, **ctx.factor_counts())
    out = dict(card=name, power_limit_w=power, frames=args.frames, warmup=args.warmup, tracks_per_frame=int(np.median(tracks[args.warmup:])),
               iterations=ITERATIONS, window=sizes)
    for v, ts in times.items():
        out[v] = dict(median_ms=float(np.median(ts)), min_ms=float(np.min(ts)))
    print(json.dumps(out))
    for r in runners:
        r.ctx.close()


if __name__ == "__main__":
    main()
