#!/usr/bin/env python
"""bench.py -- factor evals/s & GN-iters/s of the B200 hot path (BASELINE.json metric).

A "step" is one Levenberg-Marquardt / Gauss-Newton iteration of the sliding-window problem: evaluate
every factor (residual + Jacobian) -> loss reweighting -> J^T J / J^T r -> landmark Schur complement
-> [one ncclAllReduce of the packed band-only system at N > 1] -> banded-arrow Cholesky -> back-substitution
-> retraction -> cost at the trial point -> accept/reject, captured as ONE CUDA graph at every N.
`value` = factors per second with everything resident in HBM; `e2e` = the same through
hb200_optimize() with the variable blocks in pinned HOST memory (H2D + D2H inside the timed region).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config 1] [--impl reference] [--dump-outputs DIR]
N > 1: launched by torch.distributed.run, one rank per GPU, weak scaling on the headline workload (each rank
owns one cfg-sized factor shard of an N-times larger window) plus strong-scaling sections on the large
BASELINE configs (cfg3: 500 k pixel factors, cfg4: 1 M factors) sharded over the N ranks.
torch.distributed only ships the NCCL unique id / IPC handles and takes the max over ranks of the timings;
the communicator and every collective on the iteration path live inside libhyperb200.so.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from hyperslam_b200 import synthetic  # noqa: E402

METRIC = "factor_evals_per_s"
UNIT = "factor evals/s"


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=300)
    p.add_argument("--warmup", type=int, default=10)
    p.add_argument("--config", type=int, default=1, help="index into BASELINE.json configs (default 1 = headline)")
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-large", action="store_true", help="skip the large-window sections (cfg2 / cfg3 / cfg4)")
    p.add_argument("--no-parity", action="store_true", help="skip the N-rank vs oracle check at N > 1")
    p.add_argument("--sweep", action="store_true", help="factor-count sweep of the 1 M-factor window (BASELINE config 5)")
    p.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (float64, single GPU)")
    return p.parse_args()


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f)["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def make_global_window(config, world):
    cfg = dict(synthetic.CONFIGS[config])
    cfg["num_landmarks"] *= world
    cfg["num_imu"] *= world
    return synthetic.make_window(seed=synthetic.SEED_BASE + config + 1, constant_knots=2, **cfg)


def algorithmic_bytes(win):
    """Per-launch algorithmic bytes of the factor kernels (DESIGN.md 'HBM layout'): per factor, inputs + residual +
    Jacobian blocks; the shared window state once per launch."""
    k, kb = win.order, win.bias_order
    K, L, C = win.knots.shape[0], win.landmarks.shape[0], win.cameras.shape[0]
    pix_per = 8 + 16 + 16 + 16 + 2 * 6 * k * 8 + 48            # stamp, pixel, idx | r, Jp, Jl
    imu_per = 8 + 48 + 16 + 48 + 6 * 6 * k * 8 + 2 * kb * 8 + 96  # stamp, meas, idx | r, Jp, wg, wa, Jg
    shared = K * 224
    pix = win.v_stamp.size * pix_per + (shared + L * 24 + C * 160 if win.v_stamp.size else 0)
    imu = win.i_stamp.size * imu_per + (shared + 48 * 8 + (win.gyro_bias.size + win.accel_bias.size) * 8 if win.i_stamp.size else 0)
    return dict(pixel_eval_kernel=pix, inertial_eval_kernel=imu, factor_eval_kernel=pix + imu, pixel_per_factor=pix_per, inertial_per_factor=imu_per)


class ClockSampler:
    """SM clock / throttle reasons sampled through NVML every 2 ms from BEFORE the warm-up to the end of the timed
    region (nvidia-smi -lms as the fallback); `mark()` brackets the timed region so both counts are reported."""
    NAMES = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, device):
        self.device = device
        self.rows = []          # (t, sm_mhz, reasons bitmask)
        self.max_mhz = None
        self.stop_flag = False
        self.thread = None
        self.marks = []
        self.backend = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            index = int(visible.split(",")[self.device]) if visible and visible.split(",")[0].isdigit() else self.device
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml
            self.backend = "nvml"
            self.thread = threading.Thread(target=self._poll_nvml, daemon=True)
        except Exception:
            self.backend = "nvidia-smi"
            self.thread = threading.Thread(target=self._poll_smi, daemon=True)
        self.thread.start()

    def _poll_nvml(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((time.perf_counter(), float(mhz), int(reasons)))
            except Exception:
                pass
            time.sleep(0.002)

    def _poll_smi(self):
        fields = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                  "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), f"--query-gpu={fields}", "--format=csv,noheader,nounits", "-lms", "5"],
                                    stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            return
        bits = [0x8, 0x40, 0x20, 0x4]
        for line in proc.stdout:
            if self.stop_flag:
                break
            r = [x.strip() for x in line.split(",")]
            try:
                mask = sum(b for b, v in zip(bits, r[2:6]) if v.lower().startswith("active"))
                self.rows.append((time.perf_counter(), float(r[0]), mask))
                self.max_mhz = float(r[1])
            except (ValueError, IndexError):
                continue
        proc.terminate()

    def mark(self):
        self.marks.append(time.perf_counter())

    def stop(self):
        self.stop_flag = True
        if self.thread:
            self.thread.join(timeout=2)
        if not self.rows:
            return dict(sm_mhz=None, sm_max_mhz=self.max_mhz, reasons=["no samples"], samples=0, backend=self.backend)
        lo, hi = (self.marks[0], self.marks[-1]) if len(self.marks) >= 2 else (-1e300, 1e300)
        timed = [r for r in self.rows if lo <= r[0] <= hi]
        use = timed if len(timed) >= 3 else self.rows   # a very short timed region: fall back to warm-up + timed samples
        mask = 0
        for r in self.rows:
            mask |= r[2]
        return dict(sm_mhz=statistics.median(r[1] for r in use), sm_max_mhz=self.max_mhz,
                    reasons=sorted(n for b, n in self.NAMES.items() if mask & b), samples=len(self.rows), samples_in_timed_region=len(timed),
                    backend=self.backend, period_ms=2 if self.backend == "nvml" else 5)


def best_thread_count(ow, fn):
    """The CPU arm gets the thread count that serves it best (hyper-threads usually hurt)."""
    import psutil
    cands = sorted({c for c in (psutil.cpu_count(logical=False), os.cpu_count(), 32, 16, 8) if c and c <= (os.cpu_count() or 1)})
    best, best_t = cands[-1], float("inf")
    for c in cands:
        fn(c)
        t0 = time.perf_counter(); fn(c); fn(c); dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = c, dt
    return best


def run_reference(args, rank, world):
    """CPU arm: the oracle (a restatement -- the reference cannot be built here) on the host cores."""
    if rank != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as ol
    win = make_global_window(args.config, 1)
    ow = ol.OracleWindow(win)
    nf = win.num_factors
    cores = best_thread_count(ow, lambda c: ow.iterate(apply=False, outputs=False, nthreads=c))
    for _ in range(max(args.warmup, 1)):
        ow.iterate(apply=False, outputs=False, nthreads=cores)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ow.iterate(apply=False, outputs=False, nthreads=cores)
    dt = (time.perf_counter() - t0) / max(args.steps, 1)
    value = nf / dt
    ev_cores = best_thread_count(ow, lambda c: ow.evaluate(want_J=True, outputs=False, nthreads=c))
    t1 = time.perf_counter()
    reps = 0
    while time.perf_counter() - t1 < 2.0:
        ow.evaluate(want_J=True, outputs=False, nthreads=ev_cores); reps += 1
    ev = nf * reps / (time.perf_counter() - t1)
    line = dict(impl="reference", metric=METRIC, value=value, unit=UNIT, n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=dt * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64", data="synthetic",
                config=dict(workload=synthetic.CONFIG_NAMES[args.config], factors_per_step=nf, note="CPU oracle (restatement of the reference path; Ceres/Eigen/HyperState are not installable here), built -O3 -march=x86-64-v3 (the reference builds -O3 -march=native), OpenMP over factors, serial assembly + Schur + dense Cholesky"),
                cpu_baseline=dict(value=value, unit=UNIT, cores=cores, kind="port", sample=f"{args.steps} full LM iterations of {nf} factors each",
                                  evaluate_only_value=ev, evaluate_only_cores=ev_cores, gn_iters_per_s=1.0 / dt),
                e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gn_iters_per_s=1.0 / dt,
                evaluate_sweep=dict(evals_per_s=ev))
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------------------
class Harness:
    """One rank's view of one window: context, L2 flush, device-timed steps (max over ranks)."""

    def __init__(self, torch, dist, runtime, local_rank, rank, world, gwin, flush):
        self.torch, self.dist, self.rank, self.world, self.local_rank = torch, dist, rank, world, local_rank
        self.gwin = gwin
        self.win = gwin.shard(rank, world) if world > 1 else gwin
        self.ctx = runtime.Context(local_rank, use_graph=True)
        self.ctx.load_window(self.win)
        self.comm = self.ctx.connect_torch_distributed(dist) if world > 1 else dict(nranks=1, nccl=False, peer_mailbox=False)
        self.ext = torch.cuda.ExternalStream(self.ctx.stream, device=torch.device("cuda", local_rank))
        self.flush_buf = flush
        self.ctx.snapshot()

    def l2_flush(self):
        with self.torch.cuda.stream(self.ext):
            self.flush_buf.fill_(1.0)

    def maxreduce(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed_steps(self, step_fn, steps, warmup, sampler=None):
        torch, dist, ctx = self.torch, self.dist, self.ctx
        for _ in range(warmup):
            ctx.restore(); self.l2_flush(); step_fn()
        ctx.synchronize(); torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        stops = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        launches0 = ctx.launch_count
        if sampler:
            sampler.mark()
        for i in range(steps):
            ctx.restore(); self.l2_flush()
            starts[i].record(self.ext)
            step_fn()
            stops[i].record(self.ext)
        ctx.synchronize(); torch.cuda.synchronize()
        if sampler:
            sampler.mark()
        if self.world > 1:
            dist.barrier()
        ms = sum(s.elapsed_time(e) for s, e in zip(starts, stops))
        return self.maxreduce(ms), ctx.launch_count - launches0

    def kernel_profile(self, reps):
        """Per-launch durations of one iteration (CUDA event after every launch; same kernels, same fusion as the graph,
        side-stream forks serialised).  Collective at N > 1: every rank calls it."""
        self.ctx.restore()
        seq = self.ctx.profile_iteration(reps=reps)
        agg = {}
        for name, ms in seq:
            agg[name] = agg.get(name, 0.0) + ms
        first = {}
        for name, ms in seq:
            first.setdefault(name, ms)
        return seq, agg, first

    def close(self):
        self.ctx.close()


def dump_outputs(out_dir, ctx):
    """What a caller of the timed step receives: the window state after the last timed LM iteration, and the pose /
    landmark step that iteration solved for.  The window is seeded, so two builds can be compared array by array, to
    rounding (DESIGN.md section 6); the largest config, cfg4, writes about 4 MB."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = ctx.state()
    arrays["delta_p"], arrays["delta_l"] = ctx.delta()
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.ascontiguousarray(a, dtype=np.float64))


def roofline_entry(name, nbytes, ms, peak):
    ach = nbytes / (ms * 1e-3) / 1e9
    return dict(kernel=name, algorithmic_bytes_per_launch=int(nbytes), launch_ms=ms, achieved=ach, frac=ach / peak)


def comm_entry(h, agg, reps_total=1):
    """NVLink side of the iteration: payload and bus bandwidth of the one system all-reduce."""
    info = h.ctx.comm_info()
    pay = info["payload_doubles"] * 8
    peer = info.get("peer_reduce")
    ms = agg.get("peer_reduce_kernel") if peer else agg.get("ncclAllReduce(system)")
    n = h.world
    what = ("1 fused barrier + all-reduce kernel over NVLink peer memory (peer_reduce_kernel: flag exchange, then every rank sums the N partial "
            "systems out of its peers' HBM in rank order); no NCCL call on the iteration path") if peer else "1 ncclAllReduce (packed band-only system)"
    out = dict(allreduce_bytes=pay, mode="peer-memory" if peer else "nccl", collectives_per_iteration=what + (
        " + peer-memory scalar exchange fused in accept_kernel" if info.get("peer_mailbox") else " + 1 ncclAllReduce (8 scalars)"),
        comm_ms=ms)
    if ms:
        out["nvlink_algbw_gbs"] = pay / (ms * 1e-3) / 1e9
        out["nvlink_busbw_gbs"] = pay * 2 * (n - 1) / n / (ms * 1e-3) / 1e9
        out["note"] = "payload is latency-bound (NVLink 5: 900 GB/s per direction); comm_ms is the launch-to-completion time of the all-reduce on the iteration stream, max wait for the slowest rank included"
    return out


def large_section(torch, dist, runtime, local_rank, rank, world, flush, config, scale, peak, iters=5):
    """Strong-scaling section: one large BASELINE window sharded over the ranks (single GPU: the whole window)."""
    gwin = synthetic.make_config(config, scale=scale, constant_knots=2)
    h = Harness(torch, dist, runtime, local_rank, rank, world, gwin, flush)
    total_ms, _ = h.timed_steps(lambda: h.ctx.iterate(1, records=False), iters, 3)
    ms = total_ms / iters
    sweep_ms, _ = h.timed_steps(lambda: h.ctx.evaluate(jacobians=True), iters, 2)
    sweep_ms /= iters
    seq, agg, first = h.kernel_profile(3)
    out = None
    ab = algorithmic_bytes(h.win)
    info = h.ctx.comm_info()
    if rank == 0:
        out = dict(workload=synthetic.CONFIG_NAMES[config] + (f" x{scale:g}" if scale != 1.0 else ""), factors=gwin.num_factors, factors_per_gpu=h.win.num_factors,
                   n_gpus=world, reduced_system_size=h.ctx.reduced_size(), block_half_bandwidth=h.ctx.bandwidth(), ms_per_iteration=ms,
                   factor_evals_per_s=gwin.num_factors / (ms * 1e-3), gn_iters_per_s=1e3 / ms,
                   evaluate_sweep_ms=sweep_ms, evaluate_sweep_evals_per_s=gwin.num_factors / (sweep_ms * 1e-3), peak=peak, unit="GB/s",
                   iteration_kernel_ms={k_: round(v, 4) for k_, v in agg.items()}, graph=info["graph"],
                   per_launch_source="hb200_profile_iteration: the iteration's own kernels (fused J^T J included), CUDA event after every launch")
        for kname in ("pixel_eval_kernel", "inertial_eval_kernel", "factor_eval_kernel"):
            if kname in first and ab[kname]:
                out[kname] = roofline_entry(kname + " (Jacobian pass, in-iteration)", ab[kname], first[kname], peak)
        hbm_bytes = ab["pixel_eval_kernel"] + ab["inertial_eval_kernel"]
        out["iteration_hbm_gbs_per_gpu"] = hbm_bytes / (ms * 1e-3) / 1e9
        if world > 1:
            out["comm"] = comm_entry(h, agg)
    h.close()
    return out


def sliding_section(torch, runtime, local_rank, frames=20):
    """Steady-state frame loop through the device-side window bookkeeping (SURVEY.md 8f rank 3): per frame one state element
    is appended, the frame's factors and new landmarks are added (bound on the device), the window's lower bound moves on
    (expired landmarks / factors / leading state elements are compacted away), five LM iterations run and the state is
    read back -- wall clock per frame, host bookkeeping and all copies included."""
    K0, k = 50, 4
    full = synthetic.make_window(order=k, num_knots=K0 + frames + 2, num_landmarks=1000 + 25 * frames, frames_per_landmark=5, num_cameras=2,
                                 num_imu=2000 + 45 * frames, seed=synthetic.SEED_BASE + 4242)
    st = full.knots[:, 7]
    order_v, order_i = np.argsort(full.v_stamp, kind="stable"), np.argsort(full.i_stamp, kind="stable")
    v = dict(stamp=full.v_stamp[order_v], cam=full.v_cam[order_v], gid=full.v_lm[order_v], pixel=full.v_pixel[order_v])
    im = dict(stamp=full.i_stamp[order_i], meas=full.i_meas[order_i])
    hi = st[K0 - 2]
    vm, mm = v["stamp"] < hi, im["stamp"] < hi
    ids = list(dict.fromkeys(v["gid"][vm].tolist()))
    pos = {g: p for p, g in enumerate(ids)}
    import dataclasses
    kc = np.zeros(K0, np.uint8); kc[:2] = 1
    win = dataclasses.replace(full, knots=full.knots[:K0].copy(), landmarks=full.landmarks[ids], v_stamp=v["stamp"][vm], v_cam=v["cam"][vm],
                              v_lm=np.array([pos[g] for g in v["gid"][vm].tolist()], np.int32), v_pixel=v["pixel"][vm], i_stamp=im["stamp"][mm],
                              i_meas=im["meas"][mm], knot_const=kc, truth=None)
    ctx = runtime.Context(local_rank)
    ctx.load_window(win)
    ctx.iterate(5, records=False)
    times, sizes = [], []
    alive = list(ids)
    last_seen = {}
    for g, t in zip(v["gid"][vm].tolist(), v["stamp"][vm].tolist()):
        last_seen[g] = t
    prev_hi = hi
    for f in range(frames):
        hi = st[K0 + f - 1]
        sel_v = (v["stamp"] >= prev_hi) & (v["stamp"] < hi)
        sel_i = (im["stamp"] >= prev_hi) & (im["stamp"] < hi)
        prev_hi = hi
        new_ids = [g for g in dict.fromkeys(v["gid"][sel_v].tolist()) if g not in pos]
        lower = st[f + 1] + 1e-9   # the window keeps its length: one element in, one out
        # host-side id bookkeeping of the caller (which landmark sits where), mirrored from the rules
        for g, t in zip(v["gid"][sel_v].tolist(), v["stamp"][sel_v].tolist()):
            last_seen[g] = t
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ctx.append_knots(1)
        ctx.append_landmarks(full.landmarks[new_ids].reshape(-1, 3))
        alive += new_ids
        pos = {g: p for p, g in enumerate(alive)}
        ctx.append_pixel_factors(v["stamp"][sel_v], v["cam"][sel_v], np.array([pos[g] for g in v["gid"][sel_v].tolist()], np.int32), v["pixel"][sel_v])
        ctx.append_inertial_factors(im["stamp"][sel_i], im["meas"][sel_i])
        stats = ctx.slide(lower, drop_inertial=True)
        ctx.iterate(5, records=False)
        state = ctx.state()
        times.append(time.perf_counter() - t0)
        alive = [g for g in alive if last_seen.get(g, np.inf) >= lower]
        pos = {g: p for p, g in enumerate(alive)}
        assert len(alive) == stats["landmarks"], (len(alive), stats)
        sizes.append((stats["knots"], stats["landmarks"], stats["visual_factors"], stats["inertial_factors"]))
    ctx.close()
    med = statistics.median(times[3:])
    Kw, Lw, Nvw, Niw = sizes[-1]
    return dict(frames=frames, ms_per_frame_median=med * 1e3, ms_per_frame_min=min(times[3:]) * 1e3, window=dict(knots=Kw, landmarks=Lw, pixel_factors=Nvw, inertial_factors=Niw),
                per_frame="append 1 state element + ~%d pixel / ~%d inertial factors + new landmarks (H2D), hb200_slide, 5 LM iterations, state read-back (D2H); wall clock" % (
                    int(np.mean([s_[2] for s_ in sizes]) / (Kw - 3)), int(np.mean([s_[3] for s_ in sizes]) / (Kw - 3))),
                factor_evals_per_s=5 * (Nvw + Niw) / med)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and (world > 1 or args.impl != "b200"):
        raise SystemExit("--dump-outputs covers --impl b200 on one GPU (at N > 1 a rank's landmarks are only its own shard's)")
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")

    import torch
    import torch.distributed as dist
    from hyperslam_b200 import runtime

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")  # 256 MiB > 126 MB L2
    peak, peak_src = load_peaks()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    gwin = make_global_window(args.config, world)
    h = Harness(torch, dist, runtime, local_rank, rank, world, gwin, flush)
    ctx, win = h.ctx, h.win
    nf_total, nf_local = gwin.num_factors, win.num_factors
    n_reduced = ctx.reduced_size()

    # ---- device-resident steps ---------------------------------------------------------------
    total_ms, launches = h.timed_steps(lambda: ctx.iterate(1, records=False), args.steps, max(args.warmup, 3), sampler if rank == 0 else None)
    ms_per_step = total_ms / args.steps
    value = nf_total / (ms_per_step * 1e-3)
    info = ctx.comm_info()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, ctx)   # before the evaluate sweep below restores the snapshot

    # evaluate-only sweep (knot table + factor kernels, residual + Jacobian)
    sweep_ms, _ = h.timed_steps(lambda: ctx.evaluate(jacobians=True), args.steps, 3)
    sweep_ms /= args.steps

    # ---- end to end through hb200_optimize with pinned host buffers ---------------------------
    def pinned(a):
        t = torch.empty(a.shape, dtype=torch.float64).pin_memory()
        t.numpy()[...] = a
        return t
    init = dict(knots=win.knots, gyro=win.gyro_bias, accel=win.accel_bias, gravity=win.gravity, landmarks=win.landmarks)
    src = {k_: pinned(v) for k_, v in init.items()}
    work = {k_: pinned(v) for k_, v in init.items()}
    h2d = sum(v.numel() * 8 for v in work.values())
    d2h = h2d + 56

    def e2e_step():
        for k_ in work:
            work[k_].copy_(src[k_])   # host-side reset of the in/out buffers (not device work)
        ctx.restore()                 # trust-region state back to the initial radius
        h.l2_flush()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ctx.optimize(1, work["knots"].numpy(), work["gyro"].numpy(), work["accel"].numpy(), work["gravity"].numpy(),
                     work["landmarks"].numpy(), records=True)
        return time.perf_counter() - t0

    for _ in range(max(args.warmup, 3)):
        e2e_step()
    if world > 1:
        dist.barrier()
    e2e_t = h.maxreduce(sum(e2e_step() for _ in range(args.steps)) / args.steps)
    e2e_value = nf_total / e2e_t
    clocks = sampler.stop() if rank == 0 else None

    # ---- attribution: per-kernel durations of the iteration's own launch sequence (collective at N > 1) -------
    seq, kernel_ms, first = h.kernel_profile(10)
    total_k = sum(kernel_ms.values())
    shares = {k_: round(v / total_k, 4) for k_, v in kernel_ms.items()}
    ab = algorithmic_bytes(win)
    dominant = max(kernel_ms, key=kernel_ms.get)
    roof_kernel = "factor_eval_kernel" if "factor_eval_kernel" in first else "pixel_eval_kernel"
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    tj = {}
    if os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f)
        traffic = tj.get(roof_kernel + "_dram_bytes")
    roofline = roofline_entry(f"{roof_kernel}<{win.order},4,J,FUSE> -- the factor kernel of the timed graph (residual + Jacobian of every visual and inertial factor, fused pixel J^T J)",
                              ab[roof_kernel], first[roof_kernel], peak)
    roofline.update(bound="hbm", peak=peak, unit="GB/s", traffic=traffic, peak_source=peak_src, dominant_kernel_by_time=dominant,
                    kernel_share_of_step=shares, launch_sequence=[n for n, _ in seq],
                    kernel_ms_source="hb200_profile_iteration: the graph's launch sequence run with a CUDA event after every launch (measured live)",
                    whole_step=dict(algorithmic_bytes=ab["factor_eval_kernel"], ms=ms_per_step, achieved=ab["factor_eval_kernel"] / (ms_per_step * 1e-3) / 1e9,
                                    frac=ab["factor_eval_kernel"] / (ms_per_step * 1e-3) / 1e9 / peak),
                    note="cfg1 moves 7.8 MB per sweep (1.2 us at peak): latency-bound by construction (SURVEY.md 8d); large_windows holds the bandwidth-relevant fractions of the same in-iteration kernels",
                    traffic_note="dram__bytes_read + write of one launch from the committed ncu capture (profiles/traffic.json): far below the algorithmic bytes at cfg1 because the 7 MB of residuals / Jacobians the launch writes stay in the 126 MB L2 until the J^T J / Schur kernels have consumed them; on the 1M-factor window the same kernels write through (profiles/r02_ncu_full.md)")
    try:
        roofline["fp64_peak_tflops_measured"] = ctx.measure_fp64_peak()
    except Exception as e:  # noqa: BLE001
        roofline["fp64_peak_tflops_measured"] = None
        roofline["fp64_peak_error"] = str(e)
    comm = comm_entry(h, kernel_ms) if world > 1 else None

    # ---- N-rank == single-process oracle, on this very window (outside every timed region) -------------------
    parity = None
    if world > 1 and not args.no_parity:
        ctx.restore()
        recs = ctx.iterate(3)
        state = ctx.state()
        knots = torch.from_numpy(state["knots"]).cuda()
        ref = knots.clone()
        dist.broadcast(ref, 0)
        same = torch.tensor([1.0 if torch.equal(knots, ref) else 0.0], device="cuda")
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        if rank == 0:
            sys.path.insert(0, os.path.join(ROOT, "tests"))
            import oracle_lib as ol
            ow = ol.OracleWindow(gwin)
            worst_c, worst_n, acc_ok = 0.0, 0.0, True
            for rec in recs:
                o = ow.iterate(apply=True)
                worst_c = max(worst_c, abs(rec["cost"] - o["cost"]) / abs(o["cost"]))
                worst_n = max(worst_n, abs(rec["cost_new"] - o["cost_new"]) / abs(o["cost_new"]))
                acc_ok = acc_ok and rec["accepted"] == o["accepted"] and rec["spd"] == 1
            dk = float(np.abs(state["knots"] - ow.state()["knots"]).max())
            parity = dict(nrank_vs_oracle=dict(ok=bool(worst_c < 1e-7 and worst_n < 1e-6 and acc_ok and dk < 1e-6 and same.item() == 1.0),
                                               iterations=3, cost_rel_err=worst_c, trial_cost_rel_err=worst_n, accept_decisions_equal=acc_ok,
                                               knots_max_abs_diff=dk, replicas_bit_identical=bool(same.item() == 1.0),
                                               window=f"{nf_total} factors sharded over {world} ranks vs the single-process CPU oracle"))

    # dense library bar asked for by SURVEY.md 2.2: cuSOLVER potrf + potrs (through torch.linalg) on the same reduced system
    dense_bar = None
    if world == 1:
        try:
            ctx.restore(); ctx.evaluate(jacobians=True); ctx.build_system()
            S, b = ctx.system()
            Sd, bd = torch.from_numpy(S).cuda(), torch.from_numpy(b).cuda().unsqueeze(1)
            for _ in range(3):
                Lc = torch.linalg.cholesky(Sd); torch.cholesky_solve(bd, Lc)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(20):
                Lc = torch.linalg.cholesky(Sd); xs = torch.cholesky_solve(bd, Lc)
            e1.record(); torch.cuda.synchronize()
            ctx.solve(); dp, _ = ctx.delta()
            dense_bar = dict(cusolver_potrf_potrs_ms=e0.elapsed_time(e1) / 20, n=int(S.shape[0]), band_solve_kernel_ms=kernel_ms.get("band_solve_kernel"),
                             solution_rel_diff=float(np.abs(xs.squeeze(1).cpu().numpy() - dp).max() / (np.abs(dp).max() + 1e-300)),
                             note="torch.linalg.cholesky + cholesky_solve (cuSOLVER) on the dense damped system; library code, comparison only")
        except Exception as e:  # noqa: BLE001
            dense_bar = dict(error=str(e))

    h.close()

    sliding = None
    if world == 1 and not args.no_large:
        try:
            sliding = sliding_section(torch, runtime, local_rank)
        except Exception as e:  # noqa: BLE001
            sliding = dict(error=str(e))

    # ---- large windows: the BASELINE configs beyond the headline, at their GPU counts ------------------------
    large = {}
    if not args.no_large:
        plan = [(2, 1.0), (4, 1.0)] if world == 1 else ([(3, 1.0)] + ([(4, 1.0)] if world >= 8 else []))
        if args.sweep:
            plan += [(4, s) for s in (0.01, 0.1, 0.3)]
        for config, scale in plan:
            sec = large_section(torch, dist, runtime, local_rank, rank, world, flush, config, scale, peak)
            if rank == 0:
                key = f"cfg{config}" + (f"_x{scale:g}" if scale != 1.0 else "")
                large[key] = sec
        if rank == 0 and tj.get("large_window"):
            large["ncu_traffic"] = tj["large_window"]

    if rank != 0:
        if world > 1:
            dist.barrier(); dist.destroy_process_group()
        return

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle_lib as ol
        ow = ol.OracleWindow(gwin)
        cores = best_thread_count(ow, lambda c: ow.iterate(apply=False, outputs=False, nthreads=c))
        ow.iterate(apply=False, outputs=False, nthreads=cores)
        t0 = time.perf_counter(); reps = 0
        while time.perf_counter() - t0 < 6.0:
            ow.iterate(apply=False, outputs=False, nthreads=cores); reps += 1
        it_s = (time.perf_counter() - t0) / reps
        ev_cores = best_thread_count(ow, lambda c: ow.evaluate(want_J=True, outputs=False, nthreads=c))
        t0 = time.perf_counter(); r2 = 0
        while time.perf_counter() - t0 < 3.0:
            ow.evaluate(want_J=True, outputs=False, nthreads=ev_cores); r2 += 1
        ev_all = nf_total * r2 / (time.perf_counter() - t0)
        t0 = time.perf_counter(); r3 = 0
        while time.perf_counter() - t0 < 3.0:
            ow.evaluate(want_J=True, outputs=False, nthreads=1); r3 += 1
        ev_one = nf_total * r3 / (time.perf_counter() - t0)
        cpu = dict(value=nf_total / it_s, unit=UNIT, cores=cores, kind="port",
                   sample=f"{reps} full LM iterations + {r2} all-core and {r3} single-thread Evaluate sweeps of {nf_total} factors (oracle restatement; Ceres cannot be built here)",
                   gn_iters_per_s=1.0 / it_s, evaluate_only_all_cores=ev_all, evaluate_only_cores=ev_cores, evaluate_only_one_thread=ev_one)

    step_desc = "one LM iteration (evaluate r+J, JtJ, Schur, " + (("1 peer-memory all-reduce kernel, " if info.get("peer_reduce") else "1 NCCL all-reduce, ") if world > 1 else "") + \
                "banded Cholesky, retract, trial cost, accept) " + ("as one CUDA graph" if info["graph"] else "direct launches (graph capture unavailable)")
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3), ms_per_step=ms_per_step,
                higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f64", data="synthetic",
                config=dict(workload=synthetic.CONFIG_NAMES[args.config], factors_per_step=nf_total, factors_per_gpu=nf_local,
                            reduced_system_size=n_reduced, spline_order=win.order, knots=int(win.knots.shape[0]),
                            landmarks=int(gwin.landmarks.shape[0]), parallelism=f"factor-sharded x{world}" if world > 1 else "single GPU",
                            l2="flushed between timed steps (256 MiB device write)", step=step_desc),
                e2e=dict(value=e2e_value, unit=UNIT, h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h, ms_per_step=e2e_t * 1e3,
                         api="hb200_optimize(1 iteration) with pinned host variable blocks"),
                gpu_launches=int(launches), clocks=clocks, gn_iters_per_s=1e3 / ms_per_step,
                evaluate_sweep=dict(ms=sweep_ms, evals_per_s=nf_total / (sweep_ms * 1e-3)), kernel_ms={k_: round(v, 5) for k_, v in kernel_ms.items()},
                roofline=roofline)
    if large:
        line["roofline"]["large_windows"] = large
    if comm:
        line["comm"] = comm
    if parity:
        line["parity"] = parity
    if dense_bar:
        line["dense_solver_bar"] = dense_bar
    if sliding:
        line["e2e"]["sliding_window"] = sliding
    if cpu:
        line["cpu_baseline"] = cpu
    print(json.dumps(line))
    if world > 1:
        dist.barrier(); dist.destroy_process_group()


if __name__ == "__main__":
    main()
