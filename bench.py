#!/usr/bin/env python
"""bench.py -- HDL-64 frames/s of the LiDAR->tracks hot path (ground_removal -> component_clustering -> box_fitting ->
imm_ukf_jpda) on B200, next to the reference's own CPU implementation timed on the same host.

    python bench.py [--gpus N] [--steps K] [--warmup W]           # our CUDA path
    python bench.py ... --dump-outputs DIR                        # + the last timed step's boxes and live tracks as DIR/*.npy
    python bench.py --impl reference [--steps K] [--warmup W]     # the reference's sources (oracle/_ref) on the host CPU
    torchrun ... bench.py --gpus N ...                            # one rank per GPU, independent sensor streams (weak scaling)

One "step" = one 120,000-point synthetic HDL-64 frame (64 rings x 1875 azimuths, ~64 live tracks) through all four
stages, tracker state carried from frame to frame.  Frames are consecutive frames of ONE moving scene; every step reads
a different frame (the ring of W+K frames is larger than the 126 MB L2, so inputs never sit in L2 from the previous step).

Printed JSON (rank 0, one line):
  value     whole-job frames/s with the frames already resident in HBM (CUDA events around K steps, max over ranks)
  e2e       frames/s through the reference-facing C ABI on HOST buffers (lmot_frame_submit / lmot_frame_collect, pinned frames):
            every step copies its frame H2D, runs the four stages and reads boxes + track outputs back; timed by the C++ loop
            host/frame_loop.cpp (the reference's host language), the same loop from Python/ctypes is reported next to it
  roofline  ground_fused_kernel (the whole ground-removal stage in one cooperative launch, the only stage that streams
            the whole frame): algorithmic bytes per frame / its CUDA-event duration, vs the measured HBM peak
  cpu_baseline  the reference's own four entry points on a bounded sample of the same frames, one host thread
  parity_check  the CUDA path against the reference ON THE BENCH SCENE, frame by frame over the cpu_baseline sample: counts, boxes
            (bit-exact), trackManage (identical), UKF states of well-conditioned tracks (<= 1e-4); a failing check withholds `value`
  windows   --windows R repeats the K-step timed region R times on consecutive frames (default 1, so exactly K steps are timed;
            barrier + synchronize on both sides of each); `value`, `ms_per_step` and `e2e` are the MEDIAN window, `window_values`
            lists all of them
  latency_us    p50 / p99 per stage and per frame, one frame in flight (CUDA events) and at the pipeline's depth (host clock)
  batched_8x120k  BASELINE.json configs[3]: 8 sensor streams, one frame each per tick, one shared track table: ticks through
            lmot_batch_dev, and the ground_removal + CCL roofline of the two batched launches
"""
from __future__ import annotations

import argparse
import importlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # before CUDA initialises: one hardware queue per pipeline stream

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
PKG = "3d-lidar-multi-object-tracking_b200"

WORKLOAD = "hdl64_120k_64trk_full_pipeline"
SCENE = dict(n_objects=150, lattice_pitch=3.8, ped_fraction=0.65, seed=1)   # ~64 live tracks at steady state
KERNEL_NAMES = ("ground_fused+ccl", "tile_hist+seg_offsets", "scatter", "box_fit",
                "imm_predict_gate", "imm_update", "spawn_output")        # clustering runs in the ground kernel's last CTA (LMOT_FUSE_CCL=0: own launch)
KERNEL_NAMES_UNFUSED = ("ground_fused", "ccl_cluster") + KERNEL_NAMES[1:]
# dram__bytes_read.sum + dram__bytes_write.sum of ONE ground_fused_kernel launch at the bench workload (pipeline geometry, 74 CTAs,
# clustering fused into its tail), from the committed `ncu --set full` capture profiles/r2g_ncu_full_ground_pipeline.csv (2.07 MB read:
# the frame once, plus the polar grid and the bit planes; 0 bytes written: the 3.9 MB of output clouds stay in the 126 MB L2 within
# the measured launch)
TRAFFIC_NCU = 2.07e6
TRAFFIC_SOURCE = "constant from the committed ncu --set full capture profiles/r2g_ncu_full_ground_pipeline.csv (dram__bytes_read.sum + dram__bytes_write.sum of one launch), not measured by this run"
KERNELS_PER_FRAME = len(KERNEL_NAMES) + 2   # ground + clustering 1 (one launch) + box 3 + tracker 3, + the tracker's gate kernel + publish_kernel


def make_frames(synth, n_frames, seed_offset=0):
    cfg = synth.SceneConfig(**{**SCENE, "seed": SCENE["seed"] + seed_offset})
    ts, frames = [], []
    for t, pts in synth.frames(cfg, n_frames):
        ts.append(t)
        frames.append(pts)
    return ts, np.stack(frames)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def host_cpu_name():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


# ------------------------------------------------------------------------------------------- reference arm
def run_reference(args, synth):
    """The reference's own CPU implementation of the path (oracle/_ref = its unmodified sources, ruleBasedFilter in
    INTENDED mode like the GPU arm), single thread like the reference's ROS nodes; bounded sample per step."""
    from oracle import ref as oracle
    if oracle.have_ref("intended"):
        o, kind = oracle.RefOracle("intended"), "reference"
    else:
        o, kind = oracle.PortOracle("intended"), "port"
    K, W = args.steps, args.warmup
    ts, frames = make_frames(synth, W + K)
    o.tracker_reset()
    # The reference deploys as THREE single-threaded ROS nodes (ground | cluster | tracking) connected by topics, i.e. a
    # 3-stage pipeline on three cores.  Same here: one thread per node, queues instead of TCPROS (ctypes drops the GIL).
    import queue
    q1, q2 = queue.Queue(maxsize=4), queue.Queue(maxsize=4)
    stage = np.zeros(4)
    marks = {}

    def node_ground():
        for i in range(W + K):
            t0 = time.perf_counter()
            e, g = o.ground_remove(frames[i])
            if i >= W:
                stage[0] += time.perf_counter() - t0
            q1.put((i, e))
        q1.put(None)

    def node_cluster():
        while True:
            item = q1.get()
            if item is None:
                q2.put(None)
                return
            i, e = item
            t0 = time.perf_counter()
            grid, k = o.component_clustering(e); t1 = time.perf_counter()
            boxes, _ = o.box_fitting(e, grid, k); t2 = time.perf_counter()
            if i >= W:
                stage[1] += t1 - t0; stage[2] += t2 - t1
            q2.put((i, boxes))

    def node_tracking():
        while True:
            item = q2.get()
            if item is None:
                return
            i, boxes = item
            if i == W:
                marks["t0"] = time.perf_counter()
            t0 = time.perf_counter()
            o.tracker_step(boxes, ts[i])
            if i >= W:
                stage[3] += time.perf_counter() - t0
            marks["t1"] = time.perf_counter()

    threading.stack_size(256 * 1024 * 1024)   # the reference recurses per grid cell and passes 250 KB arrays by value
    threads = [threading.Thread(target=f) for f in (node_ground, node_cluster, node_tracking)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    t_total = marks["t1"] - marks["t0"]
    fps = K / t_total
    line = {
        "impl": "reference", "metric": "HDL-64 frames/sec (120K pts, 64 tracks)", "value": fps, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": K, "warmup": W, "ms_per_step": 1e3 * t_total / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32 points / f64 tracker", "data": "synthetic",
        "config": {"workload": WORKLOAD, "points_per_frame": int(frames.shape[1]), "scene": SCENE, "rule_filter": "INTENDED"},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": 3, "kind": kind, "host_cpu": host_cpu_name(), "host_cores": os.cpu_count(),
                         "sample": f"{K} consecutive frames of the workload after {W} warm-up frames; 3 threads = the reference's 3 ROS nodes pipelined; single-thread sum of stages = {1e3 * stage.sum() / K:.2f} ms/frame",
                         "stage_ms": {n: 1e3 * v / K for n, v in zip(("ground", "cluster", "box", "tracker"), stage)}},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------- shared track table (N > 1)
def shared_tracker_block(lmot, synth, rank, world, local_rank, ticks=10, warm=3):
    """N GPUs feeding ONE track table through the C++ shared tracker (include/lmot_shared.h, host/shared_tracker.cpp: NCCL
    all-gather of device box lists, tracker on rank 0, NCCL broadcast of count + table; nothing but a 4-byte count crosses a host).
      streams: every rank its own 120 k-point sensor stream, ONE tracker step per tick on the concatenation (configs[3] across GPUs)
      frames : ONE dense 1 M-point sensor, frame t*N + r on rank r, folded in frame order (BASELINE.json configs[4])
    Ticks are host-synchronous (the owner reads the outputs back every tick); time = host clock between barriers, max over ranks."""
    import torch
    import torch.distributed as dist
    uid = [lmot.shared_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    ctx = lmot.Lmot(device=local_rank)
    st = lmot.SharedTracker(ctx, rank, world, 0, uid[0])
    out = {"host_code": "host/shared_tracker.cpp (C++, NCCL C API) over liblmot.so", "owner_rank": 0}
    for mode in ("streams", "frames"):
        if mode == "streams":
            seq = list(synth.frames(synth.SceneConfig(**{**SCENE, "seed": SCENE["seed"] + rank}), warm + ticks))
            tick_ts = [s_[0] for s_ in seq]
            dt = 0.0
            workload = f"{world} sensor streams x 120 k points per tick"
        else:
            cfg = synth.dense_config(n_objects=400, lattice_pitch=2.3, ped_fraction=0.9, seed=11)
            seq = [(t_, p_[:1_000_000]) for t_, p_ in synth.frames(cfg, (warm + ticks) * world, only=lambda f: f % world == rank)]
            tick_ts = [synth.DT_US * (t * world + 1) for t in range(warm + ticks)]
            dt = synth.DT_US
            workload = f"one dense sensor, 1 M points per frame, {world} consecutive frames per tick (frame-sharded)"
        dev = [torch.from_numpy(np.ascontiguousarray(p_)).cuda() for _, p_ in seq]
        ctx.tracker_reset()
        m = lmot.SHARED_STREAMS if mode == "streams" else lmot.SHARED_FRAMES
        for t in range(warm):
            st.tick_dev(dev[t].data_ptr(), len(seq[t][1]), tick_ts[t], mode=m, frame_dt_us=dt)
        dist.barrier(); torch.cuda.synchronize()
        t0 = time.perf_counter()
        phases = np.zeros(4)
        for t in range(warm, warm + ticks):
            r = st.tick_dev(dev[t].data_ptr(), len(seq[t][1]), tick_ts[t], mode=m, frame_dt_us=dt)
            phases += np.array(list(st.last_us().values()))
        dist.barrier(); torch.cuda.synchronize()
        sec = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        ph = torch.tensor(phases / ticks, dtype=torch.float64, device="cuda")
        dist.all_reduce(sec, op=dist.ReduceOp.MAX)
        dist.all_reduce(ph, op=dist.ReduceOp.MAX)
        nt = torch.tensor([len(r["track_manage"]) if rank == 0 else 0, int((r["track_manage"] > 0).sum()) if rank == 0 else 0], device="cuda")
        dist.broadcast(nt, src=0)
        out[mode] = {"workload": workload, "ticks": ticks, "frames_per_s": world * ticks / float(sec[0]), "ms_per_tick": 1e3 * float(sec[0]) / ticks,
                     "tracks_in_table_end": int(nt[0]), "live_tracks_end": int(nt[1]), "table_bytes_broadcast_last_tick": int(nt[0]) * 1648,
                     "device_us_per_tick_max_over_ranks": dict(zip(("detect", "allgather_boxes", "tracker_owner", "broadcast_count_and_table"), (float(x) for x in ph)))}
        del dev
    st.close()
    ctx.close()
    return out


def run_shared_tracker(args, lmot, synth, rank, world, local_rank):
    """--shared-tracker: only the shared-table configuration (the default N > 1 line carries the same block next to the independent streams)."""
    blk = shared_tracker_block(lmot, synth, rank, world, local_rank, ticks=max(4, min(args.steps, 30)))
    if rank == 0:
        mode = blk[args.shared_tracker]
        print(json.dumps({
            "metric": "HDL-64 frames/sec (shared track table)", "value": mode["frames_per_s"], "unit": "frames/s", "n_gpus": world, "steps": mode["ticks"], "warmup": 3,
            "ms_per_step": mode["ms_per_tick"], "higher_is_better": True, "scaling": "weak" if args.shared_tracker == "streams" else "strong", "vs_baseline": None,
            "dtype": "f32 points / f64 tracker", "data": "synthetic", "config": {"workload": "shared_tracker_" + args.shared_tracker, **mode}, "shared_tracker": blk,
            "gpu_launches": KERNELS_PER_FRAME * mode["ticks"]}))


# ------------------------------------------------------------------------------------------- tracker in isolation (configs[2])
def tracker_stress(ctx, steps=40, warm=5):
    """BASELINE.json configs[2]: 1024 mature tracks (32x32 lattice, 8 m pitch) x 256 noisy detections, the tracker stage in
    isolation through lmot_track_step.  Every timed step starts from the SAME 1024-track table (re-loaded, untimed), so each
    step is exactly that workload; device time = CUDA events around the three tracker kernels."""
    rng = np.random.default_rng(0)
    T, M = 1024, 256
    gx, gy = np.meshgrid(np.arange(32) * 8.0 - 124.0, np.arange(32) * 8.0 - 124.0, indexing="ij")
    pos = np.stack([gx.ravel(), gy.ravel()], 1)
    half = np.array([[-1.0, -0.5], [-1.0, 0.5], [1.0, 0.5], [1.0, -0.5]])

    def boxes_at(p, noise):
        c = p + rng.normal(0, noise, p.shape)
        out = np.zeros((len(c), 8, 3), np.float32)
        for k in range(4):
            out[:, k, :2] = c + half[k]; out[:, k, 2] = -2.0
            out[:, 4 + k, :2] = c + half[k]; out[:, 4 + k, 2] = 0.0
        return out

    off = -0.63035 - np.pi / 2
    ctx.tracker_reset()
    ts = 0.0
    for _ in range(8):                      # frame 1 spawns, then every lattice site is observed until the tracks are mature
        ts += 1e5
        ctx.track_step(boxes_at(pos, 0.02), ts)
    state = ctx.tracker_dump()
    mature = int((state[:, 0] == 5).sum())
    det = boxes_at(pos[np.sort(rng.choice(T, M, replace=False))], 0.15)
    ctx.enable_timing(True)
    dev, host, kern = [], [], []
    for i in range(warm + steps):
        ctx.tracker_load(state, 1, ts, 0.0, off, off, -np.pi / 2)
        t0 = time.perf_counter()
        out = ctx.track_step(det, ts + 1e5)
        t1 = time.perf_counter()
        if i >= warm:
            dev.append(ctx.last_stage_ms()[3]); host.append(1e3 * (t1 - t0)); kern.append(ctx.last_kernel_ms()[:3])
    ctx.enable_timing(False)
    ctx.tracker_reset()
    dev_ms, host_ms = float(np.mean(dev)), float(np.mean(host))
    return {"workload": "imm_ukf_jpda stress: 1024 tracks x 256 detections, tracker stage in isolation (configs[2])",
            "tracks_in_table": int(len(state)), "mature_tracks": mature, "detections": M, "steps": steps,
            "device_ms_per_step": dev_ms, "track_updates_per_s_device": len(state) / (dev_ms * 1e-3),
            "host_call_ms_per_step": host_ms, "steps_per_s_through_c_abi": 1e3 / host_ms,
            "kernel_us": {n: float(1e3 * v) for n, v in zip(("imm_predict_gate", "imm_update", "spawn_output"), np.mean(np.array(kern), 0))}}


def run_native_e2e(frames, W, K, n_pts, rank, local_rank, world, windows=1, in_flight=0):
    """host/frame_loop (C++ submit / collect loop over the C ABI, pinned host frames) on this rank's GPU.
    -> (parsed JSON line, None) or (None, reason); never raises, no collectives inside."""
    import tempfile
    drv = os.path.join(ROOT, PKG, "host", "frame_loop")
    if not os.path.exists(drv):
        return None, "host/frame_loop not built"
    path = None
    try:
        where = None
        for cand in ("/dev/shm", tempfile.gettempdir(), ROOT):      # first place with room for the frames file (read once, into pinned memory)
            try:
                st_ = os.statvfs(cand)
                if os.access(cand, os.W_OK) and st_.f_bavail * st_.f_frsize > 1.2 * frames.nbytes * (world if cand == "/dev/shm" else 1):
                    where = cand
                    break
            except OSError:
                pass
        fd, path = tempfile.mkstemp(prefix=f"lmot_frames_r{rank}_", suffix=".bin", dir=where)
        os.close(fd)
        frames.tofile(path)
        env = dict(os.environ)
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        env["CUDA_VISIBLE_DEVICES"] = (vis.split(",")[local_rank] if vis else str(local_rank))
        out = subprocess.run([drv, path, str(len(frames)), str(n_pts), str(W), str(K), "100000", str(windows), str(in_flight)], env=env, stdout=subprocess.PIPE,
                             stderr=subprocess.PIPE, text=True, timeout=600)
        if out.returncode != 0:
            return None, f"frame_loop exit {out.returncode}: {out.stderr.strip()[:300]}"
        native = json.loads(out.stdout.strip().splitlines()[-1])
        if native.get("frames") != K * windows:
            return None, f"frame_loop collected {native.get('frames')} of {K * windows} frames"
        return native, None
    except Exception as ex:          # noqa: BLE001 -- a broken side measurement must not take the benchmark line down
        return None, f"{type(ex).__name__}: {ex}"
    finally:
        if path and os.path.exists(path):
            os.unlink(path)


# ------------------------------------------------------------------------------------------- parity on the bench scene
def _rel_err(a, b):
    scale = np.maximum(np.maximum(np.abs(a), np.abs(b)), 1e-3)
    err = np.abs(a - b) / scale
    err[np.isnan(a) & np.isnan(b)] = 0
    err[np.isnan(err)] = np.inf
    return err


def _pd_tracks(dump):
    """live tracks whose merged covariance is positive definite in the reference (an indefinite filter amplifies 1-ulp libm
    differences chaotically; the reference itself kills it a few frames later -- tests/test_tracker_gpu.py)"""
    ok = np.zeros(len(dump), bool)
    for i, d in enumerate(dump):
        if d[0] <= 0:
            continue
        P = d[24:49].reshape(5, 5)
        if np.all(np.isfinite(P)):
            ok[i] = np.linalg.eigvalsh((P + P.T) / 2).min() > 1e-9
    return ok


def cpu_baseline_and_parity(ctx, oracle_mod, frames, ts, n_sample, W, K, d_frames, n_pts):
    """The reference's four entry points, one host thread, on the first frames of the bench workload (timed) -- and, untimed, the
    CUDA path on the SAME frames compared with what the reference just produced."""
    o = oracle_mod.RefOracle("intended") if oracle_mod.have_ref("intended") else oracle_mod.PortOracle("intended")
    kind = "reference" if isinstance(o, oracle_mod.RefOracle) else "port"
    Wc = 10
    n = min(Wc + n_sample, len(frames))
    o.tracker_reset()
    ctx.tracker_reset()
    tt = 0.0
    chk = dict(frames=0, ok=True, first_failure=None, pd_excluded=0, tracks_compared=0, max_state_rel_err=0.0, state_frames=0)

    def fail(i, what):
        if chk["ok"]:
            chk["ok"], chk["first_failure"] = False, f"frame {i}: {what}"

    for i in range(n):
        t0 = time.perf_counter()
        e, g = o.ground_remove(frames[i]); grid, k = o.component_clustering(e); boxes, _ = o.box_fitting(e, grid, k)
        a = o.tracker_step(boxes, ts[i])
        if i >= Wc:
            tt += time.perf_counter() - t0
        ctx.frame_dev(d_frames[i].data_ptr(), n_pts, ts[i])
        r = ctx.frame_fetch()
        chk["frames"] += 1
        if (r["n_elevated"], r["n_ground"], r["num_cluster"]) != (len(e), len(g), k):
            fail(i, f"counts {(r['n_elevated'], r['n_ground'], r['num_cluster'])} vs reference {(len(e), len(g), k)}")
        elif r["boxes"].shape != boxes.shape or not np.array_equal(r["boxes"].view(np.uint32), boxes.view(np.uint32)):
            fail(i, "boxes differ (bit-exact bar)")
        elif not (np.array_equal(r["track_manage"], a["track_manage"]) and np.array_equal(r["is_static"], a["is_static"]) and np.array_equal(r["is_vis"], a["is_vis"])):
            fail(i, "trackManage / static / visible flags differ")
        if chk["ok"] and (i % 5 == 4 or i == n - 1):          # UKF states + covariances of every track, every 5th frame
            da, db = o.tracker_dump(), ctx.tracker_dump()
            if da.shape != db.shape or not np.array_equal(da[:, 0:4], db[:, 0:4]):
                fail(i, "track table integers differ")
            else:
                pd = _pd_tracks(da)
                chk["pd_excluded"] = max(chk["pd_excluded"], int((da[:, 0] > 0).sum() - pd.sum()))
                chk["tracks_compared"] = max(chk["tracks_compared"], int(pd.sum()))
                err = _rel_err(da[pd][:, 4:175], db[pd][:, 4:175])
                if err.size:
                    chk["max_state_rel_err"] = max(chk["max_state_rel_err"], float(err.max()))
                    if err.max() >= 1e-4:
                        fail(i, f"UKF state relative error {float(err.max()):.3g} > 1e-4")
                chk["state_frames"] += 1
    ns = n - Wc
    chk["bars"] = "counts + boxes bit-exact, trackManage/static/visible identical every frame; x/P/modeProb/zPred/S/K <= 1e-4 rel. every 5th frame on tracks whose reference covariance is positive definite (pd_excluded = most live tracks excluded on a frame)"
    cpu = {"value": ns / tt, "unit": "frames/s", "cores": 1, "kind": kind, "host_cpu": host_cpu_name(), "host_cores": os.cpu_count(),
           "sample": f"first {ns} frames of the same workload after {Wc} warm-up frames, single thread (the reference is single-threaded per node)"}
    return cpu, chk


def pct(a, q):
    a = np.sort(np.asarray(a, np.float64))
    return float(a[min(len(a) - 1, int(q * len(a)))]) if len(a) else None


# ------------------------------------------------------------------------------------------- batched ticks (configs[3])
def batched_block(lmot, synth, local_rank, stream, peak, ticks=12, warm=3, F=8):
    """BASELINE.json configs[3]: F sensor streams (scenes of different seeds), one frame each per tick, ONE track table.
    (a) ticks/s through lmot_batch_dev with the tick frames resident in HBM (ring of ticks > L2), (b) the ground_removal + CCL
    roofline of the two batched launches (lmot_batch_ground_ccl_dev), CUDA events on the launching stream."""
    import torch
    streams = [[p for _, p in synth.frames(synth.SceneConfig(**{**SCENE, "seed": 101 + s}), warm + ticks)] for s in range(F)]
    n = len(streams[0][0])
    dev = [torch.from_numpy(np.stack(st_)).cuda() for st_ in streams]
    ctx = lmot.Lmot(device=local_rank)
    ctx.set_stream(stream.cuda_stream)
    prepared = [ctx.batch_prepare([(dev[s_][t].data_ptr(), n) for s_ in range(F)]) for t in range(warm + ticks)]
    args = lambda t: prepared[t]
    # (b) roofline of ground + CCL
    for t in range(warm):
        ctx.batch_ground_ccl_dev(args(t))
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 3 * ticks
    e0.record(stream)
    for i in range(reps):
        ctx.batch_ground_ccl_dev(args(warm + i % ticks))
    e1.record(stream)
    torch.cuda.synchronize()
    gc_us = 1e3 * e0.elapsed_time(e1) / reps
    ne = nf = 0
    for s_ in range(F):
        r = ctx.ground_remove(streams[s_][warm]); ne += len(r["elevated"]); nf += len(r["elevated"]) + len(r["ground"])
    bytes_ground = F * (16 * n + 9600 * 24) + 16 * nf             # SURVEY.md §8d per frame, summed over the tick
    bytes_ccl = 20 * ne + F * 2 * 62500 * 4
    # (a) whole ticks, tracker included
    ctx.tracker_reset()
    for t in range(warm):
        ctx.batch_dev(args(t), 1e5 * (t + 1))
    ctx.flush(); torch.cuda.synchronize()
    e0.record(stream)
    for t in range(warm, warm + ticks):
        ctx.batch_dev(args(t), 1e5 * (t + 1))
    ctx.flush()
    e1.record(stream)
    torch.cuda.synchronize()
    tick_ms = e0.elapsed_time(e1) / ticks
    res = ctx.batch_fetch()
    ctx.enable_timing(True)
    ctx.tracker_reset()
    km = []
    for t in range(warm + ticks):
        ctx.batch_dev(args(t), 1e5 * (t + 1)); ctx.batch_fetch(want_boxes=False)
        if t >= warm:
            km.append(ctx.last_kernel_ms())
    ctx.enable_timing(False)
    names = ("ground_fused+ccl[8 frames]", "tile_hist+seg_offsets[8]", "scatter[8]", "box_fit[8]", "concat_boxes", "imm_predict_gate", "imm_update", "spawn_output")
    kus = np.mean(np.array(km), 0) * 1e3 if km and len(set(map(len, km))) == 1 else []
    if len(kus) == len(names) + 1:
        names = ("ground_fused[8 frames]", "ccl[8]") + names[1:]
    ctx.close()
    ach = (bytes_ground + bytes_ccl) / gc_us / 1e3
    return {"workload": f"{F} sensor streams x {n} points per tick, one shared track table (BASELINE.json configs[3])", "streams": F, "ticks": ticks,
            "frames_per_s": 1e3 * F / tick_ms, "ticks_per_s": 1e3 / tick_ms, "ms_per_tick": tick_ms,
            "live_tracks_end": int((res["track_manage"] > 0).sum()), "tracks_in_table_end": int(len(res["track_manage"])), "boxes_last_tick": int(len(res["boxes"])),
            "roofline": {"bound": "hbm", "kernels": "ground_removal + component clustering of the 8 frames: ONE launch (CTA groups own frames; the last CTA of a frame to finish labels its components)",
                         "algorithmic_bytes_ground": int(bytes_ground), "algorithmic_bytes_ccl": int(bytes_ccl), "us_per_tick": gc_us,
                         "achieved": ach, "unit": "GB/s", "peak": peak, "frac": ach / peak},
            "kernel_us_timing_mode": ({k_: float(v) for k_, v in zip(names, kus)} if len(kus) == len(names) else [float(v) for v in kus]),
            "l2_policy": f"every tick reads {F} frames no earlier tick of the window has read ({(warm + ticks) * F * n * 16 / 2**20:.0f} MiB ring)"}


# ------------------------------------------------------------------------------------------- our arm
PER_TRACK = ("targets", "vandyaw", "track_manage", "is_static", "is_vis")


def dump_outputs(out_dir, res):
    """One .npy per array of a frame result: float32 data as is, integer and flag arrays widened to float64 (exact).
    Per-track arrays keep the live tracks (trackManage != 0) and `track_index` gives their rows in the table: a dead
    slot stays in the append-only table with whatever state its filter ended in (NaN when it diverged, as in the
    reference), and the tracking node publishes only live tracks."""
    os.makedirs(out_dir, exist_ok=True)
    live = np.asarray(res["track_manage"]) != 0
    out = {**res, "track_index": np.flatnonzero(live)}
    for name, v in out.items():
        a = np.asarray(v)
        a = a[live] if name in PER_TRACK else a
        a = a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--windows", type=int, default=1, help="repetitions of the K-step timed window (each one times K more steps)")
    ap.add_argument("--impl", default="lmot", choices=["lmot", "reference"])
    ap.add_argument("--cpu-sample", type=int, default=60, help="frames of the CPU baseline / parity sample (rank 0, N=1)")
    ap.add_argument("--tracker-stress", type=int, default=40, help="timed steps of the 1024x256 tracker-only workload (0 = skip; rank 0, N=1)")
    ap.add_argument("--dense-frames", type=int, default=10, help="1M-point frames for the dense roofline measurement (0 = skip)")
    ap.add_argument("--batch-ticks", type=int, default=12, help="ticks of the batched 8 x 120 k configuration (0 = skip; rank 0)")
    ap.add_argument("--pipeline-depth", type=int, default=0, help="frames in flight inside the context (0 = the library default, 8)")
    ap.add_argument("--shared-ticks", type=int, default=8, help="N>1: ticks of the shared-track-table block (both modes) appended to the default line (0 = skip)")
    ap.add_argument("--shared-tracker", choices=["off", "streams", "frames"], default="off",
                    help="N>1 only: all ranks feed ONE track table (NCCL all_gather of boxes, tracker on rank 0, NCCL broadcast of the "
                         "outputs and of the table): 'streams' = N sensors per tick (configs[3]), 'frames' = one sensor, frames sharded "
                         "round-robin over the ranks (configs[4]).  Default: N independent streams, no collective.")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (boxes and live tracks, rank 0) to DIR/<name>.npy, float32 / float64")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    synth = importlib.import_module(PKG + ".synth")

    if args.impl == "reference":
        if rank == 0:
            run_reference(args, synth)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- there is no CPU fallback for the product path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lmot = importlib.import_module(PKG)
    K, W = args.steps, max(args.warmup, 3)
    R = max(1, args.windows)

    # ---- inputs: W + R*K consecutive frames of this rank's sensor stream, resident in HBM and in pinned host memory
    ts, frames = make_frames(synth, W + R * K, seed_offset=rank)
    n_pts = int(frames.shape[1])
    h_frames = torch.from_numpy(frames).pin_memory()
    d_frames = h_frames.cuda(non_blocking=True)
    torch.cuda.synchronize()
    ring_mb = d_frames.numel() * 4 / 2**20

    prm = lmot.default_params()
    if args.pipeline_depth > 0:
        prm.pipeline_depth = args.pipeline_depth
    ctx = lmot.Lmot(prm, device=local_rank)
    # a REAL stream: torch's default stream has handle 0, which lmot_set_stream reads as "use the context's own stream" --
    # CUDA events recorded on stream 0 would then not be ordered with the pipeline at all
    stream = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(stream)
    assert stream.cuda_stream != 0
    ctx.set_stream(stream.cuda_stream)
    frame_bytes = n_pts * 16

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)      # nvidia-smi samples every 100 ms across all timed passes below
    sampler.start()
    if args.shared_tracker != "off" and world > 1:
        ctx.close()
        run_shared_tracker(args, lmot, synth, rank, world, local_rank)
        dist.destroy_process_group()
        return

    # ---- (1) device-resident throughput: `value`.  R windows of exactly K steps, each bracketed by barrier + synchronize.
    ctx.tracker_reset()
    for i in range(W):
        ctx.frame_dev(d_frames[i].data_ptr(), n_pts, ts[i])
    # every timed step reads a frame no earlier step has read; with the default K the ring is 3x the 126 MB L2.  A short run
    # (ring < L2) could still find its frames in L2 from the upload above: push them out with a buffer larger than L2
    small_ring = ring_mb < 160
    if small_ring:
        l2_flush = torch.empty(192 * 2**20, dtype=torch.uint8, device="cuda")
        l2_flush.zero_()
    win_ms = []
    for r_ in range(R):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(W + r_ * K, W + (r_ + 1) * K):
            ctx.frame_dev(d_frames[i].data_ptr(), n_pts, ts[i])
        ctx.flush()                      # device-side join of the context's internal streams into the timing stream
        e1.record(stream)
        barrier()
        win_ms.append(e0.elapsed_time(e1))
    res_dev = ctx.frame_fetch()
    live_tracks = int((res_dev["track_manage"] > 0).sum())
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, res_dev)

    # ---- (2) per-stage device time of the same frames, ONE frame in flight (CUDA events on the launching stream)
    ctx.tracker_reset()
    ctx.enable_timing(True)
    per_stage, per_frame_dev = [], []
    kern_ms = None
    n_elev_sum = 0
    for i in range(W + K):
        ctx.frame_dev(d_frames[i].data_ptr(), n_pts, ts[i])
        r = ctx.frame_fetch(want_boxes=False)
        if i >= W:
            sm = ctx.last_stage_ms()
            per_stage.append(sm); per_frame_dev.append(sum(sm))
            km = np.array(ctx.last_kernel_ms())
            kern_ms = km if kern_ms is None or len(kern_ms) != len(km) else kern_ms + km
            n_elev_sum += r["n_elevated"] + r["n_ground"]
    ctx.enable_timing(False)
    per_stage = np.array(per_stage)
    stage_ms = per_stage.mean(0)
    # ... and the same, as the library runs in production: no event between the kernels (programmatic dependent launches stay on), two
    # CUDA events on the caller's stream per frame -- before lmot_frame_dev and behind lmot_flush (the stream's join with the frame)
    ctx.tracker_reset()
    n_lat = min(K, 100)
    lat_frame, lat_detect = [], []
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_lat)]
    for i in range(W + n_lat):
        a, b = evs[max(i - W, 0)]
        a.record(stream)
        ctx.frame_dev(d_frames[i].data_ptr(), n_pts, ts[i])
        ctx.flush()
        b.record(stream)
        ctx.frame_fetch(want_boxes=False)
        if i >= W:
            lat_frame.append(a.elapsed_time(b))
    for i in range(W + n_lat):
        a, b = evs[max(i - W, 0)]
        a.record(stream)
        ctx.detect_dev(d_frames[i].data_ptr(), n_pts)
        ctx.flush()
        b.record(stream)
        torch.cuda.synchronize()
        if i >= W:
            lat_detect.append(a.elapsed_time(b))
    n_f = n_elev_sum / K                                         # points that survive the range filter, per frame
    ground_bytes = 16 * n_pts + 16 * n_f + 9600 * 24             # SURVEY.md §8d: read XYZI + write both clouds + grid
    peak, peak_src = measured_peak_gbs()
    # roofline of the dominant streaming kernel at the bench workload: ground_fused_kernel launched back to back over the
    # K timed frames of the ring (each launch reads a different frame; ring > L2), CUDA events on the launching stream
    for i in range(W):
        ctx.ground_remove_dev(d_frames[i].data_ptr(), n_pts)
    torch.cuda.synchronize()
    r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    r0.record(stream)
    for i in range(W, W + K):
        ctx.ground_remove_dev(d_frames[i].data_ptr(), n_pts)
    r1.record(stream)
    torch.cuda.synchronize()
    ground_launch_ms = r0.elapsed_time(r1) / K
    achieved = ground_bytes / (ground_launch_ms * 1e-3) / 1e9

    # ---- (2b) the streaming stage on DENSE 1M-point frames (BASELINE.json configs[4] shape): the size at which an HBM
    # roofline fraction is meaningful for ground removal (at 120 k points the stage is launch / latency bound)
    dense = None
    if args.dense_frames > 0:
        dcfg = synth.dense_config(n_objects=SCENE["n_objects"], lattice_pitch=SCENE["lattice_pitch"], ped_fraction=SCENE["ped_fraction"], seed=7 + rank)
        dfr = []
        for _, p in synth.frames(dcfg, args.dense_frames):
            dfr.append(p[:1_000_000])
        d_dense = torch.from_numpy(np.stack(dfr)).cuda()
        nd = int(d_dense.shape[1])
        for i in range(3):
            ctx.ground_remove_dev(d_dense[i % len(dfr)].data_ptr(), nd)
        torch.cuda.synchronize()
        reps = 3 * len(dfr)
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record(stream)
        for i in range(reps):
            ctx.ground_remove_dev(d_dense[i % len(dfr)].data_ptr(), nd)
        g1.record(stream)
        torch.cuda.synchronize()
        ms = g0.elapsed_time(g1) / reps
        out = ctx.ground_remove(dfr[0])
        nf_d = len(out["elevated"]) + len(out["ground"])
        db = 16 * nd + 16 * nf_d + 9600 * 24
        dense = {"workload": "ground_removal stage on dense 1M-point frames", "points_per_frame": nd, "frames_in_ring": len(dfr),
                 "ring_mib": float(d_dense.numel() * 4 / 2**20), "avg_stage_ms": ms, "algorithmic_bytes_per_launch": db,
                 "how": "launches back to back on one stream (programmatic dependents, see roofline.how), every launch a different frame of the ring",
                 "achieved": db / (ms * 1e-3) / 1e9, "unit": "GB/s", "peak": peak, "frac": db / (ms * 1e-3) / 1e9 / peak}
        del d_dense

    # ---- (2c) BASELINE.json configs[3]: 8 streams x 120 k per tick, batched launches, one track table
    batched = None
    if rank == 0 and args.batch_ticks > 0:
        batched = batched_block(lmot, synth, local_rank, stream, peak, ticks=args.batch_ticks)

    # ---- H2D bandwidth of this box (context for `e2e`: every step moves the 1.92 MB frame over PCIe)
    hb0, hb1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tmp_d = torch.empty_like(d_frames[:8])
    hb0.record(stream)
    for _ in range(8):
        tmp_d.copy_(h_frames[:8], non_blocking=True)
    hb1.record(stream)
    torch.cuda.synchronize()
    h2d_gbs = 8 * tmp_d.numel() * 4 / (hb0.elapsed_time(hb1) * 1e-3) / 1e9
    # ... and one copy PER FRAME (what lmot_frame_submit issues): the per-copy set-up cost is not negligible at 1.9 MB
    hb0.record(stream)
    for i in range(64):
        tmp_d[i % 8].copy_(h_frames[i % (W + K)], non_blocking=True)
    hb1.record(stream)
    torch.cuda.synchronize()
    h2d_frame_us = 1e3 * hb0.elapsed_time(hb1) / 64
    del tmp_d

    # ---- (3) end to end through the C ABI with host buffers: `e2e` (Python loop: one window; the C++ loop below is the figure)
    ctx.tracker_reset()
    h_np = h_frames.numpy()
    depth = min(int(ctx.params.result_ring) - 1, 2 * int(ctx.params.pipeline_depth))     # frames the host may be ahead of the results it has read back
    for i in range(W):
        ctx.frame(h_np[i], ts[i])
    barrier()
    t0 = time.perf_counter()
    d2h = 0
    collected = 0
    t_submit = t_collect = 0.0
    in_flight = 0
    for i in range(W, W + R * K):        # every step: H2D of its frame; every result is read back inside the region
        if in_flight == depth:
            tc = time.perf_counter(); r = ctx.frame_collect(); t_collect += time.perf_counter() - tc
            collected += 1; in_flight -= 1
        tc = time.perf_counter(); ctx.frame_submit(h_np[i], ts[i]); t_submit += time.perf_counter() - tc
        in_flight += 1
    while in_flight > 0:
        tc = time.perf_counter(); r = ctx.frame_collect(); t_collect += time.perf_counter() - tc
        collected += 1; in_flight -= 1
    barrier()
    e2e_py_s = (time.perf_counter() - t0) / R
    assert collected == R * K
    d2h = 16 * 4 + r["boxes"].size * 4 + len(r["track_manage"]) * (12 + 16 + 4 + 1 + 1) + r["vis_bb"].size * 4
    py_live = int((r["track_manage"] > 0).sum())

    # ---- (3b) the same loop in the reference's host language: host/frame_loop.cpp (C++ over the same two C-ABI calls, pinned host
    # frames, every result collected, R windows of K steps with lmot_sync on both sides).  This is `e2e`.
    barrier()
    native, native_err = run_native_e2e(frames, W, K, n_pts, rank, local_rank, world, windows=R)
    if native is not None and not (native["tracks_last"] == len(r["track_manage"]) and native["live_tracks_last"] == py_live):
        # same frames, same tracker: the native loop must end in the state the Python loop ended in
        native_err, native = f"frame_loop ended in a different tracker state: {native} vs {len(r['track_manage'])} tracks / {py_live} live", None
    if native is not None:
        e2e_s, d2h = native["e2e_s"], native["d2h_bytes_last"]
    else:
        e2e_s = e2e_py_s             # (reported as such: e2e.driver says which loop was timed, e2e.native_driver_error why)
    # ... and once more with ONE frame in flight: the latency of a frame through the host API (submit call -> results copied out)
    lat1 = None
    if rank == 0:
        lat1, _ = run_native_e2e(frames, W, min(K, 100), n_pts, rank, local_rank, world, windows=1, in_flight=1)
    clocks = sampler.stop()

    # ---- aggregate over ranks (max time per window, then the median window)
    t = torch.tensor(win_ms + [e2e_s * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    win_max = [float(x) for x in t[:R]]
    dev_ms_max, e2e_ms_max = float(np.median(win_max)) if R % 2 else float(sorted(win_max)[(R - 1) // 2]), float(t[R])
    value = world * K / (dev_ms_max * 1e-3)
    e2e = world * K / (e2e_ms_max * 1e-3)

    cpu_baseline = parity = None
    if rank == 0 and world == 1 and args.cpu_sample > 0:
        from oracle import ref as oracle     # the checker / baseline, never the measured product
        cpu_baseline, parity = cpu_baseline_and_parity(ctx, oracle, frames, ts, args.cpu_sample, W, K, d_frames, n_pts)

    stress = None
    if rank == 0 and world == 1 and args.tracker_stress > 0:
        stress = tracker_stress(ctx, steps=args.tracker_stress)

    # ---- N > 1: the one real exchange step of the path, several GPUs feeding ONE track table (collective: every rank takes part)
    shared = None
    if world > 1 and args.shared_ticks > 0:
        shared = shared_tracker_block(lmot, synth, rank, world, local_rank, ticks=args.shared_ticks)

    if rank == 0:
        stage_names = ("ground", "cluster", "box", "tracker")
        latency = {
            "one_frame_in_flight_device": {"frame": {"p50": 1e3 * pct(per_frame_dev, 0.5), "p99": 1e3 * pct(per_frame_dev, 0.99)},
                                           **{n: {"p50": 1e3 * pct(per_stage[:, j], 0.5), "p99": 1e3 * pct(per_stage[:, j], 0.99)} for j, n in enumerate(stage_names)},
                                           "how": f"CUDA events around the stages of {K} frames submitted one at a time (lmot_frame_dev + fetch), device time, us"},
            "one_frame_in_flight_device_production": {"frame": {"p50": 1e3 * pct(lat_frame, 0.5), "p99": 1e3 * pct(lat_frame, 0.99)},
                                                      "detection": {"p50": 1e3 * pct(lat_detect, 0.5), "p99": 1e3 * pct(lat_detect, 0.99)},
                                                      "how": f"{n_lat} frames one at a time, timing mode OFF (no event between the kernels, programmatic dependent launches on): two CUDA events on the caller's stream per frame, around lmot_frame_dev + lmot_flush (all four stages) and around lmot_detect_dev (ground removal + clustering + box fitting); the per-stage figures above pay ~4 us of event record per kernel and run without programmatic launches"},
            "one_frame_in_flight_host_api": ({"frame": {"p50": lat1["latency_us_p50"], "p99": lat1["latency_us_p99"]},
                                              "how": "host clock, lmot_frame_submit call -> results copied out by lmot_frame_collect, H2D of the frame included (host/frame_loop.cpp, in_flight = 1)"} if lat1 else None),
            "pipelined_host_api": ({"frame": {"p50": native["latency_us_p50"], "p99": native["latency_us_p99"]}, "in_flight": native["in_flight"],
                                    "how": "same clock with the pipeline full: in_flight frames submitted ahead of the results read back (queueing included)"} if native else None),
        }
        ok = parity is None or parity["ok"]
        line = {
            "metric": "HDL-64 frames/sec (120K pts, 64 tracks)", "value": (value if ok else None), "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": dev_ms_max / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "windows": R, "window_values": [world * K / (w_ * 1e-3) for w_ in win_max],
            "dtype": "f32 points / f64 tracker", "data": "synthetic",
            "config": {"workload": WORKLOAD, "points_per_frame": n_pts, "scene": SCENE, "live_tracks_end": live_tracks,
                       "tracks_in_table_end": int(len(res_dev["track_manage"])), "rule_filter": "INTENDED",
                       "parallelism": f"{world} independent sensor stream(s), one per GPU, no collective on the data path",
                       "pipeline_depth": int(ctx.params.pipeline_depth), "result_ring": int(ctx.params.result_ring),
                       "l2_policy": (f"every step reads a different frame of a {ring_mb:.0f} MiB ring (> 126 MB L2)" if not small_ring else
                                     f"every step reads a different frame of a {ring_mb:.0f} MiB ring, L2 flushed (192 MiB written) before the first timed window")},
            "parity_check": parity,
            "e2e": {"value": (e2e if ok else None), "unit": "frames/s", "h2d_bytes_per_step": frame_bytes, "d2h_bytes_per_step": int(d2h),
                    "windows": (native["windows"] if native else 1), "window_values": ([world * K / w_ for w_ in native["window_s"]] if native else None),
                    "pinned_h2d_gbs_this_box": h2d_gbs, "h2d_us_per_frame_copy_this_box": h2d_frame_us, "pcie_bound_frames_per_s": 1e6 / h2d_frame_us,
                    "driver": ("host/frame_loop.cpp: C++ loop over lmot_frame_submit / lmot_frame_collect, pinned host frames" if native else "python ctypes loop"),
                    "native_driver_error": native_err,
                    "host_us_per_step": ({"submit": native["submit_us_per_frame"], "collect_incl_wait": native["collect_us_per_frame"]} if native
                                         else {"submit": 1e6 * t_submit / (R * K), "collect_incl_wait": 1e6 * t_collect / (R * K)}),
                    "python_ctypes_loop": {"value": world * K / e2e_py_s, "unit": "frames/s", "note": "same two calls from a Python loop (this rank)",
                                           "host_us_per_step": {"submit": 1e6 * t_submit / (R * K), "collect_incl_wait": 1e6 * t_collect / (R * K)}}},
            "gpu_launches": KERNELS_PER_FRAME * K * R,
            "clocks": clocks,
            "latency_us": latency,
            "roofline": {"bound": "hbm", "kernel": "ground_fused_kernel (the whole ground_removal stage: bin + polar grid + classify/partition, one launch)",
                         "achieved": achieved, "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": achieved / peak,
                         "algorithmic_bytes_per_launch": ground_bytes, "avg_launch_ms": float(ground_launch_ms),
                         "launches_timed": K, "traffic": TRAFFIC_NCU, "traffic_source": TRAFFIC_SOURCE,
                         "how": "K launches back to back on one stream, CUDA events around the K; consecutive launches are chained as programmatic dependents (no event between them: the next launch's CTAs set up while the previous grid drains and wait in griddepcontrol.wait)",
                         "note": "latency bound at 120 k points: 3.84 MB is 0.6 us of HBM time, the kernel needs two frame-wide barriers and one count exchange; see roofline_dense_1m and batched_8x120k.roofline"},
            "stage_ms": {n: float(v) for n, v in zip(stage_names, stage_ms)},
            "kernel_us_warm": ({n: float(1e3 * v / K) for n, v in zip(KERNEL_NAMES if len(kern_ms) == len(KERNEL_NAMES) else KERNEL_NAMES_UNFUSED, kern_ms)}
                               if kern_ms is not None and len(kern_ms) in (len(KERNEL_NAMES), len(KERNEL_NAMES_UNFUSED)) else None),
            "roofline_dense_1m": dense,
            "batched_8x120k": batched,
            "tracker_stress_1024x256": stress,
            "shared_tracker": shared,
            "cpu_baseline": cpu_baseline,
        }
        print(json.dumps(line))
        if not ok:
            sys.stderr.write("bench.py: parity_check FAILED (" + str(parity["first_failure"]) + ") -- value withheld\n")
    ctx.close()
    if world > 1:
        dist.destroy_process_group()
    if rank == 0 and parity is not None and not parity["ok"]:
        raise SystemExit(1)


if __name__ == "__main__":
    main()
