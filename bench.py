#!/usr/bin/env python
"""Headline benchmark: clip-frames/s of DragPoser's per-frame latent optimisation at fixed
100 iterations, 4096 synthetic clips per GPU, 6 trackers (BASELINE.json metric / configs[3]).

A "step" is one frame of the hot path for every clip of the batch: temporal-predictor
target (window 0 => every frame) + 100 x {decode, FK, tracker loss, adjoint, decoder
backward, latent Adam} + frame epilogue.  `value` has the tracker streams resident in
HBM; `e2e` goes through the host-buffer API (H2D of the step's targets and D2H of the
poses inside the timed region).  At N = 1 the same line also carries BASELINE config 3
(`configs["3trk_var_4096"]`: head + hands, variable tracker mask, window 16) and the
B = 1 latency of the DragPoserDLL C ABI (`latency`).  `--impl reference` times the CPU
oracle port of the reference loop (the reference is Python and cannot travel to the GPU
box) on all host cores.  One JSON line on stdout (rank 0).
`--dump-outputs DIR` also writes the results of the last timed step (DIR/pose.npy,
DIR/global_pos.npy; DIR/3trk_var_*.npy for config 3): the inputs are seeded, so two
builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden", "model_dancedb.npz")
FLOP_PER_CLIP_ITER = 35520.0      # decoder fwd + bwd-data GEMMs, folded 24->40->60->92 (SURVEY 8(d))
HBM_BYTES_PER_CLIP_FRAME = 1300.0  # algorithmic state + tracker + result bytes (SURVEY 8(d))
MAX_ITER = 100
# Per-core speed of the oracle port relative to the UNMODIFIED reference loop, measured in the build container (the reference
# tree does not travel to the GPU box): scripts/port_vs_reference.py, 1 clip x 3 frames x 100 fixed iterations, one thread.
PORT_VS_REFERENCE_PER_CORE = {"ratio": 1.44, "port_frames_per_s": 4.15, "reference_frames_per_s": 2.89,
                              "how": "scripts/port_vs_reference.py in the build container (8-vCPU Xeon, torch 2.11 CPU), one thread, "
                                     "same clip and targets; the port is the faster of the two, so GPU / port ratios understate GPU / reference"}

KERNEL_NAMES = {
    1: "dp_frame_simt_kernel (persistent per-frame loop; fp32 CUDA-core decoder)",
    3: "dp_frame_tc16_kernel (persistent per-frame loop; decoder GEMMs on tcgen05, fp16x2 split, weights in tensor memory)",
}
# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the dominant kernel, from the ncu --set full capture whose
# summary is committed under profiles/ (keyed by decoder path, clips per GPU, tracker config); null for other configurations
NCU_DRAM_BYTES_PER_LAUNCH = {(3, 4096, "6"): 2472448}  # profiles/r2_frame_kernel.md (final capture): 2 468 864 read + 3 584 written


def fixed_opts(cfg):
    return dict(stop_eps_pos=-1.0, stop_eps_rot=-1.0, max_iter=MAX_ITER, min_loss_incr=-float("inf"), learning_rate=1e-2,
                lambda_rot=1, lambda_temporal=cfg.lambda_temporal, temporal_future_window=cfg.temporal_future_window,
                joint_adjustment_indices=cfg.joint_adjustment, joint_adjustment_weight=cfg.joint_adjustment_weight)


def get_config(name):
    from dragposer_b200 import synthetic

    return synthetic.config_3_trackers() if name == "3" else synthetic.config_6_trackers()


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device, n_gpus=1):
        self.rows, self.proc = [], None
        self.device = str(device) if n_gpus == 1 else ",".join(str(i) for i in range(n_gpus))  # every GPU of the job

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.device)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6), ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                    if r[col].lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- CPU reference arm
def _cpu_worker(args):
    """One single-threaded worker = one clip, like the reference (B = 1, CPU, fp32)."""
    idx, n_warm, n_timed, tracker_cfg = args
    import torch

    torch.set_num_threads(1)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import dragposer_port as port
    from dragposer_b200 import model, synthetic

    cfg = get_config(tracker_cfg)
    pm = model.load_folded_npz(GOLDEN)
    npz = np.load(GOLDEN)
    wl = synthetic.make_workload(pm, npz["offsets"], cfg, 1, n_warm + n_timed, first_clip=idx)
    drag = port.PortDragPose(port.PortWeights(npz), model.random_temporal_state(2222))
    drag.set_initial_state(wl["latent0"], np.zeros((1, 3)), [[1.0, 0, 0, 0]], np.zeros((1, 6)))
    o = fixed_opts(cfg)
    kw = dict(stop_eps_pos=o["stop_eps_pos"], stop_eps_rot=o["stop_eps_rot"], max_iter=o["max_iter"], min_loss_incr=o["min_loss_incr"],
              learning_rate=o["learning_rate"], lambda_rot=1.0, lambda_temporal=o["lambda_temporal"],
              temporal_future_window=o["temporal_future_window"], joint_adjustment=o["joint_adjustment_indices"],
              joint_adjustment_weight=o["joint_adjustment_weight"])
    t0 = None
    for t in range(n_warm + n_timed):
        if t == n_warm:
            t0 = time.perf_counter()
        drag.run(wl["tgt_pos"][t], wl["tgt_rot"][t], wl["joints"], wl["weights"], **kw)
    return time.perf_counter() - t0


def cpu_reference(n_warm, n_timed, tracker_cfg, cores=None):
    """All host cores, one clip per core; returns (clip-frames/s, cores, sample text)."""
    import multiprocessing as mp

    cores = cores or os.cpu_count() or 1
    ctx = mp.get_context("spawn")
    with ctx.Pool(cores) as pool:
        times = pool.map(_cpu_worker, [(i, n_warm, n_timed, tracker_cfg) for i in range(cores)])
    value = cores * n_timed / max(times)
    sample = (f"{cores} clips x {n_timed} frames (one single-threaded process per core, B=1 like the reference), "
              f"{MAX_ITER} fixed iterations, {tracker_cfg} trackers, predictor every frame, after {n_warm} warm-up frames")
    return value, cores, sample


# ----------------------------------------------------------------------------- single-frame latency (second half of the metric)
LAT_POS = (-2.6648, 0.9977, 3.7518)
LAT_ROT = (0.6381, 0.0078, -0.7698, 0.0110)


def quat_from_matrix(m):
    """(…,3,3) rotation matrices -> (…,4) wxyz quaternions (largest-component selection)."""
    m = np.asarray(m, np.float64)
    out = np.empty(m.shape[:-2] + (4,), np.float64)
    flat_m, flat_o = m.reshape(-1, 3, 3), out.reshape(-1, 4)
    for i, r in enumerate(flat_m):
        tr = r[0, 0] + r[1, 1] + r[2, 2]
        if tr > 0:
            s = 2.0 * np.sqrt(1.0 + tr)
            q = (0.25 * s, (r[2, 1] - r[1, 2]) / s, (r[0, 2] - r[2, 0]) / s, (r[1, 0] - r[0, 1]) / s)
        elif r[0, 0] > r[1, 1] and r[0, 0] > r[2, 2]:
            s = 2.0 * np.sqrt(1.0 + r[0, 0] - r[1, 1] - r[2, 2])
            q = ((r[2, 1] - r[1, 2]) / s, 0.25 * s, (r[0, 1] + r[1, 0]) / s, (r[0, 2] + r[2, 0]) / s)
        elif r[1, 1] > r[2, 2]:
            s = 2.0 * np.sqrt(1.0 + r[1, 1] - r[0, 0] - r[2, 2])
            q = ((r[0, 2] - r[2, 0]) / s, (r[0, 1] + r[1, 0]) / s, 0.25 * s, (r[1, 2] + r[2, 1]) / s)
        else:
            s = 2.0 * np.sqrt(1.0 + r[2, 2] - r[0, 0] - r[1, 1])
            q = ((r[1, 0] - r[0, 1]) / s, (r[0, 2] + r[2, 0]) / s, (r[1, 2] + r[2, 1]) / s, 0.25 * s)
        flat_o[i] = q
    return out.astype(np.float32)


def latency_stream(n_frames):
    """The moving target stream both latency arms replay: clip 0 of the synthetic 6-tracker workload (latent random walk, SURVEY
    8d), tracker positions relative to the root and tracker rotations (matrices for the port, quaternions for the C ABI)."""
    from dragposer_b200 import model, synthetic

    cfg = synthetic.config_6_trackers()
    pm = model.load_folded_npz(GOLDEN)
    npz = np.load(GOLDEN)
    wl = synthetic.make_workload(pm, npz["offsets"], cfg, 1, n_frames)
    return wl, quat_from_matrix(wl["tgt_rot"][:, 0])


def _stats(ms):
    t = np.sort(np.asarray(ms))
    pick = lambda q: float(t[min(len(t) - 1, int(len(t) * q))])
    return {"p50_ms": pick(0.5), "p90_ms": pick(0.9), "p99_ms": pick(0.99), "max_ms": float(t[-1]), "mean_ms": float(t.mean()), "calls": int(len(t))}


def dll_latency(calls=1000):
    """Wall-clock of drag_pose through the DragPoserDLL C ABI, B = 1, host buffers in and out (SURVEY 8d), on the moving synthetic
    stream: the Unity settings (MaxIter 5 / 10, lr 0.01, window 16, the reference session's stop thresholds), the offline budget
    (MaxIter 100 with those thresholds) and a FIXED 100 iterations (thresholds and min_loss_incr off).  Frames on which the
    temporal predictor runs (every 16th) are reported separately from the others; `all` mixes them as a session sees them."""
    import ctypes as C
    import tempfile

    from dragposer_b200 import build, export_model

    class F3(C.Structure):
        _fields_ = [("x", C.c_float), ("y", C.c_float), ("z", C.c_float)]

    class Q4(C.Structure):
        _fields_ = [("w", C.c_float), ("x", C.c_float), ("y", C.c_float), ("z", C.c_float)]

    class F2(C.Structure):
        _fields_ = [("x", C.c_float), ("y", C.c_float)]

    if not os.path.exists(build.DLL_SO):  # built by build(); the benchmark compiles nothing (its tree may be read-only)
        raise SystemExit(f"bench.py: {build.DLL_SO} is missing: build it first (python -m dragposer_b200.build)")
    lib = C.CDLL(build.DLL_SO)
    V = C.c_void_p
    lib.init_drag_poser.restype = V
    lib.set_reference_skeleton.argtypes = [V, C.c_char_p]
    lib.load_models.argtypes = [V, C.c_char_p]
    lib.set_mask_and_weights.argtypes = [V, C.POINTER(C.c_float), C.POINTER(F2)]
    lib.init_drag_model.argtypes = [V, F3, Q4]
    lib.set_optim_params.argtypes = [V, C.c_float, C.c_float, C.c_int, C.c_float]
    lib.set_lambdas.argtypes = [V, C.c_float, C.c_float, C.c_int]
    lib.set_global_pos.argtypes = [V, F3]
    lib.drag_pose.argtypes = [V, C.c_int, C.POINTER(F3), C.POINTER(Q4), C.POINTER(Q4), C.POINTER(F3)]
    lib.destroy_drag_poser.argtypes = [V]
    lib.dp_last_status.argtypes = [V]
    lib.dp_get_last_iterations.argtypes = [V]
    lib.dp_set_min_loss_increment.argtypes = [V, C.c_double]
    g = np.load(os.path.join(ROOT, "tests", "golden", "ref_rundrag.npz"))
    window = 16
    n_fixed = max(160, calls // 4)
    wl, quats = latency_stream(calls + 24)
    out = {"boundary": "DragPoserDLL C ABI drag_pose, B = 1, 6 trackers, host buffers in/out, window 16",
           "stream": "clip 0 of the synthetic 6-tracker workload (latent random walk), one new target set per call",
           "predictor": "every 16th frame needs new targets (5 decoder passes, ~70 kernels, 0.41 ms on the device as a replayed CUDA graph); "
                        "its inputs end three frames in the past, so the engine issues that call three frames early on a side stream "
                        "(dp_engine.cu:run_one, DP_PRED_PREFETCH=0 turns it off) and 'predictor_frames' only wait for what is left of it: "
                        "nothing in this per-frame call sequence (DragPoser.cs:137-173; the un-timed setter calls between two drag_pose "
                        "calls are part of it), 0.28 ms for a caller that issues drag_pose back to back (scripts/latency_by_index.py); "
                        "without the early call: p50 0.56 ms on those frames (start of round 2), 0.45 ms with the graph alone"}
    settings = (("max_iter_5", 5, False, calls), ("max_iter_10", 10, False, calls), ("max_iter_100", 100, False, max(200, calls // 2)),
                ("fixed_100_iterations", 100, True, n_fixed))
    with tempfile.TemporaryDirectory() as d:
        export_model.export(GOLDEN, os.path.join(d, "model.dpm"), allow_random_temporal=True)
        for name, max_iter, fixed, n in settings:
            h = lib.init_drag_poser()
            lib.set_reference_skeleton(h, os.path.join(ROOT, "tests", "golden", "skeleton22.bvh").encode())
            lib.load_models(h, d.encode())
            mask = (C.c_float * 22)(*g["mask"].tolist())
            weights = (F2 * 22)(*[F2(*w) for w in g["weights"].tolist()])
            lib.init_drag_model(h, F3(*LAT_POS), Q4(*LAT_ROT))
            if lib.dp_last_status(h) != 0:
                raise SystemExit("bench.py: DragPoserDLL session failed to start")
            if fixed:
                lib.dp_set_min_loss_increment(h, -float("inf"))
            pos = [(F3 * 6)(*[F3(*p) for p in wl["tgt_pos"][t, 0].tolist()]) for t in range(n + 20)]
            rot = [(Q4 * 6)(*[Q4(*q) for q in quats[t].tolist()]) for t in range(n + 20)]
            res, gp = (Q4 * 22)(), (F3 * 1)()
            times, iters = [], []
            for i in range(n + 20):  # the per-frame call sequence of DragPoser.cs:137-173
                lib.set_mask_and_weights(h, mask, weights)
                if fixed:
                    lib.set_optim_params(h, -1.0, -1.0, max_iter, 0.01)
                else:
                    lib.set_optim_params(h, 0.01 * 0.01, 0.01, max_iter, 0.01)
                lib.set_lambdas(h, 1, 0.02, window)
                t0 = time.perf_counter()
                lib.drag_pose(h, 6, pos[i], rot[i], res, gp)
                times.append((time.perf_counter() - t0) * 1e3)
                iters.append(lib.dp_get_last_iterations(h))
                lib.set_global_pos(h, gp[0])
            lib.destroy_drag_poser(h)
            times, iters = np.array(times[20:]), np.array(iters[20:])
            pred = (np.arange(20, n + 20) % window) == 0  # frames on which current_index == 0: the predictor runs (5 decoder passes)
            out[name] = {"all": _stats(times), "predictor_frames": _stats(times[pred]), "other_frames": _stats(times[~pred]),
                         "mean_iterations": float(iters.mean())}
    out["p50_ms"] = out["max_iter_5"]["all"]["p50_ms"]
    return out


def port_latency(calls=30):
    """The reference arm of the latency metric: the oracle port's DragPose.run, B = 1, one core, same stream and parameters."""
    import torch

    torch.set_num_threads(1)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import dragposer_port as port
    from dragposer_b200 import model

    npz = np.load(GOLDEN)
    wl, _ = latency_stream(calls + 3)
    out = {"boundary": "oracle port of DragPose.run, B = 1, 6 trackers, one core, window 16",
           "stream": "clip 0 of the synthetic 6-tracker workload (latent random walk), one new target set per call"}
    for name, max_iter, fixed, n in (("max_iter_5", 5, False, calls), ("max_iter_10", 10, False, calls),
                                     ("fixed_100_iterations", 100, True, max(6, calls // 5))):
        drag = port.PortDragPose(port.PortWeights(npz), model.random_temporal_state(2222))
        drag.set_initial_state(wl["latent0"], np.zeros((1, 3)), [[1.0, 0, 0, 0]], np.zeros((1, 6)))
        times = []
        for t in range(n + 3):
            t0 = time.perf_counter()
            drag.run(wl["tgt_pos"][t], wl["tgt_rot"][t], wl["joints"], wl["weights"], stop_eps_pos=-1.0 if fixed else 1e-4,
                     stop_eps_rot=-1.0 if fixed else 1e-2, max_iter=max_iter, min_loss_incr=-float("inf") if fixed else 1e-5,
                     learning_rate=1e-2, lambda_rot=1.0, lambda_temporal=0.02, temporal_future_window=16, joint_adjustment=None,
                     joint_adjustment_weight=0.0)
            times.append((time.perf_counter() - t0) * 1e3)
        out[name] = {"all": _stats(times[3:])}
    out["p50_ms"] = out["max_iter_5"]["all"]["p50_ms"]
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = get_config(args.trackers)
    n_warm, n_timed = max(1, min(args.warmup, 1)), max(1, args.steps)
    value, cores, sample = cpu_reference(n_warm, n_timed, args.trackers)
    config = workload_config(args, cfg, args.clips * args.gpus)
    # what this arm actually ran: per-clip CPU cost does not depend on how many clips exist, so the bounded sample stands for the
    # workload above -- but the sample is the sample
    config["cpu_sample"] = {"clips": cores, "frames_per_clip": n_timed, "warmup_frames": n_warm, "processes": cores, "threads_per_process": 1}
    line = {
        "impl": "reference", "metric": "clip-frames/sec (fixed 100 opt iters)", "value": value, "unit": "clip-frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * cores / value,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config,
        "cpu_baseline": {"value": value, "unit": "clip-frames/s", "cores": cores, "kind": "port", "sample": sample,
                         "port_vs_unmodified_reference_per_core": PORT_VS_REFERENCE_PER_CORE},
        "e2e": {"value": value, "unit": "clip-frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not args.no_latency:
        line["latency"] = port_latency()
    print(json.dumps(line))


def workload_config(args, cfg, clips_total, trackers=None):
    trackers = trackers or args.trackers
    return {"workload": f"{trackers}-tracker synthetic streams (SURVEY 8d){', variable tracker mask' if trackers == '3' else ''}, model_dancedb "
                        f"weights, seed-2222 random-init predictor, window {cfg.temporal_future_window}, fixed {MAX_ITER} iterations",
            "clips_per_gpu": args.clips, "clips_total": clips_total, "trackers": int(trackers), "max_iter": MAX_ITER,
            "l2": "flushed between timed steps (256 MiB write)", "parallelism": f"clip-shard x{args.gpus}"}


# ----------------------------------------------------------------------------- GPU arm
def measure(args, trackers, K, W, rank, world, dev, local, clocks=None):
    """Device-timed and end-to-end throughput of one workload (tracker config) at args.clips clips per GPU; returns a dict."""
    import torch
    import torch.distributed as dist

    from dragposer_b200 import dist as dpdist
    from dragposer_b200 import model, synthetic
    from dragposer_b200.engine import BatchedDragPose, RunOptions

    cfg = get_config(trackers)
    pm = model.load_folded_npz(GOLDEN)
    offsets = np.load(GOLDEN)["offsets"]
    tm = model.temporal_from_state(model.random_temporal_state(2222))
    B = args.clips
    n_total = B * world
    T = W + K
    variable = trackers == "3"
    wl = synthetic.make_workload(pm, offsets, cfg, B, T, first_clip=rank * B, variable_mask=variable)
    eng = BatchedDragPose(pm, offsets, tm, B, device=local)
    eng.set_initial_state(wl["latent0"], np.zeros((B, 3)), np.tile([[1.0, 0, 0, 0]], (B, 1)), np.zeros((B, 6)))
    opts = RunOptions(decoder_path=args.decoder_path, **fixed_opts(cfg))
    E = wl["tgt_pos"].shape[2]
    d_tp = torch.from_numpy(wl["tgt_pos"]).to(dev)
    d_tr = torch.from_numpy(wl["tgt_rot"]).to(dev)
    if variable:
        d_j, d_w = torch.from_numpy(wl["joints_tb"]).to(dev), torch.from_numpy(wl["weights_tb"]).to(dev)
        d_ne = torch.from_numpy(wl["n_ee"]).to(dev)
    else:
        d_j = torch.from_numpy(wl["joints"].astype(np.int32)).to(dev)
        d_w = torch.from_numpy(wl["weights"]).to(dev)
        d_ne = None
    # result rows of every frame in the wire layout [pose 88 | global_pos 3 | pad], written by the frame kernel itself
    d_rows = torch.zeros((T, B, dpdist.ROW), dtype=torch.float32, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    work_stream = torch.cuda.Stream(device=dev)  # everything timed runs (and is timed) on this stream
    torch.cuda.set_stream(work_stream)
    stream = work_stream.cuda_stream

    def step(t):
        eng.run_frames_device(1, d_tp[t], d_tr[t], d_j[t] if variable else d_j, d_w[t] if variable else d_w, d_rows[t], None,
                              n_ee=d_ne[t] if variable else None, shared=not variable, ee_stride=E, stream=stream, options=opts)

    # the only collective of the job: the K frames' result rows go to rank 0 in a few chunks, each gather running while the
    # next chunk's frames are computed; only the last chunk's gather is exposed
    n_chunks = K if world > 1 else 0  # one frame per chunk: only the last frame's gather (and its D2H in the e2e leg) is exposed
    bounds = [W + (K * i) // n_chunks for i in range(n_chunks + 1)] if n_chunks else []
    recv = [torch.empty((world, bounds[i + 1] - bounds[i], B, dpdist.ROW), dtype=torch.float32, device=dev) if rank == 0 else None
            for i in range(n_chunks)]
    for t in range(W):
        step(t)
    if world > 1:  # warm the collective too (NCCL connects its channels on the first call of a shape)
        for i in range(n_chunks):
            _, h = dpdist.gather_packed(d_rows[bounds[i]:bounds[i + 1]], n_total, dst=0, out=recv[i], async_op=True)
            h.wait()
    if clocks is not None:
        clocks.start()  # before the barrier: every rank must enter the timed region at the same moment
    eng.set_profiling(True)
    l0 = eng.launch_count()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    evs, handles, chunk = [], [], 0
    for k in range(K):
        flush.zero_()  # L2 flush between timed steps (outside the event pair)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step(W + k)
        b.record()
        evs.append((a, b))
        if n_chunks and W + k + 1 == bounds[chunk + 1]:
            _, h = dpdist.gather_packed(d_rows[bounds[chunk]:bounds[chunk + 1]], n_total, dst=0, out=recv[chunk], async_op=True)
            handles.append(h)
            chunk += 1
    if handles:  # what is left of the gathers once the last frame is done
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for h in handles:
            h.wait()
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    ms = sum(a.elapsed_time(b) for a, b in evs)
    gather_tail_ms = evs[-1][0].elapsed_time(evs[-1][1]) if handles else 0.0
    launches = eng.launch_count() - l0
    ms_pred, ms_frame, nprof = eng.profile()
    eng.set_profiling(False)
    clk = clocks.stop() if clocks is not None else None
    # rows [pose 88 | global_pos 3] of the last timed step as its consumer receives them (rank 0 holds every rank's rows); copied
    # here because the e2e pass below reuses the gather buffers
    last_rows = None
    if args.dump_outputs and rank == 0:
        rows = dpdist.GatheredFrames(recv[-1], n_total).frame(0) if world > 1 else d_rows[W + K - 1]
        last_rows = rows[:, :91].cpu().numpy()
    ms_by_rank, parts_by_rank = [ms / K], None
    if world > 1:
        dist.barrier()
        every = [torch.zeros(4, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(every, torch.tensor([ms, ms_frame / max(nprof, 1), ms_pred / max(nprof, 1), gather_tail_ms], dtype=torch.float64, device=dev))
        ms_by_rank = [float(t[0].item()) / K for t in every]
        parts_by_rank = [[round(float(t[1].item()), 4), round(float(t[2].item()), 4), round(float(t[3].item()), 4)] for t in every]
        ms = max(float(t[0].item()) for t in every)  # the job is as fast as its slowest rank
    value = n_total * K / (ms * 1e-3)

    # ---- e2e.  One GPU: HOST arrays through the public API (BatchedDragPose.run_frames), every frame's staging + H2D + D2H inside
    # the timed region (the call double-buffers them against the kernels of the neighbouring frames).  Several GPUs: every rank
    # copies each step's targets from PINNED host memory to its GPU (double-buffered) and runs the frame; the results are delivered
    # twice, in two timed passes over the same K steps: (a) to rank 0's pinned host memory through the same per-frame gather as above
    # (one consumer process: `e2e.gathered_to_rank0_value`), (b) every rank's own rows to its own pinned host memory (`e2e.value`:
    # the caller keeps shards, the natural consumer of a clip-sharded batch evaluation -- no collective on the data path).  Either
    # clock stops when the last row is in host memory.
    h_tp, h_tr = wl["tgt_pos"], wl["tgt_rot"]
    host_out = (np.zeros((K, B, 88), np.float32), np.zeros((K, B, 3), np.float32))  # result arrays of the caller, reused

    def run_host(t0, t1):
        out = host_out if t1 - t0 == K else None
        if variable:
            return eng.run_frames(h_tp[t0:t1], h_tr[t0:t1], wl["joints_tb"][t0:t1], wl["weights_tb"][t0:t1], n_ee=wl["n_ee"][t0:t1],
                                  out=out, options=opts)
        return eng.run_frames(h_tp[t0:t1], h_tr[t0:t1], wl["joints"], wl["weights"], out=out, options=opts)

    if world == 1:
        run_host(0, min(W, 2))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        run_host(W, W + K)
        e2e_s = time.perf_counter() - t0
    else:
        p_tp, p_tr = torch.from_numpy(h_tp).pin_memory(), torch.from_numpy(h_tr).pin_memory()
        # the step's inputs on the device, double-buffered: the copy of step t+1 (own stream) runs under the kernels of step t
        s_tp, s_tr = [torch.empty_like(d_tp[0]) for _ in range(2)], [torch.empty_like(d_tr[0]) for _ in range(2)]
        host_recv = [torch.empty(r.shape, dtype=torch.float32).pin_memory() if r is not None else None for r in recv]
        copy_stream = torch.cuda.Stream(device=dev)
        in_stream = torch.cuda.Stream(device=dev)
        ev_in = [torch.cuda.Event() for _ in range(2)]
        ev_done = [torch.cuda.Event() for _ in range(2)]
        n_host_steps = [0]

        def step_from_host(t):
            slot = n_host_steps[0] & 1
            n_host_steps[0] += 1
            with torch.cuda.stream(in_stream):
                in_stream.wait_event(ev_done[slot])  # the frame that last read this slot has finished (no-op the first time round)
                s_tp[slot].copy_(p_tp[t], non_blocking=True)
                s_tr[slot].copy_(p_tr[t], non_blocking=True)
                ev_in[slot].record(in_stream)
            work_stream.wait_event(ev_in[slot])
            eng.run_frames_device(1, s_tp[slot], s_tr[slot], d_j[t] if variable else d_j, d_w[t] if variable else d_w, d_rows[t], None,
                                  n_ee=d_ne[t] if variable else None, shared=not variable, ee_stride=E, stream=stream, options=opts)
            ev_done[slot].record(work_stream)

        step_from_host(0)
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        chunk, handles = 0, []
        for k in range(K):
            step_from_host(W + k)
            if W + k + 1 == bounds[chunk + 1]:
                _, h = dpdist.gather_packed(d_rows[bounds[chunk]:bounds[chunk + 1]], n_total, dst=0, out=recv[chunk], async_op=True)
                handles.append(h)
                if rank == 0:
                    with torch.cuda.stream(copy_stream):
                        h.wait()  # only the copy stream waits for the collective
                        host_recv[chunk].copy_(recv[chunk], non_blocking=True)
                chunk += 1
        for h in handles:
            h.wait()
        torch.cuda.synchronize()
        e2e_gathered_s = time.perf_counter() - t0
        # (b) the caller keeps shards (one evaluation worker per GPU, as eval_drag --batch on a node would run): every rank reads ITS
        # OWN result rows of every step into its own pinned host memory; no collective at all on the data path
        host_rows = torch.empty((K, B, dpdist.ROW), dtype=torch.float32).pin_memory()
        ev_rows = [torch.cuda.Event() for _ in range(K)]
        step_from_host(W)  # re-warm after the gathered pass (the frame stream carries on from where it is: same work per step)
        torch.cuda.synchronize()
        dist.barrier()
        t0 = time.perf_counter()
        for k in range(K):
            step_from_host(W + k)
            ev_rows[k].record(work_stream)
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(ev_rows[k])
                host_rows[k].copy_(d_rows[W + k], non_blocking=True)
        torch.cuda.synchronize()
        e2e_s = time.perf_counter() - t0
        tt = torch.tensor([e2e_s, e2e_gathered_s], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e_s, e2e_gathered_s = float(tt[0].item()), float(tt[1].item())
    h2d = B * E * (3 + 9) * 4 + (B * E * (1 + 2) * 4 + B * 4 if variable else E * 12)
    d2h = B * (88 + 3) * 4
    path = eng.last_decoder_path()
    eng.close()
    torch.cuda.set_stream(torch.cuda.default_stream(dev))
    return dict(cfg=cfg, value=value, ms=ms, K=K, launches=launches, frame_ms=ms_frame / max(nprof, 1), pred_ms=ms_pred / max(nprof, 1), clk=clk,
                ms_by_rank=ms_by_rank, parts_by_rank=parts_by_rank, e2e_value=n_total * K / e2e_s, h2d=h2d, d2h=d2h, path=path, n_total=n_total,
                e2e_gathered=(n_total * K / e2e_gathered_s) if world > 1 else None, last_rows=last_rows,
                gather={"chunks": n_chunks, "to": "rank 0", "bytes_received_by_rank_0": int(max(world - 1, 0) * K * B * dpdist.ROW * 4)})


def roofline(m, B, trackers, peaks):
    # burst peak: the timed region is a few tens of milliseconds at full clock (each step is bracketed by its own events)
    tf32_peak = (peaks.get("bf16_tflops") or 1632.8) / 2.0
    hbm_peak = peaks.get("hbm_gbs") or 6650.0
    which = "measured bf16 burst / 2 = TF32 (MEASURED_PEAKS.json)" if peaks else "fallback (no MEASURED_PEAKS.json)"
    achieved_tf = B * MAX_ITER * FLOP_PER_CLIP_ITER / (m["frame_ms"] * 1e-3) / 1e12
    achieved_gbs = B * HBM_BYTES_PER_CLIP_FRAME / (m["frame_ms"] * 1e-3) / 1e9
    return {"bound": "tensor", "kernel": KERNEL_NAMES[m["path"]], "achieved": achieved_tf, "peak": tf32_peak, "unit": "TFLOP/s",
            "frac": achieved_tf / tf32_peak, "traffic": NCU_DRAM_BYTES_PER_LAUNCH.get((m["path"], B, trackers)), "peak_source": which,
            "kernel_ms_per_launch": m["frame_ms"], "predictor_ms_per_step": m["pred_ms"],
            "hbm": {"achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": achieved_gbs / hbm_peak},
            "tensor_pipe_pct_of_peak_ncu": {"dp_frame_tc16_kernel": 12.12, "tp_ff_tc_kernel": 53.9, "tp_attn_tc_kernel": 7.26,
                                            "source": "profiles/r2_frame_kernel.md, r2_predictor.md: sm__ops_path_tensor_op_utchmma_src_fp16_dst_fp32 (issued ops, % of peak sustained elapsed)"},
            "note": "dependency-latency bound path (SURVEY 8d): both fractions are small by construction"}


DUMP_BYTES = 63 << 20  # all arrays of one dump together, below 64 MB with room for the .npy headers


def dump_outputs(out_dir, rows_by_prefix):
    """Writes <prefix>pose.npy (n,88) and <prefix>global_pos.npy (n,3), float32, per workload: the last timed step's results, so
    that two builds run with the same arguments can be compared output for output.  Above the byte budget a fixed, seeded sample
    of clips (the same one on every run) is written, in clip order."""
    os.makedirs(out_dir, exist_ok=True)
    keep = DUMP_BYTES // len(rows_by_prefix) // (91 * 4)
    for prefix, rows in rows_by_prefix.items():
        if rows.shape[0] > keep:
            rows = rows[np.sort(np.random.default_rng(0).choice(rows.shape[0], keep, replace=False))]
        np.save(os.path.join(out_dir, f"{prefix}pose.npy"), np.ascontiguousarray(rows[:, :88], np.float32))
        np.save(os.path.join(out_dir, f"{prefix}global_pos.npy"), np.ascontiguousarray(rows[:, 88:91], np.float32))


def run_ours(args):
    import torch
    import torch.distributed as dist

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if os.environ.get("DP_BENCH_REVERSE_DEVICES"):  # diagnostic: is a slow rank a slow GPU or a slow process?
        local = world - 1 - local
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the engine has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    K, W = args.steps, args.warmup
    clocks = ClockSampler(local, world) if rank == 0 else None
    m = measure(args, args.trackers, K, W, rank, world, dev, local, clocks)
    line, peaks = None, {}
    if rank == 0:
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
                peaks = json.load(fh)
        except Exception:
            pass
        line = {
            "metric": "clip-frames/sec (fixed 100 opt iters)", "value": m["value"], "unit": "clip-frames/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": m["ms"] / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(args, m["cfg"], m["n_total"]),
            "roofline": roofline(m, args.clips, args.trackers, peaks),
            "e2e": {"value": m["e2e_value"], "unit": "clip-frames/s", "h2d_bytes_per_step": m["h2d"], "d2h_bytes_per_step": m["d2h"]},
            "gpu_launches": m["launches"], "clocks": m["clk"],
        }
        if world > 1:
            line["ms_per_step_by_rank"] = [round(v, 4) for v in m["ms_by_rank"]]
            line["frame_kernel_predictor_gather_tail_ms_by_rank"] = m["parts_by_rank"]
            line["gather"] = m["gather"]
            line["e2e"]["delivery"] = "every rank reads its own result rows into its own pinned host memory (the caller keeps shards)"
            line["e2e"]["gathered_to_rank0_value"] = m["e2e_gathered"]  # the same K steps with all rows gathered into rank 0's host memory
    outputs = {"": m["last_rows"]}
    if world == 1 and not args.no_config3 and args.trackers == "6":
        # BASELINE config 3 in the same record: head + hands with the hands dropping out, window 16 (the predictor runs on every 16th
        # frame with five decoder passes), 4096 clips.  The per-step cost depends on how many predictor frames (t % 16 == 0) fall
        # into the K timed frames W..W+K-1: a multiple of 16 for --steps weighs them as a long run does, and the record says how many
        m3 = measure(args, "3", K, W, rank, world, dev, local)
        outputs["3trk_var_"] = m3["last_rows"]
        window = m3["cfg"].temporal_future_window
        line["configs"] = {("3trk_var_4096" if args.clips == 4096 else f"3trk_var_{args.clips}"): {
            "value": m3["value"], "unit": "clip-frames/s", "steps": K, "ms_per_step": m3["ms"] / K,
            "predictor_steps": sum(1 for t in range(W, W + K) if t % window == 0),
            "config": workload_config(args, m3["cfg"], m3["n_total"], "3"), "roofline": roofline(m3, args.clips, "3", peaks),
            "e2e": {"value": m3["e2e_value"], "unit": "clip-frames/s", "h2d_bytes_per_step": m3["h2d"], "d2h_bytes_per_step": m3["d2h"]},
            "gpu_launches": m3["launches"]}}
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        if world == 1 and not args.no_latency:
            line["latency"] = dll_latency()
        if world == 1 and not args.no_cpu_baseline:
            v, cores, sample = cpu_reference(1, 6, args.trackers)
            line["cpu_baseline"] = {"value": v, "unit": "clip-frames/s", "cores": cores, "kind": "port", "sample": sample,
                                    "port_vs_unmodified_reference_per_core": PORT_VS_REFERENCE_PER_CORE}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--clips", type=int, default=4096, help="clips per GPU (weak scaling)")
    ap.add_argument("--trackers", default="6", choices=["6", "3"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-latency", action="store_true", help="skip the B = 1 C-ABI latency measurement")
    ap.add_argument("--no-config3", action="store_true", help="skip the second workload (BASELINE config 3) at N = 1")
    ap.add_argument("--decoder-path", type=int, default=0, choices=[0, 1, 3], help="0 auto, 1 fp32 CUDA-core decoder, 3 tcgen05 fp16x2")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the poses and root positions of the last timed step as DIR/*.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
