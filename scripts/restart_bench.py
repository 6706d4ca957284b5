"""Cost of per-clip restarts (dp_engine_restart_clips) on the GPU it runs on.

    python scripts/restart_bench.py [--out DIR]

Prints, and with --out also writes as DIR/restart_bench.json:
  * host enqueue time and device time (CUDA events on the launching stream) of one restart of 1, 64 and 512 clips (4 096-clip engine);
  * frame time at 4 096 clips, 6 trackers / window 0 and 3 trackers / window 16, 100 fixed iterations, for no restarts, aligned
    restarts (1/16 of the clips every 16 frames, at a boundary) and unaligned restarts every frame (1/16 of the clips each, 16 phases);
  * p50 / p99 host-observed frame latency at 64 clips, window 16 (BatchedDragPose.run), every clip at one phase vs four phases;
  * eval_drag.evaluate_stream (256 slots) vs evaluate_batch over the same variable-length excerpts of example_full.bvh, in real
    (unpadded) clip-frames per second of engine time and of wall time.
The GPU's name and power limit are read in the same run."""
from __future__ import annotations

import argparse
import ctypes as C
import gzip
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from dragposer_b200 import _lib, eval_drag, model, synthetic  # noqa: E402
from dragposer_b200.engine import BatchedDragPose, RunOptions  # noqa: E402

G = os.path.join(ROOT, "tests", "golden")
FIXED = dict(stop_eps_pos=-1.0, stop_eps_rot=-1.0, max_iter=100, min_loss_incr=-float("inf"), learning_rate=1e-2)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def engine(pm, off, tm, n):
    return BatchedDragPose(pm, off, tm, n)


def start(n):
    return np.zeros((n, 3), np.float32), np.tile(np.float32([[1, 0, 0, 0]]), (n, 1)), np.zeros((n, 6), np.float32)


def restart_cost(pm, off, tm):
    eng = engine(pm, off, tm, 4096)
    rng = np.random.default_rng(0)
    eng.set_initial_state(rng.standard_normal((4096, 24)).astype(np.float32) * 0.3, *start(4096))
    st = torch.cuda.Stream()
    out = {}
    for n in (1, 64, 512):
        ids = np.ascontiguousarray(rng.permutation(4096)[:n].astype(np.int32))
        z = np.ascontiguousarray(rng.standard_normal((n, 24)).astype(np.float32))
        gp, gr, ht = start(n)
        host, dev = [], []
        for rep in range(60):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(st)
            t0 = time.perf_counter()
            _lib.check(eng.lib.dp_engine_restart_clips(eng.h, n, _lib_ptr(ids), _lib_ptr(z), _lib_ptr(gp), _lib_ptr(gr), _lib_ptr(ht),
                                                       C.c_void_p(st.cuda_stream)))
            t1 = time.perf_counter()
            b.record(st)
            st.synchronize()
            if rep >= 10:
                host.append((t1 - t0) * 1e3)
                dev.append(a.elapsed_time(b))
        out[n] = dict(host_enqueue_ms=float(np.median(host)), device_ms=float(np.median(dev)))
    eng.close()
    return out


def _lib_ptr(a):
    return C.c_void_p(a.ctypes.data)


def step_times(pm, off, tm, frames=64, warm=20):  # the warm-up holds the first restart (its staging and scratch are allocated then)
    out = {}
    B = 4096
    for name, cfg in (("6trk_w0", synthetic.config_6_trackers()), ("3trk_w16", synthetic.config_3_trackers())):
        W = cfg.temporal_future_window
        wl = synthetic.make_workload(pm, off, cfg, B, 16)
        tp = torch.from_numpy(wl["tgt_pos"]).cuda()
        tr = torch.from_numpy(wl["tgt_rot"].reshape(16, B, -1, 9)).cuda()
        j = torch.from_numpy(np.asarray(wl["joints"], np.int32)).cuda()
        w = torch.from_numpy(np.asarray(wl["weights"], np.float32)).cuda()
        pose, gpos = torch.empty(1, B, 88, device="cuda"), torch.empty(1, B, 3, device="cuda")
        opt = RunOptions(**FIXED, lambda_rot=1, lambda_temporal=cfg.lambda_temporal, temporal_future_window=W,
                         joint_adjustment_indices=cfg.joint_adjustment, joint_adjustment_weight=cfg.joint_adjustment_weight)
        z = wl["latent0"]
        for mode in ("none", "aligned", "unaligned"):
            eng = engine(pm, off, tm, B)
            eng.set_initial_state(z, *start(B))
            n_restarts = 0
            for t in range(warm + frames):
                if t == warm:
                    eng.frame_stats()  # synchronise
                    t0, l0 = time.perf_counter(), eng.launch_count()
                if mode == "aligned" and t % 16 == 0 and t:
                    ids = np.arange((t // 16) % 16, B, 16)
                elif mode == "unaligned" and t:
                    ids = np.arange(t % 16, B, 16)
                else:
                    ids = None
                if ids is not None:
                    eng.restart_clips(ids, z[ids], *start(len(ids)))
                    n_restarts += t >= warm
                k = t % 16
                eng.run_frames_device(1, tp[k], tr[k], j, w, pose, gpos, options=opt)
            eng.frame_stats()
            ms = (time.perf_counter() - t0) * 1e3 / frames
            out[f"{name}_{mode}"] = dict(ms_per_frame=ms, launches_per_frame=(eng.launch_count() - l0) / frames,
                                         distinct_phases=len(set(eng.clip_index(W).tolist())) if W else 1, restarts=n_restarts)
            eng.close()
    return out


def latency(pm, off, tm, frames=400):
    cfg = synthetic.config_3_trackers()
    B = 64
    wl = synthetic.make_workload(pm, off, cfg, B, 16)
    kw = dict(stop_eps_pos=0.01 * 0.01, stop_eps_rot=0.01, max_iter=100, min_loss_incr=0.00001, learning_rate=1e-2, lambda_rot=1,
              lambda_temporal=cfg.lambda_temporal, temporal_future_window=16, joint_adjustment_indices=cfg.joint_adjustment,
              joint_adjustment_weight=cfg.joint_adjustment_weight)
    out = {}
    for mode in ("uniform", "mixed"):
        eng = engine(pm, off, tm, B)
        eng.set_initial_state(wl["latent0"], *start(B))
        ts = []
        for t in range(frames + 32):
            if mode == "mixed" and t in (1, 5, 9):  # four phases: 0, 1, 5, 9
                ids = np.arange({1: 1, 5: 2, 9: 3}[t], B, 4)
                eng.restart_clips(ids, wl["latent0"][ids], *start(len(ids)))
            k = t % 16
            t0 = time.perf_counter()
            eng.run(wl["tgt_pos"][k], wl["tgt_rot"][k], wl["joints"], wl["weights"], **kw)
            if t >= 32:
                ts.append((time.perf_counter() - t0) * 1e3)
        out[mode] = dict(p50_ms=float(np.percentile(ts, 50)), p99_ms=float(np.percentile(ts, 99)),
                         distinct_phases=len(set(eng.clip_index(16).tolist())))
        eng.close()
    return out


def stream_vs_batch(n_clips=1024, lo=40, hi=600):
    src = b""
    for part in ("example_full.bvh.gz.1", "example_full.bvh.gz.2"):
        with open(os.path.join(G, part), "rb") as fi:
            src += fi.read()
    lines = gzip.decompress(src).decode().split("\n")
    m = next(i for i, l in enumerate(lines) if l.strip().startswith("Frames:"))
    total = int(lines[m].split()[1])
    rng = np.random.default_rng(3)
    out = {}
    with tempfile.TemporaryDirectory() as d:
        paths, lens = [], []
        for i in range(n_clips):
            k = int(rng.integers(lo, hi + 1))
            a = int(rng.integers(0, total - k))
            p = os.path.join(d, f"x{i:04d}.bvh")
            with open(p, "w") as fo:
                fo.write("\n".join(lines[:m] + [f"Frames: {k}", lines[m + 1]] + lines[m + 2 + a : m + 2 + a + k]) + "\n")
            paths.append(p)
            lens.append(k)
        lat = list(rng.standard_normal((n_clips, 24)).astype(np.float32) * np.float32(0.5))
        npz = os.path.join(G, "model_dancedb.npz")
        real = float(sum(lens))
        for name, fn in (("evaluate_batch", lambda: eval_drag.evaluate_batch(npz, paths, initial_latents=lat, random_temporal=True)),
                         ("evaluate_stream_256", lambda: eval_drag.evaluate_stream(npz, paths, 256, initial_latents=lat, random_temporal=True))):
            t0 = time.perf_counter()
            res = fn()
            wall = time.perf_counter() - t0
            eng_s = res[0]["time"]
            out[name] = dict(real_clip_frames=real, engine_s=eng_s, wall_s=wall, real_clip_frames_per_s_engine=real / eng_s,
                             real_clip_frames_per_s_wall=real / wall, mean_mpjpe_cm=float(np.mean([r["mpjpe"] for r in res]) * 100))
        out["clips"] = n_clips
        out["frames_per_clip"] = [lo, hi]
        out["padded_clip_frames_batch"] = float(n_clips * max(lens))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="directory for restart_bench.json")
    ap.add_argument("--skip-eval", action="store_true")
    args = ap.parse_args()
    pm = model.load_folded_npz(os.path.join(G, "model_dancedb.npz"))
    off = np.load(os.path.join(G, "model_dancedb.npz"))["offsets"]
    tm = model.temporal_from_state(model.random_temporal_state(2222))
    res = dict(gpu=gpu_info())
    print("GPU:", res["gpu"], flush=True)
    res["restart"] = restart_cost(pm, off, tm)
    print(json.dumps(res["restart"]), flush=True)
    res["step_4096"] = step_times(pm, off, tm)
    print(json.dumps(res["step_4096"]), flush=True)
    res["latency_64_w16"] = latency(pm, off, tm)
    print(json.dumps(res["latency_64_w16"]), flush=True)
    if not args.skip_eval:
        res["eval"] = stream_vs_batch()
        print(json.dumps(res["eval"]), flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "restart_bench.json"), "w") as fo:
            json.dump(res, fo, indent=1)


if __name__ == "__main__":
    main()
