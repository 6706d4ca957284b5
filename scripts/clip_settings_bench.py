"""Cost of per-clip optimiser settings (dp_engine_set_clip_settings) on the GPU it runs on.

    python scripts/clip_settings_bench.py [--out DIR] [--rounds R] [--frames K]

Frame time (6 trackers, window 0, 100 fixed iterations: the headline workload) on the tcgen05 frame kernel at 4 096 clips and on
the fp32 frame kernel at 4 096 and 64 clips (its small-batch use), measured with CUDA events on the launching stream over K frames,
for
  * no table (every per-clip field from dp_run_params),
  * a one-entry table equal to those dp_run_params,
  * four fixed-iteration settings that differ in learning rate, loss weights and joint adjustment, dealt to the clips in turn
    (the same work per clip as the other two modes, so the difference is the cost of the table: on the tcgen05 kernel reading it,
    on the fp32 kernel one gather, launch and scatter per setting).
The modes alternate within each of R rounds; the median and the range over the rounds are reported.  Prints, and with --out also
writes as DIR/clip_settings_bench.json.  The GPU's name and power limit are read in the same run."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from dragposer_b200 import model, synthetic  # noqa: E402
from dragposer_b200.engine import BatchedDragPose, ClipOptions, RunOptions  # noqa: E402

G = os.path.join(ROOT, "tests", "golden")
FIXED = dict(stop_eps_pos=-1.0, stop_eps_rot=-1.0, max_iter=100, min_loss_incr=-float("inf"))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", help="directory for clip_settings_bench.json")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--frames", type=int, default=32)
    args = ap.parse_args()
    pm = model.load_folded_npz(os.path.join(G, "model_dancedb.npz"))
    off = np.load(os.path.join(G, "model_dancedb.npz"))["offsets"]
    tm = model.temporal_from_state(model.random_temporal_state(2222))
    cfg = synthetic.config_6_trackers()
    base = dict(FIXED, learning_rate=1e-2, lambda_rot=1, lambda_temporal=cfg.lambda_temporal, joint_adjustment_indices=cfg.joint_adjustment,
                joint_adjustment_weight=cfg.joint_adjustment_weight)
    four = [base, dict(base, learning_rate=5e-3, lambda_temporal=0.15), dict(base, lambda_rot=0.5, joint_adjustment_indices=None),
            dict(base, learning_rate=2e-2, joint_adjustment_indices=(13, 3), joint_adjustment_weight=0.1)]
    st = torch.cuda.Stream()
    res = dict(gpu=gpu_info(), frames_per_sample=args.frames, rounds=args.rounds)
    print("GPU:", res["gpu"], flush=True)
    for key, path, B in (("tcgen05_fp16x2_4096", 3, 4096), ("fp32_4096", 1, 4096), ("fp32_64", 1, 64)):
        wl = synthetic.make_workload(pm, off, cfg, B, 16)
        tp = torch.from_numpy(wl["tgt_pos"]).cuda()
        tr = torch.from_numpy(wl["tgt_rot"].reshape(16, B, -1, 9)).cuda()
        j = torch.from_numpy(np.asarray(wl["joints"], np.int32)).cuda()
        w = torch.from_numpy(np.asarray(wl["weights"], np.float32)).cuda()
        pose, gpos = torch.empty(1, B, 88, device="cuda"), torch.empty(1, B, 3, device="cuda")
        modes = {"no_table": None, "one_entry": ([ClipOptions(**base)], None),
                 "four_settings": ([ClipOptions(**s) for s in four], np.arange(B, dtype=np.int32) % 4)}
        opt = RunOptions(**base, temporal_future_window=0, decoder_path=path)
        engines = {}
        for name, table in modes.items():
            eng = BatchedDragPose(pm, off, tm, B)
            eng.set_initial_state(wl["latent0"], np.zeros((B, 3), np.float32), np.tile(np.float32([[1, 0, 0, 0]]), (B, 1)),
                                  np.zeros((B, 6), np.float32))
            if table is not None:
                eng.set_clip_options(*table)
            engines[name] = eng
        samples = {name: [] for name in modes}
        t = 0
        for rnd in range(args.rounds + 1):  # round 0 warms every engine up
            for name, eng in engines.items():
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(st)
                for k in range(args.frames):
                    eng.run_frames_device(1, tp[(t + k) % 16], tr[(t + k) % 16], j, w, pose, gpos, options=opt, stream=st.cuda_stream)
                b.record(st)
                st.synchronize()
                if rnd:
                    samples[name].append(a.elapsed_time(b) / args.frames)
            t += args.frames
        res[key] = {name: dict(ms_per_frame_median=float(np.median(v)), ms_per_frame_min=float(np.min(v)), ms_per_frame_max=float(np.max(v)),
                               decoder_path=engines[name].last_decoder_path()) for name, v in samples.items()}
        print(key, json.dumps(res[key]), flush=True)
        for eng in engines.values():
            eng.close()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "clip_settings_bench.json"), "w") as fo:
            json.dump(res, fo, indent=1)


if __name__ == "__main__":
    main()
