"""Drop-in for the reference's evaluation CLI (python/src/eval_drag.py:255-293):

    python -m dragposer_b200.eval_drag <model_dir | folded.npz> <file.bvh | dir> [--config cfg.json] [--verbose]
                                       [--batch [--slots N]]

Same arguments, same JSON tracker-config keys, same printed metrics; writes `data/eval_<name>.bvh`.  The per-frame
optimisation runs on the B200 engine; target construction from the ground-truth clip and the BVH/metric export are
host-side numpy (python/src/eval_drag.py:164-202, train.py:437-509, eval_metrics.py:6-32).
"""
from __future__ import annotations

import argparse
import os
import time

import numpy as np
import torch

from . import model as dpm
from . import motion, synthetic
from .bvh import Bvh
from .drag_pose import DragPose


def evaluate(model_path, input_path, config=None, verbose=False, max_frames=None, save=True, seed=2222, quiet=False, initial_latent=None,
             random_temporal=False):
    torch.manual_seed(seed)  # eval_drag.py:23-25
    np.random.seed(seed)
    cfg = synthetic.TrackerConfig.load(config) if config else synthetic.config_6_trackers()  # defaults: eval_drag.py:68-131
    bvh = Bvh(input_path)
    parents, offsets = bvh.skeleton()
    rots = bvh.quaternions()
    pm = dpm.load_pose_model(model_path, parents)
    tdir = model_path if os.path.isdir(model_path) else os.path.dirname(model_path)
    tm = dpm.load_temporal_model(tdir, allow_random=random_temporal)  # eval_drag.py:58-59 raises when temporal.pt is missing
    clip = motion.ClipData(rots, bvh.positions[:, 0, :], parents, offsets, pm.mean_dqs, pm.std_dqs)
    joints, weights = cfg.joints, cfg.tracker_weights
    drag = DragPose(pm, tm, offsets=offsets)
    drag.set_initial_pose(clip.dqs[0].reshape(1, 176, 1), clip.global_pos[0].reshape(1, 3, 1), clip.global_rot[0].reshape(1, 4, 1), clip.heights[0])
    if initial_latent is not None:  # tests: reproduce a recorded reparameterisation draw (torch RNG stream of the reference)
        drag.set_initial_latent(initial_latent, clip.global_pos[0], clip.global_rot[0], clip.heights[0])
    n_frames = clip.n_frames if max_frames is None else min(max_frames, clip.n_frames)
    poses, gposs, iters = np.zeros((n_frames, 88), np.float32), np.zeros((n_frames, 3), np.float32), []
    gpos = clip.global_pos[0].copy()
    start = time.time()
    for i in range(n_frames):
        if i % 100 == 0 and not quiet:
            print("Frame: {} out of {}".format(i + 1, n_frames))
        tp, tr = motion.frame_targets(clip, i, pm.mean_q, pm.std_q, parents, offsets, gpos, joints)
        pose, g = drag.run(tp, tr, joints, weights, offsets, stop_eps_pos=0.01 * 0.01, stop_eps_rot=0.01, max_iter=100, min_loss_incr=0.00001,
                           learning_rate=1e-2, lambda_rot=1, lambda_temporal=cfg.lambda_temporal,
                           temporal_future_window=cfg.temporal_future_window, joint_adjustment_indices=cfg.joint_adjustment,
                           joint_adjustment_weight=cfg.joint_adjustment_weight, verbose=verbose)
        poses[i], gposs[i] = pose.numpy(), g.numpy()
        gpos = gposs[i]
        iters.append(drag.last_iterations)
    elapsed = time.time() - start
    drag.close()
    local = motion.result_local_quats(poses, pm.mean_q, pm.std_q, parents)
    out_path = None
    if save:  # result_to_bvh: euler angles in the clip's channel order, root positions from the optimiser
        os.makedirs("data", exist_ok=True)
        out_path = os.path.join("data", "eval_" + os.path.basename(input_path))
        write_result_bvh(bvh, local, gposs, out_path)
    m, e = motion.mpjpe(rots[:n_frames], local.astype(np.float64), np.asarray(offsets, np.float64), parents)
    if not quiet:
        print("Evaluate Loss: {}".format(m + e))
        print("Mean Per Joint Position Error: {}".format(m))
        print("Mean End Effector Position Error: {}".format(e))
        print("Time: {}".format(elapsed))
    return dict(mpjpe=m, mpeepe=e, time=elapsed, iterations=np.asarray(iters), poses=poses, global_pos=gposs, out_path=out_path)


def evaluate_batch(model_path, input_paths, config=None, save=False, seed=2222, quiet=True, initial_latents=None, max_frames=None,
                   device=0, random_temporal=False):
    """Many BVH clips at once (SURVEY 8f rank 1): every clip becomes one row of a BatchedDragPose, the ground-truth tracker
    targets of ALL frames are built once in world coordinates (motion.world_targets) and the whole sequence runs through
    run_frames with targets_world=True, so nothing on the host depends on the previous frame's result.  Clips must share the
    skeleton; shorter clips are padded by repeating their last frame (their metrics only use their own frames).
    Same optimiser settings and metrics as evaluate(); returns one result dict per clip."""
    from .engine import BatchedDragPose

    torch.manual_seed(seed)
    np.random.seed(seed)
    cfg = synthetic.TrackerConfig.load(config) if config else synthetic.config_6_trackers()
    bvhs = [Bvh(p) for p in input_paths]
    parents, offsets = bvhs[0].skeleton()
    for b in bvhs[1:]:
        p2, o2 = b.skeleton()
        if list(p2) != list(parents) or not np.allclose(o2, offsets, atol=1e-6):
            raise ValueError("evaluate_batch: all clips must share one skeleton")
    pm = dpm.load_pose_model(model_path, parents)
    tdir = model_path if os.path.isdir(model_path) else os.path.dirname(model_path)
    tm = dpm.load_temporal_model(tdir, allow_random=random_temporal)
    joints, weights = cfg.joints, cfg.tracker_weights
    rots = [b.quaternions() for b in bvhs]
    clips = [motion.ClipData(r, b.positions[:, 0, :], parents, offsets, pm.mean_dqs, pm.std_dqs) for r, b in zip(rots, bvhs)]
    lens = [c.n_frames if max_frames is None else min(max_frames, c.n_frames) for c in clips]
    B, T, E = len(clips), max(lens), len(joints)
    tgt_pos, tgt_rot = np.empty((T, B, E, 3), np.float32), np.empty((T, B, E, 3, 3), np.float32)
    for b, c in enumerate(clips):
        tp, tr = motion.world_targets(c, pm.mean_q, pm.std_q, parents, offsets, joints, lens[b])
        tgt_pos[: lens[b], b], tgt_rot[: lens[b], b] = tp, tr
        tgt_pos[lens[b]:, b], tgt_rot[lens[b]:, b] = tp[-1], tr[-1]
    eng = BatchedDragPose(pm, offsets, tm, B, device=device)
    if initial_latents is not None:
        latent0 = np.stack([np.asarray(z, np.float32).reshape(-1) for z in initial_latents])
    else:  # mu + eps * exp(0.5 logvar) on the device; eps ~ torch.randn, one draw per clip in clip order (autoencoder.py:19-27)
        eps = np.concatenate([torch.randn(1, dpm.LATENT).numpy() for _ in clips])
        latent0 = eng.encode(np.stack([c.dqs[0] for c in clips]), eps)
    eng.set_initial_state(latent0, np.stack([c.global_pos[0] for c in clips]), np.stack([c.global_rot[0] for c in clips]),
                          np.stack([c.heights[0] for c in clips]))
    start = time.time()
    poses, gposs = eng.run_frames(tgt_pos, tgt_rot, joints, weights, stop_eps_pos=0.01 * 0.01, stop_eps_rot=0.01, max_iter=100,
                                  min_loss_incr=0.00001, learning_rate=1e-2, lambda_rot=1, lambda_temporal=cfg.lambda_temporal,
                                  temporal_future_window=cfg.temporal_future_window, joint_adjustment_indices=cfg.joint_adjustment,
                                  joint_adjustment_weight=cfg.joint_adjustment_weight, targets_world=True)
    elapsed = time.time() - start
    eng.close()
    results = []
    for b, (bvh, c) in enumerate(zip(bvhs, clips)):
        local = motion.result_local_quats(poses[: lens[b], b], pm.mean_q, pm.std_q, parents)
        out_path = None
        if save:
            os.makedirs("data", exist_ok=True)
            out_path = os.path.join("data", "eval_" + os.path.basename(input_paths[b]))
            write_result_bvh(bvh, local, gposs[: lens[b], b], out_path)
        m, e = motion.mpjpe(rots[b][: lens[b]], local.astype(np.float64), np.asarray(offsets, np.float64), parents)
        if not quiet:
            print("{}: MPJPE {} MPEEPE {}".format(os.path.basename(input_paths[b]), m, e))
        results.append(dict(mpjpe=m, mpeepe=e, time=elapsed, poses=poses[: lens[b], b], global_pos=gposs[: lens[b], b], out_path=out_path))
    return results


LOOKAHEAD = 4  # frames of one look-ahead predictor cycle at window 0 (DP_LOOKAHEAD, csrc/dp_internal.h)


def boundary_period(window):
    """Frames between two frames at which a clip can start without an extra predictor call: the window, or the look-ahead cycle
    at window 0."""
    return window if window > 0 else LOOKAHEAD


def slot_schedule(lengths, slots, period):
    """Continuous batching of clips of `lengths` frames over `slots` engine rows.  The first `slots` clips start at frame 0; every
    later clip, in order, takes the slot that frees first (lowest slot on a tie) at the first multiple of `period` at or after that
    slot's clip has ended, so a slot idles at most period - 1 frames.  Returns (starts, total): starts[i] = (slot, first engine
    frame) of clip i, which runs engine frames [first, first + lengths[i]); total = engine frames of the whole run."""
    import heapq

    free = [(0, s) for s in range(min(slots, len(lengths)))]
    starts = []
    for n in lengths:
        t, s = heapq.heappop(free)
        t = -(-t // period) * period
        starts.append((s, t))
        heapq.heappush(free, (t + int(n), s))
    return starts, max((t + int(n) for (_, t), n in zip(starts, lengths)), default=0)


def evaluate_stream(model_path, input_paths, slots, config=None, save=False, seed=2222, initial_latents=None, max_frames=None, device=0,
                    random_temporal=False, predictor_path=0):
    """Many BVH clips through a fixed number of engine rows (continuous batching): a slot whose clip has ended takes the next file
    at the next predictor boundary (slot_schedule), with BatchedDragPose.restart_pose / restart_clips, so the batch stays on the
    lockstep path and no frame is padded beyond the wait for that boundary.  Targets are world-space (targets_world=True) and are
    built per run of frames between two restarts.  Same optimiser settings, metrics and result dicts as evaluate_batch(); frames a
    slot spends waiting are computed and discarded.  predictor_path: 0 = tensor-core predictor, 1 = fp32 CUDA-core kernels."""
    from .engine import BatchedDragPose

    torch.manual_seed(seed)
    np.random.seed(seed)
    cfg = synthetic.TrackerConfig.load(config) if config else synthetic.config_6_trackers()
    bvhs = [Bvh(p) for p in input_paths]
    parents, offsets = bvhs[0].skeleton()
    for b in bvhs[1:]:
        p2, o2 = b.skeleton()
        if list(p2) != list(parents) or not np.allclose(o2, offsets, atol=1e-6):
            raise ValueError("evaluate_stream: all clips must share one skeleton")
    pm = dpm.load_pose_model(model_path, parents)
    tdir = model_path if os.path.isdir(model_path) else os.path.dirname(model_path)
    tm = dpm.load_temporal_model(tdir, allow_random=random_temporal)
    joints, weights = cfg.joints, cfg.tracker_weights
    rots = [b.quaternions() for b in bvhs]
    clips = [motion.ClipData(r, b.positions[:, 0, :], parents, offsets, pm.mean_dqs, pm.std_dqs) for r, b in zip(rots, bvhs)]
    lens = [c.n_frames if max_frames is None else min(max_frames, c.n_frames) for c in clips]
    W = cfg.temporal_future_window
    starts, total = slot_schedule(lens, slots, boundary_period(W))
    N, E = min(slots, len(clips)), len(joints)
    eng = BatchedDragPose(pm, offsets, tm, N, device=device)
    eng.set_predictor_path(predictor_path)
    if initial_latents is not None:
        latent0 = [np.asarray(z, np.float32).reshape(24) for z in initial_latents]
        eps = None
    else:  # one torch draw per clip in clip order, like evaluate_batch; encoded on the device when the clip starts
        eps = [torch.randn(1, dpm.LATENT).numpy() for _ in clips]

    def begin(ids, first):  # clips `ids` start now in their slots
        rows = [starts[i][0] for i in ids]
        state = (np.stack([clips[i].global_pos[0] for i in ids]), np.stack([clips[i].global_rot[0] for i in ids]),
                 np.stack([clips[i].heights[0] for i in ids]))
        if eps is None:
            z = np.stack([latent0[i] for i in ids])
        else:
            z = eng.encode(np.stack([clips[i].dqs[0] for i in ids]), np.concatenate([eps[i] for i in ids]))
        if first:
            eng.set_initial_state(z, *state)
        else:
            assert eng.frames_to_boundary(W) == 0
            eng.restart_clips(rows, z, *state)

    opts = dict(stop_eps_pos=0.01 * 0.01, stop_eps_rot=0.01, max_iter=100, min_loss_incr=0.00001, learning_rate=1e-2, lambda_rot=1,
                lambda_temporal=cfg.lambda_temporal, temporal_future_window=W, joint_adjustment_indices=cfg.joint_adjustment,
                joint_adjustment_weight=cfg.joint_adjustment_weight, targets_world=True)
    poses = [np.empty((n, 88), np.float32) for n in lens]
    gposs = [np.empty((n, 3), np.float32) for n in lens]
    by_start = {}
    for i, (_, t) in enumerate(starts):
        by_start.setdefault(t, []).append(i)
    cuts = sorted(by_start) + [total]
    current = [None] * N  # clip in each slot
    targets = {}  # world-space targets of the clips running now
    elapsed = 0.0
    for a, b in zip(cuts[:-1], cuts[1:]):
        for i in by_start[a]:
            targets.pop(current[starts[i][0]], None)  # the slot's previous clip, kept until now for the frames spent waiting
            current[starts[i][0]] = i
            targets[i] = motion.world_targets(clips[i], pm.mean_q, pm.std_q, parents, offsets, joints, lens[i])
        begin(by_start[a], a == 0)
        tp, tr = np.empty((b - a, N, E, 3), np.float32), np.empty((b - a, N, E, 3, 3), np.float32)
        for s, i in enumerate(current):
            f = np.minimum(np.arange(a, b) - starts[i][1], lens[i] - 1)  # a slot waiting for the boundary repeats its last frame
            tp[:, s], tr[:, s] = targets[i][0][f], targets[i][1][f]
        t0 = time.time()
        p, g = eng.run_frames(tp, tr, joints, weights, **opts)
        elapsed += time.time() - t0
        for s, i in enumerate(current):
            f0, f1 = a - starts[i][1], min(b - starts[i][1], lens[i])
            if f1 > f0:
                poses[i][f0:f1], gposs[i][f0:f1] = p[: f1 - f0, s], g[: f1 - f0, s]
    eng.close()
    results = []
    for i, (bvh, c) in enumerate(zip(bvhs, clips)):
        local = motion.result_local_quats(poses[i], pm.mean_q, pm.std_q, parents)
        out_path = None
        if save:
            os.makedirs("data", exist_ok=True)
            out_path = os.path.join("data", "eval_" + os.path.basename(input_paths[i]))
            write_result_bvh(bvh, local, gposs[i], out_path)
        m, e = motion.mpjpe(rots[i][: lens[i]], local.astype(np.float64), np.asarray(offsets, np.float64), parents)
        results.append(dict(mpjpe=m, mpeepe=e, time=elapsed, poses=poses[i], global_pos=gposs[i], out_path=out_path))
    return results


def write_result_bvh(bvh: Bvh, local_quats, root_pos, path):
    F = local_quats.shape[0]
    with open(path, "w") as fh:
        children = {j: [] for j in range(len(bvh.names))}
        for j in range(1, len(bvh.names)):
            children[bvh.parents[j]].append(j)
        ends = {}
        for p, off in bvh.end_sites:
            ends.setdefault(p, []).append(off)
        lines = ["HIERARCHY"]

        def emit(j, d):
            t = "\t" * d
            o = bvh.raw_offsets[j]
            lines.extend([f"{t}{'ROOT' if j == 0 else 'JOINT'} {bvh.names[j]}", t + "{", f"{t}\tOFFSET {o[0]:.6f} {o[1]:.6f} {o[2]:.6f}",
                          f"{t}\tCHANNELS {len(bvh.channels[j])} " + " ".join(bvh.channels[j])])
            for c in children[j]:
                emit(c, d + 1)
            for off in ends.get(j, []):
                lines.extend([f"{t}\tEnd Site", t + "\t{", f"{t}\t\tOFFSET {off[0]:.6f} {off[1]:.6f} {off[2]:.6f}", t + "\t}"])
            lines.append(t + "}")

        emit(0, 0)
        lines += ["MOTION", f"Frames: {F}", f"Frame Time: {bvh.frame_time:.6f}"]
        eul = [np.degrees(motion.to_euler(local_quats[:, j].astype(np.float64), bvh.rot_order[j])) for j in range(len(bvh.names))]
        rows = []
        for f in range(F):
            vals = []
            for j in range(len(bvh.names)):
                r = 0
                for ch in bvh.channels[j]:
                    if ch.lower().endswith("position"):
                        vals.append(root_pos[f, "xyz".index(ch[0].lower())] if j == 0 else bvh.positions[f, j, "xyz".index(ch[0].lower())])
                    else:
                        vals.append(eul[j][f, r])
                        r += 1
            rows.append(" ".join(f"{v:.6f}" for v in vals))
        fh.write("\n".join(lines) + "\n" + "\n".join(rows) + "\n")


def main():
    ap = argparse.ArgumentParser(description="Evaluate DragPoser (B200 engine)")
    ap.add_argument("model_path", type=str, help="path to the model folder (generator.pt, data.pt[, temporal.pt]) or a folded .npz")
    ap.add_argument("input_path", type=str, help="input .bvh file or a directory (every .bvh in it is evaluated)")
    ap.add_argument("--config", type=str, default=None, help="path to the tracker config file")
    ap.add_argument("--verbose", action="store_true", default=False, help="print additional information")
    ap.add_argument("--batch", action="store_true", default=False,
                    help="directory input: run all clips together as one batch (one engine row per clip, world-space targets)")
    ap.add_argument("--slots", type=int, default=0,
                    help="with --batch: run the clips through this many engine rows, a new clip starting in a slot whose clip has ended")
    ap.add_argument("--random-temporal", action="store_true", default=False,
                    help="temporal.pt is missing: run with the seed-2222 random-init predictor instead of failing like the reference")
    args = ap.parse_args()
    rt = args.random_temporal
    if os.path.isdir(args.input_path) and args.batch:
        files = [os.path.join(args.input_path, fn) for fn in sorted(os.listdir(args.input_path)) if fn.endswith(".bvh")]
        if args.slots > 0:
            results = evaluate_stream(args.model_path, files, args.slots, args.config, save=True, random_temporal=rt)
        else:
            results = evaluate_batch(args.model_path, files, args.config, save=True, quiet=True, random_temporal=rt)
        for fn, r in zip(files, results):
            print("Evaluate {} ------------------------".format(fn))
            print("Evaluate Loss: {}".format(r["mpjpe"] + r["mpeepe"]))
            print("Mean Per Joint Position Error: {}".format(r["mpjpe"]))
            print("Mean End Effector Position Error: {}".format(r["mpeepe"]))
            print("Time: {}".format(r["time"]))
    elif os.path.isdir(args.input_path):
        for fn in sorted(os.listdir(args.input_path)):
            if fn.endswith(".bvh"):
                print("Evaluate {} ------------------------".format(os.path.join(args.input_path, fn)))
                evaluate(args.model_path, os.path.join(args.input_path, fn), args.config, args.verbose, random_temporal=rt)
    else:
        evaluate(args.model_path, args.input_path, args.config, args.verbose, random_temporal=rt)


if __name__ == "__main__":
    main()
