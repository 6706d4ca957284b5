"""GPU: the eval_drag drop-in (BASELINE config #1 on an excerpt) against the reference's own evaluation loop."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")


def test_eval_drag_on_bvh_excerpt_matches_reference(tmp_path, monkeypatch):
    from dragposer_b200 import eval_drag, model, motion
    from dragposer_b200.bvh import Bvh

    monkeypatch.chdir(tmp_path)  # the CLI writes data/eval_<name>.bvh relative to the cwd (train.py:505-508)
    g = np.load(os.path.join(G, "ref_eval_bvh.npz"))
    cfg = tmp_path / "6.json"
    from dragposer_b200 import synthetic
    import json

    c = synthetic.config_6_trackers()
    cfg.write_text(json.dumps(dict(mask=c.mask.tolist(), weights=c.weights.tolist(), enable_joint_adjustment=True,
                                   joint_adjustment_indices=[0, 0], joint_adjustment_weight=1.0, lambda_temporal=0.02,
                                   temporal_future_window=0)))
    res = eval_drag.evaluate(os.path.join(G, "model_dancedb.npz"), os.path.join(G, "example_48f.bvh"), str(cfg), quiet=True,
                             initial_latent=g["latent0"], random_temporal=True)
    d_it = np.abs(res["iterations"] - g["iters"])
    # iteration counts: exact (+-1) while the trajectories still coincide, statistically equal afterwards (see below)
    assert d_it[:8].max() <= 1 and (d_it <= 1).mean() >= 0.9 and d_it.max() <= 5, (res["iterations"], g["iters"])
    pm = model.load_folded_npz(os.path.join(G, "model_dancedb.npz"))
    b = Bvh(os.path.join(G, "example_48f.bvh"))
    par, off = b.skeleton()
    z = np.zeros((48, 3))
    p1, _ = motion.fk_np(motion.result_local_quats(res["poses"], pm.mean_q, pm.std_q, par).astype(np.float64), z, off.astype(np.float64), par)
    p2, _ = motion.fk_np(motion.result_local_quats(g["pose"], pm.mean_q, pm.std_q, par).astype(np.float64), z, off.astype(np.float64), par)
    d = np.abs(p1 - p2).max(axis=(1, 2))
    root = np.abs(res["global_pos"] - g["gpos"]).max()
    rots = b.quaternions()
    m_ref, e_ref = motion.mpjpe(rots, motion.result_local_quats(g["pose"], pm.mean_q, pm.std_q, par).astype(np.float64), off.astype(np.float64), par)
    print(f"eval_drag excerpt: joint diff vs reference, frames 0-7: {d[:8].max()*1e3:.4f} mm, all 48: {d.max()*1e3:.2f} mm; root diff {root*1e3:.4f} mm; "
          f"MPJPE {res['mpjpe']*100:.2f} cm (reference {m_ref*100:.2f}), MPEEPE {res['mpeepe']*100:.2f} cm (reference {e_ref*100:.2f}), "
          f"{48/res['time']:.0f} frames/s")
    # Early-stopped frames run ~2 Adam steps from a FRESH optimiser state, and the first Adam step is lr*sign(g): latent
    # dimensions whose gradient sits in the fp32 noise get a +-lr kick whose sign is not reproducible across
    # implementations, so two fp32-faithful runs drift apart by ~2.5x per frame until they saturate at the ~1.5 cm scale
    # of the method's own error.  The CPU oracle port shows the SAME divergence from the reference on this excerpt
    # (1.6 mm at frame 12, 12-17 mm later; DESIGN.md section 4).  Reproducible: the first frames to 1 mm, the root
    # (snapped by the joint adjustment), the iteration counts and the accuracy metrics.
    assert d[:8].max() < 1e-3 and root < 1e-3
    assert d.max() < 0.05
    assert abs(res["mpjpe"] - m_ref) < 5e-3 and abs(res["mpeepe"] - e_ref) < 5e-3
    assert res["mpjpe"] < 0.06  # a wrong quaternion convention or FK order gives tens of centimetres (SURVEY section 4)
    # the written BVH parses back to the same local rotations
    out = Bvh(res["out_path"])
    q = out.quaternions()
    ref_q = motion.result_local_quats(res["poses"], pm.mean_q, pm.std_q, par)
    dots = np.abs(np.sum(q * ref_q / np.linalg.norm(ref_q, axis=-1, keepdims=True), axis=-1))
    assert dots.min() > 1 - 1e-6


def test_evaluate_batch_world_targets_matches_per_frame_loop(tmp_path, monkeypatch):
    """SURVEY 8(f) rank 1: whole clips streamed with world-absolute targets (the kernel subtracts the current root position)
    against the per-frame host loop of evaluate(); three rows: the clip twice and a ragged 20-frame excerpt."""
    import json

    from dragposer_b200 import eval_drag, model, motion, synthetic
    from dragposer_b200.bvh import Bvh

    monkeypatch.chdir(tmp_path)
    g = np.load(os.path.join(G, "ref_eval_bvh.npz"))
    c = synthetic.config_6_trackers()
    cfg = tmp_path / "6.json"
    cfg.write_text(json.dumps(dict(mask=c.mask.tolist(), weights=c.weights.tolist(), enable_joint_adjustment=True,
                                   joint_adjustment_indices=[0, 0], joint_adjustment_weight=1.0, lambda_temporal=0.02,
                                   temporal_future_window=0)))
    src = os.path.join(G, "example_48f.bvh")
    short = tmp_path / "short_20f.bvh"
    lines = open(src).read().split("\n")
    m = next(i for i, l in enumerate(lines) if l.strip().startswith("Frames:"))
    short.write_text("\n".join(lines[:m] + ["Frames: 20"] + lines[m + 1 : m + 2 + 20]) + "\n")
    npz = os.path.join(G, "model_dancedb.npz")
    one = eval_drag.evaluate(npz, src, str(cfg), quiet=True, initial_latent=g["latent0"], save=False, random_temporal=True)
    res = eval_drag.evaluate_batch(npz, [src, src, str(short)], str(cfg), initial_latents=[g["latent0"]] * 3, save=True, random_temporal=True)
    assert len(res) == 3 and res[0]["poses"].shape == (48, 88) and res[2]["poses"].shape == (20, 88)
    assert np.array_equal(res[0]["poses"], res[1]["poses"])  # identical rows give identical results
    assert np.array_equal(res[2]["poses"][:20], res[0]["poses"][:20])  # padding of the short clip does not leak into its frames
    pm = model.load_folded_npz(npz)
    par, off = Bvh(src).skeleton()
    z = np.zeros((48, 3))
    p1, _ = motion.fk_np(motion.result_local_quats(res[0]["poses"], pm.mean_q, pm.std_q, par).astype(np.float64), z, off.astype(np.float64), par)
    p2, _ = motion.fk_np(motion.result_local_quats(one["poses"], pm.mean_q, pm.std_q, par).astype(np.float64), z, off.astype(np.float64), par)
    d = np.abs(p1 - p2).max(axis=(1, 2))
    root = np.abs(res[0]["global_pos"] - one["global_pos"]).max()
    print(f"evaluate_batch vs per-frame loop: joint diff frames 0-7 {d[:8].max()*1e3:.4f} mm, all {d.max()*1e3:.2f} mm, root {root*1e3:.4f} mm; "
          f"MPJPE {res[0]['mpjpe']*100:.2f} vs {one['mpjpe']*100:.2f} cm")
    # same trajectory sensitivity as above: (root - origin) + R o is rounded differently from (root + R o) - origin
    assert d[:8].max() < 1e-3 and root < 1e-3 and d.max() < 0.05
    assert abs(res[0]["mpjpe"] - one["mpjpe"]) < 5e-3 and abs(res[0]["mpeepe"] - one["mpeepe"]) < 5e-3
    assert os.path.exists(res[2]["out_path"]) and Bvh(res[2]["out_path"]).quaternions().shape[0] == 20


def test_evaluate_batch_default_start_uses_device_encoder(tmp_path, monkeypatch):
    """Without recorded latents evaluate_batch encodes the first poses on the device with torch-drawn eps (seed 2222):
    runs end to end, finite, and accurate on the excerpt."""
    from dragposer_b200 import eval_drag

    monkeypatch.chdir(tmp_path)
    src = os.path.join(G, "example_48f.bvh")
    res = eval_drag.evaluate_batch(os.path.join(G, "model_dancedb.npz"), [src, src], None, max_frames=16, random_temporal=True)
    assert len(res) == 2 and res[0]["poses"].shape == (16, 88) and np.isfinite(res[0]["poses"]).all()
    assert not np.array_equal(res[0]["poses"], res[1]["poses"])  # two different reparameterisation draws
    assert res[0]["mpjpe"] < 0.06 and res[1]["mpjpe"] < 0.06


def test_device_pose_error_matches_host_metrics(tmp_path):
    """SURVEY 8(f) rank 2: MPJPE / MPEEPE on the device against motion.mpjpe (the host restatement of eval_metrics.py)."""
    from dragposer_b200 import model, motion
    from dragposer_b200.bvh import Bvh
    from dragposer_b200.engine import BatchedDragPose

    g = np.load(os.path.join(G, "ref_eval_bvh.npz"))
    pm = model.load_folded_npz(os.path.join(G, "model_dancedb.npz"))
    b = Bvh(os.path.join(G, "example_48f.bvh"))
    par, off = b.skeleton()
    tm = model.temporal_from_state(model.random_temporal_state(2222))
    clip = motion.ClipData(b.quaternions(), b.positions[:, 0, :], par, off, pm.mean_dqs, pm.std_dqs)
    # ground truth in the engine's pose format: quaternion half of the dual quats, root slot = standardised world root rotation
    gt = clip.dqs.reshape(48, 22, 8)[:, :, :4].reshape(48, 88).copy()
    gt[:, :4] = (clip.global_rot - pm.mean_q[:4]) / pm.std_q[:4]
    eng = BatchedDragPose(pm, off, tm, 64)
    mp, me = eng.pose_error(g["pose"], gt)
    eng.close()
    res_local = motion.result_local_quats(g["pose"], pm.mean_q, pm.std_q, par).astype(np.float64)
    want_m, want_e = motion.mpjpe(b.quaternions(), res_local, off.astype(np.float64), par)
    print(f"device MPJPE {mp.mean()*100:.4f} cm (host {want_m*100:.4f}), MPEEPE {me.mean()*100:.4f} cm (host {want_e*100:.4f})")
    assert abs(mp.mean() - want_m) < 1e-5 and abs(me.mean() - want_e) < 1e-5
    same_m, same_e = BatchedDragPose(pm, off, tm, 64).pose_error(gt, gt)
    assert same_m.max() == 0.0 and same_e.max() == 0.0


def test_full_clip_known_answer_matches_reference(tmp_path, monkeypatch):
    """BASELINE config #1 / SURVEY section 4 known answer: the whole of example.bvh (5 052 frames, 6-tracker config, early stopping
    on) through both drop-in evaluation paths, against the metrics the UNMODIFIED reference produced for the same clip and the same
    start latent (oracle/make_golden.py evalfull: train.result_to_bvh + eval_metrics.eval_pos_error).  Late-clip poses are not
    comparable frame by frame (DESIGN.md section 4); the accuracy metrics, the root track (snapped to the hip tracker by the joint
    adjustment every frame) and the iteration statistics are."""
    import gzip
    import json

    from dragposer_b200 import eval_drag, synthetic

    monkeypatch.chdir(tmp_path)
    g = np.load(os.path.join(G, "ref_eval_full.npz"))
    src = tmp_path / "example.bvh"
    packed = b""
    for part in ("example_full.bvh.gz.1", "example_full.bvh.gz.2"):  # the gzip file cut in two, each piece below 1 MB
        with open(os.path.join(G, part), "rb") as fi:
            packed += fi.read()
    src.write_bytes(gzip.decompress(packed))
    c = synthetic.config_6_trackers()
    cfg = tmp_path / "6.json"
    cfg.write_text(json.dumps(dict(mask=c.mask.tolist(), weights=c.weights.tolist(), enable_joint_adjustment=True,
                                   joint_adjustment_indices=[0, 0], joint_adjustment_weight=1.0, lambda_temporal=0.02,
                                   temporal_future_window=0)))
    npz = os.path.join(G, "model_dancedb.npz")
    ref_m, ref_e, ref_it = float(g["mpjpe"]), float(g["mpeepe"]), g["iters"].astype(np.float64)
    one = eval_drag.evaluate(npz, str(src), str(cfg), quiet=True, initial_latent=g["latent0"], save=True, random_temporal=True)
    assert one["poses"].shape == (5052, 88) and os.path.exists(one["out_path"])
    bat = eval_drag.evaluate_batch(npz, [str(src)], str(cfg), initial_latents=[g["latent0"]], random_temporal=True)[0]
    for name, r in (("eval_drag.evaluate (per-frame DragPose.run)", one), ("eval_drag.evaluate_batch (world targets, run_frames)", bat)):
        root = np.abs(r["global_pos"] - g["gpos"]).max()
        print(f"{name}: MPJPE {r['mpjpe']*100:.3f} cm (reference {ref_m*100:.3f}), MPEEPE {r['mpeepe']*100:.3f} cm (reference {ref_e*100:.3f}), "
              f"root track max diff {root*1e3:.3f} mm" + (f", mean iterations {r['iterations'].mean():.2f} (reference {ref_it.mean():.2f}), "
              f"{5052 / r['time']:.0f} frames/s (reference: {5052 / float(g['seconds_one_core']):.1f} on one core)" if "iterations" in r else ""))
        assert abs(r["mpjpe"] - ref_m) < 3e-3 and abs(r["mpeepe"] - ref_e) < 3e-3
        assert root < 2e-3
    assert abs(one["iterations"].mean() - ref_it.mean()) < 0.1 * ref_it.mean()
    assert np.abs(one["iterations"][:8] - g["iters"][:8]).max() <= 1
