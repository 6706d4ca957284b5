"""GPU: per-clip restarts of a running batch (dp_engine_restart_clips) against fresh engines that start exactly the restarted clips,
and continuous batching of BVH clips (eval_drag.evaluate_stream) against one-clip runs."""
import gzip
import os

import numpy as np
import pytest

import dragposer_port as port
from dragposer_b200 import synthetic
from dragposer_b200._lib import EngineError

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")

EARLY = dict(stop_eps_pos=0.01 * 0.01, stop_eps_rot=0.01, max_iter=100, min_loss_incr=0.00001, learning_rate=1e-2)
FIXED = dict(stop_eps_pos=-1.0, stop_eps_rot=-1.0, max_iter=100, min_loss_incr=-float("inf"), learning_rate=1e-2)
B, T = 64, 40
# two non-contiguous sets, restarted mid-window (window 16: indices 5 and 6) and mid-look-ahead-cycle (window 0: rows 1 and 2)
SETS = ((5, [3, 10, 17, 40, 41, 63]), (22, [1, 8, 30, 31, 55]))


def _start(n):
    return np.zeros((n, 3), np.float32), np.tile(np.float32([[1, 0, 0, 0]]), (n, 1)), np.zeros((n, 6), np.float32)


def _scenario(pose_model, offsets):
    cfg = synthetic.config_6_trackers()
    base = synthetic.make_workload(pose_model, offsets, cfg, B, T)
    fresh = [synthetic.make_workload(pose_model, offsets, cfg, len(ids), T - f, first_clip=1000 * (k + 1)) for k, (f, ids) in enumerate(SETS)]
    tp, tr = base["tgt_pos"].copy(), base["tgt_rot"].copy()
    for (f, ids), w in zip(SETS, fresh):
        tp[f:, ids], tr[f:, ids] = w["tgt_pos"], w["tgt_rot"]
    return cfg, base, fresh, tp, tr


def _run(eng, latent0, tp, tr, joints, weights, kw, window, restarts=None):
    """Frame by frame; restarts = {frame: (ids, latent)} issued before that frame.  -> poses, gpos, iters (T, n, .)"""
    eng.set_initial_state(latent0, *_start(latent0.shape[0]))
    ps, gs, its = [], [], []
    for t in range(tp.shape[0]):
        if restarts and t in restarts:
            ids, z = restarts[t]
            eng.restart_clips(ids, z, *_start(len(ids)))
        p, g = eng.run(tp[t], tr[t], joints, weights, temporal_future_window=window, **kw)
        ps.append(p), gs.append(g), its.append(eng.frame_stats()[0])
    return np.stack(ps), np.stack(gs), np.stack(its)


@pytest.mark.parametrize("window", [0, 16])
@pytest.mark.parametrize("path", [1, 3], ids=["fp32", "tcgen05-fp16x2"])
def test_restarted_clips_are_bitwise_fresh_engines_and_the_others_untouched(engine_factory, pose_model, model_npz, window, path):
    """fp32 predictor, fixed decoder path: from its restart frame on, every restarted clip is bit for bit a fresh engine that
    starts exactly those clips with the same states and targets; every other clip is bit for bit the run without restarts;
    the target rows a caller reads back and the per-clip indices agree with the fresh engines."""
    cfg, base, fresh, tp, tr = _scenario(pose_model, model_npz["offsets"])
    kw = dict(EARLY, lambda_rot=1, lambda_temporal=0.15, joint_adjustment_indices=cfg.joint_adjustment,
              joint_adjustment_weight=cfg.joint_adjustment_weight, decoder_path=path)
    joints, weights = base["joints"], base["weights"]

    def engine(n):
        e = engine_factory(n)
        e.set_predictor_path(1)
        return e

    eng = engine(B)
    out = _run(eng, base["latent0"], tp, tr, joints, weights, kw, window, {f: (ids, w["latent0"]) for (f, ids), w in zip(SETS, fresh)})
    st, idx = eng.state(window), eng.clip_index(window)
    ref = _run(engine(B), base["latent0"], base["tgt_pos"], base["tgt_rot"], joints, weights, kw, window)
    touched = sorted(sum((ids for _, ids in SETS), []))
    keep = [c for c in range(B) if c not in touched]
    for a, b in zip(out, ref):
        assert np.array_equal(a[:, keep], b[:, keep])
    for (f, ids), w in zip(SETS, fresh):
        order = np.argsort(ids)
        ids_sorted = np.asarray(ids)[order]
        e1 = engine(len(ids))
        one = _run(e1, w["latent0"][order], w["tgt_pos"][:, order], w["tgt_rot"][:, order], joints, weights, kw, window)
        for a, b in zip(out, one):
            assert np.isfinite(a).all() and np.array_equal(a[f:, ids_sorted], b)
        s1 = e1.state(window)
        assert np.array_equal(st["target_buf"][ids_sorted], s1["target_buf"])
        assert np.array_equal(idx[ids_sorted], e1.clip_index(window))
        for k in ("latent", "global_pos", "latent_buf", "disp_buf", "height_buf"):
            assert np.array_equal(st[k][ids_sorted], s1[k])
    if window:
        assert sorted(set(idx.tolist())) == sorted({(T - f) % window for f, _ in SETS} | {T % window})


def _pose_positions(pw, pose):
    import torch

    q = torch.as_tensor(pose) * pw.std_q + pw.mean_q
    q = q.reshape(q.shape[0], 22, 4)
    pos, _ = port.fk_chain(port.root_to_local(q, pw.parents), torch.zeros(q.shape[0], 3), pw.offsets, pw.parents)
    return pos.numpy()


@pytest.mark.parametrize("window", [0, 16])
def test_restarts_with_the_tensor_core_predictor(engine_factory, pose_model, model_npz, port_weights, window):
    """Default (tcgen05) predictor, 6 trackers, 100 fixed iterations: a subset predictor call may see other tile fills than the
    fresh engine's call, so the target latents are held to the predictor's own bar (2e-5) and the joints to 1 mm."""
    cfg, base, fresh, tp, tr = _scenario(pose_model, model_npz["offsets"])
    kw = dict(FIXED, lambda_rot=1, lambda_temporal=0.15, joint_adjustment_indices=cfg.joint_adjustment,
              joint_adjustment_weight=cfg.joint_adjustment_weight)
    joints, weights = base["joints"], base["weights"]
    eng = engine_factory(B)
    out = _run(eng, base["latent0"], tp, tr, joints, weights, kw, window, {f: (ids, w["latent0"]) for (f, ids), w in zip(SETS, fresh)})
    st = eng.state(window)
    for (f, ids), w in zip(SETS, fresh):
        order = np.argsort(ids)
        ids_sorted = np.asarray(ids)[order]
        e1 = engine_factory(len(ids))
        one = _run(e1, w["latent0"][order], w["tgt_pos"][:, order], w["tgt_rot"][:, order], joints, weights, kw, window)
        d_t = np.abs(st["target_buf"][ids_sorted] - e1.state(window)["target_buf"]).max()
        p_a = _pose_positions(port_weights, out[0][f:, ids_sorted].reshape(-1, 88))
        p_b = _pose_positions(port_weights, one[0].reshape(-1, 88))
        d_p = np.abs(p_a - p_b).max()
        print(f"window {window}, restart at frame {f}: target latents max diff {d_t:.2e}, joints max diff {d_p * 1e3:.4f} mm")
        assert d_t <= 2e-5 and d_p <= 1e-3


@pytest.mark.parametrize("window", [0, 16])
def test_aligned_restarts_add_no_predictor_launches(engine_factory, pose_model, model_npz, window):
    """Restarts at a boundary (frames_to_boundary == 0) keep one phase for every clip: the launch count grows by the one reset
    kernel of each restart and by nothing else.  320 clips: above the small-batch mode's early predictor call."""
    n, frames = 320, 36
    cfg = synthetic.config_6_trackers()
    wl = synthetic.make_workload(pose_model, model_npz["offsets"], cfg, n, frames)
    kw = dict(FIXED, max_iter=4, lambda_temporal=0.15, temporal_future_window=window)
    period = window or 4
    counts, restarts = [], 0
    for restart in (False, True):
        eng = engine_factory(n)
        eng.set_initial_state(wl["latent0"], *_start(n))
        c0 = eng.launch_count()
        for t in range(frames):
            assert eng.frames_to_boundary(window) == (-t) % period
            if restart and t and t % period == 0:
                ids = np.arange(t % 7, n, 9)
                eng.restart_clips(ids, wl["latent0"][ids], *_start(len(ids)))
                restarts += 1
                idx = eng.clip_index(window)
                assert (idx == 0).all()  # phases stay uniform
            eng.run(wl["tgt_pos"][t], wl["tgt_rot"][t], wl["joints"], wl["weights"], **kw)
        counts.append(eng.launch_count() - c0)
        eng.close()
    assert restarts > 0 and counts[1] - counts[0] == restarts, (counts, restarts)


@pytest.mark.parametrize("frame", [16, 30], ids=["aligned", "unaligned"])
def test_restart_while_an_early_predictor_call_is_in_flight(engine_factory, pose_model, model_npz, monkeypatch, frame):
    """Small-batch streaming (8 clips, window 16): the predictor call of frame 16 (32) is issued at frame 13 (29).  A restart before
    frame 16 (aligned) or 30 (mid-window) voids it; the results are bit for bit those of an engine without early calls."""
    cfg = synthetic.config_3_trackers()
    n, frames = 8, 40
    wl = synthetic.make_workload(pose_model, model_npz["offsets"], cfg, n, frames)
    new = synthetic.make_workload(pose_model, model_npz["offsets"], cfg, 3, 1, first_clip=77)
    kw = dict(EARLY, lambda_rot=1, lambda_temporal=cfg.lambda_temporal, joint_adjustment_indices=cfg.joint_adjustment,
              joint_adjustment_weight=cfg.joint_adjustment_weight)
    outs = []
    for prefetch in ("1", "0"):
        monkeypatch.setenv("DP_PRED_PREFETCH", prefetch)  # read when the engine is created
        eng = engine_factory(n)
        res = _run(eng, wl["latent0"], wl["tgt_pos"], wl["tgt_rot"], wl["joints"], wl["weights"], kw, 16, {frame: ([1, 4, 6], new["latent0"])})
        outs.append(res + (eng.state(16)["target_buf"], eng.clip_index(16)))
        eng.close()
    for a, b in zip(outs[0], outs[1]):
        assert np.array_equal(a, b)


def test_restart_errors_leave_the_engine_unchanged(engine_factory, pose_model, model_npz):
    cfg = synthetic.config_3_trackers()
    n = 16
    wl = synthetic.make_workload(pose_model, model_npz["offsets"], cfg, n, 8)
    kw = dict(FIXED, max_iter=4, lambda_temporal=cfg.lambda_temporal, temporal_future_window=16)
    z = wl["latent0"]
    eng = engine_factory(n)
    with pytest.raises(EngineError, match="error -3"):  # before dp_engine_init_clips
        eng.restart_clips([0], z[:1], *_start(1))
    eng.set_initial_state(z, *_start(n))
    for t in range(3):
        eng.run(wl["tgt_pos"][t], wl["tgt_rot"][t], wl["joints"], wl["weights"], **kw)

    def snapshot():
        s = eng.state(16)
        return [s[k] for k in ("latent", "global_pos", "global_rot", "latent_buf", "disp_buf", "height_buf", "target_buf")] + [
            np.asarray(s["current_index"]), eng.clip_index(16), np.asarray(eng.frames_to_boundary(16))]

    def unchanged(before):
        for a, b in zip(before, snapshot()):
            assert np.array_equal(a, b)

    before = snapshot()
    for ids in ([2, 5, 2], [3, n], [-1]):
        with pytest.raises(EngineError, match="error -1"):  # duplicate or out-of-range ids
            eng.restart_clips(ids, z[: len(ids)], *_start(len(ids)))
        unchanged(before)
    eng.restart_clips([2, 9], z[[3, 4]], *_start(2))  # mid-window: phases are now mixed
    idx = eng.clip_index(16)
    assert idx[2] == idx[9] == 0 and (np.delete(idx, [2, 9]) == 3).all()
    assert eng.frames_to_boundary(16) == 0
    before = snapshot()
    with pytest.raises(EngineError, match="error -3"):
        eng.run(wl["tgt_pos"][3], wl["tgt_rot"][3], wl["joints"], wl["weights"], **dict(kw, temporal_future_window=8))
    unchanged(before)
    with pytest.raises(EngineError, match="error -3"):
        eng.predict_targets(16)
    unchanged(before)
    with pytest.raises(EngineError, match="error -3"):
        eng.clip_index(8)
    eng.run(wl["tgt_pos"][3], wl["tgt_rot"][3], wl["joints"], wl["weights"], **kw)  # the window it runs at still works
    assert eng.frames_to_boundary(16) == 12  # the next frame whose index is some clip's phase: index 0 of the untouched clips


def _excerpts(tmp_path, n, lo, hi, seed):
    src = b""
    for part in ("example_full.bvh.gz.1", "example_full.bvh.gz.2"):
        with open(os.path.join(G, part), "rb") as fi:
            src += fi.read()
    lines = gzip.decompress(src).decode().split("\n")
    m = next(i for i, l in enumerate(lines) if l.strip().startswith("Frames:"))
    total = int(lines[m].split()[1])
    rng = np.random.default_rng(seed)
    paths = []
    for i in range(n):
        k = int(rng.integers(lo, hi + 1))
        a = int(rng.integers(0, total - k))
        p = tmp_path / f"excerpt_{i:02d}.bvh"
        p.write_text("\n".join(lines[:m] + [f"Frames: {k}", lines[m + 1]] + lines[m + 2 + a : m + 2 + a + k]) + "\n")
        paths.append(str(p))
    return paths


def _one_clip(npz, path, latent, predictor_path):
    """The clip alone in a one-clip BatchedDragPose, same settings as evaluate_stream."""
    from dragposer_b200 import model as dpm
    from dragposer_b200 import motion
    from dragposer_b200.bvh import Bvh
    from dragposer_b200.engine import BatchedDragPose

    cfg = synthetic.config_6_trackers()
    b = Bvh(path)
    par, off = b.skeleton()
    pm = dpm.load_pose_model(npz, par)
    tm = dpm.load_temporal_model(os.path.dirname(npz), allow_random=True)
    clip = motion.ClipData(b.quaternions(), b.positions[:, 0, :], par, off, pm.mean_dqs, pm.std_dqs)
    tp, tr = motion.world_targets(clip, pm.mean_q, pm.std_q, par, off, cfg.joints)
    eng = BatchedDragPose(pm, off, tm, 1)
    eng.set_predictor_path(predictor_path)
    eng.set_initial_state(latent.reshape(1, 24), clip.global_pos[:1], clip.global_rot[:1], clip.heights[:1])
    p, g = eng.run_frames(tp[:, None], tr[:, None], cfg.joints, cfg.tracker_weights, stop_eps_pos=0.01 * 0.01, stop_eps_rot=0.01,
                          max_iter=100, min_loss_incr=0.00001, learning_rate=1e-2, lambda_rot=1, lambda_temporal=cfg.lambda_temporal,
                          temporal_future_window=cfg.temporal_future_window, joint_adjustment_indices=cfg.joint_adjustment,
                          joint_adjustment_weight=cfg.joint_adjustment_weight, targets_world=True)
    eng.close()
    local = motion.result_local_quats(p[:, 0], pm.mean_q, pm.std_q, par)
    m, _ = motion.mpjpe(b.quaternions(), local.astype(np.float64), np.asarray(off, np.float64), par)
    return p[:, 0], g[:, 0], m


def test_evaluate_stream_equals_one_clip_runs(tmp_path, monkeypatch):
    """8 slots, 20 excerpts of 40-400 frames: every clip, started in a slot at a look-ahead boundary while the other slots run on,
    gives bit for bit the poses of a one-clip engine run (fp32 predictor), and with the tensor-core predictor its MPJPE is within
    0.05 cm of that run's."""
    from dragposer_b200 import eval_drag

    monkeypatch.chdir(tmp_path)
    npz = os.path.join(G, "model_dancedb.npz")
    paths = _excerpts(tmp_path, 20, 40, 400, 5)
    lat = np.random.default_rng(9).standard_normal((20, 24)).astype(np.float32) * np.float32(0.5)
    for predictor_path in (1, 0):
        res = eval_drag.evaluate_stream(npz, paths, 8, initial_latents=list(lat), random_temporal=True, predictor_path=predictor_path)
        assert len(res) == 20
        worst = 0.0
        for i, (p, r) in enumerate(zip(paths, res)):
            poses, gpos, m = _one_clip(npz, p, lat[i], predictor_path)
            assert r["poses"].shape == poses.shape
            if predictor_path == 1:
                assert np.array_equal(r["poses"], poses) and np.array_equal(r["global_pos"], gpos), i
            worst = max(worst, abs(r["mpjpe"] - m))
        print(f"evaluate_stream, predictor path {predictor_path}: worst MPJPE difference to one-clip runs {worst * 100:.4f} cm")
        assert worst < 5e-4
