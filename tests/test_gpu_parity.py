"""GPU parity tests: the CUDA engine (through the dp_engine C ABI) against the golden
vectors recorded from the unmodified reference and against the CPU oracle.

Tolerances (north_star): per-iteration latent-gradient relative error <= 1e-4, final
per-joint positions within 1 mm.  The reference's OWN fp32 gradient differs from a
float64 evaluation by ~1.3e-7 absolute (it standardises/de-standardises by 1/std up
to 1700x), so the comparison against recorded reference gradients carries that
absolute floor: |g - g_ref| <= 1e-4 |g_ref| + 5e-7.
"""
import os

import numpy as np
import pytest
import torch

import dragposer_port as port
from dragposer_b200 import synthetic

pytestmark = pytest.mark.gpu

FIXED = dict(stop_eps_pos=-1.0, stop_eps_rot=-1.0, max_iter=100, min_loss_incr=-float("inf"), learning_rate=1e-2)
EARLY = dict(stop_eps_pos=0.01 * 0.01, stop_eps_rot=0.01, max_iter=100, min_loss_incr=0.00001, learning_rate=1e-2)
GRAD_REL, GRAD_FLOOR, POS_TOL = 1e-4, 5e-7, 1e-3


def pose_positions(pw, pose_std, root_pos=None):
    """Standardised output pose (B,88) -> joint positions (B,22,3) in metres (root at origin)."""
    q = torch.as_tensor(pose_std) * pw.std_q + pw.mean_q
    q = q.reshape(q.shape[0], 22, 4)
    local = port.root_to_local(q, pw.parents)
    pos, _ = port.fk_chain(local, torch.zeros(q.shape[0], 3), pw.offsets, pw.parents)
    return pos.numpy()


@pytest.mark.parametrize("path", [1, 3], ids=["fp32", "tcgen05-fp16x2"])
def test_gradient_teacher_forced_vs_reference(golden_dir, engine_factory, port_weights, path):
    g = np.load(os.path.join(golden_dir, "ref_trace_6trk.npz"))
    eng = engine_factory(512)
    worst_rel, worst_f64 = 0.0, 0.0
    for tag in ("fixed", "early"):
        F, Cn = g[f"{tag}_iters"].shape
        for t in range(F):
            for c in range(Cn):
                n = int(g[f"{tag}_iters"][t, c])
                lat = g[f"{tag}_latent"][t, c, :n]
                args = dict(global_rot=np.tile(g[f"{tag}_grot"][t, c], (n, 1)), tgt_latent=np.tile(g[f"{tag}_tgt_latent"][t, c], (n, 1)),
                            tgt_pos=np.tile(g["tgt_pos"][t, c], (n, 1, 1)), tgt_rot=np.tile(g["tgt_rot"][t, c], (n, 1, 1, 1)),
                            joints=g["joints"], weights=g["weights"], lambda_rot=1.0, lambda_temporal=0.02)
                r = eng.eval_gradient(lat, decoder_path=path, **args)
                ref = g[f"{tag}_grad"][t, c, :n]
                err = np.linalg.norm(r["grad"] - ref, axis=1)
                bound = GRAD_REL * np.linalg.norm(ref, axis=1) + GRAD_FLOOR
                assert (err <= bound).all(), (tag, t, c, float((err / bound).max()))
                worst_rel = max(worst_rel, float((err / np.linalg.norm(ref, axis=1)).max()))
                # losses against the recorded reference values
                np.testing.assert_allclose(r["lp"], g[f"{tag}_loss"][t, c, :n, 0], rtol=2e-4, atol=1e-8)
                np.testing.assert_allclose(r["lr"], g[f"{tag}_loss"][t, c, :n, 1], rtol=2e-4, atol=1e-8)
                np.testing.assert_allclose(r["lt"], g[f"{tag}_loss"][t, c, :n, 2], rtol=2e-4, atol=1e-9)
                # float64 truth: the engine must be at least as close to it as 1e-4 relative (+floor)
                pw64 = port.PortWeights(np.load(os.path.join(golden_dir, "model_dancedb.npz")), dtype=torch.float64)
                t64 = port.loss_and_grad(pw64, lat, args["global_rot"], args["tgt_pos"], args["tgt_rot"], args["tgt_latent"],
                                         g["joints"], g["weights"], lambda_rot=1.0, lambda_temporal=0.02, dtype=torch.float64)
                e64 = np.linalg.norm(r["grad"] - t64["grad"], axis=1)
                assert (e64 <= GRAD_REL * np.linalg.norm(t64["grad"], axis=1) + GRAD_FLOOR).all()
                worst_f64 = max(worst_f64, float((e64 / np.linalg.norm(t64["grad"], axis=1)).max()))
    print(f"worst grad rel err vs reference fp32 {worst_rel:.2e}, vs float64 truth {worst_f64:.2e}")


@pytest.mark.parametrize("path", [1, 3], ids=["fp32", "tcgen05-fp16x2"])
def test_gradient_random_states_vs_float64(golden_dir, engine_factory, pose_model, model_npz, path):
    """20 random states (like SURVEY's probe): relative error <= 1e-4 with no floor, for both decoder paths."""
    rng = np.random.default_rng(11)
    n = 20
    cfg = synthetic.config_6_trackers()
    wl = synthetic.make_workload(pose_model, model_npz["offsets"], cfg, n, 1)
    lat = wl["latent0"] + 0.2 * rng.standard_normal((n, 24)).astype(np.float32)
    grot = rng.standard_normal((n, 4)).astype(np.float32)
    grot /= np.linalg.norm(grot, axis=1, keepdims=True)
    tl = rng.standard_normal((n, 24)).astype(np.float32) * 0.3
    eng = engine_factory(512)
    r = eng.eval_gradient(lat, grot, tl, wl["tgt_pos"][0], wl["tgt_rot"][0], wl["joints"], wl["weights"], lambda_rot=1.0,
                          lambda_temporal=0.02, decoder_path=path)
    pw64 = port.PortWeights(model_npz, dtype=torch.float64)
    t64 = port.loss_and_grad(pw64, lat, grot, wl["tgt_pos"][0], wl["tgt_rot"][0], tl, wl["joints"], wl["weights"],
                             lambda_rot=1.0, lambda_temporal=0.02, dtype=torch.float64)
    rel = np.linalg.norm(r["grad"] - t64["grad"], axis=1) / np.linalg.norm(t64["grad"], axis=1)
    print("decoder path %d random-state grad rel err: max %.2e median %.2e" % (path, rel.max(), np.median(rel)))
    assert rel.max() <= GRAD_REL
    np.testing.assert_allclose(r["pos"], t64["pos"], atol=2e-6)


@pytest.mark.parametrize("path", [1, 3], ids=["fp32", "tcgen05-fp16x2"])
@pytest.mark.parametrize("n_trk", [2, 22], ids=["two-trackers", "every-joint-tracked"])
def test_gradient_tracker_count_extremes_vs_float64(engine_factory, pose_model, model_npz, path, n_trk):
    """Mask handling at its extremes: the smallest set the reference can run (E = 2) and all 22 joints tracked, per-clip
    tracker tables (not shared), random weights; loss values, gradient and joint positions against the float64 port."""
    rng = np.random.default_rng(100 + n_trk)
    n = 24
    offsets = model_npz["offsets"]
    joints = np.stack([rng.permutation(22)[:n_trk] for _ in range(n)]).astype(np.int32)
    joints.sort(axis=1)
    weights = rng.uniform(0.2, 1.5, (n, n_trk, 2)).astype(np.float32)
    lat = (0.4 * rng.standard_normal((n, 24))).astype(np.float32)
    lat_t = lat + (0.1 * rng.standard_normal((n, 24))).astype(np.float32)
    p_t, R_t = synthetic.pose_fk_np(pose_model, offsets, pose_model.decode_np(lat_t))
    tp = np.take_along_axis(p_t, joints[:, :, None], 1).astype(np.float32)
    tr = np.take_along_axis(R_t, joints[:, :, None, None], 1).astype(np.float32)
    grot = np.tile(np.float32([1, 0, 0, 0]), (n, 1))
    tl = (0.3 * rng.standard_normal((n, 24))).astype(np.float32)
    eng = engine_factory(64)
    r = eng.eval_gradient(lat, grot, tl, tp, tr, joints, weights, lambda_rot=1.0, lambda_temporal=0.05, decoder_path=path)
    pw64 = port.PortWeights(model_npz, dtype=torch.float64)
    t64 = port.loss_and_grad(pw64, lat, grot, tp, tr, tl, joints, weights, lambda_rot=1.0, lambda_temporal=0.05, dtype=torch.float64)
    rel = np.linalg.norm(r["grad"] - t64["grad"], axis=1) / np.linalg.norm(t64["grad"], axis=1)
    worst = rel.max()
    assert worst <= GRAD_REL
    np.testing.assert_allclose(r["pos"], t64["pos"], atol=2e-6)
    np.testing.assert_allclose(np.stack([r["lp"], r["lr"], r["lt"]]), np.stack([t64["lp"], t64["lr"], t64["lt"]]), rtol=1e-4, atol=1e-7)  # losses are sums of squared small differences
    print(f"decoder path {path}, {n_trk} trackers per clip: worst gradient rel err {worst:.2e}")


@pytest.mark.parametrize("path", [1, 3], ids=["fp32", "tcgen05-fp16x2"])
@pytest.mark.parametrize("tag,opt,n_frames", [("fixed", FIXED, 2), ("early", EARLY, 6)])
def test_frames_6_trackers_vs_reference(golden_dir, engine_factory, port_weights, tag, opt, n_frames, path):
    g = np.load(os.path.join(golden_dir, "ref_trace_6trk.npz"))
    cfg = synthetic.config_6_trackers()
    eng = engine_factory(512)
    B = g["latent0"].shape[0]
    eng.set_initial_state(g["latent0"], np.zeros((B, 3)), np.tile([[1.0, 0, 0, 0]], (B, 1)), np.zeros((B, 6)))
    eng.enable_trace(True)
    worst_late = 0.0
    for t in range(n_frames):
        pose, gpos = eng.run(g["tgt_pos"][t], g["tgt_rot"][t], g["joints"], g["weights"], lambda_rot=1,
                             lambda_temporal=cfg.lambda_temporal, temporal_future_window=cfg.temporal_future_window,
                             joint_adjustment_indices=cfg.joint_adjustment, joint_adjustment_weight=cfg.joint_adjustment_weight,
                             decoder_path=path, **opt)
        assert eng.last_decoder_path() == path
        iters, losses = eng.frame_stats()
        ref_iters = g[f"{tag}_iters"][t]
        if tag == "fixed":
            assert (iters == 100).all()
        else:  # early stop decisions are float compares near thresholds: allow a +-1 slip, positions still within 1 mm
            assert np.abs(iters - ref_iters).max() <= 1, (t, iters, ref_iters)
        dpos = np.abs(pose_positions(port_weights, pose) - pose_positions(port_weights, g[f"{tag}_pose"][t])).max()
        dg = np.abs(gpos - g[f"{tag}_gpos"][t]).max()
        print(f"{tag} frame {t}: iters {iters} ref {ref_iters} max joint diff {dpos*1e3:.4f} mm root diff {dg*1e3:.4f} mm")
        assert dpos <= POS_TOL and dg <= POS_TOL
        # per-iteration trajectory: latents stay close to the reference's.  This is a LOOSE guard by nature -- the first Adam step
        # is lr * sign(g), so a latent dimension whose gradient sits in the fp32 noise takes a +-lr = 1e-2 kick whose sign two
        # faithful implementations need not agree on; the kick decays as Adam's moments fill.  The real per-iteration guard is the
        # teacher-forced gradient test above (1e-4 relative at the reference's own latents).  Measured here: first frame of a clip
        # (common start) <= 3e-6 from iteration 10 on; later frames inherit the carried state's difference.
        tr = eng.trace(opt["max_iter"])
        for c in range(B):
            n = int(min(iters[c], ref_iters[c]))
            assert tr["active"][c, :n].all()
            dz = np.abs(tr["latent"][c, :n] - g[f"{tag}_latent"][t, c, :n])
            assert dz.max() <= 2e-3, (t, c, dz.max())
            if n > 10:
                late = float(dz[10:].max())
                worst_late = max(worst_late, late)
                assert late <= (2e-4 if t == 0 else 1e-3), (t, c, late)
    eng.enable_trace(False)
    print(f"{tag}: worst per-iteration latent difference from iteration 10 on: {worst_late:.2e}")
    st = eng.state()
    for c in range(B):
        np.testing.assert_allclose(st["height_buf"][c], g[f"{tag}_state_height_buf_{c}"], atol=1e-3)
        np.testing.assert_allclose(st["disp_buf"][c], g[f"{tag}_state_disp_buf_{c}"], atol=1e-3)
        np.testing.assert_allclose(st["latent"][c], g[f"{tag}_state_latent_{c}"], atol=5e-3)


def test_temporal_predictor_vs_reference(golden_dir, engine_factory):
    g = np.load(os.path.join(golden_dir, "ref_temporal.npz"))
    eng = engine_factory(512)
    B = g["latent_buf"].shape[0]
    eng.set_initial_state(np.zeros((B, 24)), np.zeros((B, 3)), np.tile([[1.0, 0, 0, 0]], (B, 1)), np.zeros((B, 6)))
    eng.set_ring_buffers(g["latent_buf"], g["disp_buf"], g["height_buf"])
    for W in (0, 16):
        tb = eng.predict_targets(W)
        ref = g[f"target_buf_w{W}"]
        rows = slice(0, max(W, 1))  # row W is never read (current_index < W)
        err = np.abs(tb[:, rows] - ref[:, rows]).max()
        print(f"window {W}: predictor max abs err {err:.2e} (|ref| max {np.abs(ref).max():.2f})")
        assert err <= 2e-5


@pytest.mark.parametrize("variable", [False, True], ids=["shared-trackers", "variable-mask"])
def test_run_frames_pipelined_equals_frame_by_frame(engine_factory, pose_model, model_npz, variable):
    """dp_engine_run_frames_host (double-buffered staging and copies) must give bit-identical results to per-frame run()."""
    offsets = model_npz["offsets"]
    cfg = synthetic.config_3_trackers() if variable else synthetic.config_6_trackers()
    B, T = 200, 7
    wl = synthetic.make_workload(pose_model, offsets, cfg, B, T, variable_mask=variable)
    kw = dict(lambda_rot=1, lambda_temporal=cfg.lambda_temporal, temporal_future_window=cfg.temporal_future_window, max_iter=12,
              joint_adjustment_indices=cfg.joint_adjustment, joint_adjustment_weight=cfg.joint_adjustment_weight)
    outs = []
    for mode in ("frames", "single"):
        eng = engine_factory(256)
        eng.set_initial_state(wl["latent0"], np.zeros((B, 3)), np.tile([[1.0, 0, 0, 0]], (B, 1)), np.zeros((B, 6)))
        if mode == "frames":
            if variable:
                outs.append(eng.run_frames(wl["tgt_pos"], wl["tgt_rot"], wl["joints_tb"], wl["weights_tb"], n_ee=wl["n_ee"], **kw))
            else:
                outs.append(eng.run_frames(wl["tgt_pos"], wl["tgt_rot"], wl["joints"], wl["weights"], **kw))
        else:
            ps, gs = [], []
            for t in range(T):
                if variable:
                    p_, g_ = eng.run(wl["tgt_pos"][t], wl["tgt_rot"][t], wl["joints_tb"][t], wl["weights_tb"][t], n_ee=wl["n_ee"][t], **kw)
                else:
                    p_, g_ = eng.run(wl["tgt_pos"][t], wl["tgt_rot"][t], wl["joints"], wl["weights"], **kw)
                ps.append(p_); gs.append(g_)
            outs.append((np.stack(ps), np.stack(gs)))
        eng.close()
    assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1])
    assert np.isfinite(outs[0][0]).all()


def test_early_predictor_call_survives_window_changes_and_teardown(engine_factory, pose_model, model_npz, monkeypatch):
    """The early predictor call is tied to the window it was issued for: a caller that changes temporal_future_window between the
    early call and its use (16 -> 8 -> 4 -> 16, the reference's fresh-zero-buffer rule, drag_pose.py:237-244) gets bitwise the frames
    of the engine without early calls, and an engine can be closed while such a call is still in flight."""
    offsets = model_npz["offsets"]
    cfg = synthetic.config_6_trackers()
    B, T = 2, 65
    wl = synthetic.make_workload(pose_model, offsets, cfg, B, T)
    windows = [16] * 14 + [8] * 13 + [4] * 9 + [16] * 29  # changes right after an early call was issued (index W - 3) and mid-window
    kw = dict(lambda_rot=1, lambda_temporal=0.02, max_iter=6, joint_adjustment_indices=cfg.joint_adjustment,
              joint_adjustment_weight=cfg.joint_adjustment_weight)
    outs = []
    for prefetch in ("1", "0"):
        monkeypatch.setenv("DP_PRED_PREFETCH", prefetch)
        eng = engine_factory(4)
        eng.set_initial_state(wl["latent0"], np.zeros((B, 3)), np.tile([[1.0, 0, 0, 0]], (B, 1)), np.zeros((B, 6)))
        ps = []
        for t in range(T):
            p_, g_ = eng.run(wl["tgt_pos"][t], wl["tgt_rot"][t], wl["joints"], wl["weights"], temporal_future_window=windows[t], **kw)
            ps.append(np.concatenate([p_.ravel(), g_.ravel()]))
        outs.append(np.stack(ps))
        eng.close()  # frame 64 has index 13 of a 16-frame window: an early call was issued on it
    assert np.isfinite(outs[0]).all() and np.array_equal(outs[0], outs[1])


@pytest.mark.parametrize("mode", ["frames", "single"])
def test_predictor_issued_three_frames_early_gives_bitwise_the_same_frames(engine_factory, pose_model, model_npz, monkeypatch, mode):
    """Small-batch streaming mode (window 16): the predictor call of a window's first frame is issued three frames early on its own
    stream into a second target buffer (dp_engine.cu:run_one; its inputs end three frames in the past).  40 frames -- two such early
    calls, the second one a CUDA-graph replay -- must equal the engine that calls the predictor at the frame itself, bit for bit,
    including the target rows a caller reads back, through run() and through the pipelined multi-frame call, with a
    set_ring_buffers in the middle of a window (which voids the early call)."""
    offsets = model_npz["offsets"]
    cfg = synthetic.config_3_trackers()
    assert cfg.temporal_future_window == 16
    B, T = 3, 40
    wl = synthetic.make_workload(pose_model, offsets, cfg, B, T, variable_mask=True)
    kw = dict(lambda_rot=1, lambda_temporal=cfg.lambda_temporal, temporal_future_window=16, max_iter=8,
              joint_adjustment_indices=cfg.joint_adjustment, joint_adjustment_weight=cfg.joint_adjustment_weight)
    outs = []
    for prefetch in ("1", "0"):
        monkeypatch.setenv("DP_PRED_PREFETCH", prefetch)  # read when the engine is created
        eng = engine_factory(8)
        eng.set_initial_state(wl["latent0"], np.zeros((B, 3)), np.tile([[1.0, 0, 0, 0]], (B, 1)), np.zeros((B, 6)))
        ps, gs, tb = [], [], []
        if mode == "frames":
            p_, g_ = eng.run_frames(wl["tgt_pos"], wl["tgt_rot"], wl["joints_tb"], wl["weights_tb"], n_ee=wl["n_ee"], **kw)
            ps, gs = list(p_), list(g_)
            tb.append(eng.state(16)["target_buf"].copy())
        else:
            for t in range(T):
                if t == 30:  # between the early call (frame 29 = index 13) and its use (frame 32): the early targets are void
                    st = eng.state(16)
                    order = (np.arange(60) + 7) % 60  # any other chronological content
                    eng.set_ring_buffers(st["latent_buf"][:, order], st["disp_buf"][:, order], st["height_buf"][:, order])
                p_, g_ = eng.run(wl["tgt_pos"][t], wl["tgt_rot"][t], wl["joints_tb"][t], wl["weights_tb"][t], n_ee=wl["n_ee"][t], **kw)
                ps.append(p_); gs.append(g_)
                if t in (15, 16, 31, 32, 39):
                    tb.append(eng.state(16)["target_buf"].copy())
        outs.append((np.stack(ps), np.stack(gs), np.stack(tb)))
        eng.close()
    for a, b in zip(outs[0], outs[1]):
        assert np.isfinite(a).all() and np.array_equal(a, b)


@pytest.mark.parametrize("path", [1, 3], ids=["fp32", "tcgen05-fp16x2"])
def test_clip_order_is_exact(engine_factory, pose_model, model_npz, path):
    """Clip indexing: shuffling the clips of a batch shuffles the results and nothing else, bit for bit (a clip's arithmetic does
    not depend on which warp half, tile column, CTA or predictor part it lands in).  2 frames, variable tracker mask, 2100 clips
    (more than the 2048 that split the predictor into two parts)."""
    cfg = synthetic.config_3_trackers()
    B, T = 2100, 2
    wl = synthetic.make_workload(pose_model, model_npz["offsets"], cfg, B, T, variable_mask=True)
    perm = np.random.default_rng(1).permutation(B)
    kw = dict(lambda_rot=1, lambda_temporal=cfg.lambda_temporal, temporal_future_window=cfg.temporal_future_window, max_iter=15,
              joint_adjustment_indices=cfg.joint_adjustment, joint_adjustment_weight=cfg.joint_adjustment_weight, decoder_path=path)
    outs = []
    for order in (np.arange(B), perm):
        eng = engine_factory(B)
        eng.set_initial_state(wl["latent0"][order], np.zeros((B, 3)), np.tile([[1.0, 0, 0, 0]], (B, 1)), np.zeros((B, 6)))
        for t in range(T):
            res = eng.run(wl["tgt_pos"][t][order], wl["tgt_rot"][t][order], wl["joints_tb"][t][order], wl["weights_tb"][t][order],
                          n_ee=wl["n_ee"][t][order], **kw)
        iters, losses = eng.frame_stats()
        outs.append((res[0], res[1], iters, losses))
        eng.close()
    for a, b in zip(outs[0], outs[1]):
        assert np.array_equal(a[perm], b)


def test_device_encoder_matches_folded_encoder(engine_factory, pose_model):
    """SURVEY 8(f) rank 3: clip start-up on the device vs the host restatement of the folded encoder (model.PoseModel.encode_np)."""
    rng = np.random.default_rng(9)
    n = 300
    dqs = rng.standard_normal((n, 176)).astype(np.float32)
    eps = rng.standard_normal((n, 24)).astype(np.float32)
    eng = engine_factory(512)
    mu, logvar = pose_model.encode_np(dqs)
    got_mu = eng.encode(dqs)
    got = eng.encode(dqs, eps)
    want = mu + eps * np.exp(np.float32(0.5) * logvar)
    scale = max(1.0, float(np.abs(want).max()))
    print(f"device encoder: mu diff {np.abs(got_mu - mu).max():.2e}, latent diff {np.abs(got - want).max():.2e} (|latent| max {scale:.2f})")
    assert np.abs(got_mu - mu).max() <= 2e-5 * scale and np.abs(got - want).max() <= 2e-5 * scale
    eng.set_initial_pose(dqs, np.zeros((n, 3)), np.tile([[1.0, 0, 0, 0]], (n, 1)), np.zeros((n, 6)), eps)
    st = eng.state()
    assert np.array_equal(st["latent"], got) and np.array_equal(st["latent_buf"][:, 17], got)


@pytest.mark.parametrize("n_clips", [5000, 1])
def test_tcgen05_paths_agree_with_cuda_core_path_multi_wave(engine_factory, pose_model, model_npz, n_clips):
    """More clips than one wave of 32-clip tiles (5000 > 148 x 32) and the single-clip corner, every clip checked: teacher-forced
    gradients and joint positions of the tensor-core frame kernel against the fp32 CUDA-core kernel (deterministic), then a
    short optimisation run (robust statistic: an early Adam step is lr * sign(g), so a gradient component inside the fp32 noise
    can flip a +-lr kick between implementations on a few clips out of thousands)."""
    rng = np.random.default_rng(3)
    cfg = synthetic.config_6_trackers()
    wl = synthetic.make_workload(pose_model, model_npz["offsets"], cfg, n_clips, 2)
    lat = wl["latent0"] + 0.2 * rng.standard_normal((n_clips, 24)).astype(np.float32)
    grot = rng.standard_normal((n_clips, 4)).astype(np.float32)
    grot /= np.linalg.norm(grot, axis=1, keepdims=True)
    tl = rng.standard_normal((n_clips, 24)).astype(np.float32) * 0.3
    kw = dict(lambda_rot=1, lambda_temporal=cfg.lambda_temporal, temporal_future_window=cfg.temporal_future_window, max_iter=12,
              stop_eps_pos=-1.0, stop_eps_rot=-1.0, min_loss_incr=-float("inf"), learning_rate=1e-2,
              joint_adjustment_indices=cfg.joint_adjustment, joint_adjustment_weight=cfg.joint_adjustment_weight)
    grads, out = {}, {}
    for path in (1, 3):
        eng = engine_factory(n_clips)
        grads[path] = eng.eval_gradient(lat, grot, tl, wl["tgt_pos"][0], wl["tgt_rot"][0], wl["joints"], wl["weights"], lambda_rot=1.0,
                                        lambda_temporal=0.02, decoder_path=path)
        eng.set_initial_state(wl["latent0"], np.zeros((n_clips, 3)), np.tile([[1.0, 0, 0, 0]], (n_clips, 1)), np.zeros((n_clips, 6)))
        for t in range(2):
            out[path] = eng.run(wl["tgt_pos"][t], wl["tgt_rot"][t], wl["joints"], wl["weights"], decoder_path=path, **kw)
        assert eng.last_decoder_path() == path
        eng.close()
    for path in (3,):
        rel = np.linalg.norm(grads[path]["grad"] - grads[1]["grad"], axis=1) / np.linalg.norm(grads[1]["grad"], axis=1)
        dpos = np.abs(grads[path]["pos"] - grads[1]["pos"]).max()
        dq = np.abs((out[path][0] - out[1][0]) * pose_model.std_q).max(axis=1)  # quaternion components per clip
        dg = np.abs(out[path][1] - out[1][1]).max()
        print(f"{n_clips} clips, path {path} vs fp32 path: gradient rel diff max {rel.max():.2e}, joint positions {dpos:.2e} m; after 2 x 12 "
              f"iterations quaternion diff median {np.median(dq):.2e}, 99th percentile {np.percentile(dq, 99):.2e}, max {dq.max():.2e}, root {dg:.2e}")
        assert rel.max() <= GRAD_REL and dpos <= 1e-5  # bar: 1e-4 relative, 1 mm
        assert np.isfinite(out[path][0]).all() and np.median(dq) < 1e-5 and np.percentile(dq, 99) < 1e-3 and dq.max() < 5e-2 and dg < 1e-4


@pytest.mark.parametrize("n_clips", [1, 37, 300, 2101, 8200])
def test_temporal_predictor_tensor_core_vs_cuda_core(golden_dir, engine_factory, n_clips):
    """Every decoder length (T = 1 + W/4 up to 30 tokens), ragged last tiles, a batch large enough (>= 2048 clips) to run the
    predictor as two parts on two streams, and one (8200 clips: 449 encoder row tiles per part, the last one ragged) large enough
    that the encoder feed-forward runs without the hidden split: tcgen05 kernels vs the fp32 CUDA-core kernels."""
    g = np.load(os.path.join(golden_dir, "ref_temporal.npz"))
    rng = np.random.default_rng(5)
    reps = -(-n_clips // g["latent_buf"].shape[0])
    lat = np.tile(g["latent_buf"], (reps, 1, 1))[:n_clips] + rng.normal(0, 0.05, (n_clips, 60, 24)).astype(np.float32)
    disp = np.tile(g["disp_buf"], (reps, 1, 1))[:n_clips]
    hgt = np.tile(g["height_buf"], (reps, 1, 1))[:n_clips]
    eng = engine_factory(max(512, n_clips))
    eng.set_initial_state(np.zeros((n_clips, 24)), np.zeros((n_clips, 3)), np.tile([[1.0, 0, 0, 0]], (n_clips, 1)), np.zeros((n_clips, 6)))
    eng.set_ring_buffers(lat, disp, hgt)
    for W in (0, 4, 28, 60, 116):
        eng.set_predictor_path(0)
        tc = eng.predict_targets(W).copy()
        eng.set_predictor_path(1)
        ref = eng.predict_targets(W).copy()
        eng.set_predictor_path(0)
        rows = slice(0, max(W, 1))
        err = np.abs(tc[:, rows] - ref[:, rows]).max()
        print(f"{n_clips} clips, window {W}: tensor-core vs CUDA-core predictor max abs diff {err:.2e}")
        assert np.isfinite(tc[:, rows]).all() and err <= 2e-5


@pytest.mark.parametrize("n_clips", [1, 2, 37, 2101])
def test_single_token_decoder_pass_four_clips_per_warp_is_bitwise_the_one_clip_kernels(golden_dir, engine_factory, n_clips, monkeypatch):
    """The single-token decoder pass runs four clips per warp (every weight of its matrix-vector chains loaded once per four clips,
    dp_temporal.cuh: tp_self_attn_rows / tp_cross_attn_rows); each clip's arithmetic keeps the order of the one-clip kernels, which
    stay as the cross-check (DP_DEC_ROWS=0, read on every call): bitwise equal targets, ragged last warps (n % 4 = 1, 2) and the
    two-part split included, at window 0 (the pass is the whole decoder) and window 16 (it is the first of five passes)."""
    g = np.load(os.path.join(golden_dir, "ref_temporal.npz"))
    rng = np.random.default_rng(17)
    reps = -(-n_clips // g["latent_buf"].shape[0])
    tile = lambda a: np.tile(a, (reps, 1, 1))[:n_clips]
    eng = engine_factory(max(512, n_clips))
    eng.set_initial_state(np.zeros((n_clips, 24)), np.zeros((n_clips, 3)), np.tile([[1.0, 0, 0, 0]], (n_clips, 1)), np.zeros((n_clips, 6)))
    eng.set_ring_buffers(tile(g["latent_buf"]) + rng.normal(0, 0.05, (n_clips, 60, 24)).astype(np.float32), tile(g["disp_buf"]), tile(g["height_buf"]))
    for W in (0, 16):
        rows = slice(0, max(W, 1))
        monkeypatch.setenv("DP_DEC_ROWS", "1")
        a = eng.predict_targets(W)[:, rows].copy()
        monkeypatch.setenv("DP_DEC_ROWS", "0")
        b = eng.predict_targets(W)[:, rows].copy()
        monkeypatch.delenv("DP_DEC_ROWS")
        assert np.isfinite(a).all() and np.abs(a).max() > 1e-3 and np.array_equal(a, b)


@pytest.mark.parametrize("n_clips", [1, 2, 37, 2101])
def test_ring_copy_embedding_is_bitwise_the_gathering_embedding(engine_factory, pose_model, model_npz, n_clips, monkeypatch):
    """Look-ahead calls (window 0: four virtual clips per clip, one predictor call per four frames) embed their tokens from a coalesced
    copy of each clip's whole ring (tp_embed_ring_kernel) instead of gathering 33 inputs per token (tp_embed_kernel, DP_EMBED_RING=0,
    read on every call): same operations in the same order, so ten frames -- three look-ahead calls, the ring head moving, CTAs that
    straddle clip and part boundaries -- come out bitwise equal."""
    cfg = synthetic.config_6_trackers()
    T = 10
    wl = synthetic.make_workload(pose_model, model_npz["offsets"], cfg, n_clips, T)
    kw = dict(lambda_rot=1, lambda_temporal=cfg.lambda_temporal, temporal_future_window=0, max_iter=4,
              joint_adjustment_indices=cfg.joint_adjustment, joint_adjustment_weight=cfg.joint_adjustment_weight)
    outs = []
    for ring in ("1", "0"):
        monkeypatch.setenv("DP_EMBED_RING", ring)
        eng = engine_factory(max(512, n_clips))
        eng.set_initial_state(wl["latent0"], np.zeros((n_clips, 3)), np.tile([[1.0, 0, 0, 0]], (n_clips, 1)), np.zeros((n_clips, 6)))
        ps = []
        for t in range(T):
            p_, g_ = eng.run(wl["tgt_pos"][t], wl["tgt_rot"][t], wl["joints"], wl["weights"], **kw)
            ps.append(np.concatenate([p_.ravel(), g_.ravel()]))
        st = eng.state()
        outs.append((np.stack(ps), st["latent_buf"].copy()))
        eng.close()
    monkeypatch.delenv("DP_EMBED_RING")
    assert np.isfinite(outs[0][0]).all() and np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1])
    assert np.abs(np.diff(outs[0][0], axis=0)).max() > 1e-4  # the frames differ from one another: the targets are in play


@pytest.mark.parametrize("n_clips", [1, 37])
def test_predictor_graph_replay_is_bitwise_the_kernel_by_kernel_chain(golden_dir, engine_factory, n_clips):
    """A small predictor call is captured into a CUDA graph on its second use and replayed afterwards (dp_temporal.cu): the first
    (kernel by kernel), second (capture + launch) and third (replay) call agree bit for bit, and a replay on NEW ring contents still
    matches the fp32 CUDA-core chain, which is never captured with the same key."""
    g = np.load(os.path.join(golden_dir, "ref_temporal.npz"))
    rng = np.random.default_rng(11)
    reps = -(-n_clips // g["latent_buf"].shape[0])
    tile = lambda a: np.tile(a, (reps, 1, 1))[:n_clips]
    eng = engine_factory(64)
    eng.set_initial_state(np.zeros((n_clips, 24)), np.zeros((n_clips, 3)), np.tile([[1.0, 0, 0, 0]], (n_clips, 1)), np.zeros((n_clips, 6)))
    for W in (0, 16):
        eng.set_ring_buffers(tile(g["latent_buf"]), tile(g["disp_buf"]), tile(g["height_buf"]))
        rows = slice(0, max(W, 1))
        a = eng.predict_targets(W)[:, rows].copy()
        n0 = eng.launch_count()
        b = eng.predict_targets(W)[:, rows].copy()
        n1 = eng.launch_count()
        c = eng.predict_targets(W)[:, rows].copy()
        n2 = eng.launch_count()
        assert np.isfinite(a).all() and np.array_equal(a, b) and np.array_equal(a, c)
        assert n1 - n0 == n2 - n1 > 0  # the replay reports the kernels it launches
        lat = tile(g["latent_buf"]) + rng.normal(0, 0.05, (n_clips, 60, 24)).astype(np.float32)
        eng.set_ring_buffers(lat, tile(g["disp_buf"]), tile(g["height_buf"]))
        d = eng.predict_targets(W)[:, rows].copy()  # replay on new inputs
        eng.set_predictor_path(1)
        ref = eng.predict_targets(W)[:, rows].copy()
        eng.set_predictor_path(0)
        assert np.abs(d - a).max() > 1e-4 and np.abs(d - ref).max() <= 2e-5


@pytest.mark.parametrize("path", [1, 3], ids=["fp32", "tcgen05-fp16x2"])
def test_frames_3_trackers_variable_mask_vs_reference(golden_dir, engine_factory, port_weights, path):
    g = np.load(os.path.join(golden_dir, "ref_frames_3trk.npz"))
    cfg = synthetic.config_3_trackers()
    eng = engine_factory(512)
    T, B = g["n_ee"].shape
    eng.set_initial_state(g["latent0"], np.zeros((B, 3)), np.tile([[1.0, 0, 0, 0]], (B, 1)), np.zeros((B, 6)))
    worst = 0.0
    for t in range(T):
        pose, gpos = eng.run(g["tgt_pos"][t], g["tgt_rot"][t], g["joints_tb"][t], g["weights_tb"][t], n_ee=g["n_ee"][t],
                             lambda_rot=1, lambda_temporal=cfg.lambda_temporal, temporal_future_window=cfg.temporal_future_window,
                             joint_adjustment_indices=cfg.joint_adjustment, joint_adjustment_weight=cfg.joint_adjustment_weight,
                             decoder_path=path, **EARLY)
        iters, _ = eng.frame_stats()
        dpos = np.abs(pose_positions(port_weights, pose) - pose_positions(port_weights, g["pose"][t])).max()
        dg = np.abs(gpos - g["gpos"][t]).max()
        worst = max(worst, dpos, dg)
        assert dpos <= POS_TOL and dg <= POS_TOL, (t, dpos, dg, iters, g["iters"][t])
    print(f"3-tracker variable mask, {T} frames: worst position diff {worst*1e3:.4f} mm")
    tb = eng.state(cfg.temporal_future_window)["target_buf"]
    np.testing.assert_allclose(tb[:, :16], g["target_buf"][:, :16], atol=5e-4)


@pytest.mark.parametrize("path", [1, 3], ids=["fp32", "tcgen05-fp16x2"])
def test_batch_256_clips_vs_oracle(engine_factory, pose_model, model_npz, port_weights, temporal_model, path):
    """BASELINE config 2: 256 synthetic clips, 6 trackers, against the CPU oracle (batched port)."""
    B, T = 256, 2
    cfg = synthetic.config_6_trackers()
    wl = synthetic.make_workload(pose_model, model_npz["offsets"], cfg, B, T)
    eng = engine_factory(512)
    eng.set_initial_state(wl["latent0"], np.zeros((B, 3)), np.tile([[1.0, 0, 0, 0]], (B, 1)), np.zeros((B, 6)))
    ora = port.PortDragPose(port_weights, temporal_model.sd)
    ora.set_initial_state(wl["latent0"], np.zeros((B, 3)), np.tile([[1.0, 0, 0, 0]], (B, 1)), np.zeros((B, 6)))
    opt = dict(FIXED, max_iter=40, decoder_path=path)
    oopt = dict(FIXED, max_iter=40)
    for t in range(T):
        pose, gpos = eng.run(wl["tgt_pos"][t], wl["tgt_rot"][t], wl["joints"], wl["weights"], lambda_rot=1,
                             lambda_temporal=cfg.lambda_temporal, temporal_future_window=0,
                             joint_adjustment_indices=cfg.joint_adjustment, joint_adjustment_weight=cfg.joint_adjustment_weight, **opt)
        op, og = ora.run(wl["tgt_pos"][t], wl["tgt_rot"][t], wl["joints"], wl["weights"], lambda_rot=1.0,
                         lambda_temporal=cfg.lambda_temporal, temporal_future_window=0, joint_adjustment=cfg.joint_adjustment,
                         joint_adjustment_weight=cfg.joint_adjustment_weight, **oopt)
        dpos = np.abs(pose_positions(port_weights, pose) - pose_positions(port_weights, op.numpy())).max()
        dg = np.abs(gpos - og.numpy()).max()
        print(f"256 clips frame {t}: max joint diff {dpos*1e3:.4f} mm, root diff {dg*1e3:.4f} mm")
        assert dpos <= POS_TOL and dg <= POS_TOL
    # frame/clip indexing is exact: clip c of the batch equals clip c run alone
    solo = engine_factory(512)
    for c in (0, 17, 255):
        solo.set_initial_state(wl["latent0"][c : c + 1], np.zeros((1, 3)), [[1.0, 0, 0, 0]], np.zeros((1, 6)))
        for t in range(T):
            p1, g1 = solo.run(wl["tgt_pos"][t, c : c + 1], wl["tgt_rot"][t, c : c + 1], wl["joints"], wl["weights"], lambda_rot=1,
                              lambda_temporal=cfg.lambda_temporal, temporal_future_window=0,
                              joint_adjustment_indices=cfg.joint_adjustment, joint_adjustment_weight=cfg.joint_adjustment_weight, **opt)
        np.testing.assert_allclose(p1[0], pose[c], atol=2e-3)
        np.testing.assert_allclose(g1[0], gpos[c], atol=1e-5)


def test_clocked_instantiation_is_bitwise_identical_and_timeline_is_ordered(engine_factory, pose_model, model_npz):
    """The phase clock / timeline of the tcgen05 frame kernel lives in a second template instantiation (profiling level 2): it must
    produce bit-identical frames, its eight phase counters must be filled, and the stamps of both clip groups of CTA 0 must be
    ordered in time (loop top < forward < kinematics < barrier < two backward layers < last layer + Adam, iteration after iteration)."""
    cfg = synthetic.config_6_trackers()
    B, T = 600, 2
    wl = synthetic.make_workload(pose_model, model_npz["offsets"], cfg, B, T)
    kw = dict(lambda_rot=1, lambda_temporal=cfg.lambda_temporal, temporal_future_window=0, max_iter=60, stop_eps_pos=-1.0, stop_eps_rot=-1.0,
              min_loss_incr=-float("inf"), joint_adjustment_indices=cfg.joint_adjustment, joint_adjustment_weight=cfg.joint_adjustment_weight,
              decoder_path=3)
    outs = []
    for level in (0, 2):
        eng = engine_factory(B)
        eng.set_initial_state(wl["latent0"], np.zeros((B, 3)), np.tile([[1.0, 0, 0, 0]], (B, 1)), np.zeros((B, 6)))
        eng.set_profiling(level)
        for t in range(T):
            res = eng.run(wl["tgt_pos"][t], wl["tgt_rot"][t], wl["joints"], wl["weights"], **kw)
        outs.append(res)
        if level == 2:
            cyc = eng.phase_cycles()
            assert all(c > 0 for c in cyc[:5]), cyc
            tl = eng.timeline()  # [group][iteration 40..43][6 stamps]
            flat = tl.reshape(2, -1)
            assert (np.diff(flat, axis=1) > 0).all(), tl
            period = (tl[:, 1:, 0] - tl[:, :-1, 0]).mean()
            print(f"clocked kernel: {period:.0f} cycles per iteration, phase counters {cyc[:5]}")
        eng.close()
    assert np.array_equal(outs[0][0], outs[1][0]) and np.array_equal(outs[0][1], outs[1][1])


def test_fixed_iterations_with_a_non_finite_target_stop_like_the_reference_loop(engine_factory, pose_model, model_npz):
    """A fixed-iteration run (negative thresholds, min_loss_incr = -inf) never reads the tracker losses of an iteration except the last
    ones, and the tcgen05 kernel skips their warp sums -- but `while ... and prev_loss - loss > min_loss_incr` (drag_pose.py:296-300)
    still ends on a NaN loss.  A clip with a NaN target must therefore stop after its first iteration on both frame kernels, the other
    clips must run all iterations, and the reported final losses must be the real ones (the two kernels agree)."""
    cfg = synthetic.config_6_trackers()
    B, iters = 600, 30
    wl = synthetic.make_workload(pose_model, model_npz["offsets"], cfg, B, 1)
    tp = wl["tgt_pos"][0].copy()
    bad = [5, 301, 599]
    tp[bad[0], 2, 1] = np.nan
    tp[bad[1], 0, 0] = np.inf
    tp[bad[2], 5, 2] = np.nan
    kw = dict(lambda_rot=1, lambda_temporal=cfg.lambda_temporal, temporal_future_window=0, max_iter=iters, stop_eps_pos=-1.0, stop_eps_rot=-1.0,
              min_loss_incr=-float("inf"), joint_adjustment_indices=cfg.joint_adjustment, joint_adjustment_weight=cfg.joint_adjustment_weight)
    stats = {}
    for path in (1, 3):
        eng = engine_factory(B)
        eng.set_initial_state(wl["latent0"], np.zeros((B, 3)), np.tile([[1.0, 0, 0, 0]], (B, 1)), np.zeros((B, 6)))
        eng.run(tp, wl["tgt_rot"][0], wl["joints"], wl["weights"], decoder_path=path, **kw)
        stats[path] = eng.frame_stats()
        eng.close()
    good = np.setdiff1d(np.arange(B), bad)
    for path in (1, 3):
        it, losses = stats[path]
        assert (it[bad] == 1).all(), (path, it[bad])
        assert (it[good] == iters).all()
        assert np.isfinite(losses[good]).all() and (losses[good, 0] > 0).all() and (losses[good, 1] > 0).all()
    rel = np.abs(stats[3][1][good] - stats[1][1][good]) / np.maximum(np.abs(stats[1][1][good]), 1e-6)
    print(f"final losses of the {len(good)} finite clips, tcgen05 vs fp32 kernel: max relative difference {rel.max():.2e}")
    assert rel.max() < 5e-3
