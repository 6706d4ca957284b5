"""CPU: the oracle (oracle/dragposer_port.py) is pinned against the golden vectors recorded from the
UNMODIFIED reference (oracle/make_golden.py) and, when /root/reference is mounted, against the live reference."""
import os

import numpy as np
import pytest
import torch

import dragposer_port as port
import reference_harness as rh
from dragposer_b200 import synthetic

FIXED = dict(stop_eps_pos=-1.0, stop_eps_rot=-1.0, max_iter=100, min_loss_incr=-float("inf"), learning_rate=1e-2)
EARLY = dict(stop_eps_pos=0.01 * 0.01, stop_eps_rot=0.01, max_iter=100, min_loss_incr=0.00001, learning_rate=1e-2)


def test_port_gradient_teacher_forced_vs_reference(golden_dir, port_weights):
    g = np.load(os.path.join(golden_dir, "ref_trace_6trk.npz"))
    for tag in ("fixed", "early"):
        F, C = g[f"{tag}_iters"].shape
        for t in range(F):
            for c in range(C):
                n = int(g[f"{tag}_iters"][t, c])
                r = port.loss_and_grad(port_weights, g[f"{tag}_latent"][t, c, :n], np.tile(g[f"{tag}_grot"][t, c], (n, 1)),
                                       np.tile(g["tgt_pos"][t, c], (n, 1, 1)), np.tile(g["tgt_rot"][t, c], (n, 1, 1, 1)),
                                       np.tile(g[f"{tag}_tgt_latent"][t, c], (n, 1)), g["joints"], g["weights"], lambda_rot=1.0,
                                       lambda_temporal=0.02)
                ref = g[f"{tag}_grad"][t, c, :n]
                err = np.linalg.norm(r["grad"] - ref, axis=1)
                # two fp32 evaluations of the same function: 1e-4 relative plus the reference's own fp32 noise floor
                assert (err <= 1e-4 * np.linalg.norm(ref, axis=1) + 5e-7).all()
                np.testing.assert_allclose(r["lp"], g[f"{tag}_loss"][t, c, :n, 0], rtol=1e-4, atol=1e-9)
                np.testing.assert_allclose(r["lr"], g[f"{tag}_loss"][t, c, :n, 1], rtol=1e-4, atol=1e-9)
                np.testing.assert_allclose(r["lt"], g[f"{tag}_loss"][t, c, :n, 2], rtol=1e-4, atol=1e-10)


@pytest.mark.parametrize("tag,opt,n_frames", [("fixed", FIXED, 1), ("early", EARLY, 6)])
def test_port_frames_vs_reference(golden_dir, port_weights, temporal_model, tag, opt, n_frames):
    g = np.load(os.path.join(golden_dir, "ref_trace_6trk.npz"))
    cfg = synthetic.config_6_trackers()
    B = g["latent0"].shape[0]
    d = port.PortDragPose(port_weights, temporal_model.sd)
    d.set_initial_state(g["latent0"], np.zeros((B, 3)), np.tile([[1.0, 0, 0, 0]], (B, 1)), np.zeros((B, 6)))
    for t in range(n_frames):
        pose, gpos = d.run(g["tgt_pos"][t], g["tgt_rot"][t], g["joints"], g["weights"], lambda_rot=1.0,
                           lambda_temporal=cfg.lambda_temporal, temporal_future_window=0, joint_adjustment=cfg.joint_adjustment,
                           joint_adjustment_weight=cfg.joint_adjustment_weight, **opt)
        assert (d.iters.numpy() == g[f"{tag}_iters"][t]).all()  # identical early-stop decisions
        q = lambda p: np.asarray(p) * port_weights.std_q.numpy() + port_weights.mean_q.numpy()
        assert np.abs(q(pose.numpy()) - q(g[f"{tag}_pose"][t])).max() < 1e-5
        assert np.abs(gpos.numpy() - g[f"{tag}_gpos"][t]).max() < 1e-5


def test_port_variable_mask_frames_vs_reference(golden_dir, port_weights, temporal_model):
    g = np.load(os.path.join(golden_dir, "ref_frames_3trk.npz"))
    cfg = synthetic.config_3_trackers()
    T, B = g["n_ee"].shape
    d = port.PortDragPose(port_weights, temporal_model.sd)
    d.set_initial_state(g["latent0"], np.zeros((B, 3)), np.tile([[1.0, 0, 0, 0]], (B, 1)), np.zeros((B, 6)))
    assert set(np.unique(g["n_ee"])) == {2, 3}
    for t in range(20):
        pose, gpos = d.run(g["tgt_pos"][t], g["tgt_rot"][t], g["joints_tb"][t], g["weights_tb"][t], n_ee=g["n_ee"][t], lambda_rot=1.0,
                           lambda_temporal=cfg.lambda_temporal, temporal_future_window=cfg.temporal_future_window,
                           joint_adjustment=cfg.joint_adjustment, joint_adjustment_weight=cfg.joint_adjustment_weight, **EARLY)
        assert np.abs(d.iters.numpy() - g["iters"][t]).max() <= 1
        assert np.abs(gpos.numpy() - g["gpos"][t]).max() < 1e-4


def test_port_predictor_vs_reference(golden_dir, temporal_model):
    g = np.load(os.path.join(golden_dir, "ref_temporal.npz"))
    sd = {k: torch.as_tensor(v) for k, v in temporal_model.sd.items()}
    for W in (0, 16):
        tb = port.predict_targets(sd, torch.zeros(24), torch.ones(24), torch.as_tensor(g["latent_buf"]), torch.as_tensor(g["disp_buf"]),
                                  torch.as_tensor(g["height_buf"]), W)
        assert np.abs(tb.numpy() - g[f"target_buf_w{W}"]).max() < 5e-6
        if W:  # step-function upsampling: rows 0-3 <- pred@4, ..., 12-16 <- pred@16 (drag_pose.py:282-289)
            assert np.array_equal(tb[:, 0], tb[:, 3]) and np.array_equal(tb[:, 12], tb[:, 16]) and not np.array_equal(tb[:, 3], tb[:, 4])


def test_rundrag_local_quaternion_conversion(golden_dir, port_weights):
    """from_root_quat (train.py:409-434) on the recorded session: unit local quaternions, root-children untouched."""
    g = np.load(os.path.join(golden_dir, "ref_rundrag.npz"))
    q = g["result_pose"]
    assert np.allclose(np.linalg.norm(q, axis=-1), 1.0, atol=1e-4)


def test_port_matches_recorded_reference_one_frame(golden_dir, port_weights, temporal_model):
    """The one-frame comparison below (fresh start, early-stop thresholds capped at 25 iterations, seed-2222 predictor) against the
    reference's recorded run of frame 0 (ref_trace_6trk.npz): each clip ran past 25 iterations there, so a capped reference run is
    exactly those first 25 iterations, and the port must follow that latent path and its losses."""
    g = np.load(os.path.join(golden_dir, "ref_trace_6trk.npz"))
    cfg = synthetic.config_6_trackers()
    B, n = g["latent0"].shape[0], 25
    assert (g["early_iters"][0] > n).all()
    d = port.PortDragPose(port_weights, temporal_model.sd)
    d.set_initial_state(g["latent0"], np.zeros((B, 3)), np.tile([[1.0, 0, 0, 0]], (B, 1)), np.zeros((B, 6)))
    d.trace = []
    d.run(g["tgt_pos"][0], g["tgt_rot"][0], g["joints"], g["weights"], lambda_rot=1.0, lambda_temporal=cfg.lambda_temporal,
          temporal_future_window=0, joint_adjustment=cfg.joint_adjustment, joint_adjustment_weight=cfg.joint_adjustment_weight,
          **dict(EARLY, max_iter=n))
    assert (d.iters.numpy() == n).all() and len(d.trace) == n
    latents = np.stack([r["latent"] for r in d.trace], 1)
    assert np.abs(latents - g["early_latent"][0, :, :n]).max() < 2e-5
    np.testing.assert_allclose(np.stack([r["lp"] for r in d.trace], 1), g["early_loss"][0, :, :n, 0], rtol=1e-4, atol=1e-9)
    np.testing.assert_allclose(np.stack([r["lr"] for r in d.trace], 1), g["early_loss"][0, :, :n, 1], rtol=1e-4, atol=1e-9)


@pytest.mark.skipif(not rh.available(), reason="live reference only exists in the build container")
def test_port_matches_live_reference_one_frame(port_weights, pose_model, model_npz):
    from dragposer_b200 import model as dpm

    ref = rh.Reference()
    ref.temporal.load_state_dict(dpm.random_temporal_state(2222))
    cfg = synthetic.config_6_trackers()
    wl = synthetic.make_workload(pose_model, model_npz["offsets"], cfg, 1, 1, first_clip=99)
    drag = ref.new_drag()
    drag.set_initial_pose(torch.zeros(1, 176, 1), torch.zeros(1, 3, 1), torch.tensor([[1.0, 0, 0, 0]]).unsqueeze(-1), torch.zeros(6))
    z = torch.from_numpy(wl["latent0"].copy())
    drag.latent = z.clone().requires_grad_()
    drag.latent_buffer = torch.tile(z, (60, 1))
    opt = dict(EARLY, max_iter=25)
    pose, gpos = drag.run(torch.from_numpy(wl["tgt_pos"][0, 0]), torch.from_numpy(wl["tgt_rot"][0, 0]), torch.from_numpy(wl["joints"]).long(),
                          torch.from_numpy(wl["weights"]), ref.offsets, lambda_rot=1, lambda_temporal=cfg.lambda_temporal,
                          temporal_future_window=0, joint_adjustment_indices=cfg.joint_adjustment,
                          joint_adjustment_weight=cfg.joint_adjustment_weight, **opt)
    d = port.PortDragPose(port_weights, dpm.random_temporal_state(2222))
    d.set_initial_state(wl["latent0"], np.zeros((1, 3)), [[1.0, 0, 0, 0]], np.zeros((1, 6)))
    p2, g2 = d.run(wl["tgt_pos"][0], wl["tgt_rot"][0], wl["joints"], wl["weights"], lambda_rot=1.0, lambda_temporal=cfg.lambda_temporal,
                   temporal_future_window=0, joint_adjustment=cfg.joint_adjustment, joint_adjustment_weight=cfg.joint_adjustment_weight, **opt)
    assert np.abs(p2.numpy()[0] - pose.detach().numpy()).max() < 5e-3  # standardised space (1/std up to 1700x)
    assert np.abs(g2.numpy()[0] - gpos.detach().numpy()).max() < 1e-5
