"""SURVEY 8(f) rank 4: the reference's "Additional Losses" extension point (python/src/drag_pose.py:129-183, commented out as shipped)
and the trained-predictor path (`temporal.pt`, written by train.py:311-319 and read by train_temporal.py:474-482).

The golden vectors of the extension losses come from the reference's own loop with exactly that block re-enabled
(oracle/reference_harness.load_drag_pose_with_extension_losses; recipe: `python -B oracle/make_golden.py extlosses`)."""
import os
import struct

import numpy as np
import pytest
import torch

import dragposer_port as port

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")
ALL = 15


def _wild_args(g):
    """32 single evaluations at wild states (latent 1.5 N(0,I), random previous root rotation / position): the head / hips "forward"
    term is only active when the two face more than ~37 degrees apart, which optimisation trajectories never reach."""
    c = g["wild_clip"]
    return dict(latents=g["wild_latent"], global_rot=g["wild_grot"], tgt_latent=g["wild_tgt_latent"], tgt_pos=g["tgt_pos"][0][c],
                tgt_rot=g["tgt_rot"][0][c], global_pos=g["wild_gpos"])


def _teacher_args(g, t, c):
    n = g["latent"].shape[2]
    return dict(latents=g["latent"][t, c], global_rot=np.tile(g["grot"][t, c], (n, 1)), tgt_latent=np.tile(g["tgt_latent"][t, c], (n, 1)),
                tgt_pos=np.tile(g["tgt_pos"][t, c], (n, 1, 1)), tgt_rot=np.tile(g["tgt_rot"][t, c], (n, 1, 1, 1)),
                global_pos=np.tile(g["frame_gpos"][t, c], (n, 1)))


# ----------------------------------------------------------------------------- CPU
def test_port_extension_losses_match_reference(port_weights):
    g = np.load(os.path.join(G, "ref_extension_losses.npz"))
    F, C = g["latent"].shape[:2]
    worst = 0.0
    for t in range(F):
        for c in range(C):
            a = _teacher_args(g, t, c)
            r = port.loss_and_grad(port_weights, a["latents"], a["global_rot"], a["tgt_pos"], a["tgt_rot"], a["tgt_latent"], g["joints"], g["weights"],
                                   lambda_rot=1.0, lambda_temporal=0.02, extension_losses_mask=ALL, global_pos=a["global_pos"])
            rel = np.linalg.norm(r["grad"] - g["grad"][t, c], axis=1) / np.linalg.norm(g["grad"][t, c], axis=1)
            worst = max(worst, float(rel.max()))
            np.testing.assert_allclose(r["le"], g["extra"][t, c], rtol=1e-5, atol=1e-6)
            np.testing.assert_allclose(r["lp"], g["loss"][t, c, :, 0], rtol=2e-4, atol=1e-8)
    a = _wild_args(g)
    r = port.loss_and_grad(port_weights, a["latents"], a["global_rot"], a["tgt_pos"], a["tgt_rot"], a["tgt_latent"], g["joints"], g["weights"],
                           lambda_rot=1.0, lambda_temporal=0.02, extension_losses_mask=ALL, global_pos=a["global_pos"])
    rel = np.linalg.norm(r["grad"] - g["wild_grad"], axis=1) / np.linalg.norm(g["wild_grad"], axis=1)
    np.testing.assert_allclose(r["le"], g["wild_extra"], rtol=1e-5, atol=2e-6)
    worst = max(worst, float(rel.max()))
    print(f"port with the four extension losses vs the reference with its block re-enabled: worst gradient rel err {worst:.2e}")
    assert worst <= 1e-4


def test_extension_terms_are_all_exercised(port_weights):
    """Each of the four terms contributes on the golden states (otherwise the parity above would not cover it)."""
    g = np.load(os.path.join(G, "ref_extension_losses.npz"))
    a = _wild_args(g)
    vals = {}
    for bit in (1, 2, 4, 8):
        r = port.loss_and_grad(port_weights, a["latents"], a["global_rot"], a["tgt_pos"], a["tgt_rot"], a["tgt_latent"], g["joints"], g["weights"],
                               lambda_rot=1.0, lambda_temporal=0.02, extension_losses_mask=bit, global_pos=a["global_pos"])
        vals[bit] = int((r["le"] > 0).sum())
    print("golden states on which each extension term is active:", vals)
    assert all(v >= 8 for v in vals.values())


def test_temporal_pt_round_trip_in_reference_format(tmp_path, temporal_model):
    """A predictor written in the reference's temporal.pt layout ({"model_state_dict", "means_latent", "stds_latent"}, train.py:311-319)
    with non-trivial latent statistics loads back identically, is flagged as trained, is required by default, and the .dpm export
    records it."""
    from dragposer_b200 import export_model, model

    rng = np.random.default_rng(3)
    tm = model.TemporalModel(temporal_model.sd, rng.normal(0, 0.3, 24).astype(np.float32), rng.uniform(0.5, 1.5, 24).astype(np.float32))
    d = tmp_path / "m"
    d.mkdir()
    with pytest.raises(FileNotFoundError):
        model.load_temporal_model(str(d))  # like train_temporal.load_model: no silent random predictor
    assert not model.load_temporal_model(str(d), allow_random=True).trained
    model.save_temporal_model(tm, str(d / "temporal.pt"))
    ck = torch.load(str(d / "temporal.pt"), map_location="cpu", weights_only=True)
    assert set(ck) == {"model_state_dict", "means_latent", "stds_latent"}
    back = model.load_temporal_model(str(d))
    assert back.trained and set(back.sd) == set(tm.sd)
    for k in tm.sd:
        assert np.array_equal(back.sd[k], tm.sd[k]), k
    assert np.array_equal(back.means_latent, tm.means_latent) and np.array_equal(back.stds_latent, tm.stds_latent)
    # export: the folded pose model lies next to temporal.pt; the header flag says "trained", the statistics travel
    import shutil
    shutil.copy(os.path.join(G, "model_dancedb.npz"), d / "model_dancedb.npz")
    out = export_model.export(str(d / "model_dancedb.npz"), str(d / "model.dpm"))
    raw = open(out, "rb").read()
    version, n, flags = struct.unpack("<III", raw[4:16])
    assert version == 2 and flags & export_model.DPM_FLAG_TRAINED_TEMPORAL
    flat = np.frombuffer(raw[16:], np.float32)
    assert np.array_equal(flat[-48:-24], tm.means_latent) and np.array_equal(flat[-24:], tm.stds_latent)


def test_temporal_pt_has_the_layout_the_reference_loader_reads(tmp_path, temporal_model):
    """A file written by save_temporal_model holds what the reference's train_temporal.load_model (train_temporal.py:474-482) reads:
    the checkpoint keys, the latent statistics, and a state dict with the names and shapes of the reference Temporal module
    (golden/temporal_pt_layout.json, recorded by `python -B oracle/make_golden.py tplayout`), which its strict load_state_dict
    requires."""
    import json

    from dragposer_b200 import model

    with open(os.path.join(G, "temporal_pt_layout.json")) as fh:
        layout = json.load(fh)
    tm = model.TemporalModel(temporal_model.sd, np.full(24, 0.25, np.float32), np.full(24, 2.0, np.float32))
    path = str(tmp_path / "temporal.pt")
    model.save_temporal_model(tm, path)
    ck = torch.load(path, map_location="cpu")
    assert sorted(ck) == sorted(layout["checkpoint_keys"])
    assert {k: list(v.shape) for k, v in ck["model_state_dict"].items()} == layout["model_state_dict"]
    for k, v in ck["model_state_dict"].items():
        assert v.dtype == torch.float32 and np.array_equal(v.numpy(), tm.sd[k]), k
    for name, value in (("means_latent", 0.25), ("stds_latent", 2.0)):
        assert list(ck[name].shape) == layout[name] and ck[name].dtype == torch.float32 and torch.all(ck[name] == value), name


def test_temporal_pt_loads_into_the_reference_module(tmp_path, temporal_model):
    """When the reference tree is present: the file written by save_temporal_model is accepted by the reference's own
    train_temporal.load_model (train_temporal.py:474-482)."""
    import reference_harness as rh

    if not rh.available():
        pytest.skip("reference tree not present")
    from dragposer_b200 import model

    rh.activate()
    import train_temporal
    from temporal_transformer import Temporal

    tm = model.TemporalModel(temporal_model.sd, np.full(24, 0.25, np.float32), np.full(24, 2.0, np.float32))
    path = str(tmp_path / "temporal.pt")
    model.save_temporal_model(tm, path)
    net = Temporal(train_temporal.param, "cpu")
    means, stds = train_temporal.load_model(net, path, "cpu")
    assert torch.allclose(means, torch.full((24,), 0.25)) and torch.allclose(stds, torch.full((24,), 2.0))
    for k, v in net.state_dict().items():
        assert np.array_equal(v.numpy(), tm.sd[k]), k


# ----------------------------------------------------------------------------- GPU
@pytest.mark.gpu
def test_engine_extension_losses_gradient_vs_reference(engine_factory, port_weights, model_npz):
    g = np.load(os.path.join(G, "ref_extension_losses.npz"))
    eng = engine_factory(64)
    F, C = g["latent"].shape[:2]
    worst = 0.0
    for t in range(F):
        for c in range(C):
            a = _teacher_args(g, t, c)
            r = eng.eval_gradient(a["latents"], a["global_rot"], a["tgt_latent"], a["tgt_pos"], a["tgt_rot"], g["joints"], g["weights"], lambda_rot=1.0,
                                  lambda_temporal=0.02, decoder_path=1, extension_losses=ALL, global_pos=a["global_pos"])
            ref = g["grad"][t, c]
            err = np.linalg.norm(r["grad"] - ref, axis=1)
            assert (err <= 1e-4 * np.linalg.norm(ref, axis=1) + 5e-7).all(), (t, c, float((err / np.linalg.norm(ref, axis=1)).max()))
            worst = max(worst, float((err / np.linalg.norm(ref, axis=1)).max()))
    a = _wild_args(g)
    r = eng.eval_gradient(a["latents"], a["global_rot"], a["tgt_latent"], a["tgt_pos"], a["tgt_rot"], g["joints"], g["weights"], lambda_rot=1.0,
                          lambda_temporal=0.02, extension_losses=ALL, global_pos=a["global_pos"])
    err = np.linalg.norm(r["grad"] - g["wild_grad"], axis=1)
    assert (err <= 1e-4 * np.linalg.norm(g["wild_grad"], axis=1) + 5e-7).all(), float((err / np.linalg.norm(g["wild_grad"], axis=1)).max())
    worst = max(worst, float((err / np.linalg.norm(g["wild_grad"], axis=1)).max()))
    print(f"engine with the four extension losses vs the reference's recorded gradients: worst rel err {worst:.2e}")
    # each term on its own against the float64 port (random root positions / floor level)
    pw64 = port.PortWeights(model_npz, dtype=torch.float64)
    a = _wild_args(g)
    for bit in (1, 2, 4, 8):
        r = eng.eval_gradient(a["latents"], a["global_rot"], a["tgt_latent"], a["tgt_pos"], a["tgt_rot"], g["joints"], g["weights"], lambda_rot=1.0,
                              lambda_temporal=0.02, extension_losses=bit, floor_level=0.05, global_pos=a["global_pos"])
        t64 = port.loss_and_grad(pw64, a["latents"], a["global_rot"], a["tgt_pos"], a["tgt_rot"], a["tgt_latent"], g["joints"], g["weights"],
                                 lambda_rot=1.0, lambda_temporal=0.02, dtype=torch.float64, extension_losses_mask=bit, global_pos=a["global_pos"],
                                 floor_level=0.05)
        rel = np.linalg.norm(r["grad"] - t64["grad"], axis=1) / np.linalg.norm(t64["grad"], axis=1)
        assert rel.max() <= 1e-4, (bit, rel.max())
    with pytest.raises(RuntimeError):  # the tensor-core kernel does not carry the extension terms
        eng.eval_gradient(a["latents"], a["global_rot"], a["tgt_latent"], a["tgt_pos"], a["tgt_rot"], g["joints"], g["weights"], decoder_path=3,
                          extension_losses=ALL)


@pytest.mark.gpu
def test_engine_extension_losses_frames_vs_reference(engine_factory, port_weights):
    """Three frames of the loop with the extension losses on (30 fixed iterations), carried state included, <= 1 mm."""
    from dragposer_b200 import synthetic

    g = np.load(os.path.join(G, "ref_extension_losses.npz"))
    cfg = synthetic.config_6_trackers()
    F, C = g["latent"].shape[:2]
    eng = engine_factory(64)
    eng.set_initial_state(g["latent0"], np.tile(g["gpos0"], (C, 1)), np.tile([[1.0, 0, 0, 0]], (C, 1)), np.zeros((C, 6)))
    eng.enable_trace(True)
    pw = port_weights
    for t in range(F):
        pose, gpos = eng.run(g["tgt_pos"][t], g["tgt_rot"][t], g["joints"], g["weights"], lambda_rot=1, lambda_temporal=cfg.lambda_temporal,
                             temporal_future_window=0, joint_adjustment_indices=cfg.joint_adjustment, joint_adjustment_weight=cfg.joint_adjustment_weight,
                             stop_eps_pos=-1.0, stop_eps_rot=-1.0, max_iter=30, min_loss_incr=-float("inf"), learning_rate=1e-2,
                             extension_losses=ALL)
        assert eng.last_decoder_path() == 1
        q = lambda p: (torch.as_tensor(p) * pw.std_q + pw.mean_q).reshape(-1, 22, 4)
        fk = lambda p: port.fk_chain(port.root_to_local(q(p), pw.parents), torch.zeros(C, 3), pw.offsets, pw.parents)[0].numpy()
        dpos = np.abs(fk(pose) - fk(g["pose"][t])).max()
        dg = np.abs(gpos - g["gpos"][t]).max()
        tr = eng.trace(30)
        dz = np.abs(tr["latent"] - g["latent"][t]).max()
        print(f"extension losses, frame {t}: joints {dpos*1e3:.4f} mm, root {dg*1e3:.4f} mm, per-iteration latent diff {dz:.2e}")
        assert dpos <= 1e-3 and dg <= 1e-3
    eng.enable_trace(False)


@pytest.mark.gpu
def test_trained_predictor_file_drives_the_engine(tmp_path, pose_model, model_npz, temporal_model):
    """temporal.pt with non-trivial latent statistics -> load_temporal_model -> engine: the predicted target latents equal the oracle's
    with the same statistics (drag_pose.py:257-262,280), and differ from the ones with means 0 / stds 1."""
    from dragposer_b200 import model
    from dragposer_b200.engine import BatchedDragPose

    g = np.load(os.path.join(G, "ref_temporal.npz"))
    rng = np.random.default_rng(4)
    ml, sl = rng.normal(0, 0.3, 24).astype(np.float32), rng.uniform(0.5, 1.5, 24).astype(np.float32)
    model.save_temporal_model(model.TemporalModel(temporal_model.sd, ml, sl), str(tmp_path / "temporal.pt"))
    tm = model.load_temporal_model(str(tmp_path))
    B = g["latent_buf"].shape[0]
    eng = BatchedDragPose(pose_model, model_npz["offsets"], tm, 64)
    eng.set_initial_state(np.zeros((B, 24)), np.zeros((B, 3)), np.tile([[1.0, 0, 0, 0]], (B, 1)), np.zeros((B, 6)))
    eng.set_ring_buffers(g["latent_buf"], g["disp_buf"], g["height_buf"])
    sd = {k: torch.as_tensor(v) for k, v in tm.sd.items()}
    for W in (0, 16):
        got = eng.predict_targets(W)
        want = port.predict_targets(sd, torch.as_tensor(ml), torch.as_tensor(sl), torch.as_tensor(g["latent_buf"]), torch.as_tensor(g["disp_buf"]),
                                    torch.as_tensor(g["height_buf"]), W).numpy()
        rows = slice(0, max(W, 1))
        err = np.abs(got[:, rows] - want[:, rows]).max()
        print(f"trained-predictor path, window {W}: max abs err vs the oracle {err:.2e}")
        assert err <= 3e-5 and np.abs(got[:, rows] - g[f"target_buf_w{W}"][:, rows]).max() > 1e-2
    eng.close()
