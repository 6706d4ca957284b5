"""ORACLE-ONLY: generates the committed fixtures under tests/golden/ by running the
UNMODIFIED reference (`/root/reference/python/src`) in this container.

    python -B oracle/make_golden.py            # ~3-4 minutes on one core

Deviations forced by the mount (both documented in SURVEY.md section 0): `temporal.pt`
is a missing blob, so the predictor is the seeded random-init instance produced by
`dragposer_b200.model.random_temporal_state(2222)` loaded into the reference's
own `Temporal` module, with means_latent = 0 and stds_latent = 1.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

import reference_harness as rh  # noqa: E402
from dragposer_b200 import model as dpm  # noqa: E402
from dragposer_b200 import synthetic  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def build():
    ref = rh.Reference()
    ref.temporal.load_state_dict(dpm.random_temporal_state(2222))
    ref.temporal.eval()
    return ref


def save_model_fixture(ref):
    sd = ref.generator.state_dict()
    pm = dpm.fold_generator_state(sd, ref.means, ref.stds, ref.parents)
    path = os.path.join(OUT, "model_dancedb.npz")
    dpm.save_folded_npz(pm, path, offsets=ref.offsets_np)
    z = dict(np.load(path))
    pre = "autoencoder.decoder."
    z["dec_f_w"] = sd[pre + "f_latent.weight"].numpy()
    z["dec_f_b"] = sd[pre + "f_latent.bias"].numpy()
    for l in range(3):
        z[f"dec_U{l}"] = sd[f"{pre}layers.{l}.0.weight"].numpy()
        z[f"dec_W{l}"] = (sd[f"{pre}layers.{l}.1.weight"] * sd[f"{pre}layers.{l}.1.mask"])[..., 0].numpy()
        z[f"dec_b{l}"] = sd[f"{pre}layers.{l}.1.bias"].numpy()
    np.savez_compressed(path, **z)
    return pm


class Recorder:
    """Wraps DragPose.loss to record per-iteration latents, losses and gradients without
    touching the reference source.  `latent.grad` still holds iteration k-1's gradient when
    the loss of iteration k is evaluated (zero_grad runs after it), and the last
    iteration's gradient after `run` returns."""

    def __init__(self, drag):
        self.drag = drag
        self.rows = []
        orig_loss = drag.loss

        def loss(*a, **k):
            self._close()
            out = orig_loss(*a, **k)
            self.rows.append(dict(latent=drag.latent.detach().clone().numpy()[0], lp=float(out[0]),
                                  lr=float(out[1]), lt=float(out[2]), le=float(out[3])))
            return out

        drag.loss = loss

    def _close(self):
        if self.rows and "grad" not in self.rows[-1]:
            self.rows[-1]["grad"] = self.drag.latent.grad.clone().numpy()[0]

    def take(self):
        self._close()
        rows, self.rows = self.rows, []
        return rows


def init_drag(ref, latent0, extension_losses=False, gpos0=(0.0, 0.0, 0.0)):
    drag = ref.new_drag(extension_losses=extension_losses)
    drag.set_initial_pose(torch.zeros(1, 176, 1), torch.tensor(gpos0, dtype=torch.float32).reshape(1, 3, 1),
                          torch.tensor([[1.0, 0, 0, 0]]).unsqueeze(-1), torch.zeros(6))
    z = torch.from_numpy(latent0.copy()).reshape(1, 24)
    drag.latent = z.clone().requires_grad_()
    drag.latent_buffer = torch.tile(z, (60, 1))
    return drag


def run_frames(ref, wl, clip, n_frames, record_iters=False, n_ee=None, extension_losses=False, gpos0=(0.0, 0.0, 0.0), **opt):
    drag = init_drag(ref, wl["latent0"][clip], extension_losses, gpos0)
    rec = Recorder(drag) if record_iters else None
    poses, gposs, iters, traces, grots, tgt_lats = [], [], [], [], [], []
    offsets = ref.offsets
    for t in range(n_frames):
        E = int(wl["n_ee"][t, clip]) if "n_ee" in wl else len(wl["joints"])
        joints = wl["joints_tb"][t, clip, :E] if "joints_tb" in wl else wl["joints"]
        weights = wl["weights_tb"][t, clip, :E] if "weights_tb" in wl else wl["weights"]
        grots.append(drag.current_global_rot.detach().numpy()[0].copy())
        index = drag.current_index
        pose, gpos = drag.run(
            torch.from_numpy(wl["tgt_pos"][t, clip, :E].copy()), torch.from_numpy(wl["tgt_rot"][t, clip, :E].copy()),
            torch.from_numpy(np.asarray(joints)).long(), torch.from_numpy(np.asarray(weights).copy()), offsets,
            lambda_rot=1, lambda_temporal=wl["lambda_temporal"], temporal_future_window=wl["window"],
            joint_adjustment_indices=wl["joint_adjustment"], joint_adjustment_weight=wl["joint_adjustment_weight"],
            **opt)
        poses.append(pose.detach().numpy().copy())
        gposs.append(gpos.detach().numpy().copy())
        tgt_lats.append(drag.target_latent_buffer[index].detach().numpy().copy())
        if rec:
            rows = rec.take()
            iters.append(len(rows))
            traces.append(rows)
    state = dict(latent=drag.latent.detach().numpy()[0].copy(), grot=drag.current_global_rot.detach().numpy()[0].copy(),
                 latent_buf=drag.latent_buffer.detach().numpy().copy(), disp_buf=drag.displacement_buffer.detach().numpy().copy(),
                 height_buf=drag.heights_buffer.detach().numpy().copy(),
                 target_buf=drag.target_latent_buffer.detach().numpy().copy(),
                 frame_grot=np.stack(grots), frame_tgt_latent=np.stack(tgt_lats))
    return np.stack(poses), np.stack(gposs), iters, traces, state


def pack_traces(traces, max_iter):
    """list[frame] of list[iter] of rows -> padded arrays (F,I,...)."""
    F_ = len(traces)
    lat = np.zeros((F_, max_iter, 24), np.float32)
    grad = np.zeros((F_, max_iter, 24), np.float32)
    loss = np.zeros((F_, max_iter, 3), np.float64)
    n = np.zeros(F_, np.int32)
    for f, rows in enumerate(traces):
        n[f] = len(rows)
        for i, r in enumerate(rows):
            lat[f, i], grad[f, i] = r["latent"], r["grad"]
            loss[f, i] = (r["lp"], r["lr"], r["lt"])
    return lat, grad, loss, n


def golden_iter_traces(ref, pm):
    """6 trackers: 3 clips x 2 frames at fixed 100 iterations + 3 clips x 6 frames with
    the reference's early-stop defaults (eval_drag.py:204-222)."""
    cfg = synthetic.config_6_trackers()
    n_clips = 3
    wl = synthetic.make_workload(pm, ref.offsets_np.astype(np.float32), cfg, n_clips, 6)
    out = dict(latent0=wl["latent0"], tgt_pos=wl["tgt_pos"], tgt_rot=wl["tgt_rot"], joints=wl["joints"],
               weights=wl["weights"])
    fixed = dict(stop_eps_pos=-1.0, stop_eps_rot=-1.0, max_iter=100, min_loss_incr=-float("inf"), learning_rate=1e-2)
    early = dict(stop_eps_pos=0.01 * 0.01, stop_eps_rot=0.01, max_iter=100, min_loss_incr=0.00001, learning_rate=1e-2)
    for tag, opt, nf in (("fixed", fixed, 2), ("early", early, 6)):
        P, G, L, GR, LS, N, FR, FT = [], [], [], [], [], [], [], []
        for c in range(n_clips):
            poses, gposs, iters, traces, state = run_frames(ref, wl, c, nf, record_iters=True, **opt)
            lat, grad, loss, n = pack_traces(traces, 100)
            P.append(poses), G.append(gposs), L.append(lat), GR.append(grad), LS.append(loss), N.append(n)
            FR.append(state["frame_grot"]), FT.append(state["frame_tgt_latent"])
            out[f"{tag}_state_latent_{c}"] = state["latent"]
            out[f"{tag}_state_height_buf_{c}"] = state["height_buf"]
            out[f"{tag}_state_disp_buf_{c}"] = state["disp_buf"]
        out.update({f"{tag}_pose": np.stack(P, 1), f"{tag}_gpos": np.stack(G, 1), f"{tag}_latent": np.stack(L, 1),
                    f"{tag}_grad": np.stack(GR, 1), f"{tag}_loss": np.stack(LS, 1), f"{tag}_iters": np.stack(N, 1),
                    f"{tag}_grot": np.stack(FR, 1), f"{tag}_tgt_latent": np.stack(FT, 1)})
    np.savez_compressed(os.path.join(OUT, "ref_trace_6trk.npz"), **out)


def golden_frames_3trk(ref, pm):
    """3 trackers (head + hands), window 16, variable mask E in {2,3}: 2 clips x 40 frames,
    reference early-stop defaults."""
    cfg = synthetic.config_3_trackers()
    n_clips, n_frames = 2, 40
    # force some drops inside the short fixture so E = 2 is exercised
    keep = np.ones((n_frames, n_clips, 3), bool)
    keep[8:20, 0, 1] = False
    keep[25:33, 0, 2] = False
    keep[5:30, 1, 2] = False
    base = synthetic.make_workload(pm, ref.offsets_np.astype(np.float32), cfg, n_clips, n_frames)
    order = np.argsort(~keep, axis=-1, kind="stable")
    wl = dict(base)
    wl["n_ee"] = keep.sum(-1).astype(np.int32)
    wl["joints_tb"] = base["joints"][order].astype(np.int32)
    wl["weights_tb"] = base["weights"][order]
    wl["tgt_pos"] = np.take_along_axis(base["tgt_pos"], order[..., None], 2)
    wl["tgt_rot"] = np.take_along_axis(base["tgt_rot"], order[..., None, None], 2)
    early = dict(stop_eps_pos=0.01 * 0.01, stop_eps_rot=0.01, max_iter=100, min_loss_incr=0.00001, learning_rate=1e-2)
    P, G, N, TB = [], [], [], []
    for c in range(n_clips):
        poses, gposs, iters, _, state = run_frames(ref, wl, c, n_frames, record_iters=True, **early)
        P.append(poses), G.append(gposs), N.append(np.asarray(iters, np.int32)), TB.append(state["target_buf"])
    np.savez_compressed(
        os.path.join(OUT, "ref_frames_3trk.npz"), latent0=wl["latent0"], tgt_pos=wl["tgt_pos"], tgt_rot=wl["tgt_rot"],
        n_ee=wl["n_ee"], joints_tb=wl["joints_tb"], weights_tb=wl["weights_tb"], pose=np.stack(P, 1),
        gpos=np.stack(G, 1), iters=np.stack(N, 1), target_buf=np.stack(TB, 0))


def golden_temporal(ref):
    """Predictor I/O: random ring buffers -> target_latent_buffer for W = 0 and W = 16."""
    g = torch.Generator().manual_seed(77)
    B = 4
    lat = torch.randn(B, 60, 24, generator=g) * 0.5
    disp = torch.randn(B, 60, 3, generator=g) * 0.01
    hts = torch.randn(B, 60, 6, generator=g) * 0.3 + 0.8
    out = dict(latent_buf=lat.numpy(), disp_buf=disp.numpy(), height_buf=hts.numpy())
    for W in (0, 16):
        bufs = []
        for c in range(B):
            drag = ref.new_drag()
            drag.set_initial_pose(torch.zeros(1, 176, 1), torch.zeros(1, 3, 1),
                                  torch.tensor([[1.0, 0, 0, 0]]).unsqueeze(-1), torch.zeros(6))
            drag.latent_buffer, drag.displacement_buffer, drag.heights_buffer = lat[c].clone(), disp[c].clone(), hts[c].clone()
            pos = torch.zeros(6, 3)
            rot = torch.eye(3).expand(6, 3, 3).clone()
            drag.run(pos, rot, torch.tensor([0, 3, 7, 13, 17, 21]), torch.ones(6, 2), ref.offsets, max_iter=1,
                     temporal_future_window=W, stop_eps_pos=-1, stop_eps_rot=-1)
            bufs.append(drag.target_latent_buffer.numpy().copy())
        out[f"target_buf_w{W}"] = np.stack(bufs)
    np.savez_compressed(os.path.join(OUT, "ref_temporal.npz"), **out)


def golden_temporal_pt_layout(ref):
    """What train_temporal.load_model (train_temporal.py:474-482) reads from temporal.pt: the checkpoint's keys (train.py:311-319),
    the shapes of the latent statistics and the names and shapes of the reference Temporal module's state dict, which
    load_state_dict requires exactly."""
    import json

    layout = {"checkpoint_keys": ["model_state_dict", "means_latent", "stds_latent"], "means_latent": [24], "stds_latent": [24],
              "model_state_dict": {k: list(v.shape) for k, v in ref.temporal.state_dict().items()}}
    with open(os.path.join(OUT, "temporal_pt_layout.json"), "w") as fh:
        json.dump(layout, fh, indent=1)
        fh.write("\n")


def golden_rundrag(ref):
    """The C-ABI session of DragPoserDLL/main.cpp:17-38 driven through the reference's
    RunDrag (run_drag.py) with the example skeleton: 6 frames, MaxIter 10, lr 0.01, window 60."""
    rh.activate()
    import run_drag
    import train_temporal

    def load_random_predictor(module, path, device):  # temporal.pt is a missing blob
        module.load_state_dict(dpm.random_temporal_state(2222))
        return torch.zeros(24), torch.ones(24)

    train_temporal.load_model = load_random_predictor
    import contextlib
    import io

    with contextlib.redirect_stdout(io.StringIO()):
        rd = run_drag.RunDrag()
        rd.set_reference_skeleton(rh.EXAMPLE_BVH)
        rd.load_models(rh.MODEL_DIR)
    mask = np.array([1, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0, 1], np.float32)
    weights = np.array(synthetic._W, np.float32)
    rd.set_mask_and_weights(mask, weights)
    rd.init_drag_pose(np.array([[-2.6648, 0.9977, 3.7518]], np.float32), np.array([[0.6381, 0.0078, -0.7698, 0.0110]], np.float32))
    latent0 = rd.drag.latent.detach().numpy()[0].copy()
    rd.set_optim_params(0.01 * 0.01, 0.01, 10, 0.01)
    rd.set_lambdas(1, 0.02, 60)
    pos = np.array([[0, 0, 0], [0.0953, -0.8287, 0.0786], [-0.0835, -0.8810, 0.0721], [-0.0032, 0.6362, 0.0252],
                    [-0.1830, -0.0721, 0.1874], [-0.0642, -0.0306, -0.2561]], np.float32)
    rot = np.array([[-0.6381, -0.0078, 0.7698, -0.0110], [0.7759, 0.2940, -0.5198, 0.2034],
                    [-0.3807, -0.0448, 0.9235, -0.0174], [-0.5807, 0.0365, 0.8109, 0.0632],
                    [-0.2944, -0.4933, 0.6859, 0.4468], [0.6386, -0.5011, -0.3526, 0.4655]], np.float32)
    rng = np.random.default_rng(5)
    T = 6
    tp = pos[None] + rng.normal(0, 0.01, (T, 6, 3)).astype(np.float32)
    tp[:, 0] = 0
    res_pose, res_gpos = np.zeros((T, 22, 4), np.float32), np.zeros((T, 1, 3), np.float32)
    for t in range(T):
        rd.drag_pose(tp[t].copy(), rot.copy(), res_pose[t], res_gpos[t])
        rd.set_global_pos(res_gpos[t].copy())
    np.savez_compressed(os.path.join(OUT, "ref_rundrag.npz"), latent0=latent0, mask=mask, weights=weights, tgt_pos=tp,
                        tgt_quat=rot, result_pose=res_pose, result_gpos=res_gpos)


def golden_eval_bvh(ref, n_frames=48):
    """Config #1 of BASELINE.json on an excerpt: the evaluation loop of python/src/eval_drag.py:62-224 (the reference's own
    TestMotionData / from_root_quat / pymotion-fk / DragPose.run calls) on the first frames of example.bvh with
    config/6_trackers_config.json.  Also writes the BVH excerpt itself (data: CC BY-SA 4.0, LICENSE_data)."""
    rh.activate()
    import train
    from motion_data import TestMotionData
    from pymotion.ops.forward_kinematics_torch import fk
    from utils import from_root_quat

    src = open(rh.EXAMPLE_BVH).read().split("\n")
    m = src.index("MOTION")
    excerpt = src[: m + 1] + [f"Frames: {n_frames}", src[m + 2]] + src[m + 3 : m + 3 + n_frames]
    with open(os.path.join(OUT, "example_48f.bvh"), "w") as fh:
        fh.write("\n".join(excerpt) + "\n")
    cfg = ref.load_config("6_trackers_config.json")
    mask = torch.tensor(cfg["mask"])
    weights = torch.tensor(cfg["weights"], dtype=torch.float32)
    ds = TestMotionData(train.param, train.scale, "cpu", height_indices=[0, 4, 8, 13, 17, 21])
    ds.set_means_stds(ref.means, ref.stds)
    ds.add_motion(ref.offsets_np, ref.pos[:n_frames, 0, :], ref.rots[:n_frames], ref.parents, ref.bvh, "example_48f.bvh")
    ds.normalize()
    nm = ds.get_item(0)
    mask_indices = torch.nonzero(mask).squeeze()
    weights = weights[mask_indices]
    drag = ref.new_drag()
    inp = nm["dqs"].unsqueeze(0).permute(0, 2, 1)
    gpos, grot, heights = nm["global_pos"], nm["global_rot"], nm["heights"]
    torch.manual_seed(4242)
    drag.set_initial_pose(torch.tile(inp[..., 0:1], (1, 1, 1)), gpos[..., 0:1], grot[..., 0:1], heights[0])
    latent0 = drag.latent.detach().numpy()[0].copy()
    poses, gps, its = [], [], []
    rec = Recorder(drag)
    for i in range(n_frames):
        tq = inp[..., i : i + 1].clone().reshape((1, -1, 8, 1))[..., :4, :].flatten(1, 2)
        tq = tq * drag.stds_dqs + drag.means_dqs
        tq[:, :4, :] = grot[..., i : i + 1]
        loc = from_root_quat(tq.permute(0, 2, 1).reshape((1, 1, -1, 4)), drag.parents)
        disp = (gpos[..., i : i + 1] - drag.current_global_pos.detach().clone()).permute(0, 2, 1)
        p, R = fk(loc, disp, ref.offsets, drag.parents)
        pose, gp = drag.run(target_ee_pos=p[0, 0, mask_indices, :], target_ee_rot=R[0, 0, mask_indices, :, :], mask_joints=mask_indices,
                            weights_joints=weights, offsets=ref.offsets, stop_eps_pos=0.01 * 0.01, stop_eps_rot=0.01, max_iter=100,
                            min_loss_incr=0.00001, learning_rate=1e-2, lambda_rot=1, lambda_temporal=cfg["lambda_temporal"],
                            temporal_future_window=cfg["temporal_future_window"], height_indices=[0, 4, 8, 13, 17, 21],
                            joint_adjustment_indices=tuple(cfg["joint_adjustment_indices"]), joint_adjustment_weight=cfg["joint_adjustment_weight"])
        poses.append(pose.detach().numpy().copy())
        gps.append(gp.detach().numpy().copy())
        its.append(len(rec.take()))
    np.savez_compressed(os.path.join(OUT, "ref_eval_bvh.npz"), latent0=latent0, pose=np.stack(poses), gpos=np.stack(gps), iters=np.asarray(its, np.int32))


def _eval_loop(ref, n_frames, filename, seed=4242):
    """The evaluation loop of python/src/eval_drag.py:62-224 (6-tracker config) on the first n_frames of example.bvh through the
    reference's own objects; returns (latent0, results_pose (1,88,F), results_global_pos (1,3,F), iterations)."""
    rh.activate()
    import train
    from motion_data import TestMotionData
    from pymotion.ops.forward_kinematics_torch import fk
    from utils import from_root_quat

    cfg = ref.load_config("6_trackers_config.json")
    mask = torch.tensor(cfg["mask"])
    weights = torch.tensor(cfg["weights"], dtype=torch.float32)
    ds = TestMotionData(train.param, train.scale, "cpu", height_indices=[0, 4, 8, 13, 17, 21])
    ds.set_means_stds(ref.means, ref.stds)
    ds.add_motion(ref.offsets_np, ref.pos[:n_frames, 0, :], ref.rots[:n_frames], ref.parents, ref.bvh, filename)
    ds.normalize()
    nm = ds.get_item(0)
    mask_indices = torch.nonzero(mask).squeeze()
    weights = weights[mask_indices]
    drag = ref.new_drag()
    inp = nm["dqs"].unsqueeze(0).permute(0, 2, 1)
    gpos, grot, heights = nm["global_pos"], nm["global_rot"], nm["heights"]
    torch.manual_seed(seed)
    drag.set_initial_pose(torch.tile(inp[..., 0:1], (1, 1, 1)), gpos[..., 0:1], grot[..., 0:1], heights[0])
    latent0 = drag.latent.detach().numpy()[0].copy()
    results_pose = torch.zeros((1, 88, n_frames))
    results_gpos = torch.zeros((1, 3, n_frames))
    its = []
    rec = Recorder(drag)
    for i in range(n_frames):
        tq = inp[..., i : i + 1].clone().reshape((1, -1, 8, 1))[..., :4, :].flatten(1, 2)
        tq = tq * drag.stds_dqs + drag.means_dqs
        tq[:, :4, :] = grot[..., i : i + 1]
        loc = from_root_quat(tq.permute(0, 2, 1).reshape((1, 1, -1, 4)), drag.parents)
        disp = (gpos[..., i : i + 1] - drag.current_global_pos.detach().clone()).permute(0, 2, 1)
        p, R = fk(loc, disp, ref.offsets, drag.parents)
        pose, gp = drag.run(target_ee_pos=p[0, 0, mask_indices, :], target_ee_rot=R[0, 0, mask_indices, :, :], mask_joints=mask_indices,
                            weights_joints=weights, offsets=ref.offsets, stop_eps_pos=0.01 * 0.01, stop_eps_rot=0.01, max_iter=100,
                            min_loss_incr=0.00001, learning_rate=1e-2, lambda_rot=1, lambda_temporal=cfg["lambda_temporal"],
                            temporal_future_window=cfg["temporal_future_window"], height_indices=[0, 4, 8, 13, 17, 21],
                            joint_adjustment_indices=tuple(cfg["joint_adjustment_indices"]), joint_adjustment_weight=cfg["joint_adjustment_weight"])
        results_pose[..., i] = pose.detach()
        results_gpos[..., i] = gp.detach()
        its.append(len(rec.take()))
    return latent0, results_pose, results_gpos, np.asarray(its, np.int32), inp


def _reference_result_and_metrics(ref, results_pose, results_gpos, gt_dir, gt_name, n_frames):
    """eval_drag.py:228-247: train.result_to_bvh (writes data/eval_<name> under a scratch cwd) and eval_metrics.eval_pos_error
    on the ground-truth / result BVH pair, unmodified.  Returns (mpjpe, mpeepe, text of the written BVH)."""
    rh.activate()
    import tempfile

    import eval_metrics
    import train

    bvh = train.get_bvh_from_disk(gt_dir, gt_name)
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as d:
        os.chdir(d)
        os.makedirs("data")
        try:
            import contextlib
            import io

            with contextlib.redirect_stdout(io.StringIO()):
                path, fn = train.result_to_bvh(results_pose, None, ref.means, ref.stds, bvh, gt_name, save=True,
                                               res_global_pos=results_gpos, are_root_rot_incr=False)
                mpjpe, mpeepe = eval_metrics.eval_pos_error(train.get_bvh_from_disk(gt_dir, gt_name), train.get_bvh_from_disk(path, fn),
                                                            "cpu", downsample_gt=1)
            text = open(os.path.join(path, fn)).read()
        finally:
            os.chdir(cwd)
    return mpjpe, mpeepe, text


def golden_extension_losses(ref, pm):
    """SURVEY 8(f) rank 4: the reference loop with its commented-out "Additional Losses" block (drag_pose.py:129-183) re-enabled by
    oracle/reference_harness.load_drag_pose_with_extension_losses: 3 clips x 3 frames x 30 fixed iterations, 6 trackers, start root
    at (0.3, 0.9, -0.2) so that the feet-floor term sees a plausible height; per-iteration latents, gradients and the four loss values."""
    cfg = synthetic.config_6_trackers()
    n_clips, n_frames, iters = 3, 3, 30
    gpos0 = (0.3, 0.9, -0.2)
    wl = synthetic.make_workload(pm, ref.offsets_np.astype(np.float32), cfg, n_clips, n_frames, first_clip=40)
    fixed = dict(stop_eps_pos=-1.0, stop_eps_rot=-1.0, max_iter=iters, min_loss_incr=-float("inf"), learning_rate=1e-2)
    out = dict(latent0=wl["latent0"], tgt_pos=wl["tgt_pos"], tgt_rot=wl["tgt_rot"], joints=wl["joints"], weights=wl["weights"],
               gpos0=np.asarray(gpos0, np.float32))
    P, G, L, GR, LS, LE, FR, FT, FG = [], [], [], [], [], [], [], [], []
    for c in range(n_clips):
        drag = init_drag(ref, wl["latent0"][c], True, gpos0)
        rec = Recorder(drag)
        poses, gposs, lat, grad, loss, le, grots, tls, gps = [], [], [], [], [], [], [], [], []
        for t in range(n_frames):
            grots.append(drag.current_global_rot.detach().numpy()[0].copy())
            gps.append(drag.current_global_pos.detach().numpy()[0, :, 0].copy())
            pose, gpos = drag.run(torch.from_numpy(wl["tgt_pos"][t, c].copy()), torch.from_numpy(wl["tgt_rot"][t, c].copy()),
                                  torch.from_numpy(np.asarray(wl["joints"])).long(), torch.from_numpy(wl["weights"].copy()), ref.offsets,
                                  lambda_rot=1, lambda_temporal=wl["lambda_temporal"], temporal_future_window=wl["window"],
                                  joint_adjustment_indices=wl["joint_adjustment"], joint_adjustment_weight=wl["joint_adjustment_weight"], **fixed)
            tls.append(drag.target_latent_buffer[0].detach().numpy().copy())
            rows = rec.take()
            assert len(rows) == iters
            poses.append(pose.detach().numpy().copy()), gposs.append(gpos.detach().numpy().copy())
            lat.append(np.stack([r["latent"] for r in rows])), grad.append(np.stack([r["grad"] for r in rows]))
            loss.append(np.array([[r["lp"], r["lr"], r["lt"]] for r in rows])), le.append(np.array([r["le"] for r in rows]))
        P.append(np.stack(poses)), G.append(np.stack(gposs)), L.append(np.stack(lat)), GR.append(np.stack(grad)), LS.append(np.stack(loss))
        LE.append(np.stack(le)), FR.append(np.stack(grots)), FT.append(np.stack(tls)), FG.append(np.stack(gps))
    st = lambda x: np.stack(x, 1)  # (frames, clips, ...)
    out.update(pose=st(P), gpos=st(G), latent=st(L), grad=st(GR), loss=st(LS), extra=st(LE), grot=st(FR), tgt_latent=st(FT), frame_gpos=st(FG))
    print("extension losses: extra-loss range %.4g .. %.4g (tracker terms %.4g .. %.4g)" % (out["extra"].min(), out["extra"].max(),
          out["loss"][..., :2].sum(-1).min(), out["loss"][..., :2].sum(-1).max()))
    # Single evaluations (decode, loss, backward: drag_pose.py:309-343) at WILD states -- latent 1.5 N(0,I), random previous root
    # rotation and position -- because the head / hips "forward" term only switches on when the two face more than ~37 degrees
    # apart, which the optimisation trajectories above never reach.
    g = torch.Generator().manual_seed(31)
    n_wild = 32
    zw = 1.5 * torch.randn(n_wild, 24, generator=g)
    gq = torch.randn(n_wild, 4, generator=g)
    gq = gq / gq.norm(dim=1, keepdim=True)
    gp = torch.randn(n_wild, 3, generator=g) * torch.tensor([0.5, 0.3, 0.5]) + torch.tensor([0.0, 0.9, 0.0])
    tl = 0.3 * torch.randn(n_wild, 24, generator=g)
    drag = init_drag(ref, wl["latent0"][0], True, gpos0)
    mask = torch.from_numpy(np.asarray(wl["joints"])).long()
    wts = torch.from_numpy(wl["weights"].copy())
    W_grad, W_loss, W_extra = [], [], []
    for i in range(n_wild):
        drag.latent = zw[i : i + 1].clone().requires_grad_()
        drag.current_global_rot = gq[i : i + 1].clone()
        drag.current_global_pos = gp[i].reshape(1, 3, 1).clone()
        pose, disp = drag.decoder(drag.latent, drag.data.mean_dqs, drag.data.std_dqs)
        res = drag.loss(pose, disp, torch.from_numpy(wl["tgt_pos"][0, i % n_clips].copy()), torch.from_numpy(wl["tgt_rot"][0, i % n_clips].copy()),
                        tl[i], ref.offsets, mask, wts, 1, 0.02)
        (res[0] + res[1] + res[2] + res[3]).backward()
        W_grad.append(drag.latent.grad.numpy()[0].copy())
        W_loss.append([float(res[0]), float(res[1]), float(res[2])])
        W_extra.append(float(res[3]))
    out.update(wild_latent=zw.numpy(), wild_grot=gq.numpy(), wild_gpos=gp.numpy(), wild_tgt_latent=tl.numpy(), wild_clip=np.arange(n_wild) % n_clips,
               wild_grad=np.stack(W_grad), wild_loss=np.asarray(W_loss), wild_extra=np.asarray(W_extra))
    np.savez_compressed(os.path.join(OUT, "ref_extension_losses.npz"), **out)


def golden_encoder(ref, n=48):
    """Encoder.forward (autoencoder.py:136-143) of the shipped generator on real frames: every 100th frame of example.bvh,
    standardised dual quaternions exactly as eval_drag feeds them (TestMotionData), -> mu, logvar; plus one seeded
    reparameterisation draw (autoencoder.py:19-22)."""
    rh.activate()
    import train
    from motion_data import TestMotionData

    ds = TestMotionData(train.param, train.scale, "cpu", height_indices=[0, 4, 8, 13, 17, 21])
    ds.set_means_stds(ref.means, ref.stds)
    ds.add_motion(ref.offsets_np, ref.pos[:, 0, :], ref.rots, ref.parents, ref.bvh, "example.bvh")
    ds.normalize()
    nm = ds.get_item(0)
    frames = np.arange(n) * 100
    x = nm["dqs"][frames].unsqueeze(-1)  # (n,176,1)
    enc = ref.generator.autoencoder.encoder
    with torch.no_grad():
        mu, logvar = enc(x)
        torch.manual_seed(99)
        latent, mu2, logvar2 = ref.generator.autoencoder.forward_encoder(x)
    torch.manual_seed(99)
    eps = torch.randn_like(logvar)
    assert torch.equal(mu, mu2)
    np.savez_compressed(os.path.join(OUT, "ref_encoder.npz"), frames=frames, dqs=x[..., 0].numpy(), mu=mu.numpy(), logvar=logvar.numpy(),
                        eps=eps.numpy(), latent=latent.numpy())


def golden_result_path(ref):
    """Result path on the 48-frame excerpt: train.result_to_bvh output and eval_metrics.eval_pos_error values for the poses recorded in
    ref_eval_bvh.npz (train.py:437-509, eval_metrics.py:6-32)."""
    g = np.load(os.path.join(OUT, "ref_eval_bvh.npz"))
    F_ = g["pose"].shape[0]
    rp = torch.from_numpy(g["pose"].T.copy())[None]
    rg = torch.from_numpy(g["gpos"].T.copy())[None]
    mpjpe, mpeepe, text = _reference_result_and_metrics(ref, rp, rg, OUT, "example_48f.bvh", F_)
    with open(os.path.join(OUT, "ref_eval_48f_result.bvh"), "w") as fh:
        fh.write(text)
    np.savez_compressed(os.path.join(OUT, "ref_eval_metrics.npz"), mpjpe=np.float64(mpjpe), mpeepe=np.float64(mpeepe))
    print("excerpt: reference MPJPE %.6f MPEEPE %.6f" % (mpjpe, mpeepe))


def golden_eval_full(ref):
    """BASELINE config #1, the known answer of SURVEY section 4: the reference's evaluation on ALL frames of example.bvh with the
    6-tracker config (early stopping on, seed-2222 random-init predictor) -- about 6 minutes on one core.  Records the metrics of
    eval_metrics.eval_pos_error, the per-frame iteration counts and root positions, and ships the clip itself gzip-compressed
    (motion data: CC BY-SA 4.0, LICENSE_data) so the GPU box can run the same evaluation."""
    import gzip
    import io
    import time

    n_frames = ref.rots.shape[0]
    t0 = time.time()
    latent0, rp, rg, its, _ = _eval_loop(ref, n_frames, "example.bvh")
    secs = time.time() - t0
    mpjpe, mpeepe, _ = _reference_result_and_metrics(ref, rp, rg, os.path.dirname(rh.EXAMPLE_BVH), "example.bvh", n_frames)
    packed = io.BytesIO()
    with open(rh.EXAMPLE_BVH, "rb") as src, gzip.GzipFile("example_full.bvh.gz", "wb", 9, packed, mtime=0) as dst:
        dst.write(src.read())
    cut = 960000  # the gzip file in two pieces, each below 1 MB; `cat example_full.bvh.gz.1 example_full.bvh.gz.2` rejoins them
    for i, part in enumerate((packed.getvalue()[:cut], packed.getvalue()[cut:]), 1):
        with open(os.path.join(OUT, f"example_full.bvh.gz.{i}"), "wb") as fh:
            fh.write(part)
    np.savez_compressed(os.path.join(OUT, "ref_eval_full.npz"), latent0=latent0, mpjpe=np.float64(mpjpe), mpeepe=np.float64(mpeepe),
                        iters=its.astype(np.int16), gpos=rg[0].numpy().T.copy(), pose_every_100=rp[0].numpy().T[::100].copy(),
                        seconds_one_core=np.float64(secs))
    print("full clip: %d frames in %.1f s, mean %.2f iterations, reference MPJPE %.6f MPEEPE %.6f" % (n_frames, secs, its.mean(), mpjpe, mpeepe))


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    torch.set_num_threads(1)
    ref = build()
    pm = save_model_fixture(ref)
    which = sys.argv[1:] or ["trace", "frames3", "temporal", "tplayout", "rundrag", "evalbvh", "encoder", "resultpath", "extlosses"]
    if "trace" in which:
        golden_iter_traces(ref, pm)
    if "frames3" in which:
        golden_frames_3trk(ref, pm)
    if "temporal" in which:
        golden_temporal(ref)
    if "tplayout" in which:
        golden_temporal_pt_layout(ref)
    if "rundrag" in which:
        golden_rundrag(ref)
    if "evalbvh" in which:
        golden_eval_bvh(ref)
    if "encoder" in which:
        golden_encoder(ref)
    if "extlosses" in which:
        golden_extension_losses(ref, pm)
    if "resultpath" in which:
        golden_result_path(ref)
    if "evalfull" in which:  # not in the default list: ~6 minutes
        golden_eval_full(ref)
    print("golden fixtures written to", OUT)
