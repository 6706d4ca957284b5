"""CPU: host-side logic of the package (model folding, topology, configs, BVH, rotations, sharding)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from dragposer_b200 import bvh, dist as dpdist, export_model, model, rotations, synthetic, topology
from dragposer_b200.engine import pack_temporal

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_folded_decoder_equals_unfolded(model_npz, pose_model, port_weights):
    import dragposer_port as port

    z = torch.randn(32, 24, generator=torch.Generator().manual_seed(0))
    x = torch.nn.functional.linear(z, port_weights.f_w, port_weights.f_b)
    for l in range(3):
        x = torch.nn.functional.linear(torch.nn.functional.linear(x, port_weights.U[l]), port_weights.W[l], port_weights.b[l])
        if l != 2:
            x = torch.nn.functional.leaky_relu(x, 0.2)
    y = pose_model.decode_np(z.numpy())
    assert np.abs(y - x.numpy()).max() / np.abs(y).max() < 1e-6


def test_topology_reproduces_shipped_masks(model_npz):
    """The unfolded weights of the fixture are weight*mask: their zero pattern must lie inside our topology masks,
    and the unpool matrices must be identical (skeleton.py:133-175,213-245,341-362)."""
    layers, primal = topology.decoder_plan(list(model_npz["parents"]))
    assert primal == 24 and [u.shape for u, _ in layers] == [(40, 24), (60, 40), (92, 60)]
    for l, (U, M) in enumerate(layers):
        assert np.array_equal(U, model_npz[f"dec_U{l}"])
        W = model_npz[f"dec_W{l}"]
        assert not np.any((W != 0) & (M == 0))
        assert int(M.sum()) == [1120, 1456, 2032][l]
    enc, primal_e = topology.encoder_plan(list(model_npz["parents"]))
    assert primal_e == 48 and [m.shape[0] for m, _ in enc] == [176, 112, 72]


def test_random_init_same_architecture():
    rp = model.random_pose_model(3)
    assert [a.shape for a in rp.A] == [(40, 24), (60, 40), (92, 60)] and [a.shape for a in rp.enc_A] == [(112, 176), (72, 112), (48, 72)]
    assert np.isfinite(rp.decode_np(np.zeros((2, 24), np.float32))).all()


def test_temporal_blob_layout(temporal_model):
    blob = pack_temporal(temporal_model)
    assert blob.size == 1283976 and blob.dtype == np.float32
    w = temporal_model.sd["in_proj_encoder.weight"]  # (48,33) stored transposed first
    assert np.array_equal(blob[: 33 * 48].reshape(33, 48), w.T)
    assert np.array_equal(blob[-24:], temporal_model.sd["out_proj.bias"])
    sd2 = model.random_temporal_state(2222)  # seeded construction is reproducible and does not disturb the global RNG
    torch.manual_seed(5)
    a = torch.rand(1)
    torch.manual_seed(5)
    model.random_temporal_state(2222)
    assert torch.equal(a, torch.rand(1))
    assert all(np.array_equal(np.asarray(sd2[k]), temporal_model.sd[k]) for k in temporal_model.sd)


def test_tracker_config_json_roundtrip(tmp_path):
    cfg = synthetic.config_3_trackers()
    data = dict(mask=cfg.mask.tolist(), weights=cfg.weights.tolist(), enable_joint_adjustment=True, joint_adjustment_indices=[13, 0],
                joint_adjustment_weight=0.1, lambda_temporal=0.15, temporal_future_window=16)
    p = tmp_path / "cfg.json"
    p.write_text(json.dumps(data))
    c2 = synthetic.TrackerConfig.load(str(p))
    assert c2.joints.tolist() == [13, 17, 21] and c2.tracker_weights[0].tolist() == [20, 20]
    assert c2.joint_adjustment == (13, 0) and c2.temporal_future_window == 16
    six = synthetic.config_6_trackers()
    assert six.joints.tolist() == [0, 3, 7, 13, 17, 21] and six.lambda_temporal == 0.02 and six.temporal_future_window == 0
    with pytest.raises(ValueError):
        synthetic.TrackerConfig(dict(data, weights=[[1, 2]] * 21))


def test_synthetic_workload_is_deterministic_and_orthonormal(pose_model, model_npz):
    cfg = synthetic.config_6_trackers()
    a = synthetic.make_workload(pose_model, model_npz["offsets"], cfg, 4, 3)
    b = synthetic.make_workload(pose_model, model_npz["offsets"], cfg, 2, 3, first_clip=2)
    assert np.array_equal(a["tgt_pos"][:, 2:], b["tgt_pos"]) and np.array_equal(a["latent0"][2:], b["latent0"])  # clip c depends on c only
    R = a["tgt_rot"]
    assert np.abs(R @ np.swapaxes(R, -1, -2) - np.eye(3)).max() < 1e-5
    v = synthetic.make_workload(pose_model, model_npz["offsets"], synthetic.config_3_trackers(), 64, 200, variable_mask=True)
    assert v["n_ee"].min() >= 2 and v["n_ee"].max() == 3 and (v["joints_tb"][..., 0] == 13).all()


def test_bvh_reader_and_rotations():
    b = bvh.Bvh(os.path.join(ROOT, "tests", "golden", "skeleton22.bvh"))
    par, off = b.skeleton()
    assert par == list(model.DEFAULT_PARENTS) and off.shape == (22, 3) and np.all(off[0] == 0)
    assert np.allclose(b.quaternions(), np.tile([1.0, 0, 0, 0], (1, 22, 1)))
    rng = np.random.default_rng(0)
    q = rotations.normalize(rng.standard_normal((5, 22, 4)))
    loc = rotations.from_root_quat(q, par)
    for j in range(1, 22):  # rebuilding root-space rotations from the local ones gives q back
        p = par[j]
        back = loc[:, j] if p == 0 else rotations.mul(q[:, p], loc[:, j])
        assert np.abs(back - q[:, j]).max() < 1e-6
    v = rng.standard_normal((5, 22, 3))
    assert np.abs(np.einsum("...ij,...j->...i", rotations.to_matrix(q), v) - rotations.mul_vec(q, v)).max() < 1e-6


def test_export_model_roundtrip(tmp_path, pose_model):
    out = export_model.export(os.path.join(ROOT, "tests", "golden", "model_dancedb.npz"), str(tmp_path / "m.dpm"), allow_random_temporal=True)
    raw = open(out, "rb").read()
    assert raw[:4] == b"DPM1"
    version, n, flags = (int(v) for v in np.frombuffer(raw[4:16], np.uint32))
    assert version == 2 and flags == 0  # bit 0 clear: the predictor is the random-init stand-in, not a temporal.pt
    flat = np.frombuffer(raw[16:], np.float32)
    assert flat.size == n == sum(c for _, c in export_model.DPM_FIELDS) + 1283976 + 48
    assert np.array_equal(flat[:960].reshape(40, 24), pose_model.A[0])


def test_shard_bounds_cover_all_clips():
    for n, w in ((4096, 8), (4097, 8), (10, 4), (3, 8)):
        seen = []
        for r in range(w):
            lo, hi, per = dpdist.shard_bounds(n, w, r)
            assert hi - lo <= per
            seen += list(range(lo, hi))
        assert seen == list(range(n))


def test_gloo_world_size_2_gather_keeps_clip_order(tmp_path):
    """N > 1 path on CPU: two gloo ranks gather their result rows; row c of the result is clip c."""
    script = tmp_path / "w.py"
    script.write_text(f"""
import os, sys
sys.path.insert(0, {ROOT!r})
import torch, torch.distributed as dist
from dragposer_b200 import dist as dpdist
dist.init_process_group('gloo')
rank, world = dist.get_rank(), dist.get_world_size()
n = 7
lo, hi, per = dpdist.shard_bounds(n, world, rank)
pose = torch.arange(lo, hi, dtype=torch.float32)[:, None].repeat(1, 88) + 0.5
gpos = torch.arange(lo, hi, dtype=torch.float32)[:, None].repeat(1, 3) - 0.25
P, G = dpdist.gather_results(pose, gpos, n)
assert P.shape == (n, 88) and G.shape == (n, 3)
assert torch.equal(P[:, 0], torch.arange(n, dtype=torch.float32) + 0.5) and torch.equal(G[:, 2], torch.arange(n, dtype=torch.float32) - 0.25)
# a batch of frames in one collective, to the rank that consumes them: frame t, clip c carries 100 t + c
T = 3
pf = pose[None] + 100.0 * torch.arange(T, dtype=torch.float32)[:, None, None]
gf = gpos[None] + 100.0 * torch.arange(T, dtype=torch.float32)[:, None, None]
got = dpdist.gather_frames(pf, gf, n, dst=0)
want = 100.0 * torch.arange(T, dtype=torch.float32)[:, None] + torch.arange(n, dtype=torch.float32)[None]
if rank == 0:
    for t in range(T):
        assert got.pose(t).shape == (n, 88) and got.global_pos(t).shape == (n, 3)
        assert torch.equal(got.pose(t)[:, 5], want[t] + 0.5) and torch.equal(got.global_pos(t)[:, 1], want[t] - 0.25)
    assert torch.equal(got.clip(5)[:, 0], want[:, 5] + 0.5)  # one clip over the frames: a view into the receive buffer
else:
    assert got is None
# the engine's own wire layout (packed rows as the frame kernels write them), asynchronously, into a preallocated buffer
rows = torch.zeros((T, per, dpdist.ROW))
rows[:, : hi - lo, :88] = pf
rows[:, : hi - lo, 88:91] = gf
out = torch.empty((world, T, per, dpdist.ROW)) if rank == 1 else None
got, work = dpdist.gather_packed(rows, n, dst=1, out=out, async_op=True)
work.wait()
if rank == 1:
    assert got.buffer is out and torch.equal(got.pose(2)[:, 7], want[2] + 0.5)
else:
    assert got is None
dist.destroy_process_group()
print('rank', rank, 'ok')
""")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29617", str(script)], capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.count("ok") == 2


def test_engine_fails_loudly_without_library(monkeypatch, tmp_path):
    from dragposer_b200 import _lib

    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "ENGINE_SO", str(tmp_path / "nope.so"))
    with pytest.raises(_lib.EngineError, match="no CPU fallback"):
        _lib.load()


def test_bench_output_dump_is_a_fixed_sample_below_64_mb(tmp_path):
    """bench.py --dump-outputs: every clip while they fit; above that the same seeded sample of clips on every run, in clip order,
    with all arrays of one dump together below 64 MB."""
    import bench

    small = np.arange(5 * 91, dtype=np.float32).reshape(5, 91)
    bench.dump_outputs(str(tmp_path / "a"), {"": small})
    assert np.array_equal(np.load(tmp_path / "a" / "pose.npy"), small[:, :88])
    assert np.array_equal(np.load(tmp_path / "a" / "global_pos.npy"), small[:, 88:91])
    big = np.repeat(np.arange(200_000, dtype=np.float32)[:, None], 91, 1)  # row c holds c; 73 MB per workload
    for d in ("b", "c"):
        bench.dump_outputs(str(tmp_path / d), {"": big, "3trk_var_": big})
    assert sum(f.stat().st_size for f in (tmp_path / "b").iterdir()) <= 64 << 20
    for name in ("pose", "global_pos", "3trk_var_pose", "3trk_var_global_pos"):
        x, y = np.load(tmp_path / "b" / f"{name}.npy"), np.load(tmp_path / "c" / f"{name}.npy")
        assert x.dtype == np.float32 and np.array_equal(x, y)
    assert (np.diff(np.load(tmp_path / "b" / "pose.npy")[:, 0]) > 0).all()
