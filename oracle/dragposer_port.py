"""ORACLE -- test infrastructure, NOT part of the product path.

CPU (torch fp32 + autograd) restatement of DragPoser's per-frame latent
optimisation loop, batched over independent clips.  Only `tests/`,
`__graft_entry__.smoke()` and `bench.py`'s cpu_baseline / `--impl reference`
legs may import this file; `dragposer_b200/` never does.

Parity status: PINNED against the reference itself.  The reference ships no
tests or golden vectors (SURVEY.md section 4), so `oracle/make_golden.py` runs the
unmodified reference modules (`/root/reference/python/src`, imported through
`oracle/reference_harness.py`) and commits their inputs/outputs under
`tests/golden/`; `tests/test_oracle.py` checks this port against those vectors
(and, when /root/reference is present, against the live reference).

Each function cites the reference lines it restates:
  decode()            python/src/autoencoder.py:224-256, skeleton.py:117-130,244-245
  to_matrix4()        python/src/utils.py:34-76
  root_to_local()     python/src/utils.py:80-106
  fk_chain()          python/src/utils.py:109-149
  tracker_loss()      python/src/drag_pose.py:66-194
  adam_step()         torch/optim/adam.py:347-547 (single-tensor path)
  temporal_forward()  python/src/temporal_transformer.py:53-78 + torch nn.Transformer
  predict_targets()   python/src/drag_pose.py:234-294
  PortDragPose.run()  python/src/drag_pose.py:196-414
  from_root_quat()    python/src/utils.py:6-31 / train.py:409-434
Third-party arithmetic (upc-pymotion==0.1.10, absent here): quat mul / mul_vec /
inverse / normalize restated from its published semantics (SURVEY.md 8(c)).
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn.functional as F

PAST_ROWS = 60
SAMPLE_STEP = 4
PAST_INDEX = list(range(0, 60, 4))  # train_temporal.param["past_frames"]
HEIGHT_JOINTS = [0, 4, 8, 13, 17, 21]


# ------------------------------------------------------------------ quaternions
def qmul(a, b):
    w0, x0, y0, z0 = a.unbind(-1)
    w1, x1, y1, z1 = b.unbind(-1)
    return torch.stack(
        (
            w0 * w1 - x0 * x1 - y0 * y1 - z0 * z1,
            w0 * x1 + x0 * w1 + y0 * z1 - z0 * y1,
            w0 * y1 - x0 * z1 + y0 * w1 + z0 * x1,
            w0 * z1 + x0 * y1 - y0 * x1 + z0 * w1,
        ),
        -1,
    )


def qmul_vec(q, v):
    u = q[..., 1:]
    t = 2.0 * torch.cross(u, v, dim=-1)
    return v + q[..., 0:1] * t + torch.cross(u, t, dim=-1)


def qconj(q):
    return q * q.new_tensor([1.0, -1.0, -1.0, -1.0])


def qnormalize(q, eps=1e-8):
    return q / (torch.sqrt((q * q).sum(-1, keepdim=True)) + eps)


def to_matrix4(q):
    w, x, y, z = q.unbind(-1)
    x2, y2, z2 = x + x, y + y, z + z
    xx, yy, wx = x * x2, y * y2, w * x2
    xy, yz, wy = x * y2, y * z2, w * y2
    xz, zz, wz = x * z2, z * z2, w * z2
    zero, one = torch.zeros_like(w), torch.ones_like(w)
    rows = [
        torch.stack((1.0 - (yy + zz), xy - wz, xz + wy, zero), -1),
        torch.stack((xy + wz, 1.0 - (xx + zz), yz - wx, zero), -1),
        torch.stack((xz - wy, yz + wx, 1.0 - (xx + yy), zero), -1),
        torch.stack((zero, zero, zero, one), -1),
    ]
    return torch.stack(rows, -2)


def quat_to_matrix3(q):
    return to_matrix4(q)[..., :3, :3]


# ------------------------------------------------------------------ decoder
class PortWeights:
    """Unfolded decoder (as the reference executes it) + statistics + skeleton."""

    def __init__(self, npz, dtype=torch.float32):
        t = lambda k: torch.from_numpy(np.asarray(npz[k], dtype=np.float32)).to(dtype)
        self.f_w, self.f_b = t("dec_f_w"), t("dec_f_b")
        self.U = [t(f"dec_U{l}") for l in range(3)]
        self.W = [t(f"dec_W{l}") for l in range(3)]  # weight * mask
        self.b = [t(f"dec_b{l}") for l in range(3)]
        mean_dqs, std_dqs = t("mean_dqs"), t("std_dqs")
        self.mean_q = mean_dqs.reshape(-1, 8)[:, :4].reshape(-1).contiguous()
        self.std_q = std_dqs.reshape(-1, 8)[:, :4].reshape(-1).contiguous()
        self.mean_d, self.std_d = t("mean_d"), t("std_d")
        self.parents = [int(p) for p in npz["parents"]]
        self.offsets = t("offsets")


def decode(w: PortWeights, latent):
    """latent (B,24) -> standardised unit quats (B,88), standardised displacement (B,3)."""
    x = F.linear(latent, w.f_w, w.f_b)
    for l in range(3):
        x = F.linear(x, w.U[l])  # SkeletonUnpool: constant 0/1 matmul
        x = F.linear(x, w.W[l], w.b[l])  # SkeletonConv k=1 == masked Linear
        if l != 2:
            x = F.leaky_relu(x, 0.2)
    motion, disp = x[:, :-4], x[:, -4:-1]
    motion = motion * w.std_q + w.mean_q
    motion = qnormalize(motion.reshape(motion.shape[0], -1, 4)).reshape(motion.shape[0], -1)
    motion = (motion - w.mean_q) / w.std_q
    return motion, disp


# ------------------------------------------------------------------ kinematics
def root_to_local(q, parents):
    """(B,J,4) root-space quats -> (B,J,4,4) local rotation matrices."""
    rot = to_matrix4(q)
    inv = to_matrix4(qconj(q))
    par = torch.tensor(parents)
    deep = par != 0
    out = rot.clone()
    out[:, deep] = torch.matmul(inv[:, par[deep]], rot[:, deep])
    return out


def fk_chain(local, root_pos, offsets, parents):
    """Sequential chain M[i] = M[parent] @ M[i]; returns positions (B,J,3), rotmats (B,J,3,3)."""
    m = local.clone()
    m[..., :3, 3] = offsets
    m[:, 0, :3, 3] = root_pos
    mats = [m[:, 0]]
    for i in range(1, len(parents)):
        mats.append(torch.matmul(mats[parents[i]], m[:, i]))
    m = torch.stack(mats, 1)
    return m[..., :3, 3], m[..., :3, :3]


def from_root_quat(q, parents):
    """Root-space quats -> local quats (result side; numpy or torch (…,J,4))."""
    q = torch.as_tensor(q)
    out = q.clone()
    for j in reversed(range(1, q.shape[-2])):
        p = parents[j]
        if p == 0:
            continue
        out[..., j, :] = qmul(qconj(out[..., p, :]), out[..., j, :])
    return out


EXT_FEET_FLOOR, EXT_FORWARD, EXT_HEAD_HIPS, EXT_HIPS_FEET = 1, 2, 4, 8


def extension_losses(pos, rot, global_pos, mask, floor_level=0.0):
    """The four "Additional Losses" of drag_pose.py:129-183 (commented out in the shipped reference; y axis = 1), per clip (B,).
    pos (B,J,3) relative to the previous root, rot (B,J,3,3), global_pos (B,3) = current_global_pos."""
    B = pos.shape[0]
    total = pos.new_zeros(B)
    if mask & EXT_FEET_FLOOR:  # :133-135
        total = total + ((global_pos[:, 1:2] + (pos[:, [4, 8], 1] - floor_level)) ** 2).mean(1)
    if mask & EXT_FORWARD:  # :137-157; quat.mul_vec(quat.from_matrix(R), (0,0,1)) is the third column of R
        fh = rot[:, 13, :, 2] * pos.new_tensor([1.0, 0.0, 1.0])
        nh = fh.norm(dim=-1)
        fg = rot[:, 0, :, 2] * pos.new_tensor([1.0, 0.0, 1.0])
        fg = fg / fg.norm(dim=-1, keepdim=True)
        s = ((fh / nh[:, None].clamp(min=1e-30)) * fg).sum(-1) + 0.2
        term = (1 - torch.minimum(torch.ones_like(s), s)) ** 2
        total = total + torch.where(nh > 0.5, term, torch.zeros_like(term))
    flat = pos.new_tensor([1.0, 0.0, 1.0])
    if mask & EXT_HEAD_HIPS:  # :159-164 (global_pos cancels)
        total = total + (((pos[:, 13] - pos[:, 0]) * flat) ** 2).sum(-1)
    if mask & EXT_HIPS_FEET:  # :166-176
        for j in (3, 7):
            total = total + torch.clamp((((pos[:, 0] - pos[:, j]) * flat) ** 2).sum(-1) - 0.2 * 0.2, min=0.0)
    return total


def tracker_loss(w, latent, motion, disp, g_rot, tgt_pos, tgt_rot, tgt_latent, joints, weights, valid,
                 lambda_rot, lambda_temporal):
    """Per-clip loss terms (B,), plus the by-products the frame epilogue needs.

    joints (B,E) long, weights (B,E,2), valid (B,E) float {0,1}; the mean()
    denominators are 3*E_c and 9*E_c with E_c = valid.sum(1)."""
    B = latent.shape[0]
    qs = (motion * w.std_q + w.mean_q).reshape(B, -1, 4)
    d = disp * w.std_d + w.mean_d
    world_rot = qmul(g_rot, qs[:, 0])
    qs = torch.cat((world_rot[:, None], qs[:, 1:]), 1)
    local = root_to_local(qs, w.parents)
    world_disp = qmul_vec(world_rot, d)
    pos, rot = fk_chain(local, world_disp, w.offsets, w.parents)
    idx = joints[..., None]
    p_sel = torch.gather(pos, 1, idx.expand(-1, -1, 3))
    r_sel = torch.gather(rot, 1, idx[..., None].expand(-1, -1, 3, 3))
    n_e = valid.sum(1)
    lp = (((p_sel - tgt_pos) ** 2) * (weights[..., 0] * valid)[..., None]).sum((1, 2)) / (3.0 * n_e)
    lr = (((r_sel - tgt_rot) ** 2) * (weights[..., 1] * valid)[..., None, None]).sum((1, 2, 3)) / (9.0 * n_e)
    lt = ((latent - tgt_latent) ** 2).mean(1)
    return lp, lr * lambda_rot, lt * lambda_temporal, world_disp, d, world_rot, pos, rot


def adam_step(z, g, m, v, step, lr, active):
    """In-place single-tensor Adam (betas .9/.999, eps 1e-8) on the active rows;
    bias corrections in Python double exactly like torch."""
    b1, b2, eps = 0.9, 0.999, 1e-8
    for c in torch.nonzero(active).flatten().tolist():
        step[c] += 1
        t = int(step[c])
        m[c].lerp_(g[c], 1 - b1)
        v[c].mul_(b2).addcmul_(g[c], g[c], value=1 - b2)
        step_size = lr / (1 - b1**t)
        denom = (v[c].sqrt() / math.sqrt(1 - b2**t)).add_(eps)
        z[c].addcdiv_(m[c], denom, value=-step_size)


def adam_step_batched(z, g, m, v, step, lr, active):
    """Same arithmetic, vectorised over clips (identical fp32 op order)."""
    b1, b2, eps = 0.9, 0.999, 1e-8
    a = active
    step[a] += 1
    t = step[a].double()
    m[a] = torch.lerp(m[a], g[a], 1 - b1)
    v[a] = (v[a] * b2).addcmul(g[a], g[a], value=1 - b2)
    step_size = (lr / (1 - torch.pow(torch.tensor(b1, dtype=torch.float64), t))).float()[:, None]
    bc2 = torch.sqrt(1 - torch.pow(torch.tensor(b2, dtype=torch.float64), t)).float()[:, None]
    denom = v[a].sqrt() / bc2 + eps
    z[a] = z[a] + (-step_size * m[a]) / denom


# ------------------------------------------------------------------ temporal predictor
def _ln(x, sd, name):
    return F.layer_norm(x, (x.shape[-1],), sd[name + ".weight"], sd[name + ".bias"], 1e-5)


def _mha(q_in, kv_in, sd, name, n_heads=4):
    """torch MultiheadAttention (packed in_proj), batch-first tensors (B,T,d)."""
    d = q_in.shape[-1]
    w, b = sd[name + ".in_proj_weight"], sd[name + ".in_proj_bias"]
    q = F.linear(q_in, w[:d], b[:d])
    k = F.linear(kv_in, w[d : 2 * d], b[d : 2 * d])
    v = F.linear(kv_in, w[2 * d :], b[2 * d :])
    B, T, S, hd = q.shape[0], q.shape[1], k.shape[1], d // n_heads
    q = q.reshape(B, T, n_heads, hd).transpose(1, 2)
    k = k.reshape(B, S, n_heads, hd).transpose(1, 2)
    v = v.reshape(B, S, n_heads, hd).transpose(1, 2)
    att = torch.softmax((q * (1.0 / math.sqrt(hd))) @ k.transpose(-1, -2), -1)
    o = (att @ v).transpose(1, 2).reshape(B, T, d)
    return F.linear(o, sd[name + ".out_proj.weight"], sd[name + ".out_proj.bias"])


def temporal_forward(sd, enc_in, dec_in, n_enc=3, n_dec=3):
    """enc_in (B,14,33), dec_in (B,T,24) -> (B,T,24); eval mode, no masks."""
    pe = sd["positional_encoding.pos_encoding"]
    e = F.linear(enc_in, sd["in_proj_encoder.weight"], sd["in_proj_encoder.bias"]) + pe[: enc_in.shape[1]]
    t = F.linear(dec_in, sd["in_proj_decoder.weight"], sd["in_proj_decoder.bias"]) + pe[: dec_in.shape[1]]
    for l in range(n_enc):
        p = f"temporal.encoder.layers.{l}"
        e = _ln(e + _mha(e, e, sd, p + ".self_attn"), sd, p + ".norm1")
        ff = F.linear(F.relu(F.linear(e, sd[p + ".linear1.weight"], sd[p + ".linear1.bias"])),
                      sd[p + ".linear2.weight"], sd[p + ".linear2.bias"])
        e = _ln(e + ff, sd, p + ".norm2")
    e = _ln(e, sd, "temporal.encoder.norm")
    for l in range(n_dec):
        p = f"temporal.decoder.layers.{l}"
        t = _ln(t + _mha(t, t, sd, p + ".self_attn"), sd, p + ".norm1")
        t = _ln(t + _mha(t, e, sd, p + ".multihead_attn"), sd, p + ".norm2")
        ff = F.linear(F.relu(F.linear(t, sd[p + ".linear1.weight"], sd[p + ".linear1.bias"])),
                      sd[p + ".linear2.weight"], sd[p + ".linear2.bias"])
        t = _ln(t + ff, sd, p + ".norm3")
    t = _ln(t, sd, "temporal.decoder.norm")
    return F.linear(t, sd["out_proj.weight"], sd["out_proj.bias"])


def predict_targets(sd, means_latent, stds_latent, latent_buf, disp_buf, height_buf, window):
    """Ring buffers (B,60,·) in chronological order -> target_latent_buffer (B,W+1,24), in the dtype of the ring buffers
    (float64 rings, statistics and state dict give a float64 predictor)."""
    idx = PAST_INDEX
    lat = (latent_buf[:, idx[:-1]] - means_latent) / stds_latent
    dacc = torch.stack([disp_buf[:, j : j + SAMPLE_STEP].sum(1) for j in idx[:-1]], 1)
    enc_in = torch.cat((lat, dacc, height_buf[:, idx[:-1]]), -1)
    dec_in = ((latent_buf[:, idx[-1]] - means_latent) / stds_latent)[:, None]
    B = latent_buf.shape[0]
    buf = torch.zeros(B, window + 1, 24, dtype=latent_buf.dtype)
    with torch.no_grad():
        for i in range(0, window + 1, SAMPLE_STEP):
            out = temporal_forward(sd, enc_in, dec_in)
            dec_in = torch.cat((dec_in, out[:, -1:]), 1)
            buf[:, i] = out[:, -1]
    buf = buf * stds_latent + means_latent
    for i in range(0, window, SAMPLE_STEP):  # step-function "lerp" (linspace(1,1,..))
        buf[:, i : i + SAMPLE_STEP + 1] = buf[:, i + SAMPLE_STEP][:, None]
    return buf


# ------------------------------------------------------------------ the frame optimiser
class PortDragPose:
    def __init__(self, weights: PortWeights, temporal_sd, means_latent=None, stds_latent=None):
        self.w = weights
        self.sd = {k: torch.as_tensor(np.asarray(v), dtype=torch.float32) for k, v in temporal_sd.items()}
        self.means_latent = torch.zeros(24) if means_latent is None else torch.as_tensor(means_latent).float()
        self.stds_latent = torch.ones(24) if stds_latent is None else torch.as_tensor(stds_latent).float()
        self.target_buf = None
        self.trace = None  # set to [] to record per-iteration (latent, grad, lp, lr, lt, active)

    def set_initial_state(self, latent, global_pos, global_rot, heights):
        f = lambda x: torch.as_tensor(np.asarray(x), dtype=torch.float32).clone()
        self.latent = f(latent)
        B = self.latent.shape[0]
        self.gpos, self.grot = f(global_pos).reshape(B, 3), f(global_rot).reshape(B, 4)
        self.latent_buf = self.latent[:, None].repeat(1, PAST_ROWS, 1)
        self.disp_buf = torch.zeros(B, PAST_ROWS, 3)
        self.height_buf = f(heights).reshape(B, 1, 6).repeat(1, PAST_ROWS, 1)
        self.index = 0
        self.target_buf = None

    def run(self, tgt_pos, tgt_rot, joints, weights, n_ee=None, stop_eps_pos=1e-2, stop_eps_rot=1e-2,
            max_iter=100, min_loss_incr=1e-5, learning_rate=1e-3, lambda_rot=1.0, lambda_temporal=1.0,
            temporal_future_window=60, joint_adjustment=None, joint_adjustment_weight=0.01, extension_losses_mask=0, floor_level=0.0):
        f = lambda x: torch.as_tensor(np.asarray(x), dtype=torch.float32)
        B = self.latent.shape[0]
        tgt_pos, tgt_rot, weights = f(tgt_pos), f(tgt_rot), f(weights)
        joints = torch.as_tensor(np.asarray(joints)).long()
        if joints.dim() == 1:
            joints = joints[None].expand(B, -1)
        if weights.dim() == 2:
            weights = weights[None].expand(B, -1, -1)
        E = joints.shape[1]
        n_ee = torch.full((B,), E) if n_ee is None else torch.as_tensor(np.asarray(n_ee)).long()
        valid = (torch.arange(E)[None] < n_ee[:, None]).float()
        joints = torch.where(valid > 0, joints, torch.zeros_like(joints))
        W = temporal_future_window
        assert W % SAMPLE_STEP == 0
        if self.target_buf is None or self.target_buf.shape[1] != W + 1:
            self.target_buf = torch.zeros(B, W + 1, 24)
        if self.index == 0:
            self.target_buf = predict_targets(self.sd, self.means_latent, self.stds_latent,
                                              self.latent_buf, self.disp_buf, self.height_buf, W)
        tgt_latent = self.target_buf[:, self.index]

        m, v = torch.zeros(B, 24), torch.zeros(B, 24)
        step = torch.zeros(B, dtype=torch.long)
        prev = torch.full((B,), 1e7, dtype=torch.float64)
        incr = torch.ones(B, dtype=torch.float64)
        lp = torch.full((B,), float("inf"), dtype=torch.float64)
        lr = torch.full((B,), float("inf"), dtype=torch.float64)
        lt = torch.full((B,), float("inf"), dtype=torch.float64)
        keep = {}
        remaining = max_iter
        while remaining > 0:
            active = ((lp > stop_eps_pos) | (lr > stop_eps_rot)) & (incr > min_loss_incr)
            if not bool(active.any()):
                break
            z = self.latent.clone().requires_grad_(True)
            motion, disp = decode(self.w, z)
            l_p, l_r, l_t, wdisp, d_root, wrot, pos, rot_all = tracker_loss(
                self.w, z, motion, disp, self.grot, tgt_pos, tgt_rot, tgt_latent, joints, weights, valid,
                lambda_rot, lambda_temporal)
            total = l_p + l_r + l_t
            if extension_losses_mask:
                total = total + extension_losses(pos, rot_all, self.gpos, extension_losses_mask, floor_level)
            (total * active.float()).sum().backward()
            g = z.grad
            if self.trace is not None:
                self.trace.append(dict(latent=self.latent.clone().numpy(), grad=g.clone().numpy(),
                                       lp=l_p.detach().numpy().copy(), lr=l_r.detach().numpy().copy(),
                                       lt=l_t.detach().numpy().copy(), active=active.numpy().copy()))
            cur = dict(latent=self.latent.clone(), motion=motion.detach(), wdisp=wdisp.detach(),
                       d_root=d_root.detach(), wrot=wrot.detach(), pos=pos.detach())
            for k, val in cur.items():
                keep[k] = val if k not in keep else torch.where(
                    active.reshape((B,) + (1,) * (val.dim() - 1)), val, keep[k])
            adam_step_batched(self.latent, g, m, v, step, learning_rate, active)
            td = total.detach().double()
            lp = torch.where(active, l_p.detach().double(), lp)
            lr = torch.where(active, l_r.detach().double(), lr)
            lt = torch.where(active, l_t.detach().double(), lt)
            incr = torch.where(active, prev - td, incr)
            prev = torch.where(active, td, prev)
            remaining -= 1
        self.iters, self.last_losses = step.clone(), (lp, lr, lt)

        # ---- frame epilogue (drag_pose.py:369-414), from the last evaluated iteration
        self.gpos = self.gpos + keep["wdisp"]
        self.grot = keep["wrot"]
        d_root = keep["d_root"].clone()
        if joint_adjustment is not None:
            j, e = joint_adjustment
            adj = (tgt_pos[:, e] - keep["pos"][:, j]) * joint_adjustment_weight
            self.gpos = self.gpos + adj
            d_root = d_root + adj
        roll = lambda buf, new: torch.cat((buf[:, 1:], new[:, None]), 1)
        self.latent_buf = roll(self.latent_buf, keep["latent"])
        self.disp_buf = roll(self.disp_buf, d_root)
        self.height_buf = roll(self.height_buf, (keep["pos"] + self.gpos[:, None])[:, HEIGHT_JOINTS, 1])
        pose = keep["motion"].clone()
        pose[:, :4] = (self.grot - self.w.mean_q[:4]) / self.w.std_q[:4]
        self.index = 0 if W == 0 else (self.index + 1) % W
        return pose, self.gpos.clone()


# ------------------------------------------------------------------ CPU baseline timing
def time_reference_loop(npz_path, temporal_sd, n_clips, n_frames, max_iter, workload, n_threads=1):
    """Times the B=1 port loop (one clip at a time, like the reference) on this
    process; returns clip-frames per second.  `workload` provides per-clip
    (latent0, targets) -- see dragposer_b200.synthetic."""
    import time

    torch.set_num_threads(n_threads)
    w = PortWeights(np.load(npz_path))
    done, t0 = 0, time.perf_counter()
    for c in range(n_clips):
        drag = PortDragPose(w, temporal_sd)
        drag.set_initial_state(workload["latent0"][c : c + 1], np.zeros((1, 3)), [[1.0, 0, 0, 0]], np.zeros((1, 6)))
        for t in range(n_frames):
            drag.run(workload["tgt_pos"][t, c : c + 1], workload["tgt_rot"][t, c : c + 1], workload["joints"],
                     workload["weights"], stop_eps_pos=-1.0, stop_eps_rot=-1.0, max_iter=max_iter,
                     min_loss_incr=-float("inf"), learning_rate=1e-2, lambda_rot=1.0,
                     lambda_temporal=workload["lambda_temporal"], temporal_future_window=workload["window"],
                     joint_adjustment=workload["joint_adjustment"],
                     joint_adjustment_weight=workload["joint_adjustment_weight"])
            done += 1
    return done / (time.perf_counter() - t0)


def loss_and_grad(w: PortWeights, latent, g_rot, tgt_pos, tgt_rot, tgt_latent, joints, weights, n_ee=None,
                  lambda_rot=1.0, lambda_temporal=1.0, dtype=torch.float32, extension_losses_mask=0, global_pos=None, floor_level=0.0):
    """Teacher-forced evaluation: loss terms and d(loss)/d(latent) at given latents (B,24).
    dtype=torch.float64 (with PortWeights(..., dtype=torch.float64)) gives the float64 truth."""
    f = lambda x: torch.as_tensor(np.asarray(x), dtype=torch.float32).to(dtype)
    z = f(latent).clone().requires_grad_(True)
    B = z.shape[0]
    joints = torch.as_tensor(np.asarray(joints)).long()
    weights = f(weights)
    if joints.dim() == 1:
        joints = joints[None].expand(B, -1)
    if weights.dim() == 2:
        weights = weights[None].expand(B, -1, -1)
    E = joints.shape[1]
    n_ee = torch.full((B,), E) if n_ee is None else torch.as_tensor(np.asarray(n_ee)).long()
    valid = (torch.arange(E)[None] < n_ee[:, None]).to(dtype)
    joints = torch.where(valid > 0, joints, torch.zeros_like(joints))
    motion, disp = decode(w, z)
    lp, lr, lt, wdisp, d_root, wrot, pos, rot_all = tracker_loss(w, z, motion, disp, f(g_rot), f(tgt_pos), f(tgt_rot),
                                                        f(tgt_latent), joints, weights, valid, lambda_rot,
                                                        lambda_temporal)
    le = torch.zeros_like(lp)
    if extension_losses_mask:
        gp = torch.zeros(B, 3, dtype=dtype) if global_pos is None else f(global_pos)
        le = extension_losses(pos, rot_all, gp, extension_losses_mask, floor_level)
    (lp + lr + lt + le).sum().backward()
    return dict(lp=lp.detach().numpy(), lr=lr.detach().numpy(), lt=lt.detach().numpy(), le=le.detach().numpy(), grad=z.grad.numpy(),
                pos=pos.detach().numpy(), motion=motion.detach().numpy(), wrot=wrot.detach().numpy(),
                wdisp=wdisp.detach().numpy())
