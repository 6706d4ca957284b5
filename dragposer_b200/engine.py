"""Batched B200 engine: B independent clips optimised per frame in one launch.

Thin Python over the dp_engine_* C ABI (include/dp_engine.h, csrc/dp_engine.cu).
Semantics per clip are those of the reference's `DragPose` (python/src/drag_pose.py):
`set_initial_state` == `set_initial_pose` (:47-64) with the latent supplied by the
caller (the reference draws it from torch's RNG, :50 + autoencoder.py:19-22), `run`
== `DragPose.run` (:196-414).
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np

from . import _lib
from .model import PoseModel, TemporalModel, N_ENC, N_DEC

F32 = np.float32


def _f32(x):
    return np.ascontiguousarray(x, dtype=F32)


def _i32(x):
    return np.ascontiguousarray(x, dtype=np.int32)


def _ptr(a):
    return None if a is None else C.c_void_p(a.ctypes.data)


def pack_temporal(tm: TemporalModel) -> np.ndarray:
    """Float32 blob in the order of csrc/dp_temporal.cuh:tp_layout(); every Linear
    weight transposed to [in][out].  Keys are `Temporal.state_dict()` names
    (python/src/temporal_transformer.py:15-34)."""
    sd = tm.sd
    parts = []
    T = lambda k: parts.append(np.ascontiguousarray(sd[k].T, dtype=F32).reshape(-1))
    V = lambda k: parts.append(np.ascontiguousarray(sd[k], dtype=F32).reshape(-1))

    def attn(p):
        T(p + ".in_proj_weight"), V(p + ".in_proj_bias"), T(p + ".out_proj.weight"), V(p + ".out_proj.bias")

    def ff(p):
        T(p + ".linear1.weight"), V(p + ".linear1.bias"), T(p + ".linear2.weight"), V(p + ".linear2.bias")

    def norm(p):
        V(p + ".weight"), V(p + ".bias")

    T("in_proj_encoder.weight"), V("in_proj_encoder.bias")
    T("in_proj_decoder.weight"), V("in_proj_decoder.bias")
    V("positional_encoding.pos_encoding")
    for l in range(N_ENC):
        p = f"temporal.encoder.layers.{l}"
        attn(p + ".self_attn"), ff(p), norm(p + ".norm1"), norm(p + ".norm2")
    norm("temporal.encoder.norm")
    for l in range(N_DEC):
        p = f"temporal.decoder.layers.{l}"
        attn(p + ".self_attn"), attn(p + ".multihead_attn"), ff(p)
        norm(p + ".norm1"), norm(p + ".norm2"), norm(p + ".norm3")
    norm("temporal.decoder.norm")
    T("out_proj.weight"), V("out_proj.bias")
    for a in parts:
        assert a.size % 4 == 0
    return np.concatenate(parts)


# bits of `extension_losses`: the reference's "Additional Losses" (python/src/drag_pose.py:129-183, commented out as shipped)
EXT_FEET_FLOOR, EXT_FORWARD, EXT_HEAD_HIPS, EXT_HIPS_FEET = 1, 2, 4, 8


class RunOptions:
    """Keyword surface of DragPose.run (python/src/drag_pose.py:196-215), same defaults, plus the engine's own switches
    (decoder_path, targets_world, extension_losses / floor_level -- see include/dp_engine.h:dp_run_params)."""

    def __init__(self, stop_eps_pos=1e-2, stop_eps_rot=1e-2, max_iter=100, min_loss_incr=0.00001, learning_rate=1e-3,
                 lambda_rot=1, lambda_temporal=1, temporal_future_window=60, joint_adjustment_indices=None,
                 joint_adjustment_weight=0.01, decoder_path=0, targets_world=False, extension_losses=0, floor_level=0.0):
        self.c = _lib.RunParams(
            float(stop_eps_pos), float(stop_eps_rot), float(min_loss_incr), int(max_iter), float(learning_rate),
            float(lambda_rot), float(lambda_temporal), int(temporal_future_window),
            -1 if joint_adjustment_indices is None else int(joint_adjustment_indices[0]),
            0 if joint_adjustment_indices is None else int(joint_adjustment_indices[1]),
            float(joint_adjustment_weight), int(decoder_path), int(bool(targets_world)), int(extension_losses), float(floor_level))


class ClipOptions:
    """The per-clip keywords of DragPose.run (python/src/drag_pose.py:196-215), same defaults: one clip's optimiser settings in a
    batch whose clips run with different settings (BatchedDragPose.set_clip_options; include/dp_engine.h:dp_clip_settings)."""

    def __init__(self, stop_eps_pos=1e-2, stop_eps_rot=1e-2, max_iter=100, min_loss_incr=0.00001, learning_rate=1e-3,
                 lambda_rot=1, lambda_temporal=1, joint_adjustment_indices=None, joint_adjustment_weight=0.01):
        self.c = _lib.ClipSettings(
            float(stop_eps_pos), float(stop_eps_rot), float(min_loss_incr), int(max_iter), float(learning_rate), float(lambda_rot),
            float(lambda_temporal), -1 if joint_adjustment_indices is None else int(joint_adjustment_indices[0]),
            0 if joint_adjustment_indices is None else int(joint_adjustment_indices[1]), float(joint_adjustment_weight))


class BatchedDragPose:
    def __init__(self, pose: PoseModel, offsets, temporal: TemporalModel, max_clips: int, device: int = 0):
        self.lib = _lib.load()
        self.pose, self.temporal = pose, temporal
        self.offsets = _f32(offsets).reshape(22, 3)
        self.max_clips = int(max_clips)
        h = C.c_void_p()
        _lib.check(self.lib.dp_engine_create(C.byref(h), int(device), self.max_clips))
        self.h = h
        self.device = int(device)
        keep = [_f32(pose.A[0]), _f32(pose.b[0]), _f32(pose.A[1]), _f32(pose.b[1]), _f32(pose.A[2]), _f32(pose.b[2]),
                _f32(pose.mean_q), _f32(pose.std_q), _f32(pose.mean_d), _f32(pose.std_d)]
        par = _i32(pose.parents)
        pm = _lib.PoseModelC(*[a.ctypes.data_as(_lib.c_float_p) for a in keep], par.ctypes.data_as(_lib.c_int32_p),
                             self.offsets.ctypes.data_as(_lib.c_float_p))
        _lib.check(self.lib.dp_engine_set_pose_model(self.h, C.byref(pm)))
        if pose.enc_A:  # folded encoder: clip start-up on the device (encode / set_initial_pose)
            enc = [_f32(pose.enc_A[0]), _f32(pose.enc_b[0]), _f32(pose.enc_A[1]), _f32(pose.enc_b[1]), _f32(pose.enc_A[2]), _f32(pose.enc_b[2]),
                   _f32(pose.enc_mu[0]), _f32(pose.enc_mu[1]), _f32(pose.enc_logvar[0]), _f32(pose.enc_logvar[1])]
            em = _lib.EncoderModelC(*[a.ctypes.data_as(_lib.c_float_p) for a in enc])
            _lib.check(self.lib.dp_engine_set_encoder_model(self.h, C.byref(em)))
        if temporal is not None:
            blob = pack_temporal(temporal)
            assert blob.size == self.lib.dp_engine_temporal_blob_floats(), (blob.size, self.lib.dp_engine_temporal_blob_floats())
            ml, sl = _f32(temporal.means_latent), _f32(temporal.stds_latent)
            _lib.check(self.lib.dp_engine_set_temporal_model(self.h, _ptr(blob), blob.size, _ptr(ml), _ptr(sl)))
        self.n_clips = 0

    def close(self):
        if getattr(self, "h", None):
            self.lib.dp_engine_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ state
    def set_initial_state(self, latent, global_pos, global_rot, heights):
        latent = _f32(latent).reshape(-1, 24)
        B = latent.shape[0]
        gp, gr, ht = _f32(global_pos).reshape(B, 3), _f32(global_rot).reshape(B, 4), _f32(heights).reshape(B, 6)
        _lib.check(self.lib.dp_engine_init_clips(self.h, B, _ptr(latent), _ptr(gp), _ptr(gr), _ptr(ht)))
        self.n_clips = B

    def initial_latent(self, dqs_std, eps=None):
        """Encoder + reparameterisation (autoencoder.py:19-27): mu + eps * exp(0.5 logvar);
        eps = None gives mu (the reference draws eps ~ N(0,I) from torch's RNG)."""
        mu, logvar = self.pose.encode_np(_f32(dqs_std).reshape(-1, 176))
        return mu if eps is None else mu + _f32(eps) * np.exp(F32(0.5) * logvar)

    def set_global_pos(self, global_pos, first_clip=0):
        gp = _f32(global_pos).reshape(-1, 3)
        _lib.check(self.lib.dp_engine_set_global_pos(self.h, int(first_clip), gp.shape[0], _ptr(gp)))

    def state(self, window=None):
        B = self.n_clips
        out = dict(latent=np.empty((B, 24), F32), global_pos=np.empty((B, 3), F32), global_rot=np.empty((B, 4), F32),
                   latent_buf=np.empty((B, 60, 24), F32), disp_buf=np.empty((B, 60, 3), F32),
                   height_buf=np.empty((B, 60, 6), F32))
        tb = None if window is None else np.empty((B, window + 1, 24), F32)
        idx = C.c_int(0)
        _lib.check(self.lib.dp_engine_get_state(self.h, _ptr(out["latent"]), _ptr(out["global_pos"]), _ptr(out["global_rot"]),
                                                _ptr(out["latent_buf"]), _ptr(out["disp_buf"]), _ptr(out["height_buf"]),
                                                _ptr(tb), C.byref(idx)))
        out["target_buf"], out["current_index"] = tb, idx.value
        return out

    def set_ring_buffers(self, latent_buf, disp_buf, height_buf):
        B = self.n_clips
        a, b, c = _f32(latent_buf).reshape(B, 60, 24), _f32(disp_buf).reshape(B, 60, 3), _f32(height_buf).reshape(B, 60, 6)
        _lib.check(self.lib.dp_engine_set_ring_buffers(self.h, _ptr(a), _ptr(b), _ptr(c)))

    def encode(self, dqs, eps=None):
        """Folded pose-VAE encoder + reparameterisation on the device: standardised dual quats (n,176) and optional standard-normal
        draws eps (n,24) -> latent (n,24) = mu + eps * exp(0.5 logvar) (autoencoder.py:19-27,136-143); eps=None gives mu."""
        x = _f32(dqs).reshape(-1, 176)
        n = x.shape[0]
        e = None if eps is None else _f32(eps).reshape(n, 24)
        out = np.empty((n, 24), F32)
        _lib.check(self.lib.dp_engine_encode_host(self.h, n, _ptr(x), _ptr(e), _ptr(out)))
        return out

    def set_initial_pose(self, dqs, global_pos, global_rot, heights, eps=None):
        """Batched DragPose.set_initial_pose (drag_pose.py:47-64): encode the first pose of every clip on the device, then
        initialise the clips (ring buffers tiled with the initial latent / heights)."""
        self.set_initial_state(self.encode(dqs, eps), global_pos, global_rot, heights)

    def restart_clips(self, clips, latent, global_pos, global_rot, heights):
        """Restart the clips `clips` (unique ids < n_clips) with latent (n,24), global_pos (n,3), global_rot (n,4), heights (n,6),
        like set_initial_state does for every clip, while the others keep running.  Each restarted clip's next frame is its own
        frame 0.  Restarting when frames_to_boundary(window) == 0 keeps the lockstep path; elsewhere the restarted clips get
        their own predictor phase (include/dp_engine.h:dp_engine_restart_clips)."""
        ids = _i32(clips).reshape(-1)
        n = ids.shape[0]
        z, gp = _f32(latent).reshape(n, 24), _f32(global_pos).reshape(n, 3)
        gr, ht = _f32(global_rot).reshape(n, 4), _f32(heights).reshape(n, 6)
        _lib.check(self.lib.dp_engine_restart_clips(self.h, n, _ptr(ids), _ptr(z), _ptr(gp), _ptr(gr), _ptr(ht), None))

    def restart_pose(self, clips, dqs, global_pos, global_rot, heights, eps=None):
        """restart_clips with the latent encoded on the device from standardised dual quats (n,176) (see set_initial_pose)."""
        self.restart_clips(clips, self.encode(dqs, eps), global_pos, global_rot, heights)

    def set_clip_options(self, options, which=None):
        """Per-clip optimiser settings: clip c runs with options[which[c]] (which: (n_clips,) ints; None = options[0] for every
        clip), bit for bit as a batch of only the clips of that entry would run with those keywords.  While they are set, the
        per-clip keywords of run / run_frames / run_frames_device are ignored; their temporal_future_window, decoder_path,
        targets_world, extension_losses and floor_level still apply to the whole batch.  options=None clears them.
        set_initial_state clears them too; restart_clips keeps every clip's entry.  On the fp32 frame kernel each entry in use runs as
        a batch of its own, one after the other (DESIGN.md section 3.4)."""
        if options is None:
            _lib.check(self.lib.dp_engine_set_clip_settings(self.h, 0, None, None))
            return
        options = list(options)
        table = (_lib.ClipSettings * max(1, len(options)))(*[o.c for o in options])
        idx = None if which is None else _i32(which).reshape(-1)
        if idx is not None and idx.shape[0] != self.n_clips:
            raise ValueError(f"which must hold one index per clip ({self.n_clips}), got {idx.shape[0]}")
        _lib.check(self.lib.dp_engine_set_clip_settings(self.h, len(options), C.cast(table, C.c_void_p), _ptr(idx)))

    def clip_index(self, window):
        """Own temporal index of every clip for the next frame run with `window` (B,) -- DragPose.current_index per clip."""
        out = np.empty(self.n_clips, np.int32)
        _lib.check(self.lib.dp_engine_get_clip_index(self.h, int(window), _ptr(out)))
        return out

    def frames_to_boundary(self, window):
        """Frames until the next frame at which a restart costs no extra predictor call (0 = the next frame)."""
        rc = self.lib.dp_engine_frames_to_boundary(self.h, int(window))
        if rc < 0:
            _lib.check(rc)
        return int(rc)

    def pose_error(self, pose_a, pose_b):
        """Per-row MPJPE and MPEEPE (metres) between two sets of poses in the engine's output format (n,88), computed on the
        device (eval_metrics.py:6-32 with the root at the origin) -> (mpjpe (n,), mpeepe (n,))."""
        a, b = _f32(pose_a).reshape(-1, 88), _f32(pose_b).reshape(-1, 88)
        assert a.shape == b.shape
        err = np.empty((a.shape[0], 2), F32)
        _lib.check(self.lib.dp_engine_pose_error_host(self.h, a.shape[0], _ptr(a), _ptr(b), _ptr(err)))
        return err[:, 0], err[:, 1]

    def predict_targets(self, window):
        _lib.check(self.lib.dp_engine_predict_targets(self.h, int(window), None))
        return self.state(window)["target_buf"]

    # ------------------------------------------------------------------ frames
    def _trackers(self, joints, weights, n_ee, B, E):
        joints, weights = _i32(joints), _f32(weights)
        shared = int(joints.ndim == 1)
        if shared:
            assert joints.shape == (E,) and weights.shape == (E, 2)
        else:
            assert joints.shape == (B, E) and weights.shape == (B, E, 2)
        ne = None if n_ee is None else _i32(n_ee).reshape(B)
        return joints, weights, shared, ne

    def run_frames(self, target_ee_pos, target_ee_rot, mask_joints, weights_joints, n_ee=None, out=None, **opts):
        """T consecutive frames from HOST arrays in one call: target_ee_pos (T,B,E,3), target_ee_rot (T,B,E,3,3),
        mask_joints (E,) / weights_joints (E,2) shared by every clip and frame or (T,B,E) / (T,B,E,2), n_ee (T,B) or None
        -> poses (T,B,88), global_pos (T,B,3).  Same results as T calls of run(); the staging and host<->device copies of
        neighbouring frames overlap the kernels (dp_engine_run_frames_host).  `out` = (poses, global_pos) float32 C-contiguous
        arrays to write into (a long-running caller reuses them; fresh numpy pages cost a page fault per 4 KB)."""
        B = self.n_clips
        tp = _f32(target_ee_pos)
        T = tp.shape[0]
        tp = tp.reshape(T, B, -1, 3)
        E = tp.shape[2]
        tr = _f32(target_ee_rot).reshape(T, B, E, 9)
        joints, weights = _i32(mask_joints), _f32(weights_joints)
        shared = int(joints.ndim == 1)
        if shared:
            assert joints.shape == (E,) and weights.shape == (E, 2)
        else:
            assert joints.shape == (T, B, E) and weights.shape == (T, B, E, 2)
        ne = None if n_ee is None else _i32(n_ee).reshape(T, B)
        p = opts["options"].c if "options" in opts else RunOptions(**opts).c
        if out is None:
            pose, gpos = np.empty((T, B, 88), F32), np.empty((T, B, 3), F32)
        else:
            pose, gpos = out
            assert pose.dtype == F32 and gpos.dtype == F32 and pose.flags.c_contiguous and gpos.flags.c_contiguous
            assert pose.shape == (T, B, 88) and gpos.shape == (T, B, 3)
        _lib.check(self.lib.dp_engine_run_frames_host(self.h, C.byref(p), T, _ptr(ne), _ptr(joints), _ptr(weights), shared,
                                                      _ptr(tp), _ptr(tr), E, _ptr(pose), _ptr(gpos)))
        return pose, gpos

    def run(self, target_ee_pos, target_ee_rot, mask_joints, weights_joints, n_ee=None, **opts):
        """HOST buffers in, host arrays out (copies + one sync inside the call).
        target_ee_pos (B,E,3), target_ee_rot (B,E,3,3), mask_joints (E,) or (B,E),
        weights_joints (E,2) or (B,E,2) -> pose (B,88), global_pos (B,3)."""
        B = self.n_clips
        tp = _f32(target_ee_pos).reshape(B, -1, 3)
        E = tp.shape[1]
        tr = _f32(target_ee_rot).reshape(B, E, 9)
        joints, weights, shared, ne = self._trackers(mask_joints, weights_joints, n_ee, B, E)
        p = opts["options"].c if "options" in opts else RunOptions(**opts).c
        pose, gpos = np.empty((B, 88), F32), np.empty((B, 3), F32)
        _lib.check(self.lib.dp_engine_run_frame_host(self.h, C.byref(p), _ptr(ne), _ptr(joints), _ptr(weights), shared,
                                                     _ptr(tp), _ptr(tr), E, _ptr(pose), _ptr(gpos)))
        return pose, gpos

    def run_frames_device(self, n_frames, tgt_pos, tgt_rot, joints, weights, out_pose, out_gpos, n_ee=None, shared=True,
                          ee_stride=None, stream=None, options: RunOptions = None):
        """DEVICE-resident torch tensors (float32 / int32, contiguous); enqueues
        n_frames frames on `stream` (an int cudaStream_t or None) without synchronising.  out_gpos=None: out_pose is a packed
        (n_frames, B, 92) tensor of result rows [pose 88 | global_pos 3 | pad] (the wire layout of dist.gather_frames)."""
        dp = lambda t: None if t is None else C.c_void_p(t.data_ptr())
        E = int(ee_stride if ee_stride is not None else tgt_pos.shape[-2])
        _lib.check(self.lib.dp_engine_run_frames_device(
            self.h, C.byref(options.c), int(n_frames), dp(n_ee), dp(joints), dp(weights), int(bool(shared)), dp(tgt_pos),
            dp(tgt_rot), E, dp(out_pose), dp(out_gpos), None if stream is None else C.c_void_p(stream)))

    def frame_stats(self):
        B = self.n_clips
        iters, losses = np.empty(B, np.int32), np.empty((B, 3), F32)
        _lib.check(self.lib.dp_engine_get_frame_stats(self.h, _ptr(iters), _ptr(losses)))
        return iters, losses

    def enable_trace(self, on=True):
        _lib.check(self.lib.dp_engine_enable_trace(self.h, int(on)))

    def trace(self, max_iter):
        rows = np.empty((self.n_clips, max_iter, 52), F32)
        _lib.check(self.lib.dp_engine_get_trace(self.h, _ptr(rows), int(max_iter)))
        return dict(latent=rows[..., :24], grad=rows[..., 24:48], loss=rows[..., 48:51], active=rows[..., 51] > 0)

    def eval_gradient(self, latents, global_rot, tgt_latent, tgt_pos, tgt_rot, joints, weights, n_ee=None, lambda_rot=1.0,
                      lambda_temporal=1.0, decoder_path=0, extension_losses=0, floor_level=0.0, global_pos=None):
        """Teacher-forced loss + d(loss)/d(latent) at given latents; no state change."""
        z = _f32(latents).reshape(-1, 24)
        n = z.shape[0]
        g, t = _f32(global_rot).reshape(n, 4), _f32(tgt_latent).reshape(n, 24)
        tp = _f32(tgt_pos).reshape(n, -1, 3)
        E = tp.shape[1]
        tr = _f32(tgt_rot).reshape(n, E, 9)
        joints, weights, shared, ne = self._trackers(joints, weights, n_ee, n, E)
        grad, losses, pos = np.empty((n, 24), F32), np.empty((n, 3), F32), np.empty((n, 22, 3), F32)
        gp = None if global_pos is None else _f32(global_pos).reshape(n, 3)
        _lib.check(self.lib.dp_engine_eval_gradient(self.h, n, _ptr(z), _ptr(g), _ptr(t), _ptr(ne), _ptr(joints), _ptr(weights),
                                                    shared, _ptr(tp), _ptr(tr), E, float(lambda_rot), float(lambda_temporal),
                                                    int(decoder_path), _ptr(grad), _ptr(losses), _ptr(pos), int(extension_losses),
                                                    float(floor_level), _ptr(gp)))
        return dict(grad=grad, lp=losses[:, 0], lr=losses[:, 1], lt=losses[:, 2], pos=pos)

    def last_decoder_path(self):
        """1 = fp32 CUDA-core frame kernel, 3 = tcgen05 (fp16x2) frame kernel."""
        return int(self.lib.dp_engine_last_decoder_path(self.h))

    def set_predictor_path(self, path):
        """0 = tcgen05 fp16x2 attention + feed-forward (default), 1 = fp32 CUDA-core kernels (cross-check)."""
        _lib.check(self.lib.dp_engine_set_predictor_path(self.h, int(path)))

    def set_profiling(self, on=True):
        _lib.check(self.lib.dp_engine_set_profiling(self.h, int(on)))

    def phase_cycles(self):
        """Phase clock of CTA 0 of the tcgen05 frame kernel since set_profiling(2): cycles in [decoder forward, scaling + barrier,
        decoder backward, Adam, kinematics pass, 0, 0, 0] (include/dp_engine.h)."""
        out = (C.c_ulonglong * 8)()
        _lib.check(self.lib.dp_engine_get_phase_cycles(self.h, out))
        return [int(v) for v in out]

    def timeline(self):
        """Stamps (device clock) of the two clip groups of CTA 0 over iterations 40..43 of the last frame run under set_profiling(2):
        array [group][iteration][loop top, forward, kinematics, barrier, two backward layers, last layer + Adam] (include/dp_engine.h)."""
        out = (C.c_ulonglong * 48)()
        _lib.check(self.lib.dp_engine_get_timeline(self.h, out))
        return np.array(list(out), dtype=np.int64).reshape(2, 4, 6)

    def profile(self):
        """(ms in the temporal predictor, ms in the frame kernel, frames) since set_profiling(True)."""
        a, b, n = C.c_double(0), C.c_double(0), C.c_longlong(0)
        _lib.check(self.lib.dp_engine_get_profile(self.h, C.byref(a), C.byref(b), C.byref(n)))
        return a.value, b.value, n.value

    def launch_count(self):
        return int(self.lib.dp_engine_launch_count(self.h))
