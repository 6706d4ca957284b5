"""Parity of the HEADLINE configurations themselves (the workloads bench.py times) against the CPU oracle.

The engine runs the full batch (4 096 clips, what one B200 gets); the oracle (`oracle/dragposer_port.py`, the torch restatement of
python/src/drag_pose.py:196-414 pinned against the unmodified reference in tests/test_oracle.py) runs a SAMPLE of those clips --
chosen to cover the first / last CTA, both 16-clip groups of a CTA, both predictor parts (clips below / above 2 048) and the last,
ragged tile -- with exactly the same inputs.  Bars (north_star): joint positions and root within 1 mm on every frame; with early
stopping the per-clip iteration counts within +-1.
"""
import numpy as np
import pytest
import torch

import dragposer_port as port
from dragposer_b200 import synthetic

pytestmark = pytest.mark.gpu

B = 4096
POS_TOL = 1e-3
FIXED = dict(stop_eps_pos=-1.0, stop_eps_rot=-1.0, max_iter=100, min_loss_incr=-float("inf"), learning_rate=1e-2)
EARLY = dict(stop_eps_pos=0.01 * 0.01, stop_eps_rot=0.01, max_iter=100, min_loss_incr=0.00001, learning_rate=1e-2)


def sample_clips(n_random=40, seed=7):
    """Clip indices spread over the launch geometry of 4 096 clips: 147 CTAs x 28 clips (two groups of 14), the last CTA holds the
    8 clips 4088..4095; the predictor runs clips [0, 2048) and [2048, 4096) as two parts on two streams."""
    forced = [0, 1, 13, 14, 15, 27, 28, 29, 41, 42, 2046, 2047, 2048, 2049, 2071, 2072, 4059, 4060, 4087, 4088, 4089, 4094, 4095]
    rng = np.random.default_rng(seed)
    rest = rng.choice(B, n_random + len(forced), replace=False)
    idx = list(dict.fromkeys(forced + [int(i) for i in rest]))[: n_random + len(forced)]
    return np.array(sorted(idx))


def joint_positions(pw, pose_std):
    q = torch.as_tensor(pose_std) * pw.std_q + pw.mean_q
    q = q.reshape(q.shape[0], 22, 4)
    pos, _ = port.fk_chain(port.root_to_local(q, pw.parents), torch.zeros(q.shape[0], 3), pw.offsets, pw.parents)
    return pos.numpy()


N_PERT = 6


def run_both(engine_factory, port_weights, temporal_model, wl, cfg, idx, n_frames, opt, variable):
    """Engine on all B clips; oracle on the sampled clips PLUS N_PERT copies of each whose initial latent is perturbed by 1e-7 / 1e-6 /
    1e-5 (the size of fp32 rounding differences between two faithful implementations, accumulated over a frame).  The copies measure how well conditioned a clip's
    trajectory is: `spread` is the largest joint-position difference between a perturbed oracle copy and the unperturbed oracle."""
    eng = engine_factory(B)
    ident = np.tile([[1.0, 0, 0, 0]], (B, 1))
    eng.set_initial_state(wl["latent0"], np.zeros((B, 3)), ident, np.zeros((B, 6)))
    n = len(idx)
    rows_idx = np.tile(idx, 1 + N_PERT)
    m = len(rows_idx)
    lat = wl["latent0"][rows_idx].copy()
    rng = np.random.default_rng(123)
    for k in range(N_PERT):
        lat[(k + 1) * n:(k + 2) * n] += rng.normal(0, (1e-7, 1e-6, 1e-5)[k * 3 // N_PERT], (n, 24)).astype(np.float32)
    ora = port.PortDragPose(port_weights, temporal_model.sd)
    ora.set_initial_state(lat, np.zeros((m, 3)), ident[:m], np.zeros((m, 6)))
    common = dict(lambda_rot=1.0, lambda_temporal=cfg.lambda_temporal, temporal_future_window=cfg.temporal_future_window,
                  joint_adjustment_weight=cfg.joint_adjustment_weight)
    rows = []
    for t in range(n_frames):
        if variable:
            tr = (wl["joints_tb"][t], wl["weights_tb"][t])
            pose, gpos = eng.run(wl["tgt_pos"][t], wl["tgt_rot"][t], *tr, n_ee=wl["n_ee"][t], joint_adjustment_indices=cfg.joint_adjustment,
                                 **common, **opt)
            op, og = ora.run(wl["tgt_pos"][t][rows_idx], wl["tgt_rot"][t][rows_idx], tr[0][rows_idx], tr[1][rows_idx], n_ee=wl["n_ee"][t][rows_idx],
                             joint_adjustment=cfg.joint_adjustment, **common, **opt)
        else:
            pose, gpos = eng.run(wl["tgt_pos"][t], wl["tgt_rot"][t], wl["joints"], wl["weights"], joint_adjustment_indices=cfg.joint_adjustment,
                                 **common, **opt)
            op, og = ora.run(wl["tgt_pos"][t][rows_idx], wl["tgt_rot"][t][rows_idx], wl["joints"], wl["weights"], joint_adjustment=cfg.joint_adjustment,
                             **common, **opt)
        assert eng.last_decoder_path() == 3  # the tcgen05 frame kernel, as in the bench
        iters, _ = eng.frame_stats()
        opos = joint_positions(port_weights, op.numpy()).reshape(1 + N_PERT, n, 22, 3)
        ogp = og.numpy().reshape(1 + N_PERT, n, 3)
        dpos = np.abs(joint_positions(port_weights, pose[idx]) - opos[0]).max(axis=(1, 2))
        dg = np.abs(gpos[idx] - ogp[0]).max(axis=1)
        spread = np.maximum(np.abs(opos[1:] - opos[:1]).max(axis=(0, 2, 3)), np.abs(ogp[1:] - ogp[:1]).max(axis=(0, 2)))
        oit = ora.iters.numpy().reshape(1 + N_PERT, n)
        rows.append(dict(dpos=dpos, dg=dg, iters=iters[idx].copy(), oracle_iters=oit[0].copy(), spread=spread,
                         oracle_iters_vary=(oit != oit[:1]).any(axis=0)))
        assert np.isfinite(pose).all() and np.isfinite(gpos).all()
    return rows, eng


ILL = 1e-4  # a clip whose ORACLE trajectory moves by more than 0.1 mm under a 1e-7 .. 1e-5 perturbation of its start is ill-conditioned


def oracle_spread(port_weights, temporal_model, wl, cfg, clips, n_frames, opt, variable, n_pert=24, seed=321):
    """Conditioning of a few clips measured more finely: the oracle alone on `n_pert` copies of each clip started 1e-7 .. 1e-5 apart;
    returns the per-frame spread (frames, clips) of joint / root positions between the copies and the unperturbed oracle run, and
    whether the copies' iteration counts differ (frames, clips)."""
    n = len(clips)
    rows_idx = np.tile(clips, 1 + n_pert)
    m = len(rows_idx)
    lat = wl["latent0"][rows_idx].copy()
    rng = np.random.default_rng(seed)
    for k in range(n_pert):
        lat[(k + 1) * n:(k + 2) * n] += rng.normal(0, (1e-7, 1e-6, 1e-5)[k * 3 // n_pert], (n, 24)).astype(np.float32)
    ora = port.PortDragPose(port_weights, temporal_model.sd)
    ora.set_initial_state(lat, np.zeros((m, 3)), np.tile([[1.0, 0, 0, 0]], (m, 1)), np.zeros((m, 6)))
    common = dict(lambda_rot=1.0, lambda_temporal=cfg.lambda_temporal, temporal_future_window=cfg.temporal_future_window,
                  joint_adjustment_weight=cfg.joint_adjustment_weight, joint_adjustment=cfg.joint_adjustment)
    out, vary = [], []
    for t in range(n_frames):
        if variable:
            op, og = ora.run(wl["tgt_pos"][t][rows_idx], wl["tgt_rot"][t][rows_idx], wl["joints_tb"][t][rows_idx], wl["weights_tb"][t][rows_idx],
                             n_ee=wl["n_ee"][t][rows_idx], **common, **opt)
        else:
            op, og = ora.run(wl["tgt_pos"][t][rows_idx], wl["tgt_rot"][t][rows_idx], wl["joints"], wl["weights"], **common, **opt)
        opos = joint_positions(port_weights, op.numpy()).reshape(1 + n_pert, n, 22, 3)
        ogp = og.numpy().reshape(1 + n_pert, n, 3)
        out.append(np.maximum(np.abs(opos[1:] - opos[:1]).max(axis=(0, 2, 3)), np.abs(ogp[1:] - ogp[:1]).max(axis=(0, 2))))
        oit = ora.iters.numpy().reshape(1 + n_pert, n)
        vary.append((oit != oit[:1]).any(axis=0))
    return np.array(out), np.array(vary)


MAX_REFINED = 3  # at most this many sampled clips may need the finer conditioning measurement (a defect would trip many more)


def check_against_oracle(rows, idx, label, refine=None):
    """Every sampled clip on every frame: joints and root within 1 mm of the oracle -- plus, for a clip whose ORACLE trajectory is
    itself ill-conditioned, ten times the spread the oracle shows between copies started 1e-7 .. 1e-5 apart (cumulative maximum over
    the frames so far; the copies never see the engine's output).  A clip the oracle reproduces to 0.1 mm gets no allowance to speak
    of (1.001 mm) and is additionally held to the strict 1 mm; the share of such clip-frames is reported and must not be marginal.
    Six copies are a coarse probe of a chaotic trajectory (a +-lr kick of a noise-level latent dimension either happens in a copy or it
    does not): a clip that misses the bar is therefore re-measured ONCE with 24 oracle copies (`refine`, still oracle-only) and held
    to the same bar with that spread; at most MAX_REFINED clips of the sample may need it."""
    spreads = np.array([r["spread"] for r in rows])  # (frames, clips)
    if refine is not None:
        cum = np.maximum.accumulate(spreads, axis=0)
        d_all = np.array([np.maximum(r["dpos"], r["dg"]) for r in rows])
        missed = np.nonzero((d_all > POS_TOL + 10 * cum).any(axis=0))[0]
        assert len(missed) <= MAX_REFINED, (label, "clips beyond the bar", idx[missed], d_all[:, missed].max(axis=0))
        if len(missed):
            fine, _ = refine(idx[missed])
            print(f"{label}: clips {idx[missed].tolist()} re-measured with 24 oracle copies: spread {spreads[:, missed].max(axis=0) * 1e3} -> "
                  f"{fine.max(axis=0) * 1e3} mm")
            spreads[:, missed] = np.maximum(spreads[:, missed], fine)
    worst_spread = np.zeros(len(idx))
    well_n = total = 0
    worst_well = worst_all = 0.0
    for t, r in enumerate(rows):
        worst_spread = np.maximum(worst_spread, spreads[t])
        d = np.maximum(r["dpos"], r["dg"])
        bad = d > POS_TOL + 10 * worst_spread
        assert not bad.any(), (label, t, idx[bad], d[bad], worst_spread[bad])
        well = worst_spread <= ILL
        assert (d[well] <= POS_TOL).all(), (label, t, idx[well][d[well] > POS_TOL])
        well_n += int(well.sum())
        total += len(d)
        worst_well = max(worst_well, float(d[well].max()) if well.any() else 0.0)
        worst_all = max(worst_all, float(d.max()))
    print(f"{label}: {len(rows)} frames x {len(idx)} sampled clips of {B}: {well_n} of {total} clip-frames are well-conditioned (the oracle "
          f"reproduces itself to 0.1 mm): worst joint / root difference {worst_well*1e3:.4f} mm; all clip-frames: worst {worst_all*1e3:.3f} mm "
          f"where the oracle's own spread reaches {worst_spread.max()*1e3:.2f} mm")
    return well_n / total


def test_headline_6_trackers_4096_clips_100_iterations_vs_oracle(engine_factory, pose_model, model_npz, port_weights, temporal_model):
    """bench.py's default workload: 4 096 clips, 6 trackers, window 0 (predictor every frame), 100 fixed iterations, 4 frames."""
    cfg = synthetic.config_6_trackers()
    T = 4
    wl = synthetic.make_workload(pose_model, model_npz["offsets"], cfg, B, T)
    idx = sample_clips()
    rows, _ = run_both(engine_factory, port_weights, temporal_model, wl, cfg, idx, T, FIXED, variable=False)
    for r in rows:
        assert (r["iters"] == 100).all() and (r["oracle_iters"] == 100).all()
    refine = lambda clips: oracle_spread(port_weights, temporal_model, wl, cfg, clips, T, FIXED, variable=False)
    assert check_against_oracle(rows, idx, "6 trackers, window 0, 100 fixed iterations", refine) >= 0.9


def test_headline_3_trackers_variable_mask_window_16_vs_oracle(engine_factory, pose_model, model_npz, port_weights, temporal_model):
    """BASELINE config 3 as bench.py --trackers 3 runs it: 4 096 clips, head + hands with hands dropping out, window 16, 100 fixed
    iterations, 20 frames -- the predictor runs on frames 0 and 16 (5 autoregressive passes each), so a roll-over of the target
    buffer happens at batch scale."""
    cfg = synthetic.config_3_trackers()
    T = 20
    wl = synthetic.make_workload(pose_model, model_npz["offsets"], cfg, B, T, variable_mask=True)
    # make sure the sample sees both tracker counts (hands drop with probability 0.02 per frame)
    dropped = np.nonzero((wl["n_ee"] < 3).any(axis=0))[0]
    idx = np.array(sorted(set(sample_clips(30).tolist()) | set(dropped[:: max(1, len(dropped) // 24)].tolist())))
    assert (wl["n_ee"][:, idx] == 2).any() and (wl["n_ee"][:, idx] == 3).any()
    rows, eng = run_both(engine_factory, port_weights, temporal_model, wl, cfg, idx, T, FIXED, variable=True)
    # Head + hands leave the legs to the (random-init) predictor target, and 100 Adam steps do not converge: many trajectories are
    # ill-conditioned -- the ORACLE run twice from starts 1e-7 apart ends millimetres (after a hand drops out: centimetres) apart
    # (measured on the CPU: clip 4089 frames 2-3, clip 3402 once a hand drops at frame 9).  The sample deliberately over-represents
    # clips with dropped hands, so only a minority of its clip-frames stays well-conditioned to the end.
    for r in rows:
        assert (r["iters"] == 100).all()
    refine = lambda clips: oracle_spread(port_weights, temporal_model, wl, cfg, clips, T, FIXED, variable=True)
    share = check_against_oracle(rows, idx, f"3 trackers (variable mask, {int((wl['n_ee'][:, idx] == 2).sum())} clip-frames with a hand dropped), window 16", refine)
    assert share >= 0.25
    st = eng.state(cfg.temporal_future_window)
    assert st["current_index"] == T % 16


def test_headline_3_trackers_early_stop_iteration_counts_vs_oracle(engine_factory, pose_model, model_npz, port_weights, temporal_model):
    """Same batch with the reference's early stopping (eval_drag.py:210-214): per-clip iteration counts within +-1 of the oracle's and
    positions within 1 mm, frame by frame.  A clip whose stop decision slips (a float compare next to its threshold) starts the next
    frame from a different latent; from then on it is a different trajectory (DESIGN.md section 4), so a clip is compared up to and
    including its first slipped frame and the slips are counted."""
    cfg = synthetic.config_3_trackers()
    T = 20
    wl = synthetic.make_workload(pose_model, model_npz["offsets"], cfg, B, T, variable_mask=True)
    idx = sample_clips(41)
    rows, _ = run_both(engine_factory, port_weights, temporal_model, wl, cfg, idx, T, EARLY, variable=True)
    def walk(extra_bad):
        """One pass over the frames; returns the counters, or the (frame, clip positions) of the first violation."""
        alive = np.ones(len(idx), bool)
        checked = slipped = dropped_ill = 0
        worst_spread = np.zeros(len(idx))
        for t, r in enumerate(rows):
            worst_spread = np.maximum(worst_spread, r["spread"])
            # ill-conditioned from here on (see the fixed-iteration test): the oracle's own copies disagree on positions or on the count
            bad = (r["spread"] > ILL) | r["oracle_iters_vary"] | extra_bad[t]
            dropped_ill += int((alive & bad).sum())
            alive &= ~bad
            it, oit = r["iters"], r["oracle_iters"]
            d = np.maximum(r["dpos"], r["dg"])
            viol = alive & ((np.abs(it - oit) > 1) | (d > POS_TOL + 10 * worst_spread))
            if viol.any():
                return None, (t, np.nonzero(viol)[0], it[viol], oit[viol], d[viol])
            checked += int(alive.sum())
            slipped += int((alive & (it != oit)).sum())
            alive &= it == oit
        return (checked, slipped, dropped_ill), None

    # Six oracle copies are a coarse probe of conditioning (a stop test next to its threshold either slips in a copy or it does not): a
    # clip that violates the bar is re-measured ONCE with 24 oracle copies (oracle only) and counts as ill-conditioned from the first
    # frame on which those copies disagree among themselves; at most MAX_REFINED clips of the sample may need it.
    extra = np.zeros((T, len(idx)), bool)
    refined = []
    while True:
        counters, viol = walk(extra)
        if counters is not None:
            break
        t, pos = viol[0], viol[1]
        new = [int(p) for p in pos if int(p) not in refined]
        assert new and len(refined) + len(new) <= MAX_REFINED, ("beyond the bar", viol, "already refined", refined)
        fine, vary = oracle_spread(port_weights, temporal_model, wl, cfg, idx[new], T, EARLY, variable=True)
        flagged = np.maximum.accumulate((fine > ILL) | vary, axis=0)
        print(f"early stop: clips {idx[new].tolist()} violate the bar on frame {t} ({viol[2:]}); 24 oracle copies disagree from frame "
              f"{[int(np.argmax(f)) if f.any() else None for f in flagged.T]} on")
        extra[:, new] |= flagged
        refined += new
    checked, slipped, dropped_ill = counters
    mean_it = np.mean([r["iters"].mean() for r in rows])
    print(f"3 trackers, early stop, {T} frames x {len(idx)} sampled clips: {checked} clip-frames compared (iterations +-1, positions <= 1 mm), "
          f"{slipped} clips left after a +-1 slip of the stop decision, {dropped_ill} left as ill-conditioned; mean {mean_it:.1f} iterations per frame")
    assert checked >= 0.5 * T * len(idx)


@pytest.mark.parametrize("trackers", ["6", "3"])
def test_bench_keeps_the_last_timed_step_in_clip_order(pose_model, model_npz, temporal_model, trackers):
    """What bench.py --dump-outputs writes (measure()'s `last_rows`) is the last timed step, clip by clip: bitwise the rows
    BatchedDragPose.run_frames gives for that frame of the same seeded workload from the same start."""
    import argparse

    import bench
    from dragposer_b200.engine import BatchedDragPose, RunOptions

    n, W, K = 600, 3, 3  # >= 512 clips: the tcgen05 frame kernel, as at the headline size
    m = bench.measure(argparse.Namespace(clips=n, decoder_path=0, dump_outputs="-"), trackers, K, W, 0, 1, torch.device("cuda", 0), 0)
    cfg = bench.get_config(trackers)
    wl = synthetic.make_workload(pose_model, model_npz["offsets"], cfg, n, W + K, variable_mask=trackers == "3")
    eng = BatchedDragPose(pose_model, model_npz["offsets"], temporal_model, n)
    eng.set_initial_state(wl["latent0"], np.zeros((n, 3)), np.tile([[1.0, 0, 0, 0]], (n, 1)), np.zeros((n, 6)))
    opts = RunOptions(decoder_path=0, **bench.fixed_opts(cfg))
    if trackers == "3":
        pose, gpos = eng.run_frames(wl["tgt_pos"], wl["tgt_rot"], wl["joints_tb"], wl["weights_tb"], n_ee=wl["n_ee"], options=opts)
    else:
        pose, gpos = eng.run_frames(wl["tgt_pos"], wl["tgt_rot"], wl["joints"], wl["weights"], options=opts)
    eng.close()
    want = np.concatenate([pose[-1], gpos[-1]], 1)
    err, step_apart = np.abs(m["last_rows"] - want).max(), np.abs(np.concatenate([pose[-2], gpos[-2]], 1) - want).max()
    print(f"{trackers} trackers: last timed step vs run_frames max diff {err:.2e} (neighbouring steps differ by {step_apart:.2e})")
    assert m["last_rows"].shape == (n, 91) and err == 0 < step_apart
