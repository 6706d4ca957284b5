"""GPU: per-clip optimiser settings (dp_engine_set_clip_settings / BatchedDragPose.set_clip_options).  A batch whose clips run with
different settings is checked bit for bit against one engine per setting that holds exactly that setting's clips and runs it as
plain dp_run_params, on both frame kernels."""
import numpy as np
import pytest

from dragposer_b200 import synthetic
from dragposer_b200._lib import EngineError
from dragposer_b200.engine import ClipOptions, RunOptions

pytestmark = pytest.mark.gpu
INF = float("inf")

# Between them the four settings vary every per-clip field: a fixed-iteration one, early-stopping ones with smaller and larger
# budgets, three learning rates and loss weights, joint adjustment off and on with two (joint, slot, weight) triples.
SETTINGS = [
    dict(stop_eps_pos=-1.0, stop_eps_rot=-1.0, min_loss_incr=-INF, max_iter=12, learning_rate=1e-2, lambda_rot=1.0,
         lambda_temporal=0.02, joint_adjustment_indices=None),
    dict(stop_eps_pos=1e-4, stop_eps_rot=1e-2, min_loss_incr=1e-5, max_iter=6, learning_rate=5e-3, lambda_rot=0.5,
         lambda_temporal=0.15, joint_adjustment_indices=(0, 0), joint_adjustment_weight=1.0),
    dict(stop_eps_pos=1e-3, stop_eps_rot=3e-2, min_loss_incr=1e-6, max_iter=20, learning_rate=2e-2, lambda_rot=2.0,
         lambda_temporal=0.5, joint_adjustment_indices=(13, 3), joint_adjustment_weight=0.1),
    dict(stop_eps_pos=1e-4, stop_eps_rot=1e-3, min_loss_incr=1e-6, max_iter=9, learning_rate=1e-3, lambda_rot=1.0,
         lambda_temporal=0.02, joint_adjustment_indices=None),
]


def _need(s):
    """Trackers a clip must have on for its joint-adjustment slot."""
    ja = s.get("joint_adjustment_indices")
    return 1 if ja is None else ja[1] + 1


def _workload(pose_model, model_npz, n, frames, which, seed, settings=SETTINGS):
    """6 trackers with per-clip weights and a per-frame, per-clip number of active trackers that covers each clip's slot."""
    cfg = synthetic.config_6_trackers()
    wl = synthetic.make_workload(pose_model, model_npz["offsets"], cfg, n, frames, first_clip=seed)
    rng = np.random.default_rng(seed)
    E = len(cfg.joints)
    joints = np.tile(np.asarray(cfg.joints, np.int32), (n, 1))
    weights = (cfg.tracker_weights[None] * rng.uniform(0.5, 2.0, (n, 1, 1))).astype(np.float32)
    lo = np.array([max(2, _need(settings[s])) for s in which])
    n_ee = rng.integers(lo[None, :], E + 1, (frames, n)).astype(np.int32)
    return dict(latent0=wl["latent0"], tp=wl["tgt_pos"], tr=wl["tgt_rot"], joints=joints, weights=weights, n_ee=n_ee)


def _engine(engine_factory, n):
    e = engine_factory(n)
    e.set_predictor_path(1)  # fp32 predictor: its targets do not depend on which other clips share the call
    return e


def _start(n):
    return np.zeros((n, 3), np.float32), np.tile(np.float32([[1, 0, 0, 0]]), (n, 1)), np.zeros((n, 6), np.float32)


def _frames(eng, wl, rows, frames, kw, stats=True):
    """Frames `frames` of the clips `rows` of the workload -> poses, gpos, iters, losses stacked over the frames."""
    out = [[], [], [], []]
    for t in frames:
        p, g = eng.run(wl["tp"][t][rows], wl["tr"][t][rows], wl["joints"][rows], wl["weights"][rows], n_ee=wl["n_ee"][t][rows], **kw)
        it, ls = eng.frame_stats() if stats else (None, None)
        for o, v in zip(out, (p, g, it, ls)):
            o.append(v)
    return [np.stack(o) for o in out] if stats else [np.stack(o) for o in out[:2]]


STATE_KEYS = ("latent", "global_pos", "global_rot", "latent_buf", "disp_buf", "height_buf", "target_buf")


def _mixed_vs_uniform(engine_factory, wl, which, window, path, frames, batch_kw=None, settings=SETTINGS):
    n = len(which)
    rows = np.arange(n)
    kw = dict(temporal_future_window=window, decoder_path=path, **(batch_kw or {}))
    mixed = _engine(engine_factory, n)
    mixed.set_initial_state(wl["latent0"], *_start(n))
    mixed.set_clip_options([ClipOptions(**s) for s in settings], which)
    # the per-clip keywords of the frame call are not read while the table is set
    out = _frames(mixed, wl, rows, range(frames), dict(kw, max_iter=1, learning_rate=1.0, lambda_rot=9.0))
    st = mixed.state(window)
    assert mixed.last_decoder_path() == path
    for s, setting in enumerate(settings):
        ids = np.flatnonzero(which == s)
        assert len(ids) > 0
        uni = _engine(engine_factory, len(ids))
        uni.set_initial_state(wl["latent0"][ids], *_start(len(ids)))
        ref = _frames(uni, wl, ids, range(frames), dict(kw, **setting))
        for a, b in zip(out, ref):
            assert np.array_equal(a[:, ids], b), s
        su = uni.state(window)
        for k in STATE_KEYS:
            assert np.array_equal(st[k][ids], su[k]), (s, k)
        assert (out[2][:, ids] <= setting["max_iter"]).all()
        uni.close()
    return out


@pytest.mark.parametrize("window", [0, 16])
@pytest.mark.parametrize("path,n", [(3, 576), (3, 40), (1, 1200), (1, 40)], ids=["tcgen05-576", "tcgen05-40", "fp32-1200", "fp32-40"])
def test_mixed_batch_is_bitwise_the_uniform_batches(engine_factory, pose_model, model_npz, window, path, n):
    """Clips assigned to four settings in a shuffled pattern, variable n_ee and per-clip trackers, frames across predictor calls:
    each clip's poses, positions, iteration counts, losses and carried state are bitwise those of a batch of only its setting's
    clips run with that setting as plain dp_run_params on the same kernel.  At 1 200 clips the fp32 kernel runs two clips per warp."""
    which = np.random.default_rng(n + window).permutation(np.arange(n) % len(SETTINGS)).astype(np.int32)
    wl = _workload(pose_model, model_npz, n, 20, which, 100 + window)
    out = _mixed_vs_uniform(engine_factory, wl, which, window, path, 20)
    assert len(np.unique(out[2])) > 3  # the early-stopping settings stop at different counts


def test_mixed_batch_with_extension_losses(engine_factory, pose_model, model_npz):
    """fp32 kernel with every extension loss on: the mixed batch is bitwise the uniform batches."""
    n = 24
    which = np.random.default_rng(5).permutation(np.arange(n) % len(SETTINGS)).astype(np.int32)
    wl = _workload(pose_model, model_npz, n, 8, which, 300)
    _mixed_vs_uniform(engine_factory, wl, which, 16, 1, 8, dict(extension_losses=15, floor_level=-0.05))


def test_all_fixed_iteration_table(engine_factory, pose_model, model_npz):
    """Every setting in use runs a fixed number of iterations, with budgets that split the clip pairs of the tcgen05 kernel's warps:
    the launch skips the loss sums except at each clip's last iteration, and the result is bitwise the uniform batches."""
    fixed = [dict(SETTINGS[0], max_iter=m, learning_rate=lr, lambda_rot=lrot, joint_adjustment_indices=ja)
             for m, lr, lrot, ja in ((12, 1e-2, 1.0, None), (5, 5e-3, 0.5, (0, 0)), (17, 2e-2, 2.0, (13, 3)), (1, 1e-3, 1.0, None))]
    n = 600
    which = np.random.default_rng(7).permutation(np.arange(n) % len(fixed)).astype(np.int32)
    wl = _workload(pose_model, model_npz, n, 6, which, 800, fixed)
    out = _mixed_vs_uniform(engine_factory, wl, which, 16, 3, 6, settings=fixed)
    for s, f in enumerate(fixed):
        assert (out[2][:, which == s] == f["max_iter"]).all()


@pytest.mark.parametrize("path,n", [(3, 520), (1, 16)], ids=["tcgen05", "fp32"])
def test_one_entry_table_is_the_plain_run(engine_factory, pose_model, model_npz, path, n):
    setting = SETTINGS[2]
    which = np.full(n, 2, np.int32)
    wl = _workload(pose_model, model_npz, n, 6, which, 400)
    kw = dict(temporal_future_window=16, decoder_path=path)
    rows = np.arange(n)
    outs, states = [], []
    for table in (False, True):
        eng = _engine(engine_factory, n)
        eng.set_initial_state(wl["latent0"], *_start(n))
        if table:
            eng.set_clip_options([ClipOptions(**setting)])
        outs.append(_frames(eng, wl, rows, range(6), dict(kw, **setting)))
        states.append(eng.state(16))
        eng.close()
    for a, b in zip(*outs):
        assert np.array_equal(a, b)
    for k in STATE_KEYS:
        assert np.array_equal(states[0][k], states[1][k]), k


@pytest.mark.parametrize("path", [1, 3], ids=["fp32", "tcgen05"])
def test_trace_and_iteration_counts_follow_each_clips_max_iter(engine_factory, pose_model, model_npz, path):
    n = 32
    which = (np.arange(n) % len(SETTINGS)).astype(np.int32)
    wl = _workload(pose_model, model_npz, n, 3, which, 500)
    eng = _engine(engine_factory, n)
    eng.set_initial_state(wl["latent0"], *_start(n))
    eng.set_clip_options([ClipOptions(**s) for s in SETTINGS], which)
    eng.enable_trace(True)
    top = max(s["max_iter"] for s in SETTINGS)
    cap = np.array([SETTINGS[s]["max_iter"] for s in which])
    for t in range(3):
        eng.run(wl["tp"][t], wl["tr"][t], wl["joints"], wl["weights"], n_ee=wl["n_ee"][t], temporal_future_window=16, decoder_path=path)
        iters, _ = eng.frame_stats()
        assert (iters >= 1).all() and (iters <= cap).all()
        assert (iters[which == 0] == SETTINGS[0]["max_iter"]).all()  # the fixed-iteration setting runs its whole budget
        active = eng.trace(top)["active"]
        for c in range(n):
            assert active[c, : iters[c]].all() and not active[c, iters[c]:].any(), c


@pytest.mark.parametrize("path", [1, 3], ids=["fp32", "tcgen05"])
def test_restarted_rows_take_a_new_setting_and_init_clears_the_table(engine_factory, pose_model, model_npz, path):
    """Restart rows mid-window and give them another setting: from their restart on they are bitwise a fresh engine with that
    setting, the other rows bitwise the run without the restart.  set_initial_state then clears the table."""
    n, frames, f = 24, 14, 5
    which = (np.arange(n) % 3).astype(np.int32)  # settings 0..2; the restarted rows move to setting 3
    wl = _workload(pose_model, model_npz, n, frames, which, 600)
    wl["n_ee"][:] = 6
    restarted = np.array([2, 7, 8, 19])
    new = synthetic.make_workload(pose_model, model_npz["offsets"], synthetic.config_6_trackers(), len(restarted), 1, first_clip=77)
    kw = dict(temporal_future_window=16, decoder_path=path)
    opts = [ClipOptions(**s) for s in SETTINGS]
    rows = np.arange(n)

    eng = _engine(engine_factory, n)
    eng.set_initial_state(wl["latent0"], *_start(n))
    eng.set_clip_options(opts, which)
    a = _frames(eng, wl, rows, range(f), kw)
    eng.restart_clips(restarted, new["latent0"], *_start(len(restarted)))
    which2 = which.copy()
    which2[restarted] = 3
    eng.set_clip_options(opts, which2)
    b = _frames(eng, wl, rows, range(f, frames), kw)
    out = [np.concatenate(x) for x in zip(a, b)]

    ref = _engine(engine_factory, n)
    ref.set_initial_state(wl["latent0"], *_start(n))
    ref.set_clip_options(opts, which)
    base = _frames(ref, wl, rows, range(frames), kw)
    keep = np.setdiff1d(rows, restarted)
    for x, y in zip(out, base):
        assert np.array_equal(x[:, keep], y[:, keep])

    fresh = _engine(engine_factory, len(restarted))
    fresh.set_initial_state(new["latent0"], *_start(len(restarted)))
    one = _frames(fresh, wl, restarted, range(f, frames), dict(kw, **SETTINGS[3]))
    for x, y in zip(out, one):
        assert np.array_equal(x[f:, restarted], y)
    st, sf = eng.state(16), fresh.state(16)
    for k in STATE_KEYS:
        assert np.array_equal(st[k][restarted], sf[k]), k

    # set_initial_state clears the table: the next frames read dp_run_params again
    plain = _engine(engine_factory, n)
    for e in (eng, plain):
        e.set_initial_state(wl["latent0"], *_start(n))
    x = _frames(eng, wl, rows, range(3), dict(kw, **SETTINGS[1]))
    y = _frames(plain, wl, rows, range(3), dict(kw, **SETTINGS[1]))
    for u, v in zip(x, y):
        assert np.array_equal(u, v)


def test_refused_calls_leave_the_engine_unchanged(engine_factory, pose_model, model_npz):
    n, frames = 16, 5
    which = (np.arange(n) % len(SETTINGS)).astype(np.int32)
    wl = _workload(pose_model, model_npz, n, frames, which, 700)
    kw = dict(temporal_future_window=16, decoder_path=3)
    opts = [ClipOptions(**s) for s in SETTINGS]
    rows = np.arange(n)
    engines = []
    for refused in (True, False):
        eng = _engine(engine_factory, n)
        eng.set_initial_state(wl["latent0"], *_start(n))
        eng.set_clip_options(opts, which)
        first = _frames(eng, wl, rows, range(1), kw)
        if refused:
            bad = which.copy()
            bad[3] = len(opts)
            with pytest.raises(EngineError, match="error -1"):  # an index out of range
                eng.set_clip_options(opts, bad)
            bad[3] = -1
            with pytest.raises(EngineError, match="error -1"):
                eng.set_clip_options(opts, bad)
            with pytest.raises(EngineError, match="error -1"):  # more settings than DP_MAX_CLIP_SETTINGS
                eng.set_clip_options(opts * 9, which)
            with pytest.raises(EngineError, match="error -1"):  # max_iter 0
                eng.set_clip_options(opts[:3] + [ClipOptions(**dict(SETTINGS[3], max_iter=0))], which)
            # clip 2 (setting 2: joint adjustment at slot 3) with only three trackers on
            n_ee = wl["n_ee"][1].copy()
            n_ee[2] = 3
            with pytest.raises(EngineError, match="error -1"):
                eng.run(wl["tp"][1], wl["tr"][1], wl["joints"], wl["weights"], n_ee=n_ee, **kw)
            # three tracker slots per clip: setting 2's slot 3 is beyond them
            with pytest.raises(EngineError, match="error -1"):
                eng.run(wl["tp"][1][:, :3], wl["tr"][1][:, :3], wl["joints"][:, :3], wl["weights"][:, :3], **kw)
        rest = _frames(eng, wl, rows, range(1, frames), kw)
        engines.append((first, rest, eng.state(16)))
    (f0, r0, s0), (f1, r1, s1) = engines
    for x, y in zip(f0 + r0, f1 + r1):
        assert np.array_equal(x, y)
    for k in STATE_KEYS:
        assert np.array_equal(s0[k], s1[k]), k
