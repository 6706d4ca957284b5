"""GPU: the engine's temporal predictor, and the bookkeeping that decides which predicted row each frame reads, against a float64
predictor (oracle/dragposer_port.predict_targets in float64, see tests/test_host_predictor_float64.py).

Bar: differences in standardised units (divided by stds_latent) <= 4 e32 + 2e-6, where e32 is the fp32 port's own max error against
float64 on the same clips, model and window.  The rows checked are every row a frame can read (0..W-1; row 0 at window 0).

- predict_targets at every window 0..116, both predictor paths (tcgen05 fp16x2 and fp32 CUDA cores), 1 / 37 / 300 clips every clip,
  2 101 (two parts) and 8 200 clips (no hidden split) on sampled clips;
- four stress models (peaked attention, LayerNorm gains and biases far from 1 and 0, larger feed-forward activations, small latent
  stds) through their own engines;
- teacher-forced frames: before every frame the test reads the rings, the latent and clip_index back, keeps its own copy of the
  reference's target buffer and current_index per clip (drag_pose.py:237-244,399-402: predictor at index 0, a fresh zero buffer
  with the index kept when the window changes, index -> (index + 1) % W), and after the frame checks the index, the row the
  engine holds for that frame, and that the frame kernel's temporal loss is the one of that row."""
import time

import numpy as np
import pytest
import torch

from dragposer_b200 import synthetic
from dragposer_b200.engine import BatchedDragPose
from test_host_predictor_float64 import BAR_FLOOR, WINDOWS, Oracle, predict, readable_rows, stress_model, tiled_rings

pytestmark = pytest.mark.gpu

LOOP = dict(stop_eps_pos=0.01 * 0.01, stop_eps_rot=0.01, max_iter=1, min_loss_incr=0.00001, learning_rate=1e-2, lambda_rot=1,
            lambda_temporal=1.0)
LT_REL = 1e-4


@pytest.fixture(scope="module", autouse=True)
def _report_runtime():
    t0 = time.perf_counter()
    yield
    print(f"\n{__name__}: {time.perf_counter() - t0:.1f} s including the CPU oracle")


def _engine(pose_model, model_npz, tm, max_clips):
    return BatchedDragPose(pose_model, model_npz["offsets"], tm, max_clips)


def _start(eng, n, rings, latent0=None):
    z = np.zeros((n, 24), np.float32) if latent0 is None else latent0
    eng.set_initial_state(z, np.zeros((n, 3)), np.tile([[1.0, 0, 0, 0]], (n, 1)), np.zeros((n, 6)))
    eng.set_ring_buffers(*rings)


def sample_clips(n, seed=0):
    """80 clips: the first and last 16, 16 on each side of the two-part boundary, and 16 others."""
    per = (n + 1) // 2
    edges = np.concatenate([np.arange(16), np.arange(per - 16, per + 16), np.arange(n - 16, n)])
    rest = np.setdiff1d(np.arange(n), edges)
    return np.unique(np.concatenate([edges, np.random.default_rng(seed).choice(rest, 16, replace=False)]))


def _check_predict_targets(eng, orc, windows, clips=None, label=""):
    worst = {0: 0.0, 1: 0.0}
    for w in windows:
        rows = readable_rows(w)
        want, bar = orc.rows(w), orc.bar(w)
        errs = []
        for path in (0, 1):
            eng.set_predictor_path(path)
            got = eng.predict_targets(w)
            got = got[:, rows] if clips is None else got[clips][:, rows]
            assert np.isfinite(got).all()
            err = float((np.abs(got.astype(np.float64) - want) / orc.std).max())
            errs.append(err)
            worst[path] = max(worst[path], err)
        print(f"{label} window {w:3d}: tensor-core {errs[0]:.2e}, CUDA-core {errs[1]:.2e}, bar {bar:.2e} (e32 {orc.e32(w):.2e})")
        assert max(errs) <= bar, (label, w, errs, bar)
    eng.set_predictor_path(0)
    return worst


# ----------------------------------------------------------------------------- a. predict_targets, every window
@pytest.mark.parametrize("n_clips", [1, 37, 300])
def test_predict_targets_every_window_vs_float64(pose_model, model_npz, temporal_model, n_clips):
    rings = tiled_rings(n_clips, 5)
    orc = Oracle(temporal_model, *rings)
    eng = _engine(pose_model, model_npz, temporal_model, max(512, n_clips))
    try:
        _start(eng, n_clips, rings)
        worst = _check_predict_targets(eng, orc, WINDOWS, label=f"{n_clips} clips")
    finally:
        eng.close()
    print(f"{n_clips} clips, windows 0..116: max err tensor-core {worst[0]:.2e}, CUDA-core {worst[1]:.2e}")


@pytest.mark.parametrize("n_clips", [2101, 8200], ids=["two-parts", "no-hidden-split"])
def test_predict_targets_large_batches_vs_float64(pose_model, model_npz, temporal_model, n_clips):
    """Sampled clips: the first and last tile, both sides of the part boundary, and 16 others."""
    rings = tiled_rings(n_clips, 6)
    clips = sample_clips(n_clips)
    orc = Oracle(temporal_model, *(r[clips] for r in rings))
    eng = _engine(pose_model, model_npz, temporal_model, n_clips)
    try:
        _start(eng, n_clips, rings)
        _check_predict_targets(eng, orc, (0, 16, 116), clips, label=f"{n_clips} clips ({len(clips)} sampled)")
    finally:
        eng.close()


# ----------------------------------------------------------------------------- b. stress models
@pytest.mark.parametrize("kind", ["sharp", "ln", "ff", "stats"])
def test_predict_targets_stress_models_vs_float64(pose_model, model_npz, temporal_model, kind):
    """300 clips, windows 0, 16 and 116, both predictor paths.  A miss on the tensor-core path alone points at the fp16x2 split
    products or the epilogues."""
    rings = tiled_rings(300, 7)
    tm = stress_model(temporal_model, kind, rings)
    orc = Oracle(tm, *rings)
    eng = _engine(pose_model, model_npz, tm, 512)
    try:
        _start(eng, 300, rings)
        _check_predict_targets(eng, orc, (0, 16, 116), label=f"{kind}, 300 clips")
    finally:
        eng.close()


# ----------------------------------------------------------------------------- c. teacher-forced frames
class ReferenceBookkeeping:
    """The reference's per-clip target buffer and current_index (drag_pose.py:237-244,399-402), with float64 predictions from the
    rings the engine holds before each frame.  `track`: the clips followed (all of them, or a sample of a large batch)."""

    def __init__(self, tm, n, track):
        self.tm, self.track = tm, track
        self.std = tm.stds_latent.astype(np.float64)
        self.window = None
        self.buf = np.zeros((n, 117, 24))
        self.bar = np.full(n, BAR_FLOOR)
        self.idx = np.zeros(n, np.int64)
        self.calls = []

    def restart(self, clips):
        """A restarted clip is a fresh DragPose: no buffer yet, index 0."""
        self.buf[clips] = 0.0
        self.bar[clips] = BAR_FLOOR
        self.idx[clips] = 0

    def set_window(self, w):
        if w != self.window:  # a fresh zero buffer; the index is kept
            self.buf[:] = 0.0
            self.bar[:] = BAR_FLOOR
            # the one documented divergence (dp_engine.cu:TargetSchedule::index_at): an index beyond the new buffer, an IndexError in
            # the reference, restarts the cycle
            self.idx[self.idx > w] = 0
            self.window = w

    def before_frame(self, w, st):
        self.set_window(w)
        need = self.track[self.idx[self.track] == 0]
        if need.size:
            rings = (st["latent_buf"][need], st["disp_buf"][need], st["height_buf"][need])
            t64 = predict(self.tm, *rings, w)
            t32 = predict(self.tm, *rings, w, torch.float32)
            rows = readable_rows(w)
            e32 = float((np.abs(t32[:, rows].astype(np.float64) - t64[:, rows]) / self.std).max())
            self.buf[need, : w + 1] = t64
            self.bar[need] = 4.0 * e32 + BAR_FLOOR
            self.calls.append((w, need.size, e32))

    def rows(self):
        return self.buf[self.track, self.idx[self.track]], self.bar[self.track]

    def after_frame(self, w):
        self.idx = np.zeros_like(self.idx) if w == 0 else (self.idx + 1) % w


def _restart(eng, bk, clips, rng, window, boundary):
    """restart_pose on `clips` with random standardised dual quaternions, at a predictor boundary of `window` or between two; the
    rings read back are the set_initial_pose fill."""
    assert (eng.frames_to_boundary(window) == 0) == boundary
    n = len(clips)
    dqs = rng.standard_normal((n, 176)).astype(np.float32)
    hgt = rng.uniform(0.0, 1.7, (n, 6)).astype(np.float32)
    eng.restart_pose(clips, dqs, np.zeros((n, 3)), np.tile([[1.0, 0, 0, 0]], (n, 1)), hgt)
    z = eng.encode(dqs)
    st = eng.state()
    assert np.array_equal(st["latent"][clips], z)
    assert np.array_equal(st["latent_buf"][clips], np.repeat(z[:, None], 60, 1))
    assert np.array_equal(st["height_buf"][clips], np.repeat(hgt[:, None], 60, 1))
    assert not st["disp_buf"][clips].any()
    bk.restart(clips)


def _replace_rings(eng, bk, rng):
    """set_ring_buffers with other chronological content: the rows in use stay, the next window predicts from the new rings."""
    st = eng.state()
    order = (np.arange(60) + 7) % 60
    n = st["latent_buf"].shape[0]
    eng.set_ring_buffers(st["latent_buf"][:, order] + rng.normal(0, 0.05, (n, 60, 24)).astype(np.float32), st["disp_buf"][:, order],
                         st["height_buf"][:, order])


def _teacher_forced(eng, tm, wl, windows, track, events=None, label=""):
    n = eng.n_clips
    bk = ReferenceBookkeeping(tm, n, track)
    T = wl["tgt_pos"].shape[0]
    worst_ratio, worst_err, worst_lt, n_checked = 0.0, 0.0, 0.0, 0
    for t, w in enumerate(windows):
        if events and t in events:
            events[t](eng, bk)
        st = eng.state()
        bk.before_frame(w, st)
        got_idx = eng.clip_index(w)[track]
        assert np.array_equal(got_idx, bk.idx[track]), (label, t, w, np.flatnonzero(got_idx != bk.idx[track])[:8])
        path = 1 if t % 2 == 0 else 3  # both frame kernels
        eng.run(wl["tgt_pos"][t % T], wl["tgt_rot"][t % T], wl["joints"], wl["weights"], temporal_future_window=w, decoder_path=path,
                **LOOP)
        assert eng.last_decoder_path() == path
        tb = eng.state(w)["target_buf"]
        got = (tb[track, 0] if w == 0 else tb[track, bk.idx[track]]).astype(np.float64)
        want, bar = bk.rows()
        err = (np.abs(got - want) / bk.std).max(1)
        bad = np.flatnonzero(~(err <= bar))
        assert bad.size == 0, (label, t, w, track[bad[:8]], err[bad[:8]], bar[bad[:8]], bk.idx[track[bad[:8]]])
        worst_ratio, worst_err = max(worst_ratio, float((err / bar).max())), max(worst_err, float(err.max()))
        lt = eng.frame_stats()[1][track, 2].astype(np.float64)
        lt_want = LOOP["lambda_temporal"] * ((st["latent"][track].astype(np.float64) - got) ** 2).mean(1)
        rel = np.abs(lt - lt_want) / lt_want
        assert rel.max() <= LT_REL, (label, t, w, path, float(rel.max()))
        worst_lt = max(worst_lt, float(rel.max()))
        bk.after_frame(w)
        n_checked += track.size
    e32 = max((c[2] for c in bk.calls), default=0.0)
    print(f"{label}: {len(windows)} frames, {len(bk.calls)} float64 predictor calls, {n_checked} clip-frames; row max err "
          f"{worst_err:.2e} (worst err/bar {worst_ratio:.2f}, max e32 {e32:.2e}); temporal loss max rel err {worst_lt:.1e} (bar {LT_REL:.0e})")
    return bk


def _predict_targets(eng, bk, w):
    """predict_targets at another window: the same window change as a frame at w, before that frame."""
    eng.predict_targets(w)
    bk.set_window(w)


def _cycles(w, n):
    """`n` predictor calls at window w, the first at frame 0."""
    return [w] * ((n - 1) * max(w, 1) + 1)


SCENARIOS = {}
for _w in (4, 8, 12, 16, 28, 60, 116):
    for _p in ("1", "0"):  # enough calls for an early call at index W - 3 and a graph replay (third call of one shape and target)
        SCENARIOS[f"w{_w}-prefetch{_p}"] = dict(n=37, windows=_cycles(_w, 6 if _w <= 16 else 3 if _w <= 60 else 2), prefetch=_p)
for _n in (1, 300, 520):  # 520 clips: the look-ahead runs as 2 080 virtual clips, two parts
    SCENARIOS[f"w0-{_n}clips"] = dict(n=_n, windows=[0] * 10)
SCENARIOS["w16-2101clips-sampled"] = dict(n=2101, windows=_cycles(16, 2), sample=True)
# 16 -> 8 at index 5 (rows 5..7 of the zero buffer) -> 16 at index 3 -> 4 at index 6 (beyond the new buffer) -> 0 at index 2 -> 16
SCENARIOS["window-sequence"] = dict(n=37, windows=[16] * 5 + [8] * 14 + [16] * 19 + [4] * 6 + [0] * 6 + [16] * 18)
for _pp, _name in ((0, "tc"), (1, "fp32")):
    # two sets mid-window (indices 5 and 11; clip 9 twice), three phases afterwards
    SCENARIOS[f"restart-mixed-phases-{_name}"] = dict(n=37, windows=[16] * 50, pred_path=_pp,
                                                      restarts={5: [2, 9, 17, 30], 11: [9, 21, 36]})
    SCENARIOS[f"restart-lookahead-{_name}"] = dict(n=37, windows=[0] * 13, pred_path=_pp, restarts={6: [1, 5, 36]})
    SCENARIOS[f"restart-boundary-{_name}"] = dict(n=37, windows=[16] * 34, pred_path=_pp, restarts={16: [0, 7, 8]})
# predict_targets(4) at index 11 of window 16 (beyond the new buffer): the frames at window 4 start at index 0
SCENARIOS["predict-targets-window-change"] = dict(n=37, windows=[16] * 11 + [4] * 9, predict_targets={11: 4})
SCENARIOS["set-ring-buffers"] = dict(n=37, windows=_cycles(16, 4), replace_rings=(14, 37))  # after the early call; mid-window
SCENARIOS["sharp-w0"] = dict(n=37, windows=[0] * 10, model="sharp")
SCENARIOS["sharp-w16"] = dict(n=37, windows=_cycles(16, 3), model="sharp")


@pytest.mark.parametrize("name", list(SCENARIOS))
def test_teacher_forced_frames_vs_float64_bookkeeping(pose_model, model_npz, temporal_model, monkeypatch, name):
    """One iteration per frame (its losses are iteration 0's), both frame kernels in turn; per frame: the index, the row the engine
    holds for the frame within the bar, and the frame kernel's temporal loss against that row within 1e-4 relative."""
    sc = SCENARIOS[name]
    n, windows = sc["n"], sc["windows"]
    monkeypatch.setenv("DP_PRED_PREFETCH", sc.get("prefetch", "1"))  # read when the engine is created
    rings = tiled_rings(n, 8)
    tm = stress_model(temporal_model, sc["model"], rings) if "model" in sc else temporal_model
    wl = synthetic.make_workload(pose_model, model_npz["offsets"], synthetic.config_6_trackers(), n, min(len(windows), 16))
    track = sample_clips(n) if sc.get("sample") else np.arange(n)
    rng = np.random.default_rng(9)
    events = {}
    for f, clips in sc.get("restarts", {}).items():
        boundary = name.startswith("restart-boundary")
        events[f] = lambda eng, bk, clips=np.array(clips), w=windows[f]: _restart(eng, bk, clips, rng, w, boundary)
    for f in sc.get("replace_rings", ()):
        events[f] = lambda eng, bk: _replace_rings(eng, bk, rng)
    for f, w in sc.get("predict_targets", {}).items():
        events[f] = lambda eng, bk, w=w: _predict_targets(eng, bk, w)
    eng = _engine(pose_model, model_npz, tm, max(64, n))
    try:
        eng.set_predictor_path(sc.get("pred_path", 0))
        _start(eng, n, rings, wl["latent0"])
        _teacher_forced(eng, tm, wl, windows, track, events, label=name)
    finally:
        eng.close()
