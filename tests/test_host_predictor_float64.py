"""The temporal predictor in float64 (oracle/dragposer_port.predict_targets with float64 rings, statistics and weights) as the
reference the engine's predictor is measured against (tests/test_gpu_targets_float64.py), and the stress models those tests use.

What holds here, on the CPU:
- the float64 oracle matches the targets recorded from the unmodified reference (golden/ref_temporal.npz);
- the fp32 port matches the float64 oracle at every window: that difference, e32, sets the GPU tests' bar (4 e32 + 2e-6);
- rows 0..W-1 of the window-W buffer are rows 0..W-1 of the window-116 buffer (the decoder is autoregressive and the step fill only
  looks back), so one window-116 call gives every row a frame can read at any window W > 0;
- every bookkeeping error the GPU tests are meant to see moves the float64 targets by at least ten times that bar, on every model.

Differences are in standardised units: divided by the model's stds_latent, the scale of the predictor's own outputs."""
import os

import numpy as np
import pytest
import torch

import dragposer_port as port

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")
WINDOWS = list(range(0, 117, 4))
BAR_FLOOR = 2e-6
STRESS = ("sharp", "ln", "ff", "stats")


def tiled_rings(n, seed):
    """The golden rings (4 clips) tiled to n clips, latents plus N(0, 0.05) noise: float32 (latent, disp, height)."""
    g = np.load(os.path.join(G, "ref_temporal.npz"))
    rng = np.random.default_rng(seed)
    reps = -(-n // g["latent_buf"].shape[0])
    lat = np.tile(g["latent_buf"], (reps, 1, 1))[:n] + rng.normal(0, 0.05, (n, 60, 24)).astype(np.float32)
    return lat.astype(np.float32), np.tile(g["disp_buf"], (reps, 1, 1))[:n], np.tile(g["height_buf"], (reps, 1, 1))[:n]


def stress_model(base, kind, rings=None):
    """A TemporalModel derived from `base` (float32, fixed seeds) that drives the predictor's arithmetic away from the benign random
    init: "sharp" Q and K rows of every in_proj_weight x4 (attention logits x16), "ln" LayerNorm gains U(0.2, 4) and biases N(0, 1),
    "ff" every linear1 / linear2 weight x4, "stats" means_latent = the mean of `rings`' latents and stds_latent = 0.1 (standardised
    inputs ten times larger)."""
    from dragposer_b200 import model

    rng = np.random.default_rng({"sharp": 1, "ln": 2, "ff": 3, "stats": 4}[kind])
    sd = {k: v.copy() for k, v in base.sd.items()}
    ml, sl = base.means_latent.copy(), base.stds_latent.copy()
    for k, v in sd.items():
        if kind == "sharp" and k.endswith("in_proj_weight"):
            d = v.shape[1]
            v[: 2 * d] *= 4.0
        elif kind == "ln" and "norm" in k and k.endswith(".weight"):
            sd[k] = rng.uniform(0.2, 4.0, v.shape).astype(np.float32)
        elif kind == "ln" and "norm" in k and k.endswith(".bias"):
            sd[k] = rng.normal(0.0, 1.0, v.shape).astype(np.float32)
        elif kind == "ff" and (k.endswith("linear1.weight") or k.endswith("linear2.weight")):
            v *= 4.0
    if kind == "stats":
        ml = rings[0].reshape(-1, 24).mean(0).astype(np.float32)
        sl = np.full(24, 0.1, np.float32)
    return model.TemporalModel(sd, ml, sl)


def predict(tm, lat, disp, hgt, window, dtype=torch.float64):
    """oracle predict_targets in `dtype` on the float32 weights, statistics and rings of the engine -> (B, window + 1, 24) ndarray."""
    t = lambda a: torch.as_tensor(np.asarray(a, np.float32)).to(dtype)
    sd = {k: t(v) for k, v in tm.sd.items()}
    return port.predict_targets(sd, t(tm.means_latent), t(tm.stds_latent), t(lat), t(disp), t(hgt), window).numpy()


def readable_rows(window):
    """The rows a frame can read at `window`: 0..W-1, row 0 at window 0 (row W is never read: current_index < W)."""
    return slice(0, max(window, 1))


class Oracle:
    """Float64 and fp32 targets of one set of rings under one model, for every window: rows 0..W-1 of window W > 0 come from one
    window-116 call, row 0 of window 0 from a window-0 call (test_rows_of_every_window_are_rows_of_window_116 shows they are equal
    to separate calls)."""

    def __init__(self, tm, lat, disp, hgt, fp32=True):
        self.std = tm.stds_latent.astype(np.float64)
        self.t64 = {w: predict(tm, lat, disp, hgt, w) for w in (0, 116)}
        self.t32 = {w: predict(tm, lat, disp, hgt, w, torch.float32) for w in (0, 116)} if fp32 else None

    def rows(self, window, which=None):
        src = self.t64 if which is None else self.t32
        return src[0][:, :1] if window == 0 else src[116][:, :window]

    def e32(self, window):
        """fp32 port vs float64, standardised, over the rows readable at `window`."""
        return float((np.abs(self.rows(window, 32).astype(np.float64) - self.rows(window)) / self.std).max())

    def bar(self, window):
        return 4.0 * self.e32(window) + BAR_FLOOR


def std_err(got, want, std):
    return float((np.abs(np.asarray(got, np.float64) - np.asarray(want, np.float64)) / std).max())


# ----------------------------------------------------------------------------- tests
def test_float64_oracle_matches_the_reference(temporal_model):
    """Ties the float64 predictor to the unmodified reference: its recorded targets (4 clips, windows 0 and 16) within 5e-6, the
    bar the fp32 port meets (test_oracle.test_port_predictor_vs_reference)."""
    g = np.load(os.path.join(G, "ref_temporal.npz"))
    for w in (0, 16):
        got = predict(temporal_model, g["latent_buf"], g["disp_buf"], g["height_buf"], w)
        assert got.dtype == np.float64
        rows = readable_rows(w)
        err = np.abs(got[:, rows] - g[f"target_buf_w{w}"][:, rows]).max()
        print(f"window {w}: float64 oracle vs the reference's recorded targets {err:.2e}")
        assert err <= 5e-6


def test_fp32_port_matches_float64_at_every_window(temporal_model):
    """37 clips (golden rings tiled, plus noise), every window 0, 4, ..., 116: the fp32 port is within 2e-6 of float64.  And the rows
    a frame can read at window W are bitwise rows 0..W-1 of the window-116 buffer, in both precisions (what Oracle relies on)."""
    lat, disp, hgt = tiled_rings(37, 0)
    full = {dt: predict(temporal_model, lat, disp, hgt, 116, dt) for dt in (torch.float64, torch.float32)}
    worst = 0.0
    for w in WINDOWS:
        rows = readable_rows(w)
        t64 = predict(temporal_model, lat, disp, hgt, w)
        t32 = predict(temporal_model, lat, disp, hgt, w, torch.float32)
        assert t64.shape == (37, w + 1, 24) and t32.dtype == np.float32
        if w > 0:
            assert np.array_equal(t64[:, rows], full[torch.float64][:, rows]) and np.array_equal(t32[:, rows], full[torch.float32][:, rows])
        err = np.abs(t32[:, rows].astype(np.float64) - t64[:, rows]).max()
        worst = max(worst, float(err))
        assert err <= 2e-6, (w, err)
    print(f"fp32 port vs float64, windows 0..116: max abs err {worst:.2e}")


def _perturbations(tm, lat, disp, hgt, window):
    """Float64 targets of the bookkeeping errors the GPU tests must see, each next to the correct ones: standardised max difference
    over the readable rows."""
    lat, disp, hgt = (np.asarray(a, np.float64) for a in (lat, disp, hgt))
    rows = readable_rows(window)
    ref = predict(tm, lat, disp, hgt, window)
    roll = lambda a: np.roll(a, 1, axis=1)
    dec57 = lat.copy()
    dec57[:, 56] = lat[:, 57]  # decoder token read one row late; rows 0..52 (the encoder's) unchanged
    cases = {
        "ring head one row off": (roll(lat), roll(disp), roll(hgt)),
        "decoder token from row 57": (dec57, disp, hgt),
        "heights one row off": (lat, disp, roll(hgt)),
        "displacement sums one row off": (lat, roll(disp), hgt),
    }
    std = tm.stds_latent.astype(np.float64)
    out = {k: std_err(predict(tm, *v, window)[:, rows], ref[:, rows], std) for k, v in cases.items()}
    full = predict(tm, lat, disp, hgt, 116)
    out["step fill one prediction late"] = std_err(full[:, 4 : window + 4], full[:, :window], std)  # row r from raw[4(r//4) + 8]
    return out


@pytest.mark.parametrize("kind", ("base",) + STRESS)
def test_bookkeeping_errors_move_the_float64_targets_far_beyond_the_bar(temporal_model, kind):
    """Power table, window 16, 37 clips: each error moves the float64 targets by at least ten times the GPU bar (4 e32 + 2e-6) of the
    same model and clips, so a check at that bar cannot miss it -- on the random-init model and on every stress model."""
    rings = tiled_rings(37, 0)
    tm = temporal_model if kind == "base" else stress_model(temporal_model, kind, rings)
    bar = Oracle(tm, *rings).bar(16)
    table = _perturbations(tm, *rings, 16)
    print(f"{kind}: bar {bar:.2e}; " + ", ".join(f"{k} {v:.2e}" for k, v in table.items()))
    for k, v in table.items():
        assert v >= 10 * bar, (kind, k, v, bar)


def test_stress_models_are_what_they_claim(temporal_model):
    """Each stress model changes exactly its own tensors and is deterministic."""
    rings = tiled_rings(37, 0)
    for kind in STRESS:
        a, b = stress_model(temporal_model, kind, rings), stress_model(temporal_model, kind, rings)
        changed = {k for k in a.sd if not np.array_equal(a.sd[k], temporal_model.sd[k])}
        assert all(np.array_equal(a.sd[k], b.sd[k]) for k in a.sd) and np.array_equal(a.means_latent, b.means_latent)
        if kind == "sharp":
            assert changed == {k for k in a.sd if k.endswith("in_proj_weight")}
        elif kind == "ln":
            assert changed == {k for k in a.sd if "norm" in k} and all(a.sd[k].min() >= 0.2 for k in changed if k.endswith(".weight"))
        elif kind == "ff":
            assert changed == {k for k in a.sd if k.endswith(("linear1.weight", "linear2.weight"))}
        else:
            assert not changed and np.all(a.stds_latent == np.float32(0.1)) and np.abs(a.means_latent).max() > 0
