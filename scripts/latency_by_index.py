"""B = 1 streaming through BatchedDragPose.run (window 16, MaxIter 5): host-observed call time by position in the predictor window."""
import os, sys, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from dragposer_b200 import model, synthetic
from dragposer_b200.engine import BatchedDragPose
npz = os.path.join(ROOT, "tests/golden/model_dancedb.npz")
pm = model.load_folded_npz(npz); off = np.load(npz)["offsets"]
tm = model.temporal_from_state(model.random_temporal_state(2222))
cfg = synthetic.config_6_trackers()
T = 336
wl = synthetic.make_workload(pm, off, cfg, 1, T)
eng = BatchedDragPose(pm, off, tm, 1)
eng.set_initial_state(wl["latent0"], np.zeros((1, 3)), [[1.0, 0, 0, 0]], np.zeros((1, 6)))
kw = dict(stop_eps_pos=1e-4, stop_eps_rot=1e-2, max_iter=5, min_loss_incr=1e-5, learning_rate=1e-2, lambda_rot=1, lambda_temporal=0.02, temporal_future_window=16)
ts = np.zeros(T)
for t in range(T):
    t0 = time.perf_counter(); eng.run(wl["tgt_pos"][t], wl["tgt_rot"][t], wl["joints"], wl["weights"], **kw); ts[t] = time.perf_counter() - t0
ts = ts[64:].reshape(-1, 16)
print("DP_PRED_PREFETCH=%s  median call time (us) by window index:" % os.environ.get("DP_PRED_PREFETCH", "1"))
print(" ".join(f"{1e6 * v:.0f}" for v in np.median(ts, axis=0)), f"| mean {1e6 * ts.mean():.1f}")
eng.close()
