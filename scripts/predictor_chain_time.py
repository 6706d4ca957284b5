"""B = 1 predictor call at window 16 (5 decoder passes, ~70 kernels): wall time of dp_engine_predict_targets + device synchronisation.
From the second call of a shape on, everything after the embedding kernel is a replayed CUDA graph; the first five calls are not counted."""
import os, sys, time
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from dragposer_b200 import _lib, model
from dragposer_b200.engine import BatchedDragPose

B = int(sys.argv[1]) if len(sys.argv) > 1 else 1
npz = os.path.join(ROOT, "tests/golden/model_dancedb.npz")
pm = model.load_folded_npz(npz); off = np.load(npz)["offsets"]
tm = model.temporal_from_state(model.random_temporal_state(2222))
eng = BatchedDragPose(pm, off, tm, B)
eng.set_initial_state(np.zeros((B, 24)), np.zeros((B, 3)), np.tile([[1.0, 0, 0, 0]], (B, 1)), np.zeros((B, 6)))
for W in (16, 0):
    ts, te = [], []
    for i in range(60):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _lib.check(eng.lib.dp_engine_predict_targets(eng.h, W, None))
        t1 = time.perf_counter()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0); te.append(t1 - t0)
    print(f"{B} clip(s), window {W}: enqueue p50 {1e6 * np.median(te[5:]):.0f} us, "
          f"enqueue + device p50 {1e6 * np.median(ts[5:]):.0f} us")
eng.close()
