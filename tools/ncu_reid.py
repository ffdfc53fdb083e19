"""One OSNet-x1.0 embedding pass (batch 64) bracketed by cudaProfilerStart/Stop, for ncu."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from object_detection_tracking_b200.reid import ReidEngine  # noqa: E402
from object_detection_tracking_b200.synth import synth_osnet_state  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 64
eng = ReidEngine(B, precision=sys.argv[2] if len(sys.argv) > 2 else "split")
eng.load_state(synth_osnet_state(4321))
crops = np.random.default_rng(0).integers(0, 256, (B, 256, 128, 3)).astype(np.uint8)
eng.embed(crops)
torch.cuda.synchronize()
torch.cuda.profiler.start()
f = eng.embed(crops)
torch.cuda.synchronize()
torch.cuda.profiler.stop()
print("profiled pass:", f.shape, eng.num_launches())
