"""One EfficientDet pass bracketed by cudaProfilerStart/Stop, for ncu:
  ncu --profile-from-start off --metrics gpu__time_duration.sum --clock-control none --csv \
      --log-file gpurun_out/effdet_launches.csv python tools/effdet_ncu_pass.py [det] [H] [W] [precision]
A number printed under ncu is never a bench value."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from gpu_effnet_probe import synth_frame  # noqa: E402
from object_detection_tracking_b200.effdet import EffdetEngine  # noqa: E402
from object_detection_tracking_b200.effdet_config import BACKBONE_OF, make_effdet_config  # noqa: E402
from object_detection_tracking_b200.synth import synth_effdet_weights, synth_efficientnet_weights  # noqa: E402

det = sys.argv[1] if len(sys.argv) > 1 else "efficientdet-d7"
H = int(sys.argv[2]) if len(sys.argv) > 2 else 1536
W = int(sys.argv[3]) if len(sys.argv) > 3 else 1536
prec = sys.argv[4] if len(sys.argv) > 4 else "split"
cfg = make_effdet_config(det, H, W)
Wt = dict(synth_effdet_weights(cfg))
Wt.update(synth_efficientnet_weights(BACKBONE_OF[det]))
eng = EffdetEngine(cfg, Wt, precision=prec, backbone=BACKBONE_OF[det])
frame = synth_frame(1080, 1920)
eng.detect(frame)
torch.cuda.synchronize()
torch.cuda.profiler.start()
out = eng.detect(frame)
torch.cuda.synchronize()
torch.cuda.profiler.stop()
print("profiled pass: %d detections" % len(out["final_probs"]))
