"""The float64 ("exact", oracle.frcnn.exact()) evaluation of EfficientDet-D7 at 1536x1536 on the frame of
tests/test_effdet_gpu.py::test_d7_full_size_matches_oracle: final detections + backbone endpoints' statistics.  It takes
half a minute on 8 cores here but eight minutes on the GPU box's host (no fast float64 conv path there), so the test reads
this fixture instead of recomputing it; the float32 oracle is still evaluated live.  Run: python tests/golden/make_golden_d7_exact.py"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, os.path.dirname(HERE))
from test_effdet_gpu import _condition_d7_heads, _frame  # noqa: E402
from object_detection_tracking_b200.effdet_config import BACKBONE_OF, make_effdet_config  # noqa: E402
from object_detection_tracking_b200.synth import synth_effdet_weights, synth_efficientnet_weights  # noqa: E402
from oracle import effdet as oe  # noqa: E402
from oracle import efficientnet as on  # noqa: E402
from oracle import frcnn  # noqa: E402

det = "efficientdet-d7"
bb = BACKBONE_OF[det]
cfg = make_effdet_config(det, 1536, 1536)
Wt = dict(synth_effdet_weights(cfg))
Wt.update(synth_efficientnet_weights(bb))
_condition_d7_heads(Wt)
frame = _frame(1080, 1920)
img, scale = on.preprocess(frame, 1536, 1536)
with frcnn.exact():
    f64 = on.forward(img, Wt, bb, stages=False)
    r64 = oe.forward_from_features(cfg, Wt, {l: f64[l] for l in (3, 4, 5)}, image_scale=scale, stages=False)
np.savez_compressed(os.path.join(HERE, "d7_exact.npz"), final_boxes=r64["final_boxes"], final_probs=r64["final_probs"],
                    final_labels=r64["final_labels"], levels=r64["levels"],
                    c3=f64[3][:, ::8, ::8], c4=f64[4][:, ::4, ::4], c5=f64[5][:, ::4, ::4],     # strided samples of the endpoints
                    frame_checksum=np.int64(frame.astype(np.int64).sum()))
print("written", os.path.join(HERE, "d7_exact.npz"))
