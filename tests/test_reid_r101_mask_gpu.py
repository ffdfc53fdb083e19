"""GPU parity of the two engines that build their own launch sequences on conv_tc_kernel beyond the detector: the vehicle
ReID ResNet-101 (torchreid/models/resnet.py:441-455) against reference-generated activations (resnet101_reid.npz), and the
Mask-RCNN head (--add_mask, models.py:934-961,1173-1199) against oracle.frcnn.maskrcnn_head.  First B200 run: round 2, 5/5 green."""
import hashlib
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def r101(golden_dir):
    return np.load(os.path.join(golden_dir, "resnet101_reid.npz"))


def golden_crops(g):
    """The ragged uint8 noise crops the fixture was generated from (seeded as in tests/golden/make_golden_tmot.py),
    checked byte for byte against the hashes stored with it."""
    rng = np.random.default_rng(15)
    crops = [rng.integers(0, 256, (int(rng.integers(40, 200)), int(rng.integers(60, 320)), 3), dtype=np.uint8)
             for _ in range(4)]
    assert [c.shape for c in crops] == [tuple(s) for s in g["crop_shapes"]]
    assert [hashlib.sha256(c.tobytes()).hexdigest() for c in crops] == list(g["crop_sha256"])
    return crops


def test_torch_style_strided_convs_single_op():
    """The two strided geometries the torchreid ResNet adds, as single ops against torch fp32: 3x3 stride 2 pad 1 and
    1x1 stride 2 on even extents (run as (1,0,1,0) / (0,-1,0,-1), which is the same convolution there)."""
    import torch
    import torch.nn.functional as F
    from object_detection_tracking_b200 import engine
    rng = np.random.default_rng(21)
    for (H, W, cin, cout, k, pad_run) in ((32, 64, 64, 64, 3, (1, 0, 1, 0)), (16, 32, 256, 512, 1, (0, -1, 0, -1)),
                                          (8, 16, 256, 256, 3, (1, 0, 1, 0))):
        x = rng.standard_normal((2, H, W, cin)).astype(np.float32)
        w = (rng.standard_normal((k, k, cin, cout)) / np.sqrt(k * k * cin)).astype(np.float32)
        ref = F.conv2d(torch.from_numpy(x).permute(0, 3, 1, 2), torch.from_numpy(w).permute(3, 2, 0, 1).contiguous(),
                       stride=2, padding=k // 2).permute(0, 2, 3, 1).numpy()
        out = engine.op_conv2d(x, w, None, None, stride=2, dil=1, pad=pad_run, relu=False, res_shift=0, impl="tcgen05",
                               split=True)
        assert out.shape == ref.shape
        assert np.abs(out - ref).max() <= 2e-5 * np.abs(ref).max()


def test_resnet101_reid_embedding_matches_reference(r101):
    """torchreid resnet101 (vehicle extractor, single_video_reid.py:410-415): features and intermediate activations
    against the reference model run on the CPU (tests/golden/make_golden_tmot.py: resnet101_reid)."""
    from object_detection_tracking_b200.reid import ReidEngine
    from object_detection_tracking_b200.synth import synth_resnet101_reid_state
    eng = ReidEngine(batch=4, precision="split", model="resnet101")
    eng.load_state(synth_resnet101_reid_state(2468))
    feats = eng.embed(r101["resized"])
    ref = r101["feats"]
    assert feats.shape == ref.shape == (4, 2048)
    mp = eng.get_activation("maxpool")
    assert mp.shape == (4, 32, 64, 64)
    assert np.abs(mp[:1, :8] - r101["maxpool"]).max() <= 1e-5 * np.abs(r101["maxpool"]).max()
    for name in ("layer1.0", "layer2.0", "layer3.22"):
        act = eng.get_activation(name)
        m = r101[name + "_mean"]
        assert np.abs(act.mean(axis=(1, 2)) - m).max() <= 2e-5 * max(1.0, float(r101[name + "_absmax"]))
    l4 = eng.get_activation("layer4")
    assert l4.shape == (4, 4, 8, 2048)
    assert np.abs(l4[:2] - r101["layer4"]).max() <= 3e-5 * np.abs(r101["layer4"]).max()     # fp32-class through 101 layers
    assert np.abs(feats - ref).max() <= 3e-5 * np.abs(ref).max()
    again = eng.embed(r101["resized"][:2])                                                     # graph replay, smaller n
    np.testing.assert_array_equal(again, feats[:2])
    assert eng.num_launches() > 100
    eng.close()


def test_resnet101_feature_extractor_drop_in(r101):
    from object_detection_tracking_b200.reid import FeatureExtractor
    from object_detection_tracking_b200.synth import synth_resnet101_reid_state
    ext = FeatureExtractor("resnet101", model_path="", image_size=(128, 256), device="cuda:0", batch=4,
                           state_dict=synth_resnet101_reid_state(2468))
    crops = golden_crops(r101)
    got = ext(crops).numpy()
    assert got.shape == (4, 2048)
    assert np.abs(got - r101["feats"]).max() <= 3e-5 * np.abs(r101["feats"]).max()
    with pytest.raises(NotImplementedError):
        FeatureExtractor("resnet101", image_size=(256, 128), state_dict={})


def test_mask_head_matches_oracle():
    """--add_mask (models.py:934-961, 1173-1199): ROIAlign 14x14 of the final boxes, 4 x conv3x3, 2x2/2 transposed conv,
    conv1x1, own-class sigmoid -- final_masks and all class logits against the oracle on the 192x256 frame."""
    from object_detection_tracking_b200 import _lib
    from object_detection_tracking_b200.config import make_config
    from object_detection_tracking_b200.engine import Detector
    from object_detection_tracking_b200.synth import synth_frame, synth_weights
    from oracle import frcnn
    H, W = 192, 256
    cfg = make_config(resnet_num_block=(1, 1, 2, 1), max_size=W, short_edge_size=H, add_mask=True)
    Wt = synth_weights(cfg, 1234)
    frame = synth_frame(H, W, 5).astype(np.float32)
    det = Detector(cfg, 1, H, W, device=0, precision="split", use_cuda_graph=False)
    det.load_weights(Wt)
    out = det.detect_host(frame[None])
    ref = frcnn.forward(cfg, Wt, frame, stages=True)
    r = int(out["valid"][0])
    assert r == ref["final_boxes"].shape[0] > 0
    # final_masks: [R,28,28] sigmoid of the own-class logits; order may differ between near-tied scores -> match by box
    masks = det.get_masks()[0]
    d = (np.abs(out["boxes"][0, :r, None, :] - ref["final_boxes"][None, :, :]).max(-1)
         + 10.0 * (out["labels"][0, :r, None] != ref["final_labels"][None, :]))
    match = d.argmin(1)
    assert d.min(1).max() < 2e-3
    assert np.abs(masks[:r] - ref["final_masks"][match]).max() < 2e-4
    assert (masks[r:] == 0).all()
    # all class logits of the live rows
    ml = det.get_stage("mask_logits")                                   # [B*R, 196*4, ld, 1]
    ld = ml.shape[2]
    ml = ml.reshape(-1, 14, 14, 2, 2, ld)[:r, ..., :cfg.num_class - 1]  # [r, y, x, dy, dx, c]
    got = ml.transpose(0, 5, 1, 3, 2, 4).reshape(r, cfg.num_class - 1, 28, 28)
    refl = ref["mask_logits"][match]
    assert np.abs(got - refl).max() <= 1e-4 * max(1.0, float(np.abs(refl).max()))


def test_mask_head_graph_replay_and_backend_fetch():
    from object_detection_tracking_b200.backend import Session, get_model
    from object_detection_tracking_b200.config import make_config
    from object_detection_tracking_b200.synth import synth_frame, synth_weights
    H, W = 192, 256
    cfg = make_config(resnet_num_block=(1, 1, 2, 1), max_size=W, short_edge_size=H, add_mask=True)
    model = get_model(cfg, gpuid=0)
    model.set_weights(synth_weights(cfg, 1234))
    sess = Session()
    frame = synth_frame(H, W, 5).astype(np.float32)
    fetches = [model.final_boxes, model.final_labels, model.final_probs, model.final_masks]
    a = sess.run(fetches, feed_dict=model.get_feed_dict_forward(frame))
    b = sess.run(fetches, feed_dict=model.get_feed_dict_forward(frame))           # CUDA-graph replay
    assert a[3].shape == (len(a[0]), 28, 28) and a[3].dtype == np.float32 and len(a[0]) > 0
    assert ((a[3] > 0) & (a[3] < 1)).all()
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)
