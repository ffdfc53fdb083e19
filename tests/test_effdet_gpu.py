"""EfficientDet BiFPN + class/box nets + post-processing on the GPU (b2_effdet_* C ABI) vs oracle/effdet.py.
Tolerances: stage tensors fp32-class (split precision); integer outputs (labels, levels, count) exact; boxes within
1e-3 px; scores 1e-6."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _features(cfg, seed=5):
    from object_detection_tracking_b200.effdet_config import feat_sizes
    rng = np.random.default_rng(seed)
    fs = feat_sizes(cfg)
    return {l: np.abs(rng.standard_normal((cfg.backbone_channels[l - 3],) + fs[l])).astype(np.float32) for l in (3, 4, 5)}


def _case(name, h, w, precision="split", **over):
    from object_detection_tracking_b200.effdet import EffdetEngine
    from object_detection_tracking_b200.effdet_config import make_effdet_config
    from object_detection_tracking_b200.synth import synth_effdet_weights
    from oracle import effdet as oe
    cfg = make_effdet_config(name, h, w, **over)
    W = synth_effdet_weights(cfg)
    feats = _features(cfg)
    ref = oe.forward_from_features(cfg, W, feats, image_scale=1.25, stages=True)
    eng = EffdetEngine(cfg, W, precision=precision)
    out = eng.run_features(feats, image_scale=1.25)
    return cfg, eng, out, ref, feats


@pytest.fixture(scope="module")
def d0():
    c = _case("efficientdet-d0", 256, 384, fpn_cell_repeats=2, box_class_repeats=2)
    yield c
    c[1].close()


def test_bifpn_levels_match_oracle(d0):
    cfg, eng, out, ref, _ = d0
    for l in range(3, 8):
        g, r = eng.stage("fpn%d" % l), ref["fpn"][l].transpose(1, 2, 0)
        assert g.shape == r.shape
        assert np.abs(g - r).max() <= 2e-5 * max(1.0, np.abs(r).max())


def test_class_and_box_outputs_match_oracle(d0):
    cfg, eng, out, ref, _ = d0
    for l in range(3, 8):
        for k, key in (("cls", "cls_out"), ("box", "box_out")):
            g, r = eng.stage("%s%d" % (k, l)), ref[key][l]
            assert g.shape == r.shape
            assert np.abs(g - r).max() <= 2e-5 * max(1.0, np.abs(r).max())


def test_detections_match_oracle(d0):
    cfg, eng, out, ref, _ = d0
    assert len(out["final_probs"]) == len(ref["final_probs"]) > 0
    np.testing.assert_array_equal(out["final_labels"], ref["final_labels"])
    np.testing.assert_array_equal(out["levels"], ref["levels"])
    assert np.abs(out["final_boxes"] - ref["final_boxes"]).max() <= 1e-3
    assert np.abs(out["final_probs"] - ref["final_probs"]).max() <= 1e-6
    assert np.abs(out["fpn_box_feat"] - ref["fpn_box_feat"]).max() <= 2e-5 * max(1.0, np.abs(ref["fpn_box_feat"]).max())


def test_graph_replay_is_deterministic_and_scale_is_live(d0):
    cfg, eng, out, ref, feats = d0
    again = eng.run_features(feats, image_scale=1.25)
    for k in out:
        np.testing.assert_array_equal(again[k], out[k])
    other = eng.run_features(feats, image_scale=2.0)            # image_scale is read on the device, not baked in
    np.testing.assert_array_equal(other["final_labels"], out["final_labels"])
    np.testing.assert_allclose(other["final_boxes"], out["final_boxes"] * np.float32(2.0 / 1.25), rtol=1e-6)
    assert eng.num_launches > 100


def test_sum_method_and_padded_filters():
    # D1 width (88 filters -> padded to 128 operand channels), un-normalised "sum" combine (the D6/D7 setting)
    cfg, eng, out, ref, _ = _case("efficientdet-d1", 256, 256, fpn_cell_repeats=2, box_class_repeats=1,
                                  fpn_weight_method="sum")
    for l in range(3, 8):
        g, r = eng.stage("fpn%d" % l), ref["fpn"][l].transpose(1, 2, 0)
        assert np.abs(g - r).max() <= 2e-5 * max(1.0, np.abs(r).max())
    np.testing.assert_array_equal(out["final_labels"], ref["final_labels"])
    np.testing.assert_array_equal(out["levels"], ref["levels"])
    assert np.abs(out["final_boxes"] - ref["final_boxes"]).max() <= 1e-3
    eng.close()


def test_d7_width_small_frame():
    # the headline family's width (384 filters, 8 cells, 5 head repeats, anchor_scale 5, "sum") on a small frame
    cfg, eng, out, ref, _ = _case("efficientdet-d7", 128, 256)
    np.testing.assert_array_equal(out["final_labels"], ref["final_labels"])
    np.testing.assert_array_equal(out["levels"], ref["levels"])
    assert np.abs(out["final_boxes"] - ref["final_boxes"]).max() <= 1e-3
    assert np.abs(out["fpn_box_feat"] - ref["fpn_box_feat"]).max() <= 5e-5 * max(1.0, np.abs(ref["fpn_box_feat"]).max())
    eng.close()


def test_fp16_precision_is_close():
    cfg, eng, out, ref, _ = _case("efficientdet-d0", 256, 384, precision="fp16", fpn_cell_repeats=2, box_class_repeats=2)
    for l in range(3, 8):
        g, r = eng.stage("cls%d" % l), ref["cls_out"][l]
        assert np.abs(g - r).max() <= 2e-2 * max(1.0, np.abs(r).max())
    # set-based: near-tied candidates may swap order at fp16 accuracy
    hits = 0
    for b, lab in zip(out["final_boxes"], out["final_labels"]):
        d = np.abs(ref["final_boxes"] - b).max(axis=1)
        j = int(np.argmin(d))
        hits += int(d[j] < 0.5 and ref["final_labels"][j] == lab)
    assert hits >= 0.9 * len(ref["final_labels"])
    eng.close()


def test_ties_resolve_to_lowest_index():
    # all class logits equal (zero pointwise kernel, constant bias): tf.nn.top_k keeps the lowest flat indices
    from object_detection_tracking_b200.effdet import EffdetEngine
    from object_detection_tracking_b200.effdet_config import make_effdet_config
    from object_detection_tracking_b200.synth import synth_effdet_weights
    from oracle import effdet as oe
    cfg = make_effdet_config("efficientdet-d0", 128, 128, fpn_cell_repeats=1, box_class_repeats=1, max_detection_topk=700)
    W = synth_effdet_weights(cfg)
    W["class_net/class-predict/pointwise_kernel"] = np.zeros_like(W["class_net/class-predict/pointwise_kernel"])
    W["class_net/class-predict/bias"] = np.full_like(W["class_net/class-predict/bias"], -1.0)
    feats = _features(cfg)
    ref = oe.forward_from_features(cfg, W, feats, image_scale=1.0)
    eng = EffdetEngine(cfg, W)
    out = eng.run_features(feats, image_scale=1.0)
    np.testing.assert_array_equal(out["final_labels"], ref["final_labels"])
    np.testing.assert_array_equal(out["levels"], ref["levels"])
    assert np.abs(out["final_boxes"] - ref["final_boxes"]).max() <= 1e-3
    eng.close()


def test_missing_weight_fails_loudly():
    from object_detection_tracking_b200.effdet import EffdetEngine
    from object_detection_tracking_b200.effdet_config import make_effdet_config
    from object_detection_tracking_b200.synth import synth_effdet_weights
    cfg = make_effdet_config("efficientdet-d0", 128, 128, fpn_cell_repeats=1, box_class_repeats=1)
    W = synth_effdet_weights(cfg)
    del W["box_net/box-predict/bias"]
    with pytest.raises(RuntimeError, match="missing weight"):
        EffdetEngine(cfg, W)


# ---- pre-processing + EfficientNet backbone + whole-frame detect (a16, a17) ------------------------------------------
def _frame(h, w, seed=3):
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (h // 8 + 1, w // 8 + 1, 3)).astype(np.float32)
    img = np.kron(base, np.ones((8, 8, 1), np.float32))[:h, :w]
    return np.clip(img + rng.standard_normal((h, w, 3)) * 12, 0, 255).astype(np.uint8)


def _condition_d7_heads(Wt):
    """The seeded weights are conditioned for the shallow test nets; through D7's 8 cells and 5-deep heads the predict
    layers reach |box logit| ~ 18 (exp -> boxes of 1e7 px) and |class logit| ~ 280 (every score exactly 1).  Scaling the
    two predict kernels brings the outputs back to a trained detector's range (boxes inside the frame, spread scores)."""
    Wt["class_net/class-predict/pointwise_kernel"] = Wt["class_net/class-predict/pointwise_kernel"] * np.float32(0.03)
    Wt["box_net/box-predict/pointwise_kernel"] = Wt["box_net/box-predict/pointwise_kernel"] * np.float32(0.08)


def _full_case(det, H, W, fh, fw, precision="split", tweak=None, **over):
    from object_detection_tracking_b200.effdet import EffdetEngine
    from object_detection_tracking_b200.effdet_config import BACKBONE_OF, make_effdet_config
    from object_detection_tracking_b200.synth import synth_effdet_weights, synth_efficientnet_weights
    from oracle import effdet as oe
    from oracle import efficientnet as on
    bb = BACKBONE_OF[det]
    cfg = make_effdet_config(det, H, W, **over)
    Wt = dict(synth_effdet_weights(cfg))
    Wt.update(synth_efficientnet_weights(bb))
    if tweak is not None:
        tweak(Wt)
    frame = _frame(fh, fw)
    img, scale = on.preprocess(frame, H, W)
    feats = on.forward(img, Wt, bb, stages=True)
    ref = oe.forward_from_features(cfg, Wt, {l: feats[l] for l in (3, 4, 5)}, image_scale=scale, stages=True)
    eng = EffdetEngine(cfg, Wt, precision=precision, backbone=bb)
    out = eng.detect(frame)
    return cfg, eng, out, ref, feats, img, scale, frame, Wt


@pytest.fixture(scope="module")
def full_d0():
    c = _full_case("efficientdet-d0", 256, 384, 300, 500, fpn_cell_repeats=2, box_class_repeats=2)
    yield c
    c[1].close()


def test_preprocess_is_bit_exact(full_d0):
    cfg, eng, out, ref, feats, img, scale, frame, _ = full_d0
    np.testing.assert_array_equal(eng.stage("image"), img)
    assert out["image_scale"] == pytest.approx(float(scale), rel=1e-7)


def test_backbone_blocks_and_endpoints_match_oracle(full_d0):
    cfg, eng, out, ref, feats, img, scale, frame, _ = full_d0
    st = feats["stages"]
    g = eng.stage("stem", real=st["stem"].shape[0])
    assert np.abs(g - st["stem"].transpose(1, 2, 0)).max() <= 2e-5 * max(1.0, np.abs(st["stem"]).max())
    for i in range(len(st) - 1):
        r = st["block_%d" % i].transpose(1, 2, 0)
        g = eng.stage("block_%d" % i, real=r.shape[2])
        assert g.shape == r.shape
        assert np.abs(g - r).max() <= 2e-5 * max(1.0, np.abs(r).max()), "block_%d" % i
    for l in (3, 4, 5):
        r = feats[l].transpose(1, 2, 0)
        assert np.abs(eng.stage("c%d" % l) - r).max() <= 2e-5 * max(1.0, np.abs(r).max())


def test_whole_frame_detections_match_oracle(full_d0):
    cfg, eng, out, ref, feats, img, scale, frame, _ = full_d0
    assert len(out["final_probs"]) == len(ref["final_probs"]) > 0
    np.testing.assert_array_equal(out["final_labels"], ref["final_labels"])
    np.testing.assert_array_equal(out["levels"], ref["levels"])
    assert np.abs(out["final_boxes"] - ref["final_boxes"]).max() <= 1e-3
    assert np.abs(out["final_probs"] - ref["final_probs"]).max() <= 5e-6
    assert np.abs(out["fpn_box_feat"] - ref["fpn_box_feat"]).max() <= 2e-5 * max(1.0, np.abs(ref["fpn_box_feat"]).max())
    again = eng.detect(frame)                                        # CUDA-graph replay, SE-scaled weights rewritten per frame
    for k in ("final_boxes", "final_probs", "final_labels", "fpn_box_feat"):
        np.testing.assert_array_equal(again[k], out[k])
    other = eng.detect(_frame(240, 320, seed=9))                     # a different frame size through the same context
    assert other["image_scale"] != out["image_scale"]
    back = eng.detect(frame)
    np.testing.assert_array_equal(back["final_boxes"], out["final_boxes"])


def test_backbone_5x5_stride2_and_wider_trunk():
    # b1 trunk (23 blocks) on a square input whose frame is taller than wide (height-limited scale)
    cfg, eng, out, ref, feats, img, scale, frame, _ = _full_case("efficientdet-d1", 256, 256, 200, 190,
                                                                 fpn_cell_repeats=1, box_class_repeats=1)
    np.testing.assert_array_equal(eng.stage("image"), img)
    for l in (3, 4, 5):
        r = feats[l].transpose(1, 2, 0)
        assert np.abs(eng.stage("c%d" % l) - r).max() <= 2e-5 * max(1.0, np.abs(r).max())
    np.testing.assert_array_equal(out["final_labels"], ref["final_labels"])
    assert np.abs(out["final_boxes"] - ref["final_boxes"]).max() <= 1e-3
    eng.close()


def test_d7_full_size_matches_oracle():
    """BASELINE configs[2]: EfficientDet-D7 (EfficientNet-b6 trunk, 8 BiFPN cells of 384 filters, 5-deep heads) at
    1536x1536 on one 1080x1920 frame, whole-frame detect against the oracle (efficientdet_wrapper.py:40-61,367-474).

    The 1e-3 px bar of the north star is BELOW float32 rounding noise for this configuration: the float32 oracle is itself
    7.6e-3 px away from the float64 evaluation of the same graph (oracle.frcnn.exact(), measured on the CPU: relative
    error 5e-6 on c5, 6e-6 ... 8e-6 on the box logits, times anchors of up to 800 px).  Integer outputs (count, class ids,
    levels) must be exact, scores within 1e-5; for the boxes the GPU must be as close to the exact evaluation as a
    float32 implementation can be: within 2x the float32 port's own distance (and 2e-2 px absolute)."""
    import json
    import os
    cfg, eng, out, ref, feats, img, scale, frame, Wt = _full_case("efficientdet-d7", 1536, 1536, 1080, 1920, tweak=_condition_d7_heads)
    try:
        # the float64 evaluation of the same frame / weights: fixture of tests/golden/make_golden_d7_exact.py (8 minutes on
        # the GPU box's host, so not recomputed here)
        gx = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "d7_exact.npz"))
        assert int(gx["frame_checksum"]) == int(frame.astype(np.int64).sum())
        ref64 = {k: gx[k] for k in ("final_boxes", "final_probs", "final_labels", "levels")}
        strides = {3: 8, 4: 4, 5: 4}
        f64 = {l: gx["c%d" % l] for l in (3, 4, 5)}
        np.testing.assert_array_equal(eng.stage("image"), img)
        rec = {"config": "C3", "final": len(out["final_probs"]), "final_ref": len(ref["final_probs"])}
        rec["c_rel"] = [float(np.abs(eng.stage("c%d" % l) - feats[l].transpose(1, 2, 0)).max() / np.abs(feats[l]).max())
                        for l in (3, 4, 5)]
        rec["c_rel_exact"] = [float(np.abs(eng.stage("c%d" % l)[::strides[l], ::strides[l]] - f64[l].transpose(1, 2, 0)).max() /
                                    np.abs(f64[l]).max()) for l in (3, 4, 5)]       # on the fixture's strided sample
        rec["c_rel_oracle32_exact"] = [float(np.abs(feats[l][:, ::strides[l], ::strides[l]] - f64[l]).max() / np.abs(f64[l]).max())
                                       for l in (3, 4, 5)]
        rec["fpn_rel"] = [float(np.abs(eng.stage("fpn%d" % l) - ref["fpn"][l].transpose(1, 2, 0)).max() /
                                max(1.0, np.abs(ref["fpn"][l]).max())) for l in range(3, 8)]
        rec["cls_rel"] = [float(np.abs(eng.stage("cls%d" % l) - ref["cls_out"][l]).max() / max(1.0, np.abs(ref["cls_out"][l]).max()))
                          for l in range(3, 8)]
        rec["box_rel"] = [float(np.abs(eng.stage("box%d" % l) - ref["box_out"][l]).max() / max(1.0, np.abs(ref["box_out"][l]).max()))
                          for l in range(3, 8)]
        # (label, box, prob) triples as sets: candidates whose scores agree to 1e-6 may swap places in the score order
        trip = lambda o: np.concatenate([o["final_labels"][:, None] * 10.0, o["final_boxes"], o["final_probs"][:, None]], 1).astype(np.float64)

        def sd(a, b):
            d = np.abs(trip(a)[:, None, :] - trip(b)[None, :, :]).max(-1)
            return float(max(d.min(1).max(), d.min(0).max()))
        rec["gpu_to_oracle32"], rec["gpu_to_exact"], rec["oracle32_to_exact"] = sd(out, ref), sd(out, ref64), sd(ref, ref64)
        rec["prob_maxabs"] = float(np.abs(np.sort(out["final_probs"]) - np.sort(ref["final_probs"])).max())
        rec["order_equal"] = bool(len(out["final_labels"]) == len(ref["final_labels"]) and
                                  np.array_equal(out["final_labels"], ref["final_labels"]) and np.array_equal(out["levels"], ref["levels"]))
        root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        os.makedirs(os.path.join(root, "gpurun_out"), exist_ok=True)
        with open(os.path.join(root, "gpurun_out", "baseline_parity.jsonl"), "a") as f:
            f.write(json.dumps(rec) + "\n")
        assert max(rec["c_rel"]) < 5e-5 and max(rec["fpn_rel"]) < 1e-4 and max(rec["cls_rel"]) < 1e-4, rec
        assert rec["final"] == rec["final_ref"] > 0
        np.testing.assert_array_equal(np.sort(out["final_labels"]), np.sort(ref["final_labels"]))
        np.testing.assert_array_equal(np.sort(out["levels"]), np.sort(ref["levels"]))
        assert rec["prob_maxabs"] <= 1e-5
        assert rec["gpu_to_exact"] <= 2e-2 and rec["gpu_to_exact"] <= 2.0 * rec["oracle32_to_exact"], rec
        if rec["order_equal"]:
            assert np.abs(out["fpn_box_feat"] - ref["fpn_box_feat"]).max() <= 1e-4 * max(1.0, np.abs(ref["fpn_box_feat"]).max())
    finally:
        eng.close()


def test_efficientdet_model_object_drop_in():
    # the reference call surface: models.get_model(config) -> EfficientDet; sess.run(fetches, feed_dict)
    from types import SimpleNamespace
    from object_detection_tracking_b200.backend import EfficientDet, Session, get_model
    from object_detection_tracking_b200.effdet_config import make_effdet_config
    from object_detection_tracking_b200.synth import synth_effdet_weights, synth_efficientnet_weights
    from oracle import effdet as oe
    from oracle import efficientnet as on
    config = SimpleNamespace(is_efficientdet=True, efficientdet_modelname="efficientdet-d0", short_edge_size=256, max_size=384,
                             efficientdet_min_level=3, efficientdet_max_level=7, efficientdet_max_detection_topk=5000,
                             result_score_thres=1e-4, result_per_im=100, use_partial_classes=True,
                             partial_classes=["person", "car", "bus", "truck", "bicycle"], is_load_from_pb=False)
    model = get_model(config, gpuid=0, controller="/cpu:0")
    assert isinstance(model, EfficientDet)
    cfg_full = make_effdet_config("efficientdet-d0", 256, 384)
    Wt = dict(synth_effdet_weights(cfg_full))
    Wt.update(synth_efficientnet_weights("efficientnet-b0"))
    with pytest.raises(RuntimeError):
        Session().run([model.final_boxes], feed_dict=model.get_feed_dict_forward(_frame(300, 500)))   # no weights yet
    model.set_weights(Wt)
    frame = _frame(300, 500).astype(np.float32)                      # the drivers feed the float32 resized frame
    sess = Session()
    boxes, labels, probs, feat = sess.run([model.final_boxes, model.final_labels, model.final_probs, model.fpn_box_feat],
                                          feed_dict=model.get_feed_dict_forward(frame))
    assert boxes.shape[1] == 4 and len(boxes) == len(labels) == len(probs) == len(feat) > 0
    assert labels.min() >= 1 and labels.max() <= 5                   # 1..len(partial_classes)
    # oracle with the same class gather (wrapper :398-404)
    idx = model.partial_class_idxs
    img, scale = on.preprocess(frame.astype(np.uint8), 256, 384)
    feats = on.forward(img, Wt, "efficientnet-b0")
    ref = oe.forward_from_features(cfg_full, Wt, feats, image_scale=scale, partial_class_idxs=idx)
    np.testing.assert_array_equal(labels, ref["final_labels"])
    assert np.abs(boxes - ref["final_boxes"]).max() <= 1e-3
    assert np.abs(probs - ref["final_probs"]).max() <= 5e-6
