"""Generates the committed golden fixtures by running the REFERENCE's own importable code
(/root/reference: generate_anchors.py, deep_sort/*).  Run once in the authoring container:
    python tests/golden/make_golden.py
The fixtures travel with the repo; /root/reference does not exist on the GPU box."""
import hashlib
import os
import sys

import numpy as np
import scipy.linalg  # noqa: F401  (import before the np.float shim, SURVEY.md 8c)
import scipy.optimize  # noqa: F401

np.float = float   # deep_sort/detection.py:30 uses the removed alias
np.int = int
sys.path.insert(0, "/root/reference")
HERE = os.path.dirname(os.path.abspath(__file__))

from generate_anchors import generate_anchors  # noqa: E402
from deep_sort import nn_matching  # noqa: E402
from deep_sort.detection import Detection  # noqa: E402
from deep_sort.tracker import Tracker  # noqa: E402


def anchors():
    out = {}
    for stride, size in zip((4, 8, 16, 32, 64), (32, 64, 128, 256, 512)):
        out["s%d" % stride] = generate_anchors(stride, scales=np.array([size], dtype=np.float64) / stride,
                                               ratios=np.array((0.5, 1, 2), dtype=np.float64))
    out["default"] = generate_anchors()
    np.savez(os.path.join(HERE, "anchors.npz"), **out)


def cosine():
    rng = np.random.default_rng(7)
    T, N, D, budget = 23, 37, 256, 5
    seg = [0]
    gal = []
    for t in range(T):
        n = int(rng.integers(1, budget + 1))
        gal.append(np.abs(rng.standard_normal((n, D))).astype(np.float32) + 0.1)
        seg.append(seg[-1] + n)
    dets = (np.abs(rng.standard_normal((N, D))) + 0.1).astype(np.float32)
    m = nn_matching.NearestNeighborDistanceMetric("cosine", 0.5, budget)
    m.samples = {t: list(gal[t]) for t in range(T)}
    cost = m.distance(dets, list(range(T)))
    np.savez(os.path.join(HERE, "deepsort_cosine.npz"), gallery=np.concatenate(gal), seg=np.asarray(seg, np.int32),
             dets=dets, cost=cost)


def euclid():
    """NearestNeighborDistanceMetric('euclidean') of the reference on signed features (nn_matching.py:5-28,57-75)."""
    rng = np.random.default_rng(17)
    T, N, D, budget = 9, 13, 128, 4
    m = nn_matching.NearestNeighborDistanceMetric("euclidean", 0.3, budget)
    feats = rng.standard_normal((60, D)).astype(np.float32)
    targets = np.asarray([i % T for i in range(60)])
    m.partial_fit(feats, targets, list(range(T)))
    dets = rng.standard_normal((N, D)).astype(np.float32)
    order = [4, 0, 2, 8, 1]
    np.savez(os.path.join(HERE, "deepsort_euclid.npz"), feats=feats, targets=targets, dets=dets,
             order=np.asarray(order), cost=m.distance(dets, order), budget=budget, T=T)


def tracker_run():
    """8 frames of synthetic moving objects through the reference Tracker (this fork's defaults,
    tracker.py:40) -> per-frame (track_id, tlwh) of confirmed tracks."""
    rng = np.random.default_rng(11)
    D, n_obj, n_frames = 256, 6, 10
    proto = np.abs(rng.standard_normal((n_obj, D))).astype(np.float32) + 0.05
    pos = rng.uniform(100, 900, (n_obj, 2))
    vel = rng.uniform(-12, 12, (n_obj, 2))
    size = rng.uniform(40, 120, (n_obj, 2))
    frames = []
    metric = nn_matching.NearestNeighborDistanceMetric("cosine", 0.5, 5)
    tracker = Tracker(metric)
    results = []
    for f in range(n_frames):
        dets_f = []
        for o in range(n_obj):
            if rng.uniform() < 0.15:
                continue   # missed detection
            p = pos[o] + vel[o] * f + rng.normal(0, 1.0, 2)
            feat = proto[o] + np.abs(rng.standard_normal(D)).astype(np.float32) * 0.05
            dets_f.append(np.concatenate([p, size[o], [0.9], feat]).astype(np.float32))
        dets_f = np.asarray(dets_f, dtype=np.float32).reshape(-1, 5 + D)
        frames.append(dets_f)
        detections = [Detection(r[:4], r[4], r[5:]) for r in dets_f]
        tracker.predict()
        tracker.update(detections)
        for t in tracker.tracks:
            if t.is_confirmed() and t.time_since_update <= 1:
                results.append([f, t.track_id] + t.to_tlwh().tolist())
    np.savez(os.path.join(HERE, "deepsort_tracker.npz"), results=np.asarray(results, dtype=np.float64),
             **{"frame%d" % i: fr for i, fr in enumerate(frames)})


def tracker_crowd():
    """90 frames, up to 22 objects with crossing paths, look-alike appearance vectors, misses, false positives, objects that
    leave (so that tracks age out after max_age = 60 misses) and late arrivals, through the reference Tracker + pre-tracker
    NMS inputs -> rows (frame, track_id, tlwh) of the confirmed tracks, plus every live track's (id, state, hits, age,
    time_since_update) after each frame (life-cycle bookkeeping)."""
    rng = np.random.default_rng(23)
    D, n_obj, n_frames = 32, 22, 90
    base = np.abs(rng.standard_normal((6, D))).astype(np.float32) + 0.05
    proto = np.stack([base[o % 6] + 0.35 * np.abs(rng.standard_normal(D)).astype(np.float32) for o in range(n_obj)])
    pos = rng.uniform(80, 1100, (n_obj, 2))
    vel = rng.uniform(-9, 9, (n_obj, 2))
    size = rng.uniform(30, 110, (n_obj, 2))
    t_in = np.where(rng.uniform(size=n_obj) < 0.3, rng.integers(5, 40, n_obj), 0)
    t_out = np.where(rng.uniform(size=n_obj) < 0.35, rng.integers(8, 25, n_obj), n_frames)
    metric = nn_matching.NearestNeighborDistanceMetric("cosine", 0.5, 5)
    tracker = Tracker(metric, max_iou_distance=0.5)
    frames, results, life = [], [], []
    for f in range(n_frames):
        rows = []
        for o in range(n_obj):
            if f < t_in[o] or f >= t_out[o] or rng.uniform() < 0.2:
                continue
            p = pos[o] + vel[o] * f + rng.normal(0, 1.5, 2)
            feat = proto[o] + np.abs(rng.standard_normal(D)).astype(np.float32) * 0.08
            rows.append(np.concatenate([p, size[o] * rng.uniform(0.95, 1.05, 2), [rng.uniform(0.5, 1.0)], feat]))
        for _ in range(rng.integers(0, 3)):       # false positives
            rows.append(np.concatenate([rng.uniform(50, 1100, 2), rng.uniform(30, 90, 2), [rng.uniform(0.3, 0.7)],
                                        np.abs(rng.standard_normal(D)) + 0.05]))
        dets_f = np.asarray(rows, dtype=np.float32).reshape(-1, 5 + D)
        frames.append(dets_f)
        tracker.predict()
        tracker.update([Detection(r[:4], r[4], r[5:]) for r in dets_f])
        for t in tracker.tracks:
            life.append([f, t.track_id, t.state, t.hits, t.age, t.time_since_update])
            if t.is_confirmed() and t.time_since_update <= 1:
                results.append([f, t.track_id] + t.to_tlwh().tolist())
    np.savez_compressed(os.path.join(HERE, "deepsort_tracker_crowd.npz"), results=np.asarray(results, dtype=np.float64),
                        life=np.asarray(life, dtype=np.int64), **{"frame%d" % i: fr for i, fr in enumerate(frames)})
    print("tracker_crowd: %d result rows, %d ids, max live tracks %d" % (
        len(results), len(set(int(r[1]) for r in results)), max(np.bincount(np.asarray(life)[:, 0]))))


def track_nms():
    """application_util/preprocessing.non_max_suppression on seeded boxes (with and without scores)."""
    import types
    sys.modules.setdefault("cv2", types.ModuleType("cv2"))     # preprocessing.py imports cv2 at module top, unused here
    from application_util import preprocessing
    rng = np.random.default_rng(5)
    out = {}
    for case in range(6):
        n = int(rng.integers(1, 40))
        boxes = np.concatenate([rng.uniform(0, 300, (n, 2)), rng.uniform(20, 120, (n, 2))], axis=1)
        scores = rng.uniform(0.1, 1.0, n)
        thr = float(rng.choice([0.3, 0.5, 0.85, 1.0]))
        out["boxes%d" % case] = boxes
        out["scores%d" % case] = scores
        out["thr%d" % case] = np.float64(thr)
        out["keep_scored%d" % case] = np.asarray(preprocessing.non_max_suppression(boxes, thr, scores), dtype=np.int64)
        out["keep_plain%d" % case] = np.asarray(preprocessing.non_max_suppression(boxes, thr), dtype=np.int64)
    np.savez(os.path.join(HERE, "track_nms.npz"), **out)


def osnet():
    """Reference torchreid osnet_x1_0 (eval) on seeded crops with the seeded synthetic state_dict."""
    import torch
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from object_detection_tracking_b200.synth import synth_osnet_state
    from torchreid.feature_extractor import FeatureExtractor
    from torchreid import distance
    state = synth_osnet_state(4321)
    ext = FeatureExtractor("osnet_x1_0", model_path="", device="cpu", verbose=False)
    sd = ext.model.state_dict()
    for k, v in state.items():
        assert tuple(sd[k].shape) == v.shape, (k, sd[k].shape, v.shape)
        sd[k].copy_(torch.from_numpy(v))
    ext.model.load_state_dict(sd)
    ext.model.eval()
    rng = np.random.default_rng(5)
    crops = [rng.integers(0, 256, (int(rng.integers(60, 300)), int(rng.integers(30, 160)), 3), dtype=np.uint8)
             for _ in range(6)]
    feats = ext(crops).numpy()
    # also the model on already-resized crops (isolates the network from PIL)
    resized = np.stack([np.asarray(ext.to_pil(c).resize((128, 256), 2)) for c in crops])   # 2 = PIL BILINEAR
    d_cos = distance.compute_distance_matrix(torch.from_numpy(feats[:4]), torch.from_numpy(feats[2:]), "cosine").numpy()
    d_euc = distance.compute_distance_matrix(torch.from_numpy(feats[:4]), torch.from_numpy(feats[2:]), "euclidean").numpy()
    # the crops are regenerated from the seed by the tests; their hashes pin that they are the same bytes
    np.savez_compressed(os.path.join(HERE, "osnet.npz"), feats=feats, resized=resized, d_cos=d_cos, d_euc=d_euc,
                        crop_shapes=np.array([c.shape for c in crops], np.int64),
                        crop_sha256=np.array([hashlib.sha256(c.tobytes()).hexdigest() for c in crops]))


def effdet_numpy():
    """The numpy halves of efficientdet/anchors.py (anchor grid, box decode, sigmoid) -- importable once the
    TensorFlow import at the top of the module is stubbed (TF itself is absent here; only numpy code is executed)."""
    from unittest.mock import MagicMock
    for m in ("tensorflow", "tensorflow.compat", "tensorflow.compat.v1", "tensorflow.compat.v2", "tensorflow.python",
              "tensorflow.python.tpu", "tensorflow.python.tpu.tpu_function", "absl", "absl.logging"):
        sys.modules.setdefault(m, MagicMock())
    from efficientdet import anchors as ra
    out = {}
    for tag, (h, w, scale) in {"a": (256, 384, 4.0), "b": (512, 640, 5.0)}.items():
        fs = [{"height": h, "width": w}]
        for _ in range(7):
            fs.append({"height": (fs[-1]["height"] - 1) // 2 + 1, "width": (fs[-1]["width"] - 1) // 2 + 1})
        cfgs = ra._generate_anchor_configs(fs, 3, 7, 3, [(1.0, 1.0), (1.4, 0.7), (0.7, 1.4)])
        out["anchors_" + tag] = ra._generate_anchor_boxes((h, w), scale, cfgs)       # float64 [N,4]
    rng = np.random.default_rng(11)
    anc = out["anchors_a"][rng.integers(0, out["anchors_a"].shape[0], 64)].astype(np.float32)
    codes = (rng.standard_normal((64, 4)) * 0.3).astype(np.float32)
    out["dec_anchors"], out["dec_codes"] = anc, codes
    out["dec_boxes"] = ra.decode_box_outputs(codes.swapaxes(0, 1), anc.swapaxes(0, 1))
    logits = (rng.standard_normal(64) * 3).astype(np.float32)
    out["sig_logits"], out["sig_scores"] = logits, ra.sigmoid(logits)
    # filter / repeat rounding of the backbone (efficientnet_model.py:137-159) for b0..b7
    from types import SimpleNamespace
    from efficientdet.backbone import efficientnet_model as em
    table = {"b0": (1.0, 1.0), "b1": (1.0, 1.1), "b2": (1.1, 1.2), "b3": (1.2, 1.4), "b4": (1.4, 1.8), "b5": (1.6, 2.2),
             "b6": (1.8, 2.6), "b7": (2.0, 3.1)}
    base_f, base_r = [32, 16, 24, 40, 80, 112, 192, 320, 1280], [1, 2, 3, 4]
    rf, rr = [], []
    for k in sorted(table):
        gp = SimpleNamespace(width_coefficient=table[k][0], depth_coefficient=table[k][1], depth_divisor=8, min_depth=None)
        rf.append([em.round_filters(f, gp) for f in base_f])
        rr.append([em.round_repeats(r, gp) for r in base_r])
    out["round_filters"], out["round_repeats"] = np.array(rf, np.int64), np.array(rr, np.int64)
    # COCO category table (class_ids.py:526-549)
    import class_ids as rc
    ids = sorted(rc.coco_id_mapping)
    out["coco_ids"] = np.array(ids, np.int64)
    out["coco_names"] = np.array([rc.coco_id_mapping[i] for i in ids])
    out["coco_dense"] = np.array([rc.coco_obj_class_to_id[rc.coco_id_mapping[i]] for i in ids], np.int64)
    np.savez_compressed(os.path.join(HERE, "effdet_numpy.npz"), **out)


if __name__ == "__main__":
    anchors()
    cosine()
    tracker_run()
    tracker_crowd()
    track_nms()
    osnet()
    effdet_numpy()
    print("golden fixtures written to", HERE)
