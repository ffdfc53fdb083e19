"""GPU parity of the section-8f widening that composes already-verified kernels (the tensor-core GEMM behind
b2_distance_matrix) with small new ones: TMOT embedding distance, the JDE tracker with its embedding cost on the GPU, and
the multi-camera track-pair cost (b2_track_pair_cost), device-side frame resize, given-box features, the detect -> track
loop.  First B200 run: round 2, 12/12 green (gpurun_out/widen_tests.log -> profiles/r2_first_gpu_call.txt)."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def cdist64(a, b):
    a, b = a.astype(np.float64), b.astype(np.float64)
    return np.sqrt(np.maximum(0.0, ((a[:, None, :] - b[None, :, :]) ** 2).sum(-1)))


def test_tmot_embedding_distance_matches_cdist(golden_dir):
    from object_detection_tracking_b200 import tmot
    g = np.load(os.path.join(golden_dir, "tmot_matching.npz"))
    got = tmot.embedding_distance(g["track_feats"], g["det_feats"])
    # unit vectors: d^2 = 2 - 2ab carries ~1e-7 absolute error, so d is good to ~1e-7 / d (3e-4 at d -> 0)
    assert np.abs(got - g["emb"]).max() < 1e-3
    far = g["emb"] > 0.1
    assert np.abs(got[far] - g["emb"][far]).max() < 5e-6
    rng = np.random.default_rng(2)
    a = rng.standard_normal((150, 512)).astype(np.float32)
    b = rng.standard_normal((90, 512)).astype(np.float32)
    assert np.abs(tmot.embedding_distance(a, b) - cdist64(a, b)).max() < 1e-3
    assert tmot.embedding_distance(np.zeros((0, 8), np.float32), b[:, :8]).shape == (0, 90)


def test_jde_tracker_on_gpu_reproduces_reference_ids(golden_dir):
    """Same 80-frame, two-tracker sequence as tests/test_tmot_cpu.py, embedding cost from the tensor cores."""
    from object_detection_tracking_b200.tmot import JDETracker, _IdGroup
    g = np.load(os.path.join(golden_dir, "tmot_jde.npz"))
    grp = _IdGroup()
    trackers = [JDETracker(0.5, track_max_second_lost=4.0, frame_gap=8., frame_rate=30., id_group=grp) for _ in range(2)]
    rows = []
    for f in range(80):
        for k, trk in enumerate(trackers):
            fr = g["s%d_f%d" % (k, f)]
            for t in trk.update([(r[:4].astype(np.float64), float(r[4]), r[5:].copy()) for r in fr]):
                rows.append([f, k, t.track_id] + t.tlwh.tolist())
    got = np.asarray(rows, dtype=np.float64)
    assert got.shape[0] == g["out"].shape[0]
    np.testing.assert_array_equal(got[:, :3], g["out"][:, :3])          # frame, tracker, track id: bit-exact
    assert np.abs(got[:, 3:7] - g["out"][:, 3:7]).max() < 1e-6
    for t in trackers:
        t.close()


def test_track_pair_cost_matches_reference(golden_dir):
    from object_detection_tracking_b200 import reid
    g = np.load(os.path.join(golden_dir, "reid_pairs.npz"))
    cams = []
    for name in ("c1", "c2"):
        cams.append({int(t): (g["%s_t%d_rows" % (name, t)], g["%s_t%d_feat" % (name, t)]) for t in g[name + "_ids"]})
    fd = reid.compute_feature_dist(cams[0], cams[1], g["spatial"])
    np.testing.assert_array_equal(fd == 999.0, g["feature"] == 999.0)
    scale = max(float((c[t][1].astype(np.float64) ** 2).sum(1).max()) for c in cams for t in c)
    assert np.abs(fd - g["feature"]).max() <= 2e-6 * scale
    got = reid.match_tracks(cams[0], cams[1], frame_offset=4, tol=50,
                            ignore_pairs=[list(g["ignore0"]), list(g["ignore1"])])
    ids1, ids2 = sorted(cams[0]), sorted(cams[1])
    assert got == [(ids1[i], ids2[int(j)]) for i, j in enumerate(g["x"]) if j >= 0]


def test_track_pair_cost_large_ungated():
    """50 x 40 tracks with 1..12 crops each, D = 512, no gate, plus empty tracks -> `fill`."""
    from object_detection_tracking_b200 import _lib
    rng = np.random.default_rng(9)
    N, M, D = 50, 40, 512
    ka, kb = rng.integers(1, 13, N), rng.integers(1, 9, M)
    ka[7] = 0
    kb[3] = 0
    sa = np.concatenate([[0], np.cumsum(ka)]).astype(np.int32)
    sb = np.concatenate([[0], np.cumsum(kb)]).astype(np.int32)
    a = rng.standard_normal((sa[-1], D)).astype(np.float32)
    b = rng.standard_normal((sb[-1], D)).astype(np.float32)
    out = np.zeros((N, M), np.float32)
    _lib.check(_lib.load().b2_track_pair_cost(0, _lib.ptr(a), _lib.ptr(sa), N, _lib.ptr(b), _lib.ptr(sb), M, D, None, 999.0, 1,
                                              _lib.ptr(out)), "b2_track_pair_cost")
    a64, b64 = a.astype(np.float64), b.astype(np.float64)
    full = (a64 ** 2).sum(1)[:, None] + (b64 ** 2).sum(1)[None, :] - 2 * a64 @ b64.T
    ref = np.full((N, M), 999.0)
    for i in range(N):
        for j in range(M):
            blk = full[sa[i]:sa[i + 1], sb[j]:sb[j + 1]]
            if blk.size:
                ref[i, j] = max(blk.min(), 0.0)
    assert (ref[7] == 999.0).all() and (ref[:, 3] == 999.0).all()
    assert np.abs(out - ref).max() <= 5e-6 * np.abs(full).max()


def test_resize_kernel_matches_oracle_and_cv2_fixture(golden_dir):
    """b2_resize_frames (the ingest resize alone) is bit-exact with the cv2-pinned oracle."""
    from object_detection_tracking_b200.engine import resize_frames
    from oracle import resize
    g = np.load(os.path.join(golden_dir, "resize_cv2.npz"))
    for k in range(6):
        nw, nh = (int(v) for v in g["size%d" % k])
        got = resize_frames(g["src%d" % k][None], nw, nh)[0]
        np.testing.assert_array_equal(got, g["dst%d" % k])
    rng = np.random.default_rng(4)
    src = rng.integers(0, 256, (2, 1080, 1920, 3)).astype(np.uint8)        # BASELINE frame source size, batch of 2
    got = resize_frames(src, 1280, 720)
    for b in range(2):
        np.testing.assert_array_equal(got[b], resize.resize_linear(src[b], 1280, 720))


def test_detect_with_device_resize_equals_host_resize_path():
    """b2_detect_host_resize(uint8 source frames) == b2_detect_host(oracle-resized float32 frames), bit for bit."""
    from object_detection_tracking_b200.config import make_config
    from object_detection_tracking_b200.engine import Detector, get_new_hw
    from object_detection_tracking_b200.synth import synth_frame, synth_weights
    from oracle import resize
    cfg = make_config(resnet_num_block=(1, 1, 2, 1), max_size=256, short_edge_size=144)
    src = np.stack([synth_frame(216, 384, s) for s in (3, 4)])                      # 1.5x larger than the network input
    nw, nh = get_new_hw(216, 384, 144, 256)
    assert (nw, nh) == (256, 144)
    det = Detector(cfg, 2, nh, nw, device=0, precision="split", use_cuda_graph=True)
    det.load_weights(synth_weights(cfg, 1234))
    a = det.detect_host_resize(src)
    a = {k: v.copy() for k, v in a.items()}
    b = det.detect_host(np.stack([resize.resize_linear(f, nw, nh) for f in src]))
    assert int(a["valid"].sum()) > 0
    for k in ("valid", "labels", "boxes", "probs"):
        np.testing.assert_array_equal(a[k], b[k])


def test_feature_aggregation_modes_match_host_aggregation():
    """feat_mode 1 / 2 / 3 (mean, max, "spatial": obj_detect_tracking_multi_queuer_tmot.py:511-525) computed on the device
    equal the same aggregation of the full [R,256,7,7] features done on the host."""
    from object_detection_tracking_b200.config import make_config
    from object_detection_tracking_b200.engine import Detector
    from object_detection_tracking_b200.synth import synth_frame, synth_weights
    H, W = 192, 256
    cfg = make_config(resnet_num_block=(1, 1, 2, 1), max_size=W, short_edge_size=H)
    det = Detector(cfg, 1, H, W, device=0, precision="split", use_cuda_graph=True)
    det.load_weights(synth_weights(cfg, 1234))
    frame = synth_frame(H, W, 5).astype(np.float32)[None]
    full = det.detect_host(frame, feat_mode=0)
    r = int(full["valid"][0])
    assert r > 0
    f = full["feat"][:r]
    mean = det.detect_host(frame, feat_mode=1)["feat"][:r]
    mx = det.detect_host(frame, feat_mode=2)["feat"][:r]
    sp = det.detect_host(frame, feat_mode=3)["feat"][:r]
    scale = float(np.abs(f).max())
    assert np.abs(mean - f.mean(axis=(2, 3))).max() <= 1e-6 * scale
    np.testing.assert_array_equal(mx, f.max(axis=(2, 3)))
    assert sp.shape == (r, 49) and np.abs(sp - f.mean(axis=1).reshape(r, 49)).max() <= 1e-5 * scale


def test_given_box_features_match_oracle():
    """RCNN_FPN_givenbox (models.py:1816-1967) through get_model_feat / Session.run: 130 boxes (two chunks of 100), some
    touching the frame border where the uncropped levels matter."""
    from object_detection_tracking_b200.backend import Session, get_model_feat
    from object_detection_tracking_b200.config import make_config
    from object_detection_tracking_b200.synth import synth_frame, synth_weights
    from oracle import frcnn
    H, W = 192, 256
    cfg = make_config(resnet_num_block=(1, 1, 2, 1), max_size=W, short_edge_size=H)
    Wt = synth_weights(cfg, 1234)
    frame = synth_frame(H, W, 5).astype(np.float32)
    rng = np.random.default_rng(6)
    xy = rng.uniform(0, [W - 20, H - 20], (130, 2))
    wh = rng.uniform(6, [W / 1.5, H / 1.5], (130, 2))
    boxes = np.concatenate([xy, np.minimum(xy + wh, [W, H])], 1).astype(np.float32)
    boxes[:4] = [[0, 0, W, H], [W - 30, H - 30, W, H], [0, H - 12, 40, H], [W - 9, 0, W, 50]]
    model = get_model_feat(cfg, gpuid=0)
    model.set_weights(Wt)
    got, = Session().run([model.final_box_features], feed_dict=model.get_feed_dict(frame, boxes))
    ref = frcnn.forward_givenbox(cfg, Wt, frame, boxes)
    assert got.shape == ref.shape == (130, 256)
    assert np.abs(got - ref).max() <= 2e-5 * np.abs(ref).max()
    assert Session().run([model.final_box_features], feed_dict=model.get_feed_dict(frame, np.zeros((0, 4))))[0].shape == (0, 256)


def test_pipelined_resize_ingest_equals_synchronous_call():
    """b2_submit_host_resize / b2_wait (two slots) == b2_detect_host_resize on the same uint8 source batches."""
    from object_detection_tracking_b200.config import make_config
    from object_detection_tracking_b200.engine import Detector
    from object_detection_tracking_b200.synth import synth_frame, synth_weights
    cfg = make_config(resnet_num_block=(1, 1, 2, 1), max_size=256, short_edge_size=144)
    det = Detector(cfg, 2, 144, 256, device=0, precision="split", use_cuda_graph=True)
    det.load_weights(synth_weights(cfg, 1234))
    batches = [np.stack([synth_frame(216, 384, 10 * j + i) for i in range(2)]) for j in range(3)]
    ref = [{k: v.copy() for k, v in det.detect_host_resize(b).items()} for b in batches]
    outs = [det.alloc_outputs(), det.alloc_outputs()]
    got = []
    det.submit_host_resize(batches[0], outs[0], 0)
    for j in range(1, 3):
        det.submit_host_resize(batches[j], outs[j & 1], j & 1)
        det.wait((j - 1) & 1)
        got.append({k: v.copy() for k, v in outs[(j - 1) & 1].items()})
    det.wait(0)
    got.append({k: v.copy() for k, v in outs[0].items()})
    for a, b in zip(got, ref):
        assert int(b["valid"].sum()) > 0
        for k in ("valid", "labels", "boxes", "probs"):
            np.testing.assert_array_equal(a[k], b[k])


def test_detect_then_track_loop_end_to_end():
    """The per-frame loop of obj_detect_tracking.py:597-696 with every piece swapped in: sess.run on the model object,
    create_obj_infos, pre-tracker NMS, native Tracker with the GPU appearance metric; and the TMOT variant
    (preprocess_detections + JDETracker).  The same frame is fed repeatedly, so every detection must keep its track id."""
    from object_detection_tracking_b200.backend import Session, get_model
    from object_detection_tracking_b200.config import make_config
    from object_detection_tracking_b200.synth import synth_frame, synth_weights
    from object_detection_tracking_b200.tmot import JDETracker, _IdGroup
    from object_detection_tracking_b200.tracking import (GpuNearestNeighborDistanceMetric, Tracker, create_obj_infos,
                                                         non_max_suppression, preprocess_detections)
    H, W = 192, 256
    cfg = make_config(resnet_num_block=(1, 1, 2, 1), max_size=W, short_edge_size=H)
    model = get_model(cfg, gpuid=0)
    model.set_weights(synth_weights(cfg, 1234))
    sess = Session()
    frame = synth_frame(H, W, 5).astype(np.float32)
    id2class = {i: "class%d" % i for i in range(1, cfg.num_class)}
    tracker = Tracker(GpuNearestNeighborDistanceMetric("cosine", 0.5, 5), max_iou_distance=0.5)
    jde = JDETracker(0.0, id_group=_IdGroup())
    seen, seen_jde, target = [], [], None
    for f in range(5):
        boxes, labels, probs, feats = sess.run([model.final_boxes, model.final_labels, model.final_probs, model.fpn_box_feat],
                                               feed_dict=model.get_feed_dict_forward(frame))
        assert len(feats) == len(boxes) > 0                                  # obj_detect_tracking.py:648
        if target is None:
            target = id2class[int(np.bincount(labels).argmax())]            # the most frequent class of this frame
        dets = create_obj_infos(f, boxes, probs, labels, feats, id2class, [target], 0.0, 0, 1.0)
        keep = non_max_suppression(np.array([d.tlwh for d in dets]), 0.85, np.array([d.confidence for d in dets]))
        dets = [dets[i] for i in keep]
        tracker.predict()
        tracker.update(dets)
        seen.append(sorted(t.track_id for t in tracker.tracks if t.is_confirmed() and t.time_since_update <= 1))
        tm = preprocess_detections(boxes, probs, labels, feats, id2class, [target], 0.0, 1.0)
        tm = [tm[i] for i in non_max_suppression(np.array([d[0] for d in tm]), 0.85, np.array([d[1] for d in tm]))]
        seen_jde.append(sorted(t.track_id for t in jde.update(tm)))
    n = len(dets)
    assert n > 0 and seen[1] == seen[-1] == list(range(1, n + 1))            # n_init = 1: confirmed at the first match
    assert seen_jde[0] == [] and seen_jde[1] == seen_jde[-1] == list(range(1, n + 1))   # activated at the second frame
    tracker.close()
    jde.close()


def test_distance_calls_from_the_persistent_workspace_equal_the_per_call_path():
    """The default grow-only workspace + cached GEMM plans behind b2_cosine_cost / b2_distance_matrix returns the same bits,
    across growing and shrinking shapes and both metrics, as each call made as the first call of a fresh process (a new
    workspace sized for that call alone, with no leftovers of earlier calls)."""
    import subprocess
    import sys
    import tempfile
    code = (
        "import numpy as np, sys; sys.path.insert(0, %r)\n"
        "from object_detection_tracking_b200.engine import cosine_cost\n"
        "from object_detection_tracking_b200.reid import compute_distance_matrix\n"
        "only = sys.argv[2] if len(sys.argv) > 2 else None   # run just this call\n"
        "rng = np.random.default_rng(0); out = {}\n"
        "for k, (T, per, N, D) in enumerate([(5, 3, 7, 64), (40, 5, 90, 256), (3, 2, 4, 256), (100, 5, 100, 256), (9, 4, 33, 48)]):\n"
        "    gal = np.abs(rng.standard_normal((T * per, D))).astype(np.float32) + 0.1\n"
        "    seg = (np.arange(T + 1) * per).astype(np.int32)\n"
        "    det = np.abs(rng.standard_normal((N, D))).astype(np.float32) + 0.1\n"
        "    calls = {'cos%%d' %% k: lambda: cosine_cost(gal, seg, det),\n"
        "             'euc%%d' %% k: lambda: compute_distance_matrix(gal, det, 'euclidean').numpy(),\n"
        "             'cdm%%d' %% k: lambda: compute_distance_matrix(det, gal, 'cosine').numpy()}\n"
        "    for name, call in calls.items():\n"
        "        if only in (None, name):\n"
        "            out[name] = call()\n"
        "np.savez(sys.argv[1], **out)\n") % os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    names = ["%s%d" % (kind, k) for k in range(5) for kind in ("cos", "euc", "cdm")]
    fresh = {}
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "reused.npz")
        subprocess.run([sys.executable, "-c", code, path], check=True, timeout=300)
        reused = dict(np.load(path))
        for name in names:
            path = os.path.join(tmp, name + ".npz")
            subprocess.run([sys.executable, "-c", code, path, name], check=True, timeout=300)
            fresh.update(np.load(path))
    assert set(reused) == set(fresh) == set(names)
    for k in names:
        np.testing.assert_array_equal(fresh[k], reused[k])


def test_euclidean_nearest_neighbor_metric():
    """NearestNeighborDistanceMetric('euclidean') (deep_sort/nn_matching.py:8-28,57-75,156-177): min over a track's gallery
    rows of the squared euclidean distance, clamped at 0."""
    from object_detection_tracking_b200.tracking import GpuNearestNeighborDistanceMetric
    rng = np.random.default_rng(14)
    D = 128
    m = GpuNearestNeighborDistanceMetric("euclidean", 0.3, budget=4)
    feats = rng.standard_normal((30, D)).astype(np.float32)
    m.partial_fit(feats, [i % 6 for i in range(30)], list(range(6)))          # budget keeps the last 4 per target
    q = rng.standard_normal((11, D)).astype(np.float32)
    got = m.distance(q, [4, 0, 2])
    ref = np.zeros((3, 11))
    for r, t in enumerate([4, 0, 2]):
        g = np.asarray(m.samples[t], dtype=np.float64)
        assert len(g) == 4
        d = (g * g).sum(1)[:, None] + (q.astype(np.float64) ** 2).sum(1)[None, :] - 2 * g @ q.astype(np.float64).T
        ref[r] = np.maximum(0.0, d.min(axis=0))
    assert got.shape == (3, 11) and got.dtype == np.float64
    assert np.abs(got - ref).max() <= 5e-6 * np.abs(ref).max()
    with pytest.raises(ValueError):
        GpuNearestNeighborDistanceMetric("manhattan", 0.3)
