"""ctypes binding of libb200det.so (include/b200det.h).  Loading never needs a GPU; every compute
entry point fails loudly (RuntimeError with b2_last_error()) instead of falling back to the CPU."""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int32, c_int64, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb200det.so")


class B2Config(ctypes.Structure):
    _fields_ = [
        ("batch", c_int32), ("height", c_int32), ("width", c_int32), ("input_dtype", c_int32),
        ("num_class", c_int32), ("resnet_blocks", c_int32 * 4), ("use_dilations", c_int32),
        ("class_agnostic", c_int32), ("rpn_topk", c_int32), ("result_per_im", c_int32),
        ("fpn_num_channel", c_int32), ("fc_head_dim", c_int32), ("precision", c_int32),
        ("conv_impl", c_int32), ("use_cuda_graph", c_int32),
        ("max_size", c_float), ("rpn_min_size", c_float), ("rpn_nms_thres", c_float),
        ("fastrcnn_nms_iou_thres", c_float), ("result_score_thres", c_float),
        ("anchor_strides", c_float * 5), ("anchor_sizes", c_float * 5), ("anchor_ratios", c_float * 3),
        ("bbox_reg_weights", c_float * 4), ("accum_chunk", c_int32), ("multi_semantics", c_int32),
        ("add_mask", c_int32),
    ]


class B2EffdetConfig(ctypes.Structure):
    _fields_ = [
        ("image_h", c_int32), ("image_w", c_int32), ("min_level", c_int32), ("max_level", c_int32),
        ("fpn_num_filters", c_int32), ("fpn_cell_repeats", c_int32), ("box_class_repeats", c_int32),
        ("num_classes", c_int32), ("num_scales", c_int32), ("num_aspects", c_int32),
        ("aspect_ratios", (c_float * 2) * 3), ("anchor_scale", c_float), ("fpn_weight_method", c_int32),
        ("backbone_channels", c_int32 * 3), ("max_detection_topk", c_int32), ("result_per_im", c_int32),
        ("nms_iou_threshold", c_float), ("result_score_thres", c_float), ("precision", c_int32), ("backbone", c_int32),
    ]


# every symbol include/b200det.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("b2_last_error", c_char_p, []),
    ("b2_version", c_int, []),
    ("b2_create", c_int, [POINTER(c_void_p), c_int, POINTER(B2Config)]),
    ("b2_destroy", None, [c_void_p]),
    ("b2_load_weights", c_int, [c_void_p, POINTER(c_char_p), POINTER(c_void_p), POINTER(c_int64), c_int]),
    ("b2_detect", c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int]),
    ("b2_detect_host", c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int]),
    ("b2_detect_host_resize", c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int]),
    ("b2_resize_frames", c_int, [c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    ("b2_submit_host", c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int]),
    ("b2_wait", c_int, [c_void_p, c_int]),
    ("b2_submit_host_resize", c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int]),
    ("b2_box_features", c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    ("b2_get_masks", c_int, [c_void_p, c_void_p, c_int64]),
    ("b2_stage_shape", c_int, [c_void_p, c_char_p, POINTER(c_int64), POINTER(c_int32)]),
    ("b2_get_stage", c_int, [c_void_p, c_char_p, c_void_p, c_int64]),
    ("b2_set_stage", c_int, [c_void_p, c_char_p, c_void_p, c_int64]),
    ("b2_run_phases", c_int, [c_void_p, c_int]),
    ("b2_phase_times", c_int, [c_void_p, POINTER(c_float)]),
    ("b2_kernel_launches", c_int, [c_void_p]),
    ("b2_num_steps", c_int, [c_void_p]),
    ("b2_profile_steps", c_int, [c_void_p, c_int, POINTER(c_float), c_int, POINTER(c_int)]),
    ("b2_step_info", c_int, [c_void_p, c_int, ctypes.c_char_p, c_int, POINTER(ctypes.c_double), POINTER(ctypes.c_double), POINTER(c_int)]),
    ("b2_cosine_cost", c_int, [c_int, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p]),
    ("b2_tracker_create", c_int, [POINTER(c_void_p), c_int, ctypes.c_double, c_int, c_int, ctypes.c_double, c_int, c_int, c_int]),
    ("b2_tracker_destroy", None, [c_void_p]),
    ("b2_tracker_set_cost_fn", c_int, [c_void_p, c_void_p, c_void_p]),
    ("b2_tracker_predict", c_int, [c_void_p]),
    ("b2_tracker_update", c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int]),
    ("b2_tracker_num_tracks", c_int, [c_void_p]),
    ("b2_tracker_get_tracks", c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    ("b2_linear_sum_assignment", c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    ("b2_track_nms", c_int, [c_void_p, c_void_p, c_int, ctypes.c_double, c_void_p]),
    ("b2_lapjv", c_int, [c_void_p, c_int, c_int, ctypes.c_double, c_void_p, c_void_p, POINTER(ctypes.c_double)]),
    ("b2_tmot_iou_distance", c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p]),
    ("b2_tmot_fuse_motion", c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, ctypes.c_double]),
    ("b2_tmot_embedding_distance", c_int, [c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p]),
    ("b2_jde_create", c_int, [POINTER(c_void_p), c_int] + [ctypes.c_double] * 8 + [c_int, c_int, c_void_p]),
    ("b2_jde_destroy", None, [c_void_p]),
    ("b2_jde_set_cost_fn", c_int, [c_void_p, c_void_p, c_void_p]),
    ("b2_jde_reset", c_int, [c_void_p]),
    ("b2_jde_reset_ids", c_int, [c_void_p]),
    ("b2_jde_update", c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int]),
    ("b2_jde_get_tracks", c_int, [c_void_p, c_int, c_int] + [c_void_p] * 12),
    ("b2_reid_create", c_int, [POINTER(c_void_p), c_int, c_int, c_int]),
    ("b2_reid_create_model", c_int, [POINTER(c_void_p), c_int, c_int, c_int, c_int]),
    ("b2_reid_destroy", None, [c_void_p]),
    ("b2_reid_load_weights", c_int, [c_void_p, POINTER(c_char_p), POINTER(c_void_p), POINTER(c_int64), c_int]),
    ("b2_reid_embed", c_int, [c_void_p, c_void_p, c_int, c_void_p]),
    ("b2_reid_embed_dev", c_int, [c_void_p, c_void_p, c_int, c_void_p]),
    ("b2_reid_feat_dim", c_int, [c_void_p]),
    ("b2_reid_num_launches", c_int, [c_void_p]),
    ("b2_reid_get_activation", c_int, [c_void_p, c_char_p, c_void_p, c_int64, POINTER(c_int64)]),
    ("b2_effdet_create", c_int, [POINTER(c_void_p), POINTER(B2EffdetConfig), c_int]),
    ("b2_effdet_destroy", None, [c_void_p]),
    ("b2_effdet_load_weights", c_int, [c_void_p, POINTER(c_char_p), POINTER(c_void_p), POINTER(c_int64), c_int]),
    ("b2_effdet_run_features", c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_float] + [c_void_p] * 6),
    ("b2_effdet_detect", c_int, [c_void_p, c_void_p, c_int, c_int] + [c_void_p] * 7),
    ("b2_effdet_get_stage", c_int, [c_void_p, c_char_p, c_void_p, c_int64, POINTER(c_int64)]),
    ("b2_effdet_num_launches", c_int, [c_void_p]),
    ("b2_effdet_profile_steps", c_int, [c_void_p, c_int, POINTER(c_float), c_int, POINTER(c_int)]),
    ("b2_effdet_step_info", c_int, [c_void_p, c_int, ctypes.c_char_p, c_int, POINTER(ctypes.c_double), POINTER(ctypes.c_double), POINTER(c_int)]),
    ("b2_distance_matrix", c_int, [c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    ("b2_track_pair_cost", c_int, [c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_float, c_int, c_void_p]),
    ("b2_track_pair_cost_dev", c_int, [c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_float, c_int, c_void_p]),
    ("b2_gallery_create", c_int, [c_int, c_void_p, c_int, c_int, POINTER(c_void_p), c_void_p]),
    ("b2_gallery_open", c_int, [c_int, c_void_p, POINTER(c_void_p)]),
    ("b2_gallery_close", c_int, [c_int, c_void_p]),
    ("b2_gallery_free", c_int, [c_int, c_void_p]),
    ("b2_track_spatial_dist", c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, ctypes.c_double, c_void_p]),
    ("b2_op_conv2d", c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p] + [c_int] * 19 + [c_void_p]),
    ("b2_conv_pair_launches", c_int64, []),
]

PHASES = dict(BACKBONE=1, FPN=2, RPN_HEAD=4, PROPOSALS=8, ROI=16, HEAD_FC=32, POST=64, BOX_FEAT=128, ALL=255)
PHASE_NAMES = ["backbone", "fpn", "rpn_head", "proposals", "roi", "head_fc", "post", "box_feat"]

_lib = None


def load(build_if_missing: bool = True) -> ctypes.CDLL:
    """Load (building in-tree if needed) libb200det.so and declare all prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        if not build_if_missing:
            raise RuntimeError("libb200det.so is not built: run `python -m object_detection_tracking_b200.build`")
        from . import build as _build
        _build.build()
    lib = ctypes.CDLL(LIB_PATH)
    for name, res, args in SYMBOLS:
        fn = getattr(lib, name)          # AttributeError if the export is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = "libb200det"):
    if rc != 0:
        msg = load().b2_last_error()
        raise RuntimeError("%s failed: %s" % (what, msg.decode() if msg else "unknown error"))


def ptr(a) -> c_void_p:
    """Raw pointer of a numpy array / torch tensor / None."""
    if a is None:
        return c_void_p(0)
    if isinstance(a, np.ndarray):
        return c_void_p(a.ctypes.data)
    return c_void_p(a.data_ptr())          # torch.Tensor


def make_config(cfg, batch: int, height: int, width: int, input_dtype: str = "float32", precision: str = "split",
                conv_impl: str = "tcgen05", use_cuda_graph: bool = True, multi_semantics: bool = False,
                accum_chunk: int = 0) -> B2Config:
    """Translate the reference-style namespace (config.py / obj_detect_tracking.py:236-389)."""
    c = B2Config()
    c.batch, c.height, c.width = int(batch), int(height), int(width)
    c.input_dtype = {"float32": 0, "uint8": 1}[input_dtype]
    c.num_class = int(cfg.num_class)
    for i, v in enumerate(cfg.resnet_num_block):
        c.resnet_blocks[i] = int(v)
    c.use_dilations = int(bool(cfg.use_dilations))
    c.class_agnostic = int(bool(getattr(cfg, "use_frcnn_class_agnostic", False)))
    c.rpn_topk = int(cfg.rpn_test_post_nms_topk)
    c.result_per_im = int(cfg.result_per_im)
    c.fpn_num_channel = int(cfg.fpn_num_channel)
    c.fc_head_dim = int(cfg.fpn_frcnn_fc_head_dim)
    c.precision = {"fp16": 0, "split": 1}[precision]
    c.conv_impl = {"tcgen05": 0, "simt": 1}[conv_impl]
    c.use_cuda_graph = int(bool(use_cuda_graph))
    c.max_size = float(cfg.max_size)
    c.rpn_min_size = float(cfg.rpn_min_size)
    c.rpn_nms_thres = float(cfg.rpn_proposal_nms_thres)
    c.fastrcnn_nms_iou_thres = float(cfg.fastrcnn_nms_iou_thres)
    c.result_score_thres = float(cfg.result_score_thres)
    for i in range(5):
        c.anchor_strides[i] = float(cfg.anchor_strides[i])
        c.anchor_sizes[i] = float(cfg.anchor_sizes[i])
    for i in range(3):
        c.anchor_ratios[i] = float(cfg.anchor_ratios[i])
    for i in range(4):
        c.bbox_reg_weights[i] = float(cfg.fastrcnn_bbox_reg_weights[i])
    c.multi_semantics = int(bool(multi_semantics))
    c.accum_chunk = int(accum_chunk)
    c.add_mask = int(bool(getattr(cfg, "add_mask", False)))
    return c
