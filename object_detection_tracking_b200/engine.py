"""Python owner of a b2_ctx: the thin host layer above the C ABI (ctypes only; torch/numpy arrays are
just buffers).  One Detector = one device = one fixed (batch, H, W) launch plan."""
from __future__ import annotations

import ctypes
from ctypes import c_char_p, c_float, c_int32, c_int64, c_void_p

import numpy as np

from . import _lib
from .config import normalize_config


class Detector:
    def __init__(self, cfg, batch: int, height: int, width: int, device: int = 0, input_dtype: str = "float32",
                 precision: str = "split", conv_impl: str = "tcgen05", use_cuda_graph: bool = True,
                 multi_semantics: bool = False, accum_chunk: int = 0):
        self.lib = _lib.load()
        self.cfg = normalize_config(cfg)
        self.batch, self.height, self.width = int(batch), int(height), int(width)
        self.device = int(device)
        self.input_dtype = input_dtype
        self.precision = precision
        self._c = _lib.make_config(self.cfg, batch, height, width, input_dtype, precision, conv_impl, use_cuda_graph,
                                   multi_semantics, accum_chunk)
        self._ctx = c_void_p(0)
        _lib.check(self.lib.b2_create(ctypes.byref(self._ctx), self.device, ctypes.byref(self._c)), "b2_create")
        self.R = int(self.cfg.result_per_im)
        self.C = int(self.cfg.fpn_num_channel)
        self._pinned = None

    # -- lifetime ---------------------------------------------------------------------------------
    def close(self):
        if getattr(self, "_ctx", None) is not None and self._ctx.value:
            self.lib.b2_destroy(self._ctx)
            self._ctx = c_void_p(0)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- weights ----------------------------------------------------------------------------------
    def load_weights(self, weights: dict):
        """`weights`: name -> float32 ndarray in the reference's Tensorpack-npz naming."""
        names = sorted(weights.keys())
        arrs = [np.ascontiguousarray(weights[k], dtype=np.float32) for k in names]
        n = len(names)
        c_names = (c_char_p * n)(*[k.encode() for k in names])
        c_data = (c_void_p * n)(*[a.ctypes.data for a in arrs])
        c_numel = (c_int64 * n)(*[a.size for a in arrs])
        _lib.check(self.lib.b2_load_weights(self._ctx, c_names, c_data, c_numel, n), "b2_load_weights")

    # -- the hot call -----------------------------------------------------------------------------
    def _np_dtype(self):
        return np.uint8 if self.input_dtype == "uint8" else np.float32

    def alloc_outputs(self, feat_mode: int = 0, pinned: bool = False):
        B, R, C = self.batch, self.R, self.C
        shapes = dict(boxes=((B, R, 4), np.float32), probs=((B, R), np.float32), labels=((B, R), np.int32),
                      valid=((B,), np.int32),
                      feat=({0: (B * R, C, 7, 7), 1: (B * R, C), 2: (B * R, C), 3: (B * R, 49)}[feat_mode], np.float32))
        if pinned:
            import torch
            tmap = {np.float32: torch.float32, np.int32: torch.int32}
            return {k: torch.empty(s, dtype=tmap[d]).pin_memory() for k, (s, d) in shapes.items()}
        return {k: np.empty(s, dtype=d) for k, (s, d) in shapes.items()}

    def detect_host(self, frames, out: dict | None = None, feat_mode: int = 0, want_feat: bool = True):
        """frames: [B,H,W,3] host array (numpy or pinned torch) of the configured dtype.  Returns dict of
        host arrays (boxes [B,100,4], probs, labels, valid, feat)."""
        if isinstance(frames, np.ndarray):
            frames = np.ascontiguousarray(frames, dtype=self._np_dtype())
            assert frames.shape == (self.batch, self.height, self.width, 3), frames.shape
        if out is None:
            out = self.alloc_outputs(feat_mode)
        _lib.check(self.lib.b2_detect_host(self._ctx, _lib.ptr(frames), _lib.ptr(out["boxes"]), _lib.ptr(out["probs"]),
                                           _lib.ptr(out["labels"]), _lib.ptr(out["valid"]),
                                           _lib.ptr(out["feat"]) if want_feat else c_void_p(0), feat_mode),
                   "b2_detect_host")
        return out

    def detect_host_resize(self, frames_u8, out: dict | None = None, feat_mode: int = 0, want_feat: bool = True):
        """Source-resolution uint8 frames [B,h,w,3] (BGR): upload, resize on the device to the configured height x width
        (cv2.resize INTER_LINEAR arithmetic, nn.py:1540-1545), then the pass.  Needs input_dtype="float32"."""
        frames_u8 = np.ascontiguousarray(frames_u8, dtype=np.uint8)
        assert frames_u8.ndim == 4 and frames_u8.shape[0] == self.batch and frames_u8.shape[3] == 3, frames_u8.shape
        if out is None:
            out = self.alloc_outputs(feat_mode)
        _lib.check(self.lib.b2_detect_host_resize(self._ctx, _lib.ptr(frames_u8), int(frames_u8.shape[1]),
                                                  int(frames_u8.shape[2]), _lib.ptr(out["boxes"]), _lib.ptr(out["probs"]),
                                                  _lib.ptr(out["labels"]), _lib.ptr(out["valid"]),
                                                  _lib.ptr(out["feat"]) if want_feat else c_void_p(0), feat_mode),
                   "b2_detect_host_resize")
        return out

    def box_features(self, frame, boxes) -> np.ndarray:
        """RCNN_FPN_givenbox (models.py:1816-1967): [n, 256] mean-pooled ROI features of the given boxes on one frame
        (batch-1 context)."""
        frame = np.ascontiguousarray(frame, dtype=self._np_dtype())
        assert frame.shape == (self.height, self.width, 3), frame.shape
        boxes = np.ascontiguousarray(boxes, dtype=np.float32).reshape(-1, 4)
        out = np.empty((len(boxes), self.C), dtype=np.float32)
        _lib.check(self.lib.b2_box_features(self._ctx, _lib.ptr(frame), _lib.ptr(boxes), len(boxes), _lib.ptr(out)),
                   "b2_box_features")
        return out

    def get_masks(self) -> np.ndarray:
        """final_masks of the last pass (config.add_mask): [B, result_per_im, 28, 28] float32 (models.py:958-961)."""
        out = np.empty((self.batch, int(self.cfg.result_per_im), 28, 28), dtype=np.float32)
        _lib.check(self.lib.b2_get_masks(self._ctx, _lib.ptr(out), out.nbytes), "b2_get_masks")
        return out

    def submit_host(self, frames, out: dict, slot: int, feat_mode: int = 0, want_feat: bool = True):
        """Asynchronous detect_host: enqueue upload + pass + download for `slot` (0/1) and return; `frames` and the
        arrays of `out` must stay alive (pinned for real overlap) until wait(slot).  Streaming drivers alternate slots
        so that the upload of the next batch overlaps the pass of the current one."""
        if isinstance(frames, np.ndarray):
            frames = np.ascontiguousarray(frames, dtype=self._np_dtype())     # a copy only when the caller's array needs one
            assert frames.shape == (self.batch, self.height, self.width, 3), frames.shape
        if not hasattr(self, "_inflight"):
            self._inflight = {}
        self._inflight[int(slot)] = (frames, out)                             # keep the buffers alive until wait()
        _lib.check(self.lib.b2_submit_host(self._ctx, _lib.ptr(frames), _lib.ptr(out["boxes"]), _lib.ptr(out["probs"]),
                                           _lib.ptr(out["labels"]), _lib.ptr(out["valid"]),
                                           _lib.ptr(out["feat"]) if want_feat else c_void_p(0), feat_mode, int(slot)),
                   "b2_submit_host")

    def submit_host_resize(self, frames_u8, out: dict, slot: int, feat_mode: int = 0, want_feat: bool = True):
        """submit_host for uint8 source frames [B,h,w,3] that are resized on the device (detect_host_resize, pipelined)."""
        if isinstance(frames_u8, np.ndarray):
            frames_u8 = np.ascontiguousarray(frames_u8, dtype=np.uint8)
        assert frames_u8.shape[0] == self.batch and frames_u8.shape[3] == 3, frames_u8.shape
        if not hasattr(self, "_inflight"):
            self._inflight = {}
        self._inflight[int(slot)] = (frames_u8, out)
        _lib.check(self.lib.b2_submit_host_resize(self._ctx, _lib.ptr(frames_u8), int(frames_u8.shape[1]),
                                                  int(frames_u8.shape[2]), _lib.ptr(out["boxes"]), _lib.ptr(out["probs"]),
                                                  _lib.ptr(out["labels"]), _lib.ptr(out["valid"]),
                                                  _lib.ptr(out["feat"]) if want_feat else c_void_p(0), feat_mode, int(slot)),
                   "b2_submit_host_resize")

    def wait(self, slot: int):
        _lib.check(self.lib.b2_wait(self._ctx, int(slot)), "b2_wait")
        getattr(self, "_inflight", {}).pop(int(slot), None)

    def detect_device(self, frames_dev, out_dev: dict | None = None, feat_mode: int = 0, sync: bool = True):
        """frames_dev / out_dev: torch CUDA tensors (or None to leave results in the context)."""
        o = out_dev or {}
        _lib.check(self.lib.b2_detect(self._ctx, _lib.ptr(frames_dev), _lib.ptr(o.get("boxes")),
                                      _lib.ptr(o.get("probs")), _lib.ptr(o.get("labels")), _lib.ptr(o.get("valid")),
                                      _lib.ptr(o.get("feat")), feat_mode, int(sync)), "b2_detect")
        return out_dev

    # -- stage access (parity tests) ----------------------------------------------------------------
    def stage_shape(self, name: str):
        shape = (c_int64 * 4)()
        dt = c_int32(0)
        _lib.check(self.lib.b2_stage_shape(self._ctx, name.encode(), shape, ctypes.byref(dt)), "b2_stage_shape")
        return tuple(int(v) for v in shape), (np.int32 if dt.value == 1 else np.float32)

    def get_stage(self, name: str) -> np.ndarray:
        shape, dt = self.stage_shape(name)
        a = np.empty(shape, dtype=dt)
        _lib.check(self.lib.b2_get_stage(self._ctx, name.encode(), _lib.ptr(a), a.nbytes), "b2_get_stage")
        return a

    def set_stage(self, name: str, value: np.ndarray):
        if name == "image":
            a = np.ascontiguousarray(value, dtype=self._np_dtype())
        else:
            _, dt = self.stage_shape(name)
            a = np.ascontiguousarray(value, dtype=dt)
        _lib.check(self.lib.b2_set_stage(self._ctx, name.encode(), _lib.ptr(a), a.nbytes), "b2_set_stage")

    def run_phases(self, mask: int = 255):
        _lib.check(self.lib.b2_run_phases(self._ctx, int(mask)), "b2_run_phases")

    def phase_times(self) -> dict:
        ms = (c_float * 8)()
        _lib.check(self.lib.b2_phase_times(self._ctx, ms), "b2_phase_times")
        return {n: float(ms[i]) for i, n in enumerate(_lib.PHASE_NAMES)}

    def kernel_launches(self) -> int:
        return int(self.lib.b2_kernel_launches(self._ctx))

    def profile_steps(self, reps: int = 3) -> list:
        """Per launch group: dict(name, kind, ms, flops, bytes) -- device time from CUDA events."""
        n = int(self.lib.b2_num_steps(self._ctx))
        ms = (c_float * n)()
        nout = ctypes.c_int(0)
        _lib.check(self.lib.b2_profile_steps(self._ctx, int(reps), ms, n, ctypes.byref(nout)), "b2_profile_steps")
        out = []
        buf = ctypes.create_string_buffer(256)
        for i in range(nout.value):
            fl, by, kind = ctypes.c_double(0), ctypes.c_double(0), ctypes.c_int(0)
            _lib.check(self.lib.b2_step_info(self._ctx, i, buf, 256, ctypes.byref(fl), ctypes.byref(by),
                                             ctypes.byref(kind)), "b2_step_info")
            out.append(dict(name=buf.value.decode(), kind=kind.value, ms=float(ms[i]), flops=fl.value, bytes=by.value))
        return out


def cosine_cost(gallery: np.ndarray, seg_offsets: np.ndarray, dets: np.ndarray, device: int = 0,
                precision: str = "split") -> np.ndarray:
    """[T, N] appearance cost = per-track min over gallery rows of (1 - cosine) on the GPU."""
    lib = _lib.load()
    gallery = np.ascontiguousarray(gallery, dtype=np.float32)
    dets = np.ascontiguousarray(dets, dtype=np.float32)
    seg = np.ascontiguousarray(seg_offsets, dtype=np.int32)
    T = seg.shape[0] - 1
    N, D = dets.shape
    cost = np.zeros((T, N), dtype=np.float32)
    if T == 0 or N == 0:
        return cost
    _lib.check(lib.b2_cosine_cost(device, _lib.ptr(gallery), _lib.ptr(seg), T, _lib.ptr(dets), N, D,
                                  {"fp16": 0, "split": 1}[precision], _lib.ptr(cost)), "b2_cosine_cost")
    return cost


def op_conv2d(x, w, bias=None, res=None, stride=1, dil=1, pad=(0, 0, 0, 0), relu=False, res_shift=0,
              impl="tcgen05", split=True, a_mode=-1, epi_mode=-1, device=0) -> np.ndarray:
    """Single convolution through the C ABI (NHWC activations, HWIO kernel) -- used by the kernel tests."""
    lib = _lib.load()
    x = np.ascontiguousarray(x, dtype=np.float32)
    w = np.ascontiguousarray(w, dtype=np.float32)
    B, H, W, Cin = x.shape
    R, S, _, Cout = w.shape
    pt, pb, pl, pr = pad
    Ho = (H + pt + pb - ((R - 1) * dil + 1)) // stride + 1
    Wo = (W + pl + pr - ((S - 1) * dil + 1)) // stride + 1
    out = np.zeros((B, Ho, Wo, Cout), dtype=np.float32)
    b = None if bias is None else np.ascontiguousarray(bias, dtype=np.float32)
    r = None if res is None else np.ascontiguousarray(res, dtype=np.float32)
    _lib.check(lib.b2_op_conv2d(device, _lib.ptr(x), _lib.ptr(w), _lib.ptr(b), _lib.ptr(r), B, H, W, Cin, R, S, Cout,
                                stride, dil, pt, pb, pl, pr, int(relu), int(res_shift),
                                {"tcgen05": 0, "simt": 1}[impl], int(split), int(a_mode), int(epi_mode),
                                _lib.ptr(out)),
               "b2_op_conv2d")
    return out


def get_new_hw(h, w, size, max_size):
    """nn.py:1548-1560: (neww, newh) of resizeImage for an h x w frame."""
    scale = size * 1.0 / min(h, w)
    if h < w:
        newh, neww = size, scale * w
    else:
        newh, neww = scale * h, size
    if max(newh, neww) > max_size:
        scale = max_size * 1.0 / max(newh, neww)
        newh = newh * scale
        neww = neww * scale
    return int(neww + 0.5), int(newh + 0.5)


def resize_frames(frames_u8, new_w, new_h, device=0):
    """The ingest resize alone: uint8 [n,h,w,3] -> float32 [n,new_h,new_w,3] on the GPU (b2_resize_frames)."""
    frames_u8 = np.ascontiguousarray(frames_u8, dtype=np.uint8)
    n, h, w, _ = frames_u8.shape
    out = np.empty((n, int(new_h), int(new_w), 3), dtype=np.float32)
    _lib.check(_lib.load().b2_resize_frames(int(device), _lib.ptr(frames_u8), n, h, w, int(new_h), int(new_w), _lib.ptr(out)),
               "b2_resize_frames")
    return out
