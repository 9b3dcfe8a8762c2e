"""Thin Python handle over the C-ABI engine (include/yolonano_b200.h).

PyTorch is used here only for device memory and the current stream; every
computation happens inside libyolonano_b200.so.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence, Tuple

import torch

from . import _lib
from .topology import conv_table, num_anchor_boxes


class EngineError(RuntimeError):
    pass


def _ptr(t: Optional[torch.Tensor]) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


def _stream_ptr(device: torch.device) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


class Engine:
    """One engine per (GPU, stream).  Not thread-safe (same as the C handle)."""

    def __init__(self, device: torch.device, input_size: int, num_classes: int,
                 anchor_size: Sequence[Sequence[float]], conf_thresh: float = 0.001,
                 nms_thresh: float = 0.5, diou_nms: bool = False,
                 gemm_mode: int = _lib.GEMM_TC_3XTF32, max_batch: int = 1):
        self.lib = _lib.load()
        device = torch.device(device)
        if device.type != "cuda":
            raise EngineError("the B200 engine only runs on a CUDA device (no CPU fallback)")
        self.device = torch.device("cuda", device.index if device.index is not None
                                   else torch.cuda.current_device())
        flat = [float(v) for wh in anchor_size for v in wh]
        if len(flat) != 18:
            raise EngineError("anchor_size must hold 9 [w,h] pairs (3 levels x 3 anchors)")
        cfg = _lib.YnbConfig()
        cfg.abi_version = _lib.YNB_ABI_VERSION
        cfg.device = self.device.index
        cfg.input_size = int(input_size)
        cfg.num_classes = int(num_classes)
        cfg.num_anchors = 3
        cfg.anchors = (C.c_float * 18)(*flat)
        cfg.conf_thresh = float(conf_thresh)
        cfg.nms_thresh = float(nms_thresh)
        cfg.diou_nms = int(bool(diou_nms))
        cfg.gemm_mode = int(gemm_mode)
        cfg.max_batch = int(max_batch)
        self.num_classes = int(num_classes)
        self.input_size = int(input_size)
        self.table = conv_table(self.num_classes)
        self._h = C.c_void_p()
        rc = self.lib.ynb_create(C.byref(cfg), C.byref(self._h))
        if rc != _lib.YNB_OK:
            msg = self.lib.ynb_last_error(None)
            self._h = C.c_void_p()
            raise EngineError(f"ynb_create failed ({rc}): {msg.decode() if msg else '?'}")

    # -- plumbing -----------------------------------------------------------------
    def _check(self, rc: int, what: str):
        if rc != _lib.YNB_OK:
            msg = self.lib.ynb_last_error(self._h)
            raise EngineError(f"{what} failed ({rc}): {msg.decode() if msg else '?'}")

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self.lib.ynb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def num_boxes(self) -> int:
        return int(self.lib.ynb_num_boxes(self._h))

    @property
    def launch_count(self) -> int:
        return int(self.lib.ynb_launch_count(self._h))

    def workspace_bytes(self, batch: int) -> int:
        return int(self.lib.ynb_workspace_bytes(self._h, batch))

    def set_grid(self, input_size: int):
        self._check(self.lib.ynb_set_grid(self._h, int(input_size)), "ynb_set_grid")
        self.input_size = int(input_size)

    def set_thresholds(self, conf: float, nms: float, diou: bool):
        self._check(self.lib.ynb_set_thresholds(self._h, float(conf), float(nms), int(bool(diou))),
                    "ynb_set_thresholds")

    def set_gemm_mode(self, mode: int):
        self._check(self.lib.ynb_set_gemm_mode(self._h, int(mode)), "ynb_set_gemm_mode")

    # -- weights ------------------------------------------------------------------
    def load_weights(self, fused: Dict[str, Tuple[torch.Tensor, torch.Tensor]]):
        """`fused[name] = (W [cout,cin/g,k,k], b [cout])`, BN already folded, any device."""
        for spec in self.table:
            w, b = fused[spec.name]
            w = w.detach().to("cpu", torch.float32).contiguous()
            b = b.detach().to("cpu", torch.float32).contiguous()
            if tuple(w.shape) != spec.weight_shape() or b.numel() != spec.cout:
                raise EngineError(f"{spec.name}: weight {tuple(w.shape)} / bias {tuple(b.shape)} "
                                  f"do not match {spec.weight_shape()}")
            self._check(self.lib.ynb_load_conv(self._h, spec.name.encode(), _ptr(w), w.numel(),
                                               _ptr(b), b.numel()), f"ynb_load_conv({spec.name})")
        self._check(self.lib.ynb_commit_weights(self._h), "ynb_commit_weights")

    # -- the path -----------------------------------------------------------------
    def _check_input(self, x: torch.Tensor) -> torch.Tensor:
        if not x.is_cuda:
            raise EngineError("input must live on the engine's GPU (no CPU fallback)")
        if x.device != self.device:
            raise EngineError(f"input on {x.device}, engine on {self.device}")
        if x.dtype != torch.float32 or x.dim() != 4 or x.shape[1] != 3:
            raise EngineError("input must be float32 [B,3,S,S]")
        s = self.input_size
        if x.shape[2] != s or x.shape[3] != s:
            # the reference fails with a broadcasting RuntimeError here (SURVEY §8b)
            raise RuntimeError(f"input is {tuple(x.shape[2:])} but the grid is set for {s}x{s}; "
                               "call set_grid first")
        return x.contiguous()

    def forward_raw(self, x: torch.Tensor):
        x = self._check_input(x)
        b, s = x.shape[0], self.input_size
        ch = 3 * (1 + self.num_classes + 4)
        outs = [torch.empty((b, ch, s // st, s // st), device=self.device, dtype=torch.float32)
                for st in (8, 16, 32)]
        self._check(self.lib.ynb_forward_raw(self._h, _ptr(x), b, _ptr(outs[0]), _ptr(outs[1]),
                                             _ptr(outs[2]), _stream_ptr(self.device)),
                    "ynb_forward_raw")
        return outs

    def forward_train_loss(self, x: torch.Tensor, target: torch.Tensor):
        """backbone + neck + heads, then the training branch (models/yolo_nano.py:333-358) on the
        engine's own NHWC head maps: (losses [4] on the device, gradients [B, H*W, ld] x 3)."""
        x = self._check_input(x)
        b, s = x.shape[0], self.input_size
        n = self.num_boxes
        if (not target.is_cuda or target.dtype != torch.float32 or not target.is_contiguous()
                or tuple(target.shape) != (b, n, 11)):
            raise EngineError(f"target must be a contiguous float32 CUDA tensor [B={b}, N={n}, 11]")
        ld = int(self.lib.ynb_raw_ld(self._h))
        grads = [torch.empty((b, (s // st) ** 2, ld), device=self.device, dtype=torch.float32) for st in (8, 16, 32)]
        losses = torch.empty(4, device=self.device, dtype=torch.float32)
        wsb = int(self.lib.ynb_train_loss_workspace_bytes(b, s))
        ws = torch.empty(wsb, device=self.device, dtype=torch.uint8)
        self._check(self.lib.ynb_forward_train_loss(self._h, _ptr(x), b, _ptr(target), _ptr(losses), _ptr(grads[0]),
                                                    _ptr(grads[1]), _ptr(grads[2]), _ptr(ws), wsb,
                                                    _stream_ptr(self.device)), "ynb_forward_train_loss")
        return losses, grads

    def forward_decode(self, x: torch.Tensor):
        x = self._check_input(x)
        b, n = x.shape[0], self.num_boxes
        boxes = torch.empty((b, n, 4), device=self.device, dtype=torch.float32)
        scores = torch.empty((b, n), device=self.device, dtype=torch.float32)
        cls = torch.empty((b, n), device=self.device, dtype=torch.int32)
        self._check(self.lib.ynb_forward_decode(self._h, _ptr(x), b, _ptr(boxes), _ptr(scores),
                                                _ptr(cls), _stream_ptr(self.device)),
                    "ynb_forward_decode")
        return boxes, scores, cls

    def forward_detect(self, x: torch.Tensor, out=None):
        """Returns device tensors (boxes [B,N,4], scores [B,N], cls [B,N] i32, counts [B] i32)."""
        x = self._check_input(x)
        b, n = x.shape[0], self.num_boxes
        if out is None:
            out = self.alloc_outputs(b)
        boxes, scores, cls, counts = out
        self._check(self.lib.ynb_forward_detect(self._h, _ptr(x), b, _ptr(boxes), _ptr(scores),
                                                _ptr(cls), _ptr(counts), _stream_ptr(self.device)),
                    "ynb_forward_detect")
        return boxes, scores, cls, counts

    def alloc_outputs(self, batch: int, pinned_host: bool = False):
        n = self.num_boxes
        kw = dict(device="cpu", pin_memory=True) if pinned_host else dict(device=self.device)
        return (torch.empty((batch, n, 4), dtype=torch.float32, **kw),
                torch.empty((batch, n), dtype=torch.float32, **kw),
                torch.empty((batch, n), dtype=torch.int32, **kw),
                torch.empty((batch,), dtype=torch.int32, **kw))

    def _check_host_shape(self, t: torch.Tensor, channels_last: bool, what: str):
        """The C side copies 3*S*S*batch elements using the engine's CURRENT grid size: a buffer built for
        another size (e.g. before a set_grid) must be an error, not an out-of-bounds read."""
        s = self.input_size
        want = (s, s, 3) if channels_last else (3, s, s)
        if tuple(t.shape[1:]) != want:
            raise EngineError(f"{what}: buffer is {tuple(t.shape)} but the grid is set for {s}x{s} "
                              f"(expected [B,{want[0]},{want[1]},{want[2]}]); call set_grid first")

    def detect_host(self, x_host: torch.Tensor, out_host=None):
        """Host buffers in, host buffers out; copies happen inside the call."""
        if x_host.is_cuda or x_host.dtype != torch.float32 or x_host.dim() != 4:
            raise EngineError("detect_host wants a float32 host tensor [B,3,S,S]")
        self._check_host_shape(x_host, False, "detect_host")
        x_host = x_host.contiguous()
        b = x_host.shape[0]
        if out_host is None:
            out_host = self.alloc_outputs(b, pinned_host=True)
        boxes, scores, cls, counts = out_host
        self._check(self.lib.ynb_detect_host(self._h, _ptr(x_host), b, _ptr(boxes), _ptr(scores),
                                             _ptr(cls), _ptr(counts), _stream_ptr(self.device)),
                    "ynb_detect_host")
        return boxes, scores, cls, counts

    def submit_host(self, slot: int, x_host: torch.Tensor, out_host):
        """Asynchronous half of detect_host: H2D + compute are enqueued, nothing is waited for.
        `x_host` and `out_host` (pinned) must stay alive until wait_host(slot)."""
        if x_host.is_cuda or x_host.dtype != torch.float32 or x_host.dim() != 4 or not x_host.is_contiguous():
            raise EngineError("submit_host wants a contiguous float32 host tensor [B,3,S,S]")
        self._check_host_shape(x_host, False, "submit_host")
        boxes, scores, cls, counts = out_host
        self._check(self.lib.ynb_submit_host(self._h, int(slot), _ptr(x_host), x_host.shape[0], _ptr(boxes),
                                             _ptr(scores), _ptr(cls), _ptr(counts), _stream_ptr(self.device)),
                    "ynb_submit_host")

    def submit_host_u8(self, slot: int, img_host: torch.Tensor, out_host, rects_host: torch.Tensor = None):
        """submit_host for uint8 images [B,S,S,3] BGR (letterboxed to S x S on the host); `rects_host`
        int32 [B,4] = (x0, y0, w, h) of the content, None = whole canvas.  Normalize + ToTensor of
        data/transforms.py run on the device."""
        if img_host.is_cuda or img_host.dtype != torch.uint8 or img_host.dim() != 4 or img_host.shape[-1] != 3 \
                or not img_host.is_contiguous():
            raise EngineError("submit_host_u8 wants a contiguous uint8 host tensor [B,S,S,3]")
        self._check_host_shape(img_host, True, "submit_host_u8")
        if rects_host is not None and (rects_host.dtype != torch.int32 or tuple(rects_host.shape) != (img_host.shape[0], 4)
                                       or not rects_host.is_contiguous() or rects_host.is_cuda):
            raise EngineError("rects_host must be a contiguous int32 host tensor [B,4]")
        boxes, scores, cls, counts = out_host
        self._check(self.lib.ynb_submit_host_u8(self._h, int(slot), _ptr(img_host),
                                                _ptr(rects_host) if rects_host is not None else None,
                                                img_host.shape[0], _ptr(boxes), _ptr(scores), _ptr(cls), _ptr(counts),
                                                _stream_ptr(self.device)), "ynb_submit_host_u8")

    def preprocess_u8(self, img: torch.Tensor, rects: torch.Tensor = None) -> torch.Tensor:
        """uint8 [B,S,S,3] BGR device tensor -> the float32 [B,3,S,S] RGB tensor of ValTransforms."""
        if not img.is_cuda or img.dtype != torch.uint8 or img.dim() != 4 or not img.is_contiguous():
            raise EngineError("preprocess_u8 wants a contiguous uint8 CUDA tensor [B,S,S,3]")
        self._check_host_shape(img, True, "preprocess_u8")
        if rects is not None and (not rects.is_cuda or rects.dtype != torch.int32 or not rects.is_contiguous()
                                  or tuple(rects.shape) != (img.shape[0], 4)):
            raise EngineError("rects must be a contiguous int32 CUDA tensor [B,4]")
        b, s = img.shape[0], img.shape[1]
        x = torch.empty((b, 3, s, s), dtype=torch.float32, device=img.device)
        self._check(self.lib.ynb_preprocess_u8(self._h, _ptr(img), _ptr(rects) if rects is not None else None, b,
                                               _ptr(x), _stream_ptr(self.device)), "ynb_preprocess_u8")
        return x

    @staticmethod
    def letterbox_desc(h0: int, w0: int, size: int):
        """Geometry of the reference's Resize (data/transforms.py:73-119) for one image: (nw, nh, left, top, mode,
        scale_x, scale_y) and the evaluators' (scale[4], offset[4]) as float64 — the same Python expressions."""
        if h0 > w0:
            nw, nh = int(w0 / h0 * size), size
            left, top = (nh - nw) // 2, 0
            offset, scale = [left / nh, 0., left / nh, 0.], [nw / nh, 1., nw / nh, 1.]
        elif h0 < w0:
            nw, nh = size, int(h0 / w0 * size)
            left, top = 0, (nw - nh) // 2
            offset, scale = [0., top / nw, 0., top / nw], [1., nh / nw, 1., nh / nw]
        else:
            nw, nh, left, top = size, size, 0, 0
            offset, scale = [0., 0., 0., 0.], [1., 1., 1., 1.]
        if nw < 1 or nh < 1:
            raise EngineError(f"image {h0}x{w0} collapses at size {size}")
        sx, sy = 1.0 / (nw / w0), 1.0 / (nh / h0)
        eps = 2.220446049250313e-16
        mode = 0 if (h0 == w0 == size) else (2 if abs(sx - 2) < eps and abs(sy - 2) < eps else 1)
        return nw, nh, left, top, mode, sx, sy, scale, offset

    def preprocess_images(self, images):
        """ValTransforms (letterbox Resize + Normalize + ToTensor) of a list of uint8 BGR HWC arrays of ANY shapes, on
        the device in one launch: returns (x float32 [B,3,S,S], maps float64 [B,12] = offset, scale, size for
        `map_boxes`).  Bit-identical to the reference transform (cv2 bilinear restated)."""
        import numpy as np
        s = self.input_size
        descs = np.zeros(len(images), dtype=np.dtype([("offset", "<i8"), ("h0", "<i4"), ("w0", "<i4"), ("nw", "<i4"),
                                                      ("nh", "<i4"), ("left", "<i4"), ("top", "<i4"), ("mode", "<i4"),
                                                      ("reserved", "<i4"), ("sx", "<f8"), ("sy", "<f8")]))
        maps = np.zeros((len(images), 12), dtype=np.float64)
        off = 0
        for i, im in enumerate(images):
            if im.dtype != np.uint8 or im.ndim != 3 or im.shape[2] != 3:
                raise EngineError("preprocess_images wants uint8 [H,W,3] BGR arrays")
            h0, w0 = int(im.shape[0]), int(im.shape[1])
            nw, nh, left, top, mode, sx, sy, scale, offset = self.letterbox_desc(h0, w0, s)
            descs[i] = (off, h0, w0, nw, nh, left, top, mode, 0, sx, sy)
            maps[i, 0:4], maps[i, 4:8], maps[i, 8:12] = offset, scale, [w0, h0, w0, h0]
            off += (h0 * w0 * 3 + 15) // 16 * 16
        packed = torch.empty(off, dtype=torch.uint8).pin_memory()
        pk = packed.numpy()
        for i, im in enumerate(images):
            o = int(descs[i]["offset"])
            pk[o:o + im.size] = np.ascontiguousarray(im).reshape(-1)
        # pinned staging + non_blocking: the host does not wait for the copies (a batch loop stays asynchronous)
        src = packed.to(self.device, non_blocking=True)
        d_desc = torch.from_numpy(descs.view(np.uint8).reshape(-1)).pin_memory().to(self.device, non_blocking=True)
        x = torch.empty((len(images), 3, s, s), dtype=torch.float32, device=self.device)
        self._check(self.lib.ynb_preprocess_letterbox_u8(self._h, _ptr(src), _ptr(d_desc), len(images), _ptr(x),
                                                         _stream_ptr(self.device)), "ynb_preprocess_letterbox_u8")
        return x, torch.from_numpy(maps).pin_memory().to(self.device, non_blocking=True)

    def map_boxes(self, boxes: torch.Tensor, counts: torch.Tensor, maps: torch.Tensor):
        """In place: boxes [B,N,4] (normalised, NMS output) -> original image pixels, rows [0, counts[b])
        (evaluator/cocoapi_evaluator.py:85-87)."""
        if not (boxes.is_cuda and boxes.dtype == torch.float32 and boxes.is_contiguous() and boxes.dim() == 3
                and maps.is_cuda and maps.dtype == torch.float64 and tuple(maps.shape) == (boxes.shape[0], 12)
                and counts.is_cuda and counts.dtype == torch.int32):
            raise EngineError("map_boxes wants boxes f32 [B,N,4], counts i32 [B], maps f64 [B,12] on the GPU")
        self._check(self.lib.ynb_map_boxes(_ptr(boxes), _ptr(counts), _ptr(maps.contiguous()), boxes.shape[0],
                                           boxes.shape[1], _stream_ptr(self.device)), "ynb_map_boxes")
        return boxes

    def set_normalization(self, mean_bgr, std_bgr):
        m = (C.c_float * 3)(*[float(v) for v in mean_bgr])
        sd = (C.c_float * 3)(*[float(v) for v in std_bgr])
        self._check(self.lib.ynb_set_normalization(self._h, m, sd), "ynb_set_normalization")

    def wait_host(self, slot: int):
        self._check(self.lib.ynb_wait_host(self._h, int(slot)), "ynb_wait_host")

    def profile(self, x: torch.Tensor):
        """One forward_detect with a CUDA-event pair around every kernel launch.
        Returns [(label, kernel family, ms, algorithmic bytes, flops), ...]."""
        self._check(self.lib.ynb_set_profiling(self._h, 1), "ynb_set_profiling")
        try:
            self.forward_detect(x)
        finally:
            self.lib.ynb_set_profiling(self._h, 0)
        out = []
        name, kind = C.c_char_p(), C.c_char_p()
        ms, by, fl = C.c_float(), C.c_double(), C.c_double()
        for i in range(self.lib.ynb_profile_count(self._h)):
            self._check(self.lib.ynb_profile_entry(self._h, i, C.byref(name), C.byref(kind), C.byref(ms),
                                                   C.byref(by), C.byref(fl)), "ynb_profile_entry")
            out.append((name.value.decode(), kind.value.decode(), ms.value, by.value, fl.value))
        return out

    def read_tap(self, name: str, batch: int) -> torch.Tensor:
        c, h, w = C.c_int32(), C.c_int32(), C.c_int32()
        self._check(self.lib.ynb_tap_shape(self._h, name.encode(), C.byref(c), C.byref(h), C.byref(w)),
                    f"ynb_tap_shape({name})")
        out = torch.empty((batch, c.value, h.value, w.value), device=self.device, dtype=torch.float32)
        self._check(self.lib.ynb_read_tap(self._h, name.encode(), batch, _ptr(out),
                                          _stream_ptr(self.device)), f"ynb_read_tap({name})")
        return out
