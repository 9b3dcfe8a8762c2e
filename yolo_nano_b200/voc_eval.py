"""VOC mAP on the device: what `VOCAPIEvaluator.evaluate` does after detection — write_voc_results_file, then
do_python_eval -> voc_eval -> voc_ap for every class (evaluator/vocapi_evaluator.py, ssd.pytorch lineage) — without
the det files.  `add` turns each batch of kept detections into det-file lines on the device (one int32 row per line,
the decimal fields the text would carry); `evaluate` sorts, matches, scans and returns the per-class APs.

Detections of equal score are taken in file order (image, then kept row), the order the NMS defines for its own ties;
voc_eval's default np.argsort leaves that order to the platform's sort.
"""
from __future__ import annotations

import ctypes as C
from typing import Sequence, Tuple

import numpy as np
import torch

from . import _lib
from .engine import EngineError, _ptr, _stream_ptr

ROW_FIELDS = ("image", "class", "milli", "x1", "y1", "x2", "y2")


class VOCDetections:
    """A device arena of det-file lines for one evaluation.  Not thread-safe."""

    def __init__(self, device, num_classes: int, capacity: int):
        self.lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise EngineError("VOCDetections runs on a CUDA device (no CPU fallback)")
        self.num_classes = int(num_classes)
        self.capacity = int(capacity)
        self.rows = torch.empty((self.capacity, len(ROW_FIELDS)), dtype=torch.int32, device=self.device)
        # [rows appended (counted past the capacity too), rejected values]
        self.state = torch.zeros(2, dtype=torch.int64, device=self.device)
        self.num_images = 0

    def add(self, boxes: torch.Tensor, scores: torch.Tensor, cls: torch.Tensor, counts: torch.Tensor):
        """Append the kept rows [0, counts[b]) of every image of a batch (pixel boxes f32 [B,N,4] after map_boxes,
        scores f32 [B,N], cls i32 [B,N], counts i32 [B], all on the device) as the next B images.  No sync."""
        b = int(counts.shape[0])
        n = int(scores.shape[1]) if scores.dim() == 2 else -1
        ok = (boxes.dtype == torch.float32 and scores.dtype == torch.float32 and cls.dtype == torch.int32
              and counts.dtype == torch.int32 and tuple(boxes.shape) == (b, n, 4) and tuple(scores.shape) == (b, n)
              and tuple(cls.shape) == (b, n) and counts.dim() == 1
              and all(t.device == self.device and t.is_contiguous() for t in (boxes, scores, cls, counts)))
        if not ok:
            raise EngineError(f"add wants contiguous boxes f32 [B,N,4], scores f32 [B,N], cls i32 [B,N], counts i32 [B] "
                              f"on {self.device}")
        if b == 0 or n == 0:
            return
        rc = self.lib.ynb_voc_append(_ptr(boxes), _ptr(scores), _ptr(cls), _ptr(counts), b, n, self.num_images,
                                     self.num_classes, _ptr(self.rows), self.capacity, _ptr(self.state),
                                     _stream_ptr(self.device))
        if rc != _lib.YNB_OK:
            msg = self.lib.ynb_last_error(None)
            raise EngineError(f"ynb_voc_append failed ({rc}): {msg.decode() if msg else '?'}")
        self.num_images += b

    def num_rows(self) -> int:
        """Rows appended so far, including any past the capacity (synchronises)."""
        return int(self.state[0])

    def _checked_rows(self) -> int:
        n, bad = (int(v) for v in self.state.cpu())
        if n > self.capacity:
            raise EngineError(f"{n} detection rows exceed the capacity of {self.capacity}; rows past it were dropped")
        if bad:
            raise EngineError(f"{bad} detections had a class outside [0, {self.num_classes}), a score outside [0, 1] "
                              "or a non-finite / out-of-range box")
        return n

    def pack_gt(self, gt: Sequence[Tuple[np.ndarray, np.ndarray, np.ndarray]]):
        """Per-image (boxes [G,4], labels [G], difficult [G]) -> device (boxes f64 [G,4], difficult u8 [G],
        start i32 [images * classes + 1]) bucketed by (image, class) in annotation order."""
        if len(gt) != self.num_images:
            raise EngineError(f"gt covers {len(gt)} images but {self.num_images} were added")
        nc = self.num_classes
        sizes = [len(np.asarray(lab).reshape(-1)) for _, lab, _ in gt]
        boxes = np.concatenate([np.asarray(b, dtype=np.float64).reshape(-1, 4) for b, _, _ in gt] or
                               [np.zeros((0, 4))]).reshape(-1, 4)
        labels = np.concatenate([np.asarray(lab).reshape(-1) for _, lab, _ in gt] or [np.zeros(0)]).astype(np.int64)
        diff = np.concatenate([np.asarray(d).reshape(-1) for _, _, d in gt] or [np.zeros(0)]).astype(bool)
        if boxes.shape[0] != labels.shape[0] or diff.shape[0] != labels.shape[0]:
            raise EngineError("gt: boxes, labels and difficult must have one entry per object")
        if labels.size and (labels.min() < 0 or labels.max() >= nc):
            raise EngineError(f"gt labels must lie in [0, {nc})")
        if not np.isfinite(boxes).all():
            raise EngineError("gt boxes must be finite")
        img = np.repeat(np.arange(len(gt), dtype=np.int64), sizes)
        bucket = img * nc + labels
        order = np.argsort(bucket, kind="stable")
        start = np.zeros(len(gt) * nc + 1, dtype=np.int32)
        start[1:] = np.cumsum(np.bincount(bucket, minlength=len(gt) * nc))
        dev = self.device
        return (torch.from_numpy(np.ascontiguousarray(boxes[order])).to(dev),
                torch.from_numpy(diff[order].astype(np.uint8)).to(dev),
                torch.from_numpy(start).to(dev), int(labels.size))

    def evaluate(self, gt, ovthresh: float = 0.5, use_07_metric: bool = True, details: bool = False):
        """voc_eval of every class against `gt` (one (boxes [G,4], labels [G], difficult [G]) per added image, boxes in
        voc_eval's coordinates).  Returns (aps float64 [C], mAP) with mAP = np.mean(aps), the -1 of classes without
        detections included as the reference does; with details=True also (npos [C], order [R] = arena row of each
        sorted position, flags [R] = 1 TP / 2 FP / 0 ignored) as host arrays."""
        n = self._checked_rows()
        gb, gd, gs, n_gt = self.pack_gt(gt)
        nc, dev = self.num_classes, self.device
        wsb = int(self.lib.ynb_voc_eval_workspace_bytes(n, nc, n_gt))
        if wsb < 0:
            raise EngineError("ynb_voc_eval_workspace_bytes: bad sizes")
        ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
        ap = torch.empty(nc, dtype=torch.float64, device=dev)
        npos = torch.empty(nc, dtype=torch.int32, device=dev)
        order = torch.empty(n, dtype=torch.int32, device=dev) if details else None
        flags = torch.empty(n, dtype=torch.int8, device=dev) if details else None
        rc = self.lib.ynb_voc_eval(_ptr(self.rows), n, nc, self.num_images, _ptr(gb), _ptr(gd), _ptr(gs), n_gt,
                                   C.c_double(float(ovthresh)), int(bool(use_07_metric)), _ptr(ap), _ptr(npos),
                                   _ptr(order), _ptr(flags), _ptr(ws), wsb, _stream_ptr(dev))
        if rc != _lib.YNB_OK:
            msg = self.lib.ynb_last_error(None)
            raise EngineError(f"ynb_voc_eval failed ({rc}): {msg.decode() if msg else '?'}")
        aps = ap.cpu().numpy()
        out = (aps, float(np.mean(aps)))
        if details:
            out += (npos.cpu().numpy(), order.cpu().numpy(), flags.cpu().numpy())
        return out
