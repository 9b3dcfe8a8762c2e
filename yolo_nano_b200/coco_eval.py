"""COCO AP on the device: what `COCOAPIEvaluator.evaluate` does after detection (evaluator/cocoapi_evaluator.py) —
the results JSON, `cocoGt.loadRes`, then pycocotools' `COCOeval(cocoGt, cocoDt, 'bbox')` with `params.imgIds = ids`,
`evaluate()`, `accumulate()` and `summarize()` — without the JSON, the Python dicts or pycocotools.  `add` turns each
batch of kept detections into results entries on the device (one int32 row per entry, the float32 values the JSON
would carry); `evaluate` runs evaluateImg and accumulate on the device and the 12 summary means on the host.

COCOeval's sorts are all stable (mergesort) and its arithmetic is short IEEE float64 chains, so the precision and
recall arrays, and with them the stats, are the ones pycocotools computes, bit for bit.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Sequence

import numpy as np
import torch

from . import _lib
from .engine import EngineError, _ptr, _stream_ptr

ROW_FIELDS = ("image", "class", "score_bits", "x1_bits", "y1_bits", "x2_bits", "y2_bits")

# Params.setDetParams (pycocotools/cocoeval.py), bbox defaults
IOU_THRS = np.linspace(.5, 0.95, int(np.round((0.95 - .5) / .05)) + 1, endpoint=True)
REC_THRS = np.linspace(.0, 1.00, int(np.round((1.00 - .0) / .01)) + 1, endpoint=True)
MAX_DETS = [1, 10, 100]
AREA_RNG_LBL = ['all', 'small', 'medium', 'large']


def summarize(precision: np.ndarray, recall: np.ndarray) -> np.ndarray:
    """COCOeval.summarize -> _summarizeDets: the 12 stats from precision [T,R,K,A,M] and recall [T,K,A,M]."""
    def _summarize(ap=1, iouThr=None, areaRng='all', maxDets=100):
        aind = [i for i, aRng in enumerate(AREA_RNG_LBL) if aRng == areaRng]
        mind = [i for i, mDet in enumerate(MAX_DETS) if mDet == maxDets]
        if ap == 1:
            s = precision
            if iouThr is not None:
                t = np.where(iouThr == IOU_THRS)[0]
                s = s[t]
            s = s[:, :, :, aind, mind]
        else:
            s = recall
            if iouThr is not None:
                t = np.where(iouThr == IOU_THRS)[0]
                s = s[t]
            s = s[:, :, aind, mind]
        if len(s[s > -1]) == 0:
            mean_s = -1
        else:
            mean_s = np.mean(s[s > -1])
        return mean_s

    stats = np.zeros((12,))
    stats[0] = _summarize(1)
    stats[1] = _summarize(1, iouThr=.5, maxDets=MAX_DETS[2])
    stats[2] = _summarize(1, iouThr=.75, maxDets=MAX_DETS[2])
    stats[3] = _summarize(1, areaRng='small', maxDets=MAX_DETS[2])
    stats[4] = _summarize(1, areaRng='medium', maxDets=MAX_DETS[2])
    stats[5] = _summarize(1, areaRng='large', maxDets=MAX_DETS[2])
    stats[6] = _summarize(0, maxDets=MAX_DETS[0])
    stats[7] = _summarize(0, maxDets=MAX_DETS[1])
    stats[8] = _summarize(0, maxDets=MAX_DETS[2])
    stats[9] = _summarize(0, areaRng='small', maxDets=MAX_DETS[2])
    stats[10] = _summarize(0, areaRng='medium', maxDets=MAX_DETS[2])
    stats[11] = _summarize(0, areaRng='large', maxDets=MAX_DETS[2])
    return stats


def pack_gt(gt: Dict, image_ids: Sequence[int], class_ids: Sequence[int], num_classes: int):
    """The instances dict -> the evaluation's host arrays, as COCOeval._prepare selects them:
    image_rank [images] (position of each added image's id among the sorted ids), class_cat [num_classes]
    (index of class_ids[c] among the sorted GT category ids, -1 when it is none), and the GT of the evaluated images
    and categories in annotation-file order, bucketed by (rank, category index): boxes f64 [G,4] xywh, area f64 [G],
    iscrowd u8 [G], start i32 [images * K + 1].  Returns a dict of NumPy arrays and K."""
    ids = [int(i) for i in image_ids]
    uniq = np.unique(np.asarray(ids, dtype=np.int64))
    if len(uniq) != len(ids):
        raise EngineError("image_ids must be unique (one per added image)")
    known = {int(im["id"]) for im in gt["images"]}
    missing = [i for i in ids if i not in known]
    if missing:
        raise EngineError(f"image ids not in gt['images'] (loadRes would refuse them): {missing[:5]}")
    if len(class_ids) < num_classes:
        raise EngineError(f"class_ids has {len(class_ids)} entries for {num_classes} classes")
    cat_ids = sorted(int(c["id"]) for c in gt["categories"])
    K = len(cat_ids)
    if K == 0:
        raise EngineError("gt has no categories")
    cat_index = {c: k for k, c in enumerate(cat_ids)}
    class_cat = np.array([cat_index.get(int(class_ids[c]), -1) for c in range(num_classes)], dtype=np.int32)
    rank_of = {int(i): r for r, i in enumerate(uniq)}
    anns = gt.get("annotations", [])
    ann_ids = [int(a["id"]) for a in anns]
    if len(set(ann_ids)) != len(ann_ids):
        raise EngineError("gt annotation ids must be unique")
    cell, boxes, area, crowd = [], [], [], []
    for a in anns:
        r = rank_of.get(int(a["image_id"]))
        k = cat_index.get(int(a["category_id"]))
        if r is None or k is None:
            continue
        if "iscrowd" not in a:
            raise EngineError(f"annotation {a['id']} has no iscrowd field")
        if int(a["id"]) <= 0:
            raise EngineError(f"annotation id {a['id']} <= 0: COCOeval reads a match on id 0 as no match")
        cell.append(r * K + k)
        boxes.append([float(v) for v in a["bbox"]])
        area.append(float(a["area"]))
        crowd.append(1 if a["iscrowd"] else 0)
    cell = np.asarray(cell, dtype=np.int64)
    order = np.argsort(cell, kind="stable")
    start = np.zeros(len(ids) * K + 1, dtype=np.int32)
    start[1:] = np.cumsum(np.bincount(cell, minlength=len(ids) * K))
    boxes = np.asarray(boxes, dtype=np.float64).reshape(-1, 4)[order]
    area = np.asarray(area, dtype=np.float64)[order]
    if not (np.isfinite(boxes).all() and np.isfinite(area).all()):
        raise EngineError("gt boxes and areas must be finite")
    return {"image_rank": np.searchsorted(uniq, np.asarray(ids, dtype=np.int64)).astype(np.int32),
            "class_cat": class_cat, "boxes": np.ascontiguousarray(boxes), "area": np.ascontiguousarray(area),
            "iscrowd": np.asarray(crowd, dtype=np.uint8)[order], "start": start}, K


class COCODetections:
    """A device arena of COCO results entries for one evaluation.  Not thread-safe."""

    def __init__(self, device, num_classes: int, capacity: int):
        self.lib = _lib.load()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise EngineError("COCODetections runs on a CUDA device (no CPU fallback)")
        self.num_classes = int(num_classes)
        self.capacity = int(capacity)
        # one row at least: an empty tensor has no address to hand to the library
        self.rows = torch.empty((max(self.capacity, 1), len(ROW_FIELDS)), dtype=torch.int32, device=self.device)
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
        if b == 0:
            return
        if n > 0:
            rc = self.lib.ynb_coco_append(_ptr(boxes), _ptr(scores), _ptr(cls), _ptr(counts), b, n, self.num_images,
                                          self.num_classes, _ptr(self.rows), self.capacity, _ptr(self.state),
                                          _stream_ptr(self.device))
            if rc != _lib.YNB_OK:
                msg = self.lib.ynb_last_error(None)
                raise EngineError(f"ynb_coco_append failed ({rc}): {msg.decode() if msg else '?'}")
        self.num_images += b

    def num_rows(self) -> int:
        """Rows appended so far, including any past the capacity (synchronises)."""
        return int(self.state[0])

    def _checked_rows(self) -> int:
        n, bad = (int(v) for v in self.state.cpu())
        if n > self.capacity:
            raise EngineError(f"{n} detection rows exceed the capacity of {self.capacity}; rows past it were dropped")
        if bad:
            raise EngineError(f"{bad} detections had a class outside [0, {self.num_classes}) or a non-finite score or "
                              "box")
        return n

    def evaluate(self, gt: Dict, image_ids: Sequence[int], class_ids: Sequence[int], details: bool = False):
        """COCOeval 'bbox' of the added detections against `gt` (the instances JSON as a dict), with
        params.imgIds = image_ids (the COCO id of each added image, in add order) and category ids
        class_ids[cls] (the reference's dataset.class_ids).  Returns stats float64 [12] (the reference's
        (ap50, ap50_95) are stats[1] and stats[0]); with details=True also (precision [10,101,K,4,3],
        recall [10,K,4,3]) as host arrays."""
        if len(image_ids) != self.num_images:
            raise EngineError(f"image_ids covers {len(image_ids)} images but {self.num_images} were added")
        n = self._checked_rows()
        p, K = pack_gt(gt, image_ids, class_ids, self.num_classes)
        dev, ni = self.device, self.num_images
        n_gt = int(p["area"].shape[0])
        t = {k: torch.from_numpy(v).to(dev) for k, v in p.items()}
        wsb = int(self.lib.ynb_coco_eval_workspace_bytes(n, ni, K, n_gt))
        if wsb < 0:
            raise EngineError("ynb_coco_eval_workspace_bytes: bad sizes")
        ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
        precision = torch.empty((len(IOU_THRS), len(REC_THRS), K, len(AREA_RNG_LBL), len(MAX_DETS)),
                                dtype=torch.float64, device=dev)
        recall = torch.empty((len(IOU_THRS), K, len(AREA_RNG_LBL), len(MAX_DETS)), dtype=torch.float64, device=dev)
        dbl = C.POINTER(C.c_double)
        iou_thrs = np.ascontiguousarray(IOU_THRS, dtype=np.float64)
        rec_thrs = np.ascontiguousarray(REC_THRS, dtype=np.float64)
        rc = self.lib.ynb_coco_eval(_ptr(self.rows), n, self.num_classes, ni, _ptr(t["image_rank"]),
                                    _ptr(t["class_cat"]), K, _ptr(t["boxes"]), _ptr(t["area"]), _ptr(t["iscrowd"]),
                                    _ptr(t["start"]), n_gt, iou_thrs.ctypes.data_as(dbl), rec_thrs.ctypes.data_as(dbl),
                                    _ptr(precision), _ptr(recall), _ptr(ws), wsb, _stream_ptr(dev))
        if rc != _lib.YNB_OK:
            msg = self.lib.ynb_last_error(None)
            raise EngineError(f"ynb_coco_eval failed ({rc}): {msg.decode() if msg else '?'}")
        prec, rec = precision.cpu().numpy(), recall.cpu().numpy()
        stats = summarize(prec, rec)
        return (stats, (prec, rec)) if details else stats
