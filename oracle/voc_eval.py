"""Restatement of the reference's VOC mAP (evaluator/vocapi_evaluator.py: write_voc_results_file, voc_eval, voc_ap;
ssd.pytorch lineage) — the checker of yolo_nano_b200.voc_eval, never its path.

Two points where this lineage differs from py-faster-rcnn's voc_eval live in one place each:
  * overlaps without the +1 pixel convention ............................ `overlaps`
  * ap = -1 for a class whose det file has no lines ....................... `NO_LINES_AP`

Three forms:
  * `voc_eval_literal`  the reference's voc_eval line by line: parses det files and an annots.pkl from disk, sorts
                        with the given argsort kind (the reference uses NumPy's default, whose tie order is the
                        platform's; 'stable' gives file order).
  * `result_rows` + `voc_eval_rows`  the same numbers from integer det-file rows (the device's arena format), stable
                        order, and the order-independent claim rule: a detection with ovmax > thr on a non-difficult
                        jmax is TP iff it is the first in sorted order aiming at that GT.
  * `decimal_ints`      the rounding of '{:.1f}' / '{:.3f}' (half-even on the exact float32 value) in integers.
This restatement has not yet been pinned by a golden from the real voc_eval (`python -m oracle.gen_voc_golden`
records one wherever the reference tree exists).
"""
from __future__ import annotations

import os
import pickle
from typing import List, Sequence, Tuple

import numpy as np

NO_LINES_AP = -1.
NEG_ZERO = np.iinfo(np.int32).min      # arena encoding of a '-0.0' field
EPS64 = np.finfo(np.float64).eps


def overlaps(bb, BBGT):
    """IoU of a detection with GT boxes, no +1 (voc_eval's inner block); works on [4] vs [G,4] and on broadcast
    [..., 4] arrays alike — the same IEEE float64 operations elementwise."""
    ixmin = np.maximum(BBGT[..., 0], bb[..., 0])
    iymin = np.maximum(BBGT[..., 1], bb[..., 1])
    ixmax = np.minimum(BBGT[..., 2], bb[..., 2])
    iymax = np.minimum(BBGT[..., 3], bb[..., 3])
    iw = np.maximum(ixmax - ixmin, 0.)
    ih = np.maximum(iymax - iymin, 0.)
    inters = iw * ih
    uni = ((bb[..., 2] - bb[..., 0]) * (bb[..., 3] - bb[..., 1]) +
           (BBGT[..., 2] - BBGT[..., 0]) * (BBGT[..., 3] - BBGT[..., 1]) - inters)
    with np.errstate(invalid="ignore", divide="ignore"):
        return inters / uni


def voc_ap(rec, prec, use_07_metric=True):
    """evaluator/vocapi_evaluator.py voc_ap."""
    if use_07_metric:
        ap = 0.
        for t in np.arange(0., 1.1, 0.1):
            if np.sum(rec >= t) == 0:
                p = 0
            else:
                p = np.max(prec[rec >= t])
            ap = ap + p / 11.
    else:
        mrec = np.concatenate(([0.], rec, [1.]))
        mpre = np.concatenate(([0.], prec, [0.]))
        for i in range(mpre.size - 1, 0, -1):
            mpre[i - 1] = np.maximum(mpre[i - 1], mpre[i])
        i = np.where(mrec[1:] != mrec[:-1])[0]
        ap = np.sum((mrec[i + 1] - mrec[i]) * mpre[i + 1])
    return ap


def _rec_prec(tp, fp, npos):
    fp = np.cumsum(fp)
    tp = np.cumsum(tp)
    with np.errstate(invalid="ignore", divide="ignore"):
        rec = tp / float(npos)
    prec = tp / np.maximum(tp + fp, EPS64)
    return rec, prec


# ---- det files and the literal voc_eval ---------------------------------------------------------------------------
def write_det_files(template: str, image_names: Sequence[str], dets, labelmap: Sequence[str]):
    """write_voc_results_file: dets[i] = (pixel boxes f32 [K,4], scores [K], cls [K]) of image i, through
    evalfmt.voc_class_dets / voc_result_lines (pinned to the real writer by golden g6)."""
    from yolo_nano_b200 import evalfmt
    per_image = [evalfmt.voc_class_dets(b, s, c, len(labelmap)) for b, s, c in dets]
    for j, cls in enumerate(labelmap):
        with open(template.format(cls), "wt") as f:
            for i, name in enumerate(image_names):
                d = per_image[i][j]
                if len(d) == 0:
                    continue
                f.writelines(evalfmt.voc_result_lines(name, d))


def write_annots(cachefile: str, imagesetfile: str, image_names: Sequence[str], gt, labelmap: Sequence[str]):
    """The annots.pkl cache voc_eval reads (recs[imagename] = [{'name', 'bbox', 'difficult'}, ...]) and the image
    set file; gt[i] = (boxes [G,4] in voc_eval's coordinates, labels [G], difficult [G])."""
    recs = {}
    for name, (b, lab, d) in zip(image_names, gt):
        recs[name] = [{"name": labelmap[int(l_)], "bbox": [float(v) for v in bx], "difficult": int(df)}
                      for bx, l_, df in zip(np.asarray(b, np.float64).reshape(-1, 4), np.asarray(lab).reshape(-1),
                                            np.asarray(d).reshape(-1))]
    with open(cachefile, "wb") as f:
        pickle.dump(recs, f)
    with open(imagesetfile, "wt") as f:
        f.writelines(n + "\n" for n in image_names)


def voc_eval_literal(detpath, imagesetfile, classname, cachefile, ovthresh=0.5, use_07_metric=True, kind=None):
    """voc_eval (evaluator/vocapi_evaluator.py) line by line, annots read from the pickle cache; `kind` is the
    argsort kind (None = NumPy's default, as in the reference)."""
    with open(imagesetfile, 'r') as f:
        lines = f.readlines()
    imagenames = [x.strip() for x in lines]
    with open(cachefile, 'rb') as f:
        recs = pickle.load(f)
    class_recs = {}
    npos = 0
    for imagename in imagenames:
        R = [obj for obj in recs[imagename] if obj['name'] == classname]
        bbox = np.array([x['bbox'] for x in R])
        difficult = np.array([x['difficult'] for x in R]).astype(bool)
        det = [False] * len(R)
        npos = npos + sum(~difficult)
        class_recs[imagename] = {'bbox': bbox, 'difficult': difficult, 'det': det}
    detfile = detpath.format(classname)
    with open(detfile, 'r') as f:
        lines = f.readlines()
    if any(lines) == 1:
        splitlines = [x.strip().split(' ') for x in lines]
        image_ids = [x[0] for x in splitlines]
        confidence = np.array([float(x[1]) for x in splitlines])
        BB = np.array([[float(z) for z in x[2:]] for x in splitlines])
        sorted_ind = np.argsort(-confidence, kind=kind)
        BB = BB[sorted_ind, :]
        image_ids = [image_ids[x] for x in sorted_ind]
        nd = len(image_ids)
        tp = np.zeros(nd)
        fp = np.zeros(nd)
        for d in range(nd):
            R = class_recs[image_ids[d]]
            bb = BB[d, :].astype(float)
            ovmax = -np.inf
            BBGT = R['bbox'].astype(float)
            if BBGT.size > 0:
                ov = overlaps(bb, BBGT)
                ovmax = np.max(ov)
                jmax = np.argmax(ov)
            if ovmax > ovthresh:
                if not R['difficult'][jmax]:
                    if not R['det'][jmax]:
                        tp[d] = 1.
                        R['det'][jmax] = 1
                    else:
                        fp[d] = 1.
            else:
                fp[d] = 1.
        rec, prec = _rec_prec(tp, fp, npos)
        ap = voc_ap(rec, prec, use_07_metric)
    else:
        ap = NO_LINES_AP
    return ap


def eval_files(tmpdir: str, dets, gt, num_classes: int, ovthresh=0.5, use_07_metric=True, kind="stable"):
    """The whole reference round trip in `tmpdir`: det files + annots, then voc_eval per class.  Returns aps [C]."""
    names = [f"{i:06d}" for i in range(len(dets))]
    labelmap = [f"class{j:03d}" for j in range(num_classes)]
    template = os.path.join(tmpdir, "det_test_{}.txt")
    cachefile, imageset = os.path.join(tmpdir, "annots.pkl"), os.path.join(tmpdir, "test.txt")
    write_det_files(template, names, dets, labelmap)
    write_annots(cachefile, imageset, names, gt, labelmap)
    return np.array([voc_eval_literal(template, imageset, c, cachefile, ovthresh, use_07_metric, kind)
                     for c in labelmap], dtype=np.float64)


# ---- integer rows -------------------------------------------------------------------------------------------------
def decimal_ints(v, digits: int) -> np.ndarray:
    """The integer of '{:.<digits>f}' of float32 values (round half-even on the exact binary value), int64; a '-0'
    result is NEG_ZERO."""
    v = np.ascontiguousarray(v, dtype=np.float32)
    if not np.isfinite(v).all():
        raise ValueError("decimal_ints: non-finite value")
    u = v.view(np.uint32).astype(np.int64)
    ex, fr = (u >> 23) & 0xff, u & 0x7fffff
    m = np.where(ex > 0, fr | 0x800000, fr)
    e = np.where(ex > 0, ex - 150, -149)
    big = m * 10 ** digits
    s = np.clip(-e, 1, 62)
    q_neg = big >> s
    rem = big & ((np.int64(1) << s) - 1)
    half = np.int64(1) << (s - 1)
    q_neg = q_neg + ((rem > half) | ((rem == half) & (q_neg & 1 == 1)))
    q = np.where(e >= 0, big << np.clip(e, 0, 62), q_neg)
    q = np.where(-e >= 40, 0, q)
    neg = (u >> 31) == 1
    return np.where(neg, np.where(q == 0, NEG_ZERO, -q), q)


def tenths_to_float(n) -> np.ndarray:
    n = np.asarray(n, dtype=np.int64)
    return np.where(n == NEG_ZERO, -0.0, n / 10.0)


def result_rows(dets) -> np.ndarray:
    """Det-file lines as int32 rows [image, class, milli, x1, y1, x2, y2] in file order (image, kept row):
    dets[i] = (pixel boxes f32 [K,4], scores f32 [K], cls [K]) of image i."""
    out = []
    for i, (b, s, c) in enumerate(dets):
        b = np.asarray(b, np.float32).reshape(-1, 4)
        r = np.empty((len(b), 7), np.int64)
        r[:, 0] = i
        r[:, 1] = np.asarray(c).reshape(-1)
        r[:, 2] = decimal_ints(np.asarray(s, np.float32), 3)
        r[:, 3:] = decimal_ints(b + np.float32(1), 1)
        out.append(r)
    return np.concatenate(out or [np.zeros((0, 7), np.int64)]).astype(np.int32)


def voc_eval_rows(rows: np.ndarray, gt, num_classes: int, ovthresh=0.5, use_07_metric=True, chunk=200_000):
    """voc_eval of every class from integer rows: returns (aps [C], npos [C], per class (arena rows in sorted order,
    flags 1 TP / 2 FP / 0 ignored))."""
    rows = np.asarray(rows, np.int64).reshape(-1, 7)
    sizes = np.array([len(np.asarray(lab).reshape(-1)) for _, lab, _ in gt], np.int64)
    gb = np.concatenate([np.asarray(b, np.float64).reshape(-1, 4) for b, _, _ in gt] or [np.zeros((0, 4))])
    gl = np.concatenate([np.asarray(lab).reshape(-1) for _, lab, _ in gt] or [np.zeros(0)]).astype(np.int64)
    gd = np.concatenate([np.asarray(d).reshape(-1) for _, _, d in gt] or [np.zeros(0)]).astype(bool)
    gi = np.repeat(np.arange(len(gt)), sizes)
    aps, npos_all, detail = [], [], []
    for c in range(num_classes):
        sel = np.nonzero(rows[:, 1] == c)[0]
        npos = int(np.sum((gl == c) & ~gd))
        npos_all.append(npos)
        if len(sel) == 0:
            aps.append(NO_LINES_AP)
            detail.append((sel, np.zeros(0, np.int8)))
            continue
        confidence = rows[sel, 2] / 1000.0
        srt = sel[np.argsort(-confidence, kind="stable")]
        # GT of class c bucketed per image, annotation order kept
        gidx_c = np.nonzero(gl == c)[0]
        cnt = np.bincount(gi[gidx_c], minlength=len(gt))
        start = np.concatenate([[0], np.cumsum(cnt)])
        gmax = max(int(cnt.max()) if len(cnt) else 0, 1)
        flags = np.empty(len(srt), np.int8)
        slot = np.full(len(srt), -1, np.int64)
        for a in range(0, len(srt), chunk):
            r = rows[srt[a:a + chunk]]
            img = r[:, 0]
            bb = tenths_to_float(r[:, 3:7])
            k = np.arange(gmax)[None, :]
            valid = k < cnt[img][:, None]
            g = gidx_c[np.minimum(start[img][:, None] + k, max(len(gidx_c) - 1, 0))] if len(gidx_c) else \
                np.zeros((len(r), gmax), np.int64)
            BBGT = gb[g] if len(gidx_c) else np.zeros((len(r), gmax, 4))
            ov = np.where(valid, overlaps(bb[:, None, :], BBGT), -np.inf)
            jmax = np.argmax(ov, axis=1)
            ovmax = ov[np.arange(len(r)), jmax]
            gj = g[np.arange(len(r)), jmax]
            hit = ovmax > ovthresh
            dif = gd[gj] if len(gidx_c) else np.zeros(len(r), bool)
            f = np.full(len(r), 2, np.int8)
            f[hit & dif] = 0
            cand = hit & ~dif
            slot[a:a + chunk][cand] = gj[cand]
            flags[a:a + chunk] = f
        cand = np.nonzero(slot >= 0)[0]
        _, first = np.unique(slot[cand], return_index=True)
        flags[cand[first]] = 1
        tp = (flags == 1).astype(np.float64)
        fp = (flags == 2).astype(np.float64)
        rec, prec = _rec_prec(tp, fp, npos)
        aps.append(voc_ap(rec, prec, use_07_metric))
        detail.append((srt, flags))
    return np.array(aps, dtype=np.float64), np.array(npos_all), detail


def default_vs_stable(dets, gt, num_classes: int, tmpdir: str, use_07_metric=True) -> Tuple[np.ndarray, np.ndarray]:
    """APs of the literal voc_eval with NumPy's default argsort and with a stable one, on the same det files."""
    a = eval_files(tmpdir, dets, gt, num_classes, use_07_metric=use_07_metric, kind=None)
    b = eval_files(tmpdir, dets, gt, num_classes, use_07_metric=use_07_metric, kind="stable")
    return a, b


def random_set(n_images: int, num_classes: int, seed: int, max_gt: int = 8, dets_per_gt: float = 3.0,
               difficult_rate: float = 0.1, score_levels: int = 40) -> Tuple[List, List]:
    """A tie-heavy synthetic evaluation set: per image GT boxes (integer pixel coordinates, like parse_rec's) and
    detections that are jittered copies of them plus clutter, scores on a coarse grid so that '{:.3f}' ties are
    everywhere.  Returns (dets, gt) in the shapes evaluate / eval_files take."""
    rng = np.random.default_rng(seed)
    dets, gt = [], []
    for i in range(n_images):
        w, h = rng.integers(200, 640, 2)
        g = int(rng.integers(0, max_gt + 1))
        x1 = rng.integers(0, w - 20, g)
        y1 = rng.integers(0, h - 20, g)
        gbox = np.stack([x1, y1, np.minimum(x1 + rng.integers(8, 200, g), w - 1),
                         np.minimum(y1 + rng.integers(8, 200, g), h - 1)], 1).astype(np.float64)
        glab = rng.integers(0, num_classes, g)
        gdif = rng.random(g) < difficult_rate
        gt.append((gbox, glab, gdif))
        k = int(rng.poisson(dets_per_gt * max(g, 1)))
        src = rng.integers(0, max(g, 1), k)
        if g:
            base = gbox[src] + rng.normal(0, 6, (k, 4))
            lab = np.where(rng.random(k) < 0.85, glab[src], rng.integers(0, num_classes, k))
        else:
            base = np.zeros((k, 4))
            lab = rng.integers(0, num_classes, k)
        clutter = rng.random(k) < 0.3
        cx, cy = rng.uniform(0, w, k), rng.uniform(0, h, k)
        base[clutter] = np.stack([cx, cy, cx + rng.uniform(1, 150, k), cy + rng.uniform(1, 150, k)], 1)[clutter]
        b = (base - 1).astype(np.float32)             # the writer adds 1 back
        s = (rng.integers(1, score_levels + 1, k) / score_levels).astype(np.float32)
        dets.append((b, s, lab.astype(np.int64)))
    return dets, gt
