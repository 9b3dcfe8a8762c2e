"""Restatement of the reference's COCO AP (evaluator/cocoapi_evaluator.py: the results JSON, `cocoGt.loadRes`, then
pycocotools' `COCOeval(cocoGt, cocoDt, 'bbox')` with `params.imgIds = ids`, evaluate / accumulate / summarize) — the
checker of yolo_nano_b200.coco_eval, never its path.

Two forms:
  * `coco_eval_literal`  the parts of pycocotools 2.0 that 'bbox' uses, line by line and named after them: COCO's
                         index (createIndex, getAnnIds / loadAnns order), loadRes, COCOeval._prepare, computeIoU with
                         maskUtils.iou's bbIou in Python floats, evaluateImg, accumulate and summarize.  It runs on the
                         JSON round trip of evalfmt.coco_result_rows (pinned to the real evaluator by golden g6).
  * `arena_rows` + `coco_eval_rows`  the same arrays from int32 results rows (the device's arena format),
                         vectorised over cells for million-row sets.  evaluateImg's greedy scan becomes: among GT not
                         yet matched at (t, a) (crowd GT stay available) with IoU >= min(t, 1 - 1e-10), the largest IoU
                         among non-ignored GT, the later one on equal IoU; only if there is none, the same among
                         ignored GT.
pycocotools is not a dependency of this project, and no golden from the real COCOeval has pinned this restatement
yet: `python -m oracle.gen_coco_golden` records one wherever pycocotools is installed.  Until then it rests on the
pycocotools 2.0 sources it transcribes and on hand-derived known answers (tests/test_coco_eval_oracle.py).
"""
from __future__ import annotations

import copy
import itertools
import json
from collections import defaultdict
from typing import Dict, List, Sequence, Tuple

import numpy as np

IOU_THRS = np.linspace(.5, 0.95, int(np.round((0.95 - .5) / .05)) + 1, endpoint=True)
REC_THRS = np.linspace(.0, 1.00, int(np.round((1.00 - .0) / .01)) + 1, endpoint=True)
MAX_DETS = [1, 10, 100]
AREA_RNG = [[0 ** 2, 1e5 ** 2], [0 ** 2, 32 ** 2], [32 ** 2, 96 ** 2], [96 ** 2, 1e5 ** 2]]
AREA_RNG_LBL = ['all', 'small', 'medium', 'large']


# ---- the literal form ---------------------------------------------------------------------------------------------
class COCO:
    """pycocotools.coco.COCO: the index and the calls COCOeval makes."""

    def __init__(self, dataset: Dict):
        self.dataset = dataset
        self.createIndex()

    def createIndex(self):
        anns, cats, imgs = {}, {}, {}
        imgToAnns, catToImgs = defaultdict(list), defaultdict(list)
        if 'annotations' in self.dataset:
            for ann in self.dataset['annotations']:
                imgToAnns[ann['image_id']].append(ann)
                anns[ann['id']] = ann
        if 'images' in self.dataset:
            for img in self.dataset['images']:
                imgs[img['id']] = img
        if 'categories' in self.dataset:
            for cat in self.dataset['categories']:
                cats[cat['id']] = cat
        if 'annotations' in self.dataset and 'categories' in self.dataset:
            for ann in self.dataset['annotations']:
                catToImgs[ann['category_id']].append(ann['image_id'])
        self.anns, self.imgToAnns, self.catToImgs, self.imgs, self.cats = anns, imgToAnns, catToImgs, imgs, cats

    def getAnnIds(self, imgIds=[], catIds=[], areaRng=[], iscrowd=None):
        imgIds = imgIds if _isArrayLike(imgIds) else [imgIds]
        catIds = catIds if _isArrayLike(catIds) else [catIds]
        if len(imgIds) == len(catIds) == len(areaRng) == 0:
            anns = self.dataset['annotations']
        else:
            if not len(imgIds) == 0:
                lists = [self.imgToAnns[imgId] for imgId in imgIds if imgId in self.imgToAnns]
                anns = list(itertools.chain.from_iterable(lists))
            else:
                anns = self.dataset['annotations']
            anns = anns if len(catIds) == 0 else [ann for ann in anns if ann['category_id'] in catIds]
            anns = anns if len(areaRng) == 0 else [ann for ann in anns if ann['area'] > areaRng[0] and
                                                   ann['area'] < areaRng[1]]
        if iscrowd is not None:
            ids = [ann['id'] for ann in anns if ann['iscrowd'] == iscrowd]
        else:
            ids = [ann['id'] for ann in anns]
        return ids

    def getCatIds(self):
        return [cat['id'] for cat in self.dataset['categories']]

    def getImgIds(self):
        return self.imgs.keys()

    def loadAnns(self, ids=[]):
        if _isArrayLike(ids):
            return [self.anns[id] for id in ids]
        elif type(ids) == int:
            return [self.anns[ids]]

    def loadRes(self, anns: List[Dict]):
        """loadRes for a list of bbox results (the JSON file already parsed)."""
        res = COCO({'images': [img for img in self.dataset['images']]})
        assert type(anns) == list, 'results in not an array of objects'
        annsImgIds = [ann['image_id'] for ann in anns]
        assert set(annsImgIds) == (set(annsImgIds) & set(self.getImgIds())), \
            'Results do not correspond to current coco set'
        assert 'bbox' in anns[0] and not anns[0]['bbox'] == []
        res.dataset['categories'] = copy.deepcopy(self.dataset['categories'])
        for id, ann in enumerate(anns):
            bb = ann['bbox']
            x1, x2, y1, y2 = [bb[0], bb[0] + bb[2], bb[1], bb[1] + bb[3]]
            if 'segmentation' not in ann:
                ann['segmentation'] = [[x1, y1, x1, y2, x2, y2, x2, y1]]
            ann['area'] = bb[2] * bb[3]
            ann['id'] = id + 1
            ann['iscrowd'] = 0
        res.dataset['annotations'] = anns
        res.createIndex()
        return res


def _isArrayLike(obj):
    return hasattr(obj, '__iter__') and hasattr(obj, '__len__')


def bbIou(dt, gt, iscrowd) -> np.ndarray:
    """maskUtils.iou for boxes (common/maskApi.c bbIou) in Python floats; [D, G]."""
    m, n = len(dt), len(gt)
    o = np.zeros((m, n))
    for g in range(n):
        G = gt[g]
        ga = G[2] * G[3]
        crowd = iscrowd[g]
        for d in range(m):
            D = dt[d]
            da = D[2] * D[3]
            w = min(D[2] + D[0], G[2] + G[0]) - max(D[0], G[0])
            if w <= 0:
                continue
            h = min(D[3] + D[1], G[3] + G[1]) - max(D[1], G[1])
            if h <= 0:
                continue
            i = w * h
            u = da if crowd else da + ga - i
            o[d, g] = i / u
    return o


class Params:
    def __init__(self):
        self.imgIds = []
        self.catIds = []
        self.iouThrs = IOU_THRS
        self.recThrs = REC_THRS
        self.maxDets = list(MAX_DETS)
        self.areaRng = [list(a) for a in AREA_RNG]
        self.areaRngLbl = list(AREA_RNG_LBL)
        self.useCats = 1


class COCOeval:
    def __init__(self, cocoGt, cocoDt):
        self.cocoGt, self.cocoDt = cocoGt, cocoDt
        self.params = Params()
        self.params.imgIds = sorted(cocoGt.getImgIds())
        self.params.catIds = sorted(cocoGt.getCatIds())

    def _prepare(self):
        p = self.params
        gts = self.cocoGt.loadAnns(self.cocoGt.getAnnIds(imgIds=p.imgIds, catIds=p.catIds))
        dts = self.cocoDt.loadAnns(self.cocoDt.getAnnIds(imgIds=p.imgIds, catIds=p.catIds))
        for gt in gts:
            gt['ignore'] = gt['ignore'] if 'ignore' in gt else 0
            gt['ignore'] = 'iscrowd' in gt and gt['iscrowd']
        self._gts = defaultdict(list)
        self._dts = defaultdict(list)
        for gt in gts:
            self._gts[gt['image_id'], gt['category_id']].append(gt)
        for dt in dts:
            self._dts[dt['image_id'], dt['category_id']].append(dt)
        self.evalImgs = defaultdict(list)
        self.eval = {}

    def evaluate(self):
        p = self.params
        p.imgIds = list(np.unique(p.imgIds))
        p.maxDets = sorted(p.maxDets)
        self.params = p
        self._prepare()
        catIds = p.catIds
        self.ious = {(imgId, catId): self.computeIoU(imgId, catId) for imgId in p.imgIds for catId in catIds}
        maxDet = p.maxDets[-1]
        self.evalImgs = [self.evaluateImg(imgId, catId, areaRng, maxDet)
                         for catId in catIds for areaRng in p.areaRng for imgId in p.imgIds]
        self._paramsEval = copy.deepcopy(self.params)

    def computeIoU(self, imgId, catId):
        p = self.params
        gt = self._gts[imgId, catId]
        dt = self._dts[imgId, catId]
        if len(gt) == 0 and len(dt) == 0:
            return []
        inds = np.argsort([-d['score'] for d in dt], kind='mergesort')
        dt = [dt[i] for i in inds]
        if len(dt) > p.maxDets[-1]:
            dt = dt[0:p.maxDets[-1]]
        g = [g['bbox'] for g in gt]
        d = [d['bbox'] for d in dt]
        iscrowd = [int(o['iscrowd']) for o in gt]
        if len(d) == 0 or len(g) == 0:
            return []
        return bbIou(d, g, iscrowd)

    def evaluateImg(self, imgId, catId, aRng, maxDet):
        p = self.params
        gt = self._gts[imgId, catId]
        dt = self._dts[imgId, catId]
        if len(gt) == 0 and len(dt) == 0:
            return None
        for g in gt:
            if g['ignore'] or (g['area'] < aRng[0] or g['area'] > aRng[1]):
                g['_ignore'] = 1
            else:
                g['_ignore'] = 0
        gtind = np.argsort([g['_ignore'] for g in gt], kind='mergesort')
        gt = [gt[i] for i in gtind]
        dtind = np.argsort([-d['score'] for d in dt], kind='mergesort')
        dt = [dt[i] for i in dtind[0:maxDet]]
        iscrowd = [int(o['iscrowd']) for o in gt]
        ious = self.ious[imgId, catId][:, gtind] if len(self.ious[imgId, catId]) > 0 else self.ious[imgId, catId]
        T = len(p.iouThrs)
        G = len(gt)
        D = len(dt)
        gtm = np.zeros((T, G))
        dtm = np.zeros((T, D))
        gtIg = np.array([g['_ignore'] for g in gt])
        dtIg = np.zeros((T, D))
        if not len(ious) == 0:
            for tind, t in enumerate(p.iouThrs):
                for dind, d in enumerate(dt):
                    iou = min([t, 1 - 1e-10])
                    m = -1
                    for gind, g in enumerate(gt):
                        if gtm[tind, gind] > 0 and not iscrowd[gind]:
                            continue
                        if m > -1 and gtIg[m] == 0 and gtIg[gind] == 1:
                            break
                        if ious[dind, gind] < iou:
                            continue
                        iou = ious[dind, gind]
                        m = gind
                    if m == -1:
                        continue
                    dtIg[tind, dind] = gtIg[m]
                    dtm[tind, dind] = gt[m]['id']
                    gtm[tind, m] = d['id']
        a = np.array([d['area'] < aRng[0] or d['area'] > aRng[1] for d in dt]).reshape((1, len(dt)))
        dtIg = np.logical_or(dtIg, np.logical_and(dtm == 0, np.repeat(a, T, 0)))
        return {'image_id': imgId, 'category_id': catId, 'aRng': aRng, 'maxDet': maxDet,
                'dtIds': [d['id'] for d in dt], 'gtIds': [g['id'] for g in gt], 'dtMatches': dtm, 'gtMatches': gtm,
                'dtScores': [d['score'] for d in dt], 'gtIgnore': gtIg, 'dtIgnore': dtIg}

    def accumulate(self):
        p = self.params
        T = len(p.iouThrs)
        R = len(p.recThrs)
        K = len(p.catIds)
        A = len(p.areaRng)
        M = len(p.maxDets)
        precision = -np.ones((T, R, K, A, M))
        recall = -np.ones((T, K, A, M))
        _pe = self._paramsEval
        catIds = _pe.catIds
        setK = set(catIds)
        setA = set(map(tuple, _pe.areaRng))
        setM = set(_pe.maxDets)
        setI = set(_pe.imgIds)
        k_list = [n for n, k in enumerate(p.catIds) if k in setK]
        m_list = [m for n, m in enumerate(p.maxDets) if m in setM]
        a_list = [n for n, a in enumerate(map(lambda x: tuple(x), p.areaRng)) if a in setA]
        i_list = [n for n, i in enumerate(p.imgIds) if i in setI]
        I0 = len(_pe.imgIds)
        A0 = len(_pe.areaRng)
        for k, k0 in enumerate(k_list):
            Nk = k0 * A0 * I0
            for a, a0 in enumerate(a_list):
                Na = a0 * I0
                for m, maxDet in enumerate(m_list):
                    E = [self.evalImgs[Nk + Na + i] for i in i_list]
                    E = [e for e in E if e is not None]
                    if len(E) == 0:
                        continue
                    dtScores = np.concatenate([e['dtScores'][0:maxDet] for e in E])
                    inds = np.argsort(-dtScores, kind='mergesort')
                    dtm = np.concatenate([e['dtMatches'][:, 0:maxDet] for e in E], axis=1)[:, inds]
                    dtIg = np.concatenate([e['dtIgnore'][:, 0:maxDet] for e in E], axis=1)[:, inds]
                    gtIg = np.concatenate([e['gtIgnore'] for e in E])
                    npig = np.count_nonzero(gtIg == 0)
                    if npig == 0:
                        continue
                    tps = np.logical_and(dtm, np.logical_not(dtIg))
                    fps = np.logical_and(np.logical_not(dtm), np.logical_not(dtIg))
                    tp_sum = np.cumsum(tps, axis=1).astype(dtype=np.float64)
                    fp_sum = np.cumsum(fps, axis=1).astype(dtype=np.float64)
                    for t, (tp, fp) in enumerate(zip(tp_sum, fp_sum)):
                        tp = np.array(tp)
                        fp = np.array(fp)
                        nd = len(tp)
                        rc = tp / npig
                        pr = tp / (fp + tp + np.spacing(1))
                        q = np.zeros((R,))
                        if nd:
                            recall[t, k, a, m] = rc[-1]
                        else:
                            recall[t, k, a, m] = 0
                        pr = pr.tolist()
                        q = q.tolist()
                        for i in range(nd - 1, 0, -1):
                            if pr[i] > pr[i - 1]:
                                pr[i - 1] = pr[i]
                        inds = np.searchsorted(rc, p.recThrs, side='left')
                        try:
                            for ri, pi in enumerate(inds):
                                q[ri] = pr[pi]
                        except IndexError:
                            pass
                        precision[t, :, k, a, m] = np.array(q)
        self.eval = {'params': p, 'counts': [T, R, K, A, M], 'precision': precision, 'recall': recall}

    def summarize(self):
        def _summarize(ap=1, iouThr=None, areaRng='all', maxDets=100):
            p = self.params
            aind = [i for i, aRng in enumerate(p.areaRngLbl) if aRng == areaRng]
            mind = [i for i, mDet in enumerate(p.maxDets) if mDet == maxDets]
            if ap == 1:
                s = self.eval['precision']
                if iouThr is not None:
                    t = np.where(iouThr == p.iouThrs)[0]
                    s = s[t]
                s = s[:, :, :, aind, mind]
            else:
                s = self.eval['recall']
                if iouThr is not None:
                    t = np.where(iouThr == p.iouThrs)[0]
                    s = s[t]
                s = s[:, :, aind, mind]
            if len(s[s > -1]) == 0:
                mean_s = -1
            else:
                mean_s = np.mean(s[s > -1])
            return mean_s

        def _summarizeDets():
            stats = np.zeros((12,))
            stats[0] = _summarize(1)
            stats[1] = _summarize(1, iouThr=.5, maxDets=self.params.maxDets[2])
            stats[2] = _summarize(1, iouThr=.75, maxDets=self.params.maxDets[2])
            stats[3] = _summarize(1, areaRng='small', maxDets=self.params.maxDets[2])
            stats[4] = _summarize(1, areaRng='medium', maxDets=self.params.maxDets[2])
            stats[5] = _summarize(1, areaRng='large', maxDets=self.params.maxDets[2])
            stats[6] = _summarize(0, maxDets=self.params.maxDets[0])
            stats[7] = _summarize(0, maxDets=self.params.maxDets[1])
            stats[8] = _summarize(0, maxDets=self.params.maxDets[2])
            stats[9] = _summarize(0, areaRng='small', maxDets=self.params.maxDets[2])
            stats[10] = _summarize(0, areaRng='medium', maxDets=self.params.maxDets[2])
            stats[11] = _summarize(0, areaRng='large', maxDets=self.params.maxDets[2])
            return stats
        self.stats = _summarizeDets()


def summarize(precision: np.ndarray, recall: np.ndarray) -> np.ndarray:
    """COCOeval.summarize on given arrays (the literal code, with the default params)."""
    E = COCOeval.__new__(COCOeval)
    E.params = Params()
    E.eval = {'precision': precision, 'recall': recall}
    E.summarize()
    return E.stats


def result_json(dets, image_ids: Sequence[int], class_ids: Sequence[int]) -> List[Dict]:
    """The reference's results file, parsed back: evalfmt.coco_result_rows per image (dets[i] = (pixel boxes f32
    [K,4], scores f32 [K], cls [K]) of image image_ids[i]) through json.dumps / json.loads."""
    from yolo_nano_b200 import evalfmt
    rows = []
    for (b, s, c), iid in zip(dets, image_ids):
        rows += evalfmt.coco_result_rows(int(iid), np.asarray(b, np.float32).reshape(-1, 4),
                                         np.asarray(s, np.float32), np.asarray(c), class_ids)
    return json.loads(json.dumps(rows))


def coco_eval_literal(gt_dataset: Dict, result_rows: List[Dict], image_ids: Sequence[int]):
    """COCOAPIEvaluator.evaluate after detection: loadRes, COCOeval 'bbox' with params.imgIds = image_ids,
    evaluate / accumulate / summarize.  Returns (stats [12], precision [T,R,K,A,M], recall [T,K,A,M])."""
    cocoGt = COCO(copy.deepcopy(gt_dataset))
    cocoDt = cocoGt.loadRes(copy.deepcopy(result_rows))
    cocoEval = COCOeval(cocoGt, cocoDt)
    cocoEval.params.imgIds = list(image_ids)
    cocoEval.evaluate()
    cocoEval.accumulate()
    cocoEval.summarize()
    return cocoEval.stats, cocoEval.eval['precision'], cocoEval.eval['recall']


# ---- the vectorised form on arena rows ----------------------------------------------------------------------------
def arena_rows(dets) -> np.ndarray:
    """Results entries as int32 rows [image, class, score bits, x1, y1, x2, y2 bits] in file order (image, kept row):
    dets[i] = (pixel boxes f32 [K,4], scores f32 [K], cls [K]) of the i-th added image."""
    out = []
    for i, (b, s, c) in enumerate(dets):
        b = np.asarray(b, np.float32).reshape(-1, 4)
        r = np.empty((len(b), 7), np.int32)
        r[:, 0] = i
        r[:, 1] = np.asarray(c).reshape(-1)
        r[:, 2] = np.asarray(s, np.float32).reshape(-1).view(np.int32)
        r[:, 3:] = b.view(np.int32)
        out.append(r)
    return np.concatenate(out or [np.zeros((0, 7), np.int32)])


def _gt_cells(gt: Dict, uniq: np.ndarray, cat_ids: List[int]):
    """GT of the evaluated images and categories in annotation order, stable-sorted by cell (rank, k)."""
    rank = {int(i): r for r, i in enumerate(uniq)}
    kix = {c: k for k, c in enumerate(cat_ids)}
    K = len(cat_ids)
    cell, box, area, crowd = [], [], [], []
    for a in gt.get('annotations', []):
        r, k = rank.get(a['image_id']), kix.get(a['category_id'])
        if r is None or k is None:
            continue
        cell.append(r * K + k)
        box.append(a['bbox'])
        area.append(a['area'])
        crowd.append(bool(a['iscrowd']))
    cell = np.asarray(cell, np.int64)
    o = np.argsort(cell, kind='stable')
    return (cell[o], np.asarray(box, np.float64).reshape(-1, 4)[o], np.asarray(area, np.float64)[o],
            np.asarray(crowd, bool)[o])


def _bbiou_vec(d, g, crowd):
    """bbIou elementwise on broadcast [..., 4] xywh arrays (the same float64 operations)."""
    da = d[..., 2] * d[..., 3]
    ga = g[..., 2] * g[..., 3]
    w = np.minimum(d[..., 2] + d[..., 0], g[..., 2] + g[..., 0]) - np.maximum(d[..., 0], g[..., 0])
    h = np.minimum(d[..., 3] + d[..., 1], g[..., 3] + g[..., 1]) - np.maximum(d[..., 1], g[..., 1])
    i = w * h
    u = np.where(crowd, da, da + ga - i)
    with np.errstate(invalid='ignore', divide='ignore'):
        return np.where((w > 0) & (h > 0), i / u, 0.0)


def _last_argmax(x):
    return x.shape[-1] - 1 - np.argmax(x[..., ::-1], axis=-1)


def coco_eval_rows(rows: np.ndarray, image_ids: Sequence[int], gt: Dict, class_ids: Sequence[int],
                   cell_budget: int = 1 << 22):
    """COCOeval 'bbox' from int32 arena rows (image = add index into image_ids).  Returns (stats [12],
    precision [T,R,K,A,M], recall [T,K,A,M])."""
    rows = np.asarray(rows, np.int32).reshape(-1, 7)
    T, R, A, M = len(IOU_THRS), len(REC_THRS), len(AREA_RNG), len(MAX_DETS)
    ids = np.asarray(image_ids, np.int64)
    uniq = np.unique(ids)
    cat_ids = sorted(c['id'] for c in gt['categories'])
    K = len(cat_ids)
    kix = {c: k for k, c in enumerate(cat_ids)}
    class_cat = np.array([kix.get(int(c), -1) for c in class_ids], np.int64)
    rank_of_add = np.searchsorted(uniq, ids)
    f = rows[:, 2:7].copy().view(np.float32).astype(np.float64)
    score = f[:, 0]
    box = np.stack([f[:, 1], f[:, 2], f[:, 3] - f[:, 1], f[:, 4] - f[:, 2]], 1)    # loadRes' xywh
    darea = box[:, 2] * box[:, 3]
    kd = class_cat[rows[:, 1]] if len(rows) else np.zeros(0, np.int64)
    sel = np.nonzero(kd >= 0)[0]
    cellkey = rank_of_add[rows[sel, 0]] * K + kd[sel]
    # cell order: (rank, k), score descending, file order; the first 100 of each cell
    o = np.lexsort((-score[sel], cellkey))
    order, ck = sel[o], cellkey[o]
    _, first, inv = np.unique(ck, return_index=True, return_inverse=True)
    pos = np.arange(len(order)) - first[inv]
    keep = pos < MAX_DETS[-1]
    order, ck, pos = order[keep], ck[keep], pos[keep]
    nk = len(order)
    # GT cells
    gcell, gbox, garea, gcrowd = _gt_cells(gt, uniq, cat_ids)
    lo = np.array([a[0] for a in AREA_RNG], np.float64)
    hi = np.array([a[1] for a in AREA_RNG], np.float64)
    gign = gcrowd[None, :] | (garea[None, :] < lo[:, None]) | (garea[None, :] > hi[:, None])       # [A, G]
    npig = np.zeros((K, A), np.int64)
    for a in range(A):
        np.add.at(npig[:, a], gcell[~gign[a]] % K, 1)
    # evaluateImg: per kept detection, TP / ignored per (a, t)
    tp = np.zeros((nk, A, T), bool)
    ig = np.zeros((nk, A, T), bool)
    dout = (darea[order][:, None] < lo[None, :]) | (darea[order][:, None] > hi[None, :])            # [nk, A]
    t_eff = np.minimum(IOU_THRS, 1 - 1e-10)
    cells, cstart, cnt = np.unique(ck, return_index=True, return_counts=True)
    gs = np.searchsorted(gcell, cells, 'left')
    gn = np.searchsorted(gcell, cells, 'right') - gs
    with_gt = np.nonzero(gn > 0)[0]
    gpad = 1 << np.ceil(np.log2(np.maximum(gn[with_gt], 1))).astype(np.int64)
    for gp in np.unique(gpad):
        bucket = with_gt[gpad == gp]
        step = max(1, cell_budget // (MAX_DETS[-1] * int(gp) * A * T))
        for c0 in range(0, len(bucket), step):
            cb = bucket[c0:c0 + step]
            C, Dm = len(cb), int(cnt[cb].max())
            di = cstart[cb][:, None] + np.arange(Dm)[None, :]
            dvalid = np.arange(Dm)[None, :] < cnt[cb][:, None]
            di = np.where(dvalid, di, cstart[cb][:, None])
            gi = gs[cb][:, None] + np.arange(gp)[None, :]
            gvalid = np.arange(gp)[None, :] < gn[cb][:, None]
            gi = np.where(gvalid, gi, gs[cb][:, None])
            iou = _bbiou_vec(box[order[di]][:, :, None, :], gbox[gi][:, None, :, :], gcrowd[gi][:, None, :])
            crowd = gcrowd[gi]                                                           # [C, G]
            ign = gign[:, gi].transpose(1, 0, 2)                                         # [C, A, G]
            matched = np.zeros((C, A, T, gp), bool)
            for d in range(Dm):
                v = iou[:, d, :][:, None, None, :]
                elig = (gvalid[:, None, None, :] & ~(matched & ~crowd[:, None, None, :])
                        & (v >= t_eff[None, None, :, None]))
                g1 = elig & ~ign[:, :, None, :]
                g2 = elig & ign[:, :, None, :]
                has1, has2 = g1.any(-1), g2.any(-1)
                m1 = _last_argmax(np.where(g1, v, -1.0))
                m2 = _last_argmax(np.where(g2, v, -1.0))
                mm = np.where(has1, m1, m2)
                hit = (has1 | has2) & dvalid[:, d][:, None, None]
                mark = hit & ~np.take_along_axis(np.broadcast_to(crowd[:, None, None, :], matched.shape),
                                                  mm[..., None], -1)[..., 0]
                cc, aa, tt = np.nonzero(mark)
                matched[cc, aa, tt, mm[cc, aa, tt]] = True
                rows_d = di[:, d][dvalid[:, d]]
                tp[rows_d] = has1[dvalid[:, d]]
                ig[rows_d] = has2[dvalid[:, d]] & ~has1[dvalid[:, d]]
    ig |= ~tp & ~ig & dout[:, :, None] if nk else ig
    # accumulate: per category, the cell order stable-sorted by score
    kk = ck % K if nk else np.zeros(0, np.int64)
    o2 = np.lexsort((-score[order], kk))
    kk2 = kk[o2]
    precision = -np.ones((T, R, K, A, M))
    recall = -np.ones((T, K, A, M))
    for k in range(K):
        idx = o2[np.searchsorted(kk2, k, 'left'):np.searchsorted(kk2, k, 'right')]
        for a in range(A):
            if npig[k, a] == 0:
                continue
            for m, maxDet in enumerate(MAX_DETS):
                sub = idx[pos[idx] < maxDet]
                tps = tp[sub, a, :].T
                fps = ~tps & ~ig[sub, a, :].T
                tp_sum = np.cumsum(tps, axis=1).astype(np.float64)
                fp_sum = np.cumsum(fps, axis=1).astype(np.float64)
                nd = len(sub)
                for t in range(T):
                    rc = tp_sum[t] / npig[k, a]
                    pr = tp_sum[t] / (fp_sum[t] + tp_sum[t] + np.spacing(1))
                    recall[t, k, a, m] = rc[-1] if nd else 0
                    pr = np.maximum.accumulate(pr[::-1])[::-1]
                    inds = np.searchsorted(rc, REC_THRS, side='left')
                    precision[t, :, k, a, m] = np.where(inds < nd, pr[np.minimum(inds, max(nd - 1, 0))] if nd else 0,
                                                        0.0)
    return summarize(precision, recall), precision, recall


# ---- synthetic sets -----------------------------------------------------------------------------------------------
def random_set(n_images: int, num_classes: int, seed: int, max_gt: int = 8, dets_per_gt: float = 3.0,
               crowd_rate: float = 0.05, score_levels: int = 40, num_cats: int = None) -> Tuple[List, Dict, List, List]:
    """A tie-heavy synthetic COCO evaluation: GT boxes on an integer grid (some crowd, areas both from the box and
    given), detections that are jittered copies plus clutter with scores on a coarse grid, image ids shuffled and
    non-contiguous, and class_ids whose last entry is not a GT category.  Returns (dets, gt, image_ids,
    class_ids)."""
    rng = np.random.default_rng(seed)
    num_cats = num_cats or max(num_classes - 1, 1)
    cat_ids = sorted(rng.choice(np.arange(1, 4 * num_classes + 10), num_cats, replace=False).tolist())
    class_ids = cat_ids[:num_classes] + [10_000 + j for j in range(num_classes - len(cat_ids[:num_classes]))]
    image_ids = (rng.permutation(n_images * 3)[:n_images] + 1).tolist()
    gt = {'images': [], 'annotations': [], 'categories': [{'id': int(c), 'name': f'c{c}'} for c in cat_ids]}
    dets = []
    aid = 1
    for i, iid in enumerate(image_ids):
        w, h = (int(v) for v in rng.integers(120, 640, 2))
        gt['images'].append({'id': int(iid), 'width': w, 'height': h})
        g = int(rng.integers(0, max_gt + 1))
        x = rng.integers(0, w - 8, g)
        y = rng.integers(0, h - 8, g)
        bw = rng.integers(2, 160, g)
        bh = rng.integers(2, 160, g)
        glab = rng.integers(0, min(num_classes, len(cat_ids)), g)
        for j in range(g):
            crowd = int(rng.random() < crowd_rate)
            area = float(bw[j] * bh[j]) if rng.random() < 0.5 else float(bw[j] * bh[j]) * float(rng.uniform(0.5, 1))
            gt['annotations'].append({'id': aid, 'image_id': int(iid), 'category_id': int(cat_ids[glab[j]]),
                                      'bbox': [float(x[j]), float(y[j]), float(bw[j]), float(bh[j])], 'area': area,
                                      'iscrowd': crowd})
            aid += 1
        k = int(rng.poisson(dets_per_gt * max(g, 1)))
        src = rng.integers(0, max(g, 1), k)
        if g:
            base = np.stack([x[src], y[src], x[src] + bw[src], y[src] + bh[src]], 1) + rng.normal(0, 4, (k, 4))
            lab = np.where(rng.random(k) < 0.85, glab[src], rng.integers(0, num_classes, k))
        else:
            base = np.zeros((k, 4))
            lab = rng.integers(0, num_classes, k)
        clutter = rng.random(k) < 0.3
        cx, cy = rng.uniform(0, w, k), rng.uniform(0, h, k)
        base[clutter] = np.stack([cx, cy, cx + rng.uniform(1, 150, k), cy + rng.uniform(1, 150, k)], 1)[clutter]
        s = (rng.integers(1, score_levels + 1, k) / score_levels).astype(np.float32)
        dets.append((base.astype(np.float32), s, lab.astype(np.int64)))
    return dets, gt, image_ids, class_ids
