"""The COCO AP restatement (oracle/coco_eval.py): the literal pycocotools transcription and the vectorised form on
arena rows agree bit for bit, and both give the answers derived by hand from COCOeval's definition.  CPU only."""
import numpy as np
import pytest

from oracle import coco_eval as O

P1 = 1 / (1 + np.spacing(1))        # pr of one TP and no FP: tp / ((fp + tp) + 2^-52), just below 1
P_HALF = 1 / (2 + np.spacing(1))    # one TP after one FP


def _gt(anns, cats=(1,), images=(1,)):
    out = {'images': [{'id': i} for i in images], 'categories': [{'id': c} for c in cats], 'annotations': []}
    for j, a in enumerate(anns):
        x, y, w, h = a['bbox']
        out['annotations'].append({'id': j + 1, 'image_id': a.get('image_id', images[0]),
                                   'category_id': a.get('category_id', cats[0]), 'bbox': [x, y, w, h],
                                   'area': a.get('area', float(w * h)), 'iscrowd': a.get('iscrowd', 0)})
    return out


def _det(boxes, scores, cls):
    return (np.asarray(boxes, np.float32).reshape(-1, 4), np.asarray(scores, np.float32), np.asarray(cls, np.int64))


def _both(dets, gt, image_ids, class_ids):
    """Literal (on the JSON results) and vectorised (on arena rows) results, checked bit for bit against each other."""
    lit = O.coco_eval_literal(gt, O.result_json(dets, image_ids, class_ids), image_ids)
    vec = O.coco_eval_rows(O.arena_rows(dets), image_ids, gt, class_ids)
    for name, a, b in zip(("stats", "precision", "recall"), lit, vec):
        assert a.shape == b.shape, name
        assert np.array_equal(a.view(np.int64), b.view(np.int64)), (name, np.argwhere(a != b)[:5])
    return lit


def test_one_perfect_small_detection():
    gt = _gt([{'bbox': [0, 0, 10, 10]}])
    stats, prec, rec = _both([_det([[0, 0, 10, 10]], [0.9], [0])], gt, [1], [1])
    assert np.all(prec[:, :, 0, 0:2, :] == P1) and np.all(prec[:, :, 0, 2:, :] == -1)
    assert np.all(rec[:, 0, 0:2, :] == 1) and np.all(rec[:, 0, 2:, :] == -1)
    want = np.array([1, 1, 1, 1, -1, -1, 1, 1, 1, 1, -1, -1], float)
    np.testing.assert_allclose(stats, want, rtol=0, atol=4e-16)


def test_iou_exactly_one_half():
    """GT [0,0,10,10] against the detection [0,0,10,5]: IoU = 50 / (100 + 50 - 50) = 0.5, a TP at t = 0.5 only."""
    gt = _gt([{'bbox': [0, 0, 10, 10]}])
    stats, prec, rec = _both([_det([[0, 0, 10, 5]], [0.9], [0])], gt, [1], [1])
    assert np.all(prec[0, :, 0, 0, :] == P1) and np.all(prec[1:, :, 0, 0, :] == 0)
    assert np.all(rec[0, 0, 0, :] == 1) and np.all(rec[1:, 0, 0, :] == 0)
    np.testing.assert_allclose(stats[:3], [0.1, 1, 0], rtol=0, atol=4e-16)


def test_false_positive_above_a_true_positive():
    gt = _gt([{'bbox': [0, 0, 10, 10]}])
    dets = [_det([[50, 50, 60, 60], [0, 0, 10, 10]], [0.9, 0.8], [0, 0])]
    stats, prec, rec = _both(dets, gt, [1], [1])
    assert np.all(prec[:, :, 0, 0, 1:] == P_HALF)       # maxDets 10 and 100: the envelope is 1/2 at every recall
    assert np.all(prec[:, :, 0, 0, 0] == 0)             # maxDets 1: only the FP
    assert stats[6] == 0 and stats[8] == 1              # AR@1, AR@100


def test_detection_inside_a_crowd_box_is_ignored():
    """A detection inside a crowd GT has IoU 1 (the detection's area is the union) and is ignored at every
    threshold: the TP below it keeps precision P1 (an FP above it would give 1/2)."""
    gt = _gt([{'bbox': [0, 0, 100, 100], 'iscrowd': 1}, {'bbox': [200, 200, 10, 10]}])
    dets = [_det([[10, 10, 30, 30], [200, 200, 210, 210]], [0.9, 0.8], [0, 0])]
    stats, prec, rec = _both(dets, gt, [1], [1])
    assert np.all(prec[:, :, 0, 0, 1:] == P1)
    assert np.all(prec[:, :, 0, 0, 0] == 0) and np.all(rec[:, 0, 0, 0] == 0)   # maxDets 1 keeps only the ignored one
    only_crowd = _gt([{'bbox': [0, 0, 100, 100], 'iscrowd': 1}])
    stats, prec, rec = _both([dets[0]], only_crowd, [1], [1])
    assert np.all(prec == -1) and np.all(stats == -1)     # no non-ignored GT anywhere


def test_gt_of_area_1024_counts_small_and_medium():
    gt = _gt([{'bbox': [0, 0, 32, 32]}])
    stats, prec, rec = _both([_det([[0, 0, 32, 32]], [0.5], [0])], gt, [1], [1])
    assert np.all(prec[:, :, 0, 1:3, :] == P1) and np.all(prec[:, :, 0, 3, :] == -1)
    np.testing.assert_allclose(stats[3:6], [1, 1, -1], rtol=0, atol=4e-16)


def test_category_with_gt_but_no_detections_has_precision_zero():
    gt = _gt([{'bbox': [0, 0, 10, 10], 'category_id': 1}, {'bbox': [0, 0, 50, 50], 'category_id': 2}], cats=(1, 2))
    stats, prec, rec = _both([_det([[0, 0, 10, 10]], [0.9], [0])], gt, [1], [1, 2])
    assert np.all(prec[:, :, 1, 0, :] == 0) and np.all(rec[:, 1, 0, :] == 0)
    assert np.all(prec[:, :, 0, 0, :] == P1)


def _edge_set():
    """Several hundred GT in one cell, > 100 detections in a cell, equal IoU against two GT, score ties within and
    across images, an image without GT, one without detections, one with neither, a class outside the GT
    categories, image ids out of order."""
    rng = np.random.default_rng(5)
    image_ids = [42, 7, 19, 3, 100]
    cats = (1, 5, 9)
    anns = []
    for j in range(300):                                              # image 42, category 5: 300 GT
        x, y = float(rng.integers(0, 600)), float(rng.integers(0, 600))
        anns.append({'image_id': 42, 'category_id': 5, 'bbox': [x, y, 20.0, 20.0], 'iscrowd': int(j % 37 == 0)})
    anns += [{'image_id': 7, 'category_id': 1, 'bbox': [0, 0, 10, 10]},
             {'image_id': 7, 'category_id': 1, 'bbox': [0, 0, 10, 10]},               # equal IoU: the later GT wins
             {'image_id': 7, 'category_id': 1, 'bbox': [100, 100, 96, 96]},           # area 96^2
             {'image_id': 7, 'category_id': 1, 'bbox': [300, 300, 32, 32], 'area': 1024.0},
             {'image_id': 7, 'category_id': 9, 'bbox': [0, 0, 400, 400], 'iscrowd': 1},
             {'image_id': 3, 'category_id': 9, 'bbox': [5, 5, 50, 50], 'area': 20000.0},  # out-of-range area
             {'image_id': 3, 'category_id': 9, 'bbox': [5, 5, 50, 50]}]
    gt = _gt(anns, cats=cats, images=image_ids + [555])
    d42 = rng.uniform(0, 600, (160, 2))
    d42 = np.concatenate([d42, d42 + rng.uniform(5, 30, (160, 2))], 1)
    dets = [
        _det(d42, np.round(rng.uniform(0, 1, 160) * 8) / 8, np.full(160, 1)),
        _det([[0, 0, 10, 10], [0, 0, 10, 10], [0, 0, 10, 5], [100, 100, 196, 196], [300, 300, 332, 332],
              [0, 0, 10, 7.5], [10, 10, 100, 100], [20, 20, 30, 30]],
             [0.5, 0.5, 0.5, 0.25, 0.25, 0.5, 0.125, 0.5], [0, 0, 0, 0, 0, 0, 2, 3]),
        _det([[10, 10, 20, 20]], [0.5], [0]),                            # image 19: no GT
        _det(np.zeros((0, 4)), [], []),                                  # image 3: GT, no detections
        _det(np.zeros((0, 4)), [], []),                                  # image 100: neither
    ]
    class_ids = [1, 5, 9, 77]
    return dets, gt, image_ids, class_ids


def test_edge_set_literal_equals_vectorised():
    dets, gt, image_ids, class_ids = _edge_set()
    stats, prec, rec = _both(dets, gt, image_ids, class_ids)
    assert (prec > 0).any() and (stats > 0).any()


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_random_tie_heavy_sets(seed):
    dets, gt, image_ids, class_ids = O.random_set(60, 6, seed=seed, max_gt=10, score_levels=6)
    stats, prec, rec = _both(dets, gt, image_ids, class_ids)
    assert (prec > 0).any()


def test_package_summarize_and_gt_packing():
    """The package's host half: summarize equals the literal one bit for bit, and pack_gt refuses what COCOeval
    would mis-read."""
    from yolo_nano_b200 import coco_eval as P
    from yolo_nano_b200.engine import EngineError
    dets, gt, image_ids, class_ids = O.random_set(40, 5, seed=9)
    _, prec, rec = O.coco_eval_rows(O.arena_rows(dets), image_ids, gt, class_ids)
    assert np.array_equal(P.summarize(prec, rec), O.summarize(prec, rec))
    assert np.array_equal(P.IOU_THRS, O.IOU_THRS) and np.array_equal(P.REC_THRS, O.REC_THRS)
    p, K = P.pack_gt(gt, image_ids, class_ids, 5)
    assert K == len(gt['categories']) and p['start'][-1] == len(p['area'])
    assert list(p['image_rank']) == list(np.argsort(np.argsort(image_ids)))
    with pytest.raises(EngineError):
        P.pack_gt(gt, image_ids[:-1] + image_ids[:1], class_ids, 5)              # duplicate image id
    with pytest.raises(EngineError):
        P.pack_gt(gt, image_ids[:-1] + [10 ** 9], class_ids, 5)                 # not a GT image
    bad = {**gt, 'annotations': [dict(a) for a in gt['annotations']]}
    bad['annotations'][0]['id'] = 0
    with pytest.raises(EngineError):
        P.pack_gt(bad, image_ids, class_ids, 5)
    del bad['annotations'][0]['iscrowd']
    bad['annotations'][0]['id'] = 10 ** 6
    with pytest.raises(EngineError):
        P.pack_gt(bad, image_ids, class_ids, 5)
