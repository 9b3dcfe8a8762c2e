"""COCO AP on the device (yolo_nano_b200.coco_eval) against the restated COCOeval (oracle/coco_eval.py): the results
rows, precision, recall and all 12 stats bit for bit."""
import contextlib
import io

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import coco_eval as O  # noqa: E402
from oracle import weights as W  # noqa: E402

DEV = torch.device("cuda", 0)


def _model(size, classes, weights):
    import yolo_nano_b200 as pkg
    sd = W.reference_init(classes, seed=3) if weights == "refinit" else W.calibrated(classes, seed=4)
    with contextlib.redirect_stdout(io.StringIO()):
        m = pkg.YOLONano(DEV, size, classes, anchor_size=W.anchors_for(classes))
    m.load_state_dict(sd)
    return m.to(DEV).eval()


def _images(n, seed):
    """Original uint8 BGR images of COCO-like shapes (smooth content, so that detections vary between images)."""
    rng = np.random.default_rng(seed)
    shapes = [(480, 640), (640, 480), (427, 640), (640, 640), (360, 640), (500, 375)]
    out = []
    for i in range(n):
        h, w = shapes[int(rng.integers(len(shapes)))]
        small = rng.integers(0, 256, (h // 16 + 2, w // 16 + 2, 3), dtype=np.uint8)
        out.append(np.ascontiguousarray(np.repeat(np.repeat(small, 16, 0), 16, 1)[:h, :w]))
    return out


def _engine_dets(m, imgs, batch=64):
    """Engine detections after map_boxes, on the device per batch and as host triples."""
    out_dev, host = [], []
    for a in range(0, len(imgs), batch):
        eng = m.engine(len(imgs[a:a + batch]))
        x, maps = eng.preprocess_images(imgs[a:a + batch])
        boxes, scores, cls, counts = eng.forward_detect(x)
        eng.map_boxes(boxes, counts, maps)
        out_dev.append((boxes.clone(), scores.clone(), cls.clone(), counts.clone()))
        ch = counts.cpu().numpy()
        bh, sh, clh = boxes.cpu().numpy(), scores.cpu().numpy(), cls.cpu().numpy()
        host += [(bh[i, :ch[i]].copy(), sh[i, :ch[i]].copy(), clh[i, :ch[i]].astype(np.int64)) for i in range(len(ch))]
    return out_dev, host


def _padded(dets):
    """Host triples -> device batch tensors as the engine lays them out (rows past counts[b] are junk)."""
    b = len(dets)
    n = max([len(s) for _, s, _ in dets] + [1])
    boxes = np.full((b, n, 4), 7.7, np.float32)
    scores = np.full((b, n), 0.5, np.float32)
    cls = np.full((b, n), 99, np.int32)
    for i, (bx, s, c) in enumerate(dets):
        boxes[i, :len(s)], scores[i, :len(s)], cls[i, :len(s)] = bx, s, c
    counts = np.array([len(s) for _, s, _ in dets], np.int32)
    return tuple(torch.from_numpy(a).to(DEV) for a in (boxes, scores, cls, counts))


def _device_eval(dets, gt, image_ids, class_ids, nc, batch=64, capacity=None):
    from yolo_nano_b200 import COCODetections
    total = sum(len(s) for _, s, _ in dets)
    cd = COCODetections(DEV, nc, total if capacity is None else capacity)
    for a in range(0, len(dets), batch):
        cd.add(*_padded(dets[a:a + batch]))
    return cd, cd.evaluate(gt, image_ids, class_ids, details=True)


def _same(a, b):
    return a.shape == b.shape and np.array_equal(np.ascontiguousarray(a).view(np.int64),
                                                 np.ascontiguousarray(b).view(np.int64))


def _check(dets, gt, image_ids, class_ids, nc, label, batch=64, literal=False):
    """Device vs the vectorised oracle (and the literal one on small sets); on a difference, names the first entry."""
    cd, (stats, (prec, rec)) = _device_eval(dets, gt, image_ids, class_ids, nc, batch)
    n = cd.num_rows()
    rows = O.arena_rows(dets)
    assert np.array_equal(cd.rows[:n].cpu().numpy(), rows), f"{label}: appended rows differ"
    wants = [("rows", O.coco_eval_rows(rows, image_ids, gt, class_ids))]
    if literal:
        wants.append(("literal", O.coco_eval_literal(gt, O.result_json(dets, image_ids, class_ids), image_ids)))
    for form, (ws, wp, wr) in wants:
        bad = np.argwhere(prec.view(np.int64) != wp.view(np.int64))
        assert len(bad) == 0, f"{label} vs {form}: precision differs first at [t,r,k,a,m] = {bad[0].tolist()}: " \
                              f"{prec[tuple(bad[0])]!r} != {wp[tuple(bad[0])]!r}"
        assert _same(rec, wr), f"{label} vs {form}: recall differs at {np.argwhere(rec != wr)[:3].tolist()}"
        assert _same(stats, ws), (label, form, stats, ws)
    print(f"[report] {label}: {n} rows, AP {stats[0]:.6f}, AP50 {stats[1]:.6f}, AR100 {stats[8]:.6f}")
    return stats, prec, rec


def _edge_set():
    """Crowd and out-of-range GT, GT and detection areas exactly at 32^2 and 96^2, IoU exactly 0.5 and 0.75, equal
    IoU against two GT, more than 1, 10 and 100 detections in one cell, score ties within a cell and across images
    (image ids out of order), images without GT / detections / either, a class outside the GT categories and a cell
    with several hundred GT."""
    rng = np.random.default_rng(11)
    image_ids = [42, 7, 19, 3, 100, 8]
    cats = [1, 5, 9]
    anns = []

    def ann(iid, cat, box, **kw):
        anns.append({'id': len(anns) + 1, 'image_id': iid, 'category_id': cat, 'bbox': [float(v) for v in box],
                     'area': kw.get('area', float(box[2] * box[3])), 'iscrowd': kw.get('iscrowd', 0)})

    for j in range(400):                                                 # image 42, category 5: 400 GT
        x, y = rng.integers(0, 600, 2)
        ann(42, 5, [x, y, int(rng.integers(8, 120)), int(rng.integers(8, 120))], iscrowd=int(j % 41 == 0))
    ann(7, 1, [0, 0, 10, 10])
    ann(7, 1, [0, 0, 10, 10])                                           # equal IoU: the later GT wins
    ann(7, 1, [100, 100, 96, 96])                                       # area 96^2
    ann(7, 1, [300, 300, 32, 32])                                       # area 32^2
    ann(7, 1, [500, 500, 40, 40], area=1e11)                            # outside every range
    ann(7, 9, [0, 0, 400, 400], iscrowd=1)
    ann(3, 9, [5, 5, 50, 50])
    ann(8, 1, [0, 0, 20, 20])
    gt = {'images': [{'id': i} for i in image_ids + [555]], 'categories': [{'id': c} for c in cats],
          'annotations': anns}
    g42 = np.array([a['bbox'] for a in anns[:400]])
    pick = rng.integers(0, 400, 260)
    b42 = np.concatenate([g42[pick, :2], g42[pick, :2] + g42[pick, 2:]], 1) + rng.normal(0, 3, (260, 4))
    f32 = np.float32
    dets = [
        (b42.astype(f32), (rng.integers(1, 9, 260) / 8).astype(f32), np.ones(260, np.int64)),
        (np.array([[0, 0, 10, 10], [0, 0, 10, 10], [0, 0, 10, 5], [0, 0, 10, 7.5], [100, 100, 196, 196],
                   [300, 300, 332, 332], [60, 60, 92, 92], [10, 10, 100, 100], [20, 20, 30, 30],
                   [500, 500, 540, 540]], f32),
         np.array([0.5, 0.5, 0.5, 0.5, 0.25, 0.25, 0.5, 0.125, 0.5, 0.75], f32),
         np.array([0, 0, 0, 0, 0, 0, 0, 2, 3, 0])),
        (np.array([[10, 10, 20, 20]], f32), np.array([0.5], f32), np.array([0])),           # image 19: no GT
        (np.zeros((0, 4), f32), np.zeros(0, f32), np.zeros(0, np.int64)),                 # image 3: no detections
        (np.zeros((0, 4), f32), np.zeros(0, f32), np.zeros(0, np.int64)),                 # image 100: neither
        # image 8: 120 detections of one GT (more than 1, 10 and 100), scores tied with the other images
        (np.tile(np.array([[0, 0, 20, 20]], f32), (120, 1)) + rng.integers(0, 4, (120, 4)).astype(f32),
         (rng.integers(1, 9, 120) / 8).astype(f32), np.zeros(120, np.int64)),
    ]
    return dets, gt, image_ids, [1, 5, 9, 77]


def test_edge_set(lib):
    dets, gt, image_ids, class_ids = _edge_set()
    stats, prec, rec = _check(dets, gt, image_ids, class_ids, 4, "edge", literal=True)
    assert (prec > 0).any()
    # empty arena: -1 without GT, 0 with
    _check([(np.zeros((0, 4), np.float32), np.zeros(0, np.float32), np.zeros(0, np.int64))] * 2,
           {'images': [{'id': 1}, {'id': 2}], 'categories': [{'id': 3}],
            'annotations': [{'id': 1, 'image_id': 2, 'category_id': 3, 'bbox': [0, 0, 5, 5], 'area': 25,
                             'iscrowd': 0}]}, [2, 1], [3], 1, "empty")


@pytest.mark.parametrize("seed", [0, 1])
def test_random_tie_heavy_sets(lib, seed):
    dets, gt, image_ids, class_ids = O.random_set(1200, 20, seed=100 + seed, max_gt=12, score_levels=25)
    _check(dets, gt, image_ids, class_ids, 20, f"random{seed}")


def test_splits_and_reruns(lib):
    """Batches of 1, 7 and 64 give identical rows and results; two evaluations are identical."""
    dets, gt, image_ids, class_ids = O.random_set(150, 20, seed=9)
    ref = None
    for bs in (1, 7, 64):
        cd, (stats, (prec, rec)) = _device_eval(dets, gt, image_ids, class_ids, 20, batch=bs)
        rows = cd.rows[:cd.num_rows()].cpu()
        s2, (p2, r2) = cd.evaluate(gt, image_ids, class_ids, details=True)
        assert _same(stats, s2) and _same(prec, p2) and _same(rec, r2)
        if ref is None:
            ref = (rows, stats, prec, rec)
        else:
            assert torch.equal(rows, ref[0])
            assert _same(stats, ref[1]) and _same(prec, ref[2]) and _same(rec, ref[3])


@pytest.mark.parametrize("weights", ["refinit", "calibrated"])
def test_appended_rows_equal_engine_outputs(lib, weights):
    """Engine detections at 416 (after map_boxes) -> device rows == the float32 outputs bit for bit, in file order."""
    m = _model(416, 80, weights)
    imgs = _images(6, seed=80)
    dev, host = _engine_dets(m, imgs, batch=4)
    from yolo_nano_b200 import COCODetections
    cd = COCODetections(DEV, 80, sum(len(s) for _, s, _ in host))
    for t in dev:
        cd.add(*t)
    n = cd.num_rows()
    want = O.arena_rows(host)
    print(f"[report] 80 classes, {weights}: {n} rows from {len(imgs)} images")
    assert n == len(want) and np.array_equal(cd.rows[:n].cpu().numpy(), want)


def _gt_from_dets(host, classes, image_ids, class_ids, seed):
    """COCO GT that includes jittered copies of real detections (1-40 per image, about 1 % crowd), so that the
    APs are non-trivial."""
    rng = np.random.default_rng(seed)
    anns = []
    for (b, s, c), iid in zip(host, image_ids):
        g = int(rng.integers(1, 41))
        if len(s):
            pick = rng.integers(0, len(s), g)
            box = np.round(b[pick].astype(np.float64) + rng.normal(0, 3, (g, 4)))
            lab = np.where(rng.random(g) < 0.9, c[pick], rng.integers(0, classes, g))
        else:
            box = np.tile([10., 10., 50., 60.], (g, 1))
            lab = rng.integers(0, classes, g)
        for j in range(g):
            w, h = max(box[j, 2] - box[j, 0], 1.0), max(box[j, 3] - box[j, 1], 1.0)
            anns.append({'id': len(anns) + 1, 'image_id': int(iid), 'category_id': int(class_ids[lab[j]]),
                         'bbox': [float(box[j, 0]), float(box[j, 1]), w, h], 'area': w * h,
                         'iscrowd': int(rng.random() < 0.01)})
    return {'images': [{'id': int(i)} for i in image_ids], 'categories': [{'id': int(c)} for c in class_ids],
            'annotations': anns}


def _coco_ids(classes):
    """COCO-like category ids: 1..90 with gaps."""
    ids = [i for i in range(1, 91) if i not in (12, 26, 29, 30, 45, 66, 68, 69, 71, 83)]
    return ids[:classes]


def test_engine_set_over_a_million_rows(lib):
    """One engine-produced set of >= 1 M results rows (reference-init weights at 416, 80 classes), where the cut to
    100 detections per cell dominates."""
    m = _model(416, 80, "refinit")
    host, k = [], 0
    while sum(len(s) for _, s, _ in host) < 1_000_000 and k < 16:
        _, h = _engine_dets(m, _images(64, seed=1000 + k))
        host += h
        k += 1
    assert sum(len(s) for _, s, _ in host) >= 1_000_000
    image_ids = (np.random.default_rng(5).permutation(len(host) * 2)[:len(host)] + 1).tolist()
    class_ids = _coco_ids(80)
    gt = _gt_from_dets(host, 80, image_ids, class_ids, seed=2)
    cut = 0
    for b, s, c in host:
        cut += int(np.maximum(np.bincount(c, minlength=80) - 100, 0).sum())
    print(f"[report] engine-1M: {cut} of {sum(len(s) for _, s, _ in host)} rows fall past 100 per cell")
    stats, _, _ = _check(host, gt, image_ids, class_ids, 80, "engine-1M")
    assert stats[1] > 0


def test_evaluate_coco_end_to_end(lib):
    """YOLONano.evaluate_coco == detect_raw_images -> evalfmt.coco_result_rows -> coco_eval_literal, exactly."""
    m = _model(320, 80, "calibrated")
    imgs = _images(24, seed=77)
    image_ids = [int(v) for v in np.random.default_rng(8).permutation(1000)[:24] + 1]
    class_ids = _coco_ids(80)
    host = [d for a in range(0, 24, 8) for d in m.detect_raw_images(imgs[a:a + 8])]   # evaluate_coco's batches
    gt = _gt_from_dets(host, 80, image_ids, class_ids, seed=3)
    stats = m.evaluate_coco(zip(imgs, image_ids), gt, class_ids, batch_size=8)
    want, _, _ = O.coco_eval_literal(gt, O.result_json(host, image_ids, class_ids), image_ids)
    assert _same(stats, want), (stats, want)
    print(f"[report] evaluate_coco: AP {stats[0]:.6f} AP50 {stats[1]:.6f} ({sum(len(s) for _, s, _ in host)} rows)")


def test_capacity_overflow_raises_and_writes_nothing_past_it(lib):
    from yolo_nano_b200 import COCODetections, EngineError
    dets, gt, image_ids, class_ids = O.random_set(20, 4, seed=6)
    total = sum(len(s) for _, s, _ in dets)
    cap = total // 2
    cd = COCODetections(DEV, 4, cap)
    guard = torch.full((cap + 64, 7), -123456, dtype=torch.int32, device=DEV)
    cd.rows = guard[:cap]
    cd.add(*_padded(dets[:10]))
    cd.add(*_padded(dets[10:]))
    assert cd.num_rows() == total
    with pytest.raises(EngineError):
        cd.evaluate(gt, image_ids, class_ids)
    assert bool((guard[cap:] == -123456).all())
    assert np.array_equal(guard[:cap].cpu().numpy(), O.arena_rows(dets)[:cap])


def test_rejects_bad_values_and_ids(lib):
    from yolo_nano_b200 import COCODetections, EngineError
    gt = {'images': [{'id': 1}, {'id': 2}], 'categories': [{'id': 1}], 'annotations': []}
    for bad in [(np.array([[0, 0, np.inf, 5]], np.float32), np.array([0.5], np.float32), np.array([0])),
                (np.array([[0, 0, 5, 5]], np.float32), np.array([np.nan], np.float32), np.array([0])),
                (np.array([[0, 0, 5, 5]], np.float32), np.array([0.5], np.float32), np.array([7]))]:
        cd = COCODetections(DEV, 4, 8)
        cd.add(*_padded([bad]))
        with pytest.raises(EngineError):
            cd.evaluate(gt, [1], [1, 2, 3, 4])
    good = (np.array([[0, 0, 5, 5]], np.float32), np.array([0.5], np.float32), np.array([0]))
    for ids in ([1, 1], [1, 3]):                         # duplicate id, id not in gt['images']
        cd = COCODetections(DEV, 4, 8)
        cd.add(*_padded([good, good]))
        with pytest.raises(EngineError):
            cd.evaluate(gt, ids, [1, 2, 3, 4])
