"""VOC mAP on the device (yolo_nano_b200.voc_eval) against the restated voc_eval (oracle/voc_eval.py): the det-file
rows bit for bit, the VOC07 AP bit for bit, the area AP within 1e-12 relative."""
import contextlib
import io
import tempfile

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import voc_eval as V  # noqa: E402
from oracle import weights as W  # noqa: E402

DEV = torch.device("cuda", 0)
AREA_RTOL = 1e-12


def _model(size, classes, weights):
    import yolo_nano_b200 as pkg
    sd = W.reference_init(classes, seed=3) if weights == "refinit" else W.calibrated(classes, seed=4)
    with contextlib.redirect_stdout(io.StringIO()):
        m = pkg.YOLONano(DEV, size, classes, anchor_size=W.anchors_for(classes))
    m.load_state_dict(sd)
    return m.to(DEV).eval()


def _images(n, seed):
    """Original uint8 BGR images of VOC-like shapes (smooth content, so that detections vary between images)."""
    rng = np.random.default_rng(seed)
    shapes = [(375, 500), (500, 375), (333, 500), (500, 500), (281, 500), (500, 334)]
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


def _device_eval(dets, gt, nc, batch=64, use07=True, capacity=None):
    from yolo_nano_b200 import VOCDetections
    total = sum(len(s) for _, s, _ in dets)
    vd = VOCDetections(DEV, nc, total if capacity is None else capacity)
    for a in range(0, len(dets), batch):
        vd.add(*_padded(dets[a:a + batch]))
    return vd, vd.evaluate(gt, use_07_metric=use07, details=True)


def _check(dets, gt, nc, label, batch=64):
    """Device vs oracle in both metrics; on a difference, names the first sorted detection whose flag differs."""
    rows = V.result_rows(dets)
    for use07 in (True, False):
        vd, (aps, m_ap, npos, order, flags) = _device_eval(dets, gt, nc, batch, use07)
        n = vd.num_rows()
        assert np.array_equal(vd.rows[:n].cpu().numpy(), rows), f"{label}: appended rows differ"
        want, want_npos, detail = V.voc_eval_rows(rows, gt, nc, use_07_metric=use07)
        want_order = np.concatenate([d[0] for d in detail]) if n else np.zeros(0, np.int64)
        want_flags = np.concatenate([d[1] for d in detail]) if n else np.zeros(0, np.int8)
        assert np.array_equal(npos, want_npos), label
        assert np.array_equal(order, want_order), f"{label}: sorted order differs"
        bad = np.nonzero(flags != want_flags)[0]
        assert len(bad) == 0, (f"{label}: first disagreement at sorted position {bad[0]} (arena row {order[bad[0]]}: "
                               f"{rows[order[bad[0]]].tolist()}), device flag {flags[bad[0]]}, oracle {want_flags[bad[0]]}")
        if use07:
            assert np.array_equal(aps.view(np.int64), want.view(np.int64)), (label, aps, want)
            assert m_ap == float(np.mean(want))
            ap07 = aps
        else:
            assert np.array_equal(np.isnan(aps), np.isnan(want)), (label, aps, want)
            ok = ~np.isnan(want)
            rel = np.abs(aps[ok] - want[ok]) / np.maximum(np.abs(want[ok]), 1e-300)
            worst = float(rel.max()) if rel.size else 0.0
            print(f"[report] {label}: {n} rows, mAP07 {np.mean(ap07):.6f}, area mAP {np.mean(aps):.6f}, "
                  f"area max rel diff vs np.sum {worst:.3e}")
            assert worst <= AREA_RTOL, (label, worst)
    return ap07


def _edge_set():
    f32 = np.float32
    gt = [
        (np.array([[0, 0, 10, 10], [20, 20, 30, 30], [50, 50, 60, 60]], float), np.array([0, 0, 1]),
         np.array([False, True, False])),
        (np.array([[0, 0, 10, 10], [5, 5, 5, 5]], float), np.array([0, 2]), np.array([False, False])),
        (np.zeros((0, 4)), np.zeros(0, int), np.zeros(0, bool)),
    ]
    d0 = (np.array([[0, 0, 10, 10], [0, 0, 10, 10], [20, 20, 30, 30], [50, 50, 60, 60], [0, 0, 20, 10]], f32) - 1,
          np.array([0.9, 0.9, 0.8, 0.7, 0.6], f32), np.array([0, 0, 0, 1, 3]))
    d1 = (np.array([[0, 0, 10, 5.0], [0, 0, 10, 10], [5, 5, 5, 5]], f32) - 1,
          np.array([0.95, 0.5, 0.4], f32), np.array([0, 0, 2]))
    # the second box writes '-0.0' fields: -0.04 + 1 - 1 in float32
    d2 = (np.array([[1, 1, 5, 5], [-0.04, -0.02, 3, 3]], f32) - 1, np.array([0.3, 0.0004], f32), np.array([0, 0]))
    return [d0, d1, d2], gt


def test_edge_cases(lib):
    """A difficult match, duplicate detections of one GT, overlap exactly 0.5 (strict >), a NaN overlap from
    zero-area boxes, a class with no GT (07: 0, area: NaN), a class with no lines (-1), an image with no GT, '-0.0'
    fields; and an empty set."""
    dets, gt = _edge_set()
    ap07 = _check(dets, gt, 5, "edge")
    assert ap07[4] == -1 and ap07[3] == 0
    from yolo_nano_b200 import VOCDetections
    vd = VOCDetections(DEV, 4, 16)
    vd.add(*_padded([(np.zeros((0, 4), np.float32), np.zeros(0, np.float32), np.zeros(0, np.int64))] * 3))
    aps, m_ap = vd.evaluate([(np.zeros((0, 4)), np.zeros(0, int), np.zeros(0, bool))] * 3)
    assert list(aps) == [-1.0] * 4 and m_ap == -1.0


@pytest.mark.parametrize("seed", [0, 1])
def test_random_tie_heavy_sets(lib, seed):
    dets, gt = V.random_set(1200, 20, seed=100 + seed, max_gt=12, score_levels=25)
    _check(dets, gt, 20, f"random{seed}")


def test_splits_and_reruns(lib):
    """Batches of 1, 7 and 64 give identical rows and APs; two evaluations are identical."""
    dets, gt = V.random_set(150, 20, seed=9)
    ref = None
    for bs in (1, 7, 64):
        vd, res = _device_eval(dets, gt, 20, batch=bs)
        rows = vd.rows[:vd.num_rows()].cpu()
        again = vd.evaluate(gt, details=True)
        for a, b in zip(res, again):
            assert np.array_equal(np.asarray(a), np.asarray(b))
        if ref is None:
            ref = (rows, res)
        else:
            assert torch.equal(rows, ref[0])
            for a, b in zip(res, ref[1]):
                assert np.array_equal(np.asarray(a), np.asarray(b))


@pytest.mark.parametrize("classes,weights", [(80, "refinit"), (80, "calibrated"), (20, "refinit"), (20, "calibrated")])
def test_appended_rows_equal_oracle_rows(lib, classes, weights):
    """Engine detections at 416 (after map_boxes) -> device rows == the oracle's integer rows, in file order."""
    m = _model(416, classes, weights)
    imgs = _images(6, seed=classes)
    dev, host = _engine_dets(m, imgs, batch=4)
    from yolo_nano_b200 import VOCDetections
    vd = VOCDetections(DEV, classes, sum(len(s) for _, s, _ in host))
    for t in dev:
        vd.add(*t)
    n = vd.num_rows()
    want = V.result_rows(host)
    print(f"[report] {classes} classes, {weights}: {n} rows from {len(imgs)} images")
    assert n == len(want) and np.array_equal(vd.rows[:n].cpu().numpy(), want)


def _gt_from_dets(host, classes, seed):
    """GT that includes jittered copies of real detections (1-40 per image), so that the APs are non-trivial."""
    rng = np.random.default_rng(seed)
    gt = []
    for b, s, c in host:
        g = int(rng.integers(1, 41))
        if len(s):
            pick = rng.integers(0, len(s), g)
            box = np.round(b[pick].astype(np.float64) + 1 + rng.normal(0, 3, (g, 4)))
            lab = np.where(rng.random(g) < 0.9, c[pick], rng.integers(0, classes, g))
        else:
            box = np.tile([10., 10., 50., 60.], (g, 1))
            lab = rng.integers(0, classes, g)
        gt.append((box, lab, rng.random(g) < 0.1))
    return gt


def test_engine_set_over_a_million_rows(lib):
    """One engine-produced set of >= 1 M det-file rows (reference-init weights at 416, 20 classes)."""
    m = _model(416, 20, "refinit")
    host, k = [], 0
    while sum(len(s) for _, s, _ in host) < 1_000_000 and k < 16:
        _, h = _engine_dets(m, _images(64, seed=1000 + k))
        host += h
        k += 1
    gt = _gt_from_dets(host, 20, seed=2)
    assert sum(len(s) for _, s, _ in host) >= 1_000_000
    ap07 = _check(host, gt, 20, "engine-1M")
    assert (ap07 > 0).any()


def test_evaluate_voc_end_to_end(lib):
    """YOLONano.evaluate_voc == detect_raw_images -> evalfmt det files -> voc_eval (literal, stable order), exactly."""
    m = _model(320, 20, "calibrated")
    imgs = _images(40, seed=77)
    host = [d for a in range(0, 40, 16) for d in m.detect_raw_images(imgs[a:a + 16])]   # evaluate_voc's batches
    gt = _gt_from_dets(host, 20, seed=3)
    for use07 in (True, False):
        aps, m_ap = m.evaluate_voc(imgs, gt, batch_size=16, use_07_metric=use07)
        with tempfile.TemporaryDirectory() as tmp:
            want = V.eval_files(tmp, host, gt, 20, use_07_metric=use07, kind="stable")
        if use07:
            assert np.array_equal(aps.view(np.int64), want.view(np.int64)), (aps, want)
        else:
            assert np.array_equal(np.isnan(aps), np.isnan(want))
            ok = ~np.isnan(want)
            assert np.all(np.abs(aps[ok] - want[ok]) <= AREA_RTOL * np.abs(want[ok])), (aps, want)
        print(f"[report] evaluate_voc 07={use07}: mAP {m_ap:.6f} (oracle {np.mean(want):.6f})")


def test_capacity_overflow_raises_and_writes_nothing_past_it(lib):
    from yolo_nano_b200 import VOCDetections, EngineError
    dets, gt = V.random_set(20, 4, seed=6)
    total = sum(len(s) for _, s, _ in dets)
    cap = total // 2
    vd = VOCDetections(DEV, 4, cap)
    guard = torch.full((cap + 64, 7), -123456, dtype=torch.int32, device=DEV)
    vd.rows = guard[:cap]
    vd.add(*_padded(dets[:10]))
    vd.add(*_padded(dets[10:]))
    assert vd.num_rows() == total
    with pytest.raises(EngineError):
        vd.evaluate(gt)
    assert bool((guard[cap:] == -123456).all())
    assert np.array_equal(guard[:cap].cpu().numpy(), V.result_rows(dets)[:cap])


def test_rejects_bad_values(lib):
    from yolo_nano_b200 import VOCDetections, EngineError
    for bad in [(np.array([[0, 0, np.inf, 5]], np.float32), np.array([0.5], np.float32), np.array([0])),
                (np.array([[0, 0, 5, 5]], np.float32), np.array([1.5], np.float32), np.array([0])),
                (np.array([[0, 0, 5, 5]], np.float32), np.array([0.5], np.float32), np.array([7]))]:
        vd = VOCDetections(DEV, 4, 8)
        vd.add(*_padded([bad]))
        with pytest.raises(EngineError):
            vd.evaluate([(np.zeros((0, 4)), np.zeros(0, int), np.zeros(0, bool))])
