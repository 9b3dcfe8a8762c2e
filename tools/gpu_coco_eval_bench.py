"""COCO AP on the device vs the reference's COCOeval path, at val2017 scale.

A synthetic set of 5000 original images of COCO-like shapes with about 7.4 GT boxes each (about 1 % crowd) over 80
categories with COCO's id gaps, detected at 416 with reference-init and with calibrated weights (conf_thresh 0.001,
as the evaluators run).  Reported per weight set:
  * append + evaluate on the device (CUDA events, warmed, best of --reps), with the results row count;
  * YOLONano.evaluate_coco over the whole set (host clock, ends in the one synchronise), preprocessing and detection
    included;
  * the literal COCOeval restatement (oracle/coco_eval.py, results JSON round trip included) on the first
    --oracle-images images only, and its rows per second; the device on the same subset must equal it bit for bit.
GPU name and power limit are read in the same run.

    python tools/gpu_coco_eval_bench.py --out profiles/r03_coco_eval_bench_5000.json
"""
from __future__ import annotations

import argparse
import contextlib
import ctypes as C
import io
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from oracle import coco_eval as O  # noqa: E402
from oracle import weights as W  # noqa: E402
import yolo_nano_b200 as pkg  # noqa: E402
from yolo_nano_b200 import _lib  # noqa: E402
from yolo_nano_b200 import coco_eval as CE  # noqa: E402
from yolo_nano_b200.engine import _ptr, _stream_ptr  # noqa: E402

SHAPES = [(480, 640), (640, 480), (427, 640), (640, 427), (425, 640), (640, 640), (360, 640), (500, 375)]
CLASS_IDS = [i for i in range(1, 91) if i not in (12, 26, 29, 30, 45, 66, 68, 69, 71, 83)]


def image(i: int) -> np.ndarray:
    rng = np.random.default_rng(20_000 + i)
    h, w = SHAPES[int(rng.integers(len(SHAPES)))]
    small = rng.integers(0, 256, (h // 16 + 2, w // 16 + 2, 3), dtype=np.uint8)
    return np.ascontiguousarray(np.repeat(np.repeat(small, 16, 0), 16, 1)[:h, :w])


def image_ids(n: int):
    return (np.random.default_rng(5000).permutation(600_000)[:n] + 1).tolist()


def ground_truth(n: int):
    """About 7.4 boxes per image (Poisson), log-uniform sizes so that all three area ranges are populated."""
    rng = np.random.default_rng(7)
    ids = image_ids(n)
    anns = []
    for i, iid in enumerate(ids):
        h, w = SHAPES[int(np.random.default_rng(20_000 + i).integers(len(SHAPES)))]
        for _ in range(int(rng.poisson(7.4))):
            bw, bh = (float(np.round(np.exp(rng.uniform(np.log(4), np.log(s))))) for s in (w, h))
            x, y = float(rng.integers(0, max(w - bw, 1))), float(rng.integers(0, max(h - bh, 1)))
            anns.append({'id': len(anns) + 1, 'image_id': iid, 'category_id': int(CLASS_IDS[rng.integers(80)]),
                         'bbox': [x, y, bw, bh], 'area': bw * bh * float(rng.uniform(0.4, 1.0)),
                         'iscrowd': int(rng.random() < 0.01)})
    return {'images': [{'id': i} for i in ids], 'categories': [{'id': c} for c in CLASS_IDS], 'annotations': anns}


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"unavailable ({e})"
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def run(weights: str, args, gt, dev):
    classes = 80
    sd = W.reference_init(classes, seed=0) if weights == "refinit" else W.calibrated(classes, seed=0)
    with contextlib.redirect_stdout(io.StringIO()):
        m = pkg.YOLONano(dev, args.size, classes, anchor_size=W.anchors_for(classes))
    m.load_state_dict(sd)
    m = m.to(dev).eval()
    n, bs = args.images, args.batch
    ids = image_ids(n)

    # detections of the whole set on the device, kept per batch
    outs = []
    for a in range(0, n, bs):
        imgs = [image(i) for i in range(a, min(n, a + bs))]
        eng = m.engine(len(imgs))
        x, maps = eng.preprocess_images(imgs)
        boxes, scores, cls, counts = eng.forward_detect(x)
        eng.map_boxes(boxes, counts, maps)
        outs.append((boxes, scores, cls, counts))
    rows = int(sum(int(o[3].sum()) for o in outs))

    lib = _lib.load()
    dbl = C.POINTER(C.c_double)
    best = {"append_ms": 1e30, "evaluate_ms": 1e30}
    stats = None
    for rep in range(args.reps + 1):                       # rep 0 warms up
        cd = pkg.COCODetections(dev, classes, rows)
        e0, e1, e2, e3 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
        e0.record()
        for o in outs:
            cd.add(*o)
        e1.record()
        n_rows = cd._checked_rows()
        p, K = CE.pack_gt(gt, ids, CLASS_IDS, classes)
        t = {k: torch.from_numpy(v).to(dev) for k, v in p.items()}
        n_gt = int(p["area"].shape[0])
        wsb = int(lib.ynb_coco_eval_workspace_bytes(n_rows, n, K, n_gt))
        ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
        prec = torch.empty((10, 101, K, 4, 3), dtype=torch.float64, device=dev)
        rec = torch.empty((10, K, 4, 3), dtype=torch.float64, device=dev)
        iou_thrs, rec_thrs = np.ascontiguousarray(CE.IOU_THRS), np.ascontiguousarray(CE.REC_THRS)
        torch.cuda.synchronize()
        e2.record()
        rc = lib.ynb_coco_eval(_ptr(cd.rows), n_rows, classes, n, _ptr(t["image_rank"]), _ptr(t["class_cat"]), K,
                               _ptr(t["boxes"]), _ptr(t["area"]), _ptr(t["iscrowd"]), _ptr(t["start"]), n_gt,
                               iou_thrs.ctypes.data_as(dbl), rec_thrs.ctypes.data_as(dbl), _ptr(prec), _ptr(rec),
                               _ptr(ws), wsb, _stream_ptr(dev))
        e3.record()
        torch.cuda.synchronize()
        assert rc == 0, lib.ynb_last_error(None)
        if rep:
            best["append_ms"] = min(best["append_ms"], e0.elapsed_time(e1))
            best["evaluate_ms"] = min(best["evaluate_ms"], e2.elapsed_time(e3))
        stats = CE.summarize(prec.cpu().numpy(), rec.cpu().numpy())
        assert n_rows == rows
        assert np.array_equal(stats, cd.evaluate(gt, ids, CLASS_IDS))
        del cd, ws

    # the whole evaluate_coco (preprocess + detect + map + append + evaluate), warmed on one batch first
    m.evaluate_coco([(image(i), ids[i]) for i in range(bs)], gt, CLASS_IDS, batch_size=bs, capacity=rows)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    stats2 = m.evaluate_coco(((image(i), ids[i]) for i in range(n)), gt, CLASS_IDS, batch_size=bs, capacity=rows)
    wall = time.perf_counter() - t0
    assert np.array_equal(stats2, stats)

    # the literal COCOeval restatement on a subset, and the device on the same subset
    k = min(args.oracle_images, n)
    host = []
    for o in outs:
        ch = o[3].cpu().numpy()
        bh, sh, clh = o[0].cpu().numpy(), o[1].cpu().numpy(), o[2].cpu().numpy()
        host += [(bh[i, :ch[i]], sh[i, :ch[i]], clh[i, :ch[i]].astype(np.int64)) for i in range(len(ch))]
        if len(host) >= k:
            break
    host = host[:k]
    sub_rows = sum(len(s) for _, s, _ in host)
    sub_gt = dict(gt, images=gt['images'][:k])
    t0 = time.perf_counter()
    lit_stats, lit_prec, _ = O.coco_eval_literal(sub_gt, O.result_json(host, ids[:k], CLASS_IDS), ids[:k])
    t_oracle = time.perf_counter() - t0
    cd = pkg.COCODetections(dev, classes, sub_rows)
    for a in range(0, k, bs):
        b = host[a:a + bs]
        nmax = max([len(s) for _, s, _ in b] + [1])
        bx = np.zeros((len(b), nmax, 4), np.float32)
        sc = np.zeros((len(b), nmax), np.float32)
        cl = np.zeros((len(b), nmax), np.int32)
        for i, (bb, s, c) in enumerate(b):
            bx[i, :len(s)], sc[i, :len(s)], cl[i, :len(s)] = bb, s, c
        cnt = np.array([len(s) for _, s, _ in b], np.int32)
        cd.add(*(torch.from_numpy(v).to(dev) for v in (bx, sc, cl, cnt)))
    sub_stats, (sub_prec, _) = cd.evaluate(sub_gt, ids[:k], CLASS_IDS, details=True)
    return {
        "weights": weights, "images": n, "batch": bs, "input_size": args.size, "rows": rows,
        "rows_per_image": rows / n, "gt_boxes": len(gt['annotations']),
        "device_append_ms": best["append_ms"], "device_evaluate_ms": best["evaluate_ms"],
        "device_append_plus_evaluate_ms": best["append_ms"] + best["evaluate_ms"],
        "evaluate_coco_wall_s": wall, "stats": [float(v) for v in stats],
        "oracle_subset_images": k, "oracle_subset_rows": sub_rows, "oracle_subset_s": t_oracle,
        "oracle_rows_per_s": sub_rows / t_oracle,
        "oracle_subset_stats": [float(v) for v in lit_stats],
        "device_subset_equals_literal": bool(np.array_equal(sub_stats, lit_stats) and
                                             np.array_equal(sub_prec, lit_prec)),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=5000)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--size", type=int, default=416)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--oracle-images", type=int, default=20)
    ap.add_argument("--out", default="coco_eval_bench.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gpu_coco_eval_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    res = {"gpu": gpu_info(), "note": "device times: CUDA events, best of reps after one warm-up; evaluate_coco: host "
           "clock over the whole set incl. host-side image generation and packing; oracle: the literal COCOeval "
           "restatement on the first oracle_subset_images images only (not extrapolated)", "runs": []}
    gt = ground_truth(args.images)
    for w in ("refinit", "calibrated"):
        r = run(w, args, gt, dev)
        print(json.dumps(r), flush=True)
        res["runs"].append(r)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
