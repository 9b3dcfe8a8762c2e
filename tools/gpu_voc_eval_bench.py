"""VOC mAP on the device vs the reference's det-file voc_eval, at VOC07-test scale.

A synthetic set of 4952 original images of VOC-like shapes with 1-40 GT boxes each over 20 classes, detected at 416 with
reference-init and with calibrated weights (conf_thresh 0.001, as the evaluators run).  Reported per weight set:
  * append + evaluate on the device (CUDA events, warmed, best of --reps), with the det-file row count;
  * YOLONano.evaluate_voc over the whole set (host clock, ends in the one synchronise), preprocessing and detection
    included;
  * the reference path (det files written by evalfmt, then voc_eval per class, NumPy's default argsort) on the lines of
    the first --oracle-images images only, and its lines per second.
GPU name and power limit are read in the same run.

    python tools/gpu_voc_eval_bench.py --out voc_eval_bench.json
"""
from __future__ import annotations

import argparse
import contextlib
import ctypes as C
import io
import json
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from oracle import voc_eval as V  # noqa: E402
from oracle import weights as W  # noqa: E402
import yolo_nano_b200 as pkg  # noqa: E402
from yolo_nano_b200 import _lib  # noqa: E402
from yolo_nano_b200.engine import _ptr, _stream_ptr  # noqa: E402

SHAPES = [(375, 500), (500, 375), (333, 500), (500, 500), (281, 500), (500, 334), (366, 500), (500, 353)]


def image(i: int) -> np.ndarray:
    rng = np.random.default_rng(10_000 + i)
    h, w = SHAPES[int(rng.integers(len(SHAPES)))]
    small = rng.integers(0, 256, (h // 16 + 2, w // 16 + 2, 3), dtype=np.uint8)
    return np.ascontiguousarray(np.repeat(np.repeat(small, 16, 0), 16, 1)[:h, :w])


def ground_truth(n: int, classes: int):
    rng = np.random.default_rng(4952)
    gt = []
    for i in range(n):
        h, w = SHAPES[int(np.random.default_rng(10_000 + i).integers(len(SHAPES)))]
        g = int(rng.integers(1, 41))
        x1, y1 = rng.integers(0, w - 16, g), rng.integers(0, h - 16, g)
        box = np.stack([x1, y1, np.minimum(x1 + rng.integers(8, 300, g), w - 1),
                        np.minimum(y1 + rng.integers(8, 300, g), h - 1)], 1).astype(np.float64)
        gt.append((box, rng.integers(0, classes, g), rng.random(g) < 0.1))
    return gt


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"unavailable ({e})"
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def run(weights: str, args, gt, dev):
    classes = 20
    sd = W.reference_init(classes, seed=0) if weights == "refinit" else W.calibrated(classes, seed=0)
    with contextlib.redirect_stdout(io.StringIO()):
        m = pkg.YOLONano(dev, args.size, classes, anchor_size=pkg.MULTI_ANCHOR_SIZE)
    m.load_state_dict(sd)
    m = m.to(dev).eval()
    n, bs = args.images, args.batch

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
    best = {"append_ms": 1e30, "evaluate_ms": 1e30}
    aps = None
    for rep in range(args.reps + 1):                       # rep 0 warms up
        vd = pkg.VOCDetections(dev, classes, rows)
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        for o in outs:
            vd.add(*o)
        e1.record()
        n_rows = vd._checked_rows()
        gb, gd, gs, n_gt = vd.pack_gt(gt)
        wsb = int(lib.ynb_voc_eval_workspace_bytes(n_rows, classes, n_gt))
        ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
        ap = torch.empty(classes, dtype=torch.float64, device=dev)
        npos = torch.empty(classes, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        e1b = torch.cuda.Event(enable_timing=True)
        e1b.record()
        rc = lib.ynb_voc_eval(_ptr(vd.rows), n_rows, classes, n, _ptr(gb), _ptr(gd), _ptr(gs), n_gt, C.c_double(0.5),
                              1, _ptr(ap), _ptr(npos), None, None, _ptr(ws), wsb, _stream_ptr(dev))
        e2.record()
        torch.cuda.synchronize()
        assert rc == 0, lib.ynb_last_error(None)
        if rep:
            best["append_ms"] = min(best["append_ms"], e0.elapsed_time(e1))
            best["evaluate_ms"] = min(best["evaluate_ms"], e1b.elapsed_time(e2))
        aps = ap.cpu().numpy()
        assert n_rows == rows
        assert np.array_equal(aps, vd.evaluate(gt)[0])
        del vd, ws

    # the whole evaluate_voc (preprocess + detect + map + append + evaluate), warmed on one batch first
    m.evaluate_voc([image(i) for i in range(bs)], gt[:bs], batch_size=bs)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    aps2, m_ap = m.evaluate_voc((image(i) for i in range(n)), gt, batch_size=bs, capacity=rows)
    wall = time.perf_counter() - t0
    assert np.array_equal(aps2, aps)

    # the reference path on a subset: det files + voc_eval (default argsort, as the reference runs it)
    k = min(args.oracle_images, n)
    host = []
    for o in outs:
        ch = o[3].cpu().numpy()
        bh, sh, clh = o[0].cpu().numpy(), o[1].cpu().numpy(), o[2].cpu().numpy()
        host += [(bh[i, :ch[i]], sh[i, :ch[i]], clh[i, :ch[i]].astype(np.int64)) for i in range(len(ch))]
        if len(host) >= k:
            break
    host = host[:k]
    sub_lines = sum(len(s) for _, s, _ in host)
    with tempfile.TemporaryDirectory() as tmp:
        t0 = time.perf_counter()
        ora = V.eval_files(tmp, host, gt[:k], classes, use_07_metric=True, kind=None)
        t_oracle = time.perf_counter() - t0
    # the device on the same subset, for the same-lines comparison
    vd = pkg.VOCDetections(dev, classes, sub_lines)
    for a in range(0, k, bs):
        b = host[a:a + bs]
        nmax = max([len(s) for _, s, _ in b] + [1])
        bx = np.zeros((len(b), nmax, 4), np.float32)
        sc = np.zeros((len(b), nmax), np.float32)
        cl = np.zeros((len(b), nmax), np.int32)
        for i, (bb, s, c) in enumerate(b):
            bx[i, :len(s)], sc[i, :len(s)], cl[i, :len(s)] = bb, s, c
        cnt = np.array([len(s) for _, s, _ in b], np.int32)
        vd.add(*(torch.from_numpy(t).to(dev) for t in (bx, sc, cl, cnt)))
    sub_dev, _ = vd.evaluate(gt[:k])
    with tempfile.TemporaryDirectory() as tmp:
        ora_stable = V.eval_files(tmp, host, gt[:k], classes, use_07_metric=True, kind="stable")
    return {
        "weights": weights, "images": n, "batch": bs, "input_size": args.size, "rows": rows,
        "rows_per_image": rows / n,
        "device_append_ms": best["append_ms"], "device_evaluate_ms": best["evaluate_ms"],
        "device_append_plus_evaluate_ms": best["append_ms"] + best["evaluate_ms"],
        "evaluate_voc_wall_s": wall, "mAP07": m_ap,
        "oracle_subset_images": k, "oracle_subset_lines": sub_lines, "oracle_subset_s": t_oracle,
        "oracle_lines_per_s": sub_lines / t_oracle,
        "oracle_subset_default_argsort_mAP07": float(np.mean(ora)),
        "oracle_subset_stable_mAP07": float(np.mean(ora_stable)),
        "device_subset_mAP07": float(np.mean(sub_dev)),
        "device_subset_equals_stable_oracle": bool(np.array_equal(sub_dev, ora_stable)),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=4952)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--size", type=int, default=416)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--oracle-images", type=int, default=100)
    ap.add_argument("--out", default="voc_eval_bench.json")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gpu_voc_eval_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    res = {"gpu": gpu_info(), "note": "device times: CUDA events, best of reps after one warm-up; evaluate_voc: host "
           "clock over the whole set incl. host-side image packing; oracle: the first oracle_subset_images images only",
           "runs": []}
    gt = ground_truth(args.images, 20)
    for w in ("refinit", "calibrated"):
        r = run(w, args, gt, dev)
        print(json.dumps(r), flush=True)
        res["runs"].append(r)
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
