"""Generates tests/golden/g13_coco_eval.npz by running the REAL pycocotools COCOeval 'bbox' (the evaluator's
`COCOAPIEvaluator.evaluate` after detection: results JSON, loadRes, params.imgIds, evaluate / accumulate /
summarize) on a fixed synthetic set, wherever pycocotools is installed.

    python -m oracle.gen_coco_golden

pycocotools is not a dependency of this project.  No such golden has been recorded yet, so oracle/coco_eval.py has
not been pinned by the real COCOeval: it rests on the pycocotools 2.0 sources it transcribes and on hand-derived
known answers.  Once recorded, the golden holds the set (detections, GT JSON, image and class ids) with the real
stats, precision and recall, which the restatement must reproduce bit for bit.
"""
from __future__ import annotations

import contextlib
import io
import json
import os
import tempfile

import numpy as np

from oracle import coco_eval as O
from oracle.gen_golden import OUT


def coco_eval_golden():
    from pycocotools.coco import COCO  # type: ignore
    from pycocotools.cocoeval import COCOeval  # type: ignore
    dets, gt, image_ids, class_ids = O.random_set(40, 6, seed=13, max_gt=10, score_levels=8)
    rows = O.result_json(dets, image_ids, class_ids)
    with tempfile.TemporaryDirectory() as tmp:
        gt_file, res_file = os.path.join(tmp, "gt.json"), os.path.join(tmp, "res.json")
        with open(gt_file, "w") as f:
            json.dump(gt, f)
        with open(res_file, "w") as f:
            json.dump(rows, f)
        with contextlib.redirect_stdout(io.StringIO()):
            cocoGt = COCO(gt_file)
            cocoDt = cocoGt.loadRes(res_file)
            cocoEval = COCOeval(cocoGt, cocoDt, 'bbox')
            cocoEval.params.imgIds = image_ids
            cocoEval.evaluate()
            cocoEval.accumulate()
            cocoEval.summarize()
    out = {"gt_json": np.frombuffer(json.dumps(gt).encode(), np.uint8), "image_ids": np.array(image_ids),
           "class_ids": np.array(class_ids), "stats": cocoEval.stats,
           "precision": cocoEval.eval["precision"], "recall": cocoEval.eval["recall"]}
    for i, (b, s, c) in enumerate(dets):
        out[f"img{i}.boxes"], out[f"img{i}.scores"], out[f"img{i}.cls"] = b, s, c
    np.savez_compressed(OUT / "g13_coco_eval.npz", **out)
    print("g13_coco_eval.npz:", len(rows), "results, stats", cocoEval.stats.tolist())


if __name__ == "__main__":
    coco_eval_golden()
