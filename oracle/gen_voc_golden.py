"""Generates tests/golden/g12_voc_eval.npz by running the REAL VOCAPIEvaluator.voc_eval / voc_ap
(evaluator/vocapi_evaluator.py) of the reference tree (see oracle/gen_golden.py for the recipe).

    python -m oracle.gen_voc_golden

Fixed det files written by evalfmt, a prepared annots.pkl cache and an image set in a temp dir, both metrics.  Scores
are distinct multiples of 0.001, so NumPy's default argsort and a stable one give the same order and
oracle/voc_eval.py must reproduce the recorded APs bit for bit.
"""
from __future__ import annotations

import contextlib
import io
import os
import tempfile
from types import SimpleNamespace

import numpy as np

from oracle import voc_eval as V
from oracle.gen_golden import OUT, _import_reference


def voc_eval_golden():
    _import_reference()
    with contextlib.redirect_stdout(io.StringIO()):
        from evaluator.vocapi_evaluator import VOCAPIEvaluator  # type: ignore
    num_classes = 5
    dets, gt = V.random_set(30, num_classes, seed=12, max_gt=4, dets_per_gt=2.0)
    total = sum(len(s) for _, s, _ in dets)
    assert total < 1000
    scores = (np.random.default_rng(13).permutation(999)[:total] + 1) / 1000.0
    k = 0
    for i, (b, s, c) in enumerate(dets):
        dets[i] = (b, scores[k:k + len(s)].astype(np.float32), c)
        k += len(s)
    names = [f"{i:06d}" for i in range(len(dets))]
    labelmap = [f"class{j:03d}" for j in range(num_classes)]
    out = {"num_classes": num_classes}
    with tempfile.TemporaryDirectory() as tmp:
        template = os.path.join(tmp, "det_test_{}.txt")
        cachedir = os.path.join(tmp, "annotations_cache")
        os.mkdir(cachedir)
        imageset = os.path.join(tmp, "test.txt")
        V.write_det_files(template, names, dets, labelmap)
        V.write_annots(os.path.join(cachedir, "annots.pkl"), imageset, names, gt, labelmap)
        fake = SimpleNamespace(imgsetpath=imageset, annopath=os.path.join(tmp, "%s.xml"), set_type="test")
        fake.voc_ap = lambda rec, prec, use_07_metric=True: VOCAPIEvaluator.voc_ap(fake, rec, prec, use_07_metric)
        for use07 in (True, False):
            aps = []
            for cls in labelmap:
                with contextlib.redirect_stdout(io.StringIO()):
                    _, _, ap = VOCAPIEvaluator.voc_eval(fake, detpath=template.format(cls), classname=cls,
                                                        cachedir=cachedir, ovthresh=0.5, use_07_metric=use07)
                aps.append(ap)
            out["aps07" if use07 else "aps_area"] = np.array(aps, dtype=np.float64)
    for i, ((b, s, c), (gb, gl, gd)) in enumerate(zip(dets, gt)):
        out[f"img{i}.boxes"], out[f"img{i}.scores"], out[f"img{i}.cls"] = b, s, c
        out[f"img{i}.gt_boxes"], out[f"img{i}.gt_labels"], out[f"img{i}.gt_difficult"] = gb, gl, gd
    np.savez_compressed(OUT / "g12_voc_eval.npz", **out)
    print("g12_voc_eval.npz:", total, "lines, aps07", out["aps07"].tolist())


if __name__ == "__main__":
    voc_eval_golden()
