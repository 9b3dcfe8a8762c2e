"""Generates tests/golden/*.npz by running the REAL reference (/root/reference).

Run in the build container only (the reference checkout does not exist on the GPU
box):   python -m oracle.gen_golden
The fixtures pin the oracle restatement (tests/test_oracle_golden.py) and are the
reference-side truth the CUDA path is compared with (tests/test_gpu_*.py).

Recipe = SURVEY App. C: PYTHONDONTWRITEBYTECODE (read-only tree), `np.int = int` shim for
models/yolo_nano.py:264, construct with trainable=False (no download).
"""
from __future__ import annotations

import contextlib
import io
import os
import sys
from pathlib import Path

import numpy as np
import torch

REF = "/root/reference"
OUT = Path(__file__).resolve().parent.parent / "tests" / "golden"


def _import_reference():
    sys.dont_write_bytecode = True
    np.int = int  # noqa: NPY001 - shim for the reference on NumPy >= 1.24
    if REF not in sys.path:
        sys.path.insert(0, REF)
    with contextlib.redirect_stdout(io.StringIO()):
        from models.yolo_nano import YOLONano  # type: ignore
        from data import config  # type: ignore
        from utils.fuse_conv_bn import fuse_conv_bn  # type: ignore
    return YOLONano, config, fuse_conv_bn


def _build(YOLONano, size, classes, anchors, sd=None, seed=0, **kw):
    torch.manual_seed(seed)
    with contextlib.redirect_stdout(io.StringIO()):
        m = YOLONano(device=torch.device("cpu"), input_size=size, num_classes=classes,
                     anchor_size=anchors, **kw).eval()
    if sd is not None:
        m.load_state_dict(sd, strict=True)
    return m


def _run_one(m, x1, tap_names=()):
    """Reference forward on ONE image with taps; returns dict of numpy arrays."""
    rec = {}
    hooks = []

    def hook(name):
        def f(_mod, _inp, out):
            rec[name] = out.detach().numpy().copy()
        return f

    named = dict(m.named_modules())
    tapmap = {"pool": "backbone.maxpool", "lat3": "conv1x1_0", "lat4": "conv1x1_1", "lat5": "conv1x1_2",
              "p3": "smooth_1", "p4": "smooth_2", "p5": "smooth_3", "fpn4": "smooth_0",
              "pred_s": "head_det_1", "pred_m": "head_det_2", "pred_l": "head_det_3"}
    for st, rep in ((2, 4), (3, 8), (4, 4)):
        for i in range(rep):
            tapmap[f"stage{st}.{i}"] = f"backbone.stage{st}.{i}"
    tapmap["c3"], tapmap["c4"], tapmap["c5"] = "backbone.stage2", "backbone.stage3", "backbone.stage4"
    for t in tap_names:
        hooks.append(named[tapmap[t]].register_forward_hook(hook(t)))

    orig_post = m.postprocess

    def post(all_local, all_conf):
        rec["all_bbox"] = all_local.copy()
        cls = np.argmax(all_conf, axis=1)
        rec["all_score"] = all_conf[(np.arange(all_conf.shape[0]), cls)].copy()
        rec["all_cls"] = cls.astype(np.int32)
        # 5th column carries the anchor index through the reference's own row selection
        aug = np.concatenate([all_local, np.arange(len(all_local), dtype=np.float32)[:, None]], 1)
        b, s, c = orig_post(aug, all_conf)
        rec["keep_idx"] = b[:, 4].astype(np.int64)
        return b[:, :4].copy(), s, c

    m.postprocess = post
    with torch.no_grad():
        b, s, c = m(x1)
    m.postprocess = orig_post
    for h in hooks:
        h.remove()
    rec["bboxes"], rec["scores"], rec["cls_inds"] = b, s, c.astype(np.int64)
    return rec


def main():
    from oracle import weights as W
    YOLONano, config, fuse_conv_bn = _import_reference()
    OUT.mkdir(parents=True, exist_ok=True)
    torch.set_num_threads(min(8, os.cpu_count() or 1))
    meta_common = dict(torch=torch.__version__, numpy=np.__version__)

    # ---- G1: BASELINE config C1 — 320x320, VOC-20, B=1, reference init --------------------
    m = _build(YOLONano, 320, 20, config.MULTI_ANCHOR_SIZE, seed=0)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    mine = W.reference_init(20, seed=0)
    assert list(mine.keys()) == list(sd.keys()) and all(torch.equal(mine[k], sd[k]) for k in sd), \
        "parameter containers do not reproduce the reference init"
    x = W.synthetic_input(1, 320, seed=0)
    r = _run_one(m, x, ("c3", "c4", "c5", "pred_s", "pred_m", "pred_l"))
    np.savez_compressed(OUT / "g1_voc320_refinit.npz", sd_digest=W.digest(sd), x_digest=W.digest(x),
                        size=320, classes=20, seed=0, conf_thresh=0.001, nms_thresh=0.5, **meta_common, **r)
    print("g1", r["bboxes"].shape, W.digest(sd))

    # ---- G2: 128x128, COCO-80, B=2, calibrated weights, every tap ---------------------------
    sd = W.calibrated(80, seed=1)
    m = _build(YOLONano, 128, 80, config.MULTI_ANCHOR_SIZE_COCO, sd=sd)
    x = W.synthetic_input(2, 128, seed=1)
    taps = ["pool", "c3", "c4", "c5", "lat3", "lat4", "lat5", "fpn4", "p3", "p4", "p5",
            "pred_s", "pred_m", "pred_l"] + [f"stage{s}.{i}" for s, n in ((2, 4), (3, 8), (4, 4)) for i in range(n)]
    out = {}
    for i in range(2):
        r = _run_one(m, x[i:i + 1], taps)
        for k, v in r.items():
            out[f"img{i}.{k}"] = v
    # DIoU + other thresholds on the same decoded candidates
    for tag, kw in (("diou", dict(diou_nms=True)), ("t45c10", dict(conf_thresh=0.1, nms_thresh=0.45))):
        m2 = _build(YOLONano, 128, 80, config.MULTI_ANCHOR_SIZE_COCO, sd=sd, **kw)
        for i in range(2):
            r = _run_one(m2, x[i:i + 1])
            out[f"img{i}.{tag}.keep_idx"] = r["keep_idx"]
    # fused model (utils/fuse_conv_bn.py): outputs after folding
    m3 = fuse_conv_bn(_build(YOLONano, 128, 80, config.MULTI_ANCHOR_SIZE_COCO, sd=sd))
    assert len(m3.state_dict()) == 154
    r = _run_one(m3, x[0:1], ("pred_s",))
    out["img0.fused.pred_s"] = r["pred_s"]
    out["img0.fused.keep_idx"] = r["keep_idx"]
    np.savez_compressed(OUT / "g2_coco128_calibrated.npz", sd_digest=W.digest(sd), x_digest=W.digest(x),
                        size=128, classes=80, seed=1, conf_thresh=0.001, nms_thresh=0.5, **meta_common, **out)
    print("g2", out["img0.bboxes"].shape, out["img1.bboxes"].shape, W.digest(sd))

    # ---- G3: 416x416, COCO-80 (the bench config's shape), calibrated + reference init -------
    for tag, sd, seed in (("calibrated", W.calibrated(80, seed=2), 2), ("refinit", W.reference_init(80, seed=3), 3)):
        m = _build(YOLONano, 416, 80, config.MULTI_ANCHOR_SIZE_COCO, sd=sd)
        x = W.synthetic_input(2, 416, seed=seed)
        out = {}
        for i in range(2):
            r = _run_one(m, x[i:i + 1])
            for k in ("all_bbox", "all_score", "all_cls", "keep_idx", "bboxes", "scores", "cls_inds"):
                out[f"img{i}.{k}"] = r[k]
        np.savez_compressed(OUT / f"g3_coco416_{tag}.npz", sd_digest=W.digest(sd), x_digest=W.digest(x),
                            size=416, classes=80, seed=seed, conf_thresh=0.001, nms_thresh=0.5,
                            **meta_common, **out)
        print("g3", tag, out["img0.bboxes"].shape, out["img1.bboxes"].shape)


def preprocess_golden():
    """G4: the reference's ValTransforms (data/transforms.py:445-458) on uint8 BGR images — square
    (no resize), landscape and portrait (cv2.resize + padding with mean*255).  Stored: the letterboxed
    uint8 canvas + content rectangle our pre-processing entry takes, and the reference's tensor."""
    import cv2
    sys.dont_write_bytecode = True
    if REF not in sys.path:
        sys.path.insert(0, REF)
    from data.transforms import ValTransforms  # type: ignore
    rng = np.random.default_rng(7)
    size = 64
    out = {}
    for name, (h0, w0) in (("square", (64, 64)), ("landscape", (48, 80)), ("portrait", (90, 50))):
        img = rng.integers(0, 256, (h0, w0, 3), dtype=np.uint8)
        tensor, _, _, scale, offset = ValTransforms(size)(img)
        tensor = tensor.numpy()
        # what the host side of OUR entry does: the same cv2.resize call, content placed on a canvas
        canvas = np.zeros((size, size, 3), np.uint8)
        if h0 > w0:
            content = cv2.resize(img, (int(w0 / h0 * size), size))
            left = (size - content.shape[1]) // 2
            rect = (left, 0, content.shape[1], size)
        elif h0 < w0:
            content = cv2.resize(img, (size, int(h0 / w0 * size)))
            top = (size - content.shape[0]) // 2
            rect = (0, top, size, content.shape[0])
        else:
            content = img if h0 == size else cv2.resize(img, (size, size))
            rect = (0, 0, size, size)
        canvas[rect[1]:rect[1] + rect[3], rect[0]:rect[0] + rect[2]] = content
        assert tensor.shape == (3, size, size), tensor.shape
        out[f"{name}.canvas"] = canvas
        out[f"{name}.rect"] = np.array(rect, np.int32)
        out[f"{name}.tensor"] = tensor.astype(np.float32)
    np.savez_compressed(OUT / "g4_preprocess64.npz", size=size, numpy=np.__version__, cv2=cv2.__version__, **out)
    print("g4", {k: v.shape for k, v in out.items() if k.endswith("tensor")})


def tta_golden():
    """G5: the reference's TestTimeAugmentation (utils/misc.py:90-148) driving the reference model:
    calibrated VOC-20 weights, 128^2 input, scales 96 / 128 / 160, flips, merge NMS 0.4."""
    from oracle import weights as W
    YOLONano, config, _ = _import_reference()
    from utils.misc import TestTimeAugmentation  # type: ignore
    sd = W.calibrated(20, seed=6)
    m = _build(YOLONano, 128, 20, config.MULTI_ANCHOR_SIZE, sd=sd)
    x = W.synthetic_input(1, 128, 6)
    tta = TestTimeAugmentation(num_classes=20, nms_thresh=0.4, scale_range=[96, 160, 32])
    with torch.no_grad():
        b, s, c = tta(x, m)
    np.savez_compressed(OUT / "g5_tta128_calibrated.npz", bboxes=b.astype(np.float32), scores=s.astype(np.float32),
                        labels=c.astype(np.int64), scales=np.array(tta.scales), seed=6, numpy=np.__version__,
                        torch=torch.__version__)
    print("g5", b.shape, np.bincount(c, minlength=20).tolist())


def evalfmt_golden():
    """G6: the reference evaluators' own code on fixed detections — COCOAPIEvaluator.evaluate up to the
    result JSON (evaluator/cocoapi_evaluator.py:47-112, fake dataset / model / COCO object) and
    VOCAPIEvaluator.write_voc_results_file (evaluator/vocapi_evaluator.py:142-157)."""
    import json
    import tempfile
    from types import SimpleNamespace
    _import_reference()
    with contextlib.redirect_stdout(io.StringIO()):
        from evaluator.cocoapi_evaluator import COCOAPIEvaluator  # type: ignore
        from evaluator.vocapi_evaluator import VOCAPIEvaluator  # type: ignore
    rng = np.random.default_rng(12)
    n_img, sizes = 2, [(480, 640), (500, 375)]          # (h, w)
    dets, scales, offsets = [], [], []
    for h, w in sizes:
        k = 7
        xy = rng.random((k, 2), dtype=np.float32) * 0.6
        b = np.concatenate([xy, xy + rng.random((k, 2), dtype=np.float32) * 0.3 + 0.05], 1).astype(np.float32)
        dets.append((b, rng.random(k, dtype=np.float32), rng.integers(0, 5, k).astype(np.int64)))
        if h < w:
            scales.append(np.array([1., h / w, 1., h / w])); offsets.append(np.array([[0., (w - h) // 2 / w, 0., (w - h) // 2 / w]]))
        else:
            scales.append(np.array([[w / h, 1., w / h, 1.]])); offsets.append(np.array([[(h - w) // 2 / h, 0., (h - w) // 2 / h, 0.]]))
    class_ids = [1, 3, 7, 18, 44]
    state = {"i": 0}

    class FakeModel:
        def eval(self):
            return self
        def __call__(self, x):
            b, s, c = dets[state["i"]]
            return b.copy(), s.copy(), c.copy()

    def transform(img):
        i = state["i"]
        return torch.zeros(3, 8, 8), None, None, scales[i], offsets[i]

    class FakeDataset:
        class_ids = [1, 3, 7, 18, 44]
        coco = SimpleNamespace(loadRes=lambda path: None)
        def __len__(self):
            return n_img
        def pull_image(self, index):
            state["i"] = index
            h, w = sizes[index]
            return np.zeros((h, w, 3), np.uint8), 1000 + index

    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        os.chdir(tmp)
        try:
            fake = SimpleNamespace(dataset=FakeDataset(), transform=transform, device=torch.device("cpu"), testset=True)
            with contextlib.redirect_stdout(io.StringIO()):
                COCOAPIEvaluator.evaluate(fake, FakeModel())
            coco_json = open("coco_test-dev.json").read()
            # VOC: boxes mapped exactly as evaluate() does (:72-74), per-class arrays (:76-86), then the writer
            labelmap = ["aeroplane", "bicycle", "bird", "boat", "bottle"]
            all_boxes = [[[] for _ in range(n_img)] for _ in labelmap]
            mapped = []
            for i, (h, w) in enumerate(sizes):
                b, s, c = (v.copy() for v in dets[i])
                size = np.array([[w, h, w, h]])
                b -= offsets[i]; b /= scales[i]; b *= size
                mapped.append(b.copy())
                for j in range(len(labelmap)):
                    inds = np.where(c == j)[0]
                    if len(inds) == 0:
                        all_boxes[j][i] = np.empty([0, 5], dtype=np.float32)
                        continue
                    all_boxes[j][i] = np.hstack((b[inds], s[inds][:, np.newaxis])).astype(np.float32, copy=False)
            # `if dets == []` (:150) raises on NumPy >= 2 for arrays; old NumPy answered False: same shim idea as np.int
            class _Arr(np.ndarray):
                def __eq__(self, other):
                    return False if isinstance(other, list) else np.ndarray.__eq__(self, other)
            all_boxes = [[a.view(_Arr) for a in row] for row in all_boxes]
            fake_voc = SimpleNamespace(labelmap=labelmap, display=False,
                                       dataset=SimpleNamespace(ids=[("VOC2007", "000001"), ("VOC2007", "000002")]),
                                       get_voc_results_file_template=lambda cls: os.path.join(tmp, "det_test_%s.txt" % cls))
            VOCAPIEvaluator.write_voc_results_file(fake_voc, all_boxes)
            voc_files = {cls: open(os.path.join(tmp, "det_test_%s.txt" % cls)).read() for cls in labelmap}
        finally:
            os.chdir(cwd)
    out = {"coco_json": np.array(coco_json), "class_ids": np.array(class_ids), "sizes": np.array(sizes),
           "labelmap": np.array(labelmap)}
    for i in range(n_img):
        out[f"img{i}.bboxes"], out[f"img{i}.scores"], out[f"img{i}.cls"] = dets[i]
        out[f"img{i}.scale"], out[f"img{i}.offset"], out[f"img{i}.mapped"] = scales[i], offsets[i], mapped[i]
    for cls, txt in voc_files.items():
        out[f"voc.{cls}"] = np.array(txt)
    np.savez_compressed(OUT / "g6_evalfmt.npz", **out)
    print("g6", len(json.loads(coco_json)), "coco rows;", {k: len(v.splitlines()) for k, v in voc_files.items()})


def train_labels(batch: int, seed: int):
    """Synthetic normalised labels [[xmin,ymin,xmax,ymax,cls],...] per image: random boxes plus the
    edge cases of tools.py:97-216 (a 'dirty' sub-pixel box, two boxes on the same cell/anchor, a
    box matching several anchors -> ignored (-1) entries, a box with no anchor above the threshold)."""
    rng = np.random.RandomState(seed)
    out = []
    for b in range(batch):
        labs = []
        for _ in range(6):
            cx, cy = rng.uniform(0.15, 0.85, 2)
            w, h = rng.uniform(0.05, 0.6, 2)
            labs.append([max(cx - w / 2, 0.0), max(cy - h / 2, 0.0), min(cx + w / 2, 1.0), min(cy + h / 2, 1.0),
                         float(rng.randint(0, 20))])
        labs.append([0.5, 0.5, 0.503, 0.7, 3.0])                 # dirty: narrower than one pixel
        labs.append([0.30, 0.30, 0.52, 0.50, 7.0])               # same cell and anchor ...
        labs.append([0.305, 0.305, 0.525, 0.505, 9.0])           # ... the later one wins
        labs.append([0.1, 0.4, 0.9, 0.45, 11.0])                 # extreme aspect: no anchor above 0.5
        labs.append([0.109375, 0.03125, 0.890625, 0.96875, 13.0])  # 100x120 px at 128: three anchors > 0.5
        labs.append([0.2, 0.1, 0.2 + 60 / 128, 0.1 + 90 / 128, 2.0])  # 60x90 px: two anchors > 0.5
        # the data loader hands the labels over as float32 tensors (train.py:211): keep the fixture on
        # float32-representable values so that the device entry (float32 labels) sees the same numbers
        out.append([[float(np.float32(v)) for v in lab] for lab in labs])
    return out


def train_golden():
    """g7: the reference's training branch at the head boundary (SURVEY 8 row a14): targets from
    tools.multi_gt_creator, the four losses of forward(x, target) with trainable=True (BN in eval
    mode so that the network part is the inference network), d(total)/d(raw head maps)."""
    from oracle import weights as W
    YOLONano, config, _ = _import_reference()
    import tools  # type: ignore  (reference)
    torch.set_num_threads(min(8, os.cpu_count() or 1))
    size, classes, batch, seed = 128, 20, 2, 7
    sd = W.calibrated(classes, seed=seed)
    m = _build(YOLONano, size, classes, config.MULTI_ANCHOR_SIZE, sd=sd)
    m.trainable = True           # constructing with trainable=True would download weights (:32)
    x = W.synthetic_input(batch, size, seed=seed)
    labels = train_labels(batch, seed)
    target = tools.multi_gt_creator(size, m.stride, labels, anchor_size=config.MULTI_ANCHOR_SIZE)
    rec = {}
    hooks = []
    for name, mod in (("pred_s", m.head_det_1), ("pred_m", m.head_det_2), ("pred_l", m.head_det_3)):
        def f(_mod, _inp, out, name=name):
            out.retain_grad()
            rec[name] = out
        hooks.append(mod.register_forward_hook(f))
    ls = m(x, target=target)
    sum(ls).backward()
    for h in hooks:
        h.remove()
    out = {"target": target.numpy(), "losses": np.array([float(v.detach()) for v in ls], dtype=np.float32)}
    for k, v in rec.items():
        out[k] = v.detach().numpy().copy()
        out["grad_" + k] = v.grad.numpy().copy()
    lab = np.full((batch, max(len(l) for l in labels), 5), -1.0, dtype=np.float64)
    for b, l in enumerate(labels):
        lab[b, :len(l)] = np.asarray(l)
    # one torch.optim.SGD step (train.py:167-171) on a flat vector, twice (first step / momentum)
    g = torch.Generator().manual_seed(seed)
    p0 = torch.randn(20011, generator=g)
    g1, g2 = torch.randn(20011, generator=g) * 0.1, torch.randn(20011, generator=g) * 0.1
    prm = torch.nn.Parameter(p0.clone())
    opt = torch.optim.SGD([prm], lr=1e-3, momentum=0.9, weight_decay=5e-4)
    prm.grad = g1.clone(); opt.step()
    p1 = prm.detach().clone()
    prm.grad = g2.clone(); opt.step()
    np.savez_compressed(OUT / "g7_train128.npz", size=size, classes=classes, seed=seed, labels=lab,
                        n_labels=np.array([len(l) for l in labels]), sd_digest=W.digest(sd), x_digest=W.digest(x),
                        sgd_p0=p0.numpy(), sgd_g1=g1.numpy(), sgd_g2=g2.numpy(), sgd_p1=p1.numpy(),
                        sgd_p2=prm.detach().numpy(), torch=torch.__version__, numpy=np.__version__, **out)
    print("g7 losses", out["losses"], "positives", int((target[:, :, 0] > 0).sum()), "ignored", int((target[:, :, 0] < 0).sum()))


def train_step_golden():
    """g10: the REAL reference in train() mode (BatchNorm on batch statistics): forward(x, target) with
    trainable=True, total_loss.backward() (train.py:219-229) at 128^2 / VOC-20 / batch 4, calibrated weights.
    Stored: the four losses, (sum, abs-sum, max-abs) of every parameter gradient (247 x 3), a few gradients in
    full, the running statistics of three BatchNorm layers after the step."""
    from oracle import weights as W
    YOLONano, config, _ = _import_reference()
    import tools  # type: ignore  (reference)
    torch.set_num_threads(min(8, os.cpu_count() or 1))
    size, classes, batch, seed = 128, 20, 4, 10
    sd = W.calibrated(classes, seed=seed)
    m = _build(YOLONano, size, classes, config.MULTI_ANCHOR_SIZE, sd=sd)
    m.trainable = True
    m.train()
    x = W.synthetic_input(batch, size, seed=seed)
    labels = train_labels(batch, seed)
    target = tools.multi_gt_creator(size, m.stride, labels, anchor_size=config.MULTI_ANCHOR_SIZE)
    ls = m(x, target=target)
    sum(ls).backward()
    names, stats = [], []
    out = {"size": size, "classes": classes, "batch": batch, "seed": seed, "sd_digest": W.digest(sd), "x_digest": W.digest(x),
           "target": target.numpy(), "losses": np.array([float(v.detach()) for v in ls], dtype=np.float32)}
    for k, p_ in m.named_parameters():
        g = p_.grad
        names.append(k)
        stats.append([float(g.double().sum()), float(g.double().abs().sum()), float(g.abs().max())])
    out["grad_names"] = np.array(names)
    out["grad_stats"] = np.array(stats, dtype=np.float64)
    full = ["backbone.conv1.0.weight", "backbone.conv1.1.weight", "backbone.stage2.0.branch1.0.weight",
            "backbone.stage2.1.branch2.0.weight", "backbone.stage3.3.branch2.4.bias", "backbone.stage4.3.branch2.5.weight",
            "conv1x1_1.convs.0.bias", "smooth_1.convs.1.weight", "head_det_1.0.convs.0.weight", "head_det_2.4.bias",
            "head_det_3.4.weight"]
    pd = dict(m.named_parameters())
    for k in full:
        out["grad." + k] = pd[k].grad.numpy().copy()
    msd = m.state_dict()
    for k in ("backbone.conv1.1", "backbone.stage3.0.branch2.4", "head_det_1.3.convs.1"):
        out["rm." + k] = msd[k + ".running_mean"].numpy().copy()
        out["rv." + k] = msd[k + ".running_var"].numpy().copy()
        out["nbt." + k] = msd[k + ".num_batches_tracked"].numpy().copy()
    # The reference's OWN float32 rounding sensitivity: LeakyReLU / ReLU / max-pool are piecewise linear, the forward
    # amplifies a 1-ulp input change to ~1e-4 at the deep activations, so a handful of units change side and the
    # gradients of the layers below move by per cent.  Stored per parameter: the largest change of the gradient
    # (relative to its max-abs) over four input perturbations of relative size 1e-6 — the bound any other float32
    # implementation of the same graph (different summation order) can be held to.
    base = {k: p_.grad.clone() for k, p_ in m.named_parameters()}
    sens = np.zeros(len(names))
    for trial in range(4):
        m.zero_grad()
        noise = torch.randn(x.shape, generator=torch.Generator().manual_seed(100 + trial))
        sum(m(x * (1.0 + 1e-6 * noise), target=target)).backward()
        for i, (k, p_) in enumerate(m.named_parameters()):
            sens[i] = max(sens[i], float((p_.grad - base[k]).abs().max() / base[k].abs().max().clamp_min(1e-30)))
    out["grad_sens"] = sens
    for k, p_ in m.named_parameters():
        p_.grad = base[k]
    np.savez_compressed(OUT / "g10_trainstep128.npz", torch=torch.__version__, **out)
    print("g10_trainstep128.npz: losses", out["losses"], len(names), "parameters")


def letterbox_golden():
    """g9: the REAL ValTransforms (data/transforms.py:445-458, cv2.resize inside) on uint8 BGR images of assorted
    shapes at size 96, and the evaluator's inverse box mapping (evaluator/cocoapi_evaluator.py:85-87) on fixed boxes."""
    import cv2
    sys.dont_write_bytecode = True
    if REF not in sys.path:
        sys.path.insert(0, REF)
    from data.transforms import ValTransforms  # type: ignore
    rng = np.random.default_rng(9)
    size = 96
    shapes = [(96, 96), (60, 60), (192, 192), (75, 100), (100, 75), (37, 91), (200, 131), (192, 150), (48, 192), (333, 500)]
    out = {"size": size, "n": len(shapes)}
    for i, (h0, w0) in enumerate(shapes):
        img = rng.integers(0, 256, (h0, w0, 3), dtype=np.uint8)
        tensor, _, _, scale, offset = ValTransforms(size)(img)
        boxes = rng.random((7, 4)).astype(np.float32)
        mapped = boxes.copy()
        mapped -= offset
        mapped /= scale
        mapped *= np.array([[w0, h0, w0, h0]])
        out[f"img{i}"] = img
        out[f"x{i}"] = tensor.numpy().astype(np.float32)
        out[f"boxes{i}"] = boxes
        out[f"mapped{i}"] = mapped
    np.savez_compressed(OUT / "g9_letterbox96.npz", cv2=cv2.__version__, numpy=np.__version__, **out)
    print("g9_letterbox96.npz:", len(shapes), "images")


def resize_cases():
    """Yields (h0, w0, dw, dh, image) of the cv2 resize check: fixed shapes (the exact 2x downscale fast path,
    up-scaling) and 25 random letterbox-style shapes, uint8 HWC noise images from one seeded generator."""
    rng = np.random.default_rng(1)
    shapes = [(480, 640, 416, 312), (640, 480, 312, 416), (100, 100, 416, 416), (832, 832, 416, 416), (37, 91, 416, 169)]
    for _ in range(25):
        h0, w0 = int(rng.integers(20, 700)), int(rng.integers(20, 700))
        s = int(rng.choice([320, 416, 608]))
        shapes.append((h0, w0, max(1, int(w0 / h0 * s)) if h0 > w0 else s, s if h0 >= w0 else max(1, int(h0 / w0 * s))))
    for h0, w0, dw, dh in shapes:
        yield h0, w0, dw, dh, rng.integers(0, 256, (h0, w0, 3), dtype=np.uint8)


def resize_golden():
    """g11: cv2.resize (INTER_LINEAR, the call inside ValTransforms) on the cases of resize_cases().  The outputs
    are ~10 MB of noise, so each is stored as the SHA-256 of its bytes (bit-exact check) plus 256 values at seeded
    positions (to show where a mismatch is); the input's SHA-256 pins the generated image."""
    import hashlib
    import cv2
    out = {}
    shapes = []
    for i, (h0, w0, dw, dh, img) in enumerate(resize_cases()):
        want = cv2.resize(img, (dw, dh))
        idx = np.random.default_rng(i).choice(want.size, 256, replace=False)
        shapes.append((h0, w0, dw, dh))
        out[f"in_sha{i}"] = hashlib.sha256(img.tobytes()).hexdigest()
        out[f"out_sha{i}"] = hashlib.sha256(want.tobytes()).hexdigest()
        out[f"idx{i}"] = idx
        out[f"vals{i}"] = want.reshape(-1)[idx]
    np.savez_compressed(OUT / "g11_cv2resize.npz", cv2=cv2.__version__, numpy=np.__version__,
                        shapes=np.array(shapes, dtype=np.int64), **out)
    print("g11_cv2resize.npz:", len(shapes), "cases")


def ema_golden():
    """g8: the REAL ModelEMA (utils/misc.py:67-86) over three updates of a model whose weights change between
    updates the way an optimizer would change them (deterministic perturbations)."""
    _import_reference()
    from utils.misc import ModelEMA  # type: ignore
    from oracle.train_oracle import ema_model, ema_perturb
    seed = 8
    m = ema_model(seed)
    ema = ModelEMA(m, decay=0.9999, updates=1500)
    out = {"seed": seed, "start_updates": 1500}
    g = torch.Generator().manual_seed(seed + 1)
    for step in range(3):
        ema_perturb(m, g)
        ema.update(m)
        out[f"decay{step}"] = np.float64(ema.decay(ema.updates))
    for k, v in ema.ema.state_dict().items():
        out["ema." + k] = v.numpy()
    np.savez_compressed(OUT / "g8_ema.npz", torch=torch.__version__, **out)
    print("g8_ema.npz:", len(out), "entries, updates", ema.updates)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "evalfmt":
        evalfmt_golden()
    elif len(sys.argv) > 1 and sys.argv[1] == "preprocess":
        preprocess_golden()
    elif len(sys.argv) > 1 and sys.argv[1] == "tta":
        tta_golden()
    elif len(sys.argv) > 1 and sys.argv[1] == "trainstep":
        train_step_golden()
    elif len(sys.argv) > 1 and sys.argv[1] == "letterbox":
        letterbox_golden()
    elif len(sys.argv) > 1 and sys.argv[1] == "ema":
        ema_golden()
    elif len(sys.argv) > 1 and sys.argv[1] == "resize":
        resize_golden()
    elif len(sys.argv) > 1 and sys.argv[1] == "train":
        train_golden()
    else:
        main()
        preprocess_golden()
        tta_golden()
        evalfmt_golden()
        train_golden()
