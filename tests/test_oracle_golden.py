"""Pins the oracle restatement against fixtures recorded from the REAL reference
(oracle/gen_golden.py).  CPU only."""
import numpy as np
import pytest
import torch

from oracle import weights as W
from oracle import yolo_nano_oracle as O

# The fixtures were produced by the same torch/oneDNN build; on another CPU the conv
# kernels may pick a different blocking, so network outputs get a tight tolerance while
# everything downstream of recorded tensors is checked exactly.
NET_ATOL, NET_RTOL = 2e-5, 2e-5


@pytest.fixture(scope="module")
def g1(golden):
    return golden("g1_voc320_refinit.npz")


@pytest.fixture(scope="module")
def g2(golden):
    return golden("g2_coco128_calibrated.npz")


def test_reference_init_reproduces_reference_weights(g1):
    sd = W.reference_init(20, seed=0)
    assert len(sd) == 469
    assert W.digest(sd) == str(g1["sd_digest"])
    assert W.digest(W.synthetic_input(1, 320, 0)) == str(g1["x_digest"])


def test_network_and_decode_match_reference_c1(g1):
    sd = W.reference_init(20, seed=0)
    x = W.synthetic_input(1, 320, 0)
    taps = {}
    preds = O.network(sd, x, taps)
    for k in ("c3", "c4", "c5", "pred_s", "pred_m", "pred_l"):
        np.testing.assert_allclose(taps[k].numpy(), g1[k], rtol=NET_RTOL, atol=NET_ATOL, err_msg=k)
    bbox, cls = O.decode(preds, 320, 20, W.anchors_for(20))
    np.testing.assert_allclose(bbox[0].numpy(), g1["all_bbox"], atol=1e-6)
    score, ci = O.class_scores(cls[0].numpy())
    np.testing.assert_allclose(score, g1["all_score"], rtol=1e-5, atol=1e-8)


def test_postprocess_exact_on_recorded_candidates_c1(g1):
    """NMS restatement on the reference's own decoded tensors: keep-set must be identical
    (tie order 'numpy' = the reference expression itself)."""
    b, s, c, idx = O.postprocess_flat(g1["all_bbox"], g1["all_score"], g1["all_cls"].astype(np.int64),
                                      20, 0.001, 0.5, tie="numpy")
    np.testing.assert_array_equal(idx, g1["keep_idx"])
    np.testing.assert_array_equal(b, g1["bboxes"])
    np.testing.assert_array_equal(s, g1["scores"])
    np.testing.assert_array_equal(c, g1["cls_inds"])


def test_defined_tie_break_differs_only_on_ties_c1(g1):
    """With reference-init weights scores tie massively (SURVEY §8c hazard 2): the
    'index' tie-break this build defines may keep a slightly different set.  Count it."""
    _, _, _, idx = O.postprocess_flat(g1["all_bbox"], g1["all_score"], g1["all_cls"].astype(np.int64),
                                      20, 0.001, 0.5, tie="index")
    diff = np.setxor1d(idx, g1["keep_idx"])
    assert len(diff) <= 0.02 * len(g1["keep_idx"]), f"{len(diff)} boxes differ"


def test_every_tap_matches_reference_calibrated(g2):
    sd = W.calibrated(80, seed=1)
    assert W.digest(sd) == str(g2["sd_digest"])
    x = W.synthetic_input(2, 128, 1)
    assert W.digest(x) == str(g2["x_digest"])
    for i in range(2):
        taps = {}
        O.network(sd, x[i:i + 1], taps)
        names = [k.split(".", 1)[1] for k in g2.files if k.startswith(f"img{i}.") and k.split(".", 1)[1] in taps]
        assert len(names) >= 30
        for k in names:
            np.testing.assert_allclose(taps[k].numpy(), g2[f"img{i}.{k}"], rtol=NET_RTOL, atol=NET_ATOL, err_msg=k)


def test_batched_network_equals_per_image(g2):
    """SURVEY §8c hazard 4: the batch extension is defined as 'loop the reference'."""
    sd = W.calibrated(80, seed=1)
    x = W.synthetic_input(2, 128, 1)
    preds = O.network(sd, x)
    for i in range(2):
        np.testing.assert_allclose(preds[0][i].numpy(), g2[f"img{i}.pred_s"][0], rtol=NET_RTOL, atol=NET_ATOL)


@pytest.mark.parametrize("tag,kw", [("", dict(conf=0.001, nms=0.5, diou=False)),
                                    ("diou.", dict(conf=0.001, nms=0.5, diou=True)),
                                    ("t45c10.", dict(conf=0.1, nms=0.45, diou=False))])
def test_postprocess_variants_exact_calibrated(g2, tag, kw):
    """Tie-free inputs: both tie orders must give the reference keep-set bit-exactly,
    for plain NMS, DIoU-NMS and non-default thresholds."""
    for i in range(2):
        bb, sc, cl = g2[f"img{i}.all_bbox"], g2[f"img{i}.all_score"], g2[f"img{i}.all_cls"].astype(np.int64)
        for tie in ("numpy", "index"):
            _, _, _, idx = O.postprocess_flat(bb, sc, cl, 80, kw["conf"], kw["nms"], kw["diou"], tie)
            np.testing.assert_array_equal(idx, g2[f"img{i}.{tag}keep_idx"], err_msg=f"{tag}{tie}")


def test_fused_state_dict_path(g2):
    """fuse_conv_bn (utils/fuse_conv_bn.py) on our containers gives the reference's
    fused outputs; the oracle runs a fused (154-key) state_dict as well."""
    import contextlib, io
    import yolo_nano_b200 as pkg
    sd = W.calibrated(80, seed=1)
    with contextlib.redirect_stdout(io.StringIO()):
        m = pkg.YOLONano(torch.device("cpu"), 128, 80, anchor_size=pkg.MULTI_ANCHOR_SIZE_COCO)
    m.load_state_dict(sd)
    folded_before = m.fused_weights()
    pkg.fuse_conv_bn(m)
    fsd = m.state_dict()
    assert len(fsd) == 154
    folded_after = m.fused_weights()
    for k in folded_before:
        assert torch.equal(folded_before[k][0], folded_after[k][0])
        assert torch.equal(folded_before[k][1], folded_after[k][1])
    x = W.synthetic_input(2, 128, 1)
    preds = O.network({k: v for k, v in fsd.items()}, x[0:1])
    np.testing.assert_allclose(preds[0].numpy(), g2["img0.fused.pred_s"], rtol=NET_RTOL, atol=NET_ATOL)
    # folding table used by the engine == what fuse_conv_bn wrote into the module
    tab = O.fold_state_dict(sd, pkg.conv_table(80))
    for k, (w, b) in tab.items():
        assert torch.equal(w, fsd[k + ".weight"]) and torch.equal(b, fsd[k + ".bias"])


def test_g3_keepsets(golden):
    for tag in ("calibrated", "refinit"):
        g = golden(f"g3_coco416_{tag}.npz")
        for i in range(2):
            bb, sc, cl = g[f"img{i}.all_bbox"], g[f"img{i}.all_score"], g[f"img{i}.all_cls"].astype(np.int64)
            _, _, _, idx = O.postprocess_flat(bb, sc, cl, 80, 0.001, 0.5, tie="numpy")
            np.testing.assert_array_equal(idx, g[f"img{i}.keep_idx"])
            _, _, _, idx2 = O.postprocess_flat(bb, sc, cl, 80, 0.001, 0.5, tie="index")
            if tag == "calibrated":
                np.testing.assert_array_equal(idx2, g[f"img{i}.keep_idx"])
            else:
                assert len(np.setxor1d(idx2, g[f"img{i}.keep_idx"])) <= 0.02 * len(idx)


def test_preprocess_restatement_matches_reference_valtransforms(golden):
    """oracle.preprocess_u8 against the real ValTransforms (data/transforms.py:445-458) recorded by
    oracle/gen_golden.py: square (no resize), landscape and portrait (padding with mean*255)."""
    g = golden("g4_preprocess64.npz")
    for name in ("square", "landscape", "portrait"):
        rect = g[f"{name}.rect"]
        t = O.preprocess_u8(g[f"{name}.canvas"], None if name == "square" else rect)
        np.testing.assert_array_equal(t, g[f"{name}.tensor"])


def test_tta_restatement_matches_reference_driver(golden):
    """oracle.tta against the real TestTimeAugmentation + reference model (utils/misc.py:90-148):
    3 scales x flip, merge NMS 0.4 — identical boxes, scores, labels."""
    g = golden("g5_tta128_calibrated.npz")
    sd = W.calibrated(20, seed=6)
    x = W.synthetic_input(1, 128, 6)
    b, s, c = O.tta(sd, x, 20, W.anchors_for(20), g["scales"], 0.4)
    np.testing.assert_array_equal(c, g["labels"])
    np.testing.assert_array_equal(b, g["bboxes"])
    np.testing.assert_array_equal(s, g["scores"])


def test_evaluator_glue_matches_reference_evaluators(golden):
    """yolo_nano_b200.evalfmt against the real evaluators run on fixed detections (golden g6):
    inverse letterbox mapping, COCO result rows (cocoapi_evaluator.py:85-100), VOC per-class arrays and
    det-file lines (vocapi_evaluator.py:72-86,148-157)."""
    import json
    from yolo_nano_b200 import evalfmt
    g = golden("g6_evalfmt.npz")
    class_ids = g["class_ids"].tolist()
    labelmap = [str(v) for v in g["labelmap"]]
    rows, voc = [], {c: "" for c in labelmap}
    for i, (h, w) in enumerate(g["sizes"].tolist()):
        b = g[f"img{i}.bboxes"].copy()
        evalfmt.map_to_image(b, g[f"img{i}.scale"], g[f"img{i}.offset"], w, h)
        np.testing.assert_array_equal(b, g[f"img{i}.mapped"])
        rows += evalfmt.coco_result_rows(1000 + i, b, g[f"img{i}.scores"], g[f"img{i}.cls"], class_ids)
        per_cls = evalfmt.voc_class_dets(b, g[f"img{i}.scores"], g[f"img{i}.cls"], len(labelmap))
        for c, d in zip(labelmap, per_cls):
            assert d.dtype == np.float32 and d.shape[1] == 5
            voc[c] += "".join(evalfmt.voc_result_lines(f"{i + 1:06d}", d))
    assert rows == json.loads(str(g["coco_json"]))
    for c in labelmap:
        assert voc[c] == str(g[f"voc.{c}"]), c


def test_letterbox_transform_and_box_mapping_match_reference(golden):
    """oracle.val_transform (cv2 bilinear resize restated + letterbox + Normalize + ToTensor) and
    oracle.map_boxes_to_image against the REAL ValTransforms / evaluator code (golden g9): bit-identical."""
    g9 = golden("g9_letterbox96.npz")
    size = int(g9["size"])
    for i in range(int(g9["n"])):
        img = g9[f"img{i}"]
        x, scale, offset = O.val_transform(img, size)
        np.testing.assert_array_equal(x, g9[f"x{i}"], err_msg=f"image {i} {img.shape}")
        got = O.map_boxes_to_image(g9[f"boxes{i}"], scale, offset, img.shape[1], img.shape[0])
        np.testing.assert_array_equal(got, g9[f"mapped{i}"])


def test_cv2_resize_restatement_is_bit_exact(golden):
    """The restated OpenCV bilinear uint8 resize against cv2.resize over random shapes (incl. the exact 2x
    downscale fast path and up-scaling), as recorded by oracle/gen_golden.py (golden g11: SHA-256 of every cv2
    output plus 256 sampled values)."""
    import hashlib
    from oracle.gen_golden import resize_cases
    g = golden("g11_cv2resize.npz")
    cases = list(resize_cases())
    assert [c[:4] for c in cases] == [tuple(s) for s in g["shapes"].tolist()]
    for i, (h0, w0, dw, dh, img) in enumerate(cases):
        assert hashlib.sha256(img.tobytes()).hexdigest() == str(g[f"in_sha{i}"]), f"input {i} is not the recorded one"
        got = O.cv2_resize_linear_u8(img, dw, dh)
        assert got.shape == (dh, dw, 3) and got.dtype == np.uint8, str((h0, w0, dw, dh))
        np.testing.assert_array_equal(got.reshape(-1)[g[f"idx{i}"]], g[f"vals{i}"], err_msg=str((h0, w0, dw, dh)))
        assert hashlib.sha256(got.tobytes()).hexdigest() == str(g[f"out_sha{i}"]), str((h0, w0, dw, dh))
