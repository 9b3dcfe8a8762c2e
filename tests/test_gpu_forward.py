"""End-to-end parity of the engine and the drop-in module on a real B200."""
import contextlib
import ctypes as C
import io

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import weights as W  # noqa: E402
from oracle import yolo_nano_oracle as O  # noqa: E402

TAPS = ["pool"] + [f"stage{s}.{i}" for s, n in ((2, 4), (3, 8), (4, 4)) for i in range(n)] + \
       ["c3", "c4", "c5", "lat3", "lat4", "lat5", "fpn4", "p3", "p4", "p5", "pred_s", "pred_m", "pred_l"]
# Per-layer tolerance relative to the layer's own scale, per arithmetic mode.  Rounding
# differences compound through ~45 layers: the fp32 FFMA path itself ends 3e-5 away from
# the oneDNN reference (measured), so 1e-4 is "fp32-grade"; single-pass TF32 is the
# throughput mode (reported separately, not a parity mode).
LAYER_TOL = {"ffma": 1e-4, "3xtf32": 1e-4, "tf32": 0.3}


@pytest.fixture(scope="module")
def G():
    import gpu_util
    return gpu_util


@pytest.fixture(scope="module")
def g2(golden):
    return golden("g2_coco128_calibrated.npz")


@pytest.mark.parametrize("mode", ["ffma", "3xtf32", "tf32"])
def test_every_layer_matches_reference_calibrated(G, g2, mode):
    """Per-layer parity against tensors recorded from the REAL reference with calibrated
    weights (O(1) activations everywhere; SURVEY §8c hazard 1)."""
    sd = W.calibrated(80, seed=1)
    x = W.synthetic_input(2, 128, 1).to(G.DEV)
    eng = G.make_engine(sd, 128, 80, mode)
    raw = eng.forward_raw(x)
    torch.cuda.synchronize()
    worst = {}
    for name in TAPS:
        got = eng.read_tap(name, 2).cpu().numpy()
        for i in range(2):
            worst[name] = max(worst.get(name, 0.0), G.rel_err(got[i:i + 1], g2[f"img{i}.{name}"]))
    bad = {k: v for k, v in worst.items() if not v < LAYER_TOL[mode]}
    assert not bad, f"{mode}: layers out of tolerance {bad}"
    if mode != "tf32":
        # north_star: raw head outputs within 1e-3 absolute and 1e-4 relative
        for i, k in enumerate(("pred_s", "pred_m", "pred_l")):
            for b in range(2):
                np.testing.assert_allclose(raw[i][b:b + 1].cpu().numpy(), g2[f"img{b}.{k}"], rtol=1e-4, atol=1e-3)
    eng.close()


@pytest.mark.parametrize("mode", ["ffma", "3xtf32"])
def test_c1_config_voc320_reference_init(G, golden, mode):
    """BASELINE config C1 (320x320, VOC-20, batch 1, reference init) against the reference."""
    g1 = golden("g1_voc320_refinit.npz")
    sd = W.reference_init(20, seed=0)
    x = W.synthetic_input(1, 320, 0).to(G.DEV)
    eng = G.make_engine(sd, 320, 20, mode, max_batch=1)
    raw = eng.forward_raw(x)
    for got, k in zip(raw, ("pred_s", "pred_m", "pred_l")):
        np.testing.assert_allclose(got.cpu().numpy(), g1[k], rtol=1e-4, atol=1e-3)
    for k in ("c3", "c4", "c5"):   # collapsed activations: compare relative to their own scale
        assert G.rel_err(eng.read_tap(k, 1).cpu().numpy(), g1[k]) < 2e-5, k
    boxes, scores, cls = eng.forward_decode(x)
    assert float(np.abs(boxes[0].cpu().numpy() - g1["all_bbox"]).max()) * 320 < 1e-3    # px
    np.testing.assert_allclose(scores[0].cpu().numpy(), g1["all_score"], rtol=1e-4, atol=1e-7)
    ob, os_, oc, on = eng.forward_detect(x)
    k = int(on[0])
    # keep-set: exact w.r.t. the oracle on the engine's own candidates ...
    bh, sh, ch = boxes[0].cpu().numpy(), scores[0].cpu().numpy(), cls[0].cpu().numpy().astype(np.int64)
    b, s, c, idx = O.postprocess_flat(bh, sh, ch, 20, 0.001, 0.5)
    assert k == len(idx)
    np.testing.assert_array_equal(ob[0, :k].cpu().numpy(), b)
    # ... and against the reference's own keep-set the difference is bounded and reported:
    # reference-init scores tie by the hundreds (hazard 2) and sit 1e-8 apart, so ordering
    # flips from 1-ulp score differences are expected here; the calibrated test below is exact.
    diff = np.setxor1d(idx, g1["keep_idx"])
    print(f"[report] C1 {mode}: kept {k} vs reference {len(g1['keep_idx'])}, {len(diff)} boxes differ (ties / ulp order)")
    assert len(diff) <= 0.05 * len(g1["keep_idx"])
    eng.close()


def test_detect_matches_reference_keepset_calibrated(G, g2):
    """Tie-free weights: the full CUDA path must reproduce the reference detections:
    same kept anchors, boxes within 1e-3 px, same classes.  Pairs whose IoU is within 1e-5
    of the threshold may flip (north_star exception) — counted and reported."""
    sd = W.calibrated(80, seed=1)
    x = W.synthetic_input(2, 128, 1).to(G.DEV)
    eng = G.make_engine(sd, 128, 80, "3xtf32")
    boxes, scores, cls = eng.forward_decode(x)
    ob, os_, oc, on = eng.forward_detect(x)
    total_diff = 0
    for i in range(2):
        k = int(on[i])
        bh, sh, ch = boxes[i].cpu().numpy(), scores[i].cpu().numpy(), cls[i].cpu().numpy().astype(np.int64)
        # With O(1) activations the allowed raw-output error (1e-3 + 1e-4|t|) propagates to
        # boxes as (w/2 + stride/4) * dt, i.e. up to ~0.1 px per 100 px of box: the 1e-3 px
        # criterion is asserted where it is meaningful (decode kernel on identical inputs:
        # test_decode_level; reference-init configs: test_c1_config_*), here we bound and report.
        box_px = float(np.abs(bh - g2[f"img{i}.all_bbox"]).max()) * 128
        print(f"[report] img{i}: end-to-end box error {box_px:.4f} px (calibrated weights)")
        assert box_px < 0.15
        # score = softmax * sigmoid: its relative error is the logit error (<= ~1e-3 allowed)
        np.testing.assert_allclose(sh, g2[f"img{i}.all_score"], rtol=2e-3, atol=1e-6)
        assert (ch != g2[f"img{i}.all_cls"]).mean() < 2e-3
        _, _, _, idx = O.postprocess_flat(bh, sh, ch, 80, 0.001, 0.5)
        assert k == len(idx)
        np.testing.assert_array_equal(ob[i, :k].cpu().numpy(), bh[idx])
        np.testing.assert_array_equal(oc[i, :k].cpu().numpy(), ch[idx])
        diff = np.setxor1d(idx, g2[f"img{i}.keep_idx"])
        total_diff += len(diff)
        print(f"[report] img{i}: kept {k}, reference kept {len(g2[f'img{i}.keep_idx'])}, differing {len(diff)}")
    assert total_diff <= 4, "keep-sets differ by more than near-threshold / near-tie flips explain"
    eng.close()


def test_fused_and_unfused_weights_agree(G, g2):
    """fuse_conv_bn'd module (154 keys) through the drop-in gives the same engine weights."""
    import yolo_nano_b200 as pkg
    sd = W.calibrated(80, seed=1)
    x = W.synthetic_input(2, 128, 1).to(G.DEV)
    with contextlib.redirect_stdout(io.StringIO()):
        m = pkg.YOLONano(G.DEV, 128, 80, anchor_size=pkg.MULTI_ANCHOR_SIZE_COCO)
    m.load_state_dict(sd)
    m = m.to(G.DEV).eval()
    r1 = m(x)
    pkg.fuse_conv_bn(m)
    assert len(m.state_dict()) == 154
    r2 = m(x)
    for a, b in zip(r1, r2):
        np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(np.sort(np.unique(r1[2])), np.sort(np.unique(g2["img0.cls_inds"])))


def test_dropin_module_contract(G, golden):
    """forward(x) -> (bboxes ndarray [K,4] f32 writable, scores [K] f32, cls_inds [K] i64),
    image 0 only; set_grid between calls; K=0 shapes; CPU input raises."""
    import yolo_nano_b200 as pkg
    g1 = golden("g1_voc320_refinit.npz")
    with contextlib.redirect_stdout(io.StringIO()):
        m = pkg.YOLONano(G.DEV, 320, 20, anchor_size=pkg.MULTI_ANCHOR_SIZE)
    m.load_state_dict(W.reference_init(20, 0))
    m = m.to(G.DEV).eval()
    x = W.synthetic_input(1, 320, 0).to(G.DEV)
    b, s, c = m(torch.cat([x, torch.zeros_like(x)]))          # image 1 is ignored like the reference
    assert b.dtype == np.float32 and s.dtype == np.float32 and c.dtype == np.int64
    assert b.ndim == 2 and b.shape[1] == 4 and b.flags.writeable and b.flags.owndata
    assert abs(len(b) - len(g1["bboxes"])) <= 0.05 * len(g1["bboxes"])
    assert b.min() >= 0 and b.max() <= 1
    b -= 0.1                                                    # callers rescale in place
    m.conf_thresh = 0.9                                         # nothing survives
    b0, s0, c0 = m(x)
    assert b0.shape == (0, 4) and s0.shape == (0,) and c0.shape == (0,)
    m.conf_thresh = 0.001
    m.set_grid(160)                                             # TTA / multi-scale path
    b2, _, _ = m(W.synthetic_input(1, 160, 3).to(G.DEV))
    assert b2.shape[1] == 4
    with pytest.raises(RuntimeError):
        m(x)                                                    # 320 input on a 160 grid
    with pytest.raises(pkg.EngineError):
        m(x.cpu())
    res = m.detect(W.synthetic_input(3, 160, 4).to(G.DEV))
    assert len(res) == 3


def test_batch64_equals_per_image_and_host_path(G):
    """BASELINE config 2 shape (416x416, COCO-80, batch 64): every image of the batch gives
    bit-identical detections to running it alone (batch extension = loop the reference),
    and the host-buffer entry point returns the same rows."""
    sd = W.calibrated(80, seed=2)
    bsz = 64
    x = W.synthetic_input(bsz, 416, 2).to(G.DEV)
    eng = G.make_engine(sd, 416, 80, "3xtf32", max_batch=bsz)
    ob, os_, oc, on = [t.clone() for t in eng.forward_detect(x)]
    torch.cuda.synchronize()
    assert int(on.min()) > 0
    for i in (0, 17, 63):
        b1, s1, c1, n1 = eng.forward_detect(x[i:i + 1])
        k = int(n1[0])
        assert k == int(on[i])
        assert torch.equal(b1[0, :k], ob[i, :k]) and torch.equal(s1[0, :k], os_[i, :k]) and torch.equal(c1[0, :k], oc[i, :k])
    xh = x.cpu().pin_memory()
    hb, hs, hc, hn = eng.detect_host(xh)
    assert torch.equal(hn, on.cpu())
    for i in (0, 31, 63):
        k = int(hn[i])
        assert torch.equal(hb[i, :k], ob[i, :k].cpu()) and torch.equal(hc[i, :k], oc[i, :k].cpu())
    # double-buffered streaming API: two steps in flight, same rows
    outs = [eng.alloc_outputs(bsz, pinned_host=True) for _ in range(2)]
    xh2 = torch.flip(x, dims=[0]).cpu().pin_memory()
    eng.submit_host(0, xh, outs[0])
    eng.submit_host(1, xh2, outs[1])
    with pytest.raises(Exception):
        eng.submit_host(0, xh, outs[0])                 # slot 0 still in flight
    eng.wait_host(0)
    eng.wait_host(1)
    assert torch.equal(outs[0][3], on.cpu()) and torch.equal(outs[1][3], torch.flip(on.cpu(), dims=[0]))
    k = int(outs[1][3][0])
    assert torch.equal(outs[1][0][0, :k], ob[bsz - 1, :k].cpu())
    eng.close()


def test_g3_416_against_reference(G, golden):
    g = golden("g3_coco416_calibrated.npz")
    sd = W.calibrated(80, seed=2)
    x = W.synthetic_input(2, 416, 2).to(G.DEV)
    eng = G.make_engine(sd, 416, 80, "3xtf32")
    boxes, scores, cls = eng.forward_decode(x)
    ob, os_, oc, on = eng.forward_detect(x)
    for i in range(2):
        box_px = float(np.abs(boxes[i].cpu().numpy() - g[f"img{i}.all_bbox"]).max()) * 416
        print(f"[report] 416 img{i}: end-to-end box error {box_px:.4f} px (calibrated weights)")
        assert box_px < 0.5
        k = int(on[i])
        _, _, _, idx = O.postprocess_flat(boxes[i].cpu().numpy(), scores[i].cpu().numpy(),
                                          cls[i].cpu().numpy().astype(np.int64), 80, 0.001, 0.5)
        assert k == len(idx)
        diff = np.setxor1d(idx, g[f"img{i}.keep_idx"])
        print(f"[report] 416 img{i}: kept {k}, reference {len(g[f'img{i}.keep_idx'])}, differing {len(diff)}")
        assert len(diff) <= 0.002 * k + 2
    eng.close()


@pytest.mark.parametrize("classes,size", [(80, 128), (20, 160)])
def test_fused_decode_epilogue_equals_decode_kernel(lib, G, classes, size):
    """head_det_*.4 with the decode in the GEMM epilogue (no raw map in HBM) against the same
    conv followed by decode_level_kernel: identical raw sums feed identical arithmetic, so
    boxes and scores are bit-equal; classes may differ only where two products round equal.
    The reference is the engine's raw tail (planned with the same merged accumulator as the
    fused tail), laid out NHWC again and decoded level by level by ynb_decode_level."""
    sd = W.calibrated(classes, seed=5)
    batch = 3
    x = W.synthetic_input(batch, size, 5).to(G.DEV)
    eng = G.make_engine(sd, size, classes, "3xtf32")
    bf, sf, cf = [t.cpu().numpy() for t in eng.forward_decode(x)]
    raw = eng.forward_raw(x)
    eng.close()
    ch = 3 * (1 + classes + 4)
    ld = (ch + 3) // 4 * 4
    n = sum(3 * (size // s) ** 2 for s in (8, 16, 32))
    boxes = torch.zeros(batch, n, 4, device=G.DEV)
    scores = torch.zeros(batch, n, device=G.DEV)
    cl = torch.zeros(batch, n, device=G.DEV, dtype=torch.int32)
    anchors = np.array(W.anchors_for(classes), dtype=np.float32).reshape(3, 6)
    off = 0
    for lvl, p in enumerate(raw):
        gsz = p.shape[2]
        nhwc = torch.zeros(batch, gsz * gsz, ld, device=G.DEV)
        nhwc[..., :ch] = p.permute(0, 2, 3, 1).reshape(batch, gsz * gsz, ch)
        a = (C.c_float * 6)(*anchors[lvl].tolist())
        rc = lib.ynb_decode_level(G.ptr(nhwc), ld, G.ptr(boxes), G.ptr(scores), G.ptr(cl), batch, gsz, 8 << lvl, size,
                                  a, 3, classes, n, off, G.stream())
        assert rc == 0, lib.ynb_last_error(None)
        off += gsz * gsz * 3
    bu, su, cu = boxes.cpu().numpy(), scores.cpu().numpy(), cl.cpu().numpy()
    np.testing.assert_array_equal(bf, bu)
    np.testing.assert_array_equal(sf, su)
    assert (cf != cu).mean() < 1e-4


def test_preprocess_u8_bit_exact_and_u8_entry_equals_float_entry(G, golden):
    """SURVEY 8f row 1: Normalize + ToTensor (+ Resize padding) on the device.  (1) the tensor is
    bit-identical to the real reference's ValTransforms output (golden g4); (2) the uint8 host entry
    returns exactly the detections of the float32 host entry fed with that tensor."""
    g = golden("g4_preprocess64.npz")
    names = ("square", "landscape", "portrait")
    sd = W.calibrated(20, seed=3)
    eng = G.make_engine(sd, 64, 20, "3xtf32")
    canvas = torch.from_numpy(np.stack([g[f"{n}.canvas"] for n in names]))
    rects = torch.from_numpy(np.stack([g[f"{n}.rect"] for n in names]).astype(np.int32))
    x = eng.preprocess_u8(canvas.to(G.DEV), rects.to(G.DEV))
    ref = np.stack([g[f"{n}.tensor"] for n in names])
    np.testing.assert_array_equal(x.cpu().numpy(), ref)
    # whole canvas (no rectangle) == oracle without padding
    x2 = eng.preprocess_u8(canvas.to(G.DEV))
    np.testing.assert_array_equal(x2.cpu().numpy(), np.stack([O.preprocess_u8(g[f"{n}.canvas"]) for n in names]))
    # end to end through the host entries
    out_f = eng.alloc_outputs(3, pinned_host=True)
    out_u = eng.alloc_outputs(3, pinned_host=True)
    eng.submit_host(0, torch.from_numpy(ref).pin_memory(), out_f)
    eng.wait_host(0)
    eng.submit_host_u8(1, canvas.pin_memory(), out_u, rects.pin_memory())
    eng.wait_host(1)
    assert np.array_equal(out_f[3].numpy(), out_u[3].numpy())
    for i in range(3):
        k = int(out_f[3][i])
        for a, b in zip(out_f[:3], out_u[:3]):
            np.testing.assert_array_equal(a[i, :k].numpy(), b[i, :k].numpy())
    eng.close()


def test_dropin_detect_images_equals_detect_on_reference_tensor(G, golden):
    """Drop-in class: detect_images(uint8 canvases) == detect(the reference's ValTransforms tensor)."""
    import yolo_nano_b200 as pkg
    g = golden("g4_preprocess64.npz")
    names = ("square", "landscape", "portrait")
    with contextlib.redirect_stdout(io.StringIO()):
        m = pkg.YOLONano(G.DEV, 64, 20, anchor_size=pkg.MULTI_ANCHOR_SIZE)
    m.load_state_dict(W.calibrated(20, seed=3))
    m = m.to(G.DEV).eval()
    ref = m.detect(torch.from_numpy(np.stack([g[f"{n}.tensor"] for n in names])).to(G.DEV))
    got = m.detect_images(np.stack([g[f"{n}.canvas"] for n in names]), np.stack([g[f"{n}.rect"] for n in names]))
    for r, q in zip(ref, got):
        for a, b in zip(r, q):
            np.testing.assert_array_equal(a, b)


@pytest.mark.parametrize("size,classes,batch", [(608, 80, 2), (224, 20, 5)])
def test_detect_other_sizes_keepset_exact_on_own_candidates(G, size, classes, batch):
    """BASELINE config 3 geometry (608^2, N = 22 743 anchors) and an odd small one: the whole CUDA path
    (fused decode + anchor-grid NMS, CUDA graph on the second call) against the oracle NMS run on the
    engine's own decoded candidates, reference-init weights (every anchor is a candidate)."""
    sd = W.reference_init(classes, seed=4)
    x = W.synthetic_input(batch, size, 4).to(G.DEV)
    eng = G.make_engine(sd, size, classes, "3xtf32")
    boxes, scores, cls = eng.forward_decode(x)
    for rep in range(2):                                   # eager, then graph replay
        ob, os_, oc, on = eng.forward_detect(x)
        for i in range(batch):
            bh, sh = boxes[i].cpu().numpy(), scores[i].cpu().numpy()
            ch = cls[i].cpu().numpy().astype(np.int64)
            b, s, c, idx = O.postprocess_flat(bh, sh, ch, classes, 0.001, 0.5)
            k = int(on[i])
            assert k == len(idx)
            np.testing.assert_array_equal(ob[i, :k].cpu().numpy(), b)
            np.testing.assert_array_equal(os_[i, :k].cpu().numpy(), s)
            np.testing.assert_array_equal(oc[i, :k].cpu().numpy().astype(np.int64), c)
    eng.close()


def test_resize_bilinear_matches_interpolate_and_flip(G):
    """ynb_resize_bilinear against torch.nn.functional.interpolate(bilinear, align_corners=False) and
    torch.flip (utils/misc.py:104-121): up- and down-scaling within 2e-6, identity size bit-exact."""
    import torch.nn.functional as F
    import yolo_nano_b200 as pkg
    x = W.synthetic_input(2, 128, 8)
    for s in (96, 128, 160, 320):
        got = pkg.resize_bilinear(x.to(G.DEV), s, with_flip=True).cpu()
        ref = F.interpolate(x, size=(s, s), mode="bilinear", align_corners=False)
        for b in range(2):
            if s == 128:
                assert torch.equal(got[2 * b], x[b])
            torch.testing.assert_close(got[2 * b], ref[b], rtol=0, atol=2e-6)
            assert torch.equal(got[2 * b + 1], torch.flip(got[2 * b], [-1]))
        plain = pkg.resize_bilinear(x.to(G.DEV), s).cpu()
        assert torch.equal(plain, got[0::2])


def test_tta_driver_against_reference_driver(G, golden):
    """Drop-in TestTimeAugmentation (3 scales x flip through the engine, merge NMS on the device) against
    the real reference driver's recorded result.  The merge NMS is exact on its inputs; the per-scale
    detections carry the network tolerance, so boxes are matched by label within 0.3 px."""
    import yolo_nano_b200 as pkg
    g = golden("g5_tta128_calibrated.npz")
    with contextlib.redirect_stdout(io.StringIO()):
        m = pkg.YOLONano(G.DEV, 128, 20, anchor_size=pkg.MULTI_ANCHOR_SIZE)
    m.load_state_dict(W.calibrated(20, seed=6))
    m = m.to(G.DEV).eval()
    x = W.synthetic_input(1, 128, 6).to(G.DEV)
    tta = pkg.TestTimeAugmentation(num_classes=20, nms_thresh=0.4, scale_range=[96, 160, 32])
    b, s, c = tta(x, m)
    # (a) the merge step alone is exact: ynb_nms on the union == oracle merge on the same union
    from yolo_nano_b200.tta import merge_nms
    rng = np.random.default_rng(0)
    ub = np.concatenate([g["bboxes"], np.clip(g["bboxes"] + rng.normal(0, 0.01, g["bboxes"].shape), 0, 1)]).astype(np.float32)
    us = np.concatenate([g["scores"], g["scores"] * np.float32(0.9)]).astype(np.float32)
    ul = np.concatenate([g["labels"], g["labels"]])
    mb, ms, ml = merge_nms(ub, us, ul, 20, 0.4, G.DEV)
    ob, os_, ol = O.tta_merge(ub, us, ul, 20, 0.4)
    np.testing.assert_array_equal(mb, ob)
    np.testing.assert_array_equal(ms, os_)
    np.testing.assert_array_equal(ml, ol)
    # (b) end to end against the reference driver
    gb, gl = g["bboxes"], g["labels"]
    print(f"[report] TTA: kept {len(b)} vs reference {len(gb)}")
    assert abs(len(b) - len(gb)) <= 0.01 * len(gb) + 2
    unmatched = 0
    for k in range(len(gb)):
        cand = np.nonzero(c == gl[k])[0]
        d = np.abs(b[cand] - gb[k]).max(axis=1).min() * 128 if len(cand) else 1e9
        unmatched += d > 0.3
    print(f"[report] TTA: {unmatched} of {len(gb)} reference boxes without a match within 0.3 px")
    assert unmatched <= 0.01 * len(gb) + 2


def test_detect_is_deterministic_and_batch_independent(G):
    """The NMS build appends suppressor-list entries with atomics (arbitrary order); the result must not
    depend on it: two runs of a 16-image batch are bit-identical, and image i of the batch equals the
    same image run alone (the defined batch semantics, SURVEY 8c hazard 4)."""
    sd = W.reference_init(80, seed=3)
    x = W.synthetic_input(16, 416, 11).to(G.DEV)
    eng = G.make_engine(sd, 416, 80, "3xtf32", max_batch=16)
    a = [t.clone() for t in eng.forward_detect(x)]
    b = [t.clone() for t in eng.forward_detect(x)]
    c = [t.clone() for t in eng.forward_detect(x)]          # third call: CUDA-graph replay
    assert torch.equal(a[3], b[3]) and torch.equal(a[3], c[3])
    for i in range(16):                      # rows beyond an image's count are never written: compare the valid ones
        k = int(a[3][i])
        for u, v, w_ in zip(a[:3], b[:3], c[:3]):
            assert torch.equal(u[i, :k], v[i, :k]) and torch.equal(u[i, :k], w_[i, :k])
    for i in (0, 7, 15):
        one = eng.forward_detect(x[i:i + 1].contiguous())
        k = int(one[3][0])
        assert k == int(a[3][i])
        for u, v in zip(one[:3], a[:3]):
            assert torch.equal(u[0, :k], v[i, :k])
    eng.close()


def test_raw_outputs_at_baseline_size_calibrated_reported(G):
    """north_star bar at the BASELINE size with O(1) activations (416^2, COCO-80, calibrated weights): raw
    head outputs against the fp32 oracle and against an fp64 evaluation of the same network.  Measured:
    fp32 re-association noise alone uses 0.6-0.9 of the tolerance here (our fp32 FFMA mode and the oneDNN
    oracle are equally far from fp64); 3xTF32 is ~2x that, so a few outputs per million exceed
    1e-3 + 1e-4|ref| (reported, bounded) — at 128^2 and on the reference-init benchmark weights: none."""
    sd = W.calibrated(80, seed=12)
    x = W.synthetic_input(1, 416, 12)
    ref32 = [t.numpy() for t in O.network(sd, x)]
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
    ref64 = [t.numpy() for t in O.network(sd64, x.double())]

    def worst(a, b):
        w, v, n = 0.0, 0, 0
        for r, g in zip(a, b):
            err = np.abs(g - r)
            tol = 1e-3 + 1e-4 * np.abs(r)
            w = max(w, float((err / tol).max())); v += int((err > tol).sum()); n += err.size
        return w, v, n

    res = {}
    for mode in ("ffma", "3xtf32"):
        eng = G.make_engine(sd, 416, 80, mode)
        got = [t.cpu().numpy() for t in eng.forward_raw(x.to(G.DEV))]
        eng.close()
        res[mode] = (worst(ref32, got), worst(ref64, got))
    o64 = worst(ref64, ref32)
    for mode, (a, b) in res.items():
        print(f"[report] 416 calibrated {mode}: vs fp32 oracle {a[0]:.2f} tol ({a[1]} of {a[2]} over); "
              f"vs fp64 {b[0]:.2f} tol ({b[1]} over); fp32 oracle vs fp64 {o64[0]:.2f} tol")
    assert res["ffma"][0][1] == 0                                  # true fp32: inside the bar
    w, v, n = res["3xtf32"][0]
    assert v <= 5e-5 * n and w < 2.0                               # parity mode: a few per 100 k, < 2x tol


def test_bench_workload_network_parity_416_refinit(G, golden):
    """The bench's exact workload (416^2, COCO-80, reference init seed 3): raw head maps and stage taps
    against the oracle network, decoded candidates against the REAL reference's recorded ones (golden g3),
    keep-sets against the reference's with the tie-dependent differences counted."""
    g3 = golden("g3_coco416_refinit.npz")
    seed = int(g3["seed"])
    sd = W.reference_init(80, seed=seed)
    x = W.synthetic_input(2, 416, seed)
    assert W.digest(sd) == str(g3["sd_digest"]) and W.digest(x) == str(g3["x_digest"])
    taps = {}
    ref = O.network(sd, x, taps=taps)
    eng = G.make_engine(sd, 416, 80, "3xtf32")
    raw = eng.forward_raw(x.to(G.DEV))
    for got, want in zip(raw, ref):                       # north_star: 1e-3 absolute + 1e-4 relative
        np.testing.assert_allclose(got.cpu().numpy(), want.numpy(), rtol=1e-4, atol=1e-3)
    for name in TAPS:                                     # collapsed activations: relative to each layer's own scale
        assert G.rel_err(eng.read_tap(name, 2).cpu().numpy(), taps[name].numpy()) < 1e-4, name
    boxes, scores, cls = eng.forward_decode(x.to(G.DEV))
    ob, os_, oc, on = eng.forward_detect(x.to(G.DEV))
    for i in range(2):
        assert float(np.abs(boxes[i].cpu().numpy() - g3[f"img{i}.all_bbox"]).max()) * 416 < 1e-3     # px
        np.testing.assert_allclose(scores[i].cpu().numpy(), g3[f"img{i}.all_score"], rtol=1e-4, atol=1e-7)
        bh, sh, ch = boxes[i].cpu().numpy(), scores[i].cpu().numpy(), cls[i].cpu().numpy().astype(np.int64)
        _, _, _, idx = O.postprocess_flat(bh, sh, ch, 80, 0.001, 0.5)
        k = int(on[i])
        assert k == len(idx)
        np.testing.assert_array_equal(ob[i, :k].cpu().numpy(), bh[idx])
        diff = np.setxor1d(idx, g3[f"img{i}.keep_idx"])
        print(f"[report] bench workload img{i}: kept {k} vs reference {len(g3[f'img{i}.keep_idx'])}, "
              f"{len(diff)} differ (exact score ties / 1-ulp order)")
        assert len(diff) <= 0.05 * len(g3[f"img{i}.keep_idx"])
    eng.close()


@pytest.mark.parametrize("weights", ["refinit", "calibrated"])
def test_network_parity_608(G, weights):
    """BASELINE configs[2] size (608^2, COCO-80): every stage tap and the raw head maps against the oracle.
    Reference init: inside the north_star bar; calibrated (O(1) activations in all 45 layers): per-layer 1e-4 of
    the layer's scale, raw maps bounded as at 416^2 (see test_raw_outputs_at_baseline_size_calibrated_reported)."""
    sd = W.reference_init(80, seed=4) if weights == "refinit" else W.calibrated(80, seed=4)
    x = W.synthetic_input(2, 608, 4)
    taps = {}
    ref = O.network(sd, x, taps=taps)
    eng = G.make_engine(sd, 608, 80, "3xtf32")
    raw = eng.forward_raw(x.to(G.DEV))
    for name in TAPS:
        assert G.rel_err(eng.read_tap(name, 2).cpu().numpy(), taps[name].numpy()) < 1e-4, name
    over = n = 0
    worst = 0.0
    for got, want in zip(raw, ref):
        err = np.abs(got.cpu().numpy() - want.numpy())
        tol = 1e-3 + 1e-4 * np.abs(want.numpy())
        over += int((err > tol).sum()); n += err.size; worst = max(worst, float((err / tol).max()))
    print(f"[report] 608 {weights}: worst raw error {worst:.2f} tol, {over} of {n} outputs over")
    if weights == "refinit":
        assert over == 0
    else:
        assert over <= 5e-5 * n and worst < 2.0
    eng.close()


def test_two_grid_sizes_through_one_device_buffer(G):
    """set_grid between forwards with the input living at the SAME device address and the same batch (what
    torch's caching allocator produces in the TTA scale loop / multi-scale eval): the stem's input tensor map
    must follow the size (advisor finding: the map cache was keyed by pointer and batch only)."""
    sd = W.calibrated(20, seed=2)
    eng = G.make_engine(sd, 128, 20, "3xtf32")
    buf = torch.empty(2 * 3 * 192 * 192, device=G.DEV)
    for size in (128, 192, 128, 160):
        x = W.synthetic_input(2, size, size)
        xd = buf[: x.numel()].view(2, 3, size, size)
        xd.copy_(x)
        eng.set_grid(size)
        for _ in range(3):                                   # eager, capture, graph replay
            raw = eng.forward_raw(xd)
            ob, os_, oc, on = eng.forward_detect(xd)
        ref = O.network(sd, x)
        for got, want in zip(raw, ref):
            np.testing.assert_allclose(got.cpu().numpy(), want.numpy(), rtol=1e-4, atol=1e-3)
        boxes, scores, cls = eng.forward_decode(xd)
        for i in range(2):
            bh, sh, ch = boxes[i].cpu().numpy(), scores[i].cpu().numpy(), cls[i].cpu().numpy().astype(np.int64)
            _, _, _, idx = O.postprocess_flat(bh, sh, ch, 20, 0.001, 0.5)
            assert int(on[i]) == len(idx)
            np.testing.assert_array_equal(ob[i, : len(idx)].cpu().numpy(), bh[idx])
    eng.close()


def test_host_entries_reject_buffers_of_another_grid_size(G):
    """The host entry points copy 3*S*S*batch elements using the engine's current grid: a buffer built for another
    size is an error, not an out-of-bounds read (advisor finding)."""
    from yolo_nano_b200.engine import EngineError
    sd = W.calibrated(20, seed=2)
    eng = G.make_engine(sd, 128, 20, "3xtf32")
    out = eng.alloc_outputs(1, pinned_host=True)
    with pytest.raises(EngineError):
        eng.submit_host(0, torch.zeros(1, 3, 96, 96).pin_memory(), out)
    with pytest.raises(EngineError):
        eng.submit_host_u8(0, torch.zeros(1, 96, 96, 3, dtype=torch.uint8).pin_memory(), out)
    with pytest.raises(EngineError):
        eng.detect_host(torch.zeros(1, 3, 160, 160))
    with pytest.raises(EngineError):
        eng.preprocess_u8(torch.zeros(1, 96, 96, 3, dtype=torch.uint8, device=G.DEV))
    eng.set_grid(96)
    eng.submit_host(0, torch.zeros(1, 3, 96, 96).pin_memory(), out)
    eng.wait_host(0)
    eng.close()


def test_bf16_mode_tolerance_reported(G, g2):
    """BASELINE configs[3] throughput mode (YNB_GEMM_TC_BF16): bf16 activations and weights in HBM, kind::f16 tensor
    cores, fp32 accumulation / bias / activation / depthwise taps.  Reported separately from the fp32 parity mode, with
    its tolerance stated here, against the REAL reference's tensors on the calibrated weights — the WORST case for a
    storage format: an untrained random network amplifies every rounding through its 45 layers (single-pass TF32,
    2^-11 per operand, already reaches 0.15-0.3 of the layer scale at the deepest taps: LAYER_TOL above; bf16 rounds
    at 2^-9).  Stated tolerance: one kernel <= 2e-2 of the layer scale in max norm (the stage-2 taps, 1-4 kernels
    deep, measure it); after 45 layers <= 0.6 in max norm and <= 0.35 in RMS (measured 0.41 / 0.29).  On the reference-init BASELINE
    weights the head maps are within 2e-2 absolute (next test).  The NMS stage stays exact on its inputs."""
    sd = W.calibrated(80, seed=1)
    x = W.synthetic_input(2, 128, 1).to(G.DEV)
    eng = G.make_engine(sd, 128, 80, "bf16")
    eng.forward_raw(x)
    torch.cuda.synchronize()
    worst, rms = {}, {}
    for name in TAPS:
        got = eng.read_tap(name, 2).cpu().numpy().astype(np.float64)
        want = np.concatenate([g2[f"img{i}.{name}"] for i in range(2)]).astype(np.float64)
        worst[name] = float(np.abs(got - want).max() / np.abs(want).max())
        rms[name] = float(np.sqrt(((got - want) ** 2).mean()) / np.sqrt((want ** 2).mean()))
    print("[report] bf16 per-layer max error / layer scale:", {k: round(v, 4) for k, v in worst.items()})
    print("[report] bf16 per-layer rms error / layer rms:", {k: round(v, 4) for k, v in rms.items()})
    assert all(worst[k] < 2e-2 for k in ("pool", "stage2.0", "stage2.1", "stage2.2", "stage2.3", "lat3")), worst
    assert max(worst.values()) < 0.6 and max(rms.values()) < 0.35, (worst, rms)
    boxes, scores, cls = eng.forward_decode(x)
    ob, os_, oc, on = eng.forward_detect(x)
    for i in range(2):
        bh, sh, ch = boxes[i].cpu().numpy(), scores[i].cpu().numpy(), cls[i].cpu().numpy().astype(np.int64)
        box_px = float(np.median(np.abs(bh - g2[f"img{i}.all_bbox"]).max(axis=1))) * 128
        cls_flip = float((ch != g2[f"img{i}.all_cls"]).mean())
        _, _, _, idx = O.postprocess_flat(bh, sh, ch, 80, 0.001, 0.5)
        k = int(on[i])
        assert k == len(idx)                                                   # NMS itself stays exact on its inputs
        np.testing.assert_array_equal(ob[i, :k].cpu().numpy(), bh[idx])
        ref_idx = g2[f"img{i}.keep_idx"]
        diff = len(np.setxor1d(idx, ref_idx))
        print(f"[report] bf16 img{i} (calibrated, worst case): median box error {box_px:.3f} px, class flips "
              f"{cls_flip:.4f}, kept {k} vs reference {len(ref_idx)}, {diff} boxes differ")
    eng.close()


@pytest.mark.parametrize("size,classes", [(416, 80), (320, 20)])
def test_bf16_mode_reference_init_workloads(G, size, classes):
    """bf16 mode on the BASELINE weights (reference init) at configs[3]'s size and at C1's: raw head maps against the
    fp32 oracle — tolerance 2e-2 absolute (the maps are O(1) logits dominated by the biases) —, detections run."""
    sd = W.reference_init(classes, seed=3)
    x = W.synthetic_input(2, size, 5)
    ref = O.network(sd, x)
    eng = G.make_engine(sd, size, classes, "bf16")
    raw = eng.forward_raw(x.to(G.DEV))
    worst = max(float(np.abs(g.cpu().numpy() - r.numpy()).max()) for g, r in zip(raw, ref))
    print(f"[report] bf16 {size}/{classes} reference init: worst raw head error {worst:.5f}")
    assert worst < 2e-2
    ob, os_, oc, on = eng.forward_detect(x.to(G.DEV))
    assert int(on.min()) > 0
    eng.close()


def test_letterbox_preprocess_on_device_bit_identical(G, golden):
    """SURVEY §8f row 1, the whole ValTransforms on the device: original uint8 images of assorted shapes (square,
    no-resize, exact 2x downscale, up-scaling, extreme aspect ratios) -> the float32 tensor of the REAL reference
    transform (golden g9: cv2.resize inside), bit for bit; and the evaluators' inverse box mapping on the device."""
    g9 = golden("g9_letterbox96.npz")
    size, n = int(g9["size"]), int(g9["n"])
    sd = W.calibrated(20, seed=2)
    eng = G.make_engine(sd, size, 20, "3xtf32", max_batch=n)
    imgs = [g9[f"img{i}"] for i in range(n)]
    x, maps = eng.preprocess_images(imgs)
    for i in range(n):
        np.testing.assert_array_equal(x[i].cpu().numpy(), g9[f"x{i}"], err_msg=f"image {i} {imgs[i].shape}")
    boxes = torch.from_numpy(np.stack([g9[f"boxes{i}"] for i in range(n)])).to(G.DEV).contiguous()
    counts = torch.tensor([7, 5, 7, 0, 7, 3, 7, 7, 1, 7], dtype=torch.int32, device=G.DEV)
    eng.map_boxes(boxes, counts, maps)
    for i in range(n):
        k = int(counts[i])
        np.testing.assert_array_equal(boxes[i, :k].cpu().numpy(), g9[f"mapped{i}"][:k])
        np.testing.assert_array_equal(boxes[i, k:].cpu().numpy(), g9[f"boxes{i}"][k:])      # rows past the count untouched
    eng.close()


def test_detect_raw_images_equals_reference_evaluator_loop(G, golden):
    """Drop-in: detect_raw_images(list of original images) == for each image: ValTransforms -> model -> inverse mapping
    (evaluator/cocoapi_evaluator.py:70-87), with the oracle transform (pinned to the real one by g9) as the host side."""
    import yolo_nano_b200 as pkg
    g9 = golden("g9_letterbox96.npz")
    size = int(g9["size"])
    sd = W.calibrated(20, seed=2)
    with contextlib.redirect_stdout(io.StringIO()):
        m = pkg.YOLONano(G.DEV, size, 20, anchor_size=W.anchors_for(20))
    m.load_state_dict(sd)
    m = m.to(G.DEV).eval()
    imgs = [g9[f"img{i}"] for i in (3, 4, 5, 9)]
    got = m.detect_raw_images(imgs)
    for im, (gb, gs, gc) in zip(imgs, got):
        x, scale, offset = O.val_transform(im, size)
        b, s, c = m(torch.from_numpy(x)[None].to(G.DEV))
        want = O.map_boxes_to_image(b, scale, offset, im.shape[1], im.shape[0])
        np.testing.assert_array_equal(gb, want)
        np.testing.assert_array_equal(gs, s)
        np.testing.assert_array_equal(gc, c)


@pytest.mark.parametrize("size,batch", [(96, 1), (160, 3), (224, 2), (352, 1), (512, 2), (640, 1)])
def test_odd_grid_sizes_and_batches(G, size, batch):
    """Grid sizes whose feature maps are not multiples of the kernels' tiles (12, 20, 28, 44, 64, 80 at stride 8: partial
    32x4 / 16x8 tiles of the fused unit tails, partial GEMM tiles, odd batches): raw head maps and stage outputs against
    the oracle in the fp32 parity mode, the head maps in bf16 mode within its stated tolerance, NMS exact on the
    engine's own candidates."""
    sd = W.reference_init(20, seed=size)
    x = W.synthetic_input(batch, size, size)
    taps = {}
    ref = O.network(sd, x, taps=taps)
    eng = G.make_engine(sd, size, 20, "3xtf32", max_batch=batch)
    raw = eng.forward_raw(x.to(G.DEV))
    for got, want in zip(raw, ref):
        np.testing.assert_allclose(got.cpu().numpy(), want.numpy(), rtol=1e-4, atol=1e-3)
    for name in ("c3", "c4", "c5", "p3", "p4", "p5"):
        assert G.rel_err(eng.read_tap(name, batch).cpu().numpy(), taps[name].numpy()) < 1e-4, name
    boxes, scores, cls = eng.forward_decode(x.to(G.DEV))
    ob, os_, oc, on = eng.forward_detect(x.to(G.DEV))
    for i in range(batch):
        bh, sh, ch = boxes[i].cpu().numpy(), scores[i].cpu().numpy(), cls[i].cpu().numpy().astype(np.int64)
        _, _, _, idx = O.postprocess_flat(bh, sh, ch, 20, 0.001, 0.5)
        assert int(on[i]) == len(idx)
        np.testing.assert_array_equal(ob[i, : len(idx)].cpu().numpy(), bh[idx])
    eng.close()
    engb = G.make_engine(sd, size, 20, "bf16", max_batch=batch)
    rawb = engb.forward_raw(x.to(G.DEV))
    worst = max(float(np.abs(g.cpu().numpy() - r.numpy()).max()) for g, r in zip(rawb, ref))
    assert worst < 2e-2, worst
    engb.close()


@pytest.mark.parametrize("size,batch,mode", [(416, 256, "3xtf32"), (608, 256, "3xtf32"), (416, 256, "bf16")])
def test_full_size_workloads_size_independent_properties(G, size, batch, mode):
    """BASELINE's full sizes (416^2 x 256 = the metric's workload, 608^2 x 256 = configs[2], bf16 = one GPU's share of
    configs[3] x 2), where the oracle would need minutes: properties that do not depend on the size —
      * batch independence / permutation: the batch is 8 distinct images tiled 32 times in a shuffled order; every copy
        of an image must give the bit-identical detections, wherever it sits in the batch;
      * the same images run as a batch of 8 give the same detections (batch-size independence);
      * determinism: a second run (CUDA-graph replay) is bit-identical;
      * NMS idempotence: the kept boxes of an image, fed through the per-class NMS again, are all kept (a keep set is
        a fixed point of greedy NMS), in the same order;
      * every kept score >= conf_thresh, every box inside the unit square, classes in range."""
    from yolo_nano_b200.tta import merge_nms
    classes = 80
    sd = W.reference_init(classes, seed=5)
    base = W.synthetic_input(8, size, 21)
    perm = torch.randperm(batch, generator=torch.Generator().manual_seed(1))
    idx = (torch.arange(batch) % 8)[perm]
    x = base[idx].contiguous().to(G.DEV)
    eng = G.make_engine(sd, size, classes, mode, max_batch=batch)
    a = [t.clone() for t in eng.forward_detect(x)]
    b = [t.clone() for t in eng.forward_detect(x)]
    assert torch.equal(a[3], b[3])
    kmax = int(a[3].max())
    valid = torch.arange(kmax, device=G.DEV)[None, :] < a[3][:, None]      # rows beyond an image's count are not written
    for u, v in zip(a[:3], b[:3]):
        m = valid if u.dim() == 2 else valid[..., None]
        assert torch.equal(torch.where(m, u[:, :kmax], torch.zeros_like(u[:, :kmax])),
                           torch.where(m, v[:, :kmax], torch.zeros_like(v[:, :kmax])))
    boxes, scores, cls, counts = a
    small = eng.forward_detect(base.to(G.DEV))
    first = {}
    for pos in range(batch):
        img = int(idx[pos])
        k = int(counts[pos])
        assert k == int(small[3][img]) and k > 0
        for u, v in zip((boxes, scores, cls), small[:3]):
            assert torch.equal(u[pos, :k], v[img, :k]), (pos, img)
        first.setdefault(img, pos)
    conf = 0.001
    for img, pos in first.items():
        k = int(counts[pos])
        bb, ss, cc = boxes[pos, :k].cpu().numpy(), scores[pos, :k].cpu().numpy(), cls[pos, :k].cpu().numpy()
        assert (ss >= conf).all() and (bb >= 0).all() and (bb <= 1).all() and (cc >= 0).all() and (cc < classes).all()
        if img < 2:
            kb, ks, kc = merge_nms(bb, ss, cc.astype(np.int32), classes, 0.5, G.DEV)
            assert len(ks) == k and np.array_equal(kb, bb) and np.array_equal(ks, ss) and np.array_equal(kc, cc.astype(np.int64))
    eng.close()
