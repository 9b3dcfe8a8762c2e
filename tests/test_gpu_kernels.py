"""Unit parity of the individually callable kernels, through the C ABI, on a real B200."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from oracle import weights as W  # noqa: E402
from oracle import yolo_nano_oracle as O  # noqa: E402


@pytest.fixture(scope="module")
def G():
    import gpu_util
    return gpu_util


def _nhwc(t):
    return t.permute(0, 2, 3, 1).contiguous()


@pytest.mark.parametrize("batch,ch,hw,stride,act", [
    (1, 58, 52, 1, 0), (64, 58, 52, 1, 0),      # backbone.stage2.1.branch2.3 (SURVEY §7.2)
    (1, 58, 104, 2, 0), (8, 58, 104, 2, 0),     # backbone.stage2.0.branch2.3
    (2, 116, 26, 1, 0), (2, 232, 13, 1, 0), (2, 24, 104, 2, 0),
    (2, 96, 13, 1, 2), (2, 96, 52, 1, 2),       # head depthwise + LeakyReLU
    (1, 4, 1, 1, 0), (1, 4, 3, 2, 1),           # degenerate maps
])
def test_dwconv3x3(lib, G, batch, ch, hw, stride, act):
    torch.manual_seed(ch * 7 + hw + stride)
    c4 = (ch + 3) // 4 * 4
    x = torch.randn(batch, ch, hw, hw)
    w = torch.randn(ch, 1, 3, 3)
    b = torch.randn(ch)
    ref = F.conv2d(x, w, b, stride, 1, 1, ch)
    ref = F.relu(ref) if act == 1 else (F.leaky_relu(ref, 0.1) if act == 2 else ref)
    xin = torch.zeros(batch, hw, hw, c4)
    xin[..., :ch] = _nhwc(x)
    wp = torch.zeros(9, c4)
    wp[:, :ch] = w.view(ch, 9).t()
    bp = torch.zeros(c4)
    bp[:ch] = b
    ho = ref.shape[2]
    xin, wp, bp = xin.to(G.DEV), wp.to(G.DEV), bp.to(G.DEV)
    out = torch.full((batch, ho, ho, c4), float("nan"), device=G.DEV)
    rc = lib.ynb_dwconv3x3(G.ptr(xin), c4, 0, G.ptr(out), c4, 0, 1, G.ptr(wp), G.ptr(bp),
                           batch, hw, hw, c4, stride, act, G.stream())
    assert rc == 0, lib.ynb_last_error(None)
    got = out.cpu()[..., :ch].permute(0, 3, 1, 2)
    torch.testing.assert_close(got, ref, rtol=1e-5, atol=1e-5)
    if c4 != ch:
        assert float(out[..., ch:].abs().max()) == 0.0     # channel pads stay zero


SHAPES = [(1000, 24, 58), (4321, 60, 58), (5408, 116, 116), (700, 232, 232), (338, 464, 96),
          (5408, 96, 255), (128, 32, 16), (129, 96, 96), (1, 24, 58), (64 * 2704, 60, 58)]


def _pw_problem(G, m, cin, cout, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(m, cin, generator=g).to(G.DEV)
    w = (torch.randn(cout, cin, generator=g) / cin ** 0.5).to(G.DEV)
    b = torch.randn(cout, generator=g).to(G.DEV)
    ref = (x.double() @ w.double().t() + b.double())
    return x, w, b, ref


@pytest.mark.parametrize("m,cin,cout", SHAPES)
def test_pwconv_ffma(lib, G, m, cin, cout):
    x, w, b, ref = _pw_problem(G, m, cin, cout, m + cin)
    ld = (cout + 3) // 4 * 4
    out = torch.full((m, ld), float("nan"), device=G.DEV)
    rc = lib.ynb_pwconv(G.ptr(x), cin, 0, G.ptr(out), ld, 0, 1, G.ptr(w), G.ptr(b), m, cin, cout, 1, G.stream())
    assert rc == 0, lib.ynb_last_error(None)
    torch.testing.assert_close(out[:, :cout].double(), ref.clamp_min(0), rtol=1e-5, atol=2e-5)


@pytest.mark.parametrize("mode,tol", [(1, 2e-5), (2, 2e-2)])
@pytest.mark.parametrize("m,cin,cout", SHAPES)
def test_pwconv_tcgen05(lib, G, m, cin, cout, mode, tol):
    """tcgen05 path: 3xTF32 must be fp32-grade (tolerance as the FFMA kernel), single-pass
    TF32 is the throughput mode with its own (looser) tolerance."""
    x, w, b, ref = _pw_problem(G, m, cin, cout, m + cin)
    ld = (cout + 3) // 4 * 4
    out = torch.full((m, ld), float("nan"), device=G.DEV)
    rc = lib.ynb_pwconv_tc(G.ptr(x), cin, 0, G.ptr(out), ld, 0, 1, G.ptr(w), G.ptr(b), m, cin, cout, 2, mode,
                           G.stream())
    assert rc == 0, lib.ynb_last_error(None)
    torch.cuda.synchronize()
    want = F.leaky_relu(ref, 0.1)
    torch.testing.assert_close(out[:, :cout].double(), want, rtol=tol, atol=tol)


def test_pwconv_strided_views(lib, G):
    """Channel sub-range in, interleaved slots out: chunk / cat / channel_shuffle as views."""
    m, c, h = 3000, 232, 116
    g = torch.Generator().manual_seed(3)
    xfull = torch.randn(m, c, generator=g).to(G.DEV)
    w = (torch.randn(h, h, generator=g) / h ** 0.5).to(G.DEV)
    b = torch.randn(h, generator=g).to(G.DEV)
    ref = torch.relu(xfull[:, h:].double() @ w.double().t() + b.double())
    for fn, extra in ((lib.ynb_pwconv, ()), (lib.ynb_pwconv_tc, (1,))):
        out = torch.zeros(m, c, device=G.DEV)
        rc = fn(G.ptr(xfull), c, h, G.ptr(out), c, 1, 2, G.ptr(w), G.ptr(b), m, h, h, 1, *extra, G.stream())
        assert rc == 0, lib.ynb_last_error(None)
        torch.cuda.synchronize()
        torch.testing.assert_close(out[:, 1::2].double(), ref, rtol=2e-5, atol=2e-5)
        assert float(out[:, 0::2].abs().max()) == 0.0


@pytest.mark.parametrize("mode,tol", [(1, 3e-5), (2, 2e-2), (3, 4e-3)])
@pytest.mark.parametrize("batch,h,w,c,cout,dw_act,with_pass", [
    (2, 52, 52, 60, 58, 0, True),      # stage-2 stride-1 unit tail (58 channels stored with ld 60)
    (3, 26, 26, 116, 116, 0, True),    # stage 3: streamed weight chunks
    (2, 13, 13, 116, 116, 0, True),    # one partial tile per image
    (1, 40, 40, 60, 58, 0, True),      # 320^2 input
    (2, 52, 52, 96, 96, 2, False),     # detection-head pair (LeakyReLU after the depthwise conv too)
    (5, 19, 19, 96, 96, 2, False),     # 608^2 level 5
    (1, 7, 9, 32, 16, 1, False),       # tiny non-square map, ReLU in between
])
def test_fused_dw_pw_unit_tail(lib, G, batch, h, w, c, cout, dw_act, with_pass, mode, tol):
    """dwpw_tc_kernel = depthwise 3x3 + bias (+act) -> pointwise + bias + act (+ cat/channel_shuffle with the
    pass-through half) in one launch, against torch (backbone/shufflenetv2.py:57-63,70-76; models/yolo_nano.py:50-58).
    bf16 mode (3): in / out / pass are bf16 with channels and ld multiples of 8; the float64 reference rounds what the
    kernel rounds (pointwise weights and the depthwise output, RNE), so the tolerance is the output's own rounding."""
    bf = mode == 3
    rnd = (lambda t: t.to(torch.bfloat16).double()) if bf else (lambda t: t)
    al = 8 if bf else 4
    up = lambda v: (v + al - 1) // al * al
    g = torch.Generator().manual_seed(h * 131 + c)
    creal = min(c, 58) if c == 60 else c                      # physical pads (58 -> 60, bf16: -> 64) carry zeros
    c = up(c)
    x = torch.zeros(batch, h, w, c)
    x[..., :creal] = torch.randn(batch, h, w, creal, generator=g)
    dw_w = torch.zeros(c, 3, 3)
    dw_w[:creal] = torch.randn(creal, 3, 3, generator=g) / 3
    dw_b = torch.zeros(c)
    dw_b[:creal] = torch.randn(creal, generator=g) * 0.2
    pw_w = torch.zeros(cout, c)
    pw_w[:, :creal] = torch.randn(cout, creal, generator=g) / creal ** 0.5
    pw_b = torch.randn(cout, generator=g) * 0.3
    act = 2 if dw_act == 2 else 1
    f = {0: lambda t: t, 1: torch.relu, 2: lambda t: F.leaky_relu(t, 0.1)}
    xn = rnd(x.permute(0, 3, 1, 2).double())
    mid = rnd(f[dw_act](F.conv2d(xn, dw_w.double().unsqueeze(1), dw_b.double(), 1, 1, groups=c)))
    ref = f[act](F.conv2d(mid, rnd(pw_w.double())[:, :, None, None], pw_b.double())).permute(0, 2, 3, 1)
    et = torch.bfloat16 if bf else torch.float32
    xd = x.to(G.DEV, et)
    dwp = dw_w.reshape(c, 9).t().contiguous().to(G.DEV)      # [9][C] tap-major
    dbd, pwd, pbd = dw_b.to(G.DEV), pw_w.contiguous().to(G.DEV), pw_b.to(G.DEV)
    if with_pass:
        ld = up(2 * cout) + al
        pld = up(cout) + al                                                    # pass rows are read 16 bytes at a time
        x1 = torch.randn(batch, h, w, pld, generator=g).to(G.DEV, et)
        out = torch.full((batch, h, w, ld), float("nan"), device=G.DEV, dtype=et)
        rc = lib.ynb_dwpw_tc(G.ptr(xd), c, G.ptr(dwp), G.ptr(dbd), dw_act, G.ptr(pwd), G.ptr(pbd), act, G.ptr(out), ld,
                             G.ptr(x1), pld, batch, h, w, c, cout, mode, G.stream())
        assert rc == 0, lib.ynb_last_error(None)
        torch.cuda.synchronize()
        assert torch.equal(out[..., 0:2 * cout:2], x1[..., :cout])           # pass-through half, bit for bit
        torch.testing.assert_close(out[..., 1:2 * cout:2].double().cpu(), ref, rtol=tol, atol=tol)
        # nothing written past the unit's channels (bf16: past its last 16-byte chunk, round_up(2 * cout, 8))
        assert bool(torch.isnan(out[..., up(2 * cout):]).all())
    else:
        ld = up(cout) + al
        out = torch.full((batch, h, w, ld), float("nan"), device=G.DEV, dtype=et)
        rc = lib.ynb_dwpw_tc(G.ptr(xd), c, G.ptr(dwp), G.ptr(dbd), dw_act, G.ptr(pwd), G.ptr(pbd), act, G.ptr(out), ld,
                             None, 0, batch, h, w, c, cout, mode, G.stream())
        assert rc == 0, lib.ynb_last_error(None)
        torch.cuda.synchronize()
        torch.testing.assert_close(out[..., :cout].double().cpu(), ref, rtol=tol, atol=tol)
        assert bool(torch.isnan(out[..., cout:]).all())


@pytest.mark.parametrize("batch,size", [(1, 64), (2, 128), (1, 320), (2, 416)])
def test_stem_pool(lib, G, batch, size):
    g = torch.Generator().manual_seed(size)
    x = torch.randn(batch, 3, size, size, generator=g)
    w = torch.randn(24, 3, 3, 3, generator=g) / 3
    b = torch.randn(24, generator=g) * 0.1
    ref = F.max_pool2d(F.relu(F.conv2d(x, w, b, 2, 1)), 3, 2, 1)
    wp = w.permute(1, 2, 3, 0).reshape(27, 24).contiguous().to(G.DEV)
    out = torch.full((batch, size // 4, size // 4, 24), float("nan"), device=G.DEV)
    xd, bd = x.to(G.DEV), b.to(G.DEV)
    rc = lib.ynb_stem_pool(G.ptr(xd), G.ptr(out), G.ptr(wp), G.ptr(bd), batch, size, G.stream())
    assert rc == 0, lib.ynb_last_error(None)
    torch.testing.assert_close(out.cpu().permute(0, 3, 1, 2), ref, rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("classes,size", [(20, 320), (80, 128)])
def test_decode_level(lib, G, classes, size):
    """Decode kernel vs the oracle restatement of models/yolo_nano.py:120-156,362-367."""
    g = torch.Generator().manual_seed(classes)
    ch = 3 * (1 + classes + 4)
    preds = [torch.randn(2, ch, size // s, size // s, generator=g) * 2 for s in (8, 16, 32)]
    bbox, cls = O.decode(preds, size, classes, W.anchors_for(classes))
    n = bbox.shape[1]
    boxes = torch.zeros(2, n, 4, device=G.DEV)
    scores = torch.zeros(2, n, device=G.DEV)
    cl = torch.zeros(2, n, device=G.DEV, dtype=torch.int32)
    off = 0
    anchors = np.array(W.anchors_for(classes), dtype=np.float32).reshape(3, 6)
    ld = (ch + 3) // 4 * 4
    for lvl, p in enumerate(preds):
        gsz = p.shape[2]
        raw = torch.zeros(2, gsz * gsz, ld)
        raw[..., :ch] = p.permute(0, 2, 3, 1).reshape(2, gsz * gsz, ch)
        raw = raw.to(G.DEV)
        a = (C.c_float * 6)(*anchors[lvl].tolist())
        rc = lib.ynb_decode_level(G.ptr(raw), ld, G.ptr(boxes), G.ptr(scores), G.ptr(cl), 2, gsz, 8 << lvl, size,
                                  a, 3, classes, n, off, G.stream())
        assert rc == 0, lib.ynb_last_error(None)
        off += gsz * gsz * 3
    torch.cuda.synchronize()
    # decoded boxes within 1e-3 px (BASELINE.json north_star)
    assert float((boxes.cpu() - bbox).abs().max()) * size < 1e-3
    for i in range(2):
        s_ref, c_ref = O.class_scores(cls[i].numpy())
        np.testing.assert_allclose(scores[i].cpu().numpy(), s_ref, rtol=2e-5, atol=1e-9)
        mism = cl[i].cpu().numpy() != c_ref
        # an argmax may only flip between classes whose probabilities agree to rounding
        if mism.any():
            p = cls[i].numpy()
            rows = np.nonzero(mism)[0]
            gap = np.abs(p[rows, cl[i].cpu().numpy()[rows]] - p[rows, c_ref[rows]]) / s_ref[rows]
            assert gap.max() < 1e-5 and mism.mean() < 1e-3


# ---------------------------------------------------------------------------------------------
# NMS: bit-exact keep-sets against the NumPy restatement on identical candidates
# ---------------------------------------------------------------------------------------------
def _check_nms(lib, G, boxes, scores, cls, classes, conf, thr, diou, grid_size=0):
    kept, counts, ob, os_, oc = G.run_nms(lib, boxes, scores, cls, classes, conf, thr, diou, grid_size)
    for i in range(scores.shape[0]):
        b, s, c, idx = O.postprocess_flat(boxes[i], scores[i], cls[i].astype(np.int64), classes, conf, thr, diou,
                                          tie="index")
        np.testing.assert_array_equal(kept[i], idx)
        k = counts[i]
        assert k == len(idx)
        np.testing.assert_array_equal(ob[i, :k], b)      # ascending anchor order, bit-identical rows
        np.testing.assert_array_equal(os_[i, :k], s)
        np.testing.assert_array_equal(oc[i, :k], c)


@pytest.mark.parametrize("fixture,classes", [("g1_voc320_refinit.npz", 20), ("g2_coco128_calibrated.npz", 80),
                                             ("g3_coco416_calibrated.npz", 80), ("g3_coco416_refinit.npz", 80)])
@pytest.mark.parametrize("conf,thr,diou", [(0.001, 0.5, False), (0.001, 0.5, True), (0.1, 0.45, False)])
def test_nms_on_reference_candidates(lib, G, golden, fixture, classes, conf, thr, diou):
    g = golden(fixture)
    pre = "" if "all_bbox" in g.files else "img0."
    imgs = [pre] if pre == "" else ["img0.", "img1."]
    boxes = np.stack([g[p + "all_bbox"] for p in imgs])
    scores = np.stack([g[p + "all_score"] for p in imgs])
    cls = np.stack([g[p + "all_cls"] for p in imgs])
    _check_nms(lib, G, boxes, scores, cls, classes, conf, thr, diou)
    size = {"g1": 320, "g2": 128, "g3": 416}[fixture[:2]]
    _check_nms(lib, G, boxes, scores, cls, classes, conf, thr, diou, grid_size=size)     # anchor-grid NMS


def test_nms_matches_reference_keepsets_when_tie_free(lib, G, golden):
    """Calibrated fixtures have no score ties: the CUDA keep-set must equal what the REAL
    reference kept (recorded keep_idx), not just the oracle."""
    for name, tags in (("g2_coco128_calibrated.npz", ("", "diou.", "t45c10.")), ("g3_coco416_calibrated.npz", ("",))):
        g = golden(name)
        for tag in tags:
            conf, thr, diou = (0.1, 0.45, False) if tag == "t45c10." else (0.001, 0.5, tag == "diou.")
            boxes = np.stack([g[f"img{i}.all_bbox"] for i in range(2)])
            scores = np.stack([g[f"img{i}.all_score"] for i in range(2)])
            cls = np.stack([g[f"img{i}.all_cls"] for i in range(2)])
            size = 128 if name.startswith("g2") else 416
            for grid_size in (0, size):
                kept, *_ = G.run_nms(lib, boxes, scores, cls, 80, conf, thr, diou, grid_size)
                for i in range(2):
                    np.testing.assert_array_equal(kept[i], g[f"img{i}.{tag}keep_idx"])


def test_nms_edge_cases(lib, G):
    rng = np.random.default_rng(0)
    n = 700
    xy = rng.random((2, n, 2), dtype=np.float32) * 0.8
    wh = rng.random((2, n, 2), dtype=np.float32) * 0.3
    boxes = np.concatenate([xy, np.minimum(xy + wh, 1.0)], -1).astype(np.float32)
    scores = rng.random((2, n), dtype=np.float32)
    cls = rng.integers(0, 5, (2, n)).astype(np.int32)
    # image 0: everything in one class, many exact score ties, zero-area boxes (NaN IoU, hazard 3)
    cls[0] = 3
    scores[0, ::3] = 0.5
    boxes[0, 10:40, 2:] = boxes[0, 10:40, :2]
    boxes[0, 50:60] = boxes[0, 50]                      # identical boxes
    # image 1: nothing passes the threshold
    scores[1] = 1e-6
    _check_nms(lib, G, boxes, scores, cls, 5, 0.001, 0.5, False)
    _check_nms(lib, G, boxes, scores, cls, 5, 0.001, 0.5, True)
    _check_nms(lib, G, boxes[:1, :1], scores[:1, :1], cls[:1, :1], 5, 0.001, 0.5, False)   # single box


def test_nms_large_segment_and_idempotence(lib, G):
    """BASELINE-size property checks: 608^2 anchor count (global-memory sort path), one giant
    class; NMS of the kept set keeps everything (idempotence)."""
    rng = np.random.default_rng(1)
    n = 22743
    xy = rng.random((1, n, 2), dtype=np.float32) * 0.9
    wh = rng.random((1, n, 2), dtype=np.float32) * 0.1 + 0.01
    boxes = np.concatenate([xy, np.minimum(xy + wh, 1.0)], -1).astype(np.float32)
    scores = rng.random((1, n), dtype=np.float32)
    cls = np.zeros((1, n), dtype=np.int32)
    kept, counts, ob, os_, oc = G.run_nms(lib, boxes, scores, cls, 80, 0.001, 0.5, False)
    _, _, _, idx = O.postprocess_flat(boxes[0], scores[0], cls[0].astype(np.int64), 80, 0.001, 0.5)
    np.testing.assert_array_equal(kept[0], idx)
    k = counts[0]
    kept2, counts2, *_ = G.run_nms(lib, ob[:, :k], os_[:, :k], oc[:, :k], 80, 0.001, 0.5, False)
    assert counts2[0] == k and np.array_equal(kept2[0], np.arange(k))


# ---------------------------------------------------------------------------------------------
# anchor-grid NMS (ynb_nms_grid): exact on any input, fast on decode-shaped input
def _decode_like_boxes(rng, size, batch, log_lo, log_hi, classes):
    """Boxes with the decode's structure (models/yolo_nano.py:120-156, 366): centre inside the
    anchor's cell, any size from sub-pixel to several images wide, clipped to the unit square."""
    bx, sc, cl = [], [], []
    for stride in (8, 16, 32):
        g = size // stride
        gy, gx = np.meshgrid(np.arange(g), np.arange(g), indexing="ij")
        gx = np.repeat(gx.reshape(-1), 3).astype(np.float32)
        gy = np.repeat(gy.reshape(-1), 3).astype(np.float32)
        n = gx.size
        u = rng.random((batch, n, 2), dtype=np.float32)
        u[rng.random((batch, n, 2)) < 0.02] = 0.0            # sigmoid saturating at a cell border
        u[rng.random((batch, n, 2)) < 0.02] = 1.0
        cx = (u[..., 0] + gx) * np.float32(stride)
        cy = (u[..., 1] + gy) * np.float32(stride)
        wh = np.exp(rng.uniform(log_lo, log_hi, (batch, n, 2))).astype(np.float32)
        x1 = (cx - wh[..., 0] * np.float32(0.5)) / np.float32(size)
        y1 = (cy - wh[..., 1] * np.float32(0.5)) / np.float32(size)
        x2 = (cx + wh[..., 0] * np.float32(0.5)) / np.float32(size)
        y2 = (cy + wh[..., 1] * np.float32(0.5)) / np.float32(size)
        bx.append(np.clip(np.stack([x1, y1, x2, y2], -1), 0.0, 1.0).astype(np.float32))
    boxes = np.concatenate(bx, 1)
    n = boxes.shape[1]
    scores = rng.random((batch, n), dtype=np.float32)
    scores[:, ::7] = np.float32(0.25)                          # exact ties
    cls = rng.integers(0, classes, (batch, n)).astype(np.int32)
    return boxes, scores, cls


@pytest.mark.parametrize("thr,diou", [(0.5, False), (0.5, True), (0.3, False), (0.7, False), (0.05, False),
                                      (0.0, False), (0.9, True)])
def test_nms_grid_decode_like_boxes_all_scales(lib, G, thr, diou):
    """Window search against the oracle on boxes from 0.3 px to 3 images wide, clipped at every
    border, 2 classes (long suppressor lists), conf cutting ~10 %."""
    rng = np.random.default_rng(int(thr * 100) + diou)
    size = 160
    boxes, scores, cls = _decode_like_boxes(rng, size, 3, np.log(0.3), np.log(3 * size), 2)
    _check_nms(lib, G, boxes, scores, cls, 2, 0.1, thr, diou, grid_size=size)


def test_nms_grid_uniform_scale_segments(lib, G):
    """The bench-shaped case: every (level, anchor) is one class with near-identical box sizes
    (reference-init behaviour), long dependency chains between neighbouring cells."""
    rng = np.random.default_rng(5)
    size = 256
    boxes, scores, cls = _decode_like_boxes(rng, size, 2, 0.0, 0.0, 1)
    n0, n1 = 3 * 32 * 32, 3 * 16 * 16
    for lvl, (beg, end) in enumerate(((0, n0), (n0, n0 + n1), (n0 + n1, boxes.shape[1]))):
        for a in range(3):
            anchor = np.float32((8 << lvl) * (1.5 + a))
            idx = np.arange(beg + a, end, 3)
            c = (boxes[:, idx, :2] + boxes[:, idx, 2:]) * np.float32(0.5)
            half = anchor * np.exp(rng.normal(0, 0.05, (2, idx.size, 2))).astype(np.float32) / np.float32(2 * size)
            boxes[:, idx, :2] = np.clip(c - half, 0, 1)
            boxes[:, idx, 2:] = np.clip(c + half, 0, 1)
            cls[:, idx] = (lvl * 3 + a) % 4
    _check_nms(lib, G, boxes, scores, cls, 4, 0.001, 0.5, False, grid_size=size)
    _check_nms(lib, G, boxes, scores, cls, 4, 0.001, 0.45, True, grid_size=size)


def test_nms_grid_crowded_and_irregular(lib, G):
    """More suppressors than the list holds (re-scan path), zero-area / out-of-cell / NaN-IoU
    boxes (irregular list), arbitrary boxes unrelated to the grid."""
    rng = np.random.default_rng(9)
    size = 128
    boxes, scores, cls = _decode_like_boxes(rng, size, 3, np.log(40.0), np.log(60.0), 1)   # everything overlaps
    boxes[0, 100:140, 2:] = boxes[0, 100:140, :2]          # zero area (0/0 = NaN suppresses, hazard 3)
    boxes[0, 200:210] = boxes[0, 200]                       # identical boxes in foreign cells
    n = boxes.shape[1]
    xy = rng.random((n, 2), dtype=np.float32) * 0.8         # image 2: boxes that ignore the grid entirely
    boxes[2] = np.concatenate([xy, np.minimum(xy + rng.random((n, 2), dtype=np.float32) * 0.3, 1.0)], -1)
    cls[2] = rng.integers(0, 3, n)
    for thr, diou in ((0.5, False), (0.6, True)):
        _check_nms(lib, G, boxes, scores, cls, 3, 0.001, thr, diou, grid_size=size)
    scores[1] = 1e-6                                        # nothing passes the threshold
    _check_nms(lib, G, boxes[1:2], scores[1:2], cls[1:2], 3, 0.001, 0.5, False, grid_size=size)
