"""The engine's output depends only on (weights, GEMM mode, grid, batch, thresholds): not on the order in which they
were set.  Mode switches, re-commits, grid and batch changes and CUDA-graph capture / replay must leave nothing
stale behind, and the drop-in module must notice every way its weights can change."""
import contextlib
import io

import numpy as np
import pytest
import torch

from oracle import weights as W
from oracle import yolo_nano_oracle as O

TAPS = (["pool"] + [f"stage{s}.{n}" for s, reps in O.STAGES for n in ["b1dw", "b2pw"] + list(range(reps))]
        + ["lat3", "lat4", "lat5", "fpn4", "p3", "p4", "p5"] + [f"head{l}.{n}" for l in range(3) for n in "ab"])
_SD = {}


def sd_of(name):
    """Two calibrated weight sets (O(1) activations, so a stale layer changes every output)."""
    if name not in _SD:
        _SD[name] = W.calibrated(80, seed={"A": 1, "B": 2}[name])
    return _SD[name]


def fused(name):
    from yolo_nano_b200.topology import conv_table
    return O.fold_state_dict(sd_of(name), conv_table(80))


def _mode(mode):
    import gpu_util as G
    return G.MODES[mode]


def new_engine(mode, weights, size=128, max_batch=2, **kw):
    import gpu_util as G
    from yolo_nano_b200.engine import Engine
    eng = Engine(G.DEV, size, 80, W.anchors_for(80), gemm_mode=_mode(mode), max_batch=max_batch, **kw)
    eng.load_weights(fused(weights))
    return eng


def raw_and_taps(eng, x):
    out = {n: t.cpu() for n, t in zip(("pred_s", "pred_m", "pred_l"), eng.forward_raw(x))}
    out.update({n: eng.read_tap(n, x.shape[0]).cpu() for n in TAPS})
    return out


def first_difference(got, want):
    """Names (in forward order) whose tensors are not bit-identical."""
    return [n for n in TAPS + ["pred_s", "pred_m", "pred_l"] if not torch.equal(got[n], want[n])]


def model(sd, device, size=128):
    import yolo_nano_b200 as pkg
    with contextlib.redirect_stdout(io.StringIO()):
        m = pkg.YOLONano(device, size, 80, anchor_size=pkg.MULTI_ANCHOR_SIZE_COCO)
    m.load_state_dict(sd)
    return m.to(device).eval()


# ---- GPU ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["3xtf32", "tf32"])
def test_mode_round_trip_with_recommit_equals_fresh_engine(mode):
    """create in `mode` with weights A; switch to FFMA and load B; switch back.  Raw maps and every tap must be
    bit-identical to a fresh `mode` engine loaded with B (the merged stride-2 GEMM weights included)."""
    x = W.synthetic_input(2, 128, 4).cuda()
    eng = new_engine(mode, "A")
    eng.forward_raw(x)
    eng.set_gemm_mode(_mode("ffma"))
    eng.load_weights(fused("B"))
    eng.forward_raw(x)
    eng.set_gemm_mode(_mode(mode))
    got = raw_and_taps(eng, x)
    eng.close()
    fresh = new_engine(mode, "B")
    want = raw_and_taps(fresh, x)
    fresh.close()
    diff = first_difference(got, want)
    assert not diff, f"{mode} after FFMA + re-commit: stale from {diff[0]} on ({len(diff)} tensors differ: {diff})"


def _run_three(eng, x, out):
    """forward_raw, then forward_detect three times on the same buffers: eager, graph capture, graph replay."""
    raw = [t.cpu() for t in eng.forward_raw(x)]
    dets = []
    for _ in range(3):
        b, s, c, n = [t.cpu() for t in eng.forward_detect(x, out)]
        dets.append([n] + [t[i, :int(n[i])] for i in range(len(n)) for t in (b, s, c)])   # rows past a count are unset
    return raw, dets


@pytest.mark.gpu
def test_seeded_walk_over_state_transitions_equals_fresh_engines():
    """~12 seeded steps over set_grid (96 / 128 / 160), batch 1 / 2 / 3, modes FFMA / 3xTF32 / TF32, weights A / B and
    set_thresholds on ONE engine.  After each step: forward_raw and forward_detect (eager, capture, replay) must be
    bit-identical to an engine built directly in that state (same max_batch)."""
    rng = np.random.default_rng(7)
    eng = new_engine("3xtf32", "A", size=128, max_batch=3)
    state = {"size": 128, "batch": 2, "mode": "3xtf32", "weights": "A", "thr": (0.001, 0.5, False)}
    fresh_cache = {}
    kinds = ["grid", "batch", "mode", "weights", "thr"]
    for step in range(12):
        kind = kinds[step % len(kinds)] if step < len(kinds) else kinds[int(rng.integers(len(kinds)))]
        if kind == "grid":
            state["size"] = int(rng.choice([s for s in (96, 128, 160) if s != state["size"]]))
            eng.set_grid(state["size"])
        elif kind == "batch":
            state["batch"] = int(rng.choice([b for b in (1, 2, 3) if b != state["batch"]]))
        elif kind == "mode":
            state["mode"] = str(rng.choice([m for m in ("ffma", "3xtf32", "tf32") if m != state["mode"]]))
            eng.set_gemm_mode(_mode(state["mode"]))
        elif kind == "weights":
            state["weights"] = "B" if state["weights"] == "A" else "A"
            eng.load_weights(fused(state["weights"]))
        else:
            state["thr"] = [(0.001, 0.5, False), (0.05, 0.45, True), (0.01, 0.6, False)][int(rng.integers(3))]
            eng.set_thresholds(*state["thr"])
        x = W.synthetic_input(state["batch"], state["size"], state["size"] + state["batch"]).cuda()
        raw, dets = _run_three(eng, x, eng.alloc_outputs(state["batch"]))
        key = (state["size"], state["batch"], state["mode"], state["weights"], state["thr"])
        if key not in fresh_cache:
            f = new_engine(state["mode"], state["weights"], size=state["size"], max_batch=3,
                           conf_thresh=state["thr"][0], nms_thresh=state["thr"][1], diou_nms=state["thr"][2])
            fresh_cache[key] = _run_three(f, x, f.alloc_outputs(state["batch"]))
            f.close()
        raw_f, dets_f = fresh_cache[key]
        where = f"step {step} ({kind}) -> {state}"
        for a, b in zip(raw, raw_f):
            assert torch.equal(a, b), f"{where}: raw maps differ from a fresh engine"
        for i, (d, df) in enumerate(zip(dets, dets_f)):
            for a, b in zip(d, df):
                assert torch.equal(a, b), f"{where}: forward_detect call {i} differs from a fresh engine"
    eng.close()


@pytest.mark.gpu
def test_bf16_engine_refuses_fp32_modes_and_keeps_its_output():
    from yolo_nano_b200.engine import EngineError
    x = W.synthetic_input(2, 128, 5).cuda()
    eng = new_engine("bf16", "A")
    before = raw_and_taps(eng, x)
    for m in ("ffma", "3xtf32", "tf32"):
        with pytest.raises(EngineError):
            eng.set_gemm_mode(_mode(m))
    assert not first_difference(raw_and_taps(eng, x), before), "output changed after a refused mode switch"
    eng.load_weights(fused("A"))
    assert not first_difference(raw_and_taps(eng, x), before), "output changed after re-committing the same weights"
    eng.close()


def _detections_equal(a, b):
    return all(np.array_equal(u, v) for u, v in zip(a, b))


@pytest.mark.gpu
def test_dropin_sees_assign_load_and_dtype_round_trip():
    """The drop-in re-packs the engine weights after load_state_dict(assign=True), and after a dtype round trip
    followed by an in-place update of a BatchNorm buffer."""
    dev = torch.device("cuda", 0)
    x = W.synthetic_input(1, 128, 6).to(dev)
    m = model(sd_of("A"), dev)
    out_a = m(x)
    sd_b = {k: v.to(dev) for k, v in sd_of("B").items()}
    m.load_state_dict(sd_b, assign=True)
    out_b = m(x)
    want_b = model(sd_of("B"), dev)(x)
    assert not _detections_equal(out_a, want_b), "weights A and B must give different detections"
    assert _detections_equal(out_b, want_b), "stale weights after load_state_dict(assign=True)"

    m.double()
    m.float()
    m.get_submodule("backbone.stage3.0.branch1.1").running_var.mul_(1.7)
    out_c = m(x)
    want_c = model({k: v.cpu() for k, v in m.state_dict().items()}, dev)(x)
    assert not _detections_equal(out_b, want_c), "the running_var update must change the detections"
    assert _detections_equal(out_c, want_c), "stale weights after a dtype round trip and an in-place buffer update"


# ---- CPU: the drop-in's weight fingerprint -------------------------------------------------------------------------
def test_weights_fingerprint_tracks_every_way_weights_change():
    import yolo_nano_b200 as pkg
    m = model(sd_of("A"), torch.device("cpu"))
    fp = m._weights_fingerprint()
    assert m._weights_fingerprint() == fp, "nothing changed: the fingerprint (and the engine cache) must hold"

    m.load_state_dict({k: v.clone() for k, v in sd_of("B").items()}, assign=True)
    fp2 = m._weights_fingerprint()
    assert fp2 != fp, "load_state_dict(assign=True)"
    assert m._weights_fingerprint() == fp2

    m.double()
    m.float()
    fp3 = m._weights_fingerprint()
    m.get_submodule("backbone.stage3.0.branch1.1").running_var.mul_(1.7)
    assert m._weights_fingerprint() != fp3, "dtype round trip, then an in-place buffer update"

    fp4 = m._weights_fingerprint()
    pkg.fuse_conv_bn(m)
    assert m._weights_fingerprint() != fp4, "fuse_conv_bn"
    assert len(m._weight_tensors()) == 154
