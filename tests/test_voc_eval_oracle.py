"""CPU checks of the VOC mAP restatement (oracle/voc_eval.py) that the device evaluator is compared with: the decimal
fields of the det-file lines, and the vectorised integer-row form against the literal voc_eval on real det files."""
import tempfile

import numpy as np
import pytest

from oracle import voc_eval as V


def _values(n, seed):
    rng = np.random.default_rng(seed)
    parts = [
        rng.uniform(-50, 1e4, n).astype(np.float32),
        rng.uniform(-2, 2, n // 4).astype(np.float32),
        (rng.integers(-4000, 40000, n // 4) * 0.25).astype(np.float32),       # x.25 / x.75: '{:.1f}' half-way
        (rng.integers(-1600, 16000, n // 4) / 16).astype(np.float32),        # k/16: '{:.3f}' half-way cases
        rng.random(n // 4, dtype=np.float32),                                # scores
        np.array([0.0, -0.0, -0.04, -0.05, 0.05, 0.0005, -0.0005, 1e-30, -1e-30, 9999.95, 1e4, 1.0,
                  np.float32(0.1), np.float32(0.15), np.float32(0.25), np.float32(2.5)], np.float32),
    ]
    return np.concatenate(parts)


def _parse(s):
    n = int(s.replace(".", ""))
    return V.NEG_ZERO if s.startswith("-") and n == 0 else n


@pytest.mark.parametrize("digits", [1, 3])
def test_decimal_ints_equal_python_formatting(digits):
    """decimal_ints == the integer of '{:.1f}'.format(np.float32(v) + 1) / '{:.3f}'.format(v) on > 1 M float32
    values (exact half-way cases, negatives, -0.0, up to 1e4), and n / 10**digits is what float() parses back."""
    v = _values(600_000, digits)
    x = v + np.float32(1) if digits == 1 else v                 # the writer's `dets[k, 0] + 1` in float32
    assert x.dtype == np.float32 and len(x) >= 1_000_000
    fmt = "{:.%df}" % digits
    strs = [fmt.format(t) for t in x.tolist()]                 # .tolist() = the exact float32 values as doubles
    want = np.array([_parse(s) for s in strs], np.int64)
    got = V.decimal_ints(x, digits)
    bad = np.nonzero(got != want)[0]
    assert len(bad) == 0, [(float(x[i]), strs[i], int(got[i])) for i in bad[:5]]
    back = np.array([float(s) for s in strs])
    dec = np.where(got == V.NEG_ZERO, -0.0, got / float(10 ** digits))
    assert np.array_equal(back.view(np.int64), dec.view(np.int64))     # bit for bit, sign of zero included


def test_rows_equal_fields_of_the_writer():
    """result_rows == the fields parsed back from evalfmt.voc_result_lines (the writer golden g6 pins)."""
    from yolo_nano_b200 import evalfmt
    dets, _ = V.random_set(60, 5, seed=3)
    rows = V.result_rows(dets)
    parsed = []
    for i, (b, s, c) in enumerate(dets):
        for k in range(len(s)):
            line = evalfmt.voc_result_lines("x", np.hstack([b[k:k + 1], s[k:k + 1, None]]).astype(np.float32))[0]
            f = line.split()
            parsed.append([i, int(c[k])] + [_parse(t) for t in f[1:]])
    assert np.array_equal(rows, np.array(parsed, np.int64).astype(np.int32))


def _edge_set():
    """Hand-made cases: a difficult match, duplicates of one GT, overlap exactly 0.5, a zero-area NaN overlap,
    an image without GT, a class without GT and a class without lines (5 classes)."""
    f32 = np.float32
    gt = [
        (np.array([[0, 0, 10, 10], [20, 20, 30, 30], [50, 50, 60, 60]], float), np.array([0, 0, 1]),
         np.array([False, True, False])),
        (np.array([[0, 0, 10, 10], [5, 5, 5, 5]], float), np.array([0, 2]), np.array([False, False])),
        (np.zeros((0, 4)), np.zeros(0, int), np.zeros(0, bool)),
    ]
    # boxes are written with +1: store box - 1
    d0 = (np.array([[0, 0, 10, 10], [0, 0, 10, 10], [20, 20, 30, 30], [50, 50, 60, 60], [0, 0, 20, 10]], f32) - 1,
          np.array([0.9, 0.9, 0.8, 0.7, 0.6], f32), np.array([0, 0, 0, 1, 3]))
    d1 = (np.array([[0, 0, 10, 5.0], [0, 0, 10, 10], [5, 5, 5, 5]], f32) - 1,   # IoU 0.5 exactly; then a match
          np.array([0.95, 0.5, 0.4], f32), np.array([0, 0, 2]))
    d2 = (np.array([[1, 1, 5, 5]], f32) - 1, np.array([0.3], f32), np.array([0]))
    return [d0, d1, d2], gt


@pytest.mark.parametrize("use07", [True, False])
def test_rows_form_equals_literal_voc_eval(use07):
    """voc_eval_rows (integer rows, stable order, parallel claim rule) == voc_eval_literal on det files written to a
    temp dir (stable argsort), bit for bit, on hand-made edge cases and on a random tie-heavy set."""
    for dets, gt, nc in [(*_edge_set(), 5), (*V.random_set(300, 6, seed=11), 6)]:
        with tempfile.TemporaryDirectory() as tmp:
            want = V.eval_files(tmp, dets, gt, nc, use_07_metric=use07, kind="stable")
        got, npos, _ = V.voc_eval_rows(V.result_rows(dets), gt, nc, use_07_metric=use07)
        assert np.array_equal(got.view(np.int64), want.view(np.int64)), (got, want)


def test_edge_cases_values():
    dets, gt = _edge_set()
    ap07, npos, detail = V.voc_eval_rows(V.result_rows(dets), gt, 5, use_07_metric=True)
    area, _, _ = V.voc_eval_rows(V.result_rows(dets), gt, 5, use_07_metric=False)
    assert list(npos) == [2, 1, 1, 0, 0]
    assert ap07[4] == -1 and area[4] == -1                     # no lines
    assert ap07[3] == 0 and np.isnan(area[3])                  # lines but no GT
    flags0 = detail[0][1]
    # class 0 sorted: 0.95 (IoU 0.5, FP), 0.9 TP, 0.9 duplicate FP, 0.8 difficult (ignored), 0.5 TP, 0.3 no GT FP
    assert list(flags0) == [2, 1, 2, 0, 1, 2]


def test_arange_thresholds_are_multiples_of_a_tenth():
    """The device's 07 thresholds are i * 0.1 in float64: that is what np.arange(0., 1.1, 0.1) holds."""
    t = np.arange(0., 1.1, 0.1)
    assert len(t) == 11 and np.array_equal(t, np.arange(11) * 0.1)


def test_report_default_vs_stable_argsort():
    """How far voc_eval's default (unstable) argsort moves the APs on a tie-heavy set: reported, not asserted."""
    dets, gt = V.random_set(400, 5, seed=5, score_levels=20)
    with tempfile.TemporaryDirectory() as tmp:
        a, b = V.default_vs_stable(dets, gt, 5, tmp)
    print(f"[report] default vs stable argsort: per-class |dAP| max {np.abs(a - b).max():.3e}, "
          f"mAP {a.mean():.6f} vs {b.mean():.6f}")
