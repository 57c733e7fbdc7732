"""CPU tier of the evaluation metrics: known answers for the float64 reference (tests/reference_metrics.py), its SSIM
against an independent 2-D convolution, the host-side summary, and the argument checks of pnr_eval_frame (which run
before any CUDA call, so they are exercised here without a device)."""
import ctypes as C
import re
from fractions import Fraction

import numpy as np
import pytest
import torch

import reference_metrics as RM

THING = [0, 1]          # category 0 stuff, category 1 thing


def frame(rows):
    return np.array(rows, dtype=np.int64).ravel()


def test_perfect_prediction_scores_one():
    g = np.random.default_rng(0)
    sem = g.integers(0, 5, 400)
    pan = np.where(sem >= 3, sem * 1000 + g.integers(1, 4, 400), sem * 1000)
    w = RM.frame_words(5, sem, sem, pan, pan, [0, 0, 0, 1, 1])
    m = RM.metrics(w, 5)
    assert m["miou"] == 1.0 and m["pixel_acc"] == 1.0
    assert m["pq"] == m["sq"] == m["rq"] == 1.0


def test_hand_built_frame_exact_fractions():
    """6x6: GT thing 1001 = row 0 cols 0-3, predicted 1001 = row 0 cols 1-4 (IoU 3/5); GT thing 1002 = row 2 cols 0-2
    under predicted stuff (FN); predicted thing 1007 = row 4 cols 0-2 on GT stuff (FP); everything else stuff 0."""
    gt = np.zeros((6, 6), np.int64)
    pr = np.zeros((6, 6), np.int64)
    gt[0, 0:4] = 1001
    pr[0, 1:5] = 1001
    gt[2, 0:3] = 1002
    pr[4, 0:3] = 1007
    tp, fp, fn, iou = RM.pq_stats(pr.ravel(), gt.ravel(), 2, THING)
    assert tp.tolist() == [1, 1] and fp.tolist() == [0, 1] and fn.tolist() == [0, 1]
    assert iou[1] == 0.6
    # stuff: both areas 29, intersection 36 - 11 = 25
    assert iou[0] == 25 / 33
    m = RM.metrics(RM.frame_words(2, pan_pred=pr, pan_gt=gt, is_thing=THING), 2)
    pq1 = Fraction(3, 5) / 2
    assert m["pq"] == pytest.approx(float((pq1 + Fraction(25, 33)) / 2), rel=0, abs=1e-15)
    assert m["rq"] == pytest.approx(0.75, abs=1e-15) and m["sq"] == pytest.approx(float((Fraction(3, 5) + Fraction(25, 33)) / 2), abs=1e-15)


def test_iou_of_exactly_one_half_is_not_a_match():
    gt = frame([[1001, 1001, 1001, 1001, 0, 0]])
    pr = frame([[1001, 1001, 0, 0, 0, 0]])        # |p∩g| = 2, union 4
    tp, fp, fn, iou = RM.pq_stats(pr, gt, 2, THING)
    assert (tp[1], fp[1], fn[1], iou[1]) == (0, 1, 1, 0.0)


def test_void_pixels_leave_the_union():
    gt = frame([[1001, 1001, 1001, -1, -1, -1, 0, 0]])
    pr = frame([[1001, 1001, 1001, 1001, 1001, 1001, 0, 0]])   # 3 of the 6 predicted pixels lie on GT void
    tp, fp, fn, iou = RM.pq_stats(pr, gt, 2, THING)
    assert (tp[1], fp[1], fn[1], iou[1]) == (1, 0, 0, 1.0)
    # a category id outside [0, C) is void too
    tp2, _, _, iou2 = RM.pq_stats(pr, np.where(gt < 0, 7000, gt), 2, THING)
    assert tp2[1] == 1 and iou2[1] == 1.0


def test_prediction_on_void_or_crowd_is_not_a_false_positive():
    gt = frame([[-1, -1, -1, 0, 1000, 1000, 1000, 0, 0, 0]])      # 1000 = thing category 1, instance 0: crowd
    pr = frame([[1005, 1005, 1005, 1005, 1006, 1006, 1006, 1006, 0, 0]])
    tp, fp, fn, _ = RM.pq_stats(pr, gt, 2, THING)
    assert tp[1] == 0 and fp[1] == 0 and fn[1] == 0                # the crowd region is not a missed segment either
    pr2 = frame([[1005, 0, 0, 1005, 1006, 1006, 0, 1006, 1006, 0]])  # exactly half on void / crowd is not "mostly"
    _, fp2, _, _ = RM.pq_stats(pr2, gt, 2, THING)
    assert fp2[1] == 2


def test_stuff_instance_part_is_ignored():
    gt = frame([[3, 3, 7, 7, 1001, 1001]])       # two "instances" of stuff category 0
    pr = frame([[0, 0, 0, 0, 1001, 1001]])
    tp, fp, fn, iou = RM.pq_stats(pr, gt, 2, THING)
    assert tp.tolist() == [1, 1] and fp.sum() == 0 and fn.sum() == 0 and iou.tolist() == [1.0, 1.0]


def test_segment_cap():
    ids = np.arange(1025, dtype=np.int64) + 10001            # 1025 instances of thing category 1
    assert RM.pq_stats(ids, ids, 2, THING, div=10000) is None
    assert RM.pq_stats(ids[:1024], ids[:1024], 2, THING, div=10000)[0][1] == 1024


def test_psnr_and_ssim_known_answers():
    g = np.random.default_rng(1)
    H, W = 20, 24
    img = g.random((H * W, 3))
    assert RM.ssim(img, img, H, W) == pytest.approx(1.0, abs=1e-15)
    assert RM.psnr(np.clip(img, 0.2, 0.8) + 0.1, np.clip(img, 0.2, 0.8)) == pytest.approx(20.0, abs=1e-9)
    assert RM.psnr(img, img) == float("inf")


def test_ssim_matches_a_2d_valid_convolution():
    from scipy import signal
    g = np.random.default_rng(2)
    H, W = 37, 45
    x = g.random((H, W, 3))
    y = np.clip(x + 0.1 * g.standard_normal((H, W, 3)), 0, 1)
    win = np.outer(RM.gaussian_window(), RM.gaussian_window())
    conv = lambda z: signal.convolve2d(z, win[::-1, ::-1], mode="valid")
    vals = []
    for c in range(3):
        a, b = x[..., c], y[..., c]
        mx, my = conv(a), conv(b)
        vx = np.maximum(conv(a * a) - mx ** 2, 0)
        vy = np.maximum(conv(b * b) - my ** 2, 0)
        cxy = conv(a * b) - mx * my
        vals.append((2 * mx * my + 1e-4) * (2 * cxy + 9e-4) / ((mx ** 2 + my ** 2 + 1e-4) * (vx + vy + 9e-4)))
    assert RM.ssim(x.reshape(-1, 3), y.reshape(-1, 3), H, W) == pytest.approx(float(np.mean(vals)), rel=1e-12)


def test_depth_known_answers():
    gt = np.array([0.0, -1.0, 10.0, 10.0, 200.0, 10.0], np.float32)
    pred = np.array([5.0, 5.0, 12.5, 10.0, 10.0, 0.0], np.float32)
    sums, counts = RM.depth_stats(pred, gt, 1e-3, 80.0)
    # 0 / negative / beyond max_depth excluded; a ratio of exactly 1.25 is not < 1.25; 1e-3 vs 10 fails all
    assert counts.tolist() == [3, 1, 2, 2]
    p = np.array([12.5, 10.0, np.float32(1e-3)], np.float64)
    assert sums[2] == pytest.approx(np.sum((p - 10) ** 2), rel=1e-15)


def test_host_summary_matches_the_reference_summary():
    from panopticnerf_b200.lib.evaluators import summarize_stats
    g = np.random.default_rng(3)
    R, Cn = 3000, 6
    thing = [0, 0, 1, 1, 0, 1]
    sem_gt = g.integers(-1, Cn, R)
    sem_pr = np.where(g.random(R) < 0.7, sem_gt, g.integers(0, Cn, R))
    base = np.repeat(g.integers(0, Cn, R // 50), 50)
    pan_gt = base * 1000 + np.repeat(g.integers(0, 3, R // 50), 50)
    pan_pr = np.where(g.random(R) < 0.8, pan_gt, base * 1000 + 1)
    w = RM.frame_words(Cn, sem_pr, sem_gt, pan_pr, pan_gt, thing)
    got, ref = summarize_stats(w, Cn, thing), RM.metrics(w, Cn)
    for k in ("miou", "pixel_acc", "pq", "sq", "rq"):
        assert got[k] == pytest.approx(ref[k], rel=1e-14), k
    over = w.copy()
    over[RM.OVERFLOW] = 1
    from panopticnerf_b200._capi import PnrError
    with pytest.raises(PnrError, match="1024"):
        summarize_stats(over, Cn, thing)


# ------------------------------------------------------------------------------------------------ C entry point
def _lib():
    import __graft_entry__ as g
    g.build()
    from panopticnerf_b200 import _capi
    return _capi


def test_stats_and_workspace_sizes():
    capi = _lib()
    L = capi.lib()
    assert L.pnr_eval_stats_bytes(45) == 8 * (16 + 45 * 45 + 4 * 45)
    assert L.pnr_eval_stats_bytes(0) == 8 * 16
    assert L.pnr_eval_stats_bytes(65) == 0 and L.pnr_eval_stats_bytes(-1) == 0
    small = L.pnr_eval_workspace_bytes(376 * 1408, 45, 0)
    assert small == 6 * 1024 * 8
    full = L.pnr_eval_workspace_bytes(376 * 1408, 45, 1000)
    assert full >= small + 2 * 4 * 45 * 1000 + 4 * 1024 * 1025 + 8 * 1024
    assert full < small + 2 * 4 * 45 * 1000 + 4 * 1024 * 1025 + 64 * 1024
    assert L.pnr_eval_workspace_bytes(100, 64, 1 << 20) == 0           # C * label_divisor > 2^24


@pytest.mark.parametrize("field,value,match", [
    ("C", 65, "C=65"), ("C", -1, "C=-1"), ("label_divisor", 0, "label_divisor=0"), ("H", 7, "H\\*W"),
    ("stats", None, "stats"), ("workspace_bytes", 1024, "workspace"), ("is_thing", None, "is_thing"),
    ("sem_gt", None, "sem_pred and sem_gt")])
def test_eval_frame_rejects_bad_arguments_before_touching_the_device(field, value, match):
    capi = _lib()
    L = capi.lib()
    fake = 1 << 20                                    # never dereferenced: the checks come before any CUDA call
    a = capi.PnrEvalArgs()
    a.R, a.C, a.H, a.W = 64 * 32, 45, 32, 64
    for k in ("sem_pred", "sem_gt", "pan_pred", "pan_gt", "is_thing", "rgb_pred", "rgb_gt", "depth_pred", "depth_gt",
              "stats", "workspace"):
        setattr(a, k, fake)
    a.label_divisor, a.min_depth, a.max_depth = 1000, 1e-3, 80.0
    a.workspace_bytes = L.pnr_eval_workspace_bytes(a.R, 45, 1000)
    setattr(a, field, value)
    rc = L.pnr_eval_frame(C.byref(a), None)
    assert rc == -1
    assert re.search(match, L.pnr_last_error().decode()), L.pnr_last_error().decode()
    assert L.pnr_eval_frame(None, None) == -1


def test_evaluator_refuses_cpu_tensors():
    import panopticnerf_b200 as PN
    from panopticnerf_b200 import _capi
    ev = PN.make_evaluator(PN.make_cfg("cfg1", num_classes=5, is_thing=[0, 0, 1, 1, 0]))
    out = {"rgb_map": torch.zeros(16, 3), "semantic_map": torch.zeros(16, 5)}
    with pytest.raises(_capi.PnrError, match="CUDA"):
        ev.evaluate(out, {"rgb": torch.zeros(16, 3), "semantic_gt": torch.zeros(16, dtype=torch.int32)})
    with pytest.raises(ValueError, match="is_thing"):
        PN.make_evaluator(PN.make_cfg("cfg1", num_classes=5, is_thing=[0, 1]))
