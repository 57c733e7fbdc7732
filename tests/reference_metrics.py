"""float64 numpy restatement of the evaluation metrics of include/pnr.h (pnr_eval_frame).  TEST INFRASTRUCTURE ONLY:
tests/test_cpu_eval.py pins it with known answers, tests/test_gpu_eval.py holds the kernels to it.

`frame_words` returns one frame's statistics in the layout of the device buffer (int64 words, float64 sums stored
bit-cast), so a test can compare the integer statistics exactly and the sums within a tolerance."""
from __future__ import annotations

import math
from typing import Optional

import numpy as np

HEADER_WORDS = 16
MAX_SEGMENTS = 1024
(OVERFLOW, PQ_FRAMES, PSNR_FRAMES, SSIM_FRAMES, DEPTH_VALID, DEPTH_DELTA1, DEPTH_DELTA2, DEPTH_DELTA3,
 PSNR_SUM, SSIM_SUM, ABS_REL_SUM, SQ_REL_SUM, SQ_ERR_SUM, SQ_LOG_SUM) = range(14)


def confusion(pred, gt, C: int) -> np.ndarray:
    """[C, C] int64, row = GT, column = prediction; labels outside [0, C) on either side are ignored."""
    p, g = np.asarray(pred, np.int64).ravel(), np.asarray(gt, np.int64).ravel()
    ok = (g >= 0) & (g < C) & (p >= 0) & (p < C)
    return np.bincount(g[ok] * C + p[ok], minlength=C * C).reshape(C, C).astype(np.int64)


def segment_keys(ids, C: int, div: int, is_thing) -> np.ndarray:
    """-1 for void (negative id or category outside [0, C)); stuff categories drop the instance part."""
    ids = np.asarray(ids, np.int64).ravel()
    thing = np.asarray(is_thing, bool)
    cat = np.where(ids >= 0, ids // div, -1)
    void = (ids < 0) | (cat >= C)
    catc = np.clip(cat, 0, C - 1)
    return np.where(void, -1, np.where(thing[catc], ids, catc * div))


def pq_stats(pan_pred, pan_gt, C: int, is_thing, div: int = 1000, cap: int = MAX_SEGMENTS):
    """Per category tp, fp, fn (int64 [C]) and iou_sum (float64 [C], the TPs in ascending predicted-segment id order),
    or None when a side has more than `cap` distinct segments."""
    thing = np.asarray(is_thing, bool)
    kp, kg = segment_keys(pan_pred, C, div, is_thing), segment_keys(pan_gt, C, div, is_thing)
    P, ap = np.unique(kp[kp >= 0], return_counts=True)
    G, ag = np.unique(kg[kg >= 0], return_counts=True)
    if len(P) > cap or len(G) > cap:
        return None
    area_g = dict(zip(G.tolist(), ag.tolist()))
    sel = kp >= 0
    pairs, cnt = np.unique(np.stack([kp[sel], kg[sel]], 1), axis=0, return_counts=True)
    inter = {}
    for (a, b), n in zip(pairs.tolist(), cnt.tolist()):
        inter.setdefault(a, {})[b] = n
    tp, fp, fn = (np.zeros(C, np.int64) for _ in range(3))
    iou_sum = np.zeros(C, np.float64)
    matched = set()
    crowd = lambda key: bool(thing[key // div]) and key % div == 0
    for key, area in zip(P.tolist(), ap.tolist()):
        c = key // div
        row = inter.get(key, {})
        on_void = row.get(-1, 0)
        hit = None
        for gk, n in row.items():
            if gk < 0 or gk // div != c or crowd(gk):
                continue
            denom = area + area_g[gk] - n - on_void
            if 2 * n > denom:
                hit = (gk, n / denom)
        if hit is not None:
            tp[c] += 1
            iou_sum[c] += hit[1]
            matched.add(hit[0])
        elif 2 * (on_void + (row.get(c * div, 0) if thing[c] else 0)) <= area:
            fp[c] += 1
    for gk in G.tolist():
        if gk not in matched and not crowd(gk):
            fn[gk // div] += 1
    return tp, fp, fn, iou_sum


def psnr(pred, gt) -> float:
    d = np.asarray(pred, np.float64) - np.asarray(gt, np.float64)
    mse = np.mean(d * d)
    return math.inf if mse == 0 else -10.0 * math.log10(mse)


def gaussian_window(size: int = 11, sigma: float = 1.5) -> np.ndarray:
    f = (np.arange(size, dtype=np.float64) - size // 2) / sigma
    g = np.exp(-0.5 * f * f)
    return g / g.sum()


def ssim(pred, gt, H: int, W: int) -> float:
    """Mean SSIM over the valid region and the 3 channels (11x11 Gaussian, sigma 1.5, c1 = 0.01^2, c2 = 0.03^2)."""
    g = gaussian_window()
    x = np.asarray(pred, np.float64).reshape(H, W, 3)
    y = np.asarray(gt, np.float64).reshape(H, W, 3)
    Ho, Wo = H - 10, W - 10

    def filt(z):
        h = sum(g[k] * z[:, k:k + Wo] for k in range(11))
        return sum(g[k] * h[k:k + Ho] for k in range(11))

    c1, c2 = 0.01 ** 2, 0.03 ** 2
    vals = []
    for c in range(3):
        a, b = x[..., c], y[..., c]
        mx, my = filt(a), filt(b)
        vx = np.maximum(filt(a * a) - mx * mx, 0.0)
        vy = np.maximum(filt(b * b) - my * my, 0.0)
        cxy = filt(a * b) - mx * my
        vals.append(((2 * mx * my + c1) * (2 * cxy + c2)) / ((mx * mx + my * my + c1) * (vx + vy + c2)))
    return float(np.mean(np.stack(vals)))


def depth_stats(pred, gt, min_depth: float, max_depth: float):
    """(sums abs_rel, sq_rel, sq_err, sq_log as float64 [4], counts valid, d1, d2, d3 as int64 [4])."""
    p = np.asarray(pred, np.float32).ravel()
    g = np.asarray(gt, np.float32).ravel()
    ok = (g > 0) & (g <= np.float32(max_depth))
    g = g[ok].astype(np.float64)
    p = np.clip(p[ok], np.float32(min_depth), np.float32(max_depth)).astype(np.float64)
    d = p - g
    ratio = np.maximum(p / g, g / p)
    sums = np.array([np.sum(np.abs(d) / g), np.sum(d * d / g), np.sum(d * d), np.sum((np.log(p) - np.log(g)) ** 2)])
    counts = np.array([ok.sum(), (ratio < 1.25).sum(), (ratio < 1.25 ** 2).sum(), (ratio < 1.25 ** 3).sum()], np.int64)
    return sums, counts


def frame_words(C: int, sem_pred=None, sem_gt=None, pan_pred=None, pan_gt=None, is_thing=None, div: int = 1000,
                rgb_pred=None, rgb_gt=None, H: int = 0, W: int = 0, depth_pred=None, depth_gt=None,
                min_depth: float = 1e-3, max_depth: float = 80.0, words: Optional[np.ndarray] = None) -> np.ndarray:
    """One frame's statistics added to `words` (a fresh zero buffer when None), layout of include/pnr.h."""
    w = np.zeros(HEADER_WORDS + C * C + 4 * C, np.int64) if words is None else words.copy()
    f = w.view(np.float64)
    if sem_pred is not None:
        w[HEADER_WORDS:HEADER_WORDS + C * C] += confusion(sem_pred, sem_gt, C).ravel()
    if pan_pred is not None:
        r = pq_stats(pan_pred, pan_gt, C, is_thing, div)
        if r is None:
            w[OVERFLOW] += 1
        else:
            w[PQ_FRAMES] += 1
            base = HEADER_WORDS + C * C
            for k in range(3):
                w[base + k * C:base + (k + 1) * C] += r[k]
            f[base + 3 * C:base + 4 * C] += r[3]
    if rgb_pred is not None:
        f[PSNR_SUM] += psnr(rgb_pred, rgb_gt)
        w[PSNR_FRAMES] += 1
        if H * W:
            f[SSIM_SUM] += ssim(rgb_pred, rgb_gt, H, W)
            w[SSIM_FRAMES] += 1
    if depth_pred is not None:
        sums, counts = depth_stats(depth_pred, depth_gt, min_depth, max_depth)
        f[ABS_REL_SUM:SQ_LOG_SUM + 1] += sums
        w[DEPTH_VALID:DEPTH_DELTA3 + 1] += counts
    return w


def metrics(words: np.ndarray, C: int, is_thing=None) -> dict:
    """mIoU (mean over classes with a non-empty union), PQ / SQ / RQ (means over categories with TP + FP + FN > 0)."""
    w = np.asarray(words, np.int64)
    f = w.view(np.float64)
    out = {}
    conf = w[HEADER_WORDS:HEADER_WORDS + C * C].reshape(C, C).astype(np.float64)
    union = conf.sum(0) + conf.sum(1) - np.diag(conf)
    if union.sum() > 0:
        out["miou"] = float(np.mean(np.diag(conf)[union > 0] / union[union > 0]))
        out["pixel_acc"] = float(np.trace(conf) / conf.sum())
    base = HEADER_WORDS + C * C
    tp, fp, fn = (w[base + k * C:base + (k + 1) * C].astype(np.float64) for k in range(3))
    iou_sum = f[base + 3 * C:base + 4 * C]
    present = tp + fp + fn > 0
    if present.any():
        d = (tp + 0.5 * fp + 0.5 * fn)[present]
        out["pq"] = float(np.mean(iou_sum[present] / d))
        out["sq"] = float(np.mean(np.where(tp[present] > 0, iou_sum[present] / np.maximum(tp[present], 1), 0.0)))
        out["rq"] = float(np.mean(tp[present] / d))
    if w[PSNR_FRAMES]:
        out["psnr"] = f[PSNR_SUM] / w[PSNR_FRAMES]
    if w[SSIM_FRAMES]:
        out["ssim"] = f[SSIM_SUM] / w[SSIM_FRAMES]
    return out
