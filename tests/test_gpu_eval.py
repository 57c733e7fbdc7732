"""GPU: the evaluation kernels (pnr_eval_frame through `Evaluator`) against the float64 reference of
tests/reference_metrics.py on cfg2-sized frames (376 x 1408) of seeded blocky labels, with void and crowd regions and
predictions shifted so that many IoUs sit near 1/2.  Integer statistics must be equal, floating-point sums within
1e-9 (depth 1e-6: fp32 inputs); accumulation over frames is the sum of the frames; two runs are bit-identical."""
import numpy as np
import pytest
import torch

import panopticnerf_b200 as PN
import reference_metrics as RM
from panopticnerf_b200 import _capi

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
C_SEM = 45
IS_THING = [1 if 24 <= c < 34 else 0 for c in range(C_SEM)]
H, W = 376, 1408


def synthetic_frame(seed: int, H: int = H, W: int = W, instances: int = 500):
    """Blocks of 32 x 64 pixels, half of them things with an instance each (15 % instance 0 = crowd), the others a random
    stuff category; ~5 % of the blocks are
    GT void (id -1 or category 255).  The prediction shifts every block row by 20-23 pixels (IoU (64-s)/(64+s) ~ 1/2
    for an isolated block), relabels 2 % of the pixels with ids of the frame, and leaves a few pixels void."""
    g = np.random.default_rng(seed)
    by, bx = -(-H // 32), -(-W // 64)
    stuff = np.array([c for c in range(C_SEM) if not IS_THING[c]])
    thing = g.random((by, bx)) < 0.5
    cat = np.where(thing, g.integers(24, 34, (by, bx)), stuff[g.integers(0, len(stuff), (by, bx))])
    inst = np.where(thing, np.where(g.random((by, bx)) < 0.15, 0, g.integers(1, instances + 1, (by, bx))), 0)
    ids = cat * 1000 + inst
    ids = np.where(g.random((by, bx)) < 0.03, -1, ids)
    ids = np.where(g.random((by, bx)) < 0.02, 255 * 1000, ids)
    gt = np.repeat(np.repeat(ids, 32, 0), 64, 1)[:H, :W]
    pred = np.empty_like(gt)
    for r in range(by):
        s = int(g.integers(20, 24))
        rows = slice(r * 32, min(H, r * 32 + 32))
        pred[rows] = np.roll(gt[rows], s, axis=1)
    pred = np.where(pred == 255 * 1000, g.integers(0, C_SEM) * 1000, pred)
    noise = g.random((H, W)) < 0.02
    pool = np.unique(gt[gt >= 0])
    pred = np.where(noise, pool[g.integers(0, len(pool), (H, W))], pred)
    pred = np.where(g.random((H, W)) < 0.001, -1, pred)
    pan_gt, pan_pred = gt.ravel().astype(np.int32), pred.ravel().astype(np.int32)
    sem_gt = np.where(pan_gt >= 0, pan_gt // 1000, -1).astype(np.int32)
    sem_pred = np.where(pan_pred >= 0, pan_pred // 1000, -1).astype(np.int16)
    yy, xx = np.meshgrid(np.linspace(0, 1, H), np.linspace(0, 1, W), indexing="ij")
    base = np.stack([np.sin(7 * xx + seed) * 0.4 + 0.5, yy, (xx * yy + 0.1 * g.random((H, W)))], -1)
    rgb_gt = np.clip(base, 0, 1).reshape(-1, 3).astype(np.float32)
    rgb_pred = np.clip(rgb_gt + 0.05 * g.standard_normal(rgb_gt.shape), 0, 1).astype(np.float32)
    depth_gt = (g.random(H * W) * 100).astype(np.float32)
    depth_gt[g.random(H * W) < 0.1] = 0.0
    depth_pred = (depth_gt * (1 + 0.3 * g.standard_normal(H * W)) + 0.5).astype(np.float32)
    return dict(sem_pred=sem_pred, sem_gt=sem_gt, pan_pred=pan_pred, pan_gt=pan_gt, rgb_pred=rgb_pred, rgb_gt=rgb_gt,
                depth_pred=depth_pred, depth_gt=depth_gt)


def to_render_output(f):
    t = lambda k: torch.from_numpy(f[k]).to(DEV)
    out = {"semantic": t("sem_pred"), "panoptic": t("pan_pred"), "rgb_map": t("rgb_pred"), "depth_map": t("depth_pred")}
    batch = {"semantic_gt": t("sem_gt"), "panoptic_gt": t("pan_gt"), "rgb": t("rgb_gt"), "depth": t("depth_gt")}
    return out, batch


def make_eval(**kw):
    return PN.make_evaluator(PN.make_cfg("cfg2", num_classes=C_SEM, is_thing=IS_THING, **kw))


def reference_words(f, words=None, Hs=H, Ws=W):
    return RM.frame_words(C_SEM, f["sem_pred"], f["sem_gt"], f["pan_pred"], f["pan_gt"], IS_THING, 1000,
                          f["rgb_pred"], f["rgb_gt"], Hs, Ws, f["depth_pred"], f["depth_gt"], 1e-3, 80.0, words)


FLOAT_WORDS = [RM.PSNR_SUM, RM.SSIM_SUM] + list(range(RM.ABS_REL_SUM, RM.SQ_LOG_SUM + 1))


def assert_words_match(got, ref):
    iou0 = RM.HEADER_WORDS + C_SEM * C_SEM + 3 * C_SEM
    fl = np.zeros(len(ref), bool)
    fl[FLOAT_WORDS] = True
    fl[iou0:iou0 + C_SEM] = True
    assert np.array_equal(got[~fl], ref[~fl]), np.nonzero(got[~fl] != ref[~fl])
    gf, rf = got.view(np.float64), ref.view(np.float64)
    for i in np.nonzero(fl)[0]:
        tol = 1e-6 if RM.ABS_REL_SUM <= i <= RM.SQ_LOG_SUM else 1e-9
        assert abs(gf[i] - rf[i]) <= tol * max(1.0, abs(rf[i])), (i, gf[i], rf[i])


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_single_frame_matches_reference(seed):
    f = synthetic_frame(seed)
    ev = make_eval()
    ev.evaluate(*to_render_output(f))
    got, ref = ev.raw_stats(), reference_words(f)
    assert ref[RM.OVERFLOW] == 0 and ref[RM.PQ_FRAMES] == 1
    base = RM.HEADER_WORDS + C_SEM * C_SEM
    assert ref[base:base + C_SEM].sum() > 20 and ref[base + C_SEM:base + 3 * C_SEM].sum() > 20   # TPs, FPs and FNs
    assert_words_match(got, ref)
    s, m = ev.summarize(), RM.metrics(ref, C_SEM)
    for k in ("miou", "pixel_acc", "pq", "sq", "rq", "psnr", "ssim"):
        assert abs(s[k] - m[k]) <= 1e-9 * max(1.0, abs(m[k])), k
    assert {"pq_things", "pq_stuff", "depth"} <= set(s) and s["depth"]["n"] == ref[RM.DEPTH_VALID]


def test_iou_near_one_half_is_decided_exactly():
    """Isolated thing blocks shifted by s pixels in 64: IoU (64-s)/(64+s) crosses 1/2 between s = 21 and 22."""
    cases = [20, 21, 22, 23, 21, 22, 0, 32]
    base = np.zeros((64, 128 * len(cases)), np.int32)
    pred = np.zeros_like(base)
    for k, s in enumerate(cases):
        base[16:48, 128 * k + 32:128 * k + 96] = 25 * 1000 + k + 1
        pred[16:48, 128 * k + 32 + s:128 * k + 96 + s] = 25 * 1000 + k + 1
    f = {"pan_pred": pred.ravel(), "pan_gt": base.ravel()}
    ev = make_eval()
    ev.evaluate({"panoptic": torch.from_numpy(f["pan_pred"]).to(DEV)}, {"panoptic_gt": torch.from_numpy(f["pan_gt"]).to(DEV)})
    ref = RM.frame_words(C_SEM, pan_pred=f["pan_pred"], pan_gt=f["pan_gt"], is_thing=IS_THING)
    base_w = RM.HEADER_WORDS + C_SEM * C_SEM
    assert ref[base_w + 25] == 4                      # s = 20, 21, 21, 0 match, 22, 22, 23, 32 do not
    assert_words_match(ev.raw_stats(), ref)


def test_accumulation_is_the_sum_of_frames_and_bit_reproducible():
    frames = [synthetic_frame(10 + i) for i in range(3)]
    singles = []
    for f in frames:
        ev = make_eval()
        ev.evaluate(*to_render_output(f))
        singles.append(ev.raw_stats())
    runs = []
    for _ in range(2):
        ev = make_eval()
        for f in frames:
            ev.evaluate(*to_render_output(f))
        runs.append(ev.raw_stats())
    assert np.array_equal(runs[0], runs[1])
    acc = np.zeros_like(singles[0])
    for s in singles:
        af, sf = acc.view(np.float64), s.view(np.float64)
        ints = np.ones(len(acc), bool)
        iou0 = RM.HEADER_WORDS + C_SEM * C_SEM + 3 * C_SEM
        ints[FLOAT_WORDS] = False
        ints[iou0:iou0 + C_SEM] = False
        acc[ints] += s[ints]
        af[~ints] += sf[~ints]
    assert np.array_equal(runs[0], acc)
    ref = None
    for f in frames:
        ref = reference_words(f, ref)
    assert_words_match(runs[0], ref)
    ev.reset()
    assert not ev.raw_stats().any()


def test_segment_overflow_is_raised_by_summarize():
    ids = (25 * 1000 + 1 + np.arange(64 * 40) % 999).astype(np.int32)       # 999 thing instances ...
    ids[:1100] = 26 * 1000 + 1 + np.arange(1100) % 999                       # ... plus up to 999 of another thing
    ev = make_eval()
    t = torch.from_numpy(ids).to(DEV)
    ev.evaluate({"panoptic": t, "rgb_map": torch.zeros(len(ids), 3, device=DEV)},
                {"panoptic_gt": t, "rgb": torch.zeros(len(ids), 3, device=DEV)})
    w = ev.raw_stats()
    assert w[RM.OVERFLOW] == 1 and w[RM.PQ_FRAMES] == 0 and w[RM.PSNR_FRAMES] == 1
    with pytest.raises(_capi.PnrError, match="1024"):
        ev.summarize()
    ev.reset()
    ok = torch.from_numpy(ids[:1024].copy()).to(DEV)
    ev.evaluate({"panoptic": ok}, {"panoptic_gt": ok})
    assert ev.summarize()["pq"] == 1.0


def test_end_to_end_render_fuse_evaluate():
    """A cfg3-shaped strip through Renderer.render -> fuse_panoptic -> Evaluator, held to the reference metrics of the
    GPU's own labels (near-tie argmaxes may legitimately differ from a CPU render; the evaluation must not)."""
    from panopticnerf_b200 import synthetic as S
    from panopticnerf_b200.lib.visualizers import fuse_panoptic
    rows = 24
    cfg = PN.make_cfg("cfg3")
    net = S.init_network_weights(PN.make_network(cfg)).to(DEV)
    batch = S.make_batch(cfg, row0=180, rows=rows)
    out = PN.make_renderer(cfg, net).render({k: v.to(DEV) for k, v in batch.items()})
    inst_class = torch.arange(cfg.num_instances) % C_SEM
    out.update(fuse_panoptic(out, IS_THING, inst_class))
    R = out["rgb_map"].shape[0]
    f = synthetic_frame(7, H=rows, W=cfg.W_img)
    gt = {"semantic_gt": torch.from_numpy(f["sem_gt"]).to(DEV), "panoptic_gt": torch.from_numpy(f["pan_gt"]).to(DEV),
          "rgb": torch.from_numpy(f["rgb_gt"]).to(DEV), "depth": torch.from_numpy(f["depth_gt"]).to(DEV)}
    ev = PN.make_evaluator(PN.make_cfg("cfg3", H=rows, is_thing=IS_THING))
    ev.evaluate(out, gt)
    mine = {"sem_pred": out["semantic"].cpu().numpy(), "pan_pred": out["panoptic"].cpu().numpy(),
            "rgb_pred": out["rgb_map"].cpu().numpy(), "depth_pred": out["depth_map"].cpu().numpy()}
    ref = reference_words({**f, **mine}, Hs=rows, Ws=cfg.W_img)
    ref_metrics = RM.metrics(ref, C_SEM)
    assert R == rows * cfg.W_img and ref[RM.SSIM_FRAMES] == 1
    assert_words_match(ev.raw_stats(), ref)
    s = ev.summarize()
    for k in ("miou", "pq", "psnr", "ssim"):
        assert abs(s[k] - ref_metrics[k]) <= 1e-9 * max(1.0, abs(ref_metrics[k])), k
    # without fuse_panoptic's labels: semantic labels from the argmax kernel (pnr_label_tiles), no PQ
    ev2 = PN.make_evaluator(PN.make_cfg("cfg3", H=rows, is_thing=IS_THING))
    ev2.evaluate({k: v for k, v in out.items() if k not in ("semantic", "panoptic")}, gt)
    w2 = ev2.raw_stats()
    conf = slice(RM.HEADER_WORDS, RM.HEADER_WORDS + C_SEM * C_SEM)
    assert np.array_equal(w2[conf], ref[conf]) and w2[RM.PQ_FRAMES] == 0
