"""On-device evaluation of rendered frames (the reference's `run.py --type evaluate` with its lib/evaluators
`Evaluator`): semantic confusion matrix -> IoU / mIoU / pixel accuracy, panoptic quality (PQ / SQ / RQ), PSNR / SSIM and
depth error.  Every frame is accumulated by `pnr_eval_frame` into a small device statistics buffer; `summarize()` copies
that buffer to the host once.  Definitions and the buffer layout: include/pnr.h (pnr_eval_frame)."""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import numpy as np
import torch

from ... import _capi

HEADER_WORDS = 16
(OVERFLOW, PQ_FRAMES, PSNR_FRAMES, SSIM_FRAMES, DEPTH_VALID, DEPTH_DELTA1, DEPTH_DELTA2, DEPTH_DELTA3,
 PSNR_SUM, SSIM_SUM, ABS_REL_SUM, SQ_REL_SUM, SQ_ERR_SUM, SQ_LOG_SUM) = range(14)


def summarize_stats(words: np.ndarray, C: int, is_thing=None) -> Dict[str, object]:
    """The metrics of a statistics buffer read back as int64 words (layout: include/pnr.h)."""
    w = np.asarray(words, dtype=np.int64)
    f = w.view(np.float64)
    if w[OVERFLOW]:
        raise _capi.PnrError(f"evaluation: {int(w[OVERFLOW])} frame(s) had more than 1024 distinct panoptic segments "
                             "on one side; their panoptic quality was not computed")
    res: Dict[str, object] = {}
    if C > 0:
        conf = w[HEADER_WORDS:HEADER_WORDS + C * C].reshape(C, C)
        if conf.sum() > 0:
            tp = np.diag(conf).astype(np.float64)
            union = conf.sum(0) + conf.sum(1) - np.diag(conf)
            iou = np.where(union > 0, tp / np.maximum(union, 1), np.nan)
            res["iou"] = iou
            res["miou"] = float(np.nanmean(iou))
            res["pixel_acc"] = float(tp.sum() / conf.sum())
        if w[PQ_FRAMES] > 0:
            base = HEADER_WORDS + C * C
            tp, fp, fn = (w[base + k * C:base + (k + 1) * C].astype(np.float64) for k in range(3))
            iou_sum = f[base + 3 * C:base + 4 * C]
            denom = tp + 0.5 * fp + 0.5 * fn
            present = (tp + fp + fn) > 0
            with np.errstate(invalid="ignore", divide="ignore"):
                pq = np.where(present, iou_sum / np.where(present, denom, 1.0), np.nan)
                sq = np.where(tp > 0, iou_sum / np.maximum(tp, 1.0), np.where(present, 0.0, np.nan))
                rq = np.where(present, tp / np.where(present, denom, 1.0), np.nan)
            res["pq_per_class"], res["sq_per_class"], res["rq_per_class"] = pq, sq, rq
            res["tp"], res["fp"], res["fn"] = tp.astype(np.int64), fp.astype(np.int64), fn.astype(np.int64)
            thing = np.zeros(C, dtype=bool) if is_thing is None else np.asarray(is_thing, dtype=bool)
            for name, sel in (("", np.ones(C, dtype=bool)), ("_things", thing), ("_stuff", ~thing)):
                m = sel & present
                for k, v in (("pq", pq), ("sq", sq), ("rq", rq)):
                    res[k + name] = float(v[m].mean()) if m.any() else float("nan")
    if w[PSNR_FRAMES] > 0:
        res["psnr"] = float(f[PSNR_SUM] / w[PSNR_FRAMES])
    if w[SSIM_FRAMES] > 0:
        res["ssim"] = float(f[SSIM_SUM] / w[SSIM_FRAMES])
    n = int(w[DEPTH_VALID])
    if n > 0:
        res["depth"] = {"abs_rel": float(f[ABS_REL_SUM] / n), "sq_rel": float(f[SQ_REL_SUM] / n),
                        "rmse": float(np.sqrt(f[SQ_ERR_SUM] / n)), "rmse_log": float(np.sqrt(f[SQ_LOG_SUM] / n)),
                        "a1": w[DEPTH_DELTA1] / n, "a2": w[DEPTH_DELTA2] / n, "a3": w[DEPTH_DELTA3] / n, "n": n}
    return res


class Evaluator:
    """evaluate(output, batch) per frame, summarize() at the end, reset() to start over.

    output: a `Renderer.render` result on a CUDA device.  Its `panoptic` / `semantic` entries (from `fuse_panoptic`)
    are used when present; otherwise the semantic labels are the argmax of `semantic_map` (pnr_label_tiles).
    batch (ground truth, same device or host): `rgb` [R,3], `depth` [R] (<= 0: no depth), `semantic_gt` [R] int,
    `panoptic_gt` [R] int32 (category * label_divisor + instance).  Each metric family runs when its two inputs exist.
    cfg keys: num_classes, is_thing [C], label_divisor (1000), min_depth (1e-3), max_depth (cfg.far), H / W_img (SSIM
    when H * W_img equals the frame's ray count)."""

    def __init__(self, cfg, device=None):
        self.C = int(getattr(cfg, "num_classes", 0) or 0)
        if self.C > 64:
            raise ValueError(f"Evaluator: num_classes={self.C}; the semantic / panoptic statistics support C <= 64")
        thing = getattr(cfg, "is_thing", None)
        self.is_thing = None if thing is None else [int(bool(x)) for x in thing]
        if self.is_thing is not None and len(self.is_thing) != self.C:
            raise ValueError(f"Evaluator: is_thing has {len(self.is_thing)} entries for {self.C} classes")
        self.label_divisor = int(getattr(cfg, "label_divisor", 1000))
        self.min_depth = float(getattr(cfg, "min_depth", 1e-3))
        self.max_depth = float(getattr(cfg, "max_depth", getattr(cfg, "far", 80.0)))
        self.H, self.W = int(getattr(cfg, "H", 0) or 0), int(getattr(cfg, "W_img", 0) or 0)
        self.device = None if device is None else torch.device(device)
        self.stats: Optional[torch.Tensor] = None
        self._ws: Optional[torch.Tensor] = None
        self._thing_dev: Optional[torch.Tensor] = None

    def _buffers(self, dev: torch.device, R: int, pan: bool):
        if self.stats is None:
            self.device = dev
            n = int(_capi.lib().pnr_eval_stats_bytes(self.C))
            self.stats = torch.zeros(n // 8, dtype=torch.int64, device=dev)
        elif self.stats.device != dev:
            raise ValueError(f"Evaluator: statistics live on {self.stats.device}, frame on {dev}")
        need = int(_capi.lib().pnr_eval_workspace_bytes(R, self.C, self.label_divisor if pan else 0))
        if need == 0:
            raise ValueError(f"Evaluator: C={self.C}, label_divisor={self.label_divisor} out of range")
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=dev)
        if pan and self._thing_dev is None:
            if self.is_thing is None:
                raise ValueError("Evaluator: panoptic quality needs cfg.is_thing [num_classes]")
            self._thing_dev = torch.tensor(self.is_thing, dtype=torch.uint8, device=dev)

    def evaluate(self, output: Dict[str, torch.Tensor], batch: Dict[str, torch.Tensor]) -> None:
        ref = output.get("rgb_map", output.get("semantic_map", output.get("panoptic")))
        if ref is None:
            raise ValueError("Evaluator.evaluate: the output holds none of rgb_map / semantic_map / panoptic")
        if not ref.is_cuda:
            raise _capi.PnrError(f"Evaluator.evaluate: expected CUDA tensors, got {ref.device} - panopticnerf_b200 is "
                                 "GPU-only (no CPU fallback)")
        dev, R = ref.device, ref.shape[0]
        gt = lambda k, dt: None if batch.get(k) is None else batch[k].to(dev, dt).reshape(-1).contiguous()
        keep = []                                    # keeps every converted tensor alive until the launch is enqueued

        sem_pred = sem_gt = pan_pred = pan_gt = None
        if self.C > 0 and batch.get("semantic_gt") is not None:
            sem_gt = gt("semantic_gt", torch.int32)
            if "semantic" in output:
                sem_pred = output["semantic"].to(torch.int16).contiguous()
            elif output.get("semantic_map") is not None:
                sm = output["semantic_map"].to(torch.float32).contiguous()
                sem_pred = torch.empty(R, dtype=torch.int16, device=dev)
                with torch.cuda.device(dev):
                    _capi.check(_capi.lib().pnr_label_tiles(None, None, _capi.ptr(sm, name="semantic_map"), None, R,
                                                            sm.shape[1], 0, None, None, _capi.ptr(sem_pred), None,
                                                            _capi.stream_ptr()), "pnr_label_tiles")
                keep.append(sm)
            else:
                sem_gt = None
        if self.C > 0 and batch.get("panoptic_gt") is not None and "panoptic" in output:
            pan_pred = output["panoptic"].to(torch.int32).contiguous()
            pan_gt = gt("panoptic_gt", torch.int32)
        rgb_pred = rgb_gt = depth_pred = depth_gt = None
        if output.get("rgb_map") is not None and batch.get("rgb") is not None:
            rgb_pred = output["rgb_map"].to(torch.float32).contiguous()
            rgb_gt = batch["rgb"].to(dev, torch.float32).reshape(R, 3).contiguous()
        if output.get("depth_map") is not None and batch.get("depth") is not None:
            depth_pred = output["depth_map"].to(torch.float32).reshape(-1).contiguous()
            depth_gt = gt("depth", torch.float32)
        keep += [sem_pred, sem_gt, pan_pred, pan_gt, rgb_pred, rgb_gt, depth_pred, depth_gt]

        self._buffers(dev, R, pan_pred is not None)
        a = _capi.PnrEvalArgs()
        a.R, a.C = R, self.C
        a.H, a.W = (self.H, self.W) if (rgb_pred is not None and self.H * self.W == R) else (0, 0)
        p = _capi.ptr
        a.sem_pred, a.sem_gt = p(sem_pred, torch.int16, "semantic"), p(sem_gt, torch.int32, "semantic_gt")
        a.pan_pred, a.pan_gt = p(pan_pred, torch.int32, "panoptic"), p(pan_gt, torch.int32, "panoptic_gt")
        a.is_thing = p(self._thing_dev) if pan_pred is not None else None
        a.label_divisor = self.label_divisor
        a.rgb_pred, a.rgb_gt = p(rgb_pred, torch.float32, "rgb_map"), p(rgb_gt, torch.float32, "rgb")
        a.depth_pred, a.depth_gt = p(depth_pred, torch.float32, "depth_map"), p(depth_gt, torch.float32, "depth")
        a.min_depth, a.max_depth = self.min_depth, self.max_depth
        a.stats = p(self.stats)
        a.workspace, a.workspace_bytes = p(self._ws), self._ws.numel()
        with torch.cuda.device(dev):
            _capi.check(_capi.lib().pnr_eval_frame(C.byref(a), _capi.stream_ptr()), "pnr_eval_frame")

    def raw_stats(self) -> np.ndarray:
        """The statistics buffer on the host, as int64 words (one device-to-host copy)."""
        if self.stats is None:
            return np.zeros(int(_capi.lib().pnr_eval_stats_bytes(self.C)) // 8, dtype=np.int64)
        return self.stats.cpu().numpy()

    def summarize(self) -> Dict[str, object]:
        """iou [C] / miou (mean over classes with a non-empty union) / pixel_acc; pq / sq / rq overall, _things and
        _stuff (means over categories with TP + FP + FN > 0) and per class; psnr / ssim (means of the per-frame values);
        depth {abs_rel, sq_rel, rmse, rmse_log, a1, a2, a3, n} (pixel-weighted over all frames).  Raises PnrError when
        a frame had more panoptic segments than the kernels handle.  The statistics are kept (see reset())."""
        return summarize_stats(self.raw_stats(), self.C, self.is_thing)

    def reset(self) -> None:
        if self.stats is not None:
            self.stats.zero_()


def make_evaluator(cfg, device=None) -> Evaluator:
    return Evaluator(cfg, device)
