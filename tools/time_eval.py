"""Time pnr_eval_frame (csrc/eval_kernels.cu) on a cfg2 frame (376 x 1408 rays, C = 45, label_divisor 1000), per metric
family and all together: python tools/time_eval.py [frames].  CUDA events around `frames` back-to-back calls after a
warm-up; the inputs (~20 MB) stay in L2 between frames, as they would when a frame is evaluated right after its render.
Prints the device time per frame, the algorithmic bytes of the family over that time, and the card's name and power
limit read in the same run."""
import ctypes as C
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from panopticnerf_b200 import _capi  # noqa: E402

DEV = "cuda:0"
FRAMES = int(sys.argv[1]) if len(sys.argv) > 1 else 500
H, W, NC, DIV = 376, 1408, 45, 1000
R = H * W


def frame(seed=0):
    g = torch.Generator().manual_seed(seed)
    by, bx = H // 8 + 1, W // 16 + 1
    cat = torch.randint(0, NC, (by, bx), generator=g)
    inst = torch.randint(0, 8, (by, bx), generator=g)
    ids = (cat * DIV + inst).repeat_interleave(8, 0).repeat_interleave(16, 1)[:H, :W].reshape(-1)
    pred = torch.where(torch.rand(R, generator=g) < 0.05, ids[torch.randperm(R, generator=g)], ids.roll(5))
    rgb = torch.rand(R, 3, generator=g)
    depth = torch.rand(R, generator=g) * 80
    t = lambda x, dt: x.to(DEV, dt).contiguous()
    return dict(sem_pred=t(pred // DIV, torch.int16), sem_gt=t(ids // DIV, torch.int32), pan_pred=t(pred, torch.int32),
                pan_gt=t(ids, torch.int32), rgb_pred=t((rgb + 0.05 * torch.randn(R, 3, generator=g)).clamp(0, 1), torch.float32),
                rgb_gt=t(rgb, torch.float32), depth_pred=t(depth * 1.1, torch.float32), depth_gt=t(depth, torch.float32))


FAMILIES = {   # name -> (input keys, SSIM, algorithmic bytes per frame: every input read once)
    "semantic": (("sem_pred", "sem_gt"), False, R * (2 + 4)),
    # ids read by the mark and histogram passes; the per-frame clear of the key flags and the 1024 x 1025 joint
    # histogram; the flag scan (read + write)
    "panoptic": (("pan_pred", "pan_gt"), False, R * 8 * 2 + (2 * 4 * NC * DIV + 4 * 1024 * 1025) + 2 * 2 * 4 * NC * DIV),
    "psnr": (("rgb_pred", "rgb_gt"), False, R * 24),
    "psnr+ssim": (("rgb_pred", "rgb_gt"), True, R * 24 * 2),
    "depth": (("depth_pred", "depth_gt"), False, R * 8),
}
FAMILIES["all"] = (sum((v[0] for v in FAMILIES.values()), ()), True,
                   sum(v[2] for k, v in FAMILIES.items() if k != "psnr"))


def main():
    L = _capi.lib()
    f = frame()
    thing = torch.tensor([1 if 24 <= c < 34 else 0 for c in range(NC)], dtype=torch.uint8, device=DEV)
    stats = torch.zeros(L.pnr_eval_stats_bytes(NC) // 8, dtype=torch.int64, device=DEV)
    ws = torch.empty(L.pnr_eval_workspace_bytes(R, NC, DIV), dtype=torch.uint8, device=DEV)
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print(f"card: {torch.cuda.get_device_name(0)} | nvidia-smi: {smi[0] if smi else 'n/a'}")
    print(f"frame: {H} x {W} = {R} rays, C = {NC}, label_divisor {DIV}; {FRAMES} frames per family after 20 warm-up")
    for name, (keys, ssim, nbytes) in FAMILIES.items():
        a = _capi.PnrEvalArgs()
        a.R, a.C, a.label_divisor, a.min_depth, a.max_depth = R, NC, DIV, 1e-3, 80.0
        for k in keys:
            setattr(a, k, f[k].data_ptr())
        a.H, a.W = (H, W) if ssim else (0, 0)
        a.is_thing = thing.data_ptr()
        a.stats, a.workspace, a.workspace_bytes = stats.data_ptr(), ws.data_ptr(), ws.numel()
        s = _capi.stream_ptr()
        for _ in range(20):
            _capi.check(L.pnr_eval_frame(C.byref(a), s), "pnr_eval_frame")
        torch.cuda.synchronize()
        L.pnr_launch_count(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(FRAMES):
            L.pnr_eval_frame(C.byref(a), s)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / FRAMES
        launches = L.pnr_launch_count(1) / FRAMES
        print(f"{name:10s} {ms * 1e3:8.1f} us/frame  {launches:.0f} launches  {nbytes / 1e6:6.1f} MB  "
              f"{nbytes / (ms * 1e-3) / 1e12:6.3f} TB/s ({100 * nbytes / (ms * 1e-3) / 7.7e12:5.2f} % of 7.7 TB/s)")


if __name__ == "__main__":
    main()
