"""bench.py — rays/sec of the render hot path on synthetic KITTI-360-shaped rays (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--precision fp16x3|bf16x3|fp16|bf16]
                    [--config cfg2|cfg3|cfg5] [--scaling weak|strong] [--gather maps|labels|none]
                    [--dump-outputs DIR]

A step = one pass of the hot path over one frame of rays (default: config 2 of BASELINE.json, 376 x 1408 rays,
64 samples/ray, 8 x 256 MLP, rgb + sigma, 64 bounding primitives) through the public API - Renderer.render, i.e.
ONE pnr_render_fused call: scene near/far -> ray/box intersection -> stratified depths + ids -> fused PE + MLP
(tcgen05) -> alpha compositing.
  --scaling weak   (default; config 4): every rank renders its own frame, one NCCL all-gather of the rendered tiles
                   (libpnr's pnr_allgather_outputs) rebuilds all of them on every rank inside the step;
  --scaling strong : ONE frame is ray-sharded over the ranks (config 5's layout), same gather;
  --gather labels  : the gathered tile is rgb8 | depth | semantic label | instance label (pnr_label_tiles) instead of
                   the fp32 rgb | depth | acc maps.

value  : rays/s with inputs resident in HBM (CUDA events per step, L2 flushed between steps, max over ranks)
e2e    : the same through Renderer.render from pinned HOST rays, H2D + D2H inside the timed region
roofline: dominant kernel (fused MLP) algorithmic FLOP/s vs the measured dense bf16 tensor peak
cpu_baseline / --impl reference: the CPU oracle (port of the spec; the reference source is not in the
         mount) timed on the box's host cores on a bounded strip of the same frame.

--dump-outputs DIR: after the timed steps, rank 0 writes every tensor the last timed step returned (Renderer.render's
dict, plus the gathered tiles as gathered_<name> when there is a gather) as DIR/<name>.npy, float32 (float64 stays
float64; integer and mask outputs are converted exactly).  The inputs are seeded, so two builds run with the same
arguments can be compared file by file.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

# stdout carries exactly one JSON line.  Libraries write to it too (NCCL prints its version banner there at
# NCCL_DEBUG=VERSION/WARN), so file descriptor 1 is pointed at stderr for the whole run and the JSON line is
# written to a saved copy of the real stdout.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line: dict) -> None:
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

UNIT = "rays/s"
FALLBACK_PEAKS = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}
WORKLOADS = {
    "cfg2": "cfg2: KITTI-360 perspective 376x1408, 64 samples/ray, 8x256 MLP, rgb+sigma, 64 boxes",
    "cfg3": "cfg3: the cfg2 frame + semantic (45) and instance (64) heads, coarse 64 + fine 128 samples/ray (fine pass: 192)",
    "cfg5": "cfg5: PanopticNeRF-360 equirectangular 2048x1024, 192 samples/ray, 8x256 MLP + semantic (45) / instance (64) heads",
}


def metric_name(cfg) -> str:
    if cfg.preset == "cfg2":
        return "rays/sec at 376x1408x64 samples (8x256 MLP, rgb+sigma)"
    n = f"{cfg.N_samples}" + (f"+{cfg.N_importance}" if cfg.N_importance else "")
    return f"rays/sec at {cfg.H}x{cfg.W_img}x{n} samples (8x256 MLP + semantic/instance heads)"


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        d["_src"] = "measured (MEASURED_PEAKS.json)"
        return d
    d = dict(FALLBACK_PEAKS)
    d["_src"] = "fallback (B200_PROFILING.md)"
    return d


def flops_per_sample(cfg) -> int:
    D, W = cfg.D, cfg.W
    Ex, Ed = 3 + 6 * cfg.xyz_res, 3 + 6 * cfg.view_res
    mac = Ex * W + (D - 2) * W * W + (W + Ex) * W + W + W * W + (W + Ed) * (W // 2) + (W // 2) * 3
    if cfg.num_classes:
        mac += W * (W // 2) + (W // 2) * cfg.num_classes
    if cfg.num_instances:
        mac += W * (W // 2) + (W // 2) * cfg.num_instances
    return 2 * mac


def host_threads() -> int:
    """Threads the CPU legs may really use: the scheduler affinity of this process, capped by the cgroup CPU quota
    (os.cpu_count() counts the machine's cores, not this lease's - VERDICT r1: 381 vs 2 480 rays/s at '128 cores')."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = Path(path).read_text().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, math.ceil(int(txt[0]) / int(txt[1]))))
            else:
                q = int(txt[0])
                per = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read_text())
                if q > 0:
                    n = min(n, max(1, math.ceil(q / per)))
            break
        except Exception:
            continue
    return max(1, n)


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md).  Uses NVML in-process
    (nvidia_ml_py) - spawning nvidia-smi every 100 ms perturbs the GPU - with nvidia-smi as the fallback.
    Created (NVML initialised) before the warm-up so no first-call cost lands in the timed steps."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, index: int):
        self.index, self.sm, self.mx, self.reasons = index, [], [], set()
        self._stop, self._t, self.nv, self.h = threading.Event(), None, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and vis.split(",")[index].isdigit() else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.nv = pynvml
            self._sample()
        except Exception:
            self.nv = None

    def _sample(self):
        nv = self.nv
        if nv is not None:
            self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
            self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)))
            fn = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            mask = int(fn(self.h))
            self.reasons |= {k for k, b in self.BITS.items() if mask & b}
        else:
            o = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
            r = [x.strip() for x in o.strip().split(",")]
            if len(r) >= 7:
                self.sm.append(float(r[0])); self.mx.append(float(r[1]))
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                self.reasons |= {n for n, v in zip(names, r[3:7]) if v.lower().startswith("active")}

    def start(self):
        self.sm, self.mx, self.reasons = [], [], set()

        def run():
            while not self._stop.is_set():
                try:
                    self._sample()
                except Exception:
                    pass
                self._stop.wait(0.1 if self.nv is not None else 0.5)
        self._t = threading.Thread(target=run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None,
                "sm_max_mhz": max(self.mx) if self.mx else None, "reasons": sorted(self.reasons),
                "samples": len(self.sm), "source": "nvml" if self.nv is not None else "nvidia-smi"}


# ------------------------------------------------------------------------------------------------ CPU legs
class CpuOracle:
    """The CPU oracle (port of the specification; the reference source is not in the mount) on a strip of the frame."""

    def __init__(self, cfg, threads: int):
        from oracle import reference_renderer as O
        from panopticnerf_b200 import synthetic as S
        torch.set_num_threads(threads)
        self.cfg, self.S, self.threads = cfg, S, threads
        self.net = S.init_network_weights(O.make_network(cfg))
        self.ren = O.make_renderer(cfg, self.net)

    def strip(self, rows: int):
        return self.S.make_batch(self.cfg, row0=(self.cfg.H - rows) // 2, rows=rows, num_boxes=64)

    def run(self, rows: int):
        batch = self.strip(rows)
        t0 = time.perf_counter()
        out = self.ren.render(batch)
        dt = time.perf_counter() - t0
        assert torch.isfinite(out["rgb_map"]).all()
        return batch["rays"].shape[0] / dt, dt, batch, out

    def pick_rows(self, seconds_per_step: float, max_rows: int = 16) -> int:
        """Strip height whose render takes about `seconds_per_step` (BASELINE.md section 4 asks for 16 rows; fewer
        when the host is too slow for the run to end within a few minutes).  The probe doubles as thread warm-up."""
        self.run(1)
        rate, _, _, _ = self.run(1)
        return int(max(1, min(max_rows, round(rate * seconds_per_step / self.cfg.W_img))))


def run_reference(args, cfg, rank, world):
    """--impl reference: the reference's own CPU PyTorch path.  Its source is not in the mount
    (SURVEY.md section 0), so this is the oracle port of the specification, on the host threads this process may
    use, each step a bounded strip of the same frame; rank 0 alone runs it."""
    if rank != 0:
        return
    threads = host_threads()
    orc = CpuOracle(cfg, threads)
    budget = 240.0 / max(args.steps + args.warmup, 1)              # the whole run ends within a few minutes
    rows = args.ref_rows or orc.pick_rows(min(budget, 12.0))
    for _ in range(max(args.warmup - 2, 0) if not args.ref_rows else args.warmup):
        orc.run(rows)
    secs = []
    for _ in range(args.steps):
        _, dt, _, out = orc.run(rows)
        secs.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    rays = rows * cfg.W_img
    value = rays * len(secs) / sum(secs)
    sample = (f"{rows}-row strip ({rays} rays) of the {cfg.H}x{cfg.W_img} frame per step; median step "
              f"{statistics.median(secs):.2f} s, {threads} threads")
    emit({
        "impl": "reference", "metric": metric_name(cfg), "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(secs) / len(secs),
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOADS[cfg.preset], "sample": sample,
                   "note": "CPU oracle port; reference source unavailable in /root/reference"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample,
                         "median_rays_per_s": rays / statistics.median(secs), "os_cpu_count": os.cpu_count()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


def parity_on_strip(ref_out, gpu_out, far: float) -> dict:
    """Measured end-to-end max error of the GPU render against the CPU oracle on the cpu_baseline strip, under the
    strict per-quantity floors of SURVEY 8(a) and under the end-to-end floors of tests/util.py (the ones the
    end-to-end tests assert): |x-y| / max(|y|, floor), to be compared with 1e-4."""
    strict = {"rgb_map": 1e-2, "acc_map": 1e-3, "weights": 1e-3, "depth_map": 1e-2 * far}
    relaxed = {"rgb_map": 1e-1, "acc_map": 1e-1, "weights": 1e-1, "depth_map": 1e-2 * far}
    rep = {}
    for k in strict:
        x, y = gpu_out[k].detach().double().cpu(), ref_out[k].double()
        err = (x - y).abs()
        rep[k] = {"max_abs": float(err.max()),
                  "rel_strict_floor": float((err / torch.clamp(y.abs(), min=strict[k])).max()),
                  "rel_e2e_floor": float((err / torch.clamp(y.abs(), min=relaxed[k])).max())}
    rep["masks_and_indices_equal"] = bool(torch.equal(gpu_out["hit_mask"].cpu(), ref_out["hit_mask"]) and
                                          torch.equal(gpu_out["box_id"].cpu(), ref_out["box_id"]) and
                                          torch.equal(gpu_out["z_vals"].cpu(), ref_out["z_vals"]))
    rep["tolerance"] = 1e-4
    return rep


DUMP_BUDGET = 60 << 20      # bytes of array data under --dump-outputs; the .npy headers add ~128 bytes per file


def dump_outputs(dirname: str, arrays: dict) -> None:
    """Write each tensor of `arrays` as <dirname>/<name>.npy: float64 stays float64, everything else becomes float32
    (exact for the integer ids, labels and masks).  When the whole set exceeds DUMP_BUDGET, every tensor keeps the same
    fixed, seeded sample of its rows (first dimension, ascending), so a file holds the same rays in every run."""
    import numpy as np
    arrays = {k: v.detach() for k, v in arrays.items() if torch.is_tensor(v)}
    total = sum(v.numel() * (8 if v.dtype == torch.float64 else 4) for v in arrays.values())
    keep = min(1.0, DUMP_BUDGET / total) if total else 1.0
    rows = {}
    d = Path(dirname)
    d.mkdir(parents=True, exist_ok=True)
    for name, t in sorted(arrays.items()):
        if keep < 1.0 and t.dim() > 0:
            n = t.shape[0]
            if n not in rows:
                rows[n] = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:int(n * keep)].sort().values
            t = t[rows[n].to(t.device)]
        t = t.cpu().to(torch.float64 if t.dtype == torch.float64 else torch.float32)
        np.save(d / f"{name}.npy", t.numpy())


# ------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="fp16x3", choices=["fp16x3", "bf16x3", "fp16", "bf16"])
    ap.add_argument("--config", default="cfg2", choices=["cfg2", "cfg3", "cfg5"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--gather", default="maps", choices=["maps", "labels", "none"])
    ap.add_argument("--ref-rows", type=int, default=0, help="strip height per CPU step (0 = sized to the time budget, <= 16)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-fast-mode", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the cfg3 block under 'extra'")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (at most 64 MB: a fixed, seeded sample "
                         "of the rays when the frame's outputs are larger)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    import panopticnerf_b200 as PN
    from panopticnerf_b200 import _capi, parallel, synthetic as S

    cfg = PN.make_cfg(args.config, precision=args.precision)
    if args.impl == "reference":
        run_reference(args, cfg, rank, world)
        return

    assert torch.cuda.is_available(), "bench.py (our arm) needs a GPU; there is no CPU path"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- inputs, resident in HBM.  weak: one frame per rank; strong: one frame, contiguous ray shards
    net = S.init_network_weights(PN.make_network(cfg)).to(dev)
    ren = PN.make_renderer(cfg, net)
    frame = S.make_batch(cfg, seed=rank if args.scaling == "weak" else 0, num_boxes=64)
    R_frame = frame["rays"].shape[0]
    if args.scaling == "strong" and world > 1:
        cpu_batch = parallel.shard_batch(frame, rank, world)
        R_total = R_frame                                       # rays all ranks render per step
    else:
        cpu_batch = frame
        R_total = R_frame * world
    batch = {k: v.to(dev) for k, v in cpu_batch.items()}
    R = batch["rays"].shape[0]
    N = cfg.N_samples
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)     # > 126 MB L2
    tg = parallel.TileGather(dev) if (dist is not None and args.gather != "none") else None
    R_gather = R_frame if args.scaling == "strong" else R * world       # rows of the gathered image(s)
    # weak scaling gathers `world` whole frames: rank r's tile = its frame (per = R rays each)

    def gather(out):
        if tg is None:
            return None
        return tg.gather_labels(out, R_gather) if args.gather == "labels" else tg.gather_maps(out, R_gather)

    def step():
        out = ren.render(batch)
        return out, gather(out)

    L = _capi.lib()
    sampler = ClockSampler(local_rank)
    out = gathered = None
    for _ in range(args.warmup):
        out, gathered = step()      # bound like in the timed loop: the previous step's outputs stay alive while the
                                    # next ones are allocated, so the caching allocator reaches its steady state here
                                    # (otherwise the 2nd timed step pays a cudaMalloc: 94 / 224 ms outliers, r2 logs)
    barrier()
    sampler.start()
    L.pnr_launch_count(1)
    evs = []
    barrier()
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out, gathered = step()
        b.record()
        evs.append((a, b))
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = int(L.pnr_launch_count(0))
    step_ms = [a.elapsed_time(b) for a, b in evs]
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    value = R_total * args.steps / (total_ms / 1e3)
    assert torch.isfinite(out["rgb_map"]).all()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {**out, **{f"gathered_{k}": v for k, v in (gathered or {}).items()}})
    gather_bytes = None
    if gathered is not None:
        gather_bytes = int(gathered["bytes_per_rank"]) if args.gather == "labels" else 20 * math.ceil(R_gather / world)

    # ---------------- dominant kernel: fused MLP, timed alone on the same inputs (events on torch's stream).
    # With a fine pass the fine launch (N + Ni samples, heads) is the dominant one.
    z = out["z_vals"]
    Nz = z.shape[1]
    # (the stand-alone launch materialises raw [R_m, Nz, 4+C+K]: a ray subset when that would exceed ~2 GB - a cfg5
    #  frame's raw is 170 GB - still hundreds of tiles per SM)
    raw_per_ray = Nz * (4 + cfg.num_classes + cfg.num_instances) * 4
    R_m = R if R * raw_per_ray <= (4 << 30) else max(1, (2 << 30) // raw_per_ray)
    m_rays, m_z = batch["rays"][:R_m].contiguous(), z[:R_m].contiguous()
    mlp_ms = []
    for i in range(3 + min(args.steps, 10)):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        net.forward_rays(m_rays, m_z)
        b.record()
        torch.cuda.synchronize()
        if i >= 3:
            mlp_ms.append(a.elapsed_time(b))
    clocks = sampler.stop()
    mlp_t = sum(mlp_ms) / len(mlp_ms) * (R / R_m)          # scaled to the rank's whole share when a subset was timed
    pk = peaks()
    alg_flop = flops_per_sample(cfg) * R * Nz
    achieved = alg_flop / (mlp_t / 1e3) / 1e12
    peak = float(pk["bf16_tflops_sustained"])
    traffic, traffic_src = None, None
    prof = ROOT / "profiles" / "mlp_ncu_summary.json"
    if prof.exists() and args.config == "cfg2" and R == R_frame:
        try:
            ent = json.loads(prof.read_text()).get(args.precision, {})
            traffic, traffic_src = ent.get("dram_bytes_per_launch"), ent.get("source")
        except Exception:
            traffic = None
    mlp_per_step = mlp_t * (1.0 + (N / Nz if cfg.N_importance else 0.0))    # coarse launch scaled by its samples
    roofline = {"bound": "tensor", "kernel": "mlp_fused_kernel", "achieved": achieved, "peak": peak,
                "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": traffic_src or "not captured for this configuration",
                "peak_source": f"bf16_tflops_sustained, {pk['_src']}", "kernel_ms": mlp_t,
                "kernel_share_of_step": min(1.0, mlp_per_step / (total_ms / args.steps)),
                "alg_flop_per_launch": alg_flop, "samples_per_launch": R * Nz,
                "timed_on_rays": R_m,
                "passes": 3 if args.precision.endswith("x3") else 1,
                "executed_flop_per_launch_one_pass": (flops_per_sample(cfg) - 2 * cfg.W * cfg.W) * R * Nz,
                "note": "achieved = the reference network's algorithmic FLOPs (true layer shapes, 1 pass) / time; "
                        "the kernel executes 2*W*W fewer per sample (feature_linear is folded into the view "
                        "layer at weight load, exact algebra) and the x3 modes issue 3 tensor-core passes per "
                        "product, so tensor-pipe busy is ~2.7x this fraction (bound of the fraction: 0.375)"}

    # ---------------- e2e: public API from pinned host rays, H2D + D2H inside the timed region
    host_rays = cpu_batch["rays"].pin_memory()
    dev_rays = torch.empty_like(batch["rays"])
    e2e_batch = dict(batch)
    if args.gather == "labels" and tg is not None:
        d2h_rows, d2h_width = R_gather, None
    else:
        d2h_rows, d2h_width = (R_gather if tg is not None else R), 5
    host_out = {}

    def e2e_step():
        dev_rays.copy_(host_rays, non_blocking=True)
        e2e_batch["rays"] = dev_rays
        o = ren.render(e2e_batch)
        g = gather(o)
        if g is not None and args.gather == "labels":
            res = {k: v for k, v in g.items() if torch.is_tensor(v)}
        else:
            src = g if g is not None else o
            res = {"packed": torch.cat([src["rgb_map"], src["depth_map"][:, None], src["acc_map"][:, None]], 1)}
        for k, v in res.items():
            if k not in host_out:
                host_out[k] = torch.empty(v.shape, dtype=v.dtype).pin_memory()
            host_out[k].copy_(v, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    for _ in range(2):
        e2e_step()
    barrier()
    e_evs = []
    for _ in range(args.steps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        e2e_step()
        b.record()
        e_evs.append((a, b))
    barrier()
    e_ms = torch.tensor([sum(a.elapsed_time(b) for a, b in e_evs)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(e_ms, op=dist.ReduceOp.MAX)
    e2e_value = R_total * args.steps / (float(e_ms.item()) / 1e3)
    e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": host_rays.numel() * 4,
           "d2h_bytes_per_step": sum(v.numel() * v.element_size() for v in host_out.values())}

    # ---------------- fast (1-pass) mode, reported beside the headline; not within the parity tolerance
    fast = None
    if not args.no_fast_mode and args.precision.endswith("x3") and args.config == "cfg2":
        fprec = args.precision[:-2]
        fcfg = PN.make_cfg(args.config, precision=fprec)
        fnet = PN.make_network(fcfg)
        fnet.load_state_dict(net.state_dict())
        fnet = fnet.to(dev)
        ts = []
        for i in range(3 + min(args.steps, 10)):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fnet.forward_rays(batch["rays"], z)
            b.record()
            torch.cuda.synchronize()
            if i >= 3:
                ts.append(a.elapsed_time(b))
        ft = sum(ts) / len(ts)
        fast = {"precision": fprec, "kernel_ms": ft, "achieved_tflops": alg_flop / (ft / 1e3) / 1e12,
                "frac": alg_flop / (ft / 1e3) / 1e12 / peak, "mlp_rays_per_s": R / (ft / 1e3),
                "note": "1 tensor-core pass; ~1e-3 (fp16) / ~1e-2 (bf16) relative error: outside the 1e-4 tolerance"}
        del fnet

    # ---------------- extra: config 3 (heads, coarse + fine) as a measured, first-class frame (N = 1 only)
    extra = None
    if world == 1 and args.config == "cfg2" and not args.no_extra:
        c3 = PN.make_cfg("cfg3", precision=args.precision)
        n3 = S.init_network_weights(PN.make_network(c3)).to(dev)
        r3 = PN.make_renderer(c3, n3)
        b3 = {k: v.to(dev) for k, v in S.make_batch(c3, num_boxes=64).items()}
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        base_mem = torch.cuda.memory_allocated(dev)
        ts = []
        for i in range(2 + 3):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            o3 = r3.render(b3)
            b.record()
            torch.cuda.synchronize()
            if i >= 2:
                ts.append(a.elapsed_time(b))
        ms3 = statistics.median(ts)
        flop3 = R_frame * (c3.N_samples + c3.N_samples + c3.N_importance) * flops_per_sample(c3)
        extra = {"cfg3": {"workload": WORKLOADS["cfg3"], "ms_per_frame": ms3, "rays_per_s": R_frame / (ms3 / 1e3),
                          "peak_device_memory_gb": (torch.cuda.max_memory_allocated(dev) - base_mem) / 2**30,
                          "alg_tflop_per_frame": flop3 / 1e12, "frac_of_tensor_roofline": flop3 / (ms3 / 1e3) / 1e12 / peak,
                          "outputs": sorted(k for k in o3 if k.endswith("_map")),
                          "note": "both passes run the full network (heads included), so the algorithmic FLOPs are "
                                  "256 evaluations x 1 345 792 per ray; one pnr_render_fused call, default workspace; "
                                  "compositing runs in the MLP kernel's epilogue (raw is never written)"}}
        del r3, b3, o3
        # the training step of the same network on the library's kernels (SURVEY 8(f) rank 2): 2048 rays x 192 samples,
        # forward + losses + backward to every parameter.  Informational; a failure here must not cost the bench line.
        try:
            from panopticnerf_b200.lib.train import training_step
            g3 = torch.Generator().manual_seed(0)
            Rt, Nt = 2048, 192
            rays_t = torch.cat([torch.randn(Rt, 3, generator=g3) * 0.5,
                                torch.nn.functional.normalize(torch.randn(Rt, 3, generator=g3), dim=-1)], -1).to(dev)
            z_t = torch.sort(torch.rand(Rt, Nt, generator=g3) * 6 + 0.5, -1).values.to(dev)
            batch_t = {"rgb": torch.rand(Rt, 3, generator=g3).to(dev), "depth": (torch.rand(Rt, generator=g3) * 6).to(dev),
                       "pseudo_label": torch.randint(-1, c3.num_classes, (Rt,), generator=g3).to(dev)}
            tt = []
            for i in range(2 + 3):
                for prm in n3.parameters():
                    prm.grad = None
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                training_step(n3, rays_t, z_t, batch_t, (1.0, 0.1, 1.0, 0.0))
                b.record()
                torch.cuda.synchronize()
                if i >= 2:
                    tt.append(a.elapsed_time(b))
            mst = statistics.median(tt)
            extra["train_step_cfg3"] = {
                "workload": f"{Rt} rays x {Nt} samples, cfg3 network: forward (fused MLP + compositing) + loss kernel + "
                            "backward to every parameter (trunk on the fused tensor-core kernel, the layers after it on "
                            "pnr_linear, every weight gradient on pnr_wgrad: no library GEMM)", "ms_per_step": mst, "rays_per_s": Rt / (mst / 1e3),
                "samples_per_s": Rt * Nt / (mst / 1e3)}
        except Exception as exc:   # noqa: BLE001
            extra["train_step_cfg3"] = {"error": repr(exc)[:300]}
        del n3
        # the two HBM-bound GEMM kernels of that step, timed alone against the measured copy bandwidth (operands of
        # 403 MB each: larger than L2, no flush needed).  Informational; a failure here must not cost the bench line.
        try:
            from panopticnerf_b200.lib.train.mlp_backward import wgrad, linear3x, _pow2_scale
            gg = torch.Generator().manual_seed(1)
            Sg = 393216
            dz_g = (torch.randn(Sg, 256, generator=gg) * 1e-6).to(dev)
            x_g = torch.relu(torch.randn(Sg, 256, generator=gg)).to(dev)
            w_g = (torch.randn(256, 256, generator=gg) / 16.0).to(dev)
            sc_g = _pow2_scale(dz_g)

            def _median_ms(fn, reps=5, warm=2):
                ts = []
                for i in range(warm + reps):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    fn()
                    b.record()
                    torch.cuda.synchronize()
                    if i >= warm:
                        ts.append(a.elapsed_time(b))
                return statistics.median(ts)

            t_w = _median_ms(lambda: wgrad(dz_g, x_g, precision="fp16x3", scale=sc_g))
            t_l = _median_ms(lambda: linear3x(x_g, w_g, precision="fp16x3"))
            hbm = float(peaks()["hbm_gbs"])
            byt = 4.0 * Sg * 512
            extra["train_gemms"] = {
                "workload": f"{Sg} samples x 256 x 256, fp16x3: pnr_wgrad (dW = dZ^T X + column sums; reads dZ and X) and "
                            "pnr_linear (y = x W^T; reads x, writes y); algorithmic bytes = 2 KB per sample each",
                "wgrad": {"ms": t_w, "achieved_gbs": byt / t_w / 1e6, "frac_of_hbm_peak": byt / t_w / 1e6 / hbm},
                "linear": {"ms": t_l, "achieved_gbs": byt / t_l / 1e6, "frac_of_hbm_peak": byt / t_l / 1e6 / hbm},
                "peak_gbs": hbm, "bound": "hbm"}
            del dz_g, x_g, w_g
        except Exception as exc:   # noqa: BLE001
            extra["train_gemms"] = {"error": repr(exc)[:300]}

    # ---------------- CPU baseline (rank 0, N=1): oracle port on the host cores, bounded strip + measured parity
    cpu_baseline, parity = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = host_threads()
        orc = CpuOracle(cfg, threads)
        rows = args.ref_rows or orc.pick_rows(6.0)
        runs = [orc.run(rows) for _ in range(3)]
        rates = sorted(r[0] for r in runs)
        cpu_baseline = {"value": rates[1], "unit": UNIT, "cores": threads, "kind": "port",
                        "sample": f"{rows}-row strip ({rows * cfg.W_img} rays) of the frame, median of 3 "
                                  f"({sum(r[1] for r in runs):.1f} s of CPU work)",
                        "all_runs": [round(x, 1) for x in rates], "os_cpu_count": os.cpu_count(),
                        "note": "in-repo oracle (reference source not in the mount)"}
        _, _, sbatch, sref = runs[-1]
        # same weights as the oracle's network (both are init_network_weights(seed 0) of the same architecture)
        sgpu = ren.render({k: v.to(dev) for k, v in sbatch.items()})
        parity = parity_on_strip(sref, sgpu, float(sref["far"].max()))

    if rank == 0:
        passes = "3 tensor-core passes hi*hi + lo*hi + hi*lo" if args.precision.endswith("x3") else "1 tensor-core pass"
        line = {
            "metric": metric_name(cfg), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None,
            "dtype": f"{args.precision} ({args.precision[:4]} operands, fp32 accumulate; {passes})", "data": "synthetic",
            "config": {"workload": WORKLOADS[args.config] + (", one frame per GPU" if args.scaling == "weak" else
                                                            f", ONE frame ray-sharded over {world} GPU(s)"),
                       "gather": (f"NCCL all-gather (pnr_allgather_outputs) of {args.gather} tiles, "
                                  f"{gather_bytes} bytes per rank" if tg is not None else "none (1 GPU)"),
                       "rays_per_gpu_per_step": R, "samples_per_ray": N, "importance_samples": cfg.N_importance,
                       "precision": args.precision, "parallelism": f"ray-sharded x{world}",
                       "l2": "flushed between steps (256 MiB memset, outside the events)",
                       "api": "Renderer.render -> one pnr_render_fused call per frame",
                       "wall_s_timed_region": t_wall, "step_ms": [round(x, 2) for x in step_ms]},
            "roofline": roofline, "e2e": e2e, "cpu_baseline": cpu_baseline, "parity_vs_cpu_oracle": parity,
            "gpu_launches": launches, "gpu_launches_source": "pnr_launch_count(): kernels libpnr enqueued inside the timed region",
            "clocks": clocks, "fast_mode": fast, "extra": extra,
        }
        emit(line)
    if tg is not None:
        tg.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
