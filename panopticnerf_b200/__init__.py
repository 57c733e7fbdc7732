"""panopticnerf_b200 — B200-native (sm_100a) implementation of the PanopticNeRF per-ray render path
behind the reference's lib/networks plugin surface (make_network, make_renderer, Renderer.render,
batchify_rays, raw2outputs, sample_pdf).  All compute is hand-written CUDA in libpnr.so (C ABI,
include/pnr.h); there is no CPU or PyTorch fallback."""
from .config import make_cfg, PRESETS  # noqa: F401

__all__ = ["make_cfg", "PRESETS", "make_network", "make_renderer", "make_evaluator"]


def make_network(cfg):
    from .lib.networks import make_network as _mk
    return _mk(cfg)


def make_evaluator(cfg, device=None):
    from .lib.evaluators import make_evaluator as _mk
    return _mk(cfg, device)


def make_renderer(cfg, network, network_fine=None):
    from .lib.networks import make_renderer as _mk
    return _mk(cfg, network, network_fine)
