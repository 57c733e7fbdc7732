"""Generates tests/golden/render_golden.pt from the CPU oracle (run here, CPU only):
    python tests/golden/make_golden.py
The reference has no golden vectors (its source is not in the mount), so these fixtures pin the ORACLE
against drift and give the GPU tests a committed target that does not depend on importing anything at
run time.  Inputs are seeded; everything is fp32/int32/int64 and the file is small (< 1 MB, see save_deflated)."""
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
from oracle import reference_renderer as O  # noqa: E402
from panopticnerf_b200 import make_cfg, synthetic as S  # noqa: E402


def build():
    torch.manual_seed(0)
    torch.set_num_threads(1)
    g = torch.Generator().manual_seed(123)
    out = {}
    # ---- stage fixtures
    cfg = make_cfg("cfg2")
    rays = S.make_rays(cfg, rows=1, row0=180)[::11].contiguous()                   # 128 rays
    boxes = S.make_boxes(48, 45, 64, seed=5)
    hit, bid, tin, tout = O.intersect(rays[:, :3], rays[:, 3:], boxes["box_center"], boxes["box_half"], boxes["box_rot"], 4)
    near, far = O.scene_near_far(rays[:, :3], rays[:, 3:], torch.tensor(S.SCENE_AABB), cfg.near, cfg.far)
    t = torch.linspace(0, 1, 64)
    u = torch.rand(rays.shape[0], 64, generator=g)
    z = O.stratified_z(near, far, t, 1.0, u)
    sb = O.tag_samples(z, bid, tin, tout)
    w = torch.rand(rays.shape[0], 64, generator=g) ** 3
    uf = torch.linspace(0, 1, 32)[None].expand(rays.shape[0], 32).contiguous()
    z_f, idx = O.sample_pdf(0.5 * (z[:, 1:] + z[:, :-1]), w[:, 1:-1], 32, u=uf)
    out["stage"] = dict(rays=rays, boxes=boxes, hit=hit, box_id=bid, t_in=tin, t_out=tout, near=near, far=far,
                        t_vals=t, u=u, z=z, sample_box=sb, weights=w, u_fine=uf, z_fine=z_f, idx=idx,
                        z_all=O.merge_sorted(z, z_f))
    raw = torch.randn(rays.shape[0], 64, 4 + 5 + 6, generator=g)
    comp = O.raw2outputs(raw, z, rays[:, 3:], num_classes=5, num_instances=6, sample_box=sb,
                         box_sem=boxes["box_sem"] % 5, box_inst=boxes["box_inst"] % 6)
    out["composite"] = dict(raw=raw, box_sem=boxes["box_sem"] % 5, box_inst=boxes["box_inst"] % 6, out=comp)
    x = (torch.rand(64, 3, generator=g) - 0.5) * 100
    out["embed"] = dict(x=x, e10=O.embed(x, 10), e4=O.embed(x, 4))
    # ---- network + end-to-end fixture (config 1: 4 x 64 MLP, heads, coarse + fine)
    cfg1 = make_cfg("cfg1", num_classes=5, num_instances=6, N_importance=16, max_hits=3)
    net = S.init_network_weights(O.make_network(cfg1), seed=7)
    pts = torch.rand(200, 3, generator=g) * 20 - 5
    vd = torch.nn.functional.normalize(torch.randn(200, 3, generator=g), dim=-1)
    with torch.no_grad():
        raw_net = net(pts, vd)
    batch = S.make_batch(cfg1, rows=4, row0=30, num_boxes=32)
    ren = O.make_renderer(cfg1, net).render(batch)
    keep = ("hit_mask", "box_id", "z_vals_0", "rgb_map_0", "acc_map_0", "depth_map_0", "semantic_map_0",
            "instance_map_0", "weights_0", "near", "far")
    out["net"] = dict(cfg=dict(vars(cfg1)), state={k: v.clone() for k, v in net.state_dict().items()},
                      pts=pts, viewdirs=vd, raw=raw_net, batch=batch, render={k: ren[k] for k in keep})
    return out


def save_deflated(obj, dst: Path) -> None:
    """torch.save stores its zip members uncompressed (1.09 MB for these fixtures).  Deflating the members that
    deflate to under half their size (integer ids, indices, the pickle) keeps the file under 1 MB; the random
    fp32 members stay stored.  torch.load reads both kinds of member."""
    import io
    import zipfile
    import zlib
    buf = io.BytesIO()
    torch.save(obj, buf)
    with zipfile.ZipFile(buf) as src, zipfile.ZipFile(dst, "w") as out:
        for member in src.infolist():
            data = src.read(member.filename)
            deflate = len(zlib.compress(data, 9)) < len(data) // 2
            out.writestr(member.filename, data, compress_type=zipfile.ZIP_DEFLATED if deflate else zipfile.ZIP_STORED,
                         compresslevel=9)


if __name__ == "__main__":
    dst = Path(__file__).with_name("render_golden.pt")
    save_deflated(build(), dst)
    print(dst, dst.stat().st_size, "bytes")
