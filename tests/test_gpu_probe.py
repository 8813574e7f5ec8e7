"""GPU: point growing on the device.  probe_full (render_full + pnb_probe_maps) against the eager probe outputs of the drop-in
forward(opt.prob = 1) and against the reference fixture; probe_frame (pnb_probe_select) against the reference chunk loop restated
through forward() (probe_frame_chunked); probe_holes' accumulation; grow + render end to end."""
import os

import numpy as np
import pytest
import torch

from pointnerf_b200 import harness, runner, scene

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
AVG_KEYS = ("ray_max_far_dist", "shading_avg_color", "shading_avg_dir", "shading_avg_conf", "shading_avg_embedding")


def _dev(rays):
    return {k: (v.to(DEV) if isinstance(v, torch.Tensor) else v) for k, v in rays.items()}


def _block(x0, y0, w, h):
    px, py = np.meshgrid(np.arange(x0, x0 + w), np.arange(y0, y0 + h))
    return np.stack((px, py), -1).reshape(-1, 2).astype(np.float32)


def _close(a, b, what, rel=1e-6):
    scale = max(b.abs().max().item(), 1e-30)
    d = (a - b).abs().max().item() if a.numel() else 0.0
    assert d <= rel * scale, "%s: max abs diff %.3e (max abs %.3e)" % (what, d, scale)


def _eager_unmasked(net, r):
    """forward() with opt.prob = 1, then unmask (neural_points_volumetric_model.py:125-131) to all R rays."""
    net.opt.prob = 1
    try:
        with torch.no_grad():
            out = net(r["campos"], r["raydir"], bg_color=r["bg_color"], camrotc2w=r["camrotc2w"], near=r["near"], far=r["far"])
    finally:
        net.opt.prob = 0
    mask = out["ray_mask"][0]
    inds = torch.nonzero(mask)[:, 0]
    R = mask.shape[0]
    full = {"ray_mask": mask}
    for k in ("ray_max_sample_loc_w", "ray_max_shading_opacity") + AVG_KEYS:
        v = out[k][0].reshape(inds.shape[0], -1)
        full[k] = torch.zeros((R, v.shape[1]), device=DEV).index_copy_(0, inds, v)
    full["slot"] = torch.full((R,), -1, dtype=torch.long, device=DEV)
    full["slot"][inds] = torch.max(out["coarse_point_opacity"][0], dim=-1)[1]
    return full


@pytest.mark.parametrize("name,pixels", [
    ("tiny", None),                                            # full 64x64 frame: hits and misses
    ("lego_render", "centre64"),                               # every ray hits
    ("lego_render", (640, 388, 96, 24)),                       # silhouette strip: grazing hits, partial neighbourhoods, misses
])
def test_probe_maps_match_eager_path(name, pixels):
    cfg = scene.CONFIGS[name]
    net, _, _ = harness.build_model(cfg, DEV, alpha_bias=3.0)
    pix = None if pixels is None else scene.centre_patch(cfg, 64) if pixels == "centre64" else _block(*pixels)
    r = _dev(scene.make_rays(cfg, pix))
    with torch.no_grad():
        p = net.probe_full(r["campos"], r["raydir"], r["camrotc2w"], float(r["near"]), float(r["far"]), r["bg_color"], want_argmax=True)
    net.check_errors()
    e = _eager_unmasked(net, r)
    assert torch.equal(p["ray_mask"][0], e["ray_mask"])
    hit = e["ray_mask"] > 0
    assert hit.any()
    if pixels != "centre64":
        assert not hit.all()
    assert torch.equal(p["ray_max_slot"][0].long(), e["slot"])
    assert torch.equal(p["ray_max_sample_loc_w"][0], e["ray_max_sample_loc_w"])
    assert torch.equal(p["ray_max_shading_opacity"][0], e["ray_max_shading_opacity"])
    for k in AVG_KEYS:
        _close(p[k][0], e[k], k)
    for k in ("ray_max_sample_loc_w", "ray_max_shading_opacity") + AVG_KEYS:      # unmask: zeros without a neighbour
        assert torch.all(p[k][0][~hit] == 0), k


def test_probe_full_matches_reference_fixture(golden_dir):
    """Same criteria as the drop-in forward's fixture test (tests/test_gpu_shade.py) for the fused probe."""
    fx = np.load(os.path.join(golden_dir, "tiny_probe.npz"))
    wfx = np.load(os.path.join(golden_dir, "tiny_opaque.npz"))
    cfg = scene.CONFIGS["tiny"]
    net, _, _ = harness.build_model(cfg, DEV, max_o=100000)
    net.aggregator.load_state_dict({k[4:]: torch.from_numpy(wfx[k]) for k in wfx.files if k.startswith("mlp.")})
    r = _dev(scene.make_rays(cfg, fx["pixels"]))
    with torch.no_grad():
        out = net.probe_full(r["campos"], r["raydir"], r["camrotc2w"], float(r["near"]), float(r["far"]), r["bg_color"])
    net.check_errors()
    hit = out["ray_mask"][0] > 0
    assert int(hit.sum()) == fx["ray_max_sample_loc_w"].shape[0]
    loc = out["ray_max_sample_loc_w"][0][hit].cpu().numpy()
    same = np.abs(loc - fx["ray_max_sample_loc_w"]).max(-1) == 0
    assert same.mean() > 0.98
    for k, tol in (("ray_max_shading_opacity", 1e-4), ("ray_max_far_dist", 1e-6), ("shading_avg_color", 1e-5),
                   ("shading_avg_dir", 1e-5), ("shading_avg_conf", 1e-5), ("shading_avg_embedding", 1e-5)):
        a = out[k][0][hit].cpu().numpy().reshape(fx[k].shape)
        assert np.abs(a - fx[k])[same].max() <= tol, k


# ------------------------------------------------------------------------------------------------ selection
def _tiny_net():
    return harness.build_model(scene.CONFIGS["tiny"], DEV, alpha_bias=3.0)[0]


def _render_colour(net, data, H, W):
    d = {k: v for k, v in data.items() if k != "pixel_idx"}
    return runner.render_image(net, d, H, W)["coarse_raycolor"].reshape(-1, 3)


def _gt_with_holes(net, data, H, W, pattern):
    """GT = the rendered colour where a ray hits (no far-branch hits, no misses there); at misses 0.25 grey where `pattern` is
    set (holes the probe must find), the background colour elsewhere."""
    col = _render_colour(net, data, H, W)
    miss = torch.all(col == 1.0, dim=-1)                       # bg colour 1 and the scene never renders exactly white
    gt = col.clone()
    gt[miss & pattern.reshape(-1)] = 0.25
    return gt


def _compare(net, data, H, W, gt, opacity_thresh, far_thresh=-1, prob_mul=1.0, min_n=1):
    a = runner.probe_frame(net, data, H, W, gt, opacity_thresh, far_thresh, prob_mul)
    b = runner.probe_frame_chunked(net, data, H, W, gt, opacity_thresh, far_thresh, prob_mul, chunk_size=2304)
    for k in runner.PROBE_KEYS:
        assert a["prob_maps"][k].shape == b["prob_maps"][k].shape, k
    assert torch.equal(a["prob_maps"]["ray_mask"], b["prob_maps"]["ray_mask"])
    assert a["add_xyz"].shape[0] >= min_n
    for k, c in (("add_xyz", 3), ("add_embedding", 32), ("add_color", 3), ("add_dir", 3), ("add_conf", 1)):
        assert a[k].shape == b[k].shape == (b["add_xyz"].shape[0], c), k
    assert torch.equal(a["add_xyz"], b["add_xyz"])             # same pixels, same (row-major) order, same bits
    for k in ("add_embedding", "add_color", "add_dir", "add_conf"):
        if b[k].numel():
            _close(a[k], b[k], k)
    return a, b


def _opacity_median(net, data):
    with torch.no_grad():
        p = net.probe_full(data["campos"], data["raydir"], data["camrotc2w"], float(data["near"]), float(data["far"]), data["bg_color"])
    hit = p["ray_mask"][0] > 0
    return p, float(p["ray_max_shading_opacity"][0][hit].median())


def test_select_full_frame_matches_chunk_loop():
    cfg = scene.CONFIGS["tiny"]
    net = _tiny_net()
    data = _dev(scene.make_rays(cfg))
    del data["pixel_idx"]
    yy, xx = torch.meshgrid(torch.arange(cfg.H, device=DEV), torch.arange(cfg.W, device=DEV), indexing="ij")
    gt = _gt_with_holes(net, data, cfg.H, cfg.W, (xx + yy) % 3 != 0)
    _, med = _opacity_median(net, data)
    _compare(net, data, cfg.H, cfg.W, gt, med, min_n=0)        # the median itself as threshold: the strict '>' on the tie
    _compare(net, data, cfg.H, cfg.W, gt, 0.0, prob_mul=0.4)


def test_select_bloat_clamp_at_all_four_edges():
    """A square crop around the tiny scene's disk as a frame of its own, sized so that the corners miss and the middles of the four
    edges hit: hit pixels on every image edge have misses inside their clipped 3x3 window."""
    cfg = scene.CONFIGS["tiny"]
    net = _tiny_net()
    whole = _dev(scene.make_rays(cfg))
    del whole["pixel_idx"]
    hit = runner.render_image(net, whole, cfg.H, cfg.W)["ray_mask"] > 0       # a ray's mask does not depend on the other rays
    c = cfg.W // 2
    for s in range(4, c):
        m = hit[c - s:c + s, c - s:c + s]
        if all(e.any() and not e.all() for e in (m[0], m[-1], m[:, 0], m[:, -1])):
            break
    else:
        pytest.fail("no square crop whose four edges all cross the silhouette")
    H = W = 2 * s
    data = _dev(scene.make_rays(cfg, _block(c - s, c - s, W, H)))
    del data["pixel_idx"]
    gt = _gt_with_holes(net, data, H, W, torch.ones((H, W), dtype=torch.bool, device=DEV))
    a, _ = _compare(net, data, H, W, gt, 0.0)
    assert torch.equal(a["prob_maps"]["ray_mask"][..., 0] > 0, m)


def test_select_far_branch_matches_chunk_loop():
    cfg = scene.CONFIGS["tiny"]
    net = _tiny_net()
    data = _dev(scene.make_rays(cfg))
    del data["pixel_idx"]
    gt = _gt_with_holes(net, data, cfg.H, cfg.W, torch.zeros((cfg.H, cfg.W), dtype=torch.bool, device=DEV))    # no GT holes
    p, _ = _opacity_median(net, data)
    hit = p["ray_mask"][0] > 0
    far_thresh = float(p["ray_max_far_dist"][0][hit].median())
    a, _ = _compare(net, data, cfg.H, cfg.W, gt, 0.0, far_thresh)
    assert 0 < a["add_xyz"].shape[0] < int(hit.sum())


def test_select_pixel_subset_matches_chunk_loop():
    """A row-major subset of the pixels (pixel_idx, the reference's edge_mask): pixels not given neither count as misses nor
    become points."""
    cfg = scene.CONFIGS["tiny"]
    net = _tiny_net()
    full = scene.make_rays(cfg)
    keep = ((torch.arange(cfg.H * cfg.W) % 5) != 2).nonzero()[:, 0]
    data = _dev({k: (v[:, keep] if k in ("raydir", "pixel_idx") else v) for k, v in full.items()})
    datafull = _dev(full)
    del datafull["pixel_idx"]
    yy, xx = torch.meshgrid(torch.arange(cfg.H, device=DEV), torch.arange(cfg.W, device=DEV), indexing="ij")
    gt = _gt_with_holes(net, datafull, cfg.H, cfg.W, (xx + 2 * yy) % 4 != 0)[keep.to(DEV)]
    a, _ = _compare(net, data, cfg.H, cfg.W, gt, 0.0)
    given = torch.zeros(cfg.H * cfg.W, dtype=torch.bool, device=DEV)
    given[keep.to(DEV)] = True
    assert torch.all(a["prob_maps"]["ray_mask"].reshape(-1)[~given] == 0)


def test_select_zero_candidates():
    cfg = scene.CONFIGS["tiny"]
    net = _tiny_net()
    data = _dev(scene.make_rays(cfg))
    gt = _gt_with_holes(net, {k: v for k, v in data.items() if k != "pixel_idx"}, cfg.H, cfg.W,
                        torch.ones((cfg.H, cfg.W), dtype=torch.bool, device=DEV))
    a, b = _compare(net, data, cfg.H, cfg.W, gt, 2.0, min_n=0)        # opacity never exceeds 2
    assert a["add_xyz"].shape == (0, 3) and a["add_embedding"].shape == (0, 32) and a["add_conf"].shape == (0, 1)


def test_select_every_pixel_hit():
    """lego 64x64 centre patch as a frame: no misses, candidates only through the far branch."""
    cfg = scene.CONFIGS["lego_render"]
    net = harness.build_model(cfg, DEV, alpha_bias=3.0)[0]
    H = W = 64
    data = _dev(scene.make_rays(cfg, scene.centre_patch(cfg, 64)))
    del data["pixel_idx"]
    p, _ = _opacity_median(net, data)
    assert torch.all(p["ray_mask"] > 0)
    gt = _render_colour(net, data, H, W)
    far_thresh = float(p["ray_max_far_dist"][0].median())
    _compare(net, data, H, W, gt, 0.0, -1, min_n=0)
    a, _ = _compare(net, data, H, W, gt, 0.0, far_thresh)
    assert a["add_xyz"].shape[0] > 0


# ------------------------------------------------------------------------------------------------ accumulation, end to end
def _three_frames(net):
    cfg = scene.CONFIGS["tiny"]
    full = scene.make_rays(cfg)
    yy, xx = torch.meshgrid(torch.arange(cfg.H, device=DEV), torch.arange(cfg.W, device=DEV), indexing="ij")
    frames = []
    for i in range(3):
        fr = _dev(full)
        del fr["pixel_idx"]
        fr["gt_image"] = _gt_with_holes(net, fr, cfg.H, cfg.W, (xx + yy + i) % 3 == 0)
        fr["height"], fr["width"] = cfg.H, cfg.W
        frames.append(fr)
    return frames


def test_probe_holes_accumulates_like_probe_hole():
    net = _tiny_net()
    frames = _three_frames(net)
    got = runner.probe_holes(net, frames, 0.0, -1, 0.4)
    parts = [runner.probe_frame_chunked(net, fr, fr["height"], fr["width"], fr["gt_image"], 0.0, -1) for fr in frames]
    n = len(frames)
    want = [torch.cat([p[k] for p in parts]) for k in ("add_xyz", "add_embedding", "add_color", "add_dir")]
    want.append(torch.cat([p["add_conf"] * 0.4 ** (n - i) for i, p in enumerate(parts)]))
    assert all(p["add_xyz"].shape[0] > 0 for p in parts)
    assert torch.equal(got[0], want[0])
    for g, w, k in zip(got[1:], want[1:], ("add_embedding", "add_color", "add_dir", "add_conf")):
        assert g.shape == w.shape, k
        _close(g, w, k)


def test_grow_then_render_and_probe_again():
    """grow_points(*probe_holes(...)) rebuilds the voxel grid and the hoisted table; the grown cloud renders, fills holes, and a
    second probe no longer proposes points at pixels whose holes were filled."""
    cfg = scene.CONFIGS["tiny"]
    net = _tiny_net()
    fr = _three_frames(net)[0]
    H, W = cfg.H, cfg.W
    first = runner.probe_frame(net, fr, H, W, fr["gt_image"], 0.0)
    n0 = net.neural_points.xyz.shape[0]
    add = runner.probe_holes(net, [fr], 0.0, -1, 1.0)
    assert add[0].shape[0] == first["add_xyz"].shape[0] > 0
    net.neural_points.grow_points(*add)
    assert net.neural_points.xyz.shape[0] == n0 + add[0].shape[0]
    img = runner.render_image(net, {k: v for k, v in fr.items() if k not in ("gt_image", "height", "width")}, H, W)
    second = runner.probe_frame(net, fr, H, W, fr["gt_image"], 0.0)
    m1 = first["prob_maps"]["ray_mask"][..., 0] > 0
    m2 = second["prob_maps"]["ray_mask"][..., 0] > 0
    assert torch.equal(img["ray_mask"] > 0, m2)
    hole = (torch.norm(fr["gt_image"].view(H, W, 3) - 1.0, dim=-1) > 0.002)
    miss1, miss2 = hole & ~m1, hole & ~m2
    assert int(miss2.sum()) < int(miss1.sum()), "the new points must fill some holes"

    def windows(miss):                                           # pixels with a hole in their clipped 3x3 window
        w = torch.nn.functional.max_pool2d(miss[None, None].float(), 3, stride=1, padding=1)[0, 0] > 0
        return w
    sel1 = runner.select_holes(first["prob_maps"], fr["gt_image"].view(H, W, 3), torch.ones_like(m1), torch.ones(3, device=DEV), 0.0, -1)
    sel2 = runner.select_holes(second["prob_maps"], fr["gt_image"].view(H, W, 3), torch.ones_like(m2), torch.ones(3, device=DEV), 0.0, -1)
    assert int(sel2.sum()) == second["add_xyz"].shape[0]
    filled = sel1 & ~windows(miss2)                              # candidates of the first probe whose every hole is now filled
    assert filled.any(), "no first-round candidate had all its holes filled"
    assert not (sel2 & filled).any()
    assert not (sel2 & ~windows(miss2)).any()
