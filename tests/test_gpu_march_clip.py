"""The march clips every ray to the bounding box (PNB_GC_BOX_*) and the bounding sphere (PNB_GC_SPHERE_R2) of the dilated occupancy
before it walks its steps.  Skipped steps lie at least one voxel outside any occupied voxel, so the march must keep exactly the steps,
counts and order of the full march.  The full march is the same kernel with the box and the sphere widened to cover all space.  The K-NN that follows looks cells up column by column; its results
are compared as well (cand_pidx in canonical slot order)."""
import dataclasses

import numpy as np
import pytest
import torch

from pointnerf_b200 import harness, lib as L, scene

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
BOX = slice(L.GC["box_x0"], L.GC["box_z1"] + 1)
CLIP = slice(L.GC["box_x0"], L.GC["sphere_r2"] + 1)          # box and sphere
NO_CLIP = [-(1 << 24)] * 3 + [1 << 24] * 3 + [int(np.array(1e30, np.float32).view(np.int32))]


def _grid_counters(grid):
    off = int(grid.desc.counters) - grid.buf.data_ptr()
    return grid.buf[off:off + 64].view(torch.int32)


def _view(q, ptr, n, dtype):
    off = int(ptr) - q.ws.data_ptr()
    return q.ws[off:off + n * torch.tensor([], dtype=dtype).element_size()].view(dtype)


def _snapshot(q):
    """nsamp [R], the kept steps of every ray, and the neighbours of every candidate (host copies)."""
    R, SR, K = q.R, q.SR, q.K
    nsamp = _view(q, q.desc.nsamp, R, torch.int32).cpu().numpy().copy()
    steps = _view(q, q.desc.steps, R * SR, torch.int16).cpu().numpy().view(np.uint16).reshape(R, SR).copy()
    steps[np.arange(SR)[None, :] >= nsamp[:, None]] = 0          # slots past nsamp are not written
    n_cand = int(_view(q, q.desc.samp_off, R + 1, torch.int32)[R].item())
    pidx = _view(q, q.desc.cand_pidx, n_cand * K, torch.int32).cpu().numpy().copy()
    return nsamp, steps, pidx, dict(q.counters)


def _query(net, cfg, raydir, campos=None):
    qr = net.neural_points.querier
    q = qr.run_query(net.neural_points.xyz.detach(), raydir.to(DEV).contiguous(), list(campos or cfg.campos), cfg.near, cfg.far,
                     want_counters=True)
    torch.cuda.synchronize()
    return q


def _clip_vs_full(net, cfg, raydir, campos=None):
    """Runs the query with the grid's box and sphere and with both covering all space; asserts equal results, returns the clipped
    ones."""
    q = _query(net, cfg, raydir, campos)
    grid = net.neural_points.querier._grid
    gc = _grid_counters(grid)
    clip = gc[CLIP].clone()
    clipped = _snapshot(q)
    gc[CLIP] = torch.tensor(NO_CLIP, dtype=torch.int32, device=DEV)
    try:
        full = _snapshot(_query(net, cfg, raydir, campos))
    finally:
        gc[CLIP] = clip
    for a, b, what in zip(clipped, full, ("nsamp", "steps", "cand_pidx", "counters")):
        if isinstance(a, dict):
            assert a == b, what
        else:
            assert np.array_equal(a, b), what
    return clipped


def _occupied_voxels(grid):
    """Voxel coordinates [3, n] of the set bits of occ_bits, from the bit array itself."""
    dim = [int(v) for v in grid.desc.dim]
    nw = int(grid.desc.n_words)
    off = int(grid.desc.occ_bits) - grid.buf.data_ptr()
    words = grid.buf[off:off + 4 * nw].view(torch.int32).cpu().numpy().view(np.uint32)
    bits = np.unpackbits(words.view(np.uint8), bitorder="little")[:dim[0] * dim[1] * dim[2]].reshape(dim)
    return np.array(np.nonzero(bits))


def _box_rays(net, cfg, campos, frac):
    """Unit directions from campos to points on the world extent of the occupied box: its 8 corners and its 12 edge midpoints,
    each moved by `frac` of a voxel outwards (> 0) or inwards (< 0): rays that graze the box."""
    grid = net.neural_points.querier._grid
    b = _grid_counters(grid)[BOX].cpu().numpy()
    lo, svs = np.array(grid.desc.lo, np.float64), np.array(grid.desc.svs, np.float64)
    wlo, whi = lo + b[:3] * svs - frac * svs, lo + (b[3:] + 1) * svs + frac * svs
    pts = []
    for i in range(27):
        sel = [(i // 9) % 3, (i // 3) % 3, i % 3]
        if sum(s == 1 for s in sel) > 1:
            continue
        pts.append([(wlo[a], 0.5 * (wlo[a] + whi[a]), whi[a])[sel[a]] for a in range(3)])
    d = np.array(pts) - np.array(campos, np.float64)[None]
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return torch.tensor(d, dtype=torch.float32)


def test_grid_box_is_the_occupancy_box():
    for name in ("tiny", "lego_render"):
        net, _, _ = harness.build_model(scene.CONFIGS[name], DEV)
        cfg = scene.CONFIGS[name]
        _query(net, cfg, scene.make_rays(cfg, scene.centre_patch(cfg, 8))["raydir"][0])
        grid = net.neural_points.querier._grid
        gc = _grid_counters(grid).cpu().numpy()
        v = _occupied_voxels(grid)
        assert gc[BOX].tolist() == [int(x) for x in v.min(1)] + [int(x) for x in v.max(1)]
        # every corner of every occupied voxel lies inside the sphere about the grid centre
        lo, svs, dim = (np.array(getattr(grid.desc, k), np.float64) for k in ("lo", "svs", "dim"))
        ctr = lo + 0.5 * dim * svs
        far = np.maximum(np.abs(lo[:, None] + v * svs[:, None] - ctr[:, None]), np.abs(lo[:, None] + (v + 1) * svs[:, None] - ctr[:, None]))
        r2 = float(gc[L.GC["sphere_r2"]:L.GC["sphere_r2"] + 1].view(np.float32)[0])
        assert (far ** 2).sum(0).max() <= r2 * (1 + 1e-5)


@pytest.mark.parametrize("name,side,SR", [("lego_render", None, 24), ("lego_render", None, 80), ("tiny", None, 24),
                                          ("chair_plumbing", 96, 24)])
def test_clipped_march_matches_full_march(name, side, SR):
    """Whole frames (most lego rays miss the cloud) and a chair patch; SR 80 keeps more steps per ray."""
    cfg = scene.CONFIGS[name]
    net, _, _ = harness.build_model(cfg, DEV, SR=SR)
    rays = scene.make_rays(cfg, None if side is None else scene.centre_patch(cfg, side))
    _, _, _, cnt = _clip_vs_full(net, cfg, rays["raydir"][0])
    assert cnt["n_valid"] > 0


@pytest.mark.parametrize("frac", [-1e-3, 1e-3, 0.5, 1.0, 1.5])
def test_clipped_march_grazing_rays(frac):
    """Rays aimed at the corners and edges of the box's world extent, just inside, just outside, and half a voxel to 1.5 voxels
    outside (the widened box's own edge)."""
    cfg = scene.CONFIGS["tiny"]
    net, _, _ = harness.build_model(cfg, DEV)
    _query(net, cfg, scene.make_rays(cfg, scene.centre_patch(cfg, 8))["raydir"][0])
    _clip_vs_full(net, cfg, _box_rays(net, cfg, cfg.campos, frac))


def test_clipped_march_camera_inside_box():
    """The camera sits inside the occupied box: the clip starts at the first step, in every direction."""
    cfg = scene.CONFIGS["tiny"]
    net, _, _ = harness.build_model(cfg, DEV)
    _query(net, cfg, scene.make_rays(cfg, scene.centre_patch(cfg, 8))["raydir"][0])
    inside = (0.05, -0.02, 0.03)
    g = torch.Generator().manual_seed(3)
    d = torch.randn(512, 3, generator=g)
    d = torch.cat([d, _box_rays(net, cfg, inside, 0.0)])
    d = d / d.norm(dim=1, keepdim=True)
    nsamp, _, _, _ = _clip_vs_full(net, dataclasses.replace(cfg, near=0.01, far=2.0), d, campos=inside)
    assert (nsamp > 0).any()


def test_clipped_march_rays_that_miss():
    """Rays turned away from the cloud and rays along the axes past it: no step is marched, nothing is found."""
    cfg = scene.CONFIGS["tiny"]
    net, _, _ = harness.build_model(cfg, DEV)
    rays = scene.make_rays(cfg, scene.centre_patch(cfg, 16))["raydir"][0]
    axes = torch.tensor([[1., 0., 0.], [0., 1., 0.], [-1., 0., 0.], [0., -1., 0.], [0., 0., -1.]])
    nsamp, _, _, cnt = _clip_vs_full(net, cfg, torch.cat([-rays, axes]))
    assert (nsamp == 0).all() and cnt["n_cand"] == 0
