"""Tile queue of the frozen-cloud pair kernel k_shade_tc8: the CTAs take 128-row tiles from a device counter instead of the static
stride blockIdx.x + t * gridDim.x (pnb_dbg_flags bit 4 keeps the static schedule).  Which CTA computes a tile does not enter the
arithmetic, so both schedules must give equal bits."""
import ctypes as C

import pytest
import torch

from pointnerf_b200 import harness, lib as L, scene

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
STATIC = 16          # pnb_dbg_flags bit 4: static tile schedule
KEYS = ("coarse_raycolor", "coarse_point_opacity", "coarse_is_background")


def _render(net, cfg, rays):
    with torch.no_grad():
        out = net.render_full(list(cfg.campos), rays["raydir"].to(DEV), torch.eye(3), cfg.near, cfg.far, [1., 1., 1.])
    net.check_errors()
    return out


def _pair(name, **over):
    cfg = scene.CONFIGS[name]
    queue, _, _ = harness.build_model(cfg, DEV, alpha_bias=3.0, **over)
    static, _, _ = harness.build_model(cfg, DEV, alpha_bias=3.0, pnb_dbg_flags=STATIC, **over)
    return cfg, queue, static


def _queue_state(net):
    """(n_quads, tile counter) of the last call, from the pair kernel's workspace."""
    ptrs = [C.c_void_p() for _ in range(4)]
    L.check(L.load().pnb_shade_tc_tables(net._tc_ws.data_ptr(), net._tc_ws.numel(), net._max_valid, *[C.byref(p) for p in ptrs]), "tables")
    off = ptrs[3].value - net._tc_ws.data_ptr()
    n_quads, ctr = net._tc_ws[off:off + 8].view(torch.int32).cpu().tolist()
    return n_quads, ctr


def _assert_equal(a, b):
    for k in KEYS:
        assert torch.equal(a[k], b[k]), k


def _n_valid(net):
    return int(net.last.counters_tensor()[L.QC["n_valid"]].item())


@pytest.mark.parametrize("name,side", [("lego_render", None), ("tiny", None), ("tiny", 8)])
def test_tile_queue_matches_static_schedule(name, side):
    """The whole lego frame (~1,100 tiles per CTA), the tiny frame and an 8 x 8 patch of it (fewer tiles than SMs: some CTAs only
    receive the end signal).  Every CTA takes one tile past the end before it stops, so the counter ends at n_tiles + grid size."""
    cfg, queue, static = _pair(name)
    rays = scene.make_rays(cfg, None if side is None else scene.centre_patch(cfg, side))
    oq, os_ = _render(queue, cfg, rays), _render(static, cfg, rays)
    _assert_equal(oq, os_)
    assert oq["coarse_point_opacity"].max().item() > 0.0
    n_quads, ctr = _queue_state(queue)
    n_tiles = (n_quads + 3) // 4
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    assert ctr == n_tiles + n_sm
    if side == 8:
        assert 0 < n_tiles < n_sm


def test_tile_queue_without_valid_samples():
    """Rays pointing away from the cloud: no valid sample, no tile, every CTA gets the end signal first."""
    cfg, queue, static = _pair("tiny")
    rays = scene.make_rays(cfg)
    rays["raydir"] = -rays["raydir"]
    oq, os_ = _render(queue, cfg, rays), _render(static, cfg, rays)
    assert _n_valid(queue) == 0
    _assert_equal(oq, os_)
    assert _queue_state(queue) == (0, torch.cuda.get_device_properties(0).multi_processor_count)


def test_tile_queue_is_reset_between_calls():
    """Back-to-back calls on different ray sets: each call hands out all of its tiles again (the counter is zeroed by the row packing
    of the same call).  A stale counter would skip tiles and leave the previous call's h-bar / sigma in the workspace."""
    cfg, queue, static = _pair("lego_render")
    patches = [scene.make_rays(cfg, scene.centre_patch(cfg, s)) for s in (96, 64, 96)]
    for rays in patches:
        _assert_equal(_render(queue, cfg, rays), _render(static, cfg, rays))
        n_quads, ctr = _queue_state(queue)
        assert ctr == (n_quads + 3) // 4 + torch.cuda.get_device_properties(0).multi_processor_count
