"""CPU: the host restatement of point growing's hole test (runner.select_holes, run/train_ft.py:493-505) and of probe_hole's
accumulation (runner.accumulate_new_points, :508-512) on hand-built maps with known answers.  The GPU tests pin the CUDA selection
(pnb_probe_select) to this restatement."""
import torch

from pointnerf_b200 import runner

H, W = 5, 6
BG = torch.ones(3)
ALL = torch.ones((H, W), dtype=torch.bool)


def _maps(hit, op=0.9, far=0.0, color=0.5):
    return {"ray_mask": hit[..., None].to(torch.int8).clone(),
            "ray_max_shading_opacity": torch.full((H, W, 1), op) if not torch.is_tensor(op) else op[..., None].clone(),
            "ray_max_far_dist": torch.full((H, W, 1), far) if not torch.is_tensor(far) else far[..., None].clone(),
            "coarse_raycolor": torch.full((H, W, 3), color)}


def _selected(mask):
    return sorted(map(tuple, mask.nonzero().tolist()))


def test_miss_window_is_clamped_at_the_image_border():
    """A miss in each corner and one on an edge: the 3x3 windows are clipped to the image, only hit pixels are selected."""
    hit = torch.ones((H, W), dtype=torch.bool)
    for y, x in ((0, 0), (0, W - 1), (H - 1, 0), (H - 1, W - 1), (2, W - 1)):
        hit[y, x] = False
    gt = torch.full((H, W, 3), 0.5)                          # GT differs from the background everywhere: every miss counts
    sel = runner.select_holes(_maps(hit), gt, ALL, BG, 0.5, -1)
    want = {(0, 1), (1, 0), (1, 1), (0, W - 2), (1, W - 2), (H - 2, 0), (H - 1, 1), (H - 2, 1), (H - 1, W - 2), (H - 2, W - 2),
            (1, W - 1), (3, W - 1), (2, W - 2), (3, W - 2)}
    assert _selected(sel) == sorted(want)


def test_background_coloured_and_not_given_misses_do_not_count():
    hit = torch.ones((H, W), dtype=torch.bool)
    hit[2, 2] = False
    hit[0, 5] = False
    gt = torch.full((H, W, 3), 0.5)
    gt[2, 2] = BG + 0.001                                    # |gt - bg| = 0.0017 <= 0.002: the background, not a hole
    edge = ALL.clone()
    edge[0, 5] = False                                       # not among the given pixels
    sel = runner.select_holes(_maps(hit), gt, edge, BG, 0.5, -1)
    assert not sel.any()
    gt[2, 2] = BG - 0.01
    sel = runner.select_holes(_maps(hit), gt, edge, BG, 0.5, -1)
    assert _selected(sel) == sorted((y, x) for y in (1, 2, 3) for x in (1, 2, 3) if (y, x) != (2, 2))


def test_opacity_threshold_is_strict():
    hit = torch.ones((H, W), dtype=torch.bool)
    hit[2, 2] = False
    op = torch.full((H, W), 0.7)
    op[1, 1] = 0.7000001
    op[3, 3] = 0.6
    sel = runner.select_holes(_maps(hit, op=op), torch.full((H, W, 3), 0.5), ALL, BG, 0.7, -1)
    assert _selected(sel) == [(1, 1)]


def test_far_branch():
    """far_thresh > 0 also selects hit pixels whose arg-max sample is far from its neighbours and whose colour matches the GT."""
    hit = torch.ones((H, W), dtype=torch.bool)
    hit[4, 0] = False
    far = torch.zeros((H, W))
    far[0, 3] = 0.5                                          # far, colour matches: selected
    far[1, 3] = 0.5                                          # far, colour off by 0.2: not selected
    far[2, 3] = 0.1                                          # not farther than the threshold
    far[4, 0] = 0.5                                          # far but no neighbour (the miss itself): not selected
    gt = torch.full((H, W, 3), 0.5)
    gt[4, 0] = BG                                            # a background-coloured miss: marks nothing
    gt[1, 3] = 0.7
    m = _maps(hit, far=far, color=0.5)
    assert _selected(runner.select_holes(m, gt, ALL, BG, 0.5, 0.1)) == [(0, 3)]
    assert not runner.select_holes(m, gt, ALL, BG, 0.5, -1).any()          # far_thresh <= 0: branch off


def test_bloat_inds_clamps():
    inds = torch.tensor([[0, 0], [4, 5]])
    out = runner.bloat_inds(inds, 1, H, W)
    assert out.shape == (18, 2)
    assert set(map(tuple, out[:9].tolist())) == {(0, 0), (0, 1), (1, 0), (1, 1)}
    assert set(map(tuple, out[9:].tolist())) == {(4, 5), (3, 5), (4, 4), (3, 4)}


def test_prob_mul_compounds_over_frames():
    """probe_hole multiplies ALL of add_conf by prob_mul after every frame: frame i of n ends up scaled by prob_mul**(n - i)."""
    acc = tuple(torch.zeros((0, c)) for c in (3, 32, 3, 3, 1))
    for i in range(3):
        new = [torch.full((2, c), float(i)) for c in (3, 32, 3, 3)] + [torch.ones((2, 1))]
        acc = runner.accumulate_new_points(acc, new, 0.4)
    assert acc[0].shape == (6, 3) and torch.equal(acc[0][:, 0], torch.tensor([0., 0., 1., 1., 2., 2.]))
    want = torch.tensor([0.4 ** 3] * 2 + [0.4 ** 2] * 2 + [0.4] * 2)
    assert torch.allclose(acc[4][:, 0], want, rtol=1e-6, atol=0)
