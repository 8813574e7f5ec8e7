"""CPU: pins oracle/shade_oracle.py against numbers produced by the reference's own Python
(PointAggregator / NeuralPointsRayMarching / ray_march run unmodified on CPU, oracle/make_golden.py),
forward values and autograd gradients."""
import os

import numpy as np
import pytest
import torch

from oracle import shade_oracle
from pointnerf_b200 import scene


def _mlp_from(fx, prefix="mlp."):
    return {k[len(prefix):]: torch.from_numpy(fx[k]) for k in fx.files if k.startswith(prefix)}


@pytest.mark.parametrize("name", ["tiny_opaque", "tiny_thin_sr8", "tiny_order1"])
def test_shade_oracle_matches_reference_fixture(name, golden_dir):
    fx = np.load(os.path.join(golden_dir, name + ".npz"))
    order = int(fx["agg_intrp_order"]) if "agg_intrp_order" in fx.files else 2
    cfg = scene.CONFIGS["tiny"]
    pts = scene.make_points(cfg)
    rays = scene.make_rays(cfg, fx["pixels"])
    mask = torch.from_numpy(fx["ray_mask"]) > 0
    pts_g = {k: v.clone().requires_grad_(k in ("embedding", "color", "dir", "conf")) for k, v in pts.items()}
    mlp = {k: v.clone().requires_grad_(True) for k, v in _mlp_from(fx).items()}
    sh = shade_oracle.shade(pts_g, mlp, torch.from_numpy(fx["sample_pidx"]), torch.from_numpy(fx["sample_loc_w"]),
                            rays["raydir"][0][mask], torch.tensor(cfg.campos), torch.eye(3), [cfg.vsize] * 3, torch.ones(3),
                            agg_intrp_order=order)
    # forward: same torch build, same op order -> tight
    for a, b in (("ray_color", "coarse_raycolor"), ("opacity", "coarse_point_opacity"), ("weight", "weight"),
                 ("conf_coefficient", "conf_coefficient"), ("sample_loc", "sample_loc")):
        assert np.abs(sh[a].detach().numpy() - fx[b]).max() <= 1e-6, a
    assert np.abs(sh["bg_T"].detach().numpy() - fx["coarse_is_background"]).max() <= 1e-6
    assert np.abs(sh["blend_weight"].detach().numpy() - fx["blend_weight"]).max() <= 1e-6
    # backward oracle = autograd through the restatement
    loss = (sh["ray_color"] ** 2).sum() + 1e-3 * sh["conf_coefficient"].sum()
    loss.backward()
    for k, g in (("embedding", "grad_embedding"), ("color", "grad_color"), ("dir", "grad_dir"), ("conf", "grad_conf")):
        ref = fx[g]
        assert np.abs(pts_g[k].grad.numpy() - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max()), k
    for k in mlp:
        ref = fx["gradmlp." + k]
        assert np.abs(mlp[k].grad.numpy() - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max()), k


def test_fill_invalid(golden_dir):
    fx = np.load(os.path.join(golden_dir, "tiny_opaque.npz"))
    mask = torch.from_numpy(fx["ray_mask"]) > 0
    out = shade_oracle.fill_invalid(mask, torch.from_numpy(fx["coarse_raycolor"]), torch.from_numpy(fx["coarse_point_opacity"]),
                                    torch.from_numpy(fx["coarse_is_background"]), torch.zeros(int(mask.sum()), 3), torch.ones(3))
    assert out["coarse_raycolor"].shape == (mask.shape[0], 3)
    assert torch.all(out["coarse_raycolor"][~mask] == 1) and torch.all(out["coarse_is_background"][~mask] == 1)
    assert torch.all(out["coarse_point_opacity"][~mask] == 0)


def test_positional_encoding_matches_reference(golden_dir):
    """vs the reference's models/helpers/networks.py positional_encoding on a seeded input (oracle/make_golden.py)."""
    fx = np.load(os.path.join(golden_dir, "positional_encoding.npz"))
    x = torch.from_numpy(fx["x"])
    for freqs, ori in ((3, False), (5, False), (4, True)):
        assert torch.equal(torch.from_numpy(fx["pe_%d_%d" % (freqs, int(ori))]), shade_oracle.positional_encoding(x, freqs, ori=ori))
