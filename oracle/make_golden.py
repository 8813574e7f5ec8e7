"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.npz by running the reference's OWN, unmodified
Python hot path (imported from /root/reference through oracle/ref_shim.py) on CPU, with the pybind op
woord_query_grid_point_index served by oracle/query_oracle.c.  Run in the build container:

    python -m oracle.make_golden

The fixtures pin (a) oracle/shade_oracle.py + oracle/pipeline.py (tests/test_oracle_*.py, CPU) and
(b) the CUDA path (tests/test_gpu_*.py) against numbers the reference code itself produced.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_shim, query_oracle  # noqa: E402
from pointnerf_b200 import scene  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def build_reference_net(cfg, alpha_bias, SR=24, is_train=False, extra_flags=()):
    ref_shim.install()
    from models.neural_points_volumetric_model import NeuralPointsRayMarching
    from models.neural_points.neural_points import NeuralPoints
    from models.aggregators.point_aggregators import PointAggregator
    from models.rendering.diff_render_func import find_render_function, find_blend_function, find_tone_map
    vs = str(cfg.vsize)
    opt = ref_shim.make_opt(["--vsize", vs, vs, vs, "--P", str(cfg.P), "--SR", str(SR), "--K", str(cfg.K),
                             "--kernel_size"] + [str(cfg.kernel_size)] * 3 + ["--query_size"] + [str(cfg.query_size)] * 3 +
                            ["--ranges"] + [str(v) for v in scene.ranges_for(cfg)] + list(extra_flags), is_train=is_train)
    pts = scene.make_points(cfg)
    torch.manual_seed(0)
    agg = PointAggregator(opt)
    with torch.no_grad():
        agg.alpha_branch[0].bias += alpha_bias
    npts = NeuralPoints(32, 8192, opt, torch.device("cpu"))
    npts.querier.device = "cpu"   # point_query.py:31 hard-codes "cuda"; instance attribute only, source untouched
    npts.set_points(pts["xyz"], pts["embedding"], points_color=pts["color"], points_dir=pts["dir"],
                    points_conf=pts["conf"], parameter=True)
    net = NeuralPointsRayMarching(tonemap_func=find_tone_map("off"), render_func=find_render_function("radiance"),
                                  blend_func=find_blend_function("alpha"), aggregator=agg, neural_points=npts, opt=opt,
                                  num_pos_freqs=10, num_viewdir_freqs=4)
    return net, agg, npts, pts, opt


def golden_case(name, cfg, pixels, alpha_bias, SR=24, extra_flags=()):
    net, agg, npts, pts, opt = build_reference_net(cfg, alpha_bias, SR=SR, extra_flags=extra_flags)
    rays = scene.make_rays(cfg, pixels)
    out = net(rays["campos"], rays["raydir"], bg_color=rays["bg_color"], camrotc2w=rays["camrotc2w"],
              pixel_idx=rays["pixel_idx"], near=rays["near"], far=rays["far"], h=rays["h"], w=rays["w"],
              intrinsic=rays["intrinsic"])
    # what the querier returned (recompute through the reference class to capture intermediates)
    q = npts.querier
    rng_t, vsz, sdim = q.get_hyperparameters(opt.vsize, npts.xyz[None], ranges=opt.ranges)
    qp = q.query_points(rays["pixel_idx"].to(torch.int32), npts.w2pers(npts.xyz, rays["camrotc2w"], rays["campos"]),
                        npts.xyz[None], torch.tensor([npts.xyz.shape[0]], dtype=torch.int32), 0, 0, None,
                        np.float32(cfg.near), np.float32(cfg.far), rays["raydir"], rays["campos"], rays["camrotc2w"])
    loss = (out["coarse_raycolor"] ** 2).sum() + 1e-3 * out["conf_coefficient"].sum()
    loss.backward()
    g = {n: p.grad for n, p in net.named_parameters() if p.grad is not None}
    fx = dict(
        alpha_bias=np.float32(alpha_bias), SR=np.int32(SR), pixels=np.asarray(pixels, np.float32), agg_intrp_order=np.int32(opt.agg_intrp_order),
        ranges6=rng_t.detach().numpy(), scaled_vdim=sdim, counters=np.array([query_oracle.last_counters[k] for k in query_oracle.COUNTER_NAMES], np.int32),
        ray_mask=out["ray_mask"][0].numpy(), sample_pidx=qp[0][0].numpy(), sample_loc=qp[1][0].detach().numpy(),
        sample_loc_w=qp[2][0].numpy(),
        coarse_raycolor=out["coarse_raycolor"][0].detach().numpy(),
        coarse_point_opacity=out["coarse_point_opacity"][0].detach().numpy(),
        coarse_is_background=out["coarse_is_background"][0].detach().numpy(),
        weight=out["weight"][0].numpy(), conf_coefficient=out["conf_coefficient"][0].detach().numpy(),
        blend_weight=out["blend_weight"][0].numpy(),
        grad_embedding=g["neural_points.points_embeding"].numpy(), grad_color=g["neural_points.points_color"].numpy(),
        grad_dir=g["neural_points.points_dir"].numpy(), grad_conf=g["neural_points.points_conf"].numpy(),
    )
    for k, v in agg.state_dict().items():
        fx["mlp." + k] = v.detach().numpy()
        fx["gradmlp." + k] = g["aggregator." + k].numpy()
    os.makedirs(OUT, exist_ok=True)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **fx)
    print(name, "R'=%d" % fx["sample_pidx"].shape[0], "bgT mean %.3f" % fx["coarse_is_background"].mean(),
          {k: query_oracle.last_counters[k] for k in ("n_occ", "max_pts", "n_valid_samples", "n_valid_pairs")})


def golden_probe(name, cfg, pixels, alpha_bias):
    """opt.prob == 1 outputs (neural_points_volumetric_model.py:331-351) of the reference module; same MLP weights as
    golden_case(..., alpha_bias) (seed 0), so the fixture stores outputs only."""
    net, agg, npts, pts, opt = build_reference_net(cfg, alpha_bias)
    opt.prob = 1
    rays = scene.make_rays(cfg, pixels)
    with torch.no_grad():
        out = net(rays["campos"], rays["raydir"], bg_color=rays["bg_color"], camrotc2w=rays["camrotc2w"],
                  pixel_idx=rays["pixel_idx"], near=rays["near"], far=rays["far"], h=rays["h"], w=rays["w"],
                  intrinsic=rays["intrinsic"])
    keys = ["ray_max_shading_opacity", "ray_max_sample_loc_w", "ray_max_far_dist", "shading_avg_color", "shading_avg_dir",
            "shading_avg_conf", "shading_avg_embedding"]
    fx = {k: out[k][0].numpy() for k in keys}
    fx["pixels"] = np.asarray(pixels, np.float32)
    fx["alpha_bias"] = np.float32(alpha_bias)
    np.savez_compressed(os.path.join(OUT, name + ".npz"), **fx)
    print(name, {k: fx[k].shape for k in keys})


def golden_hyper():
    """get_hyperparameters of the reference class for every BASELINE config (cheap, a few ints/floats each)."""
    ref_shim.install()
    fx = {}
    for name in ("chair_plumbing", "lego_render", "tiny"):
        cfg = scene.CONFIGS[name]
        net, agg, npts, pts, opt = build_reference_net(cfg, 0.0)
        rng_t, vsz, sdim = npts.querier.get_hyperparameters(opt.vsize, npts.xyz[None], ranges=opt.ranges)
        fx[name + ".ranges6"] = rng_t.detach().numpy()
        fx[name + ".scaled_vdim"] = sdim
        fx[name + ".scaled_vsize"] = npts.querier.scaled_vsize_np
        fx[name + ".radius_limit"] = npts.querier.radius_limit_np
    from models.rendering.diff_ray_marching import near_far_linear_ray_generation
    for (near, far, D) in ((2.0, 6.0, 400), (0.0, 3.5, 400), (0.1, 8.0, 400), (2.0, 6.0, 37)):
        _, _, _, ts = near_far_linear_ray_generation(torch.zeros(1, 3), torch.ones(1, 1, 3), D, near=near, far=far, jitter=0.)
        fx["t_%g_%g_%d" % (near, far, D)] = ts.reshape(-1).numpy()
    np.savez_compressed(os.path.join(OUT, "hyper.npz"), **fx)
    print("hyper", {k: v.tolist() for k, v in fx.items() if k.endswith("scaled_vdim")})


def golden_checkpoint_layout():
    """Key names / shapes / dtypes of the reference module's own state_dict, i.e. of the `{epoch}_net_ray_marching.pth`
    files written by models/base_model.py:85-99 (the checkpoint wire format, SURVEY 8(f) rank 3)."""
    import json
    cfg = scene.CONFIGS["tiny"]
    net, agg, npts, pts, opt = build_reference_net(cfg, 0.0)
    layout = {k: [list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in net.state_dict().items()}
    with open(os.path.join(OUT, "checkpoint_layout.json"), "w") as f:
        json.dump(dict(n_points=int(pts["xyz"].shape[0]), layout=layout), f, indent=1, sort_keys=True)
    print("checkpoint_layout:", len(layout), "tensors")


def golden_output_keys():
    """Key sets (and per-key trailing shapes) of the dict the reference NeuralPointsRayMarching.forward returns in the three modes the
    runners use (neural_points_volumetric_model.py:252-364): evaluation, training (zero_one_loss_items = conf_coefficient) and the
    point-growing probe (opt.prob == 1).  tests/test_gpu_shade.py asserts the drop-in forward returns exactly these."""
    import json
    cfg = scene.CONFIGS["tiny"]
    pixels = scene.centre_patch(cfg, 12)
    rays = scene.make_rays(cfg, pixels)
    res = {}
    for mode in ("eval", "train", "probe"):
        net, agg, npts, pts, opt = build_reference_net(cfg, 4.0, is_train=(mode == "train"))
        if mode == "probe":
            opt.prob = 1
        ctx = torch.enable_grad() if mode == "train" else torch.no_grad()
        with ctx:
            out = net(rays["campos"], rays["raydir"], bg_color=rays["bg_color"], camrotc2w=rays["camrotc2w"],
                      pixel_idx=rays["pixel_idx"], near=rays["near"], far=rays["far"], h=rays["h"], w=rays["w"],
                      intrinsic=rays["intrinsic"])
        res[mode] = {k: (list(v.shape[2:]) if isinstance(v, torch.Tensor) and v.dim() >= 2 else None) for k, v in out.items() if v is not None}
    with open(os.path.join(OUT, "output_keys.json"), "w") as f:
        json.dump(res, f, indent=1, sort_keys=True)
    print("output_keys:", {m: sorted(v) for m, v in res.items()})


def _param_names(fn):
    import inspect
    return [p.name for p in inspect.signature(fn).parameters.values() if p.kind in (p.POSITIONAL_OR_KEYWORD, p.KEYWORD_ONLY)]


def golden_reference_api():
    """The parts of the reference's interface that the drop-in seams of INTEGRATION.md must match, as the reference's own classes report
    them: method parameter names, the argparse namespace of the shipped flags, the aggregator's state-dict layout (in order) and the key
    set of its evaluation-mode forward.  tests/test_reference_contract.py checks pointnerf_b200 against this file."""
    import json
    ref_shim.install()
    from models.neural_points.point_query import lighting_fast_querier as RefQuerier
    from models.neural_points.neural_points import NeuralPoints as RefPoints
    from models.neural_points_volumetric_model import NeuralPointsRayMarching as RefMarch
    sig = {}
    for cls, names in ((RefQuerier, ("__init__", "query_points", "get_hyperparameters", "clean_up")),
                       (RefPoints, ("prune", "grow_points", "set_points")), (RefMarch, ("forward",))):
        for n in names:
            sig["%s.%s" % (cls.__name__, n)] = _param_names(getattr(cls, n))
    cfg = scene.CONFIGS["tiny"]
    net, agg, npts, pts, opt = build_reference_net(cfg, 4.0)
    rays = scene.make_rays(cfg, scene.centre_patch(cfg, 12))
    with torch.no_grad():
        out = net(rays["campos"], rays["raydir"], bg_color=rays["bg_color"], camrotc2w=rays["camrotc2w"], pixel_idx=rays["pixel_idx"],
                  near=rays["near"], far=rays["far"], h=rays["h"], w=rays["w"], intrinsic=rays["intrinsic"])
    res = dict(signatures=sig, opt=vars(opt),
               aggregator_state_dict=[[k, list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in agg.state_dict().items()],
               net_state_dict_keys=sorted(net.state_dict().keys()),
               forward_eval_keys=sorted(k for k, v in out.items() if v is not None))
    with open(os.path.join(OUT, "reference_api.json"), "w") as f:
        json.dump(res, f, indent=1, sort_keys=True)
    # positional_encoding of models/helpers/networks.py on a seeded input, for the (freqs, ori) pairs the hot path uses
    from models.helpers.networks import positional_encoding
    g = torch.Generator().manual_seed(0)
    x = torch.randn(7, 5, generator=g)
    fx = dict(x=x.numpy())
    for freqs, ori in ((3, False), (5, False), (4, True)):
        fx["pe_%d_%d" % (freqs, int(ori))] = positional_encoding(x, freqs, ori=ori).numpy()
    np.savez_compressed(os.path.join(OUT, "positional_encoding.npz"), **fx)
    print("reference_api:", len(sig), "signatures,", len(res["opt"]), "options")


if __name__ == "__main__":
    assert ref_shim.available(), "needs /root/reference"
    if len(sys.argv) > 1 and sys.argv[1] == "keys":
        golden_output_keys()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "api":
        golden_reference_api()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "order1":
        tiny = scene.CONFIGS["tiny"]
        golden_case("tiny_order1", tiny, scene.centre_patch(tiny, 40), alpha_bias=4.0, extra_flags=["--agg_intrp_order", "1"])
        sys.exit(0)
    tiny = scene.CONFIGS["tiny"]
    golden_case("tiny_opaque", tiny, scene.centre_patch(tiny, 40), alpha_bias=4.0)
    golden_case("tiny_thin_sr8", tiny, scene.centre_patch(tiny, 40), alpha_bias=0.0, SR=8)
    # agg_intrp_order = 1 (point_aggregators.py:573-599: alpha_branch on the K-aggregated feature), SURVEY 8(f) rank 4
    golden_case("tiny_order1", tiny, scene.centre_patch(tiny, 40), alpha_bias=4.0, extra_flags=["--agg_intrp_order", "1"])
    golden_probe("tiny_probe", tiny, scene.centre_patch(tiny, 40), alpha_bias=4.0)
    golden_hyper()
    golden_checkpoint_layout()
    golden_output_keys()
    golden_reference_api()
