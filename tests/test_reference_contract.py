"""CPU: the drop-in seams of INTEGRATION.md checked against what the reference's OWN classes report about themselves,
recorded in tests/golden/reference_api.json by oracle/make_golden.py (`python -m oracle.make_golden api`, which imports the
reference un-modified through oracle/ref_shim.py) -- the closest available proxy for "run/train_ft.py and run/render_vid.py drop in
unchanged" (the runners themselves do not import here: SURVEY 8c).

  seam A  lighting_fast_querier: constructor / query_points / get_hyperparameters / clean_up signatures
  seam B  NeuralPointsRayMarching.forward signature, install_into() on a class shaped as the reference's (its parameter names), option
          surface (check_opt on the reference's own argparse namespace), state-dict keys / shapes (= checkpoint wire format), optimiser
          parameter split (neural_points_volumetric_model.py:155-190), NeuralPoints.prune / grow_points / set_points signatures
  output  key sets of the reference forward in eval / train / probe mode == tests/golden/output_keys.json (the GPU tests assert the
          drop-in returns exactly those)
"""
import argparse
import inspect
import json
import os

import pytest
import torch
from torch import nn


@pytest.fixture(scope="module")
def ref(golden_dir):
    with open(os.path.join(golden_dir, "reference_api.json")) as f:
        return json.load(f)


def _names(fn):
    return [p.name for p in inspect.signature(fn).parameters.values() if p.kind in (p.POSITIONAL_OR_KEYWORD, p.KEYWORD_ONLY)]


def test_querier_seam_signatures(ref):
    from pointnerf_b200.point_query import lighting_fast_querier as Ours
    for m in ("__init__", "query_points", "get_hyperparameters", "clean_up"):
        # the class is resolved by NAME (neural_points.py:330-339): same name on purpose
        assert _names(getattr(Ours, m)) == ref["signatures"]["%s.%s" % (Ours.__name__, m)], m


def test_ray_marching_forward_signature_and_points_api(ref):
    from pointnerf_b200 import ray_marching as P
    sig = ref["signatures"]
    r, ours = sig["NeuralPointsRayMarching.forward"], _names(P.NeuralPointsRayMarching.forward)
    assert ours[:len(r)] == r, (r, ours)
    for m in ("prune", "grow_points"):
        assert _names(getattr(P.NeuralPoints, m)) == sig["NeuralPoints." + m], m
    # set_points: every keyword the reference accepts is accepted (ours ignores the ones the hot path does not use via **_)
    r = sig["NeuralPoints.set_points"]
    o = inspect.signature(P.NeuralPoints.set_points).parameters
    assert all((n in o) or any(p.kind == p.VAR_KEYWORD for p in o.values()) for n in r), r
    assert [n for n in r[:3]] == [n for n in list(o)[:3]]


def _reference_shaped_net(ref, golden_dir):
    """A module with the reference NeuralPointsRayMarching's parameter names and shapes (its checkpoint layout) and the reference's own
    argparse namespace as .opt."""
    with open(os.path.join(golden_dir, "checkpoint_layout.json")) as f:
        layout = json.load(f)["layout"]

    class NeuralPointsRayMarching(nn.Module):
        def __init__(self):
            super().__init__()
            self.neural_points, self.aggregator = nn.Module(), nn.Module()
            for k, (shape, dtype) in layout.items():
                *path, leaf = k.split(".")
                m = self
                for p in path:
                    if not hasattr(m, p):
                        m.add_module(p, nn.Module())
                    m = getattr(m, p)
                m.register_parameter(leaf, nn.Parameter(torch.zeros(shape, dtype=getattr(torch, dtype))))
            self.opt = argparse.Namespace(**ref["opt"])

        def forward(self, *args, **kwargs):
            raise AssertionError("the eager reference forward must have been replaced")

    return NeuralPointsRayMarching()


def test_option_surface_and_install_into_the_real_class(ref, golden_dir):
    from pointnerf_b200 import ray_marching as P
    net = _reference_shaped_net(ref, golden_dir)
    opt = net.opt
    P.check_opt(opt)                                      # the reference's own argparse namespace with the shipped flags is accepted
    bad = type(opt)(**vars(opt)); bad.agg_intrp_order = 0
    with pytest.raises(NotImplementedError):
        P.check_opt(bad)
    bad = type(opt)(**vars(opt)); bad.xyz_grad = 1
    with pytest.raises(NotImplementedError):
        P.check_opt(bad)
    cls = type(net)
    saved = {n: cls.__dict__.get(n) for n in P._PATCHED}
    try:
        P.install_into(cls)
        assert all(getattr(cls, n) is getattr(P.NeuralPointsRayMarching, n) for n in P._PATCHED)
        P._init_state(net)                                # launch state is created on the reference-shaped instance (no CUDA needed for this)
        assert net._pnb_ready and net.precision == "bf16x3" and net.frozen_ok
        # the model shell splits the optimisers on the parameter NAMES (neural_points_volumetric_model.py:176-190)
        names = [n for n, _ in net.named_parameters()]
        assert any(n.startswith("neural_points.") for n in names) and any(n.startswith("aggregator.") for n in names)
    finally:
        for n, v in saved.items():
            if v is None:
                delattr(cls, n)
            else:
                setattr(cls, n, v)


def test_state_dict_is_the_reference_wire_format(ref, golden_dir):
    from pointnerf_b200 import harness, scene
    from pointnerf_b200.ray_marching import PointAggregator
    mine = PointAggregator(harness.make_opt(scene.CONFIGS["tiny"])).state_dict()
    assert [[k, list(v.shape), str(v.dtype).replace("torch.", "")] for k, v in mine.items()] == ref["aggregator_state_dict"]
    layout = json.load(open(os.path.join(golden_dir, "checkpoint_layout.json")))["layout"]
    sd = ref["net_state_dict_keys"]
    assert sorted(sd) == sorted(layout.keys())              # the committed layout fixture is what the reference writes
    pt_keys = sorted(k for k in sd if k.startswith("neural_points."))
    assert pt_keys == ["neural_points.points_color", "neural_points.points_conf", "neural_points.points_dir",
                       "neural_points.points_embeding", "neural_points.xyz"]


def test_output_key_fixture_matches_the_reference(ref, golden_dir):
    """The eval-mode key set the reference's forward returned == the committed fixture the GPU tests use (guards the fixture itself)."""
    want = json.load(open(os.path.join(golden_dir, "output_keys.json")))
    assert ref["forward_eval_keys"] == sorted(want["eval"].keys())
