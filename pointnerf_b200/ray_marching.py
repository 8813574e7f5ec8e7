"""Host-side mirror of the reference's hot-path modules on top of libpnb200.so:

  PointAggregator        parameter container with the reference's names/shapes
                         (/root/reference/models/aggregators/point_aggregators.py:276-348:
                         block1.{0,2}, block3.{0,2}, alpha_branch.0, color_branch.{0,2,4,6})
  NeuralPoints           parameter container (xyz, points_embeding, points_conf, points_dir, points_color,
                         Rw2c) + querier (/root/reference/models/neural_points/neural_points.py:231-344)
  NeuralPointsRayMarching.forward(campos, raydir, ...)  -> the reference's output dict
                         (/root/reference/models/neural_points_volumetric_model.py:252-364)
  render_full(...)       the same computation with full-R outputs (fill_invalid already applied,
                         :87-123) and NO host synchronisation -- what bench.py times.
  probe_full(...)        render_full + the probe outputs of point growing (:331-351) for all rays, one kernel
                         (pnb_probe_maps) -- what runner.probe_frame / probe_holes use.

Only the shipped hot-path configuration (SURVEY.md section 8 head) is implemented; any other option
value raises NotImplementedError (no silent fallback).
"""
import math
import os

import torch
import torch.nn as nn

from . import lib as _lib
from .point_query import lighting_fast_querier, make_cam_opts

MLP_KEYS = ("block1.0", "block1.2", "block3.0", "block3.2", "alpha_branch.0",
            "color_branch.0", "color_branch.2", "color_branch.4", "color_branch.6")
MLP_SHAPES = ((256, 284), (256, 256), (256, 263), (256, 256), (1, 256), (128, 280), (128, 128), (128, 128), (3, 128))
MLP_KPAD = (288, 256, 272, 256, 256, 288, 128, 128, 128)  # rows of the W^T buffers handed to the kernels

_REQUIRED = dict(
    agg_dist_pers=20, agg_distance_kernel="linear", apply_pnt_mask=1, num_feat_freqs=3,
    dist_xyz_freq=5, dist_xyz_deno=0, num_viewdir_freqs=4, view_ori=0, shading_feature_mlp_layer1=2,
    shading_feature_mlp_layer2=0, shading_feature_mlp_layer3=2, shading_alpha_mlp_layer=1,
    shading_color_mlp_layer=4, shading_feature_num=256, act_type="LeakyReLU", act_super=1,
    point_features_dim=32, agg_feat_xyz_mode="None", agg_alpha_xyz_mode="None", agg_color_xyz_mode="None",
    which_agg_model="viewmlp", agg_weight_norm=1, point_conf_mode="1", point_dir_mode="1", point_color_mode="1",
)
_DEFAULTS = dict(view_ori=0, act_super=1, agg_weight_norm=1, apply_pnt_mask=1, which_agg_model="viewmlp",
                 dist_xyz_deno=0, agg_feat_xyz_mode="None", agg_alpha_xyz_mode="None", agg_color_xyz_mode="None",
                 shading_feature_mlp_layer2=0)


def check_opt(opt):
    """Reject (loudly) every option value outside the implemented configuration (SURVEY 8b)."""
    for k, want in _REQUIRED.items():
        have = getattr(opt, k, _DEFAULTS.get(k, want))
        if isinstance(want, (int, float)) and not isinstance(want, bool):
            ok = float(have) == float(want)
        else:
            ok = str(have) == str(want)
        if not ok:
            raise NotImplementedError("pnb200: option %s=%r is outside the implemented hot path (needs %r)" % (k, have, want))
    order = int(getattr(opt, "agg_intrp_order", 2))
    if order not in (1, 2):
        # agg_intrp_order 0 (features interpolated before the MLP) does not run in the reference either: viewmlp raises a shape error with
        # the shipped colour / direction inputs (point_aggregators.py:563 vs :552-555) and another one without them (block1 is built for
        # 224 inputs, :279-280, but receives the position encoding as well)
        raise NotImplementedError("pnb200: agg_intrp_order=%d is outside the implemented hot path (2, the shipped value, or 1)" % order)
    aw = getattr(opt, "agg_axis_weight", None)
    if aw is not None and any(float(a) != 1.0 for a in aw):
        raise NotImplementedError("pnb200: agg_axis_weight must be None or 1 1 1")
    if getattr(opt, "prob", 0) not in (0, 1):
        raise NotImplementedError("pnb200: opt.prob must be 0 or 1")
    if float(getattr(opt, "xyz_grad", 0) or 0) > 0:
        # the fused backward produces no d/d(xyz) (every shipped script has xyz_grad = 0): refuse instead of silently freezing xyz
        raise NotImplementedError("pnb200: xyz_grad > 0 (point positions as trainable parameters) is outside the implemented hot path")


def _to_list(x):
    if isinstance(x, torch.Tensor):
        return x.detach().reshape(-1).cpu().tolist()
    import numpy as np
    return [float(v) for v in np.asarray(x, dtype=np.float64).reshape(-1)]


class PointAggregator(nn.Module):
    """Parameters of the reference aggregator for the shipped viewmlp configuration; same state-dict keys."""

    def __init__(self, opt=None, seed=0):
        super().__init__()
        if opt is not None:
            check_opt(opt)
        self.opt = opt
        act = lambda: nn.LeakyReLU(inplace=True)
        self.block1 = nn.Sequential(nn.Linear(284, 256), act(), nn.Linear(256, 256), act())
        self.block3 = nn.Sequential(nn.Linear(263, 256), act(), nn.Linear(256, 256), act())
        self.alpha_branch = nn.Sequential(nn.Linear(256, 1))
        self.color_branch = nn.Sequential(nn.Linear(280, 128), act(), nn.Linear(128, 128), act(),
                                          nn.Linear(128, 128), act(), nn.Linear(128, 3))
        g = torch.Generator().manual_seed(seed)
        with torch.no_grad():
            for m in self.modules():
                if isinstance(m, nn.Linear):  # xavier-uniform, zero bias (helpers/networks.py:120-141)
                    bound = math.sqrt(6.0 / (m.in_features + m.out_features))
                    m.weight.copy_((torch.rand(m.weight.shape, generator=g) * 2 - 1) * bound)
                    m.bias.zero_()

    def mlp_dict(self):
        sd = self.state_dict()
        return {k: sd[k] for k in sd}


class MlpPack:
    """W^T (zero padded) buffers for the kernels, refreshed when any parameter's version changes."""

    def __init__(self):
        self.key = None
        self.wt = None
        self.bias = None
        self.desc = None
        self.packed = None   # tcgen05 operand images of block1/block3 (hi/lo bf16)
        self.key_l1 = None   # version key of block1.0 (weight, bias): what the hoisted per-point table depends on

    def get(self, agg):
        sd = {k: v for k, v in agg.named_parameters()}
        ws = [sd[k + ".weight"] for k in MLP_KEYS]
        bs = [sd[k + ".bias"] for k in MLP_KEYS]
        key = tuple((t.data_ptr(), t._version) for t in ws + bs)
        if key != self.key:
            self.wt, self.bias = [], []
            for w, b, shp, kp in zip(ws, bs, MLP_SHAPES, MLP_KPAD):
                assert tuple(w.shape) == shp, "MLP tensor shape %s != %s" % (tuple(w.shape), shp)
                wt = torch.zeros((kp, shp[0]), dtype=torch.float32, device=w.device)
                wt[:shp[1]].copy_(w.detach().t())
                self.wt.append(wt.contiguous())
                self.bias.append(b.detach().contiguous().float())
            d = _lib.Mlp()
            for i in range(9):
                d.w[i] = self.wt[i].data_ptr()
                d.b[i] = self.bias[i].data_ptr()
            self.desc = d
            self.key = key
            self.key_l1 = (key[0], key[9])
            lib = _lib.load()
            nb = lib.pnb_mlp_pack_bytes()
            if self.packed is None or self.packed.device != ws[0].device:
                self.packed = torch.empty(nb, dtype=torch.uint8, device=ws[0].device)
            _lib.check(lib.pnb_mlp_pack(_lib.C.byref(d), self.packed.data_ptr(), nb,
                                        torch.cuda.current_stream(ws[0].device).cuda_stream), "pnb_mlp_pack")
        return self.desc


def points_desc_of(npnts):
    """pnb_points_t over the parameter tensors of a NeuralPoints-like module (ours or the reference's)."""
    if npnts.Rw2c is not None and npnts.Rw2c.dim() != 2:
        raise NotImplementedError("pnb200: per-point Rw2c is not part of the implemented hot path")
    for name in ("points_embeding", "points_color", "points_dir", "points_conf"):
        if getattr(npnts, name, None) is None:
            raise NotImplementedError("pnb200: neural_points.%s is None; the hot path needs point_{conf,dir,color}_mode=1" % name)
    p = _lib.Points()
    tens = (npnts.xyz, npnts.points_embeding, npnts.points_color, npnts.points_dir, npnts.points_conf)
    for t in tens:
        if not (t.is_cuda and t.is_contiguous() and t.dtype == torch.float32):
            raise _lib.PnbError("pnb200: point tensors must be contiguous fp32 CUDA tensors")
    if npnts.points_embeding.shape[-1] != 32:
        raise NotImplementedError("pnb200: point_features_dim must be 32")
    p.xyz, p.emb, p.color, p.dir, p.conf = (t.data_ptr() for t in tens)
    p.N = npnts.xyz.shape[0]
    return p


def rw2c_host_of(npnts):
    """Rw2c as 9 host floats, cached on the module per tensor version (one tiny D2H copy when it changes)."""
    R = npnts.Rw2c
    if R is None:
        return None
    key = (R.data_ptr(), R._version)
    if getattr(npnts, "_pnb_rw2c_key", None) != key:
        npnts._pnb_rw2c_host = _to_list(R)
        npnts._pnb_rw2c_key = key
    return npnts._pnb_rw2c_host


class NeuralPoints(nn.Module):
    """Parameter container + querier with the reference's attribute names (neural_points.py:231-344)."""

    def __init__(self, opt, device):
        super().__init__()
        self.opt = opt
        self.device = device
        self.xyz = None
        self.points_embeding = self.points_conf = self.points_dir = self.points_color = None
        self.Rw2c = torch.eye(3)
        self.querier = lighting_fast_querier(device, opt)

    def set_points(self, points_xyz, points_embeding, points_color=None, points_dir=None, points_conf=None,
                   parameter=True, Rw2c=None, **_):
        mk = (lambda t, g: nn.Parameter(t.contiguous(), requires_grad=g)) if parameter else (lambda t, g: t.contiguous())
        o = self.opt
        self.xyz = mk(points_xyz, getattr(o, "xyz_grad", 0) > 0)
        self.points_embeding = mk(points_embeding, getattr(o, "feat_grad", 1) > 0)
        self.points_color = mk(points_color, getattr(o, "color_grad", 1) > 0)
        self.points_dir = mk(points_dir, getattr(o, "dir_grad", 1) > 0)
        self.points_conf = mk(points_conf, getattr(o, "conf_grad", 1) > 0)
        if "Rw2c" in self._parameters:
            del self._parameters["Rw2c"]
        # a supplied Rw2c is part of the state dict, as in the reference (neural_points.py:463-467); the default stays a plain eye(3)
        self.Rw2c = torch.eye(3, device=points_xyz.device) if Rw2c is None else \
            nn.Parameter(Rw2c.to(points_xyz.device).float().contiguous(), requires_grad=False)
        self.querier.clean_up()

    def reset_querier(self):
        self.querier.clean_up()

    def _wrap(self, t, grad_flag):
        t = nn.Parameter(t.contiguous())
        t.requires_grad = grad_flag
        return t

    def prune(self, thresh):
        """/root/reference/models/neural_points/neural_points.py:347-370: keep points with conf >= thresh.
        Parameters are re-created (the caller rebuilds its optimisers, run/train_ft.py:834-842); the cached voxel
        grid is invalidated."""
        o = self.opt
        mask = self.points_conf[0, ..., 0] >= thresh
        self.xyz = self._wrap(self.xyz[mask, :], getattr(o, "xyz_grad", 0) > 0)
        self.points_embeding = self._wrap(self.points_embeding[:, mask, :], getattr(o, "feat_grad", 1) > 0)
        self.points_conf = self._wrap(self.points_conf[:, mask, :], getattr(o, "conf_grad", 1) > 0)
        self.points_dir = self._wrap(self.points_dir[:, mask, :], getattr(o, "dir_grad", 1) > 0)
        self.points_color = self._wrap(self.points_color[:, mask, :], getattr(o, "color_grad", 1) > 0)
        self.querier.clean_up()
        return int((~mask).sum())

    def grow_points(self, add_xyz, add_embedding, add_color, add_dir, add_conf, add_eulers=None, add_Rw2c=None):
        """/root/reference/models/neural_points/neural_points.py:373-399: append points (new parameters)."""
        o = self.opt
        self.xyz = self._wrap(torch.cat([self.xyz, add_xyz], dim=0), getattr(o, "xyz_grad", 0) > 0)
        self.points_embeding = self._wrap(torch.cat([self.points_embeding, add_embedding[None, ...]], dim=1), getattr(o, "feat_grad", 1) > 0)
        self.points_conf = self._wrap(torch.cat([self.points_conf, add_conf[None, ...]], dim=1), getattr(o, "conf_grad", 1) > 0)
        self.points_dir = self._wrap(torch.cat([self.points_dir, add_dir[None, ...]], dim=1), getattr(o, "dir_grad", 1) > 0)
        self.points_color = self._wrap(torch.cat([self.points_color, add_color[None, ...]], dim=1), getattr(o, "color_grad", 1) > 0)
        self.querier.clean_up()

    def points_desc(self):
        return points_desc_of(self)


class _RenderFn(torch.autograd.Function):
    """Differentiable face of the fused path: ray_color[R,3] = f(points_embeding, points_color, points_dir,
    points_conf, 18 MLP tensors).  Backward = pnb_shade_backward (activations recomputed, layer GEMMs on tcgen05 / BF16x3)."""

    @staticmethod
    def forward(ctx, mod, run_args, emb, color, pdir, conf, *mlp_params):
        q, ray_color, opacity, bg_T, ray_mask = mod._run(*run_args)
        ctx.mod = mod
        ctx.q = q
        ctx.generation = mod._generation          # the backward recomputes from the query / sigma_rgb buffers of THIS run
        ctx.o = mod._last_opts
        ctx.n_valid = q.counters["n_valid"]
        ctx.n_pairs = q.counters["n_pairs"]
        ctx.sigma_rgb = mod._sigma_rgb          # forward (sigma, rgb) per candidate; valid until the next _run
        ctx.needs = [t.requires_grad for t in (emb, color, pdir, conf)]
        ctx.mlp_shapes = [tuple(t.shape) for t in mlp_params]
        ctx.mark_non_differentiable(opacity, bg_T, ray_mask)
        return ray_color, opacity, bg_T, ray_mask

    @staticmethod
    def backward(ctx, g_color, g_op, g_bg, g_mask):
        lib = _lib.load()
        mod, q = ctx.mod, ctx.q
        if mod._generation != ctx.generation:
            raise _lib.PnbError("pnb200: backward() of a forward whose query / sigma_rgb buffers were overwritten by a later call of the "
                                "same module (two forwards before one backward, or an eval render in between); call backward() "
                                "before the next forward")
        npnts = mod.neural_points
        dev = g_color.device
        g_color = g_color.contiguous().float()
        N = npnts.xyz.shape[0]
        outs = []
        for need, shape in zip(ctx.needs, ((1, N, 32), (1, N, 3), (1, N, 3), (1, N, 1))):
            outs.append(torch.zeros(shape, dtype=torch.float32, device=dev) if need else None)
        dwt = [torch.zeros_like(w) for w in mod._mlp.wt]
        dbs = [torch.zeros_like(b) for b in mod._mlp.bias]
        nb = lib.pnb_backward_bytes(max(ctx.n_valid, 1), q.desc.cap_samples)
        if getattr(mod, "_bwd_ws", None) is None or mod._bwd_ws.numel() < nb:
            mod._bwd_ws = torch.empty(nb, dtype=torch.uint8, device=dev)
        wp = (_lib.C.c_void_p * 9)(*[t.data_ptr() for t in dwt])
        bp = (_lib.C.c_void_p * 9)(*[t.data_ptr() for t in dbs])
        pts = points_desc_of(npnts)
        mlp = mod._mlp.get(mod.aggregator)
        stream = torch.cuda.current_stream(dev).cuda_stream
        ptr = lambda t: t.data_ptr() if t is not None else None
        if getattr(mod, "_bwd_err", None) is None or mod._bwd_err.device != dev:
            mod._bwd_err = torch.zeros(4, dtype=torch.int32, device=dev)     # checked (synchronising) by check_errors()
        # opt.pnb_bwd_fp32: 0 tensor-core GEMMs (default) | 1 fp32 CUDA-core GEMMs | 4 fp32 recompute + tensor-core dX / dW
        # (fp32-faithful LeakyReLU masks) | 2 (diagnostic) three-part split in every tensor-core GEMM
        flags = int(getattr(mod.opt, "pnb_bwd_fp32", 0))
        _lib.check(lib.pnb_shade_backward(_lib.C.byref(q.desc), _lib.C.byref(pts), _lib.C.byref(mlp), _lib.C.byref(ctx.o),
                                          ctx.sigma_rgb.data_ptr(), g_color.data_ptr(), int(ctx.n_valid), int(ctx.n_pairs), ptr(outs[0]),
                                          ptr(outs[1]), ptr(outs[2]), ptr(outs[3]), wp, bp, mod._bwd_ws.data_ptr(),
                                          mod._bwd_ws.numel(), flags, mod._bwd_err.data_ptr(), stream), "pnb_shade_backward")
        grads = []
        for i, shp in enumerate(MLP_SHAPES):                 # W^T [K_pad, N] -> nn.Linear weight [N, K]
            grads.append(dwt[i][:shp[1]].t().contiguous().view(ctx.mlp_shapes[2 * i]))
            grads.append(dbs[i].view(ctx.mlp_shapes[2 * i + 1]))
        return (None, None, outs[0], outs[1], outs[2], outs[3], *grads)


class _AuxFn(torch.autograd.Function):
    """`weight`, `conf_coefficient`, `blend_weight` of the reference's output dict for the R' hit rays, one kernel on the compacted
    query (pnb_aux_outputs) instead of a dense export + ~20 eager torch ops; differentiable with respect to points_conf through
    conf_coefficient (straight-through clamp, neural_points.py:713; pnb_aux_conf_backward)."""

    @staticmethod
    def forward(ctx, mod, q, inds, opacity, conf):
        lib = _lib.load()
        npnts = mod.neural_points
        dev = opacity.device
        n = int(inds.shape[0])
        SR, K = int(q.desc.SR), int(q.desc.K)
        wgt = torch.empty((n, SR, K), dtype=torch.float32, device=dev)
        cc = torch.empty((n, SR, K), dtype=torch.float32, device=dev)
        blend = torch.empty((n, SR), dtype=torch.float32, device=dev)
        pts = points_desc_of(npnts)
        stream = torch.cuda.current_stream(dev).cuda_stream
        _lib.check(lib.pnb_aux_outputs(_lib.C.byref(q.desc), _lib.C.byref(pts), inds.data_ptr(), n, opacity.data_ptr(), wgt.data_ptr(),
                                       cc.data_ptr(), blend.data_ptr(), stream), "pnb_aux_outputs")
        ctx.mod, ctx.q, ctx.inds, ctx.generation = mod, q, inds, mod._generation
        ctx.conf_shape = tuple(conf.shape)
        ctx.mark_non_differentiable(wgt, blend)
        return wgt, cc, blend

    @staticmethod
    def backward(ctx, g_w, g_cc, g_b):
        if g_cc is None:
            return None, None, None, None, None
        mod, q = ctx.mod, ctx.q
        if mod._generation != ctx.generation:
            raise _lib.PnbError("pnb200: backward() of a forward whose query buffers were overwritten by a later call of the same module")
        lib = _lib.load()
        g_cc = g_cc.contiguous().float()
        g_conf = torch.zeros(ctx.conf_shape, dtype=torch.float32, device=g_cc.device)
        stream = torch.cuda.current_stream(g_cc.device).cuda_stream
        _lib.check(lib.pnb_aux_conf_backward(_lib.C.byref(q.desc), ctx.inds.data_ptr(), int(ctx.inds.shape[0]), g_cc.data_ptr(),
                                             g_conf.data_ptr(), stream), "pnb_aux_conf_backward")
        return None, None, None, None, g_conf


def _init_state(mod):
    """Per-module launch state (weight packs, workspaces).  Works on our module and on the reference's
    NeuralPointsRayMarching after install_into()."""
    opt = mod.opt
    check_opt(opt)
    for k, want in (("which_render_func", "radiance"), ("which_blend_func", "alpha"), ("which_tonemap_func", "off")):
        if getattr(opt, k, want) != want:
            raise NotImplementedError("pnb200: %s=%r unsupported (needs %r)" % (k, getattr(opt, k), want))
    mod._mlp = MlpPack()
    mod._sigma_rgb = None
    mod._tc_ws = None
    mod._err = None
    mod._generation = 0
    mod._pre = None              # hoisted layer-1 table of the frozen pipeline + the versions it was computed from
    mod._pre_key = None
    mod._valid_per_ray = 0.0     # densest call seen so far (valid samples per ray): sizes the shading workspace
    mod._status_pending = []     # (event, pinned [err, query counters], R) of render_full() calls not yet checked
    mod._status_free = []
    mod._max_valid = 0
    # "bf16x3": per-pair MLPs on tcgen05 tensor cores with the error-compensated split (default);
    # "fp32": the exact-fp32 CUDA-core kernel.
    mod.precision = getattr(opt, "pnb_precision", "bf16x3")
    if mod.precision not in ("bf16x3", "fp32"):
        raise NotImplementedError("pnb200: pnb_precision=%r (bf16x3 | fp32)" % mod.precision)
    # pnb_frozen: 1 (default) = calls that need no gradient (rendering, evaluation) run the frozen-cloud pair kernel
    # (k_shade_tc8: the point-only inputs of block1.0 hoisted into a per-point table, rebuilt when points_embeding or
    # block1.0 change); 0 = always the general kernel (k_shade_tc7), which is what training steps use in either case.
    mod.frozen_ok = bool(int(getattr(opt, "pnb_frozen", 1)))
    mod.dbg_flags = int(getattr(opt, "pnb_dbg_flags", 0)) | int(os.environ.get("PNB_DBG_FLAGS_DEFAULT", "0"))   # (env: kernel experiments under the test-suite)
    mod.last = None
    mod._pnb_ready = True


_PATCHED = ("forward", "_run", "check_errors", "render_full", "_point_pre", "_poll_status", "_queue_status", "probe_full")


def install_into(reference_cls):
    """Patch the reference's models.neural_points_volumetric_model.NeuralPointsRayMarching class in place: its
    instances keep their own parameters (self.neural_points.*, self.aggregator.*) and gain the fused forward
    (INTEGRATION.md, seam B).  self.neural_points.querier must be pointnerf_b200's lighting_fast_querier (seam A)."""
    for name in _PATCHED:
        setattr(reference_cls, name, getattr(NeuralPointsRayMarching, name))
    return reference_cls


def reference_forward(self, *args, **kwargs):
    """Function form of the patched forward (bind it as NeuralPointsRayMarching.forward of the reference)."""
    for name in _PATCHED[1:]:
        if not hasattr(type(self), name):
            setattr(type(self), name, getattr(NeuralPointsRayMarching, name))
    return NeuralPointsRayMarching.forward(self, *args, **kwargs)


class NeuralPointsRayMarching(nn.Module):
    """forward() keeps the reference's signature and output dict (neural_points_volumetric_model.py:252-364)."""

    def __init__(self, aggregator=None, neural_points=None, opt=None, **kwargs):
        super().__init__()
        self.aggregator = aggregator
        self.neural_points = neural_points
        self.opt = opt
        _init_state(self)

    # -------------------------------------------------------------------------------------------------
    def _point_pre(self, mlp_desc, pts_desc, stream):
        """Hoisted layer-1 table of the frozen pipeline (pnb_point_pre), rebuilt when points_embeding or block1.0 changed."""
        emb = self.neural_points.points_embeding
        key = (emb.data_ptr(), emb._version, emb.shape[1], self._mlp.key_l1)
        if key != self._pre_key:
            lib = _lib.load()
            nb = lib.pnb_point_pre_bytes(int(pts_desc.N))
            if self._pre is None or self._pre.numel() * 4 < nb or self._pre.device != emb.device:
                self._pre = torch.empty((nb + 3) // 4, dtype=torch.float32, device=emb.device)
            _lib.check(lib.pnb_point_pre(_lib.C.byref(pts_desc), _lib.C.byref(mlp_desc), self._pre.data_ptr(), self._pre.numel() * 4,
                                         stream), "pnb_point_pre")
            self._pre_key = key
        return self._pre

    def _poll_status(self, block=False):
        """Deferred device status of earlier render_full() / forward() calls ([err, query counters, backward err] copied to pinned
        memory behind the kernels).  Non-blocking unless `block`; raises PnbError for a call that dropped samples or timed out."""
        pend = self._status_pending
        while pend and (block or pend[0][0].query()):
            ev, host, R = pend.pop(0)
            ev.synchronize()
            err, n_valid, bwd_err = int(host[0]), int(host[1 + _lib.QC["n_valid"]]), int(host[17])
            self._status_free.append(host)
            if bwd_err != 0:
                self._bwd_err.zero_()
                raise _lib.PnbError("pnb200: tcgen05 GEMM pipeline time-out in an earlier backward pass (code %d)" % bwd_err)
            self._valid_per_ray = max(self._valid_per_ray, n_valid / max(R, 1))
            if err == 9:
                raise _lib.PnbOverflow("pnb200: an earlier render_full() produced %d valid samples, more than its shading workspace held "
                                       "(the extra samples were dropped); the workspace has been enlarged - render the frame again, or "
                                       "call check_errors() after each frame, or set opt.pnb_max_valid_per_ray" % n_valid)
            if err != 0:
                raise _lib.PnbError("pnb200: tcgen05 pipeline time-out (code %d) in an earlier render_full()" % err)

    # -------------------------------------------------------------------------------------------------
    def _run(self, campos, raydir, camrotc2w, near, far, bg_color, want_counters, t=None, frozen=False):
        if not getattr(self, "_pnb_ready", False):
            _init_state(self)           # reference module patched by install_into(): state is created lazily
        lib = _lib.load()
        npnts, opt = self.neural_points, self.opt
        raydir = raydir[0].contiguous() if raydir.dim() == 3 else raydir.contiguous()
        dev = raydir.device
        self._poll_status(block=False)
        # camera scalars go to the kernels by value: host lists / CPU tensors cost nothing, device tensors
        # cost one small D2H copy (the reference does the same with near/far/intrinsic, neural_points.py:704)
        cp, rt, bg = _to_list(campos)[:3], _to_list(camrotc2w)[:9], _to_list(bg_color)[:3]
        q = npnts.querier.run_query(npnts.xyz.detach(), raydir, cp, float(near), float(far), t=t, want_counters=want_counters)
        o = make_cam_opts(cp, rt, Rw2c=rw2c_host_of(npnts),
                          vsize_z=float(opt.vsize[2]), bg_color=bg, raydist_mode_unit=int(getattr(opt, "raydist_mode_unit", 0)),
                          agg_intrp_order=int(getattr(opt, "agg_intrp_order", 2)))
        cap = q.desc.cap_samples
        self._generation += 1
        if self._sigma_rgb is None or self._sigma_rgb.shape[0] < cap or self._sigma_rgb.device != dev:
            self._sigma_rgb = torch.empty((cap, 4), dtype=torch.float32, device=dev)
        mlp = self._mlp.get(self.aggregator)
        pts = points_desc_of(npnts)
        stream = torch.cuda.current_stream(dev).cuda_stream
        if self.precision == "fp32":
            _lib.check(lib.pnb_shade_forward(_lib.C.byref(q.desc), _lib.C.byref(pts), _lib.C.byref(mlp), _lib.C.byref(o),
                                             self._sigma_rgb.data_ptr(), None, 0, stream), "pnb_shade_forward")
        else:
            # capacity of the shading workspace in valid samples (1 KB each): exact when the caller paid for the counters
            # (forward()), otherwise the densest frame seen so far with 25 % head-room, at least opt.pnb_max_valid_per_ray per ray;
            # an overflow is safe on the device (dropped samples contribute nothing) and is reported by check_errors() /
            # the next call (_poll_status)
            per_ray = max(float(getattr(opt, "pnb_max_valid_per_ray", 10)), 1.25 * self._valid_per_ray)
            max_valid = int(min(q.R * q.SR, max(min(1 << 20, q.R * q.SR), math.ceil(q.R * per_ray))))
            if want_counters and getattr(q, "counters", None):
                n_valid = int(q.counters.get("n_valid", 0))
                self._valid_per_ray = max(self._valid_per_ray, n_valid / max(q.R, 1))
                max_valid = max(max_valid, n_valid)
            max_valid = max(max_valid, 128)
            self._max_valid = max_valid
            nb = lib.pnb_shade_tc_bytes(max_valid)
            if self._tc_ws is None or self._tc_ws.numel() < nb or self._tc_ws.device != dev:
                self._tc_ws = None
                self._tc_ws = torch.empty(nb, dtype=torch.uint8, device=dev)
            if self._err is None or self._err.device != dev:
                self._err = torch.zeros(512, dtype=torch.int32, device=dev)   # [0] status, [2:64] cycle counters, [64:] per-CTA cycles (int64)
            else:
                self._err[:1].zero_()
            flags = _lib.TC_PAIRS | _lib.TC_COLOR | (self.dbg_flags << 8)
            pre_ptr = None
            if frozen and self.frozen_ok:
                pre_ptr = self._point_pre(mlp, pts, stream).data_ptr()
                flags |= _lib.TC_FROZEN
            _lib.check(lib.pnb_shade_forward_tc(_lib.C.byref(q.desc), _lib.C.byref(pts), _lib.C.byref(mlp),
                                                self._mlp.packed.data_ptr(), pre_ptr, _lib.C.byref(o), self._sigma_rgb.data_ptr(),
                                                self._tc_ws.data_ptr(), self._tc_ws.numel(), max_valid, flags,
                                                self._err.data_ptr(), stream), "pnb_shade_forward_tc")
        R, SR = q.R, q.SR
        ray_color = torch.empty((R, 3), dtype=torch.float32, device=dev)
        opacity = torch.empty((R, SR), dtype=torch.float32, device=dev)
        bg_T = torch.empty((R,), dtype=torch.float32, device=dev)
        ray_mask = torch.empty((R,), dtype=torch.int8, device=dev)
        _lib.check(lib.pnb_composite_forward(_lib.C.byref(q.desc), _lib.C.byref(o), self._sigma_rgb.data_ptr(),
                                             ray_color.data_ptr(), opacity.data_ptr(), bg_T.data_ptr(),
                                             ray_mask.data_ptr(), stream), "pnb_composite_forward")
        self.last = q
        self._last_opts = o
        return q, ray_color, opacity, bg_T, ray_mask

    def check_errors(self):
        """Synchronising check of the device-side status of the tensor-core path: raises PnbOverflow (after enlarging the
        workspace for the next call) when the last call dropped samples, PnbError on a pipeline time-out."""
        if getattr(self, "_status_pending", None):
            self._poll_status(block=True)
        be = getattr(self, "_bwd_err", None)
        if be is not None:
            code = int(be[0].item())
            if code != 0:
                be.zero_()
                raise _lib.PnbError("pnb200: tcgen05 GEMM pipeline time-out in the backward pass (code %d)" % code)
        if self._err is not None:
            code = int(self._err[0].item())
            if code != 0:
                self._err[:1].zero_()
            if code == 9:
                n_valid = int(self.last.counters_tensor()[_lib.QC["n_valid"]].item())
                self._valid_per_ray = max(self._valid_per_ray, n_valid / max(self.last.R, 1))
                raise _lib.PnbOverflow("pnb200: %d valid samples, more than the shading workspace held (%d): the extra samples were dropped; "
                                       "the workspace has been enlarged for the next call (or set opt.pnb_max_valid_per_ray)"
                                       % (n_valid, self._max_valid))
            if code != 0:
                raise _lib.PnbError("pnb200: tcgen05 pipeline time-out (code %d)" % code)

    def _queue_status(self, q, dev):
        """Copies the device status of the call just issued to pinned memory behind its kernels (no host synchronisation); a later
        call (_poll_status) or check_errors() raises it."""
        if self._err is None or self.precision == "fp32":
            return
        host = self._status_free.pop() if self._status_free else torch.zeros(18, dtype=torch.int32).pin_memory()
        host[:1].copy_(self._err[:1], non_blocking=True)
        host[1:17].copy_(q.counters_tensor(), non_blocking=True)
        be = getattr(self, "_bwd_err", None)
        if be is not None:
            host[17:18].copy_(be[:1], non_blocking=True)
        else:
            host[17] = 0
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(dev))
        self._status_pending.append((ev, host, q.R))

    def render_full(self, campos, raydir, camrotc2w, near, far, bg_color, t=None):
        """Full-R outputs, fill_invalid semantics, no host sync: dict(coarse_raycolor [1,R,3],
        coarse_point_opacity [1,R,SR], coarse_is_background [1,R,1], ray_mask [1,R]).  No gradients (frozen-cloud pipeline).
        The device status of the call (workspace overflow, time-out) is copied to pinned memory behind the kernels and raised
        by a LATER call or by check_errors(); runner.render_image checks it before returning."""
        q, ray_color, opacity, bg_T, ray_mask = self._run(campos, raydir, camrotc2w, near, far, bg_color, False, t=t, frozen=True)
        self._queue_status(q, ray_color.device)
        return dict(coarse_raycolor=ray_color[None], coarse_point_opacity=opacity[None],
                    coarse_is_background=bg_T[None, :, None], ray_mask=ray_mask[None])

    def probe_full(self, campos, raydir, camrotc2w, near, far, bg_color, t=None, want_argmax=False):
        """render_full() plus the probe outputs of point growing for all R rays (neural_points_volumetric_model.py:331-351 followed by
        fill_invalid / unmask, :87-123; one pnb_probe_maps kernel on the compacted query, no dense export, no host sync).  Adds
        ray_max_shading_opacity [1,R,1], ray_max_sample_loc_w [1,R,3], ray_max_far_dist [1,R,1], shading_avg_color [1,R,3],
        shading_avg_dir [1,R,3], shading_avg_conf [1,R,1], shading_avg_embedding [1,R,32] (zeros on rays without a neighbour) and,
        with want_argmax, ray_max_slot [1,R] int32 (the arg-max sample slot, -1 without a neighbour).  Status as render_full."""
        q, ray_color, opacity, bg_T, ray_mask = self._run(campos, raydir, camrotc2w, near, far, bg_color, False, t=t, frozen=True)
        dev = ray_color.device
        R = q.R
        # one allocation carved into contiguous maps; the embedding block comes first (16-byte aligned rows for pnb_probe_select)
        flat = torch.empty((R * 44,), dtype=torch.float32, device=dev)
        emb = flat[:R * 32].view(R, 32)
        loc, col, pdir = (flat[R * o:R * (o + 3)].view(R, 3) for o in (32, 35, 38))
        op_max, far_d, conf = (flat[R * o:R * (o + 1)].view(R, 1) for o in (41, 42, 43))
        argmax = torch.empty((R,), dtype=torch.int32, device=dev) if want_argmax else None
        lib = _lib.load()
        pts = points_desc_of(self.neural_points)
        _lib.check(lib.pnb_probe_maps(_lib.C.byref(q.desc), _lib.C.byref(pts), opacity.data_ptr(), op_max.data_ptr(), loc.data_ptr(),
                                      far_d.data_ptr(), col.data_ptr(), pdir.data_ptr(), conf.data_ptr(), emb.data_ptr(),
                                      argmax.data_ptr() if argmax is not None else None,
                                      torch.cuda.current_stream(dev).cuda_stream), "pnb_probe_maps")
        self._queue_status(q, dev)
        out = dict(coarse_raycolor=ray_color[None], coarse_point_opacity=opacity[None], coarse_is_background=bg_T[None, :, None],
                   ray_mask=ray_mask[None], ray_max_shading_opacity=op_max[None], ray_max_sample_loc_w=loc[None],
                   ray_max_far_dist=far_d[None], shading_avg_color=col[None], shading_avg_dir=pdir[None], shading_avg_conf=conf[None],
                   shading_avg_embedding=emb[None])
        if argmax is not None:
            out["ray_max_slot"] = argmax[None]
        return out

    def forward(self, campos, raydir, gt_image=None, bg_color=None, camrotc2w=None, pixel_idx=None, near=None,
                far=None, focal=None, h=None, w=None, intrinsic=None, **kargs):
        if "bg_ray" in kargs:
            raise NotImplementedError("pnb200: bg_ray input is not part of the implemented hot path")
        near_f = float(torch.min(near)) if isinstance(near, torch.Tensor) else float(near)
        far_f = float(torch.max(far)) if isinstance(far, torch.Tensor) else float(far)
        bg = bg_color if bg_color is not None else torch.zeros(3)
        run_args = (campos, raydir, camrotc2w, near_f, far_f, bg, True)
        npnts, agg = self.neural_points, self.aggregator
        train = torch.is_grad_enabled() and any(
            t is not None and t.requires_grad for t in
            [npnts.points_embeding, npnts.points_color, npnts.points_dir, npnts.points_conf] + list(agg.parameters()))
        if train:
            sd = dict(agg.named_parameters())
            mlp_params = []
            for k in MLP_KEYS:
                mlp_params += [sd[k + ".weight"], sd[k + ".bias"]]
            ray_color, opacity, bg_T, ray_mask = _RenderFn.apply(self, run_args, npnts.points_embeding, npnts.points_color,
                                                                 npnts.points_dir, npnts.points_conf, *mlp_params)
            q = self.last
        else:
            q, ray_color, opacity, bg_T, ray_mask = self._run(*run_args, frozen=True)
        # the shading workspace was sized from the query counters (no overflow possible); a pipeline time-out of this call or of the
        # previous backward is raised by the next call / check_errors() instead of stalling the host here until the forward has finished
        self._queue_status(q, ray_color.device)
        # compact to the R' rays the reference returns (one host sync already paid for the counters)
        # (the number of hit rays is already on the host with the query counters: no second synchronisation for the compaction)
        inds = torch.nonzero_static(ray_mask, size=int(q.counters["R2"]))[:, 0] if getattr(q, "counters", None) else torch.nonzero(ray_mask)[:, 0]
        out = {}
        out["coarse_raycolor"] = ray_color[inds][None]
        out["coarse_point_opacity"] = opacity[inds][None]
        out["coarse_is_background"] = bg_T[inds][None, :, None]
        # queried_shading: 1 where no sample of the ray is valid (:290) -- rays in R' always have one
        out["queried_shading"] = torch.zeros((1, inds.shape[0], 3), dtype=torch.float32, device=ray_color.device)
        out["ray_mask"] = ray_mask[None]
        opt = self.opt
        want_aux = (getattr(opt, "sparse_loss_weight", 0) > 0) or ("conf_coefficient" in getattr(opt, "zero_one_loss_items", [])) \
            or getattr(opt, "prob", 0) != 0                       # point_aggregators.py:812-813
        if want_aux and inds.shape[0] > 0 and getattr(opt, "prob", 0) != 1:
            # weight / conf_coefficient / blend_weight of the reference dict (:325-329): one kernel on the compacted query
            wgt, conf_coefficient, blend = _AuxFn.apply(self, q, inds, opacity, npnts.points_conf)
            out["weight"] = wgt[None]
            out["blend_weight"] = blend[None, ..., None]
            out["conf_coefficient"] = conf_coefficient[None]
        elif want_aux and inds.shape[0] > 0:
            # probe pass (opt.prob == 1, point growing): the same three outputs with eager torch ops on the dense export, which the
            # probe outputs below need anyway
            cam = make_cam_opts(_to_list(campos)[:3], _to_list(camrotc2w)[:9])
            ex = q.export(cam, want_pers=False, want_dirs=False)
            pidx = ex["sample_pidx"]
            mask = pidx >= 0
            idx = pidx.clamp(min=0).long()
            d = npnts.xyz.detach()[idx] - ex["sample_loc_w"][:, :, None, :]
            wgt = mask * (1.0 / torch.clamp(torch.norm(d, dim=-1), min=1e-6))
            wgt = wgt / torch.clamp(torch.sum(wgt, dim=-1, keepdim=True), min=1e-8)
            # index_select (as the reference, neural_points.py:717): its backward is one index_add_, not a sort-based scatter
            c0 = torch.index_select(npnts.points_conf[0, :, 0], 0, idx.reshape(-1)).view(idx.shape)
            conf_coefficient = c0 - (c0 - torch.clamp(c0, min=0.0001, max=1)).detach()
            op = out["coarse_point_opacity"][0].detach()
            acc = torch.cumprod(1. - op + 1e-10, dim=-1)
            acc_T = torch.cat([torch.ones_like(acc[:, :1]), acc[:, :-1]], dim=-1)
            out["weight"] = wgt[None].detach()
            out["blend_weight"] = (op * acc_T)[None, ..., None]
            out["conf_coefficient"] = conf_coefficient[None]
            if getattr(opt, "prob", 0) == 1:
                # probe outputs for point growing (neural_points_volumetric_model.py:331-351), same torch ops on the
                # dense export: arg-max-opacity sample of every ray and the weighted average of its neighbours
                K = pidx.shape[-1]
                omax, oind = torch.max(out["coarse_point_opacity"], dim=-1, keepdim=True)          # [1,R',1]
                out["ray_max_shading_opacity"] = omax
                oi = oind[0, :, 0]
                rows = torch.arange(pidx.shape[0], device=pidx.device)
                loc_max = ex["sample_loc_w"][rows, oi]                                                # [R',3]
                out["ray_max_sample_loc_w"] = loc_max[None]
                wsel = (wgt * conf_coefficient.detach())[rows, oi][..., None]                         # [R',K,1]
                idx_max = idx[rows, oi]                                                               # [R',K] (clamped, :707)
                xyz_max = npnts.xyz.detach()[idx_max]
                out["ray_max_far_dist"] = torch.min(torch.norm(xyz_max - loc_max[:, None, :], dim=-1), dim=-1, keepdim=True)[0][None]
                out["shading_avg_color"] = torch.sum(npnts.points_color.detach()[0][idx_max] * wsel, dim=-2)[None]
                out["shading_avg_dir"] = torch.sum(npnts.points_dir.detach()[0][idx_max] * wsel, dim=-2)[None]
                out["shading_avg_conf"] = torch.sum(npnts.points_conf.detach()[0][idx_max] * wsel, dim=-2)[None]
                out["shading_avg_embedding"] = torch.sum(npnts.points_embeding.detach()[0][idx_max] * wsel, dim=-2)[None]
        elif getattr(opt, "prob", 0) == 1:
            dev = ray_color.device                                                                    # :352-361
            out.update({"ray_max_shading_opacity": torch.zeros([0, 0, 1, 1], device=dev), "ray_max_sample_loc_w": torch.zeros([0, 0, 3], device=dev),
                        "ray_max_far_dist": torch.zeros([0, 0, 1], device=dev), "shading_avg_color": torch.zeros([0, 0, 3], device=dev),
                        "shading_avg_dir": torch.zeros([0, 0, 3], device=dev), "shading_avg_conf": torch.zeros([0, 0, 1], device=dev),
                        "shading_avg_embedding": torch.zeros([0, 0, 32], device=dev)})
        return out
