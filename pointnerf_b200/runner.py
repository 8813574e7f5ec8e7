"""Whole-image entry points either side of the seam (SURVEY.md 8(f) rank 2).

The reference renders an image as a host loop over `random_sample_size**2`-ray chunks
(`/root/reference/run/render_vid.py:45-71`, `/root/reference/run/train_ft.py:283-320`): per chunk `model.set_input`,
`model.test()`, `.cpu().numpy()` of every `*color` visual into a `[H*W,3]` host array, then `fill_invalid`
(`neural_points_volumetric_model.py:87-123`) — 278 launches + host syncs for an 800x800 frame at the shipped 2304-ray
chunk.  `render_image` is the same computation as ONE call (rays of the whole frame resident on the device, fill_invalid
applied in-kernel, no host sync until the caller reads the result); `render_image_chunked` reproduces the reference loop
through the drop-in `forward()` and is what the parity test compares it with (a ray's colour is bit-identical whichever
rays share its call).
"""
import numpy as np
import torch


def _near_far(near, far):
    n = float(torch.min(near)) if isinstance(near, torch.Tensor) else float(near)
    f = float(torch.max(far)) if isinstance(far, torch.Tensor) else float(far)
    return n, f


def render_image(net, data, height, width, check=True):
    """data: the dict a reference dataset item carries (`campos [1,3]`, `raydir [1,H*W,3]`, `camrotc2w [1,3,3]`, `near`, `far`,
    `bg_color`).  Returns device tensors: `coarse_raycolor [H,W,3]`, `coarse_point_opacity [H,W,SR]`,
    `coarse_is_background [H,W,1]`, `ray_mask [H,W]` (all rays, background filled as fill_invalid does).
    check=True (default): the device status of the frame is read before returning (one stream synchronisation; the caller is
    about to read the image anyway) and a frame whose shading workspace was too small is rendered again with the exact size;
    check=False: fully asynchronous, the status surfaces at a later call or through `net.check_errors()`."""
    near, far = _near_far(data["near"], data["far"])
    raydir = data["raydir"]
    if raydir.shape[1] != height * width:
        raise ValueError("render_image: %d rays for a %dx%d image" % (raydir.shape[1], height, width))
    bg = data.get("bg_color", None)
    from .lib import PnbOverflow
    with torch.no_grad():
        for attempt in range(2):
            out = net.render_full(data["campos"], raydir, data["camrotc2w"], near, far, bg if bg is not None else torch.zeros(3))
            if not check:
                break
            try:
                net.check_errors()
                break
            except PnbOverflow:
                if attempt == 1:
                    raise
    sr = out["coarse_point_opacity"].shape[-1]
    return dict(coarse_raycolor=out["coarse_raycolor"][0].view(height, width, 3),
                coarse_point_opacity=out["coarse_point_opacity"][0].view(height, width, sr),
                coarse_is_background=out["coarse_is_background"][0].view(height, width, 1),
                ray_mask=out["ray_mask"][0].view(height, width))


def render_image_chunked(net, data, height, width, chunk_size):
    """The reference chunk loop (render_vid.py:45-71) through the drop-in `forward()` + fill_invalid on the host:
    returns `{"coarse_raycolor": np.ndarray [H,W,3]}` exactly as the reference assembles `visuals`."""
    near, far = _near_far(data["near"], data["far"])
    raydir = data["raydir"]
    total = height * width
    bg = data.get("bg_color", None)
    bgv = (bg if bg is not None else torch.zeros(3)).reshape(-1)[:3].cpu().numpy().astype(np.float32)
    img = np.zeros((total, 3), dtype=np.float32)
    with torch.no_grad():
        for start in range(0, total, chunk_size):
            end = min(start + chunk_size, total)
            out = net(data["campos"], raydir[:, start:end, :], bg_color=bg, camrotc2w=data["camrotc2w"],
                      near=near, far=far)
            mask = out["ray_mask"][0].bool().cpu().numpy()
            chunk = np.tile(bgv[None, :], (end - start, 1))                      # fill_invalid: background where no neighbour
            chunk[mask] = out["coarse_raycolor"][0].cpu().numpy()
            img[start:end] = chunk
    return dict(coarse_raycolor=img.reshape(height, width, 3))


# ------------------------------------------------------------------------------------------------ point growing (probe_hole)
# The reference grows points between optimisation loops with `probe_hole` (`/root/reference/run/train_ft.py:417-530`): per frame a
# host loop of `random_sample_size**2`-ray chunks through `model.test()` with opt.prob = 1, the nine per-pixel maps below scattered
# into [H,W,C] tensors, then a hole test and boolean-mask compaction of the new points.  `probe_frame` is the same computation as one
# render (`probe_full`: render_full + the pnb_probe_maps kernel) and one selection (`pnb_probe_select`) per frame, with ONE host
# synchronisation (the number of new points); `probe_frame_chunked` restates the reference loop through the drop-in forward() and is
# its parity partner.

PROBE_KEYS = ("coarse_raycolor", "ray_mask", "ray_max_sample_loc_w", "ray_max_far_dist", "ray_max_shading_opacity",
              "shading_avg_color", "shading_avg_dir", "shading_avg_conf", "shading_avg_embedding")
_UNMASK_KEYS = PROBE_KEYS[2:]
_ADD_KEYS = ("add_xyz", "add_embedding", "add_color", "add_dir", "add_conf")
_ADD_SRC = ("ray_max_sample_loc_w", "shading_avg_embedding", "shading_avg_color", "shading_avg_dir", "shading_avg_conf")


def _pixel_ids(data, n_rays, height, width, device):
    """Linear pixel id (y * W + x) of every ray: data["pixel_idx"] [1,R,2] as (x, y) when given, row-major order otherwise."""
    pix = data.get("pixel_idx", None)
    if pix is None:
        if n_rays != height * width:
            raise ValueError("probe: %d rays for a %dx%d frame and no pixel_idx" % (n_rays, height, width))
        return None
    pix = pix.reshape(-1, 2).to(device).long()
    if pix.shape[0] != n_rays:
        raise ValueError("probe: pixel_idx has %d entries for %d rays" % (pix.shape[0], n_rays))
    return pix[:, 1] * width + pix[:, 0]


def _bg_of(data, device):
    bg = data.get("bg_color", None)
    return (bg if bg is not None else torch.zeros(3)).reshape(-1)[:3].to(device).float()


def bloat_inds(inds, shift, height, width):
    """train_ft.py:532-540: every (y, x) of `inds` [N,2] expanded to its (2*shift+1)^2 window, clamped to the image."""
    inds = inds[:, None, :]
    r = torch.arange(-shift, shift + 1, dtype=torch.long, device=inds.device)
    sx, sy = torch.meshgrid(r, r, indexing="ij")
    inds = (inds + torch.stack([sx, sy], dim=-1).reshape(1, -1, 2)).reshape(-1, 2)
    inds[..., 0] = torch.clamp(inds[..., 0], min=0, max=height - 1)
    inds[..., 1] = torch.clamp(inds[..., 1], min=0, max=width - 1)
    return inds


def select_holes(prob_maps, gt_image, edge_mask, bg, opacity_thresh, far_thresh):
    """The hole test of train_ft.py:493-505 as the reference writes it (torch ops on any device): prob_maps [H,W,C] maps, gt_image
    [H,W,3] (0 outside edge_mask), edge_mask [H,W] bool (the pixels given), bg [3].  Returns the [H,W] bool mask of new points."""
    height, width = edge_mask.shape
    bg = bg.reshape(1, 1, 3).to(gt_image.device, gt_image.dtype)
    ray_mask = prob_maps["ray_mask"]
    miss_ray_mask = (ray_mask < 1) * (torch.norm(gt_image - bg, dim=-1, keepdim=True) > 0.002)
    miss_ray_inds = (edge_mask.reshape(height, width, 1) * miss_ray_mask).squeeze(-1).nonzero()
    neighbor_inds = bloat_inds(miss_ray_inds, 1, height, width)
    nmm = torch.zeros_like(gt_image[..., 0])
    nmm[neighbor_inds[..., 0], neighbor_inds[..., 1]] = 1
    if far_thresh > 0:
        far_ray_mask = (ray_mask > 0) * (prob_maps["ray_max_far_dist"] > far_thresh) * \
            (torch.norm(gt_image - prob_maps["coarse_raycolor"], dim=-1, keepdim=True) < 0.1)
        nmm += far_ray_mask.squeeze(-1)
    return (ray_mask.squeeze(-1) > 0) * nmm * (prob_maps["ray_max_shading_opacity"].squeeze(-1) > opacity_thresh) > 0


def accumulate_new_points(acc, new, prob_mul):
    """One frame of probe_hole's accumulation (train_ft.py:508-512): concatenate, and scale ALL of add_conf (earlier frames
    included) by prob_mul.  acc / new: (add_xyz, add_embedding, add_color, add_dir, add_conf)."""
    out = [torch.cat([a, n], dim=0) for a, n in zip(acc, new)]
    out[4] = out[4] * prob_mul
    return tuple(out)


def probe_frame(net, data, height, width, gt_image, opacity_thresh, far_thresh=-1, prob_mul=1.0):
    """Probe one frame for holes and return the new points it proposes (probe_hole's per-frame body, train_ft.py:456-512).

    data: the reference dataset item (`campos`, `raydir [1,R,3]`, `camrotc2w`, `near`, `far`, `bg_color`, optional
    `pixel_idx [1,R,2]` as (x, y) for a subset of the pixels; without it the rays are the full frame in row-major order).
    gt_image: the ground-truth colour of every ray, R*3 values in ray order.  A pixel becomes a new point when it has a neighbour
    (ray_mask > 0), its arg-max opacity exceeds opacity_thresh (strictly), and a given pixel in its 3x3 window has no neighbour
    while its GT differs from the background (|gt - bg| > 0.002), or (far_thresh > 0) its arg-max sample lies farther than
    far_thresh from its neighbours while its colour is close to the GT (< 0.1).

    Returns dict(prob_maps={the nine [H,W,C] maps of probe_hole, zeros at pixels not given}, add_xyz [n,3], add_embedding [n,32],
    add_color [n,3], add_dir [n,3], add_conf [n,1] (shading_avg_conf * prob_mul)); new points in row-major pixel order.
    One host synchronisation: reading n.  The device status of the render is checked then as well; a frame whose shading workspace
    was too small is probed again with the enlarged workspace (as render_image does).
    The GT colour is paired with its pixel through pixel_idx; the reference pairs the given GT values with the given pixels in
    row-major order, which is the same whenever pixel_idx is row-major sorted (every full frame and strided subset)."""
    from . import lib as _lib
    near, far = _near_far(data["near"], data["far"])
    raydir = data["raydir"]
    dev = raydir.device
    R = raydir.shape[1]
    HW = height * width
    lin = _pixel_ids(data, R, height, width, dev)
    bg = _bg_of(data, dev)
    gt = torch.as_tensor(gt_image).to(dev).float().reshape(-1, 3).contiguous()
    if gt.shape[0] != R:
        raise ValueError("probe_frame: gt_image has %d colours for %d rays" % (gt.shape[0], R))
    lib = _lib.load()
    stream = torch.cuda.current_stream(dev).cuda_stream
    ws = torch.empty(lib.pnb_probe_select_bytes(height, width), dtype=torch.uint8, device=dev)
    count = torch.zeros(1, dtype=torch.int32, device=dev)
    bg_c = (_lib.C.c_float * 3)(*bg.cpu().tolist())
    with torch.no_grad():
        for attempt in range(2):
            out = net.probe_full(data["campos"], raydir, data["camrotc2w"], near, far, bg)
            if lin is None:
                maps = {k: out[k][0].reshape(height, width, -1) for k in PROBE_KEYS}
                present, gt_full = None, gt
            else:
                maps = {}
                for k in PROBE_KEYS:
                    v = out[k][0].reshape(R, -1)
                    maps[k] = torch.zeros((HW, v.shape[1]), dtype=v.dtype, device=dev).index_copy_(0, lin, v).view(height, width, -1)
                present = torch.zeros(HW, dtype=torch.uint8, device=dev).index_fill_(0, lin, 1)
                gt_full = torch.zeros((HW, 3), dtype=torch.float32, device=dev).index_copy_(0, lin, gt)
            src = [maps[k] for k in ("ray_mask",)] + [gt_full] + [maps[k] for k in ("coarse_raycolor", "ray_max_far_dist",
                                                                                    "ray_max_shading_opacity") + _ADD_SRC]
            ptrs = [t.data_ptr() for t in src]
            args = ptrs[:1] + [present.data_ptr() if present is not None else None] + ptrs[1:]

            def select(cap, bufs):
                _lib.check(lib.pnb_probe_select(height, width, *args, bg_c, float(opacity_thresh), float(far_thresh), ws.data_ptr(),
                                                ws.numel(), cap, *[b.data_ptr() if b is not None else None for b in bufs],
                                                count.data_ptr(), stream), "pnb_probe_select")

            select(0, [None] * 5)                       # count only
            n = int(count.item())                       # the one host synchronisation of the frame
            try:
                net._poll_status(block=True)            # the render's status is already on the host (its event has completed)
                break
            except _lib.PnbOverflow:
                if attempt == 1:
                    raise
        flat = torch.empty((max(n, 1) * 42,), dtype=torch.float32, device=dev)
        add_emb = flat[:n * 32].view(n, 32)
        add_xyz, add_color, add_dir = (flat[n * o:n * (o + 3)].view(n, 3) for o in (32, 35, 38))
        add_conf = flat[n * 41:n * 42].view(n, 1)
        if n > 0:
            # same maps, same scan: writes exactly the n rows counted above
            select(n, [add_xyz, add_emb, add_color, add_dir, add_conf])
        if prob_mul != 1.0:
            add_conf = add_conf * prob_mul
    return dict(prob_maps=maps, add_xyz=add_xyz, add_embedding=add_emb, add_color=add_color, add_dir=add_dir, add_conf=add_conf)


def _frame_hw(frame):
    h = frame.get("height", frame.get("h"))
    w = frame.get("width", frame.get("w"))
    if h is None or w is None:
        raise ValueError("probe_holes: every frame needs its size as height / width (or the dataset item's h / w)")
    return int(torch.as_tensor(h).reshape(-1)[0]), int(torch.as_tensor(w).reshape(-1)[0])


def probe_holes(net, frames, opacity_thresh, far_thresh, prob_mul):
    """probe_hole (train_ft.py:417-530) over `frames`, single rank: returns (add_xyz [n,3], add_embedding [n,32], add_color [n,3],
    add_dir [n,3], add_conf [n,1]) for `net.neural_points.grow_points(*...)`.  Each frame is a dataset item as `probe_frame` takes
    it plus `gt_image` (the GT colour of each ray) and its size (`height` / `width`, or the item's `h` / `w`).

    The accumulation keeps the reference's compounding: after each frame ALL of add_conf is multiplied by prob_mul
    (`add_conf = cat([add_conf, new]) * prob_mul`), so the points of frame i of n (0-based) end up scaled by prob_mul**(n - i),
    and the first frame's the most.  With the frames sharded over ranks (parallel.shard_frames, merged by allgather_new_points)
    each rank compounds over its own frames only, so the exponents differ from a single-rank run over all frames."""
    dev = net.neural_points.xyz.device
    acc = (torch.zeros((0, 3), device=dev), torch.zeros((0, 32), device=dev), torch.zeros((0, 3), device=dev),
           torch.zeros((0, 3), device=dev), torch.zeros((0, 1), device=dev))
    for fr in frames:
        h, w = _frame_hw(fr)
        r = probe_frame(net, fr, h, w, fr["gt_image"], opacity_thresh, far_thresh)
        acc = accumulate_new_points(acc, [r[k] for k in _ADD_KEYS], prob_mul)
    return acc


def probe_frame_chunked(net, data, height, width, gt_image, opacity_thresh, far_thresh=-1, prob_mul=1.0, chunk_size=2304):
    """The reference's per-frame probe (train_ft.py:456-512) restated through the drop-in forward() with opt.prob = 1: chunks of
    `chunk_size` rays, fill_invalid / unmask on the host, the nine maps scattered per chunk, `select_holes`, boolean-mask
    compaction.  Same arguments and returns as probe_frame (the parity partner of probe_frame, as render_image_chunked is of
    render_image).  GT values are placed as the reference places them: into the given pixels in row-major order."""
    near, far = _near_far(data["near"], data["far"])
    raydir = data["raydir"]
    dev = raydir.device
    R = raydir.shape[1]
    lin = _pixel_ids(data, R, height, width, dev)
    if lin is None:
        lin = torch.arange(R, device=dev)
    bg = _bg_of(data, dev)
    gt = torch.as_tensor(gt_image).to(dev).float().reshape(-1, 3)
    opt = net.opt
    prob0 = getattr(opt, "prob", 0)
    opt.prob = 1
    maps = {}
    try:
        with torch.no_grad():
            for start in range(0, R, chunk_size):
                end = min(start + chunk_size, R)
                n = end - start
                out = net(data["campos"], raydir[:, start:end, :], bg_color=bg, camrotc2w=data["camrotc2w"], near=near, far=far)
                mask = out["ray_mask"][0]
                inds = torch.nonzero(mask)[:, 0]
                full = {"coarse_raycolor": bg[None, :].repeat(n, 1), "ray_mask": mask[:, None]}         # fill_invalid
                full["coarse_raycolor"][inds] = out["coarse_raycolor"][0]
                for k in _UNMASK_KEYS:                                                                 # unmask
                    v = out[k][0].reshape(inds.shape[0], -1) if inds.shape[0] else out[k].reshape(0, out[k].shape[-1])
                    full[k] = torch.zeros((n, v.shape[1]), dtype=v.dtype, device=dev)
                    full[k][inds] = v
                for k in PROBE_KEYS:
                    if k not in maps:
                        maps[k] = torch.zeros((height * width, full[k].shape[1]), dtype=full[k].dtype, device=dev)
                    maps[k][lin[start:end]] = full[k]
    finally:
        opt.prob = prob0
    maps = {k: v.view(height, width, -1) for k, v in maps.items()}
    edge_mask = torch.zeros(height * width, dtype=torch.bool, device=dev)
    edge_mask[lin] = True
    gt_full = torch.zeros((height * width, 3), dtype=torch.float32, device=dev)
    gt_full[edge_mask] = gt
    sel = select_holes(maps, gt_full.view(height, width, 3), edge_mask.view(height, width), bg, opacity_thresh, far_thresh)
    res = {k: maps[s][sel] for k, s in zip(_ADD_KEYS, _ADD_SRC)}
    res["add_conf"] = res["add_conf"] * prob_mul
    res["prob_maps"] = maps
    return res
