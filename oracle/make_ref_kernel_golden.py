"""TEST INFRASTRUCTURE ONLY -- records what the reference's own CUDA query kernel returns, as the fixtures
tests/golden/ref_kernel_<case>.npz that tests/test_gpu_ref_kernel.py compares libpnb200 against.

It runs `woord_query_grid_point_index` of the reference's un-modified `query_worldcoords_cuda` extension (compiled for sm_100a
into oracle/_ref/ by oracle/build_ref.py) on a GPU, with the 18 arguments of the reference's point_query.py:85-93, for every
case in CASES.  Each fixture holds
  ray_mask   the reference's ray mask over all rays of the case (np.packbits, little bit order);
  rays       int32 [n]: a fixed, seeded sample of the rays the reference kept, in increasing order;
  pidx       int32 [n, SR, K]: their neighbour index sets, sorted along K (only the sets are comparable: in-voxel order
             depends on the kernel's atomics);
  locw       float32 [n, SR, 3]: their world sample positions.
The sample is the shortest prefix of a seeded permutation of the kept rays that holds `target` filled samples, so that each
fixture stays a few tens of kB.

    python -m oracle.make_ref_kernel_golden [OUT_DIR]        # needs a GPU and oracle/_ref/ (default OUT_DIR: tests/golden)
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from pointnerf_b200 import harness, scene  # noqa: E402


def block(x0, y0, w, h):
    px, py = np.meshgrid(np.arange(x0, x0 + w), np.arange(y0, y0 + h))
    return np.stack((px, py), -1).reshape(-1, 2).astype(np.float32)


# case -> (config, pixels (None = full frame), option overrides, filled samples to store)
CASES = {
    "tiny_full_frame": ("tiny", None, {}, 1300),
    "chair": ("chair_plumbing", scene.centre_patch(scene.CONFIGS["chair_plumbing"], 96), {}, 1300),
    "lego_chunk_sr24": ("lego_render", scene.centre_patch(scene.CONFIGS["lego_render"], 48), dict(SR=24), 1300),
    "lego_chunk_sr80": ("lego_render", scene.centre_patch(scene.CONFIGS["lego_render"], 48), dict(SR=80), 1300),
    "lego_silhouette": ("lego_render", block(400 + 240, 388, 96, 24), {}, 1300),
    "truck_chunk": ("truck_8gpu", scene.centre_patch(scene.CONFIGS["truck_8gpu"], 32), {}, 1300),
    "truck_strip": ("truck_8gpu", block(860, 0, 100, 16), {}, 700),
    "scannet_chunk": ("scannet_8gpu", scene.centre_patch(scene.CONFIGS["scannet_8gpu"], 24), {}, 1300),
}


def path(golden_dir, case):
    return os.path.join(golden_dir, "ref_kernel_%s.npz" % case)


def run_ours(case, dev):
    """libpnb200's query through the drop-in lighting_fast_querier.query_points on the rays of `case`."""
    cfg_name, pixels, over, _ = CASES[case]
    cfg = scene.CONFIGS[cfg_name]
    net, pts, opt = harness.build_model(cfg, dev, **over)
    rays = scene.make_rays(cfg, pixels)
    r = {k: (v.to(dev) if isinstance(v, torch.Tensor) else v) for k, v in rays.items()}
    querier = net.neural_points.querier
    xyz = net.neural_points.xyz.detach().contiguous()
    npts = torch.tensor([xyz.shape[0]], dtype=torch.int32, device=dev)
    pix = r["pixel_idx"].to(torch.int32)
    raydir = r["raydir"].contiguous()
    ours = querier.query_points(pix, None, xyz[None], npts, r["h"], r["w"], r["intrinsic"], np.float32(cfg.near),
                                np.float32(cfg.far), raydir, r["campos"], r["camrotc2w"])
    return dict(cfg=cfg, opt=opt, net=net, querier=querier, xyz=xyz, npts=npts, pix=pix, raydir=raydir, r=r, ours=ours)


def run_reference(ext, s):
    """The reference kernel on the same points, rays and hyper-parameters."""
    cfg, opt, querier, xyz, raydir, r = s["cfg"], s["opt"], s["querier"], s["xyz"], s["raydir"], s["r"]
    dev = xyz.device
    R = raydir.shape[1]
    ranges_tensor, ranges_np, vsize_np, scaled_vdim_np = querier._hyper
    t = querier._t_for(cfg.near, cfg.far, R, dev)
    # ray generation of diff_ray_marching.py:386-388 as torch runs it on the device: one mul kernel, one add kernel
    raypos = (r["campos"][:, None, None, :] + raydir[:, :, None, :] * t[None, None, :, None]).contiguous()
    max_o = int(opt.max_o) if opt.max_o is not None else int(xyz.shape[0])
    out = ext.woord_query_grid_point_index(
        s["pix"], raypos, xyz[None], s["npts"], querier.kernel_size_tensor, querier.query_size_tensor, int(opt.SR), int(opt.K), R,
        raypos.shape[2], torch.as_tensor(scaled_vdim_np, device=dev), max_o, int(opt.P), float(querier.radius_limit_np),
        ranges_tensor.to(dev), querier.scaled_vsize_tensor, 1024, 2)
    torch.cuda.synchronize()
    return out[0][0].cpu().numpy(), out[1][0].cpu().numpy(), out[2][0].reshape(-1).cpu().numpy() > 0


def sample(pidx, locw, mask, target, seed=0):
    rays = np.nonzero(mask)[0]
    filled = ((pidx >= 0).any(-1) | (locw != 0).any(-1)).sum(-1)                  # per kept ray
    perm = np.random.RandomState(seed).permutation(rays.shape[0])
    n = min(int(np.searchsorted(np.cumsum(filled[perm]), target)) + 1, perm.shape[0])
    rows = np.sort(perm[:n])
    return dict(ray_mask=np.packbits(mask.astype(np.uint8), bitorder="little"), rays=rays[rows].astype(np.int32),
                pidx=np.sort(pidx[rows], -1).astype(np.int32), locw=locw[rows].astype(np.float32))


def main(out_dir):
    from oracle import build_ref
    ext = build_ref.load_prebuilt()
    assert ext is not None, "oracle/_ref/query_worldcoords_cuda.so is missing: python -m oracle.build_ref"
    os.makedirs(out_dir, exist_ok=True)
    dev = torch.device("cuda:0")
    for case in CASES:
        s = run_ours(case, dev)
        gc = s["querier"].last_grid_counters
        assert gc["overflow_o"] == 0 and gc["overflow_p"] == 0, "fixture cases must not overflow max_o / P"
        pidx, locw, mask = run_reference(ext, s)
        fx = sample(pidx, locw, mask, CASES[case][3])
        np.savez_compressed(path(out_dir, case), **fx)
        print("%-16s rays %d kept %d stored %d (%d kB)" % (case, mask.shape[0], int(mask.sum()), fx["rays"].shape[0],
                                                          os.path.getsize(path(out_dir, case)) // 1024))
        del s
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden"))
