"""Point growing: one frame's probe on the device (runner.probe_frame: render + pnb_probe_maps + pnb_probe_select, one host sync)
against the reference's chunk loop restated through the drop-in forward() (runner.probe_frame_chunked) at the shipped chunk sizes
(random_sample_size 48 -> 2304 rays, 60 -> 3600).  Times are CUDA-event spans of whole frames after one warm-up frame per path; the
two new kernels are also timed alone (events around 20 back-to-back launches on the frame's own buffers) to give their share of
the probe_frame time.  Prints one JSON line per (config, thresholds) run.

  python tools/probe_bench.py [--configs lego_render scannet_8gpu] [--reps 5] [--chunked-reps 2]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pointnerf_b200 import harness, lib as L, runner, scene   # noqa: E402

# (config, opacity threshold, far threshold): prob_thresh 0.7 and far_thresh -1 (NeRF-Synthetic) / 0.005 (some ScanNet scenes) are
# the shipped values.  On the synthetic lego shell the pixels next to a miss are grazing rays whose arg-max opacity stays below 0.7,
# so that run proposes no point; the run with threshold 0 selects every hit pixel next to a GT hole.
RUNS = {"lego_render": [(0.7, -1.0), (0.0, -1.0)], "scannet_8gpu": [(0.7, 0.005)]}


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return "nvidia-smi unavailable (%s)" % e


def span(fn, reps):
    """Mean CUDA-event time (ms) of `reps` calls of fn (each may synchronise the host inside)."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def frame(cfg_name, opacity_thresh, far_thresh, dev, reps, chunked_reps):
    cfg = scene.CONFIGS[cfg_name]
    net, _, _ = harness.build_model(cfg, dev, alpha_bias=3.0)
    data = {k: (v.to(dev) if isinstance(v, torch.Tensor) else v) for k, v in scene.make_rays(cfg).items()}
    del data["pixel_idx"]                                            # full frame, row-major
    H, W = cfg.H, cfg.W
    col = runner.render_image(net, data, H, W)["coarse_raycolor"].reshape(-1, 3)
    miss = torch.all(col == 1.0, dim=-1)
    idx = torch.arange(H * W, device=dev)
    gt = col.clone()
    gt[miss & (((idx // W) + (idx % W)) % 2 == 0)] = 0.25           # GT holes: half of the miss pixels are not background
    st = dict(opacity_thresh=opacity_thresh, far_thresh=far_thresh)
    run = lambda: runner.probe_frame(net, data, H, W, gt, st["opacity_thresh"], st["far_thresh"], 0.4)
    res = run()                                                      # warm-up (grid, hoisted table, workspace sizes)
    n = int(res["add_xyz"].shape[0])
    out = dict(config=cfg_name, H=H, W=W, N=cfg.N, SR=cfg.SR, K=cfg.K, candidates=n, **st,
               hit_pixels=int((res["prob_maps"]["ray_mask"] > 0).sum()))
    out["probe_frame_ms"] = span(run, reps)
    # the two new kernels alone, on this frame's buffers
    lib = L.load()
    stream = torch.cuda.current_stream(dev).cuda_stream
    with torch.no_grad():
        p = net.probe_full(data["campos"], data["raydir"], data["camrotc2w"], float(data["near"]), float(data["far"]), data["bg_color"])
    net.check_errors()
    q, pts = net.last, net.neural_points.points_desc()
    R = H * W
    bufs = [torch.empty((R, c), device=dev) for c in (1, 3, 1, 3, 3, 1, 32)]
    opacity = p["coarse_point_opacity"][0]
    maps_call = lambda: L.check(lib.pnb_probe_maps(L.C.byref(q.desc), L.C.byref(pts), opacity.data_ptr(), *[b.data_ptr() for b in bufs],
                                                   None, stream), "pnb_probe_maps")
    out["k_probe_maps_ms"] = span(maps_call, 20)
    m = res["prob_maps"]
    ws = torch.empty(lib.pnb_probe_select_bytes(H, W), dtype=torch.uint8, device=dev)
    cnt = torch.zeros(1, dtype=torch.int32, device=dev)
    outs = [torch.empty((max(n, 1), c), device=dev) for c in (3, 32, 3, 3, 1)]
    src = [m["ray_mask"], None, gt, m["coarse_raycolor"], m["ray_max_far_dist"], m["ray_max_shading_opacity"], m["ray_max_sample_loc_w"],
           m["shading_avg_embedding"], m["shading_avg_color"], m["shading_avg_dir"], m["shading_avg_conf"]]
    bg = (L.C.c_float * 3)(1.0, 1.0, 1.0)

    def sel(cap):
        L.check(lib.pnb_probe_select(H, W, *[t.data_ptr() if t is not None else None for t in src], bg, st["opacity_thresh"],
                                     st["far_thresh"], ws.data_ptr(), ws.numel(), cap,
                                     *[o.data_ptr() if cap else None for o in outs], cnt.data_ptr(), stream), "pnb_probe_select")
    out["probe_select_count_ms"] = span(lambda: sel(0), 20)
    out["probe_select_write_ms"] = span(lambda: sel(n), 20)
    k = out["k_probe_maps_ms"] + out["probe_select_count_ms"] + out["probe_select_write_ms"]
    out["new_kernels_ms"] = k
    out["new_kernels_share_of_probe_frame"] = k / out["probe_frame_ms"]
    for chunk in (2304, 3600):
        run_c = lambda: runner.probe_frame_chunked(net, data, H, W, gt, st["opacity_thresh"], st["far_thresh"], 0.4, chunk_size=chunk)
        ref = run_c()                                                # warm-up, and the parity check of this frame
        same = ref["add_xyz"].shape == res["add_xyz"].shape and torch.equal(ref["add_xyz"], res["add_xyz"])
        ms = span(run_c, chunked_reps)
        out["chunked_%d" % chunk] = dict(ms=ms, calls=(R + chunk - 1) // chunk, add_xyz_equal=bool(same),
                                         speedup=ms / out["probe_frame_ms"])
    net.check_errors()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="+", default=["lego_render", "scannet_8gpu"])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--chunked-reps", type=int, default=2)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("probe_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    print(json.dumps(dict(card=card(), torch=torch.__version__)), flush=True)
    for c in a.configs:
        for ot, ft in RUNS[c]:
            print(json.dumps(frame(c, ot, ft, dev, a.reps, a.chunked_reps)), flush=True)
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
