"""Per-kernel device time of the bench.py main workload (lego frame, 800x800, K=8, 400k points, SR=24), from torch.profiler.

Renders `--frames` frames after a warm-up and prints, per kernel name, the launches per frame and the device ms per frame, with the
card's name and power limit.  Run it alone: the profiler slows the host, so its frame times are not bench numbers.

usage: python tools/kernel_times.py [--frames 10] [--sr 24]
"""
import argparse
import os
import re
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pointnerf_b200 import harness, scene  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=10)
    ap.add_argument("--sr", type=int, default=24)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()[0]
    cfg = scene.CONFIGS["lego_render"]
    cfg.SR = args.sr
    net, _, _ = harness.build_model(cfg, dev, seed=0, alpha_bias=3.0)
    raydir = scene.make_rays(cfg)["raydir"].to(dev)
    cam = (list(cfg.campos), torch.eye(3), cfg.near, cfg.far, [1., 1., 1.])

    def frame():
        with torch.no_grad():
            net.render_full(cam[0], raydir, cam[1], cam[2], cam[3], cam[4])

    for _ in range(3):
        frame()
    torch.cuda.synchronize(dev)
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(args.frames):
            frame()
        torch.cuda.synchronize(dev)
    net.check_errors()
    agg = {}
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        name = re.sub(r"^(void )?(pnb::)?", "", e.name)
        name = re.sub(r"[(<].*$", "", name)[:48]
        a = agg.setdefault(name, [0, 0.0])
        a[0] += 1
        a[1] += e.time_range.elapsed_us() / 1e3
    total = sum(v[1] for v in agg.values()) / args.frames
    print("# card %s | lego_render 800x800 SR=%d, %d frames under torch.profiler" % (card, args.sr, args.frames))
    print("%-48s %8s %10s %7s" % ("kernel", "n/frame", "ms/frame", "share"))
    for name, (n, ms) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
        print("%-48s %8.1f %10.4f %6.1f%%" % (name, n / args.frames, ms / args.frames, 100 * ms / args.frames / total))
    print("%-48s %8s %10.4f" % ("total", "", total))


if __name__ == "__main__":
    main()
