#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config, measured on B200.

Metric: Mrays/s (whole job) for full-image renders of the synthetic "lego_render" scene (BASELINE configs[1]:
800x800 = 640,000 rays per image, K=8, N=400,000 neural points, SR=24 shading samples per ray, D=400 march steps, fp32 I/O).
A "step" = one full image per GPU through the hot path (voxel query -> row packing -> fused pair MLPs -> colour MLP ->
composite), ONE `render_full` call.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--sr 24] [--only main] [--dump-outputs DIR]

N>1 is launched by torchrun (one rank per GPU, NCCL).  The JSON line of every N carries
  value / ms_per_step  WEAK scaling: N distinct camera poses (rolls about the view axis), rank g renders frame g, one all-gather of
                       the [R,3] colours per step inside the timed region, issued on a side stream so that it overlaps the next frame;
  strong               ONE 800x800 frame, rays interleave-sharded (ray i -> rank i % N), tile all-gather inside the timed region;
  truck                BASELINE configs[3]: N=2M points, 960x540, kernel_size 5, one frame interleave-sharded over the N ranks;
  train                BASELINE configs[2] (N=1..8) per-scene optimisation step: 3600 rays per step split over the ranks,
                       forward + backward + gradient all-reduce + 2x Adam (parallel.TrainStep);
  scannet              BASELINE configs[4]: N=5M points (P=30), the same step with the sparse touched-rows gradient exchange, plus one
                       prune + probe + grow cycle (variable-length all-gather of the new points);
  cold, sr80           (N=1) first frame of a new point cloud (voxel grid + per-point table built inside the timed region); SR=80.

`--dump-outputs DIR` writes what the last of the K timed steps of the main line returned (rank 0's frame) as DIR/<name>.npy, float32:
the render_full outputs coarse_raycolor [1,R,3], coarse_is_background [1,R,1] and ray_mask [1,R] in full, and coarse_point_opacity
[1,R,SR] for a fixed, seeded sample of DUMP_OPACITY_RAYS rays (their indices in coarse_point_opacity_rays.npy).  The scene, weights and
rays are seeded: the same arguments give the same inputs on every run, so two builds can be compared output for output.

`--impl reference` times the reference's own CPU path (the oracle port: oracle/query_oracle.c + oracle/shade_oracle.py, i.e. the
reference's algorithm on the host cores) on a bounded, stratified sample of the same frame.  The oracle is used here ONLY as the
measured CPU baseline, never inside the GPU arm.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from pointnerf_b200 import harness, scene  # noqa: E402

METRIC = "Mrays/s (800x800 render, K=8, 400k pts, SR=24), whole job"
FLOPS_PER_PAIR = 542720.0    # SURVEY.md 8(d): 2*(284*256 + 256*256 + 263*256 + 256*256 + 256)
FLOPS_PER_SAMPLE = 137984.0  # 2*(280*128 + 128*128 + 128*128 + 128*3)
# kernels of libpnb200.so launched per render_full (memsets / torch fills are not counted): march, 2 scans x 3, expand, knn, valid_list,
# count_rays (query = 11); k_pack_quads, k_pack_scan, k_pack_place, pair kernel, colour kernel (tcgen05 shading = 5); composite (1)
LAUNCHES_PER_STEP_TC = 11 + 5 + 1
LAUNCHES_PER_STEP_FP32 = 11 + 1 + 1
MMA_FLOPS = 2.0 * 128 * 256 * 16                      # one tcgen05.mma M128 N256 K16
MMAS_PER_TILE = {True: 159, False: 201}               # frozen (k_shade_tc8) / general (k_shade_tc7) pair kernel, per 128-row tile
DUMP_OPACITY_RAYS = 65536                             # the full [R,SR] opacity of an 800x800 frame alone is 61 MB


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d["hbm_gbs"], bf16_tflops=d["bf16_tflops"], bf16_tflops_sustained=d.get("bf16_tflops_sustained"),
                    source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback")


class ClockSampler:
    """nvidia-smi polled every 25 ms from before the warm-up (its start-up latency would otherwise eat a 0.2-s timed region);
    stop(t0, t1) keeps the samples whose timestamps fall inside the timed region [t0, t1] (host wall clock)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                       "-lms", "25"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self, t0=None, t1=None):
        import datetime
        if self.p is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.05)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)

        def collect(lo, hi):
            sm, mx, reasons, pw = [], [], set(), []
            for r in rows:
                try:
                    ts = datetime.datetime.strptime(r[0].strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    if lo is not None and not (lo <= ts <= hi):
                        continue
                    sm.append(float(r[1])); mx.append(float(r[2])); pw.append(float(r[3]))
                except Exception:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            return sm, mx, reasons, pw

        window = "timed region"
        sm, mx, reasons, pw = collect(t0, t1)
        if len(sm) < 2 and t0 is not None:          # very short region: fall back to everything since the warm-up started (also under load)
            sm, mx, reasons, pw = collect(None, None)
            window = "warm-up + timed region"
        if not sm:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["no samples"])
        return dict(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), power_w_max=float(max(pw)), samples=len(sm),
                    window=window, reasons=sorted(reasons))


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own path on the host cores = oracle port (C query + torch-CPU shading).  A pool of worker
# processes (each with a few intra-op threads: 128-thread eager torch on 1e5-row tensors is slower than 8 threads)
# renders reference-sized chunks of the frame concurrently, so that every host core is used.
_W = {}
CPU_GRID = 16          # the frame's central 768 x 768 pixels = 16 x 16 blocks of 48 x 48 = the reference's 2304-ray chunk (train_ft.py:773)


def _cpu_worker_init(sr, threads):
    import torch as _t
    from oracle import query_oracle
    from pointnerf_b200.ray_marching import PointAggregator
    _t.set_num_threads(threads)
    query_oracle.build()
    cfg = scene.CONFIGS["lego_render"]
    cfg.SR = sr
    opt = harness.make_opt(cfg)
    agg = PointAggregator(opt, seed=0)
    with _t.no_grad():
        agg.alpha_branch[0].bias += 3.0
    _W.update(cfg=cfg, opt=opt, pts=scene.make_points(cfg), mlp=harness.mlp_cpu(agg))


def cpu_block_of(i):
    """Block i of a fixed stratified order over the 16 x 16 block grid (a stride-101 walk visits every block once per 256 and
    spreads any prefix over the frame: hits in the disc of the shell, misses in the corners, the limb in between)."""
    b = (i * 101) % (CPU_GRID * CPU_GRID)
    return b % CPU_GRID, b // CPU_GRID


def _cpu_worker_chunk(i):
    """Render one 2304-ray chunk = 48 x 48 block `cpu_block_of(i)` of the 800 x 800 frame (margin 16 px)."""
    from oracle import pipeline
    cfg, opt, pts, mlp = _W["cfg"], _W["opt"], _W["pts"], _W["mlp"]
    bx, by = cpu_block_of(i)
    x0, y0 = 16 + 48 * bx, 16 + 48 * by
    px, py = np.meshgrid(np.arange(x0, x0 + 48), np.arange(y0, y0 + 48))
    rays = scene.make_rays(cfg, np.stack((px, py), -1).reshape(-1, 2).astype(np.float32))
    t0 = time.perf_counter()
    out = pipeline.render(pts, mlp, rays["raydir"][0], cfg.campos, np.eye(3, dtype=np.float32), cfg.near, cfg.far, opt.vsize,
                          opt.vscale, opt.kernel_size, opt.query_size, opt.ranges, opt.SR, opt.K, opt.P, pts["xyz"].shape[0], D=cfg.D)
    return 2304, time.perf_counter() - t0, int(out["ray_mask"].sum())


class CpuArm:
    def __init__(self, sr):
        import multiprocessing as mp
        self.cores = os.cpu_count() or 1
        self.threads = 8 if self.cores >= 16 else self.cores
        self.workers = max(1, self.cores // self.threads)
        self.pool = mp.get_context("spawn").Pool(self.workers, initializer=_cpu_worker_init, initargs=(sr, self.threads))
        self.hit = 0
        self.rays = 0

    def step(self, k=0):
        """One step = every worker renders one chunk concurrently.  Returns (rays, seconds)."""
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_worker_chunk, [k * self.workers + j for j in range(self.workers)])
        self.hit += sum(h for _, _, h in res)
        self.rays += sum(r for r, _, _ in res)
        return sum(r for r, _, _ in res), time.perf_counter() - t0

    def close(self):
        self.pool.close()
        self.pool.join()

    def describe(self, steps, secs):
        return ("%d steps x %d concurrent 2304-ray chunks = 48x48 blocks of the 800x800 frame in a stratified order over the whole frame "
                "(stride walk over the 16x16 block grid: hits, misses and the limb in frame proportion; %.0f %% of the sampled rays hit); "
                "%d worker processes x %d torch threads; voxel grid rebuilt per chunk as the reference does; %.1f s"
                % (steps, self.workers, 100.0 * self.hit / max(self.rays, 1), self.workers, self.threads, secs))


WORKLOAD = "lego_render: 800x800 image per GPU, K=8, N=400000 points, SR=%d, D=400, P=16, vsize 0.004 x vscale 2"      # both arms


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    arm = CpuArm(args.sr)
    for i in range(args.warmup):
        arm.step(i)
    arm.hit = arm.rays = 0
    rays = 0
    t0 = time.perf_counter()
    for i in range(args.steps):
        r, _ = arm.step(args.warmup + i)
        rays += r
    dt = time.perf_counter() - t0
    arm.close()
    val = rays / dt / 1e6
    line = dict(impl="reference", metric=METRIC, value=val, unit="Mrays/s", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=dt / args.steps * 1e3, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic", config=dict(workload=WORKLOAD % args.sr, rays_per_step_sampled=rays // max(args.steps, 1),
                            note="each step = a bounded stratified sample of the frame (see cpu_baseline.sample); value = rays of the sample / time"),
                cpu_baseline=dict(value=val, unit="Mrays/s", cores=arm.workers * arm.threads, kind="port", sample=arm.describe(args.steps, dt)),
                e2e=dict(value=val, unit="Mrays/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))
    return 0


def cpu_baseline_leg(sr, budget_s=20.0):
    """Bounded sample of the same workload on the host cores (rank 0, N=1 only)."""
    arm = CpuArm(sr)
    arm.step(0)
    arm.hit = arm.rays = 0
    rays, n, t0 = 0, 0, time.perf_counter()
    while True:
        r, _ = arm.step(1 + n)
        rays += r
        n += 1
        if time.perf_counter() - t0 > budget_s or n >= 6:
            break
    dt = time.perf_counter() - t0
    arm.close()
    return dict(value=rays / dt / 1e6, unit="Mrays/s", cores=arm.workers * arm.threads, kind="port", sample=arm.describe(n, dt))


# ---------------------------------------------------------------------------------------------------------------------
def roll(k, n):
    """Camera-to-world rotation of pose k of n: a roll about the view axis (the shell is symmetric under it: equal work per pose)."""
    a = 2.0 * math.pi * k / max(n, 1)
    return torch.tensor([[math.cos(a), -math.sin(a), 0.0], [math.sin(a), math.cos(a), 0.0], [0.0, 0.0, 1.0]], dtype=torch.float32)


class Dist:
    """Thin wrapper: world-1 runs need no process group."""

    def __init__(self, dev):
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.dev = dev
        self.comm = None
        if self.world > 1:
            import torch.distributed as dist
            self.dist = dist
            dist.init_process_group("nccl", device_id=dev)
            self.comm = torch.cuda.Stream(dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize(self.dev)

    def max_over_ranks(self, x):
        if self.world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def gather_async(self, col, out):
        """all_gather of this rank's colours into out[world, R, 3] on the side stream (overlaps the next frame's kernels)."""
        if self.world == 1:
            return
        main = torch.cuda.current_stream(self.dev)
        self.comm.wait_stream(main)
        col.record_stream(self.comm)
        with torch.cuda.stream(self.comm):
            self.dist.all_gather_into_tensor(out.view(-1, 3), col)

    def join(self):
        if self.world > 1:
            torch.cuda.current_stream(self.dev).wait_stream(self.comm)

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def time_region(D, flush, fn, steps):
    """EXACTLY `steps` steps between a barrier + synchronize on both sides; one CUDA event pair on the launching stream around the
    whole region (the side-stream collectives are joined before the closing event); L2 flushed before every step (inside the
    region: a 160 MB fill, ~0.03 ms).  Returns total ms, max over ranks."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    D.barrier()
    e0.record()
    for k in range(steps):
        flush.fill_(1)
        fn(k)
    D.join()
    e1.record()
    D.barrier()
    return D.max_over_ranks(e0.elapsed_time(e1))


def render_section(D, net, cam_list, rays_host, steps, warmup, flush, e2e=False):
    """Times `steps` frames.  rays_host: this rank's pinned [R,3] ray directions; cam_list: (campos, camrot, near, far, bg).
    Resident mode: rays already on the device.  e2e mode: H2D of the rays and D2H of the colours inside every step.
    Returns (ms, R, the render_full outputs of the last step)."""
    dev = D.dev
    R = rays_host.shape[0]
    rays_dev = rays_host.to(dev)
    gathered = [torch.empty((D.world, R, 3), dtype=torch.float32, device=dev) for _ in range(2)] if D.world > 1 else None
    out_host = torch.empty((R, 3), dtype=torch.float32).pin_memory()
    last = {}

    def step(k):
        rd = rays_host.to(dev, non_blocking=True) if e2e else rays_dev
        with torch.no_grad():
            out = net.render_full(cam_list[0], rd, cam_list[1], cam_list[2], cam_list[3], cam_list[4])
        if k == steps - 1:
            last["out"] = out
        col = out["coarse_raycolor"][0]
        if D.world > 1:
            D.gather_async(col, gathered[k & 1])
        if e2e:
            out_host.copy_(col, non_blocking=True)

    from pointnerf_b200.lib import PnbOverflow
    for attempt in range(2):
        for k in range(warmup):
            step(k)
        D.join()
        D.barrier()
        try:
            net.check_errors()
            break
        except PnbOverflow:                     # a scene denser than the workspace heuristic: the workspace has grown, warm up again
            if attempt == 1 or warmup == 0:
                raise
    last.clear()
    ms = time_region(D, flush, step, steps)
    net.check_errors()
    return ms, R, last.get("out")


def dump_outputs(out, directory):
    """render_full outputs -> directory/<name>.npy (float32); coarse_point_opacity for a seeded sample of the rays."""
    os.makedirs(directory, exist_ok=True)
    arrays = {k: out[k].float().cpu().numpy() for k in ("coarse_raycolor", "coarse_is_background", "ray_mask")}
    R = out["coarse_point_opacity"].shape[1]
    rays = np.sort(np.random.RandomState(0).choice(R, min(R, DUMP_OPACITY_RAYS), replace=False))
    arrays["coarse_point_opacity"] = out["coarse_point_opacity"][:, torch.from_numpy(rays).to(out["coarse_point_opacity"].device)].cpu().numpy()
    arrays["coarse_point_opacity_rays"] = rays.astype(np.float32)
    for k, v in arrays.items():
        np.save(os.path.join(directory, k + ".npy"), v)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", type=str, default="pnb200")
    ap.add_argument("--sr", type=int, default=24)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--only", type=str, default="", help="comma list of sub-results to run besides the main line: strong,truck,train,scannet,cold,sr80 (default: all)")
    ap.add_argument("--precision", type=str, default="bf16x3", help="bf16x3 (tcgen05, default) | fp32 (CUDA cores)")
    ap.add_argument("--frozen", type=int, default=1, help="1 (default): frozen-cloud pair kernel k_shade_tc8 (point-only layer-1 inputs hoisted per point) | 0: general kernel k_shade_tc7")
    ap.add_argument("--dump-outputs", type=str, default=None, metavar="DIR",
                    help="write the outputs of the last timed step of the main line to DIR/<name>.npy (float32, rank 0)")
    args = ap.parse_args()
    if args.impl == "reference":
        return run_reference_arm(args)
    want = set(x for x in args.only.split(",") if x) or {"strong", "truck", "train", "scannet", "cold", "sr80"}

    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    D = Dist(dev)
    rank, world = D.rank, D.world
    assert world == args.gpus, "WORLD_SIZE %d != --gpus %d (launch N>1 with torchrun)" % (world, args.gpus)
    W = max(args.warmup, 3)
    flush = torch.empty(160 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    cfg = scene.CONFIGS["lego_render"]
    cfg.SR = args.sr
    net, pts, opt = harness.build_model(cfg, dev, seed=0, alpha_bias=3.0, pnb_precision=args.precision, pnb_frozen=args.frozen)
    full = scene.make_rays(cfg)
    dirs_cam = full["raydir"][0]                                   # camera-frame directions (z = 1), pose 0 = identity
    R_img = dirs_cam.shape[0]
    bg = [1., 1., 1.]

    # ---------------- main line: WEAK scaling, rank g renders the frame of pose g
    Rg = roll(rank, world)
    mine = (dirs_cam @ Rg.t()).contiguous().pin_memory()
    cam = (list(cfg.campos), Rg, cfg.near, cfg.far, bg)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    render_section(D, net, cam, mine, 1, W, flush)                # warm-up (also sizes the workspaces)
    # the timed region of the contract: EXACTLY K steps, barrier + synchronize on both sides -> `value` / `ms_per_step`.  It is followed by
    # ONE repeat of the same region, reported next to it (`config.timed_regions_ms_per_step`) and not used for the value: the GPU boxes
    # share their host, and a stalled launching thread occasionally adds milliseconds to a region that has nothing to do with the GPU
    # work - the repeat makes such a run recognisable
    regions = []
    for i in range(2):
        t_w0 = time.time()
        ms_i, R, out_i = render_section(D, net, cam, mine, args.steps, 0, flush)
        regions.append((ms_i, t_w0, time.time()))
        if i == 0 and args.dump_outputs and rank == 0:
            dump_outputs(out_i, args.dump_outputs)
        del out_i
    ms_res, t_w0, t_w1 = regions[0]
    clocks = sampler.stop(t_w0, t_w1) if sampler else None
    # workload counters (oracle-independent: the library's own device counters)
    qc = net.neural_points.querier.run_query(net.neural_points.xyz.detach(), mine.to(dev), cam[0], cam[2], cam[3], want_counters=True).counters
    gc = net.neural_points.querier.last_grid_counters
    with torch.no_grad():
        net.render_full(cam[0], mine.to(dev), cam[1], cam[2], cam[3], cam[4])     # net.last = a full query again
    torch.cuda.synchronize(dev)

    # ---------------- dominant kernel alone: CUDA events around the launch on the launching stream, same inputs, L2 flushed
    from pointnerf_b200 import lib as _lib
    from pointnerf_b200.point_query import make_cam_opts
    l = _lib.load()
    q = net.last
    mlp = net._mlp.get(net.aggregator)
    ptsd = net.neural_points.points_desc()
    o = make_cam_opts(cam[0], cam[1], Rw2c=None, vsize_z=float(opt.vsize[2]), bg_color=cam[4], raydist_mode_unit=opt.raydist_mode_unit)
    stream = torch.cuda.current_stream(dev).cuda_stream
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def time_kernel(launch):
        ms = []
        for i in range(args.steps + 1):
            flush.fill_(1)
            e0.record()
            launch()
            e1.record()
            torch.cuda.synchronize(dev)
            if i > 0:
                ms.append(e0.elapsed_time(e1))
        return float(np.mean(ms))

    frozen = bool(net.frozen_ok) and args.precision != "fp32"
    if args.precision == "fp32":
        shade_avg = time_kernel(lambda: _lib.check(l.pnb_shade_forward(
            _lib.C.byref(q.desc), _lib.C.byref(ptsd), _lib.C.byref(mlp), _lib.C.byref(o), net._sigma_rgb.data_ptr(), None, 0, stream),
            "pnb_shade_forward"))
        color_avg = None
        kname = "k_shade_fwd (fp32 CUDA-core kernel: pair MLPs + colour branch)"
        kflops = FLOPS_PER_PAIR * qc["n_pairs"] + FLOPS_PER_SAMPLE * qc["n_valid"]
        issued = None
        n_launch = LAUNCHES_PER_STEP_FP32
    else:
        pre_ptr = net._point_pre(mlp, ptsd, stream).data_ptr() if frozen else None

        def tc(flags):
            _lib.check(l.pnb_shade_forward_tc(_lib.C.byref(q.desc), _lib.C.byref(ptsd), _lib.C.byref(mlp), net._mlp.packed.data_ptr(), pre_ptr,
                                              _lib.C.byref(o), net._sigma_rgb.data_ptr(), net._tc_ws.data_ptr(), net._tc_ws.numel(),
                                              net._max_valid, flags | (_lib.TC_FROZEN if frozen else 0), net._err.data_ptr(), stream),
                       "pnb_shade_forward_tc")
        shade_avg = time_kernel(lambda: tc(_lib.TC_PAIRS))
        color_avg = time_kernel(lambda: tc(_lib.TC_COLOR))
        kname = ("k_shade_tc8 (frozen cloud: the 224 point-only inputs of block1.0 hoisted into a per-point table)" if frozen else "k_shade_tc7") + \
            " incl. the 3 row-packing kernels (tcgen05 BF16x3 pair MLPs 284-256-256 | 263-256-256 + alpha + K-reduction)"
        kflops = FLOPS_PER_PAIR * qc["n_pairs"]
        n_tiles = math.ceil(qc["n_pairs"] / 0.993 / 128.0)       # packed rows: 99.3 % fill (tools/tc_profile.py prints the exact count)
        issued = MMAS_PER_TILE[frozen] * MMA_FLOPS * n_tiles
        n_launch = LAUNCHES_PER_STEP_TC
        net.check_errors()

    # ---------------- e2e: host buffers, H2D of the rays + D2H of the colours inside the timed region
    ms_e2e, _, _ = render_section(D, net, cam, mine, args.steps, 2, flush, e2e=True)

    total_rays = R * world * args.steps
    value = total_rays / (ms_res * 1e-3) / 1e6
    e2e_val = total_rays / (ms_e2e * 1e-3) / 1e6
    pk = peaks()
    traffic = None
    tfile = os.path.join(ROOT, "profiles", "r02_ncu_dram_traffic.json")
    if os.path.exists(tfile) and args.precision != "fp32" and args.sr == 24:
        traffic = json.load(open(tfile)).get("k_shade_tc8" if frozen else "k_shade_tc7", None)
    achieved = kflops / (shade_avg * 1e-3) / 1e12
    peak = pk["bf16_tflops"]

    sub = {}
    # ---------------- strong scaling: ONE frame, rays interleave-sharded over the ranks
    if "strong" in want:
        mine_s = dirs_cam[rank::world].contiguous().pin_memory()
        cam0 = (list(cfg.campos), torch.eye(3), cfg.near, cfg.far, bg)
        ms_s, Rs, _ = render_section(D, net, cam0, mine_s, args.steps, W, flush)
        sub["strong"] = dict(value=R_img * args.steps / (ms_s * 1e-3) / 1e6, unit="Mrays/s", ms_per_frame=ms_s / args.steps,
                             rays_per_rank=Rs, what="one 800x800 frame, ray i -> rank i %% %d, all-gather of the [R/N,3] tiles inside the timed "
                             "region (side stream, double-buffered)" % world)
    # ---------------- cold: new point cloud every step (voxel grid + frozen table rebuilt inside the timed region)
    if "cold" in want and world == 1:
        def cold_step(k):
            net.neural_points.querier.clean_up()
            net._pre_key = None
            with torch.no_grad():
                net.render_full(cam[0], q.raydir, cam[1], cam[2], cam[3], cam[4])
        cold_step(0)
        ms_cs = [time_region(D, flush, cold_step, 3) for _ in range(2)]      # host synchronisations inside: the faster of two regions (shared host)
        ms_c = min(ms_cs)
        sub["cold"] = dict(value=R_img * 3 / (ms_c * 1e-3) / 1e6, unit="Mrays/s", ms_per_frame=ms_c / 3, regions_ms_per_frame=[m / 3 for m in ms_cs],
                           what="voxel grid build (incl. its host synchronisation for the counters) + per-point layer-1 table inside every step")
    del net
    torch.cuda.empty_cache()
    # ---------------- SR = 80 (the shipped value of the NeRF-Synthetic scripts)
    if "sr80" in want and world == 1 and args.sr != 80:
        cfg80 = scene.CONFIGS["lego_render"]
        cfg80.SR = 80
        net80, _, _ = harness.build_model(cfg80, dev, seed=0, alpha_bias=3.0, pnb_precision=args.precision, pnb_frozen=args.frozen)
        ms80, _, _ = render_section(D, net80, cam, mine, 5, W, flush)
        sub["sr80"] = dict(value=R_img * 5 / (ms80 * 1e-3) / 1e6, unit="Mrays/s", ms_per_frame=ms80 / 5)
        cfg80.SR = args.sr
        del net80
        torch.cuda.empty_cache()
    # ---------------- config 4: Truck, 2M points, 960x540, kernel_size 5, one frame sharded over the ranks
    if "truck" in want:
        tcfg = scene.CONFIGS["truck_8gpu"]
        tnet, _, topt = harness.build_model(tcfg, dev, seed=0, alpha_bias=3.0, pnb_precision=args.precision, pnb_frozen=args.frozen)
        tdirs = scene.make_rays(tcfg)["raydir"][0]
        tmine = tdirs[rank::world].contiguous().pin_memory()
        tcam = (list(tcfg.campos), torch.eye(3), tcfg.near, tcfg.far, bg)
        ms_t, Rt, _ = render_section(D, tnet, tcam, tmine, 5, W, flush)
        tq = tnet.neural_points.querier.run_query(tnet.neural_points.xyz.detach(), tmine.to(dev), tcam[0], tcam[2], tcam[3], want_counters=True).counters
        sub["truck"] = dict(value=tdirs.shape[0] * 5 / (ms_t * 1e-3) / 1e6, unit="Mrays/s", ms_per_frame=ms_t / 5, rays_per_rank=Rt,
                            workload="truck_8gpu: 960x540, N=2000000 points, kernel_size 5, vsize 0.002, SR=24, one frame interleave-sharded x%d" % world,
                            rank0_counters=dict(hit_rays=tq["R2"], valid_samples=tq["n_valid"], valid_pairs=tq["n_pairs"]),
                            point_table_mb=round(2e6 * 168 / 1e6), hoisted_table_mb=round(2e6 * 1024 / 1e6))
        del tnet
        torch.cuda.empty_cache()
    # ---------------- config 3: per-scene optimisation step (3600 rays per step over the ranks)
    if "train" in want:
        sub["train"] = train_section(D, args, dev)
    # ---------------- config 5: ScanNet-sized cloud (5M points, P=30): optimisation step with the sparse exchange + one prune/grow cycle
    if "scannet" in want:
        sub["scannet"] = train_section(D, args, dev, cfg_name="scannet_8gpu", sparse=True, n_steps=10, grow_cycle=True)

    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            cpu = cpu_baseline_leg(args.sr)
        line = dict(
            metric=METRIC, value=value, unit="Mrays/s", n_gpus=world, steps=args.steps, warmup=W,
            ms_per_step=ms_res / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
            dtype=("f32 (bf16x3 split on tcgen05, fp32 accumulate)" if args.precision != "fp32" else "f32"),
            data="synthetic",
            config=dict(workload=WORKLOAD % args.sr,
                        rays_per_step_per_gpu=R,
                        timed_regions_ms_per_step=[r[0] / args.steps for r in regions],
                        timing="value / ms_per_step = the first region of exactly K steps (barrier + synchronize on both sides); the second entry is one repeat of the same region, for comparison only",
                        parallelism=("%d distinct poses (rolls about the view axis), rank g renders frame g; points / grid / MLP replicated%s"
                                     % (world, "; one all-gather of the colours per step on a side stream" if world > 1 else "")),
                        l2="flushed before every timed step (160 MiB fill inside the region); the per-frame working set (410 MB per-point "
                           "table, 3.5 GB h-bar) exceeds the 126 MB L2 anyway",
                        workload_counters=dict(hit_rays=qc["R2"], valid_samples=qc["n_valid"], valid_pairs=qc["n_pairs"],
                                               candidate_samples=qc["n_cand"], occupied_voxels=gc["n_occ"], max_pts_per_voxel=gc["max_pts"])),
            e2e=dict(value=e2e_val, unit="Mrays/s", h2d_bytes_per_step=int(mine.numel() * 4 * world),
                     d2h_bytes_per_step=int(R * 3 * 4 * world), ms_per_step=ms_e2e / args.steps),
            gpu_launches=n_launch * args.steps,
            clocks=clocks,
            roofline=dict(bound="tensor", kernel=kname, achieved=achieved, peak=peak, unit="TFLOP/s",
                          frac=achieved / peak, traffic=traffic, peak_source="%s bf16 cuBLAS burst (MEASURED_PEAKS.json)" % pk["source"],
                          algorithmic_flops_per_launch=kflops, kernel_ms=shade_avg,
                          kernel_share_of_step=shade_avg / (ms_res / args.steps),
                          issued_mma_flops_per_launch=issued,
                          tensor_pipe_frac_issued=(issued / (shade_avg * 1e-3) / 1e12 / peak if issued else None),
                          note=("algorithmic = SURVEY 8(d) formula (542,720 FLOP per valid pair); the frozen pipeline computes 21 % of "
                                "them once per point instead of once per pair, issued = the tcgen05.mma actually launched (BF16x3: 3 per product)"
                                if frozen else None),
                          colour_branch_kernel_ms=color_avg),
            cpu_baseline=cpu,
        )
        line.update(sub)
        if _RETRY_NOTE:
            line["retried_after"] = _RETRY_NOTE        # the first attempt tripped the in-kernel watchdog (see __main__)
        print(json.dumps(line))
    D.close()
    return 0


def train_section(D, args, dev, cfg_name="ship_optimise", sparse=False, n_steps=20, grow_cycle=False):
    """Per-scene optimisation step (run/train_ft.py): 3600 random rays of one view per step (lego_cuda.sh:109), train jitter on,
    forward + backward + gradient exchange + 2x Adam (parallel.TrainStep).  The step's rays are split over the ranks
    (ray i -> rank i % world).  cfg_name: ship_optimise = BASELINE configs[2] (N=600k); scannet_8gpu = configs[4] (N=5M, P=30,
    sparse touched-rows exchange of the point gradients, plus one prune + probe + grow cycle when grow_cycle)."""
    from pointnerf_b200 import parallel
    cfg = scene.CONFIGS[cfg_name]
    net, pts, opt = harness.build_model(cfg, dev, alpha_bias=3.0, is_train=True, pnb_precision=args.precision)
    ts = parallel.TrainStep(net, world=D.world, rank=D.rank, sparse_points=sparse)
    rng = np.random.RandomState(0)
    g = torch.Generator().manual_seed(1)
    n_warm = 4
    acc = dict(forward=0.0, backward=0.0, exchange=0.0, adam=0.0)
    tot = 0.0
    hit = 0
    host = 0.0

    def batch():
        px = rng.randint(0, cfg.W, size=(3600,)).astype(np.float32)
        py = rng.randint(0, cfg.H, size=(3600,)).astype(np.float32)
        gt = torch.rand(3600, 3, generator=g)
        sel = np.arange(D.rank, 3600, D.world)
        # the per-ray tensors go to the device; the camera scalars (position, rotation, near / far, intrinsics) stay host tensors, as a
        # data loader delivers them (the kernels take them by value: device copies would cost one synchronising D2H read each)
        rays = {k: (v.to(dev) if k in ("raydir", "pixel_idx") else v) for k, v in scene.make_rays(cfg, np.stack([px, py], -1)[sel]).items()}
        kw = dict(campos=rays["campos"], raydir=rays["raydir"], bg_color=rays["bg_color"], camrotc2w=rays["camrotc2w"], pixel_idx=rays["pixel_idx"],
                  near=rays["near"], far=rays["far"], h=rays["h"], w=rays["w"], intrinsic=rays["intrinsic"])
        return kw, gt[sel].to(dev)

    for it in range(n_warm + n_steps):
        kw, gt = batch()
        evs = []

        def mark(name):
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            evs.append((name, e))
        t_h0 = time.perf_counter()
        ts.step(kw, gt, mark=mark)
        t_h1 = time.perf_counter()
        torch.cuda.synchronize(dev)
        if os.environ.get("PNB_TRAIN_PROFILE") and D.rank == 0:
            st = torch.cuda.memory_stats(dev)
            sys.stderr.write("[train step %2d] %.2f ms  host %.2f ms  cudaMalloc calls %d  reserved %.2f GB  hit %d\n" % (
                it, evs[0][1].elapsed_time(evs[-1][1]), (t_h1 - t_h0) * 1e3, st.get("num_device_alloc", -1), st["reserved_bytes.all.current"] / 1e9,
                int(ts.last["n_hit_terms"] / 3)))
        if it >= n_warm:
            host += t_h1 - t_h0
            for (n0, a), (n1, b) in zip(evs[:-1], evs[1:]):
                acc[n1] += a.elapsed_time(b)
            tot += evs[0][1].elapsed_time(evs[-1][1])
            hit += int(ts.last["n_hit_terms"] / 3)
    if os.environ.get("PNB_TRAIN_PROFILE") and D.rank == 0:      # diagnostic: per-kernel device time of 5 more steps (stderr)
        from torch.profiler import profile, ProfilerActivity
        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            for _ in range(5):
                ts.step(*batch())
            torch.cuda.synchronize(dev)
        rows = sorted(prof.key_averages(), key=lambda e: -e.device_time_total)
        sys.stderr.write("[train profile %s] device time per step %.3f ms, %d events\n" % (cfg_name, sum(e.device_time_total for e in rows) / 5e3, sum(e.count for e in rows) // 5))
        for e in rows[:8]:
            sys.stderr.write("   %8.3f ms/step x%-4d %s\n" % (e.device_time_total / 5e3, e.count // 5, e.key[:90]))
        rows = sorted(prof.key_averages(), key=lambda e: -e.self_cpu_time_total)
        for e in rows[:12]:
            sys.stderr.write("   cpu %8.3f ms/step x%-4d %s\n" % (e.self_cpu_time_total / 5e3, e.count // 5, e.key[:90]))
    ms = D.max_over_ranks(tot / n_steps)
    out = dict(steps_per_s=1e3 / ms, ms_per_step=ms, ms_fwd=acc["forward"] / n_steps, ms_bwd=acc["backward"] / n_steps,
               ms_exchange=acc["exchange"] / n_steps, ms_adam=acc["adam"] / n_steps, ms_host_issue=host / n_steps * 1e3, mrays_per_s=3600 / ms / 1e3,
               hit_rays_per_step=hit / n_steps,
               what="%s: N=%d, 3600 rays per step over %d rank(s), fwd (tcgen05) + bwd (tcgen05 GEMMs) + %s + 2x Adam over all N rows; "
                    "per-phase ms are rank 0's, ms_per_step the max over ranks"
                    % (cfg_name, cfg.N, D.world, "sparse touched-rows exchange of the point gradients + flat all-reduce of the MLP gradients" if sparse
                       else "one flat gradient all-reduce"))
    if grow_cycle:
        # prune (deterministic function of the replicated points_conf, neural_points.py:347-370: no communication), then a probe pass
        # (opt.prob = 1 outputs, run/train_ft.py:417-530) on this rank's share of one frame's rays, new points = the arg-max-opacity
        # sample locations with their averaged attributes, merged across ranks (allgather_new_points), grow, optimisers rebuilt,
        # and one more step on the new cloud (voxel grid rebuilt inside it)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        t_host = time.perf_counter()
        e0.record()
        n0 = net.neural_points.xyz.shape[0]
        pruned = net.neural_points.prune(0.12)
        opt.prob = 1
        opt.is_train = False
        kw, _ = batch()
        with torch.no_grad():
            pr = net(**kw)
        opt.prob = 0
        opt.is_train = True
        keep = pr["ray_max_shading_opacity"][0, :, 0] > 0.5 if pr["ray_max_shading_opacity"].numel() else torch.zeros(0, dtype=torch.bool, device=dev)
        keep = keep & (torch.arange(keep.shape[0], device=dev) % 4 == 0)
        add = [pr["ray_max_sample_loc_w"][0][keep], pr["shading_avg_embedding"][0][keep], pr["shading_avg_color"][0][keep],
               pr["shading_avg_dir"][0][keep], pr["shading_avg_conf"][0][keep]] if keep.numel() else None
        if add is None:
            z = lambda c: torch.zeros((0, c), device=dev)
            add = [z(3), z(32), z(3), z(3), z(1)]
        merged = parallel.allgather_new_points(*add, D.world)
        net.neural_points.grow_points(*merged)
        ts = parallel.TrainStep(net, world=D.world, rank=D.rank, sparse_points=sparse)     # new parameters -> new optimisers (train_ft.py:834-842)
        kw, gt = batch()
        ts.step(kw, gt)
        e1.record()
        torch.cuda.synchronize(dev)
        out["grow_cycle"] = dict(ms=D.max_over_ranks(e0.elapsed_time(e1)), host_ms=(time.perf_counter() - t_host) * 1e3, points_before=n0,
                                 pruned=int(pruned), grown=int(merged[0].shape[0]), points_after=int(net.neural_points.xyz.shape[0]),
                                 what="prune(conf < 0.12) + probe pass (opt.prob = 1) + variable-length all-gather of the new points + grow + "
                                      "optimiser rebuild + one optimisation step on the new cloud (voxel grid rebuilt)")
    del net, ts
    torch.cuda.empty_cache()
    return out


_RETRY_NOTE = None

if __name__ == "__main__":
    try:
        rc = main()
    except Exception as e:  # noqa: BLE001
        from pointnerf_b200.lib import PnbError
        single = int(os.environ.get("WORLD_SIZE", "1")) == 1       # with several ranks a one-sided retry would hang the collectives
        if isinstance(e, PnbError) and "time-out" in str(e) and single:
            # every in-kernel mbarrier wait is bounded (2 s): a protocol stall surfaces as this error instead of a hung GPU.
            # Never seen on the final pipeline; if it ever happens the run is re-measured once and the JSON line says so.
            print("bench.py: %s -- re-measuring once" % e, file=sys.stderr)
            _RETRY_NOTE = str(e)
            rc = main()
        else:
            raise
    sys.exit(rc)
