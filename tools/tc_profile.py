"""Run on the GPU box, lego_render frame: per-CTA cycle counts of the pair kernel (dbg flag 4: cycles + SM id of every CTA into
d_err[64..]) and the cycles per 128-row tile they imply.  PNB_FROZEN=0 selects the general kernel (k_shade_tc7), default the
frozen-cloud kernel (k_shade_tc8; PNB_DBG_FLAGS=16: static tile schedule instead of the tile queue); PNB_NO_WEIGHTS=1 removes the weight traffic (garbage results, timing experiment);
PNB_SR / PNB_CONFIG override the workload."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from pointnerf_b200 import harness, scene, lib as L
dev = torch.device("cuda:0")
cfg = scene.CONFIGS[os.environ.get("PNB_CONFIG", "lego_render")]
over = {}
if os.environ.get("PNB_SR"):
    over["SR"] = int(os.environ["PNB_SR"])
net, pts, opt = harness.build_model(cfg, dev, alpha_bias=3.0, pnb_frozen=int(os.environ.get("PNB_FROZEN", "1")), **over)
rays = scene.make_rays(cfg)
rd = rays["raydir"].to(dev)
for i in range(3):
    with torch.no_grad():
        ref_out = net.render_full(list(cfg.campos), rd, torch.eye(3), cfg.near, cfg.far, [1., 1., 1.])
ref_col, ref_opa = ref_out["coarse_raycolor"].clone(), ref_out["coarse_point_opacity"].clone()
net.check_errors()
net.dbg_flags = 4 | int(os.environ.get("PNB_DBG_FLAGS", "0")) | (1 if os.environ.get("PNB_PROF") else 0)       # frozen kernel: +8 = the non-deferred last epilogue (k_shade_tc8<.., DEFER = false>)
if os.environ.get("PNB_NO_WEIGHTS"):
    net.dbg_flags |= 0          # (the no-weights bit is a top-level flag)
    L.TC_PAIRS |= L.TC_DBG_NO_WEIGHTS
torch.cuda.synchronize()
with torch.no_grad():
    out = net.render_full(list(cfg.campos), rd, torch.eye(3), cfg.near, cfg.far, [1., 1., 1.])
torch.cuda.synchronize()
print("vs the default variant: max |d colour| %.3e  max |d opacity| %.3e" % (float((out["coarse_raycolor"] - ref_col).abs().max()),
                                                                             float((out["coarse_point_opacity"] - ref_opa).abs().max())))
per = net._err.cpu().view(torch.int64)[32:32 + 148].tolist()
n_quads = int(net._err.cpu().view(torch.int64)[32 + 192])
cyc = [(v & 0xffffffffffff) for v in per]
cnt = net.last.counters_tensor().cpu().tolist()
n_tiles = (n_quads + 3) // 4
print("kernel", "k_shade_tc8 (frozen, dbg %d)" % net.dbg_flags if net.frozen_ok else "k_shade_tc7 (general)", "| status", int(net._err[0]),
      "| n_valid", cnt[L.QC["n_valid"]], "n_pairs", cnt[L.QC["n_pairs"]], "n_quads", n_quads, "tiles", n_tiles,
      "row fill %.4f" % (cnt[L.QC["n_pairs"]] / max(n_quads * 32, 1)))
print("per-CTA cycles: min %.2f M  max %.2f M  mean %.2f M -> %.1f k cycles per 128-row tile (tiles per CTA %.1f)"
      % (min(cyc) / 1e6, max(cyc) / 1e6, sum(cyc) / len(cyc) / 1e6, sum(cyc) / len(cyc) / (n_tiles / 148.0) / 1e3, n_tiles / 148.0))
print("per-CTA kernel cycles (M) @smid:", " ".join("%.1f@%d" % ((v & 0xffffffffffff) / 1e6, v >> 48) for v in per))

if os.environ.get("PNB_PROF") and net.frozen_ok:
    c = net._err.cpu().view(torch.int64)[1:23].tolist()
    names = ["loader: wait empty", "issuer: wait acc_full (l>0)", "issuer: wait final (l=0)", "issuer: wait a1_ready", "issuer: wait drain",
             "issuer: wait kblk (slow path)", "issuer: wait weights (slow path)", "issuer: MMA issue + commits + fast probes",
             "builder q0: wait a1_free", "builder q0: build", "builder q0: wait final", "builder q0: last-epilogue share", "builder q0: wait alpha",
             "epi warp 0: wait prow", "epi warp 0: wait acc_full (E1)", "epi warp 0: E1 busy", "epi warp 0: wait acc_full (E2,E3)", "epi warp 0: E2+E3 busy",
             "epi warp 0: wait final", "epi warp 0: last-epilogue share (DEFER: drain only)", "kernel total (thread 0)",
             "epi warp 0: deferred last-epilogue chunks (gaps A-C of the next tile)"]
    tiles0 = int(net._err.cpu().view(torch.int64)[32 + 193]) or (n_tiles - 1) // 148 + 1     # tiles block 0 processed (k_shade_tc8)
    print("block 0 accounting (%d tiles), cycles per tile:" % tiles0)
    for n, v in zip(names, c):
        print("  %-46s %9.0f  (%5.1f %% of the kernel)" % (n, v / tiles0, 100.0 * v / max(c[20], 1)))
