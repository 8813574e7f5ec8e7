// Point growing: the per-ray probe outputs and the per-frame hole selection of the reference's probe_hole
// (run/train_ft.py:417-530), on the device.
//
//   k_probe_maps     neural_points_volumetric_model.py:331-351 followed by fill_invalid / unmask (:87-123), full-R, straight from the
//                    sample-compacted query and the [R,SR] opacity of k_composite (no dense [R',SR,K] export).  One warp per ray.
//   k_probe_mark     train_ft.py:493-505 on the H x W pixel grid: GT miss mask, 3x3 bloat (bloat_inds with its border clamp),
//                    the far_thresh branch and the opacity threshold -> one flag per pixel.  One thread per pixel.
//   k_probe_compact  the boolean-mask indexing of train_ft.py:508-512: selected pixels in row-major order (exclusive scan of the flags,
//                    deterministic) -> add_xyz / add_embedding / add_color / add_dir / add_conf and the device-side count.
#include "common.cuh"

namespace pnb {

struct ProbeMapParams {
    pnb_query_t q;
    pnb_points_t pts;
    const float* opacity;   // [R, SR] (k_composite)
    float* op_max;          // [R]
    float* loc;             // [R, 3]
    float* far_dist;        // [R]
    float* avg_color;       // [R, 3]
    float* avg_dir;         // [R, 3]
    float* avg_conf;        // [R]
    float* avg_emb;         // [R, 32]
    int32_t* argmax;        // [R] or null
};

// torch.max(dim) order: NaN above everything, then the larger value, ties to the lower index
__device__ __forceinline__ bool probe_better(float a, int ia, float b, int ib) {
    const bool na = a != a, nb = b != b;
    if (na != nb) return na;
    if (!na && a != b) return a > b;
    return ia < ib;
}

__global__ void __launch_bounds__(256) k_probe_maps(ProbeMapParams p) {
    const pnb_query_t& q = p.q;
    const int lane = threadIdx.x & 31;
    const long long r_ll = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r_ll >= q.R) return;                                    // whole warps leave together
    const int r = (int)r_ll, SR = q.SR, K = q.K;
    if (q.ray_hit[r] == 0) {                                    // unmask: zeros outside the hit rays
        p.avg_emb[(size_t)r * PNB_FEAT + lane] = 0.f;
        if (lane < 3) { p.loc[3 * r + lane] = 0.f; p.avg_color[3 * r + lane] = 0.f; p.avg_dir[3 * r + lane] = 0.f; }
        if (lane == 0) { p.op_max[r] = 0.f; p.far_dist[r] = 0.f; p.avg_conf[r] = 0.f; if (p.argmax) p.argmax[r] = -1; }
        return;
    }
    // arg-max opacity over all SR slots (unfilled slots hold 0), first index on ties
    const float* op = p.opacity + (size_t)r * SR;
    float best = -INFINITY;
    int bi = 0x7fffffff;
    for (int j = lane; j < SR; j += 32) {
        const float v = op[j];
        if (probe_better(v, j, best, bi)) { best = v; bi = j; }
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, best, d);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, d);
        if (probe_better(ov, oi, best, bi)) { best = ov; bi = oi; }
    }
    // world position of the slot, as pnb_query_export forms it (fp32 mul then add); an unfilled slot is the origin with no neighbours
    float lx = 0.f, ly = 0.f, lz = 0.f;
    int pid = -1;
    if (bi < q.nsamp[r]) {
        const float t = q.t[(size_t)r * q.t_ray_stride + q.steps[(size_t)r * SR + bi]];
        lx = raypos1(q.campos[0], q.raydir[3 * r], t);
        ly = raypos1(q.campos[1], q.raydir[3 * r + 1], t);
        lz = raypos1(q.campos[2], q.raydir[3 * r + 2], t);
        if (lane < K) pid = q.cand_pidx[(size_t)(q.samp_off[r] + bi) * K + lane];
    }
    // lane k < K: neighbour k (index clamped to 0 as the reference gathers it), its distance and inverse-distance weight
    const int idx = pid > 0 ? pid : 0;
    float dist = INFINITY, w = 0.f;
    if (lane < K) {
        const float dx = __ldg(&p.pts.xyz[3 * idx]) - lx, dy = __ldg(&p.pts.xyz[3 * idx + 1]) - ly, dz = __ldg(&p.pts.xyz[3 * idx + 2]) - lz;
        dist = sqrtf(dx * dx + dy * dy + dz * dz);
        w = pid >= 0 ? 1.0f / fmaxf(dist, 1e-6f) : 0.f;
    }
    float wsum = 0.f, far = INFINITY;
    for (int k = 0; k < K; ++k) {                              // ascending slot order, the same sum on every lane
        wsum += __shfl_sync(0xffffffffu, w, k);
        far = fminf(far, __shfl_sync(0xffffffffu, dist, k));   // min over all K slots, clamped point-0 slots included
    }
    float wsel = 0.f;
    if (lane < K) wsel = (w / fmaxf(wsum, 1e-8f)) * fminf(fmaxf(__ldg(&p.pts.conf[idx]), 1e-4f), 1.0f);
    // weighted averages, added in ascending slot order: lane = embedding channel; lanes 0-2 colour, 3-5 direction, 6 conf
    float acc = 0.f, acc_s = 0.f;
    const float* small = lane < 3 ? p.pts.color + lane : lane < 6 ? p.pts.dir + (lane - 3) : p.pts.conf;
    const int small_stride = lane < 6 ? 3 : 1;
    for (int k = 0; k < K; ++k) {
        const float wk = __shfl_sync(0xffffffffu, wsel, k);
        const int ik = __shfl_sync(0xffffffffu, idx, k);
        acc = __fadd_rn(acc, __fmul_rn(__ldg(&p.pts.emb[(size_t)ik * PNB_FEAT + lane]), wk));
        if (lane < 7) acc_s = __fadd_rn(acc_s, __fmul_rn(__ldg(&small[(size_t)ik * small_stride]), wk));
    }
    p.avg_emb[(size_t)r * PNB_FEAT + lane] = acc;
    if (lane < 3) p.avg_color[3 * r + lane] = acc_s;
    else if (lane < 6) p.avg_dir[3 * r + lane - 3] = acc_s;
    else if (lane == 6) p.avg_conf[r] = acc_s;
    if (lane == 0) {
        p.op_max[r] = best;
        p.loc[3 * r] = lx; p.loc[3 * r + 1] = ly; p.loc[3 * r + 2] = lz;
        p.far_dist[r] = far;
        if (p.argmax) p.argmax[r] = bi;
    }
}

struct ProbeSelectParams {
    int H, W;
    const int8_t* ray_mask;     // [H*W] (0 where no ray was cast)
    const uint8_t* present;     // [H*W] pixels given (edge_mask) or null = all
    const float* gt;            // [H*W, 3] (0 where not present)
    const float* color;         // [H*W, 3] coarse_raycolor
    const float* far_dist;      // [H*W]
    const float* op_max;        // [H*W]
    const float* loc;           // [H*W, 3]
    const float* emb;           // [H*W, 32]
    const float* avg_color;     // [H*W, 3]
    const float* avg_dir;       // [H*W, 3]
    const float* avg_conf;      // [H*W]
    float bg[3];
    float opacity_thresh, far_thresh;
    uint8_t* flags;             // [H*W] scratch
    const uint32_t* offs;       // [H*W + 1] exclusive scan of flags
    int cap;
    float *add_xyz, *add_emb, *add_color, *add_dir, *add_conf;
    int32_t* count;
};

__device__ __forceinline__ float norm3(float x, float y, float z) { return sqrtf(x * x + y * y + z * z); }

__global__ void __launch_bounds__(256) k_probe_mark(ProbeSelectParams p) {
    const int HW = p.H * p.W;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= HW) return;
    const int y = i / p.W, x = i - y * p.W;
    const bool hit = p.ray_mask[i] > 0;
    bool sel = false;
    if (hit && p.op_max[i] > p.opacity_thresh) {
        // a GT-visible miss in the 3x3 window clipped to the image (bloat_inds with its clamp marks exactly these pixels)
        bool marked = false;
        for (int yy = max(y - 1, 0); yy <= min(y + 1, p.H - 1) && !marked; ++yy)
            for (int xx = max(x - 1, 0); xx <= min(x + 1, p.W - 1); ++xx) {
                const int n = yy * p.W + xx;
                if ((p.present == nullptr || p.present[n]) && p.ray_mask[n] < 1 &&
                    norm3(p.gt[3 * n] - p.bg[0], p.gt[3 * n + 1] - p.bg[1], p.gt[3 * n + 2] - p.bg[2]) > 0.002f) { marked = true; break; }
            }
        if (!marked && p.far_thresh > 0.f)
            marked = p.far_dist[i] > p.far_thresh &&
                     norm3(p.gt[3 * i] - p.color[3 * i], p.gt[3 * i + 1] - p.color[3 * i + 1], p.gt[3 * i + 2] - p.color[3 * i + 2]) < 0.1f;
        sel = marked;
    }
    p.flags[i] = sel ? 1 : 0;
}

__global__ void __launch_bounds__(256) k_probe_compact(ProbeSelectParams p) {
    const int HW = p.H * p.W;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) *p.count = (int32_t)p.offs[HW];
    if (i >= HW || !p.flags[i]) return;
    const uint32_t o = p.offs[i];
    if (o >= (uint32_t)p.cap) return;
    for (int c = 0; c < 3; ++c) {
        p.add_xyz[3 * o + c] = p.loc[3 * i + c];
        p.add_color[3 * o + c] = p.avg_color[3 * i + c];
        p.add_dir[3 * o + c] = p.avg_dir[3 * i + c];
    }
    p.add_conf[o] = p.avg_conf[i];
    const float4* s = (const float4*)(p.emb + (size_t)i * PNB_FEAT);
    float4* d = (float4*)(p.add_emb + (size_t)o * PNB_FEAT);
#pragma unroll
    for (int c = 0; c < PNB_FEAT / 4; ++c) d[c] = s[c];
}

struct ProbeSelectLayout {
    uint8_t* flags;
    uint32_t* offs;
    uint32_t* scan_tmp;
    size_t bytes;
};

static ProbeSelectLayout carve_select(void* ws, size_t n) {
    Carver c(ws, 0);
    ProbeSelectLayout L;
    L.flags = c.take<uint8_t>(n);
    L.offs = c.take<uint32_t>(n + 1);
    L.scan_tmp = c.take<uint32_t>(scan_tmp_elems(n));
    L.bytes = align_up(c.off);
    return L;
}

}  // namespace pnb

using namespace pnb;

extern "C" int pnb_probe_maps(const pnb_query_t* q, const pnb_points_t* pts, const float* d_opacity, float* d_op_max, float* d_loc,
                              float* d_far_dist, float* d_avg_color, float* d_avg_dir, float* d_avg_conf, float* d_avg_emb,
                              int32_t* d_argmax, pnb_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    PNB_REQUIRE(q && pts && d_opacity && d_op_max && d_loc && d_far_dist && d_avg_color && d_avg_dir && d_avg_conf && d_avg_emb,
                PNB_ERR_INVALID, "pnb_probe_maps: null argument");
    PNB_REQUIRE(pts->xyz && pts->emb && pts->color && pts->dir && pts->conf, PNB_ERR_INVALID, "pnb_probe_maps: null point tensor");
    PNB_REQUIRE(q->K >= 1 && q->K <= PNB_MAX_K, PNB_ERR_UNSUPPORTED, "pnb_probe_maps: K=%d unsupported", q->K);
    PNB_REQUIRE(q->SR >= 1 && q->SR <= PNB_MAX_SR, PNB_ERR_UNSUPPORTED, "pnb_probe_maps: SR=%d unsupported", q->SR);
    if (q->R <= 0) return PNB_OK;
    ProbeMapParams p;
    p.q = *q; p.pts = *pts; p.opacity = d_opacity; p.op_max = d_op_max; p.loc = d_loc; p.far_dist = d_far_dist;
    p.avg_color = d_avg_color; p.avg_dir = d_avg_dir; p.avg_conf = d_avg_conf; p.avg_emb = d_avg_emb; p.argmax = d_argmax;
    const long long threads = (long long)q->R * 32;
    k_probe_maps<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(p);
    PNB_CHECK_CUDA(cudaGetLastError());
    return PNB_OK;
}

extern "C" size_t pnb_probe_select_bytes(int H, int W) {
    if (H <= 0 || W <= 0) return 0;
    return carve_select(nullptr, (size_t)H * W).bytes;
}

extern "C" int pnb_probe_select(int H, int W, const int8_t* d_ray_mask, const uint8_t* d_present, const float* d_gt,
                                const float* d_color, const float* d_far_dist, const float* d_op_max, const float* d_loc,
                                const float* d_avg_emb, const float* d_avg_color, const float* d_avg_dir, const float* d_avg_conf,
                                const float bg_color[3], float opacity_thresh, float far_thresh, void* ws, size_t ws_bytes, int cap,
                                float* d_add_xyz, float* d_add_emb, float* d_add_color, float* d_add_dir, float* d_add_conf,
                                int32_t* d_count, pnb_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    PNB_REQUIRE(H > 0 && W > 0 && (long long)H * W < (1ll << 31) - 1, PNB_ERR_INVALID, "pnb_probe_select: bad size %dx%d", H, W);
    PNB_REQUIRE(d_ray_mask && d_gt && d_color && d_far_dist && d_op_max && d_loc && d_avg_emb && d_avg_color && d_avg_dir && d_avg_conf &&
                bg_color && ws && d_count, PNB_ERR_INVALID, "pnb_probe_select: null argument");
    PNB_REQUIRE(cap >= 0, PNB_ERR_INVALID, "pnb_probe_select: cap=%d", cap);
    PNB_REQUIRE(cap == 0 || (d_add_xyz && d_add_emb && d_add_color && d_add_dir && d_add_conf), PNB_ERR_INVALID,
                "pnb_probe_select: null output with cap=%d", cap);
    PNB_REQUIRE(((uintptr_t)d_avg_emb & 15) == 0 && ((uintptr_t)d_add_emb & 15) == 0, PNB_ERR_INVALID,
                "pnb_probe_select: embedding buffers must be 16-byte aligned");
    const size_t n = (size_t)H * W;
    ProbeSelectLayout L = carve_select(ws, n);
    PNB_REQUIRE(L.bytes <= ws_bytes, PNB_ERR_WORKSPACE, "pnb_probe_select: workspace %zu < required %zu", ws_bytes, L.bytes);
    ProbeSelectParams p;
    p.H = H; p.W = W; p.ray_mask = d_ray_mask; p.present = d_present; p.gt = d_gt; p.color = d_color; p.far_dist = d_far_dist;
    p.op_max = d_op_max; p.loc = d_loc; p.emb = d_avg_emb; p.avg_color = d_avg_color; p.avg_dir = d_avg_dir; p.avg_conf = d_avg_conf;
    for (int i = 0; i < 3; ++i) p.bg[i] = bg_color[i];
    p.opacity_thresh = opacity_thresh; p.far_thresh = far_thresh;
    p.flags = L.flags; p.offs = L.offs; p.cap = cap;
    p.add_xyz = d_add_xyz; p.add_emb = d_add_emb; p.add_color = d_add_color; p.add_dir = d_add_dir; p.add_conf = d_add_conf;
    p.count = d_count;
    const unsigned nb = (unsigned)((n + 255) / 256);
    k_probe_mark<<<nb, 256, 0, stream>>>(p);
    PNB_CHECK_CUDA(cudaGetLastError());
    int rc = exclusive_scan_u32(L.flags, 2, L.offs, (uint32_t)n, L.scan_tmp, stream);
    if (rc) return rc;
    k_probe_compact<<<nb, 256, 0, stream>>>(p);
    PNB_CHECK_CUDA(cudaGetLastError());
    return PNB_OK;
}
