// Ray march + first-SR sample selection + layered voxel K-NN, sample-compacted.
//
// Replaces (per call):
//   near_far_linear_ray_generation  /root/reference/models/rendering/diff_ray_marching.py:349-392
//        (raypos [1,R,400,3] is never materialised; positions are campos + raydir*t[d] in-kernel)
//   mask_raypos                     /root/reference/models/neural_points/cuda/query_worldcoords.cu:165-189
//   host glue (cumsum / first SR)   :381-391
//   get_shadingloc                  :192-214
//   query_neigh_along_ray_layered   :217-302
//   host glue (ray drop)            :425-429
// The integer decisions follow the canonical serial semantics of SURVEY.md 8(a) bit for bit: voxel index by
// IEEE sub+div+floor, distance fmaf(dz,dz,fmaf(dx,dx,dy*dy)), traversal x-major then y, z, list order,
// replace-farthest K buffer with strict '<', shell early-out once K candidates were seen.
#include "common.cuh"

namespace pnb {

struct QueryParams {
    GridDev g;
    float campos[3];
    const float* raydir;
    const float* t;
    int t_ray_stride;
    int R, D, SR, K;
    int ks0;  // kernel_size[0]
    float r2;
    int cap;
};

// First index d of the non-decreasing row tr[0, D) with tr[d] >= v (LE = false) or tr[d] > v (LE = true); D if there is none.
// Warp-cooperative: every round probes 32 evenly spaced entries and keeps the gap where the predicate turns (2 rounds for D = 400).
template <bool LE>
__device__ __forceinline__ int warp_search(const float* tr, int D, float v, int lane) {
    int lo = 0, hi = D;  // the answer lies in [lo, hi]; hi == D or tr[hi] passes
    while (lo < hi) {
        const int step = (hi - lo + 31) / 32;
        const int i = lo + lane * step;
        bool below = false;
        if (i < hi) {
            const float t = tr[i];
            below = LE ? !(t > v) : (t < v);
        }
        const int k = __popc(__ballot_sync(0xffffffffu, below));  // probes 0..k-1 fail, probe k (if any) passes
        if (k == 0) break;
        const int last = lo + (k - 1) * step;
        lo = last + 1;
        hi = min(hi, last + step);
    }
    return lo;
}

// One warp per ray: 32 march steps per iteration, ballot -> ordered slots.
//
// Only the steps that can land in the occupied box (PNB_GC_BOX_*, the bounding box of occ_bits) are marched.  A step hits only if
// its voxel floor(fdiv(fsub(p, lo), svs)) lies in the box, with p = fadd(c, fmul(d, t)).  Such a p lies within a few ulps of the
// box's world extent [lo + b0 * svs, lo + (b1 + 1) * svs], and c + d * t (exact) within a few more ulps of p.  The box is widened by
// one voxel on every side before the ray is clipped, so the clipped t-interval [t0, t1], computed in fp32 with errors of a few ulps
// of t, still holds every t that can hit as long as a voxel is far wider than those rounding errors (|d| ulp(t) + ulp(p) against
// svs: 1e-6 against 8e-3 for the shipped scenes).  The steps kept are those from the last one before t0 to the first one after t1,
// one more step on each side than the interval needs.  Every skipped step is outside the widened box, so it is at least one voxel
// away from any occupied voxel and its exact per-step test would fail: slots, counts and order are those of the full march.
// The same holds for the bounding sphere (PNB_GC_SPHERE_R2, about the grid centre): every point of an occupied voxel lies within
// its radius, which is widened by one voxel before the ray is clipped.  For a rounded object it removes most of the steps of the
// rays that cross the box's corners without meeting the object.  Setting the box and the radius to cover everything (tests) gives
// the full march.
__global__ void __launch_bounds__(256) k_march(QueryParams p, int* __restrict__ nsamp, uint16_t* __restrict__ steps) {
    int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (warp >= p.R) return;
    const int r = warp;
    const float dx = p.raydir[3 * r], dy = p.raydir[3 * r + 1], dz = p.raydir[3 * r + 2];
    const float* tr = p.t + (size_t)r * p.t_ray_stride;
    // clip the ray to the widened box
    const float c3[3] = {p.campos[0], p.campos[1], p.campos[2]}, d3[3] = {dx, dy, dz};
    float t0 = -INFINITY, t1 = INFINITY;
    bool miss = false;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const int b0 = __ldg(&p.g.counters[PNB_GC_BOX_X0 + a]), b1 = __ldg(&p.g.counters[PNB_GC_BOX_X1 + a]);
        const float wlo = p.g.lo[a] + (float)(b0 - 1) * p.g.svs[a], whi = p.g.lo[a] + (float)(b1 + 2) * p.g.svs[a];
        miss |= b0 > b1;
        if (d3[a] != 0.f) {
            const float ta = (wlo - c3[a]) / d3[a], tb = (whi - c3[a]) / d3[a];
            t0 = fmaxf(t0, fminf(ta, tb));
            t1 = fminf(t1, fmaxf(ta, tb));
        } else {
            miss |= c3[a] < wlo || c3[a] > whi;
        }
    }
    // and to the bounding sphere, widened by one voxel; |d|^2 t^2 + 2 (d . oc) t + |oc|^2 - rad^2 = 0
    {
        float oc[3], a2 = 0.f, b = 0.f, k = 0.f, svs_max = 0.f;
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            oc[a] = c3[a] - grid_centre(p.g.lo[a], p.g.svs[a], p.g.dim[a]);
            a2 += d3[a] * d3[a]; b += d3[a] * oc[a]; k += oc[a] * oc[a];
            svs_max = fmaxf(svs_max, p.g.svs[a]);
        }
        const float rad = sqrtf(__int_as_float(__ldg(&p.g.counters[PNB_GC_SPHERE_R2]))) + svs_max;
        const float disc = b * b - a2 * (k - rad * rad);
        if (disc >= 0.f && a2 > 0.f) {
            const float sq = sqrtf(disc);
            t0 = fmaxf(t0, (-b - sq) / a2);
            t1 = fminf(t1, (-b + sq) / a2);
        } else {
            miss = true;
        }
    }
    miss |= !(t0 <= t1);
    int count = 0;
    if (!miss) {
        const int first = max(warp_search<false>(tr, p.D, t0, lane) - 1, 0);   // first step with t >= t0, one step earlier
        const int end = min(warp_search<true>(tr, p.D, t1, lane) + 1, p.D);    // past the last step with t <= t1, one step later
        for (int base = first; base < end; base += 32) {
            int d = base + lane;
            bool hit = false;
            if (d < end) {
                float t = tr[d];
                int x = vox1(raypos1(p.campos[0], dx, t), p.g.lo[0], p.g.svs[0]);
                int y = vox1(raypos1(p.campos[1], dy, t), p.g.lo[1], p.g.svs[1]);
                int z = vox1(raypos1(p.campos[2], dz, t), p.g.lo[2], p.g.svs[2]);
                if (in_grid(x, y, z, p.g.dim)) {
                    uint32_t c = cell_index(x, y, z, p.g.dim);
                    hit = (__ldg(&p.g.occ_bits[c >> 5]) >> (c & 31)) & 1u;
                }
            }
            uint32_t m = __ballot_sync(0xffffffffu, hit);
            int slot = count + __popc(m & ((1u << lane) - 1u));
            if (hit && slot < p.SR) steps[(size_t)r * p.SR + slot] = (uint16_t)d;
            count += __popc(m);
            if (count >= p.SR) break;
        }
    }
    if (lane == 0) nsamp[r] = count < p.SR ? count : p.SR;
}

// candidates of ray r -> packed (ray, slot); one thread per ray
__global__ void __launch_bounds__(256) k_expand(int R, int cap, const int* __restrict__ nsamp, const uint32_t* __restrict__ samp_off,
                                                uint32_t* __restrict__ samp_ray, int* counters) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    bool first = false;
    if (r < R) {
        const int n = nsamp[r];
        const uint32_t off = samp_off[r];
        first = n > 0 && off < (uint32_t)cap;
        for (int j = 0; j < n; ++j) {
            if (off + j >= (uint32_t)cap) { counters[PNB_QC_OVERFLOW] = 1; break; }
            samp_ray[off + j] = ((uint32_t)r << 7) | (uint32_t)j;
        }
    }
    const uint32_t m = __ballot_sync(0xffffffffu, first);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(&counters[PNB_QC_R1], __popc(m));
}

// One thread per candidate sample: canonical layered K-NN.
__global__ void __launch_bounds__(128) k_knn(QueryParams p, const uint32_t* __restrict__ samp_off,
                                             const uint32_t* __restrict__ samp_ray, const uint16_t* __restrict__ steps,
                                             int* __restrict__ cand_pidx, uint8_t* __restrict__ samp_nvalid,
                                             uint8_t* __restrict__ ray_hit, int* counters) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t n_cand = min(samp_off[p.R], (uint32_t)p.cap);
    if (s >= n_cand) return;
    uint32_t pk = samp_ray[s];
    int r = (int)(pk >> 7), j = (int)(pk & 127u);
    int d = steps[(size_t)r * p.SR + j];
    float t = p.t[(size_t)r * p.t_ray_stride + d];
    const float cx = raypos1(p.campos[0], p.raydir[3 * r], t);
    const float cy = raypos1(p.campos[1], p.raydir[3 * r + 1], t);
    const float cz = raypos1(p.campos[2], p.raydir[3 * r + 2], t);
    const int fx = vox1(cx, p.g.lo[0], p.g.svs[0]);
    const int fy = vox1(cy, p.g.lo[1], p.g.svs[1]);
    const int fz = vox1(cz, p.g.lo[2], p.g.svs[2]);
    const int dead = p.g.parity_slot0 ? p.g.counters[PNB_GC_SLOT0_CELL] : -1;

    int idx[PNB_MAX_K];
    float buf[PNB_MAX_K];
#pragma unroll
    for (int m = 0; m < PNB_MAX_K; ++m) { idx[m] = -1; buf[m] = 0.f; }
    int kid = 0, far_ind = 0;
    float far2 = 0.f;
    const int nlayer = (p.ks0 + 1) / 2;
    for (int layer = 0; layer < nlayer; ++layer) {
        const int xa = max(-fx, -layer), xb = min(p.g.dim[0] - fx, layer + 1);
        const int ya = max(-fy, -layer), yb = min(p.g.dim[1] - fy, layer + 1);
        const int za = max(-fz, -layer), zb = min(p.g.dim[2] - fz, layer + 1);
        for (int x = xa; x < xb; ++x)
            for (int y = ya; y < yb; ++y) {
                // The shell cells of column (x, y) are consecutive in z, so they are looked up together: one or two pt_bits words
                // give their occupancy, one word_rank load their consecutive dense slots, and their cell_start entries share a line.
                // On the shell's rim every z of [za, zb) is visited, inside it only z = -layer and z = +layer.
                const bool rim = max(abs(x), abs(y)) == layer;
                for (int zc = za; zc < zb; zc += 32) {
                    const int n = min(zb - zc, 32);  // cells zc .. zc + n - 1
                    const uint32_t span = n == 32 ? 0xffffffffu : (1u << n) - 1u;
                    const uint32_t want = rim ? span : ((zc == -layer ? 1u : 0u) | (zc + n == layer + 1 ? 1u << (n - 1) : 0u));
                    if (!want) continue;
                    const uint32_t c0 = cell_index(fx + x, fy + y, fz + zc, p.g.dim);
                    const uint32_t wi = c0 >> 5, sh = c0 & 31u;
                    uint64_t W = __ldg(&p.g.pt_bits[wi]);
                    if (sh + (uint32_t)n > 32u) W |= (uint64_t)__ldg(&p.g.pt_bits[wi + 1]) << 32;  // the column straddles two words
                    const uint32_t occ = (uint32_t)(W >> sh) & span;                              // bit i: cell c0 + i holds points
                    uint32_t todo = occ & want;
                    if (!todo) continue;
                    // word_rank[wi + 1] = word_rank[wi] + popc(pt_bits[wi]): one rank serves both words
                    const uint32_t slot0 = __ldg(&p.g.word_rank[wi]) + __popcll(W & ((1ull << sh) - 1ull));
                    while (todo) {
                        const int i = __ffs(todo) - 1;
                        todo &= todo - 1u;
                        if ((int)(c0 + i) == dead) continue;  // query_worldcoords.cu:147 (slot 0 never filled)
                        const uint32_t slot = slot0 + __popc(occ & ((1u << i) - 1u));
                        uint32_t a = __ldg(&p.g.cell_start[slot]), b = __ldg(&p.g.cell_start[slot + 1]);
                        if (b - a > (uint32_t)p.g.P) b = a + (uint32_t)p.g.P;
                        for (uint32_t g = a; g < b; ++g) {
                            float4 q = __ldg(&p.g.spts[g]);
                            float xv = __fsub_rn(q.x, cx), yv = __fsub_rn(q.y, cy), zv = __fsub_rn(q.z, cz);
                            float d2 = __fmaf_rn(zv, zv, __fmaf_rn(xv, xv, __fmul_rn(yv, yv)));
                            if (p.r2 == 0.f || d2 <= p.r2) {
                                int pi = __float_as_int(q.w);
                                if (kid++ < p.K) {
                                    int slotk = kid - 1;
#pragma unroll
                                    for (int m = 0; m < PNB_MAX_K; ++m)
                                        if (m == slotk) { idx[m] = pi; buf[m] = d2; }
                                    if (d2 > far2) { far2 = d2; far_ind = slotk; }
                                } else if (d2 < far2) {
#pragma unroll
                                    for (int m = 0; m < PNB_MAX_K; ++m)
                                        if (m == far_ind) { idx[m] = pi; buf[m] = d2; }
                                    far2 = d2;
#pragma unroll
                                    for (int m = 0; m < PNB_MAX_K; ++m)
                                        if (m < p.K && buf[m] > far2) { far2 = buf[m]; far_ind = m; }
                                }
                            }
                        }
                    }
                }
            }
        if (kid >= p.K) break;
    }
    int nv = kid < p.K ? kid : p.K;
#pragma unroll
    for (int m = 0; m < PNB_MAX_K; ++m)
        if (m < p.K) cand_pidx[(size_t)s * p.K + m] = idx[m];
    samp_nvalid[s] = (uint8_t)nv;
    if (nv > 0) {
        ray_hit[r] = 1;
        atomicAdd(&counters[PNB_QC_N_PAIRS], nv);
    }
}

__global__ void __launch_bounds__(256) k_valid_list(int R, int cap, const uint32_t* __restrict__ samp_off,
                                                    const uint8_t* __restrict__ samp_nvalid,
                                                    const uint32_t* __restrict__ valid_rank, uint32_t* __restrict__ valid_list,
                                                    int* counters) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t n_cand = min(samp_off[R], (uint32_t)cap);
    if (s == 0) {
        counters[PNB_QC_N_CAND] = (int)n_cand;
        counters[PNB_QC_N_VALID] = (int)valid_rank[n_cand];
    }
    if (s >= n_cand) return;
    if (samp_nvalid[s] > 0) valid_list[valid_rank[s]] = s;
}

__global__ void __launch_bounds__(256) k_count_rays(int R, const uint8_t* __restrict__ ray_hit, int* counters) {
    int r = blockIdx.x * blockDim.x + threadIdx.x;
    int v = (r < R && ray_hit[r]) ? 1 : 0;
    uint32_t m = __ballot_sync(0xffffffffu, v);
    if ((threadIdx.x & 31) == 0 && m) atomicAdd(&counters[PNB_QC_R2], __popc(m));
}

// Dense reference layout: rows of rays with ray_hit, in ray order.
__global__ void __launch_bounds__(128) k_export(pnb_query_t q, float R00, float R10, float R20, float R01, float R11,
                                                float R21, float R02, float R12, float R22,
                                                const uint32_t* __restrict__ ray_rank, int32_t* __restrict__ ray_row,
                                                int8_t* __restrict__ ray_mask, int32_t* __restrict__ sample_pidx,
                                                float* __restrict__ sample_loc_w, float* __restrict__ sample_loc,
                                                float* __restrict__ sample_ray_dirs) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;  // (ray, slot)
    if (i >= q.R * q.SR) return;
    int r = i / q.SR, j = i - r * q.SR;
    bool hit = q.ray_hit[r] != 0;
    if (j == 0) { ray_mask[r] = hit ? 1 : 0; ray_row[r] = hit ? (int)ray_rank[r] : -1; }
    if (!hit) return;
    size_t row = (size_t)ray_rank[r] * q.SR + j;
    float lx = 0.f, ly = 0.f, lz = 0.f;
    int n = q.nsamp[r];
    if (j < n) {
        uint32_t s = q.samp_off[r] + j;
        int d = q.steps[(size_t)r * q.SR + j];
        float t = q.t[(size_t)r * q.t_ray_stride + d];
        lx = raypos1(q.campos[0], q.raydir[3 * r], t);
        ly = raypos1(q.campos[1], q.raydir[3 * r + 1], t);
        lz = raypos1(q.campos[2], q.raydir[3 * r + 2], t);
        for (int k = 0; k < q.K; ++k) sample_pidx[row * q.K + k] = q.cand_pidx[(size_t)s * q.K + k];
    } else {
        for (int k = 0; k < q.K; ++k) sample_pidx[row * q.K + k] = -1;
    }
    sample_loc_w[row * 3] = lx; sample_loc_w[row * 3 + 1] = ly; sample_loc_w[row * 3 + 2] = lz;
    if (sample_loc) {  // point_query.py:101-108
        float sx = lx - q.campos[0], sy = ly - q.campos[1], sz = lz - q.campos[2];
        float xc = sx * R00 + sy * R10 + sz * R20;
        float yc = sx * R01 + sy * R11 + sz * R21;
        float zc = sx * R02 + sy * R12 + sz * R22;
        sample_loc[row * 3] = xc / zc; sample_loc[row * 3 + 1] = yc / zc; sample_loc[row * 3 + 2] = zc;
    }
    if (sample_ray_dirs) {
        sample_ray_dirs[row * 3] = q.raydir[3 * r];
        sample_ray_dirs[row * 3 + 1] = q.raydir[3 * r + 1];
        sample_ray_dirs[row * 3 + 2] = q.raydir[3 * r + 2];
    }
}

struct QueryLayout {
    int* nsamp;
    uint32_t* samp_off;
    uint16_t* steps;
    uint32_t* samp_ray;
    int* cand_pidx;
    uint8_t* samp_nvalid;
    uint32_t* valid_list;
    uint32_t* valid_rank;
    uint8_t* ray_hit;
    int* counters;
    uint32_t* scan_tmp;
    uint32_t* ray_rank;
    size_t bytes;
};

static QueryLayout carve_query(void* ws, size_t cap_bytes, int R, int SR, int K, int cap) {
    Carver c(ws, cap_bytes);
    QueryLayout L;
    size_t r = (size_t)(R > 0 ? R : 1), cs = (size_t)(cap > 0 ? cap : 1);
    L.counters = c.take<int>(16);
    L.nsamp = c.take<int>(r);
    L.samp_off = c.take<uint32_t>(r + 1);
    L.steps = c.take<uint16_t>(r * SR);
    L.samp_ray = c.take<uint32_t>(cs);
    L.cand_pidx = c.take<int>(cs * K);
    L.samp_nvalid = c.take<uint8_t>(cs);
    L.valid_list = c.take<uint32_t>(cs);
    L.valid_rank = c.take<uint32_t>(cs + 1);
    L.ray_hit = c.take<uint8_t>(r);
    L.ray_rank = c.take<uint32_t>(r + 1);
    L.scan_tmp = c.take<uint32_t>(scan_tmp_elems(cs > r ? cs : r));
    L.bytes = align_up(c.off);
    return L;
}

}  // namespace pnb

using namespace pnb;

static inline int default_cap(int R, int SR, int cap) { return cap > 0 ? cap : R * SR; }

extern "C" size_t pnb_query_bytes(int R, int SR, int K, int cap_samples) {
    return carve_query(nullptr, 0, R, SR, K, default_cap(R, SR, cap_samples)).bytes;
}

extern "C" int pnb_query(pnb_query_t* q, void* ws, size_t ws_bytes, const pnb_grid_t* grid, const float campos[3],
                         const float* d_raydir, int R, const float* d_t, int t_ray_stride, int D, int SR, int K,
                         float radius_limit, const int32_t kernel_size[3], int cap_samples, pnb_stream_t stream_,
                         int32_t* h_counters) {
    cudaStream_t stream = (cudaStream_t)stream_;
    PNB_REQUIRE(q && ws && grid && d_raydir && d_t, PNB_ERR_INVALID, "pnb_query: null argument");
    PNB_REQUIRE(R > 0 && R < (1 << 25), PNB_ERR_INVALID, "pnb_query: R=%d out of range [1, 2^25)", R);
    PNB_REQUIRE(K >= 1 && K <= PNB_MAX_K, PNB_ERR_UNSUPPORTED,
                "pnb_query: K=%d unsupported (reference kernel buffer is KN=8, query_worldcoords.cu:14)", K);
    PNB_REQUIRE(SR >= 1 && SR <= PNB_MAX_SR, PNB_ERR_UNSUPPORTED, "pnb_query: SR=%d unsupported (1..%d)", SR, PNB_MAX_SR);
    PNB_REQUIRE(D >= 1 && D <= 65535, PNB_ERR_UNSUPPORTED, "pnb_query: D=%d unsupported (1..65535)", D);
    PNB_REQUIRE(t_ray_stride == 0 || t_ray_stride >= D, PNB_ERR_INVALID, "pnb_query: bad t_ray_stride");
    PNB_REQUIRE((long long)R * SR < (1ll << 31), PNB_ERR_UNSUPPORTED, "pnb_query: R*SR too large");
    int cap = default_cap(R, SR, cap_samples);
    QueryLayout L = carve_query(ws, ws_bytes, R, SR, K, cap);
    PNB_REQUIRE(L.bytes <= ws_bytes, PNB_ERR_WORKSPACE, "pnb_query: workspace %zu < required %zu", ws_bytes, L.bytes);

    QueryParams p;
    p.g = to_dev(*grid);
    for (int i = 0; i < 3; ++i) p.campos[i] = campos[i];
    p.raydir = d_raydir; p.t = d_t; p.t_ray_stride = t_ray_stride;
    p.R = R; p.D = D; p.SR = SR; p.K = K; p.ks0 = kernel_size[0];
    p.r2 = radius_limit * radius_limit;  // query_worldcoords.cu:410
    p.cap = cap;

    PNB_CHECK_CUDA(cudaMemsetAsync(L.counters, 0, 16 * sizeof(int), stream));
    PNB_CHECK_CUDA(cudaMemsetAsync(L.ray_hit, 0, (size_t)R, stream));
    PNB_CHECK_CUDA(cudaMemsetAsync(L.samp_nvalid, 0, (size_t)cap, stream));  // tail beyond n_cand must scan as 0
    {
        long long threads = (long long)R * 32;
        k_march<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(p, L.nsamp, L.steps);
    }
    int rc;
    rc = exclusive_scan_u32(L.nsamp, 3, L.samp_off, (uint32_t)R, L.scan_tmp, stream);
    if (rc) return rc;
    k_expand<<<(R + 255) / 256, 256, 0, stream>>>(R, cap, L.nsamp, L.samp_off, L.samp_ray, L.counters);
    k_knn<<<(cap + 127) / 128, 128, 0, stream>>>(p, L.samp_off, L.samp_ray, L.steps, L.cand_pidx, L.samp_nvalid,
                                                  L.ray_hit, L.counters);
    PNB_CHECK_CUDA(cudaGetLastError());
    // valid-sample list (ascending candidate id)
    rc = exclusive_scan_u32(L.samp_nvalid, 2, L.valid_rank, (uint32_t)cap, L.scan_tmp, stream);
    if (rc) return rc;
    k_valid_list<<<(cap + 255) / 256, 256, 0, stream>>>(R, cap, L.samp_off, L.samp_nvalid, L.valid_rank, L.valid_list,
                                                         L.counters);
    k_count_rays<<<(R + 255) / 256, 256, 0, stream>>>(R, L.ray_hit, L.counters);
    PNB_CHECK_CUDA(cudaGetLastError());

    q->R = R; q->SR = SR; q->K = K; q->D = D; q->cap_samples = cap;
    q->nsamp = L.nsamp; q->samp_off = L.samp_off; q->steps = L.steps; q->samp_ray = L.samp_ray;
    q->cand_pidx = L.cand_pidx; q->samp_nvalid = L.samp_nvalid; q->valid_list = L.valid_list;
    q->valid_rank = L.valid_rank; q->ray_hit = L.ray_hit; q->counters = L.counters;
    q->ray_rank = L.ray_rank; q->scan_tmp = L.scan_tmp;
    q->raydir = d_raydir; q->t = d_t; q->t_ray_stride = t_ray_stride;
    for (int i = 0; i < 3; ++i) q->campos[i] = campos[i];
    if (h_counters) {
        PNB_CHECK_CUDA(cudaMemcpyAsync(h_counters, L.counters, 16 * sizeof(int), cudaMemcpyDeviceToHost, stream));
        PNB_CHECK_CUDA(cudaStreamSynchronize(stream));
    }
    return PNB_OK;
}

extern "C" int pnb_query_export(const pnb_query_t* q, const pnb_shade_opts_t* cam, int32_t* d_ray_row, int8_t* d_ray_mask,
                                int32_t* d_sample_pidx, float* d_sample_loc_w, float* d_sample_loc,
                                float* d_sample_ray_dirs, pnb_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    PNB_REQUIRE(q && cam && d_ray_row && d_ray_mask && d_sample_pidx && d_sample_loc_w, PNB_ERR_INVALID,
                "pnb_query_export: null argument");
    int rc = exclusive_scan_u32(q->ray_hit, 2, q->ray_rank, (uint32_t)q->R, q->scan_tmp, stream);
    if (rc) return rc;
    const float* M = cam->camrotc2w;
    k_export<<<(q->R * q->SR + 127) / 128, 128, 0, stream>>>(*q, M[0], M[3], M[6], M[1], M[4], M[7], M[2], M[5], M[8],
                                                              q->ray_rank, d_ray_row, d_ray_mask, d_sample_pidx,
                                                              d_sample_loc_w, d_sample_loc, d_sample_ray_dirs);
    PNB_CHECK_CUDA(cudaGetLastError());
    return PNB_OK;
}
