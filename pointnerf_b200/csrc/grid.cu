// Voxel grid build: bitmask + rank + CSR of points sorted voxel-major (deterministic).
//
// Replaces, for the lifetime of one point-cloud version, what the reference rebuilds on every ray chunk:
//   claim_occ      /root/reference/models/neural_points/cuda/query_worldcoords.cu:18-78
//   map_coor2occ   :80-115
//   fill_occ2pnts  :117-162
// and the three dense int32 grids of :314-319.  Layout here (B200: everything the ray march touches is a
// 1-bit-per-voxel mask that stays in L2/L1; points of one voxel are contiguous 16-byte records):
//   occ_bits   dilated occupancy, the reference's coor_occ
//   pt_bits    voxels holding points; slot(cell) = word_rank[cell>>5] + popc(pt_bits[cell>>5] & below)
//   cell_start CSR offsets; spts[] = (x,y,z,index) ordered by (voxel, ascending point index)
// Canonical semantics (SURVEY 8a Q1-Q3): ascending index inside a voxel == the serial order of
// fill_occ2pnts; first P by index are kept; the voxel of the lowest-index in-range point ("slot 0") holds
// no points when parity_slot0 is set (query_worldcoords.cu:147 tests voxel_idx > 0).
#include <stdarg.h>

#include "common.cuh"

namespace pnb {

static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

// ------------------------------------------------------------------------------------------ scan
__device__ __forceinline__ uint32_t scan_load(const void* in, int mode, uint32_t i) {
    if (mode == 0) return ((const uint32_t*)in)[i];
    if (mode == 1) return __popc(((const uint32_t*)in)[i]);
    if (mode == 2) return ((const uint8_t*)in)[i] > 0 ? 1u : 0u;
    return (uint32_t)((const int*)in)[i];
}

__global__ void __launch_bounds__(256) k_scan_partial(const void* in, int mode, uint32_t n, uint32_t* bsum) {
    __shared__ uint32_t red[8];
    uint32_t base = blockIdx.x * 1024u, s = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        uint32_t i = base + threadIdx.x * 4 + j;
        if (i < n) s += scan_load(in, mode, i);
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = 0;
        for (int w = 0; w < 8; ++w) t += red[w];
        bsum[blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(1024) k_scan_bsum(uint32_t* bsum, uint32_t nb) {
    // single block, serial over chunks of 1024 block sums
    __shared__ uint32_t sh[1024];
    __shared__ uint32_t carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < nb; base += 1024) {
        uint32_t i = base + threadIdx.x;
        uint32_t v = i < nb ? bsum[i] : 0;
        sh[threadIdx.x] = v;
        __syncthreads();
        for (int o = 1; o < 1024; o <<= 1) {
            uint32_t a = threadIdx.x >= o ? sh[threadIdx.x - o] : 0;
            __syncthreads();
            sh[threadIdx.x] += a;
            __syncthreads();
        }
        uint32_t incl = sh[threadIdx.x], c = carry;
        __syncthreads();
        if (i < nb) bsum[i] = c + incl - v;  // exclusive
        if (threadIdx.x == 1023) carry = c + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) bsum[nb] = carry;  // total
}

__global__ void __launch_bounds__(256) k_scan_final(const void* in, int mode, uint32_t n, const uint32_t* bsum,
                                                    uint32_t* out) {
    __shared__ uint32_t wsum[8];
    uint32_t base = blockIdx.x * 1024u;
    uint32_t v[4], s = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        uint32_t i = base + threadIdx.x * 4 + j;
        v[j] = i < n ? scan_load(in, mode, i) : 0;
        s += v[j];
    }
    uint32_t incl = s;
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t a = __shfl_up_sync(0xffffffffu, incl, o);
        if ((threadIdx.x & 31) >= o) incl += a;
    }
    if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = incl;
    __syncthreads();
    uint32_t woff = 0;
    for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) woff += wsum[w];
    uint32_t run = bsum[blockIdx.x] + woff + incl - s;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        uint32_t i = base + threadIdx.x * 4 + j;
        if (i < n) out[i] = run;
        run += v[j];
    }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) out[n] = bsum[gridDim.x];
}

int exclusive_scan_u32(const void* in, int mode, uint32_t* out, uint32_t n, uint32_t* tmp, cudaStream_t stream) {
    uint32_t nb = (n + 1023) / 1024;
    if (nb == 0) {
        PNB_CHECK_CUDA(cudaMemsetAsync(out, 0, sizeof(uint32_t), stream));
        return PNB_OK;
    }
    k_scan_partial<<<nb, 256, 0, stream>>>(in, mode, n, tmp);
    k_scan_bsum<<<1, 1024, 0, stream>>>(tmp, nb);
    k_scan_final<<<nb, 256, 0, stream>>>(in, mode, n, tmp, out);
    PNB_CHECK_CUDA(cudaGetLastError());
    return PNB_OK;
}

// ------------------------------------------------------------------------------------------ grid kernels
struct BuildParams {
    float lo[3], svs[3];
    int dim[3], qs[3];
    int N, P, max_o;
};

// pass 1: voxel of every point -> pt_cell[i] (0xffffffff = outside), set pt_bits, track lowest in-range index.
__global__ void __launch_bounds__(256) k_mark(const float* __restrict__ xyz, BuildParams p, uint32_t* pt_bits,
                                              uint32_t* pt_cell, int* counters) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.N) return;
    int x = vox1(xyz[3 * i], p.lo[0], p.svs[0]);
    int y = vox1(xyz[3 * i + 1], p.lo[1], p.svs[1]);
    int z = vox1(xyz[3 * i + 2], p.lo[2], p.svs[2]);
    if (!in_grid(x, y, z, p.dim)) { pt_cell[i] = 0xffffffffu; return; }
    uint32_t c = cell_index(x, y, z, p.dim);
    pt_cell[i] = c;
    atomicOr(&pt_bits[c >> 5], 1u << (c & 31));
    atomicMin(&counters[PNB_GC_FIRST_PT], i);
    atomicAdd(&counters[PNB_GC_N_INRANGE], 1);
    // Squared distance from the grid centre to the farthest corner of the voxels that k_dilate marks around this point: the
    // farthest point of an axis-aligned box from a centre is the corner that is farthest along every axis.
    const int vv[3] = {x, y, z};
    float r2 = 0.f;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float ctr = grid_centre(p.lo[a], p.svs[a], p.dim[a]);
        const float e0 = p.lo[a] + (float)(vv[a] - p.qs[a] / 2) * p.svs[a], e1 = p.lo[a] + (float)(vv[a] + (p.qs[a] + 1) / 2) * p.svs[a];
        const float m = fmaxf(fabsf(e0 - ctr), fabsf(e1 - ctr));
        r2 += m * m;
    }
    // box of the voxels holding points (k_finish dilates it) and the sphere; reduced over the warp first, so that the counters see
    // one atomic per warp and value instead of one per point (r2 >= 0: its bits order as the floats do)
    const uint32_t act = __activemask();
    const int r2max = __reduce_max_sync(act, __float_as_int(r2));
    const int v[6] = {__reduce_min_sync(act, x), __reduce_min_sync(act, y), __reduce_min_sync(act, z),
                      __reduce_max_sync(act, x), __reduce_max_sync(act, y), __reduce_max_sync(act, z)};
    if ((threadIdx.x & 31) == __ffs(act) - 1) {
        for (int a = 0; a < 3; ++a) { atomicMin(&counters[PNB_GC_BOX_X0 + a], v[a]); atomicMax(&counters[PNB_GC_BOX_X1 + a], v[3 + a]); }
        atomicMax(&counters[PNB_GC_SPHERE_R2], r2max);
    }
}

// pass 2: cell -> slot, count points per slot.
__global__ void __launch_bounds__(256) k_count(BuildParams p, const uint32_t* __restrict__ pt_bits,
                                               const uint32_t* __restrict__ word_rank, uint32_t* pt_cell,
                                               uint32_t* cell_cnt, int* counters) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.N) return;
    uint32_t c = pt_cell[i];
    if (c == 0xffffffffu) return;
    uint32_t w = pt_bits[c >> 5];
    uint32_t slot = word_rank[c >> 5] + __popc(w & ((1u << (c & 31)) - 1u));
    pt_cell[i] = slot;
    atomicAdd(&cell_cnt[slot], 1u);
    if (i == counters[PNB_GC_FIRST_PT]) counters[PNB_GC_SLOT0_CELL] = (int)c;
}

// pass 3: scatter into CSR (order inside a voxel fixed by k_sort_cells).
__global__ void __launch_bounds__(256) k_scatter(const float* __restrict__ xyz, BuildParams p,
                                                 const uint32_t* __restrict__ pt_cell,
                                                 const uint32_t* __restrict__ cell_start, uint32_t* cell_fill,
                                                 float4* spts) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= p.N) return;
    uint32_t slot = pt_cell[i];
    if (slot == 0xffffffffu) return;
    uint32_t pos = cell_start[slot] + atomicAdd(&cell_fill[slot], 1u);
    spts[pos] = make_float4(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2], __int_as_float(i));
}

// pass 4: ascending point index inside every voxel (canonical serial order), statistics.
__global__ void __launch_bounds__(128) k_sort_cells(BuildParams p, uint32_t n_occ_cap,
                                                    const uint32_t* __restrict__ cell_start, float4* spts,
                                                    int* counters) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t n_occ = (uint32_t)counters[PNB_GC_N_OCC];
    if (s >= n_occ || s >= n_occ_cap) return;
    uint32_t a = cell_start[s], b = cell_start[s + 1];
    for (uint32_t i = a + 1; i < b; ++i) {
        float4 v = spts[i];
        int key = __float_as_int(v.w);
        uint32_t j = i;
        while (j > a && __float_as_int(spts[j - 1].w) > key) { spts[j] = spts[j - 1]; --j; }
        spts[j] = v;
    }
    int cnt = (int)(b - a);
    atomicMax(&counters[PNB_GC_MAX_PTS], cnt);
    if (cnt > p.P) counters[PNB_GC_OVERFLOW_P] = 1;
}

// pass 5: dilate occupied voxels by query_size (map_coor2occ :105-112).
__global__ void __launch_bounds__(256) k_dilate(BuildParams p, uint32_t n_words, const uint32_t* __restrict__ pt_bits,
                                                uint32_t* occ_bits) {
    uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= n_words) return;
    uint32_t bits = pt_bits[w];
    while (bits) {
        int b = __ffs(bits) - 1;
        bits &= bits - 1;
        uint32_t c = w * 32u + (uint32_t)b;
        int z = (int)(c % (uint32_t)p.dim[2]);
        uint32_t t = c / (uint32_t)p.dim[2];
        int y = (int)(t % (uint32_t)p.dim[1]);
        int x = (int)(t / (uint32_t)p.dim[1]);
        int x0 = max(0, x - p.qs[0] / 2), x1 = min(p.dim[0], x + (p.qs[0] + 1) / 2);
        int y0 = max(0, y - p.qs[1] / 2), y1 = min(p.dim[1], y + (p.qs[1] + 1) / 2);
        int z0 = max(0, z - p.qs[2] / 2), z1 = min(p.dim[2], z + (p.qs[2] + 1) / 2);
        for (int xx = x0; xx < x1; ++xx)
            for (int yy = y0; yy < y1; ++yy)
                for (int zz = z0; zz < z1; ++zz) {
                    uint32_t cc = cell_index(xx, yy, zz, p.dim);
                    uint32_t m = 1u << (cc & 31);
                    if (!(occ_bits[cc >> 5] & m)) atomicOr(&occ_bits[cc >> 5], m);
                }
    }
}

__global__ void k_finish(BuildParams p, const uint32_t* word_rank, uint32_t n_words, int max_o, int* counters) {
    int n_occ = (int)word_rank[n_words];
    counters[PNB_GC_N_OCC] = n_occ;
    if (n_occ > max_o) counters[PNB_GC_OVERFLOW_O] = 1;
    // the point box grown by k_dilate's window: [c - qs/2, c + (qs+1)/2) clipped to the grid (an empty box stays empty)
    if (n_occ > 0) {
        for (int a = 0; a < 3; ++a) {
            counters[PNB_GC_BOX_X0 + a] = max(0, counters[PNB_GC_BOX_X0 + a] - p.qs[a] / 2);
            counters[PNB_GC_BOX_X1 + a] = min(p.dim[a] - 1, counters[PNB_GC_BOX_X1 + a] + (p.qs[a] + 1) / 2 - 1);
        }
    }
}

struct GridLayout {
    uint32_t *occ_bits, *pt_bits, *word_rank, *cell_start, *pt_cell, *cell_fill, *scan_tmp;
    float4* spts;
    int* counters;
    size_t bytes;
};

static GridLayout carve_grid(void* buf, size_t cap, int N, const int32_t dim[3]) {
    Carver c(buf, cap);
    GridLayout L;
    size_t vol = (size_t)dim[0] * dim[1] * dim[2];
    size_t nw = (vol + 31) / 32;
    size_t nn = (size_t)(N > 0 ? N : 1);
    L.counters = c.take<int>(16);
    L.occ_bits = c.take<uint32_t>(nw);
    L.pt_bits = c.take<uint32_t>(nw);
    L.word_rank = c.take<uint32_t>(nw + 1);
    L.cell_start = c.take<uint32_t>(nn + 1);
    L.spts = c.take<float4>(nn);
    L.pt_cell = c.take<uint32_t>(nn);
    L.cell_fill = c.take<uint32_t>(nn + 1);
    L.scan_tmp = c.take<uint32_t>(scan_tmp_elems(nw > nn ? nw : nn));
    L.bytes = align_up(c.off);
    return L;
}

}  // namespace pnb

using namespace pnb;

extern "C" int pnb_version(void) { return 100; }
extern "C" const char* pnb_last_error(void) { return pnb::g_err; }
extern "C" size_t pnb_struct_size(int which) {
    switch (which) {
        case 0: return sizeof(pnb_grid_t);
        case 1: return sizeof(pnb_query_t);
        case 2: return sizeof(pnb_shade_opts_t);
        case 3: return sizeof(pnb_mlp_t);
        case 4: return sizeof(pnb_points_t);
        default: return 0;
    }
}

extern "C" size_t pnb_grid_bytes(int N, const int32_t dim[3]) { return carve_grid(nullptr, 0, N, dim).bytes; }

extern "C" int pnb_grid_build(pnb_grid_t* grid, void* buf, size_t buf_bytes, const float* d_xyz, int N,
                              const float lo[3], const float svs[3], const int32_t dim[3],
                              const int32_t query_size[3], int max_o, int P, int parity_slot0,
                              pnb_stream_t stream_, int32_t* h_counters) {
    cudaStream_t stream = (cudaStream_t)stream_;
    PNB_REQUIRE(grid && buf && d_xyz, PNB_ERR_INVALID, "pnb_grid_build: null argument");
    PNB_REQUIRE(N > 0, PNB_ERR_INVALID, "pnb_grid_build: N must be > 0 (got %d)", N);
    PNB_REQUIRE(dim[0] > 0 && dim[1] > 0 && dim[2] > 0, PNB_ERR_INVALID, "pnb_grid_build: bad dim %d %d %d", dim[0],
                dim[1], dim[2]);
    double vol = (double)dim[0] * dim[1] * dim[2];
    PNB_REQUIRE(vol < 4.0e9, PNB_ERR_UNSUPPORTED, "pnb_grid_build: %g voxels exceed the 32-bit cell index", vol);
    PNB_REQUIRE(svs[0] > 0 && svs[1] > 0 && svs[2] > 0, PNB_ERR_INVALID, "pnb_grid_build: voxel size must be > 0");
    PNB_REQUIRE(P > 0, PNB_ERR_INVALID, "pnb_grid_build: P must be > 0");
    GridLayout L = carve_grid(buf, buf_bytes, N, dim);
    PNB_REQUIRE(L.bytes <= buf_bytes, PNB_ERR_WORKSPACE, "pnb_grid_build: buffer %zu < required %zu", buf_bytes, L.bytes);

    BuildParams p;
    for (int i = 0; i < 3; ++i) { p.lo[i] = lo[i]; p.svs[i] = svs[i]; p.dim[i] = dim[i]; p.qs[i] = query_size[i]; }
    p.N = N; p.P = P; p.max_o = max_o;
    uint32_t nw = (uint32_t)(((size_t)vol + 31) / 32);

    PNB_CHECK_CUDA(cudaMemsetAsync(L.counters, 0, 16 * sizeof(int), stream));
    PNB_CHECK_CUDA(cudaMemsetAsync(L.occ_bits, 0, nw * sizeof(uint32_t), stream));
    PNB_CHECK_CUDA(cudaMemsetAsync(L.pt_bits, 0, nw * sizeof(uint32_t), stream));
    PNB_CHECK_CUDA(cudaMemsetAsync(L.cell_start, 0, ((size_t)N + 1) * sizeof(uint32_t), stream));
    PNB_CHECK_CUDA(cudaMemsetAsync(L.cell_fill, 0, ((size_t)N + 1) * sizeof(uint32_t), stream));
    int init[16];
    for (int i = 0; i < 16; ++i) init[i] = 0;
    init[PNB_GC_FIRST_PT] = 0x7fffffff;
    init[PNB_GC_SLOT0_CELL] = -1;
    for (int a = 0; a < 3; ++a) { init[PNB_GC_BOX_X0 + a] = 0x7fffffff; init[PNB_GC_BOX_X1 + a] = -1; }
    PNB_CHECK_CUDA(cudaMemcpyAsync(L.counters, init, sizeof(init), cudaMemcpyHostToDevice, stream));

    int nbN = (N + 255) / 256;
    k_mark<<<nbN, 256, 0, stream>>>(d_xyz, p, L.pt_bits, L.pt_cell, L.counters);
    int rc = exclusive_scan_u32(L.pt_bits, 1, L.word_rank, nw, L.scan_tmp, stream);
    if (rc) return rc;
    k_finish<<<1, 1, 0, stream>>>(p, L.word_rank, nw, max_o, L.counters);
    // cell_cnt is accumulated in cell_fill, scanned into cell_start, then cell_fill is re-zeroed as cursor
    k_count<<<nbN, 256, 0, stream>>>(p, L.pt_bits, L.word_rank, L.pt_cell, L.cell_fill, L.counters);
    rc = exclusive_scan_u32(L.cell_fill, 0, L.cell_start, (uint32_t)N, L.scan_tmp, stream);
    if (rc) return rc;
    PNB_CHECK_CUDA(cudaMemsetAsync(L.cell_fill, 0, ((size_t)N + 1) * sizeof(uint32_t), stream));
    k_scatter<<<nbN, 256, 0, stream>>>(d_xyz, p, L.pt_cell, L.cell_start, L.cell_fill, L.spts);
    k_sort_cells<<<(N + 127) / 128, 128, 0, stream>>>(p, (uint32_t)N, L.cell_start, L.spts, L.counters);
    k_dilate<<<(nw + 255) / 256, 256, 0, stream>>>(p, nw, L.pt_bits, L.occ_bits);
    PNB_CHECK_CUDA(cudaGetLastError());

    for (int i = 0; i < 3; ++i) { grid->lo[i] = lo[i]; grid->svs[i] = svs[i]; grid->dim[i] = dim[i]; }
    grid->P = P; grid->parity_slot0 = parity_slot0; grid->n_points = N; grid->n_words = nw;
    grid->occ_bits = L.occ_bits; grid->pt_bits = L.pt_bits; grid->word_rank = L.word_rank;
    grid->cell_start = L.cell_start; grid->spts = (float*)L.spts; grid->counters = L.counters;
    if (h_counters) {
        PNB_CHECK_CUDA(cudaMemcpyAsync(h_counters, L.counters, 16 * sizeof(int), cudaMemcpyDeviceToHost, stream));
        PNB_CHECK_CUDA(cudaStreamSynchronize(stream));
    }
    return PNB_OK;
}
