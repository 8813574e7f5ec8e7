// Shared device/host helpers of libpnb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/pnb200.h"

namespace pnb {

void set_error(const char* fmt, ...);

#define PNB_CHECK_CUDA(expr)                                                              \
    do {                                                                                  \
        cudaError_t _e = (expr);                                                          \
        if (_e != cudaSuccess) {                                                          \
            pnb::set_error("%s:%d CUDA error %s: %s", __FILE__, __LINE__, #expr,          \
                           cudaGetErrorString(_e));                                       \
            return PNB_ERR_CUDA;                                                          \
        }                                                                                 \
    } while (0)

#define PNB_REQUIRE(cond, code, ...)                                                      \
    do {                                                                                  \
        if (!(cond)) {                                                                    \
            pnb::set_error(__VA_ARGS__);                                                  \
            return code;                                                                  \
        }                                                                                 \
    } while (0)

static inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

// Bump allocator over a caller-provided workspace.
struct Carver {
    char* base;
    size_t off, cap;
    Carver(void* p, size_t bytes) : base((char*)p), off(0), cap(bytes) {}
    template <typename T>
    T* take(size_t n) {
        size_t o = align_up(off);
        off = o + n * sizeof(T);
        return (T*)(base ? base + o : nullptr);
    }
    bool ok() const { return off <= cap; }
};

// Grid parameters by value for kernels.
struct GridDev {
    float lo[3];
    float svs[3];
    int dim[3];
    int P;
    int parity_slot0;
    const uint32_t* occ_bits;
    const uint32_t* pt_bits;
    const uint32_t* word_rank;
    const uint32_t* cell_start;
    const float4* spts;
    const int* counters;
};

static inline GridDev to_dev(const pnb_grid_t& g) {
    GridDev d;
    for (int i = 0; i < 3; ++i) { d.lo[i] = g.lo[i]; d.svs[i] = g.svs[i]; d.dim[i] = g.dim[i]; }
    d.P = g.P; d.parity_slot0 = g.parity_slot0;
    d.occ_bits = g.occ_bits; d.pt_bits = g.pt_bits; d.word_rank = g.word_rank;
    d.cell_start = g.cell_start; d.spts = (const float4*)g.spts; d.counters = g.counters;
    return d;
}

#ifdef __CUDACC__
// Voxel coordinate exactly as query_worldcoords.cu:40-42: IEEE fp32 subtract, IEEE fp32 divide, floor.
__device__ __forceinline__ int vox1(float p, float lo, float svs) {
    return (int)floorf(__fdiv_rn(__fsub_rn(p, lo), svs));
}
// Sample position as the reference's torch ops form it (diff_ray_marching.py:386): mul, then add, no FMA.
__device__ __forceinline__ float raypos1(float c, float dir, float t) {
    return __fadd_rn(c, __fmul_rn(dir, t));
}
// Centre of the grid along axis a: the centre of the bounding sphere PNB_GC_SPHERE_R2.
__device__ __forceinline__ float grid_centre(float lo, float svs, int dim) { return lo + 0.5f * (float)dim * svs; }
__device__ __forceinline__ bool in_grid(int x, int y, int z, const int* dim) {
    return (x >= 0) & (x < dim[0]) & (y >= 0) & (y < dim[1]) & (z >= 0) & (z < dim[2]);
}
__device__ __forceinline__ uint32_t cell_index(int x, int y, int z, const int* dim) {
    return ((uint32_t)x * (uint32_t)dim[1] + (uint32_t)y) * (uint32_t)dim[2] + (uint32_t)z;
}
#endif

// Device-wide exclusive scan of uint32 (3 small kernels; build-time / per-call bookkeeping, not a hot loop).
// mode 0: in[i];  mode 1: popc(in[i]);  mode 2: (in_u8[i] > 0);  mode 3: in_i32[i]
int exclusive_scan_u32(const void* in, int mode, uint32_t* out /* n+1 */, uint32_t n, uint32_t* tmp /* >= n/1024+2 */,
                       cudaStream_t stream);
static inline size_t scan_tmp_elems(size_t n) { return n / 1024 + 4; }

}  // namespace pnb
