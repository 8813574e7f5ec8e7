// Fused per-pair shading on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a.
//
//   gather + weights + positional encoding  ->  block1 (284->256->256)  ->  cat extras  ->  block3 (263->256->256)
//   ->  alpha branch + K-reduction  ->  colour branch (280->128->128->128->3)
//   (reference: /root/reference/models/aggregators/point_aggregators.py:488-644, 727-814; gather
//   /root/reference/models/neural_points/neural_points.py:706-717)
//
// Kernels of this file (one persistent CTA per SM each):
//   k_pack_*      row packing: the valid (sample, neighbour) pairs -> 32-row quadrants of 128-row MMA tiles (first fit)
//   k_shade_tc7   pair MLPs, every layer D[128x256] = A[128xK] * W[256xK]^T on tcgen05.mma (kind::f16, BF16 operands, FP32
//                 accumulate in TMEM), TMEM role ping-pong between layers, K-reduction, writes h-bar + sigma
//   k_shade_tc8   the same for a FROZEN point cloud (render): the 224 point-only inputs of block1.0 are hoisted into a
//                 per-point table (k_point_pre), layer 1 runs on the 64 sample-dependent inputs only
//   k_color_tc2   colour branch per 128 valid samples, fed by h-bar in its own operand format (one bulk copy per tile)
// The reference computes these layers in fp32 (cuBLAS SGEMM, TF32 off) and the parity bar is 1e-4 on the rendered
// radiance, which a single BF16/TF32 pass misses (SURVEY.md section 7) -> error-compensated split:
//   A = A_hi + A_lo, W = W_hi + W_lo (bf16 each);   D = A_hi*W_hi + A_lo*W_hi + A_hi*W_lo    (3 MMAs per k-step)
// Weight images are pre-packed in the UMMA operand layout (pnb_mlp_pack) and streamed L2 -> shared memory with cp.async.bulk
// (TMA engine) through an mbarrier ring.  Earlier pipeline generations (v2 serialized, v3 TS form, v5 unpacked rows, v6 CTA
// pairs / cta_group::2, CUDA-core colour branch) were removed in round 2; their measurements stay in profiles/r01_* and DESIGN.md.
#include "common.cuh"
#include "umma.cuh"
#include <type_traits>

namespace pnb {
using namespace umma;

namespace tc {
constexpr int LAYOUT = LAYOUT_NONE;
constexpr int TM = 128;                 // pair rows per tile
constexpr int IMG = 256 * 64;           // bytes of one weight image ([256 x 32] bf16)
constexpr int ABLK = 128 * 64;          // bytes of one A block ([128 x 32] bf16)
constexpr int NKB_MAX = 9;
__host__ __device__ constexpr int nkb_of(int l) { return (l == 0 || l == 2) ? 9 : 8; }
__host__ __device__ constexpr int img_base(int l) { return l == 0 ? 0 : l == 1 ? 9 : l == 2 ? 17 : 26; }  // in blocks
constexpr int NBLK_TOTAL = 34;
constexpr int IMGS_PER_TILE = 2 * NBLK_TOTAL;
constexpr float LEAKY = 0.01f;
constexpr int XE = 128 * 32;            // bytes of one [128 x 16] bf16 extras operand (LBO = 128, SBO = 256)
__device__ __forceinline__ uint32_t xe_offset(int r, int k) { return (uint32_t)((r >> 3) * 256 + (k >> 3) * 128 + (r & 7) * 16 + (k & 7) * 2); }
}  // namespace tc

struct ShadeTcParams {
    pnb_query_t q;
    pnb_points_t pts;
    pnb_shade_opts_t o;
    const unsigned char* wimg;   // packed weight images (N = 256 per image)
    const float* bias[4];
    const float* wa;             // alpha_branch.0 weight [256]
    const float* ba;             // alpha_branch.0 bias [1]
    float* hbar;                 // [n_valid][256]
    float* sigma;                // [n_valid]
    int hbar_cap;
    int* err;
    int dbg_no_weights;          // timing experiment only: the loader signals the ring without copying (results are garbage)
    int dbg_flags;               // bit 0: cycle accounting of block 0; bit 2: per-CTA cycles; bit 3: v8 non-deferred last epilogue;
                                 // bit 4: v8 static tile schedule instead of the tile queue
    const unsigned char* vcnt;   // v7 row packing: neighbours per PACKED position [n_valid] (vcntp of k_pack_quads)
    const uint32_t* vorder;      // v7: valid-sample index of every packed position [n_valid]
    const uint32_t* quad_first;  // v7: first valid sample of every 32-row quadrant [n_quads + 1]
    const int* pack_cnt;         // v7: [0] = n_quads
    const float* pre;            // v8: per-point hoisted layer-1 pre-activation [N][256] (k_point_pre)
    int hbar_fmt;                // 0: hbar[n_valid][256] fp32;  1: bf16 hi/lo A-operand blocks of k_color_tc2 (per 128 samples: 8 K blocks x {hi,lo} x [128x32])
    int* tile_ctr;               // v8: tile queue, next 128-row tile to hand out (= pack_cnt + 1, zeroed by k_pack_scan)
};
__device__ __forceinline__ void prof_add(const ShadeTcParams& p, int slot, long long cyc) {
    if ((p.dbg_flags & 1) && blockIdx.x == 0) atomicAdd(reinterpret_cast<unsigned long long*>(p.err) + 1 + slot, (unsigned long long)cyc);
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

__device__ __forceinline__ void rot3t(const float* M, float x, float y, float z, float& ox, float& oy, float& oz) {
    ox = x * M[0] + y * M[1] + z * M[2];
    oy = x * M[3] + y * M[4] + z * M[5];
    oz = x * M[6] + y * M[7] + z * M[8];
}
__device__ __forceinline__ void w2pers_t(const pnb_shade_opts_t& o, float px, float py, float pz, float& xp, float& yp, float& zp) {
    float sx = px - o.campos[0], sy = py - o.campos[1], sz = pz - o.campos[2];
    const float* M = o.camrotc2w;
    float xc = sx * M[0] + sy * M[3] + sz * M[6];
    float yc = sx * M[1] + sy * M[4] + sz * M[7];
    float zc = sx * M[2] + sy * M[5] + sz * M[8];
    xp = xc / zc; yp = yc / zc; zp = zc;
}

// sin/cos of x*2^j, j = 0..NF-1: one accurate sincosf + angle doubling (abs error < 1e-6 after 4 doublings; the
// fp32 kernel keeps NF independent sincosf calls).  out[2j] = sin, out[2j+1] = cos  (networks.py:175-190 layout).
template <int NF>
__device__ __forceinline__ void pe_doubling(float x, float* out) {
    float s, c;
    sincosf(x, &s, &c);
    out[0] = s; out[1] = c;
#pragma unroll
    for (int j = 1; j < NF; ++j) {
        float s2 = 2.0f * s * c, c2 = fmaf(c, c, -s * s);
        s = s2; c = c2;
        out[2 * j] = s; out[2 * j + 1] = c;
    }
}

template <class SmemT>
__device__ __forceinline__ void store_chunk8_a1(SmemT& sm, int r, int kb, int k8, const float* v) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) split_bf16x2(v[2 * i], v[2 * i + 1], h[i], l[i]);
    uint32_t off = (uint32_t)kb * tc::ABLK + tile_offset_bytes<tc::LAYOUT>(r, k8);
    *reinterpret_cast<uint4*>(sm.a_hi + off) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(sm.a_lo + off) = make_uint4(l[0], l[1], l[2], l[3]);
}

// One pair row of the block1 operand (gather, distance weights, PE by angle doubling, hi/lo split -> shared memory),
// its block3 extras operand and its weight*conf factor.  PART 2: the whole row (v3 / v5: one builder thread per row);
// PART 0 / 1: the two halves of a row for the v6 pipeline (two builder threads per row):
//   part 0 = operand columns 0..151   (raw features, PE of features 0..19)
//   part 1 = operand columns 152..287 (PE of features 20..31, PE of the 6 distances), extras operand, weight*conf
// Sum of v over the lanes st .. st+cnt-1 of the warp (cnt <= 8; every lane calls it, lanes outside any segment pass st = lane,
// cnt = 1).  The order of the additions depends on cnt only, not on where the segment sits in the warp.
__device__ __forceinline__ float seg_scan8(float v, int lane, int st) {          // inclusive scan within the segment
#pragma unroll
    for (int d = 1; d <= 4; d <<= 1) {
        const float tv = __shfl_up_sync(0xffffffffu, v, d);
        if (lane - d >= st) v += tv;
    }
    return v;
}
__device__ __forceinline__ float seg_sum8(float v, int lane, int st, int cnt) {
    return __shfl_sync(0xffffffffu, seg_scan8(v, lane, st), st + cnt - 1);
}

// PACKED = false: row = 8 * (sample in tile) + neighbour slot, 16 samples per tile (rows of empty slots are zero).
// PACKED = true (v7): the caller has packed only the valid (sample, neighbour) pairs into the rows: row `row` is neighbour `pk` of
// valid sample `pvi` (pvi < 0: unused row), and the rows of that sample are lanes pst .. pst+pcnt-1 of this warp.
template <int PART, bool PACKED = false, class SmemT>
__device__ __forceinline__ void build_pair_part(SmemT& sm, const ShadeTcParams& p, int tile, int t, int row, int n_valid, int pvi = -1,
                                                int pk = 0, int pst = 0, int pcnt = 1) {
    using namespace tc;
    constexpr bool P0 = PART != 1, P1 = PART != 0;
    constexpr int G_LO = P0 ? 0 : 5, G_HI = P1 ? 8 : 5;      // feature groups (4 features each) whose PE this part builds
    const pnb_query_t& q = p.q;
    const int k = PACKED ? pk : (row & 7);
    const int vi = PACKED ? pvi : tile * (TM / PNB_MAX_K) + (row >> 3);
    int pidx = -1;
    float lx = 0.f, ly = 0.f, lz = 0.f, vx = 0.f, vy = 0.f, vz = 0.f;
    if (vi >= 0 && vi < n_valid) {
        uint32_t s = q.valid_list[vi];
        if (P1) {
            uint32_t pk = q.samp_ray[s];
            int r = (int)(pk >> 7), j = (int)(pk & 127u);
            int d = q.steps[(size_t)r * q.SR + j];
            float tt = q.t[(size_t)r * q.t_ray_stride + d];
            vx = q.raydir[3 * r]; vy = q.raydir[3 * r + 1]; vz = q.raydir[3 * r + 2];
            lx = raypos1(q.campos[0], vx, tt); ly = raypos1(q.campos[1], vy, tt); lz = raypos1(q.campos[2], vz, tt);
        }
        if (k < q.K) pidx = q.cand_pidx[(size_t)s * q.K + k];
    }
    const bool valid = pidx >= 0;
    const int pi = valid ? pidx : 0;
    float dist[6];
    float ovx = 0.f, ovy = 0.f, ovz = 0.f;
    if (P1) {
        rot3t(p.o.Rw2c, vx, vy, vz, ovx, ovy, ovz);
        float px = __ldg(&p.pts.xyz[3 * pi]), py = __ldg(&p.pts.xyz[3 * pi + 1]), pz = __ldg(&p.pts.xyz[3 * pi + 2]);
        dist[0] = px - lx; dist[1] = py - ly; dist[2] = pz - lz;
        float xpp, ypp, zpp, xsp, ysp, zsp;
        w2pers_t(p.o, px, py, pz, xpp, ypp, zpp);
        w2pers_t(p.o, lx, ly, lz, xsp, ysp, zsp);
        dist[3] = xpp * zpp - xsp * zsp; dist[4] = ypp * zpp - ysp * zsp; dist[5] = zpp - zsp;
        float nrm = sqrtf(dist[0] * dist[0] + dist[1] * dist[1] + dist[2] * dist[2]);
        float w = valid ? 1.0f / fmaxf(nrm, 1e-6f) : 0.f;
        float wsum = w;
        if (PACKED) {
            wsum = seg_sum8(w, row & 31, pst, pcnt);
        } else {                               // 8 consecutive lanes = the 8 rows of one sample
            wsum += __shfl_xor_sync(0xffffffffu, wsum, 1);
            wsum += __shfl_xor_sync(0xffffffffu, wsum, 2);
            wsum += __shfl_xor_sync(0xffffffffu, wsum, 4);
        }
        w = w / fmaxf(wsum, 1e-8f);
        float cf = __ldg(&p.pts.conf[pi]);
        sm.wc[t % SmemT::NWC][row] = valid ? w * fminf(fmaxf(cf, 1e-4f), 1.0f) : 0.f;
        float d0, d1, d2;
        rot3t(p.o.Rw2c, dist[0], dist[1], dist[2], d0, d1, d2);
        dist[0] = d0; dist[1] = d1; dist[2] = d2;
    }
    float ex[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (valid) {
        const float4* ep = (const float4*)&p.pts.emb[(size_t)pi * PNB_FEAT];
#pragma unroll
        for (int g = G_LO; g < G_HI; ++g) {    // 4 features per step
            float4 fv = __ldg(ep + g);
            float f[4] = {fv.x, fv.y, fv.z, fv.w};
            float pe[24];
#pragma unroll
            for (int e = 0; e < 4; ++e) pe_doubling<3>(f[e], pe + e * 6);
            const int col = 32 + 24 * g;
#pragma unroll
            for (int c = 0; c < 3; ++c) store_chunk8_a1(sm, row, (col + 8 * c) >> 5, (col + 8 * c) & 31, pe + 8 * c);
        }
        if (P0) {
#pragma unroll
            for (int g = 0; g < 4; ++g) {      // raw features, 8 per chunk (re-read: L1 hit)
                float4 a = __ldg(ep + 2 * g), b = __ldg(ep + 2 * g + 1);
                float f8[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
                store_chunk8_a1(sm, row, 0, 8 * g, f8);
            }
        }
        if (P1) {
            float dp[60];
#pragma unroll
            for (int e = 0; e < 6; ++e) pe_doubling<5>(dist[e], dp + 10 * e);
            float z4[8] = {dp[56], dp[57], dp[58], dp[59], 0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int c = 0; c < 7; ++c) store_chunk8_a1(sm, row, (224 + 8 * c) >> 5, (224 + 8 * c) & 31, dp + 8 * c);
            store_chunk8_a1(sm, row, 8, 24, z4);
            float ddx, ddy, ddz;
            rot3t(p.o.Rw2c, __ldg(&p.pts.dir[3 * pi]), __ldg(&p.pts.dir[3 * pi + 1]), __ldg(&p.pts.dir[3 * pi + 2]), ddx, ddy, ddz);
            ex[0] = __ldg(&p.pts.color[3 * pi]); ex[1] = __ldg(&p.pts.color[3 * pi + 1]); ex[2] = __ldg(&p.pts.color[3 * pi + 2]);
            ex[3] = ddx - ovx; ex[4] = ddy - ovy; ex[5] = ddz - ovz;
            ex[6] = ddx * ovx + ddy * ovy + ddz * ovz;
        }
    } else {
        float z8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        constexpr int C_LO = P0 ? 0 : 19, C_HI = P1 ? 36 : 19;   // 16-byte chunks: column / 8
        for (int c = C_LO; c < C_HI; ++c) store_chunk8_a1(sm, row, c >> 2, (c & 3) * 8, z8);
    }
    if (P1) {   // block3 extras operand [128 x 16]: chunk 0 = extras, chunk 1 = 0
        uint32_t h[4], l[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) split_bf16x2(ex[2 * i], ex[2 * i + 1], h[i], l[i]);
        uint32_t off = tc::xe_offset(row, 0);
        *reinterpret_cast<uint4*>(sm.xe_hi[t & 1] + off) = make_uint4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<uint4*>(sm.xe_lo[t & 1] + off) = make_uint4(l[0], l[1], l[2], l[3]);
        *reinterpret_cast<uint4*>(sm.xe_hi[t & 1] + off + 128) = make_uint4(0u, 0u, 0u, 0u);
        *reinterpret_cast<uint4*>(sm.xe_lo[t & 1] + off + 128) = make_uint4(0u, 0u, 0u, 0u);
    }
}
// ------------------------------------------------------------------------------------------ weight packing
// W^T fp32 [Kpad][256] (rows >= K are zero) -> per K-block: hi image then lo image, each [256 x 32] bf16 in the
// UMMA operand layout.
__global__ void __launch_bounds__(256) k_pack_weights(const float* __restrict__ wt, int Kpad, int nkb, int N, unsigned char* __restrict__ out,
                                                      int ldn = -1, int n_off = 0) {
    if (ldn < 0) ldn = N;
    int i = blockIdx.x * blockDim.x + threadIdx.x;   // (kb, n, k)
    if (i >= nkb * N * BK) return;
    int kb = i / (N * BK), rem = i - kb * N * BK;
    int n = rem / BK, k = rem - n * BK;
    int kg = kb * BK + k;
    float v = kg < Kpad ? wt[(size_t)kg * ldn + n_off + n] : 0.f;
    __nv_bfloat16 h, l;
    split_bf16(v, h, l);
    uint32_t off = tile_offset_bytes<tc::LAYOUT>(n, k);
    const size_t img = (size_t)N * 64;
    *(__nv_bfloat16*)(out + (size_t)(2 * kb) * img + off) = h;
    *(__nv_bfloat16*)(out + (size_t)(2 * kb + 1) * img + off) = l;
}

// =====================================================================================================================
// v7: v5 with PACKED ROWS.  v5 gives every valid sample 8 rows (one per neighbour slot) although only 75 % of the slots
// hold a neighbour on the lego frame (P_v / (8 S_v)): a quarter of every MMA multiplies zero rows.  Here a 128-row tile
// is four 32-row quadrants (= the TMEM lane quarter of one warp), and each quadrant holds whole samples packed back to
// back, only their valid neighbours (first-fit packing with a 64-sample look-ahead, k_pack_*: the packed order is the
// permutation `vorder`): 99.3 % of the rows carry a pair on the lego frame.
// The K-reduction over the rows of a sample (1..8 consecutive lanes, never crossing a quadrant) is a segmented
// warp-shuffle scan; its addition order depends on the neighbour count only, so a ray's colour is still independent of
// which rays share the call.  Two builder threads per row and the last epilogue shared between the epilogue and the
// builder warps (as v6); TMEM role ping-pong, chunk hand-off, weight ring and issuer are v5's.
namespace tc7 {
constexpr int NEPI_WARPS = 8, NGRP = NEPI_WARPS / 4, NCH = 16 / NGRP;
constexpr int NEPI = NEPI_WARPS * 32, NBUILD = 256, NTHR = NEPI + NBUILD + 64;     // two builder threads per row (as v6)
constexpr int NSTAGE = 4;
constexpr int PACK_S = 512;             // samples per independently packed super-chunk (its last quadrant may stay partly empty)
constexpr int PACK_WIN = 64;            // look-ahead of the first-fit packing
struct Smem {
    static constexpr int NWC = 2;          // reuse ordered through bar_alpha: the builders run their share of the last epilogue
    unsigned char a_hi[tc::NKB_MAX * tc::ABLK];
    unsigned char a_lo[tc::NKB_MAX * tc::ABLK];
    unsigned char b[NSTAGE][tc::IMG];
    unsigned char xe_hi[2][tc::XE];
    unsigned char xe_lo[2][tc::XE];
    float wc[NWC][tc::TM];
    float alpha_part[2][tc::TM];         // builder groups' partial alpha dot products
    float alpha_e[tc::TM];               // sum of the two epilogue groups' partials (two addends onto 0: order-independent)
    uint32_t qhead[NWC][4], qfirst[NWC][4], qtotal[NWC][4];   // per quadrant: bit r = row r starts a sample; first valid-sample index; rows used
    uint64_t bar_full[NSTAGE], bar_empty[NSTAGE], bar_a1_ready, bar_a1_free, bar_acc_full, bar_final, bar_alpha, bar_drain, bar_kblk[8];
    uint32_t tmem_base;
};
}  // namespace tc7

// ---- row packing (runs before the pair kernel; all sizes come from device counters, nothing synchronises)
// First-fit packing of the valid samples (1..8 rows each = their neighbour count) into 32-row quadrants, independently per
// super-chunk of PACK_S samples: samples are taken in order while they fit; a sample that does not fit stays first in line for
// the next quadrant while up to PACK_WIN later, smaller samples may fill the remaining rows (so the order inside a super-chunk
// becomes a permutation, vorder).  tests/test_host_logic.py restates the algorithm in Python; tests/test_gpu_shade.py compares
// the tables of these kernels with that restatement.
//   k_pack_quads  one WARP per super-chunk (counts in shared memory; the sequential "take while it fits" loop over the 64-entry
//                 window becomes <= 32 rounds of one warp scan each: a round takes the maximal prefix of still-fitting
//                 candidates and rejects the first one that does not fit).  Writes vorder / vcntp (final positions: the
//                 packing only permutes inside a super-chunk) and the quadrant boundaries super-chunk-locally.
//   k_pack_scan   exclusive scan of the per-super-chunk quadrant counts (one block), n_quads, sentinel
//   k_pack_place  quadrant boundaries -> their global position (fully parallel)
__global__ void __launch_bounds__(256) k_pack_quads(pnb_query_t q, int cap, uint32_t* __restrict__ sc_quads, uint32_t* __restrict__ quad_local,
                                                    uint32_t* __restrict__ vorder, unsigned char* __restrict__ vcntp,
                                                    float4* __restrict__ sigma_rgb) {
    __shared__ unsigned char cnt[8][tc7::PACK_S];
    const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int sc = blockIdx.x * 8 + wib;
    const int n_all = q.counters[PNB_QC_N_VALID];
    const int n_valid = min(n_all, cap);
    if (n_all > cap) {
        // workspace overflow (flagged as err 9 by the pair kernel): the samples that are dropped must not reach the compositing
        // kernel uninitialised -> they contribute nothing (sigma = 0)
        for (int vi = cap + blockIdx.x * blockDim.x + threadIdx.x; vi < n_all; vi += gridDim.x * blockDim.x)
            sigma_rgb[q.valid_list[vi]] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    const int i0 = sc * tc7::PACK_S;
    if (i0 >= n_valid) return;
    const int n = min(tc7::PACK_S, n_valid - i0);
    unsigned char* c = cnt[wib];                  // neighbour counts of this super-chunk; 0 = already placed
    for (int i = lane; i < n; i += 32) c[i] = q.samp_nvalid[q.valid_list[i0 + i]];
    __syncwarp();
    const uint32_t lt = (1u << lane) - 1u;
    int pos = 0, emitted = 0, nq = 0;
    while (pos < n) {                             // one quadrant per iteration (warp-uniform)
        if (lane == 0) quad_local[i0 + nq] = (uint32_t)(i0 + emitted);     // nq <= emitted: every quadrant holds >= 1 sample
        const int lim = min(n, pos + tc7::PACK_WIN);
        const int ia = pos + lane, ib = pos + 32 + lane;
        int ca = ia < lim ? (int)c[ia] : 0, cb = ib < lim ? (int)c[ib] : 0;
        int rows = 0, start = 0;                  // candidates with window index < start have been decided for this quadrant
        for (;;) {
            const int room = 32 - rows;
            const int va = (lane >= start && ca <= room) ? ca : 0, vb = (32 + lane >= start && cb <= room) ? cb : 0;
            int pa = va, pb = vb;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int ta = __shfl_up_sync(0xffffffffu, pa, d), tb = __shfl_up_sync(0xffffffffu, pb, d);
                if (lane >= d) { pa += ta; pb += tb; }
            }
            pb += __shfl_sync(0xffffffffu, pa, 31);
            const bool fa = va != 0 && pa <= room, fb = vb != 0 && pb <= room;
            const uint32_t ma = __ballot_sync(0xffffffffu, fa), mb = __ballot_sync(0xffffffffu, fb);
            const uint32_t na = __ballot_sync(0xffffffffu, va != 0 && pa > room), nb = __ballot_sync(0xffffffffu, vb != 0 && pb > room);
            const int cnt_a = __popc(ma);
            if (fa) { const int e = i0 + emitted + __popc(ma & lt); vorder[e] = (uint32_t)(i0 + ia); vcntp[e] = (unsigned char)ca; c[ia] = 0; }
            if (fb) { const int e = i0 + emitted + cnt_a + __popc(mb & lt); vorder[e] = (uint32_t)(i0 + ib); vcntp[e] = (unsigned char)cb; c[ib] = 0; }
            // rows taken this round = the largest fitting prefix sum
            int took = fb ? pb : (fa ? pa : 0);
#pragma unroll
            for (int d = 16; d >= 1; d >>= 1) took = max(took, __shfl_xor_sync(0xffffffffu, took, d));
            if (fa) ca = 0;
            if (fb) cb = 0;
            emitted += cnt_a + __popc(mb);
            rows += took;
            if (rows >= 32 || (na | nb) == 0u) break;
            start = na ? __ffs(na) : 32 + __ffs(nb);          // first rejected candidate + 1
            if (start >= 64) break;
        }
        __syncwarp();
        // first entry still unplaced (the window's entries keep their order; everything beyond the window is untouched)
        const uint32_t ra = __ballot_sync(0xffffffffu, ca != 0), rb = __ballot_sync(0xffffffffu, cb != 0);
        pos = ra ? pos + __ffs(ra) - 1 : (rb ? pos + 32 + __ffs(rb) - 1 : lim);
        ++nq;
    }
    if (lane == 0) sc_quads[sc] = (uint32_t)nq;
}
// exclusive scan of the per-super-chunk quadrant counts (one block): sc_quads[0 .. n_sc] (last = total), total -> pack_cnt[0],
// sentinel quad_first[n_quads] = n_valid; also zeroes the tile queue counter pack_cnt[1] of k_shade_tc8 (no extra launch per call)
__global__ void __launch_bounds__(1024) k_pack_scan(pnb_query_t q, int cap, uint32_t* __restrict__ sc_quads, uint32_t* __restrict__ quad_first,
                                                    int* __restrict__ pack_cnt) {
    __shared__ uint32_t wsum[32];
    const int n_valid = min(q.counters[PNB_QC_N_VALID], cap);
    const int n_sc = (n_valid + tc7::PACK_S - 1) / tc7::PACK_S;
    const int per = (n_sc + 1023) / 1024;
    const int b0 = threadIdx.x * per, b1 = min(b0 + per, n_sc);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t sum = 0;
    for (int i = b0; i < b1; ++i) sum += sc_quads[i];
    uint32_t incl = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += t; }
    if (lane == 31) wsum[w] = incl;
    __syncthreads();
    if (w == 0) {
        uint32_t v = wsum[lane], iv = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, iv, d); if (lane >= d) iv += t; }
        wsum[lane] = iv - v;
        if (lane == 31) { pack_cnt[0] = (int)iv; pack_cnt[1] = 0; quad_first[iv] = (uint32_t)n_valid; sc_quads[n_sc] = iv; }
    }
    __syncthreads();
    uint32_t run = wsum[w] + incl - sum;
    for (int i = b0; i < b1; ++i) { const uint32_t v = sc_quads[i]; sc_quads[i] = run; run += v; }
}
__global__ void __launch_bounds__(256) k_pack_place(pnb_query_t q, int cap, const uint32_t* __restrict__ sc_quads, const uint32_t* __restrict__ quad_local,
                                                    uint32_t* __restrict__ quad_first) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int n_valid = min(q.counters[PNB_QC_N_VALID], cap);
    if (i >= n_valid) return;
    const int sc = i / tc7::PACK_S, j = i - sc * tc7::PACK_S;
    const uint32_t first = sc_quads[sc], nq = sc_quads[sc + 1] - first;
    if ((uint32_t)j < nq) quad_first[first + j] = quad_local[i];
}

// Last epilogue with packed rows, one warp's share (chunks G, G+NG, ...): +bias, LeakyReLU, partial alpha dot product (returned),
// weight*conf scaling, then the K-reduction over the rows of each sample as a segmented inclusive scan (segments = samples,
// <= 8 lanes, first lane st); the last row of a sample (swrite) holds the sums and writes h-bar.
// EARLY (v8): ALL chunks of this warp are read into registers first and `drain_bar` is signalled right away - the accumulator region
// is then free for layer 2 of the next tile ~2 k cycles after the last MMA instead of after the whole reduction (~10 k).
// bias / wa: bias of block3.2 and the alpha weight (k_shade_tc8 passes its shared-memory copies: plain loads, no __ldg).
// O1: agg_intrp_order == 1 as a COMPILE-TIME flag (as a run-time flag ptxas if-converted the order-1 dot product: 16 extra loads + FMAs per
// chunk executed speculatively on the shipped order-2 path, seen in the ncu source page).
template <int NG, int NCHUNK, bool EARLY = false, bool O1 = false>
__device__ __forceinline__ float last_chunks_packed(const ShadeTcParams& p, const float* bias, const float* wa, uint32_t accb, int G, float wrow, int st,
                                                    bool swrite, int sidx, int lane, uint64_t* drain_bar = nullptr) {
    using namespace tc;
    constexpr bool order1 = O1;
    float apart = 0.f;
    uint32_t vv[EARLY ? NCHUNK : 2][16];
    if (EARLY) {
#pragma unroll
        for (int i = 0; i < NCHUNK; ++i) tmem_ld16(accb + (uint32_t)(16 * (G + NG * i)), vv[i]);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(drain_bar);
    } else {
        tmem_ld16(accb + (uint32_t)(16 * G), vv[0]);
    }
#pragma unroll
    for (int i = 0; i < NCHUNK; ++i) {
        const int c0 = 16 * (G + NG * i);
        const uint32_t* v = vv[EARLY ? i : (i & 1)];
        if (!EARLY) {
            tmem_ld_wait();
            if (i + 1 < NCHUNK) tmem_ld16(accb + (uint32_t)(c0 + 16 * NG), vv[(i + 1) & 1]);      // next chunk in flight under this one's math
        }
        float z[16];
#pragma unroll
        for (int e4 = 0; e4 < 4; ++e4) {
            const float4 bb = reinterpret_cast<const float4*>(bias + c0)[e4], ww = reinterpret_cast<const float4*>(wa + c0)[e4];
            const float bq[4] = {bb.x, bb.y, bb.z, bb.w}, wq[4] = {ww.x, ww.y, ww.z, ww.w};
#pragma unroll
            for (int e1 = 0; e1 < 4; ++e1) {
                const int e = 4 * e4 + e1;
                float y = __uint_as_float(v[e]) + bq[e1];
                y = fmaxf(y, LEAKY * y);
                if (!order1) apart = fmaf(y, wq[e1], apart);
                z[e] = y * wrow;
            }
        }
#pragma unroll
        for (int e = 0; e < 16; ++e) z[e] = seg_scan8(z[e], lane, st);
        if (order1) {       // agg_intrp_order 1: the alpha dot product runs over the K-aggregated feature (complete on the sample's last row)
#pragma unroll
            for (int e = 0; e < 16; ++e) apart = fmaf(z[e], wa[c0 + e], apart);
        }
        if (swrite) {
            if (p.hbar_fmt) {       // the colour kernel's operand image (bf16 hi / lo, core-matrix layout): two 16-byte rows each
                uint32_t hh[8], ll[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) split_bf16x2(z[2 * e], z[2 * e + 1], hh[e], ll[e]);
                unsigned char* dst = reinterpret_cast<unsigned char*>(p.hbar) + ((size_t)(sidx >> 7) * 8 + (c0 >> 5)) * (2 * 8192) +
                                     tile_offset_bytes<LAYOUT_NONE>(sidx & 127, c0 & 31);
                *reinterpret_cast<uint4*>(dst) = make_uint4(hh[0], hh[1], hh[2], hh[3]);
                *reinterpret_cast<uint4*>(dst + 128) = make_uint4(hh[4], hh[5], hh[6], hh[7]);
                *reinterpret_cast<uint4*>(dst + 8192) = make_uint4(ll[0], ll[1], ll[2], ll[3]);
                *reinterpret_cast<uint4*>(dst + 8192 + 128) = make_uint4(ll[4], ll[5], ll[6], ll[7]);
            } else {
                float4* dst = reinterpret_cast<float4*>(p.hbar + (size_t)sidx * 256 + c0);
                dst[0] = make_float4(z[0], z[1], z[2], z[3]);
                dst[1] = make_float4(z[4], z[5], z[6], z[7]);
                dst[2] = make_float4(z[8], z[9], z[10], z[11]);
                dst[3] = make_float4(z[12], z[13], z[14], z[15]);
            }
        }
    }
    return apart;
}
// One 16-column chunk of the last epilogue from REGISTERS (the deferred form of last_chunks_packed<.., EARLY = true>: identical
// arithmetic in identical order, so the two forms give bit-identical h-bar / alpha sums): columns c0 .. c0+15 of this lane's row in v.
template <bool O1>
__device__ __forceinline__ void last_chunk_from_regs(const ShadeTcParams& p, const float* bias, const float* wa, int c0, const uint32_t* v, float wrow, int st,
                                                     bool swrite, int sidx, int lane, float& apart) {
    using namespace tc;
    constexpr bool order1 = O1;
    float z[16];
#pragma unroll
    for (int e4 = 0; e4 < 4; ++e4) {
        const float4 bb = reinterpret_cast<const float4*>(bias + c0)[e4], ww = reinterpret_cast<const float4*>(wa + c0)[e4];
        const float bq[4] = {bb.x, bb.y, bb.z, bb.w}, wq[4] = {ww.x, ww.y, ww.z, ww.w};
#pragma unroll
        for (int e1 = 0; e1 < 4; ++e1) {
            const int e = 4 * e4 + e1;
            float y = __uint_as_float(v[e]) + bq[e1];
            y = fmaxf(y, LEAKY * y);
            if (!order1) apart = fmaf(y, wq[e1], apart);
            z[e] = y * wrow;
        }
    }
#pragma unroll
    for (int e = 0; e < 16; ++e) z[e] = seg_scan8(z[e], lane, st);
    if (order1) {
#pragma unroll
        for (int e = 0; e < 16; ++e) apart = fmaf(z[e], wa[c0 + e], apart);
    }
    if (swrite) {
        if (p.hbar_fmt) {
            uint32_t hh[8], ll[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) split_bf16x2(z[2 * e], z[2 * e + 1], hh[e], ll[e]);
            unsigned char* dst = reinterpret_cast<unsigned char*>(p.hbar) + ((size_t)(sidx >> 7) * 8 + (c0 >> 5)) * (2 * 8192) +
                                 tile_offset_bytes<LAYOUT_NONE>(sidx & 127, c0 & 31);
            *reinterpret_cast<uint4*>(dst) = make_uint4(hh[0], hh[1], hh[2], hh[3]);
            *reinterpret_cast<uint4*>(dst + 128) = make_uint4(hh[4], hh[5], hh[6], hh[7]);
            *reinterpret_cast<uint4*>(dst + 8192) = make_uint4(ll[0], ll[1], ll[2], ll[3]);
            *reinterpret_cast<uint4*>(dst + 8192 + 128) = make_uint4(ll[4], ll[5], ll[6], ll[7]);
        } else {
            float4* dst = reinterpret_cast<float4*>(p.hbar + (size_t)sidx * 256 + c0);
            dst[0] = make_float4(z[0], z[1], z[2], z[3]);
            dst[1] = make_float4(z[4], z[5], z[6], z[7]);
            dst[2] = make_float4(z[8], z[9], z[10], z[11]);
            dst[3] = make_float4(z[12], z[13], z[14], z[15]);
        }
    }
}
// Compiler-level anchor for registers written by an asynchronous tcgen05.ld: placed after tcgen05.wait::ld it makes the 16 values "defined
// here", so no copy of them can be scheduled between the load and its wait when they live across a loop back-edge.
__device__ __forceinline__ void pin16(uint32_t* v) {
    asm volatile("" : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]),
                      "+r"(v[8]), "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15]));
}
// warpgroup register re-allocation (setmaxnreg: all 4 warps of an aligned warpgroup execute it, convergent)
template <int N> __device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N> __device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }
// segment bookkeeping of one quadrant row: first row / index of its sample, whether it is the sample's last row
struct QuadRow { int st, j; bool live, is_end; };
__device__ __forceinline__ QuadRow quad_row(uint32_t head, int tot, int lane) {
    QuadRow r;
    r.live = lane < tot;
    const uint32_t below = head & (0xffffffffu >> (31 - lane));
    r.st = r.live ? 31 - __clz(below) : lane;
    r.j = r.live ? __popc(below) - 1 : 0;
    const uint32_t nxt = lane < 31 ? (head >> (lane + 1)) : 0u;
    r.is_end = r.live && lane == (nxt ? lane + __ffs(nxt) - 1 : tot - 1);
    return r;
}

template <bool O1>
__global__ void __launch_bounds__(tc7::NTHR, 1) k_shade_tc7(ShadeTcParams p) {
    using namespace tc;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    tc7::Smem& sm = *reinterpret_cast<tc7::Smem*>(smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u));
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const pnb_query_t& q = p.q;
    const int n_valid = min(q.counters[PNB_QC_N_VALID], p.hbar_cap);
    const int n_quads = p.pack_cnt[0];
    const int n_tiles = (n_quads + 3) >> 2;
    const int my_tiles = n_tiles > (int)blockIdx.x ? (n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    constexpr int W_BUILD = tc7::NEPI_WARPS, W_LOAD = W_BUILD + tc7::NBUILD / 32, W_ISSUE = W_LOAD + 1;

    if (tid == 0) {
        for (int s = 0; s < tc7::NSTAGE; ++s) { mbar_init(&sm.bar_full[s], 1); mbar_init(&sm.bar_empty[s], 1); }
        mbar_init(&sm.bar_a1_ready, tc7::NBUILD / 32);              // one arrive per builder warp
        mbar_init(&sm.bar_a1_free, 1);
        mbar_init(&sm.bar_acc_full, 1);
        mbar_init(&sm.bar_final, 1);
        mbar_init(&sm.bar_alpha, tc7::NEPI_WARPS);
        mbar_init(&sm.bar_drain, tc7::NEPI_WARPS + tc7::NBUILD / 32);     // one arrive per warp that reads the layer-4 accumulator
        for (int c = 0; c < 8; ++c) mbar_init(&sm.bar_kblk[c], 4 * 2);   // one arrive per warp and chunk (32 same-address arrives serialise)
        mbar_fence_init();
        if (blockIdx.x == 0 && q.counters[PNB_QC_N_VALID] > p.hbar_cap) atomicExch(p.err, 9);
    }
    if (tid < TM) sm.alpha_e[tid] = 0.f;
    if (warp == W_ISSUE) tmem_alloc<512>(&sm.tmem_base);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tP = sm.tmem_base, tQ = sm.tmem_base + 256u;
    const long long _tk0 = clock64();

    if (warp == W_LOAD) {
        if (lane == 0) {
            const uint32_t total = (uint32_t)my_tiles * IMGS_PER_TILE;
            for (uint32_t n = 0; n < total; ++n) {
                const uint32_t s = n & (tc7::NSTAGE - 1), ph = (n >> 2) & 1u;
                if (!mbar_wait(&sm.bar_empty[s], ph ^ 1u, p.err, 91)) break;
                if (p.dbg_no_weights) { mbar_arrive(&sm.bar_full[s]); continue; }
                mbar_arrive_expect_tx(&sm.bar_full[s], IMG);
                bulk_g2s(sm.b[s], p.wimg + (size_t)(n % IMGS_PER_TILE) * IMG, IMG, &sm.bar_full[s]);
            }
        }
    } else if (warp == W_ISSUE) {
        // ============================================================ MMA issuer (identical to v5)
        const uint32_t idesc = make_idesc_bf16(128, 256);
        const uint32_t hiw = desc_hi<LAYOUT>(), xe_hiw = (256u >> 4) | (1u << 14);
        const uint32_t b0_lo = desc_lo<LAYOUT>(smem_u32(sm.b[0]));
        const uint32_t ahi_lo = desc_lo<LAYOUT>(smem_u32(sm.a_hi)), alo_lo = desc_lo<LAYOUT>(smem_u32(sm.a_lo));
        const uint32_t xeh_lo0 = desc_lo<LAYOUT_NONE>(smem_u32(sm.xe_hi[0])), xel_lo0 = desc_lo<LAYOUT_NONE>(smem_u32(sm.xe_lo[0]));
        constexpr uint32_t KADV = kstep_adv16<LAYOUT>();
        uint32_t n = 0, c_acc = 0, c_pack = 0;
        bool ok = true;
        for (int t = 0; t < my_tiles && ok; ++t) {
            const uint32_t xeh_lo = xeh_lo0 + (uint32_t)(t & 1) * (tc::XE >> 4), xel_lo = xel_lo0 + (uint32_t)(t & 1) * (tc::XE >> 4);
            for (int l = 0; l < 4 && ok; ++l) {
                const uint32_t acc = (l & 1) ? tP : tQ;
                const uint32_t ab = (l & 1) ? tQ : tP;
                if (l > 0) { if (!mbar_wait(&sm.bar_acc_full, c_acc & 1u, p.err, 92)) { ok = false; break; } ++c_acc; }
                else if (t > 0) { if (!mbar_wait(&sm.bar_final, (uint32_t)(t - 1) & 1u, p.err, 92)) { ok = false; break; } }
                if (l == 0) { if (!mbar_wait(&sm.bar_a1_ready, (uint32_t)t & 1u, p.err, 93)) { ok = false; break; } }
                if (l == 1 && t > 0) { if (!mbar_wait(&sm.bar_drain, (uint32_t)(t - 1) & 1u, p.err, 94)) { ok = false; break; } }
                tc_fence_after();
                const int nkb = nkb_of(l);
                for (int kb = 0; kb < nkb && ok; ++kb) {
                    const uint32_t s0 = n & (tc7::NSTAGE - 1), ph0 = (n >> 2) & 1u;
                    const uint32_t s1 = (n + 1) & (tc7::NSTAGE - 1), ph1 = ((n + 1) >> 2) & 1u;
                    const bool need_chunks = (l >= 1 && kb < 8);
                    uint64_t* cb0 = need_chunks ? &sm.bar_kblk[kb] : &sm.bar_full[s0];
                    const uint32_t cp0 = need_chunks ? (c_pack & 1u) : ph0;
                    if (!mbar_try_wait4(&sm.bar_full[s0], ph0, &sm.bar_full[s1], ph1, cb0, cp0, &sm.bar_full[s1], ph1)) {
                        if (need_chunks && !mbar_wait(cb0, cp0, p.err, 95)) { ok = false; break; }
                        if (!mbar_wait(&sm.bar_full[s0], ph0, p.err, 96)) { ok = false; break; }
                        if (!mbar_wait(&sm.bar_full[s1], ph1, p.err, 96)) { ok = false; break; }
                    }
                    tc_fence_after();
                    const uint32_t akb_hi = ahi_lo + (uint32_t)kb * (ABLK >> 4), akb_lo = alo_lo + (uint32_t)kb * (ABLK >> 4);
                    const uint32_t tcol = ab + (uint32_t)(kb * 32);
                    const uint32_t bl = b0_lo + s0 * (IMG >> 4), bl2 = b0_lo + s1 * (IMG >> 4);
                    if (l == 0) {
                        mma_ss2_w(acc, akb_hi, hiw, bl, hiw, idesc, kb ? 1u : 0u);
                        mma_ss2_w(acc, akb_lo, hiw, bl, hiw, idesc, 1u);
                        mma_ss2_w(acc, akb_hi + KADV, hiw, bl + KADV, hiw, idesc, 1u);
                        mma_ss2_w(acc, akb_lo + KADV, hiw, bl + KADV, hiw, idesc, 1u);
                        mma_commit_w(&sm.bar_empty[s0]);
                        mma_ss2_w(acc, akb_hi, hiw, bl2, hiw, idesc, 1u);
                        mma_ss2_w(acc, akb_hi + KADV, hiw, bl2 + KADV, hiw, idesc, 1u);
                        mma_commit_w(&sm.bar_empty[s1]);
                    } else if (kb == 8) {
                        mma_ss2_w(acc, xeh_lo, xe_hiw, bl, hiw, idesc, 1u);
                        mma_ss2_w(acc, xel_lo, xe_hiw, bl, hiw, idesc, 1u);
                        mma_commit_w(&sm.bar_empty[s0]);
                        mma_ss2_w(acc, xeh_lo, xe_hiw, bl2, hiw, idesc, 1u);
                        mma_commit_w(&sm.bar_empty[s1]);
                    } else {
                        mma_ts2_w(acc, tcol, bl, hiw, idesc, kb ? 1u : 0u);
                        mma_ts2_w(acc, tcol + 8u, bl, hiw, idesc, 1u);
                        mma_ts2_w(acc, tcol + 16u, bl + KADV, hiw, idesc, 1u);
                        mma_ts2_w(acc, tcol + 24u, bl + KADV, hiw, idesc, 1u);
                        mma_commit_w(&sm.bar_empty[s0]);
                        mma_ts2_w(acc, tcol, bl2, hiw, idesc, 1u);
                        mma_ts2_w(acc, tcol + 16u, bl2 + KADV, hiw, idesc, 1u);
                        mma_commit_w(&sm.bar_empty[s1]);
                    }
                    n += 2;
                }
                if (!ok) break;
                if (l >= 1) ++c_pack;
                mma_commit_w(l < 3 ? &sm.bar_acc_full : &sm.bar_final);      // layers 1-3 -> epilogue warps; layer 4 -> every warp's share of the last epilogue
                if (l == 0) mma_commit_w(&sm.bar_a1_free);
            }
        }
    } else if (warp >= W_BUILD) {
        // ============================================================ builders: two warps per quadrant (operand columns 0..151 | 152..287),
        // lane = row; the same warps run chunk groups 2, 3 of the last epilogue of the previous tile (they are idle under layer 1)
        const int bw = warp - W_BUILD, qw = bw & 3, part = bw >> 2, row = qw * 32 + lane;
        const uint32_t tlane = (uint32_t)(qw * 32) << 16;
        bool ok = true;
        for (int t = 0; t <= my_tiles && ok; ++t) {
            if (t < my_tiles) {
                const int tile = (int)blockIdx.x + t * (int)gridDim.x;
                if (t > 0 && !mbar_wait(&sm.bar_a1_free, (uint32_t)(t - 1) & 1u, p.err, 97)) { ok = false; break; }
                const int qd = tile * 4 + qw;
                uint32_t first = 0, nsamp = 0;
                if (qd < n_quads) { first = p.quad_first[qd]; nsamp = p.quad_first[qd + 1] - first; }
                const int c = lane < (int)nsamp ? (int)p.vcnt[first + lane] : 0;
                int incl = c;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += v; }
                const uint32_t head = __reduce_or_sync(0xffffffffu, lane < (int)nsamp ? (1u << (incl - c)) : 0u);
                const int total = __shfl_sync(0xffffffffu, incl, 31);
                const QuadRow qr = quad_row(head, total, lane);
                const int cj = __shfl_sync(0xffffffffu, c, qr.j);
                if (lane == 0 && part == 1) { sm.qhead[t & 1][qw] = head; sm.qfirst[t & 1][qw] = first; sm.qtotal[t & 1][qw] = (uint32_t)total; }
                const int pvi = qr.live ? (int)p.vorder[first + qr.j] : -1;
                if (part == 0) build_pair_part<0, true>(sm, p, tile, t, row, n_valid, pvi, lane - qr.st, qr.st, qr.live ? cj : 1);
                else build_pair_part<1, true>(sm, p, tile, t, row, n_valid, pvi, lane - qr.st, qr.st, qr.live ? cj : 1);
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(&sm.bar_a1_ready);
            }
            if (t > 0) {
                const int tf = t - 1;
                if (!mbar_wait(&sm.bar_final, (uint32_t)tf & 1u, p.err, 99)) { ok = false; break; }
                tc_fence_after();
                const QuadRow qr = quad_row(sm.qhead[tf & 1][qw], (int)sm.qtotal[tf & 1][qw], lane);
                const int sidx = qr.live ? (int)p.vorder[sm.qfirst[tf & 1][qw] + qr.j] : 0;
                const bool swrite = qr.is_end && sidx < n_valid;
                const float wrow = sm.wc[tf & 1][row];
                const float apart = last_chunks_packed<4, 4, false, O1>(p, p.bias[3], p.wa, tP + tlane, 2 + part, wrow, qr.st, swrite, sidx, lane);
                tc_fence_before();
                sm.alpha_part[part][row] = apart;
                named_bar_sync(2, tc7::NBUILD);
                if (!mbar_wait(&sm.bar_alpha, (uint32_t)tf & 1u, p.err, 100)) { ok = false; break; }      // the epilogue warps' partial sums
                if (part == 0) {
                    const float a = (sm.alpha_part[0][row] + sm.alpha_part[1][row]) + sm.alpha_e[row] + __ldg(p.ba) - 1.0f;
                    sm.alpha_e[row] = 0.f;
                    const float sp = a > 20.f ? a : log1pf(expf(a));
                    // order 2: density per neighbour, weighted sum over the sample's rows; order 1: `a` is already the sample's value (its last row)
                    const float zz = O1 ? sp : seg_scan8(sp * wrow, lane, qr.st);
                    if (swrite) p.sigma[sidx] = zz;
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&sm.bar_drain);                 // after the alpha_e reads
                named_bar_sync(2, tc7::NBUILD);
            }
        }
    } else {
        // ============================================================ epilogue warps
        const int quad = warp & 3, grp = warp >> 2;
        const int erow = quad * 32 + lane;
        const uint32_t tlane = (uint32_t)(quad * 32) << 16;
        uint32_t n_acc = 0;
        bool ok = true;
        for (int t = 0; t < my_tiles && ok; ++t) {
            for (int l = 0; l < 3 && ok; ++l, ++n_acc) {        // the layer-4 (last) epilogue is shared with the builder warps
                if (!mbar_wait(&sm.bar_acc_full, n_acc & 1u, p.err, 98)) { ok = false; break; }
                tc_fence_after();
                const uint32_t accb = ((l & 1) ? tP : tQ) + tlane;
                {
                    const float* bias = p.bias[l];
#pragma unroll
                    for (int i = 0; i < tc7::NCH; ++i) {
                        const int g = grp + tc7::NGRP * i, c0 = 16 * g;
                        uint32_t v[16];
                        tmem_ld16(accb + (uint32_t)c0, v);
                        tmem_ld_wait();
                        uint32_t hh[8], ll[8];
#pragma unroll
                        for (int e = 0; e < 8; ++e) {
                            float2 bb = __ldg(reinterpret_cast<const float2*>(bias + c0) + e);
                            float y0 = __uint_as_float(v[2 * e]) + bb.x, y1 = __uint_as_float(v[2 * e + 1]) + bb.y;
                            y0 = fmaxf(y0, LEAKY * y0); y1 = fmaxf(y1, LEAKY * y1);
                            split_bf16x2(y0, y1, hh[e], ll[e]);
                        }
                        tmem_st8(accb + (uint32_t)c0, hh);
                        tmem_st8(accb + (uint32_t)c0 + 8u, ll);
                        tmem_st_wait();
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&sm.bar_kblk[g >> 1]);
                    }
                }
            }
            if (!ok) break;
            {   // this warp's share of the LAST epilogue (chunk groups 0, 1; the builder warps take 2, 3)
                if (!mbar_wait(&sm.bar_final, (uint32_t)t & 1u, p.err, 101)) { ok = false; break; }
                tc_fence_after();
                const QuadRow qr = quad_row(sm.qhead[t & 1][quad], (int)sm.qtotal[t & 1][quad], lane);
                const int sidx = qr.live ? (int)p.vorder[sm.qfirst[t & 1][quad] + qr.j] : 0;
                const float apart = last_chunks_packed<4, 4, false, O1>(p, p.bias[3], p.wa, tP + tlane, grp, sm.wc[t & 1][erow], qr.st, qr.is_end && sidx < n_valid, sidx, lane);
                tc_fence_before();
                atomicAdd(&sm.alpha_e[erow], apart);
                __syncwarp();
                if (lane == 0) { mbar_arrive(&sm.bar_alpha); mbar_arrive(&sm.bar_drain); }
            }
        }
    }
    if (tid == 0 && (p.dbg_flags & 4) && blockIdx.x < 192) {      // per-CTA cycles and SM id; [32 + 192] = number of quadrants
        uint32_t smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        reinterpret_cast<long long*>(p.err)[32 + blockIdx.x] = ((clock64() - _tk0) & 0xffffffffffffll) | ((long long)smid << 48);
        if (blockIdx.x == 0) reinterpret_cast<long long*>(p.err)[32 + 192] = n_quads;
    }
    tc_fence_before();
    __syncthreads();
    if (warp == W_ISSUE) tmem_dealloc<512>(sm.tmem_base);
}

// =====================================================================================================================
// v8: the v7 pipeline for a FROZEN point cloud (rendering; opt.pnb_frozen, default when no point/MLP tensor needs a gradient).
// The first 224 of the 284 inputs of block1.0 ([f, PE3(f)]) depend on the POINT only, not on the sample, so their
// contribution to the layer-1 pre-activation is hoisted out of the per-pair work: k_point_pre computes
//     pre[n][0..255] = b1 + W1[:, :224] . [f_n, PE3(f_n)]      (fp32, once per point-cloud / weight version, 1 KB per point)
// and the layer-1 epilogue adds pre[pidx] to the accumulator where v7 adds the bias.  What remains of layer 1 is the 60
// sample-dependent inputs PE5(dists) = 2 K blocks instead of 9:
//   * 159 MMAs per 128-row tile instead of 201, and 192 of the 252 sin/cos pairs per pair disappear (one builder thread per row);
//   * the layer-1 operand shrinks from 144 KB to 32 KB of shared memory, which buys a weight ring whose stage is a WHOLE K block
//     (hi + lo image, 32 KB, 5 stages): one tcgen05.commit per K block instead of one per image (27 + 5 per tile instead of 73;
//     a commit costs ~140 tensor-pipe cycles, profiles/r01_umma_pair_commit_cost.log);
//   * the per-pair gather becomes 1 KB of `pre` (read by the epilogue warps, 64 B per thread and 16-column chunk, prefetched
//     PF chunks ahead) instead of the 128 B feature row: L2 traffic, the table of a 400 k cloud is 410 MB.
// Pipeline otherwise as v7 (TMEM role ping-pong P/Q, chunk-granular hand-off, packed rows, shared last epilogue).
// Warps (448 threads): 0-7 epilogue (quadrant = w & 3, chunk group = w >> 2), 8-11 builders (thread = row), 12 loader, 13 issuer.
namespace tc8 {
constexpr int NBUILD = 128;
constexpr int NGRP = 2;                   // epilogue warps per TMEM lane quarter (4 measured slower: the quarter's TMEM port is shared)
constexpr int NEPI_WARPS = 4 * NGRP, NCH = 16 / NGRP;
constexpr int NTHR = NEPI_WARPS * 32 + NBUILD + 64;
constexpr int NTHR_DEFER = 512;           // DEFER variant: 4 whole warpgroups (2 x epilogue, builders, {loader, issuer, 2 idle warps}) for setmaxnreg
constexpr int REG_EPI = 168, REG_BUILD = 136, REG_CTRL = 40;     // 256 x 168 + 128 x 136 + 128 x 40 = 65536 registers
constexpr int STAGE = 2 * tc::IMG;        // ring stage = one K block: hi image + lo image
constexpr int NKB1 = 2;                   // K blocks of the frozen layer 1 (operand columns 224..287 of block1.0)
constexpr int KB1_FIRST = 7;
constexpr int STAGES_PER_TILE = NKB1 + 8 + 9 + 8;
constexpr int XPOSE = 2048;               // per-warp transpose buffer of the coalesced `pre` gather: 32 rows x 64 B
template <int NSTAGE_, bool COOP>
struct Smem {
    static constexpr int NWC = 2, NSTAGE = NSTAGE_;
    unsigned char a_hi[NKB1 * tc::ABLK];
    unsigned char a_lo[NKB1 * tc::ABLK];
    unsigned char b[NSTAGE][STAGE];
    unsigned char xe_hi[2][tc::XE];
    unsigned char xe_lo[2][tc::XE];
    unsigned char xpose[COOP ? NEPI_WARPS : 1][COOP ? XPOSE : 16];
    float wc[NWC][tc::TM];
    float alpha_part[2][NGRP][tc::TM];    // [tile parity][epilogue group] partial alpha dot products (own slot each: summed in a fixed order)
    int prow[2][tc::TM];                  // point index of every row (-1: unused row)
    alignas(16) float bias[3][256];       // copies of the layer 2..4 biases and the alpha weight: the epilogues read them per chunk as
    alignas(16) float wa[256];            // warp-broadcast LDS.128 instead of __ldg (LSU data pipe shared with tcgen05.ld/st and the gather)
    int tile_slot[2];                     // tile index of this CTA's tile t in [t & 1] (-1: no tile left), written by builder warp 0
    uint32_t qhead[NWC][4], qfirst[NWC][4], qtotal[NWC][4];
    uint64_t bar_full[NSTAGE], bar_empty[NSTAGE], bar_a1_ready, bar_a1_free, bar_acc_full, bar_final, bar_alpha, bar_drain, bar_kblk[8], bar_prow[2],
             bar_tile[2];
    uint32_t tmem_base;
};
}  // namespace tc8

// pre[n][c] = b1[c] + sum_{k<224} W1^T[k][c] * x_n[k],  x_n = [f (32), PE3(f) (192, column 32 + 6*feature + 2*j + {sin, cos})]:
// exactly the first 7 K blocks of the operand build_pair_part writes.  fp32 FMAs in ascending k.  Block = 32 points x 256 columns.
__global__ void __launch_bounds__(256) k_point_pre(const float* __restrict__ emb, int N, const float* __restrict__ w1t, const float* __restrict__ b1,
                                                   float* __restrict__ pre) {
    __shared__ __align__(16) float x[32][224 + 4];
    const int n0 = blockIdx.x * 32;
    for (int i = threadIdx.x; i < 32 * PNB_FEAT; i += 256) {
        const int pl = i >> 5, f = i & 31, n = n0 + pl;
        const float v = n < N ? __ldg(&emb[(size_t)n * PNB_FEAT + f]) : 0.f;
        float pe[6];
        pe_doubling<3>(v, pe);
        x[pl][f] = v;
#pragma unroll
        for (int e = 0; e < 6; ++e) x[pl][32 + 6 * f + e] = pe[e];
    }
    __syncthreads();
    const int c = threadIdx.x;
    float acc[32];
    const float bc = __ldg(&b1[c]);
#pragma unroll
    for (int i = 0; i < 32; ++i) acc[i] = 0.f;
    for (int k = 0; k < 224; k += 4) {
        const float w0 = __ldg(&w1t[(size_t)k * 256 + c]), w1 = __ldg(&w1t[(size_t)(k + 1) * 256 + c]);
        const float w2 = __ldg(&w1t[(size_t)(k + 2) * 256 + c]), w3 = __ldg(&w1t[(size_t)(k + 3) * 256 + c]);
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            const float4 xv = *reinterpret_cast<const float4*>(&x[i][k]);
            acc[i] = fmaf(xv.w, w3, fmaf(xv.z, w2, fmaf(xv.y, w1, fmaf(xv.x, w0, acc[i]))));
        }
    }
#pragma unroll
    for (int i = 0; i < 32; ++i)
        if (n0 + i < N) pre[(size_t)(n0 + i) * 256 + c] = acc[i] + bc;
}

// One pair row of the frozen pipeline: the PE5(dists) K blocks of the layer-1 operand (operand columns 224..287 -> blocks 0, 1),
// the block3 extras operand, weight*conf and the row's point index.  Same arithmetic as build_pair_part<PART 1, PACKED>.
template <class SmemT>
__device__ __forceinline__ void build_pair_frozen(SmemT& sm, const ShadeTcParams& p, int t, int row, int n_valid, int pvi, int pk, int pst, int pcnt) {
    using namespace tc;
    const pnb_query_t& q = p.q;
    int pidx = -1;
    float lx = 0.f, ly = 0.f, lz = 0.f, vx = 0.f, vy = 0.f, vz = 0.f;
    if (pvi >= 0 && pvi < n_valid) {
        const uint32_t s = q.valid_list[pvi];
        const uint32_t sr = q.samp_ray[s];
        const int r = (int)(sr >> 7), j = (int)(sr & 127u);
        const int d = q.steps[(size_t)r * q.SR + j];
        const float tt = q.t[(size_t)r * q.t_ray_stride + d];
        vx = q.raydir[3 * r]; vy = q.raydir[3 * r + 1]; vz = q.raydir[3 * r + 2];
        lx = raypos1(q.campos[0], vx, tt); ly = raypos1(q.campos[1], vy, tt); lz = raypos1(q.campos[2], vz, tt);
        if (pk < q.K) pidx = q.cand_pidx[(size_t)s * q.K + pk];
    }
    const bool valid = pidx >= 0;
    const int pi = valid ? pidx : 0;
    sm.prow[t & 1][row] = pidx;
    float dist[6];
    float ovx, ovy, ovz;
    rot3t(p.o.Rw2c, vx, vy, vz, ovx, ovy, ovz);
    const float px = __ldg(&p.pts.xyz[3 * pi]), py = __ldg(&p.pts.xyz[3 * pi + 1]), pz = __ldg(&p.pts.xyz[3 * pi + 2]);
    dist[0] = px - lx; dist[1] = py - ly; dist[2] = pz - lz;
    float xpp, ypp, zpp, xsp, ysp, zsp;
    w2pers_t(p.o, px, py, pz, xpp, ypp, zpp);
    w2pers_t(p.o, lx, ly, lz, xsp, ysp, zsp);
    dist[3] = xpp * zpp - xsp * zsp; dist[4] = ypp * zpp - ysp * zsp; dist[5] = zpp - zsp;
    const float nrm = sqrtf(dist[0] * dist[0] + dist[1] * dist[1] + dist[2] * dist[2]);
    float w = valid ? 1.0f / fmaxf(nrm, 1e-6f) : 0.f;
    const float wsum = seg_sum8(w, row & 31, pst, pcnt);
    w = w / fmaxf(wsum, 1e-8f);
    const float cf = __ldg(&p.pts.conf[pi]);
    sm.wc[t & 1][row] = valid ? w * fminf(fmaxf(cf, 1e-4f), 1.0f) : 0.f;
    float d0, d1, d2;
    rot3t(p.o.Rw2c, dist[0], dist[1], dist[2], d0, d1, d2);
    dist[0] = d0; dist[1] = d1; dist[2] = d2;
    float ex[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (valid) {
        float dp[64];
#pragma unroll
        for (int e = 0; e < 6; ++e) pe_doubling<5>(dist[e], dp + 10 * e);
        dp[60] = dp[61] = dp[62] = dp[63] = 0.f;
#pragma unroll
        for (int c = 0; c < 8; ++c) store_chunk8_a1(sm, row, c >> 2, (c & 3) * 8, dp + 8 * c);
        float ddx, ddy, ddz;
        rot3t(p.o.Rw2c, __ldg(&p.pts.dir[3 * pi]), __ldg(&p.pts.dir[3 * pi + 1]), __ldg(&p.pts.dir[3 * pi + 2]), ddx, ddy, ddz);
        ex[0] = __ldg(&p.pts.color[3 * pi]); ex[1] = __ldg(&p.pts.color[3 * pi + 1]); ex[2] = __ldg(&p.pts.color[3 * pi + 2]);
        ex[3] = ddx - ovx; ex[4] = ddy - ovy; ex[5] = ddz - ovz;
        ex[6] = ddx * ovx + ddy * ovy + ddz * ovz;
    } else {
        const float z8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int c = 0; c < 8; ++c) store_chunk8_a1(sm, row, c >> 2, (c & 3) * 8, z8);
    }
    uint32_t h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) split_bf16x2(ex[2 * i], ex[2 * i + 1], h[i], l[i]);
    const uint32_t off = tc::xe_offset(row, 0);
    *reinterpret_cast<uint4*>(sm.xe_hi[t & 1] + off) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(sm.xe_lo[t & 1] + off) = make_uint4(l[0], l[1], l[2], l[3]);
    *reinterpret_cast<uint4*>(sm.xe_hi[t & 1] + off + 128) = make_uint4(0u, 0u, 0u, 0u);
    *reinterpret_cast<uint4*>(sm.xe_lo[t & 1] + off + 128) = make_uint4(0u, 0u, 0u, 0u);
}

// The layer-1 epilogue adds pre[point of the row][column]: 1 KB per row, gathered from L2 / HBM.
// Reading it "lane = row" (each lane 64 B of its own row per chunk) makes every LDG.128 touch 32 different 128-byte lines = 32
// wavefronts of the LSU data pipe: 8192 per tile, measured to be what bounds the layer-1 epilogue (ncu: the pipe is 51 % busy over
// the WHOLE kernel, profiles/r02_ncu_full_summary.txt; E1 8.0 k cycles vs 4.0 k for the bias-only layers).  COOP: the warp reads
// coalesced instead - LDG j, lane l -> row 8j + l/4, 16-byte quarter l%4 of the chunk: 4 lines per request - and transposes through a
// 2 KB per-warp shared-memory buffer (XOR-swizzled, conflict-free both ways) into the lane = row order tcgen05.ld delivers.
template <bool COOP, int PF_ = 3>
struct Tc8Pf {                                    // chunks of `pre` in flight per epilogue thread (layer 1)
    static constexpr int PF = PF_;                  // (6 in flight measured slower: 40.0 k vs 37.3 k cycles per tile)
    float4 v[PF][4];
    const float4* src[COOP ? 4 : 1];              // COOP: rows 8j + lane/4 (+ this lane's quarter); else: this lane's row
    __device__ __forceinline__ void init(const float* __restrict__ pre, const int* prow, int lane) {
        if (COOP) {
#pragma unroll
            for (int j = 0; j < 4; ++j) src[j] = reinterpret_cast<const float4*>(pre + (size_t)max(prow[8 * j + (lane >> 2)], 0) * 256) + (lane & 3);
        } else {
            src[0] = reinterpret_cast<const float4*>(pre + (size_t)max(prow[lane], 0) * 256);   // unused rows: any finite values
        }
    }
    __device__ __forceinline__ void load(int slot, int g) {      // chunk g (16 columns) into v[slot]
#pragma unroll
        for (int e = 0; e < 4; ++e) v[slot][e] = COOP ? __ldg(src[e] + 4 * g) : __ldg(src[0] + 4 * g + e);
    }
    __device__ __forceinline__ void prefetch(int grp) {
#pragma unroll
        for (int i = 0; i < PF; ++i) load(i, grp + tc8::NGRP * i);
    }
    // the 16 values of this lane's row for the chunk held in v[slot]
    __device__ __forceinline__ void fetch(int slot, unsigned char* xp, int lane, float4 (&out)[4]) {
        if (COOP) {
            const int m = lane >> 2, q = lane & 3;
            __syncwarp();                         // the previous chunk's reads of the buffer are done
#pragma unroll
            for (int j = 0; j < 4; ++j) *reinterpret_cast<float4*>(xp + q * 512 + j * 128 + ((m + 2 * q) & 7) * 16) = v[slot][j];
            __syncwarp();
#pragma unroll
            for (int e = 0; e < 4; ++e) out[e] = *reinterpret_cast<const float4*>(xp + e * 512 + (lane >> 3) * 128 + (((lane & 7) + 2 * e) & 7) * 16);
        } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) out[e] = v[slot][e];
        }
    }
};

// One epilogue layer of a warp: chunks grp, grp+NGRP, ... (16 accumulator columns each): accumulator -> (+ bias (shared memory) or + pre[point]) ->
// LeakyReLU -> bf16 hi/lo -> the same columns, one mbarrier arrive per warp and chunk.
template <bool FIRST, bool COOP, class SmemT, class PfT>
__device__ __forceinline__ void tc8_epi_layer(SmemT& sm, uint32_t accb, int grp, const float* __restrict__ bias, PfT& pfs, unsigned char* xp) {
    using namespace tc;
    constexpr int NGRP = tc8::NGRP, NCH = tc8::NCH, PF = PfT::PF;
    const int lane = threadIdx.x & 31;
    const bool lane0 = lane == 0;                 // ONE mbarrier arrive per warp and chunk
    uint32_t v[16];
#pragma unroll
    for (int i = 0; i < NCH; ++i) {
        const int g = grp + NGRP * i, c0 = 16 * g;
        tmem_ld16(accb + (uint32_t)c0, v);
        float4 b4[4];
        if (FIRST) pfs.fetch(i % PF, xp, lane, b4);
        else {
#pragma unroll
            for (int e = 0; e < 4; ++e) b4[e] = reinterpret_cast<const float4*>(bias + c0)[e];     // shared-memory copy
        }
        if (FIRST && i + PF < NCH) pfs.load(i % PF, g + NGRP * PF);
        tmem_ld_wait();
        uint32_t hh[8], ll[8];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            float y0 = __uint_as_float(v[4 * e]) + b4[e].x, y1 = __uint_as_float(v[4 * e + 1]) + b4[e].y;
            float y2 = __uint_as_float(v[4 * e + 2]) + b4[e].z, y3 = __uint_as_float(v[4 * e + 3]) + b4[e].w;
            y0 = fmaxf(y0, LEAKY * y0); y1 = fmaxf(y1, LEAKY * y1); y2 = fmaxf(y2, LEAKY * y2); y3 = fmaxf(y3, LEAKY * y3);
            split_bf16x2(y0, y1, hh[2 * e], ll[2 * e]);
            split_bf16x2(y2, y3, hh[2 * e + 1], ll[2 * e + 1]);
        }
        tmem_st8(accb + (uint32_t)c0, hh);
        tmem_st8(accb + (uint32_t)c0 + 8u, ll);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane0) mbar_arrive(&sm.bar_kblk[g >> 1]);
    }
}

// NSTAGE: stages of the weight ring; COOP: coalesced + transposed gather of the hoisted table (see Tc8Pf).
// DEFER: the last epilogue of tile t no longer sits between layer 4 of tile t and the layer-1 epilogue of tile t+1.  Every warp still drains
// its chunks of the layer-4 accumulator into registers right away (bar_drain), but the epilogue warps then go straight on to tile t+1 and
// work their held chunks off in the gaps where they would otherwise wait for the tensor pipe (before the layer-2 / layer-3 / layer-4
// accumulator barriers of tile t+1); the builder warps process theirs at once and finalise sigma one tile later.  Holding 128 x 256 fp32
// next to the layer-1 epilogue's working set needs more registers per epilogue thread than a uniform split of the file gives: the
// warpgroups re-allocate (setmaxnreg): epilogue 168, builders 136, loader / issuer 40.  Same arithmetic in the same order -> results
// bit-identical to the non-deferred form.
// SCHED (DEFER only): how the 5 held chunks are spread over the gaps of the next tile - before the layer-1 (A) / layer-2 (B) / layer-3 (C)
// accumulator barriers and before the layer-4 barrier (D): 0 = 2/2/1/0, 1 = 1/2/1/1, 2 = 0/2/2/1 (default: nothing in gap A, which sits on the
// layer 4 -> layer 1 -> layer 2 critical path).  PFN: chunks of `pre` in flight in the layer-1 epilogue (2 with DEFER: registers).
// UNI: the issuer's code is a provably uniform region (operands in uniform registers); false = the previous form (A/B).
// XF: layers are queued back to back (tcgen05.mma execute in issue order: a layer's accumulator region is the previous layer's dead operand
// region, so the issuer need not wait for the previous layer's completion barrier - only for the per-K-block operand barriers), and layer 3
// issues its extras K block (operand from shared memory, independent of the layer-2 epilogue) FIRST, into the layer turn-around bubble.
// TILE QUEUE: the tiles are handed out in increasing order by one device counter (p.tile_ctr, zeroed by k_pack_scan of the same call), so
// a CTA that runs slower simply takes fewer tiles (static striding made the kernel as long as its slowest CTA; dbg bit 4 keeps it for A/B).
// Builder warp 0 takes tile t of this CTA right after bar_a1_free(t-1) (and, DEFER, bar_drain(t-2)), i.e. about one tile ahead, writes it -
// or -1 when none is left - into tile_slot[t & 1] and arrives on bar_tile[t & 1].  The other builder warps and the loader wait on bar_tile;
// the issuer and the epilogue warps read the slot after bar_a1_ready(t) / bar_prow(t), which the builders arrive on also for the -1 (then
// without an operand) so that every role leaves its loop at the same t.  No waiter is overtaken by two phase completions, and the slot is
// not rewritten before every reader of tile t has read it: bar_tile[t & 1] / tile_slot[t & 1] next change for tile t+2, after builder warp 0
// has seen bar_a1_free(t+1) - the issuer has then taken tile t+1 (so it read slot t), the loader has streamed the layer-1 weights of tile
// t+1 (so it passed its bar_tile(t) wait), and the other builder warps have arrived on bar_a1_ready(t+1) (so they passed theirs).  The
// epilogue warps read slot t before their drain of tile t: DEFER, warp 0 also waits for bar_drain(t) first; non-deferred, it has waited for
// bar_alpha(t) one iteration earlier (finish_sigma).  bar_a1_ready / bar_prow keep their previous arguments; the -1 is their last phase.
template <int NSTAGE, bool COOP, bool DEFER, bool O1 = false, int SCHED = 0, int PFN = 3, bool UNI = true, bool XF = true>
__global__ void __launch_bounds__(DEFER ? tc8::NTHR_DEFER : tc8::NTHR, 1) k_shade_tc8(ShadeTcParams p) {
    using SmemT = tc8::Smem<NSTAGE, COOP>;
    constexpr int NGRP = tc8::NGRP;
    using namespace tc;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    SmemT& sm = *reinterpret_cast<SmemT*>(smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u));
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    // the issuer's role branch is taken on a warp index that is uniform BY CONSTRUCTION (constant-lane shuffle): ptxas then treats the issuer's
    // code as a uniform region and keeps the MMA operands in uniform registers.  (Only the issuer: with uniform branches for the other
    // roles too, the epilogue code got 40 % slower - 37.0 k vs 30 k cycles per tile, profiles/r02_tc8_experiments.log #12.)
    const int warp_u = UNI ? __shfl_sync(0xffffffffu, tid >> 5, 0) : warp;
    const pnb_query_t& q = p.q;
    const int n_valid = min(q.counters[PNB_QC_N_VALID], p.hbar_cap);
    const int n_quads = p.pack_cnt[0];
    const int n_tiles = (n_quads + 3) >> 2;
    const bool static_sched = (p.dbg_flags & 16) != 0;      // tile t of a CTA = blockIdx.x + t * gridDim.x (A/B against the queue)
    int n_done = 0;                                          // tiles this CTA processed (per-CTA statistics, dbg bit 2)
    constexpr int NEPI_WARPS = tc8::NEPI_WARPS;
    constexpr int W_BUILD = NEPI_WARPS, W_LOAD = W_BUILD + tc8::NBUILD / 32, W_ISSUE = W_LOAD + 1;
    // last epilogue: 16 chunks over the NGRP epilogue warps + 1 builder warp of a quadrant; the builder warp takes group 0
    constexpr int NG4 = NGRP + 1, NCH4_B = (16 + NG4 - 1) / NG4, NCH4_E = 16 / NG4;
    static_assert(NCH4_B + NGRP * NCH4_E == 16, "last-epilogue chunk split");

    if (tid == 0) {
        for (int s = 0; s < NSTAGE; ++s) { mbar_init(&sm.bar_full[s], 1); mbar_init(&sm.bar_empty[s], 1); }
        mbar_init(&sm.bar_a1_ready, tc8::NBUILD / 32);              // one arrive per builder warp
        mbar_init(&sm.bar_a1_free, 1);
        mbar_init(&sm.bar_acc_full, 1);
        mbar_init(&sm.bar_final, 1);
        mbar_init(&sm.bar_alpha, NEPI_WARPS);
        mbar_init(&sm.bar_drain, NEPI_WARPS + tc8::NBUILD / 32);     // one arrive per warp that reads the layer-4 accumulator
        for (int c = 0; c < 8; ++c) mbar_init(&sm.bar_kblk[c], 4 * 2);   // 4 quadrant warps x 2 chunks of 16 columns, one arrive per warp
        mbar_init(&sm.bar_prow[0], tc8::NBUILD / 32);
        mbar_init(&sm.bar_prow[1], tc8::NBUILD / 32);
        mbar_init(&sm.bar_tile[0], 1);
        mbar_init(&sm.bar_tile[1], 1);
        mbar_fence_init();
        if (blockIdx.x == 0 && q.counters[PNB_QC_N_VALID] > p.hbar_cap) atomicExch(p.err, 9);
    }
    for (int i = tid; i < 4 * 256; i += (int)blockDim.x) {
        if (i < 3 * 256) sm.bias[i >> 8][i & 255] = __ldg(p.bias[1 + (i >> 8)] + (i & 255));
        else sm.wa[i - 3 * 256] = __ldg(p.wa + (i - 3 * 256));
    }
    if (warp == W_ISSUE) tmem_alloc<512>(&sm.tmem_base);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tP = sm.tmem_base, tQ = sm.tmem_base + 256u;
    const long long _tk0 = clock64();
    // in-kernel cycle accounting of block 0 (dbg bit 0, tools/tc_profile.py PNB_PROF=1): TW(slot, wait) adds the cycles a role spends
    // in a wait, TB(slot) the cycles since the previous mark of this thread; off in production (a kernel-parameter flag)
    const bool prof = (p.dbg_flags & 1) && blockIdx.x == 0 && (warp == 0 || warp == W_BUILD || warp == W_LOAD || warp == W_ISSUE);
    long long _tm = _tk0;
#define TW(slot, expr) [&]() { if (!prof) return (expr); const long long _t0 = clock64(); const bool _r = (expr); _tm = clock64(); if (lane == 0) prof_add(p, slot, _tm - _t0); return _r; }()
#define TB(slot) do { if (prof) { const long long _t1 = clock64(); if (lane == 0) prof_add(p, slot, _t1 - _tm); _tm = _t1; } } while (0)

    if (warp_u >= W_LOAD) {          // (uniform branch: see warp_u)
        if (DEFER) reg_dec<tc8::REG_CTRL>();
    }
    if (warp_u == W_ISSUE) {
        // ============================================================ MMA issuer (whole warp, warp-uniform; one commit per K block)
        // every value the MMA operands are computed from is made uniform BY CONSTRUCTION (uni32 / uni, umma.cuh)
        const bool prof = (p.dbg_flags & 1) && blockIdx.x == 0;      // (shadows the per-role flag: this one is provably uniform)
        auto uni32 = [](uint32_t x) -> uint32_t { return UNI ? pnb::uni32(x) : x; };
        auto uni = [](bool b) -> bool { return UNI ? pnb::uni(b) : b; };
        const uint32_t idesc = make_idesc_bf16(128, 256);
        const uint32_t hiw = desc_hi<LAYOUT>(), xe_hiw = (256u >> 4) | (1u << 14);
        const uint32_t b0_lo = uni32(desc_lo<LAYOUT>(smem_u32(sm.b[0])));
        const uint32_t ahi_lo = uni32(desc_lo<LAYOUT>(smem_u32(sm.a_hi))), alo_lo = uni32(desc_lo<LAYOUT>(smem_u32(sm.a_lo)));
        const uint32_t xeh_lo0 = uni32(desc_lo<LAYOUT_NONE>(smem_u32(sm.xe_hi[0]))), xel_lo0 = uni32(desc_lo<LAYOUT_NONE>(smem_u32(sm.xe_lo[0])));
        const uint32_t uP = uni32(sm.tmem_base), uQ = uP + 256u;
        constexpr uint32_t KADV = kstep_adv16<LAYOUT>();
        uint32_t s = 0, ph = 0, c_acc = 0, c_pack = 0;
        bool ok = true;
        for (int t = 0; ok; ++t) {
            if (!uni(TW(3, mbar_wait(&sm.bar_a1_ready, (uint32_t)t & 1u, p.err, 93)))) { ok = false; break; }
            if ((int)uni32((uint32_t)sm.tile_slot[t & 1]) < 0) break;           // no tile left (the builders' end signal)
            const uint32_t xeh_lo = xeh_lo0 + (uint32_t)(t & 1) * (XE >> 4), xel_lo = xel_lo0 + (uint32_t)(t & 1) * (XE >> 4);
            for (int l = 0; l < 4 && ok; ++l) {
                const uint32_t acc = (l & 1) ? uP : uQ;
                const uint32_t ab = (l & 1) ? uQ : uP;
                if (!XF) {
                    if (l > 0) { if (!uni(TW(1, mbar_wait(&sm.bar_acc_full, c_acc & 1u, p.err, 92)))) { ok = false; break; } ++c_acc; }
                    else if (t > 0) { if (!uni(TW(2, mbar_wait(&sm.bar_final, (uint32_t)(t - 1) & 1u, p.err, 92)))) { ok = false; break; } }
                }
                if (l == 1 && t > 0) { if (!uni(TW(4, mbar_wait(&sm.bar_drain, (uint32_t)(t - 1) & 1u, p.err, 94)))) { ok = false; break; } }
                tc_fence_after();
                const int nkb = l == 0 ? tc8::NKB1 : nkb_of(l);
                for (int kk = 0; kk < nkb && ok; ++kk) {
                    const int kb = (XF && l == 2) ? (kk == 0 ? 8 : kk - 1) : kk;          // XF: layer 3 starts with its extras K block
                    const bool need_chunks = (l >= 1 && kb < 8);
                    uint64_t* cb0 = need_chunks ? &sm.bar_kblk[kb] : &sm.bar_full[s];
                    const uint32_t cp0 = need_chunks ? (c_pack & 1u) : ph;
                    TB(7);
                    if (!uni(mbar_try_wait2(&sm.bar_full[s], ph, cb0, cp0))) {
                        if (need_chunks && !uni(TW(5, mbar_wait(cb0, cp0, p.err, 95)))) { ok = false; break; }
                        if (!uni(TW(6, mbar_wait(&sm.bar_full[s], ph, p.err, 96)))) { ok = false; break; }
                    }
                    tc_fence_after();
                    const uint32_t bh = b0_lo + s * (uint32_t)(tc8::STAGE >> 4), bl = bh + (uint32_t)(IMG >> 4);
                    if (l == 0) {
                        const uint32_t akb_hi = ahi_lo + (uint32_t)kb * (ABLK >> 4), akb_lo = alo_lo + (uint32_t)kb * (ABLK >> 4);
                        mma_ss2_w(acc, akb_hi, hiw, bh, hiw, idesc, kb ? 1u : 0u);
                        mma_ss2_w(acc, akb_lo, hiw, bh, hiw, idesc, 1u);
                        mma_ss2_w(acc, akb_hi + KADV, hiw, bh + KADV, hiw, idesc, 1u);
                        mma_ss2_w(acc, akb_lo + KADV, hiw, bh + KADV, hiw, idesc, 1u);
                        mma_ss2_w(acc, akb_hi, hiw, bl, hiw, idesc, 1u);
                        mma_ss2_w(acc, akb_hi + KADV, hiw, bl + KADV, hiw, idesc, 1u);
                    } else if (kb == 8) {
                        mma_ss2_w(acc, xeh_lo, xe_hiw, bh, hiw, idesc, kk ? 1u : 0u);
                        mma_ss2_w(acc, xel_lo, xe_hiw, bh, hiw, idesc, 1u);
                        mma_ss2_w(acc, xeh_lo, xe_hiw, bl, hiw, idesc, 1u);
                    } else {
                        const uint32_t tcol = ab + (uint32_t)(kb * 32);
                        mma_ts2_w(acc, tcol, bh, hiw, idesc, kk ? 1u : 0u);
                        mma_ts2_w(acc, tcol + 8u, bh, hiw, idesc, 1u);
                        mma_ts2_w(acc, tcol + 16u, bh + KADV, hiw, idesc, 1u);
                        mma_ts2_w(acc, tcol + 24u, bh + KADV, hiw, idesc, 1u);
                        mma_ts2_w(acc, tcol, bl, hiw, idesc, 1u);
                        mma_ts2_w(acc, tcol + 16u, bl + KADV, hiw, idesc, 1u);
                    }
                    mma_commit_w(&sm.bar_empty[s]);
                    if (++s == (uint32_t)NSTAGE) { s = 0; ph ^= 1u; }
                }
                if (!ok) break;
                if (l >= 1) ++c_pack;
                mma_commit_w(l < 3 ? &sm.bar_acc_full : &sm.bar_final);
                if (l == 0) mma_commit_w(&sm.bar_a1_free);
            }
        }
    } else if (warp == W_LOAD) {
        // ============================================================ weight ring: one K block (hi + lo image, 32 KB) per stage
        if (lane == 0) {
            uint32_t s = 0, ph = 0;
            bool ok = true;
            for (int t = 0; ok; ++t) {
                // tile t exists?  (published by builder warp 0 right after it took the tile, a layer or more ahead of the ring)
                if (!mbar_wait(&sm.bar_tile[t & 1], (uint32_t)(t >> 1) & 1u, p.err, 106) || sm.tile_slot[t & 1] < 0) break;
                for (uint32_t j = 0; j < (uint32_t)tc8::STAGES_PER_TILE; ++j) {
                    if (!TW(0, mbar_wait(&sm.bar_empty[s], ph ^ 1u, p.err, 91))) { ok = false; break; }
                    uint32_t blk = j < (uint32_t)tc8::NKB1 ? (uint32_t)tc8::KB1_FIRST + j : 9u + (j - (uint32_t)tc8::NKB1);
                    // XF: layer 3 (stages NKB1 + 8 .. NKB1 + 16 of a tile, weight blocks 17 .. 25) takes its extras block (25) FIRST
                    if (XF && j >= (uint32_t)tc8::NKB1 + 8u && j < (uint32_t)tc8::NKB1 + 17u) blk = j == (uint32_t)tc8::NKB1 + 8u ? 25u : blk - 1u;
                    if (p.dbg_no_weights) mbar_arrive(&sm.bar_full[s]);
                    else {
                        mbar_arrive_expect_tx(&sm.bar_full[s], tc8::STAGE);
                        const unsigned char* src = p.wimg + (size_t)blk * tc8::STAGE;
                        bulk_g2s(sm.b[s], src, IMG, &sm.bar_full[s]);
                        bulk_g2s(sm.b[s] + IMG, src + IMG, IMG, &sm.bar_full[s]);
                    }
                    if (++s == (uint32_t)NSTAGE) { s = 0; ph ^= 1u; }
                }
            }
        }
    } else if (warp > W_ISSUE) {
        // (DEFER: two idle warps complete the control warpgroup)
    } else if (warp >= W_BUILD) {
        // ============================================================ builders: one warp per quadrant, lane = row; the same warps run
        // chunk group 0 of the last epilogue of the previous tile
        if (DEFER) reg_inc<tc8::REG_BUILD>();
        const int qw = warp - W_BUILD, row = qw * 32 + lane;
        const uint32_t tlane = (uint32_t)(qw * 32) << 16;
        bool ok = true;
        // sigma of a tile = softplus(alpha dot product - 1) summed over the rows of a sample; the dot product is this warp's partial sum + the
        // epilogue warps' (bar_alpha), added in a fixed order
        const float ba = __ldg(p.ba);
        auto finish_sigma = [&](int tf, float apart, float wrow, int st, bool swrite, int sidx) -> bool {
            if (!TW(12, mbar_wait(&sm.bar_alpha, (uint32_t)tf & 1u, p.err, 100))) return false;
            float a = apart;
#pragma unroll
            for (int gq = 0; gq < NGRP; ++gq) a += sm.alpha_part[tf & 1][gq][row];          // fixed order: deterministic
            a += ba - 1.0f;
            const float sp = a > 20.f ? a : log1pf(expf(a));
            const float zz = O1 ? sp : seg_scan8(sp * wrow, lane, st);      // (order 1: see k_shade_tc7)
            if (swrite) p.sigma[sidx] = zz;
            return true;
        };
        float pd_apart = 0.f, pd_wrow = 0.f;          // DEFER: this warp's share of the tile drained one iteration ago (sigma still to be finished)
        int pd_st = 0, pd_sidx = 0;
        bool pd_sw = false;
        int t = 0;
        for (;; ++t) {
            if (t > 0 && !TW(8, mbar_wait(&sm.bar_a1_free, (uint32_t)(t - 1) & 1u, p.err, 97))) { ok = false; break; }
            // DEFER: the per-tile slots (tile_slot / qhead / qfirst / qtotal / wc, parity t & 1) were last read when tile t-2 was drained
            if (DEFER && t > 1 && !mbar_wait(&sm.bar_drain, (uint32_t)(t - 2) & 1u, p.err, 103)) { ok = false; break; }
            int tile;                                     // this CTA's tile t, -1: none left
            if (qw == 0) {
                int v = 0;
                if (lane == 0) {
                    v = static_sched ? (int)blockIdx.x + t * (int)gridDim.x : atomicAdd(p.tile_ctr, 1);
                    if (v >= n_tiles) v = -1;
                    sm.tile_slot[t & 1] = v;
                    mbar_arrive(&sm.bar_tile[t & 1]);
                }
                tile = __shfl_sync(0xffffffffu, v, 0);
            } else {
                if (!mbar_wait(&sm.bar_tile[t & 1], (uint32_t)(t >> 1) & 1u, p.err, 105)) { ok = false; break; }
                tile = sm.tile_slot[t & 1];
            }
            if (tile < 0) {                               // end: wake the issuer and the epilogue warps, which read the slot
                if (lane == 0) { mbar_arrive(&sm.bar_a1_ready); mbar_arrive(&sm.bar_prow[t & 1]); }
            } else {
                const int qd = tile * 4 + qw;
                uint32_t first = 0, nsamp = 0;
                if (qd < n_quads) { first = p.quad_first[qd]; nsamp = p.quad_first[qd + 1] - first; }
                const int c = lane < (int)nsamp ? (int)p.vcnt[first + lane] : 0;
                int incl = c;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += v; }
                const uint32_t head = __reduce_or_sync(0xffffffffu, lane < (int)nsamp ? (1u << (incl - c)) : 0u);
                const int total = __shfl_sync(0xffffffffu, incl, 31);
                const QuadRow qr = quad_row(head, total, lane);
                const int cj = __shfl_sync(0xffffffffu, c, qr.j);
                if (lane == 0) { sm.qhead[t & 1][qw] = head; sm.qfirst[t & 1][qw] = first; sm.qtotal[t & 1][qw] = (uint32_t)total; }
                const int pvi = qr.live ? (int)p.vorder[first + qr.j] : -1;
                build_pair_frozen(sm, p, t, row, n_valid, pvi, lane - qr.st, qr.st, qr.live ? cj : 1);
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) { mbar_arrive(&sm.bar_a1_ready); mbar_arrive(&sm.bar_prow[t & 1]); }
                TB(9);
            }
            // DEFER: sigma of tile t-2 (drained one iteration ago; the epilogue warps finished it in gap C of tile t-1).  This wait must come
            // BEFORE this warp's arrival on bar_drain for tile t-1 below: the epilogue warps publish tile t-1 (the next bar_alpha phase) only
            // after that drain barrier, so this waiter can never be overtaken by two phase completions.
            if (DEFER && t > 1 && !finish_sigma(t - 2, pd_apart, pd_wrow, pd_st, pd_sw, pd_sidx)) { ok = false; break; }
            if (t > 0) {
                const int tf = t - 1;
                if (!TW(10, mbar_wait(&sm.bar_final, (uint32_t)tf & 1u, p.err, 99))) { ok = false; break; }
                tc_fence_after();
                const QuadRow qr = quad_row(sm.qhead[tf & 1][qw], (int)sm.qtotal[tf & 1][qw], lane);
                const int sidx = qr.live ? (int)p.vorder[sm.qfirst[tf & 1][qw] + qr.j] : 0;
                const bool swrite = qr.is_end && sidx < n_valid;
                const float wrow = sm.wc[tf & 1][row];
                const float apart = last_chunks_packed<NG4, NCH4_B, true, O1>(p, sm.bias[2], sm.wa, tP + tlane, 0, wrow, qr.st, swrite, sidx, lane, &sm.bar_drain);
                TB(11);
                if (!DEFER) {
                    if (!finish_sigma(tf, apart, wrow, qr.st, swrite, sidx)) { ok = false; break; }
                } else {
                    // the epilogue warps finish tile tf under tile tf+1: its sigma is completed in the next iteration
                    pd_apart = apart; pd_wrow = wrow; pd_st = qr.st; pd_sw = swrite; pd_sidx = sidx;
                }
            }
            if (tile < 0) break;
        }
        if (DEFER && ok && t > 0) finish_sigma(t - 1, pd_apart, pd_wrow, pd_st, pd_sw, pd_sidx);
    } else {
        // ============================================================ epilogue warps
        const int quad = warp & 3, grp = warp >> 2;
        const int erow = quad * 32 + lane;
        const uint32_t tlane = (uint32_t)(quad * 32) << 16;
        if (DEFER) reg_inc<tc8::REG_EPI>();
        uint32_t n_acc = 0;
        bool ok = true;
        // DEFER: this warp's chunks of the previous tile's layer-4 accumulator, held in registers and worked off in the gaps of this tile
        uint32_t hv[DEFER ? NCH4_E : 1][16];
        float d_wrow = 0.f, d_apart = 0.f;
        int d_st = 0, d_sidx = 0;
        bool d_sw = false;
        auto held = [&](auto first, auto count) {          // chunks [first, first + count) of the held tile (compile-time indices: registers)
            if constexpr (DEFER) {
#pragma unroll
                for (int i = decltype(first)::value; i < decltype(first)::value + decltype(count)::value; ++i)
                    last_chunk_from_regs<O1>(p, sm.bias[2], sm.wa, 16 * (1 + grp + NG4 * i), hv[i], d_wrow, d_st, d_sw, d_sidx, lane, d_apart);
            }
        };
        auto held_done = [&](int tf) -> bool {             // the held tile is finished: publish this warp's alpha partial sum
            // alpha_part[tf & 1] last held tile tf-2, which the builder warps read before they drained tile tf-1
            if (!mbar_wait(&sm.bar_drain, (uint32_t)tf & 1u, p.err, 104)) return false;
            sm.alpha_part[tf & 1][grp][erow] = d_apart;
            __syncwarp();
            if (lane == 0) mbar_arrive(&sm.bar_alpha);
            return true;
        };
        static_assert(!DEFER || NCH4_E == 5, "the deferred schedules split 5 held chunks");
        constexpr int GA = SCHED == 0 ? 2 : SCHED == 1 ? 1 : 0, GB = 2, GC = SCHED == 2 ? 2 : 1, GD = 5 - GA - GB - GC;
        using I0 = std::integral_constant<int, 0>;
        using NA = std::integral_constant<int, GA>; using NB_ = std::integral_constant<int, GB>; using NC = std::integral_constant<int, GC>;
        using ND = std::integral_constant<int, GD>; using NR = std::integral_constant<int, 5 - GA>;
        using FB = std::integral_constant<int, GA>; using FC = std::integral_constant<int, GA + GB>; using FD = std::integral_constant<int, GA + GB + GC>;
        int t = 0;
        for (; ok; ++t) {
            if (DEFER && t > 0 && GA > 0) { held(I0{}, NA{}); TB(21); }          // gap A: the layer-1 MMAs of this tile are running
            // ---- layer 1: accumulator + pre[point of this row] (the hoisted 224 inputs and the bias)
            if (!TW(13, mbar_wait(&sm.bar_prow[t & 1], (uint32_t)(t >> 1) & 1u, p.err, 102))) { ok = false; break; }
            if (sm.tile_slot[t & 1] < 0) break;                  // no tile left
            Tc8Pf<COOP, PFN> pfs;
            pfs.init(p.pre, &sm.prow[t & 1][quad * 32], lane);
            pfs.prefetch(grp);                                   // in flight under the wait for the layer-1 MMAs
            if (!TW(14, mbar_wait(&sm.bar_acc_full, n_acc & 1u, p.err, 98))) { ok = false; break; }
            ++n_acc;
            tc_fence_after();
            tc8_epi_layer<true, COOP>(sm, tQ + tlane, grp, nullptr, pfs, sm.xpose[COOP ? warp : 0]);
            TB(15);
            // ---- layers 2, 3
            for (int l = 1; l < 3 && ok; ++l, ++n_acc) {
                if (DEFER && t > 0) {                       // gaps B, C: the layer-2 / layer-3 MMAs are running
                    if (l == 1) held(FB{}, NB_{});
                    else { held(FC{}, NC{}); if (GD == 0 && !held_done(t - 1)) { ok = false; break; } }
                    TB(21);
                }
                if (!TW(16, mbar_wait(&sm.bar_acc_full, n_acc & 1u, p.err, 98))) { ok = false; break; }
                tc_fence_after();
                tc8_epi_layer<false, COOP>(sm, ((l & 1) ? tP : tQ) + tlane, grp, sm.bias[l - 1], pfs, nullptr);
                TB(17);
            }
            if (!ok) break;
            if (DEFER && t > 0 && GD > 0) {                 // gap D: the layer-4 MMAs are running
                held(FD{}, ND{});
                if (!held_done(t - 1)) { ok = false; break; }
                TB(21);
            }
            {   // this warp's share of the LAST epilogue (chunk groups 1..NGRP of NGRP+1; the builder warps take group 0)
                if (!TW(18, mbar_wait(&sm.bar_final, (uint32_t)t & 1u, p.err, 101))) { ok = false; break; }
                tc_fence_after();
                const QuadRow qr = quad_row(sm.qhead[t & 1][quad], (int)sm.qtotal[t & 1][quad], lane);
                const int sidx = qr.live ? (int)p.vorder[sm.qfirst[t & 1][quad] + qr.j] : 0;
                if constexpr (!DEFER) {
                    const float apart = last_chunks_packed<NG4, NCH4_E, true, O1>(p, sm.bias[2], sm.wa, tP + tlane, 1 + grp, sm.wc[t & 1][erow], qr.st, qr.is_end && sidx < n_valid, sidx,
                                                                              lane, &sm.bar_drain);
                    sm.alpha_part[t & 1][grp][erow] = apart;
                    __syncwarp();
                    TB(19);
                    if (lane == 0) mbar_arrive(&sm.bar_alpha);
                } else {
                    // drain only: accumulator -> registers, release the TMEM region; the arithmetic happens in the gaps of the next tile
#pragma unroll
                    for (int i = 0; i < NCH4_E; ++i) tmem_ld16(tP + tlane + (uint32_t)(16 * (1 + grp + NG4 * i)), hv[i]);
                    d_wrow = sm.wc[t & 1][erow]; d_st = qr.st; d_sidx = sidx; d_sw = qr.is_end && sidx < n_valid; d_apart = 0.f;
                    tmem_ld_wait();
#pragma unroll
                    for (int i = 0; i < NCH4_E; ++i) pin16(hv[i]);        // the values exist from here on (tcgen05.ld is asynchronous up to the wait)
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&sm.bar_drain);
                    TB(19);
                }
            }
        }
        if (DEFER && ok && t > 0) { held(FB{}, NR{}); held_done(t - 1); }    // (chunks before FB went in gap A of the end iteration)
        n_done = t;
    }
    if (prof && tid == 0) prof_add(p, 20, clock64() - _tk0);
#undef TW
#undef TB
    if (tid == 0 && (p.dbg_flags & 4) && blockIdx.x < 192) {      // per-CTA cycles and SM id; [32 + 192] = number of quadrants
        uint32_t smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        reinterpret_cast<long long*>(p.err)[32 + blockIdx.x] = ((clock64() - _tk0) & 0xffffffffffffll) | ((long long)smid << 48);
        if (blockIdx.x == 0) { reinterpret_cast<long long*>(p.err)[32 + 192] = n_quads; reinterpret_cast<long long*>(p.err)[32 + 193] = n_done; }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == W_ISSUE) tmem_dealloc<512>(sm.tmem_base);
}

// =====================================================================================================================
// Colour branch: packed weight images of colour_branch.{0,2,4} ([128 x 32] bf16 hi / lo per K block) and the kernel parameters.
namespace ctc {
constexpr int IMG = 128 * 64;                 // [128 x 32] bf16 weight image
constexpr int NBLK = 9 + 4 + 4;               // K blocks of the three layers
constexpr int IMGS_PER_TILE = 2 * NBLK;
__host__ __device__ constexpr int nkb_of(int l) { return l == 0 ? 9 : 4; }
__host__ __device__ constexpr int img_base(int l) { return l == 0 ? 0 : l == 1 ? 9 : 13; }
}  // namespace ctc

struct ColorTcParams {
    pnb_query_t q;
    pnb_shade_opts_t o;
    const unsigned char* wimg;      // packed colour_branch.{0,2,4} images
    const float* bias[3];
    const float* w3t;               // colour_branch.6 W^T [128][3]
    const float* b3;
    const float* hbar;
    const float* sigma;
    int hbar_cap;
    float4* sigma_rgb;
    int* err;
};

// =====================================================================================================================
// Colour branch, pipelined.  The pair kernel writes h-bar already split into bf16 hi / lo and laid out as the
// tcgen05 A-operand blocks of this kernel: per 128 consecutive valid samples 8 K-blocks x {hi, lo} x [128 x 32]
// (interleaved core-matrix layout) = one contiguous 128 KB region.  So the layer-1 operand is ONE bulk copy (TMA engine)
// per tile - no builder warps, no register traffic - issued as soon as the previous tile's layer-1 MMAs have completed,
// and it lands under that tile's layers 2-3.  Same TMEM role ping-pong / in-place accumulator->operand conversion and
// chunk-granular hand-off as the pair kernel; two accumulator sets (tile parity) so a tile's final epilogue
// (128 -> 3 on CUDA cores + sigmoid) runs under the next tile's layer 1.  One tcgen05.commit per K block.
//   layer 1: A smem (8 K-blocks h-bar + 1 K-block PE(view)), acc X      layer 2: A = X, acc Y      layer 3: A = Y, acc X
//   X = 256*(t&1), Y = X + 128 (TMEM columns)
// Warps (480 threads): 0-7 epilogue (quadrant = w & 3, chunk group = w >> 2), 8-11 PE(view) builders (thread = row),
// 12 operand loader, 13 weight loader, 14 issuer (whole warp, warp-uniform).
namespace ctc2 {
constexpr int NEPI_WARPS = 8, NGRP = 2, NCH = 8 / NGRP;     // 8 chunks of 16 accumulator columns per layer
constexpr int NEPI = NEPI_WARPS * 32, NTHR = NEPI + 128 + 96;
constexpr int NSTAGE = 4;
constexpr int BLK = 128 * 64;                // [128 x 32] bf16 block (operand block and weight image)
constexpr int NKB = 9 + 4 + 4;               // K blocks per tile
constexpr int TILE_BYTES = 8 * 2 * BLK;      // h-bar operand of one tile in global memory
struct Smem {
    unsigned char a[8][2][BLK];              // layer-1 operand: K block, hi/lo
    unsigned char pe[2][BLK];                // PE(view) K block, hi/lo
    unsigned char b[NSTAGE][2][BLK];         // weight ring: hi / lo image of one K block
    float part[128][4];
    float4 w3[128];                          // colour_branch.6 W^T rows (x, y, z, 0)
    float bias[3][128];                      // colour_branch.{0,2,4} biases
    float b3[4];
    uint64_t bar_full[NSTAGE], bar_empty[NSTAGE], bar_a_full, bar_a_free, bar_pe_ready, bar_acc_full, bar_drain, bar_kblk[4];
    uint32_t tmem_base;
};
__host__ __device__ constexpr int nkb_of(int l) { return l == 0 ? 9 : 4; }
}  // namespace ctc2

__global__ void __launch_bounds__(ctc2::NTHR, 1) k_color_tc2(ColorTcParams p) {
    using namespace ctc2;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    Smem& sm = *reinterpret_cast<Smem*>(smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u));
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const pnb_query_t& q = p.q;
    const int n_valid = min(q.counters[PNB_QC_N_VALID], p.hbar_cap);
    const int n_tiles = (n_valid + 127) / 128;
    const int my_tiles = n_tiles > (int)blockIdx.x ? (n_tiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;
    constexpr int W_PE = NEPI_WARPS, W_LOADA = W_PE + 4, W_LOADW = W_LOADA + 1, W_ISSUE = W_LOADW + 1;

    if (tid == 0) {
        for (int s = 0; s < NSTAGE; ++s) { mbar_init(&sm.bar_full[s], 1); mbar_init(&sm.bar_empty[s], 1); }
        mbar_init(&sm.bar_a_full, 1);
        mbar_init(&sm.bar_a_free, 1);
        mbar_init(&sm.bar_pe_ready, 128);
        mbar_init(&sm.bar_acc_full, 1);
        mbar_init(&sm.bar_drain, NEPI_WARPS);
        for (int c = 0; c < 4; ++c) mbar_init(&sm.bar_kblk[c], 4 * 2);      // 4 quadrant warps x 2 chunks of 16 columns
        mbar_fence_init();
    }
    if (warp == W_ISSUE) tmem_alloc<512>(&sm.tmem_base);
    // the epilogue's small parameters, read as warp-broadcast shared loads
    for (int i = tid; i < 3 * 128; i += NTHR) sm.bias[i >> 7][i & 127] = __ldg(p.bias[i >> 7] + (i & 127));
    for (int i = tid; i < 128; i += NTHR) sm.w3[i] = make_float4(__ldg(p.w3t + 3 * i), __ldg(p.w3t + 3 * i + 1), __ldg(p.w3t + 3 * i + 2), 0.f);
    if (tid < 3) sm.b3[tid] = __ldg(p.b3 + tid);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tbase = sm.tmem_base;

    if (warp == W_LOADA) {
        // ============================================================ layer-1 operand: one 128 KB region per tile
        if (lane == 0) {
            for (int t = 0; t < my_tiles; ++t) {
                const int tile = (int)blockIdx.x + t * (int)gridDim.x;
                if (t > 0 && !mbar_wait(&sm.bar_a_free, (uint32_t)(t - 1) & 1u, p.err, 81)) break;
                mbar_arrive_expect_tx(&sm.bar_a_full, TILE_BYTES);
                const unsigned char* src = reinterpret_cast<const unsigned char*>(p.hbar) + (size_t)tile * TILE_BYTES;
#pragma unroll 1
                for (int c = 0; c < 8; ++c) bulk_g2s(sm.a[c][0], src + (size_t)c * 2 * BLK, 2 * BLK, &sm.bar_a_full);
            }
        }
    } else if (warp == W_LOADW) {
        // ============================================================ weight ring: hi + lo image of one K block per stage
        if (lane == 0) {
            const uint32_t total = (uint32_t)my_tiles * NKB;
            for (uint32_t n = 0; n < total; ++n) {
                const uint32_t s = n & (NSTAGE - 1), ph = (n >> 2) & 1u;
                if (!mbar_wait(&sm.bar_empty[s], ph ^ 1u, p.err, 82)) break;
                mbar_arrive_expect_tx(&sm.bar_full[s], 2 * BLK);
                bulk_g2s(sm.b[s][0], p.wimg + (size_t)(n % NKB) * 2 * BLK, 2 * BLK, &sm.bar_full[s]);
            }
        }
    } else if (warp == W_ISSUE) {
        // ============================================================ MMA issuer (whole warp, warp-uniform)
        const uint32_t idesc = make_idesc_bf16(128, 128);
        const uint32_t hiw = desc_hi<tc::LAYOUT>();
        const uint32_t b0_lo = desc_lo<tc::LAYOUT>(smem_u32(sm.b[0][0]));
        const uint32_t a0_lo = desc_lo<tc::LAYOUT>(smem_u32(sm.a[0][0])), pe_lo = desc_lo<tc::LAYOUT>(smem_u32(sm.pe[0]));
        constexpr uint32_t KADV = kstep_adv16<tc::LAYOUT>(), BADV = BLK >> 4;
        uint32_t n = 0, c_acc = 0, c_pack = 0;
        bool ok = true;
        for (int t = 0; t < my_tiles && ok; ++t) {
            const uint32_t tX = tbase + 256u * (uint32_t)(t & 1), tY = tX + 128u;
            for (int l = 0; l < 3 && ok; ++l) {
                const uint32_t acc = (l == 1) ? tY : tX, ab = (l == 1) ? tX : tY;
                // WAR on tensor memory: the MMAs of the previous layer read this layer's accumulator region as their A operand and must
                // be complete.  Every completion of bar_acc_full is consumed before the commit of the next one is issued (a parity
                // wait overtaken by two completions would never return): layer 3 of the previous tile is consumed inside layer 1,
                // before its last K block (see below); the previous tile's drain here, where it is complete in steady state.
                if (l == 1 && t > 0) {
                    if (!mbar_wait(&sm.bar_drain, (uint32_t)(t - 1) & 1u, p.err, 86)) { ok = false; break; }
                }
                if (l > 0) { if (!mbar_wait(&sm.bar_acc_full, c_acc & 1u, p.err, 83)) { ok = false; break; } ++c_acc; }
                if (l == 0) {
                    if (!mbar_wait(&sm.bar_a_full, (uint32_t)t & 1u, p.err, 84)) { ok = false; break; }
                    if (!mbar_wait(&sm.bar_pe_ready, (uint32_t)t & 1u, p.err, 85)) { ok = false; break; }
                }
                tc_fence_after();
                const int nkb = nkb_of(l);
                for (int kb = 0; kb < nkb && ok; ++kb, ++n) {
                    const uint32_t s = n & (NSTAGE - 1), ph = (n >> 2) & 1u;
                    const bool need_chunks = l >= 1;
                    if (l == 0 && t > 0 && kb == nkb - 1) {      // layer 3 of the previous tile: complete by now (ring depth < 8 K blocks)
                        if (!mbar_wait(&sm.bar_acc_full, c_acc & 1u, p.err, 83)) { ok = false; break; }
                        ++c_acc;
                    }
                    uint64_t* cb0 = need_chunks ? &sm.bar_kblk[kb] : &sm.bar_full[s];
                    const uint32_t cp0 = need_chunks ? (c_pack & 1u) : ph;
                    if (!mbar_try_wait4(&sm.bar_full[s], ph, cb0, cp0, &sm.bar_full[s], ph, cb0, cp0)) {
                        if (need_chunks && !mbar_wait(cb0, cp0, p.err, 87)) { ok = false; break; }
                        if (!mbar_wait(&sm.bar_full[s], ph, p.err, 88)) { ok = false; break; }
                    }
                    tc_fence_after();
                    const uint32_t bh = b0_lo + s * (2 * BADV), bl = bh + BADV;
                    if (l == 0) {
                        const uint32_t ah = (kb < 8) ? a0_lo + (uint32_t)kb * (2 * BADV) : pe_lo, al = ah + BADV;
                        mma_ss2_w(acc, ah, hiw, bh, hiw, idesc, kb ? 1u : 0u);
                        mma_ss2_w(acc, al, hiw, bh, hiw, idesc, 1u);
                        mma_ss2_w(acc, ah + KADV, hiw, bh + KADV, hiw, idesc, 1u);
                        mma_ss2_w(acc, al + KADV, hiw, bh + KADV, hiw, idesc, 1u);
                        mma_ss2_w(acc, ah, hiw, bl, hiw, idesc, 1u);
                        mma_ss2_w(acc, ah + KADV, hiw, bl + KADV, hiw, idesc, 1u);
                    } else {
                        const uint32_t tcol = ab + (uint32_t)(kb * 32);        // in-place packed operand: 16-column chunk = 8 hi | 8 lo
                        mma_ts2_w(acc, tcol, bh, hiw, idesc, kb ? 1u : 0u);
                        mma_ts2_w(acc, tcol + 8u, bh, hiw, idesc, 1u);
                        mma_ts2_w(acc, tcol + 16u, bh + KADV, hiw, idesc, 1u);
                        mma_ts2_w(acc, tcol + 24u, bh + KADV, hiw, idesc, 1u);
                        mma_ts2_w(acc, tcol, bl, hiw, idesc, 1u);
                        mma_ts2_w(acc, tcol + 16u, bl + KADV, hiw, idesc, 1u);
                    }
                    mma_commit_w(&sm.bar_empty[s]);
                }
                if (!ok) break;
                if (l >= 1) ++c_pack;
                mma_commit_w(&sm.bar_acc_full);
                if (l == 0) mma_commit_w(&sm.bar_a_free);
            }
        }
    } else if (warp >= W_PE) {
        // ============================================================ PE(view) K block of the next tile (thread = sample row)
        const int row = (warp - W_PE) * 32 + lane;
        for (int t = 0; t < my_tiles; ++t) {
            const int tile = (int)blockIdx.x + t * (int)gridDim.x;
            if (t > 0 && !mbar_wait(&sm.bar_a_free, (uint32_t)(t - 1) & 1u, p.err, 89)) break;
            const int vi = tile * 128 + row;
            float pe[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) pe[i] = 0.f;
            if (vi < n_valid) {
                const uint32_t s = q.valid_list[vi];
                const int r = (int)(q.samp_ray[s] >> 7);
                float ov[3];
                rot3t(p.o.Rw2c, q.raydir[3 * r], q.raydir[3 * r + 1], q.raydir[3 * r + 2], ov[0], ov[1], ov[2]);
#pragma unroll
                for (int d = 0; d < 3; ++d) {     // ori=True layout: sin block (d*4+j) then cos block
                    float sc[8];
                    pe_doubling<4>(ov[d], sc);
#pragma unroll
                    for (int j = 0; j < 4; ++j) { pe[d * 4 + j] = sc[2 * j]; pe[12 + d * 4 + j] = sc[2 * j + 1]; }
                }
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                uint32_t h[4], l[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) split_bf16x2(pe[8 * c + 2 * i], pe[8 * c + 2 * i + 1], h[i], l[i]);
                const uint32_t off = tile_offset_bytes<tc::LAYOUT>(row, 8 * c);
                *reinterpret_cast<uint4*>(sm.pe[0] + off) = make_uint4(h[0], h[1], h[2], h[3]);
                *reinterpret_cast<uint4*>(sm.pe[1] + off) = make_uint4(l[0], l[1], l[2], l[3]);
            }
            fence_proxy_async();
            mbar_arrive(&sm.bar_pe_ready);
        }
    } else {
        // ============================================================ epilogue warps
        const int quad = warp & 3, grp = warp >> 2;
        const int erow = quad * 32 + lane;
        const uint32_t tlane = (uint32_t)(quad * 32) << 16;
        uint32_t n_acc = 0;
        bool ok = true;
        for (int t = 0; t < my_tiles && ok; ++t) {
            const int tile = (int)blockIdx.x + t * (int)gridDim.x;
            const uint32_t tX = tbase + 256u * (uint32_t)(t & 1), tY = tX + 128u;
            for (int l = 0; l < 3 && ok; ++l, ++n_acc) {
                if (!mbar_wait(&sm.bar_acc_full, n_acc & 1u, p.err, 90)) { ok = false; break; }
                tc_fence_after();
                const uint32_t accb = ((l == 1) ? tY : tX) + tlane;
                const float* bias = sm.bias[l];
                if (l < 2) {
#pragma unroll
                    for (int i = 0; i < NCH; ++i) {
                        const int g = grp + NGRP * i, c0 = 16 * g;
                        uint32_t v[16];
                        tmem_ld16(accb + (uint32_t)c0, v);
                        tmem_ld_wait();
                        uint32_t hh[8], ll[8];
#pragma unroll
                        for (int e = 0; e < 8; ++e) {
                            float2 bb = reinterpret_cast<const float2*>(bias + c0)[e];
                            float y0 = __uint_as_float(v[2 * e]) + bb.x, y1 = __uint_as_float(v[2 * e + 1]) + bb.y;
                            y0 = fmaxf(y0, tc::LEAKY * y0); y1 = fmaxf(y1, tc::LEAKY * y1);
                            split_bf16x2(y0, y1, hh[e], ll[e]);
                        }
                        tmem_st8(accb + (uint32_t)c0, hh);
                        tmem_st8(accb + (uint32_t)c0 + 8u, ll);
                        tmem_st_wait();
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&sm.bar_kblk[g >> 1]);
                    }
                } else {
                    float d0 = 0.f, d1 = 0.f, d2 = 0.f;
#pragma unroll
                    for (int i = 0; i < NCH; ++i) {
                        const int c0 = 16 * (grp + NGRP * i);
                        uint32_t v[16];
                        tmem_ld16(accb + (uint32_t)c0, v);
                        tmem_ld_wait();
#pragma unroll
                        for (int e = 0; e < 16; ++e) {
                            float y = __uint_as_float(v[e]) + bias[c0 + e];
                            y = fmaxf(y, tc::LEAKY * y);
                            const float4 wr = sm.w3[c0 + e];
                            d0 = fmaf(y, wr.x, d0); d1 = fmaf(y, wr.y, d1); d2 = fmaf(y, wr.z, d2);
                        }
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&sm.bar_drain);          // this warp's share of accumulator set X drained
                    if (grp == 1) { sm.part[erow][0] = d0; sm.part[erow][1] = d1; sm.part[erow][2] = d2; }
                    named_bar_sync(1, NEPI);
                    if (grp == 0) {
                        const int vi = tile * 128 + erow;
                        if (vi < n_valid) {
                            const uint32_t s = q.valid_list[vi];
                            float4 o4;
                            o4.x = p.sigma[vi];
                            const float r0 = d0 + sm.part[erow][0] + sm.b3[0];
                            const float r1 = d1 + sm.part[erow][1] + sm.b3[1];
                            const float r2 = d2 + sm.part[erow][2] + sm.b3[2];
                            o4.y = 1.0f / (1.0f + expf(-r0)) * (1.0f + 2.0f * 0.001f) - 0.001f;
                            o4.z = 1.0f / (1.0f + expf(-r1)) * (1.0f + 2.0f * 0.001f) - 0.001f;
                            o4.w = 1.0f / (1.0f + expf(-r2)) * (1.0f + 2.0f * 0.001f) - 0.001f;
                            p.sigma_rgb[s] = o4;
                        }
                    }
                    named_bar_sync(1, NEPI);
                }
            }
        }
    }
    __syncwarp();
    tc_fence_before();
    __syncthreads();
    if (warp == W_ISSUE) tmem_dealloc<512>(sm.tmem_base);
}

}  // namespace pnb

using namespace pnb;

static size_t pack_pairs_bytes() { return (size_t)tc::NBLK_TOTAL * 2 * tc::IMG; }
static size_t pack_color_bytes() { return (size_t)ctc::NBLK * 2 * ctc::IMG; }
extern "C" size_t pnb_mlp_pack_bytes(void) { return pack_pairs_bytes() + pack_color_bytes(); }

// Packs block1/block3 weights (pnb_mlp_t W^T buffers, fp32) into tcgen05 operand images.  Call once per weight version.
extern "C" int pnb_mlp_pack(const pnb_mlp_t* mlp, void* d_out, size_t out_bytes, pnb_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    PNB_REQUIRE(mlp && d_out, PNB_ERR_INVALID, "pnb_mlp_pack: null argument");
    PNB_REQUIRE(out_bytes >= pnb_mlp_pack_bytes(), PNB_ERR_WORKSPACE, "pnb_mlp_pack: buffer too small");
    const int kpad[4] = {288, 256, 272, 256};
    for (int l = 0; l < 4; ++l) {
        int nkb = tc::nkb_of(l);
        int n = nkb * 256 * umma::BK;
        k_pack_weights<<<(n + 255) / 256, 256, 0, stream>>>(mlp->w[l], kpad[l], nkb, 256, (unsigned char*)d_out + (size_t)tc::img_base(l) * 2 * tc::IMG);
    }
    const int ckpad[3] = {288, 128, 128};   // colour_branch.{0,2,4}: W^T [K_pad][128]
    for (int l = 0; l < 3; ++l) {
        int nkb = ctc::nkb_of(l);
        int n = nkb * 128 * umma::BK;
        k_pack_weights<<<(n + 255) / 256, 256, 0, stream>>>(mlp->w[5 + l], ckpad[l], nkb, 128,
                                                            (unsigned char*)d_out + pack_pairs_bytes() + (size_t)ctc::img_base(l) * 2 * ctc::IMG);
    }
    PNB_CHECK_CUDA(cudaGetLastError());
    return PNB_OK;
}

// Hoisted layer-1 table of a frozen point cloud (k_point_pre): d_pre [N][256] fp32.
extern "C" size_t pnb_point_pre_bytes(int N) { return (size_t)(N > 0 ? N : 0) * 256 * sizeof(float); }
extern "C" int pnb_point_pre(const pnb_points_t* pts, const pnb_mlp_t* mlp, float* d_pre, size_t pre_bytes, pnb_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    PNB_REQUIRE(pts && mlp && d_pre, PNB_ERR_INVALID, "pnb_point_pre: null argument");
    PNB_REQUIRE(pre_bytes >= pnb_point_pre_bytes(pts->N), PNB_ERR_WORKSPACE, "pnb_point_pre: buffer too small");
    if (pts->N > 0) k_point_pre<<<(pts->N + 31) / 32, 256, 0, stream>>>(pts->emb, pts->N, mlp->w[0], mlp->b[0], d_pre);
    PNB_CHECK_CUDA(cudaGetLastError());
    return PNB_OK;
}

static size_t pack_sc_max(int cap) { return (size_t)cap / tc7::PACK_S + 3; }
namespace {
struct TcWs {   // carve-up of the caller's workspace (all sizes from max_valid_samples; the kernels read the live counts on the device)
    float* hbar; float* sigma; uint32_t* sc_quads; uint32_t* quad_local; uint32_t* quad_first; uint32_t* vorder; unsigned char* vcntp; int* pack_cnt;
    TcWs(void* ws, size_t ws_bytes, int cap) {
        Carver c(ws, ws_bytes);
        hbar = c.take<float>(((size_t)cap + 127) / 128 * 128 * 256);   // whole 128-sample colour tiles
        sigma = c.take<float>((size_t)cap);
        sc_quads = c.take<uint32_t>(pack_sc_max(cap));
        quad_local = c.take<uint32_t>((size_t)cap + 2);
        quad_first = c.take<uint32_t>((size_t)cap + 2);
        vorder = c.take<uint32_t>((size_t)cap + 2);
        vcntp = c.take<unsigned char>((size_t)cap + 16);
        pack_cnt = c.take<int>(4);                                    // [0] n_quads, [1] tile queue of k_shade_tc8
    }
};
}  // namespace
extern "C" size_t pnb_shade_tc_bytes(int max_valid_samples) {
    const size_t cap = (size_t)max_valid_samples;
    return align_up((cap + 127) / 128 * 128 * 256 * sizeof(float)) + align_up(cap * sizeof(float)) + align_up(pack_sc_max(max_valid_samples) * 4) +
           3 * align_up((cap + 2) * 4) + align_up(cap + 16) + align_up(16) + 256;
}
// diagnostics / tests: device pointers of the row-packing tables inside a workspace laid out for max_valid_samples
extern "C" int pnb_shade_tc_tables(void* ws, size_t ws_bytes, int max_valid_samples, void** vorder, void** vcntp, void** quad_first, void** pack_cnt) {
    PNB_REQUIRE(ws && ws_bytes >= pnb_shade_tc_bytes(max_valid_samples), PNB_ERR_WORKSPACE, "pnb_shade_tc_tables: workspace too small");
    TcWs w(ws, ws_bytes, max_valid_samples);
    if (vorder) *vorder = w.vorder;
    if (vcntp) *vcntp = w.vcntp;
    if (quad_first) *quad_first = w.quad_first;
    if (pack_cnt) *pack_cnt = w.pack_cnt;
    return PNB_OK;
}

// Tensor-core forward: row packing, per-pair MLPs and colour branch on tcgen05 (BF16x3).  ws: >= pnb_shade_tc_bytes.
extern "C" int pnb_shade_forward_tc(const pnb_query_t* q, const pnb_points_t* pts, const pnb_mlp_t* mlp, const void* d_packed,
                                    const float* d_point_pre, const pnb_shade_opts_t* opts, float* d_sigma_rgb, void* ws, size_t ws_bytes,
                                    int max_valid_samples, int flags, int* d_err, pnb_stream_t stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    PNB_REQUIRE(q && pts && mlp && d_packed && opts && d_sigma_rgb && ws && d_err, PNB_ERR_INVALID, "pnb_shade_forward_tc: null argument");
    PNB_REQUIRE(q->K >= 1 && q->K <= PNB_MAX_K, PNB_ERR_UNSUPPORTED, "pnb_shade_forward_tc: K=%d unsupported", q->K);
    PNB_REQUIRE(max_valid_samples > 0, PNB_ERR_INVALID, "pnb_shade_forward_tc: max_valid_samples must be positive");
    PNB_REQUIRE(ws_bytes >= pnb_shade_tc_bytes(max_valid_samples), PNB_ERR_WORKSPACE, "pnb_shade_forward_tc: workspace too small");
    const bool frozen = (flags & PNB_TC_FROZEN) != 0;
    PNB_REQUIRE(!frozen || d_point_pre, PNB_ERR_INVALID, "pnb_shade_forward_tc: PNB_TC_FROZEN needs the table of pnb_point_pre");
    static int configured[64] = {0}, n_sm_of[64] = {0};      // per device of this process (one process per GPU is the norm)
    int dev = 0;
    PNB_CHECK_CUDA(cudaGetDevice(&dev));
    PNB_REQUIRE(dev >= 0 && dev < 64, PNB_ERR_UNSUPPORTED, "pnb_shade_forward_tc: device ordinal %d", dev);
    // interleaved (non-swizzled) operand layout: 128-byte alignment of the carve-out is sufficient
    constexpr size_t kSmemMax = 232448;   // 227 KB opt-in limit per block on sm_100
    const size_t smem_tc7 = sizeof(tc7::Smem) + 128, smem_tc8 = sizeof(tc8::Smem<4, true>) + 128, smem_ctc2 = sizeof(ctc2::Smem) + 128;
    static_assert(sizeof(tc7::Smem) + 128 <= kSmemMax, "v7 shared-memory carve-out exceeds the per-block limit");
    static_assert(sizeof(tc8::Smem<4, true>) + 128 <= kSmemMax, "v8 shared-memory carve-out exceeds the per-block limit");
    static_assert(sizeof(ctc2::Smem) + 128 <= kSmemMax, "colour kernel shared-memory carve-out exceeds the per-block limit");
    static_assert(tc7::NSTAGE == 4, "the v7 issuer assumes a 4-stage ring");
    if (!configured[dev]) {
        PNB_CHECK_CUDA(cudaFuncSetAttribute(k_shade_tc7<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tc7));
        PNB_CHECK_CUDA(cudaFuncSetAttribute(k_shade_tc7<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tc7));
        PNB_CHECK_CUDA(cudaFuncSetAttribute(k_shade_tc8<4, true, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tc8));
        PNB_CHECK_CUDA(cudaFuncSetAttribute(k_shade_tc8<4, true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tc8));
        PNB_CHECK_CUDA(cudaFuncSetAttribute(k_shade_tc8<4, true, true, false, 2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tc8));
        PNB_CHECK_CUDA(cudaFuncSetAttribute(k_shade_tc8<4, true, true, true, 2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_tc8));
        PNB_CHECK_CUDA(cudaFuncSetAttribute(k_color_tc2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_ctc2));
        PNB_CHECK_CUDA(cudaDeviceGetAttribute(&n_sm_of[dev], cudaDevAttrMultiProcessorCount, dev));
        configured[dev] = 1;
    }
    const int n_sm = n_sm_of[dev];
    TcWs w(ws, ws_bytes, max_valid_samples);
    ShadeTcParams p;
    p.q = *q; p.pts = *pts; p.o = *opts; p.wimg = (const unsigned char*)d_packed;
    for (int l = 0; l < 4; ++l) p.bias[l] = mlp->b[l];
    p.wa = mlp->w[4];
    p.ba = mlp->b[4];
    p.hbar = w.hbar; p.sigma = w.sigma; p.hbar_cap = max_valid_samples; p.err = d_err;
    p.dbg_no_weights = (flags & PNB_TC_DBG_NO_WEIGHTS) ? 1 : 0;
    p.dbg_flags = (flags >> 8) & 0xff;
    p.vcnt = w.vcntp; p.vorder = w.vorder; p.quad_first = w.quad_first; p.pack_cnt = w.pack_cnt;
    p.tile_ctr = w.pack_cnt + 1;
    p.pre = d_point_pre;
    p.hbar_fmt = 1;                                           // h-bar in the colour kernel's operand format
    if (flags & PNB_TC_PAIRS) {
        const int cap = max_valid_samples, n_sc = (int)pack_sc_max(cap);
        k_pack_quads<<<(n_sc + 7) / 8, 256, 0, stream>>>(p.q, cap, w.sc_quads, w.quad_local, w.vorder, w.vcntp, (float4*)d_sigma_rgb);
        k_pack_scan<<<1, 1024, 0, stream>>>(p.q, cap, w.sc_quads, w.quad_first, w.pack_cnt);
        k_pack_place<<<(cap + 255) / 256, 256, 0, stream>>>(p.q, cap, w.sc_quads, w.quad_local, w.quad_first);
        if (frozen) {
            // 4-stage weight ring + coalesced gather of the hoisted table (variants measured: profiles/r02_tc8_experiments.log)
            // deferred last epilogue (default; dbg bit 3 = the non-deferred form, bit-identical results)
            // (schedules / prefetch depths measured: profiles/r02_tc8_experiments.log #10)
            const bool o1 = opts->agg_intrp_order == 1;          // a compile-time flag of the kernels (see last_chunks_packed)
            if (p.dbg_flags & 8) {                                // non-deferred last epilogue
                if (o1) k_shade_tc8<4, true, false, true><<<n_sm, tc8::NTHR, smem_tc8, stream>>>(p);
                else k_shade_tc8<4, true, false, false><<<n_sm, tc8::NTHR, smem_tc8, stream>>>(p);
            } else if (o1) k_shade_tc8<4, true, true, true, 2, 2><<<n_sm, tc8::NTHR_DEFER, smem_tc8, stream>>>(p);
            else k_shade_tc8<4, true, true, false, 2, 2><<<n_sm, tc8::NTHR_DEFER, smem_tc8, stream>>>(p);
        }
        else if (opts->agg_intrp_order == 1) k_shade_tc7<true><<<n_sm, tc7::NTHR, smem_tc7, stream>>>(p);
        else k_shade_tc7<false><<<n_sm, tc7::NTHR, smem_tc7, stream>>>(p);
    }
    if (flags & PNB_TC_COLOR) {
        ColorTcParams ct;
        ct.q = *q; ct.o = *opts; ct.wimg = (const unsigned char*)d_packed + pack_pairs_bytes();
        for (int i = 0; i < 3; ++i) ct.bias[i] = mlp->b[5 + i];
        ct.w3t = mlp->w[8]; ct.b3 = mlp->b[8];
        ct.hbar = w.hbar; ct.sigma = w.sigma; ct.hbar_cap = max_valid_samples; ct.sigma_rgb = (float4*)d_sigma_rgb; ct.err = d_err;
        k_color_tc2<<<n_sm, ctc2::NTHR, smem_ctc2, stream>>>(ct);
    }
    PNB_CHECK_CUDA(cudaGetLastError());
    return PNB_OK;
}
