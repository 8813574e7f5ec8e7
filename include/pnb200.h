/*
 * pnb200 -- C ABI of the B200-native Point-NeRF per-ray hot path (libpnb200.so).
 *
 * Plain C: pointers, sizes, a CUDA stream handle.  No torch types, no hidden allocations: every
 * device buffer (inputs, outputs, workspaces) is owned by the caller; *_bytes() functions report the
 * workspace sizes.  Every entry point returns 0 on success or a negative pnb_status; the text of the
 * last error of the calling thread is available through pnb_last_error().  Nothing here synchronises
 * the stream unless its comment says so.
 *
 * Each entry point names the reference interface it replaces
 * (paths are into the reference tree, Xharlie/pointnerf):
 *   pnb_grid_build        models/neural_points/cuda/query_worldcoords.cu:18-162   (claim_occ, map_coor2occ,
 *                         fill_occ2pnts) + the allocations of :314-319 -- run ONCE per point-cloud version
 *                         instead of once per ray chunk.
 *   pnb_query             query_worldcoords.cu:165-302,381-391 (mask_raypos, first-SR selection,
 *                         get_shadingloc, query_neigh_along_ray_layered) and the ray generation of
 *                         models/rendering/diff_ray_marching.py:349-392 (positions are formed in-kernel from
 *                         campos + raydir * t[d], never materialised).
 *   pnb_query_export      query_worldcoords.cu:425-432 + models/neural_points/point_query.py:95-98: dense
 *                         [R',SR,K] / [R',SR,3] tensors in the reference layout for the drop-in
 *                         lighting_fast_querier.query_points().
 *   pnb_shade_forward     models/neural_points/neural_points.py:706-717 (gather),
 *                         models/aggregators/point_aggregators.py:727-814,488-644 (weights, PE, MLPs).
 *   pnb_composite_forward models/neural_points_volumetric_model.py:271-305, models/rendering/
 *                         diff_ray_marching.py:508-554 (ray distances, alpha compositing) and :87-123
 *                         (fill_invalid: results are written at full R).
 *   pnb_shade_backward / pnb_composite_backward: the autograd of the above (loss.backward() in
 *                         models/mvs_points_volumetric_model.py:98-118).
 *   pnb_probe_maps / pnb_probe_select: the probe pass of point growing (run/train_ft.py:417-530 with
 *                         models/neural_points_volumetric_model.py:331-351), one call each per frame.
 */
#ifndef PNB200_H
#define PNB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* pnb_stream_t; /* cudaStream_t */

typedef enum {
    PNB_OK = 0,
    PNB_ERR_INVALID = -1,    /* bad argument (message in pnb_last_error) */
    PNB_ERR_CUDA = -2,       /* CUDA runtime error */
    PNB_ERR_WORKSPACE = -3,  /* workspace too small */
    PNB_ERR_UNSUPPORTED = -4 /* option value outside the implemented hot-path configuration */
} pnb_status;

#define PNB_MAX_K 8    /* query_worldcoords.cu:14 (#define KN 8) */
#define PNB_MAX_SR 128 /* sample slots per ray */
#define PNB_FEAT 32    /* point_features_dim of every shipped script */

/* counters written by pnb_grid_build (device int32[16], copied to host on request) */
enum {
    PNB_GC_N_OCC = 0,      /* occupied voxels */
    PNB_GC_MAX_PTS = 1,    /* max points in one voxel (before the P cap) */
    PNB_GC_OVERFLOW_O = 2, /* n_occ > max_o  (reference: random reservoir; here: all voxels kept, flagged) */
    PNB_GC_OVERFLOW_P = 3, /* some voxel > P (reference: random reservoir; here: first P by index, flagged) */
    PNB_GC_N_INRANGE = 4,  /* points inside the grid */
    PNB_GC_SLOT0_CELL = 5, /* linear index of the voxel that holds the lowest-index in-range point (Q1) */
    PNB_GC_FIRST_PT = 6,   /* that point's index */
    /* bounding box of the dilated occupancy (occ_bits), inclusive voxel coordinates; empty (lo > hi) when no point is in range.
     * pnb_query marches only the steps of a ray that can reach it (a wider box is always safe, a narrower one is not). */
    PNB_GC_BOX_X0 = 7,
    PNB_GC_BOX_Y0 = 8,
    PNB_GC_BOX_Z0 = 9,
    PNB_GC_BOX_X1 = 10,
    PNB_GC_BOX_Y1 = 11,
    PNB_GC_BOX_Z1 = 12,
    /* squared radius (fp32 bits) of a sphere about the grid centre lo + dim * svs / 2 that holds every voxel of occ_bits; the march
     * also skips the steps outside it */
    PNB_GC_SPHERE_R2 = 13
};

/* counters written by pnb_query (device int32[16]) */
enum {
    PNB_QC_N_CAND = 0,   /* candidate samples (occupied march steps kept, <= SR per ray) */
    PNB_QC_N_VALID = 1,  /* samples with >= 1 neighbour (S_v) */
    PNB_QC_N_PAIRS = 2,  /* valid (sample,k) pairs (P_v) */
    PNB_QC_R1 = 3,       /* rays with >= 1 candidate sample */
    PNB_QC_R2 = 4,       /* rays with >= 1 neighbour (R') */
    PNB_QC_OVERFLOW = 5  /* 1 if the candidate capacity was exceeded (results truncated) */
};

/* The voxel grid (device pointers into the caller's buffer) -- plain data, filled by pnb_grid_build. */
typedef struct {
    float lo[3];          /* grid origin = ranges[0:3] of point_query.py:64-66 */
    float svs[3];         /* scaled voxel size = vsize * vscale */
    int32_t dim[3];       /* scaled_vdim */
    int32_t P;            /* per-voxel point cap */
    int32_t parity_slot0; /* 1: replicate query_worldcoords.cu:147 (slot-0 voxel holds no points) */
    int32_t n_points;     /* N */
    uint32_t n_words;     /* ceil(dim0*dim1*dim2 / 32) */
    uint32_t* occ_bits;   /* dilated occupancy (coor_occ), 1 bit per voxel, z fastest */
    uint32_t* pt_bits;    /* voxels that hold >= 1 point */
    uint32_t* word_rank;  /* exclusive prefix of popc(pt_bits[w]): voxel -> dense slot */
    uint32_t* cell_start; /* [n_occ+1] CSR offsets into spts */
    float* spts;          /* [n_inrange] float4 (x, y, z, bitcast point index), voxel-major, ascending index */
    int32_t* counters;    /* device int32[16], see PNB_GC_* */
} pnb_grid_t;

/* Outputs of pnb_query (device pointers into the caller's workspace) -- sample-compacted layout. */
typedef struct {
    int32_t R, SR, K, D;
    int32_t cap_samples;     /* capacity of the per-candidate arrays */
    int32_t* nsamp;          /* [R]   candidate samples of ray r (0..SR) */
    uint32_t* samp_off;      /* [R+1] exclusive prefix of nsamp */
    uint16_t* steps;         /* [R*SR] march step index of candidate j of ray r */
    uint32_t* samp_ray;      /* [cap] ray of candidate s  (r*SR + j packed as r<<7 | j) */
    int32_t* cand_pidx;      /* [cap*K] neighbour point indices, -1 padded, canonical slot order */
    uint8_t* samp_nvalid;    /* [cap] number of neighbours (0..K) */
    uint32_t* valid_list;    /* [cap] candidate ids of valid samples, ascending */
    uint32_t* valid_rank;    /* [cap+1] exclusive prefix of (nvalid>0) */
    uint8_t* ray_hit;        /* [R] 1 if the ray has >= 1 neighbour (ray_mask of the reference) */
    uint32_t* ray_rank;      /* [R+1] scratch: exclusive prefix of ray_hit (filled by pnb_query_export) */
    uint32_t* scan_tmp;      /* scratch of the device-wide scans */
    int32_t* counters;       /* device int32[16], see PNB_QC_* */
    const float* raydir;     /* [R*3] as passed (borrowed) */
    const float* t;          /* borrowed */
    int32_t t_ray_stride;
    float campos[3];
} pnb_query_t;

/* Camera + scalar options of the shading / compositing stage. */
typedef struct {
    float campos[3];
    float camrotc2w[9]; /* row-major */
    float Rw2c[9];      /* row-major, points' world->canonical rotation (neural_points.Rw2c) */
    float vsize_z;      /* un-scaled opt.vsize[2]  (neural_points_volumetric_model.py:272) */
    float bg_color[3];
    int32_t raydist_mode_unit;
    int32_t agg_intrp_order; /* opt.agg_intrp_order (point_aggregators.py:573-633): 2 = density per neighbour, then the weighted sum
                              * (every shipped script; 0 is read as 2); 1 = alpha_branch on the K-aggregated feature */
} pnb_shade_opts_t;

/* MLP parameters, fp32, W^T layout [in][out] (transposed once per optimiser step by the host side). */
typedef struct {
    const float* w[9]; /* block1.0 block1.2 block3.0 block3.2 alpha_branch.0 color_branch.0 .2 .4 .6 */
    const float* b[9];
} pnb_mlp_t;

/* Neural point attributes (the reference's parameter tensors, read in place). */
typedef struct {
    const float* xyz;   /* [N,3] */
    const float* emb;   /* [N,32] points_embeding */
    const float* color; /* [N,3] */
    const float* dir;   /* [N,3] */
    const float* conf;  /* [N]   */
    int32_t N;
} pnb_points_t;

int pnb_version(void);
const char* pnb_last_error(void);
/* sizeof() of the POD structs above as the library was compiled (0 grid, 1 query, 2 shade_opts, 3 mlp,
 * 4 points) -- lets a foreign-language binding verify its mirror of the layout. */
size_t pnb_struct_size(int which);

/* ---- voxel grid ---- */
size_t pnb_grid_bytes(int N, const int32_t dim[3]);
/* Builds the grid into `buf` (>= pnb_grid_bytes).  h_counters (optional, int32[16]) receives the counters
 * AFTER a stream synchronise; pass NULL for a fully asynchronous build. */
int pnb_grid_build(pnb_grid_t* grid, void* buf, size_t buf_bytes, const float* d_xyz, int N,
                   const float lo[3], const float svs[3], const int32_t dim[3], const int32_t query_size[3],
                   int max_o, int P, int parity_slot0, pnb_stream_t stream, int32_t* h_counters);

/* ---- query ---- */
size_t pnb_query_bytes(int R, int SR, int K, int cap_samples);
/* cap_samples <= 0 -> R*SR (can never overflow).  t: [D] (t_ray_stride 0) or [R,D] (t_ray_stride D), every row non-decreasing
 * (as near-far linear ray generation makes it: the march finds the steps inside the grid's occupied box by binary search). */
int pnb_query(pnb_query_t* q, void* ws, size_t ws_bytes, const pnb_grid_t* grid, const float campos[3],
              const float* d_raydir, int R, const float* d_t, int t_ray_stride, int D, int SR, int K,
              float radius_limit, const int32_t kernel_size[3], int cap_samples, pnb_stream_t stream,
              int32_t* h_counters /* optional: synchronises */);
/* Dense reference layout.  d_ray_index [R] scratch (compacted row of each hit ray); outputs hold R rows of
 * capacity; rows >= R' are untouched.  ray_mask [R] int8.  sample_loc (perspective) may be NULL. */
int pnb_query_export(const pnb_query_t* q, const pnb_shade_opts_t* cam, int32_t* d_ray_row,
                     int8_t* d_ray_mask, int32_t* d_sample_pidx, float* d_sample_loc_w, float* d_sample_loc,
                     float* d_sample_ray_dirs, pnb_stream_t stream);

/* ---- shading + compositing, forward ---- */
size_t pnb_shade_bytes(int cap_samples);
/* sigma_rgb: [cap_samples] float4 per candidate sample (zeros for samples without neighbours). */
int pnb_shade_forward(const pnb_query_t* q, const pnb_points_t* pts, const pnb_mlp_t* mlp,
                      const pnb_shade_opts_t* opts, float* d_sigma_rgb, void* ws, size_t ws_bytes,
                      pnb_stream_t stream);
/* Full-R outputs (fill_invalid semantics): ray_color [R,3], opacity [R,SR], bg_T [R], ray_mask [R] int8. */
int pnb_composite_forward(const pnb_query_t* q, const pnb_shade_opts_t* opts, const float* d_sigma_rgb,
                          float* d_ray_color, float* d_opacity, float* d_bg_T, int8_t* d_ray_mask,
                          pnb_stream_t stream);

/* ---- auxiliary training outputs ----
 * `weight` [R',SR,K], `conf_coefficient` [R',SR,K] and `blend_weight` [R',SR] of the reference's output dict
 * (models/neural_points_volumetric_model.py:325-329; point_aggregators.py:421-429,727-732; neural_points.py:706-717;
 * diff_ray_marching.py:536-541) for the R' hit rays listed in d_rows (int64 ray ids, ascending), straight from the compacted query.
 * d_opacity: the [R,SR] opacity of pnb_composite_forward.  Empty slots follow the reference (weight 0, conf of point 0). */
int pnb_aux_outputs(const pnb_query_t* q, const pnb_points_t* pts, const long long* d_rows, int n_rows,
                    const float* d_opacity, float* d_weight, float* d_conf_coefficient, float* d_blend_weight,
                    pnb_stream_t stream);
/* d(loss)/d(points_conf) [N] (accumulated into) from d(loss)/d(conf_coefficient) [R',SR,K]: the clamp of neural_points.py:713 is a
 * straight-through estimator, every entry adds its gradient to the conf of its (clamped-to-0) point index. */
int pnb_aux_conf_backward(const pnb_query_t* q, const long long* d_rows, int n_rows,
                          const float* d_grad_conf_coefficient, float* d_grad_conf, pnb_stream_t stream);

/* ---- point growing: probe outputs and hole selection (run/train_ft.py:417-530) ----
 * pnb_probe_maps: the probe outputs of models/neural_points_volumetric_model.py:331-351 followed by fill_invalid / unmask (:87-123),
 * for all R rays of a query, from the compacted query and the [R,SR] opacity of pnb_composite_forward (no dense export).  Per hit ray:
 * j* = arg-max opacity over the SR slots (first index on ties), op_max [R] = opacity[j*], loc [R,3] = world position of slot j*
 * (origin for an unfilled slot), far_dist [R] = min over the K slots of |xyz[max(pidx,0)] - loc|, and avg_{color [R,3], dir [R,3],
 * conf [R], emb [R,32]} = sum over k of attr[max(pidx_k,0)] * w_k * clamp(conf, 1e-4, 1) with the normalised inverse-distance weights.
 * Rays without a neighbour get zeros.  d_argmax [R] (optional, may be NULL): j*, -1 for rays without a neighbour. */
int pnb_probe_maps(const pnb_query_t* q, const pnb_points_t* pts, const float* d_opacity, float* d_op_max, float* d_loc,
                   float* d_far_dist, float* d_avg_color, float* d_avg_dir, float* d_avg_conf, float* d_avg_emb, int32_t* d_argmax,
                   pnb_stream_t stream);
/* pnb_probe_select: the hole test of run/train_ft.py:493-512 on an H x W frame, maps in row-major [H*W] layout as probe_hole builds
 * them (ray_mask int8, 0 where no ray was cast; d_present uint8 = the pixels given (edge_mask), NULL = all; d_gt [H*W,3], 0 where
 * not given).  A pixel is selected when ray_mask > 0, op_max > opacity_thresh, and either a given pixel with ray_mask < 1 and
 * |gt - bg| > 0.002 lies in its 3x3 window (clipped to the image), or far_thresh > 0, far_dist > far_thresh and |gt - color| < 0.1.
 * The selected pixels are compacted in row-major order: the first min(n, cap) go to add_xyz [cap,3] (from d_loc),
 * add_emb [cap,32], add_color [cap,3], add_dir [cap,3], add_conf [cap]; d_count (device int32) receives n.  Deterministic.
 * ws >= pnb_probe_select_bytes(H, W); the embedding buffers must be 16-byte aligned. */
size_t pnb_probe_select_bytes(int H, int W);
int pnb_probe_select(int H, int W, const int8_t* d_ray_mask, const uint8_t* d_present, const float* d_gt, const float* d_color,
                     const float* d_far_dist, const float* d_op_max, const float* d_loc, const float* d_avg_emb,
                     const float* d_avg_color, const float* d_avg_dir, const float* d_avg_conf, const float bg_color[3],
                     float opacity_thresh, float far_thresh, void* ws, size_t ws_bytes, int cap, float* d_add_xyz,
                     float* d_add_emb, float* d_add_color, float* d_add_dir, float* d_add_conf, int32_t* d_count,
                     pnb_stream_t stream);

/* ---- shading forward on the tensor cores (tcgen05 / TMEM, BF16x3 error-compensated split) ---- */
/* Packs block1 / block3 / colour-branch weights of a pnb_mlp_t (fp32 W^T buffers) into tcgen05 operand images (hi/lo bf16, UMMA
 * shared-memory layout).  Call once per weight version.  d_out: >= pnb_mlp_pack_bytes() bytes. */
size_t pnb_mlp_pack_bytes(void);
int pnb_mlp_pack(const pnb_mlp_t* mlp, void* d_out, size_t out_bytes, pnb_stream_t stream);
/* Frozen point cloud (rendering): the 224 point-only inputs [f, PE3(f)] of block1.0
 * (models/aggregators/point_aggregators.py:547-571) are hoisted out of the per-pair work into a per-point table
 * d_pre[N][256] = b1 + W1[:, :224] . [f_n, PE3(f_n)] (fp32).  Call once per (points_embeding, block1.0) version. */
size_t pnb_point_pre_bytes(int N);
int pnb_point_pre(const pnb_points_t* pts, const pnb_mlp_t* mlp, float* d_pre, size_t pre_bytes, pnb_stream_t stream);
enum {
    PNB_TC_PAIRS = 1,           /* row packing + per-pair MLPs + K-reduction -> h-bar, sigma */
    PNB_TC_COLOR = 2,           /* colour branch -> sigma_rgb (both = a forward) */
    PNB_TC_FROZEN = 4,          /* pair kernel of a frozen cloud (k_shade_tc8): needs d_point_pre */
    PNB_TC_DBG_NO_WEIGHTS = 64  /* timing experiment: no weight traffic (garbage results) */
    /* bits 8..15: profiling flags of tools/tc_profile.py (1024: per-CTA cycles into d_err[64..], needs a 512-int d_err) */
};
/* Same contract as pnb_shade_forward; the MLPs run as tcgen05.mma tiles.  mlp->w[5] must be zero padded to 288 rows.
 * ws >= pnb_shade_tc_bytes(max_valid_samples).  d_err: device int32[>= 64], 0 on success, 9 if the query produced more valid
 * samples than max_valid_samples (the extra samples are dropped: their sigma_rgb is zeroed, every other result is exact),
 * any other non-zero value = an internal pipeline time-out (a bounded 2-s mbarrier wait expired; results invalid). */
size_t pnb_shade_tc_bytes(int max_valid_samples);
int pnb_shade_forward_tc(const pnb_query_t* q, const pnb_points_t* pts, const pnb_mlp_t* mlp, const void* d_packed,
                         const float* d_point_pre /* NULL unless PNB_TC_FROZEN */, const pnb_shade_opts_t* opts,
                         float* d_sigma_rgb, void* ws, size_t ws_bytes, int max_valid_samples, int flags, int* d_err,
                         pnb_stream_t stream);
/* Diagnostics / tests: device pointers of the row-packing tables inside a workspace laid out for max_valid_samples
 * (vorder uint32[n_valid], vcntp uint8[n_valid], quad_first uint32[n_quads + 1], pack_cnt int32[1] = n_quads). */
int pnb_shade_tc_tables(void* ws, size_t ws_bytes, int max_valid_samples, void** vorder, void** vcntp, void** quad_first,
                        void** pack_cnt);

/* ---- backward (per-scene optimisation batches) ----
 * Replaces loss.backward() through the reference's eager autograd graph
 * (models/mvs_points_volumetric_model.py:98-118): given d(loss)/d(ray_color) [R,3] (full-R layout of
 * pnb_composite_forward) accumulates gradients of points_embeding [N,32], points_color [N,3], points_dir [N,3],
 * points_conf [N] (any may be NULL) and of the 9 MLP layers in the layout of pnb_mlp_t (W^T [K_pad][N] and bias; the
 * caller zero-initialises all accumulators).  d_sigma_rgb_fwd: the forward's per-candidate (sigma, rgb) buffer.
 * n_valid / n_pairs: host copies of counters[PNB_QC_N_VALID] / [PNB_QC_N_PAIRS] (the pair-level buffers hold one row per valid pair).  ws >= pnb_backward_bytes.  The activations are recomputed and every layer
 * GEMM (recompute, dX, dW) runs on the tensor cores (tcgen05, BF16x3 split, fp32 accumulate; dW by a deterministic split-K);
 * the recomputed pre-activations carry the BF16x3 error, so ~1e-6 of the LeakyReLU masks differ from an fp32 forward's (each changes
 * one pair's gradient by ~1/256; see the flags).  d_err: device int32,
 * set non-zero if a bounded pipeline wait of the tensor-core GEMMs expires (results invalid). */
enum {
    PNB_BWD_FP32_GEMM = 1,      /* every GEMM on the fp32 CUDA-core tiles (parity reference of the tensor-core engine) */
    PNB_BWD_FP32_RECOMPUTE = 4  /* forward recompute on the fp32 tiles (LeakyReLU masks of an fp32 forward), dX / dW on the tensor cores */
};
size_t pnb_backward_bytes(int n_valid, int cap_samples);
int pnb_shade_backward(const pnb_query_t* q, const pnb_points_t* pts, const pnb_mlp_t* mlp, const pnb_shade_opts_t* opts,
                       const float* d_sigma_rgb_fwd, const float* d_ray_color, int n_valid, int n_pairs, float* d_emb, float* d_color,
                       float* d_dir, float* d_conf, float* const* d_mlp_w, float* const* d_mlp_b, void* ws,
                       size_t ws_bytes, int flags, int* d_err, pnb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* PNB200_H */
