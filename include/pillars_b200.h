/*
 * pillars_b200.h -- C ABI of libpillars_b200.so: the B200 (sm_100a) pillar LiDAR-encoder hot path.
 *
 * Drop-in boundary.  The reference (Advaith-Sajeev/LiDAR-Vision-VQA, src/lidar-encoder = vendored OpenPCDet)
 * has no native code on this path: grouping is a third-party CPU call, the feature net and the BEV scatter
 * are eager PyTorch.  Its native-extension idiom elsewhere is "pybind11 function -> raw-pointer launcher on the
 * default stream" (src/lidar-encoder/pcdet/ops/ingroup_inds/src/ingroup_inds.cpp:15-54,
 * ingroup_inds_kernel.cu:47-77).  This header is that launcher layer for the pillar path, as plain C so that
 * Python binds it with ctypes (INTEGRATION.md shows the stub a maintainer adds to pcdet).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer on the caller's current device unless its name ends in _host;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream); all work is enqueued on it and
 *     the call returns without synchronising;
 *   - return value: 0 on success, otherwise a cudaError_t value or a negative PILLARS_E_* code;
 *     pillars_last_error() returns a thread-local message.  Nothing throws.
 *   - no hidden device allocation: scratch comes from the caller's workspace, sized by
 *     pillars_workspace_bytes().  The workspace content is opaque and may be reused by the next call
 *     on the same stream.
 *   - there is NO CPU fallback: on a machine without an sm_100 device every compute entry point fails.
 *
 * Entry point                          replaces (reference file:line, paths under src/lidar-encoder/pcdet/)
 *   pillars_frame_offsets              datasets/dataset.py:237-244        (batch-index column of the collated points)
 *   pillars_voxelize                   datasets/processor/data_processor.py:16-61,133-180
 *                                      (VoxelGeneratorWrapper.generate -> spconv point_to_voxel) + the collate of
 *                                      datasets/dataset.py:232-244
 *   pillars_pfn_dense                  models/backbones_3d/vfe/pillar_vfe.py:94-123 (PillarVFE.forward) with
 *                                      :29-49 (PFNLayer.forward), eval mode
 *   pillars_scatter_bev                models/backbones_2d/map_to_bev/pointpillar_scatter.py:14-37
 *                                      (PointPillarScatter.forward)
 *   pillars_encode_bev                 the three above fused: raw points -> pillar_features, voxel_coords,
 *                                      spatial_features, i.e. module_list[vfe, map_to_bev] of
 *                                      models/detectors/pointpillar.py:9-11 fed by `points` the way
 *                                      models/backbones_3d/vfe/dynamic_pillar_vfe.py:90-142 is
 *   pillars_tokens_prepare,            src/encoder-decoder/training/models/vat_lidar.py:206-253: the BEV tokeniser at the
 *   pillars_bev_tokens[_map|_dense]    head of VATLiDAR.forward (refine -> proj -> norm_tokens -> + geo PE -> + view embed),
 *                                      the first consumer of spatial_features; geometry tables per :123-185
 */
#ifndef PILLARS_B200_H_
#define PILLARS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PILLARS_ABI_VERSION 5

/* error codes (negative; positive values are cudaError_t) */
#define PILLARS_E_BADARG (-1)      /* NULL pointer, bad size, unsupported combination */
#define PILLARS_E_WORKSPACE (-2)   /* workspace too small / misaligned */
#define PILLARS_E_UNSUPPORTED (-3) /* shape outside what the kernels are instantiated for */
#define PILLARS_E_NODEVICE (-4)    /* no CUDA device / not an sm_100 part */

/* Voxel grid + grouping limits: the `transform_points_to_voxels` block of a PCDet yaml
 * (data_processor.py:133-149).  range/voxel are the fp32 values spconv stores; grid = round((max-min)/voxel)
 * computed by the caller exactly as data_processor.py:135-136 does. */
typedef struct pillars_grid {
    float range[6];     /* xmin ymin zmin xmax ymax zmax */
    float voxel[3];     /* vx vy vz */
    int32_t grid[3];    /* nx ny nz */
    int32_t max_points; /* MAX_POINTS_PER_VOXEL (P) */
    int32_t max_voxels; /* MAX_NUMBER_OF_VOXELS, per frame */
} pillars_grid_t;

/* One PFN layer in eval mode (pillar_vfe.py:8-49) with BatchNorm folded by the caller:
 *   y = relu( (x . W^T) * scale + shift ),  scale = gamma / sqrt(var + eps), shift = beta - mean * scale
 * (USE_NORM false: scale = 1, shift = linear.bias).  Feature layout of x follows pillar_vfe.py:105-113. */
typedef struct pillars_pfn {
    int32_t c_point;          /* C: channels of a raw point incl. xyz (num_point_features) */
    int32_t c_in;             /* in_features of the linear = C (+3 if use_absolute_xyz... see pillar_vfe.py:59-62) */
    int32_t f_out;            /* out_features (64) */
    int32_t use_absolute_xyz; /* USE_ABSLOTE_XYZ */
    int32_t with_distance;    /* WITH_DISTANCE */
    float offset[3];          /* voxel/2 + range_min per axis, computed in double by the caller (pillar_vfe.py:79-81) */
    const float *weight;      /* [f_out, c_in] row-major = nn.Linear.weight */
    const float *scale;       /* [f_out] */
    const float *shift;       /* [f_out] */
    /* Optional: the layer regrouped around the pillar centre, PILLARS_FOLDED_FLOATS floats on the device, written once
     * per model by pillars_fold_pfn().  NULL: pillars_encode_bev folds into its workspace on every call (one extra
     * single-block launch).  Used by the streaming feature kernel (USE_ABSLOTE_XYZ, no WITH_DISTANCE, C <= 5). */
    const float *folded;
} pillars_pfn_t;

#define PILLARS_FOLDED_FLOATS (13 * 64)

/* what pillars_encode_bev / pillars_voxelize write; any pointer may be NULL to skip that output */
typedef struct pillars_outputs {
    int64_t pillar_capacity;  /* rows available in the per-pillar arrays below (>= sum of per-frame pillars) */
    float *pillar_features;   /* [capacity, F]        batch_dict['pillar_features']                        */
    int32_t *voxel_coords;    /* [capacity, 4] (b,z,y,x)  batch_dict['voxel_coords']                       */
    int32_t *voxel_num_points;/* [capacity]           batch_dict['voxel_num_points'] (capped at P)         */
    float *voxels;            /* [capacity, P, C] zero padded   batch_dict['voxels']                       */
    int32_t *point_pillar;    /* [n_points] row of the pillar holding the point, -1 if rejected/dropped    */
    int32_t *point_slot;      /* [n_points] slot inside the pillar, -1 if over the cap / rejected          */
    int32_t *pillar_count;    /* [n_frames + 1] pillars per frame, total in the last entry                 */
    float *bev;               /* [n_frames, F*nz, ny, nx]  batch_dict['spatial_features'] (encode_bev only) */
    void *bev_half;           /* same canvas as IEEE float16 (round to nearest even), the dtype the product stores:
                                 src/get-data/precompute_bev_features.py:394; may be given instead of or beside bev */
    int32_t want_index_map;   /* non-zero: leave the BEV index map [n_frames, ny, nx] (row of the pillar in each cell, -1 =
                                 empty) in the workspace at pillars_workspace_cell_row_offset() even when no canvas is asked
                                 for -- the input of pillars_conv_forward / pillars_bev_tokens_map (nz == 1 grids) */
} pillars_outputs_t;

int pillars_abi_version(void);
const char *pillars_last_error(void);

/* 0 if device `device` (or the current one when < 0) can run this library (compute capability 10.x). */
int pillars_device_ok(int device);

/* Scratch bytes needed by pillars_voxelize / pillars_encode_bev for n_points total points in n_frames frames;
 * by pillars_scatter_bev when n_points == 0 (then only the index map counts). */
size_t pillars_workspace_bytes(int64_t n_points, int32_t n_frames, const pillars_grid_t *grid);

/* points_b: collated batch_dict['points'] [n, row_stride] with the frame index in column 0, rows sorted by frame.
 * Writes frame_offsets[0..n_frames] (frame b owns rows [offsets[b], offsets[b+1])). */
int pillars_frame_offsets(const float *points_b, int64_t n, int32_t row_stride, int32_t n_frames,
                          int32_t *frame_offsets, void *stream);

/* Hard voxelisation of a batch: first-appearance pillar ids per frame, first-P points per pillar in point order,
 * new pillars dropped once max_voxels exist.  points is [n, row_stride] fp32; x,y,z,... start at column `col0`
 * (0 for packed frames, 1 for the collated PCDet layout); c_point channels are copied into `voxels`.
 * Fills out->{voxel_coords, voxel_num_points, voxels, point_pillar, point_slot, pillar_count} (each optional). */
int pillars_voxelize(const float *points, int64_t n, int32_t row_stride, int32_t col0, int32_t c_point,
                     const int32_t *frame_offsets, int32_t n_frames, const pillars_grid_t *grid,
                     const pillars_outputs_t *out, void *workspace, size_t workspace_bytes, void *stream);

/* Prepares pfn->folded: `folded` (device, PILLARS_FOLDED_FLOATS floats) from pfn->weight/scale/shift.  Fails with
 * PILLARS_E_UNSUPPORTED when the layer is not one the streaming kernel covers (then leave pfn->folded NULL). */
int pillars_fold_pfn(const pillars_pfn_t *pfn, float *folded, void *stream);

/* PillarVFE.forward on already grouped voxels (the reference's own input format).
 * voxels [m, P, C] fp32; num_points [m] and coords [m,4] (b,z,y,x) are int32, or fp32 when *_is_float != 0
 * (models/__init__.py:36 casts everything to float).  out is [m, F]. */
int pillars_pfn_dense(const float *voxels, const void *num_points, int32_t num_points_is_float,
                      const void *coords, int32_t coords_is_float, int64_t m, int32_t max_points,
                      const pillars_pfn_t *pfn, const float voxel_size[3], float *out, void *stream);

/* PointPillarScatter.forward: bev[b][f][y][x] = feats[m][f] for coords[m] = (b,z,y,x), zero elsewhere (nz == 1), and
 * PointPillarScatter3d.forward (pointpillar_scatter.py:40-73) for nz > 1: bev[b][f][z*ny*nx + y*nx + x], which viewed as
 * [B, f*nz, ny, nx] is exactly the reference's output.
 * m_dev, when not NULL, is a device int32 holding the live row count (<= m); rows beyond it are ignored.
 * variant: 0 = default (channel-group 256-bit stores where the shape allows, else plain), 1 = plain vector stores,
 *          4 = same as 0.  (The store paths that were measured slower are archived under profiles/micro/.) */
int pillars_scatter_bev(const float *feats, const void *coords, int32_t coords_is_float, int64_t m,
                        const int32_t *m_dev, int32_t n_frames, int32_t f, int32_t nx, int32_t ny, int32_t nz, float *bev,
                        void *workspace, size_t workspace_bytes, int32_t variant, void *stream);

/* PointPillarScatter.forward followed by the extractor's `.astype(np.float16)` (precompute_bev_features.py:394) in one
 * pass: bev_half is [n_frames, f*nz, ny, nx] float16.  Needs nx*ny*nz % 8 == 0 and f % 8 == 0. */
int pillars_scatter_bev_half(const float *feats, const void *coords, int32_t coords_is_float, int64_t m,
                             const int32_t *m_dev, int32_t n_frames, int32_t f, int32_t nx, int32_t ny, int32_t nz,
                             void *bev_half, void *workspace, size_t workspace_bytes, void *stream);

/* Multi-GPU hand-over (no counterpart in the reference: its frames go to disk; the gather helper it ships,
 * pcdet/utils/commu_utils.py:50-111, is the shape this replaces).  Compact BEV tokens gathered from several ranks lie in
 * n_segments segments of rows_per_segment rows of (b,z,y,x) int32 coordinates; segment s starts at
 * coords + s * segment_stride (int32 elements, >= 4 * rows_per_segment) and has segment_counts[s * count_stride] live rows,
 * numbered with rank-local frame indices.  Adds s * frames_per_segment to the frame index of live rows and writes -1 into
 * the frame index of padding rows, which pillars_scatter_bev and pillars_bev_tokens skip; sets *overflow (optional) to 1
 * when a count exceeds rows_per_segment.  Everything stays on the device: no count ever visits the host. */
int pillars_rebase_segments(int32_t *coords, int32_t n_segments, int64_t rows_per_segment, int64_t segment_stride,
                            const int32_t *segment_counts, int64_t count_stride, int32_t frames_per_segment,
                            int32_t *overflow, void *stream);

/* The fused path: raw points -> pillar features -> BEV.  Same grouping semantics as pillars_voxelize, same
 * feature semantics as pillars_pfn_dense on its output, same canvas as pillars_scatter_bev. */
int pillars_encode_bev(const float *points, int64_t n, int32_t row_stride, int32_t col0,
                       const int32_t *frame_offsets, int32_t n_frames, const pillars_grid_t *grid,
                       const pillars_pfn_t *pfn, const pillars_outputs_t *out, void *workspace,
                       size_t workspace_bytes, int32_t scatter_variant, void *stream);

/* ---- general feature stacks: two-layer PFN, DynamicPillarVFE, DynamicPillarVFESimple2D ---------------------------------
 * replaces (paths under src/lidar-encoder/pcdet/models/backbones_3d/vfe/):
 *   pillars_pfn_dense_stack   pillar_vfe.py:94-123 with a ModuleList of two PFNLayers (:18-19,44-49,119-120)
 *   pillars_encode_stack      mode HARD:    data_processor.py voxelisation + the same stack (any NUM_FILTERS of 1-2 entries)
 *                             mode DYNAMIC: dynamic_pillar_vfe.py:90-142 (DynamicPillarVFE.forward, PFNLayerV2 :35-46) and
 *                                           :193-240 (DynamicPillarVFESimple2D.forward) with layout SIMPLE2D            */
#define PILLARS_LAYOUT_PILLAR_VFE 0 /* features = [point channels, f_cluster, f_center (, distance)]  pillar_vfe.py:105-113 */
#define PILLARS_LAYOUT_SIMPLE2D 1   /* features = [f_center, point channels (, distance)]   dynamic_pillar_vfe.py:209-224 */
#define PILLARS_MODE_HARD 0         /* first-appearance rows, MAX_POINTS_PER_VOXEL / MAX_NUMBER_OF_VOXELS caps, padded-slot row */
#define PILLARS_MODE_DYNAMIC 1      /* rows by sorted key b*nx*ny + ix*ny + iy, no caps, x/y range check only */

typedef struct pillars_pfn_stack {
    int32_t n_layers;         /* 1 or 2 */
    int32_t c_point;          /* channels of a raw point incl. xyz */
    int32_t out_features[2];  /* out_features of each layer's linear (layer 0 of two: NUM_FILTERS[0] / 2, at most 32) */
    int32_t use_absolute_xyz;
    int32_t with_distance;
    int32_t layout;           /* PILLARS_LAYOUT_* */
    float offset[3];          /* voxel/2 + range_min per axis */
    const float *weight[2];   /* [out, in] row-major; in of layer 1 = 2 * out_features[0] */
    const float *scale[2];    /* folded BatchNorm (or 1) */
    const float *shift[2];    /* folded BatchNorm (or the linear's bias) */
} pillars_pfn_stack_t;

/* in_features of layer 0 for this stack (C + 6, C + 3, ... see the layouts above), or a negative error code. */
int pillars_pfn_stack_in_features(const pillars_pfn_stack_t *stack);

/* PillarVFE.forward on padded voxels with a one- or two-layer stack; out is [m, out_features[n_layers-1]]. */
int pillars_pfn_dense_stack(const float *voxels, const void *num_points, int32_t num_points_is_float,
                            const void *coords, int32_t coords_is_float, int64_t m, int32_t max_points,
                            const pillars_pfn_stack_t *stack, const float voxel_size[3], float *out, void *stream);

/* Raw points -> pillar features (+ BEV in mode HARD when out->bev is set) through a feature stack.
 * NUM_FILTERS [64, 64] (mode HARD) and [64] / [64, 64] (mode DYNAMIC, 4-column coords) in the standard feature layout
 * (absolute xyz, no distance, <= 5 point channels) run on the streaming feature kernel; every other stack on the general one.
 * coords_cols: 4 writes out->voxel_coords as (b,z,y,x) -- (b,0,y,x) in mode DYNAMIC, dynamic_pillar_vfe.py:132-138;
 *              3 writes (b,y,x), the `pillar_coords` of DynamicPillarVFESimple2D (:232-238).
 * In mode DYNAMIC grid->max_points / max_voxels are ignored and out->voxel_num_points receives the uncapped counts. */
int pillars_encode_stack(const float *points, int64_t n, int32_t row_stride, int32_t col0,
                         const int32_t *frame_offsets, int32_t n_frames, const pillars_grid_t *grid,
                         const pillars_pfn_stack_t *stack, int32_t mode, int32_t coords_cols,
                         const pillars_outputs_t *out, void *workspace, size_t workspace_bytes,
                         int32_t scatter_variant, void *stream);

/* ---- BEV tokeniser: VATLiDAR.forward up to the tokens its blocks attend over --------------------------------------------
 * replaces src/encoder-decoder/training/models/vat_lidar.py:206-253 (eval mode):
 *   x = GELU(conv3x3_depthwise(bev) + b)  :82-85,211   y = LayerNorm(conv1x1(x))  :88-89,222-225
 *   tokens = y + geo_mlp(geom) + view_embed[sector]     :229-245        -> [n_frames, h*w, d_model]
 * Supported shapes: c_in % 4 == 0, c_in <= 512; d_model % 128 == 0, d_model <= 1024.  All pointers 16-byte aligned. */
typedef struct pillars_tokenizer {
    int32_t c_in;               /* channels of the canvas = refine / proj in_channels */
    int32_t d_model;
    const float *dw_weight;     /* [c_in, 9]      refine.0.weight [c_in,1,3,3]                        */
    const float *dw_bias;       /* [c_in]         refine.0.bias                                       */
    const float *proj_weight_t; /* [c_in, d_model] proj.weight [d_model,c_in,1,1] TRANSPOSED by the caller */
    const float *proj_bias;     /* [d_model]      proj.bias                                           */
    const float *ln_weight;     /* [d_model]      norm_tokens.weight                                  */
    const float *ln_bias;       /* [d_model]      norm_tokens.bias                                    */
    float ln_eps;               /* norm_tokens.eps (1e-5)                                             */
    const float *pe;            /* [h*w, d_model] written by pillars_tokens_prepare                   */
    const float *background;    /* [d_model]      written by pillars_tokens_prepare                   */
    const float *proj_umma;     /* [2*c_in*d_model] optional: the projection as the shared-memory image of the tcgen05 variant
                                   (tf32 hi | lo halves, K-major, 128-byte swizzle), written by pillars_tokens_prepare.  When set
                                   (c_in 32 or 64, d_model 128 or 256) and a workspace is given, the active cells of the batch are
                                   compacted into 128-row tiles and projected with tcgen05.mma.kind::tf32 (accumulator in TMEM) */
} pillars_tokenizer_t;

/* Once per (weights, h, w): pe_out[cell] = geo_mlp.2(GELU(geo_mlp.0(geom[cell]))) + view_embed[sector[cell]] and
 * background_out = LayerNorm(proj(GELU(refine bias))), the token (before PE) of a cell whose 3x3 window is all zero.
 * geom [h*w,5] / sector [h*w] are the tables of VATLiDAR._grid (:123-185), computed by the caller;
 * geo_w1 [d,5] = geo_mlp.0.weight, geo_w2_t [d,d] = geo_mlp.2.weight TRANSPOSED, view_embed [6,d].
 * proj_umma_out (2*c_in*d_model floats, may be NULL) receives the table for tk->proj_umma.
 * Reads tk->{c_in,d_model,dw_bias,proj_weight_t,proj_bias,ln_*}; tk->pe / background / proj_umma are not read. */
int pillars_tokens_prepare(const pillars_tokenizer_t *tk, const float *geom, const int32_t *sector, int32_t h, int32_t w,
                           const float *geo_w1, const float *geo_b1, const float *geo_w2_t, const float *geo_b2,
                           const float *view_embed, float *pe_out, float *background_out, float *proj_umma_out, void *stream);

/* Scratch bytes: index map + pair list (dense == 0, for pillars_bev_tokens / _map) or those + compacted rows (dense != 0). */
size_t pillars_tokens_workspace_bytes(int32_t n_frames, int32_t c_in, int32_t h, int32_t w, int32_t dense);

/* Tokens straight from pillar rows, no dense canvas: feats [m, c_in] and coords [m,4] (b,z,y,x) exactly as
 * pillars_scatter_bev takes them (h = ny, w = nx, nz == 1).  tokens is [n_frames, h*w, d_model]. */
int pillars_bev_tokens(const float *feats, const void *coords, int32_t coords_is_float, int64_t m, const int32_t *m_dev,
                       int32_t n_frames, int32_t h, int32_t w, const pillars_tokenizer_t *tk, float *tokens,
                       void *workspace, size_t workspace_bytes, void *stream);

/* Same with an index map that already exists: cell_row [n_frames, h, w] int32, row of the pillar in the cell or -1.
 * workspace (pillars_tokens_workspace_bytes(..., 0) bytes) is only needed by the tcgen05 variant (tk->proj_umma); with
 * workspace == NULL that variant is not used. */
int pillars_bev_tokens_map(const float *feats, const int32_t *cell_row, int32_t n_frames, int32_t h, int32_t w,
                           const pillars_tokenizer_t *tk, float *tokens, void *workspace, size_t workspace_bytes,
                           void *stream);

/* VATLiDAR's own input: a dense canvas bev [n_frames, c_in, h, w].  Cells with a non-zero channel are compacted into rows
 * (workspace), then the same kernel runs; on a canvas without zeros every cell takes the arithmetic path. */
int pillars_bev_tokens_dense(const float *bev, int32_t n_frames, int32_t h, int32_t w, const pillars_tokenizer_t *tk,
                             float *tokens, void *workspace, size_t workspace_bytes, void *stream);

/* Byte offset, inside a workspace of pillars_encode_bev for the same (n_points, n_frames, grid), of the BEV index map
 * [n_frames, ny, nx] that call leaves behind when it wrote a canvas -- the cell_row argument of pillars_bev_tokens_map. */
size_t pillars_workspace_cell_row_offset(int64_t n_points, int32_t n_frames, const pillars_grid_t *grid);

/* ---- BEV backbone convolutions (SURVEY 8 f-3: BaseBEVBackbone, backbones_2d/base_bev_backbone.py:29-112) -------------
 * One layer = Conv2d / ConvTranspose2d (bias=False) + eval-mode BatchNorm2d(eps=1e-3) + ReLU, as ONE implicit-GEMM kernel on
 * the tcgen05 tensor cores (tf32 operands, fp32 accumulation: what nn.Conv2d itself does on this GPU under PyTorch's default
 * cudnn.allow_tf32).  Activations between layers are NHWC fp32.  Supported: c_in a multiple of 32; c_out in {64,128,256};
 * (k, stride, pad) in {(3,1,1), (1,1,0), (3,2,1), (2,2,0)}; up in {2, 4} = ConvTranspose2d(kernel = stride = up), given as k = 1. */
typedef struct {
    int32_t c_in, c_out;
    int32_t k, stride, pad;
    int32_t up;        /* 1 = convolution; 2 / 4 = transposed convolution with kernel = stride = up (k = 1, stride = 1, pad = 0) */
    int32_t relu;      /* apply ReLU after the BatchNorm shift */
    int32_t round_out; /* store tf32-rounded activations (for layers that feed another layer of this kind) */
} pillars_conv_t;

/* Bytes of the prepared weight image of a layer. */
size_t pillars_conv_weight_bytes(const pillars_conv_t *cv);

/* Builds the image: weight is the module's tensor ([c_out,c_in,k,k] for Conv2d, [c_in,c_out,up,up] for the transposed case);
 * bn_scale [c_out] = gamma / sqrt(running_var + eps) is folded into it (NULL = 1).  The matching shift
 * beta - running_mean * bn_scale is passed to pillars_conv_forward.  Replaces nn.Conv2d + nn.BatchNorm2d state
 * (base_bev_backbone.py:31-45,50-58). */
int pillars_conv_prepare(const pillars_conv_t *cv, const float *weight, const float *bn_scale, void *image, void *stream);

/* Runs the layer.  Input: in_nhwc [n_frames, h_in, w_in, c_in], or (in_nhwc == NULL) pillar rows [m, c_in] plus the BEV index
 * map cell_row [n_frames, h_in, w_in] (-1 = empty cell) -- the dense canvas is then never read.  Output pixel (oy, ox) of
 * channel n goes to out[b, oy', ox', out_c_off + n] of an NHWC image with out_c_total channels (out_nchw == 0) or to
 * out[b, out_c_off + n, oy', ox'] (out_nchw != 0), (oy', ox') = (oy, ox) or, for up == 2, the four phase positions.
 * error_word: optional device uint32, set non-zero if a bounded wait inside the kernel expired (never in a correct run).
 * Replaces blocks[i] / deblocks[i] of BaseBEVBackbone.forward (base_bev_backbone.py:92-106). */
int pillars_conv_forward(const pillars_conv_t *cv, const void *image, const float *bn_shift, const float *in_nhwc,
                         const float *rows, const int32_t *cell_row, int32_t n_frames, int32_t h_in, int32_t w_in, float *out,
                         int32_t out_c_total, int32_t out_c_off, int32_t out_nchw, uint32_t *error_word, void *stream);

/* Dense canvas [n_frames, c, h, w] -> (rows of its non-zero cells, index map): the input form pillars_conv_forward and the
 * tokeniser gather from.  rows must hold n_frames*h*w*c floats in the worst case; counter is one device uint32 (row count). */
int pillars_canvas_to_rows(const float *bev, int32_t n_frames, int32_t c, int32_t h, int32_t w, int32_t *cell_row, float *rows,
                           uint32_t *counter, void *stream);

/* Number of kernel launches (incl. memsets) the last successful compute call on this thread enqueued. */
int pillars_last_launch_count(void);

/* Measurement hook (bench.py): four cudaEvent_t (as void*) that pillars_encode_bev / pillars_voxelize record on the
 * call's stream at: [0] entry, [1] grouping done, [2] pillar features done, [3] scatter done.  NULL clears the hook.
 * Thread-local; costs four cudaEventRecord per call while set. */
int pillars_set_stage_events(void *const *events4);

/* Grouping implementation used by pillars_voxelize / pillars_encode_bev / pillars_encode_stack (thread-local):
 *   0  automatic: the direct-mapped cell table when n_frames * cells <= 16 * n_points + 2^22 (every pillar grid of the
 *      reference's configs), else the open-addressing hash table;
 *   1  always the hash table;   2  the direct-mapped table whenever n_frames * cells < 2^31.
 * Both produce bit-identical outputs (tests run every grouping case through both).  pillars_workspace_bytes() covers
 * either choice. */
int pillars_set_grouping(int mode);

/* Canvas occupancy bitmaps for the next pillars_encode_bev or pillars_encode_stack on this thread, which consumes and
 * clears them whether it succeeds or fails.  A canvas the library wrote before is mostly zeros already; with the bitmaps
 * the scatter writes only the cells that are occupied now or were occupied in the canvas's previous contents.
 * Layout: words [n_frames][ceil(nx*ny / 256)] of uint32 (device memory); bit k of word w of frame b covers the 8 cells
 * 256*w + 8*k .. 256*w + 8*k + 7 of that frame's ny*nx plane (row-major y, x), set = "may be non-zero".
 *   prev  the bitmap the last call on this canvas wrote into its next, describing what the canvas holds now; NULL when the
 *         contents are unknown (fresh or written by anyone else): the whole canvas is written.
 *   next  receives the occupancy this call leaves (all ones when it writes the canvas with the plain kernel).  Must not
 *         alias prev: the caller keeps two bitmaps per canvas and swaps them after every call.
 * The canvas, prev and next must be ordered with the call like the canvas alone (same stream or events).  It is an error
 * for a call with bitmaps to write both bev and bev_half.  NULL, NULL clears the hook. */
int pillars_set_canvas_occupancy(const uint32_t *prev, uint32_t *next);

/* Measurement hook (thread-local): a zeroed device buffer of 32 uint64 that the grouping / feature kernels of subsequent calls
 * stamp with %globaltimer nanoseconds per phase (even slot: earliest stamp, stored complemented; odd slot: latest stamp);
 * NULL switches it off.  profiles/scripts/phase_times.py decodes it. */
int pillars_set_debug_times(void *buffer32);

/* Test / measurement hook (thread-local): non-zero sends every call to the general feature kernel instead of the
 * streaming one -- pillars_encode_bev to k_pillar_features, pillars_encode_stack to the general stack kernel,
 * pillars_pfn_dense to the faithful padded kernel (pfn->folded is then ignored). */
int pillars_force_generic_features(int on);

#ifdef __cplusplus
}
#endif
#endif /* PILLARS_B200_H_ */
