/* sassd_b200 — C ABI of the B200-native SA-SSD inference hot path.
 *
 * Drop-in boundary (DESIGN.md §Boundary, SURVEY.md §8b): these are the entry
 * points a binding of the reference's native extensions for this path would
 * call.  Plain C: device pointers, sizes, a CUDA stream; no torch types.
 *
 * Conventions (differences from the reference ABI are deliberate and listed):
 *  - every pointer is a DEVICE pointer unless the name says host_;
 *  - every function takes the stream to launch on (the reference launches on
 *    the legacy default stream, iou3d_kernel.cu:359-386) and returns an int
 *    status (SASSD_OK or a negative SASSD_ERR_*); nothing exits the process
 *    (the reference calls exit(), iou3d.cpp:13-21) and nothing is allocated or
 *    freed inside a call (the reference cudaMalloc/cudaFree's per NMS call,
 *    iou3d.cpp:87,98) — scratch comes in through `ws` with a *_workspace_bytes query;
 *  - data-dependent sizes (voxel counts, active rows, guided anchors, kept boxes)
 *    live in device memory (`d_*` int32 counters) so that a whole frame runs
 *    without a host round trip and can be captured in a CUDA graph; buffers are
 *    sized by capacity (`*_cap`).  A capacity overflow truncates the output and
 *    sets a bit in the int32 word `d_status` (SASSD_FLAG_*).
 *  - layouts: points [N,4] f32 (x,y,z,r); voxel coordinates int32 (b,z,y,x);
 *    boxes [x,y,z(bottom),w,l,h,ry]; BEV boxes [x1,y1,x2,y2,ry];
 *    feature matrices row-major [rows, channels]; dense maps NHWC.
 */
#ifndef SASSD_B200_H
#define SASSD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* sassd_stream_t; /* cudaStream_t */

enum {
    SASSD_OK = 0,
    SASSD_ERR_ARG = -1,       /* bad argument (null pointer, unsupported size) */
    SASSD_ERR_LAUNCH = -2,    /* CUDA reported a launch error */
    SASSD_ERR_WORKSPACE = -3, /* workspace too small */
    SASSD_ERR_UNSUPPORTED = -4
};

enum { /* bits of *d_status */
    SASSD_FLAG_VOXEL_CAP = 1,   /* more voxel rows than the output capacity */
    SASSD_FLAG_ROWS_CAP = 2,    /* strided-conv output rows exceed capacity */
    SASSD_FLAG_GUIDED_CAP = 4,  /* guided anchors per frame exceed capacity */
    SASSD_FLAG_NMS_CAP = 8,     /* NMS candidates per frame exceed capacity */
    SASSD_FLAG_HASH_FULL = 16,
    SASSD_FLAG_DET_CAP = 32     /* boxes kept by the NMS exceed the detection capacity */
};

int sassd_version(void);
/* Launch hint, process-wide: on != 0 launches the tensor-core conv kernels as programmatic dependents of their
 * predecessors (their prologues overlap the previous layer's tail); -1 restores the default (environment SASSD_PDL,
 * else off).  Worth ~2 % for a step that runs alone on the GPU, costs throughput when several steps are in flight, so set
 * it around the capture of a latency-oriented graph only.  Returns the previous setting.  Results never change. */
int sassd_set_pdl(int on);

/* ------------------------------------------------------------------------
 * Voxelization.  Replaces mmdet/ops/points_op/points_ops.py:104-164
 * (points_to_voxel, reverse_index=True) called from
 * mmdet/core/point_cloud/voxel_generator.py:22-25, fused with
 * SingleStageDetector.merge_second_batch's batch-index padding
 * (mmdet/models/detectors/single_stage.py:57-65) and SimpleVoxel.forward
 * (mmdet/models/backbones/vxnet.py:110-116).
 *
 * points: frames concatenated, frame b = rows [pt_off[b], pt_off[b+1]).
 * Outputs are bit-identical to the sequential reference per frame (first-touch
 * voxel order, first `max_points` points, stop at voxel `max_voxels`), rows of
 * frame b start at sum of the previous frames' counts:
 *   voxels [rows_cap, max_points, 4] (zero padded), coors [rows_cap,4] (b,z,y,x),
 *   num_points [rows_cap], mean [rows_cap,4] (may be NULL),
 *   d_frame_rows [batch+1] = exclusive row offsets, last = total rows.
 * ---------------------------------------------------------------------- */
typedef struct {
    float voxel_size[3];  /* x, y, z */
    float range_min[3];   /* x, y, z */
    int32_t grid[3];      /* x, y, z cells (1408, 1600, 40 under car_cfg) */
    int32_t max_points;   /* <= 8 */
    int32_t max_voxels;
} sassd_voxel_params;

size_t sassd_voxelize_workspace_bytes(int n_points_cap, int batch, int slots_per_frame);
int sassd_voxelize(const float* points, const int32_t* d_pt_off, int n_points_cap, int batch,
                   const sassd_voxel_params* host_params, int slots_per_frame,
                   float* voxels, int32_t* coors, int32_t* num_points, float* mean, int rows_cap,
                   int32_t* d_frame_rows, int32_t* d_status, void* ws, size_t ws_bytes, sassd_stream_t stream);

/* SimpleVoxel.forward alone (vxnet.py:110-116): mean[r,:] = sum_s voxels[r,s,:4] / num_points[r]. */
int sassd_voxel_mean(const float* voxels, const int32_t* num_points, const int32_t* d_rows, int rows_cap,
                     int max_points, float* mean, sassd_stream_t stream);

/* ------------------------------------------------------------------------
 * anchors_mask.  Replaces mmdet/datasets/kitti.py:333-343 +
 * mmdet/core/bbox3d/geometry.py:675-709 (occupancy count, two cumsums,
 * integral-image lookup, `> threshold`).  rects [n_anchors,4] int32 are the
 * clamped cell indices (c0,c1,c2,c3) of each anchor's near-axis-aligned
 * footprint — static, computed once on the host with the reference's fp32
 * arithmetic.  mask [batch, n_anchors] uint8.
 * ---------------------------------------------------------------------- */
size_t sassd_anchor_mask_workspace_bytes(int batch, int H, int W);
int sassd_anchor_mask(const int32_t* coors, const int32_t* d_rows, int rows_cap, int batch, int H, int W,
                      const int32_t* rects, int n_anchors, int threshold, uint8_t* mask,
                      void* ws, size_t ws_bytes, sassd_stream_t stream);

/* ------------------------------------------------------------------------
 * Rulebooks.  Replace spconv v1.0 `get_indice_pairs` (third-party; call sites
 * mmdet/models/necks/cmn.py:139-173,197-212).  The hot path uses a neighbour
 * table nbr[n_out, 27] (input row feeding output row o through kernel offset
 * k = (kz*3+ky)*3+kx, -1 = none); sassd_rulebook_pairs re-indexes it into the
 * spconv-v1 tables indice_pairs[2,27,n_cap] / indice_pair_num[27] (canonical
 * order: per offset ascending output row).
 * ---------------------------------------------------------------------- */
/* hash index over active coordinates: keys/vals [slots] int32, slots a power of two >= 2*n_cap. */
int sassd_hash_build(const int32_t* coors, const int32_t* d_rows, int rows_cap, int batch, int D, int H, int W,
                     int32_t* keys, int32_t* vals, int slots, int32_t* d_status, sassd_stream_t stream);
/* submanifold 3x3x3: output sites == input sites. */
/* tile_mask (optional): int32 [ceil(rows_cap / 128)], bit k of entry t = some row of rows [128t, 128t+128) has a
 * neighbour at offset k (consumed by sassd_spconv_f16x3 to skip absent taps). */
int sassd_rulebook_subm(const int32_t* coors, const int32_t* d_rows, int rows_cap, int D, int H, int W,
                        const int32_t* keys, const int32_t* vals, int slots, int32_t* nbr, int32_t* tile_mask,
                        sassd_stream_t stream);
/* strided conv (k=3,s=2,p=1): active output set, sorted by flattened (b,z,y,x). */
size_t sassd_rulebook_conv_workspace_bytes(int batch, int Do, int Ho, int Wo);
int sassd_rulebook_conv_outputs(const int32_t* coors_in, const int32_t* d_rows_in, int rows_cap_in, int batch,
                                int D, int H, int W, int32_t* coors_out, int32_t* d_rows_out, int rows_cap_out,
                                int32_t* d_status, void* ws, size_t ws_bytes, sassd_stream_t stream);
/* Same, and every output row is inserted into the hash index of the OUTPUT level as it is written (keys_out / vals_out
 * [slots_out], slots_out a power of two >= 2 * rows_cap_out; cleared here), which replaces that level's
 * sassd_hash_build launch.  Two kernels: mark (bitmap over the output grid) and a single-pass compaction (block scan
 * + decoupled look-back over the chunks of the bitmap). */
int sassd_rulebook_conv_outputs_hash(const int32_t* coors_in, const int32_t* d_rows_in, int rows_cap_in, int batch,
                                     int D, int H, int W, int32_t* coors_out, int32_t* d_rows_out, int rows_cap_out,
                                     int32_t* keys_out, int32_t* vals_out, int slots_out, int32_t* d_status, void* ws,
                                     size_t ws_bytes, sassd_stream_t stream);
/* neighbour table of the strided conv: nbr[o][k] = row of input cell 2*o - 1 + k. */
int sassd_rulebook_conv_nbr(const int32_t* coors_out, const int32_t* d_rows_out, int rows_cap_out, int D, int H, int W,
                            const int32_t* keys_in, const int32_t* vals_in, int slots_in, int32_t* nbr,
                            int32_t* tile_mask, sassd_stream_t stream);
int sassd_rulebook_pairs(const int32_t* nbr, const int32_t* d_rows_out, int rows_cap, int32_t* indice_pairs,
                         int32_t* indice_pair_num, sassd_stream_t stream);

/* ------------------------------------------------------------------------
 * Gathered implicit-GEMM convolution — one kernel family for
 *   SubMConv3d / SparseConv3d  (spconv v1.0 indice_conv; cmn.py:145-173,192-231)
 *   SparseConv3d 1x1x1         (cmn.py:208-212)
 *   nn.Conv2d 3x3 / 1x1 + BatchNorm2d(eval) + ReLU (BEVNet cmn.py:233-282,
 *     SSDRotateHead ssd_rotate_head.py:120-125,218-231, PSWarpHead.convs :424-429)
 *   out[m, :] = act( (sum_t in[row(m,t), :] @ W[t]) * scale + shift )
 * mode TABLE : row(m,t) = nbr[m*taps + t]            (sparse layers)
 * mode CONV2D: rows are pixels of a [batch,H,W] NHWC map, taps = 3x3 window, zero padding
 * mode ROWS  : taps == 1, row(m,0) = m                (1x1 convs / plain GEMM)
 * weight [taps, Cin, Cout] f32; scale/shift [Cout] (folded BatchNorm or bias); Cin % 4 == 0.
 * precision: SASSD_PREC_FP32 = CUDA-core FFMA; SASSD_PREC_TF32X3 / SASSD_PREC_F16X3 = tcgen05 tensor cores with a
 * 3-product hi/lo split of both operands (tf32: 21 bits, any range; fp16: 22 bits, |x| < 65504, 2x the MMA rate).
 * ---------------------------------------------------------------------- */
enum { SASSD_GCONV_TABLE = 0, SASSD_GCONV_CONV2D = 1, SASSD_GCONV_ROWS = 2 };
enum { SASSD_PREC_FP32 = 0, SASSD_PREC_TF32X3 = 1, SASSD_PREC_F16X3 = 2 };
typedef struct {
    int32_t mode, precision;
    int32_t cin, cout, taps;
    int32_t in_stride, out_stride; /* floats per row */
    int32_t rows_cap;              /* upper bound of rows (grid sizing) */
    int32_t batch, H, W;           /* CONV2D only */
    int32_t relu;
} sassd_gconv_desc;
int sassd_gconv(const sassd_gconv_desc* host_desc, const float* in, const float* weight, const float* scale,
                const float* shift, const int32_t* nbr, const int32_t* d_rows, float* out, sassd_stream_t stream);

/* The tensor-core precisions take their weights pre-split (hi / lo) and pre-swizzled for the shared-memory
 * operand layout: pack once per layer with sassd_gconv_pack (weight [taps,cin,cout] fp32 -> packed,
 * sassd_gconv_pack_bytes bytes) and pass `packed` as `weight`. */
size_t sassd_gconv_pack_bytes(int taps, int cin, int cout, int precision);
int sassd_gconv_pack(const float* weight, int taps, int cin, int cout, int precision, void* packed,
                     sassd_stream_t stream);

/* Dense NHWC conv (3x3 pad 1, or 1x1) + folded BatchNorm + ReLU on the "split map" activation format — the
 * BEVNet / head convolutions (cmn.py:264-282, ssd_rotate_head.py:218-231,424-429) with the activation operand
 * moved by TMA (cp.async.bulk.tensor) instead of producer warps.  A split map is two fp16 planes
 * [2][batch][H][W][C] (C % 64 == 0): hi = half(x), lo = half((x - hi) * 2048).  Outputs: fp32 NHWC
 * (out_f32, stride out_f32_stride) and/or the next layer's split map (out_split, out_split_ch channels).
 * wpack: sassd_gconv_pack(..., SASSD_PREC_F16X3).  16 < cout <= 256.  The stored input channels [cin, cin_stored)
 * must be zero.  What is written, per pixel of the map: the kernel computes N = cout rounded up to 32, 64, 128 or
 * 256 channels; of each output it writes channels [0, min(N, width)) (width = out_f32_stride or out_split_ch),
 * channels [cout, min(N, width)) as +0.0, and leaves channels [N, width) and all memory outside the buffers
 * untouched - a split map read as the next layer's input with out_split_ch > N must be zeroed beforehand.  Both
 * outputs carry the same values (the split one is the split of the fp32 one) and do not depend on which outputs
 * are requested, on tile_order or on n_split. */
typedef struct {
    int32_t batch, H, W;
    int32_t cin, cin_stored;       /* valid / stored input channels */
    int32_t cout, taps, relu;
    int32_t out_f32_stride, out_split_ch;
    int32_t tile_order;            /* sassd_conv2d_f16x3_occ: 0 = tiles round-robin over the CTAs (best with several steps
                                      in flight), 1 = computed tiles first, constant tiles after (best for one step at a
                                      time: no CTA gets two computed tiles while others only store constants) */
    int32_t n_split;               /* 0 / 1 = a work unit is a whole tile (all cout channels); 2 (cout > 128 only) = a unit
                                      is one half of a tile's output channels, N = 128 instructions: finer units for one
                                      step at a time on maps of a few hundred tiles (B <= 4), where whole tiles quantise
                                      badly over 148 SMs; costs a second read of the activation tile from L2 */
} sassd_conv2d_desc;
int sassd_conv2d_f16x3(const sassd_conv2d_desc* host_desc, const void* in_split, const void* wpack, const float* scale,
                       const float* shift, float* out_f32, void* out_split, sassd_stream_t stream);
/* Same, for maps that descend from a scattered sparse tensor and are therefore constant over large regions.
 * tile_dist[(b * tiles_y + ty) * tiles_x + tx] (written by sassd_split_rows_to_bev / sassd_sparse_to_bev_split into a
 * buffer pre-filled with a large value) is the Chebyshev distance in pixels from the SASSD_CONV2D_TILE_H x
 * SASSD_CONV2D_TILE_W tile to the nearest active cell of the scattered map.  `reach` = number of 3x3 convolutions
 * between that map and this layer's OUTPUT (1 for the first conv): a tile with tile_dist > reach that does not lie on
 * the image border (border tiles are always computed once reach >= 2, because the zero padding differs from the
 * constant) sees a constant input, so its output is the constant vector `const_out[cout]` (the caller obtains it by
 * running this same function on a small constant map - bit-identical to computing the tile).  Such tiles skip loads
 * and MMAs and only store.  tile_dist == NULL: plain sassd_conv2d_f16x3. */
#define SASSD_CONV2D_TILE_H 8
#define SASSD_CONV2D_TILE_W 16
#define SASSD_TILE_DIST_MAX 9          /* distances beyond this are stored as any larger value */
int sassd_conv2d_f16x3_occ(const sassd_conv2d_desc* host_desc, const void* in_split, const void* wpack,
                           const float* scale, const float* shift, float* out_f32, void* out_split,
                           const int32_t* tile_dist, int reach, const float* const_out, int32_t* counters,
                           sassd_stream_t stream);     /* counters: optional int32[2], += tiles computed, += tiles */
/* dense() of the last sparse tensor straight into a (pre-zeroed) split map [2,batch,H,W,D*C]. */
int sassd_sparse_to_bev_split(const float* feat, const int32_t* coors, const int32_t* d_rows, int rows_cap, int C,
                              int D, int H, int W, int batch, void* bev_split, int32_t* tile_dist,
                              sassd_stream_t stream);   /* tile_dist: optional, pre-filled with a large value, see above */

/* Ruled sparse conv on "split rows" (two fp16 planes [2][rows][C], C % 8 == 0; hi = half(x), lo = half((x-hi)*2048)):
 * same semantics as sassd_gconv TABLE / ROWS mode with SASSD_PREC_F16X3, but the gather is 16-byte cp.async copies
 * straight into the tensor-core operand tiles and the epilogue writes the next layer's planes (out_split, out_ch
 * channels) and/or fp32 rows.  taps == 1: row(m) = m.  cin <= 64, cout <= 64.  Only rows m < min(*d_rows, rows_cap)
 * are written; rows beyond them and all memory outside the buffers are left untouched.  The kernel computes N = cout
 * rounded up to 16, 32 or 64 channels; of each row it writes channels [0, min(N, width)) (width = out_ch or
 * out_f32_stride, rounded down to whole 8 / 4-channel groups), channels [cout, min(N, width)) as +0.0, and leaves
 * channels [N, width) untouched. */
typedef struct {
    int32_t cin, cout, taps;         /* cin = stored channels of the input planes */
    int32_t rows_cap, in_rows_cap;   /* output rows capacity; rows of the input planes (plane stride) */
    int32_t relu, out_ch, out_f32_stride;
} sassd_spconv_desc;
/* wpack for sassd_spconv_f16x3: weight [taps, cin, cout] fp32 -> sassd_spconv_pack_bytes(taps, cin_stored, cout)
 * bytes.  Narrow inputs are tap-packed: a 64-wide K chunk holds 64 / cin_stored taps (cin_stored 8, 16, 32). */
size_t sassd_spconv_pack_bytes(int taps, int cin_stored, int cout);
int sassd_spconv_pack(const float* weight, int taps, int cin, int cin_stored, int cout, void* packed,
                      sassd_stream_t stream);
/* tile_mask (optional, taps <= 27): int32 per SASSD_SPCONV_TILE_ROWS-row tile of the OUTPUT rows, bit t set when some
 * row of the tile has a neighbour at tap t (written by sassd_rulebook_subm / sassd_rulebook_conv_nbr); K chunks whose
 * taps are all absent are skipped (an absent pair contributes exactly zero, so the result is unchanged).
 * ws (optional, sassd_spconv_workspace_bytes()): scratch for the tap split - when the layer has at most half as many
 * tiles as CTAs, the two CTAs of a cluster share one tile's chunks and the peer's fp32 partial sums travel through
 * it.  counters (optional, int32[2], caller-zeroed): += executed (tile, chunk) pairs, += tiles (instrumentation). */
#define SASSD_SPCONV_TILE_ROWS 128
size_t sassd_spconv_workspace_bytes(void);
int sassd_spconv_f16x3(const sassd_spconv_desc* host_desc, const void* in_split, const void* wpack, const float* scale,
                       const float* shift, const int32_t* nbr, const int32_t* tile_mask, const int32_t* d_rows,
                       void* out_split, float* out_f32, void* ws, size_t ws_bytes, int32_t* counters,
                       sassd_stream_t stream);
/* fp32 rows [rows, cin] -> split rows [2][rows_cap][cs] (cs >= cin, cs % 8 == 0, padding channels +0.0).  Rows at or
 * beyond *d_rows (d_rows == NULL: rows_cap) are not written. */
int sassd_features_to_split(const float* feat, const int32_t* d_rows, int rows_cap, int cin, int cs, void* out_split,
                            sassd_stream_t stream);
/* dense() of split rows into a (pre-zeroed) split BEV map [2,batch,H,W,D*C]. */
int sassd_split_rows_to_bev(const void* feat_split, const int32_t* coors, const int32_t* d_rows, int rows_cap, int C,
                            int D, int H, int W, int batch, void* bev_split, int32_t* tile_dist, sassd_stream_t stream);
                            /* tile_dist: optional, pre-filled with a large value (sassd_conv2d_f16x3_occ) */

/* SparseConvTensor.dense() + view (cmn.py:112-114) into the NHWC BEV map the
 * neck consumes: bev[b, y, x, d*C + c] = feat[row, c]  (reference channel c*D+d;
 * the permutation is folded into the first BEV conv's weights).  The map must be
 * zeroed by the caller (cudaMemsetAsync). */
int sassd_sparse_to_bev(const float* feat, const int32_t* coors, const int32_t* d_rows, int rows_cap, int C,
                        int D, int H, int W, float* bev, sassd_stream_t stream);

/* ------------------------------------------------------------------------
 * second_box_decode + get_guided_anchors (ssd_rotate_head.py:53-91,307-372):
 * head [batch,H,W,head_stride] NHWC holds conv_box | conv_cls | conv_dir_cls
 * channels back to back; anchors [n_anchors,7] in (class,y,x,rot) order, one table shared by the
 * batch (anchors_per_frame = 0) or one per frame [batch,n_anchors,7] (anchors_per_frame = 1, the
 * reference's signature: ssd_rotate_head.py:316 indexes anchors[i]);
 * mask [batch,n_anchors] uint8.  Per frame, in anchor order: keep mask &&
 * max_c sigmoid(cls) > thr, decode, flip direction.  Outputs (capacity k_cap per frame):
 * boxes [batch,k_cap,7], labels [batch,k_cap] i32, index [batch,k_cap] i32
 * (anchor id), d_k [batch].
 * ---------------------------------------------------------------------- */
size_t sassd_decode_select_workspace_bytes(int batch, int n_anchors);
int sassd_decode_select(const float* head, int head_stride, int batch, int H, int W, int num_class,
                        const float* anchors, int anchors_per_frame, const uint8_t* mask, int n_anchors, float thr,
                        float* boxes, int32_t* labels, int32_t* index, int32_t* d_k, int k_cap,
                        int32_t* d_status, void* ws, size_t ws_bytes, sassd_stream_t stream);

/* PSWarpHead sampling (ssd_rotate_head.py:374-414,431-447): feat [batch,H,W,feat_stride]
 * NHWC with >= num_parts channels; part p = i*7+j samples channel p bilinearly at
 * the (i,j) tap of the 4x7 window of each guided box; score = mean over parts (logit). */
int sassd_pswarp(const float* feat, int feat_stride, int batch, int H, int W, const float* boxes,
                 const int32_t* d_k, int k_cap, float off_x, float off_y, float spatial_scale,
                 float* scores, sassd_stream_t stream);

/* ------------------------------------------------------------------------
 * get_rescore_bboxes (ssd_rotate_head.py:487-533) = sigmoid(score) > score_thr,
 * boxes3d_to_bev_torch (iou3d_utils.py:47-60), nms_gpu (iou3d_utils.py:114-128,
 * iou3d.cpp:73-120, iou3d_kernel.cu:250-292) with the greedy sweep on the
 * device, gather.  Sort is stable (score descending, then candidate order).
 * det [batch,det_cap,9] = (x,y,z,w,l,h,ry,score,label); d_ndet [batch].
 * Per frame the candidates are rows [0, min(d_k, k_cap)); rows beyond are not read.  More than nms_cap passing
 * candidates: the first nms_cap of them in candidate order go on (not the best-scoring ones), SASSD_FLAG_NMS_CAP.
 * More than det_cap kept boxes: det holds the first det_cap in score order, SASSD_FLAG_DET_CAP.  det rows at or
 * beyond d_ndet are not written.
 * ---------------------------------------------------------------------- */
size_t sassd_rescore_nms_workspace_bytes(int batch, int k_cap, int nms_cap);
int sassd_rescore_nms(const float* boxes, const float* scores, const int32_t* labels, const int32_t* d_k,
                      int batch, int k_cap, float score_thr, float iou_thr, int nms_cap,
                      float* det, int32_t* d_ndet, int det_cap, int32_t* d_status,
                      void* ws, size_t ws_bytes, sassd_stream_t stream);

/* iou3d_cuda.nms_gpu alone (iou3d.cpp:73-120): boxes [n,5] already sorted by
 * score; mask [n, ceil(n/64)] u64 in the reference layout (only columns j > i
 * are filled; the reference also fills the unused lower triangle); keep [n]
 * int64 indices, *d_nkeep their number.  ws: sassd_nms_workspace_bytes(n) bytes (0 for n == 0, where ws may be
 * NULL). */
size_t sassd_nms_workspace_bytes(int n);
int sassd_nms_mask(const float* boxes5, int n, float thr, uint64_t* mask, sassd_stream_t stream);
int sassd_nms_sorted(const float* boxes5, int n, float thr, int64_t* keep, int32_t* d_nkeep,
                     void* ws, size_t ws_bytes, sassd_stream_t stream);
/* iou3d_cuda.boxes_iou_bev_gpu (iou3d.cpp:52-71): dense [na, nb] rotated BEV IoU. */
int sassd_boxes_iou_bev(const float* boxes_a, int na, const float* boxes_b, int nb, float* iou, sassd_stream_t stream);

/* ---- KITTI evaluation support (SURVEY.md section 8 row f4) ----------------------------------------------------
 * Rotated-box overlap of the reference's evaluator (mmdet/core/post_processing/rotate_nms_gpu.py:536-627
 * rotate_iou_gpu_eval), batched over frames: boxes / query are concatenated [sum, 5] (x, y, dx, dy, angle) arrays
 * with per-frame offsets [nframes + 1]; out[out_off[f] + n * nq_f + k] = overlap(box n, query k) of frame f.
 * criterion: -1 IoU, 0 intersection / area(query), 1 intersection / area(box), 2 intersection area. */
int sassd_rotate_overlap_eval(const float* boxes, const int32_t* box_off, const float* query, const int32_t* query_off,
                              const int64_t* out_off, int nframes, int criterion, int max_pairs_per_frame, float* out,
                              sassd_stream_t stream);
/* HOST function (all pointers are host memory): greedy GT<->detection matching of the KITTI protocol
 * (mmdet/core/evaluation/kitti_eval.py:164-283, :295-342).  nthresh == 0: collect the scores of the true positives
 * (tp_scores capacity = number of gt rows); nthresh > 0: pr[t] += (tp, fp, fn, similarity) for every threshold. */
int sassd_kitti_match(int nframes, const double* overlaps, const int64_t* ov_off, const int32_t* gt_off,
                      const int32_t* dt_off, const int32_t* dc_off, const double* gt_alpha, const double* dt_alpha,
                      const double* dt_score, const double* dt_bbox, const double* dc_bbox, const int32_t* ign_gt,
                      const int32_t* ign_dt, int metric, double min_overlap, int compute_aos, int nthresh,
                      const double* thresholds, double* pr, double* tp_scores, int64_t* n_tp_scores);

#ifdef __cplusplus
}
#endif
#endif /* SASSD_B200_H */
