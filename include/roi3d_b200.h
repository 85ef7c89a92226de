/*
 * roi3d_b200.h -- C ABI of libroi3d_b200.so: the B200-native (sm_100a) 3D R-CNN RoI hot path.
 *
 * This is the drop-in boundary.  Each entry point replaces one native entry point (or the torch-op
 * composition) of the reference arthur801031/3d-multi-resolution-rcnn; the reference interface is cited
 * per function as file:line under /root/reference.  The reference binds its natives with pybind11 over
 * at::Tensor; here the boundary is plain pointers + sizes + a CUDA stream, so any host (the Python
 * mirror in 3d-multi-resolution-rcnn_b200/roi3d_b200, ctypes, cffi, C++) can bind it.  INTEGRATION.md
 * shows the stub a reference maintainer adds to mmdet/ops.
 *
 * Conventions
 *   - Every `const float*`/`float*` named *_dev is a DEVICE pointer on the current CUDA device; entry
 *     points ending in `_host` take HOST pointers and do their own H2D/D2H.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  All device entry
 *     points are asynchronous on that stream and never synchronise the host.
 *   - Return value: 0 on success, a negative ROI3D_E* code on failure; roi3d_last_error() returns a
 *     thread-local message.  Nothing prints, nothing calls exit() (the reference does both:
 *     roi_align_cuda.cpp:80-83, roi_align_kernel.cu:679-682).
 *   - Boxes are (x1,y1,x2,y2,z1,z2) in input-image pixels with the +1 size convention
 *     (nms_kernel.cu:23-33); RoIs are (batch_idx, x1,y1,x2,y2,z1,z2) fp32 (roi_align_kernel.cu:231-238).
 *   - Feature layout: ROI3D_NCDHW is the reference's contiguous [B,C,D,H,W]; ROI3D_NDHWC is the same
 *     logical tensor stored channels-last ([B,D,H,W,C] in memory, torch.channels_last_3d).  The FORWARD
 *     entries take either: channels-last levels feed the streamed / per-warp kernels, NCDHW levels are read
 *     in place -- by the streamed kernel's NCDHW twin (7 x 7 x PD outputs, C % 64 == 0) or the planar kernel
 *     (square 7- or 14-wide outputs); both want 16-byte aligned levels and W % 4 == 0, other NCDHW shapes
 *     return ROI3D_EINVAL: convert with roi3d_ncdhw_to_ndhwc.  The BACKWARD entries
 *     accumulate into channels-last (ROI3D_NDHWC) gradients only.
 */
#ifndef ROI3D_B200_H_
#define ROI3D_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ROI3D_ABI_VERSION 1

#define ROI3D_NCDHW 0
#define ROI3D_NDHWC 1

#define ROI3D_OK 0
#define ROI3D_EINVAL (-1)  /* bad argument (shape, alignment, unsupported size) */
#define ROI3D_ECUDA (-2)   /* CUDA runtime / launch error */
#define ROI3D_ENOMEM (-3)  /* workspace too small / allocation failed */

#define ROI3D_MAX_LEVELS 8

int roi3d_abi_version(void);
const char *roi3d_last_error(void);
/* SM count / name of the current device (for grid sizing in the host mirror and for bench.py). */
int roi3d_device_info(int *sm_count, int *cc_major, int *cc_minor, size_t *l2_bytes);

/* ------------------------------------------------------------------------------------------------
 * One FPN level as the RoI extractor sees it.
 * Replaces: the (features, spatial_scale, spatial_scale_depth) triple held by each RoIAlign3D module,
 * mmdet/ops/roi_align/modules/roi_align_3d.py:7-18, built per stride pair in
 * mmdet/models/roi_extractors/single_level.py:45-56.
 * ---------------------------------------------------------------------------------------------- */
typedef struct roi3d_level {
  const float *feats_dev; /* forward input; may be NULL for backward-only calls */
  float *grad_dev;        /* backward output (same shape/layout as feats), accumulated into */
  int32_t layout;         /* ROI3D_NCDHW or ROI3D_NDHWC */
  int32_t D, H, W;
  float spatial_scale;       /* 1/stride      (x,y) */
  float spatial_scale_depth; /* 1/depth_stride (z)  */
} roi3d_level_t;

/* ------------------------------------------------------------------------------------------------
 * RoIAlign3D forward.
 * Replaces: roi_align_cuda.forward3d -> roi_align_forward_cuda_3d -> ROIAlignForwardLaucher3D,
 *   mmdet/ops/roi_align/src/roi_align_cuda.cpp:68-94, roi_align_kernel.cu:316-337 (kernel :214-291).
 * out_dev: [K, C, PD, PH, PW] contiguous, fully overwritten (no pre-zeroing needed, unlike
 *   functions/roi_align_3d.py:32).  feats: [B,C,D,H,W] in `layout` (ROI3D_NDHWC or ROI3D_NCDHW, see above).
 * ---------------------------------------------------------------------------------------------- */
int roi3d_roi_align3d_forward(const float *feats_dev, int layout, int B, int C, int D, int H, int W,
                              const float *rois_dev, int K, int PD, int PH, int PW, float spatial_scale,
                              float spatial_scale_depth, int sample_num, float *out_dev, void *stream);

/* Forward with an output row map: the tile of RoI k is written to row out_rows_dev[k] of out_dev (NULL = row k).
 * out_dev may be mapped pinned host memory (the kernel's streaming stores then cross PCIe directly), which is how
 * roi3d_roi_align3d_forward_host returns results while later z slabs of the volume are still being uploaded. */
int roi3d_roi_align3d_forward_rows(const float *feats_dev, int layout, int B, int C, int D, int H, int W,
                                   const float *rois_dev, int K, int PD, int PH, int PW, float spatial_scale,
                                   float spatial_scale_depth, int sample_num, float *out_dev,
                                   const int32_t *out_rows_dev, void *stream);

/* ------------------------------------------------------------------------------------------------
 * RoIAlign3D backward.
 * Replaces: roi_align_cuda.backward3d -> ROIAlignBackwardLaucher3D,
 *   roi_align_cuda.cpp:123-150, roi_align_kernel.cu:666-692 (kernel :519-636).
 * grad_in_dev [B,C,D,H,W], `layout` must be ROI3D_NDHWC, is ACCUMULATED into (caller zero-fills, as
 *   functions/roi_align_3d.py:84 does); pass zero_fill=1 to have the library clear it first.
 * bug_compat=1 reproduces the reference's top_diff index for non-cubic outputs
 *   (roi_align_kernel.cu:554-555; SURVEY F2); default 0 = the mathematically correct gradient.
 * ---------------------------------------------------------------------------------------------- */
int roi3d_roi_align3d_backward(const float *grad_out_dev, const float *rois_dev, int K, int PD, int PH, int PW,
                               float spatial_scale, float spatial_scale_depth, int sample_num,
                               float *grad_in_dev, int layout, int B, int C, int D, int H, int W,
                               int zero_fill, int bug_compat, void *stream);

/* ------------------------------------------------------------------------------------------------
 * FPN level mapping.
 * Replaces: SingleRoIExtractor.map_roi_levels, mmdet/models/roi_extractors/single_level.py:58-82
 *   (about 8 torch elementwise launches).  lvls_dev: int64[K].
 * ---------------------------------------------------------------------------------------------- */
int roi3d_map_roi_levels(const float *rois_dev, int K, int num_levels, float finest_scale, int64_t *lvls_dev,
                         void *stream);

/* ------------------------------------------------------------------------------------------------
 * Fused multi-level RoI extractor, forward and backward: level mapping + per-level RoIAlign3D +
 * scatter into one [K,C,PD,PH,PW] tensor in ONE launch, no host sync.
 * Replaces: SingleRoIExtractor.forward, single_level.py:84-104 (per-level mask, .any() sync,
 *   boolean-index gather, RoIAlign3D launch, index-add), and its autograd backward.
 * All levels share B and C.  lvls_out_dev may be NULL.
 * ---------------------------------------------------------------------------------------------- */
int roi3d_extract_forward(const roi3d_level_t *levels, int num_levels, int B, int C, const float *rois_dev,
                          int K, int PD, int PH, int PW, int sample_num, float finest_scale, float *out_dev,
                          int64_t *lvls_out_dev, void *stream);
int roi3d_extract_backward(const roi3d_level_t *levels, int num_levels, int B, int C, const float *rois_dev,
                           int K, int PD, int PH, int PW, int sample_num, float finest_scale,
                           const float *grad_out_dev, int zero_fill, int bug_compat, void *stream);

/* Deterministic form of roi3d_extract_backward: the same gradient, the same bits on every run (no float atomics; what
 * torch.use_deterministic_algorithms(True) asks for).  Each gradient voxel is written once by its owner, which adds
 * the contributions of the RoIs that touch it in ascending RoI index.  accumulate=0: every voxel of every level's
 * grad_dev is overwritten, K == 0 included (zeros; no memset needed); accumulate=1: each voxel's finished sum is added
 * to its old value with one fp32 add.  num_levels == 1 is the plain RoIAlign3D backward.  Channels-last (ROI3D_NDHWC)
 * gradients only; any output size and channel count; no bug_compat (the correct gradient only). */
int roi3d_extract_backward_deterministic(const roi3d_level_t *levels, int num_levels, int B, int C,
                                         const float *rois_dev, int K, int PD, int PH, int PW, int sample_num,
                                         float finest_scale, const float *grad_out_dev, int accumulate, void *stream);

/* Layout conversion of one level, [B,C,D,H,W] <-> channels-last; used by the host mirror when a caller
 * hands the reference's NCDHW-contiguous tensors to the channels-last kernels. */
int roi3d_ncdhw_to_ndhwc(const float *src_dev, float *dst_dev, int B, int C, int D, int H, int W, void *stream);
int roi3d_ndhwc_to_ncdhw(const float *src_dev, float *dst_dev, int B, int C, int D, int H, int W, void *stream);

/* ------------------------------------------------------------------------------------------------
 * 3D IoU NMS, batched over independent segments (one segment = one (volume, level) or one class).
 * Replaces: nms_cuda.nms_3d -> nms_cuda_3d, mmdet/ops/nms/src/nms_cuda.cpp:16-21,
 *   nms_kernel.cu:196-257 (kernel :81-129): device sort, 64x64 IoU bitmask, blocking D2H copy of
 *   the mask and a host sweep.  Here the order, the mask (upper triangle only) and the sweep all run
 *   on the device.
 * dets_dev: [nseg, n_max, 7] fp32 (x1,y1,x2,y2,z1,z2,score); segment s uses its first
 *   seg_counts_dev[s] rows (seg_counts_dev == NULL: every segment has n_max rows).
 * keep_dev: int64 [nseg, n_max]: kept ORIGINAL row indices, ascending (nms_kernel.cu:253-256).
 * keep_by_score_dev (optional, may be NULL): the same indices in descending-score order
 *   (what `dets[inds][:nms_post]` needs when the input was already score-sorted).
 * num_keep_dev: int32 [nseg].
 * Order rule for equal scores: lower original index first (SURVEY F6).
 * ---------------------------------------------------------------------------------------------- */
size_t roi3d_nms3d_workspace_bytes(int nseg, int n_max);
int roi3d_nms3d_batched(const float *dets_dev, const int32_t *seg_counts_dev, int nseg, int n_max,
                        float iou_thr, int64_t *keep_dev, int64_t *keep_by_score_dev, int32_t *num_keep_dev,
                        void *workspace_dev, size_t workspace_bytes, void *stream);

/* Same as roi3d_nms3d_batched; presorted_dev (optional uint8 [nseg]) marks segments whose rows the caller already
 * holds in (score descending, equal scores by ascending row) order -- rows straight out of roi3d_topk_segmented --
 * so the ranking pass is skipped for them.  A segment marked presorted that is not gives undefined keep lists. */
int roi3d_nms3d_batched_presorted(const float *dets_dev, const int32_t *seg_counts_dev, const uint8_t *presorted_dev,
                                  int nseg, int n_max, float iou_thr, int64_t *keep_dev, int64_t *keep_by_score_dev,
                                  int32_t *num_keep_dev, void *workspace_dev, size_t workspace_bytes, void *stream);

/* Same as roi3d_nms3d_batched_presorted with an early stop for the proposal path, which only uses the first nms_post
 * kept boxes of a score-sorted level (`proposals[:nms_post]`, rpn_head_3d.py:135): for a segment flagged presorted the
 * greedy sweep ends with the 64-box tile in which the kept count reaches max_keep_presorted.  num_keep of such a segment
 * is then between max_keep_presorted and max_keep_presorted + 63, keep_by_score holds that prefix of the full list and
 * keep (ascending index) the same boxes.  Segments not flagged, and max_keep_presorted <= 0, are swept in full. */
int roi3d_nms3d_batched_limited(const float *dets_dev, const int32_t *seg_counts_dev, const uint8_t *presorted_dev,
                                int nseg, int n_max, float iou_thr, int max_keep_presorted, int64_t *keep_dev,
                                int64_t *keep_by_score_dev, int32_t *num_keep_dev, void *workspace_dev,
                                size_t workspace_bytes, void *stream);

/* Evaluation-time flavour of the same NMS (SURVEY section 8f, N1).
 * Replaces: nms_3d_python, mmdet/core/evaluation/coco_utils.py:245-282 (numpy float64, per volume, called from
 *   apply_nms :306-332 with thr 0.1): IoU evaluated in float64 in numpy's operation order on the fp32 boxes,
 *   a box is dropped unless iou <= iou_thr (so a NaN iou drops it).  keep_by_score_dev is the reference's return
 *   order (descending score; equal scores: lower index first); keep_dev (ascending index) must be non-NULL too. */
int roi3d_nms3d_eval_batched(const float *dets_dev, const int32_t *seg_counts_dev, int nseg, int n_max, double iou_thr,
                             int64_t *keep_dev, int64_t *keep_by_score_dev, int32_t *num_keep_dev,
                             void *workspace_dev, size_t workspace_bytes, void *stream);

/* Host-buffer form of one NMS call: what mmdet.ops.nms(dets_numpy, thr, device_id) does
 * (mmdet/ops/nms/nms_wrapper.py:29-32,42-52).  keep_host capacity n; returns count in *num_keep_host. */
int roi3d_nms3d_host(const float *dets_host, int n, float iou_thr, int64_t *keep_host, int32_t *num_keep_host);

/* ------------------------------------------------------------------------------------------------
 * Training-time glue between the proposal path and RoIAlign (SURVEY section 8f, N2).
 *
 * roi3d_bbox_overlaps3d: dense IoU matrix iou[m, n] of boxes1[m] x boxes2[n] (rows of `stride` floats, the first six
 *   are x1,y1,x2,y2,z1,z2).  Replaces: bbox_overlaps, 6-column non-aligned branch, mmdet/core/bbox/geometry.py:49-60.
 * roi3d_assign_max_iou: MaxIoUAssigner.assign -> assign_wrt_overlaps, mmdet/core/bbox/assigners/
 *   max_iou_assigner.py:100,128-171, fused over the IoU (the [k, n] matrix is never stored).  Rules in order:
 *   -1 by default; 0 where neg_iou_lo <= max_overlap < neg_iou_hi (a float neg_iou_thr t is the pair (0, t));
 *   argmax + 1 where max_overlap >= pos_iou_thr; then for every gt i in ascending order with
 *   gt_max[i] >= min_pos_iou: i + 1 for every box whose IoU equals gt_max[i] (gt_max_assign_all) or for the
 *   lowest-index such box.  Ties of the per-box argmax go to the lowest gt index.  assigned_labels_dev (optional)
 *   = gt_labels[assigned - 1] for positives, 0 otherwise.  n == 0 or k == 0 is an error like the reference's
 *   ValueError.
 * roi3d_assign_max_iou_ignore: the same with the ignore-region branch (max_iou_assigner.py:101-111): boxes whose
 *   ignore_flags_dev byte is non-zero have their whole column of the overlap matrix read -1, so they stay -1
 *   ("ignore") unless they attain a gt's maximum of -1.  The caller derives the flags from
 *   roi3d_bbox_overlaps3d(bboxes, gt_bboxes_ignore) > ignore_iof_thr -- for 6-column boxes the reference's
 *   bbox_overlaps ignores mode='iof' and returns the IoU (geometry.py:49-60).  NULL flags = the plain entry.
 * roi3d_bbox2delta3d: bbox2delta3d, mmdet/core/bbox/transforms.py:33-63; deltas [n, 6] = (dx, dy, dw, dh, dz, dd);
 *   means6 / stds6 are HOST pointers to six floats (NULL = 0 / 1).
 * ---------------------------------------------------------------------------------------------- */
/* Anchors of one level in closed form and / or their inside flags, one launch (SURVEY section 8f, N3).
 * Replaces: AnchorGenerator3D.grid_anchors + valid_flags, mmdet/core/anchor/anchor_generator_3d.py:56-92 (numpy
 *   meshgrid + H2D per call) and anchor_inside_flags, mmdet/core/anchor/anchor_target.py:203-217.
 * anchors_dev [A*D*H*W, 6] fp32 and flags_dev [A*D*H*W] uint8 (either may be NULL); flat index
 * ((y*W + x)*D + z)*A + a; flag = x < valid_w && y < valid_h && z < valid_d, and if allowed_border >= 0 also
 * x1,y1,z1 >= -border, x2 < img_w + border, y2 < img_h + border, z2 < img_d + border.  base_anchors_host: [A,6]. */
int roi3d_grid_anchors(int A, int D, int H, int W, float stride, float depth_stride, const float *base_anchors_host,
                       int valid_d, int valid_h, int valid_w, float img_h, float img_w, float img_d, int allowed_border,
                       float *anchors_dev, uint8_t *flags_dev, void *stream);
int roi3d_bbox_overlaps3d(const float *boxes1_dev, int m, int stride1, const float *boxes2_dev, int n, int stride2,
                          float *iou_dev, void *stream);
size_t roi3d_assign_workspace_bytes(int n, int k);
int roi3d_assign_max_iou(const float *bboxes_dev, int n, int stride, const float *gt_dev, int k,
                         const int64_t *gt_labels_dev, float pos_iou_thr, float neg_iou_lo, float neg_iou_hi,
                         float min_pos_iou, int gt_max_assign_all, int64_t *assigned_gt_inds_dev,
                         float *max_overlaps_dev, int64_t *assigned_labels_dev, void *workspace_dev,
                         size_t workspace_bytes, void *stream);
int roi3d_assign_max_iou_ignore(const float *bboxes_dev, int n, int stride, const float *gt_dev, int k,
                                const int64_t *gt_labels_dev, const uint8_t *ignore_flags_dev, float pos_iou_thr,
                                float neg_iou_lo, float neg_iou_hi, float min_pos_iou, int gt_max_assign_all,
                                int64_t *assigned_gt_inds_dev, float *max_overlaps_dev, int64_t *assigned_labels_dev,
                                void *workspace_dev, size_t workspace_bytes, void *stream);
int roi3d_bbox2delta3d(const float *proposals_dev, int stride_p, const float *gt_dev, int stride_g, int n,
                       const float *means6, const float *stds6, float *deltas_dev, void *stream);
/* delta2bbox3D for class-wise deltas (the bbox head's decode; mmdet/core/bbox/transforms.py:105-160): deltas [n, 6k]
 * applied to rois [n, >= 6] (row stride stride_r), out [n, 6k].  dw, dh, dz AND dd are clamped with |log(wh_ratio_clip)|
 * as the reference does (:122-128; its d_ratio_clip argument is unused).  img_w <= 0: no clamp to the image
 * (max_shape=None); otherwise x in [0, img_w - 1], y in [0, img_h - 1], z in [0, img_d - 1]. */
int roi3d_delta2bbox3d(const float *rois_dev, int stride_r, const float *deltas_dev, int n, int num_classes,
                       const float *means6, const float *stds6, float wh_ratio_clip, float img_h, float img_w, float img_d,
                       float *out_dev, void *stream);

/* ------------------------------------------------------------------------------------------------
 * Mask paste (SURVEY section 8f, N4): per detection sigmoid -> resize to the box -> threshold.
 * Replaces: FCNMaskHead3D.get_seg_masks, mmdet/models/mask_heads/fcn_mask_head_3d.py:144-187 (host numpy +
 *   skimage.transform.resize per detection).  mask_logits_dev [n, Dm, Hm, Wm] fp32 (the class channel already
 *   selected); boxes_dev int32 [n, 6] = (x1, y1, x2, y2, z1, z2) after the reference's `(bbox / scale).astype(int32)`;
 *   detection i's binary mask of max(z2-z1+1,1) x max(y2-y1+1,1) x max(x2-x1+1,1) voxels (z, y, x order) is written
 *   at out_dev + offsets_dev[i].  The resize restates scikit-image 0.18.0 `resize` (n-D branch: gaussian
 *   anti-aliasing + order-1 map_coordinates, mode reflect) in float64 like scipy.
 * ---------------------------------------------------------------------------------------------- */
int roi3d_mask_paste(const float *mask_logits_dev, int n, int Dm, int Hm, int Wm, const int32_t *boxes_dev,
                     const int64_t *offsets_dev, float thr, uint8_t *out_dev, void *stream);

/* Mask targets (SURVEY section 8f, N4, training half).
 * Replaces: mask_target_single, mmdet/core/mask/mask_target.py:17-50 (per positive proposal on the host: crop of the
 *   assigned ground-truth mask to the proposal's int32 box, `255 * skimage.transform.resize(crop, (Md, Mh, Mw))`,
 *   `.astype(uint8)`, non-zero -> 1).  gt_masks_dev uint8 [G, D, H, W]; boxes_host int32 [n, 6] = (x1,y1,x2,y2,z1,z2)
 *   after the reference's `.astype(np.int32)`; gt_inds_host int64 [n]; out_dev fp32 [n, Md, Mh, Mw] of 0 / 1.
 *   The crop is clipped to the volume like a numpy slice; an empty crop gives an all-zero target (the reference's
 *   resize raises on it).  The resize restates scikit-image 0.18.0 `resize` on a uint8 input (img_as_float, gaussian
 *   anti-aliasing, order-1 map_coordinates, mode reflect, clip) in float64.
 *   crop_dhw_host for the workspace query: int32 [n, 3] = clipped (d, h, w) of every crop. */
size_t roi3d_mask_target_workspace_bytes(const int32_t *crop_dhw_host, int n);
int roi3d_mask_target(const uint8_t *gt_masks_dev, int G, int D, int H, int W, const int32_t *boxes_host,
                      const int64_t *gt_inds_host, int n, int Md, int Mh, int Mw, float *out_dev, void *workspace_dev,
                      size_t workspace_bytes, void *stream);

/* Experiment knob (not part of the reference surface): key 0 = forward kernel variant (0 = auto, 1 = one channel per
 * lane, 50 = per-warp ring kernel where the streamed kernel would apply, 60 = planar kernel on channels-last 7-wide
 * outputs, 99 = literal reference-order path); key 1 = backward kernel variant (0 = auto: streamed / planar where they
 * apply, 50 = per-warp kernel, 60 = planar backward on 7-wide outputs, 1, 3 = per-warp tables, 99 = literal); key 2 =
 * sub-items one ring-kernel warp walks per RoI (0 = auto); key 4 = volume size in KB from which
 * roi3d_roi_align3d_forward_host pipelines its copies (0 = auto, 32 MB; -1 = never); key 6 = NMS mask kernel variant;
 * key 7 = ring geometry of the streamed forward kernel (0 = 3 x 42 KB, 1 = 4 x 32 KB, 2 = 5 x 24 KB); key 9 = streamed
 * kernel experiments (bit 0: no arithmetic, bit 1: no output store, bit 2: no largest-first order); key 10 = plane
 * storage of the planar kernels per CTA in floats (0 = 18432); key 11 = top-k sieve path (0 = on where it applies,
 * -1 = digit passes only, 2 = the sieve gives up on every segment so that its fallback runs -- tests). */
int roi3d_set_tuning(int key, int value);

/* Measurement hook (not part of the reference surface): two cudaEvent_t (as void*) that the calling thread's next
 * roi3d_roi_align3d_forward / roi3d_extract_forward calls record right before and right after the launch of the streamed
 * forward kernel, so that a benchmark can time the dominant kernel by itself; NULL, NULL switches it off.  With the
 * events set the plan kernel no longer overlaps the main kernel's start (the event sits between the two launches). */
int roi3d_set_kernel_timing_events(void *start_event, void *stop_event);

/* Host-buffer form of RoIAlign3D forward (H2D feats+rois, kernel, D2H out): the e2e path bench.py times. */
int roi3d_roi_align3d_forward_host(const float *feats_host, int layout, int B, int C, int D, int H, int W,
                                   const float *rois_host, int K, int PD, int PH, int PW, float spatial_scale,
                                   float spatial_scale_depth, int sample_num, float *out_host);

/* ------------------------------------------------------------------------------------------------
 * RPN proposal path pieces (RPNHead3D.get_bboxes_single,
 * mmdet/models/anchor_heads/rpn_head_3d.py:72-149).
 * ---------------------------------------------------------------------------------------------- */

/* Segmented top-k by radix select: for each segment s (n_s = seg_len[s] scores starting at
 * scores_dev + seg_off[s]) the k_s = min(k, n_s) largest, DESCENDING, ties -> lower index.
 * Replaces: scores.topk(cfg.nms_pre), rpn_head_3d.py:108-112, and the final topk :147.
 * apply_sigmoid=1 ranks sigmoid(x) = 1/(1+exp(-x)) (rpn_head_3d.py:90) and returns those values.
 * seg_off/seg_len are HOST arrays (int64) of length nseg.
 * seg_adhw (HOST int32 [nseg,4] = A,D,H,W, or NULL): when given (A>0), segment s is an [A,D,H,W] score map
 *   and indices are LOGICAL positions after permute(2,3,1,0).reshape(-1) (rpn_head_3d.py:87-89), i.e.
 *   ((y*W + x)*D + z)*A + a -- the order grid_anchors enumerates anchors in -- both for the returned index
 *   and for the tie rule; memory is still read in its native order.
 * out_idx_dev: int64 [nseg, k] (index within the segment); out_val_dev: fp32 [nseg, k];
 * rows beyond k_s are filled with -1 / 0. */
size_t roi3d_topk_workspace_bytes(int nseg, int k);
/* Workspace that additionally holds one u32 key per score (total_len = sum of seg_len): when the workspace passed to
 * the top-k entries is at least this large, the first digit pass stores every element's order-preserving key
 * (sigmoid, mask lookup and the HBM read happen once) and the later full passes read the keys back from L2. */
size_t roi3d_topk_workspace_bytes_keys(int nseg, int k, int64_t total_len);
int roi3d_topk_segmented(const float *scores_dev, const int64_t *seg_off, const int64_t *seg_len,
                         const int32_t *seg_adhw, int nseg, int k, int apply_sigmoid, int64_t *out_idx_dev,
                         float *out_val_dev, void *workspace_dev, size_t workspace_bytes, void *stream);
/* Same, with the reference's "sort a level only if it has more than nms_pre anchors" rule
 * (rpn_head_3d.py:96,108-112): with small_segments_in_index_order != 0 a segment no longer than k is returned in
 * ascending logical index (all of it), not in score order. */
int roi3d_topk_segmented_ex(const float *scores_dev, const int64_t *seg_off, const int64_t *seg_len,
                            const int32_t *seg_adhw, int nseg, int k, int apply_sigmoid,
                            int small_segments_in_index_order, int64_t *out_idx_dev, float *out_val_dev,
                            void *workspace_dev, size_t workspace_bytes, void *stream);

/* Same, with the head's cached inside-flag masks (RPNHead3D.pos_indices / pos_indices_test, set at
 * mmdet/models/anchor_heads/anchor_head_3d.py:212,239-243 and applied as `scores = scores[pos_indices]` before the
 * top-k, rpn_head_3d.py:97-106): seg_mask_dev_ptrs is a HOST array [nseg] of DEVICE pointers (NULL entry, or a NULL
 * array, = no mask) to uint8 masks indexed by the segment's LOGICAL index; only elements with a non-zero mask byte take
 * part, and a segment's length for the k / small-segment rules is its masked-in count.  Returned indices are logical
 * positions in the unmasked segment (what the decode step needs), in the order `scores[pos_indices].topk(k)` yields.
 * out_count_dev (optional int32 [nseg]): rows returned per segment; out_sorted_dev (optional uint8 [nseg]): 1 = rows in
 * score order, 0 = small segment returned in ascending index order.  Both are written on the device (no host read). */
int roi3d_topk_segmented_masked(const float *scores_dev, const int64_t *seg_off, const int64_t *seg_len,
                                const int32_t *seg_adhw, const uint8_t *const *seg_mask_dev_ptrs, int nseg, int k,
                                int apply_sigmoid, int small_segments_in_index_order, int64_t *out_idx_dev,
                                float *out_val_dev, int32_t *out_count_dev, uint8_t *out_sorted_dev, void *workspace_dev,
                                size_t workspace_bytes, void *stream);

/* Tail of RPNHead3D.get_bboxes_single for all (image, level) segments (rpn_head_3d.py:135-148): the first
 * min(num_keep, nms_post) kept rows of every level, in NMS return order, concatenated per image in level order.
 * dets_dev [B*L, k, 7]; keep lists [B*L, k] from roi3d_nms3d_batched; use_index_order_dev (optional uint8 [B*L]):
 * 1 = take keep_by_index for that segment (levels that were not score-sorted).  Outputs: cat_props_dev
 * [B, L*P, 7], cat_scores_dev [B, L*P] (-inf past the valid rows), n_valid_dev int32 [B]; P = min(nms_post, k). */
int roi3d_rpn_collect(const float *dets_dev, int num_images, int num_levels, int k, const int64_t *keep_by_score_dev,
                      const int64_t *keep_by_index_dev, const int32_t *num_keep_dev,
                      const uint8_t *use_index_order_dev, int nms_post, float *cat_props_dev, float *cat_scores_dev,
                      int32_t *n_valid_dev, void *stream);
/* out[s][j] = rows[s][idx[s][j]] for 7-float rows (idx < 0 -> zeros): the final `proposals[topk_inds]`, :147-148. */
int roi3d_gather_rows7(const float *rows_dev, int nseg, int rows_per_seg, const int64_t *idx_dev, int n,
                       float *out_dev, void *stream);

/* Anchor base + decode of selected anchors for one level, fused:
 *   anchors as AnchorGenerator3D.grid_anchors would generate them
 *   (mmdet/core/anchor/anchor_generator_3d.py:56-71: flat index = ((y*W + x)*D + z)*A + a),
 *   deltas gathered from bbox_pred [6A, D, H, W] as permute(2,3,1,0).reshape(-1,6) would
 *   (rpn_head_3d.py:94), then delta2bbox3D (mmdet/core/bbox/transforms.py:105-160) with the
 *   img_shape clamp, and the score appended (rpn_head_3d.py:133).
 * idx_dev: int64[n] flat anchor indices (e.g. from roi3d_topk_segmented); -1 entries produce a zero row.
 * base_anchors_host: [A,6] fp32 HOST.  out_dev: [n,7]. */
int roi3d_decode_proposals(const float *bbox_pred_dev, int A, int D, int H, int W, float stride,
                           float depth_stride, const float *base_anchors_host, const int64_t *idx_dev,
                           const float *scores_dev, int n, const float *means6_host, const float *stds6_host,
                           float img_h, float img_w, float img_d, float *out_dev, void *stream);

/* Batched form of roi3d_decode_proposals: every (image, level) segment in one launch.
 * bbox_pred_dev_ptrs: HOST array [nseg] of device pointers to that segment's [6A,D,H,W] map; seg_adhw HOST int32
 * [nseg,4]; seg_level HOST int32 [nseg] (index into the per-level tables); seg_img_hwd HOST fp32 [nseg,3] =
 * (img H, W, D) or NULL for no clamp; base_anchors_host [num_levels, A, 6]; strides per level.
 * idx_dev/scores_dev: [nseg,k] (e.g. straight from roi3d_topk_segmented); out_dev: [nseg,k,7]. */
int roi3d_decode_proposals_batched(const float *const *bbox_pred_dev_ptrs, const int32_t *seg_adhw,
                                   const int32_t *seg_level, const float *seg_img_hwd, int nseg, int num_levels,
                                   int A, const float *base_anchors_host, const float *strides_host,
                                   const float *depth_strides_host, const int64_t *idx_dev, const float *scores_dev,
                                   int k, const float *means6_host, const float *stds6_host, float *out_dev,
                                   void *stream);

#ifdef __cplusplus
}
#endif
#endif /* ROI3D_B200_H_ */
