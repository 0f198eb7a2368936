/*
 * sfod_b200.h -- C ABI of libsfod_b200.so: the B200 (sm_100a) implementation of the
 * simple-SFOD teacher-student pseudo-labelling hot path (SURVEY.md section 8).
 *
 * The reference (EPFL-IMOS/simple-SFOD) is pure Python and has NO FFI of its own: its
 * arithmetic is reached through detectron2 0.6 -> torchvision / ATen operators.  Every
 * entry point below therefore cites the reference call site (file:line, relative to the
 * reference root) whose native work it replaces, and the operator signature it mirrors.
 * INTEGRATION.md shows the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions (all entry points):
 *   - plain pointers and sizes only; no torch / C++ types; `int` status return
 *     (0 = SFOD_OK, otherwise an sfod_status value; >= 1000 encodes 1000 + cudaError_t);
 *   - no exceptions, no logging, re-entrant; the only process-wide state is (i) a monotonically increasing diagnostic
 *     launch counter (sfod_debug_launch_count) and (ii) two write-once capability caches (the largest thread-block cluster
 *     the device accepts for the NMS kernels, csrc/nms.cuh) whose initialisation is idempotent -- nothing a kernel result
 *     depends on is kept between calls;
 *   - every buffer is owned by the caller (inputs, outputs, workspace); workspace sizes
 *     come from the matching *_workspace_bytes() query; all device pointers must be
 *     valid on the current CUDA device; fp32 buffers must be 16-byte aligned unless noted;
 *   - kernels are enqueued on `stream` and the call returns without synchronising;
 *     variable-length results are returned as a device-side count plus a max-sized buffer;
 *   - indices are int64 on the API (torch convention) unless noted.
 */
#ifndef SFOD_B200_H
#define SFOD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st *sfod_stream_t; /* identical to cudaStream_t */

enum sfod_status {
  SFOD_OK = 0,
  SFOD_ERR_INVALID_ARG = 1,
  SFOD_ERR_WORKSPACE_TOO_SMALL = 2,
  SFOD_ERR_UNSUPPORTED = 3,
  SFOD_ERR_ALIGNMENT = 4,
  SFOD_ERR_CUDA_BASE = 1000
};

enum sfod_layout { SFOD_NCHW = 0, SFOD_NHWC = 1 };
enum sfod_dtype { SFOD_F32 = 0, SFOD_I64 = 1, SFOD_U8 = 2 };

/* Changes whenever an entry point keeps its name but changes its arguments, or a parameter record field changes its meaning;
 * a binding refuses a library of another version. */
int sfod_abi_version(void);
/* sizeof() of the parameter structs as this library was compiled (which: 0 sfod_ema_tensor, 1 sfod_rpn_params,
 * 2 sfod_frcnn_params, 3 sfod_p2p_comm, 4 sfod_jitter_params, 5 sfod_erase_params, 6 sfod_resize_image, 7 sfod_coco_eval_params;
 * 0 for anything else) -- lets a foreign
 * binding (ctypes / cffi struct mirrors) check its layout against the C one before the first call. */
size_t sfod_abi_sizeof(int which);
const char *sfod_status_string(int status);
/* Number of kernel launches the library has issued in this process so far (diagnostic, monotonically
 * increasing; bench.py reports the difference across its timed region as "gpu_launches"). */
uint64_t sfod_debug_launch_count(void);

/* ------------------------------------------------------------------------------------
 * Mean-teacher EMA.  Replaces the per-tensor loop of
 *   daod/engine/trainers/source_free_adaptive_teacher.py:593-603 (_update_teacher_model)
 *   (same body: adaptive_teacher.py:339-358).
 * teacher[i] = fp32(student[i] * fp32(1-k)) + fp32(teacher[i] * fp32(k)), two separately
 * rounded products and one rounded sum (no FMA), written in place into the teacher tensor
 * (what load_state_dict's copy_ does).  int64 tensors (BatchNorm num_batches_tracked) are
 * promoted to fp32, blended, and truncated back, exactly like the reference.
 * One launch covers every tensor of the state dict through a chunk table ("plan").
 * The plan is built on the host from the tensor table and uploaded by the caller. */
typedef struct sfod_ema_tensor {
  const void *student; /* device pointer */
  void *teacher;       /* device pointer, updated in place */
  int64_t numel;
  int32_t dtype; /* enum sfod_dtype */
  int32_t reserved;
} sfod_ema_tensor;

int64_t sfod_ema_plan_chunks(const sfod_ema_tensor *tensors, int n_tensors);
size_t sfod_ema_plan_bytes(int64_t n_chunks);
int sfod_ema_plan_build(const sfod_ema_tensor *tensors, int n_tensors, void *host_plan, size_t host_plan_bytes);
int sfod_ema_multi_tensor(const void *device_plan, int64_t n_chunks, double keep_rate, sfod_stream_t stream);

/* ------------------------------------------------------------------------------------
 * ROIAlign / ROIPool, forward and backward.  Replace torchvision.ops.roi_align / roi_pool
 * as reached from d2 ROIPooler, built at
 *   daod/modeling/roi_heads/source_free_adaptive_teacher_roi_heads.py:42-47, called :117
 * (pooler_type "ROIAlignV2" -> aligned=1, "ROIAlign" -> aligned=0, "ROIPool" -> roi_pool).
 * input (N,C,H,W) fp32 in `layout`; rois (R,5) = [batch_index, x1, y1, x2, y2];
 * output (R,C,PH,PW) contiguous (torchvision layout).  `exact` != 0 selects the kernel that
 * reproduces torchvision's per-sample summation order bit for bit (NCHW gather); exact == 0
 * selects the separable channels-last kernel (<= 1e-5 relative, see DESIGN.md), whose
 * workspace also holds one table record per ROI (hence R in the query). */
size_t sfod_roi_align_fwd_workspace_bytes(int N, int C, int H, int W, int R, int layout, int exact);
int sfod_roi_align_fwd(const float *input, int layout, const float *rois, int N, int C, int H, int W, int R, int PH,
                       int PW, float spatial_scale, int sampling_ratio, int aligned, int exact, float *output,
                       void *workspace, size_t workspace_bytes, sfod_stream_t stream);
/* grad_in (N,C,H,W) in `layout` is fully overwritten (zero-filled then accumulated). */
size_t sfod_roi_align_bwd_workspace_bytes(int N, int C, int H, int W, int layout);
int sfod_roi_align_bwd(const float *grad_out, const float *rois, int N, int C, int H, int W, int R, int PH, int PW,
                       float spatial_scale, int sampling_ratio, int aligned, float *grad_in, int layout,
                       void *workspace, size_t workspace_bytes, sfod_stream_t stream);
int sfod_roi_pool_fwd(const float *input, const float *rois, int N, int C, int H, int W, int R, int PH, int PW,
                      float spatial_scale, float *output, int32_t *argmax, sfod_stream_t stream);
int sfod_roi_pool_bwd(const float *grad_out, const float *rois, const int32_t *argmax, int N, int C, int H, int W,
                      int R, int PH, int PW, float *grad_in, sfod_stream_t stream);

/* ------------------------------------------------------------------------------------
 * NMS with torchvision semantics.  Replaces torchvision.ops.nms / batched_nms as reached
 * from d2 find_top_rpn_proposals (called by daod/modeling/proposal_generator/rpn.py:54-56)
 * and from daod/modeling/roi_heads/fast_rcnn.py:133.
 * boxes (n,4) xyxy fp32, scores (n) fp32, idxs (n) int64 or NULL (plain nms).
 * keep_out (n) int64 receives the kept indices in score-descending order (ties: lower
 * index first = torchvision CPU's stable sort); *num_keep_dev (device int64) the count.
 * IoU arithmetic: inter / (area_i + area_j - inter) in separately rounded fp32, suppress
 * iff (double)iou > iou_threshold.  With idxs != NULL and n <= coord_trick_max_n the boxes
 * are first offset by idx * (max_coordinate + 1) in fp32, reproducing torchvision's
 * _batched_nms_coordinate_trick rounding (CPU switches strategy at numel > 4000, i.e.
 * coord_trick_max_n = 1000); above it suppression is per class on the raw boxes
 * (_batched_nms_vanilla). */
size_t sfod_nms_workspace_bytes(int64_t n);
int sfod_nms(const float *boxes, const float *scores, const int64_t *idxs, int64_t n, double iou_threshold,
             int64_t coord_trick_max_n, int64_t *keep_out, int64_t *num_keep_dev, void *workspace,
             size_t workspace_bytes, sfod_stream_t stream);

/* ------------------------------------------------------------------------------------
 * RPN proposal selection for one feature level (every shipped config is single-level).
 * Replaces d2 RPN.predict_proposals = _decode_proposals + find_top_rpn_proposals as called
 * at daod/modeling/proposal_generator/rpn.py:54-56, for all N images in one call:
 *   per image: stable descending sort of the HWA logits, keep top pre_nms_topk;
 *   decode anchor (+) delta (Box2BoxTransform weights, dw/dh clamp), fp32 ops in d2's order;
 *   drop non-finite (counted in invalid_count_dev; d2 raises in training), clip to (h,w),
 *   drop boxes with w <= min_box_size or h <= min_box_size; greedy NMS (iou_threshold);
 *   first post_nms_topk survivors.
 * head_layout 0: logits (N,HWA) and deltas (N,HWA,4) are the flattened head outputs of rpn.py:28-41.
 * head_layout 1: logits (N,A,Hf,Wf) and deltas (N,4A,Hf,Wf) are the RPN head's convolution outputs AS THEY LIE (what
 *   rpn.py:28-41 permutes and copies): the flatten is folded into the key build and the top-k gather, indices
 *   (out_src_index, anchors) keep the flattened (Hf,Wf,A) numbering.  Needs A, Hf, Wf (also with an anchor tensor).
 * anchors: (HWA,4) device tensor, or NULL to recompute d2's DefaultAnchorGenerator grid in
 * closed form from cell_anchors (A,4) host floats, feature size (Hf,Wf), stride and offset.
 * image_hw_dev: (N,2) int32 device [h, w].
 * Outputs: out_boxes (N,post_nms_topk,4), out_logits (N,post_nms_topk), out_src_index
 * (N,post_nms_topk) int64 flat anchor index of each proposal, out_count_dev (N) int32. */
typedef struct sfod_rpn_params {
  int N, HWA, A, Hf, Wf, stride;
  float anchor_offset;
  float weights[4];
  float scale_clamp;
  int pre_nms_topk, post_nms_topk;
  float min_box_size;
  double nms_thresh;
  float cell_anchors[64 * 4]; /* up to 64 cell anchors, used when anchors == NULL */
  int head_layout;            /* 0: flattened (N,HWA) / (N,HWA,4); 1: head outputs (N,A,Hf,Wf) / (N,4A,Hf,Wf) */
} sfod_rpn_params;

size_t sfod_rpn_select_workspace_bytes(const sfod_rpn_params *p);
int sfod_rpn_select(const sfod_rpn_params *p, const float *logits, const float *deltas, const float *anchors,
                    const int32_t *image_hw_dev, float *out_boxes, float *out_logits, int64_t *out_src_index,
                    int32_t *out_count_dev, int32_t *invalid_count_dev, void *workspace, size_t workspace_bytes,
                    sfod_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Fast R-CNN post-processing + pseudo-label filter for all N images in one call.
 * Replaces FastRCNNOutputLayers.inference (called at
 * daod/modeling/roi_heads/source_free_adaptive_teacher_roi_heads.py:161) =
 * predict_boxes + predict_probs + fast_rcnn_inference_single_image
 * (on-disk statement: daod/modeling/roi_heads/fast_rcnn.py:108-142), followed by
 * threshold_bbox(proposal_type="roih") of
 * daod/engine/trainers/source_free_adaptive_teacher.py:167-181.
 * cls_logits (R,K+1), deltas (R,4K) (or (R,4) when class_agnostic), proposals (R,4);
 * rows of image i are [row_offsets_dev[i], row_offsets_dev[i+1]) (int32, N+1 entries); or, with rows_stride > 0 (packed
 * layout, R == N * rows_stride), rows [i * rows_stride, i * rows_stride + row_offsets_dev[i]) where row_offsets_dev holds
 * the N DEVICE-side row counts (e.g. out_count_dev of sfod_rpn_select) -- no host knowledge of the counts is needed.
 * mode 0: inference (score > score_thresh, per-class NMS, top-k);
 * Outputs per image, padded to topk: det_boxes (N,topk,4), det_scores (N,topk),
 * det_classes (N,topk) int64, det_rows (N,topk) int64 (row within the image),
 * det_count_dev (N) int32, pseudo_count_dev (N) int32 = #detections with score >
 * pseudo_thresh (detections are score-descending, so the pseudo-label set is that prefix).
 * probs_out (R,K+1) optional (may be NULL) receives the softmax probabilities;
 * boxes_out (R,4K) optional receives the decoded (unclipped) boxes (predict_boxes). */
typedef struct sfod_frcnn_params {
  int N, R, K;
  int class_agnostic;
  int max_rows_per_image;
  float weights[4];
  float scale_clamp;
  float score_thresh;
  double nms_thresh;
  int topk;
  float pseudo_thresh;
  int64_t coord_trick_max_n; /* 1000 reproduces torchvision-CPU's strategy switch */
  int rows_stride;           /* 0: row_offsets_dev are prefix offsets; > 0: packed layout with device row counts */
} sfod_frcnn_params;

size_t sfod_frcnn_postprocess_workspace_bytes(const sfod_frcnn_params *p);
int sfod_frcnn_postprocess(const sfod_frcnn_params *p, const float *cls_logits, const float *deltas,
                           const float *proposals, const int32_t *row_offsets_dev, const int32_t *image_hw_dev,
                           float *det_boxes, float *det_scores, int64_t *det_classes, int64_t *det_rows,
                           int32_t *det_count_dev, int32_t *pseudo_count_dev, float *probs_out, float *boxes_out,
                           void *workspace, size_t workspace_bytes, sfod_stream_t stream);

/* Box2BoxTransform.apply_deltas (d2 box_regression; SURVEY.md A-2) and softmax as separate
 * operators: deltas (R,4k), boxes (R,4) -> out (R,4k).  Used by predict_boxes /
 * convert_bbox_scores (daod/modeling/roi_heads/source_free_fast_rcnn.py:15-17). */
int sfod_apply_deltas(const float *deltas, const float *boxes, int64_t R, int k, const float *weights4_host,
                      float scale_clamp, float *out, sfod_stream_t stream);
int sfod_softmax_lastdim(const float *x, int64_t R, int K1, float *out, sfod_stream_t stream);

/* Generic confidence filter: threshold_bbox (source_free_adaptive_teacher.py:150-183).
 * For S segments laid out with fixed stride: values (S,stride), counts_dev (S) int32 valid
 * entries; writes the indices (ascending) of entries with value > thres to out_index
 * (S,stride) int64 and their number to out_count_dev (S) int32. */
int sfod_threshold_select(const float *values, const int32_t *counts_dev, int S, int stride, float thres,
                          int64_t *out_index, int32_t *out_count_dev, sfod_stream_t stream);

/* Adaptive per-class threshold variant of the pseudo-label filter (SURVEY.md 8f rank 2; reference
 * daod/modeling/adaptive_thresh/adaptive_confidence.py:21-33 as used by adaptive_threshold_bbox / prediction_threshold_bbox,
 * daod/engine/trainers/source_free_adaptive_teacher.py:185-254): same segment layout as sfod_threshold_select, entry j of
 * segment s is kept iff values[s][j] >= class_thresh_dev[classes[s][j]] (K device floats; note >=).  classes outside
 * [0, K) are dropped. */
int sfod_class_threshold_select(const float *values, const int64_t *classes, const int32_t *counts_dev, int S, int stride,
                                int K, const float *class_thresh_dev, int64_t *out_index, int32_t *out_count_dev,
                                sfod_stream_t stream);
/* count_label_prediction (source_free_adaptive_teacher.py:282-296) for the whole batch in one launch: hist_dev (K) int64
 * receives, per class, the number of entries with value > thres over all S segments (zeroed by the call). */
int sfod_class_histogram(const float *values, const int64_t *classes, const int32_t *counts_dev, int S, int stride, int K,
                         float thres, int64_t *hist_dev, sfod_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Image preprocessing (SURVEY.md 8f rank 3, normalise / pad / batch part).  Replaces
 * GeneralizedRCNN.preprocess_image = `(x - pixel_mean) / pixel_std` + ImageList.from_tensors
 * (daod/modeling/meta_arch/rcnn.py:92-104) for N equally sized CHW images that are
 * `image_stride` elements apart (N = 1 for a list of differently sized images: one call per
 * image into its slot of the padded batch).  images: uint8 (SFOD_U8) or float32 (SFOD_F32) on
 * the device; mean/std: C floats on the HOST (C <= 8); out: (N,C,Hp,Wp) fp32 in `layout`,
 * fl(fl(x - mean[c]) / std[c]) inside (H,W) and 0.0 in the padding. */
int sfod_normalize_pad(const void *images, int dtype, int64_t image_stride, int N, int C, int H, int W, const float *mean,
                       const float *stdv, int Hp, int Wp, int layout, float *out, sfod_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Fused pairwise_iou + Matcher (SURVEY.md 8f rank 1).  Replaces, per image,
 * detectron2.structures.pairwise_iou followed by detectron2.modeling.matcher.Matcher.__call__ as
 * reached from RPN.label_and_sample_anchors (called by daod/modeling/proposal_generator/rpn.py:45)
 * and label_and_sample_proposals
 * (daod/modeling/roi_heads/source_free_adaptive_teacher_roi_heads.py:165-215).
 * gt_boxes (M,4), boxes (N,4) xyxy fp32 on the device; thresholds (num_thresholds ascending
 * floats) and labels (num_thresholds + 1 ints in {-1,0,1}) on the HOST: label[k] is given to
 * predictions whose best IoU v satisfies thresholds[k-1] <= v < thresholds[k].
 * matches (N) int64 = index of the first gt with the maximal IoU (0 when M == 0); match_labels
 * (N) int8; matched_vals (N) float or NULL.  allow_low_quality != 0 applies
 * Matcher.set_low_quality_matches_ literally: every prediction whose IoU with some gt equals
 * that gt's maximum over all predictions gets label 1.  The M x N matrix is never stored. */
size_t sfod_iou_match_workspace_bytes(int M);
int sfod_iou_match(const float *gt_boxes, const float *boxes, int M, int N, const float *thresholds, const int *labels,
                   int num_thresholds, int allow_low_quality, int64_t *matches, int8_t *match_labels, float *matched_vals,
                   void *workspace, size_t workspace_bytes, sfod_stream_t stream);

/* Batched detectron2 `subsample_labels` (SURVEY.md 8f rank 1): for each of `num_segments` label segments
 * labels[offsets[s] .. offsets[s+1]) (labels: int64 on the device; offsets: num_segments + 1 ints in HOST memory, passed to the
 * kernel by value; -1 = ignore, bg_label = negative, anything else positive) select
 * num_pos = min(#positive, max_positive) positives and num_neg = min(#negative, num_samples - num_pos) negatives uniformly at
 * random, as the per-image calls of ROIHeads._sample_proposals (reference
 * daod/modeling/roi_heads/source_free_adaptive_teacher_roi_heads.py:177-186) and RPN.label_and_sample_anchors (called at
 * daod/modeling/proposal_generator/rpn.py:45) do with two torch.randperm + two nonzero host syncs per image.
 * sampled: (num_segments, num_samples) int64 segment-local indices, positives first, each group in ascending order of the
 * counter-based key hash(seed, segment, index) (the k smallest keys = a uniform k-subset in random order), padded with -1;
 * counts: (num_segments, 2) int32 (num_pos, num_neg), on the device.  max_positive = int(num_samples * positive_fraction)
 * (computed by the caller with Python's float arithmetic, like the reference).  2 * num_samples <= 1024. */
int sfod_subsample_labels(const int64_t *labels, const int32_t *offsets, int num_segments, int num_samples, int max_positive,
                          int64_t bg_label, uint64_t seed, int64_t *sampled, int32_t *counts, sfod_stream_t stream);

/* ------------------------------------------------------------------------------------
 * BatchNorm train-mode forward / AdaBN statistic recomputation.  Replaces the
 * nn.BatchNorm2d train-mode forwards driven by test_refinement
 * (daod/engine/trainers/base.py:274-299, after reset_bn_stats :318-323) and by the teacher
 * forward under no_grad (source_free_adaptive_teacher.py:385-390).
 * Phase 1 (sfod_bn_partial_stats): per-channel (sum x, sum x^2) over (N,H,W) accumulated
 *   in fp64 into stats_dev (C,2) doubles, and the element count N*H*W into stats_dev[2C]
 *   (zeroed and written by the call).  These 2C+1 doubles are the payload a multi-GPU caller
 *   sums over the ranks before phase 2: with an all-reduce of its own (NCCL), or with the
 *   peer-memory exchange below.
 * Phase 2 (sfod_bn_finalize_apply): mean, biased var (fp64) from the totals and the count,
 *   both read on the device (a multi-GPU AdaBN forward needs no host read between its two
 *   phases: reference daod/engine/trainers/base.py:270-337 on several ranks; SURVEY.md 8e
 *   collective 2), running stats r = (1-m) r + m stat with the unbiased variance n/(n-1),
 *   num_batches_tracked += 1, y = (x-mean)*invstd*weight+bias (optionally fused ReLU); y may
 *   alias x.  x or y NULL: statistics and running statistics only.
 * comm (both phases; NULL = the statistics in stats_dev are used as they are): the peer-memory exchange below.
 * stats_dev must hold sfod_bn_stats_bytes(C) bytes: the 2C+1 payload, then scratch of the
 * library (scale/shift of phase 2, replicated partial totals of the channels-last pass). */
size_t sfod_bn_stats_bytes(int C);
typedef struct sfod_p2p_comm sfod_p2p_comm_t; /* defined with the peer-memory exchange below */
/* pre_bias (C floats, may be NULL): a per-channel bias added to x before everything else -- the bias of the
 * convolution that feeds the BatchNorm (reference daod/modeling/meta_arch/vgg.py:17-19: Conv2d(bias=True) -> BatchNorm2d),
 * so that the convolution can run bias-free and its separate elementwise pass over the activation disappears.
 * Statistics, running statistics and output are those of fl(x + pre_bias[c]), bit-identical to adding the bias first. */
int sfod_bn_partial_stats(const float *x, const float *pre_bias, int layout, int N, int C, int64_t HW, double *stats_dev,
                          const sfod_p2p_comm_t *comm, sfod_stream_t stream);
/* residual (same shape and layout as x, may be NULL; SFOD_ERR_ALIGNMENT unless it has x's 16-byte phase):
 * y = [relu](fl(bn(x)) + residual) -- the tail of a detectron2 BottleneckBlock (conv3+norm, `out += shortcut`, `relu_`),
 * which the R101-C4 configs of the reference (configs/r101_c4_cs_foggy_adaptive_teacher_source_free.yaml:5-7,
 * RESNETS.NORM "BN") execute as three elementwise passes.
 * fuse_maxpool2 != 0: y is the (N,C,H/2,W/2) result of MaxPool2d(kernel_size=2, stride=2) applied to the normalised
 * (+ReLU) activation (vgg.py:15), written directly (x is read once, the full-resolution activation is never stored);
 * y must not alias x and residual must be NULL in that mode. */
int sfod_bn_finalize_apply(const float *x, const float *pre_bias, const float *residual, float *y, int layout, int N, int C,
                           int H, int W, double *stats_dev, const sfod_p2p_comm_t *comm, const float *weight, const float *bias,
                           float *running_mean, float *running_var, int64_t *num_batches_tracked, double momentum, double eps,
                           int fuse_relu, int fuse_maxpool2, sfod_stream_t stream);
/* Single-launch variant of phase 1 + phase 2 for NCHW activations that (mostly) fit the 126 MB L2 (late VGG layers, res3 / res4
 * of R101-C4): a cooperative persistent kernel computes the statistics, crosses one grid barrier and normalises the chunks it has
 * just read in reverse order, so the second read of x comes from L2 (~8 instead of 12 B/element of HBM traffic, 1 launch instead
 * of 4).  Same arithmetic as the two-phase path (fp64 totals, ATen's running-stat update).  y may alias x.
 * SFOD_ERR_UNSUPPORTED: no cooperative launch possible -- use the two-phase entry points. */
int sfod_bn_train_fused(const float *x, const float *pre_bias, const float *residual, float *y, int N, int C, int H, int W,
                        double *stats_dev, const float *weight, const float *bias, float *running_mean, float *running_var,
                        int64_t *num_batches_tracked, double momentum, double eps, int fuse_relu, sfod_stream_t stream);
/* FrozenBatchNorm2d / eval-mode BatchNorm with the same fusions: y = [relu](x * scale + shift [+ residual]),
 * scale = weight / sqrt(running_var + eps), shift = bias - running_mean * scale.  detectron2 freezes the stem and res2 of
 * the R101-C4 backbone (MODEL.BACKBONE.FREEZE_AT = 2 is not overridden by configs/r101_c4_cs_foggy_adaptive_teacher_source_free.yaml),
 * so 11 of its 94 norm layers run in this mode even while the teacher is in train().  `scratch` holds
 * sfod_bn_frozen_scratch_bytes(C) bytes. */
size_t sfod_bn_frozen_scratch_bytes(int C);
int sfod_bn_frozen_apply(const float *x, const float *residual, float *y, int layout, int N, int C, int H, int W,
                         const float *weight, const float *bias, const float *running_mean, const float *running_var,
                         double eps, int fuse_relu, void *scratch, sfod_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------------
 * Multi-GPU AdaBN statistics over NVLink peer memory (SURVEY.md 8e, collective (2)): the all-reduce of the per-layer
 * (sum x, sum x^2, count) payload that makes every rank normalise with the statistics of the concatenated batch when
 * test_refinement (reference daod/engine/trainers/base.py:270-337) or the teacher forward
 * (source_free_adaptive_teacher.py:385-390) runs data-parallel.  Instead of a collective launch per layer (NCCL
 * all-reduce of 2C+1 doubles: the baseline, see simple-sfod_b200/engine/adabn_dist.py) the exchange is fused into phase 2:
 * sfod_bn_finalize_apply with comm != NULL runs one kernel that stores the local payload into every peer's inbox with P2P
 * stores (every element tagged with the exchange's epoch), polls for the peers' elements, adds the payloads in rank order
 * (bit-identical totals on every rank), leaves these totals of the concatenated batch in stats_dev and computes the
 * coefficients.  sfod_bn_partial_stats with comm != NULL computes the same statistics; in addition the CTA of the statistics
 * kernel that finishes last delivers the payload to the peers' inboxes (NCHW layers covered by one launch; otherwise phase 2
 * delivers it), so the NVLink transfer overlaps the launch gap between the two phases.  It must then be followed by
 * sfod_bn_finalize_apply on the same stream, comm and stats_dev.  With comm != NULL both calls return SFOD_ERR_INVALID_ARG
 * unless 1 <= world <= SFOD_P2P_MAX_RANKS, 0 <= rank < world and every inbox[r] is set, and SFOD_ERR_UNSUPPORTED for
 * C > sfod_p2p_max_channels().
 *
 * An inbox is sfod_p2p_inbox_bytes() of device memory allocated by sfod_p2p_alloc (cudaMalloc + zero fill), which also
 * returns its 64-byte CUDA IPC handle; the caller ships the handle to the other processes of the node (any host channel:
 * torch.distributed.all_gather_object in simple-sfod_b200/engine/p2p.py) and maps theirs with sfod_p2p_open.  Ranks sharing
 * one process (tests) put each other's inbox pointers into the comm directly.  All ranks must issue the same sequence of
 * exchanges.  A peer that never arrives is abandoned after ~3 s (sfod_p2p_status reports the number of such timeouts; the
 * results of a timed-out exchange are invalid) -- the GPU is never left spinning. */
#define SFOD_P2P_MAX_RANKS 8
#define SFOD_P2P_HANDLE_BYTES 64
struct sfod_p2p_comm {
  int32_t rank, world;                 /* world <= SFOD_P2P_MAX_RANKS */
  void *inbox[SFOD_P2P_MAX_RANKS];     /* inbox[r]: rank r's inbox as mapped into THIS process (inbox[rank] = own allocation) */
};
size_t sfod_p2p_inbox_bytes(void);
int sfod_p2p_max_channels(void);       /* largest C one exchange carries (2051: covers the 2048-channel res5 of the reference backbones) */
int sfod_p2p_alloc(void **inbox, unsigned char *handle /* SFOD_P2P_HANDLE_BYTES, may be NULL */);
int sfod_p2p_open(const unsigned char *handle, void **peer_inbox);
int sfod_p2p_close(void *peer_inbox);
int sfod_p2p_free(void *inbox);
/* Synchronous read of the own inbox header: exchanges completed, exchanges abandoned on a timeout. */
int sfod_p2p_status(const sfod_p2p_comm_t *comm, uint64_t *exchanges, uint32_t *timeouts);

/* ---------------------------------------------------------------------------------------------------------------------
 * Strong augmentation of the student's input on the device (SURVEY.md 8f rank 3).  Replaces the PIL / torchvision CPU
 * pipeline of reference daod/data/detection_utils.py:7-37, applied per image at
 * daod/data/mappers/two_crop_augmentation_mapper.py:141-157: RandomApply(ColorJitter(0.4, 0.4, 0.4, 0.1), 0.8),
 * RandomGrayscale(0.2), RandomApply(GaussianBlur((0.1, 2.0)), 0.5), 3 x RandomErasing(value="random").
 * Images are (N, 3, H, W) uint8, RGB planes.  The random decisions are drawn by the caller (as torchvision draws them) and
 * passed as per-image parameter records in DEVICE memory.  The pixel arithmetic is Pillow's, bit for bit: the reference's mapper
 * hands PIL images to the transforms, so torchvision's PIL path is what it executes. */
typedef struct sfod_jitter_params {
  int32_t n_ops;          /* 0 = ColorJitter not applied; else 4 */
  int32_t op[4];          /* order of application: 0 brightness, 1 contrast, 2 saturation, 3 hue */
  float factor[4];        /* blend alpha of op[k] (brightness / contrast / saturation) */
  int32_t hue_shift[4];   /* hue op: the shift byte uint8(int32(255 * hue)); ignored for the other ops */
  int32_t grayscale;      /* != 0: RandomGrayscale hit (3-channel gray after the jitter) */
} sfod_jitter_params;
/* ColorJitter + RandomGrayscale: Image.blend against a black / mean-gray / gray degenerate image (ImageEnhance.Brightness /
 * Contrast / Color), convert("L") = (19595 R + 38470 G + 7471 B + 0x8000) >> 16, adjust_hue through convert("HSV").
 * Bit-exact against torchvision's PIL path (tests).  workspace: N * 8 bytes.  out may alias images. */
int sfod_color_jitter_pil(const uint8_t *images, int N, int H, int W, const sfod_jitter_params *params_dev, void *workspace,
                          size_t workspace_bytes, uint8_t *out, sfod_stream_t stream);
/* Pillow's ImageFilter.GaussianBlur bit for bit -- the filter the reference actually applies (reference
 * daod/data/transforms/augmentations.py:18-21): three extended-box-blur passes per axis in 8.24 fixed point, each rounded to
 * uint8, edges replicated (Pillow src/libImaging/BoxBlur.c).  Per image: radius_dev[n] = integer box radius (-1: copy the image,
 * i.e. a RandomApply miss), ww_dev[n] / fw_dev[n] = the fixed-point weights of the inner / outermost taps; the host derives all
 * three from sigma exactly as Pillow does (simple-sfod_b200/ops.py::pil_blur_params).  max_radius = max over n (<= 9). */
int sfod_gaussian_blur_pil(const uint8_t *images, int N, int H, int W, const int32_t *radius_dev, const uint32_t *ww_dev,
                           const uint32_t *fw_dev, int max_radius, uint8_t *out, sfod_stream_t stream);
typedef struct sfod_erase_params {
  int32_t n_rects;        /* 0..4 rectangles, applied in order (a later one overwrites an earlier one) */
  int32_t rect[4][4];     /* (top, left, height, width) */
} sfod_erase_params;
/* In place: every rectangle is filled with byte(255 * v), v ~ N(0, 1) from a counter-based generator keyed by `seed`, or
 * v = noise[n][k][c][y][x] when `noise` ((N, 4, 3, H, W) floats) is given -- what ToTensor -> RandomErasing(value="random") ->
 * ToPILImage leave in the rectangle. */
int sfod_random_erase(uint8_t *images, int N, int H, int W, const sfod_erase_params *params_dev, const float *noise,
                      uint64_t seed, sfod_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------------
 * Weak augmentation of the input on the device (SURVEY.md 8f rank 3): detectron2's ResizeShortestEdge + RandomFlip, the
 * augmentations the reference's data mapper applies before the strong chain (reference
 * daod/data/mappers/two_crop_augmentation_mapper.py, `T.apply_augmentations(self.augmentation, aug_input)` with the list of
 * detectron2 build_augmentation).  For uint8 images detectron2's ResizeTransform.apply_image is
 * `Image.fromarray(img).resize((new_w, new_h), Image.BILINEAR)`; HFlipTransform is `np.flip(img, axis=1)` after it.
 * This call reproduces Pillow's 8-bit resampler (src/libImaging/Resample.c) bit for bit: horizontal pass over the input rows the
 * vertical taps use, rounded to a uint8 intermediate, then the vertical pass; every output is
 * clip8(2^21 + sum in[xmin + k] * tap[k]) in int32 with 22 fraction bits.  The taps come from the caller (the host computes them
 * in double exactly as Pillow does: simple-sfod_b200/ops.py::pil_resize_coeffs).
 * Per image one record; the source is read through three byte strides, so HWC (stride_px = 3, stride_ch = 1) and CHW planes
 * (stride_px = 1, stride_ch = H * W, i.e. a permuted view) take the same path.  The result is written as CHW planes
 * (3, out_h, out_w) at out + out_offset (the mapper's HWC -> CHW transpose is fused), mirrored horizontally when hflip != 0.
 * A coefficient table (int32, at coeffs + k*_offset) holds out (xmin, xmax) pairs followed by out x k*_size taps, zero-padded
 * to k*_size = 2 * ceil(max(in / out, 1)) + 1.  Down-scales up to 4 per axis (k*_size <= 9) and any up-scale are supported. */
typedef struct sfod_resize_image {
  const uint8_t *src;                         /* device pointer: pixel (0, 0), channel 0 */
  int64_t stride_row, stride_px, stride_ch;   /* bytes */
  int32_t in_h, in_w, out_h, out_w;
  int64_t out_offset;                         /* bytes from `out` to this image's (3, out_h, out_w) planes */
  int32_t hflip;                              /* != 0: write column x to out_w - 1 - x */
  int32_t kx_offset, kx_size;                 /* horizontal table: int32 offset into coeffs, taps per output column */
  int32_t ky_offset, ky_size;                 /* vertical table */
  int32_t reserved;
} sfod_resize_image;
/* One launch for the whole batch.  records_dev: N records in DEVICE memory; max_out_h / max_out_w / max_ksize: maxima over the
 * records (they size the grid and the shared-memory tiles; a record beyond them is skipped, its output left unwritten).
 * SFOD_ERR_INVALID_ARG for null pointers, N < 0, non-positive maxima, or max_out_h * max_out_w beyond an int32 plane index;
 * SFOD_ERR_UNSUPPORTED for max_ksize > 9 (a down-scale beyond 4). */
int sfod_resize_pil(const sfod_resize_image *records_dev, int N, const int32_t *coeffs_dev, uint8_t *out, int max_out_h,
                    int max_out_w, int max_ksize, sfod_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------------
 * Fully connected layer of the box head in fp32 on the tensor cores: y = act(x W^T + b) with x (M, K), W (N, K) and y (M, N)
 * row-major fp32 (nn.Linear's layout), b (N) or NULL, act 0 = none, 1 = ReLU (NaN propagates as in torch.relu).
 * 3xTF32 arithmetic: every operand is split into hi = tf32(v) and lo = tf32(v - hi), and x W^T is accumulated as
 * lo*hi + hi*lo + hi*hi in fp32, which keeps fp32-level accuracy (the dropped lo*lo term is <= 2^-22 relative per product).
 * The workspace holds the hi and lo planes of W and of x, rebuilt on every call (W may change in place between calls).
 * SFOD_ERR_INVALID_ARG for null x / w / y, M < 0, non-positive K or N, or another act; SFOD_ERR_UNSUPPORTED for K % 4 != 0,
 * N % 16 != 0 or M beyond 65535 * 128; SFOD_ERR_ALIGNMENT unless x, w, y and the workspace are 16-byte aligned.  All
 * checks happen before any launch.  M == 0 launches nothing. */
size_t sfod_linear_3xtf32_workspace_bytes(int64_t M, int N, int K);
int sfod_linear_3xtf32(const float *x, int64_t M, int K, const float *w, int N, const float *bias, int act, float *y,
                       void *workspace, size_t workspace_bytes, sfod_stream_t stream);

/* ---------------------------------------------------------------------------------------------------------------------
 * COCO box AP (SURVEY.md 8f row f-5): pycocotools' COCOeval(iouType="bbox").evaluate() + accumulate(), bit-equal, as the
 * reference reaches it through detectron2's COCOEvaluator (reference daod/evaluation/; test_refinement at
 * daod/engine/trainers/base.py:300, the --eval-only runs of train_net*.py, EvalHook).  summarize() stays with the caller.
 * Images are the I ground-truth images in ascending image-id order; categories the K ground-truth categories in ascending id
 * order (an index outside [0, K) is never evaluated, as a result of another category id).
 * Ground truth (n_gt = gt_offsets[I] entries, device arrays, sorted by image): the gt of image i are rows
 *   [gt_offsets[i], gt_offsets[i+1]) in annotation order; gt_offsets is HOST memory (I + 1 entries, gt_offsets[0] = 0).
 *   gt_boxes (n_gt, 4) fp64 XYWH, gt_area fp64 (the annotation's "area", not w * h), gt_iscrowd uint8 (!= 0: crowd),
 *   gt_ids int64 (the annotation id: a match to id 0 counts as a false positive, as in COCOeval), gt_categories int64.
 * Detections (device arrays, one padded row of P = dt_stride slots per image, in the order of the caller's result list):
 *   dt_boxes (I, P, 4) fp32 XYWH (16-byte aligned), dt_scores (I, P) fp32, dt_classes (I, P) int64, dt_counts (I) int32 valid
 *   slots per row -- device-side, so a detector's padded output is evaluated without reading its counts on the host.
 * Outputs (device fp64, COCOeval's layouts and -1 conventions): precision and scores (T, R, K, A, M), recall (T, K, A, M).
 * Thresholds and ranges are taken as given (the caller computes iouThrs / recThrs with numpy's linspace, as Params does).
 * SFOD_ERR_INVALID_ARG for a null pointer, non-positive sizes, a maxDets entry < 1, gt_offsets[0] != 0 or decreasing gt
 * offsets (gt not sorted by image); SFOD_ERR_UNSUPPORTED for K > SFOD_COCO_MAX_CATEGORIES, P > 1024, more than 1024 gt in one
 * image, a maxDets entry > 128, more thresholds / ranges than the arrays below hold, or I * P >= 2^24; SFOD_ERR_ALIGNMENT
 * for dt_boxes.  All checks happen before any launch. */
#define SFOD_COCO_MAX_CATEGORIES 254
#define SFOD_COCO_MAX_IOU_THRS 16
#define SFOD_COCO_MAX_REC_THRS 128
#define SFOD_COCO_MAX_AREA_RNGS 4
#define SFOD_COCO_MAX_MAX_DETS 4
typedef struct sfod_coco_eval_params {
  int32_t n_images;                               /* I */
  int32_t n_categories;                           /* K */
  int32_t dt_stride;                              /* P: detection slots per image row */
  int32_t n_iou_thrs, n_rec_thrs, n_area_rngs, n_max_dets;   /* T, R, A, M */
  int32_t max_dets[SFOD_COCO_MAX_MAX_DETS];       /* maxDets; the last one truncates every (image, category) */
  int32_t reserved;
  double iou_thrs[SFOD_COCO_MAX_IOU_THRS];
  double rec_thrs[SFOD_COCO_MAX_REC_THRS];
  double area_rng[SFOD_COCO_MAX_AREA_RNGS][2];    /* inclusive [lo, hi] on the area */
} sfod_coco_eval_params;
size_t sfod_coco_eval_workspace_bytes(const sfod_coco_eval_params *p);
int sfod_coco_eval(const sfod_coco_eval_params *p, const int64_t *gt_offsets, const double *gt_boxes, const double *gt_area,
                   const uint8_t *gt_iscrowd, const int64_t *gt_ids, const int64_t *gt_categories, const float *dt_boxes,
                   const float *dt_scores, const int64_t *dt_classes, const int32_t *dt_counts, double *precision, double *scores,
                   double *recall, void *workspace, size_t workspace_bytes, sfod_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SFOD_B200_H */
