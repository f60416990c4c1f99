/*
 * dgod_b200.h — C ABI of the DGOD detection-head hot path on NVIDIA B200 (sm_100a).
 *
 * This is the drop-in boundary (SURVEY.md §8b): one entry point per kernel family, plain
 * pointers and sizes, no torch types.  Every pointer marked "device" must be CUDA device
 * memory valid on `stream`; arrays marked "host" are read on the calling thread before the
 * call returns.  The library never allocates, frees or synchronises: outputs and scratch
 * ("workspace") are caller-owned, kernels are enqueued on the stream passed in, and the only
 * state is a thread-local error string.  Return value: DGOD_OK (0) or a negative DGOD_ERR_*;
 * on error dgod_last_error() describes it.
 *
 * Reference interfaces replaced (TV = torchvision 0.26.0, the reference's un-pinned
 * dependency, /root/reference/requirements.txt:17; call sites in /root/reference/*.py):
 *   dgod_box_iou            TV ops/boxes.py:344-370            (fasterrcnn.py:187 via TV rpn.py:208)
 *   dgod_matcher            TV models/detection/_utils.py:357-416
 *   dgod_iou_match          TV rpn.py:193-229 and TV roi_heads.py:580-613 (fasterrcnn.py:187,272)
 *   dgod_fcos_assign        fcos.py:510-548 and fcos.py:136-158
 *   dgod_fcos_loss_fwd/_bwd fcos.py:149-202 (focal + GIoU + centre-ness losses of FCOSHead.compute_loss)
 *   dgod_fcos_candidates    fcos.py:576-597 (FCOS.postprocess_detections up to the NMS: score, threshold, top-k, decode, clip)
 *   dgod_balanced_sample    TV models/detection/_utils.py:11-71 (BalancedPositiveNegativeSampler; fasterrcnn.py:119-123,272)
 *   dgod_sample_rois        TV roi_heads.py:615-678 after the sampler (sampled boxes, labels, regression targets)
 *   dgod_nms_batched        TV ops/boxes.py:20-120 -> torchvision::nms (TV rpn.py:289,
 *                           TV roi_heads.py:728, fcos.py:608)
 *   dgod_rpn_proposals      fasterrcnn.py:174-182 -> TV _utils.py:162-224, TV rpn.py:231-297,
 *                           TV anchor_utils.py:115-133
 *   dgod_rpn_filter         TV rpn.py:242-297 (fasterrcnn.py:182) on already-decoded proposals
 *   dgod_msroi_align_fwd    TV ops/poolers.py:147-227 -> torchvision::roi_align (fasterrcnn.py:278)
 *   dgod_msroi_align_bwd    torchvision::_roi_align_backward (autograd of the above)
 *   dgod_box_decode         TV _utils.py:162-224 (TV roi_heads.py:692, fasterrcnn.py:294)
 *   dgod_detect_candidates  TV roi_heads.py:692-724 (softmax, clip, score/size filters)
 *   dgod_grl_scale          DGcommon.py:33-45 (GRLayer.backward)
 *   dgod_image_batch        TV models/detection/transform.py:102-255 (GeneralizedRCNNTransform: normalize, resize, batch;
 *                           fasterrcnn.py:439-441, fcos.py:483)
 *   dgod_nchw_to_nhwc       layout helper (no reference counterpart: torch's .contiguous(channels_last))
 *   dgod_fpn_merge_fwd/_bwd TV ops/feature_pyramid_network.py FeaturePyramidNetwork.forward (lateral bias add, nearest
 *                           upsample, add) and its autograd (upsample_nearest2d_backward + accumulation)
 *   dgod_stem_pool_fwd      TV models/resnet.py ResNet._forward_impl: bn1 shift (folded), relu, maxpool of a frozen stem
 *   dgod_shift_relu_fwd     TV models/resnet.py Bottleneck.forward: bn1-3 and downsample shifts (folded), residual add, relu
 *   dgod_bias_add_fwd       the bias add of a cuDNN convolution: TV ops/feature_pyramid_network.py FPN layer blocks
 *   dgod_*_bf16             the four backbone entry points above on bf16 maps: the same modules under
 *                           torch.autocast("cuda", dtype=torch.bfloat16)
 *   dgod_map_match          torchmetrics MeanAveragePrecision (pycocotools backend): COCOeval.computeIoU / evaluateImg,
 *                           maskApi.c bbIou (DGcommon.py:127,154-172: the validation metric)
 *   dgod_map_accumulate     the same: COCOeval.accumulate
 *   dgod_linear_tc          TV models/detection/faster_rcnn.py TwoMLPHead (fasterrcnn.py:331-352): fc6 / fc7 Linear
 *                           forward (bias, ReLU) and their autograd products, fp32-accurate on the tensor cores
 *   dgod_rpn_head_fwd/_bwd  TV models/detection/rpn.py RPNHead.forward after its 3x3 conv (fasterrcnn.py:165): bias, relu,
 *                           the two 1x1 predictors, and their autograd (dgrads, threshold_backward, weight / bias grads)
 */
#ifndef DGOD_B200_H_
#define DGOD_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* dgod_stream_t; /* a cudaStream_t (0 = legacy default stream) */

#define DGOD_ABI_VERSION 9

enum {
  DGOD_OK = 0,
  DGOD_ERR_ARG = -1,       /* bad argument (null pointer, negative size, unsupported shape) */
  DGOD_ERR_WORKSPACE = -2, /* workspace_bytes smaller than dgod_*_workspace_bytes(...) */
  DGOD_ERR_CUDA = -3       /* a CUDA runtime call failed (launch, attribute, ...) */
};

enum { DGOD_F32 = 0, DGOD_BF16 = 1 };

#define DGOD_MAX_LEVELS 8
#define DGOD_MAX_CELL_ANCHORS 16

int dgod_abi_version(void);
/* Thread-local, never NULL; valid until the next failing call on this thread. */
const char* dgod_last_error(void);
/* Number of kernel launches enqueued by this library on the calling process so far. */
uint64_t dgod_launch_count(void);

/* ------------------------------------------------------------------ box_iou / Matcher */

/* iou[n1,n2] = IoU(boxes1[i], boxes2[j]) with torchvision's fp32 operation order
 * inter / ((area1 + area2) - inter), no FMA contraction (bit-exact with the CPU op). */
int dgod_box_iou(const float* boxes1 /*device [n1,4]*/, int n1,
                 const float* boxes2 /*device [n2,4]*/, int n2,
                 float* iou /*device [n1,n2]*/, dgod_stream_t stream);

size_t dgod_matcher_workspace_bytes(int m);
/* Matcher.__call__ on an explicit quality matrix (M ground truths x N predictions).
 * matches[n] = argmax_m (first index on ties), or -1 (below low) / -2 (between thresholds);
 * with allow_low_quality, predictions tying a ground truth's row maximum get their argmax back.
 * Thresholds are compared in fp32 like torch does with a Python scalar. m,n must be > 0. */
int dgod_matcher(const float* quality /*device [m,n]*/, int m, int n,
                 double high_threshold, double low_threshold, int allow_low_quality,
                 int64_t* matches /*device [n]*/,
                 void* workspace, size_t workspace_bytes, dgod_stream_t stream);

size_t dgod_iou_match_workspace_bytes(int n_img, int total_gt);
/* Fused box_iou + Matcher + label gather for a batch of images; the [M,N] matrix is never
 * materialised.  gt boxes of image i are gt_boxes[gt_offsets[i] .. gt_offsets[i+1]).
 * Candidate boxes, in one of three layouts:
 *   shared   (box_offsets == NULL, box_counts == NULL): all images share boxes[0..n_boxes) (RPN
 *            anchors); outputs are [n_img, n_boxes].
 *   ragged   (box_offsets): image i owns boxes[box_offsets[i]..box_offsets[i+1]); outputs are
 *            [n_boxes] (n_boxes = total).  max_boxes_per_img bounds the per-image count.
 *   padded   (box_counts, device [n_img]): boxes is [n_img, n_boxes, 4] and image i's candidate j
 *            is boxes[i, j] for j < box_counts[i], its ground truth j - box_counts[i] for
 *            j < box_counts[i] + n_gt_i (TV roi_heads.py:574-578 add_gt_proposals, without the
 *            copy), and an empty slot after that.  Outputs are [n_img, max_boxes_per_img]
 *            (max_boxes_per_img >= n_boxes + the largest n_gt_i); an empty slot gets
 *            matched_idx = -2, labels -1, clamped_idx 0, matched_boxes 0.  The counts stay on the
 *            device: no host synchronisation.
 * An image with zero ground truths gets matched_idx = -1 everywhere (TV rpn.py:202-206,
 * roi_heads.py:586-592 semantics follow from the derived outputs below).
 * Optional outputs (NULL to skip):
 *   labels_f32    1 / 0 / -1 as float (TV rpn.py:216-225)
 *   labels_i64    gt_labels[clamp(idx,0)], 0 below low, -1 between (TV roi_heads.py:599-609)
 *   clamped_idx   max(idx, 0)
 *   matched_boxes gt_boxes[clamp(idx,0)] (zeros when the image has no ground truth)        */
int dgod_iou_match(const float* gt_boxes /*device [total_gt,4]*/,
                   const int64_t* gt_labels /*device [total_gt] or NULL*/,
                   const int32_t* gt_offsets /*device [n_img+1]*/, int n_img, int total_gt,
                   const float* boxes /*device*/, const int32_t* box_offsets /*device or NULL*/,
                   const int32_t* box_counts /*device or NULL*/, int n_boxes, int max_boxes_per_img,
                   double high_threshold, double low_threshold, int allow_low_quality,
                   int64_t* matched_idx, float* labels_f32, int64_t* labels_i64,
                   int64_t* clamped_idx, float* matched_boxes,
                   void* workspace, size_t workspace_bytes, dgod_stream_t stream);

/* ------------------------------------------------------------------ FCOS assignment */

/* Location -> ground-truth assignment of fcos.py:510-548 including its area expression
 * (y1-x1)*(y2-y1) (fcos.py:543) and, for the optional target gather, the `len(labels) <= 1`
 * rule of fcos.py:139.  anchors are shared by all images ([n_anchors,4]); n_first / n_last are
 * num_anchors_per_level[0] / [-1].  Outputs are [n_img, n_anchors(, ...)]; optional ones may
 * be NULL: cls_targets (int64, -1 = background), box_targets (fp32 [..,4]),
 * onehot (fp32 [.., num_classes], fcos.py:157-158,201). */
int dgod_fcos_assign(const float* anchors /*device [n_anchors,4]*/, int n_anchors,
                     int n_first, int n_last, double center_sampling_radius,
                     const float* gt_boxes /*device [total_gt,4]*/,
                     const int64_t* gt_labels /*device [total_gt] or NULL*/,
                     const int32_t* gt_offsets /*device [n_img+1]*/, int n_img,
                     int64_t* matched_idx, int64_t* cls_targets, float* box_targets,
                     float* onehot, int num_classes, dgod_stream_t stream);

/* FCOS loss tail (SURVEY.md §8f rank 3): fcos.py:149-202 after the target gather — sigmoid focal loss
 * (alpha, gamma 2) over [n_img, n_anchors, num_classes] logits with one_hot(cls_targets), GIoU loss of
 * the decoded boxes (BoxLinearCoder, normalize_by_size) and BCE of the centre-ness logit against
 * sqrt(min(l,r)/max(l,r) * min(t,b)/max(t,b)) over the foreground (cls_targets >= 0), each divided by
 * max(1, #foreground).  losses: device fp32 [4] = classification, bbox_regression, bbox_ctrness,
 * #foreground (no host sync).  All tensors fp32 contiguous, box tensors 16-byte aligned; cls_targets /
 * box_targets are what dgod_fcos_assign writes.  The backward takes d(total)/d(losses[0..2]) as a
 * device fp32 [3] and writes dense gradients of the three head outputs (zeros on the background). */
size_t dgod_fcos_loss_workspace_bytes(long long n_locations);
int dgod_fcos_loss_fwd(const float* cls_logits, const float* bbox_regression, const float* bbox_ctrness,
                       const float* anchors /*device [n_anchors,4]*/, const int64_t* cls_targets,
                       const float* box_targets, int n_img, int n_anchors, int num_classes, float alpha,
                       float* losses /*device [4]*/, void* workspace, size_t workspace_bytes,
                       dgod_stream_t stream);
int dgod_fcos_loss_bwd(const float* cls_logits, const float* bbox_regression, const float* bbox_ctrness,
                       const float* anchors, const int64_t* cls_targets, const float* box_targets,
                       int n_img, int n_anchors, int num_classes, float alpha,
                       const float* losses /*device [4] from the forward*/,
                       const float* grad_losses /*device [3]*/, float* grad_cls_logits,
                       float* grad_bbox_regression, float* grad_bbox_ctrness, dgod_stream_t stream);

/* FCOS eval post-processing up to the NMS (SURVEY.md §8a row A12, fcos.py:576-597) for a batch in one launch: per
 * image and level score = sqrt(sigmoid(cls) * sigmoid(ctrness)) over [locations x classes], `> score_thresh`, the topk
 * (<= 1024) best in descending score (equal scores: ascending location * classes + class), BoxLinearCoder decode with
 * normalize_by_size (fcos.py:72-100) and clip to the image.  Head outputs are the concatenated [n_img, n_anchors, ...]
 * tensors (fp32, contiguous); level l owns anchors level_offsets[l] .. level_offsets[l+1] (device int32 [n_levels+1]).
 * Outputs have fixed capacity [n_img, n_levels * topk] (boxes [..,4], scores, labels int64, valid uint8; rows past
 * out_count[img * n_levels + l] are zero / invalid) so that dgod_nms_batched can run on them with its `valid` mask and
 * n_levels * topk boxes per segment — no host synchronisation. */
int dgod_fcos_candidates(const float* cls_logits, const float* bbox_regression, const float* bbox_ctrness,
                         const float* anchors /*device [n_anchors,4]*/, int n_anchors, int num_classes,
                         const int32_t* level_offsets /*device [n_levels+1]*/, int n_levels, int n_img,
                         const float* image_sizes /*device [n_img,2] = (h, w)*/, float score_thresh, int topk,
                         float* out_boxes, float* out_scores, int64_t* out_labels, uint8_t* out_valid,
                         int32_t* out_count /*device [n_img * n_levels]*/, dgod_stream_t stream);

/* ------------------------------------------------------------------ balanced sampler (SURVEY.md §8f rank 1) */

/* BalancedPositiveNegativeSampler for a batch in one launch, no host synchronisation.  labels [n_img, n] (fp32 as the RPN
 * produces them, or int64 as the RoI heads do): >= 1 positive, 0 negative, < 0 ignored.  keys [n_img, n] fp32: one
 * uniform random number per candidate; per image the min(#pos, num_pos) positives and the min(#neg, batch - #picked_pos)
 * negatives with the SMALLEST keys are selected (equal keys: ascending index) — a uniformly random subset like upstream's
 * randperm.  Outputs: pos_idx [n_img, min(num_pos, n)], neg_idx [n_img, min(batch, n)] (int64, ascending index, zero past
 * the count), pos_valid / neg_valid (uint8, same shapes), counts int32 [n_img, 2] = (#pos picked, #neg picked). */
int dgod_balanced_sample(const void* labels, int labels_are_int64, const float* keys, int n_img, int n,
                         int num_pos, int batch_size_per_image, int64_t* pos_idx, uint8_t* pos_valid,
                         int64_t* neg_idx, uint8_t* neg_valid, int32_t* counts, dgod_stream_t stream);

/* The RoI heads' sampled RoIs (TV roi_heads.py:615-678 after the sampler) for a batch in one launch, no host
 * synchronisation.  Inputs: dgod_balanced_sample's pos_idx/pos_valid [n_img, cap_pos] and neg_idx/neg_valid
 * [n_img, cap_neg] over the candidates of dgod_iou_match's padded layout (boxes [n_img, n_boxes, 4] with box_counts,
 * ground truths appended), and that call's labels / clamped_idx [n_img, n_slots].  Per image the picked candidates in
 * ascending index order (the union of the two ascending lists) fill batch_size_per_image slots:
 *   s_props     [n_img, batch, 4] the candidate's box; 0 in an empty slot
 *   s_labels    [n_img, batch]    int64, its label; -100 in an empty slot
 *   reg_targets [n_img, batch, 4] BoxCoder(weights).encode of its matched ground truth (ground truth 0 of the image in an
 *                                 empty slot, zeros for an image without any) against its box, or against (0,0,1,1)
 *                                 in an empty slot; the arithmetic of the eager torch composition, op for op.
 * cap_pos, cap_neg, batch_size_per_image <= 1024. */
int dgod_sample_rois(const int64_t* pos_idx, const uint8_t* pos_valid, int cap_pos, const int64_t* neg_idx,
                     const uint8_t* neg_valid, int cap_neg, const int64_t* labels, const int64_t* clamped_idx, int n_img,
                     int n_slots, const float* boxes, const int32_t* box_counts, int n_boxes, const float* gt_boxes,
                     const int32_t* gt_offsets, int batch_size_per_image, float wx, float wy, float ww, float wh,
                     float* s_props, int64_t* s_labels, float* reg_targets, dgod_stream_t stream);

/* ------------------------------------------------------------------ batched NMS */

size_t dgod_nms_workspace_bytes(int n_total, int n_seg, int max_seg_len);
/* Greedy NMS for n_seg independent segments (images) in one call; within a segment boxes of
 * different `groups` never suppress each other.  Suppression iff fp32 IoU, widened to double,
 * is > iou_threshold (the CPU op's comparison).  Order: descending score, equal scores by
 * ascending index.  offset_mode=1 reproduces _batched_nms_coordinate_trick's arithmetic
 * (boxes + group*(max+1) in fp32, one run per segment); offset_mode=0 is _batched_nms_vanilla.
 * valid (optional) masks boxes out before NMS.  keep_out[s*out_stride + j] are segment-relative
 * indices, out_stride = max_out_per_seg > 0 ? max_out_per_seg : max_seg_len; keep_count[s] is
 * min(kept, out_stride).  status[0] != 0 afterwards means group ids were outside [0,65535] and
 * the result is invalid (caller must densify the ids and retry). */
int dgod_nms_batched(const float* boxes /*device [n_total,4]*/, const float* scores /*device*/,
                     const int64_t* groups /*device [n_total] or NULL*/,
                     const uint8_t* valid /*device [n_total] or NULL*/,
                     const int32_t* seg_offsets /*device [n_seg+1]*/,
                     int n_seg, int n_total, int max_seg_len,
                     double iou_threshold, int offset_mode, int max_out_per_seg,
                     int64_t* keep_out /*device*/, int32_t* keep_count /*device [n_seg]*/,
                     int32_t* status /*device [1]*/,
                     void* workspace, size_t workspace_bytes, dgod_stream_t stream);

/* ------------------------------------------------------------------ RPN proposals */

typedef struct {
  int n_img, n_levels, anchors_per_loc;
  int height[DGOD_MAX_LEVELS], width[DGOD_MAX_LEVELS];       /* feature grid per level */
  int stride_h[DGOD_MAX_LEVELS], stride_w[DGOD_MAX_LEVELS];  /* image_size // grid (TV anchor_utils.py:119-125) */
  float cell_anchors[DGOD_MAX_LEVELS][DGOD_MAX_CELL_ANCHORS][4]; /* rounded base anchors (TV anchor_utils.py:58-74) */
  int pre_nms_top_n, post_nms_top_n;
  double nms_thresh;
  float min_size, score_thresh;
  float bbox_xform_clip; /* log(1000/16) */
} dgod_rpn_config;

size_t dgod_rpn_workspace_bytes(const dgod_rpn_config* cfg);
/* From the raw RPN head outputs to post-NMS proposals, anchors generated analytically and only
 * the per-level top-k survivors decoded.  objectness[l] is [n_img, A, H_l, W_l], deltas[l] is
 * [n_img, 4A, H_l, W_l] (NCHW, fp32).  image_sizes is device [n_img,2] = (h, w) as float.
 * out_boxes [n_img, post_nms_top_n, 4], out_scores [n_img, post_nms_top_n] (rows past
 * out_count[i] are zero), out_count [n_img]. */
int dgod_rpn_proposals(const dgod_rpn_config* cfg /*host*/,
                       const float* const* objectness /*host array of device ptrs*/,
                       const float* const* deltas /*host array of device ptrs*/,
                       const float* image_sizes /*device [n_img,2]*/,
                       float* out_boxes, float* out_scores, int32_t* out_count,
                       void* workspace, size_t workspace_bytes, dgod_stream_t stream);

/* Same stages as TV rpn.py:242-297 on already-decoded proposals [n_img, A_total, 4] and
 * objectness logits [n_img, A_total] in torchvision's concatenated (level, y, x, a) order.
 * cfg supplies n_img, n_levels, height*width*anchors_per_loc per level and the thresholds. */
int dgod_rpn_filter(const dgod_rpn_config* cfg /*host*/,
                    const float* proposals /*device*/, const float* objectness /*device*/,
                    const float* image_sizes /*device [n_img,2]*/,
                    float* out_boxes, float* out_scores, int32_t* out_count,
                    void* workspace, size_t workspace_bytes, dgod_stream_t stream);

/* ------------------------------------------------------------------ MultiScaleRoIAlign */

typedef struct {
  int n_levels;                     /* 1 = plain roi_align, no level mapping */
  int batch, channels;
  int height[DGOD_MAX_LEVELS], width[DGOD_MAX_LEVELS];
  float spatial_scale[DGOD_MAX_LEVELS];
  int channels_last;                /* 0: NCHW contiguous, 1: NHWC (channels_last) memory */
  int dtype;                        /* DGOD_F32 or DGOD_BF16 (features, output, grads) */
  int pooled_h, pooled_w, sampling_ratio, aligned;
  int k_min, k_max;                 /* LevelMapper (TV ops/poolers.py:47-84) */
  float canonical_scale, canonical_level, eps;
} dgod_roi_config;

/* rois: device [K,5] fp32 (batch index, x1, y1, x2, y2) in image coordinates (TV
 * ops/poolers.py:87-95).  roi_img_offsets (optional, device [batch+1]) promises that rois are
 * grouped by image; the backward uses it to bound its per-tile scan.  out: [K,C,PH,PW]. */
size_t dgod_msroi_align_fwd_workspace_bytes(int n_rois);
/* workspace (optional, 128-byte aligned, dgod_msroi_align_fwd_workspace_bytes(n_rois) bytes) holds the
 * per-RoI plans of the TMA kernel (channels_last, 7x7 bins, sampling_ratio 1..2, C in {64,128,256});
 * without it, or for other shapes, the table-driven / generic kernels run. */
int dgod_msroi_align_fwd(const dgod_roi_config* cfg /*host*/,
                         const void* const* feats /*host array of device ptrs*/,
                         const float* rois, int n_rois, void* out,
                         void* workspace, size_t workspace_bytes, dgod_stream_t stream);
size_t dgod_msroi_align_bwd_workspace_bytes(int n_rois);
/* Workspace for the configuration at hand (>= the size above): additionally holds the per-tile RoI lists of the
 * owner-computes kernel, whose size depends on the level geometry. */
size_t dgod_msroi_align_bwd_workspace_bytes_cfg(const dgod_roi_config* cfg /*host*/, int n_rois);
/* grad_feats[l] is fully overwritten (zero where no RoI contributes): no memset required.
 * algo 0 picks the owner-computes kernel when the shape allows (channels_last, 7x7 bins, sampling_ratio 1..2,
 * C % 64 == 0) and the workspace has dgod_msroi_align_bwd_workspace_bytes_cfg bytes: every tile of the gradient
 * maps is accumulated on chip and written once, deterministic.  Else the TMA bulk-reduce kernel (C in
 * {64,128,256}, cooperative launch), else the vector-RED / atomic scatter (fp32) or the deterministic tile
 * gather (bf16); 1 forces the scatter, 2 the tile gather, 3 the TMA bulk-reduce kernel, 4 owner-computes.
 * workspace: 128-byte aligned (RoI plans, tile lists, counters). */
int dgod_msroi_align_bwd(const dgod_roi_config* cfg /*host*/,
                         const void* grad_out /*device [K,C,PH,PW]*/,
                         const float* rois, int n_rois,
                         const int32_t* roi_img_offsets /*device [batch+1] or NULL*/,
                         void* const* grad_feats /*host array of device ptrs*/,
                         int algo /*0 auto, 1 scatter, 2 tile gather, 3 TMA bulk reduce, 4 owner-computes, 5 owner-computes with claimed work items*/,
                         void* workspace, size_t workspace_bytes, dgod_stream_t stream);

/* ------------------------------------------------------------------ box head post-processing */

/* BoxCoder.decode_single (TV _utils.py:186-224): rel_codes [n, n_cls*4], boxes [n,4]
 * -> out [n, n_cls*4]. */
int dgod_box_decode(const float* rel_codes, const float* boxes, int n, int n_cls,
                    float wx, float wy, float ww, float wh, float xform_clip,
                    float* out, dgod_stream_t stream);

/* TV roi_heads.py:692-724 for a batch: decode, softmax, clip to the image, drop the
 * background column, then flag candidates with score > score_thresh and both sides >= min_size.
 * Rows of image i are box_offsets[i]..box_offsets[i+1).  Outputs are laid out
 * [n_rows, n_cls-1]: cand_boxes [..,4], cand_scores, cand_labels (int64), cand_valid (uint8). */
int dgod_detect_candidates(const float* class_logits /*[n_rows,n_cls]*/,
                           const float* box_regression /*[n_rows,n_cls*4]*/,
                           const float* proposals /*[n_rows,4]*/,
                           const int32_t* box_offsets /*device [n_img+1]*/,
                           const float* image_sizes /*device [n_img,2]*/,
                           int n_img, int n_rows, int n_cls,
                           float wx, float wy, float ww, float wh, float xform_clip,
                           float score_thresh, float min_size,
                           float* cand_boxes, float* cand_scores, int64_t* cand_labels,
                           uint8_t* cand_valid, dgod_stream_t stream);

/* ------------------------------------------------------------------ input side (SURVEY.md §8f rank 4) */

/* GeneralizedRCNNTransform.forward for a batch in one launch: per image normalize with mean/std (host
 * [channels], channels <= 4), bilinear resize [channels,in_h,in_w] -> [out_h,out_w] with ATen's
 * align_corners=False source coordinates (scale = in/out), written zero-padded into
 * out [n_img, channels, pad_h, pad_w] (NCHW, fully overwritten).  images: host array of device pointers
 * to contiguous fp32 [channels, in_h, in_w]; the size arrays are host arrays.  The caller computes out_h /
 * out_w (floor(in * min(min_size/min(h,w), max_size/max(h,w))), TV transform.py:25-83) and the padded size. */
int dgod_image_batch(const float* const* images, const int* in_h, const int* in_w, const int* out_h,
                     const int* out_w, int n_img, int channels, const float* mean, const float* std,
                     float* out, int pad_h, int pad_w, dgod_stream_t stream);
/* The same for uint8 images [channels, in_h, in_w] with values 0..255, as they leave the decoder: every tap is divided by 255
 * on load — the dataset's `image / 255.0` (DrivingDataset.py:53), bit-identical to doing it on the host — so that the
 * host->device copy moves a quarter of the bytes. */
int dgod_image_batch_u8(const uint8_t* const* images, const int* in_h, const int* in_w, const int* out_h,
                        const int* out_w, int n_img, int channels, const float* mean, const float* std,
                        float* out, int pad_h, int pad_w, dgod_stream_t stream);

/* ------------------------------------------------------------------ layout */

/* [batch][channels][hw] -> [batch][hw][channels] (NCHW -> NHWC), fp32 or bf16.  Used by the host
 * layer to give NCHW feature maps (torchvision's default layout, fasterrcnn.py:317) the
 * channels_last RoIAlign kernels. */
int dgod_nchw_to_nhwc(const void* src, void* dst, int batch, int channels, int hw, int dtype,
                      dgod_stream_t stream);

/* ------------------------------------------------------------------ backbone: bottleneck epilogue, FPN top-down merge, stem */

/* Maps are fp32 [n, c, h, w] in NCHW (channels_last = 0) or NHWC memory (channels_last = 1: c % 4 == 0 and every
 * pointer 16-byte aligned).  All of them are bit-exact with the ATen ops they replace.
 *
 * FPN merge: out = (lat + bias[c]) + nearest_upsample(coarse [n, c, hc, wc]) to [h, w], the two adds in that order, the
 * source pixel as ATen's nearest mode computes it (min(floor(y * ((float)hc / h)), hc - 1), likewise x).  out may be
 * the same buffer as lat. */
int dgod_fpn_merge_fwd(const float* lat, const float* bias /*device [c]*/, const float* coarse, float* out, int n, int h,
                       int w, int hc, int wc, int c, int channels_last, dgod_stream_t stream);
/* Its backward for the coarse level: g_coarse = g_lb + (sum of g_fine [n, c, h, w] over the fine pixels of ATen's
 * upsample_nearest2d_backward: rows [ceil(yc * s), ceil((yc + 1) * s)) clamped to h, s = (float)h / hc, likewise
 * columns; summed row-major into a float starting at 0).  g_lb (the coarse level's other gradient) may be NULL (zero)
 * and may be the same buffer as g_coarse. */
int dgod_fpn_merge_bwd(const float* g_fine, const float* g_lb, float* g_coarse, int n, int h, int w, int hc, int wc,
                       int c, int channels_last, dgod_stream_t stream);
/* Frozen ResNet stem epilogue: out [n, c, ho, wo] = max_pool2d(relu(conv + shift[c]), 3, stride 2, pad 1) with
 * ho = (h - 1) / 2 + 1, wo = (w - 1) / 2 + 1; NaN propagates as through clamp_min and max_pool2d.  No backward. */
int dgod_stem_pool_fwd(const float* conv, const float* shift /*device [c]*/, float* out, int n, int h, int w, int c,
                       int ho, int wo, int channels_last, dgod_stream_t stream);

/* Folded ResNet Bottleneck epilogue, one pass per convolution: out [n, c, h, w] = relu(conv + shift[c]) (conv1, conv2),
 * relu((conv + shift[c]) + res) (identity block tail) or relu((conv + shift[c]) + (res + res_shift[c])) (downsample
 * block tail: res is the downsample conv's output without its shift).  res and res_shift may be NULL (res_shift only
 * with res).  Same layout rules as above for every map; bit-exact with ATen's adds in that order and relu_
 * (clamp_min: NaN passes).  No backward: the gradient is threshold_backward(grad_out, out, 0) for conv and res. */
int dgod_shift_relu_fwd(const float* conv, const float* shift /*device [c]*/, const float* res,
                        const float* res_shift /*device [c]*/, float* out, int n, int h, int w, int c, int channels_last,
                        dgod_stream_t stream);
/* The same pass without the ReLU: out = conv + bias[c], a convolution's bias add, bit-exact with ATen's add_. */
int dgod_bias_add_fwd(const float* conv, const float* bias /*device [c]*/, float* out, int n, int h, int w, int c,
                      int channels_last, dgod_stream_t stream);

/* The same four on bf16 maps (__nv_bfloat16 [n, c, h, w]; channels_last needs c % 8 == 0 and 16-byte aligned pointers);
 * biases and shifts stay fp32.  Bit-exact with the ATen bf16 ops under autocast: fp32 math, every add's result rounded
 * to bf16 (round to nearest even), each bias / shift rounded to bf16 before it is added (autocast casts a conv's bias),
 * and the merge backward's window sum rounded once to bf16 before g_lb is added. */
int dgod_fpn_merge_fwd_bf16(const void* lat, const float* bias /*device [c]*/, const void* coarse, void* out, int n,
                            int h, int w, int hc, int wc, int c, int channels_last, dgod_stream_t stream);
int dgod_fpn_merge_bwd_bf16(const void* g_fine, const void* g_lb, void* g_coarse, int n, int h, int w, int hc, int wc,
                            int c, int channels_last, dgod_stream_t stream);
int dgod_stem_pool_fwd_bf16(const void* conv, const float* shift /*device [c]*/, void* out, int n, int h, int w, int c,
                            int ho, int wo, int channels_last, dgod_stream_t stream);
int dgod_shift_relu_fwd_bf16(const void* conv, const float* shift /*device [c]*/, const void* res,
                             const float* res_shift /*device [c]*/, void* out, int n, int h, int w, int c,
                             int channels_last, dgod_stream_t stream);

/* ------------------------------------------------------------------ validation mAP (COCO bbox, no crowd, area "all") */

#define DGOD_MAP_MAX_DETS_PER_IMAGE 4096
#define DGOD_MAP_MAX_GTS_PER_IMAGE 1024
#define DGOD_MAP_MAX_IOU_THRESHOLDS 32

/* Greedy matching of n_img images, one CTA each.  Detections (det_boxes [n,4] xyxy fp32, 16-byte aligned; det_scores
 * [n] fp32; det_labels [n] int64) and ground truths (gt_boxes [m,4], gt_labels [m]) are concatenated over the images,
 * image i owning rows [off[i], off[i+1]) of det_offsets / gt_offsets (device int32 [n_img+1]).  max_dets_per_image /
 * max_gts_per_image bound every image's counts (they size shared memory; <= the caps above).  iou_thresholds: device
 * double [n_thr], 1 <= n_thr <= 32.
 * Per (image, label): detections in descending score order (stable; -0.0 ties +0.0), the first max_det kept; for each
 * threshold t (as min(t, 1 - 1e-10)) each kept detection in turn takes the unmatched GT of its label with the largest
 * IoU >= t, the later GT on equal IoU; IoU = pycocotools bbIou in double on the boxes converted to xywh in fp32.
 * Writes, at every detection's own row: tp_mask (bit t set = matched at threshold t) and kept (1 = within max_det). */
int dgod_map_match(const float* det_boxes, const float* det_scores, const int64_t* det_labels, const int* det_offsets,
                   const float* gt_boxes, const int64_t* gt_labels, const int* gt_offsets, int n_img,
                   int max_dets_per_image, int max_gts_per_image, const double* iou_thresholds, int n_thr, int max_det,
                   uint32_t* tp_mask, uint8_t* kept, dgod_stream_t stream);
/* Per-class precision / recall tables (COCOeval.accumulate), one CTA per (class, threshold).  tp_mask [n_records]: the
 * kept detections' masks grouped by class and, within a class, in descending score order (ties: earlier image, then
 * the image's own order); class k owns rows [seg_offsets[k], seg_offsets[k+1]) (device int32 [n_classes+1]; rows
 * past the last segment are ignored); gt_counts: device int32 [n_classes]; rec_thresholds: device double [n_rec_thr].
 * Writes precision [n_thr, n_rec_thr, n_classes] and recall [n_thr, n_classes] (float64; -1 for a class without
 * ground truth).  Workspace: dgod_map_accumulate_workspace_bytes(n_records, n_thr). */
size_t dgod_map_accumulate_workspace_bytes(int n_records, int n_thr);
int dgod_map_accumulate(const uint32_t* tp_mask, const int* seg_offsets, const int* gt_counts, int n_classes,
                        int n_records, const double* rec_thresholds, int n_rec_thr, int n_thr, double* precision,
                        double* recall, void* workspace, size_t workspace_bytes, dgod_stream_t stream);

/* ------------------------------------------------------------------ fp32 matrix product (box head) */

/* C [m, n] = epilogue(A B^T) on the tcgen05 tensor cores, fp32-accurate (3xTF32: each operand split into two tf32
 * parts, three products accumulated in fp32; NaN / inf propagate to the same positions as in an fp32 SGEMM, where
 * SGEMM gives +-inf this may give NaN).  A [m, k] is `a` stored [m, k] row-major, or with a_trans the transpose of
 * `a` stored [k, m]; B [n, k] likewise from `b` ([n, k], or [k, n] with b_trans).  Epilogue, in this order: + bias[n]
 * (device [n] or NULL), ReLU if relu (NaN passes), C *= (mask > 0) with mask device [m, n] or NULL.  c: device [m, n].
 * m, k >= 1, n % 32 == 0, every pointer 16-byte aligned.  Workspace: dgod_linear_tc_workspace_bytes(m, n, k) (the
 * split operands; 0 for invalid sizes). */
size_t dgod_linear_tc_workspace_bytes(int m, int n, int k);
int dgod_linear_tc(const float* a, int a_trans, const float* b, int b_trans, int m, int n, int k, const float* bias,
                   int relu, const float* mask, float* c, void* workspace, size_t workspace_bytes, dgod_stream_t stream);

/* ------------------------------------------------------------------ RPN head (after its 3x3 conv) */

/* All n_levels (<= DGOD_MAX_LEVELS) levels in one launch.  c[l]: the 3x3 conv's output WITHOUT its bias, NHWC fp32
 * [n_img, height[l], width[l], channels] (16-byte aligned); channels == 256 and anchors == 3 only.  bias [channels]
 * (the 3x3 conv's), w_cls [anchors, channels], b_cls [anchors], w_bbox [4 anchors, channels], b_bbox [4 anchors]:
 * device fp32, weights and bias 16-byte aligned.  With t = relu_(c + bias) (clamp_min: NaN passes):
 * objectness[l] [n_img, anchors, h, w] = W_cls t + b_cls and deltas[l] [n_img, 4 anchors, h, w] = W_bbox t + b_bbox,
 * NCHW-contiguous, each product an fp32 fma chain over the channels in ascending order. */
int dgod_rpn_head_fwd(const float* const* c, int n_levels, const int* height, const int* width, int n_img, int channels,
                      int anchors, const float* bias, const float* w_cls, const float* b_cls, const float* w_bbox,
                      const float* b_bbox, float* const* objectness, float* const* deltas, dgod_stream_t stream);
/* Its backward from the incoming gradients grad_objectness[l] / grad_deltas[l] (NCHW-contiguous, shapes of the
 * outputs above): grad_c[l] (NHWC like c) = (t <= 0) ? 0 : W_cls^T g_obj + W_bbox^T g_deltas (threshold_backward), and
 * grad_params [256 * 15 + 256 + 15] = dW_cls [3, 256], dW_bbox [12, 256], d bias [256], d b_cls [3], d b_bbox [12],
 * each summed over every pixel of every level.  Deterministic (fixed partition and summation order, no atomics).  Two
 * launches, the second a programmatic dependent launch.  Workspace: dgod_rpn_head_workspace_bytes() (depends on the
 * current device's SM count; 0 if it cannot be queried). */
size_t dgod_rpn_head_workspace_bytes(void);
int dgod_rpn_head_bwd(const float* const* c, int n_levels, const int* height, const int* width, int n_img, int channels,
                      int anchors, const float* bias, const float* w_cls, const float* w_bbox,
                      const float* const* grad_objectness, const float* const* grad_deltas, float* const* grad_c,
                      float* grad_params, void* workspace, size_t workspace_bytes, dgod_stream_t stream);

/* ------------------------------------------------------------------ gradient reversal */

/* out[i] = (-grad[i]) * alpha  (DGcommon.py:40-42; out may alias grad). */
int dgod_grl_scale(const void* grad, void* out, int64_t n, float alpha, int dtype,
                   dgod_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* DGOD_B200_H_ */
