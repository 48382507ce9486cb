/*
 * det_b200.h -- C ABI of libdet_b200.so: the B200-native (sm_100a) post-backbone detection hot path.
 *
 * The reference (andompesta/object-detection-pytorch-rust) has NO native/FFI layer: its boundary for this
 * path is a set of Python callables (SURVEY.md section 8b).  Each entry point below names the reference
 * callable it replaces (paths relative to the reference root).  The Python package `det_b200` mirrors those
 * callables 1:1 and forwards here through ctypes; INTEGRATION.md shows the binding a maintainer would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`; plain pointers + sizes only;
 *   - the library never allocates, frees or retains memory: outputs and workspaces are caller-owned;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), no internal synchronisation;
 *   - return value: DET_OK (0) or a negative DET_ERR_* code; det_last_error() gives a message;
 *   - boxes are fp32 XYXY rows, indices int64, labels int8, counts int32 (reference dtypes, SURVEY 8b);
 *   - all floating-point work is IEEE fp32 with FMA contraction disabled, so IoU / keep decisions are
 *     bit-identical to the reference's CPU torch path.
 */
#ifndef DET_B200_H
#define DET_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DET_OK 0
#define DET_ERR_BAD_ARG (-1)      /* null pointer, negative size, inconsistent shape            */
#define DET_ERR_UNSUPPORTED (-2)  /* size beyond a documented limit                              */
#define DET_ERR_WORKSPACE (-3)    /* workspace too small (see the matching *_workspace_bytes)    */
#define DET_ERR_CUDA (-4)         /* a CUDA runtime call failed; see det_last_error()            */
#define DET_ERR_ALIGN (-5)        /* pointer not aligned as documented                           */

#define DET_ABI_VERSION 3

/* element type of a detection head passed to the *_typed entry points.  A 16-bit head is widened to fp32 as it is
 * loaded (exact) and then takes the fp32 path's instructions: every output is bit-identical to the fp32 entry point
 * fed the same head converted to fp32.  Outputs keep their documented dtypes. */
#define DET_DTYPE_F32 0
#define DET_DTYPE_BF16 1
#define DET_DTYPE_F16 2

#if defined(__GNUC__)
#define DET_API __attribute__((visibility("default")))
#else
#define DET_API
#endif

DET_API int det_abi_version(void);
DET_API const char* det_last_error(void);
/* number of SMs of the current device (grid sizing); negative on error */
DET_API int det_sm_count(void);

/* ------------------------------------------------------------------------------------------------------------
 * (2) pairwise box overlap -- replaces pairwise_iou / pairwise_ioa / pairwise_intersection /
 *     matched_boxlist_iou, python/src/structures/boxes.py:193, :217, :173, :235.
 * ---------------------------------------------------------------------------------------------------------- */
#define DET_OVERLAP_IOU 0
#define DET_OVERLAP_IOA 1
#define DET_OVERLAP_INTERSECTION 2
/* out[n*m + j]; boxes1 (n,4), boxes2 (m,4), 16-byte aligned rows */
DET_API int det_pairwise_overlap(const float* boxes1, int64_t n, const float* boxes2, int64_t m, int mode, float* out,
                         void* stream);
/* out[i] = IoU(boxes1[i], boxes2[i]) without the empty-box guard (0/0 -> NaN), boxes.py:235 */
DET_API int det_matched_iou(const float* boxes1, const float* boxes2, int64_t n, float* out, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * (1) box codec -- replaces Box2BoxTransform.apply_deltas / get_deltas,
 *     python/src/models/components/box_regression.py:75 and :33.
 * ---------------------------------------------------------------------------------------------------------- */
/* deltas (m, k*4), boxes (m,4) -> out (m, k*4).  weights = (wx,wy,ww,wh). */
DET_API int det_apply_deltas(const float* deltas, const float* boxes, int64_t m, int k, float wx, float wy, float ww,
                     float wh, float scale_clamp, float* out, void* stream);
/* backward of det_apply_deltas (the reference's apply_deltas is differentiable through autograd; its GIoU loss and any
 * ROI box head rely on that): grad_out (m, k*4) -> grad_deltas (m, k*4) and/or grad_boxes (m,4), either may be NULL. */
DET_API int det_apply_deltas_backward(const float* deltas, const float* boxes, const float* grad_out, int64_t m, int k,
                              float wx, float wy, float ww, float wh, float scale_clamp, float* grad_deltas,
                              float* grad_boxes, void* stream);
/* src (m,4), tgt (m,4) -> out (m,4).  *invalid_flag (device int32, caller-zeroed) is set to 1 if any src width
 * <= 0 (the reference asserts, box_regression.py:72). */
DET_API int det_get_deltas(const float* src, const float* tgt, int64_t m, float wx, float wy, float ww, float wh, float* out,
                   int32_t* invalid_flag, void* stream);
/* grid anchors of one level, order (h,w,a) -- replaces AnchorGenerator._grid_anchors,
 * python/src/models/modules/anchor_generators.py:158.  cell_anchors (a,4) device. out (h*w*a,4). */
DET_API int det_grid_anchors(const float* cell_anchors, int a, int h, int w, int stride, float offset, float* out,
                     void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * (1) RPN head decode, DELTA mode -- replaces the layout change + _decode_proposals,
 *     python/src/models/rpn.py:270-284 and :330-348 (anchors synthesised in-kernel, never read).
 *     objectness (n,a,h,w) NCHW, deltas (n,a*4,h,w) NCHW -> logits_out (n,h*w*a), boxes_out (n,h*w*a,4).
 *     `out_img_stride` = number of anchors between consecutive images in the outputs (>= h*w*a) and
 *     `out_offset` the first anchor slot of this level, so all levels can land in one (n,R[,4]) buffer.
 * ---------------------------------------------------------------------------------------------------------- */
DET_API int det_rpn_decode_level(const float* objectness, const float* deltas, int n, int a, int h, int w, int stride,
                         float offset, const float* cell_anchors, float wx, float wy, float ww, float wh,
                         float scale_clamp, float* logits_out, float* boxes_out, int64_t out_img_stride,
                         int64_t out_offset, void* stream);

/* All pyramid levels of the RPN head in ONE launch (csrc/box_ops.cu rpn_decode_flat_kernel: a warp per 128-position
 * tile, outputs staged in shared memory and written as contiguous spans).  Every level shares n and a; level l:
 * objectness (n,a,h,w), deltas (n,a*4,h,w), cell_anchors (a,4), first output row out_offset.  Levels whose h*w is not
 * a multiple of 4 (or whose heads are not 16-byte aligned) ride along with scalar loads; unaligned cell anchors or
 * a > 4 fall back to one det_rpn_decode_level launch per level -- same results. */
typedef struct det_rpn_level {
    const float* objectness;
    const float* deltas;
    const float* cell_anchors;
    int32_t h, w, stride, reserved;
    int64_t out_offset;
} det_rpn_level_t;
DET_API int det_rpn_decode(const det_rpn_level_t* levels_host, int num_levels, int n, int a, float offset, float wx, float wy,
                   float ww, float wh, float scale_clamp, float* logits_out, float* boxes_out, int64_t out_img_stride,
                   void* stream);
/* det_rpn_decode on a head of element type head_dtype (DET_DTYPE_*): the objectness and deltas pointers of every level
 * point at elements of that type (the `reserved` field stays unread).  A level streams with vector loads when h*w % 4 == 0
 * and both planes are aligned to 4 elements; others ride along with scalar loads.  Unknown head_dtype: DET_ERR_BAD_ARG.
 * det_rpn_decode is this call with DET_DTYPE_F32. */
DET_API int det_rpn_decode_typed(const det_rpn_level_t* levels_host, int num_levels, int n, int a, float offset, float wx,
                         float wy, float ww, float wh, float scale_clamp, float* logits_out, float* boxes_out,
                         int64_t out_img_stride, int head_dtype, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * (3) batched, category-partitioned NMS -- replaces batched_nms, python/src/utils.py:96 (and through it
 *     torchvision.ops.batched_nms / nms), for a whole batch of images in one call.
 *
 *   boxes (n, m_max, 4), scores (n, m_max), categories (n, m_max) int64 or NULL (single category),
 *   counts (n) int32 or NULL (every image has m_max boxes).
 *   keep (n, max_out) int64: kept indices into the image's own m_max rows, by descending score, ties by
 *   lower index; keep_counts (n) int32 = min(#kept, max_out).
 *   mode: DET_NMS_AUTO reproduces the reference's CPU rule per image (count <= 1000 -> torchvision's
 *         coordinate-offset trick evaluated in fp32, else per-category); the other two force a branch.
 *   limits: m_max <= 131071, 0 <= category < 32768.
 * ---------------------------------------------------------------------------------------------------------- */
#define DET_NMS_AUTO 0
#define DET_NMS_PER_CATEGORY 1
#define DET_NMS_OFFSET_TRICK 2
DET_API int64_t det_nms_workspace_bytes(int n, int64_t m_max);
DET_API int det_nms_batched(const float* boxes, const float* scores, const int64_t* categories, const int32_t* counts,
                    int n, int64_t m_max, double iou_threshold, int mode, int64_t max_out, int64_t* keep,
                    int32_t* keep_counts, void* workspace, int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * (3) RPN proposal selection for the whole batch -- replaces find_top_rpn_proposals,
 *     python/src/models/utils.py:9-109: per-level top-k, finite filter, clip, small-box filter, per-level NMS,
 *     post-NMS top-k.  Input: all levels concatenated, boxes (n, r, 4), logits (n, r); level_sizes_host[l] =
 *     anchors of level l (sum = r, l < 16); image_sizes (n,2) int32 device (h,w).
 *     out_boxes (n, post_nms_topk, 4), out_logits (n, post_nms_topk), out_counts (n) int32.
 *     *nonfinite_flag (device int32, caller-zeroed) is set if a selected box/logit is Inf/NaN (the reference
 *     raises FloatingPointError in training, models/utils.py:82).
 * ---------------------------------------------------------------------------------------------------------- */
DET_API int64_t det_rpn_proposals_workspace_bytes(int n, int64_t r);
DET_API int det_rpn_proposals(const float* boxes, const float* logits, int n, int64_t r, const int64_t* level_sizes_host,
                      int num_levels, const int32_t* image_sizes, double nms_thresh, int64_t pre_nms_topk,
                      int64_t post_nms_topk, float min_box_size, float* out_boxes, float* out_logits,
                      int32_t* out_counts, int32_t* nonfinite_flag, void* workspace, int64_t workspace_bytes,
                      void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * (1)+(3) YOLO-grid head: fused decode + score threshold + per-class NMS, one launch for the batch.
 *     No reference implementation exists (SURVEY.md 8 row a15); the specification is oracle/ref_torch.py
 *     yolo_decode / yolo_select_nms.  head (n, s, s, b*5+c) channels-last fp32; priors (b,2) device (w,h).
 *     Optional dense outputs (NULL to skip): boxes (n,p,4), conf (n,p), scores (n,p,c), p = s*s*b.
 *     Detections: det_flat (n,max_det) int64 = predictor*c + class, det_boxes (n,max_det,4), det_scores
 *     (n,max_det), det_count (n) int32, by descending score.  limit: p*c <= 4096, c <= 1024.
 * ---------------------------------------------------------------------------------------------------------- */
DET_API int det_yolo_decode_nms(const float* head, int n, int s, int b, int c, int img_h, int img_w, const float* priors,
                        float scale_clamp, int clip, float score_thresh, double iou_threshold, int mode,
                        float* dense_boxes, float* dense_conf, float* dense_scores, int64_t max_det,
                        int64_t* det_flat, float* det_boxes, float* det_scores, int32_t* det_count, void* stream);

/* the same call with 32-bit detection indices (same values; p*c <= 4096 always fits): the serving wire format of
 * det_b200.YoloHostPipeline -- 4 bytes less per detection to move over PCIe. */
DET_API int det_yolo_decode_nms_i32(const float* head, int n, int s, int b, int c, int img_h, int img_w, const float* priors,
                            float scale_clamp, int clip, float score_thresh, double iou_threshold, int mode,
                            float* dense_boxes, float* dense_conf, float* dense_scores, int64_t max_det,
                            int32_t* det_flat32, float* det_boxes, float* det_scores, int32_t* det_count, void* stream);

/* both of the above for a head of element type head_dtype (DET_DTYPE_*), aligned to 4 elements: det_flat is int64
 * (index_bytes 8) or int32 (index_bytes 4).  Unknown head_dtype or index_bytes: DET_ERR_BAD_ARG.  det_yolo_decode_nms
 * and det_yolo_decode_nms_i32 are this call with DET_DTYPE_F32. */
DET_API int det_yolo_decode_nms_typed(const void* head, int head_dtype, int n, int s, int b, int c, int img_h, int img_w,
                              const float* priors, float scale_clamp, int clip, float score_thresh,
                              double iou_threshold, int mode, float* dense_boxes, float* dense_conf, float* dense_scores,
                              int64_t max_det, void* det_flat, int index_bytes, float* det_boxes, float* det_scores,
                              int32_t* det_count, void* stream);

/* dense anchor head (YOLOv3-style, NCHW): head (n, a*(5+c), h, w) -> boxes (n,h*w*a,4), best score, best class.
 * anchors_wh (a,2) device.  Output slots as in det_rpn_decode_level. */
DET_API int det_dense_decode_level(const float* head, int n, int a, int c, int h, int w, int stride, const float* anchors_wh,
                           float scale_clamp, float* boxes_out, float* score_out, int64_t* class_out,
                           int64_t out_img_stride, int64_t out_offset, void* stream);

/* All pyramid levels of a dense anchor head in ONE launch (flat 16-byte streaming kernel, csrc/dense_decode.cu).
 * Every level shares n, a, c; level l: head (n, a*(5+c), h, w) device, anchors_wh (a,2) device, first output row
 * out_offset.  Levels whose h*w is not a multiple of 4 (or whose head is not 16-byte aligned) ride in the same launch
 * with scalar loads.  limit: h*w < 2^30 per level. */
typedef struct det_dense_level {
    const float* head;
    const float* anchors_wh;
    int32_t h, w, stride, reserved;
    int64_t out_offset;
} det_dense_level_t;
DET_API int det_dense_decode(const det_dense_level_t* levels_host, int num_levels, int n, int a, int c, float scale_clamp,
                     float* boxes_out, float* score_out, int64_t* class_out, int64_t out_img_stride, void* stream);
/* det_dense_decode on a head of element type head_dtype (DET_DTYPE_*): every level's `head` points at elements of that
 * type (the `reserved` field stays unread).  Every pyramid is one launch: a level streams with vector loads when
 * h*w % 4 == 0 and its head is aligned to 4 elements; other levels ride along with scalar loads.  Unknown
 * head_dtype: DET_ERR_BAD_ARG.  det_dense_decode is this call with DET_DTYPE_F32. */
DET_API int det_dense_decode_typed(const det_dense_level_t* levels_host, int num_levels, int n, int a, int c,
                           float scale_clamp, float* boxes_out, float* score_out, int64_t* class_out,
                           int64_t out_img_stride, int head_dtype, void* stream);

/* Dense anchor head as a detector runs it (BASELINE configs[3]): decode -> score > score_thresh -> per-class NMS ->
 * top max_det, two launches for the whole batch and no dense output.  Specification: oracle/ref_torch.py
 * dense_select_nms over dense_decode (own; SURVEY.md 8 row a15), i.e. per image
 *     cand = nonzero(score > score_thresh);  keep = batched_nms(boxes[cand], score[cand], class[cand], iou)[:max_det]
 * with batched_nms = python/src/utils.py:96-119 (`mode` as in det_nms_batched).
 *   det_idx (n,max_det) int64 = row of the detection in the (level,h,w,a) order of det_dense_decode,
 *   det_boxes (n,max_det,4), det_scores (n,max_det), det_classes (n,max_det) int64, det_count (n) int32,
 *   by descending score, ties by lower row.
 *   cand_cap (<= 4096): capacity of the per-image candidate list.  An image with more candidates gets
 *   det_count = -1 and *overflow_flag (device int32, may be NULL; written by the call) = 1 -- nothing is guessed.
 *   gate bit 0: read the objectness plane first and skip the class/box planes of positions that cannot pass
 *   (exact: score <= sigmoid(objectness)); clear = stream the whole head.
 *   gate bit 1: the per-image counters at the head of the workspace are known to
 *   be zero.  The call always LEAVES them zero (the NMS CTA of an image resets its counter), so a caller that zeroes
 *   the first det_dense_detect_counter_bytes(n) bytes of a workspace once and then uses it for nothing else may set
 *   this bit on every call: exactly two launches, no memset node.  Clear = the call clears the counters itself.
 *   limits: every level h*w % 4 == 0 and 16-byte aligned heads (else DET_ERR_UNSUPPORTED). */
DET_API int64_t det_dense_detect_workspace_bytes(int n, int64_t cand_cap);
DET_API int64_t det_dense_detect_counter_bytes(int n); /* size of the counter block at the head of the workspace */
DET_API int det_dense_detect(const det_dense_level_t* levels_host, int num_levels, int n, int a, int c, float scale_clamp,
                     float score_thresh, double iou_threshold, int mode, int gate, int64_t cand_cap, int64_t max_det,
                     int64_t* det_idx, float* det_boxes, float* det_scores, int64_t* det_classes, int32_t* det_count,
                     int32_t* overflow_flag, void* workspace, int64_t workspace_bytes, void* stream);
/* det_dense_detect on a head of element type head_dtype (DET_DTYPE_*), as in det_dense_decode_typed.  Limits: every level
 * h*w % 4 == 0 and heads aligned to 4 elements (else DET_ERR_UNSUPPORTED).  Unknown head_dtype: DET_ERR_BAD_ARG.
 * det_dense_detect is this call with DET_DTYPE_F32. */
DET_API int det_dense_detect_typed(const det_dense_level_t* levels_host, int num_levels, int n, int a, int c,
                           float scale_clamp, float score_thresh, double iou_threshold, int mode, int gate,
                           int64_t cand_cap, int64_t max_det, int64_t* det_idx, float* det_boxes, float* det_scores,
                           int64_t* det_classes, int32_t* det_count, int32_t* overflow_flag, void* workspace,
                           int64_t workspace_bytes, int head_dtype, void* stream);

/* Row-ordered candidate compaction and the final gather of the UNFUSED detector path (det_dense_decode ->
 * det_threshold_compact -> det_nms_batched -> det_gather_detections): the exact route for images that overflow
 * det_dense_detect's candidate list and for pyramids outside its limits.  Same specification as det_dense_detect
 * (oracle/ref_torch.py dense_select_nms): cand = nonzero(score > score_thresh) in row order.
 *   boxes (n,r,4), scores (n,r), classes (n,r) int64 or NULL -> cand_rows (n,cap) int64 (row of every candidate),
 *   cand_boxes (n,cap,4), cand_scores (n,cap), cand_classes (n,cap) int64, cand_counts (n) int32 = min(#candidates, cap).
 * det_gather_detections: keep (n,max_det) int64 indices into an image's candidate list + keep_counts (n) (the outputs of
 *   det_nms_batched) -> det_idx (original rows; the candidate index when cand_rows is NULL), det_boxes, det_scores,
 *   det_classes, each (n,max_det[,4]); entries past keep_counts stay untouched. */
DET_API int det_threshold_compact(const float* boxes, const float* scores, const int64_t* classes, int n, int64_t r,
                          float score_thresh, int64_t cap, int64_t* cand_rows, float* cand_boxes, float* cand_scores,
                          int64_t* cand_classes, int32_t* cand_counts, void* stream);
DET_API int det_gather_detections(const int64_t* keep, const int32_t* keep_counts, int n, int64_t max_det,
                          const int64_t* cand_rows, const float* cand_boxes, const float* cand_scores,
                          const int64_t* cand_classes, int64_t cap, int64_t* det_idx, float* det_boxes, float* det_scores,
                          int64_t* det_classes, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * (4a) IoU target assignment -- replaces pairwise_iou + Matcher.__call__ + set_low_quality_matches_ as driven
 *      by label_and_sample_anchors, python/src/models/rpn.py:161-168 / components/matcher.py:53-120, for the
 *      whole batch and without materialising the (G,R) matrix.
 *      gt_boxes (sum_g,4) concatenated, gt_offsets (n+1) int32, anchors (r,4).
 *      thresholds_host (num_thresholds) ascending, labels_host (num_thresholds+1) in {-1,0,1}.
 *      matched_idx (n,r) int64, labels (n,r) int8, matched_iou (n,r) fp32 or NULL.
 * ---------------------------------------------------------------------------------------------------------- */
DET_API int64_t det_match_workspace_bytes(int n, int64_t r, int64_t sum_g);
DET_API int det_match_anchors(const float* gt_boxes, const int32_t* gt_offsets, int n, int64_t sum_g, const float* anchors,
                      int64_t r, const float* thresholds_host, const int32_t* labels_host, int num_thresholds,
                      int allow_low_quality, int64_t* matched_idx, int8_t* labels, float* matched_iou,
                      void* workspace, int64_t workspace_bytes, void* stream);
/* The same assignment for GRID anchors -- the (R,4) table AnchorGenerator.forward produces
 * (python/src/models/modules/anchor_generators.py:158-179: per level h*w positions x `a` cell anchors, order (h,w,a),
 * levels concatenated) -- in ONE streaming pass (csrc/assign_grid.cu): a gt-centric kernel marks the 8 x 4-position tiles
 * each box can overlap and evaluates every row maximum on the closed-form window where it can be attained, then one
 * anchor-centric kernel (a tile per warp) writes labels and matched indices including the low-quality promotion.
 * Results are bit-identical to det_match_anchors.  levels_host[l] = {h, w, stride, 0, first_row}; rows must be consecutive and sum to r;
 * a in {1, 3, 9}, num_levels * a <= 32, num_levels <= 8 (else DET_ERR_UNSUPPORTED: use det_match_anchors).
 * Optional per-image statistics for det_subsample_labels_grid (both NULL to skip): stats (n,4) int32 = {#positives,
 * #ignored (label -1), 0, 0} (written by the call), pos_list (n, list_cap) int32 = anchor row | label << 24 of the
 * first list_cap positives in arrival order (needs r < 2^24). */
typedef struct det_anchor_level {
    int32_t h, w, stride, reserved;
    int64_t first_row;
} det_anchor_level_t;
DET_API int64_t det_match_grid_workspace_bytes(int n, int64_t sum_g, const det_anchor_level_t* levels_host, int num_levels);
DET_API int det_match_grid(const float* gt_boxes, const int32_t* gt_offsets, int n, int64_t sum_g, const float* anchors,
                   int64_t r, const det_anchor_level_t* levels_host, int num_levels, int a,
                   const float* thresholds_host, const int32_t* labels_host, int num_thresholds, int allow_low_quality,
                   int64_t* matched_idx, int8_t* labels, float* matched_iou, int32_t* stats, int32_t* pos_list,
                   int list_cap, void* workspace, int64_t workspace_bytes, void* stream);
/* Matcher on a materialised quality matrix (g,r) -- Matcher.__call__, matcher.py:53. */
DET_API int det_match_quality(const float* quality, int64_t g, int64_t r, const float* thresholds_host,
                      const int32_t* labels_host, int num_thresholds, int allow_low_quality, int64_t* matched_idx,
                      int8_t* labels, int32_t* negative_flag, void* workspace, int64_t workspace_bytes, void* stream);

/* Uniform random fg/bg subsample on the device (statistically, not stream-, equivalent to subsample_labels +
 * _subsample_labels, python/src/utils.py:34 / models/rpn.py:108): keeps min(#pos, int(s*f)) positives and
 * min(#neg, s-#pos) negatives per image, everything else becomes -1.  labels (n,r) int8 in place.  int(s*f) is the
 * reference's Python double product truncated (utils.py:63), hence the double argument. */
DET_API int det_subsample_labels(int8_t* labels, int n, int64_t r, int num_samples, double positive_fraction, uint64_t seed,
                         void* stream);

/* det_subsample_labels driven by det_match_grid's statistics: same result bit for bit (same hash keys, same
 * permutation walk), but the label row is never read in full -- positives are ranked from pos_list, negatives found by
 * the walk, the row is overwritten with -1 and the survivors written back.  Images outside the fast path's
 * preconditions (positives not sparse, negatives not dense or not thinned, list overflow) run det_subsample_labels'
 * code.  Optional sample list for det_rpn_loss_sampled (both NULL to skip): samples (n, sample_cap) int32 = anchor row |
 * label << 24 of every anchor whose final label is not -1, sample_count (n) int32. */
DET_API int det_subsample_labels_grid(int8_t* labels, int n, int64_t r, int num_samples, double positive_fraction,
                              uint64_t seed, const int32_t* stats, const int32_t* pos_list, int list_cap,
                              int32_t* samples, int32_t* sample_count, int sample_cap, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * (4b) fused RPN loss forward + backward -- replaces losses + _dense_box_regression_loss + get_deltas,
 *      python/src/models/rpn.py:187-244, components/box_regression.py:128-168, :33-73, and autograd's backward.
 *      logits (n,r), deltas (n,r,4), labels (n,r) int8, matched_idx (n,r) int64, gt as above, anchors (r,4).
 *      loss_type 0 = smooth-L1(beta) (beta<1e-5 -> L1), 1 = GIoU.
 *      accumulators: 16 floats of device scratch owned by the caller, ZERO BEFORE THE FIRST CALL; every launch leaves
 *      them zero again (the kernel's last CTA re-arms them), so no memset surrounds the call.  One buffer per stream.
 *      sums_out (8) fp32, written by that last CTA: [0] = objectness BCE sum * grad_scale_cls, [1] = localisation sum *
 *      grad_scale_loc -- with grad_scale_x = loss_weight_x / (batch_size_per_image * n_global) these ARE the reference's
 *      weighted, normalised losses (rpn.py:238-243) -- [2] = #pos, [3] = #neg, rest 0.
 *      grad_logits (n,r) / grad_deltas (n,r,4): d(sum)/d(input) * grad_scale_{cls,loc} [* upstream[0|1]];
 *      NULL to skip backward.  upstream: device float[2] (d total / d cls_loss, d total / d loc_loss) or NULL (= 1),
 *      read by the kernel so an autograd backward needs no host synchronisation.
 * ---------------------------------------------------------------------------------------------------------- */
DET_API int det_rpn_loss(const float* logits, const float* deltas, const int8_t* labels, const int64_t* matched_idx,
                 const float* gt_boxes, const int32_t* gt_offsets, const float* anchors, int n, int64_t r, float wx,
                 float wy, float ww, float wh, float scale_clamp, int loss_type, float smooth_l1_beta,
                 float grad_scale_cls, float grad_scale_loc, const float* upstream, float* accumulators, float* sums_out,
                 float* grad_logits, float* grad_deltas, void* stream);

/* Sample-list-only ("lazy") assignment for GRID anchors: label_and_sample_anchors (rpn.py:132-185) reduced to what the
 * losses read -- per image the <= num_samples sampled anchors (anchor row | label << 24), the matched gt index of each
 * and their number -- without computing, writing or reading anything for the other ~R anchors.  Positives are found from
 * the gt side (closed-form windows where IoU >= the lowest positive threshold, or IoU == the row maximum, can occur),
 * negatives by the sampler's permutation walk, which labels only the anchors it visits; every label is the same fp32
 * arithmetic as det_match_grid, so the lists equal det_match_grid + det_subsample_labels_grid's as sets whenever that
 * sampler walks too (dense, thinned negatives -- any realistic image).  Images whose positives are dense (a gt with row
 * maximum 0 promotes every anchor, matcher.py:110-113) are labelled in full into scratch_labels (n, r) int8 (device
 * scratch, otherwise untouched).  labels_host[0] must be 0 or -1.  samples / sample_gt (n, sample_cap) int32,
 * sample_count (n) int32.  Feed them to det_rpn_loss_sampled (matched_idx = NULL). */
DET_API int64_t det_assign_sampled_workspace_bytes(int n, int64_t sum_g, int list_cap);
DET_API int det_assign_sampled(const float* gt_boxes, const int32_t* gt_offsets, int n, int64_t sum_g, const float* anchors,
                       int64_t r, const det_anchor_level_t* levels_host, int num_levels, int a,
                       const float* thresholds_host, const int32_t* labels_host, int num_thresholds,
                       int allow_low_quality, int num_samples, double positive_fraction, uint64_t seed,
                       int8_t* scratch_labels, int32_t* samples, int32_t* sample_gt, int32_t* sample_count,
                       int sample_cap, void* workspace, int64_t workspace_bytes, void* stream);

/* The same loss on the SAMPLED anchors only (the labels of everything else are -1 and contribute nothing, rpn.py:222-236),
 * reading the head where the convolutions left it and writing the gradients in the same layout -- O(samples) traffic
 * instead of O(r), no layout change (rpn.py:270-284), no (n,r) label sweep.
 *   layout: num_levels >= 1: levels_host[l] = per-level NCHW planes objectness (n,a,h,w), deltas (n,a*4,h,w) (channel =
 *   a*4 + component, rpn.py:278-280) and their gradient planes (all NULL to skip backward); the *_flat pointers are
 *   ignored.  num_levels == 0: logits_flat (n,r), deltas_flat (n,r,4), grad_*_flat or NULL.
 *   samples / sample_count / sample_cap: from det_subsample_labels_grid, with matched_idx (n,r) from det_match_grid and
 *   sample_gt = NULL -- or from det_assign_sampled, with its sample_gt (n, sample_cap) and matched_idx = NULL.
 *   Gradient buffers are NOT swept: zero them once (cudaMemset) -- or keep them persistent and pass the PREVIOUS step's
 *   sample list as clear_samples / clear_count (NULL, NULL otherwise): those entries are reset to zero first.
 *   accumulators: 8 floats of device scratch, zero before the first call (the kernel re-arms them).
 *   sums_out (8): [0] = objectness BCE sum * scale_cls, [1] = localisation sum * scale_loc, [2] = #pos, [3] = #neg, rest 0
 *   -- written by the kernel's last CTA, so no memset and no scaling op surround the call.  Gradients are
 *   d(sum)/d(input) * scale_{cls,loc} [* upstream[0|1]]. */
typedef struct det_head_level {
    const float* objectness;
    const float* deltas;
    float* grad_objectness;
    float* grad_deltas;
    int32_t h, w;
} det_head_level_t;
DET_API int det_rpn_loss_sampled(const det_head_level_t* levels_host, int num_levels, int a, const float* logits_flat,
                         const float* deltas_flat, float* grad_logits_flat, float* grad_deltas_flat,
                         const int32_t* samples, const int32_t* sample_count, int sample_cap,
                         const int32_t* clear_samples, const int32_t* clear_count, const int64_t* matched_idx,
                         const int32_t* sample_gt, const float* gt_boxes, const int32_t* gt_offsets, const float* anchors,
                         int n, int64_t r,
                         float wx, float wy, float ww, float wh, float scale_clamp, int loss_type,
                         float smooth_l1_beta, float scale_cls, float scale_loc, const float* upstream,
                         float* accumulators, float* sums_out, void* stream);

/* YOLO-grid fused loss forward + backward (own specification: oracle/ref_torch.py yolo_loss).
 * head (n,s,s,b*5+c); labels (n,p) int8; matched_idx (n,p) int64; gt_classes (sum_g) int64.
 * accumulators: as for det_rpn_loss.  sums_out (8): [0] = lambda_coord * loc * grad_scale, [1] = obj * grad_scale,
 * [2] = cls * grad_scale, [3] = #pos, [4] = #neg, rest 0 (grad_scale = 1 / normaliser: the reported losses).
 * grad_head same shape as head (fully written) or NULL.
 * grad = d(lambda_coord*loc + obj + cls)/d(head) * grad_scale [* upstream[0..2] per term], upstream device float[3] or NULL. */
DET_API int det_yolo_loss(const float* head, const int8_t* labels, const int64_t* matched_idx, const float* gt_boxes,
                  const int64_t* gt_classes, const int32_t* gt_offsets, int n, int s, int b, int c, int img_h,
                  int img_w, const float* priors, float lambda_coord, float lambda_noobj, float grad_scale,
                  const float* upstream, float* accumulators, float* sums_out, float* grad_head, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * (next tier, SURVEY 8f rank 2) FPN level assignment + ROIAlign / ROIPool over a feature pyramid -- replaces
 *      assign_boxes_to_levels / ROIPooler.forward / ROIAlign.forward,
 *      python/src/models/modules/roi_poolers.py:103-131, :269-331, :55-72 (torchvision.ops.roi_align underneath),
 *      and the ROIPool pooler type, roi_poolers.py:224-231 (torchvision.ops.roi_pool underneath).
 *      det_roi_levels: level_out[i] = clamp(floor(canonical_level + log2(sqrt(area_i)/canonical_box_size + 1e-8)),
 *      min_level, max_level) - min_level, boxes (m,4).
 *      Every pooling entry: box i (boxes (m,4) fp32, 16-byte aligned) samples the level `level[i]` (int64; NULL when
 *      num_levels == 1) of image batch_index[i] (int32); level l: data (n, c, h, w) contiguous, spatial_scale =
 *      1/stride.  out / grad_out (m, c, out_h, out_w).  m == 0 returns DET_OK without reading any pointer.
 *
 *      Feature dtypes (feat_dtype / grad_dtype = DET_DTYPE_*; all levels and the output share it): every element is
 *      widened to fp32 on load, the arithmetic is fp32, and the output is rounded once to the feature dtype
 *      (__float2bfloat16_rn / __float2half_rn).  So a bf16 / fp16 result is bit-identical to the fp32 call on the
 *      widened features followed by torch's .to(dtype) -- torchvision's autocast rule for roi_align / roi_pool.  An
 *      unknown dtype: DET_ERR_BAD_ARG before any CUDA call.  Gradients always accumulate into fp32 buffers.
 *
 *      det_roi_align_levels_typed: torchvision roi_align; sampling_ratio <= 0: ceil(roi / bins) samples per bin;
 *      aligned != 0: half-pixel shift (ROIAlignV2).  det_roi_align_levels is this call with DET_DTYPE_F32.
 *      det_roi_align_levels_backward_typed: levels' `data` are the fp32 GRADIENT buffers (n, c, h, w), zeroed by the
 *      caller and accumulated into with atomics; grad_out of grad_dtype.  det_roi_align_levels_backward is this call
 *      with DET_DTYPE_F32.
 *      det_roi_pool_levels: torchvision roi_pool (max pooling).  start = round(x * spatial_scale) in fp32, halves away
 *      from zero; roi size max(end - start + 1, 1); bin p of an axis covers [floor(p * bin), ceil((p + 1) * bin)) +
 *      start, clamped to [0, h] / [0, w].  An empty bin outputs 0; otherwise the max, scanned rows then columns with a
 *      strict `>` from -FLT_MAX (first maximum wins, NaN never taken; a bin of NaN / -inf gives -FLT_MAX, -inf in 16
 *      bit).  argmax (m, c, out_h, out_w) int32 = h*W + w inside the box's level plane, -1 when nothing was taken; NULL:
 *      not written (inference).  sampling_ratio and aligned do not apply.  Every level needs h*w < 2^31.
 *      det_roi_pool_levels_backward: grad level[batch_index[i]][c][argmax] += grad_out for every argmax >= 0, fp32
 *      atomics into the zeroed fp32 gradient buffers `grad_levels_host[l].data`; argmax from the forward.
 * ---------------------------------------------------------------------------------------------------------- */
typedef struct det_feature_level {
    const float* data;  /* the *_typed and pool entries: elements of their feat_dtype, cast to this pointer type */
    int32_t h, w;
    float spatial_scale;
    int32_t reserved;
} det_feature_level_t;
DET_API int det_roi_levels(const float* boxes, int64_t m, int min_level, int max_level, float canonical_box_size,
                   int canonical_level, int64_t* level_out, void* stream);
DET_API int det_roi_align_levels(const det_feature_level_t* levels_host, int num_levels, int n, int c, const float* boxes,
                         const int32_t* batch_index, const int64_t* level, int64_t m, int out_h, int out_w,
                         int sampling_ratio, int aligned, float* out, void* stream);
DET_API int det_roi_align_levels_typed(const det_feature_level_t* levels_host, int num_levels, int n, int c,
                                       const float* boxes, const int32_t* batch_index, const int64_t* level, int64_t m,
                                       int out_h, int out_w, int sampling_ratio, int aligned, void* out, int feat_dtype,
                                       void* stream);
DET_API int det_roi_align_levels_backward(const det_feature_level_t* grad_levels_host, int num_levels, int n, int c,
                                  const float* boxes, const int32_t* batch_index, const int64_t* level, int64_t m,
                                  int out_h, int out_w, int sampling_ratio, int aligned, const float* grad_out,
                                  void* stream);
DET_API int det_roi_align_levels_backward_typed(const det_feature_level_t* grad_levels_host, int num_levels, int n,
                                                int c, const float* boxes, const int32_t* batch_index,
                                                const int64_t* level, int64_t m, int out_h, int out_w,
                                                int sampling_ratio, int aligned, const void* grad_out, int grad_dtype,
                                                void* stream);
DET_API int det_roi_pool_levels(const det_feature_level_t* levels_host, int num_levels, int n, int c, const float* boxes,
                                const int32_t* batch_index, const int64_t* level, int64_t m, int out_h, int out_w,
                                void* out, int32_t* argmax, int feat_dtype, void* stream);
DET_API int det_roi_pool_levels_backward(const det_feature_level_t* grad_levels_host, int num_levels, int n, int c,
                                         const int32_t* batch_index, const int64_t* level, int64_t m, int out_h,
                                         int out_w, const int32_t* argmax, const void* grad_out, int grad_dtype,
                                         void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Second-stage (Fast R-CNN box predictor) inference -- what detectron2's FastRCNNOutputLayers.inference /
 *      fast_rcnn_inference_single_image do with the box head's outputs, for the whole batch in two launches and no
 *      host synchronisation.  The reference never wrote the ROI predictor (SURVEY.md section 0); the specification is
 *      tests/fast_rcnn_oracle.py fast_rcnn_inference_single_image ("parity unpinned by reference").  Per image, P its rows and
 *      K = num_classes:
 *        probs = softmax(logits) with the row sum taken in column order (e[0] + e[1] + ... + e[K]);
 *        boxes = apply_deltas(deltas, proposals) with k = K, or k = 1 (class_agnostic, deltas (m,4));
 *        a row is valid iff all its boxes and all its K+1 probabilities are finite -- invalid rows are dropped;
 *        boxes clipped to (h, w) as Boxes.clip;  candidates (i, c), c < K, with probs[i, c] > score_thresh in
 *        row-major order;  keep = batched_nms(box, score, c, iou_threshold)[:max_det] (`mode` as in det_nms_batched).
 *      Deviation from detectron2: i is the proposal's row among the image's ORIGINAL rows (detectron2 counts the rows
 *      left after the validity filter).
 *
 *   Inputs: class_logits (m, K+1) and box_deltas (m, K*4) or (m, 4), both of element type head_dtype (DET_DTYPE_*;
 *   16-bit rows are widened on load, so results are bit-identical to the fp32 call on the widened values); rows read
 *   with 16-byte loads where the row pitch and base allow, scalar loads otherwise.  proposals (m, 4) fp32, 16-byte
 *   aligned.  row_offsets (n+1) int32: image b owns rows [row_offsets[b], row_offsets[b+1]) (row_offsets[0] = 0,
 *   non-decreasing, row_offsets[n] = m).  image_sizes (n, 2) int32 (h, w).  weights (wx, wy, ww, wh) and scale_clamp of
 *   Box2BoxTransform (ROI heads: 10, 10, 5, 5 and log(1000/16)).
 *   det_roi_detect_typed outputs: det_idx (n, max_det) int64 = i*K + c, det_boxes (n, max_det, 4), det_scores (n, max_det),
 *   det_classes (n, max_det) int64, det_count (n) int32; by descending score, ties by lower flat id; entries past the
 *   count are undefined.  Workspace, gate bit 1, cand_cap and the overflow report are det_dense_detect's: an image with
 *   more than cand_cap candidates gets det_count = -1 and sets *overflow_flag (may be NULL; written by the call); gate
 *   bit 0 is ignored.  m == 0: det_count = 0 for every image, no input pointer is read.
 *   det_roi_decode_dense_typed: the dense form for the exact route taken by overflowing images -- scores_out
 *   (n, p_max, K) and boxes_out (n, p_max, K, 4, 16-byte aligned), row i of image b at [b, i]; the probability and clipped
 *   box of every (row, class), NaN for every class of an invalid row and of the rows i >= the image's count.  Rows past
 *   p_max are not decoded (p_max >= every image's count).  det_threshold_compact over the (n, p_max*K) view (classes =
 *   flat % K) -> det_nms_batched -> det_gather_detections then gives det_roi_detect's result.  decoded != 0: the rows
 *   are probabilities (m, K+1) and boxes (m, K*4) / (m, 4) already (detectron2's fast_rcnn_inference inputs); they are
 *   taken as they are -- validity rule, clip and padding only -- and proposals / weights are not read.
 *   limits: num_classes <= 4096 and m * num_classes < 2^31 (every flat id fits int32), cand_cap in [1, 4096]: otherwise
 *   DET_ERR_UNSUPPORTED.  Unknown head_dtype, unknown mode, max_det < 1, null pointers: DET_ERR_BAD_ARG.
 * ---------------------------------------------------------------------------------------------------------- */
DET_API int64_t det_roi_detect_workspace_bytes(int n, int64_t cand_cap);
DET_API int64_t det_roi_detect_counter_bytes(int n); /* size of the counter block at the head of the workspace */
DET_API int det_roi_detect_typed(const void* class_logits, const void* box_deltas, int head_dtype, const float* proposals,
                                 const int32_t* row_offsets, int n, int64_t m, int num_classes, int class_agnostic,
                                 const int32_t* image_sizes, float wx, float wy, float ww, float wh, float scale_clamp,
                                 float score_thresh, double iou_threshold, int mode, int gate, int64_t cand_cap,
                                 int64_t max_det, int64_t* det_idx, float* det_boxes, float* det_scores,
                                 int64_t* det_classes, int32_t* det_count, int32_t* overflow_flag, void* workspace,
                                 int64_t workspace_bytes, void* stream);
DET_API int det_roi_decode_dense_typed(const void* class_logits, const void* box_deltas, int head_dtype,
                                       const float* proposals, const int32_t* row_offsets, int n, int64_t m,
                                       int num_classes, int class_agnostic, const int32_t* image_sizes, float wx,
                                       float wy, float ww, float wh, float scale_clamp, int decoded, int p_max,
                                       float* scores_out, float* boxes_out, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Second-stage (Fast R-CNN box predictor) training losses, forward and backward in one launch -- what detectron2's
 *      FastRCNNOutputLayers.losses (softmax cross-entropy + box_reg_loss) and _log_classification_stats compute, and
 *      autograd's backward of both.  Own specification ("parity unpinned by reference"): tests/fast_rcnn_loss_oracle.py.
 *      Over the m rows the box head saw (packed over the batch), K = num_classes, fg = 0 <= gt < K:
 *        loss_cls = scale_cls * sum_i (logsumexp(x_i) - x_i[gt_i])
 *        loss_box_reg = scale_loc * sum_{fg i} L(d_i, proposal_i, gt_box_i), d_i = the 4 deltas of class gt_i (the row's
 *        only 4 when class_agnostic); L = smooth-L1(beta) on get_deltas(proposal, gt_box) (beta < 1e-5: L1), loss_type 0,
 *        or GIoU on apply_deltas(d, proposal) with scale_clamp, loss_type 1; weights (wx, wy, ww, wh) as Box2BoxTransform.
 *      With scale_x = loss_weight_x / m these are detectron2's losses (F.cross_entropy mean, box loss / m).
 *
 *   Inputs: class_logits (m, K+1) with background last and box_deltas (m, K*4) or (m, 4), both of element type
 *   head_dtype (DET_DTYPE_*; 16-bit rows are widened on load, so sums are the fp32 call's on the widened values).
 *   proposals, gt_boxes (m, 4) fp32, 16-byte aligned (a row without gt carries any box: it is read only for fg rows).
 *   gt_classes (m) int64.  A label outside [0, K] contributes to neither sum, gets zero gradient rows and is counted.
 *   accumulators: 16 floats of device scratch, zero before the first call; the last CTA re-arms them (one per stream).
 *   sums_out (8) fp32, written by that last CTA: [loss_cls, loss_box_reg, num_fg, num_accurate, fg_num_accurate,
 *   num_false_negative, num_bad_labels, 0] -- counts exact; pred = argmax of the row (first maximum, NaN the largest,
 *   first NaN wins).  grad_logits / grad_deltas: shaped and typed like the inputs, both or neither (forward only);
 *   written in full: (softmax - onehot(gt)) * s_cls and, for fg rows, d L / d d_i * s_loc in the 4 columns of class gt,
 *   0 everywhere else; s_x = scale_x * upstream[x] with upstream device float[2] or NULL (= 1), so a backward launch
 *   needs no host synchronisation.  16-bit gradients are the fp32 values rounded once (torch's .to(dtype)).
 *   m == 0: sums_out = 0 and no input pointer is read.  Limits: num_classes <= 4096, m < 2^24: DET_ERR_UNSUPPORTED.
 *   Null pointers, unknown head_dtype or loss_type: DET_ERR_BAD_ARG, before any CUDA call.
 * ---------------------------------------------------------------------------------------------------------- */
DET_API int det_fast_rcnn_loss_typed(const void* class_logits, const void* box_deltas, int head_dtype,
                                     const float* proposals, const int64_t* gt_classes, const float* gt_boxes,
                                     int64_t m, int num_classes, int class_agnostic, float wx, float wy, float ww,
                                     float wh, float scale_clamp, int loss_type, float smooth_l1_beta, float scale_cls,
                                     float scale_loc, const float* upstream, float* accumulators, float* sums_out,
                                     void* grad_logits, void* grad_deltas, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Batched ROI-head proposal sampling -- replaces label_and_sample_proposals + _sample_proposals,
 *      python/src/models/roi.py:68-193, add_ground_truth_to_proposals, models/utils.py:111-155, and
 *      subsample_labels, utils.py:34-76, for the whole batch in two launches, no host synchronisation, no allocation
 *      and no memset (CUDA-graph capturable).
 *   Inputs: proposals (n, p_stride, 4) fp32, image b's P_b = proposal_counts[b] (device int32) rows first -- rows past
 *   P_b are never read (rpn_proposals_batched's padded output).  gt_boxes (sum_g, 4) fp32 with gt_offsets (n+1) int32
 *   (Matcher.pack_gt), gt_classes (sum_g) int64, num_classes K.  The Matcher rule as det_match_anchors'.
 *   seed: device uint64 read by the kernel, so a replayed graph that advances it draws new samples.
 *   Per image, candidates j = 0 .. P_b-1 are the proposals, then (append_gt) P_b .. P_b+G_b-1 the gt boxes:
 *     label: pair_iou(gt, candidate) -> column max (first maximum) -> threshold buckets -> low-quality promotion
 *       (IoU == a gt's row maximum; a row maximum of 0 promotes every candidate) -> class gt_classes[matched], K for
 *       matcher label 0, -1 for label -1; every candidate of an image without gt is background (K).
 *     counts: fg = class neither -1 nor K; want_fg = min(#fg, int(S*f)) with S*f in double, want_bg = min(#bg,
 *       S - want_fg).  S = batch_size_per_image.
 *     selection: candidate j's key is sample_key(image_seed(*seed, b), j) (csrc/assign.cuh), a bijection of j; each class
 *       keeps its want smallest keys (a uniformly random subset; the stream differs from torch.randperm's).
 *   Outputs, padded (n, S): foreground rows first, then background, each in ascending j.  out_boxes (n,S,4) = the
 *   candidate's box; out_gt_classes (n,S) int64; out_gt_boxes (n,S,4) = gt[matched] for every row of an image with gt,
 *   the row's own box for an image without; out_matched (n,S) int32 = index into the image's gt (-1 without gt);
 *   out_src (n,S) int32 = j.  out_count (n) int32 = want_fg + want_bg, out_num_fg (n) int32 = want_fg.  Rows past the
 *   count: src = -1, gt_classes = -1, matched = -1, zero boxes.  *underfull_flag (device int32, written by the call) = 1
 *   iff some image has count < S.
 *   workspace: det_roi_sample_workspace_bytes(n, p_stride, sum_g) bytes, 16-byte aligned, ALL ZERO BEFORE THE FIRST
 *   CALL; every call leaves it zero again (so a larger one fits every smaller call).  One workspace per stream.
 *   Limits: n <= 65535, p_stride < 2^24, sum_g < 2^24, S < 2^24, n * p_stride + sum_g < 2^31: DET_ERR_UNSUPPORTED.
 *   Null pointers (proposals may be NULL when p_stride == 0, gt_boxes / gt_classes when sum_g == 0), S < 1, f outside
 *   [0, 1], num_classes < 1, a bad rule: DET_ERR_BAD_ARG, before any CUDA call.  n == 0: DET_OK, nothing is read.
 * ---------------------------------------------------------------------------------------------------------- */
DET_API int64_t det_roi_sample_workspace_bytes(int n, int64_t p_stride, int64_t sum_g);
DET_API int det_roi_sample_proposals(const float* proposals, const int32_t* proposal_counts, int n, int64_t p_stride,
                                     const float* gt_boxes, const int32_t* gt_offsets, const int64_t* gt_classes,
                                     int64_t sum_g, int num_classes, const float* thresholds_host,
                                     const int32_t* labels_host, int num_thresholds, int allow_low_quality,
                                     int batch_size_per_image, double positive_fraction, int append_gt,
                                     const uint64_t* seed, float* out_boxes, int64_t* out_gt_classes,
                                     float* out_gt_boxes, int32_t* out_matched, int32_t* out_src, int32_t* out_count,
                                     int32_t* out_num_fg, int32_t* underfull_flag, void* workspace,
                                     int64_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * (e) the training path's one collective over NVLink peer memory instead of NCCL: SUM of the `width`-float loss/count
 *     vector (the sums the reference logs per step, python/src/models/rpn.py:216-220, 238-241) over `world` ranks.
 *     Every rank owns a buffer of slots * world * 16 floats that is mapped into every peer (symmetric memory);
 *     peers_dev = device array of the `world` buffer base pointers as seen from this rank.
 *     publish: store this rank's vector + the step stamp into record [slot][rank] of every peer's buffer.
 *     collect: wait until all `world` records of [slot] in the LOCAL buffer carry `stamp`, write their sum (rank
 *     order) to out.  A wait longer than timeout_ns writes NaN and sets *error_flag (may be NULL) -- never hangs.
 *     Issue publish(t), collect(t - 1) in stream order with slots >= 4 (csrc/peer.cu explains the slot reuse).
 * ---------------------------------------------------------------------------------------------------------- */
DET_API int det_peer_sums_publish(const float* sums, int width, int rank, int world, const void* peers_dev, int slots,
                          int slot, uint32_t stamp, void* stream);
DET_API int det_peer_sums_collect(float* out, int width, int world, const float* local_buf, int slots, int slot,
                          uint32_t stamp, int64_t timeout_ns, int32_t* error_flag, void* stream);
/* compute + collective in ONE kernel: det_yolo_loss whose last CTA publishes the batch's finished `sums_out` vector
 * (`width` <= 8 floats) as step `stamp` and collects step stamp - lag into `out`.  done_counter is unused since ABI 2
 * (the accumulators carry the arrival ticket).  The out buffer of step t must stay untouched until step t + 1's. */
typedef struct det_peer_ctx {
    const void* peers_dev;
    float* out;
    int32_t* error_flag;
    int32_t* done_counter;
    int64_t timeout_ns;
    int32_t width, rank, world, slots;
    uint32_t stamp, lag;
    uint32_t* stamp_counter; /* device, may be NULL.  Non-NULL: the kernel stamps with ++(*stamp_counter) and ignores
                                `stamp`, so a captured CUDA graph can be replayed (same number of replays on every rank) */
} det_peer_ctx_t;
DET_API int det_yolo_loss_peer(const float* head, const int8_t* labels, const int64_t* matched_idx, const float* gt_boxes,
                       const int64_t* gt_classes, const int32_t* gt_offsets, int n, int s, int b, int c, int img_h,
                       int img_w, const float* priors, float lambda_coord, float lambda_noobj, float grad_scale,
                       const float* upstream, float* accumulators, float* sums_out, float* grad_head,
                       const det_peer_ctx_t* peer, void* stream);
/* both in one launch per training step: publish step `stamp` (slot stamp % slots), then collect step stamp - lag into
 * out (nothing is collected while stamp <= lag). */
DET_API int det_peer_sums_exchange(const float* sums, float* out, int width, int rank, int world, const void* peers_dev,
                           int slots, uint32_t stamp, uint32_t lag, int64_t timeout_ns, int32_t* error_flag, void* stream);
/* det_peer_sums_exchange with the step stamp kept on the device: the kernel uses ++(*stamp_counter) (uint32, zero before
 * the first step) as this step's stamp, so the call can be captured in a CUDA graph and replayed -- every rank must
 * replay the same number of times.  `out` receives the world sum of step stamp - lag (untouched on the first steps). */
DET_API int det_peer_sums_exchange_dev(const float* sums, float* out, int width, int rank, int world, const void* peers_dev,
                               int slots, uint32_t* stamp_counter, uint32_t lag, int64_t timeout_ns, int32_t* error_flag,
                               void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DET_B200_H */
