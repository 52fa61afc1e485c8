/*
 * misob200.h — C ABI of libmisob200.so: the B200 (sm_100a) implementation of the detection
 * post-processing + region-feature hot path behind miso's torchvision Faster/Mask R-CNN
 * pipelines (microfossil/particle-object-detection).
 *
 * Citations: `ref:` = the reference repo, `tv:` = torchvision 0.26.0 Python layer (the
 * third-party code the reference calls), `tv-csrc:` = torchvision native sources (dispatcher
 * registration sites; see SURVEY.md). Each entry point names the reference interface it
 * replaces. INTEGRATION.md shows the reference-side binding (ctypes) for every symbol.
 *
 * Conventions (SURVEY.md §8 b3):
 *  - every pointer is a DEVICE pointer unless the name ends in _host or the comment says so;
 *  - the caller owns all memory including the workspace; the library never allocates,
 *    frees or synchronises; all work is enqueued on `stream`;
 *  - return value: MB_OK, a negative MB_ERR_* argument error, or a positive cudaError_t;
 *  - data-dependent counts are written to device memory;
 *  - fp32 boxes are (x1, y1, x2, y2); indices are int64 where torchvision returns int64.
 */
#ifndef MISOB200_H
#define MISOB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MB_ABI_VERSION 1

#define MB_OK 0
#define MB_ERR_INVALID_ARG (-1)
#define MB_ERR_WORKSPACE (-2)   /* workspace too small */
#define MB_ERR_UNSUPPORTED (-3) /* configuration outside the implemented envelope */

#define MB_MAX_LEVELS 8
#define MB_MAX_ANCHORS_PER_LOC 16
#define MB_MAX_IMAGES 64

typedef struct CUstream_st* mb_stream_t;

int mb_abi_version(void);
/* "sm_100a;<kernel list>" — lets the host assert the CUDA build is the one loaded */
const char* mb_build_info(void);

/* ------------------------------------------------------------------------------------
 * Non-maximum suppression.
 * Replaces torchvision::nms (tv:ops/boxes.py:20-48 -> tv-csrc:ops/cuda/nms_kernel.cu:204,
 * semantics of the CPU kernel tv-csrc:ops/cpu/nms_kernel.cpp:116) and both batched_nms
 * strategies (tv:ops/boxes.py:86-120).
 *   mode 0  plain nms (groups ignored)
 *   mode 1  per-group NMS on raw coordinates ("vanilla"); groups[i] in [0, num_groups);
 *           rows with a negative group are ignored (padding of fixed-capacity inputs)
 *   mode 2  coordinate trick: boxes + fl(fl(group) * fl(max(boxes) + 1)), then plain nms
 * keep_out [num_boxes] receives original indices in descending-score order (ties: lower
 * index first). status_out[0] = number kept, or -1 if the mask workspace was too small, in
 * which case status_out[1] = mask words (8 bytes each) required; status_out has 4 int64.
 * ------------------------------------------------------------------------------------ */
#define MB_NMS_PLAIN 0
#define MB_NMS_VANILLA 1
#define MB_NMS_TRICK 2
size_t mb_nms_workspace_bytes(int64_t num_boxes, int32_t num_groups);
int mb_nms(const float* boxes, const float* scores, const int64_t* groups, int64_t num_boxes,
           int32_t num_groups, int32_t mode, double iou_threshold, int64_t* keep_out,
           int64_t* status_out, void* workspace, size_t workspace_bytes, void* mask_workspace,
           size_t mask_workspace_bytes, mb_stream_t stream);

/* ------------------------------------------------------------------------------------
 * RoIAlign.
 * mb_roi_align replaces torchvision::roi_align forward (tv:ops/roi_align.py:203-260 ->
 * tv-csrc:ops/cuda/roi_align_kernel.cu:470; arithmetic of the CPU kernel
 * tv-csrc:ops/cpu/roi_align_kernel.cpp:393): input NCHW fp32, rois [K,5] =
 * (batch, x1, y1, x2, y2), out [K, C, PH, PW].
 * mb_multiscale_roi_align replaces MultiScaleRoIAlign.forward's per-level loop
 * (tv:ops/poolers.py:147-227) in ONE launch: level assignment (LevelMapper, :73-84) is
 * evaluated on the device as area thresholds derived by the host from the mapper, every
 * output element is written exactly once. level_thresholds[i] = smallest fp32 box area
 * mapped to level > i (num_levels-1 entries, ascending).
 * exact != 0 reproduces the CPU kernel's operation order bit for bit (no FMA contraction).
 * ------------------------------------------------------------------------------------ */
typedef struct {
    int32_t num_levels;
    int32_t num_images;
    int32_t channels;
    int32_t pooled_h, pooled_w;
    int32_t sampling_ratio;
    int32_t aligned;
    int32_t exact;
    int32_t height[MB_MAX_LEVELS], width[MB_MAX_LEVELS];
    float spatial_scale[MB_MAX_LEVELS];
    float level_thresholds[MB_MAX_LEVELS];
    const float* features[MB_MAX_LEVELS]; /* device, NCHW contiguous */
    /* Alternative RoI layout (the fused RPN stage's output): boxes_per_image > 0 means `rois`
     * is [num_images, boxes_per_image, 4] and the batch index of row k is k / boxes_per_image;
     * box_counts (device, nullable) gives the live rows per image, rows beyond it produce zeros. */
    int32_t boxes_per_image;
    const int32_t* box_counts;
    /* != 0: every feature map is stored channels-last ([N, H, W, C] in memory — what a
     * torch.channels_last cuDNN backbone produces). The kernel then gathers 128-byte channel
     * vectors straight from global memory / L1 and needs no shared-memory staging. */
    int32_t channels_last;
    /* route for channels-last maps: 0 = library default (the register-gather kernel k_roi_align_nhwc4d; the TMA-staged
     * kernel if the environment variable MB_ROI_TMA=1), 1 = register-gather kernel, 2 = TMA-staged kernel
     * (k_roi_geom + k_roi_align_tma). Identical results. */
    int32_t force_gather;
} mb_roi_align_params;
/* Workspace: holds the per-RoI tap-table records of the TMA-staged kernel (channels-last maps, sampling_ratio 2,
 * aligned = 0) and, for NCHW maps whose RoIs cover the pyramid several times over, one channels-last copy of the
 * maps (transposed once per call). Without it the call still works and takes the register-gather kernels. */
size_t mb_roi_align_workspace_bytes(const mb_roi_align_params* params_host, int64_t num_rois);
int mb_multiscale_roi_align(const mb_roi_align_params* params_host, const float* rois, int64_t num_rois,
                            float* out, int32_t* levels_out /* nullable, [K] */, void* workspace,
                            size_t workspace_bytes, mb_stream_t stream);
/* Number of calls of this process that took the TMA-staged kernel (k_roi_geom + k_roi_align_tma); the others took
 * the gather kernels. Lets tests and the bench assert which route produced a result. */
int64_t mb_roi_align_tma_launches(void);

/* ------------------------------------------------------------------------------------
 * Element-wise box operators.
 *  mb_box_decode      BoxCoder.decode_single (tv:models/detection/_utils.py:183-224):
 *                     rel_codes [M, 4*C], boxes [M,4] -> out [M, C, 4]
 *  mb_clip_boxes      clip_boxes_to_image (tv:ops/boxes.py:149-182)
 *  mb_box_convert     box_convert for xyxy/xywh/cxcywh (tv:ops/boxes.py:185-270); fmt 0/1/2
 *  mb_remove_small    remove_small_boxes (tv:ops/boxes.py:123-146): ascending indices, count
 *  mb_resize_boxes    resize_boxes (tv:models/detection/transform.py:306-319)
 *  mb_grid_anchors    AnchorGenerator.grid_anchors for one level (tv:.../anchor_utils.py:84-113)
 * ------------------------------------------------------------------------------------ */
int mb_box_decode(const float* rel_codes, const float* boxes, int64_t num_boxes, int32_t num_classes,
                  float wx, float wy, float ww, float wh, float bbox_xform_clip, float* out,
                  mb_stream_t stream);
int mb_clip_boxes(const float* boxes, int64_t num_boxes, float height, float width, float* out,
                  mb_stream_t stream);
int mb_box_convert(const float* boxes, int64_t num_boxes, int32_t in_fmt, int32_t out_fmt, float* out,
                   mb_stream_t stream);
int mb_remove_small(const float* boxes, int64_t num_boxes, float min_size, int64_t* keep_out,
                    int64_t* count_out, mb_stream_t stream);
int mb_resize_boxes(const float* boxes, int64_t num_boxes, float ratio_h, float ratio_w, float* out,
                    mb_stream_t stream);
int mb_grid_anchors(const float* base_anchors_host, int32_t num_base, int32_t grid_h, int32_t grid_w,
                    int32_t stride_h, int32_t stride_w, float* out, mb_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Fused RPN post-head stage: anchors + per-level top-k + decode + clip + small-box and
 * score filter + per-level NMS + post-NMS top-n, straight from the head's NCHW outputs.
 * Replaces AnchorGenerator.forward, concat_box_prediction_layers, BoxCoder.decode and
 * RegionProposalNetwork.filter_proposals (tv:models/detection/anchor_utils.py:115-133,
 * rpn.py:81-110, _utils.py:162-224, rpn.py:231-297).
 * ------------------------------------------------------------------------------------ */
typedef struct {
    int32_t num_images, num_levels;
    int32_t feat_h[MB_MAX_LEVELS], feat_w[MB_MAX_LEVELS];
    int32_t stride_h[MB_MAX_LEVELS], stride_w[MB_MAX_LEVELS];
    int32_t anchors_per_loc[MB_MAX_LEVELS];
    float base_anchors[MB_MAX_LEVELS][MB_MAX_ANCHORS_PER_LOC][4];
    int32_t image_h[MB_MAX_IMAGES], image_w[MB_MAX_IMAGES]; /* images.image_sizes (pre-padding) */
    int32_t pre_nms_top_n, post_nms_top_n;
    double nms_thresh;
    float score_thresh, min_size;
    float wx, wy, ww, wh, bbox_xform_clip;
    int64_t trick_numel; /* batched_nms strategy rule (tv:ops/boxes.py:80): 4000 cpu, 100000 cuda, -1 vanilla */
    const float* objectness[MB_MAX_LEVELS]; /* [N, A, H, W] logits */
    const float* deltas[MB_MAX_LEVELS];     /* [N, 4A, H, W] */
} mb_rpn_params;
size_t mb_rpn_workspace_bytes(const mb_rpn_params* params_host);
/* proposals_out [N, post_nms_top_n, 4], scores_out [N, post_nms_top_n], counts_out [N] int32.
 * Optional debug outputs (nullable): topk_idx_out [N, sum_l min(pre, A_l)] int64 flattened
 * anchor indices in the reference's (level, h, w, a) order. */
int mb_rpn_proposals(const mb_rpn_params* params_host, float* proposals_out, float* scores_out,
                     int32_t* counts_out, int64_t* topk_idx_out, void* workspace,
                     size_t workspace_bytes, mb_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Fused detection post-processing: softmax + decode + clip + score/small filters + per-class
 * NMS + top detections_per_img + resize to the original image size.
 * Replaces RoIHeads.postprocess_detections (tv:models/detection/roi_heads.py:680-737) and
 * GeneralizedRCNNTransform.postprocess / resize_boxes (transform.py:257-277, :306-319).
 * ------------------------------------------------------------------------------------ */
typedef struct {
    int32_t num_images, num_classes; /* classes incl. background */
    int32_t max_props_per_image;     /* row capacity of proposals per image */
    int32_t detections_per_img;
    int32_t image_h[MB_MAX_IMAGES], image_w[MB_MAX_IMAGES]; /* resized (network) sizes */
    int32_t orig_h[MB_MAX_IMAGES], orig_w[MB_MAX_IMAGES];   /* original sizes; 0 -> no resize */
    double nms_thresh;
    float score_thresh, min_size;
    float wx, wy, ww, wh, bbox_xform_clip;
    int64_t trick_numel;
} mb_det_params;
size_t mb_det_workspace_bytes(const mb_det_params* params_host);
/* class_logits [sumR, C], box_regression [sumR, 4C], proposals [N, max_props, 4] with
 * prop_counts [N] live rows each; logits/regression rows are packed in image order
 * (row offset of image n = sum of earlier counts) when packed != 0, else strided by max_props.
 * Outputs: det_boxes [N, dpi, 4] (original image scale), det_boxes_net [N, dpi, 4] (network
 * scale, nullable), det_scores [N, dpi], det_labels [N, dpi] int64, det_counts [N] int32. */
int mb_det_postprocess(const mb_det_params* params_host, const float* class_logits,
                       const float* box_regression, const float* proposals, const int32_t* prop_counts,
                       int32_t packed, float* det_boxes, float* det_boxes_net, float* det_scores,
                       int64_t* det_labels, int32_t* det_counts, void* workspace, size_t workspace_bytes,
                       mb_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Score filter + crop extraction.
 * Replaces miso's `scores > threshold` filter and xyxy->xywh annotation
 * (ref:miso/object_detection/inference.py:53-64), RectangleAnnotation.coords_int
 * (ref:miso/object_detection/dataset/annotation.py:120-127) and the crop slice
 * (ref:miso/object_detection/crop.py:28-30).
 * mb_crop_plan: per image n, detections [N, cap, 4]/[N, cap] with det_counts[n] live rows;
 *   writes, for every detection passing the filter (original order), rects [N*cap, 4] int32 =
 *   (x_begin, y_begin, width, height) after numpy slice resolution, xywh [N*cap, 4] fp32,
 *   src index [N*cap] int32 (n*cap + i), byte offsets [N*cap+1] int64 into the packed crop
 *   buffer, and totals[0] = number of crops, totals[1] = total bytes.
 * mb_crop_gather: copies the pixels. images: one uint8 HWC device pointer per image. If
 *   totals[1] exceeds crops_capacity_bytes nothing is copied and totals[2] is set to 1.
 * ------------------------------------------------------------------------------------ */
typedef struct {
    int32_t num_images, capacity, channels;
    int32_t image_h[MB_MAX_IMAGES], image_w[MB_MAX_IMAGES];
    const uint8_t* images[MB_MAX_IMAGES]; /* device, HWC uint8, row pitch = w*channels */
    float threshold;
    int32_t boxes_are_xywh; /* != 0: det_boxes rows already are annotation bounds (x, y, w, h) */
} mb_crop_params;
int mb_crop_plan(const mb_crop_params* params_host, const float* det_boxes, const float* det_scores,
                 const int32_t* det_counts, int32_t* rects_out, float* xywh_out, int32_t* src_out,
                 int64_t* offsets_out, int64_t* totals_out, mb_stream_t stream);
int mb_crop_gather(const mb_crop_params* params_host, const int32_t* rects, const int32_t* src,
                   const int64_t* offsets, int64_t* totals, uint8_t* crops_out,
                   int64_t crops_capacity_bytes, mb_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Tiled-mosaic exchange, element-wise ends (SURVEY.md section 8e; the reference never tiles, so
 * there is no reference line to cite; the score filter is miso's
 * ref:miso/object_detection/inference.py:53 `scores > threshold`).
 * mb_mosaic_pack: detections of this rank's tiles ([tiles, dpi, 4] boxes in tile coordinates,
 *   [tiles, dpi] scores and int64 labels, det_counts[tiles] live rows, origins_yx [tiles, 2] fp32
 *   tile origins) -> block_out [rows, 6] = (x1, y1, x2, y2, score, label) in mosaic coordinates,
 *   label -1 for dead / filtered / padding rows (rows >= tiles*dpi).
 * mb_mosaic_unpack: gathered blocks [rows, 6] -> boxes [rows, 4], scores [rows], labels [rows]
 *   int64 — the inputs of mb_nms mode 1, which ignores negative labels.
 * ------------------------------------------------------------------------------------ */
int mb_mosaic_pack(const float* det_boxes, const float* det_scores, const int64_t* det_labels,
                   const int32_t* det_counts, const float* origins_yx, int32_t tiles, int32_t dpi,
                   float threshold, int64_t rows, float* block_out, mb_stream_t stream);
int mb_mosaic_unpack(const float* block, int64_t rows, float* boxes_out, float* scores_out,
                     int64_t* labels_out, mb_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Sparse seam NMS (SURVEY.md section 8e): the same result as mb_nms mode 1 (torchvision's
 * _batched_nms_vanilla, tv:ops/boxes.py:106-120, CPU kernel arithmetic) over all rows of a gathered block
 * [rows, 6] = (x1, y1, x2, y2, score, label; label < 0 = ignore), computed on the sparse "may suppress" graph:
 * rows come in groups of rows_per_tile consecutive rows (one tile's detections) and only rows of tiles whose
 * bounding boxes intersect are compared. iou_threshold must be >= 0 (MB_ERR_UNSUPPORTED otherwise: with a
 * negative threshold disjoint boxes suppress each other — use mb_nms). rows_per_tile <= 1024.
 * state_out [rows] int32: 1 kept, 2 suppressed, 3 ignored row. keep_out (nullable) [rows] int64: kept row
 * indices ascending. status_out [4] int64: [0] = number kept (0 if keep_out is null) or -1 if edge_capacity was
 * too small, [1] = suppression edges found (the capacity to retry with).
 * mb_seam_select: rows [row_lo, row_lo+num_rows) -> boxes [num_rows, 4], scores [num_rows] with -inf for rows
 * that were not kept: the inputs of mb_crop_plan (one image, capacity num_rows) for a rank's own tiles.
 * ------------------------------------------------------------------------------------ */
size_t mb_seam_nms_workspace_bytes(int64_t rows, int32_t rows_per_tile, int64_t edge_capacity);
int mb_seam_nms(const float* block, int64_t rows, int32_t rows_per_tile, double iou_threshold,
                int64_t edge_capacity, int32_t* state_out, int64_t* keep_out, int64_t* status_out,
                void* workspace, size_t workspace_bytes, mb_stream_t stream);
int mb_seam_select(const float* block, const int32_t* state, int64_t row_lo, int64_t num_rows,
                   float* boxes_out, float* scores_out, mb_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Training-side siblings (SURVEY.md section 8f row 4; reached from ref:miso/object_detection/engine/engine.py:33
 * `model(images, targets)`).
 *  mb_box_iou       torchvision.ops.box_iou (tv:ops/boxes.py:299-330): boxes1 [n1,4], boxes2 [n2,4] -> [n1,n2].
 *  mb_match_encode  assign_targets_to_anchors / assign_targets_to_proposals fused (tv:models/detection/rpn.py:193-229,
 *                   roi_heads.py:580-614): Matcher (_utils.py:345-426) on box_iou(gt, anchors) without materialising
 *                   the [M,N] matrix + BoxCoder.encode_single (_utils.py:85-127) of gt[matches.clamp(min=0)].
 *                   matches_out [N] int64 (gt index, -1 below low, -2 between), matched_vals_out [N] (nullable),
 *                   targets_out [N,4] (nullable). num_gt >= 1 (the reference handles empty targets in Python).
 *  mb_roi_align_backward  torchvision::_roi_align_backward (tv-csrc:ops/cuda/roi_align_kernel.cu): grad [K,C,PH,PW],
 *                   rois [K,5] -> grad_input [batch,C,H,W] (NCHW, zero-filled by the call, then atomically accumulated).
 * ------------------------------------------------------------------------------------ */
int mb_box_iou(const float* boxes1, int64_t n1, const float* boxes2, int64_t n2, float* iou_out, mb_stream_t stream);
size_t mb_match_encode_workspace_bytes(int64_t num_gt, int64_t num_anchors);
int mb_match_encode(const float* gt_boxes, int64_t num_gt, const float* anchors, int64_t num_anchors,
                    float high_threshold, float low_threshold, int32_t allow_low_quality_matches, float wx, float wy,
                    float ww, float wh, int64_t* matches_out, float* matched_vals_out, float* targets_out,
                    void* workspace, size_t workspace_bytes, mb_stream_t stream);
int mb_roi_align_backward(const float* grad, const float* rois, int64_t num_rois, float spatial_scale, int32_t channels,
                          int32_t height, int32_t width, int32_t pooled_h, int32_t pooled_w, int32_t sampling_ratio,
                          int32_t aligned, int32_t batch_size, float* grad_input, mb_stream_t stream);

/* ------------------------------------------------------------------------------------
 * paste_masks_in_image (tv:models/detection/roi_heads.py:375-501, called from
 * GeneralizedRCNNTransform.postprocess tv:models/detection/transform.py:269-272).
 * masks [R, 1, M, M] fp32 mask probabilities, boxes [R, 4] fp32 xyxy in image coordinates ->
 * out [R, 1, im_h, im_w] fp32 (every element written). M + 2*padding <= 64, R <= 65535.
 * ------------------------------------------------------------------------------------ */
int mb_paste_masks(const float* masks, const float* boxes, int64_t num_masks, int32_t mask_side,
                   int32_t padding, int32_t im_h, int32_t im_w, float* out, mb_stream_t stream);
/* Per-crop instance masks: paste_masks_in_image (tv:models/detection/roi_heads.py:375-501) evaluated only
 * at the pixels of the crop rectangles of mb_crop_plan, thresholded. Crop j of slot s = src[j] with
 * rect (x, y, w, h): mask_j[r, c] = 255 if paste(mask_probs[s], paste_boxes[s], frame (fh, fw))
 * [y + r - y0, x + c - x0] > mask_threshold (fp32, strict) else 0, and 0 outside the frame.
 * The frame of slot s is frames[s / rows_per_frame] = (x0, y0, fw, fh) in rect coordinates
 * (ceil(num_images*capacity / rows_per_frame) rows); frames NULL: frame f is image f at (0, 0), which
 * needs rows_per_frame >= capacity. paste_boxes are xyxy in frame coordinates, mask_probs
 * [num_images*capacity, M, M] by slot. masks_out receives h*w bytes per crop, packed in crop order at
 * offsets[j] / channels (mb_crop_gather need not run). If totals[1] / channels exceeds
 * masks_capacity_bytes nothing is written and totals[3] is set to 1, else totals[3] = 0.
 * M + 2*padding <= 64. */
int mb_crop_masks(const mb_crop_params* params_host, const float* mask_probs, const float* paste_boxes,
                  int32_t mask_side, int32_t padding, const int32_t* frames, int32_t rows_per_frame,
                  float mask_threshold, const int32_t* rects, const int32_t* src, const int64_t* offsets,
                  int64_t* totals, uint8_t* masks_out, int64_t masks_capacity_bytes, mb_stream_t stream);
/* Per-crop region measurements from the masks of mb_crop_masks (skimage.measure.regionprops of (mask > 0) with
 * one label). The region of crop j is the set of non-zero bytes of its h*w mask at masks + offsets[j] / channels;
 * (r, c) are crop-local row / column, rect (x, y, w, h). Exact int64 sums over the set pixels: A = sum 1,
 * S_r, S_c, S_rr, S_cc, S_rc (sums of r, c, r*r, c*c, r*c), P_k = sum of pixel byte k, read from
 * params.images[src[j] / capacity] at the rect (the pixel gather need not have run). out receives
 * MB_MORPH_FIELDS fp64 per crop, at row j of [num_images*capacity, MB_MORPH_FIELDS], all 0 when A = 0:
 *   0 area = A
 *   1 perimeter (4-neighbourhood): E = mask with every pixel cleared that has a 4-neighbour outside it,
 *     B = mask and not E; per p in B, code = 1 + 2 * (4-neighbours in B) + 10 * (diagonal neighbours in B);
 *     n1 = #codes in {5,7,15,17,25,27}, n2 = #{21,33}, n3 = #{13,23};
 *     perimeter = (n1 + sqrt2 * n2) + ((1 + sqrt2) / 2) * n3
 *   2, 3 centroid_x = x + S_c / A, centroid_y = y + S_r / A
 *   4, 5 major / minor_axis_length = 4 sqrt(l1), 4 sqrt(l2) with a = u_cc, b = -u_rc, c = u_rr,
 *     u_rr = (A S_rr - S_r^2) / (A * A) (numerator exact in 128 bits, converted once; A * A in fp64), likewise
 *     u_cc, u_rc = (A S_rc - S_r S_c) / (A * A); l1,2 = ((a + c) +- sqrt((a - c)^2 + 4 (b * b))) / 2, clipped at 0
 *   6 orientation = a == c ? (b < 0 ? -pi/4 : pi/4) : atan2(-2 b, c - a) / 2
 *   7 eccentricity = l1 == 0 ? 0 : sqrt(1 - l2 / l1)
 *   8 equivalent_diameter = sqrt(4 A / pi)
 *   9..12 mean_intensity_k = P_k / A for k < channels, else 0
 * The count is totals[0] (device); if totals[3] (mask overflow) is set nothing is written. workspace: at least
 * mb_mask_morphology_workspace_bytes(params) = 128 * num_images * capacity bytes (zeroed by the call).
 * MB_ERR_UNSUPPORTED for channels > 4 or an image side > 32768 (which keeps every int64 sum exact). */
#define MB_MORPH_FIELDS 13
size_t mb_mask_morphology_workspace_bytes(const mb_crop_params* params_host);
int mb_mask_morphology(const mb_crop_params* params_host, const uint8_t* masks, const int32_t* rects,
                       const int32_t* src, const int64_t* offsets, const int64_t* totals, void* workspace,
                       size_t workspace_bytes, double* out, mb_stream_t stream);
/* Lossless PNG files of the packed crops (mb_crop_gather, channels == params.channels) or masks (mb_crop_masks,
 * channels == 1): one complete stream per crop, packed in crop order at png_offsets_out[j]
 * ([num_images*capacity + 1] int64; crop j is png_offsets_out[j + 1] - png_offsets_out[j] bytes, 0 when h*w == 0).
 * Crop j (rect (x, y, w, h)) is read at packed + offsets[j] / params.channels * channels, h*w*channels bytes.
 * The bytes depend only on the crop's pixels, h, w and channels:
 *   framing  PNG signature, IHDR (w, h, bit depth 8, colour type 0 / 4 / 2 / 6 for 1 / 2 / 3 / 4 channels, no
 *            interlace), one IDAT, IEND; no other chunks
 *   filter   per row, the type 0..4 with the least sum over the row of |(int8) filtered byte| (ties: lower type);
 *            row -1 is zeros
 *   zlib     header 78 01; the filtered bytes (h * (1 + w*channels)) cut every 32768 bytes into blocks coded
 *            independently; each block is non-final and followed by an empty stored block; the stream ends with an
 *            empty final fixed-Huffman block (03 00) and the Adler-32 of the filtered bytes
 *   tokens   per maximal run of n equal bytes inside a block: a literal, then the n - 1 repeats as length-258
 *            matches at distance 1, then the m = (n - 1) % 258 left: one match of length m if m >= 3, else m literals
 *   codes    dynamic per block: lengths by package-merge (limit 15; 7 for the code-length code) over the used symbols
 *            sorted by (frequency, index), leaves before packages of equal weight; fewer than two used symbols: the
 *            lowest unused indices get length 1 too (the distance code is always [1, 1]); HLIT = last used literal /
 *            length symbol + 1, HDIST = 2; the code lengths run-length coded per tree by zlib's scan_tree / send_tree
 *   stored   a block whose dynamic form plus its empty stored block is not shorter than L + 10 bytes (the block
 *            stored, plus the empty stored block) is stored
 * mb_png_bound_bytes: a capacity no packed set of `crops` crops of packed_bytes bytes (h*w*channels summed) can
 *   exceed: 75 * crops + F + 10 * (F / 32768) with F = packed_bytes + ceil(packed_bytes / channels); -1 for bad input.
 * mb_png_workspace_bytes: for packed crops of up to packed_capacity_bytes (h*w*channels summed); 0 for bad input.
 * png_status_out [2] int64: [0] total bytes, [1] 1 if that exceeds png_capacity_bytes (nothing is written), 2 if the
 * workspace is too small for the crops (nothing is encoded), else 0. A pixel or mask overflow flag in totals (totals[2],
 * totals[3]) means nothing is encoded (no crops). Channels outside 1..4: MB_ERR_UNSUPPORTED. */
int64_t mb_png_bound_bytes(int64_t packed_bytes, int64_t crops, int32_t channels);
size_t mb_png_workspace_bytes(const mb_crop_params* params_host, int64_t packed_capacity_bytes, int32_t channels);
int mb_png_encode(const mb_crop_params* params_host, const uint8_t* packed, int32_t channels, const int32_t* rects,
                  const int64_t* offsets, const int64_t* totals, void* workspace, size_t workspace_bytes,
                  uint8_t* png_out, int64_t png_capacity_bytes, int64_t* png_offsets_out, int64_t* png_status_out,
                  mb_stream_t stream);
/* Baseline JPEG files of the packed crops (mb_crop_gather), channels 1 (mode L) or 3 (RGB): one complete file per crop,
 * packed in crop order at jpeg_offsets_out[j] ([num_images*capacity + 1] int64; 0 bytes when h*w == 0). Crop j (rect
 * (x, y, w, h)) is read at packed + offsets[j] / params.channels * channels. The file is byte for byte what
 * PIL.Image.fromarray(crop).save(f, "JPEG") writes with default arguments (libjpeg-turbo):
 *   framing  SOI; APP0 JFIF 1.1, no units, density 1:1, no thumbnail; DQT luminance (and chrominance for 3 channels);
 *            SOF0 (8 bit, h, w; components 1, 2, 3 with sampling 0x22, 0x11, 0x11 and tables 0, 1, 1, or one
 *            component 0x11); DHT DC0, AC0 (and DC1, AC1), the Annex K tables; SOS over 0..63; the scan; EOI. No
 *            other markers, no restart intervals. Headers are 328 (grey) and 623 (colour) bytes.
 *   quant    Annex K tables at quality 75: q = clamp((std * 50 + 50) / 100, 1, 255), written in zigzag order
 *   colour   jccolor.c with FIX(x) = (int)(x * 65536 + 0.5): Y = (FIX(.299) r + FIX(.587) g + FIX(.114) b + 2^15) >> 16,
 *            Cb = (-FIX(.16874) r - FIX(.33126) g + FIX(.5) b + (128 << 16) + 2^15 - 1) >> 16,
 *            Cr = (FIX(.5) r - FIX(.41869) g - FIX(.08131) b + (128 << 16) + 2^15 - 1) >> 16
 *   edges    luma padded to 8 ceil(w/8) x 8 ceil(h/8) by replicating the last column and row; chroma: the full-resolution
 *            plane padded by replication to 2 ceil(h/2) rows and 16 ceil(ceil(w/2)/8) columns, downsampled 2x2 as
 *            (sum of 4 + bias) >> 2 with bias 1, 2, 1, 2, ... along each output row, then the downsampled rows padded
 *            by replication to a whole block row
 *   DCT      jfdctint.c islow on samples - 128: rows (PASS1_BITS 2), then columns; CONST_BITS 13,
 *            DESCALE(x, n) = (x + 2^(n-1)) >> n; quantised as (|c| + 4q) / 8q with the sign of c
 *   scan     MCU 16x16 (Y0 Y1 Y2 Y3 Cb Cr) or one 8x8 block; a DC predictor per component from 0; blocks of an MCU past
 *            the component's last real block column or row are dummy blocks (zero AC, the DC of the block before
 *            them in the MCU); Huffman codes with ZRL and EOB, negative amplitudes v + 2^n - 1, 0x00 after every 0xFF
 *            data byte, the last byte padded with 1-bits
 * mb_jpeg_bound_bytes: a capacity no packed set of `crops` crops of packed_bytes bytes can exceed: every block at
 *   1660 bits (DC <= 11 + 11, each AC <= 16 + 10) and every data byte stuffed, on crops 1 pixel wide, which have the
 *   most blocks per pixel: crops * (H + 2) + 416 * B with H the header bytes and, for P = packed_bytes / channels
 *   pixels, B = P / 8 + crops (grey) or 6 * (P / 16 + crops) (colour); -1 for bad input.
 * mb_jpeg_workspace_bytes: enough for any packed crops of up to packed_capacity_bytes: 16 B of record per block plus
 *   its unstuffed codes (at most 208 B), B blocks as above, plus 40 B per slot. The codes take their exact size, so
 *   less suffices for real content (large photographic crops need about 0.5 B per pixel: 16 B per 64 or 43 pixels
 *   plus the file size); a workspace too small for the crops at hand sets flag 2.
 * jpeg_status_out [2] int64: [0] total bytes, [1] 1 if that exceeds jpeg_capacity_bytes (nothing is written), 2 if the
 * workspace is too small for the crops (nothing is encoded), else 0. A pixel overflow flag in totals (totals[2]) means
 * nothing is encoded (no crops). Channels other than 1 or 3, or an image side above 65535: MB_ERR_UNSUPPORTED. */
int64_t mb_jpeg_bound_bytes(int64_t packed_bytes, int64_t crops, int32_t channels);
size_t mb_jpeg_workspace_bytes(const mb_crop_params* params_host, int64_t packed_capacity_bytes, int32_t channels);
int mb_jpeg_encode(const mb_crop_params* params_host, const uint8_t* packed, int32_t channels, const int32_t* rects,
                   const int64_t* offsets, const int64_t* totals, void* workspace, size_t workspace_bytes,
                   uint8_t* jpeg_out, int64_t jpeg_capacity_bytes, int64_t* jpeg_offsets_out, int64_t* jpeg_status_out,
                   mb_stream_t stream);
/* maskrcnn_inference (tv:models/detection/roi_heads.py:56-82): mask_logits [R, C, M, M], labels [R] int64 ->
 * out [R, 1, M, M] = sigmoid(mask_logits[r, labels[r]]). Labels outside [0, C) are the caller's error. */
int mb_mask_prob(const float* mask_logits, const int64_t* labels, int64_t num_masks, int32_t num_classes,
                 int32_t mask_side, float* out, mb_stream_t stream);

/* ------------------------------------------------------------------------------------
 * Input transform: ToTensor (ref:miso/object_detection/inference.py:117) +
 * GeneralizedRCNNTransform.normalize / resize / batch_images
 * (tv:models/detection/transform.py:165-173, 175-201 with _resize_image_and_masks :23-70, 231-255)
 * for uint8 HWC images on the device. The caller computes the resized sizes out_h/out_w like the
 * reference (fp32 scale factor, floor) and the padded batch size; out is [N, channels, pad_h, pad_w]
 * fp32, every element written (zeros outside each image's out_h x out_w).
 * ------------------------------------------------------------------------------------ */
typedef struct {
    int32_t num_images, channels;           /* channels <= 4 */
    const uint8_t* images[MB_MAX_IMAGES];   /* device, HWC uint8, dense */
    int32_t in_h[MB_MAX_IMAGES], in_w[MB_MAX_IMAGES], out_h[MB_MAX_IMAGES], out_w[MB_MAX_IMAGES];
    float mean[4], std[4];
    int32_t pad_h, pad_w;
} mb_transform_params;
int mb_image_transform(const mb_transform_params* params_host, float* out, mb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* MISOB200_H */
