// api.cu — version / build identification of libmisob200.so.
#include "common.cuh"

extern "C" int mb_abi_version(void) { return MB_ABI_VERSION; }

extern "C" const char* mb_build_info(void) {
    return "libmisob200 sm_100a cuda " __DATE__
           ";kernels="
           "k_box_convert,k_box_decode,k_box_iou,k_box_max,k_clip_boxes,k_crop_gather,k_crop_masks,k_crop_plan,"
           "k_crop_plan_chunks,k_det_candidates,k_det_finalize,k_det_init,k_emit_single,k_emit_sorted,"
           "k_grid_anchors,k_group_hist,k_image_transform,k_kept_bucket,k_mask_prob,k_match_best,k_match_finish,"
           "k_mosaic_pack,k_mosaic_unpack,k_nchw_to_nhwc,k_nms_fixpoint,k_nms_mask,k_nms_sweep,k_nms_sweep_small,"
           "k_nms_sweep_wide,k_paste_masks,k_rank_in_segment,k_remove_small,k_resize_boxes,k_roi_align_backward,"
           "k_roi_align_direct,k_roi_align_nhwc,k_roi_align_nhwc4d,k_roi_align_sr2,k_roi_align_staged,"
           "k_roi_align_tma,k_roi_geom,k_rpn_decode,k_rpn_finalize,k_rpn_hist,k_rpn_select,k_scatter_boxes,"
           "k_seam_emit,k_seam_finish,k_seam_pairs,k_seam_prep,k_seam_resolve,k_seam_select,k_seg_meta,"
           "k_single_segment";
}
