/*
 * b200det.h -- C-ABI of libb200det.so: B200 (sm_100a) kernels for the detection
 * post-backbone hot path of pengfeidip/pytorch-faster-rcnn.
 *
 * The reference has no FFI: the path sits behind plain Python call sites and the
 * lib.builder.MODULES registry (SURVEY 8(b)).  Each entry point below therefore
 * cites the reference *Python* function it replaces (file:line under the
 * reference root); INTEGRATION.md shows the ctypes binding a maintainer adds.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer unless the name ends in _host;
 *  - boxes are column-major [4, n] fp32 (row 0 = x1, 1 = y1, 2 = x2, 3 = y2), the
 *    reference layout (lib/utils.py:52); "ld" is the row pitch in elements;
 *  - batched entry points are image-major: tensor[b] starts at b * (rows * ld);
 *  - `stream` is a cudaStream_t passed as void*;
 *  - return 0 on success, B2D_ERR_ARG (-1) for argument errors, else a positive
 *    cudaError_t; b2d_last_error_string() describes the last failure;
 *  - no entry point allocates, synchronises or throws; scratch memory is passed
 *    in by the caller (sizes from the b2d_*_workspace_bytes queries).
 */
#ifndef B200DET_H_
#define B200DET_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define B2D_API __attribute__((visibility("default")))
#else
#define B2D_API
#endif

#define B2D_OK 0
#define B2D_ERR_ARG (-1)
#define B2D_MAX_LEVELS 8
#define B2D_MAX_ANCHORS 16

/* One pyramid level of an anchor head (lib/heads/anchor_head.py:33-36,66-67). */
typedef struct b2d_level {
    int H, W, A;        /* grid size, anchors per cell */
    int center_lt;      /* lib/anchor.py:82 */
    float stride;       /* == base size */
    float ws[B2D_MAX_ANCHORS], hs[B2D_MAX_ANCHORS]; /* lib/anchor.py:92-99, fp32 */
    long long offset;   /* first flattened anchor of this level (level-major concat) */
} b2d_level;

typedef struct b2d_pyramid {
    int num_levels;
    int _pad;
    long long total;    /* anchors per image over all levels */
    b2d_level lv[B2D_MAX_LEVELS];
} b2d_pyramid;

B2D_API const char* b2d_last_error_string(void);
B2D_API int b2d_version(void);
/* re-read the B2D_* development knobs from the environment (they are otherwise read once, at first use) */
B2D_API void b2d_reload_knobs(void);

/* ---- K1: AnchorCreator.__call__ (lib/anchor.py:107-129) -> out [4, A, H, W] */
B2D_API int b2d_anchor_grid(float* out, const float* ws, const float* hs, int A, int H, int W, float stride,
                    int center_lt, void* stream);
/* inside_anchor_mask (lib/region.py:19-29); anchors [4,n] -> mask u8[n]; border<0 => all 1 */
B2D_API int b2d_inside_anchor_mask(uint8_t* mask, const float* anchors, long long n, float img_h, float img_w,
                           float border, void* stream);
/* inside_grid_mask (lib/region.py:10-16) -> flags fp32 [A,H,W]; in_h/in_w computed by the host */
B2D_API int b2d_inside_grid_mask(float* flags, int A, int H, int W, int in_h, int in_w, void* stream);

/* ---- a3: calc_iou / elem_iou (lib/utils.py:151-182) */
B2D_API int b2d_calc_iou(float* out /*[N,K]*/, const float* a /*[4,N]*/, long long N, const float* b /*[4,K]*/,
                 long long K, void* stream);
B2D_API int b2d_elem_iou(float* out /*[N]*/, const float* a, const float* b, long long N, void* stream);

/* ---- K2: MaxIoUAssigner.__call__ (lib/region.py:75-107), batched over B images.
 * Box source: explicit `boxes` [B][4][box_ld] with optional per-image counts, or
 * (boxes == NULL) the anchors of `pyr` generated in registers and masked by
 * inside_anchor_mask & inside_grid_mask against img_hw[b] = (img_h, img_w)
 * (lib/heads/anchor_head.py:92-100); masked-out anchors get label -1, iou 0.
 * gt [B][4][gt_ld], gt_count int32[B] (every count must be >= 1).
 * prepend_gt != 0 reproduces lib/bbox.py:27-29: outputs get gt_count[b] leading
 * rows (labels 1..K, iou 1) and the boxes follow; out_ld is the row pitch of
 * labels/max_iou.  census int32[B][4] = {#pos, #neg, #pos appended, 0}; pos_list
 * int32[B][pos_cap] receives the indices (into the output row) of positives in
 * unspecified order (may be NULL).  workspace: B * gt_ld * 4 bytes. */
B2D_API int b2d_assign_max_iou(int64_t* labels, float* max_iou, long long out_ld, const float* boxes,
                       long long box_ld, const int* box_count, long long N, const b2d_pyramid* pyr_host,
                       const float* img_hw, float border, const float* gt, int gt_ld, const int* gt_count,
                       int B, float pos_iou, float neg_iou, float min_pos_iou, int prepend_gt, int* census,
                       int* pos_list, int pos_cap, void* workspace, size_t ws_bytes, void* stream);

/* ---- a5: device-RNG sampler (RandomSampler semantics, lib/region.py:43-57,112-126;
 * the RNG stream is this library's own, see DESIGN.md "Samplers").  One image per
 * block.  chosen int32[B][max_num] ascending (padded with -1), n_chosen int32[B].
 * labels int64[B][ld]; count int32[B] (NULL => n for all); census/pos_list from
 * b2d_assign_max_iou or b2d_label_census. */
B2D_API int b2d_sample_labels(int* chosen, int* n_chosen, const int64_t* labels, long long ld, const int* count,
                      const int* count_add /* optional int32[B] added to count */, long long n, const int* census, const int* pos_list, int pos_cap, int B, int max_num,
                      int pos_num, unsigned long long seed, const unsigned long long* seed_step /* optional device counter added to seed */, void* stream);
/* *cell += inc on the stream: the per-step counter of the device-RNG samplers lives in device memory, so that a step
 * captured in a CUDA graph draws a fresh random stream on every replay (a by-value seed is frozen by the capture) */
B2D_API int b2d_counter_add(unsigned long long* cell, unsigned long long inc, void* stream);
/* census + positive list of an arbitrary labels vector (for the sampler classes) */
B2D_API int b2d_label_census(int* census, int* pos_list, int pos_cap, const int64_t* labels, long long ld,
                     const int* count, long long n, int B, void* stream);
/* out[b][i] = -1 everywhere except out[b][chosen] = labels[b][chosen] (lib/region.py:120-126) */
B2D_API int b2d_scatter_sampled(int64_t* out, const int64_t* labels, long long ld, long long n, const int* chosen,
                        const int* n_chosen, int max_num, int B, void* stream);

/* ---- K8: bbox2param (lib/utils.py:47-70) / param2bbox (:83-92) elementwise, [4,n] */
B2D_API int b2d_bbox2param(float* out, const float* base, const float* bbox, long long n, const float* means_host,
                   const float* stds_host, void* stream);
B2D_API int b2d_param2bbox(float* out, const float* base, const float* param, long long n, const float* means_host,
                   const float* stds_host, int clamp, float img_h, float img_w, void* stream);
B2D_API int b2d_clamp_bbox(float* out, const float* bbox, long long n, float img_h, float img_w, void* stream);

/* ---- fused target gather + encode for the sampled rows (lib/anchor.py:44-73,
 * lib/bbox.py:55-77).  Candidate i of image b is: GT i (if prepend_gt and i < K),
 * else box (i - K) taken from `boxes` or generated from `pyr`.  Outputs are
 * [B][4][max_num] / [B][max_num] with n_chosen[b] valid columns. */
B2D_API int b2d_encode_targets(float* tar_box, float* tar_gt, float* tar_param, int64_t* tar_label, int64_t* tar_is_gt,
                       const int* chosen, const int* n_chosen, int max_num, const int64_t* labels,
                       long long label_ld, const float* boxes, long long box_ld, const b2d_pyramid* pyr_host,
                       const float* gt, int gt_ld, const int* gt_count, const int64_t* gt_label,
                       int prepend_gt, const float* means_host, const float* stds_host, int B, void* stream);

/* ---- a13 in ONE launch: bbox_target (lib/bbox.py:6-82) for explicit boxes (N <= 4096,
 * gt_ld <= 512, max_num <= 1024): b2d_assign_max_iou + b2d_sample_labels +
 * b2d_encode_targets with identical outputs (same sampler specification and seed
 * convention), one CTA per image.  Arguments as in those three entry points. */
B2D_API int b2d_roi_targets_fused(int64_t* labels, float* max_iou, long long out_ld, const float* boxes, long long box_ld,
                          const int* box_count, long long N, const float* gt, int gt_ld, const int* gt_count,
                          const int64_t* gt_label, int B, float pos_iou, float neg_iou, float min_pos_iou,
                          int prepend_gt, int* census, int* pos_list, int pos_cap, int* chosen, int* n_chosen,
                          int max_num, int pos_num, unsigned long long seed, const unsigned long long* seed_step,
                          float* tar_box, float* tar_gt, float* tar_param, int64_t* tar_label, int64_t* tar_is_gt,
                          const float* means_host, const float* stds_host, void* stream);

/* gather of the head outputs at the sampled anchors (lib/anchor.py:49-56), batched:
 * cls_ptrs_host[l] -> [B, C, n_l], reg_ptrs_host[l] -> [B, 4, n_l] (the views of
 * lib/heads/anchor_head.py:82-83) -> tar_cls [B][C][max_num], tar_reg [B][4][max_num]. */
B2D_API int b2d_gather_head_outputs(float* tar_cls, float* tar_reg, const void* const* cls_ptrs_host,
                            const void* const* reg_ptrs_host, const b2d_pyramid* pyr_host, int cls_channels,
                            const int* chosen, const int* n_chosen, int max_num, int B, void* stream);

/* ---- K3: fused RPN proposal selection, all images and levels per launch
 * (RPNHead.predict_single_image, lib/heads/rpn_head.py:68-120; AnchorHead
 * .predict_single_image top-k part, lib/heads/anchor_head.py:224-248).
 * cls_ptrs_host[l] -> [B, A*C, H, W] logits, reg_ptrs_host[l] -> [B, 4A, H, W]
 * (channel = coord*A + a, lib/heads/anchor_head.py:82-83).  score_mode: 0 = one
 * sigmoid channel, 1 = two-channel softmax (score = p[1]), 2 = max over C sigmoid
 * channels (selection on the best class logit), 3 = max over the foreground classes
 * c >= 1 of a C-channel softmax (AnchorHead with use_sigmoid = False).  Outputs: props [B][4][max_num], scores [B][max_num], count int32[B]
 * (plus, if non-NULL, prov int32[B][max_num] = flattened anchor index). */
typedef struct b2d_rpn_cfg {
    int pre_nms, post_nms, max_num; /* <= 0 means "no limit" like the reference */
    int score_mode, num_cls_channels;
    float nms_thr_f;                /* largest fp32 <= the python-double threshold */
    float min_size;                 /* scale_factor * min_bbox_size */
    float means[4], stds[4];
    int do_nms;                     /* 0: stop after decode (AnchorHead path) */
    float* records;                 /* optional DEVICE buffer [B][max_num][5]: (x1, y1, x2, y2, score) per proposal, zero rows past
                                       count -- the packed record that is all-gathered over NCCL (SURVEY 8(e)); NULL = not written */
    void* event_after_select;       /* optional cudaEvent_t recorded on `stream` once the selection stage (K3) has been issued:
                                       lets a caller start independent work (the RPN-target kernels) behind K3 instead of
                                       beside it; NULL = none */
} b2d_rpn_cfg;

/* The arguments of b2d_roi_targets_fused (below) as one struct, for b2d_rpn_proposals_targets. */
typedef struct b2d_roi_target_args {
    int64_t* labels; float* max_iou; long long out_ld;          /* [B][out_ld] assignment of GT rows + proposals */
    const float* gt; int gt_ld; const int* gt_count; const int64_t* gt_label;
    float pos_iou, neg_iou, min_pos_iou; int prepend_gt;
    int* census; int* pos_list; int pos_cap;
    int* chosen; int* n_chosen; int max_num, pos_num;
    unsigned long long seed; const unsigned long long* seed_step;
    float* tar_box; float* tar_gt; float* tar_param; int64_t* tar_label; int64_t* tar_is_gt;
    float means[4], stds[4];
} b2d_roi_target_args;

B2D_API size_t b2d_rpn_proposals_workspace_bytes(const b2d_pyramid* pyr_host, int B, const b2d_rpn_cfg* cfg_host);
/* development aid: byte offset inside the workspace of the globaltimer stamps written when B2D_DBG=10
 * (u64 [B][64 CTAs][16 stamps]) */
/* kernels + memset nodes the last b2d_rpn_proposals call of this thread issued (bench.py gpu_launches) */
B2D_API int b2d_last_launch_count(void);
B2D_API size_t b2d_rpn_proposals_debug_offset(const b2d_pyramid* pyr_host, int B, const b2d_rpn_cfg* cfg_host);
B2D_API int b2d_rpn_proposals(float* props, float* scores, int* count, int* prov, const void* const* cls_ptrs_host,
                      const void* const* reg_ptrs_host, const b2d_pyramid* pyr_host, const float* img_hw,
                      int B, const b2d_rpn_cfg* cfg_host, void* workspace, size_t ws_bytes, void* stream);

/* b2d_rpn_proposals followed by bbox_target on its own output (lib/detectors/cascade_rcnn.py:111-126:
 * predict_bboxes_from_output -> bbox_targets), i.e. b2d_roi_targets_fused with boxes = props, box_count = count.  When
 * the proposal stage runs as cluster kernels the target stage is the TAIL of the same kernel (assignment spread over
 * the image's cluster, sampler + encode in its first CTA): no extra launch.  Otherwise the two entry points are called
 * one after the other; results are identical either way. */
B2D_API int b2d_rpn_proposals_targets(float* props, float* scores, int* count, int* prov, const void* const* cls_ptrs_host,
                              const void* const* reg_ptrs_host, const b2d_pyramid* pyr_host, const float* img_hw,
                              int B, const b2d_rpn_cfg* cfg_host, void* workspace, size_t ws_bytes,
                              const b2d_roi_target_args* tg_host, void* stream);

/* generic segmented top-k (descending, ties -> lowest index): values [S][ld] with
 * per-segment counts -> idx int32[S][k] (padded -1), out_count int32[S]. */
B2D_API size_t b2d_topk_workspace_bytes(long long n_max, int S, int k);
B2D_API int b2d_topk(int* idx, int* out_count, const float* values, long long ld, const int* counts, long long n,
             int S, int k, void* workspace, size_t ws_bytes, void* stream);

/* ---- K4: NMS (torchvision.ops.nms CPU semantics: stable descending score order,
 * areas without +1, suppress iff (double)iou > thr).  Segmented: boxes [S][n_ld][4]
 * ROW-major (the torchvision boundary, lib/heads/rpn_head.py:103), scores [S][n_ld],
 * counts int32[S] (NULL => n).  keep int64[S][n_ld] original indices in score order,
 * keep_count int32[S].  presorted != 0 skips the sort. */
B2D_API size_t b2d_nms_workspace_bytes(long long n_max, int S);
B2D_API int b2d_nms(int64_t* keep, int* keep_count, const float* boxes, const float* scores, long long n_ld,
            const int* counts, long long n, int S, float thr_f, int max_keep, int presorted, void* workspace,
            size_t ws_bytes, void* stream);

/* ---- index glue as kernels (round 2): multiclass / batched NMS front-end, RoI scaling, IoU-balanced sampler.
 * utils.multiclass_nms (lib/utils.py:224-269): bbox [n][4] (box_classes 1) or [n][4*C] viewed (n,4,C), score [n][C],
 * chan_mask_host = 2 x u64 bitmap of nms_channel, score_factor [n] or NULL, strict = mode 'strict'.  Outputs ROW-major
 * like the reference returns them: out_box [max_keep][4], out_score, out_label int64, out_count int32[1];
 * *overflow = 1 if more than `cap` (<= 16384) candidates passed the test. */
B2D_API size_t b2d_multiclass_nms_workspace_bytes(int cap);
B2D_API int b2d_multiclass_nms(float* out_box, float* out_score, int64_t* out_label, int* out_count, const float* bbox,
                       int box_classes, const float* score, long long n, int C, const unsigned long long* chan_mask_host,
                       float min_score, const float* score_factor, int strict, float nms_thr_f, int max_keep, int cap,
                       int* overflow, void* workspace, size_t ws_bytes, void* stream);
/* the candidate stage of b2d_multiclass_nms alone, into caller arrays of `cap` entries (cand_box / nms_box [cap][4]):
 * for candidate sets larger than b2d_nms takes (16384) */
B2D_API int b2d_multiclass_candidates(float* cand_box, float* nms_box, float* cand_score, int* cand_label, int* cand_count,
                              int* overflow, const float* bbox, int box_classes, const float* score, long long n, int C,
                              const unsigned long long* chan_mask_host, float min_score, const float* score_factor,
                              int strict, int cap, void* stream);
/* utils.batched_nms (lib/utils.py:211-221): out [n][4] = bbox + fp32(label * max(bbox)) -- the boxes handed to nms */
B2D_API int b2d_batched_nms_boxes(float* out, const float* bbox, const int64_t* label, long long n, void* stream);
/* GA-RPN call sites (GARPNHead.predict_bboxes_single_image, lib/heads/guided_head.py:621-669): guided anchors are explicit
 * per-location boxes [4][n_l] with a location mask (torch.bool [n_l]) per level.  b2d_ga_pack_scores writes the logits of all
 * levels as rows of one [L][ld] array with -inf at masked / padded places (the input of ONE segmented b2d_topk over the
 * levels); b2d_ga_decode gathers anchor + deltas of the selected places, decodes and clamps them (utils.param2bbox with
 * img_size, lib/utils.py:83-120) into box [L][k][4] (row-major, the layout b2d_nms takes), score = sigmoid(logit) or -inf
 * for masked rows and for boxes below min_size, nvalid int32[L] = selected unmasked places per level. */
B2D_API int b2d_ga_pack_scores(float* out, long long ld, const void* const* cls_ptrs_host, const void* const* mask_ptrs_host,
                       const int* n_host, int L, void* stream);
B2D_API int b2d_ga_decode(float* box, float* score, int* nvalid, const int* idx, const float* packed, long long ld, int k,
                  const void* const* cls_ptrs_host, const void* const* mask_ptrs_host, const void* const* anchor_ptrs_host,
                  const void* const* reg_ptrs_host, const int* n_host, int L, const float* means_host, const float* stds_host,
                  float img_h, float img_w, float min_size, void* stream);
/* ScalableRoICrop.scale_bbox (lib/region.py:220-225) on [4][ld] boxes */
B2D_API int b2d_scale_rois(float* out, const float* rois, long long ld, long long n, float scale, void* stream);
/* IoUBalancedNegSampler (lib/region.py:128-172).  Bins are given HIGHEST IoU range first (the reference's walk order),
 * bounds already rounded to fp32 like torch's tensor-vs-python-scalar comparison.  ids: 0 positive, 1 + j bin j, -1 none. */
B2D_API int b2d_iou_bin_ids(int* ids, const int64_t* labels, const float* iou, long long n, int num_bins,
                    const float* bin_lo_host, const float* bin_hi_host, void* stream);
B2D_API int b2d_sample_iou_balanced(int64_t* out_labels, const int64_t* labels, const float* iou, long long n, int max_num,
                            int pos_num, int num_bins, const float* bin_lo_host, const float* bin_hi_host,
                            unsigned long long seed, void* stream);
/* CrossEntropyLoss on sampled rows (lib/losses.py:129-156; callers lib/heads/anchor_head.py:113-139 and
 * lib/heads/bbox_head.py:56-80): logits [C][ld] (row_major 0: the reference's tar_cls_out) or [rows][ld] (row_major 1),
 * target int64[rows] (< 0: ignored).  fwd: partial [64][2] = per-block (sum of row losses, rows counted);
 * bwd: grad (same layout as logits) = scale[0] * dloss/dlogit. */
B2D_API size_t b2d_sampled_ce_workspace_bytes(void);
B2D_API int b2d_sampled_ce_fwd(float* partial, const float* logits, long long ld, int C, int row_major, int sigmoid,
                       const int64_t* target, long long rows, void* stream);
B2D_API int b2d_sampled_ce_bwd(float* grad, const float* scale, const float* logits, long long ld, int C, int row_major,
                       int sigmoid, const int64_t* target, long long rows, void* stream);

/* ---- SURVEY 8(f-2): loss reductions adjacent to the path, fused with the target gather.
 * AnchorHead.calc_loss for a head without sampler (lib/heads/anchor_head.py:113-139):
 * sigmoid_focal_loss (lib/losses.py:33-61) over every non-ignored anchor and
 * smooth_l1_loss_v2 (:77-83) over the positives, read straight from the head maps
 * (cls_ptrs_host[l] -> [B, A*C, H, W], reg_ptrs_host[l] -> [B, 4A, H, W]) with the class
 * target / encoded deltas rebuilt from the assignment labels (int64 [B][label_ld], gt
 * index + 1 / 0 / -1) -- no [C, s] gathers.  out3 = {sum focal, sum smooth-L1, #pos}
 * (sums, not yet divided by the averaging factor).  _bwd writes scale2[0] * d(sum focal)/d(cls)
 * and scale2[1] * d(sum smooth-L1)/d(reg) in the maps' layout (scale2: device float[2]). */
B2D_API size_t b2d_anchor_loss_workspace_bytes(const b2d_pyramid* pyr_host, int B);
B2D_API int b2d_anchor_loss_fwd(float* out3, const void* const* cls_ptrs_host, const void* const* reg_ptrs_host,
                        const b2d_pyramid* pyr_host, const int64_t* labels, long long label_ld, const float* gt, int gt_ld,
                        const int64_t* gt_label, int cls_channels, float alpha, float gamma, float beta,
                        const float* means_host, const float* stds_host, int B, void* workspace, size_t ws_bytes,
                        void* stream);
B2D_API int b2d_anchor_loss_bwd(void* const* dcls_ptrs_host, void* const* dreg_ptrs_host, const float* scale2,
                        const void* const* cls_ptrs_host, const void* const* reg_ptrs_host, const b2d_pyramid* pyr_host,
                        const int64_t* labels, long long label_ld, const float* gt, int gt_ld, const int64_t* gt_label,
                        int cls_channels, float alpha, float gamma, float beta, const float* means_host,
                        const float* stds_host, int B, void* stream);

/* ---- SURVEY 8(f-4): plain FCOS target assignment, FCOSHead.single_image_targets
 * (lib/heads/fcos_head.py:371-416): per cell the smallest-area GT whose ltrb are all > 0 and
 * whose max(ltrb) lies in [level_thr[l], level_thr[l+1]) (level_scale_thr, :167).  Same
 * tensors and output layout as b2d_atss_assign; level_thr_host float[num_levels + 1]. */
B2D_API int b2d_fcos_targets(int64_t* cls_tar, float* reg_tar, float* ctr_tar, const b2d_pyramid* pyr_host, const float* gt,
                     int gt_ld, const int* gt_count, const int64_t* gt_label, const float* img_hw,
                     const float* level_thr_host, int B, void* stream);

/* ---- SURVEY 8(f-3): RCNN test-time detections, BBoxHead.predict_bboxes_single_image
 * (lib/heads/bbox_head.py:122-146): softmax(cls_out) -> per-class decode + clamp
 * (batched_param2bbox, lib/utils.py:96-106; reg channel = coord * C + class) ->
 * multiclass_nms over classes 1..C-1 (lib/utils.py:224-269; strict != 0: arg-max class
 * only) -> first max_per_img.  props [B][4][ld] (counts int32[B] or NULL => n),
 * cls_out [B][ld][C] logits, reg_out [B][ld][4 * reg_classes] (reg_classes = C, or 1 for
 * class-agnostic regression), img_hw float[B][2] or NULL (no clamp).  Outputs
 * out_box [B][4][max_per_img], out_score / out_label [B][max_per_img], out_count int32[B].
 * cap = candidate slots per image (<= 16384); *overflow is set to 1 if an image had more
 * candidates (they are then truncated in enumeration order). */
B2D_API size_t b2d_rcnn_detect_workspace_bytes(int cap, int B);
B2D_API int b2d_rcnn_detect(float* out_box, float* out_score, int64_t* out_label, int* out_count, const float* props,
                    long long ld, const int* counts, long long n, const float* cls_out, const float* reg_out, int C,
                    int reg_classes, const float* means_host, const float* stds_host, const float* img_hw,
                    float min_score, float nms_thr_f, int max_per_img, int strict, int cap, int B, int* overflow,
                    void* workspace, size_t ws_bytes, void* stream);
/* b2d_rcnn_detect plus the packed detection records of dist.pack_detections: records fp32
 * [B][max_per_img][6] = (x1, y1, x2, y2, score, float(label)), rows past out_count[b] zero --
 * the payload of dist.gather_detections, written by the gather kernel itself. */
B2D_API int b2d_rcnn_detect_records(float* out_box, float* out_score, int64_t* out_label, int* out_count, float* records,
                            const float* props, long long ld, const int* counts, long long n, const float* cls_out,
                            const float* reg_out, int C, int reg_classes, const float* means_host, const float* stds_host,
                            const float* img_hw, float min_score, float nms_thr_f, int max_per_img, int strict, int cap,
                            int B, int* overflow, void* workspace, size_t ws_bytes, void* stream);

/* ---- dense-head test-time detections: utils.multiclass_nms (lib/utils.py:224-269) for B images at once, as
 * AnchorHead.predict_single_image (lib/heads/anchor_head.py:207-258, RetinaNet) and FCOSHead.predict_single_image
 * (lib/heads/fcos_head.py:570-631) call it after their selection.  Rows: boxes [B][4][ld] already decoded
 * (class-agnostic), counts int32[B], rows int32[B][ld] = the flat anchor / point index of each row.  The C class values
 * of a row with flat index f in level l (lv.offset[l] <= f < lv.offset[l + 1]) are
 * lv.base[l][b * lv.img_stride[l] + c * lv.class_stride[l] + (f - lv.offset[l])] -- e.g. RetinaNet's logit maps
 * cls_l.view(B, C, -1) in place, or FCOS's score [B][C][total] as one level.  transform: 0 the values are scores, 1
 * sigmoid, 2 softmax over the C values.  min_score is tested on that score; the candidate's score is score *
 * score_factor[b][f] (score_factor [B][factor_ld] or NULL).  chan_mask_host: 2 x u64 bitmap of nms_channel; strict:
 * only the first maximal channel of a row, if it is an NMS channel.  Candidates are ordered row-major, channel minor;
 * the NMS offset is channel * max(candidate boxes); label_add is added to the written labels only (1 for a sigmoid head's
 * 1-based labels).  Outputs and records as b2d_rcnn_detect(_records); workspace b2d_rcnn_detect_workspace_bytes(cap, B);
 * cap <= 16384 candidates per image, *overflow = 1 if an image had more.  events_host: NULL, or two cudaEvent_t (either
 * may be NULL) recorded after the candidate stage and after the NMS. */
typedef struct b2d_dense_levels {
    int num_levels, _pad;
    long long offset[B2D_MAX_LEVELS];       /* first flat index of the level (offset[0] == 0, ascending) */
    const float* base[B2D_MAX_LEVELS];      /* DEVICE pointer of the level's class values (image 0, class 0, index 0) */
    long long img_stride[B2D_MAX_LEVELS], class_stride[B2D_MAX_LEVELS];
} b2d_dense_levels;
B2D_API int b2d_dense_detect(float* out_box, float* out_score, int64_t* out_label, int* out_count, const float* boxes,
                     long long ld, const int* counts, const int* rows, const b2d_dense_levels* lv_host, int C, int transform,
                     const float* score_factor, long long factor_ld, const unsigned long long* chan_mask_host,
                     float min_score, int label_add, float nms_thr_f, int max_per_img, int strict, int cap, int B,
                     int* overflow, void* workspace, size_t ws_bytes, void* const* events_host, void* stream);
B2D_API int b2d_dense_detect_records(float* out_box, float* out_score, int64_t* out_label, int* out_count, float* records,
                             const float* boxes, long long ld, const int* counts, const int* rows,
                             const b2d_dense_levels* lv_host, int C, int transform, const float* score_factor,
                             long long factor_ld, const unsigned long long* chan_mask_host, float min_score, int label_add,
                             float nms_thr_f, int max_per_img, int strict, int cap, int B, int* overflow, void* workspace,
                             size_t ws_bytes, void* const* events_host, void* stream);

/* ---- K5/K6: FPN level-mapped RoIAlign (BasicRoIExtractor, lib/region.py:243-306 +
 * torchvision RoIAlign aligned=False).  rois [4, R] column-major, roi_img int32[R]
 * (NULL => image 0).  feat_ptrs_host[l] -> level l features, fp32 NCHW [B,C,H,W]
 * (layout 0) or NHWC [B,H,W,C] (layout 1) or bf16 NHWC (layout 2).  Level map:
 * floor(log2(sqrt((w+1)(h+1))/finest_scale + 1e-6)) clamped (lib/region.py:256-264);
 * levels int32[R] if non-NULL overrides the map.  out [R, C, PH, PW] fp32. */
typedef struct b2d_roi_cfg {
    int num_levels, C, PH, PW, sampling_ratio, aligned, layout;
    float finest_scale;
    int H[B2D_MAX_LEVELS], W[B2D_MAX_LEVELS];
    float spatial_scale[B2D_MAX_LEVELS];
} b2d_roi_cfg;

B2D_API int b2d_roi_align_fwd(float* out, const void* const* feat_ptrs_host, const float* rois, long long roi_ld,
                      const int* roi_img, const int* levels, long long R, const b2d_roi_cfg* cfg_host,
                      void* stream);
/* image-major variant for the fused pipeline: rois [B][4][ld] with counts int32[B];
 * out [B*ld, C, PH, PW]; rows past counts[b] are left untouched. */
B2D_API int b2d_roi_align_fwd_batched(float* out, const void* const* feat_ptrs_host, const float* rois, long long ld,
                              const int* counts, int B, const b2d_roi_cfg* cfg_host, void* stream);
B2D_API size_t b2d_roi_align_bwd_workspace_bytes(long long R, int B, const b2d_roi_cfg* cfg_host);
B2D_API int b2d_roi_align_bwd(void* const* grad_feat_ptrs_host, const float* grad_out, const float* rois,
                      long long roi_ld, const int* roi_img, const int* levels, long long R, int B,
                      const b2d_roi_cfg* cfg_host, void* workspace, size_t ws_bytes, void* stream);
/* fp32 NCHW [B,C,H,W] -> NHWC [B,H,W,C]: reference-layout FPN features (lib/necks.py:69-90)
 * to the channels-last layout the vectorised RoIAlign kernels read. */
B2D_API int b2d_nchw_to_nhwc(float* dst, const float* src, int B, int C, int H, int W, void* stream);
B2D_API int b2d_roi_levels(int* levels, const float* rois, long long roi_ld, long long R, float finest_scale,
                   int num_levels, void* stream);

/* ---- sparse host -> device feature transfer for the RoI extractor (csrc/roi_fetch.cu).
 * BasicRoIExtractor (lib/region.py:299-375) reads only the cells under the bilinear taps of the RoIs.  When the
 * pyramid is channels-last in PINNED (mapped) HOST memory, b2d_roi_mark_cells writes a bitmap with one bit per
 * (level, image, y, x) -- levels in order, each padded to whole 32-bit words, b2d_roi_cell_bitmap_bytes in total --
 * holding the cells under the bilinear taps of every RoI (rois [B][4][ld], counts int32[B], as
 * b2d_roi_align_fwd_batched; the same level map and sample geometry, so exactly the cells RoIAlign reads are marked), and b2d_fetch_marked_cells copies the
 * marked cells from src (device-visible pointers of the host tensors, [B,H,W,C] per level) to the same offsets of
 * dst (device tensors of the same shape) with SM-issued loads; *moved_cells (device, may be NULL) is incremented by
 * the number of cells copied.  Needs cfg.layout 1 or 2 and a fixed sampling_ratio. */
B2D_API size_t b2d_roi_cell_bitmap_bytes(int B, const b2d_roi_cfg* cfg_host);
B2D_API int b2d_roi_mark_cells(void* bitmap, const float* rois, long long ld, const int* counts, int B,
                       const b2d_roi_cfg* cfg_host, void* stream);
B2D_API int b2d_fetch_marked_cells(void* const* dst_ptrs_host, const void* const* src_ptrs_host, const void* bitmap,
                           int B, const b2d_roi_cfg* cfg_host, unsigned long long* moved_cells, void* stream);

/* ---- K7: RoIPool (torchvision.ops.roi_pool semantics), single level, NCHW fp32.
 * argmax int32 [R,C,PH,PW] (index into the H*W plane, -1 = empty). */
B2D_API int b2d_roi_pool_fwd(float* out, int* argmax, const float* feat, int B, int C, int H, int W, const float* rois,
                     long long roi_ld, const int* roi_img, long long R, float spatial_scale, int PH, int PW,
                     void* stream);
B2D_API int b2d_roi_pool_bwd(float* grad_feat, const float* grad_out, const int* argmax, int B, int C, int H, int W,
                     const float* rois, long long roi_ld, const int* roi_img, long long R, float spatial_scale,
                     int PH, int PW, void* workspace, size_t ws_bytes, void* stream);

/* ---- a17: BBoxHead.refine_bboxes_single_image (lib/heads/bbox_head.py:100-120), batched.
 * props [B][4][ld] with counts int32[B] (NULL => n); label int64 [B][ld]; reg_out [B][ld][4*C]
 * row-major with channel = coord*C + class (C = 1 when class-agnostic, label may then be NULL);
 * is_gt int64 [B][ld] or NULL.  out [B][4][ld] receives the non-GT columns in order, decoded with
 * means/stds and (clamp != 0) clamped to img_hw[b]; out_count int32[B]. */
B2D_API int b2d_refine_bboxes(float* out, int* out_count, const float* props, long long ld, const int* counts,
                      long long n, const int64_t* label, const float* reg_out, int C, const int64_t* is_gt,
                      const float* means_host, const float* stds_host, int clamp, const float* img_hw, int B,
                      void* stream);
/* Test-time form (CascadeRCNN.forward_test, lib/detectors/cascade_rcnn.py:186-190): the label of
 * row i is argmax(cls_out[b][i][0..num_classes)) -- the first maximal index, background
 * included, as torch.argmax -- computed in the kernel; no GT columns, nothing dropped
 * (out_count = counts).  cls_out [B][ld][num_classes] raw logits; reg_out [B][ld][4*reg_classes]
 * (reg_classes = num_classes, or 1 when class-agnostic); always clamped to img_hw[b].
 * Rows at or past counts[b] are neither read nor written. */
B2D_API int b2d_refine_bboxes_argmax(float* out, int* out_count, const float* props, long long ld, const int* counts,
                             long long n, const float* cls_out, int num_classes, const float* reg_out,
                             int reg_classes, const float* means_host, const float* stds_host, const float* img_hw,
                             int B, void* stream);

/* ---- a18 / K9: ATSS target assignment (FCOSHead.single_image_targets_atss,
 * lib/heads/fcos_head.py:283-368 with topk_by_center :106-116 read as integer division).
 * pyr: one anchor per cell (ws = hs = stride * atss scale).  Outputs are level-major over the
 * pyr->total cells of an image: cls_tar int64 [B][total], reg_tar fp32 [B][total][4] (ltrb),
 * ctr_tar fp32 [B][total].  Distance ties are broken by the lowest cell index. */
B2D_API size_t b2d_atss_workspace_bytes(const b2d_pyramid* pyr_host, int B);
B2D_API int b2d_atss_assign(int64_t* cls_tar, float* reg_tar, float* ctr_tar, const b2d_pyramid* pyr_host,
                    const float* gt, int gt_ld, const int* gt_count, const int64_t* gt_label, const float* img_hw,
                    int B, int topk, void* workspace, size_t ws_bytes, void* stream);

/* ---- a19: FCOS decode (FCOSHead.predict_single_image, lib/heads/fcos_head.py:578-604 +
 * ltrb2bbox :63-75): per cell ltrb*std+mean -> xyxy, clamp to img_hw[b], strict min-size test.
 * cls_ptrs_host[l] -> [B, C, H, W] logits, reg_ptrs_host[l] -> [B, 4, H, W], ctr_ptrs_host
 * (NULL or [l] -> [B, 1, H, W]).  boxes [B][4][total], score [B][C][total] = sigmoid(cls),
 * ctr_score [B][total] = sigmoid(ctr), key [B][total] = max_c score (* ctr_score), -inf where the
 * size test fails (the per-level top-k of :605-613 runs on key). */
B2D_API int b2d_fcos_decode(float* boxes, float* key, float* score, float* ctr_score, const void* const* cls_ptrs_host,
                    const void* const* reg_ptrs_host, const void* const* ctr_ptrs_host, const b2d_pyramid* pyr_host,
                    int cls_channels, float reg_mean, float reg_std, float min_size, const float* img_hw, int B,
                    void* stream);
/* FCOS per-level selection (lib/heads/fcos_head.py:602-613), batched and without host reads: on key [B][total] of
 * b2d_fcos_decode (-inf = failed the size test), levels of level_sizes_host[l] points in order.  Per (image, level): more
 * than pre_nms valid points -> the top pre_nms by key, descending, ties to the lowest index (b2d_topk); otherwise all
 * valid points in ascending index order; levels concatenated.  idx int32 [B][P], P = sum_l min(pre_nms, n_l)
 * (pre_nms <= 0: n_l), receives flat point indices (-1 past count[b]); count int32[B].  sel_boxes (optional, with
 * boxes [B][4][total]): [B][4][P] the boxes of the selected points (zero past count[b]).  The workspace query returns
 * 0 for an unsupported configuration (a level top-k over 16384). */
B2D_API size_t b2d_dense_select_workspace_bytes(const int* level_sizes_host, int num_levels, int B, int pre_nms);
B2D_API int b2d_dense_select(int* idx, int* count, float* sel_boxes, const float* key, const float* boxes,
                     const int* level_sizes_host, int num_levels, int B, int pre_nms, void* workspace, size_t ws_bytes,
                     void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200DET_H_ */
