/*
 * odhead.h — C ABI of libodhead.so: the B200 (sm_100a) detection-head hot path.
 *
 * Drop-in boundary for the reference's layer classes (citations relative to the
 * reference tree, Sardhendu/ObjectDetection):
 *
 *   od_proposal_forward            replaces  Proposals.build                MaskRCNN/building_blocks/proposals_tf.py:136-214
 *   od_proposal_forward_levels     replaces  the same, fed by the RPN head's per-level outputs: rpn.py:50-67 (reshape +
 *                                            softmax), training.py:146-166 (concat over P2..P6) + proposals_tf.py:136-214
 *   od_apply_box_deltas            replaces  apply_box_deltas               proposals_tf.py:23-65
 *   od_clip_boxes                  replaces  clip_boxes_to_01               proposals_tf.py:67-94
 *   od_norm_boxes                  replaces  norm_boxes / norm_boxes_tf     utils.py:181-210
 *   od_topk                        replaces  tf.nn.top_k call sites         proposals_tf.py:169, detection.py:221
 *   od_nms                         replaces  tf.image.non_max_suppression   proposals_tf.py:234, detection.py:177
 *   od_gen_anchors                 replaces  gen_anchors / gen_anchors_pixel_coord   utils.py:336-369
 *   od_pyramid_roi_align_forward   replaces  MaskRCNN.roi_pooling           maskrcnn.py:74-187
 *   od_crop_and_resize             replaces  tf.image.crop_and_resize       maskrcnn.py:152, FasterRCNN/building_blocks/fastrcnn.py:68
 *   od_detection_target_forward    replaces  BuildDetectionTargets.build_detection_target   data_processor.py:512-652
 *   od_detection_forward           replaces  DetectionLayer.build           detection.py:80-260
 *   od_unmold_detections           replaces  unmold_detection + denorm_boxes   detection.py:8-53, utils.py:212-227
 *   od_rpn_target_forward          replaces  PreprareTrainData.build_rpn_targets   data_processor.py:173-294
 *   od_rpn_loss_forward            replaces  Loss.rpn_class_loss / rpn_box_loss       loss_optimize.py:11-87
 *   od_mrcnn_loss_forward          replaces  Loss.mrcnn_class_loss / mrcnn_box_loss   loss_optimize.py:89-201
 *   od_frcnn_proposal_forward      replaces  FasterRCNN Proposals.build     FasterRCNN/building_blocks/proposals.py:392-512
 *   od_roi_pool_forward            replaces  roi_pool                       FasterRCNN/building_blocks/fastrcnn.py:22-70
 *
 * Conventions
 *   - Tensors cross the boundary as DLPack `DLTensor*` (zero copy). Device must be
 *     kDLCUDA, data C-contiguous unless a function says "any strides", dtype checked.
 *   - Outputs and workspace are caller-allocated. Query sizes with *_workspace_bytes.
 *   - Every call enqueues kernels on `stream` (a cudaStream_t passed as void*) and
 *     returns without synchronising. No global state; re-entrant; the caller selects
 *     the device (cudaSetDevice) before calling.
 *   - Return value: OD_OK (0) or a negative od_status. Never throws, never frees
 *     caller memory. od_strerror() gives a static message; od_last_error_detail()
 *     a thread-local detail string for the last failing call on this thread.
 *   - There is no CPU path behind this ABI.
 */
#ifndef ODHEAD_H_
#define ODHEAD_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- DLPack ABI subset (layout-compatible with dlpack.h >= 0.6) ---------- */
#ifndef DLPACK_DLPACK_H_
#define DLPACK_DLPACK_H_
typedef enum {
  kDLCPU = 1,
  kDLCUDA = 2,
  kDLCUDAHost = 3,
  kDLCUDAManaged = 13
} DLDeviceType;
typedef struct { DLDeviceType device_type; int32_t device_id; } DLDevice;
typedef enum {
  kDLInt = 0U, kDLUInt = 1U, kDLFloat = 2U, kDLOpaqueHandle = 3U, kDLBfloat = 4U, kDLBool = 6U
} DLDataTypeCode;
typedef struct { uint8_t code; uint8_t bits; uint16_t lanes; } DLDataType;
typedef struct {
  void* data;
  DLDevice device;
  int32_t ndim;
  DLDataType dtype;
  int64_t* shape;
  int64_t* strides;      /* in elements; NULL = compact row-major */
  uint64_t byte_offset;
} DLTensor;
#endif /* DLPACK_DLPACK_H_ */

/* ---- status codes --------------------------------------------------------- */
typedef enum {
  OD_OK = 0,
  OD_ERR_NULL = -1,       /* required pointer is NULL */
  OD_ERR_DTYPE = -2,      /* wrong dtype */
  OD_ERR_SHAPE = -3,      /* wrong rank / extent / inconsistent sizes */
  OD_ERR_DEVICE = -4,     /* not a CUDA tensor, or tensors on different devices */
  OD_ERR_LAYOUT = -5,     /* not contiguous / misaligned */
  OD_ERR_WORKSPACE = -6,  /* workspace too small or NULL */
  OD_ERR_CUDA = -7,       /* a CUDA runtime call or launch failed */
  OD_ERR_PARAM = -8       /* parameter out of supported range */
} od_status;

/* every entry point below has default ELF visibility (the library is built -fvisibility=hidden) */
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

int od_version(void);                       /* 10000*major + 100*minor + patch */
const char* od_source_hash(void);           /* sha1 of the sources this library was compiled from (build.py) */
const char* od_strerror(int status);
const char* od_last_error_detail(void);     /* thread-local, never NULL */
/* Kernels launched by this library in this process so far (statistics only; a relaxed atomic counter). */
int64_t od_launch_count(void);

/* ---- anchors (utils.py:230-369) ------------------------------------------- */
#define OD_MAX_LEVELS 8
#define OD_MAX_RATIOS 8
typedef struct od_anchor_spec {
  int32_t num_levels;                 /* len(scales) == len(feature_map_shapes) */
  int32_t num_ratios;
  double scales[OD_MAX_LEVELS];       /* RPN_ANCHOR_SCALES, one per level */
  double ratios[OD_MAX_RATIOS];       /* RPN_ANCHOR_RATIOS */
  int32_t fmap_h[OD_MAX_LEVELS];      /* get_resnet_stage_shapes */
  int32_t fmap_w[OD_MAX_LEVELS];
  int32_t fmap_stride[OD_MAX_LEVELS]; /* RESNET_STRIDES */
  int32_t anchor_stride;              /* RPN_ANCHOR_STRIDE */
  int32_t image_h, image_w;           /* normalisation: (box - [0,0,1,1]) / (h-1, w-1, h-1, w-1) */
} od_anchor_spec;

int64_t od_anchor_count(const od_anchor_spec* spec);
/* anchors: [B,A,4] f32 normalised (gen_anchors) when normalized != 0, or
 * [A,4] f64 pixel coordinates (gen_anchors_pixel_coord) when normalized == 0.
 * Ordering: level-major, then y, x, ratio (ratio fastest). */
int od_gen_anchors(const od_anchor_spec* spec, int normalized, DLTensor* anchors, void* stream);

/* ---- box decode / clip (proposals_tf.py:23-94) ----------------------------- */
/* boxes, deltas, out: [B,K,4] f32. deltas are already multiplied by the stddev. */
int od_apply_box_deltas(const DLTensor* boxes, const DLTensor* deltas, DLTensor* out, void* stream);
/* window: [4] (shared) or [B,4] f32; out = max(min(v, hi), lo) per coordinate. */
int od_clip_boxes(const DLTensor* boxes, const DLTensor* window, DLTensor* out, void* stream);
/* Pixel -> normalised coordinates, (box - [0,0,1,1]) / (h-1, w-1, h-1, w-1), out [...,4] f32.
 * tf_float32 == 0: utils.norm_boxes (utils.py:181-196; boxes i32 | f32 | f64, evaluated in float64, rounded once) -
 *                  the window of DetectionLayer (detection.py:66) and of unmold_detection (detection.py:17);
 * tf_float32 != 0: utils.norm_boxes_tf (utils.py:198-210; boxes f32, every operation in float32 with
 *                  scale = float32(h) - 1.0f) - the in-graph normalisation of the GT boxes (training.py:135). */
int od_norm_boxes(const DLTensor* boxes, int32_t image_h, int32_t image_w, int32_t tf_float32, DLTensor* out, void* stream);

/* ---- top-k: k largest per row, sorted descending, ties -> lower index ------ */
size_t od_topk_workspace_bytes(int64_t rows, int64_t cols, int64_t k);
/* scores: [B,A] f32, ANY strides (e.g. the probs[:,:,1] view of [B,A,2]).
 * values: [B,k] f32 or NULL; indices: [B,k] i32. */
int od_topk(const DLTensor* scores, int64_t k, DLTensor* values, DLTensor* indices,
            void* ws, size_t ws_bytes, void* stream);

/* ---- greedy hard NMS with tf.image.non_max_suppression semantics ---------- */
size_t od_nms_workspace_bytes(int64_t batch, int64_t num_boxes);
/* boxes [B,K,4] f32 (any corner order; canonicalised like TF), scores [B,K] f32,
 * num_valid [B] i32 or NULL (only the first num_valid[b] boxes of image b take part).
 * Candidates are visited by (score desc, index asc); box i is dropped iff IoU > thr
 * with an already kept box. keep_idx [B,max_out] i32 in selection order, -1 padded;
 * num_kept [B] i32 (may be NULL). */
int od_nms(const DLTensor* boxes, const DLTensor* scores, const DLTensor* num_valid,
           float iou_threshold, int64_t max_out, DLTensor* keep_idx, DLTensor* num_kept,
           void* ws, size_t ws_bytes, void* stream);

/* ---- ProposalLayer (proposals_tf.py:98-326) -------------------------------- */
typedef struct od_proposal_params {
  float bbox_stddev[4];     /* RPN_BBOX_STDDEV as float32 */
  int32_t pre_nms_limit;    /* PRE_NMS_ROIS_COUNT; K = min(pre_nms_limit, A) */
  int32_t post_nms_count;   /* POST_NMS_ROIS_{TRAINING,INFERENCE} = N */
  float nms_threshold;      /* RPN_NMS_THRESHOLD */
} od_proposal_params;

/* Optional intermediates (the reference's DEBUG=True outputs, proposals_tf.py:202-214).
 * Any member may be NULL. */
typedef struct od_proposal_debug {
  DLTensor* ix;                    /* [B,K] i32   top-k anchor indices */
  DLTensor* scores;                /* [B,K] f32   gathered fg scores */
  DLTensor* bbox_delta;            /* [B,K,4] f32 gathered rpn_bbox * stddev */
  DLTensor* anchors;               /* [B,K,4] f32 gathered anchors */
  DLTensor* anchor_delta;          /* [B,K,4] f32 decoded, unclipped */
  DLTensor* anchor_delta_clipped;  /* [B,K,4] f32 decoded, clipped to [0,0,1,1] */
  DLTensor* keep_idx;              /* [B,N] i32   NMS keep positions into the K list, -1 padded */
  DLTensor* num_kept;              /* [B] i32 */
} od_proposal_debug;

size_t od_proposal_workspace_bytes(int64_t batch, int64_t num_anchors, const od_proposal_params* p);
/* Head outputs in bf16. The arguments that carry a network head's output (the RPN logits and deltas here, mrcnn_bbox
 * and mrcnn_class_probs of od_detection_forward, the predictions of the two loss entry points) are f32 or bf16
 * (kDLBfloat, 16 bits; float16 and every other dtype are refused with OD_ERR_DTYPE), each argument on its own and
 * every level of a level list of one dtype (a mixed list is refused with OD_ERR_DTYPE, naming the level). A bf16
 * tensor must be aligned to the kernel's load (OD_ERR_LAYOUT otherwise): 2 bytes for a scalar, 4 for a (bg,fg) logit
 * pair, 8 for a 4-value delta or box row. A bf16 value is widened to fp32 exactly (bits << 16: sign, NaN payload and
 * subnormals survive; the library is built without flush-to-zero) and everything after the load is the f32 path, so
 * every output and DEBUG tensor (all f32) equals that of the call on the widened f32 tensors bit for bit. Every other
 * argument keeps its f32 / i32 dtype.
 *
 * rpn_class_probs [B,A,2] f32 (bg,fg), rpn_bbox [B,A,4] f32 or bf16 (dy,dx,log dh,log dw),
 * anchors [B,A,4] f32 normalised, or NULL with a non-NULL `spec` (anchors are then
 * regenerated in fp64 from the index inside the decode kernel).
 * proposals [B,N,4] f32, rows after the kept ones are zero. */
int od_proposal_forward(const DLTensor* rpn_class_probs, const DLTensor* rpn_bbox,
                        const DLTensor* anchors, const od_anchor_spec* spec,
                        const od_proposal_params* params, DLTensor* proposals,
                        const od_proposal_debug* debug,
                        void* ws, size_t ws_bytes, void* stream);

/* The same layer fed by the RPN head's conv outputs in their native per-level layout (SURVEY 8(f)3): no
 * [B,A,2] / [B,A,4] concatenation is materialised.
 * class_logits[l]: [B,H_l,W_l,2a] f32 or bf16 NHWC ('rpn_class_raw', rpn.py:50; a anchors per location, (bg,fg) pairs),
 * bbox[l]:         [B,H_l,W_l,4a] f32 or bf16 NHWC ('rpn_bbox_pred', rpn.py:63), l < num_levels. The logits and the
 * deltas each have one dtype for every level, chosen independently (bf16 as for od_proposal_forward).
 * The reference reshapes each to [B,-1,2] / [B,-1,4], takes the softmax of the pairs (rpn.py:54-59) and concatenates
 * the levels along the anchor axis (training.py:163-166); anchor i of that concatenation is what `anchors`/`spec`,
 * debug.ix etc. refer to. The fg probability exp(fg-m)/(exp(bg-m)+exp(fg-m)), m = max(bg,fg), is computed in fp32
 * for every anchor into the workspace ([B,A] f32) and ranked; deltas are read from their level only for the
 * pre_nms_limit selected anchors. */
size_t od_proposal_levels_workspace_bytes(int64_t batch, int64_t num_anchors, const od_proposal_params* p);
int od_proposal_forward_levels(const DLTensor* const* class_logits, const DLTensor* const* bbox, int32_t num_levels,
                               const DLTensor* anchors, const od_anchor_spec* spec,
                               const od_proposal_params* params, DLTensor* proposals,
                               const od_proposal_debug* debug,
                               void* ws, size_t ws_bytes, void* stream);

/* ---- PyramidROIAlign (maskrcnn.py:74-187) ---------------------------------- */
/* fmaps[l]: [B,H_l,W_l,D] f32 or bf16 NHWC for level (min_level + l), l < num_levels, every level of one dtype;
 * rois [B,N,4] f32 normalised (y1,x1,y2,x2);
 * pooled: [1,B*N,P_h,P_w,D] (or [B*N,P_h,P_w,D]) f32 or bf16, whatever the maps' dtype; row b*N+n <-> rois[b,n];
 * roi_level: [B,N] i32 or NULL. D must be a multiple of 4, and of 8 when the maps or pooled are bf16 (kDLBfloat, 16 bits;
 * float16 is refused like every other dtype).
 * Numerics: the blend is fp32 in the reference's order; bf16 map values are widened exactly, so an f32 pooled result from
 * bf16 maps equals the f32 path on the widened maps bit for bit. A bf16 pooled value is that fp32 value rounded to the
 * nearest bf16, ties to even (overflow to inf; NaN stays NaN, its payload may differ). The same holds for
 * od_crop_and_resize, whose extrapolation_value is rounded the same way. */
int od_pyramid_roi_align_forward(const DLTensor* const* fmaps, int32_t num_levels, int32_t min_level,
                                 const DLTensor* rois, int32_t image_h, int32_t image_w,
                                 int32_t pool_h, int32_t pool_w,
                                 DLTensor* pooled, DLTensor* roi_level, void* stream);
/* The same call with a small PERSISTENT workspace (od_pyramid_roi_align_workspace_bytes() bytes, 8-byte aligned, device
 * memory of the tensors' GPU) that lets the persistent CTAs of the D = 256 kernel draw ROIs dynamically instead of in a
 * fixed round robin. The caller zero-initialises it ONCE (e.g. cudaMemset after allocating it); every launch leaves it
 * zeroed again. One workspace must not be used by two launches that can run concurrently (one per stream is safe). */
size_t od_pyramid_roi_align_workspace_bytes(void);
/* A workspace of ..._bytes_n(B*N) bytes additionally holds a processing order of the ROIs (level by level, top to bottom),
 * computed by a short pre-pass of every launch, so that ROIs reading the same feature pixels run close in time and every
 * pixel is fetched from HBM once. Only the first od_pyramid_roi_align_workspace_bytes() bytes must be (and stay) zeroed.
 * The results do not depend on the order. */
size_t od_pyramid_roi_align_workspace_bytes_n(int64_t n_rois);
/* The processing order as a tensor of its own: order [B*N] i32, a permutation of 0..B*N-1 (N <= 4096 per image). A caller
 * that pools the SAME rois with several pool shapes (the 7x7 and the 14x14 pooling of one step) computes it once and passes
 * it to od_pyramid_roi_align_forward_ordered, which then skips its pre-pass; order == NULL behaves like ..._forward_ws.
 * Entries outside [0, B*N) are skipped (their rows are not written), nothing is read or written out of bounds. */
int od_roi_processing_order(const DLTensor* rois, int32_t image_h, int32_t image_w, int32_t min_level, int32_t num_levels,
                            DLTensor* order, void* stream);
int od_pyramid_roi_align_forward_ordered(const DLTensor* const* fmaps, int32_t num_levels, int32_t min_level,
                                         const DLTensor* rois, int32_t image_h, int32_t image_w,
                                         int32_t pool_h, int32_t pool_w,
                                         DLTensor* pooled, DLTensor* roi_level, const DLTensor* order,
                                         void* ws, size_t ws_bytes, void* stream);
int od_pyramid_roi_align_forward_ws(const DLTensor* const* fmaps, int32_t num_levels, int32_t min_level,
                                    const DLTensor* rois, int32_t image_h, int32_t image_w,
                                    int32_t pool_h, int32_t pool_w,
                                    DLTensor* pooled, DLTensor* roi_level, void* ws, size_t ws_bytes, void* stream);

/* tf.image.crop_and_resize(method="bilinear"): image [B,H,W,D] f32 or bf16 NHWC,
 * boxes [n,4] f32, box_ind [n] i32 (out-of-range -> that crop is left untouched),
 * out [n,crop_h,crop_w,D] f32 or bf16 (dtypes, D and numerics as od_pyramid_roi_align_forward). */
int od_crop_and_resize(const DLTensor* image, const DLTensor* boxes, const DLTensor* box_ind,
                       int32_t crop_h, int32_t crop_w, float extrapolation_value,
                       DLTensor* out, void* stream);

/* ---- DetectionTargetLayer (data_processor.py:430-658) ----------------------- */
typedef struct od_target_params {
  int32_t rois_per_image;   /* MRCNN_TRAIN_ROIS_PER_IMAGE = R */
  float bbox_stddev[4];     /* BBOX_STD_DEV as float32 */
  int32_t mask_h, mask_w;   /* mask target size (28,28); only read when gt_masks != NULL */
  int32_t use_mini_mask;    /* != 0: gt_masks are mini masks cropped to their GT box (USE_MINI_MASK, config.py:57-58):
                               the ROI is re-expressed in the GT box's frame before the crop */
  int32_t mask_layout_hwg;  /* 0: gt_masks [B,G,Mh,Mw]; != 0: [B,Mh,Mw,G] (batch_gt_masks, data_processor.py:386) */
} od_target_params;

/* Optional intermediates (data_processor.py:629-652); members may be NULL. */
typedef struct od_target_debug {
  DLTensor* iou;            /* [B,N,G] f32; rows/cols in compacted order, rest untouched */
  DLTensor* roi_iou_max;    /* [B,N] f32 */
  DLTensor* pos_indices;    /* [B,N] i32  where(max>=0.5) before shuffling, -1 padded */
  DLTensor* neg_indices;    /* [B,N] i32  where(max<0.5)  before shuffling, -1 padded */
  DLTensor* counts;         /* [B,6] i32: n_prop, n_gt, n_pos_all, n_neg_all, pos_count, neg_count */
  DLTensor* sampled_pos;    /* [B,R] i32 sampled positive indices, -1 padded */
  DLTensor* sampled_neg;    /* [B,R] i32 sampled negative indices, -1 padded */
  DLTensor* gt_assignment;  /* [B,R] i32 argmax GT (compacted index) per sampled positive, -1 padded */
} od_target_debug;

size_t od_detection_target_workspace_bytes(int64_t batch, int64_t num_proposals, int64_t num_gt);
/* proposals [B,N,4] f32 (zero-padded), gt_class_ids [B,G] i32 (0 = pad), gt_boxes [B,G,4] f32,
 * perm_pos / perm_neg [B,N] i32: permutations of 0..N-1 standing in for tf.random_shuffle
 * (data_processor.py:587,:597): the j-th entry of the shuffled list is
 * list[q_j] where q = (p for p in perm if p < len(list)), in perm order.
 * rois [B,R,4] f32, roi_gt_class_ids [B,R] i32, roi_gt_box_deltas [B,R,4] f32.
 * gt_masks [B,G,Mh,Mw] (or [B,Mh,Mw,G], see mask_layout_hwg) and mask_targets [B,R,mask_h,mask_w] f32 are optional
 * (both NULL or both set): target[r] = round(crop_and_resize(gt_mask[assigned GT of r], box_r, [mask_h,mask_w])) for
 * the sampled positives, zero rows elsewhere (north-star extension: the reference prepares the masks but its mask
 * head is commented out; semantics of the model it re-writes).
 * gt_masks is f32, u8 (kDLUInt, 8 bits) or bool (kDLBool, 8 bits), the dtypes mask datasets store masks in; every other
 * dtype (float16, bf16, int8, float64, ...) is refused with OD_ERR_DTYPE. A byte mask needs no alignment (f32: 4 bytes).
 * Each byte is widened to fp32 exactly (bool 0 / 1, u8 0..255) and everything after the load is the f32 path, so the
 * targets equal those of the f32 call on the widened masks bit for bit. mask_targets is always f32. */
int od_detection_target_forward(const DLTensor* proposals, const DLTensor* gt_class_ids,
                                const DLTensor* gt_boxes, const DLTensor* perm_pos, const DLTensor* perm_neg,
                                const od_target_params* params,
                                DLTensor* rois, DLTensor* roi_gt_class_ids, DLTensor* roi_gt_box_deltas,
                                const DLTensor* gt_masks, DLTensor* mask_targets,
                                const od_target_debug* debug,
                                void* ws, size_t ws_bytes, void* stream);

/* ---- RPN targets (data_processor.py:173-294; SURVEY.md §8f "next" row) --------- */
typedef struct od_rpn_target_params {
  int32_t max_rpn_targets;  /* RPN_TRAIN_ANCHORS_PER_IMAGE (256) */
  double bbox_stddev[4];    /* RPN_BBOX_STDDEV; the reference computes in float64 */
} od_rpn_target_params;

size_t od_rpn_target_workspace_bytes(int64_t batch, int64_t num_anchors, int64_t num_gt);
/* PreprareTrainData.build_rpn_targets, batched, float64 like the reference's numpy code.
 * anchors [A,4] f64 pixel coordinates (gen_anchors_pixel_coord), gt_boxes [B,G,4] f64 pixels with gt_count [B] i32 valid
 * rows each, perm_pos / perm_neg [B,A] i32: permutations standing in for the two np.random.choice draws (:246,:253):
 * with idx = where(label == +1 / -1), the entries idx[q] for the first `extra` values q of the permutation that
 * satisfy q < len(idx) are reset to 0.
 * rpn_target_class [B,A] i32 in {-1,0,+1}; rpn_target_bbox [B,max_rpn_targets,4] f64 (row i = i-th positive anchor in
 * ascending order, zero padded); positive_anchors [B,max_rpn_targets,4] f64 (zero padded);
 * counts [B,4] i32: positives / negatives before subsampling, positives / negatives kept. */
int od_rpn_target_forward(const DLTensor* anchors, const DLTensor* gt_boxes, const DLTensor* gt_count,
                          const DLTensor* perm_pos, const DLTensor* perm_neg, const od_rpn_target_params* params,
                          DLTensor* rpn_target_class, DLTensor* rpn_target_bbox, DLTensor* positive_anchors,
                          DLTensor* counts, void* ws, size_t ws_bytes, void* stream);

/* ---- head losses, forward values (loss_optimize.py:11-201; SURVEY.md §8f rank 4) ---------- */
/* Per-element arithmetic is fp32 in the reference's order; the sums are accumulated in fp64 in a fixed order and
 * rounded to fp32 once (deterministic; equal to TensorFlow's fp32 reductions to ~1e-7 relative).
 *
 * od_rpn_loss_forward: Loss.rpn_class_loss (:11-44) and Loss.rpn_box_loss (:47-87).
 *   rpn_target_class [B,A] or [B,A,1] i32 (+1 positive, -1 negative, 0 neutral), rpn_class_logits [B,A,2] f32 or bf16
 *   (bg,fg), rpn_target_bbox [B,T,4] f32 zero padded, rpn_pred_box [B,A,4] f32 or bf16 (both NULL: class loss only).
 *   bf16 predictions follow the head-output contract of od_proposal_forward: widened exactly, so the losses and
 *   pred_box_pos (the widened values) equal those of the f32 call on the widened tensors bit for bit.
 *   losses [2] f32 = (rpn_class_loss, rpn_box_loss); either is 0 when nothing contributes (K.switch).
 *   The r-th positive anchor of image b (ascending) pairs with rpn_target_bbox[b,r]; positives beyond T rows are
 *   ignored (the reference's shapes would not match there). pred_box_pos [P,4] f32 or NULL receives the gathered
 *   predictions of the positives in (image, anchor) order (rows past P are dropped); num_pos [1] i32 or NULL. */
size_t od_rpn_loss_workspace_bytes(int64_t batch, int64_t num_anchors);
int od_rpn_loss_forward(const DLTensor* rpn_target_class, const DLTensor* rpn_class_logits,
                        const DLTensor* rpn_target_bbox, const DLTensor* rpn_pred_box,
                        DLTensor* losses, DLTensor* pred_box_pos, DLTensor* num_pos,
                        void* ws, size_t ws_bytes, void* stream);
/* od_mrcnn_loss_forward: Loss.mrcnn_class_loss (:89-151) and Loss.mrcnn_box_loss (:154-201).
 *   mrcnn_target_class_ids [B,R] i32 zero padded; pred_logits [B,R,C] f32 or bf16 with batch_active_class_ids [B,C]
 *   f32 (row 0 is the one the reference gathers, :115) and / or target_box [B,R,4] f32 with pred_box [B,R,C,4] f32 or
 *   bf16 (bf16 as for od_rpn_loss_forward; pred_active stays f32).
 *   losses [2] f32 = (sum(ce * pred_active) / sum(pred_active), mean binary cross-entropy over the positive ROIs'
 *   boxes of their target class — K.binary_crossentropy as the reference has it — or 0 without positives);
 *   pred_active [B,R] f32 or NULL. A pair that is not passed leaves its loss at 0. */
int od_mrcnn_loss_forward(const DLTensor* mrcnn_target_class_ids, const DLTensor* pred_logits,
                          const DLTensor* batch_active_class_ids, const DLTensor* target_box,
                          const DLTensor* pred_box, DLTensor* losses, DLTensor* pred_active, void* stream);

/* ---- DetectionLayer (detection.py:56-279) ---------------------------------- */
typedef struct od_detection_params {
  float bbox_stddev[4];     /* BBOX_STD_DEV as float32 */
  float min_confidence;     /* DETECTION_MIN_THRESHOLD */
  float nms_threshold;      /* DETECTION_NMS_THRESHOLD */
  int32_t max_instances;    /* DETECTION_POST_NMS_INSTANCES */
} od_detection_params;

typedef struct od_detection_debug {
  DLTensor* class_ids;          /* [B,N] i32 */
  DLTensor* class_scores;       /* [B,N] f32 */
  DLTensor* bbox_delta;         /* [B,N,4] f32 gathered mrcnn_bbox * stddev */
  DLTensor* refined_proposals;  /* [B,N,4] f32 */
  DLTensor* clipped_proposals;  /* [B,N,4] f32 */
  DLTensor* keep_mask;          /* [B,N] i32 1 if (class>0 && score>min_conf) */
  DLTensor* nms_keep_mask;      /* [B,N] i32 1 if the ROI survives its class NMS */
} od_detection_debug;

size_t od_detection_workspace_bytes(int64_t batch, int64_t num_rois, int64_t num_classes);
/* proposals [B,N,4] f32, mrcnn_class_probs [B,N,C] f32 or bf16, mrcnn_bbox [B,N,C,4] f32 or bf16 (independently; bf16
 * under the head-output contract of od_proposal_forward: the argmax scan, its first-max and NaN rules, the score and
 * the decode are those of the f32 call on the widened values),
 * window_norm [B,4] f32 (norm_boxes of the pixel window, utils.py:181-196);
 * detections [B,max_instances,6] f32 rows (y1,x1,y2,x2,class_id,score), zero padded. */
int od_detection_forward(const DLTensor* proposals, const DLTensor* mrcnn_class_probs,
                         const DLTensor* mrcnn_bbox, const DLTensor* window_norm,
                         const od_detection_params* params, DLTensor* detections,
                         const od_detection_debug* debug,
                         void* ws, size_t ws_bytes, void* stream);

/* unmold_detection (detection.py:8-53) + denorm_boxes (utils.py:212-227) for a batch, on the device (SURVEY §8f):
 * detections [B,M,6] f32, window_norm [B,4] f32 (norm_boxes of the pixel windows), original_shape [B,2] i32 (h,w).
 * boxes [B,M,4] i32 pixel (y1,x1,y2,x2), class_ids [B,M] i32, scores [B,M] f32: the surviving rows (class_id != 0
 * prefix, zero-area boxes dropped) in order, zero padded; counts [B] i32 = rows kept. */
int od_unmold_detections(const DLTensor* detections, const DLTensor* window_norm, const DLTensor* original_shape,
                         DLTensor* boxes, DLTensor* class_ids, DLTensor* scores, DLTensor* counts, void* stream);

/* ---- Faster R-CNN single-level variants ------------------------------------ */
typedef struct od_frcnn_params {
  int32_t feat_stride;      /* RPN_FEATURE_STRIDE = 16 */
  int32_t image_h, image_w; /* clip to [0,w-1] x [0,h-1] */
  int32_t min_box_hw;       /* 16 */
  int32_t pre_nms_top_n;    /* 12000 / 6000 */
  int32_t post_nms_top_n;   /* 2000 / 300 */
  double nms_threshold;     /* suppress iff ovr >= threshold (proposals.py:163) */
  int32_t num_anchors;      /* 9 */
  double base_anchors[16 * 4]; /* (x1,y1,x2,y2) per anchor, proposals.py:188-196 */
} od_frcnn_params;

/* Largest batch the proposal layer takes: its kernels put the image on a grid y / z extent (at most 65535). A batch is
 * also refused when batch * post_nms_top_n exceeds 2^31 - 1 (int32 proposal rows). */
#define OD_FRCNN_MAX_BATCH 65535

/* Workspace of a batch of `batch` images of an fh x fw feature map; 0 for a NULL p or a batch outside
 * [0, OD_FRCNN_MAX_BATCH]. The single-image query below returns its value at batch 1. */
size_t od_frcnn_proposal_workspace_bytes_batch(int64_t batch, int64_t fh, int64_t fw, const od_frcnn_params* p);
size_t od_frcnn_proposal_workspace_bytes(int64_t fh, int64_t fw, const od_frcnn_params* p);
/* A batch of B images with one image size and one set of thresholds (params):
 * rpn_box_class_prob [B,h,w,2*na] f32|f64 (channels [:na] are read as fg, proposals.py:477), B <= OD_FRCNN_MAX_BATCH,
 * rpn_bbox [B,h,w,4*na] same dtype (dx,dy,dw,dh per anchor).
 * proposals [B*post_nms_top_n,5] f32 rows (b,x1,y1,x2,y2): the kept boxes of image 0 in visiting order, then those
 * of image 1, and so on; rows >= num_out[0] + ... + num_out[B-1] are zero.
 * num_out [B] i32: rows of image b. Each image's rows are those a batch of one gives for it.
 * Scores are ranked by a flattened stable descending order (the intended semantics of proposals.py:352-358; see
 * DESIGN.md for the reference's argsort quirk). */
int od_frcnn_proposal_forward(const DLTensor* rpn_box_class_prob, const DLTensor* rpn_bbox,
                              const od_frcnn_params* params, DLTensor* proposals, DLTensor* num_out,
                              void* ws, size_t ws_bytes, void* stream);

/* feature_map [B,h,w,D] f32, proposals [n,5] f32 rows (batch,x1,y1,x2,y2) in pixels;
 * out [n,7,7,D] = max_pool2x2(crop_and_resize(14x14)) with boxes / (H,W,H,W). */
int od_roi_pool_forward(const DLTensor* feature_map, const DLTensor* proposals,
                        float image_h, float image_w, DLTensor* out, void* stream);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif

#ifdef __cplusplus
}
#endif
#endif /* ODHEAD_H_ */
