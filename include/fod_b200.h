/*
 * fod_b200.h - C ABI of the B200-native support-guided detection head
 *              (Faster-OreFSDet hot path: correlation -> CenterNet2 proposal
 *              decode -> NMS -> relation ROI head -> class-wise NMS).
 *
 * The reference (MVME-HBUT/Faster-OreFSDet) has no native code of its own: every
 * stage below is a chain of ATen / torchvision calls made from Python.  Each
 * entry point names the reference lines it replaces (paths relative to the
 * reference root; "d2!/" = inside the vendored detectron2.7z).
 *
 * Conventions
 *   - plain C symbols, raw DEVICE pointers, explicit sizes; no torch types.
 *   - fp32 everywhere; index outputs are int64 (reference dtype) or int32 counts.
 *   - feature maps are NHWC ("channels-last": [N][H][W][128], channel innermost),
 *     128 channels (MODEL.FPN.OUT_CHANNELS).  A PyTorch NCHW tensor in
 *     torch.channels_last memory format has exactly this layout.
 *   - a "problem" is one (query image b, support class c) pair, p = b*C + c.
 *   - the caller owns every buffer; the library allocates nothing, keeps no
 *     global state (no device symbols are written: episode constants such as the
 *     support taps travel inside the launch parameters), never synchronises,
 *     never touches the default stream; every call is stream-ordered, re-entrant
 *     across streams and CUDA-graph capturable.
 *   - return value: FOD_OK or a negative FOD_ERR_* (fod_last_error() gives text).
 *     Data-dependent overflow of a fixed-capacity output is reported on the
 *     device in the caller's `status` word (FOD_STATUS_* bits) and must be
 *     checked after the caller's own final synchronisation.
 */
#ifndef FOD_B200_H
#define FOD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* fod_stream_t; /* == cudaStream_t */

#define FOD_CHANNELS 128
#define FOD_MAX_LEVELS 3
#define FOD_NMS_MAX_BOXES 8192 /* per problem, limit of the in-smem sort */

enum {
  FOD_OK = 0,
  FOD_ERR_BAD_ARG = -1,
  FOD_ERR_CAPACITY = -2,   /* a static capacity argument exceeds a kernel limit */
  FOD_ERR_CUDA = -3,       /* a CUDA runtime call failed; see fod_last_error */
  FOD_ERR_UNSUPPORTED = -4 /* device is not sm_100 */
};

/* bits of the device-side status word */
#define FOD_STATUS_CAND_OVERFLOW 1u     /* fod_decode_topk: more candidates than cand_cap   */
#define FOD_STATUS_PROPOSAL_OVERFLOW 2u /* fod_nms_proposals: ties pushed R above roi_cap   */
#define FOD_STATUS_DET_OVERFLOW 4u      /* fod_final_detect: more rows than FOD_NMS_MAX_BOXES */

int fod_version(void);
/* copies the calling thread's last error text (NUL-terminated) into buf */
int fod_last_error(char* buf, size_t len);

/* One FPN level of a batch of NHWC maps. */
typedef struct {
  int height; /* H_l */
  int width;  /* W_l */
  int stride; /* 8, 16, 32 */
} fod_level_t;

/* ---------------------------------------------------------------------------
 * Q1  support taps.  Replaces the three nn.AdaptiveAvgPool2d calls per level per
 * class per image of fewx/modeling/fsod/fsod_cen.py:458-460, 476-479, 498-500.
 *   proto : [C][h][w][128] NHWC dense-head prototype of one level
 *   taps  : [C][7][128]  rows: k11, k13[0..2] (left, centre, right), k31[0..2] (up, centre, down)
 */
int fod_support_taps(const float* proto, int num_classes, int h, int w, float* taps, fod_stream_t stream);

/* ---------------------------------------------------------------------------
 * Q2+Q3  depthwise correlation + 1x1 relation conv, fused, for ALL FPN levels and all (image, class) problems in one
 * persistent launch (tcgen05 tensor cores, 3xTF32 operand splitting = fp32 accuracy, TMA in/out).
 * Replaces fsod_cen.py:463-470 (p3), :482-491 (p4), :502-509 (p5): four depthwise
 * F.conv2d + ReLUs + adds + torch.cat + self.conv3 + ReLU.
 * q and attn are HOST arrays of num_levels DEVICE pointers; taps is a HOST array of num_levels HOST pointers:
 *   q[l]    : [B][H_l][W_l][128]      query map of level l
 *   taps[l] : [C][7][128]  HOST        the output of fod_support_taps on the level-l prototype, read back once per
 *                                      episode.  The taps are warp-uniform operands of the stencil: they are copied
 *                                      into the launch parameters (constant bank 0, 6 sets = 24 KB per launch; classes
 *                                      are processed in groups of 6 / num_levels), so no device state outlives or is
 *                                      shared between calls, and a captured graph bakes in the episode's taps.
 *   w3      : [128][256]               conv3.weight (out, in) ; in = [attn-sum | q]
 *   b3      : [128]
 *   attn[l] : [B*C][H_l][W_l][128]     problem-major output
 *   attn_amax : NULL, or per level NULL / B*C DEVICE floats (zeroed by the caller): entry p is raised to max(attn[l] of
 *               problem p) - the per-image operand bound of the convolution that consumes the maps (fod_conv2d_nhwc
 *               x_amax with amax_per_image), without a pass over them
 */
int fod_correlate_levels(const float* const* q, const float* const* taps, const fod_level_t* levels, int num_levels,
                         const float* w3, const float* b3, float* const* attn, float* const* attn_amax, int batch,
                         int num_classes, fod_stream_t stream);

/* ---------------------------------------------------------------------------
 * D1+D2+D3  heat-map sigmoid, candidate threshold, per-level top-k, box decode,
 * level concatenation.  Replaces CenterNet.inference / predict_instances /
 * predict_single_level, fewx/modeling/fsod/fsod_rpn.py:1071-1074, 1100-1110,
 * 1116-1181 and compute_grids :782-800.
 *   hm[l]   : [P][H_l][W_l]           agn_hm output (logits if hm_is_logit, else sigmoid already applied)
 *   reg[l]  : [P][H_l][W_l][4] if reg_channels_last else [P][4][H_l][W_l]; relu(scale*bbox_pred), NOT yet x stride
 *   hm_pixel_stride / reg_pixel_stride : NULL (dense: 1 and 4), or HOST arrays of num_levels pixel strides in floats:
 *               hm[l] / reg[l] then point at their first channel inside a wider NHWC buffer (the fused agn_hm | bbox_pred
 *               convolution writes [P][H][W][8] = hm, l, t, r, b, 0, 0, 0); reg_pixel_stride needs reg_channels_last
 *   reg_scale : NULL, or a HOST array of num_levels floats (the CenterNetHead Scale factors, centernet_head.py:157-160):
 *               reg[l] then is the RAW bbox_pred output and the kernel applies relu(reg_scale[l] * x) as it reads it
 *   boxes   : [P][cand_cap][4]        candidates, level-major, ascending location inside a level
 *   scores  : [P][cand_cap]           sqrt(p)
 *   loc     : [P][cand_cap] int64     location index y*W+x inside its level
 *   level_count : [P][num_levels] int32 ; cand_count : [P] int32
 * Selection rule when a level has more than pre_topk candidates: every p above
 * the k-th largest plus the lowest-location ties at it (oracle/head_oracle.py).
 * cand_cap must be >= num_levels * pre_topk.
 */
int fod_decode_topk(const float* const* hm, const float* const* reg, const fod_level_t* levels, int num_levels,
                    int num_problems, int hm_is_logit, int reg_channels_last, const int* hm_pixel_stride,
                    const int* reg_pixel_stride, const float* reg_scale, float score_thresh, int pre_topk, int cand_cap, float* boxes, float* scores, int64_t* loc, int32_t* level_count,
                    int32_t* cand_count, uint32_t* status, fod_stream_t stream);

/* The same selection with the 3x3 output convolutions (agn_hm 128 -> 1, bbox_pred 128 -> 4,
 * CenterNet2/centernet/modeling/dense_heads/centernet_head.py:152-160) folded in.  A 3x3 convolution with 5 outputs keeps the
 * tensor cores busy for 36 K-chunks per tile whatever its width; computed instead as ONE 1x1 contraction
 *   G[p][tap]            = sum_c W_hm[c][ky][kx]     * t[p][c]     (tap = ky*3 + kx; columns 9..11 unused)
 *   G[p][12 + tap*4 + j] = sum_c W_reg[j][c][ky][kx] * t[p][c]     (j = l, t, r, b; 48 columns in all)
 * (fod_conv2d_nhwc, ksize 1, 4 K-chunks per tile) it leaves nine shifted additions per output, which this op does while
 * it reads:  out(y, x)[o] = bias5[o] + sum_tap G[(y + ky - 1, x + kx - 1)][column(o, tap)]  (zero outside the map).
 *   taps[l] : [P][H_l][W_l][tap_pixel_stride[l] >= 48, multiple of 4] fp32, 16-byte aligned (tap_pixel_stride NULL = 48)
 *   bias5   : HOST, agn_hm.bias then bbox_pred.bias;  reg_scale as in fod_decode_topk (HOST, may be NULL)
 *   workspace : fod_decode_topk_taps_workspace_bytes(levels, num_levels, num_problems) bytes of device memory (the keys
 *               of every pixel, formed by a wide first kernel; the selecting CTAs read them)
 * The heat-map is taken as a logit. */
size_t fod_decode_topk_taps_workspace_bytes(const fod_level_t* levels, int num_levels, int num_problems);
int fod_decode_topk_taps(const float* const* taps, const int* tap_pixel_stride, const float* bias5, const fod_level_t* levels,
                         int num_levels, int num_problems, const float* reg_scale, float score_thresh, int pre_topk,
                         int cand_cap, float* boxes, float* scores, int64_t* loc, int32_t* level_count, int32_t* cand_count,
                         uint32_t* status, void* workspace, fod_stream_t stream);

/* ---------------------------------------------------------------------------
 * N0  class-agnostic NMS + post-NMS top-k.  Replaces nms_and_topK -> ml_nms ->
 * batched_nms -> torchvision nms and the CPU kthvalue, fsod_rpn.py:1184-1210,
 * CenterNet2/centernet/modeling/layers/ml_nms.py:4-31, d2!/layers/nms.py:10-30.
 *   boxes/scores/count : candidate lists as written by fod_decode_topk
 *   keep      : [P][roi_cap] int64    indices into the candidate list, score-descending
 *   out_boxes : [P][roi_cap][4], out_scores : [P][roi_cap], out_count : [P] int32
 * Semantics: stable descending sort, greedy suppression when
 * inter/(area_i+area_j-inter) > iou_thresh (fp32 ratio, compared as double like
 * torchvision's CPU kernel), then if more than post_topk survive keep every
 * survivor whose score >= the post_topk-th best (ties kept).  post_topk <= 0
 * disables the second step.
 */
int fod_nms_proposals(const float* boxes, const float* scores, const int32_t* count, int num_problems, int cand_cap,
                      double iou_thresh, int post_topk, int roi_cap, int64_t* keep, float* out_boxes,
                      float* out_scores, int32_t* out_count, uint32_t* status, fod_stream_t stream);

/* ---------------------------------------------------------------------------
 * N2  RPN proposal selection of the Attention-RPN (FsodRPN.predict_proposals).  Replaces find_top_rpn_proposals,
 * d2!/modeling/proposal_generator/proposal_utils.py:19-119, with the decode of Box2BoxTransform.apply_deltas,
 * d2!/modeling/box_regression.py:77-115.  A problem is one image of one class's RPN output: problem p reads image p of
 * every level's map.  Per problem and level:
 *   1. select the top k = min(H*W*A, pre_topk) objectness logits: score descending, ties by ascending anchor index,
 *      NaN above +inf (torch.sort(descending=True) made stable);
 *   2. decode them against their anchors with the separate fp32 roundings of ATen (deltas / weights as a product with
 *      the fp32 reciprocal, dw / dh clamped at log(1000/16) before the exp);
 *   3. drop rows with a non-finite box or logit, clip to the problem's image (x to [0, w], y to [0, h]), keep width and
 *      height > min_size;
 * then over the levels: the NMS of fod_batched_nms (stable score-descending visit order, torchvision's IoU arithmetic,
 * boxes offset by level * (max coordinate + 1) when num_levels > 1), and the first post_topk survivors in visit order
 * (a strict cut: no tie extension, no status bit).
 *   maps[l]    : [P][H_l][W_l][pixel_stride[l] >= 5 * num_anchors] fp32, the stacked 1x1 output of StandardRPNHead read in
 *                place: logit of anchor a in channel a, delta j (dx, dy, dw, dh) in channel num_anchors + 4a + j
 *   anchors[l] : [H_l * W_l * num_anchors][4] xyxy fp32, 16-byte aligned (DefaultAnchorGenerator, (y, x, anchor) order)
 *   levels     : only height / width are read
 *   image_hw   : [P][2] int32 (height, width) DEVICE
 *   box_weights: HOST, 4 floats (RPN.BBOX_REG_WEIGHTS)
 *   out_boxes  : [P][post_topk][4] (16-byte aligned), out_logits [P][post_topk], out_count [P] int32; rows at or beyond
 *                out_count[p] are not written
 *   workspace  : fod_rpn_proposals_workspace_bytes(...) bytes of device memory, 16-byte aligned
 * The selected candidates of a problem, sum over l of min(H_l * W_l * num_anchors, pre_topk), must not exceed
 * FOD_NMS_MAX_BOXES (FOD_ERR_CAPACITY otherwise; the caller can check it from the shapes). */
size_t fod_rpn_proposals_workspace_bytes(const fod_level_t* levels, int num_levels, int num_problems, int num_anchors,
                                         int pre_topk);
int fod_rpn_proposals(const float* const* maps, const int* pixel_stride, const float* const* anchors,
                      const fod_level_t* levels, int num_levels, int num_problems, int num_anchors, const int32_t* image_hw,
                      int pre_topk, const float* box_weights, float min_size, double iou_thresh, int post_topk,
                      float* out_boxes, float* out_logits, int32_t* out_count, void* workspace, fod_stream_t stream);

/* ---------------------------------------------------------------------------
 * R1 / P1  multi-level ROIAlign (aligned=True, sampling_ratio=0) with FPN level
 * assignment.  Replaces ROIPooler.forward + assign_boxes_to_levels +
 * torchvision.ops.roi_align, d2!/modeling/poolers.py:22-58,190-250,
 * d2!/layers/roi_align.py:49-65; call sites fsod_roi_heads.py:470-472 and
 * fsod_cen.py:355-357 (support boxes).
 *   feat[l]  : [B][H_l][W_l][128]
 *   rois     : [P][roi_cap][4] xyxy in image pixels, roi_count [P] (NULL = all roi_cap valid)
 *   problems_per_image : C (ROI row p reads image p / C)
 *   pooled   : tiled == 0: [P][roi_cap][R*R][128] (bin-major, channel innermost); rows >= count untouched.
 *              tiled == 1 (R == 8; the input format of fod_relation_head): [P][U][256][128][32] with
 *              U = ceil(roi_cap/128): unit u = ROI rows 128u..128u+127, k-chunk kc = bin*4 + channel/32, so every
 *              [128 rows x 32 k] operand tile is 16 KB of contiguous memory (one linear TMA box).
 *   out_level: [P][roi_cap] int32 assigned level (may be NULL)
 */
/*   workspace : fod_roi_align_workspace_bytes(P, roi_cap, resolution) bytes, 16-byte aligned: per ROI the box geometry
 *              and the per-bin lists of distinct rows / columns with their interpolation weights, written by a
 *              pre-pass over all ROIs (one thread per axis and bin) and read by the pooling CTAs; for resolution 8
 *              also the per-ROI scan summaries and the list of ROIs the tile-stationary kernel hands to the per-ROI one */
size_t fod_roi_align_workspace_bytes(int num_problems, int roi_cap, int resolution);
int fod_roi_align(const float* const* feat, const fod_level_t* levels, int num_levels, int batch,
                  int problems_per_image, const float* rois, const int32_t* roi_count, int roi_cap, int resolution,
                  int tiled, float* pooled, int32_t* out_level, void* workspace, fod_stream_t stream);
/* The same pooling over maps with `channels` = a multiple of 128 channels per pixel (feat[l] : [B][H_l][W_l][channels]) and
 * resolution 4, 8 or 14: the ROIPooler of the R50-C4 heads (FsodRes5ROIHeads, fewx/modeling/fsod/fsod_roi_heads.py:69-74,
 * 119-126: 1024-channel res4, 14 x 14, one level).  pooled : [P][roi_cap][R*R][channels] (tiled must be 0 unless
 * channels == 128 and R == 8). */
int fod_roi_align_wide(const float* const* feat, const fod_level_t* levels, int num_levels, int batch,
                       int problems_per_image, const float* rois, const int32_t* roi_count, int roi_cap, int resolution,
                       int channels, int tiled, float* pooled, int32_t* out_level, void* workspace, fod_stream_t stream);

/* fod_roi_align / fod_roi_align_wide pool resolution 8 over 128-channel maps (the query path R1) with the
 * tile-stationary kernel: a CTA TMA-stages a 12 x 12-pixel piece of one map into shared memory and pools every bin
 * that starts inside its 8 x 8 owned pixels, so that a map pixel leaves L2 about twice per call instead of once per
 * ROI window that covers it.  Other shapes (resolution 4 / 14, wider maps) run one CTA per ROI.  This entry point
 * forces the one-CTA-per-ROI kernel for every shape: same arguments, same workspace, bit-identical results (the
 * summation order of a bin is the same) - kept as the comparison operator of the parity tests and the A/B timing. */
int fod_roi_align_per_roi(const float* const* feat, const fod_level_t* levels, int num_levels, int batch,
                          int problems_per_image, const float* rois, const int32_t* roi_count, int roi_cap,
                          int resolution, int channels, int tiled, float* pooled, int32_t* out_level, void* workspace,
                          fod_stream_t stream);

/* ---------------------------------------------------------------------------
 * R2+R3  relation head on pooled ROI features, softmax, box decoding.
 * Replaces CustomCascadeROIHeads._run_stage fsod_roi_heads.py:482-483,509-511,520
 * (conv3/conv1/conv2 1x1 + fc1 + cls_score/bbox_pred), predict_probs
 * CenterNet2/centernet/modeling/roi_heads/custom_fast_rcnn.py:160-170,
 * Box2BoxTransform.apply_deltas d2!/modeling/box_regression.py:77-115.
 * The three 1x1 convs and fc1 have no non-linearity between them and are folded
 * on the host into one [128][8192] matrix plus a per-class bias (DESIGN.md).
 * Tensor cores (tcgen05 kind::f16) with fp32 accuracy: both operands are scaled by a power of two and split into two
 * fp16 values, three MMAs per product (the arithmetic of fod_conv2d_nhwc), TMA-fed.
 *   pooled   : [P][U][256][128][32], the tiled layout of fod_roi_align (tiled = 1)
 *   x_amax   : n_amax (1..8) DEVICE floats bounding max|pooled|; ROIAlign averages bilinear samples, so the bounds of
 *              the feature maps it read (fod_conv2d_nhwc y_amax of the FPN output convolutions, or fod_absmax) hold.
 *              Any bound >= the true maximum gives the same result up to 2^-38 of the bound.
 *   amax_per_image : x_amax is [n_amax][B] (B = num_problems / problems_per_image) and the rows of image b are scaled
 *              with the maximum of column b: an image's scores do not depend on the other images of the batch
 *   w_fold_packed : fod_conv2d_pack_weights(w_fold as a [128][8192][1][1] convolution weight, ksize 1):
 *                  fod_conv2d_packed_floats(128, 8192, 1) floats; k index = bin*128 + channel (once per weight load)
 *   bias_cls : [C][128]      per-class folded bias (support term + fc1 bias)
 *   w_out    : [6][128], b_out [6] : rows 0-1 cls_score, rows 2-5 bbox_pred
 *   reg_weights : HOST pointer, 4 floats (wx, wy, ww, wh) = ROI_BOX_CASCADE_HEAD.BBOX_REG_WEIGHTS[0]
 *   det_boxes: [P][roi_cap][4] (unclipped), det_scores [P][roi_cap] (foreground probability)
 *   logits/deltas (optional, may be NULL): [P][roi_cap][2] / [P][roi_cap][4]
 * At most 2047 problems per call.
 */
int fod_relation_head(const float* pooled, const float* x_amax, int n_amax, int amax_per_image, const float* w_fold_packed,
                      const float* bias_cls, const float* w_out, const float* b_out, const float* rois,
                      const int32_t* roi_count, int num_problems, int problems_per_image, int roi_cap,
                      const float* reg_weights, float* det_boxes, float* det_scores, float* logits, float* deltas,
                      fod_stream_t stream);

/* ---------------------------------------------------------------------------
 * R4 / N1 / O1  final class-wise NMS, top-k, rescale to the output resolution.
 * Replaces fast_rcnn_inference_single_image d2!/modeling/roi_heads/fast_rcnn.py:118-171
 * (and its N-way sibling fewx/modeling/fsod/fsod_fast_rcnn.py:84-145) followed by
 * detector_postprocess d2!/modeling/postprocessing.py:9-75.
 *   det_boxes/det_scores/roi_count : per problem, as written by fod_relation_head
 *   rows of image b = problems b*C .. b*C+C-1 in class-major order
 *   out_hw : [B][2] int32 requested output (height, width); image_hw as above
 *   out_boxes [B][max_det][4], out_scores [B][max_det], out_classes [B][max_det] int64 (class index 0..C-1),
 *   out_rows [B][max_det] int64 (c*roi_cap + r of the source row), out_count [B] int32
 * Non-finite rows are dropped, boxes clipped to the image (Boxes.clip
 * d2!/structures/boxes.py:192-207), score > score_thresh kept, boxes offset by
 * class*(max_coordinate+1) (torchvision 0.8.2 batched_nms), greedy NMS, first
 * max_det; then scale/clip/drop-empty.
 */
int fod_final_detect(const float* det_boxes, const float* det_scores, const int32_t* roi_count, int batch,
                     int problems_per_image, int roi_cap, float score_thresh, double iou_thresh, int max_det,
                     const int32_t* image_hw, const int32_t* out_hw, float* out_boxes, float* out_scores,
                     int64_t* out_classes, int64_t* out_rows, int32_t* out_count, uint32_t* status,
                     fod_stream_t stream);

/* ---------------------------------------------------------------------------
 * Generic batched_nms (operator-level boundary, d2!/layers/nms.py:10-30):
 * one problem, boxes [n][4], scores [n], idxs [n] int64 (NULL = single class).
 * keep [n] int64 score-descending, keep_count [1] int32.
 */
int fod_batched_nms(const float* boxes, const float* scores, const int64_t* idxs, int n, double iou_thresh,
                    int64_t* keep, int32_t* keep_count, fod_stream_t stream);

/* ---------------------------------------------------------------------------
 * H0  3x3 / 1x1 convolution (stride 1, or stride 2 for 3x3) over NHWC fp32 maps, zero padding ksize/2, bias and
 * optional ReLU fused; tcgen05 tensor cores with fp32 accuracy (~4e-7 relative): every operand is scaled by a power
 * of two and split into two fp16 values, three kind::f16 MMAs per product, fp32 accumulation.
 * Replaces the F.conv2d -> cuDNN calls of CenterNetHead.forward
 * (CenterNet2/centernet/modeling/dense_heads/centernet_head.py:141-161: bbox_tower conv, agn_hm, bbox_pred) and of the
 * modules that hand maps to the head (d2!/modeling/backbone/vovnet.py:205-489 conv3x3/conv1x1 + FrozenBN folded,
 * d2!/modeling/backbone/fpn.py:113-155 lateral / output convs).
 *   x       : [N][H][W] pixels of x_pixel_stride floats, the first cin of them are read
 *             (a channel slice of a wider NHWC buffer is a valid input)
 *   x_amax  : n_amax (1..8) DEVICE floats, each an upper bound of max|x| over (part of) the input view; their maximum
 *             fixes the power-of-two operand scale.  Any bound >= the true maximum gives the same result up to 2^-38 of
 *             the bound; a bound below the true maximum may overflow fp16.  fod_absmax computes it; the kernel that
 *             produced x normally reports it (y_amax below).
 *   amax_per_image : bit 0: x_amax is [n_amax][N] and image n is scaled by the maximum of column n, so that the result of
 *             an image does not depend on which other images share the batch; bit 1: y_amax is [N], max|y| per image
 *               bit 2: x is PRE-SPLIT (written by fod_stem1_u8_tc_split / fod_conv2d_nhwc_split with y_bound = this x_amax): per
 *               pixel and 16 channels [16 x fp16 hi | 16 x fp16 lo] of x * 2^e; 3x3 stride-1 layers only, cin a multiple of 16, no
 *               a_gate / a_shift; the conversion pass is skipped
 *   packed  : fod_conv2d_pack_weights output (fod_conv2d_packed_floats floats)
 *   bias    : [cout] or NULL
 *   y       : [N][Ho][Wo] pixels of y_pixel_stride floats, the first cout are written
 *   y_amax  : NULL, or a DEVICE float (zeroed by the caller) that is atomically raised to max|y|
 *   residual: NULL, or a dense NHWC map with cout channels added to the convolution (+ bias) before the activation:
 *             [N][Ho][Wo][cout], or with residual_upsample2 [N][ceil(Ho/2)][ceil(Wo/2)][cout] read at (oy/2, ox/2) -
 *             the nearest-neighbour 2x upsampling + sum of the FPN top-down path (d2!/modeling/backbone/fpn.py:139-147)
 *   a_gate  : NULL, or [N][cin] factors multiplied into x before the convolution (cin a multiple of 32)
 *   a_shift : NULL, or [N][cin] added after the factor, then ReLU if a_relu; applied to pixels inside the image only (the
 *             zero padding stays zero)
 *   colsum  : NULL, or [N][tiles per image][cout]: receives the sum of y over each 8 x 16 output tile, per channel
 *   colsumsq: NULL, or the same for y^2 (needs colsum)
 * cin, cout and both pixel strides must be multiples of 4; pointers 16-byte aligned.
 */
size_t fod_conv2d_packed_floats(int cout, int cin, int ksize);
/* w_oihw : [cout][cin][ksize][ksize] (PyTorch conv weight) -> scaled fp16 hi / lo planes [cout][ky][kx][cin_pad] + scale */
int fod_conv2d_pack_weights(const float* w_oihw, int cout, int cin, int ksize, float* packed, fod_stream_t stream);
int fod_conv2d_nhwc(const float* x, int n, int h, int w, int cin, long x_pixel_stride, const float* x_amax, int n_amax,
                    int amax_per_image, const float* packed, const float* bias, int cout, int ksize, int stride, int relu, float* y,
                    long y_pixel_stride, float* y_amax, const float* residual, int residual_upsample2, const float* a_gate,
                    const float* a_shift, int a_relu, float* colsum, float* colsumsq, fod_stream_t stream);
/* Split hand-off between convolutions: fod_conv2d_nhwc whose OUTPUT can be written in the operand format of the
 * convolution that reads it (per pixel and 16 channels [16 x fp16 hi | 16 x fp16 lo] of y * 2^e, the format of
 * fod_stem1_u8_tc_split) and whose 1x1 form can READ a concat buffer in which the later slices were written that way.
 * The consumer of a pre-split map skips the fp32 -> fp16 hi / lo conversion of its input; bytes in HBM are unchanged.
 *   y_bound  : NULL (fp32 output), or [N] / [1] device floats (like x_amax): the output is written split at the scale
 *              derived from  y_l1 * max|x| + y_beta  >= max|y|  (y_l1 = max_c sum |w[c]|, y_beta = max |bias|; needs ReLU,
 *              cout and y_pixel_stride multiples of 16), and that bound is stored to y_bound[n] for the consumer
 *   x_actual : NULL, or the actual max|x| ([N] / [1]) to use in that product when x_amax is itself such a bound (pre-split
 *              x: amax_per_image bit 2 for a 3x3 layer) - bounds then do not compound along a chain of layers
 *   x_presplit_from / slice_ch : 1x1 (or stride-2) convolution, e.g. over a concat buffer: input channels >= x_presplit_from are pre-split;
 *              x_amax row k bounds the slice that starts at channel slice_ch[k] (k < n_amax, ascending, multiples of 16),
 *              each pre-split slice at the scale of its own row; -1 / NULL: none
 * residual, a_gate, a_shift and colsumsq of fod_conv2d_nhwc are not available here. */
int fod_conv2d_nhwc_split(const float* x, int n, int h, int w, int cin, long x_pixel_stride, const float* x_amax, int n_amax,
                          int amax_per_image, const float* packed, const float* bias, int cout, int ksize, int stride, int relu,
                          float* y, long y_pixel_stride, float* y_amax, float* colsum, const float* x_actual, float* y_bound,
                          float y_l1, float y_beta, int x_presplit_from, const int* slice_ch, fod_stream_t stream);

/* GroupNorm (+ ReLU) between two convolutions without materialising the normalised map (CenterNetHead tower,
 * centernet_head.py:61-72, 145-150): the first convolution writes colsum / colsumsq, fod_group_norm_affine turns them
 * into scale / shift [maps][channels] (and the bound max|normalised map| from the bound x_amax of the raw map), the
 * second convolution applies act(x * a_gate + a_shift) to its input operand (a_gate = scale, a_shift = shift, a_relu).
 * amax_per_map: x_amax and y_amax hold one bound per map ([maps]) instead of one for the batch. */
int fod_group_norm_affine(const float* colsum, const float* colsumsq, int maps, int tiles_per_map, int channels, int groups,
                          long hw, const float* gamma, const float* beta, float eps, const float* x_amax, float* scale,
                          float* shift, float* y_amax, int amax_per_map, fod_stream_t stream);
/* eSE attention of the OSA stages (d2!/modeling/backbone/vovnet.py eSEModule: x * hsigmoid(fc(avg_pool(x)))) without a
 * pass over x: the convolution that produces x writes per-tile channel sums (colsum), fod_ese_gate turns them into
 * gate [N][C] = relu6(fc(mean) + 3) / 6, and the consumers multiply it in (fod_conv2d_nhwc a_gate, fod_maxpool3x3s2_nhwc gate).
 *   colsum : [N][fod_conv2d_tiles_per_image(Ho, Wo)][C]   fc_weight [C][C], fc_bias [C]   hw = Ho * Wo
 *   C a multiple of 4 (<= 1024), colsum 16-byte aligned; the summation order is fixed, gates do not depend on the grid */
int fod_conv2d_tiles_per_image(int ho, int wo);
int fod_ese_gate(const float* colsum, int n, int tiles_per_img, int channels, long hw, const float* fc_weight,
                 const float* fc_bias, float* gate, fod_stream_t stream);
/* max |x| of a dense fp32 array -> *out (device float; zeroed inside) */
int fod_absmax(const float* x, size_t n, float* out, fod_stream_t stream);
/* max |x| of each of `rows` arrays of row_len floats laid end to end (one per image of a batch) -> out[rows] (device
 * floats; zeroed inside): the per-image operand bounds of fod_conv2d_nhwc (amax_per_image bit 0).  row_len a multiple of 4
 * when rows > 1. */
int fod_absmax_rows(const float* x, int rows, size_t row_len, float* out, fod_stream_t stream);

/* ---------------------------------------------------------------------------
 * H0  GroupNorm (+ ReLU) over NHWC maps: the normalisation of CenterNetHead's tower
 * (CenterNet2/centernet/modeling/dense_heads/centernet_head.py:61-72, 145-150,
 * nn.GroupNorm(32, 128) then nn.ReLU).  Statistics per (map, group) over H*W and the
 * group's channels, biased variance, fp64 accumulation across threads.
 *   x, y      : [maps][hw][channels] (y may alias x)
 *   gamma/beta: [channels] or NULL
 *   y_amax    : NULL, or a DEVICE float (zeroed by the caller) raised to max|y| (the bound fod_conv2d_nhwc needs); with
 *               amax_per_map [maps] floats, one bound per map
 *   workspace : fod_group_norm_workspace_bytes(maps, groups) bytes, 16-byte aligned
 * channels / groups must be a multiple of 4.
 */
size_t fod_group_norm_workspace_bytes(int maps, int groups);
int fod_group_norm_nhwc(const float* x, int maps, long hw, int channels, int groups, const float* gamma,
                        const float* beta, float eps, int relu, float* y, float* y_amax, int amax_per_map, void* workspace,
                        fod_stream_t stream);

/* ---------------------------------------------------------------------------
 * Glue of the feature extractor (d2!/modeling/backbone/vovnet.py), memory bound.
 * fod_stem_patches: im2col of stem_1 (3x3, stride 2, pad 1 over the 3-channel normalised image):
 *   x [N][H][W][3] NHWC  ->  patches [N][ceil(H/2)][ceil(W/2)][32], k = (ky*3+kx)*3 + c, k >= 27 zero;
 *   stem_1 then is fod_conv2d_nhwc(ksize 1, cin 32) with the weight rows in the same order.
 * fod_maxpool3x3s2_nhwc: nn.MaxPool2d(kernel 3, stride 2, ceil_mode=True) of the OSA stages; `gate` (NULL or
 *   [N][C] >= 0) multiplies the result per (image, channel): the eSE gate of the producing stage.  x / y may be
 *   channel slices of wider NHWC buffers (pixel strides in floats).  Output size ceil((H-3)/2)+1.
 */
int fod_stem_patches(const float* x, int n, int h, int w, float* patches, fod_stream_t stream);
/* the same rows from the raw uint8 planar image batch x [N][3][H][W], normalised on the fly as (x - mean[c]) / std[c]
 * (CenterNet2Detector.preprocess_image, fewx/modeling/fsod/fsod_cen.py:540-555); mean3 / std3 are HOST arrays of 3 floats */
int fod_stem_patches_u8(const uint8_t* x, int n, int h, int w, const float* mean3, const float* std3, float* patches,
                        fod_stream_t stream);
/* stem_1 in one pass (CUDA cores, fp32 FMA): raw uint8 planar batch x [N][3][H][W] -> (x - mean)/std -> 3x3 / stride 2 /
 * pad 1 convolution, 64 output channels, weight [64][3][3][3] (OIHW, FrozenBN folded), bias [64] or NULL -> ReLU ->
 * y [N][ceil(H/2)][ceil(W/2)][64] NHWC; y_amax as in fod_conv2d_nhwc ([N] floats with amax_per_image).  (d2!/modeling/backbone/vovnet.py stem_1 +
 * fsod_cen.py:540-555) */
int fod_stem1_u8(const uint8_t* x, int n, int h, int w, const float* mean3, const float* std3, const float* weight,
                 const float* bias, float* y, float* y_amax, int amax_per_image, fod_stream_t stream);
/* the same layer on the tensor cores (csrc/stem1_tc.cu): a GEMM with ONE 32-wide K chunk per 128-pixel tile whose A
 * operand - the 27 im2col columns k = (ky*3 + kx)*3 + c of an output pixel, normalised, zero outside the image - is gathered
 * from the uint8 planes straight into tensor memory, so the layer is bound by its 256-byte-per-pixel output write
 * instead of by FP32 FMAs.  Same arithmetic as fod_conv2d_nhwc (fp16 hi / lo split, fp32 accumulation); the operand scale
 * is fixed by mean3 / std3, so an image's result does not depend on the batch.
 *   packed : fod_conv2d_pack_weights of the [64][32][1][1] matrix (columns in the order above, 27..31 zero; BN folded)
 *   y      : [N][ceil(H/2)][ceil(W/2)][y_pixel_stride >= 64] NHWC; y_amax as in fod_stem1_u8 */
int fod_stem1_u8_tc(const uint8_t* x, int n, int h, int w, const float* mean3, const float* std3, const float* packed,
                    const float* bias, float* y, long y_pixel_stride, float* y_amax, int amax_per_image, fod_stream_t stream);
/* fod_stem1_u8_tc with the output written in the OPERAND FORMAT of the 3x3 convolution that reads it instead of fp32:
 * per pixel and group of 16 channels 64 bytes = [16 x fp16 hi | 16 x fp16 lo] of y * 2^e (hi = fp16(y * 2^e), lo the
 * exact remainder rounded to fp16), 2^e = the scale fod_conv2d_nhwc derives from a bound on max|y|.
 *   y_bound : ONE device float >= every output value; it is known before the layer runs: the pixel range is
 *             [0, 255], so max_c (sum_k |w[c][k]| * max(|0 - mean|, |255 - mean|) / std + |bias[c]|) holds for every image.
 * The consumer is fod_conv2d_nhwc(x = y, x_amax = y_bound, n_amax = 1, amax_per_image bit 2 set): it skips the in-place
 * conversion pass of every staged tile (and the barrier behind it).  Same bytes in HBM, same accuracy class (22
 * significant bits relative to the bound), results independent of the batch (the scale depends on weights only).
 * y_amax still receives max(y) of the fp32 values. */
int fod_stem1_u8_tc_split(const uint8_t* x, int n, int h, int w, const float* mean3, const float* std3, const float* packed,
                          const float* bias, float* y, long y_pixel_stride, float* y_amax, int amax_per_image,
                          const float* y_bound, fod_stream_t stream);

int fod_maxpool3x3s2_nhwc(const float* x, int n, int h, int w, int c, long x_pixel_stride, const float* gate, float* y,
                          long y_pixel_stride, fod_stream_t stream);
/* the same pooling with the output in the split hand-off format of fod_conv2d_nhwc_split (per 16 channels [16 x fp16 hi |
 * 16 x fp16 lo] of y * 2^e): y_bound [N] device floats >= max|x| of each image (the y_amax of the convolution that wrote x;
 * the gate is <= 1, so it bounds the pooled map too); c and y_pixel_stride multiples of 16.  The readers are
 * fod_conv2d_nhwc with x_amax = y_bound and amax_per_image bit 2 (3x3) or x_presplit_from (1x1). */
int fod_maxpool3x3s2_nhwc_split(const float* x, int n, int h, int w, int c, long x_pixel_stride, const float* gate, float* y,
                                long y_pixel_stride, const float* y_bound, fod_stream_t stream);


#ifdef __cplusplus
}
#endif
#endif /* FOD_B200_H */
