/*
 * yolonano_b200.h — C ABI of the B200-native YOLO-Nano-1.0x detection forward path.
 *
 * The reference (yjh0410/YOLO-Nano) is pure Python and has no FFI of its own; the
 * boundary this library sits behind is the Python class `models.yolo_nano.YOLONano`
 * (models/yolo_nano.py:12) — see INTEGRATION.md for the ctypes stub a maintainer adds.
 * Every entry point below names the reference code it replaces (file:line under the
 * reference tree).
 *
 * Conventions
 *   - plain C symbols, opaque handle, `int` status (0 = YNB_OK), message via
 *     ynb_last_error(); no torch / C++ types cross the boundary.
 *   - all `*_dev` pointers are device pointers on the engine's GPU, owned by the caller
 *     (PyTorch allocations passed as raw addresses); `stream` is a cudaStream_t passed
 *     as void* (NULL = legacy default stream).  Calls are asynchronous on that stream
 *     unless stated otherwise.
 *   - one handle per (GPU, stream); a handle is not thread-safe; there is no global state.
 *   - tensors are float32.  Public image input is NCHW [B,3,S,S] exactly as the
 *     reference takes it; internal activations are NHWC.
 *   - there is NO CPU implementation behind any of these calls: without a usable
 *     sm_100 device ynb_create fails with YNB_ERR_NO_DEVICE.
 */
#ifndef YOLONANO_B200_H_
#define YOLONANO_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YNB_ABI_VERSION 1

/* status codes */
#define YNB_OK               0
#define YNB_ERR_INVALID      1   /* bad argument / shape                          */
#define YNB_ERR_NO_DEVICE    2   /* no CUDA device, or not compute capability 10  */
#define YNB_ERR_CUDA         3   /* a CUDA runtime / driver call failed           */
#define YNB_ERR_STATE        4   /* call order (weights not committed, ...)       */
#define YNB_ERR_UNSUPPORTED  5

/* activation codes (utils/modules.py:14, backbone/shufflenetv2.py:48) */
#define YNB_ACT_NONE  0
#define YNB_ACT_RELU  1
#define YNB_ACT_LEAKY 2          /* LeakyReLU(0.1) */

/* arithmetic mode of the dense contractions (1x1 and 3x3 convs) */
#define YNB_GEMM_FP32_FFMA   0   /* CUDA-core fp32 FMA (debug / cross-check path)            */
#define YNB_GEMM_TC_3XTF32   1   /* tcgen05 kind::tf32, 3-term split: fp32 parity mode        */
#define YNB_GEMM_TC_TF32     2   /* tcgen05 kind::tf32 single pass: throughput mode           */
#define YNB_GEMM_TC_BF16     3   /* bf16 activations + weights in HBM, tcgen05 kind::f16, fp32 accumulate:
                                    throughput mode of BASELINE configs[3] (tolerance reported separately) */

typedef struct ynb_engine ynb_engine;

/* Mirrors the constructor arguments of YOLONano (models/yolo_nano.py:13). */
typedef struct ynb_config {
  int32_t abi_version;        /* must be YNB_ABI_VERSION                                    */
  int32_t device;             /* CUDA device ordinal                                        */
  int32_t input_size;         /* S, multiple of 32                                          */
  int32_t num_classes;        /* C (20 VOC / 80 COCO)                                       */
  int32_t num_anchors;        /* A = len(anchor_size)//3 (models/yolo_nano.py:24-25), 3      */
  float   anchors[18];        /* [level][anchor][w,h] pixels (data/config.py:11-17)          */
  float   conf_thresh;        /* models/yolo_nano.py:13 default 0.001                       */
  float   nms_thresh;         /* default 0.5                                                */
  int32_t diou_nms;           /* 0: nms (:159-188), 1: diou_nms (:191-242)                   */
  int32_t gemm_mode;          /* YNB_GEMM_*                                                 */
  int32_t max_batch;          /* workspace is planned for this many images per call         */
} ynb_config;

/* ---- lifecycle ------------------------------------------------------------------ */

/* Replaces YOLONano.__init__ (models/yolo_nano.py:13-74) minus parameter creation. */
int  ynb_create(const ynb_config* cfg, ynb_engine** out);
void ynb_destroy(ynb_engine* e);
/* Message of the last failing call on `e`; with e == NULL, of the last failing ynb_create. */
const char* ynb_last_error(const ynb_engine* e);
int  ynb_abi_version(void);

/* Replaces YOLONano.set_grid / create_grid (models/yolo_nano.py:86-117): the grid is
 * analytic in the kernels, so this only re-plans the workspace for the new S. */
int  ynb_set_grid(ynb_engine* e, int32_t input_size);
/* conf_thresh / nms_thresh / diou_nms are mutable attributes in the reference. */
int  ynb_set_thresholds(ynb_engine* e, float conf_thresh, float nms_thresh, int32_t diou_nms);
int  ynb_set_gemm_mode(ynb_engine* e, int32_t gemm_mode);
/* Boxes per image N = A*(S/8)^2 + A*(S/16)^2 + A*(S/32)^2 for the current grid. */
int64_t ynb_num_boxes(const ynb_engine* e);
/* Bytes of device workspace the engine holds for `batch` images at the current S. */
int64_t ynb_workspace_bytes(const ynb_engine* e, int32_t batch);

/* ---- weights ---------------------------------------------------------------------- */

/* The 77 convolutions of the path in engine order; names are the reference
 * state_dict prefixes ("backbone.stage2.0.branch2.3", "head_det_1.4", ...). */
int32_t     ynb_num_convs(void);
const char* ynb_conv_name(int32_t index);
/* weight shape [cout, cin_per_group, k, k] of conv `index` for a given class count. */
int  ynb_conv_shape(int32_t index, int32_t num_classes, int32_t num_anchors,
                    int32_t* cout, int32_t* cin_per_group, int32_t* ksize);

/* Hands one conv's weights to the engine: `w_host` is the reference layout
 * [cout, cin/groups, k, k] with BatchNorm already folded exactly as
 * utils/fuse_conv_bn.py:6-22 does, `b_host` the folded bias [cout].  Host pointers;
 * copied before return. */
int  ynb_load_conv(ynb_engine* e, const char* name,
                   const float* w_host, int64_t w_elems,
                   const float* b_host, int64_t b_elems);
/* Packs all 77 convs into the device layouts the kernels read (permuted / padded /
 * tf32-split) and uploads them.  Synchronous. */
int  ynb_commit_weights(ynb_engine* e);

/* ---- the hot path ----------------------------------------------------------------- */

/* backbone + neck + heads, raw head outputs in the reference's NCHW order
 * [B, A*(1+C+4), H, W] for the three levels (models/yolo_nano.py:284-301).
 * Parity hook. */
int  ynb_forward_raw(ynb_engine* e, const float* x_dev, int32_t batch,
                     float* pred_s_dev, float* pred_m_dev, float* pred_l_dev, void* stream);

/* ... + re-layout, sigmoid/softmax, box decode, /S, clamp, class argmax
 * (models/yolo_nano.py:303-330, 362-367, 253-256) for EVERY image of the batch:
 *   boxes_dev  [B,N,4] x1y1x2y2 in [0,1];  scores_dev [B,N] = max_c softmax*obj;
 *   cls_dev    [B,N] int32 argmax (first max wins).
 * Parity hook for the decode stage (no threshold, no NMS). */
int  ynb_forward_decode(ynb_engine* e, const float* x_dev, int32_t batch,
                        float* boxes_dev, float* scores_dev, int32_t* cls_dev, void* stream);

/* The whole path of YOLONano.forward in eval mode (models/yolo_nano.py:282-376):
 * backbone, neck, heads, decode, score threshold, per-class (DIoU-)NMS — for every
 * image.  Outputs are compacted per image in ascending anchor order:
 *   out_boxes_dev [B,N,4], out_scores_dev [B,N], out_cls_dev [B,N] (first counts[b]
 *   rows of image b valid), out_counts_dev [B] int32. */
int  ynb_forward_detect(ynb_engine* e, const float* x_dev, int32_t batch,
                        float* out_boxes_dev, float* out_scores_dev, int32_t* out_cls_dev,
                        int32_t* out_counts_dev, void* stream);

/* Same, with HOST buffers: x_host [B,3,S,S] (pinned memory recommended), results
 * written to host arrays of the shapes above; host<->device copies are issued on
 * `stream` and the call returns after they completed (the reference's own boundary
 * is also synchronous: `.to('cpu').numpy()`, models/yolo_nano.py:370-371). */
int  ynb_detect_host(ynb_engine* e, const float* x_host, int32_t batch,
                     float* out_boxes_host, float* out_scores_host, int32_t* out_cls_host,
                     int32_t* out_counts_host, void* stream);

/* The same in two halves, double-buffered (slot 0 | 1), so that a stream of batches overlaps
 * the PCIe copy of batch i+1 with the computation of batch i:
 *   ynb_submit_host(slot)  enqueues H2D (copy stream) + the whole path (compute stream);
 *   ynb_wait_host(slot)    blocks until that step finished and its kept rows are in the
 *                          host arrays given to submit.  ynb_detect_host == submit + wait. */
int  ynb_submit_host(ynb_engine* e, int32_t slot, const float* x_host, int32_t batch,
                     float* out_boxes_host, float* out_scores_host, int32_t* out_cls_host,
                     int32_t* out_counts_host, void* stream);
int  ynb_wait_host(ynb_engine* e, int32_t slot);

/* ---- pre-processing on the device (SURVEY 8f row 1) ---------------------------------------
 * The tail of ValTransforms (data/transforms.py:445-458): Normalize (:59-70: float32(u8) / 255,
 * - mean, / std, channel-wise in BGR order), ToTensor (:394-398: BGR -> RGB, HWC -> CHW) and the
 * padding value of Resize (:73-119: mean * 255 outside the letterboxed content).  cv2.resize itself
 * stays on the host: img is uint8 [B,S,S,3] BGR already resized / letterboxed to S x S; rects
 * [B][4] = (x0, y0, w, h) of the content inside the canvas (NULL = the whole canvas).  The result is
 * bit-identical to the reference's tensor (the normalisation is a 3 x 256 table computed with the
 * reference's float32 sequence).  Inputs cross PCIe as 1 byte per element instead of 4. */
int  ynb_set_normalization(ynb_engine* e, const float* mean_bgr /*[3]*/, const float* std_bgr /*[3]*/);
int  ynb_preprocess_u8(ynb_engine* e, const uint8_t* img_dev, const int32_t* rects_dev, int32_t batch,
                       float* x_dev /*[B,3,S,S]*/, void* stream);
/* Test-time augmentation input (utils/misc.py:104-121): torch.nn.functional.interpolate(x, (s, s),
 * mode='bilinear', align_corners=False) of a float32 NCHW batch [B,3,h,w] and, with_flip != 0, the
 * torch.flip(.., [-1]) copy: out [B or 2B, 3, s, s] with out[2b] = resized, out[2b+1] = flipped. */
int  ynb_resize_bilinear(const float* in_dev, int32_t batch, int32_t h_in, int32_t w_in, float* out_dev,
                         int32_t s_out, int32_t with_flip, void* stream);
/* ynb_submit_host with uint8 images: H2D of the bytes + pre-processing + the whole path. */
int  ynb_submit_host_u8(ynb_engine* e, int32_t slot, const uint8_t* img_host, const int32_t* rects_host,
                        int32_t batch, float* out_boxes_host, float* out_scores_host,
                        int32_t* out_cls_host, int32_t* out_counts_host, void* stream);

/* After any ynb_forward_*: copy an internal activation as canonical NCHW float32 into
 * out_dev.  Names: "pool", "c3", "c4", "c5", "p3", "p4", "p5", and every backbone
 * block output "stage2.0" ... "stage4.3".  Per-layer parity hook (SURVEY §8c hazard 1). */
int  ynb_read_tap(ynb_engine* e, const char* tap, int32_t batch, float* out_dev, void* stream);
/* Shape [C,H,W] of a tap at the current grid. */
int  ynb_tap_shape(const ynb_engine* e, const char* tap, int32_t* c, int32_t* h, int32_t* w);

/* Number of kernels the engine launched since creation (bench.py's gpu_launches). */
int64_t ynb_launch_count(const ynb_engine* e);

/* Per-kernel timing for the roofline report: with profiling on, every launch of the next
 * ynb_forward_* is bracketed by CUDA events on the launching stream (the call then
 * synchronises).  Entries: launch label (reference conv name), kernel family, elapsed
 * ms, ALGORITHMIC bytes (unique unpadded inputs + outputs + weights) and flops. */
int  ynb_set_profiling(ynb_engine* e, int32_t on);
int32_t ynb_profile_count(const ynb_engine* e);
int  ynb_profile_entry(const ynb_engine* e, int32_t index, const char** name, const char** kind,
                       float* ms, double* bytes, double* flops);

/* ---- individually callable kernels (unit parity + ncu) ------------------------------
 * All take NHWC float32 device tensors with explicit channel strides (ld = floats
 * between consecutive pixels) so that channel sub-ranges of a wider tensor can be
 * read / written in place: that is how chunk / cat / channel_shuffle
 * (backbone/shufflenetv2.py:14-28,70-76) cost nothing. */

/* Depthwise 3x3, pad 1, stride 1|2, + bias + activation
 * (backbone/shufflenetv2.py:66-67 + folded BN; models/yolo_nano.py:51 for the heads).
 * w_dev is [9][C] (tap-major), b_dev [C].
 *   out[b,y,x, out_off + c*out_step] = act(b[c] + sum_t w[t][c] * in[b, y*s+dy-1, x*s+dx-1, in_off + c]) */
int  ynb_dwconv3x3(const float* in_dev, int32_t in_ld, int32_t in_off,
                   float* out_dev, int32_t out_ld, int32_t out_off, int32_t out_step,
                   const float* w_dev, const float* b_dev,
                   int32_t batch, int32_t h_in, int32_t w_in, int32_t channels,
                   int32_t stride, int32_t act, void* stream);

/* Whole ValTransforms on the device (data/transforms.py:73-119, 59-70, 394-398, 445-458): letterbox Resize
 * (cv2.resize bilinear, restated bit-exactly, + padding with mean*255) + Normalize + ToTensor from the ORIGINAL
 * uint8 BGR images of any shapes (tightly packed h0 x w0 x 3, one after the other in src_dev) to the float32
 * [batch,3,S,S] tensor of the engine's current grid size.  The caller fills one descriptor per image exactly as
 * Resize computes its geometry (yolo_nano_b200/engine.py: letterbox_desc). */
typedef struct ynb_image_desc {
  int64_t offset;            /* byte offset of the image in src_dev                                   */
  int32_t h0, w0;            /* source size                                                           */
  int32_t nw, nh;            /* content size on the S x S canvas: (int(w0/h0*S), S) | (S, int(h0/w0*S)) | (S, S) */
  int32_t left, top;         /* content position: ((nh-nw)//2, 0) | (0, (nw-nh)//2) | (0, 0)           */
  int32_t mode;              /* 0: copy (h0 == w0 == S), 1: bilinear, 2: exact 2x downscale (2x2 mean) */
  int32_t reserved;
  double  scale_x, scale_y;  /* 1 / (nw / w0), 1 / (nh / h0) in float64                               */
} ynb_image_desc;
int  ynb_preprocess_letterbox_u8(ynb_engine* e, const uint8_t* src_dev, const ynb_image_desc* descs_dev,
                                 int32_t batch, float* x_dev, void* stream);

/* The evaluators' inverse box mapping (evaluator/cocoapi_evaluator.py:85-87, test.py:133-135) on the NMS output,
 * in place:  boxes = ((boxes - offset) / scale) * size  with the reference's float64-operand roundings.
 * boxes_dev [batch][n_per_image][4], counts_dev [batch], maps_dev [batch][12] = offset[4], scale[4], size[4]. */
int  ynb_map_boxes(float* boxes_dev, const int32_t* counts_dev, const double* maps_dev, int32_t batch,
                   int64_t n_per_image, void* stream);

/* VOC mAP on the device (evaluator/vocapi_evaluator.py: write_voc_results_file + voc_eval + voc_ap, ssd.pytorch
 * lineage: overlaps without the +1 pixel, ap = -1 for a class without detection lines).
 *
 * ynb_voc_append turns the kept rows of a batch (after ynb_map_boxes: pixel boxes [batch][n_per_image][4], scores
 * [batch][n_per_image], cls [batch][n_per_image], counts [batch]) into det-file lines, one int32 row each:
 *     rows_dev[slot] = {image_base + b, class, milli, x1, y1, x2, y2}
 * milli is the integer of '{:.3f}' of the score and xk the integer of '{:.1f}' of (box_k + 1), the +1 added in
 * float32; both round half-even on the exact binary value like Python's formatting, so milli / 1000.0 and
 * xk / 10.0 are the doubles voc_eval parses back.  A '-0.0' field is stored as INT32_MIN.  Slots follow file order
 * (image, then kept row): state_dev[0] (int64, zeroed by the caller before the first batch) holds the rows
 * appended so far and is advanced on the device; rows at or past `capacity` are counted but not written.
 * state_dev[1] counts rejected values (class out of range, score outside [0, 1], non-finite or |box + 1| >= 2^27);
 * their rows are written clamped, and the caller must not evaluate them. */
int  ynb_voc_append(const float* boxes_dev, const float* scores_dev, const int32_t* cls_dev,
                    const int32_t* counts_dev, int32_t batch, int64_t n_per_image, int32_t image_base,
                    int32_t num_classes, int32_t* rows_dev, int64_t capacity, int64_t* state_dev, void* stream);

/* voc_eval of every class over rows_dev[0, n_rows) (the caller reads n_rows from state_dev[0] and checks it
 * against the capacity).  Ground truth in voc_eval's coordinates, bucketed by (image, class) in annotation order:
 * GT g has gt_boxes_dev[g][4] (float64 x1, y1, x2, y2) and gt_difficult_dev[g]; bucket (i, c) is
 * [gt_start_dev[i * num_classes + c], gt_start_dev[i * num_classes + c + 1]), gt_start_dev has
 * num_images * num_classes + 1 entries.  Detections are ordered by score descending, ties by file order; a
 * detection is TP when its best overlap (> ovthresh, strict) hits a non-difficult GT that no earlier detection
 * claimed, ignored on a difficult one.  Outputs: ap_dev [num_classes] float64 (VOC07 11-point when use_07_metric,
 * else the area under the precision envelope; -1 for a class without rows), npos_dev [num_classes] (non-difficult
 * GT per class); optional (NULL to skip) order_dev [n_rows] = arena row of each sorted position and flags_dev
 * [n_rows] = 1 TP, 2 FP, 0 ignored per sorted position.  Deterministic. */
int64_t ynb_voc_eval_workspace_bytes(int64_t n_rows, int32_t num_classes, int64_t n_gt);
int  ynb_voc_eval(const int32_t* rows_dev, int64_t n_rows, int32_t num_classes, int32_t num_images,
                  const double* gt_boxes_dev, const uint8_t* gt_difficult_dev, const int32_t* gt_start_dev,
                  int64_t n_gt, double ovthresh, int32_t use_07_metric, double* ap_dev, int32_t* npos_dev,
                  int32_t* order_dev, int8_t* flags_dev, void* workspace_dev, int64_t workspace_bytes,
                  void* stream);

/* Pointwise 1x1 conv = GEMM over pixels, + bias + activation, fp32 FFMA variant
 * (backbone/shufflenetv2.py:46,54,60; utils/modules.py:11 with k=1).
 * w_dev is [cout][cin] row-major, b_dev [cout].
 *   out[m, out_off + n*out_step] = act(b[n] + sum_k w[n][k] * in[m, in_off + k]) */
int  ynb_pwconv(const float* in_dev, int32_t in_ld, int32_t in_off,
                float* out_dev, int32_t out_ld, int32_t out_off, int32_t out_step,
                const float* w_dev, const float* b_dev,
                int64_t pixels, int32_t cin, int32_t cout, int32_t act, void* stream);

/* Same contraction on tcgen05 tensor cores (TMA-fed, TMEM accumulators);
 * mode = YNB_GEMM_TC_3XTF32 | YNB_GEMM_TC_TF32.  Requires in_ld, in_off, out_ld,
 * out_off multiples of 4 floats. */
int  ynb_pwconv_tc(const float* in_dev, int32_t in_ld, int32_t in_off,
                   float* out_dev, int32_t out_ld, int32_t out_off, int32_t out_step,
                   const float* w_dev, const float* b_dev,
                   int64_t pixels, int32_t cin, int32_t cout, int32_t act,
                   int32_t mode, void* stream);

/* Fused unit tail: depthwise 3x3 (stride 1, pad 1) + bias (+ dw_act) kept in shared memory as the A operand of
 * the pointwise 1x1 conv on tcgen05, + bias + act; one launch (yolo_nano_b200/csrc/unit_tc.cuh).  Replaces
 * branch2[3..7] of a stride-1 ShuffleV2Block (backbone/shufflenetv2.py:57-63) and, with pass_dev != NULL, the
 * torch.cat + channel_shuffle that follow it (:70-76, 14-28):
 *     out[m, 2i] = pass[m, i],  out[m, 2i+1] = act(pw(dw(in)))[m, i]          (out_ld >= 2*cout)
 * and a (depthwise Conv, pointwise Conv) pair of a detection head (models/yolo_nano.py:50-58) with
 * pass_dev == NULL: out[m, i] = act(pw(dw_act(dw(in))))[m, i].
 * in_dev: NHWC view [batch][h][w][channels of in_ld], 16-byte aligned, channels % 4 == 0; dw_w_dev [9][channels]
 * tap-major, dw_b_dev [channels]; pw_w_dev [cout][channels], pw_b_dev [cout]; cout <= 128; out_dev / pass_dev
 * 16-byte aligned with out_ld, pass_ld multiples of 4 floats.
 * mode = YNB_GEMM_TC_3XTF32 | YNB_GEMM_TC_TF32 | YNB_GEMM_TC_BF16.  In bf16 mode in_dev, out_dev and pass_dev hold
 * bf16 elements (in_ld, out_ld, channels multiples of 8; cout <= 240), the pointwise weights are rounded to bf16 and
 * the depthwise output is rounded to bf16 before the GEMM; dw_w_dev, dw_b_dev, pw_b_dev stay float32.  Rows are
 * written in whole 16-byte chunks there: with pass_dev, elements [2*cout, round_up(2*cout, 8)) of a row may be written.
 * Synchronous test hook (packs the weights on the host). */
int  ynb_dwpw_tc(const float* in_dev, int32_t in_ld, const float* dw_w_dev, const float* dw_b_dev, int32_t dw_act,
                 const float* pw_w_dev, const float* pw_b_dev, int32_t act,
                 float* out_dev, int32_t out_ld, const float* pass_dev, int32_t pass_ld,
                 int32_t batch, int32_t h, int32_t w, int32_t channels, int32_t cout, int32_t mode, void* stream);

/* Stem: Conv2d(3,24,3,2,1)+BN+ReLU then MaxPool2d(3,2,1), fused
 * (backbone/shufflenetv2.py:109-116,158-159).  x_dev NCHW [B,3,S,S];
 * out_dev NHWC [B,S/4,S/4,24]; w_dev [27][24] ((ci,ky,kx)-major), b_dev [24]. */
int  ynb_stem_pool(const float* x_dev, float* out_dev, const float* w_dev, const float* b_dev,
                   int32_t batch, int32_t input_size, void* stream);

/* Decode of raw head outputs (models/yolo_nano.py:120-156, 303-330, 362-367, 253-256).
 * raw_dev is NHWC [B, H*W, ld] for ONE level with the reference channel map
 * (obj a | cls a*C+c | box 4a+k).  Writes rows [level_off, level_off + H*W*A) of
 * boxes_dev [B,N,4], scores_dev [B,N], cls_dev [B,N]. */
int  ynb_decode_level(const float* raw_dev, int32_t raw_ld,
                      float* boxes_dev, float* scores_dev, int32_t* cls_dev,
                      int32_t batch, int32_t grid, int32_t stride_px, int32_t input_size,
                      const float* anchors_wh /* host, A*2 */, int32_t num_anchors,
                      int32_t num_classes, int64_t boxes_per_image, int64_t level_off,
                      void* stream);

/* Threshold + per-image per-class greedy NMS (models/yolo_nano.py:159-279) on decoded
 * candidates.  Inputs boxes_dev [B,N,4], scores_dev [B,N], cls_dev [B,N]; outputs as
 * ynb_forward_detect, plus keep_dev [B,N] uint8 flags (may be NULL).
 * Candidate order inside a class: score descending, ties by ascending anchor index.
 * workspace_dev: ynb_nms_workspace_bytes(batch, n) bytes. */
int64_t ynb_nms_workspace_bytes(int32_t batch, int64_t n);
int  ynb_nms(const float* boxes_dev, const float* scores_dev, const int32_t* cls_dev,
             int32_t batch, int64_t n, int32_t num_classes,
             float conf_thresh, float nms_thresh, int32_t diou,
             float* out_boxes_dev, float* out_scores_dev, int32_t* out_cls_dev,
             int32_t* out_counts_dev, uint8_t* keep_dev,
             void* workspace_dev, int64_t workspace_bytes, void* stream);

/* The same function (identical keep set and output order) for candidates that sit on the
 * model's anchor grid: n = 3 * sum_l (input_size / stride_l)^2 boxes per image in the order
 * ynb_forward_decode produces (level, cell row, cell column, anchor).  This is what
 * ynb_forward_detect runs: no sort and no serial scan — each candidate collects the preceding
 * same-class candidates that suppress it from a window of cells around itself (a pair with
 * IoU > t has bounded size ratio and centre distance), then a fixed-point pass resolves
 * kept / removed (models/yolo_nano.py:159-279).  Boxes that do not touch their own cell or have
 * no area are still handled exactly (they are compared with everything).
 * workspace_dev: ynb_nms_grid_workspace_bytes(batch, input_size) bytes; input_size % 32 == 0. */
int64_t ynb_nms_grid_workspace_bytes(int32_t batch, int32_t input_size);
int  ynb_nms_grid(const float* boxes_dev, const float* scores_dev, const int32_t* cls_dev,
                  int32_t batch, int32_t input_size, int32_t num_classes,
                  float conf_thresh, float nms_thresh, int32_t diou,
                  float* out_boxes_dev, float* out_scores_dev, int32_t* out_cls_dev,
                  int32_t* out_counts_dev, uint8_t* keep_dev,
                  void* workspace_dev, int64_t workspace_bytes, void* stream);

/* ---- training branch at the head boundary (SURVEY 8 row a14 / 8f row 4; BASELINE config 5) -----------
 * What is here: target assignment, the four losses with their gradient w.r.t. the raw head maps, the
 * SGD update, and the backward kernels of the depthwise / pointwise convolutions and activations, each
 * individually callable.  What is NOT here: BatchNorm in training mode (batch statistics) and the
 * chaining of these kernels into YOLONano.forward(x, target) — that call raises NotImplementedError. */

/* tools.multi_gt_creator (tools.py:97-216) on the device.  labels_dev [B, max_labels, 5] float32 =
 * xmin, ymin, xmax, ymax normalised to [0,1], class; counts_dev [B] int32 (NULL: all max_labels rows
 * are valid).  Writes target_dev [B, N, 11] float32 = obj (1 / 0 / -1 ignored), class, tx, ty, tw, th,
 * box-scale weight, x1, y1, x2, y2, rows in the anchor order of ynb_forward_decode.  Labels are applied
 * in order (a later label overwrites an earlier one on the same cell / anchor); float64 arithmetic in
 * the reference's operation order.  anchors_wh: host, [3][A][2] pixels. */
int  ynb_build_targets(const float* labels_dev, const int32_t* counts_dev, int32_t batch, int32_t max_labels,
                       int32_t input_size, const float* anchors_wh, int32_t num_anchors, float* target_dev,
                       void* stream);

/* The training branch of YOLONano.forward after the heads (models/yolo_nano.py:333-358): box decode
 * (no clamp) / input_size, tools.iou_score (tools.py:219-233) against the target boxes, the detached
 * IoU as objectness label, tools.loss (tools.py:236-276, MSEWithLogitsLoss :12-34).
 * raw_*_dev: NHWC [B, H*W, raw_ld] raw head maps of the three levels with the reference channel map
 * (as ynb_decode_level); target_dev [B, N, 11].  Outputs: losses_dev [4] = conf, cls, bbox (txty +
 * twth), iou, each already divided by the batch size; grad_*_dev (same layout as raw_*) =
 * d(conf + cls + bbox + iou) / d raw, the quantity train.py:222-229 back-propagates into the heads.
 * Deterministic (two-stage reduction).  workspace_dev: ynb_train_loss_workspace_bytes(batch, input_size) bytes. */
int64_t ynb_train_loss_workspace_bytes(int32_t batch, int32_t input_size);
int  ynb_train_loss(const float* raw_s_dev, const float* raw_m_dev, const float* raw_l_dev, int32_t raw_ld,
                    const float* target_dev, int32_t batch, int32_t input_size, const float* anchors_wh,
                    int32_t num_anchors, int32_t num_classes, float* losses_dev, float* grad_s_dev,
                    float* grad_m_dev, float* grad_l_dev, void* workspace_dev, int64_t workspace_bytes,
                    void* stream);

/* YOLONano.forward(x, target) with trainable = True (models/yolo_nano.py:282-358) while the BatchNorm
 * layers are in eval mode (running statistics, folded): backbone + neck + heads on the engine, then
 * ynb_train_loss directly on the engine's head maps.  grad_*_dev: [B, H*W, ynb_raw_ld(e)].  BatchNorm
 * with batch statistics (model.train()) is not built. */
int32_t ynb_raw_ld(const ynb_engine* e);
int  ynb_forward_train_loss(ynb_engine* e, const float* x_dev, int32_t batch, const float* target_dev,
                            float* losses_dev, float* grad_s_dev, float* grad_m_dev, float* grad_l_dev,
                            void* workspace_dev, int64_t workspace_bytes, void* stream);

/* One torch.optim.SGD step (train.py:167-171,230) over a flat float32 vector of n elements:
 *   d = grad_scale * g + weight_decay * p;  buf = first_step ? d : momentum * buf + d;  p -= lr * buf.
 * grad_scale = 1 / world_size folds the averaging of the data-parallel all-reduce (SURVEY 8e) into the
 * update; with grad_scale == 1 the result is bit-identical to the CPU optimiser.  16-byte aligned buffers. */
int  ynb_sgd_step(float* params_dev, const float* grads_dev, float* momentum_buf_dev, int64_t n, float lr,
                  float momentum, float weight_decay, int32_t first_step, float grad_scale, void* stream);

/* Backward of ynb_dwconv3x3 (depthwise 3x3, pad 1, stride 1|2; backbone/shufflenetv2.py:66-67,
 * models/yolo_nano.py:51) without its activation.  w_dev [9][C] as in the forward.
 *   d_in[b,yi,xi,c] = sum_t w[t][c] * d_out[b,(yi+1-dy)/s,(xi+1-dx)/s,c]  */
int  ynb_dwconv3x3_bwd_data(const float* dout_dev, int32_t dout_ld, int32_t dout_off,
                            float* din_dev, int32_t din_ld, int32_t din_off, const float* w_dev,
                            int32_t batch, int32_t h_in, int32_t w_in, int32_t channels, int32_t stride,
                            void* stream);
/* dwdb_dev [10][C]: rows 0..8 = d w[t][c] = sum d_out * in(shifted by tap t), row 9 = d bias[c]. */
int64_t ynb_dwconv3x3_bwd_weight_workspace_bytes(int32_t batch, int32_t h_in, int32_t w_in, int32_t channels,
                                                 int32_t stride);
int  ynb_dwconv3x3_bwd_weight(const float* dout_dev, int32_t dout_ld, int32_t dout_off,
                              const float* in_dev, int32_t in_ld, int32_t in_off, float* dwdb_dev,
                              int32_t batch, int32_t h_in, int32_t w_in, int32_t channels, int32_t stride,
                              void* workspace_dev, int64_t workspace_bytes, void* stream);

/* ---- pieces of the chained training step (BASELINE config 5; yolo_nano_b200/train_step.py) ---------------------
 * Stem conv UNFUSED (training needs the pre-BatchNorm output): Conv2d(3, 24, 3, stride 2, pad 1, bias=False),
 * backbone/shufflenetv2.py:109-113.  x NCHW [batch,3,S,S]; w [27][24] (index (ci*9+ky*3+kx)*24+co); out NHWC
 * [batch,S/2,S/2,24].  Its weight gradient dw [27][24] (no input gradient: the image needs none). */
int  ynb_stem_conv_fwd(const float* x_dev, const float* w2724_dev, float* out_dev, int32_t batch, int32_t input_size,
                       void* stream);
int64_t ynb_stem_conv_bwd_weight_workspace_bytes(int32_t batch, int32_t input_size);
int  ynb_stem_conv_bwd_weight(const float* dout_dev, const float* x_dev, float* dw2724_dev, int32_t batch,
                              int32_t input_size, void* workspace_dev, int64_t workspace_bytes, void* stream);
/* nn.MaxPool2d(3, 2, 1) on NHWC (backbone/shufflenetv2.py:116) and its backward (gradient to the FIRST maximum of a
 * window in row-major order, as ATen; deterministic, no atomics). */
int  ynb_maxpool3x3s2_fwd(const float* in_dev, float* out_dev, int32_t batch, int32_t h, int32_t w, int32_t channels,
                          void* stream);
int  ynb_maxpool3x3s2_bwd(const float* dout_dev, const float* in_dev, float* din_dev, int32_t batch, int32_t h, int32_t w,
                          int32_t channels, void* stream);
/* Data movement of a ShuffleV2 unit in the training step (backbone/shufflenetv2.py:14-28, 66-78), one launch each:
 * op 0  x.chunk(2): x [rows, 2*half] -> a, b [rows, half_padded] (zero-padded halves);   op 1  its adjoint (a, b -> x);
 * op 2  torch.cat + channel_shuffle: x[:, 2i] = a[:, i], x[:, 2i+1] = b[:, i];            op 3  its adjoint (x -> a, b). */
int  ynb_shuffle_unit_move(float* x_dev, float* a_dev, float* b_dev, int64_t rows, int32_t half, int32_t half_padded,
                           int32_t op, void* stream);
/* The same pair keeping the arg-max like ATen's max_pool2d_with_indices: idx_dev [B, Ho, Wo, C] uint8 = winning tap
 * (ky * 3 + kx, first maximum in row-major order); the backward is then a gather (no re-scan of the windows). */
int  ynb_maxpool3x3s2_fwd_idx(const float* in_dev, float* out_dev, uint8_t* idx_dev, int32_t batch, int32_t h, int32_t w,
                              int32_t channels, void* stream);
int  ynb_maxpool3x3s2_bwd_idx(const float* dout_dev, const uint8_t* idx_dev, float* din_dev, int32_t batch, int32_t h,
                              int32_t w, int32_t channels, void* stream);
/* FPN / PAN merge out = a + F.interpolate(a2) (models/yolo_nano.py:291-296; mode 1: a2 is (h/2 x w/2), nearest x2;
 * mode 2: a2 is (2h x 2w), [::2, ::2]) and the gradient w.r.t. a2 (d a = d out). */
int  ynb_resample_add(const float* a_dev, const float* a2_dev, float* out_dev, int32_t batch, int32_t h, int32_t w,
                      int32_t channels, int32_t mode, void* stream);
int  ynb_resample_bwd(const float* dout_dev, float* da2_dev, int32_t batch, int32_t h, int32_t w, int32_t channels,
                      int32_t mode, void* stream);
/* out = a + b: gradient accumulation where a tensor feeds two consumers. */
int  ynb_add(const float* a_dev, const float* b_dev, float* out_dev, int64_t n, void* stream);
/* Dense 3x3 conv (pad 1, stride 1) + bias + act on the tcgen05 implicit-GEMM path, standalone: forward of the
 * `smooth` convs (models/yolo_nano.py:44-47) and, with transposed / tap-reversed weights, their input gradient.
 * w_dev [cout][9][cin] tap-major, cin % 32 == 0, cout <= 256.  Synchronous hook (packs the weights on the host). */
int  ynb_conv3x3_tc(const float* in_dev, int32_t in_ld, float* out_dev, int32_t out_ld, const float* w_dev,
                    const float* b_dev, int32_t batch, int32_t h, int32_t w, int32_t cin, int32_t cout, int32_t act,
                    int32_t mode, void* stream);

/* Training-grade tensor-core convs (replace nn.Conv2d forward / the input-gradient GEMM inside train.py:222-229's
 * step): asynchronous on `stream`, no allocation, no host round trip — the hi / lo TF32 weight planes are packed by a
 * kernel into `workspace` (>= ynb_tc_async_workspace_bytes(cout, ktot) bytes, 256-byte aligned; ktot = cin, or 9 * cin
 * for the 3x3) right before the GEMM.  The last int32 of the workspace is the GEMM's pipeline-timeout flag (0 = ok).
 * pointwise: out[pixels, cout] = act(in[pixels, cin] . W^T + b) with W [w_rows x w_cols] (w_rows <= cout, w_cols <= cin,
 * zero beyond: channel padding) given as w_dev[w_rows][w_ld], or, w_trans = 1, as its transpose w_dev[w_cols][w_ld]
 * (the input gradient of the layer whose weights are w_dev, without a transpose copy). */
int64_t ynb_tc_async_workspace_bytes(int32_t cout, int32_t ktot);
int  ynb_pwconv_tc_async(const float* in_dev, int32_t in_ld, int32_t in_off, float* out_dev, int32_t out_ld,
                         int32_t out_off, int32_t out_step, const float* w_dev, int32_t w_ld, int32_t w_rows,
                         int32_t w_cols, int32_t w_trans, const float* b_dev, int64_t pixels, int32_t cin, int32_t cout, int32_t act,
                         int32_t mode, void* workspace, int64_t workspace_bytes, void* stream);
int  ynb_conv3x3_tc_async(const float* in_dev, int32_t in_ld, float* out_dev, int32_t out_ld, const float* w_dev,
                          const float* b_dev, int32_t batch, int32_t h, int32_t w, int32_t cin, int32_t cout,
                          int32_t act, int32_t mode, void* workspace, int64_t workspace_bytes, void* stream);

/* ModelEMA.update (utils/misc.py:78-86): for every floating-point state tensor  v = v * d + (1 - d) * m  with the
 * reference's two roundings (bit-identical), ALL tensors in one launch.  The caller passes device tables:
 * ema_ptrs_dev / model_ptrs_dev [T] device addresses of the float32 tensors, sizes_dev [T] element counts, and a
 * chunk map (chunk c covers elements [chunk_index[c] * E, +E) of tensor chunk_tensor[c], E = ynb_ema_chunk_elems()). */
int32_t ynb_ema_chunk_elems(void);
int  ynb_ema_update(const uint64_t* ema_ptrs_dev, const uint64_t* model_ptrs_dev, const int64_t* sizes_dev,
                    const int32_t* chunk_tensor_dev, const int32_t* chunk_index_dev, int32_t num_chunks,
                    float d, float one_minus_d, void* stream);

/* Backward of the pointwise conv (ynb_pwconv) w.r.t. weights and bias:
 *   dw[n][k] = sum_m d_out[m, dout_off + n] * in[m, in_off + k];  db[n] = sum_m d_out[m, dout_off + n].
 * (The gradient w.r.t. the input is the forward GEMM with the transposed weight matrix and no bias:
 * ynb_pwconv / ynb_pwconv_tc.)  Deterministic split-M reduction. */
int64_t ynb_pwconv_bwd_weight_workspace_bytes(int64_t pixels, int32_t cin, int32_t cout);
int  ynb_pwconv_bwd_weight(const float* dout_dev, int32_t dout_ld, int32_t dout_off,
                           const float* in_dev, int32_t in_ld, int32_t in_off, float* dw_dev, float* db_dev,
                           int64_t pixels, int32_t cin, int32_t cout,
                           void* workspace_dev, int64_t workspace_bytes, void* stream);

/* Weight / bias gradient of a dense 3x3 conv, pad 1, stride 1 (the `smooth` convs, models/yolo_nano.py:44-47;
 * utils/modules.py:11 with k = 3), NHWC views of [batch, h, w]: nine tap-shifted pointwise weight gradients on
 * the tcgen05 kernel.  dw9_dev [9][cout][cin], tap t = ky * 3 + kx  (torch: weight.grad[n][k][ky][kx]);
 * db_dev [cout].  Needs 16-byte aligned views, cin <= 255.  workspace: ynb_pwconv_bwd_weight_workspace_bytes. */
int  ynb_conv3x3_bwd_weight(const float* dout_dev, int32_t dout_ld, int32_t dout_off,
                            const float* in_dev, int32_t in_ld, int32_t in_off, float* dw9_dev, float* db_dev,
                            int32_t batch, int32_t h, int32_t w, int32_t cin, int32_t cout,
                            void* workspace_dev, int64_t workspace_bytes, void* stream);

/* Backward of ReLU / LeakyReLU(0.1) (YNB_ACT_RELU | YNB_ACT_LEAKY) from the forward OUTPUT:
 *   dpre[m, c] = dout[m, c] * (out[m, c] > 0 ? 1 : slope). */
int  ynb_act_bwd(const float* dout_dev, int32_t dout_ld, int32_t dout_off, const float* out_dev, int32_t out_ld,
                 int32_t out_off, float* dpre_dev, int32_t dpre_ld, int32_t dpre_off, int64_t pixels,
                 int32_t channels, int32_t act, void* stream);

/* nn.BatchNorm2d in TRAINING mode (utils/modules.py:13; backbone/shufflenetv2.py:47,56,61; eps 1e-5,
 * momentum 0.1) fused with the following ReLU / LeakyReLU(0.1), on an NHWC view [pixels, ld] with channels
 * [off, off + C):  mean / biased variance over the pixels -> y = act((x - mean) * rstd * gamma + beta);
 * running_mean / running_var (may be NULL) are updated in place with the unbiased variance, as torch
 * does; save_mean / save_rstd [C] are kept for the backward.  Deterministic.  channels, strides and
 * offsets multiples of 4, 16-byte aligned pointers.  workspace: ynb_bn_workspace_bytes(pixels, C). */
int64_t ynb_bn_workspace_bytes(int64_t pixels, int32_t channels);
int  ynb_bn_train_fwd(const float* x_dev, int32_t x_ld, int32_t x_off, float* y_dev, int32_t y_ld, int32_t y_off,
                      const float* gamma_dev, const float* beta_dev, float* running_mean_dev,
                      float* running_var_dev, float* save_mean_dev, float* save_rstd_dev, int64_t pixels,
                      int32_t channels, float eps, float momentum, int32_t act, void* workspace_dev,
                      int64_t workspace_bytes, void* stream);
/* Its backward, activation included (y_dev = the forward output, needed only when act != NONE):
 *   g = dy * act'(y);  dbeta = sum g;  dgamma = sum g * x_hat;
 *   dx = gamma * rstd * (g - dbeta / M - x_hat * dgamma / M).   dgamma_dbeta_dev = [dgamma[C] | dbeta[C]]. */
int  ynb_bn_train_bwd(const float* dy_dev, int32_t dy_ld, int32_t dy_off, const float* x_dev, int32_t x_ld,
                      int32_t x_off, const float* y_dev, int32_t y_ld, int32_t y_off, const float* gamma_dev,
                      const float* save_mean_dev, const float* save_rstd_dev, float* dx_dev, int32_t dx_ld,
                      int32_t dx_off, float* dgamma_dbeta_dev, int64_t pixels, int32_t channels, int32_t act,
                      void* workspace_dev, int64_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif  /* YOLONANO_B200_H_ */
