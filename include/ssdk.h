/*
 * ssdk.h -- C-ABI of the B200-native SSD hot path (libssdk.so).
 *
 * The reference (pierluigiferrari/ssd_keras) is pure Python: it has no FFI / plugin
 * interface of its own, so the drop-in boundary is its public Python surface (SURVEY.md
 * section 8b).  Each entry point below names the reference interface it replaces
 * (file:line relative to the reference root).  The Python package `ssd_keras_b200`
 * re-creates those reference names on top of this library through ctypes; see
 * INTEGRATION.md for the binding a reference maintainer would add.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no C++/torch types.
 *   - every function returns 0 on success or a negative ssdk_status; it never throws.
 *     ssdk_last_error() returns a thread-local, human readable message for the last failure.
 *   - "dev" pointers are CUDA device pointers on the context's device; "host" pointers are
 *     ordinary host memory.  Outputs are caller-allocated.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).  Calls are
 *     asynchronous with respect to the host unless stated otherwise.
 *   - a context (and the objects created from it) may be used by one host thread at a time.
 *   - there is NO CPU fallback: without a CUDA device every compute call fails with
 *     SSDK_ERR_CUDA.
 */
#ifndef SSDK_H_
#define SSDK_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SSDK_VERSION 100

typedef enum {
  SSDK_OK = 0,
  SSDK_ERR_INVALID = -1,     /* bad argument (the Python layer raises ValueError)          */
  SSDK_ERR_CUDA = -2,        /* CUDA runtime/driver failure, message has the cuda error    */
  SSDK_ERR_UNSUPPORTED = -3, /* valid in the reference but not implemented here            */
  SSDK_ERR_NOMEM = -4,
  SSDK_ERR_DEGENERATE = -5   /* degenerate ground-truth box (reference: DegenerateBoxError) */
} ssdk_status;

typedef enum { SSDK_COORDS_CENTROIDS = 0, SSDK_COORDS_CORNERS = 1, SSDK_COORDS_MINMAX = 2 } ssdk_coords;

typedef struct ssdk_ctx ssdk_ctx;
typedef struct ssdk_encoder ssdk_encoder;
typedef struct ssdk_model ssdk_model;

int ssdk_version(void);
const char* ssdk_last_error(void);

/* One context per (device, host thread).  Owns scratch workspaces. */
int ssdk_ctx_create(int device, ssdk_ctx** out);
int ssdk_ctx_destroy(ssdk_ctx* ctx);
/* Number of kernels this library launched through `ctx` since creation (bench.py's gpu_launches). */
int64_t ssdk_ctx_launch_count(const ssdk_ctx* ctx);

/* ------------------------------------------------------------------------------------------
 * Anchor boxes.  Replaces SSDInputEncoder.generate_anchor_boxes_for_layer
 * (ssd_encoder_decoder/ssd_input_encoder.py:420-548) and AnchorBoxes.call
 * (keras_layers/keras_layer_AnchorBoxes.py:133-255).  Host-side float64 arithmetic, bit-exact
 * with the reference; `out_f32` is the float32 cast the Keras layer emits (:252).
 * steps_* / offsets_* entries that are NaN mean "None" (derive step from the feature map,
 * offset 0.5).  Prior order: layers in order, ((y*W + x)*n_boxes + b) within a layer.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int img_height, img_width;
  int n_layers;
  const int* fm_height;          /* [n_layers] predictor feature-map sizes */
  const int* fm_width;           /* [n_layers] */
  const double* scales;          /* [n_layers + 1] */
  const int* n_aspect_ratios;    /* [n_layers] */
  const double* aspect_ratios;   /* concatenated, sum(n_aspect_ratios) entries */
  int two_boxes_for_ar1;
  const double* steps_h;         /* [n_layers] or NULL; NaN = None */
  const double* steps_w;
  const double* offsets_h;       /* [n_layers] or NULL; NaN = None */
  const double* offsets_w;
  int clip_boxes;
  int coords;                    /* ssdk_coords */
  int normalize_coords;
} ssdk_anchor_cfg;

int ssdk_anchors_count(const ssdk_anchor_cfg* cfg, int* out_P, int* out_n_boxes /* [n_layers] or NULL */);
int ssdk_anchors_generate(const ssdk_anchor_cfg* cfg, double* out_f64 /* host [P*4] */, float* out_f32 /* host [P*4] or NULL */);

/* ------------------------------------------------------------------------------------------
 * Ground-truth encoder.  Replaces SSDInputEncoder.__call__
 * (ssd_encoder_decoder/ssd_input_encoder.py:277-418) together with iou
 * (bounding_box_utils/bounding_box_utils.py:283-383), match_bipartite_greedy and match_multi
 * (ssd_encoder_decoder/matching_utils.py:22-116) and generate_encoding_template (:550-611).
 * IoU and matching decisions are taken in float64 like the reference; the target tensor is
 * written as float32 (what Keras feeds the loss).  One kernel launch per batch; an encoder object owns
 * scratch memory and must not be used from two streams at the same time.
 * ------------------------------------------------------------------------------------------ */
typedef struct {
  int img_height, img_width;
  int n_classes_total;       /* including background */
  int P;                     /* number of anchors */
  int background_id;
  int coords;                /* ssdk_coords: format of `anchors` and of the encoded targets */
  int matching_multi;        /* 1 = 'multi', 0 = 'bipartite' */
  double pos_iou_threshold;
  double neg_iou_limit;
  int border_d;              /* 0 'half', 1 'include', -1 'exclude' */
  int normalize_coords;
  double variances[4];
  /* Optional predictor-layer geometry (prior index = layer offset + (y*fm_width + x)*n_boxes + box): lets the encoder
   * group priors into compact blocks of feature-map cells, so that fewer ground-truth boxes touch a block.  n_layers = 0
   * (or NULL arrays): consecutive groups of 256 priors only.  The arrays are read during ssdk_encoder_create. */
  int n_layers;
  const int* fm_height;      /* [n_layers] */
  const int* fm_width;       /* [n_layers] */
  const int* n_boxes;        /* [n_layers] */
} ssdk_encode_cfg;

int ssdk_encoder_create(ssdk_ctx* ctx, const ssdk_encode_cfg* cfg, const double* anchors_host /* [P*4], in cfg->coords */,
                        ssdk_encoder** out);
int ssdk_encoder_destroy(ssdk_encoder* enc);
/* gt_boxes_dev: [sum(G_i) * 5] float32 rows (class_id, xmin, ymin, xmax, ymax) in pixels, images concatenated;
 * gt_offsets_host: [B+1] row offsets (host; the ragged shape is host knowledge in the reference too);
 * out_y_dev: [B * P * (C+12)] float32;  out_match_dev (optional): [B * P] int32, matched gt index within the
 * image, -1 = background, -2 = neutral.  status_dev (optional): one int32 that is set to the 1-based index of
 * a batch item with a degenerate box (xmax<=xmin or ymax<=ymin), else left 0 (reference raises :333-336). */
int ssdk_encode(ssdk_encoder* enc, const float* gt_boxes_dev, const int* gt_offsets_host, int B,
                float* out_y_dev, int* out_match_dev, int* status_dev, void* stream);
/* Same with float64 ground-truth rows: the reference converts whatever it is given to float64 (:330), so labels that are
 * not representable in float32 (sub-pixel coordinates after augmentation) need this entry to stay bit-exact. */
int ssdk_encode_f64(ssdk_encoder* enc, const double* gt_boxes_dev, const int* gt_offsets_host, int B,
                    float* out_y_dev, int* out_match_dev, int* status_dev, void* stream);
/* Same with the row offsets already on the device (the batch was assembled there, see ssdk_assemble_batch): nothing
 * is read from the host; total_g = gt_offsets[B] and max_g = the largest per-image box count (or an upper bound of it). */
int ssdk_encode_dev(ssdk_encoder* enc, const float* gt_boxes_dev, const int* gt_offsets_dev, int B, int total_g, int max_g,
                    float* out_y_dev, int* out_match_dev, int* status_dev, void* stream);
/* Standalone pieces, used by tests and the micro-benchmark: IoU matrix (G x P, float64, row-major). */
int ssdk_iou_matrix(ssdk_encoder* enc, const float* gt_boxes_dev, int G, double* out_dev, void* stream);
/* General IoU, replaces iou() (bounding_box_utils/bounding_box_utils.py:283-383): boxes1 [m*4], boxes2 [n*4] float64 in
 * `coords` format; elementwise=0 -> out [m*n] ('outer_product'), elementwise=1 -> out [max(m,n)] with broadcasting of a
 * single box ('element-wise').  Keeps the reference quirk: the intersection ignores border_d, the areas use it. */
int ssdk_iou(ssdk_ctx* ctx, const double* boxes1_dev, int m, const double* boxes2_dev, int n, int coords, int border_d,
             int elementwise, double* out_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * Batch assembly (the hand-off DataGenerator.generate -> label_encoder, data_generator/object_detection_2d_data_generator.py:
 * 1095-1151) and the box half of the reference's geometric augmentation ops on the device: per image a list of operations
 * with the parameters the caller's (host-side, random) augmentation logic decided, applied to every box in float64 like
 * NumPy does, boxes that fail a filter are dropped, the survivors are packed into the encoder's ragged format.
 *   CROP_PAD  a0=patch_ymin a1=patch_xmin a2=patch_height a3=patch_width; flags bit0: BoxFilter 'center_point' against the
 *             patch, bit1: clip to the patch      (CropPad.__call__, object_detection_2d_patch_sampling_ops.py:312-330;
 *             SSDExpand = negative patch origin without filter / clip, SSDRandomCrop = filter + clip)
 *   FLIP_H    a0=image width   FLIP_V  a0=image height                  (object_detection_2d_geometric_ops.py:186,194)
 *   RESIZE    a0=in_height a1=in_width a2=out_height a3=out_width; flags bit0: drop degenerate boxes afterwards (:88-100)
 *   FILTER    flags bit0: drop degenerate boxes (xmax <= xmin or ymax <= ymin), bit1: drop boxes with area < a0
 *             (BoxFilter, object_detection_2d_image_boxes_validation_utils.py:155-165; also DataGenerator's
 *             degenerate_box_handling='remove')
 * ------------------------------------------------------------------------------------------ */
typedef enum { SSDK_BOXOP_END = 0, SSDK_BOXOP_CROP_PAD = 1, SSDK_BOXOP_FLIP_H = 2, SSDK_BOXOP_FLIP_V = 3, SSDK_BOXOP_RESIZE = 4,
               SSDK_BOXOP_FILTER = 5 } ssdk_box_op_kind;
typedef struct { int op; int flags; double a0, a1, a2, a3; } ssdk_box_op;
/* gt_in_dev [total_in*5] float32 (gt_in_f64 = 0) or float64 (1) rows (class, xmin, ymin, xmax, ymax), offsets_in_dev [B+1]; ops_dev [B*max_ops] (a list ends at
 * SSDK_BOXOP_END or after max_ops entries; max_ops = 0: pack only).  Outputs: gt_out_dev [<= total_in*5], offsets_out_dev [B+1],
 * out_stats_dev (optional) [2] = total number of boxes left, largest per-image count.  Everything stays on the device: feed
 * the result to ssdk_encode_dev with total_in / the input's largest count as upper bounds. */
int ssdk_assemble_batch(ssdk_ctx* ctx, const void* gt_in_dev, int gt_in_f64, const int* offsets_in_dev, int B, int total_in,
                        const ssdk_box_op* ops_dev, int max_ops, float* gt_out_dev, int* offsets_out_dev, int* out_stats_dev,
                        void* stream);
/* The image half of the same operations, driven by the same lists: B ragged uint8 HWC 3-channel source images (the output of
 * ssdk_photometric when the chain distorts them) -> out_dev (B, out_h, out_w, 3), float32 (out_dtype 0, values 0..255) or uint8 (1).
 *   src_dev          all images' bytes; image b starts at byte src_offsets_dev[b] (int64) and is src_hw_dev[2b] x src_hw_dev[2b+1]
 *   CROP_PAD         the CropPad canvas (object_detection_2d_patch_sampling_ops.py:266-313): patch-sized, filled with the
 *                    background (flags bits 8-15 R, 16-23 G, 24-31 B), the image placed at -patch origin; a patch running past the
 *                    image is padded with the background too.  SSDExpand = negative origin with background (123, 117, 104).
 *   FLIP_H / FLIP_V  image[:, ::-1] / image[::-1]; a0 must be the current width / height
 *   RESIZE           cv2.resize(image, (a3, a2), interpolation=flags bits 8-15): 0 NEAREST, 1 LINEAR, 2 CUBIC, 3 AREA, 4 LANCZOS4
 *                    (object_detection_2d_geometric_ops.py:61-72); a0 / a1 must be the current size.  Bit-exact to OpenCV's 8-bit
 *                    arithmetic (CUBIC: to its portable implementation, see DESIGN.md section 4)
 *   FILTER           no effect on pixels
 * One fused launch, no intermediate images.  Returns SSDK_ERR_INVALID, before anything is launched, for an empty source image,
 * a crop/pad parameter that is not an integer or whose origin lies past the image (the reference's ValueError), more than one
 * RESIZE or a crop/pad / flip after it, a mode outside 0..4, sizes in a FLIP / RESIZE that are not the image's, or a final size
 * other than (out_h, out_w).  To validate, the call copies the sizes and op lists to the host and synchronises `stream`. */
int ssdk_assemble_images(ssdk_ctx* ctx, const uint8_t* src_dev, const int64_t* src_offsets_dev, const int* src_hw_dev, int B,
                         const ssdk_box_op* ops_dev, int max_ops, int out_h, int out_w, int out_dtype /* 0 f32, 1 u8 */, void* out_dev,
                         void* stream);
/* The photometric distortions that come before SSDExpand in the reference's chains (object_detection_2d_photometric_ops.py),
 * as a per-image list of pointwise pixel operations on the same ragged uint8 layout ssdk_assemble_images takes.  A pixel is in
 * uint8 state (the start) or float32 state; the list must end in uint8 state, so the result is ready to be that call's src_dev.
 *   TO_FLOAT      ConvertDataType('float32')           identity in float32 state
 *   TO_U8         ConvertDataType('uint8'): np.round (half to even) then astype(uint8); identity in uint8 state
 *   RGB2HSV       ConvertColor('RGB', 'HSV'): cv2.cvtColor on uint8, OpenCV's 8-bit integer arithmetic       (uint8 state only)
 *   HSV2RGB       ConvertColor('HSV', 'RGB'): cv2.cvtColor on uint8, bit-exact to OpenCV 4.13's default (AVX2) path: whole
 *                 32-pixel vectors of a row truncate, the last (width mod 32) pixels round (DESIGN.md section 4) (uint8 state only)
 *   BRIGHTNESS    Brightness(a0):  clip(x + f32(a0), 0, 255)                                                (float32 state only)
 *   CONTRAST      Contrast(a0):    clip(127.5 + f32(a0) * (x - 127.5), 0, 255), a0 > 0                     (float32 state only)
 *   SATURATION    Saturation(a0):  channel 1 = clip(x * f32(a0), 0, 255), a0 > 0                           (float32 state only)
 *   HUE           Hue(a0):         channel 0 = NumPy's float32 (x + f32(a0)) % 180, a0 in [-180, 180]       (float32 state only)
 *   CHANNEL_SWAP  ChannelSwap(order): x[..., order], arg = o0 | o1 << 8 | o2 << 16, each in 0..2             (either state)
 * a0 is the parameter as drawn (a Python float); NumPy 2 rounds it to float32 before combining it with a float32 image, and so
 * does the kernel.  A list ends at SSDK_PIXOP_END or after max_ops (0..64) entries.  dst_dev may equal src_dev (in place).
 * One launch.  Returns SSDK_ERR_INVALID, before anything is launched, for an empty image, an unknown operation, a colour
 * conversion in float32 state, an arithmetic operation in uint8 state, a list that does not end in uint8 state, a NaN
 * parameter or one the reference's constructors refuse.  To validate, the call copies the sizes and op lists to the host and
 * synchronises `stream`. */
typedef enum { SSDK_PIXOP_END = 0, SSDK_PIXOP_TO_FLOAT = 1, SSDK_PIXOP_TO_U8 = 2, SSDK_PIXOP_RGB2HSV = 3, SSDK_PIXOP_HSV2RGB = 4,
               SSDK_PIXOP_BRIGHTNESS = 5, SSDK_PIXOP_CONTRAST = 6, SSDK_PIXOP_SATURATION = 7, SSDK_PIXOP_HUE = 8,
               SSDK_PIXOP_CHANNEL_SWAP = 9 } ssdk_pixel_op_kind;
typedef struct { int op; int arg; double a0; } ssdk_pixel_op;
int ssdk_photometric(ssdk_ctx* ctx, const uint8_t* src_dev, uint8_t* dst_dev, const int64_t* src_offsets_dev, const int* src_hw_dev,
                     int B, const ssdk_pixel_op* ops_dev, int max_ops, void* stream);

/* ------------------------------------------------------------------------------------------
 * Evaluation.  Replaces the per-prediction Python loop of Evaluator.match_predictions
 * (eval_utils/average_precision_evaluator.py:538-736, element-wise iou at :679) and the cumulative sums of :726-727.
 * The caller sorts the predictions twice (stable): by (class, confidence desc) -- the order of the outputs -- and by
 * (class, image, confidence desc) -- the order of the pred_* inputs, whose (class, image) runs are given by seg_offsets.
 *   pred_rank[i]   position of input prediction i in the (class, confidence desc) order
 *   gt_rows        float64 (class, xmin, ymin, xmax, ymax) rows of all images, gt_offsets [n_images+1]
 *   gt_neutral     optional uint8 flags (eval_neutral, :684), gt_matched uint8 scratch zeroed by the caller
 *   tp / fp        int32 [n_pred], zeroed by the caller, in (class, confidence desc) order
 * ssdk_eval_cumsum: inclusive scans of tp / fp inside each of the n_segments ranges class_offsets[c] .. class_offsets[c+1].
 * ------------------------------------------------------------------------------------------ */
int ssdk_eval_match(ssdk_ctx* ctx, int n_pred, const int* seg_offsets_dev, int n_seg, const int* pred_image_dev,
                    const int* pred_class_dev, const float* pred_box_dev, const int* pred_rank_dev, const double* gt_rows_dev,
                    const int* gt_offsets_dev, const unsigned char* gt_neutral_dev, unsigned char* gt_matched_dev,
                    double matching_iou_threshold, int border_d, int* tp_dev, int* fp_dev, void* stream);
int ssdk_eval_cumsum(ssdk_ctx* ctx, const int* tp_dev, const int* fp_dev, const int* class_offsets_dev, int n_segments,
                     int* ctp_dev, int* cfp_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * Decoders.
 *   mode PER_CLASS + layer_semantics=1: DecodeDetections.call   (keras_layers/keras_layer_DecodeDetections.py:109-265)
 *   mode FAST      + layer_semantics=1: DecodeDetectionsFast.call (keras_layers/keras_layer_DecodeDetectionsFast.py:111-248)
 *   mode PER_CLASS + layer_semantics=0: decode_detections        (ssd_encoder_decoder/ssd_output_decoder.py:111-226)
 *   mode FAST      + layer_semantics=0: decode_detections_fast   (ssd_encoder_decoder/ssd_output_decoder.py:228-333)
 * layer_semantics=1: float32 arithmetic, tf.image.non_max_suppression IoU rule, at most nms_max_output
 *   survivors per class, output sorted by confidence (ties: lower row), zero padded to top_k rows.
 * layer_semantics=0: float32 decode stored in float64 like NumPy, float64 IoU with the border_pixels
 *   quirk, no per-class cap, strict '>' (per-class) / '>=' (fast) confidence test; out rows are the
 *   top_k set (order: confidence desc, then class-major NMS order); out_counts gives the valid rows.
 * ------------------------------------------------------------------------------------------ */
typedef enum { SSDK_DECODE_PER_CLASS = 0, SSDK_DECODE_FAST = 1 } ssdk_decode_mode;

typedef struct {
  int mode;                 /* ssdk_decode_mode */
  int layer_semantics;
  int n_classes_total;
  int P;
  double confidence_thresh; /* compared in float32 (layer) or float64 (NumPy API), like the reference */
  double iou_threshold;     /* <= 0 with layer_semantics=0 and mode FAST: skip NMS (reference :326) */
  int top_k;                /* <= 0: 'all' (NumPy API only; out must hold max_out rows) */
  int nms_max_output;       /* layer only */
  int coords;               /* input_coords */
  int normalize_coords;
  int img_height, img_width;
  int border_d;
  int max_out;              /* rows per image in `out`; layer: == top_k */
} ssdk_decode_cfg;

/* y_pred_dev [B*P*(C+12)] float32 -> out_dev [B*max_out*6] float32 rows (class, conf, xmin, ymin, xmax, ymax),
 * out_counts_dev [B] int32 valid rows, out_index_dev (optional) [B*max_out] int32 prior index of each row (-1 pad). */
int ssdk_decode(ssdk_ctx* ctx, const ssdk_decode_cfg* cfg, const float* y_pred_dev, int B,
                float* out_dev, int* out_counts_dev, int* out_index_dev, void* stream);
/* Single-class NMS micro-benchmark entry (SURVEY 8d config 5): boxes [B*n*4] corners, scores [B*n]. */
int ssdk_nms(ssdk_ctx* ctx, const float* boxes_dev, const float* scores_dev, int B, int n,
             double confidence_thresh, double iou_threshold, int nms_max_output, int top_k,
             float* out_dev /* [B*top_k*6] */, int* out_counts_dev, int* out_index_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * SSD loss.  Replaces SSDLoss.compute_loss (keras_loss_function/keras_ssd_loss.py:98-211).
 * out_loss_dev [B] float32.  bwd writes d(sum_b upstream[b]*loss[b])/d y_pred with the hard-negative
 * mask held constant (upstream_dev NULL = 1/B each, the Keras batch mean).  One cooperative kernel launch per call
 * (csrc/loss.cu): per-box losses, batch-global top-k by a two-level histogram select, masked sums / gradient.
 * ------------------------------------------------------------------------------------------ */
int ssdk_ssd_loss_fwd(ssdk_ctx* ctx, const float* y_true_dev, const float* y_pred_dev, int B, int P, int n_classes_total,
                      int neg_pos_ratio, int n_neg_min, float alpha, float* out_loss_dev,
                      int* out_stats_dev /* optional [4]: n_positive, n_neg_losses, k, ties_taken */, void* stream);
int ssdk_ssd_loss_bwd(ssdk_ctx* ctx, const float* y_true_dev, const float* y_pred_dev, int B, int P, int n_classes_total,
                      int neg_pos_ratio, int n_neg_min, float alpha, const float* upstream_dev,
                      float* out_grad_dev /* [B*P*(C+12)] */, void* stream);
/* Loss and gradient from ONE launch of the same kernel (what a training step needs). */
int ssdk_ssd_loss_fwd_bwd(ssdk_ctx* ctx, const float* y_true_dev, const float* y_pred_dev, int B, int P, int n_classes_total,
                          int neg_pos_ratio, int n_neg_min, float alpha, const float* upstream_dev, float* out_loss_dev,
                          int* out_stats_dev, float* out_grad_dev, void* stream);

/* Multi-GPU, global-batch-exact loss.  The reference's n_positive (:143) and hard-negative top-k (:179-183) run over the
 * WHOLE batch; when the batch is sharded over ranks the kernel's phases are launched one by one on a caller-provided
 * workspace and the integer counts / histograms inside it are summed over the ranks (NCCL all-reduce) in between:
 *   zero the workspace; phase 0; all-reduce(sum) counts + hist1; phase 1; all-reduce(sum) hist2; phase 2; phase 3;
 *   all-gather the int32 at ties_offset (one per rank, rank order = global image order) -> ties_all_dev; phase 4.
 * Phase 4 writes the (B,) losses of this rank's images (normalised by the global n_positive and multiplied by global_B
 * like :204-209) and / or the gradient with respect to this rank's y_pred.  Boxes whose loss equals the k-th largest are
 * taken in global flat-index order, like tf.nn.top_k on the single-process batch. */
typedef struct {
  long long bytes;            /* size of the workspace */
  long long counts_offset;    /* int64[counts_n] */
  long long counts_n;
  long long hist1_offset;     /* int32[hist_n] */
  long long hist2_offset;     /* int32[hist_n] */
  long long hist_n;
  long long ties_offset;      /* int32[1], valid after phase 3 */
} ssdk_loss_ws_layout;
int ssdk_ssd_loss_ws_layout(int B, int P, ssdk_loss_ws_layout* out);
int ssdk_ssd_loss_phase(ssdk_ctx* ctx, int phase, const float* y_true_dev, const float* y_pred_dev, int B, int P,
                        int n_classes_total, int neg_pos_ratio, int n_neg_min, float alpha, void* ws_dev, int global_B,
                        const int* ties_all_dev /* [world], phase 4 */, int rank, const float* upstream_dev,
                        float* out_loss_dev, int* out_stats_dev, float* out_grad_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * Model graph.  Replaces ssd_300 (models/keras_ssd300.py:31-457), ssd_512 (models/keras_ssd512.py:31-477)
 * and build_model (models/keras_ssd7.py:30-430) + L2Normalization
 * (keras_layers/keras_layer_L2Normalization.py:61-63): a static plan of tcgen05 implicit-GEMM
 * convolutions, pooling, normalisation and the head epilogue producing (B,P,C+12).
 * The graph is described layer by layer by the host (Python mirrors the reference builders).
 * ------------------------------------------------------------------------------------------ */
typedef enum {
  SSDK_OP_INPUT = 0,      /* preprocessing: (x - mean)/std, channel swap; source = user images (B,H,W,3) f32 */
  SSDK_OP_CONV = 1,       /* conv + bias + activation */
  SSDK_OP_MAXPOOL = 2,
  SSDK_OP_L2NORM = 3,     /* x * rsqrt(max(sum_c x^2, 1e-12)) * gamma_c */
  SSDK_OP_HEAD = 4,       /* fused conf+loc 3x3 predictor conv for one source layer -> rows of y_pred */
  SSDK_OP_TENSOR = 5      /* source = a user tensor (B,H,W,C) f32 with any channel count, taken as it is (ssdk_conv2d_fwd / ssdk_maxpool) */
} ssdk_op;

typedef enum { SSDK_ACT_NONE = 0, SSDK_ACT_RELU = 1, SSDK_ACT_ELU = 2 } ssdk_act;

typedef struct {
  int op;                   /* ssdk_op */
  int input;                /* index of the producing layer (-1 for SSDK_OP_INPUT) */
  int cout;                 /* conv/head: output channels (head: n_boxes*(C+4) is derived; give n_boxes) */
  int kh, kw, stride, dilation;
  int pad_t, pad_l, pad_b, pad_r;   /* zero padding (conv) / -inf padding (pool) */
  int act;                  /* ssdk_act */
  int n_boxes;              /* head only */
  /* Parameters, host pointers, copied at build time.  conv: kernel HWIO float32 [kh*kw*cin*cout], bias [cout];
   * optional folded batch-norm scale/shift per output channel (applied after bias, before act);
   * l2norm: gamma [c]; head: conf kernel/bias and loc kernel/bias; input: mean[3]/std[3]/swap[3]. */
  const float* kernel; const float* bias;
  const float* bn_scale; const float* bn_shift;
  const float* kernel2; const float* bias2;      /* head: loc kernel/bias (kernel/bias = conf) */
  const float* mean; const float* stddev; const int* swap;
  /* conv followed by BatchNormalization (models/keras_ssd7.py:277-309), raw parameters [cout] each.  Training plans
   * (ssdk_model_desc.training = 1) run the layer in Keras' training phase: batch statistics over (B,H,W), moving averages
   * updated with `bn_momentum`; inference plans use the folded bn_scale / bn_shift above. */
  const float* bn_gamma; const float* bn_beta; const float* bn_mean; const float* bn_var;
  float bn_eps; float bn_momentum;
} ssdk_layer_desc;

typedef struct {
  int batch;                /* plan is built for this batch size */
  int img_height, img_width, img_channels;
  int n_classes_total;
  int n_layers;
  const ssdk_layer_desc* layers;
  int precision;            /* 0 = bf16x3 split (fp32-faithful, default), 1 = single-pass bf16 */
  const float* anchors_f32; /* host [P*4] */
  float variances[4];
  int training;             /* 1: size the activation borders for the backward pass too (needed by ssdk_trainer_create) */
} ssdk_model_desc;

/* Stand-alone L2Normalization.call (keras_layers/keras_layer_L2Normalization.py:61-63) on a float32 tensor viewed as
 * [rows, C] (rows = B*H*W, channels last): out = x * rsqrt(max(sum_c x^2, 1e-12)) * gamma_c. */
int ssdk_l2_normalize(ssdk_ctx* ctx, const float* x_dev, long long rows, int C, const float* gamma_dev, float* out_dev, void* stream);

/* Stand-alone Conv2D forward (what every `Conv2D(...)` of models/keras_ssd300.py:274-335 computes; SURVEY 8b `ssdk_conv2d_fwd`):
 * y = act(conv(x, kernel) + bias) on float32 NHWC device tensors, kernel HWIO / bias on the HOST (copied and packed by the call).
 * x (B,H,W,Cin) -> y (B,Ho,Wo,Cout), Ho = (H + pad_t + pad_b - dilation*(kh-1) - 1)/stride + 1.  Runs the same tcgen05 plan the
 * model graphs use (precision 0 = bf16x3, 1 = bf16) as a one-layer graph built and destroyed inside the call: it synchronises
 * the stream and allocates -- a utility for tests and interop; steady-state users describe their layers to ssdk_model_create. */
int ssdk_conv2d_fwd(ssdk_ctx* ctx, const float* x_dev, int B, int H, int W, int Cin, const float* kernel_hwio_host,
                    const float* bias_host /* or NULL */, int Cout, int kh, int kw, int stride, int dilation,
                    int pad_t, int pad_l, int pad_b, int pad_r, int act /* ssdk_act */, int precision, float* y_dev, void* stream);
/* Stand-alone MaxPooling2D forward (models/keras_ssd300.py:276-309; -inf padding, i.e. TensorFlow 'same' when the caller passes
 * the 'same' pads): x (B,H,W,C) -> y (B,Ho,Wo,C), Ho = (H + pad_t + pad_b - kh)/stride + 1.  Same caveats as ssdk_conv2d_fwd. */
int ssdk_maxpool(ssdk_ctx* ctx, const float* x_dev, int B, int H, int W, int C, int kh, int kw, int stride,
                 int pad_t, int pad_l, int pad_b, int pad_r, float* y_dev, void* stream);

/* The two-stream schedule ssdk_model_create gives an inference plan (DESIGN.md 3.5), as a host-only function on plain arrays (no
 * device needed): kind[i] 0 = not a tensor-core GEMM launch (pool, L2Norm, input), 1 = trunk convolution, 2 = predictor head;
 * grid[i] = CTAs of that launch; input[i] = producing layer or -1; R <= 0 selects the default (sm_count / 3 + 1).
 * out_on_side[i] = 1: issued on the second stream; *out_from = first such layer (-1: single stream); *out_grid_cap = grid limit of
 * the GEMM launches that stay on the caller's stream meanwhile.  The reference has no counterpart (Keras/TF schedule their graph). */
int ssdk_schedule_preview(int n_layers, const int* kind, const int* grid, const int* input, int R, int sm_count,
                          unsigned char* out_on_side, int* out_from, int* out_grid_cap);

int ssdk_model_create(ssdk_ctx* ctx, const ssdk_model_desc* desc, ssdk_model** out);
int ssdk_model_destroy(ssdk_model* m);
int ssdk_model_num_priors(const ssdk_model* m, int* out_P);
/* Spatial size / channels of a layer's output (reference: model.get_layer(name).output_shape[1:3]). */
int ssdk_model_layer_shape(const ssdk_model* m, int layer, int* out_h, int* out_w, int* out_c);
/* images_dev (B,H,W,3) float32 NHWC -> y_pred_dev (B,P,C+12) float32. */
int ssdk_model_forward(ssdk_model* m, const float* images_dev, float* y_pred_dev, void* stream);
/* Copy a layer's activation (B,h,w,c) as float32 NHWC to out_dev (tests: per-layer parity). */
int ssdk_model_read_layer(ssdk_model* m, int layer, float* out_dev, void* stream);
/* FLOPs of one forward pass (2*MACs of every conv, SURVEY 8d) and MMA flops actually issued. */
int ssdk_model_flops(const ssdk_model* m, double* out_algorithmic, double* out_issued);
/* Time of the conv kernels of the last forward in ms (CUDA events on `stream`), when enabled. */
int ssdk_model_set_timing(ssdk_model* m, int enable);
int ssdk_model_last_conv_ms(ssdk_model* m, float* out_ms);

/* ------------------------------------------------------------------------------------------
 * Training step (BASELINE config 3).  Replaces what Keras/TensorFlow do for the reference in model.fit_generator:
 * autodiff of the graph (models/keras_ssd300.py:263-419) and of SSDLoss (keras_ssd_loss.py:98-211), the kernel_regularizer
 * l2(l2_reg) (models/keras_ssd300.py:274), SGD(lr, momentum) (ssd300_training.ipynb:169) and Adam (ssd7_training.ipynb:153).
 *   ssdk_train_backward  after ssdk_model_forward on the same images: loss + gradients of every kernel / bias / gamma into one
 *                        flat float32 buffer (so that a single NCCL all-reduce covers it).
 *   ssdk_train_apply     g = grad*grad_scale + 2*l2*w (kernels only); v = momentum*v - lr*g; w += v; re-pack the bf16 planes.
 * Parameter order in the flat buffer: layers in graph order, for each conv [kernel as (cout, kh, kw, cin) | bias | BatchNorm
 * gamma | BatchNorm beta], for each head [fused kernel (n_boxes*(C+4), 3, 3, cin) | fused bias], for L2Normalization [gamma].
 * ReLU / linear graphs (SSD300 / SSD512) and conv + BatchNormalization + ELU graphs (SSD7).
 * ------------------------------------------------------------------------------------------ */
typedef struct ssdk_trainer ssdk_trainer;
int ssdk_trainer_create(ssdk_model* m, float* flat_grad_dev /* optional, else allocated */, ssdk_trainer** out);
int ssdk_trainer_destroy(ssdk_trainer* t);
int ssdk_trainer_num_params(const ssdk_trainer* t, long long* out_n);
/* offset (in floats) and element count of a layer's kernel (which=0), bias (1), L2Normalization gamma (2), BatchNormalization
 * gamma (3) or beta (4) inside the flat buffers */
int ssdk_trainer_param_span(const ssdk_trainer* t, int layer, int which, long long* out_offset, long long* out_count);
float* ssdk_trainer_grad_buffer(ssdk_trainer* t);
int ssdk_train_backward(ssdk_trainer* t, const float* y_true_dev, const float* y_pred_dev, int neg_pos_ratio, int n_neg_min,
                        float alpha, float* out_loss_dev /* [B] */, void* stream);
/* The step in pieces, for overlapping the gradient exchange with the backward pass:
 *   ssdk_train_backward_begin   loss + d loss / d y_pred (kept inside the trainer), gradient buffer cleared;
 *   ssdk_train_backward_layers  layers hi .. lo (graph indices, top down, consecutive calls cover n_layers-1 .. 0).  In stream
 *                               order after the call the parameter gradients of exactly these layers are final, so their
 *                               span of the flat buffer (ssdk_trainer_param_span) can be all-reduced on another stream while the
 *                               lower layers are still being differentiated.  dypred_dev NULL = the trainer's own. */
int ssdk_train_backward_begin(ssdk_trainer* t, const float* y_true_dev, const float* y_pred_dev, int neg_pos_ratio, int n_neg_min,
                              float alpha, float* out_loss_dev, void* stream);
int ssdk_train_backward_layers(ssdk_trainer* t, const float* dypred_dev, int hi, int lo, void* stream);
/* The same backward pass from a gradient the caller computed: dypred_dev = d loss / d y_pred, (B,P,C+12) float32 (used with the
 * multi-GPU global-batch-exact loss, whose phases run between NCCL collectives, see ssdk_ssd_loss_phase). */
int ssdk_train_backward_dy(ssdk_trainer* t, const float* dypred_dev, void* stream);
int ssdk_train_apply(ssdk_trainer* t, float lr, float momentum, float l2_reg, float grad_scale, void* stream);
/* Adam as Keras applies it (ssd7_training.ipynb:153: Adam(lr=0.001, beta_1=0.9, beta_2=0.999, epsilon=1e-08, decay=0.0)):
 * g = grad*grad_scale + 2*l2*w (kernels); lr_t = lr*sqrt(1-beta2^t)/(1-beta1^t); m = b1*m + (1-b1)*g; v = b2*v + (1-b2)*g^2;
 * w -= lr_t*m/(sqrt(v)+eps).  `step` = t, counted from 1 by the caller. */
int ssdk_train_apply_adam(ssdk_trainer* t, float lr, float beta1, float beta2, float eps, float l2_reg, float grad_scale, int step,
                          void* stream);
/* Moving mean / variance of a BatchNormalization layer as the training passes left them (float32 [cout] each). */
int ssdk_trainer_read_bn_stats(ssdk_trainer* t, int layer, float* mean_dev, float* var_dev, void* stream);
/* Copy the current float32 master parameters (same order / layout as the gradients) to out_dev. */
int ssdk_trainer_read_params(ssdk_trainer* t, float* out_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SSDK_H_ */
