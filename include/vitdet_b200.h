/*
 * vitdet_b200.h — C ABI of the B200-native ViT-detector forward + anchor-free head decode.
 *
 * This is the drop-in boundary for ONE path of westlake-moonlight/vision_transformer_detector:
 *     create_vision_transformer_detector(...)   vision_transformer_detector.py:498-583
 *     model.predict(images) / model(images)     forward graph built by :239-495
 *     transform_predictions(logits)             :586-647
 *     0.5 / 0.5 score thresholding              :2257-2283 (visualise copy), :1359-1384 (metric copy)
 *
 * The reference has no FFI of its own (it is pure Python on Keras/TF 2.9); the entry points below
 * are what a ctypes binding of that path needs — see INTEGRATION.md for the reference-side stub.
 *
 * Conventions
 *   - every function returns 0 on success or a negative VITDET_E_* code; nothing throws across the
 *     ABI; vitdet_last_error() returns a thread-local, human-readable description of the last failure;
 *   - plain pointers and sizes only; `stream` is a cudaStream_t passed as void* (NULL = legacy
 *     default stream); all device work is asynchronous on that stream unless stated otherwise;
 *   - the caller owns every buffer it passes in; the library owns only its packed weights, its
 *     workspace and (for the *_host calls) its pinned staging buffers;
 *   - one handle per (device, stream); a handle is not thread-safe;
 *   - there is NO CPU fallback: creating a handle without an sm_100 device fails with
 *     VITDET_E_NO_DEVICE.
 */
#ifndef VITDET_B200_H_
#define VITDET_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VITDET_ABI_VERSION 2

enum {
    VITDET_OK = 0,
    VITDET_E_INVALID = -1,      /* bad argument / unsupported configuration */
    VITDET_E_NO_DEVICE = -2,    /* no CUDA device of compute capability 10.x */
    VITDET_E_CUDA = -3,         /* a CUDA runtime / driver call failed */
    VITDET_E_NOT_FOUND = -4,    /* unknown weight name */
    VITDET_E_SHAPE = -5,        /* weight shape mismatch */
    VITDET_E_UNSET = -6         /* forward called before every weight was set */
};

/* Arithmetic mode of the forward pass.
 *   BF16: bf16 operands on the tcgen05 tensor cores, f32 accumulation, f32 residual stream,
 *         LayerNorm / softmax statistics in f32  (tolerance vs the f64 oracle: 2e-2).
 *   FP32: the fp32-accumulate mode (tolerance 1e-3): float32 activations and statistics; by default the Dense layers
 *         run on the tensor cores with every operand split into two bf16 planes (hi + lo, 16 significant bits) and
 *         three tcgen05 passes per product (hi*hi + hi*lo + lo*hi, float32 accumulation, exact activations);
 *         vitdet_set_option(h, "fp32_tc", 0) selects IEEE float32 FMA kernels for every product instead. */
enum { VITDET_MODE_BF16 = 0, VITDET_MODE_FP32 = 1 };

/* Keyword arguments of create_vision_transformer_detector (det.py:498-506) plus the module
 * constants of det.py:19-43 that parameterise the head and the decode. */
typedef struct vitdet_config {
    int32_t image_h, image_w;          /* input_shape[0], input_shape[1]; default Constants.MODEL_IMAGE_SIZE = 608, 608 */
    int32_t patch_size;                /* default 17 */
    int32_t embedding_dim;             /* default 28 */
    int32_t num_heads;                 /* encoder_num_heads, default 8 */
    int32_t key_dim;                   /* encoder_key_dim, default 40; <= 128 (heads wider than 64 run one attention CTA per SM,
                                          and the fp32-accumulate mode takes its CUDA-core form for them) */
    int32_t mlp_quantities;            /* encoder_mlp_quantities, default 8 */
    int32_t repeat_times;              /* encoder_repeat_times, default 8 */
    int32_t head_last_units;           /* mlp_head_last_units, default 136 */
    int32_t head_dense_layers;         /* mlp_head_dense_layers_quantity, default 7 */
    int32_t head_block_repeats;        /* mlp_head_dense_mish_block_repeats, default 1 */
    int32_t use_mish;                  /* 1: Mish, 0: tanh-GELU (tfa.layers.GELU default) */
    int32_t num_slots;                 /* Constants.MAX_DETECT_OBJECTS_QUANTITY = 17 */
    int32_t classes;                   /* Constants.CLASSES = 80 */
    float ln_epsilon;                  /* keras LayerNormalization default 1e-3 */
} vitdet_config;

typedef struct vitdet_handle vitdet_handle;

int vitdet_abi_version(void);
const char* vitdet_last_error(void);

/* Fills *cfg with the reference defaults (det.py:498-506, :19-43). */
void vitdet_default_config(vitdet_config* cfg);

/* Replaces create_vision_transformer_detector(...) (det.py:498-583): validates the configuration,
 * allocates the packed weight storage on the current CUDA device.  Weights start unset. */
int vitdet_create(const vitdet_config* cfg, vitdet_handle** out);
void vitdet_destroy(vitdet_handle* h);

/* Derived shape facts (det.py:274, :285): tokens per image, patch vector length, parameters. */
int vitdet_tokens(const vitdet_handle* h);
int vitdet_patch_dim(const vitdet_handle* h);
int64_t vitdet_count_params(const vitdet_handle* h);

/* Weight exchange — the surface keras `model.weights` / `get_weights()` / `set_weights()` expose
 * (used by the reference at det.py:2123-2125, :2155-2157).  Weights are enumerated in Keras'
 * `model.weights` order and named by Keras variable name without the ':0' suffix
 * (e.g. "multi_head_attention_3/query/kernel"); shapes are the Keras shapes. */
int vitdet_num_weights(const vitdet_handle* h);
int vitdet_weight_info(const vitdet_handle* h, int index, char* name, int name_capacity, int* ndim,
                       int64_t shape[4]);
/* `data` is HOST float32 in Keras layout (Dense kernel = (in, units); MHA kernels (D,H,d)/(H,d,D));
 * synchronous. */
int vitdet_set_weight(vitdet_handle* h, const char* name, const float* data, int ndim, const int64_t* shape);
int vitdet_get_weight(const vitdet_handle* h, const char* name, float* data, int64_t capacity);

/* Encoder micro-batch: images pushed through the encoder per pass (bounds the workspace; the head
 * always runs over the whole batch).  Default 64. */
int vitdet_set_chunk(vitdet_handle* h, int images_per_chunk);
/* Bytes of device workspace a forward of batch B in `mode` uses. */
size_t vitdet_workspace_bytes(const vitdet_handle* h, int B, int mode);

/* Measurement hooks (no reference counterpart; bench.py's live roofline uses them).
 * profile_enable: bit c of the mask turns on CUDA-event timing (on the launching stream) around every
 * launch of kernel category c; profile_read synchronises the pending events and returns the accumulated
 * device time and launch count of one category; launch_count = kernels launched by forward calls. */
int vitdet_profile_enable(vitdet_handle* h, uint32_t category_mask);
int vitdet_profile_num_categories(const vitdet_handle* h);
const char* vitdet_profile_category_name(int category);
int vitdet_profile_read(vitdet_handle* h, int category, double* total_ms, int64_t* launches, int reset);
int64_t vitdet_launch_count(vitdet_handle* h, int reset);

/* ---- run-time switches and debug taps (no reference counterpart; used by the parity tests and A/B measurements) ----
 * Options are per handle; changing one drops the cached launch plans.  Defaults come from the environment variables of
 * the same meaning (VITDET_FUSE_LN, VITDET_FUSE_TAIL, VITDET_GEMM_PAIR, VITDET_FP32) and otherwise are the product path.
 *   "fuse_ln"    1 (default): LayerNorm runs in the epilogue of the GEMM that produces the residual-stream row; 0: stand-alone kernel
 *   "fuse_tail"  1 (default): the last three MLP layers of a block run as one kernel; 0: three GEMM launches
 *   "gemm_pair"  1 (default): CTA-pair GEMM for K >= 512 layers; 0: never; 2: wherever it is legal
 *   "fp32_tc"    1 (default): the fp32 mode's Dense layers run on the tensor cores as three-pass split-bf16 products with
 *                float32 accumulation; 0: IEEE float32 FMA kernels on the CUDA cores (the strict reference form) */
int vitdet_set_option(vitdet_handle* h, const char* key, int value);
int vitdet_get_option(const vitdet_handle* h, const char* key, int* value);

/* Debug taps: while enabled, every forward also keeps a copy of the float32 residual stream after the patch embedding
 * ("embedded_patches", det.py:305-307) and after every encoder block ("block_1" ... "block_L", det.py:408-412), plus
 * "head_last" = the input of MLP_Head_no_Sigmoid (det.py:489).  vitdet_debug_read copies one tap of the LAST forward to
 * a HOST float32 array: [B*tokens, embedding_dim] (or [B*num_slots, head_last_units] for "head_last"); synchronises. */
int vitdet_debug_taps(vitdet_handle* h, int enable);
int vitdet_debug_read(vitdet_handle* h, const char* name, float* out_host, int64_t capacity);

/* Replaces model.predict(x) / model(x, training=False):
 * images_dev: DEVICE float32 NHWC [B, image_h, image_w, 3]; logits_dev: DEVICE float32 [B, num_slots, 6]
 * raw logits (the output of 'MLP_Head_no_Sigmoid', det.py:489-493). */
int vitdet_forward(vitdet_handle* h, const float* images_dev, int B, float* logits_dev, int mode, void* stream);

/* Decode parameters: thresholds (Constants.OBJECTNESS_THRESHOLD / CLASSIFICATION_CONFIDENCE_THRESHOLD),
 * comparison rule and the image size transform_predictions scales by (det.py:637-640). */
typedef struct vitdet_decode_params {
    float objectness_threshold;        /* default 0.5 */
    float classification_threshold;    /* default 0.5 */
    int32_t strict;                    /* 1: keep iff score >  thr (metric rule, det.py:1381-1384)
                                          0: keep iff score >= thr (visualise rule, det.py:2264, :2282) */
    float image_h, image_w;            /* Constants.MODEL_IMAGE_SIZE */
    int32_t classes;                   /* Constants.CLASSES */
    int32_t use_transform_predictions; /* 1 (default): inputs are raw logits, apply transform_predictions first;
                                          0: inputs are already decoded rows (the `use_transform_predictions=False`
                                          path of MeanAveragePrecision.update_state, det.py:1340-1341) */
    float corner_scale;                /* enlarged_image_scale of visualize_predictions (det.py:2294-2325): the corner boxes are
                                          int(cx*s -/+ w*s/2), int(cy*s -/+ h*s/2) clipped to the enlarged image; 0 or 1 = no scaling */
} vitdet_decode_params;

/* Output record arrays of the decode, all DEVICE pointers, any of them may be NULL:
 *   decoded   [R,6] f32  transform_predictions output: conf, class in [0,classes-1], cx, cy, h, w (pixels)
 *   class_id  [R]   i32  round-half-even(class)                              (det.py:1366, :2271)
 *   class_conf[R]   f32  (0.5 - |class - id|) / 0.5                           (det.py:1376, :2279)
 *   keep      [R]   u8   1 iff both scores pass their thresholds
 *   corners   [R,4] i32  x0,y0,x1,y1: int() truncation then clip to the image (det.py:2300-2325)
 *   packed    [R,13] f32 the same record as one row: decoded[6] | class id | class confidence | keep | corners[4]
 *                        (integers are exact in float32) — what vitdet_gather_detections exchanges between GPUs */
#define VITDET_RECORD_FLOATS 13
typedef struct vitdet_detections {
    float* decoded;
    int32_t* class_id;
    float* class_conf;
    uint8_t* keep;
    int32_t* corners;
    float* packed;
} vitdet_detections;

/* Replaces transform_predictions (det.py:586-647) + the threshold rule on R = B*num_slots rows of
 * DEVICE logits.  Stateless: needs no handle. */
int vitdet_decode(const float* logits_dev, int R, const vitdet_decode_params* params,
                  const vitdet_detections* out, void* stream);

/* Same on HOST buffers (what a numpy caller of transform_predictions needs): logits_host [R,6] f32,
 * every non-NULL member of out_host is a HOST array; copies in, decodes on the GPU, copies back,
 * synchronises. */
int vitdet_decode_host(const float* logits_host, int R, const vitdet_decode_params* params,
                       const vitdet_detections* out_host);

/* Replaces iou_calculator(label_bbox, prediction_bbox) (det.py:761-875; "next" row N2 of the hot-path table):
 * element-wise IoU of R box pairs.  Each box is the LAST FOUR floats (cx, cy, h, w — actual pixels) of a row of
 * `width` floats (4 for plain boxes, 6 for label / decoded-prediction rows); iou[r] = I / (U + Constants.EPSILON).
 * vitdet_iou takes DEVICE pointers and is asynchronous; vitdet_iou_host takes HOST pointers and synchronises. */
int vitdet_iou(const float* label_dev, const float* pred_dev, int64_t R, int width, float* iou_dev, void* stream);
int vitdet_iou_host(const float* label_host, const float* pred_host, int64_t R, int width, float* iou_host);

/* Input side ("next" row N4): what _get_image_tensor_coco (vision_transformer_utilities.py:418-449) does after decoding
 * the file: tf.image.resize_with_pad(image, target_h, target_w) (bilinear, half-pixel centres, zero padding), clip to
 * [0, 255], / 127.5, - 1.  image: uint8 [h, w, 3]; out: float32 [target_h, target_w, 3] in [-1, 1].
 * vitdet_preprocess_image takes DEVICE pointers and is asynchronous; the _host variant takes HOST pointers. */
int vitdet_preprocess_image(const uint8_t* image_dev, int h, int w, float* out_dev, int target_h, int target_w, void* stream);
int vitdet_preprocess_image_host(const uint8_t* image_host, int h, int w, float* out_host, int target_h, int target_w);
/* The geometry resize_with_pad derives (resized height / width, top / left padding), in TF's float32 arithmetic. */
int vitdet_resize_with_pad_geometry(int h, int w, int target_h, int target_w, int* resized_h, int* resized_w, int* pad_top, int* pad_left);

/* Forward with the decode fused into the head's last Dense (one launch fewer, logits never re-read).
 * logits_dev may be NULL. */
int vitdet_forward_decode(vitdet_handle* h, const float* images_dev, int B, int mode,
                          const vitdet_decode_params* params, float* logits_dev,
                          const vitdet_detections* out, void* stream);

/* The reference-facing call with HOST buffers (what model.predict + transform_predictions +
 * thresholding do for a numpy caller): copies `images_host` to the device through pinned staging,
 * runs forward+decode, copies the requested outputs back and synchronises.  All pointers are HOST
 * pointers; any output may be NULL. */
int vitdet_predict_host(vitdet_handle* h, const float* images_host, int B, int mode,
                        const vitdet_decode_params* params, float* logits_host,
                        const vitdet_detections* out_host, void* stream);

/* ---- multi-GPU: the path's only exchange (SURVEY §8e) ----
 * Images are independent, so the batch is sharded over one process per GPU with no collective inside the forward; the
 * fixed-size detection records (vitdet_detections.packed, 13 floats per slot) of every rank are then all-gathered in
 * rank order with NCCL over NVLink.  `nccl_comm` is the caller's ncclComm_t (passed as void*: this header needs no
 * nccl.h); the library binds to the libnccl.so.2 that is already loaded in the process (or VITDET_NCCL_LIB).
 * packed_local_dev: [rows_local, 13] on this rank; packed_all_dev: [world * rows_local, 13]; asynchronous on `stream`. */
int vitdet_gather_detections(void* nccl_comm, const float* packed_local_dev, int rows_local, float* packed_all_dev, void* stream);
/* For callers without a communicator of their own: rank 0 obtains a 128-byte id and distributes it by any means (the
 * Python side broadcasts it through torch.distributed); every rank then creates the communicator on its current device. */
int vitdet_nccl_unique_id(char id_out[128]);
int vitdet_nccl_comm_create(const char id[128], int rank, int world, void** nccl_comm_out);
int vitdet_nccl_comm_destroy(void* nccl_comm);

/* ---- uint8 input ("next" row N4, fused with the patch kernel) ----
 * The reference's input pipeline turns uint8 pixels into the model's float32 input with x / 127.5 - 1
 * (vision_transformer_utilities.py:446-447).  These two entry points take the uint8 pixels themselves — NHWC
 * [B, image_h, image_w, 3], already at the model's size — and apply that normalisation inside the patch kernel, so
 * the float32 image is never materialised and the host->device copy is a quarter of the float32 one.  Results are
 * bit-identical to vitdet_forward / vitdet_predict_host on the normalised float32 images. */
/* DEVICE pointers; logits_dev may be NULL when (params, out) are given and vice versa. */
int vitdet_forward_u8(vitdet_handle* h, const uint8_t* images_dev, int B, float* logits_dev, int mode,
                      const vitdet_decode_params* params, const vitdet_detections* out, void* stream);
/* HOST pointers; same contract as vitdet_predict_host. */
int vitdet_predict_host_u8(vitdet_handle* h, const uint8_t* images_host, int B, int mode,
                           const vitdet_decode_params* params, float* logits_host,
                           const vitdet_detections* out_host, void* stream);

/* Asynchronous form of the two host calls above, for callers that stream batches: vitdet_submit_host stages and copies
 * the images (page-locked caller buffers are read directly; ordinary pageable ones are staged through pinned memory by
 * a few threads, overlapped with the copy), enqueues forward + decode + the read-back of the record block on `stream`
 * and returns a ticket; vitdet_collect waits for that ticket and fills the HOST outputs.  Up to two submissions may be
 * in flight per handle: the host->device copy of submission i+1 then overlaps the compute of submission i.
 * images_host must stay valid until the submit call returns (pageable) / until the ticket is collected (page-locked).
 * want_packed: also produce vitdet_detections.packed.  vitdet_predict_host[_u8] = submit + collect. */
int vitdet_submit_host(vitdet_handle* h, const void* images_host, int images_are_uint8, int B, int mode,
                       const vitdet_decode_params* params, int want_packed, void* stream, int* ticket);
int vitdet_collect(vitdet_handle* h, int ticket, float* logits_host, const vitdet_detections* out_host);

/* ---- evaluation metric ("next" row N2): MeanAveragePrecision of the reference (det.py:1268-2060) ----
 * The COCO-style AP of the reference: mean over the IoU thresholds tf.linspace(0.5, 0.95, 10) of the mean, over the
 * classes seen so far, of the class AP computed from the latest `latest_related_images` related images per class
 * with at most `bboxes_per_image` (confidence, IoU) rows each.  The three state tensors of the reference
 * (latest_positive_bboxes, labels_quantity_per_image, showed_up_classes; det.py:1286-1305) live on the device that
 * is current when vitdet_map_create is called. */
typedef struct vitdet_map vitdet_map;

/* MeanAveragePrecision.__init__ (det.py:1280-1308).  The reference's constants are classes = 80,
 * latest_related_images = 3 (Constants.LATEST_RELATED_IMAGES, det.py:32), bboxes_per_image = 14
 * (Constants.BBOXES_PER_IMAGE, det.py:37). */
int vitdet_map_create(int classes, int latest_related_images, int bboxes_per_image, vitdet_map** out);
void vitdet_map_destroy(vitdet_map* m);

/* reset_state (det.py:2052-2060): zero the three state tensors.  Asynchronous on `stream`. */
int vitdet_map_reset(vitdet_map* m, void* stream);

/* update_state(y_true, y_pred, use_transform_predictions) (det.py:1310-1862).  y_true_dev, y_pred_dev: DEVICE
 * float32 [batch, slots, 6] rows (objectness, class, cx, cy, h, w): labels as the reference builds them (empty
 * slots hold objectness 0 and -8 elsewhere), predictions either raw head outputs
 * (params->use_transform_predictions = 1: transform_predictions is applied first, using params->image_h/w and
 * params->classes) or already decoded rows (0).  Uses params->objectness_threshold / classification_threshold with
 * the metric's strict '>' rule (params->strict and corner_scale are ignored).  The images of the batch are taken
 * in order, as the reference's `for sample in range(batch_size)` does.  Asynchronous on `stream`; y_pred_dev can be
 * the logits buffer vitdet_forward just wrote on the same stream. */
int vitdet_map_update(vitdet_map* m, const float* y_true_dev, const float* y_pred_dev, int batch, int slots,
                      const vitdet_decode_params* params, void* stream);
/* Same with HOST arrays; copies in, updates, synchronises. */
int vitdet_map_update_host(vitdet_map* m, const float* y_true_host, const float* y_pred_host, int batch, int slots,
                           const vitdet_decode_params* params);

/* result() (det.py:1865-2049).  HOST outputs: *mean_ap; per_iou_host[10] (AP averaged over the seen classes, per
 * IoU threshold; may be NULL); per_class_host[10 * classes] (AP per threshold and class, 0 for classes not seen;
 * may be NULL).  Runs on `stream` and synchronises it. */
int vitdet_map_result(vitdet_map* m, float* mean_ap_host, float* per_iou_host, float* per_class_host, void* stream);

/* The state in the reference's layout, to HOST arrays (any may be NULL): latest_positive_bboxes
 * [classes, latest_related_images, bboxes_per_image, 2] f32, labels_quantity_per_image
 * [classes, latest_related_images] f32, showed_up_classes [classes] u8 (0/1).  Synchronises `stream`. */
int vitdet_map_state(vitdet_map* m, float* bboxes_host, float* labels_host, uint8_t* showed_host, void* stream);

/* The ten float32 IoU thresholds result() uses (tf.linspace(0.5, 0.95, num=10), det.py:1876). */
int vitdet_map_iou_thresholds(const vitdet_map* m, float* out10);

/* Number of kernels this metric object has launched so far. */
uint64_t vitdet_map_launch_count(const vitdet_map* m);

/* ---- operator-level entry points (the Keras layers the path is built from; used by the parity
 * tests to check each kernel against the oracle in isolation).  All pointers are DEVICE pointers. ---- */

/* keras.layers.Dense (+ activation + residual): out[M,N] = act(A[M,K] @ kernel[K,N] + bias) + resid.
 * A, kernel (Keras layout), bias, resid, out are float32; mode selects the tensor-core (operands
 * rounded to bf16) or the f32 CUDA-core kernel.  act: 0 none, 1 Mish, 2 tanh-GELU.  Synchronous. */
int vitdet_op_dense(const float* A, const float* kernel, const float* bias, const float* resid, float* out,
                    int M, int K, int N, int act, int mode, void* stream);
/* keras.layers.LayerNormalization(axis=-1): x, y [M,D] f32. */
int vitdet_op_layernorm(const float* x, const float* gamma, const float* beta, float* y, int M, int D,
                        float eps, void* stream);
/* Core of keras.layers.MultiHeadAttention after the q/k/v projections:
 * q,k,v,out: [B,T,H,d] f32 (q already includes its bias, NOT yet scaled by 1/sqrt(d)). Synchronous. */
int vitdet_op_attention(const float* q, const float* k, const float* v, float* out, int B, int T, int H,
                        int d, int mode, void* stream);
/* tf.image.extract_patches(SAME) + Reshape: images [B,H,W,3] f32 -> patches [B*T, 3*p*p] f32. */
int vitdet_op_patchify(const float* images, int B, int H, int W, int p, float* patches, void* stream);

/* Extras of the tensor-core Dense epilogue that the plain call above does not reach (bf16 mode only):
 *   pos / pos_period     per-row scalar pos[m % pos_period] added before the activation (the position embedding fused
 *                        into the linear_projection GEMM, det.py:291-307); NULL = none
 *   ln_gamma, ln_beta, ln_eps, ln_out
 *                        fused LayerNormalization of the finished output row (N <= 32 only): ln_out [M,N] receives, as
 *                        float32, the bf16 values the kernel hands to the next GEMM; NULL = none
 *   store_bf16           1: run the bf16-output epilogue (bias + activation on packed pairs, TMA store) and widen the stored
 *                        bf16 result to float32 in `out`; resid must be NULL.  0: the float32-output epilogue
 *   pair                 -1: choose as the forward pass does; 0: single-CTA kernel; 1: CTA-pair kernel */
typedef struct vitdet_dense_ex {
    const float* pos; int32_t pos_period;
    const float* ln_gamma; const float* ln_beta; float ln_eps; float* ln_out;
    int32_t store_bf16;
    int32_t pair;
} vitdet_dense_ex;
int vitdet_op_dense_ex(const float* A, const float* kernel, const float* bias, const float* resid, float* out,
                       int M, int K, int N, int act, const vitdet_dense_ex* ex, void* stream);
/* The fused tail of the encoder MLP pyramid (csrc/mlp_tail.cu; det.py:388-412 for the last three layers + the next
 * block's LayerNormalization det.py:353): x += act(act(act(A W0 + b0) W1 + b1) W2 + b2), ln_out = LN(x).
 * A [M,K0], kernels in Keras layout W0 [K0,N0], W1 [N0,N1], W2 [N1,N2], x [M,N2] float32 in/out, ln_out [M,N2] float32
 * (widened bf16) or NULL with ln_gamma/ln_beta.  Fails with VITDET_E_INVALID for widths the kernel does not take. */
int vitdet_op_mlp_tail(const float* A, const float* W0, const float* b0, const float* W1, const float* b1, const float* W2,
                       const float* b2, float* x, const float* ln_gamma, const float* ln_beta, float ln_eps, float* ln_out,
                       int M, int K0, int N0, int N1, int N2, int act, void* stream);
/* mlp_head first stage (det.py:454-463): Dense(D -> S) on every token of `images` images of `tokens` tokens, stored as the
 * reference's Reshape((S, -1)) lays it out: out [images*S, tokens] float32 (mode bf16: widened from the stored bf16). */
int vitdet_op_head_slots(const float* x, const float* kernel, const float* bias, float* out, int images, int tokens, int D,
                         int S, int mode, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VITDET_B200_H_ */
