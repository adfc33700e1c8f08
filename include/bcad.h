/*
 * libbcad -- B200-native predict + Grad-CAM for the vision-xai-breast-cancer-cad hot path.
 *
 * Plain C ABI: opaque handle, plain pointers and sizes, int status codes (0 = ok, <0 = error,
 * text via bcad_last_error()).  No torch types.  Device pointers are owned by the caller; the
 * handle owns only weights and workspace.  Every entry point is re-entrant per (handle, stream).
 *
 * The reference has NO FFI/plugin seam (SURVEY section 8b): its boundary is plain Python classes
 * and functions.  Each entry point below cites the reference Python interface it stands behind;
 * the ctypes binding a maintainer adds is shown in INTEGRATION.md and implemented in
 * vision-xai-breast-cancer-cad_b200/_lib.py.
 */
#ifndef BCAD_H
#define BCAD_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BCAD_MAX_CONV 8
#define BCAD_MAX_DENSE 8

/* status codes */
#define BCAD_OK 0
#define BCAD_ERR_INVALID (-1)      /* bad argument / shape / unsupported configuration (-> ValueError) */
#define BCAD_ERR_CUDA (-2)         /* CUDA runtime error (-> RuntimeError) */
#define BCAD_ERR_STATE (-3)        /* call order (weights not committed, no cached forward, ...) */
#define BCAD_ERR_NOMEM (-4)

/* cfg.flatten_order: how the CALLER's first dense weight matrix indexes the flattened pool output */
#define BCAD_FLATTEN_HWC 0         /* out.flatten() of an (h,w,C) array: Classes/CNNModel.py:178 */
#define BCAD_FLATTEN_CHW 1         /* x.reshape(B,-1) of NCHW:            ADCNNM.py:77 */
/* cfg.pool_ties: max-pool backward when several window elements equal the maximum */
#define BCAD_TIES_ALL 0            /* gradient duplicated to every tie: Classes/CNNModel.py:260,274-275 */
#define BCAD_TIES_FIRST 1          /* first maximum in row-major window order: nn.MaxPool2d (ADCNNM.py:49) */
/* cfg.head */
#define BCAD_HEAD_SOFTMAX_CLIP 0   /* probs = softmax(clip(z,+-50)) /(sum+1e-12): Classes/CNNModel.py:203-212 */
#define BCAD_HEAD_LOGITS 1         /* raw logits out, probs = softmax(logits): ADCNNM.py:78, app.py:593 */
/* cfg.precision */
#define BCAD_PREC_FP32 0           /* fp32 CUDA-core path, any shape */
#define BCAD_PREC_F16 1            /* 16-bit tcgen05 tensor-core path (fp16 operands, fp32 accumulate) where the shape allows */
#define BCAD_PREC_F16X3 2          /* tensor-core path with hi+lo fp16 split operands (3 MMAs per product): fp32-grade results;
                                    * the only tensor mode that accepts BCAD_TIES_ALL (the rule compares activations for equality) */
/* grad_mode: gradient injected at the network output for the explanation */
#define BCAD_GRAD_LOGIT 0          /* d(logit_c): pytorch_grad_cam ClassifierOutputTarget, GRADCAM.py:64 */
#define BCAD_GRAD_SOFTMAX_CE 1     /* probs - onehot(c): explainability.py:21-22 */
/* explain target (bcad_set_explain_target): which tensor of the last conv block Grad-CAM explains */
#define BCAD_TARGET_CONV_ACT 0     /* post-LeakyReLU, pre-pool output = layer['output'] / conv_act_grads (explainability.py:64): default */
#define BCAD_TARGET_CONV_PREACT 1  /* the nn.Conv2d module's own output, before F.leaky_relu: what pytorch_grad_cam captures when it hooks
                                    * model.convs[-1] of ADCNNM.CNNModel (the activation there is functional, ADCNNM.py:76) */
/* bcad_get_tensor kinds (cached by the most recent forward of <= max_batch images) */
#define BCAD_T_CONV_OUT 0          /* layer['output'] of conv block i, NHWC fp32 (Classes/CNNModel.py:169) */
#define BCAD_T_POOL_OUT 1          /* layer['output'] of pool block i, NHWC fp32 (:174) */
#define BCAD_T_DENSE_Z 2           /* layer['z'] of dense/output layer j (:181,194) */
#define BCAD_T_ALPHA 3             /* Grad-CAM channel weights alpha_k of the last explain call, [B,F] */
#define BCAD_T_CAM_LOWRES 4        /* ReLU(sum_k alpha_k A_k) before normalisation, [B,h,w] */

#if defined(__GNUC__)
#define BCAD_API __attribute__((visibility("default")))
#else
#define BCAD_API
#endif

typedef struct bcad_model bcad_model;
typedef struct bcad_unet bcad_unet;     /* tiny U-Net encoder front on the tensor cores (below) */

typedef struct bcad_config {
    int32_t in_h, in_w, in_c;               /* input_shape (H,W,C): Classes/CNNModel.py:68, ADCNNM.py:42 */
    int32_t num_classes;
    int32_t n_conv;
    int32_t conv_filters[BCAD_MAX_CONV];    /* conv_layers[i][0] */
    int32_t conv_ksize[BCAD_MAX_CONV];      /* conv_layers[i][1] */
    int32_t n_hidden;
    int32_t hidden_units[BCAD_MAX_DENSE];
    float alpha_conv;                       /* LeakyReLU slope after convs (ADCNNM.py:76 hard-wires 0.01) */
    float alpha_dense;                      /* LeakyReLU slope after hidden dense layers */
    int32_t pad;                            /* zero padding per side: 0 (NumPy CNN) or 1 (ADCNNM.py:48) */
    int32_t flatten_order;
    int32_t pool_ties;
    int32_t head;
    int32_t precision;
    int32_t max_batch;                      /* workspace is sized for this many images; larger calls are chunked */
    int32_t keep_all_activations;           /* 1: also cache every conv block's pre-pool output (compat .layers, saliency);
                                             *    on the 16-bit path: also write out the pooled first-block map, which the fused
                                             *    conv kernel otherwise keeps on chip (bcad_get_tensor(BCAD_T_POOL_OUT, 0)) */
    int32_t device;                         /* CUDA device ordinal */
    float refine_margin;                    /* BCAD_PREC_F16 only, 0 = off: an image whose two largest logits are closer than this is
                                             * re-run through the split-operand (fp32-grade) kernels inside the same call, so that the
                                             * predicted class is the fp32-grade one (north_star: classes bit-exact; the 16-bit logit
                                             * error is ~3e-3, ADCNNM.py:72-78 + app.py:589 torch.max).  Needs a shape BCAD_PREC_F16X3 covers. */
    int32_t refine_capacity;                /* images per chunk the refinement pass is sized for; 0 = max(8, max_batch/32).  Flagged images
                                             * beyond it keep their 16-bit result and are counted (bcad_refine_stats). */
} bcad_config;

/* ---- lifetime ------------------------------------------------------------------------------- */
/* CNNModel.__init__/_build_model (Classes/CNNModel.py:68-157), ADCNNM.CNNModel.__init__ (ADCNNM.py:35-70) */
BCAD_API int bcad_create(const bcad_config* cfg, bcad_model** out);
BCAD_API void bcad_destroy(bcad_model* m);
/* thread-local message of the last failing call */
BCAD_API const char* bcad_last_error(void);
BCAD_API const char* bcad_version(void);

/* ---- weights: load_weights (Classes/CNNModel.py:30-60), load_trained_model (ADCNNM.py:155-202) */
/* filters: HOST fp32 (F,k,k,C) -- the NumPy layout (Classes/CNNModel.py:94); bias: HOST fp32 (F,) */
BCAD_API int bcad_set_conv_weights(bcad_model* m, int conv_idx, const float* filters_fkkc, const float* bias);
/* W: HOST fp32 (units,in); for dense_idx 0 the `in` index follows cfg.flatten_order; bias (units,).
 * dense_idx runs over the hidden layers then the output layer (n_hidden + 1 matrices). */
BCAD_API int bcad_set_dense_weights(bcad_model* m, int dense_idx, const float* w_units_in, const float* bias);
/* optional inference-time BatchNorm fold (identity for reference models, README.md:87-93):
 * w' = w*gamma/sqrt(var+eps), b' = (b-mean)*gamma/sqrt(var+eps)+beta, applied to the staged conv. */
BCAD_API int bcad_fold_batchnorm(bcad_model* m, int conv_idx, const float* gamma, const float* beta,
                        const float* mean, const float* var, float eps);
/* packs / uploads everything staged so far; required before the first predict */
BCAD_API int bcad_commit(bcad_model* m);

/* ---- the hot path, DEVICE buffers ------------------------------------------------------------- */
/* forward(x, training=False) + predict (Classes/CNNModel.py:162-198, 524-526); model(inputs) +
 * torch.max + torch.softmax (ADCNNM.py:72-78, app.py:584-593).
 * x_dev: fp32 NHWC [B,H,W,C].  Outputs (each may be NULL): logits/probs [B,num_classes] fp32,
 * cls [B] int32 (first maximum).  stream: cudaStream_t (NULL = legacy default stream). */
BCAD_API int bcad_predict(bcad_model* m, const float* x_dev, int B, float* logits_dev, float* probs_dev,
                 int32_t* cls_dev, void* stream);

/* predict + Grad-CAM on the last conv block's post-LeakyReLU output
 * (generate_dual_class_gradcam_overlays_pytorch GRADCAM.py:31-81 with the tail of pytorch_grad_cam;
 * ExplainableAI.generate_heatmap Classes/ExplainableAI.py:14).
 * class_idx_dev: int32 [B] target classes or NULL = each image's predicted class (GRADCAM.py:60-61).
 * heatmap_dev: fp32 [B,H,W] in [0,1]. */
BCAD_API int bcad_predict_explain(bcad_model* m, const float* x_dev, int B, const int32_t* class_idx_dev,
                         int grad_mode, float* logits_dev, float* probs_dev, int32_t* cls_dev,
                         float* heatmap_dev, void* stream);

/* Same call with the heat-map bilinearly resized to out_h x out_w instead of the model's input size: pytorch_grad_cam scales the
 * low-resolution cam to the size of the image it was asked about, and the reference asks about a 512x512 image whatever its CNN
 * was fed (app.py:649-657 -> GRADCAM.py:46-64).  heatmap_dev: fp32 [B,out_h,out_w]. */
BCAD_API int bcad_predict_explain_sized(bcad_model* m, const float* x_dev, int B, const int32_t* class_idx_dev, int grad_mode,
                               float* logits_dev, float* probs_dev, int32_t* cls_dev, int out_h, int out_w, float* heatmap_dev,
                               void* stream);

/* Predict + Grad-CAM for K target classes per image from ONE forward: the deployed dual-class explanation (app.py:649-657 ->
 * GRADCAM.py:63-64 with classes_to_test) as one batched call.  1 <= K <= BCAD_MAX_EXPLAIN_CLASSES; classes_dev: int32 [B][K] on
 * the device (duplicates allowed), or NULL = column k explains class k (K <= num_classes).  out_h = out_w = 0: heat-maps of the
 * model's input size, else scaled to out_h x out_w as bcad_predict_explain_sized does.  heatmap_dev: fp32 [B][K][H][W].
 * logits / probs / cls as bcad_predict_explain (each may be NULL).  heat[:, k], logits, probs and classes are bitwise equal to
 * bcad_predict_explain_sized on the same handle with class column k (images re-run by the refinement twin included).  Afterwards
 * bcad_get_tensor(BCAD_T_ALPHA | BCAD_T_CAM_LOWRES) returns BCAD_ERR_STATE: those caches describe one class. */
#define BCAD_MAX_EXPLAIN_CLASSES 8
BCAD_API int bcad_predict_explain_classes(bcad_model* m, const float* x_dev, int B, int K, const int32_t* classes_dev, int grad_mode,
                                          float* logits_dev, float* probs_dev, int32_t* cls_dev, int out_h, int out_w,
                                          float* heatmap_dev, void* stream);

/* compute_backprops_for_explainability (explainability.py:13-68), activation-gradient part:
 * uses the activations cached by the preceding bcad_predict of the SAME B (<= max_batch,
 * keep_all_activations=1 when gradients below the last conv block are wanted).
 * conv_act_grads_dev[i]: fp32 NHWC gradient w.r.t. conv block i's post-activation output, or NULL to
 * skip (entries below the lowest requested block are not computed); d_input_dev: fp32 [B,H,W,C] or NULL. */
BCAD_API int bcad_explain_backward(bcad_model* m, int B, const int32_t* class_idx_dev, int grad_mode,
                          float* const* conv_act_grads_dev, float* d_input_dev, void* stream);

/* Input-gradient saliency (explainability.py:44-78) for K target classes per image from ONE forward.  fp32 handles with
 * keep_all_activations = 1 and no dropout masks set.  The kernels follow bcad_set_fast_training, as bcad_predict / bcad_train_backward
 * do: with it on, the eligible conv blocks and fc1 run their input gradients on the split-operand tensor-core kernels (~1e-4 relative).
 * A first block of one input channel, 32 filters, 3x3 and pad 0 / 1 runs as one fused kernel (plain fp32, summation order aside the
 * same as bcad_explain_backward's d_input).  Chunked by max_batch: one forward per chunk, then one backward per class.
 * classes_dev int32 [B][K] or NULL (column k = class k, K <= num_classes); 1 <= K <= BCAD_MAX_EXPLAIN_CLASSES; grad_mode BCAD_GRAD_*
 * (the reference uses SOFTMAX_CE).  saliency_dev fp32 [B][K][H][W] = (s - min s) / (max s - min s + 1e-8), s = max_c |d_input| per
 * image and class.  d_input_dev fp32 [B][K][H][W][C] or NULL.  logits / probs / cls as bcad_predict_explain (each may be NULL).
 * saliency[:, k] and d_input[:, k] are bitwise what a K = 1 call with class column k returns; logits / probs / cls are bitwise
 * bcad_predict's.  Afterwards the layer caches describe the last chunk's forward, as after bcad_predict. */
BCAD_API int bcad_predict_saliency_classes(bcad_model* m, const float* x_dev, int B, int K, const int32_t* classes_dev, int grad_mode,
                                           float* logits_dev, float* probs_dev, int32_t* cls_dev, float* saliency_dev,
                                           float* d_input_dev, void* stream);
/* generate_saliency_overlay (explainability.py:74-77) for [B][K] maps: heat = JET_BGR[uint8(sal * 255)] (fp32 product, truncating),
 * overlay = addWeighted(base, 0.5, heat, 0.5, 0) (round half to even, as OpenCV's 8-bit path does).  base_dev uint8 [B][H][W][base_c],
 * base_c = 1 (replicated to 3) or 3, shared by an image's K maps.  overlay_dev / heat_dev uint8 [B][K][H][W][3] (BGR), either may be NULL. */
BCAD_API int bcad_saliency_overlay(const uint8_t* base_dev, int base_c, const float* saliency_dev, int B, int K, int H, int W,
                                   uint8_t* overlay_dev, uint8_t* heat_dev, void* stream);

/* cached tensors of the most recent forward / explain (layer['output'], ['z'] ... compat) -> dst_dev */
BCAD_API int bcad_get_tensor(bcad_model* m, int kind, int index, int B, float* dst_dev, void* stream);
/* number of fp32 elements per image of that tensor */
BCAD_API int64_t bcad_tensor_elems(bcad_model* m, int kind, int index);

/* ---- the hot path, HOST buffers (the end-to-end call: H2D, compute, D2H, chunked and overlapped) */
/* x_host: fp32 [B,H,W,C]; outputs host (NULL to skip); pinned memory makes the copies asynchronous. */
BCAD_API int bcad_predict_explain_host(bcad_model* m, const float* x_host, int B, const int32_t* class_idx_host,
                              int grad_mode, float* logits_host, float* probs_host, int32_t* cls_host,
                              float* heatmap_host);
/* Same call, heat-maps as heatmap_uint8 = (cam * 255).astype(uint8) (GRADCAM.py:70, truncating) [B,H,W]: the caller that
 * only writes PNGs (app.py:715,750) gets a quarter of the device->host bytes (the call is PCIe-bound). */
BCAD_API int bcad_predict_explain_host_u8(bcad_model* m, const float* x_host, int B, const int32_t* class_idx_host_or_null,
                                 int grad_mode, float* logits_host, float* probs_host, int32_t* cls_host,
                                 uint8_t* heat_u8_host);
/* 8-bit images in: x_u8_host uint8 [B,H,W,C] (a decoded PNG / the 0-255 grey image the callers hold, app.py:629-639),
 * normalised on the device as x = float32(u8) / 255.0f (app.py:71, GRADCAM.py:46) -- a quarter of the host->device
 * bytes, results bit-identical to passing that float32 array.  Heat-maps as float32 (heatmap_host) or uint8
 * (heat_u8_host); exactly one of the two may be non-NULL, both NULL = predict only. */
BCAD_API int bcad_predict_explain_host_u8in(bcad_model* m, const uint8_t* x_u8_host, int B, const int32_t* class_idx_host_or_null,
                                   int grad_mode, float* logits_host, float* probs_host, int32_t* cls_host,
                                   float* heatmap_host, uint8_t* heat_u8_host);

/* generate_dual_class_gradcam_overlays_pytorch (GRADCAM.py:31-81) for a BATCH of 8-bit grey images, end to end: gray_u8_host uint8
 * [B,H,W] (model input size) -> img01 = u8 / 255 (GRADCAM.py:46) -> CNN input (standardise = 1: (img01 - mean) / (std + 1e-8) per
 * image as app.py:179-182 prepares CNN inputs, 0: img01 itself; replicated over in_c channels) -> predict + Grad-CAM ->
 * overlay_rgb_host uint8 [B,H,W,3] = show_cam_on_image(img_rgb, cam, use_rgb=True) (GRADCAM.py:67) and heat_u8_host uint8 [B,H,W] =
 * (cam * 255).astype(uint8) (GRADCAM.py:70); either may be NULL.  Same chunked three-stream pipeline as above. */
BCAD_API int bcad_gradcam_overlays_host(bcad_model* m, const uint8_t* gray_u8_host, int B, const int32_t* class_idx_host_or_null,
                               int grad_mode, int standardise, float* logits_host, float* probs_host, int32_t* cls_host,
                               uint8_t* overlay_rgb_host, uint8_t* heat_u8_host);

/* ---- stand-alone Grad-CAM tail (pytorch_grad_cam BaseCAM.forward / scale_cam_image) ------------ */
/* A, dA: [B,h,w,K] NHWC device, dtype 0 = fp32, 1 = bf16; out: fp32 [B,H,W].
 * alpha_k = mean_hw dA_k ; cam = ReLU(sum_k alpha_k A_k) ; min-max ; bilinear (cv2.resize) ; min-max. */
BCAD_API int bcad_gradcam_tail(const void* A_dev, const void* dA_dev, int B, int K, int h, int w, int H, int W,
                      int dtype, float* out_dev, void* stream);

/* ---- input stage of the GRADCAM.py surface, DEVICE buffers: gray_u8_dev uint8 [B,H,W] -> img01_dev fp32 [B,H,W] = u8 / 255
 * (GRADCAM.py:46) and the CNN input x_dev fp32 [B,H,W,C]: standardise = 1: (img01 - mean) / (std + 1e-8) per image (the reference's
 * CNN-input normalisation, app.py:179-182; mean / std from exact integer sums), 0: img01; the channel replicated C times. */
BCAD_API int bcad_gray_preprocess(const uint8_t* gray_u8_dev, int B, int H, int W, int C, int standardise, float* img01_dev,
                         float* x_dev, void* stream);

/* ---- overlay stage (show_cam_on_image GRADCAM.py:67, heatmap_uint8 GRADCAM.py:70) -------------- */
/* img01_dev: fp32 [B,H,W] grayscale in [0,1]; cam_dev: fp32 [B,H,W]; overlay_rgb_dev: u8 [B,H,W,3]
 * (NULL to skip); heat_u8_dev: u8 [B,H,W] (NULL to skip). */
BCAD_API int bcad_overlay(const float* img01_dev, const float* cam_dev, int B, int H, int W,
                 uint8_t* overlay_rgb_dev, uint8_t* heat_u8_dev, void* stream);

/* ---- tiny U-Net encoder front (SURVEY 8 row f1): conv2d + relu + max_pool of Classes/unet.py:13-73 ------- */
/* y = LeakyReLU_alpha(conv(x, kernel) + bias), NHWC fp32, kernel DEVICE fp32 (k,k,Cin,Cout) as unet.py holds it, bias
 * DEVICE (Cout) or NULL.  padded_output=1 reproduces conv2d(..., 'same') of unet.py:19-27: the output has the PADDED
 * size (H+2*pad, W+2*pad), the true convolution in its top-left corner and zeros elsewhere.  y [B,Ho,Wo,Cout] and/or
 * pooled [B,Ho/2,Wo/2,Cout] (2x2/2 max-pool, unet.py:32-43); either may be NULL.  alpha=0 is ReLU (unet.py:53). */
BCAD_API int bcad_conv_block(const float* x_dev, int B, int H, int W, int Cin, const float* kernel_kkcf_dev,
                    const float* bias_dev, int k, int Cout, int pad, float alpha, int padded_output,
                    float* y_dev, float* pooled_dev, void* stream);
/* non-overlapping mean pool, floor dims (Classes/ImageSegmentation.py:145-163): [B,H,W,C] -> [B,H/pool,W/pool,C] */
BCAD_API int bcad_avg_pool(const float* x_dev, int B, int H, int W, int C, int pool, float* out_dev, void* stream);

/* The same front as ONE tensor-core pipeline behind a handle (BASELINE config 3: U-Net -> CNN -> Grad-CAM at batch 256), for
 * single-channel images with H, W multiples of 4: tiny_unet_numpy (Classes/unet.py:61-73: conv(1->16)+ReLU+pool, conv(16->32)+ReLU+
 * pool, conv(32->64)+ReLU, every conv with the padded-size-output quirk of unet.py:19-27) followed by average_pool
 * (Classes/ImageSegmentation.py:145-163).  conv1 on CUDA cores (K = 9), conv2 / conv3 as tcgen05 implicit GEMMs with fp16 operands
 * and fp32 accumulation (results within 1e-2 of the map's scale; bcad_conv_block above is the fp32 route for every other shape).
 * The handle owns the weight images and the intermediate maps: no allocation on the forward path. */
BCAD_API int bcad_unet_create(int H, int W, int max_batch, int device, bcad_unet** out);
BCAD_API void bcad_unet_destroy(bcad_unet* u);
/* kernels as unet.py holds them, HOST fp32: k1 (3,3,1,16), k2 (3,3,16,32), k3 (3,3,32,64) */
BCAD_API int bcad_unet_set_kernels(bcad_unet* u, const float* k1_host, const float* k2_host, const float* k3_host);
/* output shape per image: avg_pool = 0 -> the reference's bn tensor (H/4+3, W/4+3, 64) incl. its two zero rows / columns;
 * avg_pool = p > 0 -> average_pool(bn, p): floor((H/4+3)/p) x floor((W/4+3)/p) x 64 (256x256, p = 3: 22 x 22 x 64) */
BCAD_API int bcad_unet_out_shape(bcad_unet* u, int avg_pool, int* out_h, int* out_w, int* out_c);
/* x_dev: fp32 [B,H,W] (single channel); out_dev: fp32 NHWC [B,out_h,out_w,64] */
BCAD_API int bcad_unet_forward(bcad_unet* u, const float* x_dev, int B, int avg_pool, float* out_dev, void* stream);
BCAD_API int64_t bcad_unet_launch_count(bcad_unet* u);
/* per-stage device times of the last forward's last chunk (CUDA events before every launch), stages 0..4 */
BCAD_API int bcad_unet_set_profiling(bcad_unet* u, int on);
BCAD_API int bcad_unet_profile_get(bcad_unet* u, int i, char* name_buf, int name_cap, float* ms);

/* ---- feeding producer of the basic classifier (app.py:466-489 process_bottleneck_features) ----------------------------- */
/* feat_dev: fp32 [B][C][H][W] (layout 0) or [B][H][W][C] (layout 1) -> cv2.resize(.., (out_w, out_h), INTER_LINEAR) ->
 * out_dev fp32 [B][out_h][out_w][C].  Bit-exact with OpenCV 4.13's float paths (> 4 channels: float32 coordinates). */
BCAD_API int bcad_bottleneck_resize(const float* feat_dev, int B, int C, int H, int W, int layout, int out_h, int out_w,
                           float* out_dev, void* stream);

/* ---- training step (SURVEY 8 row f4, BASELINE config 5): fp32 path, keep_all_activations=1 ------------------------ */
/* Flat gradient vector: per conv block [W packed (k*k,Cin,CoutPad) | b (CoutPad)], then per dense layer [W (out,in) | b (out)]
 * -- the layouts the device weights live in, every tensor starting on a 128-byte boundary (bcad_grad_layout gives the
 * offsets; the gaps are never read), so the optimiser and an all-reduce can treat it as one opaque fp32 buffer. */
BCAD_API int64_t bcad_grad_elems(bcad_model* m);
BCAD_API int bcad_grad_layout(bcad_model* m, int is_dense, int index, int64_t* w_off, int64_t* w_elems, int64_t* b_off,
                     int64_t* b_elems);
/* Gradients of the MEAN softmax cross-entropy over the B images of the preceding bcad_predict(x, B) w.r.t. every weight and
 * bias (_compute_sample_grads summed and divided by n: Classes/CNNModel.py:282-355, 459-464; nn.CrossEntropyLoss
 * ADCNNM.py:89).  labels_dev: int32 [B]; grads_dev: fp32 [bcad_grad_elems]; loss_dev: fp32 [B] per-sample loss or NULL. */
BCAD_API int bcad_train_backward(bcad_model* m, const float* x_dev, const int32_t* labels_dev, int B, float* grads_dev,
                        float* loss_dev, void* stream);
/* The same in two parts, for a data-parallel step that overlaps communication with the backward: part 1 = loss + dense layers
 * (their gradients -- 99.9 % of the bytes, fc1 -- are final when it returns), part 2 = the conv blocks; part 0 = both. */
BCAD_API int bcad_train_backward_part(bcad_model* m, const float* x_dev, const int32_t* labels_dev, int B, float* grads_dev,
                             float* loss_dev, int part, void* stream);
/* Dropout multipliers for the next forwards of exactly B images (B <= max_batch): masks[b][sum of hidden units] (host or
 * device pointer), hidden layers in order, each value 0 or 1/(1-rate) -- Classes/CNNModel.py:186-188, nn.Dropout of
 * ADCNNM.py:62.  The caller draws them.  NULL or B = 0 switches dropout off.  bcad_train_backward feeds the dropped
 * activations to the weight gradients; mask_backward = 1 also masks the back-propagated gradient (autograd, ADCNNM.py),
 * 0 leaves it unmasked as the NumPy reference's backward does (Classes/CNNModel.py:307-316). */
BCAD_API int bcad_set_dropout_masks(bcad_model* m, const float* masks, int B, int mask_backward, void* stream);
/* Fast training (off by default): eligible conv blocks (3x3, 32 -> 64 filters, maps <= 128 px wide) run forward / input gradient / weight
 * gradient on tcgen05 with split (hi + lo) operands; fp32 tensors in and out.  Replaces the per-block work of
 * Classes/CNNModel.py:227-240, 320-355 / torch autograd (ADCNNM.py:100-118) at ~1e-4 relative instead of fp32 rounding.
 * BCAD_ERR_INVALID when no block of the network is eligible or the handle is not BCAD_PREC_FP32. */
BCAD_API int bcad_set_fast_training(bcad_model* m, int on);

/* opt 0: w -= lr * clip(g), per-tensor L2-norm clipping at max_norm (Classes/CNNModel.py:217-222, 372-394; 0 = no clip);
 * opt 1: Adam(lr, b1, b2, eps) as torch.optim.Adam (ADCNNM.py:88).  grads_dev usually comes back from an all-reduce. */
BCAD_API int bcad_apply_update(bcad_model* m, const float* grads_dev, int opt, float lr, float max_norm, float b1, float b2,
                      float eps, void* stream);
/* current weights in the caller's layouts: filters (F,k,k,C) + bias; dense (units,in) in cfg.flatten_order + bias (HOST) */
BCAD_API int bcad_get_conv_weights(bcad_model* m, int conv_idx, float* filters_fkkc_host, float* bias_host);
BCAD_API int bcad_get_dense_weights(bcad_model* m, int dense_idx, float* w_units_in_host, float* bias_host);

/* ---- introspection ---------------------------------------------------------------------------- */
/* Grad-CAM target tensor for the following explain calls of this handle (BCAD_TARGET_*; fp32 path only for CONV_PREACT) */
BCAD_API int bcad_set_explain_target(bcad_model* m, int target);
/* refinement counters since creation (cfg.refine_margin > 0): images re-run at fp32 grade, flagged images that did not fit
 * cfg.refine_capacity (kept their 16-bit result).  Synchronises the device.  Both 0 when refinement is off. */
BCAD_API int bcad_refine_stats(bcad_model* m, int64_t* refined, int64_t* overflowed);
/* kernels launched by this handle since creation (bench.py reports the delta as gpu_launches) */
BCAD_API int64_t bcad_launch_count(bcad_model* m);
/* 1 when the handle runs the tcgen05 fast path for its conv/fc stack, 0 when it runs fp32 CUDA cores */
BCAD_API int bcad_uses_tensor_path(bcad_model* m);
/* per-kernel device times of the last DEVICE-buffer call: with bcad_set_profiling(m,1) a CUDA event is
 * recorded on the call's stream before every kernel (and one at the end); interval i is kernel i.
 * Off by default (the timed bench region runs with it off). */
BCAD_API int bcad_set_profiling(bcad_model* m, int on);
BCAD_API int bcad_profile_count(bcad_model* m);
BCAD_API int bcad_profile_get(bcad_model* m, int i, char* name_buf, int name_cap, float* ms);

/* ---- diagnostics ------------------------------------------------------------------------------ */
/* One 128 x N x (16*steps) tcgen05 UMMA problem on caller-provided shared-memory operand images and descriptor
 * fields; used by tests/test_gpu_sm100.py to pin the descriptor conventions the tensor path relies on.
 * params_host: int32 {N, steps, a_lbo, a_sbo, a_layout, b_lbo, b_sbo, b_layout, a_koff[64], b_koff[64], mode}; mode 0: bf16
 * operands, d_dev fp32 [128][N]; mode 1: fp16 operands, FP16 accumulators, d_dev = the raw 32-bit TMEM cells [128][N/2]. */
BCAD_API int bcad_selftest_umma(const void* a_img_dev, int a_bytes, const void* b_img_dev, int b_bytes,
                       const int32_t* params_host, float* d_dev, void* stream);

/* Micro-benchmark behind DESIGN.md's operand-layout choices: cycles of `reps` back-to-back 128xNx16 UMMAs and of
 * `reps` TMEM loads.  p = {N, a_layout, b_layout, a_lbo, a_sbo, b_lbo, b_sbo, reps, ld_warps, ld_x16, a_off, alternate, grid,
 * concurrent, st_warps, stores_to_hbm}; out_dev: int64[6] = {MMA cycles of CTA 0, TMEM-load cycles, -, slowest CTA's MMA cycles, loads done, stores done}. */
BCAD_API int bcad_selftest_umma_bench(const int32_t* p, long long* out_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BCAD_H */
