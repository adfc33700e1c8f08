// Launcher declarations shared between the kernel translation units and api.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/bcad.h"

namespace bcad {

// ---------------------------------------------------------------- fp32 CUDA-core path (any shape)
struct ConvArgs {
    const float* x;      // [B,H,W,Cin] NHWC
    const float* w;      // packed [k*k][Cin][CoutPad]
    const float* bias;   // [CoutPad]
    float* y;            // [B,Ho,Wo,Cout] post-activation, or nullptr
    float* p;            // [B,Hp,Wp,Cout] 2x2 max-pooled, or nullptr
    int B, H, W, Cin, Cout, CoutPad, ksize, pad, Ho, Wo, Hp, Wp;
    float alpha;         // LeakyReLU slope (1 = identity)
    int Hv = 0, Wv = 0;  // when > 0: outputs at (oy >= Hv or ox >= Wv) are forced to 0 (Classes/unet.py:19-27 quirk)
};
int launch_conv_fp32(const ConvArgs& a, cudaStream_t s);

// C[M,N] = A[M,K] * B  with B given as [N,K] (b_kmajor) or [K,N]; split-K partials in `partials`
// ([splits][M][N]) when splits > 1, reduced (+bias, optional LeakyReLU copy) by launch_splitk_reduce.
int sgemm_pick_splits(int M, int N, int K);
int launch_sgemm(const float* A, const float* Bm, float* C_or_partials, int M, int N, int K,
                 bool b_kmajor, int splits, cudaStream_t s);
int launch_splitk_reduce(const float* partials, int splits, const float* bias, float* z, float* h,
                         float alpha, int M, int N, cudaStream_t s);

int launch_head(const float* logits, float* probs, int32_t* cls, int B, int nc, int head, cudaStream_t s);
int launch_top_grad(const float* probs, const int32_t* cls, const int32_t* class_idx, float* d_top,
                    int B, int nc, int grad_mode, cudaStream_t s);
// per-image class rows [n][K] (NULL: row b is 0, 1, .., K-1) -> K contiguous class columns of ld entries: cols[k * ld + b]
int launch_class_columns(const int32_t* rows, int K, int n, int32_t* cols, int ld, cudaStream_t s);
int launch_leaky_mask_mul(float* d, const float* z, float alpha, int64_t n, cudaStream_t s);
int launch_unpool(const float* g, const float* y, float* dy, int B, int Ho, int Wo, int C, int ties,
                  cudaStream_t s);
// alpha partials from the pooled gradient (+ tie counts from y when ties==ALL): [B][splits][C]
int alpha_pool_splits(int Hp);
// pre_slope >= 0: gradients w.r.t. the PRE-activation map (routed gradient x LeakyReLU' at the window maximum)
int launch_alpha_from_pool_grad(const float* g, const float* y, float* alpha_part, int B, int Ho, int Wo,
                                int C, int ties, int splits, cudaStream_t s, float pre_slope = -1.f);
// alpha partials from a dense gradient map (fp32 or bf16 NHWC): [B][splits][C]
int launch_alpha_from_dense_grad(const void* dA, int dtype, float* alpha_part, int B, int h, int w, int C,
                                 int splits, cudaStream_t s);
// cam_lo[B,h,w] = ReLU(sum_k alpha_k A_k), alpha_k = inv_hw * sum_s alpha_part[b][s][k];
// also writes alpha_out [B][C] (may be null) and per-image min/max partials mm[B][splits][2]
int cam_splits(int h);
int launch_cam(const void* A, int dtype, const float* alpha_part, int alpha_splits, float inv_hw,
               float* alpha_out, float* cam_lo, float* mm, int B, int h, int w, int C, int splits,
               cudaStream_t s, float inv_slope = 0.f);       // inv_slope > 0 (fp32 A): undo the LeakyReLU first (pre-activation target)
int launch_upsample_norm(const float* cam_lo, const float* mm, int mm_splits, float* out, int B, int h,
                         int w, int H, int W, cudaStream_t s, const int* n_dev = nullptr,    // n_dev: live image count on the device (refine.cu)
                         size_t out_stride = 0);                                            // floats between images' maps (0 = H * W)
// non-overlapping mean pool, floor dims (Classes/ImageSegmentation.py:145-163)
int launch_avg_pool(const float* x, float* out, int B, int H, int W, int C, int pool, cudaStream_t s);
// [k][k][Cin][Cout] -> [k*k][Cin][CoutPad] (zero padded)
int launch_pad_conv_weights(const float* w, float* out, int taps, int Cin, int Cout, int CoutPad, cudaStream_t s);
int launch_overlay(const float* img01, const float* cam, int B, int H, int W, uint8_t* overlay_rgb,
                   uint8_t* heat_u8, cudaStream_t s);
// generate_saliency_overlay for [B][K] maps: base u8 [B][npix][base_c] (1 = grey, replicated; 3 = BGR), sal fp32 [B][K][npix],
// overlay / heat u8 [B][K][npix][3] BGR (either may be null)
int launch_saliency_overlay(const uint8_t* base, int base_c, const float* sal, int B, int K, int npix, uint8_t* overlay, uint8_t* heat,
                            cudaStream_t s);
// the same at the image's size: g8 u8 grey [B][hi][wi], sal fp32 [B][K][H][W] -> overlay / heat u8 [B][K][hi][wi][3] BGR (either may be
// null) = addWeighted(grey3, 0.5, cv2.resize(JET(sal), (wi, hi), INTER_LINEAR), 0.5, 0); 1 <= K <= BCAD_MAX_EXPLAIN_CLASSES, hi <= 65535
int launch_saliency_overlay_resized(const uint8_t* g8, const float* sal, int B, int K, int H, int W, int hi, int wi, uint8_t* overlay,
                                    uint8_t* heat, cudaStream_t s);

// ---------------------------------------------------------------- input-gradient saliency (saliency.cu)
// Outputs of one target class: image b's map at sal + b * out_stride (d_input: + b * out_stride * C), its min / max counters at
// mm + b * mm_ld (two uint32, zeroed before the class's first kernel).
// First block of one input channel, 32 filters, 3x3, pad 0 / 1: pool backward + LeakyReLU' + input gradient + |.| + min / max from the
// block's pooled gradient g and its output y, without the full-resolution gradient
bool saliency_conv0_supported(int Cin, int Cout, int CoutPad, int k, int pad);
int launch_saliency_conv0(const float* g, const float* y, const float* w, int B, int H, int W, int Ho, int Wo, int pad, int first_only,
                          float alpha, float* d_input, float* sal, size_t out_stride, uint32_t* mm, int mm_ld, cudaStream_t s);
// any other first block: s = max_c |d| and min / max from its input gradient d [B][hw][C]
int launch_saliency_absmax(const float* d, int B, int hw, int C, float* d_input, float* sal, size_t out_stride, uint32_t* mm, int mm_ld,
                           cudaStream_t s);
// (s - min) / (max - min + 1e-8) in place over `maps` consecutive maps of hw pixels, counters mm[2 * map ..]
int launch_saliency_norm(float* sal, int maps, int hw, const uint32_t* mm, cudaStream_t s);

// ---------------------------------------------------------------- training step (kernels_train.cu)
int launch_ce_loss_topgrad(const float* probs, const int32_t* labels, float* loss, float* dz, int B, int nc, cudaStream_t s);
int launch_heat_to_u8(const float* cam, uint8_t* out, size_t n, cudaStream_t s);
int launch_u8_to_unit(const uint8_t* src, float* dst, size_t n, cudaStream_t s);
// GRADCAM.py:46 + the CNN-input normalisation of app.py:179-182: img01 = u8 / 255; x[.., c] = standardise ? (img01 - mean) / (std + 1e-8) : img01
int launch_gray_preprocess(const uint8_t* g8, float* img01, float* x, int B, int npix, int C, int standardise, cudaStream_t s);
// u8 grey [B][hi][wi] -> x [B][H][W][C] = standardise(cv2.resize(u8 / 255.0f, (W, H), INTER_LINEAR)) (mean / std of the resized image
// in float64), the channel replicated to C; at hi x wi == H x W exactly launch_gray_preprocess (without img01)
int launch_gray_resize_preprocess(const uint8_t* g8, float* x, int B, int hi, int wi, int H, int W, int C, int standardise, cudaStream_t s);
// launch_overlay for K maps per image on img01 = u8 / 255: g8 u8 [B][npix], cam fp32 [B][K][npix] -> overlay_rgb u8 [B][K][npix][3],
// heat_u8 [B][K][npix] (either may be null); 1 <= K <= BCAD_MAX_EXPLAIN_CLASSES
int launch_overlay_classes(const uint8_t* g8, const float* cam, int B, int K, int npix, uint8_t* overlay_rgb, uint8_t* heat_u8,
                           cudaStream_t s);
int launch_bottleneck_resize(const float* src, float* dst, int B, int C, int H, int W, int chw, int oh, int ow, cudaStream_t s);
int launch_leaky_from_z(const float* z, float* h, float alpha, int64_t n, cudaStream_t s);
int launch_mul_mask(float* h, const float* mask, int B, int units, int ld, cudaStream_t s);
int launch_sgemm_tn(const float* A, const float* Bm, float* C, int M, int N, int K, cudaStream_t s);
int launch_colsum(const float* A, float* out, int K, int N, cudaStream_t s);
int conv_wgrad_band_rows(int B, int Ho, int max_ctas);
int launch_conv_wgrad(const float* dz, const float* in, float* part_w, float* part_b, float* dw, float* db, int B, int H, int W,
                      int Cin, int Cout, int CoutPad, int k, int pad, int Ho, int Wo, int band_rows, cudaStream_t s);
int launch_repack_dgrad(const float* w, float* dk, int k, int Cin, int Cout, int CoutPad, int CinPad, cudaStream_t s);
int launch_l2norm(const float* g, size_t n, float* out, cudaStream_t s);
int launch_sgd_clip_update(float* w, const float* g, const float* norm, float lr, float max_norm, size_t n, cudaStream_t s);
int launch_adam_update(float* w, const float* g, float* m1, float* m2, float lr, float b1, float b2, float eps, int step, size_t n,
                       cudaStream_t s);

// ---------------------------------------------------------------- small-margin refinement (refine.cu)
// idx[0..count) = images of the chunk whose two largest logits differ by less than `margin`, ascending; counters = {count
// clamped to cap, running total refined, running total overflowed}
int launch_refine_flag(const float* logits, int n, int nc, float margin, int cap, int32_t* idx, int32_t* counters, cudaStream_t s);
// slots [0,count): image idx[slot] (the twin's kernels read the same device-side count and skip the other slots)
// class_idx rows of K entries per image (bcad_predict_explain_classes; 1 otherwise) go to rcidx[slot * K ..]
int launch_refine_gather(const float* x, size_t img_elems, const int32_t* class_idx, const int32_t* idx, const int32_t* counters,
                         int slots, float* rx, int32_t* rcidx, cudaStream_t s, int K = 1);
struct RefineScatter {
    int n_dense;
    int sizes[8];
    const float* src_z[8];        // twin pre-activations [slots][size]
    float* dst_z[8];              // chunk pre-activations [n][size]
    const float* src_probs;
    float* dst_probs;
    const int32_t* src_cls;
    int32_t* dst_cls;
    const float* src_heat;        // [slots][hm] or nullptr
    float* dst_heat;              // [n][hm] or nullptr
    size_t hm;
    int nc;
};
int launch_refine_scatter(const RefineScatter& a, const int32_t* idx, const int32_t* counters, int slots, cudaStream_t s);

// fused dense head: fc1 split-K reduce -> remaining dense layers -> probs/class -> (explain) backward to dz1 + alpha
struct HeadArgs {
    int n_dense;                  // dense layers incl. the output layer; layer 0 comes as split-K partials
    int sizes[8];                 // output size of every dense layer (sizes[n_dense-1] = num_classes)
    int max_size;
    const float* W[8];            // (out,in) fp32 of layers 1.. (W[0] unused)
    const float* bias[8];
    float* z[8];                  // pre-activations [B][size] (kept for layer['z'] compat)
    const float* fc1_part;        // [splits][ld] partial sums of layer 0, row b at b*sizes[0]
    int fc1_splits;
    size_t fc1_ld;
    float alpha;
    int head;
    float* probs;
    int32_t* cls;
    int explain;
    const int32_t* class_idx;     // nullable = predicted class
    int grad_mode;
    float* dz1;                   // [B][sizes[0]] out, nullable
    const float* S;               // [sizes[0]][C] fp32, nullable
    int C;
    float* alpha_raw;             // [B][C]
    const int* n_dev;             // nullable DEVICE pointer: only the first *n_dev images are live (refinement twin)
};
int launch_dense_head(const HeadArgs& a, int B, cudaStream_t s);

}  // namespace bcad
