// The model handle behind bcad_model (weights, workspace, transfer pipeline).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>
#include <vector>

#include "../../include/bcad.h"
#include "kernels.h"

namespace bcad {

struct DeviceGuard {                   // make the handle's device current for the duration of a call
    int prev = -1;
    explicit DeviceGuard(int dev) {
        cudaGetDevice(&prev);
        if (prev != dev) cudaSetDevice(dev);
        else prev = -1;
    }
    ~DeviceGuard() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

struct ConvLayer {
    int Cin = 0, Cout = 0, CoutPad = 0, k = 0;
    int H = 0, W = 0, Ho = 0, Wo = 0, Hp = 0, Wp = 0;
    std::vector<float> h_w, h_b;      // staged host weights: (F,k,k,C) and (F,)
    float* d_w = nullptr;             // fp32 packed [k*k][Cin][CoutPad]
    float* d_b = nullptr;             // [CoutPad]
    float* d_w_dgrad = nullptr;       // fp32 packed flipped filters for the input gradient
    float* d_zero_bias = nullptr;
    float* y = nullptr;               // cached post-activation output (fp32 path), NHWC
    float* p = nullptr;               // cached pooled output (fp32 path), NHWC
    float* dz = nullptr;              // explain_backward scratch
    float* gp = nullptr;              // gradient w.r.t. this block's pooled output (explain_backward)
    uint8_t* tc_w = nullptr;          // fast training (sm100_train.cu): fp16 hi / lo image of d_w, and of d_w_dgrad
    uint8_t* tc_wd = nullptr;
};

struct DenseLayer {
    int in = 0, out = 0, splits = 1;
    std::vector<float> h_w, h_b;      // (out,in) with `in` in device (NHWC) order, (out,)
    float* d_w = nullptr;
    float* d_b = nullptr;
    float* z = nullptr;               // pre-activation [B,out]
    float* h = nullptr;               // LeakyReLU(z); reused as d(h) then dz by the backward
};

struct Xfer {                          // host-buffer pipeline (bcad_predict_explain_host)
    bool inited = false;
    int chunk = 0;
    cudaStream_t s_in = nullptr, s_compute = nullptr, s_out = nullptr;
    cudaEvent_t in_done[2] = {nullptr, nullptr}, compute_done[2] = {nullptr, nullptr}, out_done[2] = {nullptr, nullptr};
    float* x[2] = {nullptr, nullptr};
    float* heat[2] = {nullptr, nullptr};
    uint8_t* heat8[2] = {nullptr, nullptr};   // u8 heat-maps of a chunk (bcad_predict_explain_host_u8), allocated on first use
    uint8_t* x8[2] = {nullptr, nullptr};      // 8-bit input pixels of a chunk (bcad_predict_explain_host_u8in), allocated on first use
    float* img01[2] = {nullptr, nullptr};     // grey image / 255 of a chunk and its RGB overlays (bcad_gradcam_overlays_host), first use
    uint8_t* ov8[2] = {nullptr, nullptr};
    int32_t* cidx[2] = {nullptr, nullptr};
    // pinned host staging for the small per-image outputs (user arrays may be pageable: a pageable D2H would
    // block the host and serialise the chunk pipeline)
    void* h_small = nullptr;
    size_t h_small_bytes = 0;
    // device staging of the same outputs for a WHOLE call: every chunk writes its logits / probabilities / classes here and ONE copy at
    // the end brings them back (three tiny D2H copies per chunk sat between the heat-map copies of the link-bound output stream)
    void* d_small = nullptr;
    size_t d_small_bytes = 0;
    // both slots' staging of bcad_gradcam_overlays_classes_host (8-bit images, classes, K float / RGB / u8 maps of the image size),
    // one allocation that is replaced when a call needs more
    void* cls_arena = nullptr;
    size_t cls_arena_bytes = 0;
};

struct TrainState {                     // row f4: buffers of the training step (allocated on first use)
    bool ready = false;
    std::vector<size_t> conv_w_off, conv_b_off, dense_w_off, dense_b_off;   // offsets into the flat gradient vector
    size_t total = 0;
    std::vector<float*> dense_dz;       // dz of every dense layer [max_batch][out]
    float* hbuf = nullptr;              // LeakyReLU(z) of the layer feeding the current wgrad
    float* part_w = nullptr;            // conv wgrad per-CTA partials
    float* part_b = nullptr;
    float* norms = nullptr;             // one L2 norm per tensor
    float* adam_m = nullptr;
    float* adam_v = nullptr;
    int adam_step = 0;
    float* drop = nullptr;              // dropout multipliers [max_batch][drop_ld] (bcad_set_dropout_masks), drop_B = 0: off
    int drop_B = 0, drop_ld = 0;
    bool drop_backward = true;          // mask the gradient too (autograd); false = the NumPy reference's backward
    std::vector<int> drop_off;          // column offset of every hidden layer in a mask row
    int max_ctas = 2048;
    float* wg_part = nullptr;           // fast training: per-CTA accumulator dumps of the tensor-core weight gradient
    float* cs_part = nullptr;           //                slab partials of the bias gradient
    float* fc_part = nullptr;           //                split-K partials of the tensor-core fc1 forward
    float* c0_part = nullptr;           //                per-CTA partials of the fused first-block backward
    bool tc_dirty = true;               //                the fp16 weight images are older than the fp32 weights
};

struct TensorPath;                     // tensor_path.cu

struct Model;
struct Refine {                         // cfg.refine_margin > 0: small-margin images are re-run through a split-operand twin handle
    Model* twin = nullptr;              // BCAD_PREC_F16X3 handle of the same network, max_batch = cap
    int cap = 0;
    int32_t* idx = nullptr;             // [cap] chunk-local indices of the flagged images, in ascending order
    int32_t* counters = nullptr;        // {flagged in this chunk (clamped to cap), total refined, total overflowed}
    float* x = nullptr;                 // [cap] gathered inputs
    int32_t* cidx = nullptr;            // [cap][cidx_k] gathered target classes
    int cidx_k = 1;                     // classes per image `cidx` has room for (grows on the first bcad_predict_explain_classes call)
    float* heat = nullptr;              // [cap] heat-maps of the twin (its other outputs are read from its own workspace)
    size_t heat_elems = 0;              // per-image capacity of `heat` (grows on the first larger bcad_predict_explain_sized / _classes call)
};

struct Model {
    bcad_config cfg;
    std::vector<ConvLayer> conv;
    std::vector<DenseLayer> dense;
    int64_t flat = 0;
    bool committed = false, ws_ready = false, tensor_path = false, profiling = false, fused_head = false;
    int cached_B = 0;
    int64_t launches = 0;
    size_t ws_bytes = 0;
    std::mutex mu;
    std::mutex host_mu;                 // serialises the host-buffer calls of one handle (shared staging, streams, events)
    Refine refine;
    bool fast_train = false;            // bcad_set_fast_training: tensor-core (split-operand) kernels for the eligible conv blocks of the training step
    int sms = 0;
    int target = BCAD_TARGET_CONV_ACT;  // bcad_set_explain_target
    int heat_h = 0, heat_w = 0;         // heat-map size of the call in flight (in_h x in_w unless bcad_predict_explain_sized asks otherwise)
    const int32_t* n_dev = nullptr;     // refinement TWIN only: device pointer to the live image count of its launches
    std::vector<void*> allocs;
    // shared workspace
    float* partials = nullptr;
    float* probs = nullptr;
    int32_t* cls = nullptr;
    float* d_top = nullptr;
    float* g_flat = nullptr;
    float* alpha_part = nullptr;
    float* alpha = nullptr;
    float* cam_lo = nullptr;
    float* mm = nullptr;
    int alpha_splits = 1, cam_splits = 1;
    int32_t* class_cols = nullptr;      // [BCAD_MAX_EXPLAIN_CLASSES][max_batch]: target class column k of the chunk (bcad_predict_explain_classes)
    bool multi_class_call = false;      // the last call explained several classes: alpha / cam_lo describe none of them
    HeadArgs head_last;                 // arguments of the chunk's dense_head_kernel launch, re-launched per extra target class
    int head_n = 0;
    float* sal_din = nullptr;           // bcad_predict_saliency_classes (first use): input gradient of a first block without the fused kernel
    uint32_t* sal_mm = nullptr;         //   per-map min / max counters [max_batch][BCAD_MAX_EXPLAIN_CLASSES][2]
    cudaEvent_t call_done = nullptr;
    std::vector<cudaEvent_t> prof_pool;   // profiling marks of the last call: event i precedes kernel i
    std::vector<const char*> prof_names;
    int prof_n = 0;
    Xfer xfer;
    TrainState train;
    TensorPath* tp = nullptr;

    int alloc(void** p, size_t bytes);
    void free_all();
    int mark(const char* name, cudaStream_t s);
};

// dense backward shared by both paths: d_top -> ... -> dz of dense[0] (left in dense[0].h) and, when
// g_flat != nullptr, on to the flattened pool output
// fast training: which conv blocks run on the tensor-core kernels, and keeping their fp16 weight images current
bool tc_train_eligible(const Model* m, size_t i);
int tc_train_refresh(Model* m, cudaStream_t s);

int dense_backward(Model* m, int n, const int32_t* class_idx, int grad_mode, float* g_flat, cudaStream_t s);

// One step of the conv-block backward shared by explain_backward, the training step and the saliency call.
// conv_block_dz: conv[i].dz = gradient w.r.t. the block's pre-activation from gp (gradient w.r.t. its pooled output).  fused: pool
// backward and LeakyReLU' in one pass (unpool_mask); else unpool, then act_grad (when given) receives the gradient w.r.t. the
// post-activation output, then leaky_mask_mul unless mask is false.
int conv_block_dz(Model* m, int i, const float* gp, int B, bool fused, float* act_grad, bool mask, cudaStream_t s);
// conv_block_dgrad: the block's input gradient from conv[i].dz into dst (nullptr = conv[i - 1].gp, allocated on first use).  tc: the
// split-operand tcgen05 kernel (fast training, tc_train_eligible block); else conv_fp32 with the flipped filters, profiled as `name`.
int conv_block_dgrad(Model* m, int i, int B, float* dst, bool tc, const char* name, cudaStream_t s);

bool fused_head_ok(const Model* m);
// everything after the fc1 GEMM in one launch (dense_head_kernel); dz1 / S / alpha_raw are optional outputs
int launch_fused_head(Model* m, int n, const float* fc1_part, int splits, size_t ld, bool explain, const int32_t* class_idx,
                      int grad_mode, float* dz1, const float* S, int C, float* alpha_raw, cudaStream_t s);
// the chunk's last launch_fused_head again with another target class column (alpha_raw replaces its alpha output when it had one):
// the kernel recomputes everything from the fc1 split-K partials, which no kernel after it writes, so the forward outputs it
// rewrites come out the same and dz1 / alpha are those of the new targets
int relaunch_fused_head(Model* m, const int32_t* class_idx, float* alpha_raw, cudaStream_t s);

// ---- tensor (tcgen05) path, tensor_path.cu
int tensor_path_supported(const Model& m);          // BCAD_OK or BCAD_ERR_INVALID (+ message)
int tensor_path_commit(Model& m);
int tensor_forward_chunk(Model& m, const float* x, int n, bool explain, const int32_t* class_idx, int grad_mode, cudaStream_t s);
// K target classes: class column k at class_idx + k * col_ld, the map of class k of image b at heat + b * heat_stride + k * H * W
// (heat_stride 0 = H * W)
int tensor_explain_chunk(Model& m, int n, const int32_t* class_idx, int grad_mode, float* heat, cudaStream_t s, int K = 1,
                         size_t col_ld = 0, size_t heat_stride = 0);
int tensor_get_activation(Model& m, int kind, int index, int B, float* dst, cudaStream_t s);
void tensor_path_destroy(Model& m);

}  // namespace bcad
