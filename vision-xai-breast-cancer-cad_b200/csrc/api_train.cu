// C-ABI of the training step (SURVEY 8 row f4; BASELINE config 5): gradients of the mean softmax cross-entropy over a
// batch w.r.t. every weight and bias, optimiser updates on the device weights, weight read-back.
// Reference: Classes/CNNModel.py:282-355 (_compute_sample_grads), :372-394 (_apply_grads), :399-512 (train);
// ADCNNM.py:86-153 (Adam + CrossEntropyLoss).  fp32 path only.  Dropout: the caller draws the multipliers and hands them over with
// bcad_set_dropout_masks; the forward applies them after every hidden layer and the backward uses the dropped activations
// (and, for autograd semantics, masks the gradient too).
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "../../include/bcad.h"
#include "common.cuh"
#include "kernels.h"
#include "model.h"
#include "sm100_train.h"

namespace bcad {

#define TR_TRY(expr) do { int _rc = (expr); if (_rc != BCAD_OK) return _rc; } while (0)
#define TR_LAUNCH(m, name, expr) do { int _rc = (m)->mark(name, s); if (_rc == BCAD_OK) _rc = (expr); if (_rc != BCAD_OK) return _rc; (m)->launches += 1; } while (0)

// the one definition of the flat gradient layout: every tensor starts 128-byte aligned (vector stores in the wgrad kernels)
struct GradLayout { std::vector<size_t> conv_w, conv_b, dense_w, dense_b; size_t total = 0; };
static GradLayout grad_layout_of(const Model* m) {
    GradLayout g;
    size_t off = 0;
    auto pad32 = [](size_t n) { return (n + 31) / 32 * 32; };
    for (const ConvLayer& L : m->conv) {
        g.conv_w.push_back(off); off += pad32((size_t)L.k * L.k * L.Cin * L.CoutPad);
        g.conv_b.push_back(off); off += pad32((size_t)L.CoutPad);
    }
    for (const DenseLayer& D : m->dense) {
        g.dense_w.push_back(off); off += pad32((size_t)D.out * D.in);
        g.dense_b.push_back(off); off += pad32((size_t)D.out);
    }
    g.total = off;
    return g;
}

static int ensure_train_state(Model* m) {
    TrainState& T = m->train;
    if (T.ready) return BCAD_OK;
    const GradLayout gl = grad_layout_of(m);
    T.conv_w_off = gl.conv_w; T.conv_b_off = gl.conv_b; T.dense_w_off = gl.dense_w; T.dense_b_off = gl.dense_b;
    T.total = gl.total;
    const int mb = m->cfg.max_batch;
    int max_out = 1;
    for (DenseLayer& D : m->dense) {
        float* p = nullptr;
        TR_TRY(m->alloc((void**)&p, (size_t)mb * D.out * sizeof(float)));
        T.dense_dz.push_back(p);
        max_out = std::max(max_out, D.out);
    }
    TR_TRY(m->alloc((void**)&T.hbuf, (size_t)mb * max_out * sizeof(float)));
    size_t pw = 0, pb = 0;
    for (const ConvLayer& L : m->conv) {
        // any B <= max_batch launches at most max(max_ctas, B) CTAs (conv_wgrad_band_rows)
        const size_t ncta = (size_t)std::max(T.max_ctas, mb);
        pw = std::max(pw, ncta * (size_t)L.k * L.k * L.Cin * L.CoutPad);
        pb = std::max(pb, ncta * (size_t)L.CoutPad);
    }
    TR_TRY(m->alloc((void**)&T.part_w, pw * sizeof(float)));
    TR_TRY(m->alloc((void**)&T.part_b, pb * sizeof(float)));
    TR_TRY(m->alloc((void**)&T.norms, 2 * (m->conv.size() + m->dense.size()) * sizeof(float)));
    T.ready = true;
    return BCAD_OK;
}

// fast training (bcad_set_fast_training): conv blocks i >= 1 of the 32 -> 64 shape run forward / dgrad / wgrad on the tensor cores
bool tc_train_eligible(const Model* m, size_t i) {
    if (i == 0 || i >= m->conv.size()) return false;
    const ConvLayer& L = m->conv[i];
    return L.Cin == 32 && L.Cout == 64 && L.CoutPad == 64 && conv3x3_x3_supported(L.Cin, L.Cout, L.k, L.W, L.Wo, m->cfg.pad) &&
           conv3x3_x3_supported(L.Cout, L.Cin, L.k, L.Wo, L.W, L.k - 1 - m->cfg.pad) && wgrad3x3_x3_supported(L.Cin, L.Cout, L.k, L.W, L.Wo, m->cfg.pad);
}

int tc_train_refresh(Model* m, cudaStream_t s) {
    if (!m->fast_train || !m->train.tc_dirty) return BCAD_OK;
    for (size_t i = 0; i < m->conv.size(); ++i) {
        if (!tc_train_eligible(m, i)) continue;
        ConvLayer& L = m->conv[i];
        if (L.tc_w == nullptr) {
            TR_TRY(m->alloc((void**)&L.tc_w, conv3x3_x3_weight_bytes(L.Cin, L.Cout)));
            TR_TRY(m->alloc((void**)&L.tc_wd, conv3x3_x3_weight_bytes(L.Cout, L.Cin)));
        }
        TR_TRY(launch_pack_w_x3(L.d_w, L.tc_w, L.Cin, L.Cout, L.CoutPad, false, s));
        TR_TRY(launch_pack_w_x3(L.d_w_dgrad, L.tc_wd, L.Cout, L.Cin, cdiv(L.Cin, 32) * 32, true, s));     // bf16: multiplies the bf16-split gradient
        m->launches += 2;
    }
    m->train.tc_dirty = false;
    return BCAD_OK;
}

}  // namespace bcad

using namespace bcad;

extern "C" {

int64_t bcad_grad_elems(bcad_model* mm) {
    Model* m = reinterpret_cast<Model*>(mm);
    if (!m) return -1;
    return (int64_t)grad_layout_of(m).total;
}

int bcad_grad_layout(bcad_model* mm, int is_dense, int index, int64_t* w_off, int64_t* w_elems, int64_t* b_off, int64_t* b_elems) {
    Model* m = reinterpret_cast<Model*>(mm);
    BCAD_REQUIRE(m && w_off && w_elems && b_off && b_elems, "grad_layout: null argument");
    const GradLayout gl = grad_layout_of(m);
    if (!is_dense && index >= 0 && index < (int)m->conv.size()) {
        const ConvLayer& L = m->conv[index];
        *w_off = (int64_t)gl.conv_w[index]; *w_elems = (int64_t)L.k * L.k * L.Cin * L.CoutPad;
        *b_off = (int64_t)gl.conv_b[index]; *b_elems = L.CoutPad;
        return BCAD_OK;
    }
    if (is_dense && index >= 0 && index < (int)m->dense.size()) {
        const DenseLayer& D = m->dense[index];
        *w_off = (int64_t)gl.dense_w[index]; *w_elems = (int64_t)D.out * D.in;
        *b_off = (int64_t)gl.dense_b[index]; *b_elems = D.out;
        return BCAD_OK;
    }
    set_error("grad_layout: no such layer (%d,%d)", is_dense, index);
    return BCAD_ERR_INVALID;
}

// Gradients of the MEAN cross-entropy over the B images of the preceding bcad_predict (same x, same B, fp32 path,
// keep_all_activations=1).  grads_dev: fp32 [bcad_grad_elems]; loss_dev: fp32 [B] per-sample losses (may be NULL).
int bcad_train_backward(bcad_model* mm, const float* x, const int32_t* labels, int B, float* grads, float* loss, void* stream) {
    return bcad_train_backward_part(mm, x, labels, B, grads, loss, 0, stream);
}

// part 0: everything; part 1: loss + dense layers only (their gradients are final when it returns: a data-parallel caller can start
// all-reducing them -- 99.9 % of the bytes -- while part 2 runs); part 2: the conv blocks (needs part 1 of the same batch before it).
int bcad_train_backward_part(bcad_model* mm, const float* x, const int32_t* labels, int B, float* grads, float* loss, int part, void* stream) {
    Model* m = reinterpret_cast<Model*>(mm);
    BCAD_REQUIRE(m && x && labels && grads, "train_backward: null argument");
    BCAD_REQUIRE(part >= 0 && part <= 2, "train_backward: part must be 0 (all), 1 (dense) or 2 (conv)");
    cudaStream_t s = (cudaStream_t)stream;
    if (m->tensor_path) { set_error("training runs on the fp32 path: create the model with BCAD_PREC_FP32"); return BCAD_ERR_INVALID; }
    if (!m->committed || m->cached_B != B) {
        set_error("train_backward needs the activations of a preceding bcad_predict with the same B=%d (cached %d)", B, m->cached_B);
        return BCAD_ERR_STATE;
    }
    for (size_t i = 0; i < m->conv.size(); ++i)
        if (m->conv[i].y == nullptr) { set_error("training needs keep_all_activations=1"); return BCAD_ERR_STATE; }
    DeviceGuard g(m->cfg.device);
    std::lock_guard<std::mutex> lock(m->mu);
    TR_TRY(ensure_train_state(m));
    TrainState& T = m->train;
    BCAD_CUDA_CHECK(cudaStreamWaitEvent(s, m->call_done, 0));
    const int nc = m->cfg.num_classes, nd = (int)m->dense.size(), nconv = (int)m->conv.size();
    m->prof_n = 0;
    if (part != 2) {
    float* loss_buf = loss ? loss : T.hbuf;                  // scratch when the caller does not want the losses
    TR_LAUNCH(m, "ce_loss_topgrad", launch_ce_loss_topgrad(m->probs, labels, loss_buf, T.dense_dz[nd - 1], B, nc, s));
    // ---- dense layers, last to first
    for (int j = nd - 1; j >= 0; --j) {
        DenseLayer& D = m->dense[j];
        const float* in_j;
        if (j == 0) in_j = m->conv.back().p;
        else {
            TR_LAUNCH(m, "leaky_from_z", launch_leaky_from_z(m->dense[j - 1].z, T.hbuf, m->cfg.alpha_dense, (int64_t)B * m->dense[j - 1].out, s));
            if (T.drop_B) TR_LAUNCH(m, "dropout", launch_mul_mask(T.hbuf, T.drop + T.drop_off[j - 1], B, m->dense[j - 1].out, T.drop_ld, s));
            in_j = T.hbuf;
        }
        // fast training: the first dense layer's two GEMMs against the big weight matrix as split-operand tcgen05 GEMMs (sm100_train.cu)
        const bool tcd = m->fast_train && j == 0 && dense_bwd_x3_supported(B, D.out, D.in) && getenv("BCAD_TC_NO_DENSE") == nullptr;
        float* dst = (j > 0) ? T.dense_dz[j - 1] : m->g_flat;
        if (tcd) {
            DenseBwdArgs dw;
            dw.dz = T.dense_dz[j]; dw.src = in_j; dw.out = grads + T.dense_w_off[j]; dw.B = B; dw.units = D.out; dw.flat = D.in;
            TR_LAUNCH(m, "dense_wgrad_tcgen05_x3", launch_dense_bwd_x3(dw, 0, m->sms, s));
            TR_LAUNCH(m, "dense_bgrad", launch_colsum(T.dense_dz[j], grads + T.dense_b_off[j], B, D.out, s));
            DenseBwdArgs dg;
            dg.dz = T.dense_dz[j]; dg.src = D.d_w; dg.out = dst; dg.B = B; dg.units = D.out; dg.flat = D.in;
            TR_LAUNCH(m, "dense_dgrad_tcgen05_x3", launch_dense_bwd_x3(dg, 1, m->sms, s));
        } else {
        TR_LAUNCH(m, "dense_wgrad", launch_sgemm_tn(T.dense_dz[j], in_j, grads + T.dense_w_off[j], D.out, D.in, B, s));
        TR_LAUNCH(m, "dense_bgrad", launch_colsum(T.dense_dz[j], grads + T.dense_b_off[j], B, D.out, s));
        TR_LAUNCH(m, "dense_dgrad", launch_sgemm(T.dense_dz[j], D.d_w, dst, B, D.in, D.out, false, 1, s));
        }
        if (j > 0 && T.drop_B && T.drop_backward) TR_LAUNCH(m, "dropout", launch_mul_mask(dst, T.drop + T.drop_off[j - 1], B, m->dense[j - 1].out, T.drop_ld, s));
        if (j > 0) TR_LAUNCH(m, "leaky_mask_mul", launch_leaky_mask_mul(dst, m->dense[j - 1].z, m->cfg.alpha_dense, (int64_t)B * m->dense[j - 1].out, s));
    }
    }
    if (part == 1) {
        TR_TRY(m->mark("end", s));
        BCAD_CUDA_CHECK(cudaEventRecord(m->call_done, s));
        return BCAD_OK;
    }
    // ---- conv blocks, last to first
    const float* gp = m->g_flat;
    for (int i = nconv - 1; i >= 0; --i) {
        ConvLayer& L = m->conv[i];
        const int first_only = (m->cfg.pool_ties == BCAD_TIES_FIRST) ? 1 : 0;
        if (m->fast_train && i == 0 && L.Cin == 1 && L.Cout == 32 && L.CoutPad == 32 && L.k == 3 && getenv("BCAD_TC_NO_CONV0") == nullptr) {
            // first block, one input channel: pool backward + LeakyReLU' + dF / db in one pass, the full-resolution gradient is never written
            if (T.c0_part == nullptr) TR_TRY(m->alloc((void**)&T.c0_part, (size_t)conv0_bwd_fused_parts(m->sms) * 320 * sizeof(float)));
            TR_LAUNCH(m, "conv0_bwd_fused", launch_conv0_bwd_fused(gp, L.y, x, T.c0_part, grads + T.conv_w_off[i], grads + T.conv_b_off[i], B, L.H, L.W,
                                                                  L.Ho, L.Wo, m->cfg.pad, first_only, m->cfg.alpha_conv, m->sms, s));
            m->launches += 1;
            continue;
        }
        TR_TRY(conv_block_dz(m, i, gp, B, m->fast_train && L.Cout % 4 == 0, nullptr, true, s));
        const float* in_i = (i == 0) ? x : m->conv[i - 1].p;
        const bool tc = m->fast_train && tc_train_eligible(m, (size_t)i);
        const bool tc_w = tc && getenv("BCAD_TC_NO_WGRAD") == nullptr, tc_d = tc && getenv("BCAD_TC_NO_DGRAD") == nullptr;   // (fault isolation)
        if (tc_w) {
            // weight gradient as a pixel-contracting tcgen05 GEMM, bias gradient as a slab column sum (sm100_train.cu)
            TR_TRY(tc_train_refresh(m, s));
            if (T.wg_part == nullptr) {
                TR_TRY(m->alloc((void**)&T.wg_part, wgrad3x3_x3_partial_floats(m->sms) * sizeof(float)));
                TR_TRY(m->alloc((void**)&T.cs_part, (size_t)4096 * 64 * sizeof(float)));
            }
            TcWgradArgs w;
            w.x = in_i; w.dy = L.dz; w.partials = T.wg_part; w.B = B; w.H = L.H; w.W = L.W; w.Ho = L.Ho; w.Wo = L.Wo; w.pad = m->cfg.pad;
            TR_LAUNCH(m, "conv_wgrad_tcgen05_x3", launch_wgrad3x3_x3(w, grads + T.conv_w_off[i], L.CoutPad, m->sms, s));
            TR_LAUNCH(m, "conv_bgrad", launch_colsum64(L.dz, T.cs_part, grads + T.conv_b_off[i], (size_t)B * L.Ho * L.Wo, s));
            m->launches += 2;                                // the two reductions
        } else {
        const int rows = conv_wgrad_band_rows(B, L.Ho, T.max_ctas);
        TR_LAUNCH(m, "conv_wgrad", launch_conv_wgrad(L.dz, in_i, T.part_w, T.part_b, grads + T.conv_w_off[i], grads + T.conv_b_off[i], B, L.H, L.W,
                                                    L.Cin, L.Cout, L.CoutPad, L.k, m->cfg.pad, L.Ho, L.Wo, rows, s));
        m->launches += 2;                                    // the two partial reductions
        }
        if (i > 0) {
            TR_TRY(conv_block_dgrad(m, i, B, nullptr, tc_d, "conv_dgrad", s));
            gp = m->conv[i - 1].gp;
        }
    }
    TR_TRY(m->mark("end", s));
    BCAD_CUDA_CHECK(cudaEventRecord(m->call_done, s));
    return BCAD_OK;
}

// Dropout multipliers for the NEXT forwards of exactly B images (B <= max_batch): masks[b][sum of hidden units], hidden
// layers in order, each value 0 or 1/(1-rate) (Classes/CNNModel.py:186-188; nn.Dropout ADCNNM.py:62).  The caller draws them
// (the NumPy mirror replays np.random in the reference's order).  NULL / B = 0 switches dropout off again.
// mask_backward: 1 = the gradient is masked too (autograd, ADCNNM.py); 0 = the NumPy reference, whose backward uses d_out as
// is (Classes/CNNModel.py:307-316).
int bcad_set_dropout_masks(bcad_model* mm, const float* masks, int B, int mask_backward, void* stream) {
    Model* m = reinterpret_cast<Model*>(mm);
    BCAD_REQUIRE(m, "null model");
    if (m->tensor_path) { set_error("training runs on the fp32 path"); return BCAD_ERR_INVALID; }
    cudaStream_t s = (cudaStream_t)stream;
    DeviceGuard g(m->cfg.device);
    std::lock_guard<std::mutex> lock(m->mu);
    TrainState& T = m->train;
    if (masks == nullptr || B == 0) { T.drop_B = 0; return BCAD_OK; }
    BCAD_REQUIRE(B >= 1 && B <= m->cfg.max_batch, "dropout masks: B=%d must be within max_batch=%d", B, m->cfg.max_batch);
    BCAD_REQUIRE(m->dense.size() > 1, "the network has no hidden dense layer to drop");
    if (T.drop == nullptr) {
        T.drop_off.clear();
        T.drop_ld = 0;
        for (size_t j = 0; j + 1 < m->dense.size(); ++j) { T.drop_off.push_back(T.drop_ld); T.drop_ld += m->dense[j].out; }
        TR_TRY(m->alloc((void**)&T.drop, (size_t)m->cfg.max_batch * T.drop_ld * sizeof(float)));
    }
    BCAD_CUDA_CHECK(cudaStreamWaitEvent(s, m->call_done, 0));
    BCAD_CUDA_CHECK(cudaMemcpyAsync(T.drop, masks, (size_t)B * T.drop_ld * sizeof(float), cudaMemcpyDefault, s));
    BCAD_CUDA_CHECK(cudaEventRecord(m->call_done, s));
    T.drop_B = B;
    T.drop_backward = (mask_backward != 0);
    m->cached_B = 0;
    return BCAD_OK;
}

// Fast training: the eligible conv blocks (3x3, 32 -> 64 filters, maps up to 128 px wide) run their forward, input gradient and weight
// gradient as split-operand tcgen05 GEMMs (fp32 in / out, products from fp16 / bf16 hi + lo pairs: gradients agree with the fp32 kernels to
// ~1e-4 relative instead of 1e-6).  Off by default: the reference-pinned fp32 kernels stay the parity anchor.
int bcad_set_fast_training(bcad_model* mm, int on) {
    Model* m = reinterpret_cast<Model*>(mm);
    BCAD_REQUIRE(m, "null model");
    if (m->tensor_path) { set_error("training runs on the fp32 path: create the model with BCAD_PREC_FP32"); return BCAD_ERR_INVALID; }
    std::lock_guard<std::mutex> lock(m->mu);
    if (on) {
        bool any = false;
        for (size_t i = 0; i < m->conv.size(); ++i) any = any || tc_train_eligible(m, i);
        BCAD_REQUIRE(any, "fast training: no conv block of this network has the tensor-core shape (3x3, 32 -> 64 filters, maps <= 128 px wide)");
        if (m->sms == 0) {
            DeviceGuard g(m->cfg.device);
            BCAD_CUDA_CHECK(cudaDeviceGetAttribute(&m->sms, cudaDevAttrMultiProcessorCount, m->cfg.device));
        }
    }
    m->fast_train = (on != 0);
    m->train.tc_dirty = true;
    m->cached_B = 0;
    return BCAD_OK;
}

// optimiser step on the device weights.  opt: 0 = SGD with per-tensor L2-norm clipping at max_norm (0 = no clipping)
// (Classes/CNNModel.py:372-394), 1 = Adam (b1, b2, eps; torch.optim.Adam, ADCNNM.py:88).
int bcad_apply_update(bcad_model* mm, const float* grads, int opt, float lr, float max_norm, float b1, float b2, float eps, void* stream) {
    Model* m = reinterpret_cast<Model*>(mm);
    BCAD_REQUIRE(m && grads, "apply_update: null argument");
    BCAD_REQUIRE(opt == 0 || opt == 1, "apply_update: opt must be 0 (SGD+clip) or 1 (Adam)");
    if (m->tensor_path) { set_error("training runs on the fp32 path"); return BCAD_ERR_INVALID; }
    if (!m->committed) { set_error("weights not committed"); return BCAD_ERR_STATE; }
    cudaStream_t s = (cudaStream_t)stream;
    DeviceGuard g(m->cfg.device);
    std::lock_guard<std::mutex> lock(m->mu);
    TR_TRY(ensure_train_state(m));
    TrainState& T = m->train;
    BCAD_CUDA_CHECK(cudaStreamWaitEvent(s, m->call_done, 0));
    if (opt == 1 && T.adam_m == nullptr) {
        TR_TRY(m->alloc((void**)&T.adam_m, T.total * sizeof(float)));
        TR_TRY(m->alloc((void**)&T.adam_v, T.total * sizeof(float)));
        BCAD_CUDA_CHECK(cudaMemsetAsync(T.adam_m, 0, T.total * sizeof(float), s));
        BCAD_CUDA_CHECK(cudaMemsetAsync(T.adam_v, 0, T.total * sizeof(float), s));
    }
    if (opt == 1) ++T.adam_step;
    m->prof_n = 0;
    int tix = 0;
    auto step = [&](float* w, size_t off, size_t n) -> int {
        if (opt == 0) {
            TR_LAUNCH(m, "l2norm", launch_l2norm(grads + off, n, T.norms + tix, s));
            TR_LAUNCH(m, "sgd_clip_update", launch_sgd_clip_update(w, grads + off, T.norms + tix, lr, max_norm, n, s));
        } else {
            TR_LAUNCH(m, "adam_update", launch_adam_update(w, grads + off, T.adam_m + off, T.adam_v + off, lr, b1, b2, eps, T.adam_step, n, s));
        }
        ++tix;
        return BCAD_OK;
    };
    for (size_t i = 0; i < m->conv.size(); ++i) {
        ConvLayer& L = m->conv[i];
        TR_TRY(step(L.d_w, T.conv_w_off[i], (size_t)L.k * L.k * L.Cin * L.CoutPad));
        TR_TRY(step(L.d_b, T.conv_b_off[i], (size_t)L.CoutPad));
        TR_LAUNCH(m, "repack_dgrad", launch_repack_dgrad(L.d_w, L.d_w_dgrad, L.k, L.Cin, L.Cout, L.CoutPad, cdiv(L.Cin, 32) * 32, s));
    }
    for (size_t j = 0; j < m->dense.size(); ++j) {
        DenseLayer& D = m->dense[j];
        TR_TRY(step(D.d_w, T.dense_w_off[j], (size_t)D.out * D.in));
        TR_TRY(step(D.d_b, T.dense_b_off[j], (size_t)D.out));
    }
    m->cached_B = 0;                                         // cached activations no longer match the weights
    T.tc_dirty = true;
    TR_TRY(m->mark("end", s));
    BCAD_CUDA_CHECK(cudaEventRecord(m->call_done, s));
    return BCAD_OK;
}

// weights back in the caller's layouts (save_model Classes/CNNModel.py:530-555; state_dict ADCNNM.py:150)
int bcad_get_conv_weights(bcad_model* mm, int i, float* filters_fkkc, float* bias) {
    Model* m = reinterpret_cast<Model*>(mm);
    BCAD_REQUIRE(m && filters_fkkc, "get_conv_weights: null argument");
    BCAD_REQUIRE(i >= 0 && i < (int)m->conv.size(), "conv index %d out of range", i);
    if (!m->committed) { set_error("weights not committed"); return BCAD_ERR_STATE; }
    DeviceGuard g(m->cfg.device);
    ConvLayer& L = m->conv[i];
    BCAD_CUDA_CHECK(cudaDeviceSynchronize());
    std::vector<float> pk((size_t)L.k * L.k * L.Cin * L.CoutPad), pb(L.CoutPad);
    BCAD_CUDA_CHECK(cudaMemcpy(pk.data(), L.d_w, pk.size() * sizeof(float), cudaMemcpyDeviceToHost));
    BCAD_CUDA_CHECK(cudaMemcpy(pb.data(), L.d_b, pb.size() * sizeof(float), cudaMemcpyDeviceToHost));
    for (int f = 0; f < L.Cout; ++f) {
        if (bias) bias[f] = pb[f];
        L.h_b[f] = pb[f];
        for (int t = 0; t < L.k * L.k; ++t)
            for (int c = 0; c < L.Cin; ++c) {
                const float v = pk[((size_t)t * L.Cin + c) * L.CoutPad + f];
                filters_fkkc[((size_t)f * L.k * L.k + t) * L.Cin + c] = v;
                L.h_w[((size_t)f * L.k * L.k + t) * L.Cin + c] = v;
            }
    }
    return BCAD_OK;
}

int bcad_get_dense_weights(bcad_model* mm, int j, float* w, float* bias) {
    Model* m = reinterpret_cast<Model*>(mm);
    BCAD_REQUIRE(m && w, "get_dense_weights: null argument");
    BCAD_REQUIRE(j >= 0 && j < (int)m->dense.size(), "dense index %d out of range", j);
    if (!m->committed) { set_error("weights not committed"); return BCAD_ERR_STATE; }
    DeviceGuard g(m->cfg.device);
    DenseLayer& D = m->dense[j];
    if (D.d_w == nullptr) { set_error("dense %d has no fp32 device weights (tensor path)", j); return BCAD_ERR_STATE; }
    BCAD_CUDA_CHECK(cudaDeviceSynchronize());
    BCAD_CUDA_CHECK(cudaMemcpy(D.h_w.data(), D.d_w, D.h_w.size() * sizeof(float), cudaMemcpyDeviceToHost));
    BCAD_CUDA_CHECK(cudaMemcpy(D.h_b.data(), D.d_b, D.h_b.size() * sizeof(float), cudaMemcpyDeviceToHost));
    if (bias) memcpy(bias, D.h_b.data(), D.h_b.size() * sizeof(float));
    if (j == 0 && m->cfg.flatten_order == BCAD_FLATTEN_CHW) {
        const ConvLayer& L = m->conv.back();
        const int C = L.Cout, H = L.Hp, W = L.Wp;
        for (int u = 0; u < D.out; ++u) {
            const float* src = D.h_w.data() + (size_t)u * D.in;
            float* dst = w + (size_t)u * D.in;
            for (int c = 0; c < C; ++c)
                for (int y = 0; y < H; ++y)
                    for (int x = 0; x < W; ++x) dst[((size_t)c * H + y) * W + x] = src[((size_t)y * W + x) * C + c];
        }
    } else {
        memcpy(w, D.h_w.data(), D.h_w.size() * sizeof(float));
    }
    return BCAD_OK;
}

}  // extern "C"
