// libbcad C-ABI: model handle, weight packing, and the predict / predict+Grad-CAM drivers.
// Reference interfaces behind each entry point are cited in include/bcad.h.
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <new>
#include <vector>

#include "../../include/bcad.h"
#include "common.cuh"
#include "kernels.h"
#include "model.h"
#include "sm100_train.h"

namespace bcad {

static thread_local char g_err[1024] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int Model::alloc(void** p, size_t bytes) {
    if (bytes == 0) bytes = 16;
    cudaError_t e = cudaMalloc(p, bytes);
    if (e != cudaSuccess) {
        set_error("cudaMalloc(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
        return BCAD_ERR_NOMEM;
    }
    allocs.push_back(*p);
    ws_bytes += bytes;
    return BCAD_OK;
}

void Model::free_all() {
    for (void* p : allocs) cudaFree(p);
    allocs.clear();
    if (xfer.inited) {
        for (int i = 0; i < 2; ++i) {
            cudaEventDestroy(xfer.in_done[i]);
            cudaEventDestroy(xfer.compute_done[i]);
            cudaEventDestroy(xfer.out_done[i]);
        }
        cudaStreamDestroy(xfer.s_in);
        cudaStreamDestroy(xfer.s_compute);
        cudaStreamDestroy(xfer.s_out);
        if (xfer.h_small) cudaFreeHost(xfer.h_small);
        xfer.h_small = nullptr;
        xfer.inited = false;
    }
    for (cudaEvent_t e : prof_pool) cudaEventDestroy(e);
    prof_pool.clear();
    if (call_done) cudaEventDestroy(call_done);
}

// profiling: one CUDA event before every kernel of a call (only when switched on)
int Model::mark(const char* name, cudaStream_t s) {
    if (!profiling) return BCAD_OK;
    if (prof_n == (int)prof_pool.size()) {
        cudaEvent_t e;
        BCAD_CUDA_CHECK(cudaEventCreate(&e));
        prof_pool.push_back(e);
        prof_names.push_back(name);
    }
    prof_names[prof_n] = name;
    BCAD_CUDA_CHECK(cudaEventRecord(prof_pool[prof_n], s));
    ++prof_n;
    return BCAD_OK;
}

#define BCAD_TRY(expr)                \
    do {                              \
        int _rc = (expr);             \
        if (_rc != BCAD_OK) return _rc; \
    } while (0)

#define BCAD_LAUNCH(m, name, expr)    \
    do {                              \
        int _rc = (m)->mark(name, s); \
        if (_rc == BCAD_OK) _rc = (expr); \
        if (_rc != BCAD_OK) return _rc; \
        (m)->launches += 1;           \
    } while (0)

// -----------------------------------------------------------------------------------------------------
static int validate(const bcad_config& c) {
    BCAD_REQUIRE(c.in_h > 0 && c.in_w > 0 && c.in_c > 0, "input_shape must be positive, got (%d,%d,%d)", c.in_h, c.in_w, c.in_c);
    BCAD_REQUIRE(c.num_classes >= 1 && c.num_classes <= 1024, "num_classes %d out of range", c.num_classes);
    BCAD_REQUIRE(c.n_conv >= 1 && c.n_conv <= BCAD_MAX_CONV, "n_conv %d out of range 1..%d", c.n_conv, BCAD_MAX_CONV);
    BCAD_REQUIRE(c.n_hidden >= 0 && c.n_hidden < BCAD_MAX_DENSE, "n_hidden %d out of range 0..%d", c.n_hidden, BCAD_MAX_DENSE - 1);
    BCAD_REQUIRE(c.pad >= 0 && c.pad <= 3, "pad %d out of range 0..3", c.pad);
    BCAD_REQUIRE(c.flatten_order == BCAD_FLATTEN_HWC || c.flatten_order == BCAD_FLATTEN_CHW, "bad flatten_order %d", c.flatten_order);
    BCAD_REQUIRE(c.pool_ties == BCAD_TIES_ALL || c.pool_ties == BCAD_TIES_FIRST, "bad pool_ties %d", c.pool_ties);
    BCAD_REQUIRE(c.head == BCAD_HEAD_SOFTMAX_CLIP || c.head == BCAD_HEAD_LOGITS, "bad head %d", c.head);
    BCAD_REQUIRE(c.precision == BCAD_PREC_FP32 || c.precision == BCAD_PREC_F16 || c.precision == BCAD_PREC_F16X3, "bad precision %d", c.precision);
    BCAD_REQUIRE(c.max_batch >= 1 && c.max_batch <= 65535, "max_batch %d out of range 1..65535", c.max_batch);
    BCAD_REQUIRE(c.alpha_conv >= 0.f && c.alpha_dense >= 0.f, "negative LeakyReLU slope is not supported (pool/activation fusion assumes a monotone activation)");
    BCAD_REQUIRE(c.refine_margin >= 0.f && c.refine_margin == c.refine_margin, "refine_margin must be >= 0");
    BCAD_REQUIRE(c.refine_margin == 0.f || c.precision == BCAD_PREC_F16, "refine_margin applies to BCAD_PREC_F16 only (the other paths are fp32-grade already)");
    BCAD_REQUIRE(c.refine_capacity >= 0, "refine_capacity must be >= 0");
    return BCAD_OK;
}

}  // namespace bcad

using namespace bcad;

extern "C" {

const char* bcad_last_error(void) { return g_err; }
const char* bcad_version(void) { return "libbcad 0.1 (sm_100a)"; }

int bcad_create(const bcad_config* cfg, bcad_model** out) {
    if (cfg == nullptr || out == nullptr) {
        set_error("bcad_create: null argument");
        return BCAD_ERR_INVALID;
    }
    *out = nullptr;
    BCAD_TRY(validate(*cfg));
    int ndev = 0;
    BCAD_CUDA_CHECK(cudaGetDeviceCount(&ndev));
    BCAD_REQUIRE(cfg->device >= 0 && cfg->device < ndev, "device %d not available (%d visible)", cfg->device, ndev);
    Model* m = new (std::nothrow) Model();
    if (!m) {
        set_error("out of host memory");
        return BCAD_ERR_NOMEM;
    }
    m->cfg = *cfg;
    int h = cfg->in_h, w = cfg->in_w, c = cfg->in_c;
    for (int i = 0; i < cfg->n_conv; ++i) {
        ConvLayer L;
        L.Cin = c; L.Cout = cfg->conv_filters[i]; L.k = cfg->conv_ksize[i];
        L.H = h; L.W = w;
        L.Ho = h + 2 * cfg->pad - L.k + 1; L.Wo = w + 2 * cfg->pad - L.k + 1;
        L.Hp = L.Ho / 2; L.Wp = L.Wo / 2;
        L.CoutPad = cdiv(L.Cout, 32) * 32;
        if (L.Cout < 1 || L.k < 1 || L.k > 7 || L.Ho < 1 || L.Wo < 1 || L.Hp < 1 || L.Wp < 1) {
            set_error("conv block %d: filters=%d ksize=%d on a %dx%d map is not a valid layer (ksize 1..7, pooled map must be >= 1x1)",
                      i, L.Cout, L.k, h, w);
            delete m;
            return BCAD_ERR_INVALID;
        }
        m->conv.push_back(L);
        h = L.Hp; w = L.Wp; c = L.Cout;
    }
    m->flat = (int64_t)h * w * c;
    int prev = (int)m->flat;
    if (m->flat > 0x7fffffff) {
        set_error("flattened size %lld too large", (long long)m->flat);
        delete m;
        return BCAD_ERR_INVALID;
    }
    for (int j = 0; j <= cfg->n_hidden; ++j) {
        DenseLayer D;
        D.in = prev;
        D.out = (j < cfg->n_hidden) ? cfg->hidden_units[j] : cfg->num_classes;
        if (D.out < 1) {
            set_error("dense layer %d has %d units", j, D.out);
            delete m;
            return BCAD_ERR_INVALID;
        }
        m->dense.push_back(D);
        prev = D.out;
    }
    if (cfg->precision == BCAD_PREC_F16 || cfg->precision == BCAD_PREC_F16X3) {
        int rc = tensor_path_supported(*m);
        if (rc != BCAD_OK) {
            delete m;
            return rc;
        }
        m->tensor_path = true;
    }
    if (cfg->refine_margin > 0.f) {
        // the fp32-grade twin the small-margin images are re-run on (refine.cu)
        bcad_config c2 = *cfg;
        c2.precision = BCAD_PREC_F16X3;
        c2.refine_margin = 0.f;
        c2.refine_capacity = 0;
        c2.keep_all_activations = 0;
        int cap = cfg->refine_capacity > 0 ? cfg->refine_capacity : std::max(8, cfg->max_batch / 32);
        cap = std::min(cap, cfg->max_batch);
        c2.max_batch = cap;
        bcad_model* tw = nullptr;
        int rc = bcad_create(&c2, &tw);
        if (rc != BCAD_OK) {                       // (the twin's message says which shape limit was hit)
            delete m;
            return rc;
        }
        m->refine.twin = reinterpret_cast<Model*>(tw);
        m->refine.cap = cap;
    }
    *out = reinterpret_cast<bcad_model*>(m);
    return BCAD_OK;
}

void bcad_destroy(bcad_model* mm) {
    if (!mm) return;
    Model* m = reinterpret_cast<Model*>(mm);
    if (m->refine.twin) bcad_destroy(reinterpret_cast<bcad_model*>(m->refine.twin));
    m->refine.twin = nullptr;
    {
        DeviceGuard g(m->cfg.device);
        cudaDeviceSynchronize();
        if (m->tp) tensor_path_destroy(*m);
        m->free_all();
    }
    delete m;
}

int bcad_set_conv_weights(bcad_model* mm, int i, const float* filters, const float* bias) {
    Model* m = reinterpret_cast<Model*>(mm);
    BCAD_REQUIRE(m && filters, "set_conv_weights: null argument");
    BCAD_REQUIRE(i >= 0 && i < (int)m->conv.size(), "conv index %d out of range", i);
    std::lock_guard<std::mutex> lock(m->mu);
    ConvLayer& L = m->conv[i];
    const size_t n = (size_t)L.Cout * L.k * L.k * L.Cin;
    L.h_w.assign(filters, filters + n);
    if (bias) L.h_b.assign(bias, bias + L.Cout);
    else L.h_b.assign(L.Cout, 0.f);
    m->committed = false;
    if (m->refine.twin) return bcad_set_conv_weights(reinterpret_cast<bcad_model*>(m->refine.twin), i, filters, bias);
    return BCAD_OK;
}

int bcad_set_dense_weights(bcad_model* mm, int j, const float* w, const float* bias) {
    Model* m = reinterpret_cast<Model*>(mm);
    BCAD_REQUIRE(m && w, "set_dense_weights: null argument");
    BCAD_REQUIRE(j >= 0 && j < (int)m->dense.size(), "dense index %d out of range", j);
    std::lock_guard<std::mutex> lock(m->mu);
    DenseLayer& D = m->dense[j];
    const size_t n = (size_t)D.out * D.in;
    D.h_w.resize(n);
    if (j == 0 && m->cfg.flatten_order == BCAD_FLATTEN_CHW) {
        // caller columns are (c,h,w); the device flattens NHWC => permute to (h,w,c)  [SURVEY 7, hard part 1]
        const ConvLayer& L = m->conv.back();
        const int C = L.Cout, H = L.Hp, W = L.Wp;
        for (int u = 0; u < D.out; ++u) {
            const float* src = w + (size_t)u * D.in;
            float* dst = D.h_w.data() + (size_t)u * D.in;
            for (int c = 0; c < C; ++c)
                for (int y = 0; y < H; ++y)
                    for (int x = 0; x < W; ++x) dst[((size_t)y * W + x) * C + c] = src[((size_t)c * H + y) * W + x];
        }
    } else {
        memcpy(D.h_w.data(), w, n * sizeof(float));
    }
    if (bias) D.h_b.assign(bias, bias + D.out);
    else D.h_b.assign(D.out, 0.f);
    m->committed = false;
    if (m->refine.twin) return bcad_set_dense_weights(reinterpret_cast<bcad_model*>(m->refine.twin), j, w, bias);
    return BCAD_OK;
}

int bcad_fold_batchnorm(bcad_model* mm, int i, const float* gamma, const float* beta, const float* mean,
                        const float* var, float eps) {
    Model* m = reinterpret_cast<Model*>(mm);
    BCAD_REQUIRE(m && gamma && beta && mean && var, "fold_batchnorm: null argument");
    BCAD_REQUIRE(i >= 0 && i < (int)m->conv.size(), "conv index %d out of range", i);
    std::lock_guard<std::mutex> lock(m->mu);
    ConvLayer& L = m->conv[i];
    BCAD_REQUIRE(!L.h_w.empty(), "fold_batchnorm: conv %d has no staged weights", i);
    const size_t per = (size_t)L.k * L.k * L.Cin;
    for (int f = 0; f < L.Cout; ++f) {
        const float sc = gamma[f] / sqrtf(var[f] + eps);
        for (size_t q = 0; q < per; ++q) L.h_w[f * per + q] *= sc;
        L.h_b[f] = (L.h_b[f] - mean[f]) * sc + beta[f];
    }
    m->committed = false;
    if (m->refine.twin) return bcad_fold_batchnorm(reinterpret_cast<bcad_model*>(m->refine.twin), i, gamma, beta, mean, var, eps);
    return BCAD_OK;
}

static int upload(Model* m, float** dst, const std::vector<float>& src) {
    if (*dst == nullptr) BCAD_TRY(m->alloc((void**)dst, src.size() * sizeof(float)));
    BCAD_CUDA_CHECK(cudaMemcpy(*dst, src.data(), src.size() * sizeof(float), cudaMemcpyHostToDevice));
    return BCAD_OK;
}

int bcad_commit(bcad_model* mm) {
    Model* m = reinterpret_cast<Model*>(mm);
    BCAD_REQUIRE(m, "commit: null model");
    DeviceGuard g(m->cfg.device);
    std::lock_guard<std::mutex> lock(m->mu);
    for (size_t i = 0; i < m->conv.size(); ++i)
        if (m->conv[i].h_w.empty()) { set_error("commit: conv %zu has no weights", i); return BCAD_ERR_STATE; }
    for (size_t j = 0; j < m->dense.size(); ++j)
        if (m->dense[j].h_w.empty()) { set_error("commit: dense %zu has no weights", j); return BCAD_ERR_STATE; }
    BCAD_CUDA_CHECK(cudaDeviceSynchronize());
    const int mb = m->cfg.max_batch;
    // ---- fp32 packed weights (always kept: parity anchor, compat tensors, explain_backward)
    for (size_t i = 0; i < m->conv.size(); ++i) {
        ConvLayer& L = m->conv[i];
        std::vector<float> pk((size_t)L.k * L.k * L.Cin * L.CoutPad, 0.f), pb(L.CoutPad, 0.f);
        for (int f = 0; f < L.Cout; ++f) {
            pb[f] = L.h_b[f];
            for (int t = 0; t < L.k * L.k; ++t)
                for (int c = 0; c < L.Cin; ++c)
                    pk[((size_t)t * L.Cin + c) * L.CoutPad + f] = L.h_w[((size_t)f * L.k * L.k + t) * L.Cin + c];
        }
        BCAD_TRY(upload(m, &L.d_w, pk));
        BCAD_TRY(upload(m, &L.d_b, pb));
        // dgrad weights: correlation of dz with flipped filters, outputs = Cin  (explainability.py:60)
        const int cpad = cdiv(L.Cin, 32) * 32;
        std::vector<float> dk((size_t)L.k * L.k * L.Cout * cpad, 0.f);
        for (int f = 0; f < L.Cout; ++f)
            for (int ky = 0; ky < L.k; ++ky)
                for (int kx = 0; kx < L.k; ++kx)
                    for (int c = 0; c < L.Cin; ++c) {
                        const int t2 = (L.k - 1 - ky) * L.k + (L.k - 1 - kx);
                        dk[((size_t)t2 * L.Cout + f) * cpad + c] = L.h_w[(((size_t)f * L.k + ky) * L.k + kx) * L.Cin + c];
                    }
        BCAD_TRY(upload(m, &L.d_w_dgrad, dk));
        if (L.d_zero_bias == nullptr) {
            std::vector<float> zb(cpad, 0.f);
            BCAD_TRY(upload(m, &L.d_zero_bias, zb));
        }
    }
    for (size_t j = 0; j < m->dense.size(); ++j) {
        DenseLayer& D = m->dense[j];
        // the tensor path keeps fc1 as 16-bit tiles only (126-134 MB instead of 3x that) -- unless the tie-duplicating pool rule
        // is on: its Grad-CAM weights need the dense pooled gradient, i.e. the fp32 fc1 input-gradient GEMM
        if (!(m->tensor_path && j == 0 && m->cfg.pool_ties == BCAD_TIES_FIRST))
            BCAD_TRY(upload(m, &D.d_w, D.h_w));
        BCAD_TRY(upload(m, &D.d_b, D.h_b));
    }
    // ---- workspace (first commit only)
    if (!m->ws_ready) {
        const size_t last = m->conv.size() - 1;
        for (size_t i = 0; i < m->conv.size(); ++i) {
            ConvLayer& L = m->conv[i];
            const bool fp32_acts = !m->tensor_path;
            if (fp32_acts && (i == last || m->cfg.keep_all_activations))
                BCAD_TRY(m->alloc((void**)&L.y, (size_t)mb * L.Ho * L.Wo * L.Cout * sizeof(float)));
            if (fp32_acts) BCAD_TRY(m->alloc((void**)&L.p, (size_t)mb * L.Hp * L.Wp * L.Cout * sizeof(float)));
        }
        size_t part_elems = 16;
        for (size_t j = 0; j < m->dense.size(); ++j) {
            DenseLayer& D = m->dense[j];
            BCAD_TRY(m->alloc((void**)&D.z, (size_t)mb * D.out * sizeof(float)));
            BCAD_TRY(m->alloc((void**)&D.h, (size_t)mb * D.out * sizeof(float)));
            D.splits = sgemm_pick_splits(mb, D.out, D.in);
            part_elems = std::max(part_elems, (size_t)D.splits * mb * D.out);
        }
        BCAD_TRY(m->alloc((void**)&m->partials, part_elems * sizeof(float)));
        BCAD_TRY(m->alloc((void**)&m->probs, (size_t)mb * m->cfg.num_classes * sizeof(float)));
        BCAD_TRY(m->alloc((void**)&m->cls, (size_t)mb * sizeof(int32_t)));
        BCAD_TRY(m->alloc((void**)&m->d_top, (size_t)mb * m->cfg.num_classes * sizeof(float)));
        m->fused_head = fused_head_ok(m);
        if (!m->tensor_path || m->cfg.pool_ties != BCAD_TIES_FIRST) BCAD_TRY(m->alloc((void**)&m->g_flat, (size_t)mb * m->flat * sizeof(float)));
        const ConvLayer& T = m->conv.back();
        m->alpha_splits = alpha_pool_splits(T.Hp);
        m->cam_splits = cam_splits(T.Ho);
        BCAD_TRY(m->alloc((void**)&m->alpha_part, (size_t)mb * m->alpha_splits * T.Cout * sizeof(float)));
        BCAD_TRY(m->alloc((void**)&m->alpha, (size_t)mb * T.Cout * sizeof(float)));
        BCAD_TRY(m->alloc((void**)&m->cam_lo, (size_t)mb * T.Ho * T.Wo * sizeof(float)));
        BCAD_TRY(m->alloc((void**)&m->mm, (size_t)mb * m->cam_splits * 2 * sizeof(float)));
        BCAD_TRY(m->alloc((void**)&m->class_cols, (size_t)BCAD_MAX_EXPLAIN_CLASSES * mb * sizeof(int32_t)));
        BCAD_CUDA_CHECK(cudaEventCreateWithFlags(&m->call_done, cudaEventDisableTiming));
        m->ws_ready = true;
    }
    if (m->tensor_path) BCAD_TRY(tensor_path_commit(*m));
    if (m->refine.twin) {
        Refine& R = m->refine;
        BCAD_TRY(bcad_commit(reinterpret_cast<bcad_model*>(R.twin)));
        if (R.idx == nullptr) {
            const size_t img = (size_t)m->cfg.in_h * m->cfg.in_w * m->cfg.in_c, hm = (size_t)m->cfg.in_h * m->cfg.in_w;
            BCAD_TRY(m->alloc((void**)&R.idx, (size_t)R.cap * sizeof(int32_t)));
            BCAD_TRY(m->alloc((void**)&R.counters, 4 * sizeof(int32_t)));
            BCAD_TRY(m->alloc((void**)&R.x, (size_t)R.cap * img * sizeof(float)));
            BCAD_TRY(m->alloc((void**)&R.cidx, (size_t)R.cap * sizeof(int32_t)));
            BCAD_TRY(m->alloc((void**)&R.heat, (size_t)R.cap * hm * sizeof(float)));
            R.heat_elems = hm;
            BCAD_CUDA_CHECK(cudaMemset(R.counters, 0, 4 * sizeof(int32_t)));
            BCAD_CUDA_CHECK(cudaMemset(R.idx, 0, (size_t)R.cap * sizeof(int32_t)));
            R.twin->n_dev = R.counters;          // counters[0]: images flagged in the current chunk
        }
    }
    BCAD_CUDA_CHECK(cudaDeviceSynchronize());
    m->committed = true;
    m->cached_B = 0;
    m->train.tc_dirty = true;
    return BCAD_OK;
}

}  // extern "C"

namespace bcad {

// -----------------------------------------------------------------------------------------------------
// fp32 path: one chunk (n <= max_batch) forward, activations cached in the workspace
// -----------------------------------------------------------------------------------------------------
bool fused_head_ok(const Model* m) {
    size_t total = 0, mx = 0;
    for (const DenseLayer& D : m->dense) { total += D.out; mx = std::max(mx, (size_t)D.out); }
    return (total + 2 * mx) * sizeof(float) <= 40 * 1024 && m->dense.size() <= 8;
}

// One launch for everything after the fc1 GEMM (see dense_head_kernel).
int launch_fused_head(Model* m, int n, const float* fc1_part, int splits, size_t ld, bool explain, const int32_t* class_idx,
                      int grad_mode, float* dz1, const float* S, int C, float* alpha_raw, cudaStream_t s) {
    HeadArgs a;
    memset(&a, 0, sizeof(a));
    a.n_dense = (int)m->dense.size();
    a.max_size = 0;
    for (int j = 0; j < a.n_dense; ++j) {
        a.sizes[j] = m->dense[j].out;
        a.max_size = std::max(a.max_size, m->dense[j].out);
        a.W[j] = m->dense[j].d_w;
        a.bias[j] = m->dense[j].d_b;
        a.z[j] = m->dense[j].z;
    }
    a.fc1_part = fc1_part; a.fc1_splits = splits; a.fc1_ld = ld;
    a.alpha = m->cfg.alpha_dense; a.head = m->cfg.head; a.probs = m->probs; a.cls = m->cls;
    a.explain = explain ? 1 : 0; a.class_idx = class_idx; a.grad_mode = grad_mode;
    a.dz1 = dz1; a.S = S; a.C = C; a.alpha_raw = alpha_raw; a.n_dev = m->n_dev;
    m->head_last = a;
    m->head_n = n;
    BCAD_LAUNCH(m, "dense_head_fused", launch_dense_head(a, n, s));
    return BCAD_OK;
}

int relaunch_fused_head(Model* m, const int32_t* class_idx, float* alpha_raw, cudaStream_t s) {
    HeadArgs a = m->head_last;
    a.class_idx = class_idx;
    if (a.alpha_raw != nullptr) a.alpha_raw = alpha_raw;
    BCAD_LAUNCH(m, "dense_head_fused", launch_dense_head(a, m->head_n, s));
    return BCAD_OK;
}

static int forward_chunk_fp32(Model* m, const float* x, int n, bool explain, const int32_t* class_idx, int grad_mode,
                              cudaStream_t s) {
    const float* in = x;
    if (m->fast_train) BCAD_TRY(tc_train_refresh(m, s));
    for (size_t i = 0; i < m->conv.size(); ++i) {
        ConvLayer& L = m->conv[i];
        if (m->fast_train && i == 0 && L.Cin == 1 && L.Cout == 32 && L.CoutPad == 32 && L.k == 3 && L.y != nullptr && L.p != nullptr &&
            getenv("BCAD_TC_NO_CONV0") == nullptr) {
            // first block, one input channel: conv + bias + LeakyReLU + 2x2 pool in one pass, lane = filter (sm100_train.cu)
            BCAD_LAUNCH(m, "conv0_fwd_fused", launch_conv0_fwd_fused(in, L.d_w, L.d_b, L.y, L.p, n, L.H, L.W, L.Ho, L.Wo, m->cfg.pad, m->cfg.alpha_conv, m->sms, s));
            in = L.p;
            continue;
        }
        if (m->fast_train && tc_train_eligible(m, i) && L.y != nullptr) {
            // the block as a split-operand tcgen05 implicit GEMM on the fp32 NHWC tensors (sm100_train.cu), then the 2x2 pool
            TcConvArgs t;
            t.x = in; t.w_img = L.tc_w; t.bias = L.d_b; t.y = L.y; t.B = n; t.H = L.H; t.W = L.W; t.Ho = L.Ho; t.Wo = L.Wo;
            t.pad = m->cfg.pad; t.alpha = m->cfg.alpha_conv; t.a_bf16 = 0;
            BCAD_LAUNCH(m, "conv1_fwd_tcgen05_x3", launch_conv3x3_x3(t, L.Cin, L.Cout, m->sms, s));
            BCAD_LAUNCH(m, "maxpool2x2", launch_maxpool2x2_nhwc(L.y, L.p, n, L.Ho, L.Wo, L.Cout, s));
            in = L.p;
            continue;
        }
        ConvArgs a;
        a.x = in; a.w = L.d_w; a.bias = L.d_b; a.y = L.y; a.p = L.p;
        a.B = n; a.H = L.H; a.W = L.W; a.Cin = L.Cin; a.Cout = L.Cout; a.CoutPad = L.CoutPad;
        a.ksize = L.k; a.pad = m->cfg.pad; a.Ho = L.Ho; a.Wo = L.Wo; a.Hp = L.Hp; a.Wp = L.Wp;
        a.alpha = m->cfg.alpha_conv;
        BCAD_LAUNCH(m, i == 0 ? "conv0_fp32" : (i == 1 ? "conv1_fp32" : "convN_fp32"), launch_conv_fp32(a, s));
        in = L.p;
    }
    // fc1 as a split-K SGEMM, then either the fused head or the layer-by-layer chain
    DenseLayer& D0 = m->dense[0];
    int splits0 = std::min(D0.splits, sgemm_pick_splits(n, D0.out, D0.in));
    float* fc_part = m->partials;
    if (m->fast_train && dense_fwd_x3_supported(n, D0.out, D0.in) && getenv("BCAD_TC_NO_DENSE") == nullptr) {
        // fast training: fc1 as a split-K, split-operand tcgen05 GEMM on the fp32 tensors (sm100_train.cu)
        splits0 = dense_fwd_x3_splits(D0.in, m->sms);
        if (m->train.fc_part == nullptr) BCAD_TRY(m->alloc((void**)&m->train.fc_part, (size_t)splits0 * 64 * D0.out * sizeof(float)));
        fc_part = m->train.fc_part;
        DenseFwdArgs f;
        f.p = in; f.w = D0.d_w; f.partials = fc_part; f.B = n; f.units = D0.out; f.flat = D0.in;
        BCAD_LAUNCH(m, "fc1_fwd_tcgen05_x3", launch_dense_fwd_x3(f, m->sms, s));
    } else
    BCAD_LAUNCH(m, "fc1_sgemm", launch_sgemm(in, D0.d_w, m->partials, n, D0.out, D0.in, true, splits0, s));
    const float* drop = m->train.drop_B ? m->train.drop : nullptr;   // training forward: dropout after every hidden layer
    if (drop && m->train.drop_B != n) {
        set_error("dropout masks are set for a batch of %d, this forward has %d images (clear them with bcad_set_dropout_masks(m, NULL, 0))", m->train.drop_B, n);
        return BCAD_ERR_STATE;
    }
    if (m->fused_head && !drop) {
        BCAD_TRY(launch_fused_head(m, n, fc_part, splits0, (size_t)n * D0.out, explain, class_idx, grad_mode,
                                   explain ? D0.h : nullptr, nullptr, 0, nullptr, s));
        return BCAD_OK;
    }
    const bool only = (m->dense.size() == 1);
    BCAD_LAUNCH(m, "splitk_reduce", launch_splitk_reduce(fc_part, splits0, D0.d_b, D0.z, only ? nullptr : D0.h, m->cfg.alpha_dense, n, D0.out, s));
    if (drop && !only) BCAD_LAUNCH(m, "dropout", launch_mul_mask(D0.h, drop + m->train.drop_off[0], n, D0.out, m->train.drop_ld, s));
    in = D0.h;
    for (size_t j = 1; j < m->dense.size(); ++j) {
        DenseLayer& D = m->dense[j];
        const bool last = (j + 1 == m->dense.size());
        const int splits = std::min(D.splits, sgemm_pick_splits(n, D.out, D.in));
        BCAD_LAUNCH(m, "sgemm", launch_sgemm(in, D.d_w, m->partials, n, D.out, D.in, true, splits, s));
        BCAD_LAUNCH(m, "splitk_reduce", launch_splitk_reduce(m->partials, splits, D.d_b, D.z, last ? nullptr : D.h, m->cfg.alpha_dense, n, D.out, s));
        if (drop && !last) BCAD_LAUNCH(m, "dropout", launch_mul_mask(D.h, drop + m->train.drop_off[j], n, D.out, m->train.drop_ld, s));
        in = D.h;
    }
    BCAD_LAUNCH(m, "head", launch_head(m->dense.back().z, m->probs, m->cls, n, m->cfg.num_classes, m->cfg.head, s));
    return BCAD_OK;
}

// dense backward from d_top to the gradient w.r.t. the first dense layer's PRE-activation (dz1, in
// dense[0].d) and, when g_flat != nullptr, on to the flattened pool output (NHWC order).
int dense_backward(Model* m, int n, const int32_t* class_idx, int grad_mode, float* g_flat, cudaStream_t s) {
    const int nc = m->cfg.num_classes;
    BCAD_LAUNCH(m, "top_grad", launch_top_grad(m->probs, m->cls, class_idx, m->d_top, n, nc, grad_mode, s));
    const float* d = m->d_top;
    for (int j = (int)m->dense.size() - 1; j >= 0; --j) {
        DenseLayer& D = m->dense[j];
        // for j < last, D.h holds dL/d(LeakyReLU(z_j)) written by the step above: mask it in place into dz_j
        if (j + 1 < (int)m->dense.size()) {
            BCAD_LAUNCH(m, "leaky_mask_mul", launch_leaky_mask_mul(D.h, D.z, m->cfg.alpha_dense, (int64_t)n * D.out, s));
            d = D.h;
        }
        float* dst = (j > 0) ? m->dense[j - 1].h : g_flat;    // dense[j-1].h is dead after the forward
        if (dst == nullptr) break;
        BCAD_LAUNCH(m, "sgemm", launch_sgemm(d, D.d_w, dst, n, D.in, D.out, false, 1, s));
    }
    return BCAD_OK;
}

int conv_block_dz(Model* m, int i, const float* gp, int B, bool fused, float* act_grad, bool mask, cudaStream_t s) {
    ConvLayer& L = m->conv[i];
    const size_t elems = (size_t)B * L.Ho * L.Wo * L.Cout;
    if (L.dz == nullptr) BCAD_TRY(m->alloc((void**)&L.dz, (size_t)m->cfg.max_batch * L.Ho * L.Wo * L.Cout * sizeof(float)));
    if (fused) {
        const int first_only = (m->cfg.pool_ties == BCAD_TIES_FIRST) ? 1 : 0;
        BCAD_LAUNCH(m, "unpool_mask", launch_unpool_mask(gp, L.y, L.dz, B, L.Ho, L.Wo, L.Cout, first_only, m->cfg.alpha_conv, s));
        return BCAD_OK;
    }
    BCAD_LAUNCH(m, "unpool", launch_unpool(gp, L.y, L.dz, B, L.Ho, L.Wo, L.Cout, m->cfg.pool_ties, s));
    if (act_grad) BCAD_CUDA_CHECK(cudaMemcpyAsync(act_grad, L.dz, elems * sizeof(float), cudaMemcpyDeviceToDevice, s));
    if (mask) BCAD_LAUNCH(m, "leaky_mask_mul", launch_leaky_mask_mul(L.dz, L.y, m->cfg.alpha_conv, (int64_t)elems, s));   // explainability.py:55
    return BCAD_OK;
}

int conv_block_dgrad(Model* m, int i, int B, float* dst, bool tc, const char* name, cudaStream_t s) {
    ConvLayer& L = m->conv[i];
    if (dst == nullptr) {
        ConvLayer& P = m->conv[i - 1];
        if (P.gp == nullptr) BCAD_TRY(m->alloc((void**)&P.gp, (size_t)m->cfg.max_batch * P.Hp * P.Wp * P.Cout * sizeof(float)));
        dst = P.gp;
    }
    if (tc) {
        TcConvArgs t;
        t.x = L.dz; t.w_img = L.tc_wd; t.bias = nullptr; t.y = dst; t.B = B; t.H = L.Ho; t.W = L.Wo; t.Ho = L.H; t.Wo = L.W;
        t.pad = L.k - 1 - m->cfg.pad; t.alpha = 1.f; t.a_bf16 = 1;
        BCAD_LAUNCH(m, "conv_dgrad_tcgen05_x3", launch_conv3x3_x3(t, L.Cout, L.Cin, m->sms, s));
        return BCAD_OK;
    }
    ConvArgs a;
    a.x = L.dz; a.w = L.d_w_dgrad; a.bias = L.d_zero_bias; a.y = dst; a.p = nullptr;
    a.B = B; a.H = L.Ho; a.W = L.Wo; a.Cin = L.Cout; a.Cout = L.Cin; a.CoutPad = cdiv(L.Cin, 32) * 32;
    a.ksize = L.k; a.pad = L.k - 1 - m->cfg.pad; a.Ho = L.H; a.Wo = L.W; a.Hp = 0; a.Wp = 0; a.alpha = 1.f;
    BCAD_LAUNCH(m, name, launch_conv_fp32(a, s));
    return BCAD_OK;
}

static int tail_chunk(Model* m, const void* A, int a_dtype, int n, float* heat, size_t heat_stride, cudaStream_t s) {
    const ConvLayer& T = m->conv.back();
    const float inv_hw = 1.0f / ((float)T.Ho * (float)T.Wo);
    const float inv_slope = (m->target == BCAD_TARGET_CONV_PREACT) ? 1.0f / m->cfg.alpha_conv : 0.f;
    BCAD_LAUNCH(m, "cam", launch_cam(A, a_dtype, m->alpha_part, m->alpha_splits, inv_hw, m->alpha, m->cam_lo, m->mm, n, T.Ho,
                              T.Wo, T.Cout, m->cam_splits, s, inv_slope));
    BCAD_LAUNCH(m, "upsample_norm", launch_upsample_norm(m->cam_lo, m->mm, m->cam_splits, heat, n, T.Ho, T.Wo, m->heat_h, m->heat_w, s, nullptr, heat_stride));
    return BCAD_OK;
}

static int explain_chunk_fp32(Model* m, int n, const int32_t* class_idx, int grad_mode, float* heat, size_t heat_stride, cudaStream_t s) {
    const ConvLayer& T = m->conv.back();
    if (m->fused_head) {
        // dz1 was left in dense[0].h by the fused head: only the fc1 input gradient remains
        DenseLayer& D0 = m->dense[0];
        const float* dz1 = (m->dense.size() > 1) ? D0.h : D0.h;
        BCAD_LAUNCH(m, "fc1_dgrad_sgemm", launch_sgemm(dz1, D0.d_w, m->g_flat, n, D0.in, D0.out, false, 1, s));
    } else {
        BCAD_TRY(dense_backward(m, n, class_idx, grad_mode, m->g_flat, s));
    }
    BCAD_LAUNCH(m, "alpha_from_pool_grad", launch_alpha_from_pool_grad(m->g_flat, T.y, m->alpha_part, n, T.Ho, T.Wo, T.Cout, m->cfg.pool_ties,
                                               m->alpha_splits, s, m->target == BCAD_TARGET_CONV_PREACT ? m->cfg.alpha_conv : -1.f));
    BCAD_TRY(tail_chunk(m, T.y, 0, n, heat, heat_stride, s));
    return BCAD_OK;
}

// K = 0: one target per image, class_idx [B] (NULL = the predicted class).  K >= 1 (bcad_predict_explain_classes): class_idx
// [B][K] (NULL = column k is class k), heat [B][K][H][W]
static int run(Model* m, const float* x, int B, const int32_t* class_idx, int grad_mode, bool explain, float* logits,
               float* probs, int32_t* cls, float* heat, cudaStream_t s, int out_h = 0, int out_w = 0, int K = 0);

// cfg.refine_margin: re-run the chunk's small-margin images on the fp32-grade twin and write their results over the 16-bit ones
// (refine.cu).  Stream-ordered: the twin always runs min(cap, n) slots, the device-side count selects what is written back.
// K >= 1: ci holds the chunk's [n][K] class rows (or NULL) and each image has K maps, contiguous (bcad_predict_explain_classes)
static int refine_chunk(Model* m, const float* xc, int n, const int32_t* ci, int grad_mode, bool explain, float* heat, cudaStream_t s,
                        int K = 0) {
    Refine& R = m->refine;
    Model* t = R.twin;
    const int nc = m->cfg.num_classes, slots = std::min(R.cap, n), kc = K ? K : 1;
    const size_t img = (size_t)m->cfg.in_h * m->cfg.in_w * m->cfg.in_c, hm = (size_t)kc * m->heat_h * m->heat_w;
    if (explain && hm > R.heat_elems) {               // first call with larger or more heat-maps (_sized / _classes): grow the twin's buffer
        BCAD_CUDA_CHECK(cudaStreamSynchronize(s));
        BCAD_TRY(m->alloc((void**)&R.heat, (size_t)R.cap * hm * sizeof(float)));
        R.heat_elems = hm;
    }
    if (kc > R.cidx_k) {
        BCAD_CUDA_CHECK(cudaStreamSynchronize(s));
        BCAD_TRY(m->alloc((void**)&R.cidx, (size_t)R.cap * kc * sizeof(int32_t)));
        BCAD_CUDA_CHECK(cudaMemset(R.cidx, 0, (size_t)R.cap * kc * sizeof(int32_t)));
        R.cidx_k = kc;
    }
    BCAD_LAUNCH(m, "refine_flag", launch_refine_flag(m->dense.back().z, n, nc, m->cfg.refine_margin, slots, R.idx, R.counters, s));
    BCAD_LAUNCH(m, "refine_gather", launch_refine_gather(xc, img, ci, R.idx, R.counters, slots, R.x, R.cidx, s, kc));
    BCAD_TRY(m->mark("refine_twin_fp16x3", s));
    const int64_t l0 = t->launches;
    BCAD_TRY(run(t, R.x, slots, ci ? R.cidx : nullptr, grad_mode, explain, nullptr, nullptr, nullptr, explain ? R.heat : nullptr, s, m->heat_h, m->heat_w, K));
    m->launches += t->launches - l0;
    RefineScatter a;
    memset(&a, 0, sizeof(a));
    a.n_dense = (int)m->dense.size();
    for (int j = 0; j < a.n_dense; ++j) {
        a.sizes[j] = m->dense[j].out;
        a.src_z[j] = t->dense[j].z;
        a.dst_z[j] = m->dense[j].z;
    }
    a.src_probs = t->probs; a.dst_probs = m->probs; a.src_cls = t->cls; a.dst_cls = m->cls;
    a.src_heat = explain ? R.heat : nullptr; a.dst_heat = explain ? heat : nullptr;
    a.hm = hm; a.nc = nc;
    BCAD_LAUNCH(m, "refine_scatter", launch_refine_scatter(a, R.idx, R.counters, slots, s));
    return BCAD_OK;
}

static int run(Model* m, const float* x, int B, const int32_t* class_idx, int grad_mode, bool explain, float* logits,
               float* probs, int32_t* cls, float* heat, cudaStream_t s, int out_h, int out_w, int K) {
    BCAD_REQUIRE(m && x, "null model or input");
    BCAD_REQUIRE(out_h >= 0 && out_w >= 0 && out_h <= 16384 && out_w <= 16384 && (out_h == 0) == (out_w == 0), "bad heat-map size %dx%d", out_h, out_w);
    BCAD_REQUIRE(B >= 1, "batch must be >= 1, got %d", B);
    BCAD_REQUIRE(grad_mode == BCAD_GRAD_LOGIT || grad_mode == BCAD_GRAD_SOFTMAX_CE, "bad grad_mode %d", grad_mode);
    BCAD_REQUIRE(!explain || heat, "heatmap output pointer is null");
    BCAD_REQUIRE(!(explain && m->train.drop_B), "explanations are an inference call: clear the dropout masks first");
    if (!m->committed) { set_error("weights not committed: call bcad_commit first"); return BCAD_ERR_STATE; }
    DeviceGuard g(m->cfg.device);
    std::lock_guard<std::mutex> lock(m->mu);
    // the workspace is shared: order this call after the previous one even when it ran on another stream
    BCAD_CUDA_CHECK(cudaStreamWaitEvent(s, m->call_done, 0));
    const int mb = m->cfg.max_batch, nc = m->cfg.num_classes;
    m->heat_h = out_h ? out_h : m->cfg.in_h;
    m->heat_w = out_w ? out_w : m->cfg.in_w;
    const int kc = K ? K : 1;                                       // maps per image
    const size_t img = (size_t)m->cfg.in_h * m->cfg.in_w * m->cfg.in_c, hm = (size_t)m->heat_h * m->heat_w, hk = kc * hm;
    m->prof_n = 0;
    m->multi_class_call = (K > 1);
    for (int b0 = 0; b0 < B; b0 += mb) {
        const int n = std::min(mb, B - b0);
        const float* xc = x + (size_t)b0 * img;
        const int32_t* ci = (explain && class_idx) ? class_idx + (size_t)b0 * kc : nullptr;
        const int32_t* col = ci;                                    // target class column 0 of the chunk
        if (K) {
            // K classes: every image's class row becomes K contiguous columns, so that each backward gets a per-image target vector
            BCAD_LAUNCH(m, "class_columns", launch_class_columns(ci, K, n, m->class_cols, mb, s));
            col = m->class_cols;
        }
        if (m->tensor_path) BCAD_TRY(tensor_forward_chunk(*m, xc, n, explain, col, grad_mode, s));
        else BCAD_TRY(forward_chunk_fp32(m, xc, n, explain, col, grad_mode, s));
        if (explain) {
            float* hc = heat + (size_t)b0 * hk;
            if (m->tensor_path) BCAD_TRY(tensor_explain_chunk(*m, n, col, grad_mode, hc, s, kc, mb, hk));
            else
                for (int k = 0; k < kc; ++k) {
                    const int32_t* ck = col ? col + (size_t)k * mb : nullptr;
                    if (k > 0 && m->fused_head) BCAD_TRY(relaunch_fused_head(m, ck, nullptr, s));     // dz1 of class k
                    BCAD_TRY(explain_chunk_fp32(m, n, ck, grad_mode, hc + (size_t)k * hm, hk, s));
                }
        }
        if (m->refine.twin) BCAD_TRY(refine_chunk(m, xc, n, ci, grad_mode, explain, explain ? heat + (size_t)b0 * hk : nullptr, s, K));
        if (logits) BCAD_CUDA_CHECK(cudaMemcpyAsync(logits + (size_t)b0 * nc, m->dense.back().z, (size_t)n * nc * sizeof(float), cudaMemcpyDeviceToDevice, s));
        if (probs) BCAD_CUDA_CHECK(cudaMemcpyAsync(probs + (size_t)b0 * nc, m->probs, (size_t)n * nc * sizeof(float), cudaMemcpyDeviceToDevice, s));
        if (cls) BCAD_CUDA_CHECK(cudaMemcpyAsync(cls + b0, m->cls, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
        m->cached_B = n;
    }
    if (B > mb) m->cached_B = 0;   // the cache only describes whole calls
    BCAD_TRY(m->mark("end", s));
    BCAD_CUDA_CHECK(cudaEventRecord(m->call_done, s));
    return BCAD_OK;
}

// Saliency of one target class column ck for the chunk's cached forward (explainability.py:44-73): dense backward to the fc1 input
// gradient, the conv blocks from the last to the second with the kernels bcad_train_backward uses, then the first block's input
// gradient with |.| and the per-image min / max.  Image b's map goes to sal + b * stride (d_input: + b * stride * C).
static int saliency_class(Model* m, int n, const int32_t* ck, int grad_mode, float* sal, float* d_input, size_t stride, uint32_t* mm,
                          int mm_ld, cudaStream_t s) {
    DenseLayer& D0 = m->dense[0];
    const bool tc_fc1 = m->fast_train && dense_bwd_x3_supported(n, D0.out, D0.in);
    if (!m->fused_head) BCAD_TRY(dense_backward(m, n, ck, grad_mode, tc_fc1 ? nullptr : m->g_flat, s));
    // dz1: left in dense[0].h by the fused head or the dense chain (d_top itself when the output layer is the only dense layer)
    const float* dz1 = (m->fused_head || m->dense.size() > 1) ? D0.h : m->d_top;
    if (tc_fc1) {
        DenseBwdArgs dg;
        dg.dz = dz1; dg.src = D0.d_w; dg.out = m->g_flat; dg.B = n; dg.units = D0.out; dg.flat = D0.in;
        BCAD_LAUNCH(m, "dense_dgrad_tcgen05_x3", launch_dense_bwd_x3(dg, 1, m->sms, s));
    } else if (m->fused_head) {
        BCAD_LAUNCH(m, "fc1_dgrad_sgemm", launch_sgemm(dz1, D0.d_w, m->g_flat, n, D0.in, D0.out, false, 1, s));
    }
    const float* gp = m->g_flat;
    for (int i = (int)m->conv.size() - 1; i >= 1; --i) {
        const bool tc = m->fast_train && tc_train_eligible(m, (size_t)i);
        BCAD_TRY(conv_block_dz(m, i, gp, n, tc, nullptr, true, s));
        BCAD_TRY(conv_block_dgrad(m, i, n, nullptr, tc, "conv_fp32", s));
        gp = m->conv[i - 1].gp;
    }
    ConvLayer& L = m->conv[0];
    const int hw = L.H * L.W;
    if (saliency_conv0_supported(L.Cin, L.Cout, L.CoutPad, L.k, m->cfg.pad)) {
        BCAD_LAUNCH(m, "saliency_conv0", launch_saliency_conv0(gp, L.y, L.d_w, n, L.H, L.W, L.Ho, L.Wo, m->cfg.pad,
                                                             m->cfg.pool_ties == BCAD_TIES_FIRST ? 1 : 0, m->cfg.alpha_conv, d_input, sal,
                                                             stride, mm, mm_ld, s));
        return BCAD_OK;
    }
    if (m->sal_din == nullptr) BCAD_TRY(m->alloc((void**)&m->sal_din, (size_t)m->cfg.max_batch * hw * L.Cin * sizeof(float)));
    BCAD_TRY(conv_block_dz(m, 0, gp, n, false, nullptr, true, s));
    BCAD_TRY(conv_block_dgrad(m, 0, n, m->sal_din, false, "conv_fp32", s));
    BCAD_LAUNCH(m, "saliency_absmax", launch_saliency_absmax(m->sal_din, n, hw, L.Cin, d_input, sal, stride, mm, mm_ld, s));
    return BCAD_OK;
}

static int run_saliency(Model* m, const float* x, int B, int K, const int32_t* classes, int grad_mode, float* logits, float* probs,
                        int32_t* cls, float* saliency, float* d_input, cudaStream_t s) {
    BCAD_REQUIRE(m && x, "predict_saliency_classes: null model or input");
    if (m->tensor_path) {
        set_error("predict_saliency_classes runs on the fp32 path (the 16-bit forward keeps no first-block output): create the model with BCAD_PREC_FP32");
        return BCAD_ERR_INVALID;
    }
    BCAD_REQUIRE(m->cfg.keep_all_activations, "predict_saliency_classes needs every conv block's output: create the model with keep_all_activations=1");
    BCAD_REQUIRE(!m->train.drop_B, "predict_saliency_classes is an inference call: clear the dropout masks first (bcad_set_dropout_masks(m, NULL, 0))");
    BCAD_REQUIRE(K >= 1 && K <= BCAD_MAX_EXPLAIN_CLASSES, "predict_saliency_classes: K=%d out of range 1..%d", K, BCAD_MAX_EXPLAIN_CLASSES);
    BCAD_REQUIRE(classes || K <= m->cfg.num_classes, "predict_saliency_classes: classes=NULL explains classes 0..K-1, but K=%d > num_classes=%d",
                 K, m->cfg.num_classes);
    BCAD_REQUIRE(saliency, "predict_saliency_classes: saliency output pointer is null");
    BCAD_REQUIRE(B >= 1, "batch must be >= 1, got %d", B);
    BCAD_REQUIRE(grad_mode == BCAD_GRAD_LOGIT || grad_mode == BCAD_GRAD_SOFTMAX_CE, "bad grad_mode %d", grad_mode);
    if (!m->committed) { set_error("weights not committed: call bcad_commit first"); return BCAD_ERR_STATE; }
    DeviceGuard g(m->cfg.device);
    std::lock_guard<std::mutex> lock(m->mu);
    BCAD_CUDA_CHECK(cudaStreamWaitEvent(s, m->call_done, 0));
    if (m->sal_mm == nullptr) BCAD_TRY(m->alloc((void**)&m->sal_mm, (size_t)m->cfg.max_batch * BCAD_MAX_EXPLAIN_CLASSES * 2 * sizeof(uint32_t)));
    const int mb = m->cfg.max_batch, nc = m->cfg.num_classes;
    const size_t hw = (size_t)m->cfg.in_h * m->cfg.in_w, img = hw * m->cfg.in_c;
    m->prof_n = 0;
    m->multi_class_call = false;
    for (int b0 = 0; b0 < B; b0 += mb) {
        const int n = std::min(mb, B - b0);
        BCAD_LAUNCH(m, "class_columns", launch_class_columns(classes ? classes + (size_t)b0 * K : nullptr, K, n, m->class_cols, mb, s));
        BCAD_TRY(forward_chunk_fp32(m, x + (size_t)b0 * img, n, true, m->class_cols, grad_mode, s));
        BCAD_CUDA_CHECK(cudaMemsetAsync(m->sal_mm, 0, (size_t)n * K * 2 * sizeof(uint32_t), s));
        float* sc = saliency + (size_t)b0 * K * hw;
        for (int k = 0; k < K; ++k) {
            const int32_t* ck = m->class_cols + (size_t)k * mb;
            if (k > 0 && m->fused_head) BCAD_TRY(relaunch_fused_head(m, ck, nullptr, s));     // dz1 of class k
            BCAD_TRY(saliency_class(m, n, ck, grad_mode, sc + (size_t)k * hw, d_input ? d_input + ((size_t)b0 * K + k) * img : nullptr,
                                    (size_t)K * hw, m->sal_mm + 2 * k, 2 * K, s));
        }
        BCAD_LAUNCH(m, "saliency_norm", launch_saliency_norm(sc, n * K, (int)hw, m->sal_mm, s));
        if (logits) BCAD_CUDA_CHECK(cudaMemcpyAsync(logits + (size_t)b0 * nc, m->dense.back().z, (size_t)n * nc * sizeof(float), cudaMemcpyDeviceToDevice, s));
        if (probs) BCAD_CUDA_CHECK(cudaMemcpyAsync(probs + (size_t)b0 * nc, m->probs, (size_t)n * nc * sizeof(float), cudaMemcpyDeviceToDevice, s));
        if (cls) BCAD_CUDA_CHECK(cudaMemcpyAsync(cls + b0, m->cls, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
        m->cached_B = n;
    }
    if (B > mb) m->cached_B = 0;   // the cache only describes whole calls
    BCAD_TRY(m->mark("end", s));
    BCAD_CUDA_CHECK(cudaEventRecord(m->call_done, s));
    return BCAD_OK;
}

// -----------------------------------------------------------------------------------------------------
// host-buffer calls: H2D / compute / D2H in chunks on three streams, double-buffered
// -----------------------------------------------------------------------------------------------------
// streams, events and the model-size slot buffers of the pipeline, on first use (caller holds m->mu)
static int xfer_init(Model* m) {
    Xfer& X = m->xfer;
    if (X.inited) return BCAD_OK;
    const size_t img = (size_t)m->cfg.in_h * m->cfg.in_w * m->cfg.in_c, hm = (size_t)m->cfg.in_h * m->cfg.in_w;
    int chunk = std::min(m->cfg.max_batch, 128);
    if (const char* e = getenv("BCAD_HOST_CHUNK")) chunk = std::max(1, std::min(m->cfg.max_batch, atoi(e)));
    BCAD_CUDA_CHECK(cudaStreamCreateWithFlags(&X.s_in, cudaStreamNonBlocking));
    BCAD_CUDA_CHECK(cudaStreamCreateWithFlags(&X.s_compute, cudaStreamNonBlocking));
    BCAD_CUDA_CHECK(cudaStreamCreateWithFlags(&X.s_out, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
        BCAD_CUDA_CHECK(cudaEventCreateWithFlags(&X.in_done[i], cudaEventDisableTiming));
        BCAD_CUDA_CHECK(cudaEventCreateWithFlags(&X.compute_done[i], cudaEventDisableTiming));
        BCAD_CUDA_CHECK(cudaEventCreateWithFlags(&X.out_done[i], cudaEventDisableTiming));
        BCAD_TRY(m->alloc((void**)&X.x[i], (size_t)chunk * img * sizeof(float)));
        BCAD_TRY(m->alloc((void**)&X.heat[i], (size_t)chunk * hm * sizeof(float)));
        BCAD_TRY(m->alloc((void**)&X.cidx[i], (size_t)chunk * sizeof(int32_t)));
    }
    X.chunk = chunk;
    X.inited = true;
    return BCAD_OK;
}

// Images per chunk of a host-buffer call (after xfer_init): small enough that the PCIe pipeline fills quickly (the link, ~52 GB/s per
// direction, is the end-to-end bound), large enough to keep the kernels efficient -- a quarter of the batch, 32 .. cap images.  cap is
// 64 for float32 images (the link is the bound: at 512 images 3.6-3.7 ms with 64, 3.7-3.8 with 128) and 128 for 8-bit images (compute
// is the bound: 2.11 ms with 64, 1.73 ms with 128, 1.80 ms with 256).  BCAD_HOST_CHUNK overrides (tuning).
// Uniform chunks: measured at 512 images, 64-image chunks 3.62 ms, ramped (C/4, C/2, C, ..., C/2, C/4) 3.93 ms.
static int host_chunk(const Model* m, int B, int cap) {
    const int chunk = m->xfer.chunk;
    if (const char* e = getenv("BCAD_HOST_CHUNK")) return std::max(1, std::min(chunk, atoi(e)));
    return std::min(std::min(chunk, cap), std::max(32, ((B + 3) / 4 + 31) / 32 * 32));
}

// The checks every host-buffer call makes before any copy.  K = 0: class_idx [B] of the single-class calls; K >= 1: classes [B][K] of
// the classes calls (NULL: the default targets).  fn names the call in the messages.
static int check_host(const char* fn, Model* m, const void* image, int B, int grad_mode, const int32_t* classes, int K) {
    BCAD_REQUIRE(m && image, "%s: null model or image pointer", fn);
    BCAD_REQUIRE(B >= 1, "batch must be >= 1, got %d", B);
    if (!m->committed) { set_error("weights not committed: call bcad_commit first"); return BCAD_ERR_STATE; }
    BCAD_REQUIRE(grad_mode == BCAD_GRAD_LOGIT || grad_mode == BCAD_GRAD_SOFTMAX_CE, "bad grad_mode %d", grad_mode);
    const int nc = m->cfg.num_classes, kc = K ? K : 1;
    if (classes != nullptr)
        for (size_t i = 0; i < (size_t)B * kc; ++i)
            if (classes[i] < 0 || classes[i] >= nc) {
                if (K) set_error("classes[%zu][%zu] = %d is outside [0, %d)", i / K, i % K, classes[i], nc);
                else set_error("class_idx[%zu] = %d is outside [0, %d)", i, classes[i], nc);
                return BCAD_ERR_INVALID;
            }
    return BCAD_OK;
}

// small outputs (logits, probabilities, classes) go through pinned staging sized for the whole call (caller holds m->host_mu)
static int stage_small(Model* m, size_t bytes) {
    Xfer& X = m->xfer;
    if (X.h_small_bytes < bytes) {
        if (X.h_small) cudaFreeHost(X.h_small);
        X.h_small = nullptr;
        X.h_small_bytes = 0;
        BCAD_CUDA_CHECK(cudaMallocHost(&X.h_small, bytes));
        X.h_small_bytes = bytes;
    }
    if (X.d_small_bytes < bytes) {
        std::lock_guard<std::mutex> lock(m->mu);             // grows only when a call is larger than every call before it; the handle
        X.d_small = nullptr;                                 // owns (and frees at destroy) the smaller ones it replaces: tens of bytes per image
        X.d_small_bytes = 0;
        BCAD_TRY(m->alloc(&X.d_small, bytes));
        X.d_small_bytes = bytes;
    }
    return BCAD_OK;
}

// logits / probabilities / classes of a whole host-buffer call: written on the device per chunk, brought back by one copy behind the
// last chunk through the pinned staging of stage_small
struct SmallOutputs {
    size_t bytes = 0;
    float *dv_logits = nullptr, *dv_probs = nullptr;
    int32_t* dv_cls = nullptr;
};

static int small_outputs(Model* m, int B, SmallOutputs& o) {
    const int nc = m->cfg.num_classes;
    o.bytes = ((size_t)(2 * nc) * sizeof(float) + sizeof(int32_t)) * B;
    BCAD_TRY(stage_small(m, o.bytes));
    o.dv_logits = reinterpret_cast<float*>(m->xfer.d_small);
    o.dv_probs = o.dv_logits + (size_t)B * nc;
    o.dv_cls = reinterpret_cast<int32_t*>(o.dv_probs + (size_t)B * nc);
    return BCAD_OK;
}

static void copy_small_outputs(Model* m, int B, float* logits_host, float* probs_host, int32_t* cls_host) {
    const int nc = m->cfg.num_classes;
    const float* st_logits = reinterpret_cast<const float*>(m->xfer.h_small);
    const float* st_probs = st_logits + (size_t)B * nc;
    const int32_t* st_cls = reinterpret_cast<const int32_t*>(st_probs + (size_t)B * nc);
    if (logits_host) memcpy(logits_host, st_logits, (size_t)B * nc * sizeof(float));
    if (probs_host) memcpy(probs_host, st_probs, (size_t)B * nc * sizeof(float));
    if (cls_host) memcpy(cls_host, st_cls, (size_t)B * sizeof(int32_t));
}

// The chunk loop of every host-buffer call: per chunk c (slot c & 1, images b0 .. b0 + n) h2d(slot, b0, n) on s_in, compute(slot, b0, n)
// on s_compute, d2h(slot, b0, n) on s_out, ordered by the slot's events; the steady state runs H2D, compute and D2H of three chunks
// concurrently.  The small outputs follow the last chunk's D2H.  Returns after both streams have drained.
template <class H2D, class Compute, class D2H>
static int host_pipeline(Model* m, int B, int C0, const SmallOutputs& so, H2D h2d, Compute compute, D2H d2h) {
    Xfer& X = m->xfer;
    const int nchunks = (B + C0 - 1) / C0;
    for (int c = 0, b0 = 0; c < nchunks; ++c, b0 += C0) {
        const int slot = c & 1, n = std::min(C0, B - b0);
        if (c >= 2) {                                         // slot reuse: its previous D2H (chunk c-2) must have drained
            BCAD_CUDA_CHECK(cudaStreamWaitEvent(X.s_in, X.compute_done[slot], 0));
            BCAD_CUDA_CHECK(cudaStreamWaitEvent(X.s_compute, X.out_done[slot], 0));
        }
        BCAD_TRY(h2d(slot, b0, n));
        BCAD_CUDA_CHECK(cudaEventRecord(X.in_done[slot], X.s_in));
        BCAD_CUDA_CHECK(cudaStreamWaitEvent(X.s_compute, X.in_done[slot], 0));
        const int rc = compute(slot, b0, n);
        if (rc != BCAD_OK) { cudaDeviceSynchronize(); return rc; }
        BCAD_CUDA_CHECK(cudaEventRecord(X.compute_done[slot], X.s_compute));
        BCAD_CUDA_CHECK(cudaStreamWaitEvent(X.s_out, X.compute_done[slot], 0));
        BCAD_TRY(d2h(slot, b0, n));
        if (c + 1 == nchunks) BCAD_CUDA_CHECK(cudaMemcpyAsync(X.h_small, X.d_small, so.bytes, cudaMemcpyDeviceToHost, X.s_out));
        BCAD_CUDA_CHECK(cudaEventRecord(X.out_done[slot], X.s_out));
    }
    BCAD_CUDA_CHECK(cudaStreamSynchronize(X.s_out));
    BCAD_CUDA_CHECK(cudaStreamSynchronize(X.s_compute));
    return BCAD_OK;
}

// The single-class host-buffer calls, one image source: x_host float32 images, x8_host 8-bit pixels (x = u8 / 255 on the device) or
// gray8_host grey images of the model's size (gray_preprocess; overlay_host gets their RGB overlays).  Chunks run in the handle's Xfer
// slots, sized for up to 128 images.
static int predict_explain_host_impl(bcad_model* mm, const float* x_host, const uint8_t* x8_host, int B, const int32_t* class_idx_host,
                                     int grad_mode, float* logits_host, float* probs_host, int32_t* cls_host, float* heat_host,
                                     uint8_t* heat_u8_host, const uint8_t* gray8_host = nullptr, int standardise = 0,
                                     uint8_t* overlay_host = nullptr) {
    Model* m = reinterpret_cast<Model*>(mm);
    const void* image = gray8_host ? (const void*)gray8_host : x8_host ? (const void*)x8_host : (const void*)x_host;
    BCAD_TRY(check_host("predict_explain_host", m, image, B, grad_mode, class_idx_host, 0));
    DeviceGuard g(m->cfg.device);
    // one host-buffer call at a time per handle: the three streams, the double-buffered device slots, the events and the pinned
    // staging are shared (threaded callers -- a Flask app with one model -- queue here; separate handles run concurrently)
    std::lock_guard<std::mutex> host_lock(m->host_mu);
    Xfer& X = m->xfer;
    const int nc = m->cfg.num_classes;
    const size_t img = (size_t)m->cfg.in_h * m->cfg.in_w * m->cfg.in_c, hm = (size_t)m->cfg.in_h * m->cfg.in_w;
    {
        std::lock_guard<std::mutex> lock(m->mu);
        BCAD_TRY(xfer_init(m));
        if (heat_u8_host != nullptr && X.heat8[0] == nullptr)
            for (int i = 0; i < 2; ++i) BCAD_TRY(m->alloc((void**)&X.heat8[i], (size_t)X.chunk * hm));
        if ((x8_host != nullptr || gray8_host != nullptr) && X.x8[0] == nullptr)
            for (int i = 0; i < 2; ++i) BCAD_TRY(m->alloc((void**)&X.x8[i], (size_t)X.chunk * img));
        if (gray8_host != nullptr && X.img01[0] == nullptr)
            for (int i = 0; i < 2; ++i) {
                BCAD_TRY(m->alloc((void**)&X.img01[i], (size_t)X.chunk * hm * sizeof(float)));
                BCAD_TRY(m->alloc((void**)&X.ov8[i], (size_t)X.chunk * hm * 3));
            }
    }
    SmallOutputs so;
    BCAD_TRY(small_outputs(m, B, so));
    const bool want_heat = (heat_host != nullptr || heat_u8_host != nullptr || overlay_host != nullptr);
    BCAD_TRY(host_pipeline(m, B, host_chunk(m, B, (x8_host || gray8_host) ? 128 : 64), so,
        [&](int slot, int b0, int n) {
            if (gray8_host) BCAD_CUDA_CHECK(cudaMemcpyAsync(X.x8[slot], gray8_host + (size_t)b0 * hm, (size_t)n * hm, cudaMemcpyHostToDevice, X.s_in));
            else if (x8_host) BCAD_CUDA_CHECK(cudaMemcpyAsync(X.x8[slot], x8_host + (size_t)b0 * img, (size_t)n * img, cudaMemcpyHostToDevice, X.s_in));
            else BCAD_CUDA_CHECK(cudaMemcpyAsync(X.x[slot], x_host + (size_t)b0 * img, (size_t)n * img * sizeof(float), cudaMemcpyHostToDevice, X.s_in));
            if (class_idx_host)
                BCAD_CUDA_CHECK(cudaMemcpyAsync(X.cidx[slot], class_idx_host + b0, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, X.s_in));
            return BCAD_OK;
        },
        [&](int slot, int b0, int n) {
            int rc = BCAD_OK;
            if (gray8_host) rc = launch_gray_preprocess(X.x8[slot], X.img01[slot], X.x[slot], n, (int)hm, m->cfg.in_c, standardise, X.s_compute);
            else if (x8_host) rc = launch_u8_to_unit(X.x8[slot], X.x[slot], (size_t)n * img, X.s_compute);
            if (rc == BCAD_OK)
                rc = run(m, X.x[slot], n, class_idx_host ? X.cidx[slot] : nullptr, grad_mode, want_heat, so.dv_logits + (size_t)b0 * nc,
                         so.dv_probs + (size_t)b0 * nc, so.dv_cls + b0, X.heat[slot], X.s_compute);
            if (rc == BCAD_OK && overlay_host != nullptr)     // show_cam_on_image + heatmap_uint8 in one pass (GRADCAM.py:67,70)
                rc = launch_overlay(X.img01[slot], X.heat[slot], n, m->cfg.in_h, m->cfg.in_w, X.ov8[slot], heat_u8_host ? X.heat8[slot] : nullptr, X.s_compute);
            else if (rc == BCAD_OK && heat_u8_host != nullptr) rc = launch_heat_to_u8(X.heat[slot], X.heat8[slot], (size_t)n * hm, X.s_compute);
            return rc;
        },
        [&](int slot, int b0, int n) {
            if (heat_host) BCAD_CUDA_CHECK(cudaMemcpyAsync(heat_host + (size_t)b0 * hm, X.heat[slot], (size_t)n * hm * sizeof(float), cudaMemcpyDeviceToHost, X.s_out));
            if (heat_u8_host) BCAD_CUDA_CHECK(cudaMemcpyAsync(heat_u8_host + (size_t)b0 * hm, X.heat8[slot], (size_t)n * hm, cudaMemcpyDeviceToHost, X.s_out));
            if (overlay_host) BCAD_CUDA_CHECK(cudaMemcpyAsync(overlay_host + (size_t)b0 * hm * 3, X.ov8[slot], (size_t)n * hm * 3, cudaMemcpyDeviceToHost, X.s_out));
            return BCAD_OK;
        }));
    copy_small_outputs(m, B, logits_host, probs_host, cls_host);
    return BCAD_OK;
}

// Staging bound of the host-buffer classes calls (bcad_gradcam_overlays_classes_host, bcad_saliency_overlays_classes_host): both slots'
// 8-bit images, classes and maps stay within this many bytes of the handle's memory (the chunk shrinks to fit; a single image larger
// than half of it still runs, one image per chunk).  Grad-CAM, 512 x 512 images with K = 2: 4.25 MB per image and slot, chunks of up
// to 60 images.
static const size_t kClassesStagingBytes = (size_t)512 << 20;

static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// The checks of the classes calls on top of check_host, all made before any copy.  fn names the call in the messages.
static int check_classes_host(const char* fn, Model* m, const uint8_t* gray_u8_host, int B, int img_h, int img_w, int K,
                              const int32_t* classes_host_or_null, int grad_mode, int standardise, bool any_output) {
    BCAD_REQUIRE(any_output, "%s: the output pointers are all null", fn);
    BCAD_REQUIRE(img_h >= 1 && img_w >= 1 && img_h <= 16384 && img_w <= 16384, "%s: bad image size %dx%d", fn, img_h, img_w);
    BCAD_REQUIRE(K >= 1 && K <= BCAD_MAX_EXPLAIN_CLASSES, "%s: K=%d out of range 1..%d", fn, K, BCAD_MAX_EXPLAIN_CLASSES);
    BCAD_REQUIRE(standardise == 0 || standardise == 1, "%s: standardise must be 0 or 1", fn);
    BCAD_TRY(check_host(fn, m, gray_u8_host, B, grad_mode, classes_host_or_null, K));
    BCAD_REQUIRE(classes_host_or_null || K <= m->cfg.num_classes, "%s: classes=NULL explains classes 0..K-1, but K=%d > num_classes=%d",
                 fn, K, m->cfg.num_classes);
    return BCAD_OK;
}

// Chunk size of a classes call and the arena holding both slots of per_img_slot bytes per image (caller holds m->host_mu): host_chunk
// with the 8-bit cap, shrunk to the staging bound.  Slot i starts at arena + i * C0 * per_img_slot.
static int classes_staging(Model* m, int B, size_t per_img_slot, int& C0, uint8_t*& arena) {
    Xfer& X = m->xfer;
    std::lock_guard<std::mutex> lock(m->mu);
    BCAD_TRY(xfer_init(m));
    C0 = (int)std::max<size_t>(1, std::min<size_t>((size_t)host_chunk(m, B, 128), kClassesStagingBytes / (2 * per_img_slot)));
    const size_t need = 2 * (size_t)C0 * per_img_slot;
    if (X.cls_arena_bytes < need) {
        if (X.cls_arena != nullptr) {                     // replaced, not kept until destroy: it can be hundreds of MB
            BCAD_CUDA_CHECK(cudaFree(X.cls_arena));       // (synchronises the device: no earlier call still reads it)
            m->allocs.erase(std::find(m->allocs.begin(), m->allocs.end(), X.cls_arena));
            m->ws_bytes -= X.cls_arena_bytes;
            X.cls_arena = nullptr;
            X.cls_arena_bytes = 0;
        }
        BCAD_TRY(m->alloc(&X.cls_arena, need));
        X.cls_arena_bytes = need;
    }
    arena = reinterpret_cast<uint8_t*>(X.cls_arena);
    return BCAD_OK;
}

}  // namespace bcad

extern "C" {

int bcad_predict(bcad_model* mm, const float* x, int B, float* logits, float* probs, int32_t* cls, void* stream) {
    return run(reinterpret_cast<Model*>(mm), x, B, nullptr, BCAD_GRAD_LOGIT, false, logits, probs, cls, nullptr,
               (cudaStream_t)stream);
}

int bcad_predict_explain(bcad_model* mm, const float* x, int B, const int32_t* class_idx, int grad_mode, float* logits,
                         float* probs, int32_t* cls, float* heat, void* stream) {
    return run(reinterpret_cast<Model*>(mm), x, B, class_idx, grad_mode, true, logits, probs, cls, heat,
               (cudaStream_t)stream);
}

int bcad_predict_explain_sized(bcad_model* mm, const float* x, int B, const int32_t* class_idx, int grad_mode, float* logits,
                               float* probs, int32_t* cls, int out_h, int out_w, float* heat, void* stream) {
    BCAD_REQUIRE(out_h >= 1 && out_w >= 1, "predict_explain_sized: bad heat-map size %dx%d", out_h, out_w);
    return run(reinterpret_cast<Model*>(mm), x, B, class_idx, grad_mode, true, logits, probs, cls, heat, (cudaStream_t)stream, out_h, out_w);
}

int bcad_predict_explain_classes(bcad_model* mm, const float* x, int B, int K, const int32_t* classes, int grad_mode, float* logits,
                                 float* probs, int32_t* cls, int out_h, int out_w, float* heat, void* stream) {
    Model* m = reinterpret_cast<Model*>(mm);
    BCAD_REQUIRE(m, "predict_explain_classes: null model");
    BCAD_REQUIRE(K >= 1 && K <= BCAD_MAX_EXPLAIN_CLASSES, "predict_explain_classes: K=%d out of range 1..%d", K, BCAD_MAX_EXPLAIN_CLASSES);
    BCAD_REQUIRE(classes || K <= m->cfg.num_classes, "predict_explain_classes: classes=NULL explains classes 0..K-1, but K=%d > num_classes=%d",
                 K, m->cfg.num_classes);
    return run(m, x, B, classes, grad_mode, true, logits, probs, cls, heat, (cudaStream_t)stream, out_h, out_w, K);
}

int bcad_predict_saliency_classes(bcad_model* mm, const float* x, int B, int K, const int32_t* classes, int grad_mode, float* logits,
                                  float* probs, int32_t* cls, float* saliency, float* d_input, void* stream) {
    return run_saliency(reinterpret_cast<Model*>(mm), x, B, K, classes, grad_mode, logits, probs, cls, saliency, d_input, (cudaStream_t)stream);
}

int bcad_saliency_overlay(const uint8_t* base, int base_c, const float* saliency, int B, int K, int H, int W, uint8_t* overlay,
                          uint8_t* heat, void* stream) {
    BCAD_REQUIRE(base && saliency, "saliency_overlay: null base image or saliency");
    BCAD_REQUIRE(base_c == 1 || base_c == 3, "saliency_overlay: base_c must be 1 or 3, got %d", base_c);
    BCAD_REQUIRE(B >= 1 && K >= 1 && H >= 1 && W >= 1 && (int64_t)H * W <= 0x7fffffff, "saliency_overlay: bad sizes B=%d K=%d %dx%d", B, K, H, W);
    if (overlay == nullptr && heat == nullptr) return BCAD_OK;
    return launch_saliency_overlay(base, base_c, saliency, B, K, H * W, overlay, heat, (cudaStream_t)stream);
}

int bcad_explain_backward(bcad_model* mm, int B, const int32_t* class_idx, int grad_mode,
                          float* const* conv_act_grads, float* d_input, void* stream) {
    Model* m = reinterpret_cast<Model*>(mm);
    BCAD_REQUIRE(m, "null model");
    cudaStream_t s = (cudaStream_t)stream;
    if (!m->committed || m->cached_B != B) {
        set_error("explain_backward needs the activations of a preceding bcad_predict with the same B=%d (<= max_batch); cached B=%d", B, m->cached_B);
        return BCAD_ERR_STATE;
    }
    if (m->tensor_path) {
        set_error("explain_backward (dense activation gradients / d_input) runs on the fp32 path: create the model with BCAD_PREC_FP32");
        return BCAD_ERR_INVALID;
    }
    BCAD_REQUIRE(grad_mode == BCAD_GRAD_LOGIT || grad_mode == BCAD_GRAD_SOFTMAX_CE, "bad grad_mode %d", grad_mode);
    const int nconv = (int)m->conv.size();
    int lowest = nconv;                                    // lowest conv block whose dA is needed
    if (d_input) lowest = 0;
    else if (conv_act_grads)
        for (int i = 0; i < nconv; ++i)
            if (conv_act_grads[i]) { lowest = i; break; }
    BCAD_REQUIRE(lowest < nconv, "explain_backward: nothing requested");
    for (int i = lowest; i < nconv; ++i)
        if (m->conv[i].y == nullptr) {
            set_error("conv block %d output is not cached: create the model with keep_all_activations=1", i);
            return BCAD_ERR_STATE;
        }
    DeviceGuard g(m->cfg.device);
    std::lock_guard<std::mutex> lock(m->mu);
    BCAD_CUDA_CHECK(cudaStreamWaitEvent(s, m->call_done, 0));
    BCAD_TRY(dense_backward(m, B, class_idx, grad_mode, m->g_flat, s));
    const float* gp = m->g_flat;
    for (int i = nconv - 1; i >= lowest; --i) {
        const bool last = (i == lowest && !d_input);
        BCAD_TRY(conv_block_dz(m, i, gp, B, false, conv_act_grads ? conv_act_grads[i] : nullptr, !last, s));
        if (last) break;
        BCAD_TRY(conv_block_dgrad(m, i, B, i > 0 ? nullptr : d_input, false, "conv_fp32", s));
        gp = i > 0 ? m->conv[i - 1].gp : d_input;
    }
    BCAD_CUDA_CHECK(cudaEventRecord(m->call_done, s));
    return BCAD_OK;
}

int64_t bcad_tensor_elems(bcad_model* mm, int kind, int index) {
    Model* m = reinterpret_cast<Model*>(mm);
    if (!m) return -1;
    switch (kind) {
        case BCAD_T_CONV_OUT:
            if (index < 0 || index >= (int)m->conv.size()) return -1;
            return (int64_t)m->conv[index].Ho * m->conv[index].Wo * m->conv[index].Cout;
        case BCAD_T_POOL_OUT:
            if (index < 0 || index >= (int)m->conv.size()) return -1;
            return (int64_t)m->conv[index].Hp * m->conv[index].Wp * m->conv[index].Cout;
        case BCAD_T_DENSE_Z:
            if (index < 0 || index >= (int)m->dense.size()) return -1;
            return m->dense[index].out;
        case BCAD_T_ALPHA: return m->conv.back().Cout;
        case BCAD_T_CAM_LOWRES: return (int64_t)m->conv.back().Ho * m->conv.back().Wo;
        default: return -1;
    }
}

int bcad_get_tensor(bcad_model* mm, int kind, int index, int B, float* dst, void* stream) {
    Model* m = reinterpret_cast<Model*>(mm);
    BCAD_REQUIRE(m && dst, "get_tensor: null argument");
    const int64_t per = bcad_tensor_elems(mm, kind, index);
    BCAD_REQUIRE(per > 0, "get_tensor: bad kind/index (%d,%d)", kind, index);
    if (m->cached_B != B || B < 1) {
        set_error("get_tensor: cache holds B=%d images, asked for %d", m->cached_B, B);
        return BCAD_ERR_STATE;
    }
    cudaStream_t s = (cudaStream_t)stream;
    DeviceGuard g(m->cfg.device);
    std::lock_guard<std::mutex> lock(m->mu);
    BCAD_CUDA_CHECK(cudaStreamWaitEvent(s, m->call_done, 0));
    if (m->tensor_path && (kind == BCAD_T_CONV_OUT || kind == BCAD_T_POOL_OUT)) {
        BCAD_TRY(tensor_get_activation(*m, kind, index, B, dst, s));
        return BCAD_OK;
    }
    if ((kind == BCAD_T_ALPHA || kind == BCAD_T_CAM_LOWRES) && m->multi_class_call) {
        set_error("get_tensor: the last call explained several classes (bcad_predict_explain_classes); alpha / the low-resolution cam describe one");
        return BCAD_ERR_STATE;
    }
    const float* src = nullptr;
    switch (kind) {
        case BCAD_T_CONV_OUT: src = m->conv[index].y; break;
        case BCAD_T_POOL_OUT: src = m->conv[index].p; break;
        case BCAD_T_DENSE_Z: src = m->dense[index].z; break;
        case BCAD_T_ALPHA: src = m->alpha; break;
        case BCAD_T_CAM_LOWRES: src = m->cam_lo; break;
    }
    if (src == nullptr) {
        set_error("get_tensor: tensor (%d,%d) is not cached (keep_all_activations=0?)", kind, index);
        return BCAD_ERR_STATE;
    }
    BCAD_CUDA_CHECK(cudaMemcpyAsync(dst, src, (size_t)per * B * sizeof(float), cudaMemcpyDeviceToDevice, s));
    return BCAD_OK;
}

// -----------------------------------------------------------------------------------------------------
// host-buffer calls: chunked over three streams by host_pipeline
// -----------------------------------------------------------------------------------------------------
int bcad_predict_explain_host(bcad_model* mm, const float* x_host, int B, const int32_t* class_idx_host, int grad_mode,
                              float* logits_host, float* probs_host, int32_t* cls_host, float* heat_host) {
    return predict_explain_host_impl(mm, x_host, nullptr, B, class_idx_host, grad_mode, logits_host, probs_host, cls_host, heat_host, nullptr);
}

int bcad_predict_explain_host_u8(bcad_model* mm, const float* x_host, int B, const int32_t* class_idx_host, int grad_mode,
                                 float* logits_host, float* probs_host, int32_t* cls_host, uint8_t* heat_u8_host) {
    BCAD_REQUIRE(heat_u8_host, "predict_explain_host_u8: null heat-map pointer");
    return predict_explain_host_impl(mm, x_host, nullptr, B, class_idx_host, grad_mode, logits_host, probs_host, cls_host, nullptr, heat_u8_host);
}

int bcad_predict_explain_host_u8in(bcad_model* mm, const uint8_t* x_u8_host, int B, const int32_t* class_idx_host, int grad_mode,
                                   float* logits_host, float* probs_host, int32_t* cls_host, float* heat_host, uint8_t* heat_u8_host) {
    BCAD_REQUIRE(x_u8_host, "predict_explain_host_u8in: null image pointer");
    BCAD_REQUIRE(!(heat_host && heat_u8_host), "predict_explain_host_u8in: pass one heat-map pointer (float32 or uint8), not both");
    return predict_explain_host_impl(mm, nullptr, x_u8_host, B, class_idx_host, grad_mode, logits_host, probs_host, cls_host, heat_host, heat_u8_host);
}

int bcad_gradcam_overlays_host(bcad_model* mm, const uint8_t* gray_u8_host, int B, const int32_t* class_idx_host, int grad_mode,
                               int standardise, float* logits_host, float* probs_host, int32_t* cls_host, uint8_t* overlay_rgb_host,
                               uint8_t* heat_u8_host) {
    BCAD_REQUIRE(gray_u8_host && (overlay_rgb_host || heat_u8_host), "gradcam_overlays_host: null image / output pointer");
    BCAD_REQUIRE(standardise == 0 || standardise == 1, "gradcam_overlays_host: standardise must be 0 or 1");
    return predict_explain_host_impl(mm, nullptr, nullptr, B, class_idx_host, grad_mode, logits_host, probs_host, cls_host, nullptr,
                                     heat_u8_host, gray_u8_host, standardise, overlay_rgb_host);
}

int bcad_gradcam_overlays_classes_host(bcad_model* mm, const uint8_t* gray_u8_host, int B, int img_h, int img_w, int K,
                                       const int32_t* classes_host_or_null, int grad_mode, int standardise, float* logits_host,
                                       float* probs_host, int32_t* cls_host, uint8_t* overlay_rgb_host, uint8_t* heat_u8_host) {
    Model* m = reinterpret_cast<Model*>(mm);
    BCAD_TRY(check_classes_host("gradcam_overlays_classes_host", m, gray_u8_host, B, img_h, img_w, K, classes_host_or_null, grad_mode,
                                standardise, overlay_rgb_host || heat_u8_host));
    DeviceGuard g(m->cfg.device);
    std::lock_guard<std::mutex> host_lock(m->host_mu);
    Xfer& X = m->xfer;
    const int nc = m->cfg.num_classes;
    const size_t hw = (size_t)img_h * img_w;
    // per image and slot: 8-bit image, class row, float maps, RGB overlays, u8 heat-maps
    const size_t b_img = align256(hw), b_cls = align256((size_t)K * sizeof(int32_t)), b_heat = align256((size_t)K * hw * sizeof(float));
    const size_t b_ov = overlay_rgb_host ? align256((size_t)K * hw * 3) : 0, b_h8 = heat_u8_host ? align256((size_t)K * hw) : 0;
    const size_t per_img_slot = b_img + b_cls + b_heat + b_ov + b_h8;
    int C0;
    uint8_t* arena;
    BCAD_TRY(classes_staging(m, B, per_img_slot, C0, arena));
    uint8_t *d_img[2], *d_ov[2], *d_h8[2];
    int32_t* d_cls[2];
    float* d_heat[2];
    for (int i = 0; i < 2; ++i) {
        uint8_t* p = arena + (size_t)i * C0 * per_img_slot;
        d_img[i] = p;                                         p += (size_t)C0 * b_img;
        d_cls[i] = reinterpret_cast<int32_t*>(p);             p += (size_t)C0 * b_cls;
        d_heat[i] = reinterpret_cast<float*>(p);              p += (size_t)C0 * b_heat;
        d_ov[i] = overlay_rgb_host ? p : nullptr;             p += (size_t)C0 * b_ov;
        d_h8[i] = heat_u8_host ? p : nullptr;
    }
    SmallOutputs so;
    BCAD_TRY(small_outputs(m, B, so));
    BCAD_TRY(host_pipeline(m, B, C0, so,
        [&](int slot, int b0, int n) {
            BCAD_CUDA_CHECK(cudaMemcpyAsync(d_img[slot], gray_u8_host + (size_t)b0 * hw, (size_t)n * hw, cudaMemcpyHostToDevice, X.s_in));
            if (classes_host_or_null)
                BCAD_CUDA_CHECK(cudaMemcpyAsync(d_cls[slot], classes_host_or_null + (size_t)b0 * K, (size_t)n * K * sizeof(int32_t),
                                                cudaMemcpyHostToDevice, X.s_in));
            return BCAD_OK;
        },
        [&](int slot, int b0, int n) {
            int rc = launch_gray_resize_preprocess(d_img[slot], X.x[slot], n, img_h, img_w, m->cfg.in_h, m->cfg.in_w, m->cfg.in_c, standardise,
                                                   X.s_compute);
            if (rc == BCAD_OK)
                rc = run(m, X.x[slot], n, classes_host_or_null ? d_cls[slot] : nullptr, grad_mode, true, so.dv_logits + (size_t)b0 * nc,
                         so.dv_probs + (size_t)b0 * nc, so.dv_cls + b0, d_heat[slot], X.s_compute, img_h, img_w, K);
            if (rc == BCAD_OK) rc = launch_overlay_classes(d_img[slot], d_heat[slot], n, K, (int)hw, d_ov[slot], d_h8[slot], X.s_compute);
            return rc;
        },
        [&](int slot, int b0, int n) {
            const size_t maps = (size_t)b0 * K * hw, nmaps = (size_t)n * K * hw;
            if (overlay_rgb_host) BCAD_CUDA_CHECK(cudaMemcpyAsync(overlay_rgb_host + maps * 3, d_ov[slot], nmaps * 3, cudaMemcpyDeviceToHost, X.s_out));
            if (heat_u8_host) BCAD_CUDA_CHECK(cudaMemcpyAsync(heat_u8_host + maps, d_h8[slot], nmaps, cudaMemcpyDeviceToHost, X.s_out));
            return BCAD_OK;
        }));
    copy_small_outputs(m, B, logits_host, probs_host, cls_host);
    return BCAD_OK;
}

int bcad_saliency_overlays_classes_host(bcad_model* mm, const uint8_t* gray_u8_host, int B, int img_h, int img_w, int K,
                                        const int32_t* classes_host_or_null, int grad_mode, int standardise, float* logits_host,
                                        float* probs_host, int32_t* cls_host, float* saliency_host, uint8_t* overlay_bgr_host,
                                        uint8_t* heat_bgr_host) {
    Model* m = reinterpret_cast<Model*>(mm);
    BCAD_TRY(check_classes_host("saliency_overlays_classes_host", m, gray_u8_host, B, img_h, img_w, K, classes_host_or_null, grad_mode,
                                standardise, saliency_host || overlay_bgr_host || heat_bgr_host));
    // what run_saliency would refuse, refused before any copy
    BCAD_REQUIRE(!m->tensor_path, "saliency_overlays_classes_host runs on the fp32 path (the 16-bit forward keeps no first-block output): "
                                  "create the model with BCAD_PREC_FP32");
    BCAD_REQUIRE(m->cfg.keep_all_activations, "saliency_overlays_classes_host needs every conv block's output: create the model with "
                                              "keep_all_activations=1");
    BCAD_REQUIRE(!m->train.drop_B, "saliency_overlays_classes_host is an inference call: clear the dropout masks first "
                                   "(bcad_set_dropout_masks(m, NULL, 0))");
    DeviceGuard g(m->cfg.device);
    std::lock_guard<std::mutex> host_lock(m->host_mu);
    Xfer& X = m->xfer;
    const int nc = m->cfg.num_classes, H = m->cfg.in_h, W = m->cfg.in_w;
    const size_t hw = (size_t)img_h * img_w, mhw = (size_t)H * W;
    // per image and slot: 8-bit image, class row, model-size float saliency, BGR overlays, BGR heat-maps
    const size_t b_img = align256(hw), b_cls = align256((size_t)K * sizeof(int32_t)), b_sal = align256((size_t)K * mhw * sizeof(float));
    const size_t b_ov = overlay_bgr_host ? align256((size_t)K * hw * 3) : 0, b_ht = heat_bgr_host ? align256((size_t)K * hw * 3) : 0;
    const size_t per_img_slot = b_img + b_cls + b_sal + b_ov + b_ht;
    int C0;
    uint8_t* arena;
    BCAD_TRY(classes_staging(m, B, per_img_slot, C0, arena));
    uint8_t *d_img[2], *d_ov[2], *d_ht[2];
    int32_t* d_cls[2];
    float* d_sal[2];
    for (int i = 0; i < 2; ++i) {
        uint8_t* p = arena + (size_t)i * C0 * per_img_slot;
        d_img[i] = p;                                         p += (size_t)C0 * b_img;
        d_cls[i] = reinterpret_cast<int32_t*>(p);             p += (size_t)C0 * b_cls;
        d_sal[i] = reinterpret_cast<float*>(p);               p += (size_t)C0 * b_sal;
        d_ov[i] = overlay_bgr_host ? p : nullptr;             p += (size_t)C0 * b_ov;
        d_ht[i] = heat_bgr_host ? p : nullptr;
    }
    SmallOutputs so;
    BCAD_TRY(small_outputs(m, B, so));
    BCAD_TRY(host_pipeline(m, B, C0, so,
        [&](int slot, int b0, int n) {
            BCAD_CUDA_CHECK(cudaMemcpyAsync(d_img[slot], gray_u8_host + (size_t)b0 * hw, (size_t)n * hw, cudaMemcpyHostToDevice, X.s_in));
            if (classes_host_or_null)
                BCAD_CUDA_CHECK(cudaMemcpyAsync(d_cls[slot], classes_host_or_null + (size_t)b0 * K, (size_t)n * K * sizeof(int32_t),
                                                cudaMemcpyHostToDevice, X.s_in));
            return BCAD_OK;
        },
        [&](int slot, int b0, int n) {
            int rc = launch_gray_resize_preprocess(d_img[slot], X.x[slot], n, img_h, img_w, H, W, m->cfg.in_c, standardise, X.s_compute);
            if (rc == BCAD_OK)
                rc = run_saliency(m, X.x[slot], n, K, classes_host_or_null ? d_cls[slot] : nullptr, grad_mode, so.dv_logits + (size_t)b0 * nc,
                                  so.dv_probs + (size_t)b0 * nc, so.dv_cls + b0, d_sal[slot], nullptr, X.s_compute);
            if (rc == BCAD_OK && (overlay_bgr_host || heat_bgr_host))
                rc = launch_saliency_overlay_resized(d_img[slot], d_sal[slot], n, K, H, W, img_h, img_w, d_ov[slot], d_ht[slot], X.s_compute);
            return rc;
        },
        [&](int slot, int b0, int n) {
            const size_t maps = (size_t)b0 * K * hw * 3, bytes = (size_t)n * K * hw * 3;
            if (saliency_host)
                BCAD_CUDA_CHECK(cudaMemcpyAsync(saliency_host + (size_t)b0 * K * mhw, d_sal[slot], (size_t)n * K * mhw * sizeof(float),
                                                cudaMemcpyDeviceToHost, X.s_out));
            if (overlay_bgr_host) BCAD_CUDA_CHECK(cudaMemcpyAsync(overlay_bgr_host + maps, d_ov[slot], bytes, cudaMemcpyDeviceToHost, X.s_out));
            if (heat_bgr_host) BCAD_CUDA_CHECK(cudaMemcpyAsync(heat_bgr_host + maps, d_ht[slot], bytes, cudaMemcpyDeviceToHost, X.s_out));
            return BCAD_OK;
        }));
    copy_small_outputs(m, B, logits_host, probs_host, cls_host);
    return BCAD_OK;
}

// -----------------------------------------------------------------------------------------------------
// stand-alone tail and overlay
// -----------------------------------------------------------------------------------------------------
int bcad_gradcam_tail(const void* A, const void* dA, int B, int K, int h, int w, int H, int W, int dtype, float* out,
                      void* stream) {
    BCAD_REQUIRE(A && dA && out, "gradcam_tail: null argument");
    BCAD_REQUIRE(B >= 1 && K >= 1 && h >= 1 && w >= 1 && H >= 1 && W >= 1, "gradcam_tail: bad sizes");
    BCAD_REQUIRE(dtype == 0 || dtype == 1, "gradcam_tail: dtype must be 0 (fp32) or 1 (bf16)");
    BCAD_REQUIRE(B <= 65535, "gradcam_tail: B %d exceeds 65535 per call", B);
    cudaStream_t s = (cudaStream_t)stream;
    const int asplits = (h * w >= 4096) ? 8 : 1, csplits = cam_splits(h);
    float* scratch = nullptr;
    const size_t n_ap = (size_t)B * asplits * K, n_cam = (size_t)B * h * w, n_mm = (size_t)B * csplits * 2;
    BCAD_CUDA_CHECK(cudaMallocAsync((void**)&scratch, (n_ap + n_cam + n_mm) * sizeof(float), s));
    float* ap = scratch;
    float* cam = scratch + n_ap;
    float* mm = cam + n_cam;
    int rc = launch_alpha_from_dense_grad(dA, dtype, ap, B, h, w, K, asplits, s);
    if (rc == BCAD_OK) rc = launch_cam(A, dtype, ap, asplits, 1.0f / ((float)h * (float)w), nullptr, cam, mm, B, h, w, K, csplits, s);
    if (rc == BCAD_OK) rc = launch_upsample_norm(cam, mm, csplits, out, B, h, w, H, W, s);
    cudaFreeAsync(scratch, s);
    return rc;
}

int bcad_gray_preprocess(const uint8_t* gray_u8, int B, int H, int W, int C, int standardise, float* img01, float* x, void* stream) {
    BCAD_REQUIRE(gray_u8 && img01 && x, "gray_preprocess: null argument");
    BCAD_REQUIRE(B >= 1 && H >= 1 && W >= 1 && C >= 1 && (standardise == 0 || standardise == 1), "gray_preprocess: bad argument");
    return launch_gray_preprocess(gray_u8, img01, x, B, H * W, C, standardise, (cudaStream_t)stream);
}

int bcad_overlay(const float* img01, const float* cam, int B, int H, int W, uint8_t* overlay_rgb, uint8_t* heat_u8,
                 void* stream) {
    BCAD_REQUIRE(img01 && cam, "overlay: null argument");
    BCAD_REQUIRE(B >= 1 && H >= 1 && W >= 1, "overlay: bad sizes");
    return launch_overlay(img01, cam, B, H, W, overlay_rgb, heat_u8, (cudaStream_t)stream);
}

int bcad_gray_resize_preprocess(const uint8_t* gray_u8, int B, int img_h, int img_w, int H, int W, int C, int standardise, float* x,
                                void* stream) {
    BCAD_REQUIRE(gray_u8 && x, "gray_resize_preprocess: null argument");
    BCAD_REQUIRE(B >= 1 && img_h >= 1 && img_w >= 1 && H >= 1 && W >= 1 && C >= 1 && (int64_t)img_h * img_w <= 0x7fffffff &&
                     (int64_t)H * W <= 0x7fffffff, "gray_resize_preprocess: bad sizes B=%d %dx%d -> %dx%dx%d", B, img_h, img_w, H, W, C);
    BCAD_REQUIRE(standardise == 0 || standardise == 1, "gray_resize_preprocess: standardise must be 0 or 1");
    return launch_gray_resize_preprocess(gray_u8, x, B, img_h, img_w, H, W, C, standardise, (cudaStream_t)stream);
}

int bcad_overlay_classes(const uint8_t* gray_u8, const float* cam, int B, int K, int H, int W, uint8_t* overlay_rgb, uint8_t* heat_u8,
                         void* stream) {
    BCAD_REQUIRE(gray_u8 && cam, "overlay_classes: null image or cam");
    BCAD_REQUIRE(overlay_rgb || heat_u8, "overlay_classes: overlay and heat-map pointers are both null");
    BCAD_REQUIRE(K >= 1 && K <= BCAD_MAX_EXPLAIN_CLASSES, "overlay_classes: K=%d out of range 1..%d", K, BCAD_MAX_EXPLAIN_CLASSES);
    BCAD_REQUIRE(B >= 1 && H >= 1 && W >= 1 && (int64_t)H * W <= 0x7fffffff, "overlay_classes: bad sizes B=%d %dx%d", B, H, W);
    return launch_overlay_classes(gray_u8, cam, B, K, H * W, overlay_rgb, heat_u8, (cudaStream_t)stream);
}

int bcad_saliency_overlay_resized(const uint8_t* gray_u8, const float* saliency, int B, int K, int H, int W, int img_h, int img_w,
                                  uint8_t* overlay_bgr, uint8_t* heat_bgr, void* stream) {
    BCAD_REQUIRE(gray_u8 && saliency, "saliency_overlay_resized: null image or saliency");
    BCAD_REQUIRE(K >= 1 && K <= BCAD_MAX_EXPLAIN_CLASSES, "saliency_overlay_resized: K=%d out of range 1..%d", K, BCAD_MAX_EXPLAIN_CLASSES);
    BCAD_REQUIRE(B >= 1 && B <= 65535 && H >= 1 && W >= 1 && (int64_t)H * W <= 0x7fffffff && img_h >= 1 && img_w >= 1 && img_h <= 16384 &&
                     img_w <= 16384, "saliency_overlay_resized: bad sizes B=%d %dx%d -> %dx%d", B, H, W, img_h, img_w);
    if (overlay_bgr == nullptr && heat_bgr == nullptr) return BCAD_OK;
    return launch_saliency_overlay_resized(gray_u8, saliency, B, K, H, W, img_h, img_w, overlay_bgr, heat_bgr, (cudaStream_t)stream);
}

// -----------------------------------------------------------------------------------------------------
// stand-alone conv block / average pool: the tiny U-Net encoder front (Classes/unet.py:13-73)
// -----------------------------------------------------------------------------------------------------
int bcad_conv_block(const float* x, int B, int H, int W, int Cin, const float* kernel_kkcf, const float* bias, int k, int Cout,
                    int pad, float alpha, int padded_output, float* y, float* pooled, void* stream) {
    BCAD_REQUIRE(x && kernel_kkcf && (y || pooled), "conv_block: null argument");
    BCAD_REQUIRE(B >= 1 && H >= 1 && W >= 1 && Cin >= 1 && Cout >= 1 && k >= 1 && k <= 7 && pad >= 0 && pad <= 3, "conv_block: bad sizes");
    cudaStream_t s = (cudaStream_t)stream;
    const int Hv = H + 2 * pad - k + 1, Wv = W + 2 * pad - k + 1;           // true convolution output
    BCAD_REQUIRE(Hv >= 1 && Wv >= 1, "conv_block: kernel larger than the padded input");
    // padded_output reproduces conv2d(...,'same') of Classes/unet.py:19-27: output allocated at the padded input size,
    // the trailing rows/cols (windows skipped by the reference) stay zero
    const int Ho = padded_output ? H + 2 * pad : Hv, Wo = padded_output ? W + 2 * pad : Wv;
    const int CoutPad = cdiv(Cout, 32) * 32;
    float* scratch = nullptr;
    const size_t wn = (size_t)k * k * Cin * CoutPad;
    BCAD_CUDA_CHECK(cudaMallocAsync((void**)&scratch, (wn + CoutPad) * sizeof(float), s));
    int rc = launch_pad_conv_weights(kernel_kkcf, scratch, k * k, Cin, Cout, CoutPad, s);
    if (rc == BCAD_OK) {
        if (bias) rc = launch_pad_conv_weights(bias, scratch + wn, 1, 1, Cout, CoutPad, s);
        else if (cudaMemsetAsync(scratch + wn, 0, CoutPad * sizeof(float), s) != cudaSuccess) rc = BCAD_ERR_CUDA;
    }
    if (rc == BCAD_OK) {
        ConvArgs a;
        a.x = x; a.w = scratch; a.bias = scratch + wn; a.y = y; a.p = pooled;
        a.B = B; a.H = H; a.W = W; a.Cin = Cin; a.Cout = Cout; a.CoutPad = CoutPad; a.ksize = k; a.pad = pad;
        a.Ho = Ho; a.Wo = Wo; a.Hp = Ho / 2; a.Wp = Wo / 2; a.alpha = alpha;
        a.Hv = padded_output ? Hv : 0; a.Wv = padded_output ? Wv : 0;
        rc = launch_conv_fp32(a, s);
    }
    cudaFreeAsync(scratch, s);
    return rc;
}

int bcad_bottleneck_resize(const float* feat_dev, int B, int C, int H, int W, int layout, int out_h, int out_w, float* out_dev, void* stream) {
    BCAD_REQUIRE(feat_dev && out_dev, "bottleneck_resize: null pointer");
    BCAD_REQUIRE(B >= 1 && C >= 1 && H >= 1 && W >= 1 && out_h >= 1 && out_w >= 1, "bottleneck_resize: bad shape");
    BCAD_REQUIRE(layout == 0 || layout == 1, "bottleneck_resize: layout must be 0 (CHW) or 1 (HWC)");
    return launch_bottleneck_resize(feat_dev, out_dev, B, C, H, W, layout == 0 ? 1 : 0, out_h, out_w, (cudaStream_t)stream);
}

int bcad_avg_pool(const float* x, int B, int H, int W, int C, int pool, float* out, void* stream) {
    BCAD_REQUIRE(x && out && B >= 1 && H >= 1 && W >= 1 && C >= 1 && pool >= 1, "avg_pool: bad argument");
    return launch_avg_pool(x, out, B, H, W, C, pool, (cudaStream_t)stream);
}

int bcad_set_explain_target(bcad_model* mm, int target) {
    Model* m = reinterpret_cast<Model*>(mm);
    BCAD_REQUIRE(m, "null model");
    BCAD_REQUIRE(target == BCAD_TARGET_CONV_ACT || target == BCAD_TARGET_CONV_PREACT, "bad explain target %d", target);
    if (target == BCAD_TARGET_CONV_PREACT) {
        BCAD_REQUIRE(m->cfg.alpha_conv > 0.f, "the pre-activation map is recovered from the stored post-LeakyReLU map: needs alpha_conv > 0, "
                                              "on the tensor paths as on the fp32 path");
        if (m->tensor_path) BCAD_TRY(tensor_preact_supported(*m));
    }
    {
        std::lock_guard<std::mutex> lock(m->mu);
        m->target = target;
    }
    // the refinement twin re-runs small-margin images inside this handle's calls: it explains the same target
    if (m->refine.twin) return bcad_set_explain_target(reinterpret_cast<bcad_model*>(m->refine.twin), target);
    return BCAD_OK;
}

int bcad_refine_stats(bcad_model* mm, int64_t* refined, int64_t* overflowed) {
    Model* m = reinterpret_cast<Model*>(mm);
    BCAD_REQUIRE(m && refined && overflowed, "refine_stats: null argument");
    *refined = 0;
    *overflowed = 0;
    if (m->refine.twin == nullptr || m->refine.counters == nullptr) return BCAD_OK;
    DeviceGuard g(m->cfg.device);
    int32_t h[4] = {0, 0, 0, 0};
    BCAD_CUDA_CHECK(cudaDeviceSynchronize());
    BCAD_CUDA_CHECK(cudaMemcpy(h, m->refine.counters, sizeof(h), cudaMemcpyDeviceToHost));
    *refined = h[1];
    *overflowed = h[2];
    return BCAD_OK;
}

int64_t bcad_launch_count(bcad_model* mm) {
    Model* m = reinterpret_cast<Model*>(mm);
    return m ? m->launches : -1;
}

int bcad_uses_tensor_path(bcad_model* mm) {
    Model* m = reinterpret_cast<Model*>(mm);
    return (m && m->tensor_path) ? 1 : 0;
}

int bcad_set_profiling(bcad_model* mm, int on) {
    Model* m = reinterpret_cast<Model*>(mm);
    BCAD_REQUIRE(m, "null model");
    m->profiling = on != 0;
    return BCAD_OK;
}

int bcad_profile_count(bcad_model* mm) {
    Model* m = reinterpret_cast<Model*>(mm);
    return m ? (m->prof_n > 0 ? m->prof_n - 1 : 0) : -1;
}

int bcad_profile_get(bcad_model* mm, int i, char* name_buf, int name_cap, float* ms) {
    Model* m = reinterpret_cast<Model*>(mm);
    BCAD_REQUIRE(m && ms, "null argument");
    BCAD_REQUIRE(i >= 0 && i + 1 < m->prof_n, "profile index %d out of range (%d intervals)", i, m->prof_n - 1);
    DeviceGuard g(m->cfg.device);
    BCAD_CUDA_CHECK(cudaEventSynchronize(m->prof_pool[i + 1]));
    BCAD_CUDA_CHECK(cudaEventElapsedTime(ms, m->prof_pool[i], m->prof_pool[i + 1]));
    if (name_buf && name_cap > 0) {
        strncpy(name_buf, m->prof_names[i], name_cap - 1);
        name_buf[name_cap - 1] = 0;
    }
    return BCAD_OK;
}

}  // extern "C"
