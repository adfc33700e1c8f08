// Orchestration of the 16-bit tcgen05 path (fp16 operands, fp32 accumulation): eligibility, weight packing, per-chunk forward and explain.
//
// Pipeline per chunk of n images (n <= max_batch):
//   conv_first_pool  (CUDA cores, Cin=1)      x fp32 NHWC          -> P1 fp16 C8-planar
//   conv_igemm       (tcgen05)                P1                   -> A (target activations, fp16 C8-planar)
//                                                                     + pooled map as fc1 A-operand tiles
//   fc_splitk        (tcgen05) + fc_reduce    tiles x W1 tiles     -> z1, h1            (fp32)
//   remaining dense layers, head              (small fp32 kernels shared with the fp32 path)
//   explain: top gradient -> dense backward to dz1 -> alpha = dz1 . S / (h w)  with S[u][k] = sum_pixels W1[u][pixel,k]
//            (exact for first-index pooling: the un-pooled gradient of a window sums to the pooled gradient, so the
//             dense gradient map dA never has to exist -- SURVEY P8), cam_c8 -> upsample_norm.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "../../include/bcad.h"
#include "common.cuh"
#include "kernels.h"
#include "model.h"
#include <cuda_fp16.h>

#include "sm100_kernels.h"

namespace bcad {

struct TensorPath {
    int sms = 148;
    float* d_w0 = nullptr;          // first conv weights [9][Cout0] fp32
    float* d_b0 = nullptr;
    uint8_t* d_w0_img = nullptr;    // tensor-core first conv: [4][Cout0][8] fp16 (hi/lo split weights + bias)
    uint8_t* d_w0_plain = nullptr;  // the same without the split (fp16 mode): [2][Cout0][8] fp16 rows [w(9) b_hi b_lo 0..]
    uint8_t* d_w0_union = nullptr;  // fp16 mode, conv_fused2: patch-union image [2 chunks][4 pool classes x Cout0][8] fp16 (K slot r*4+c of the 4x4 patch)
    uint8_t* d_w1_pair = nullptr;   // conv_fused2: second-block weights [dx][Cin/8][dy = 2,1,0][Cout][8] fp16 (adjacent dy taps = N = 128 operands) + bias tile [2][2 x Cout][8]
    bool plain0 = false;            // fp16 mode: plain fp16 operands in the first block too (BCAD_CONV0_SPLIT=1 keeps the split)
    uint8_t* d_w1_img = nullptr;    // igemm weight image (fp16)
    float* d_b1 = nullptr;
    uint8_t* d_fc_w = nullptr;      // fc1 W tiles
    float* d_S = nullptr;           // [units][Cout] fp32: per-channel column sums of fc1 (alpha shortcut)
    __half* p1 = nullptr;    // conv0 pooled, C8 planar
    __half* act = nullptr;   // conv1 output, C8 planar
    uint8_t* fc_a = nullptr;        // pooled conv1 as fc1 A tiles
    float* fc_part = nullptr;
    float* alpha_raw = nullptr;     // [TF_GROUP][B][Cout] = dz1 . S
    int fc_splits = 1, kb_per_split = 1, m_pad = 128;
    bool x3 = false;                // fp16x3: hi/lo split operands everywhere (fp32-grade)
    uint8_t* d_fc_wT = nullptr;     // tie-duplicating mode: fc1 transposed as W tiles of the input-gradient GEMM [col block][k-block][hi|lo][256][128 B]
    uint8_t* dz_tiles = nullptr;    // dz1 as split A tiles [m_pad/128][units/64][hi|lo][128][128 B]
    bool p1_valid = true;           // the last forward wrote the pooled first-block map to HBM (the fused kernel only does with keep_all_activations)
    bool wide = false;              // first block has Cin > 1: nhwc_to_c8 + conv_wide (sm100_wide.cu)
    int cin_pad = 0, kc = 0, groups = 0;
    uint8_t* d_w0_wide = nullptr;   // [G][9*(KC/8)][Cout0][16 B] + bias tile
    __half* x_c8 = nullptr;         // the input converted to C8-planar fp16
};

#define TP_TRY(expr) do { int _rc = (expr); if (_rc != BCAD_OK) return _rc; } while (0)
#define TP_LAUNCH(m, name, expr) do { int _rc = (m).mark(name, s); if (_rc == BCAD_OK) _rc = (expr); if (_rc != BCAD_OK) return _rc; (m).launches += 1; } while (0)

static uint16_t f2h(float f) {                  // round-to-nearest-even fp32 -> fp16 bits (host)
    const __half h = __float2half_rn(f);
    uint16_t q;
    memcpy(&q, &h, 2);
    return q;
}
static float h2f(uint16_t q) {
    __half h;
    memcpy(&h, &q, 2);
    return __half2float(h);
}

int tensor_path_supported(const Model& m) {
    const bcad_config& c = m.cfg;
    BCAD_REQUIRE(m.conv.size() == 2, "precision=F16: the tensor path covers 2 conv blocks (got %zu); use BCAD_PREC_FP32", m.conv.size());
    const ConvLayer& c0 = m.conv[0];
    const ConvLayer& c1 = m.conv[1];
    BCAD_REQUIRE(c0.k == 3 && (c0.Cout == 16 || c0.Cout == 32 || c0.Cout == 64),
                 "precision=F16: first conv block must be 3x3 with 16/32/64 filters (got %d, k=%d)", c0.Cout, c0.k);
    if (c0.Cin > 1) {
        BCAD_REQUIRE(c0.Cout == 32 || c0.Cout == 64, "precision=F16: a multi-channel first conv block needs 32 or 64 filters (got %d)", c0.Cout);
        BCAD_REQUIRE(c0.Cin <= 1024, "precision=F16: first conv block with %d input channels (max 1024)", c0.Cin);
        BCAD_REQUIRE(c.precision != BCAD_PREC_F16X3 || c0.Cin <= 512, "precision=F16X3: first conv block with %d input channels (max 512)", c0.Cin);
    }
    BCAD_REQUIRE(c1.k == 3 && c1.Cout == 64, "precision=F16: second conv block must be 3x3 with 64 filters (got k=%d, %d)", c1.k, c1.Cout);
    BCAD_REQUIRE(c.pad == 0 || c.pad == 1, "precision=F16: pad must be 0 or 1");
    BCAD_REQUIRE(c.alpha_conv <= 1.f, "precision=F16: conv LeakyReLU slope must be <= 1 (max(v, alpha v) form)");
    // tie-duplicating pool rule (the NumPy CNN): the Grad-CAM weights need per-window tie counts, taken from activations that
    // must be fp32-grade (the rule compares for equality) -> only the split-operand mode, with an fp32 tail
    BCAD_REQUIRE(c.pool_ties == BCAD_TIES_FIRST || c.precision == BCAD_PREC_F16X3,
                 "precision=F16: the alpha shortcut needs first-index pooling (TIES_FIRST); the tie-duplicating NumPy flavour runs on "
                 "BCAD_PREC_F16X3 or BCAD_PREC_FP32");
    BCAD_REQUIRE(c.pool_ties == BCAD_TIES_FIRST || m.dense.size() > 1,
                 "precision=F16X3 with the tie-duplicating rule needs at least one hidden dense layer");
    if (c.precision == BCAD_PREC_F16X3)
        BCAD_REQUIRE(c0.Cout == 32, "precision=F16X3: the split-operand path needs 32 first-block filters (got %d)", c0.Cout);
    const int units = m.dense[0].out;
    BCAD_REQUIRE(units % 16 == 0 && units <= 256, "precision=F16: first dense layer must have a multiple of 16 units <= 256 (got %d)", units);
    return BCAD_OK;
}

int tensor_path_commit(Model& m) {
    if (m.tp == nullptr) m.tp = new TensorPath();
    TensorPath& t = *m.tp;
    t.x3 = (m.cfg.precision == BCAD_PREC_F16X3);
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&t.sms, cudaDevAttrMultiProcessorCount, dev);
    const ConvLayer& c0 = m.conv[0];
    const ConvLayer& c1 = m.conv[1];
    DenseLayer& d0 = m.dense[0];
    const int mb = m.cfg.max_batch;
    t.wide = (c0.Cin > 1);
    if (t.wide) {
        // ---- multi-channel first block: per channel group [tap][octet][Cout][8] fp16, then the bias tile
        t.cin_pad = cdiv(c0.Cin, 16) * 16;
        t.kc = conv_wide_group_channels(t.cin_pad, c0.Cout);
        t.groups = t.cin_pad / t.kc;
        const int chunks = t.kc / 8;
        const size_t wg = (size_t)9 * chunks * c0.Cout * 8;                   // halves per group
        // fp16x3: three passes over the channel groups -- inputs [x_hi | x_lo | x_hi] (launch_nhwc_to_c8_x3) against weights
        // [w_hi | w_hi | w_lo]: the plain kernel's fp32 accumulators then hold x_hi.w_hi + x_lo.w_hi + x_hi.w_lo
        const int parts = t.x3 ? 3 : 1;
        std::vector<uint16_t> img(wg * t.groups * parts + (size_t)2 * c0.Cout * 8, 0);
        for (int part = 0; part < parts; ++part)
            for (int g = 0; g < t.groups; ++g)
                for (int tap = 0; tap < 9; ++tap)
                    for (int ch = 0; ch < chunks; ++ch)
                        for (int f = 0; f < c0.Cout; ++f)
                            for (int e = 0; e < 8; ++e) {
                                const int cidx = g * t.kc + ch * 8 + e;
                                if (cidx >= c0.Cin) continue;
                                const float w = c0.h_w[((size_t)f * 9 + tap) * c0.Cin + cidx];
                                const uint16_t q = f2h(w);
                                img[((size_t)part * t.groups + g) * wg + (((size_t)tap * chunks + ch) * c0.Cout + f) * 8 + e] =
                                    (part == 2) ? f2h(w - h2f(q)) : q;
                            }
        for (int f = 0; f < c0.Cout; ++f) {
            const float bhi = h2f(f2h(c0.h_b[f]));
            img[wg * t.groups * parts + (size_t)f * 8 + 0] = f2h(bhi);
            img[wg * t.groups * parts + (size_t)f * 8 + 1] = f2h(c0.h_b[f] - bhi);
        }
        if (!t.d_w0_wide) TP_TRY(m.alloc((void**)&t.d_w0_wide, img.size() * 2));
        BCAD_CUDA_CHECK(cudaMemcpy(t.d_w0_wide, img.data(), img.size() * 2, cudaMemcpyHostToDevice));
        if (!t.x_c8) TP_TRY(m.alloc((void**)&t.x_c8, (size_t)parts * mb * c0.H * c0.W * t.cin_pad * 2));
    }
    // ---- conv0: [9][Cout] fp32
    if (!t.wide) {
        std::vector<float> w((size_t)9 * c0.Cout);
        for (int f = 0; f < c0.Cout; ++f)
            for (int tap = 0; tap < 9; ++tap) w[(size_t)tap * c0.Cout + f] = c0.h_w[(size_t)f * 9 + tap];
        if (!t.d_w0) TP_TRY(m.alloc((void**)&t.d_w0, w.size() * 4));
        if (!t.d_b0) TP_TRY(m.alloc((void**)&t.d_b0, c0.Cout * 4));
        BCAD_CUDA_CHECK(cudaMemcpy(t.d_w0, w.data(), w.size() * 4, cudaMemcpyHostToDevice));
        BCAD_CUDA_CHECK(cudaMemcpy(t.d_b0, c0.h_b.data(), c0.Cout * 4, cudaMemcpyHostToDevice));
    }
    // ---- conv0 tensor-core image: K = 32 slots per filter: [w_hi(9) b_hi | w_hi(9) b_lo | w_lo(9) 0 0 0]
    if (!t.wide && (c0.Cout == 32 || c0.Cout == 64)) {
        std::vector<uint16_t> img((size_t)4 * c0.Cout * 8, 0);
        auto put = [&](int f, int k, float v) { img[((size_t)(k >> 3) * c0.Cout + f) * 8 + (k & 7)] = f2h(v); };
        for (int f = 0; f < c0.Cout; ++f) {
            for (int tap = 0; tap < 9; ++tap) {
                const float w = c0.h_w[(size_t)f * 9 + tap];
                const float whi = h2f(f2h(w));
                put(f, tap, whi);
                put(f, 10 + tap, whi);
                put(f, 20 + tap, w - whi);
            }
            const float bhi = h2f(f2h(c0.h_b[f]));
            put(f, 9, bhi);
            put(f, 19, c0.h_b[f] - bhi);
        }
        if (!t.d_w0_img) TP_TRY(m.alloc((void**)&t.d_w0_img, img.size() * 2));
        BCAD_CUDA_CHECK(cudaMemcpy(t.d_w0_img, img.data(), img.size() * 2, cudaMemcpyHostToDevice));
        // fp16 mode: one K-step of plain fp16 weights; the bias stays an exact hi + lo pair (two slots against two ones)
        std::vector<uint16_t> pl((size_t)2 * c0.Cout * 8, 0);
        auto putp = [&](int f, int k, float v) { pl[((size_t)(k >> 3) * c0.Cout + f) * 8 + (k & 7)] = f2h(v); };
        for (int f = 0; f < c0.Cout; ++f) {
            for (int tap = 0; tap < 9; ++tap) putp(f, tap, c0.h_w[(size_t)f * 9 + tap]);
            const float bhi = h2f(f2h(c0.h_b[f]));
            putp(f, 9, bhi);
            putp(f, 10, c0.h_b[f] - bhi);
        }
        if (!t.d_w0_plain) TP_TRY(m.alloc((void**)&t.d_w0_plain, pl.size() * 2));
        BCAD_CUDA_CHECK(cudaMemcpy(t.d_w0_plain, pl.data(), pl.size() * 2, cudaMemcpyHostToDevice));
        t.plain0 = !t.x3 && getenv("BCAD_CONV0_SPLIT") == nullptr;
        // patch-union form (sm100_fused2.cu): the filter of pool class (qr, qc) sits at offset (qr, qc) inside the 4x4 input patch
        if (c0.Cout == 32) {
            std::vector<uint16_t> un((size_t)2 * 4 * c0.Cout * 8, 0);
            for (int qr = 0; qr < 2; ++qr)
                for (int qc = 0; qc < 2; ++qc)
                    for (int f = 0; f < c0.Cout; ++f)
                        for (int ty = 0; ty < 3; ++ty)
                            for (int tx = 0; tx < 3; ++tx) {
                                const int k = (qr + ty) * 4 + (qc + tx), n = (qr * 2 + qc) * c0.Cout + f;
                                un[((size_t)(k >> 3) * 4 * c0.Cout + n) * 8 + (k & 7)] = f2h(c0.h_w[(size_t)f * 9 + ty * 3 + tx]);
                            }
            if (!t.d_w0_union) TP_TRY(m.alloc((void**)&t.d_w0_union, un.size() * 2));
            BCAD_CUDA_CHECK(cudaMemcpy(t.d_w0_union, un.data(), un.size() * 2, cudaMemcpyHostToDevice));
        }
    }
    // ---- conv1 weight image: [tap*(Cin/8)+chunk][cout][8] fp16
    {
        const int chunks = c1.Cin / 8;
        const int vch = t.x3 ? 2 * chunks : chunks;                          // x3: octets [w_hi(0) w_lo(0) w_hi(1) w_lo(1) ...] per tap
        const size_t wel = (size_t)9 * vch * c1.Cout * 8;
        std::vector<uint16_t> img(wel + (size_t)2 * c1.Cout * 8, 0);         // + bias tile [2 chunks][Cout][8]
        for (int tap = 0; tap < 9; ++tap)
            for (int ch = 0; ch < chunks; ++ch)
                for (int f = 0; f < c1.Cout; ++f)
                    for (int e = 0; e < 8; ++e) {
                        const float w = c1.h_w[((size_t)f * 9 + tap) * c1.Cin + ch * 8 + e];
                        const uint16_t q = f2h(w);
                        if (!t.x3) img[(((size_t)tap * vch + ch) * c1.Cout + f) * 8 + e] = q;
                        else {                                   // halves interleaved per octet: one N = 2*Cout operand block [w_hi(ch) | w_lo(ch)]
                            img[(((size_t)tap * vch + 2 * ch) * c1.Cout + f) * 8 + e] = q;
                            img[(((size_t)tap * vch + 2 * ch + 1) * c1.Cout + f) * 8 + e] = f2h(w - h2f(q));
                        }
                    }
        for (int f = 0; f < c1.Cout; ++f) {                                 // bias K-step rows: {b_hi, b_lo, 0 ...}
            const float bhi = h2f(f2h(c1.h_b[f]));
            img[wel + (size_t)f * 8 + 0] = f2h(bhi);
            img[wel + (size_t)f * 8 + 1] = f2h(c1.h_b[f] - bhi);
        }
        if (!t.d_w1_img) TP_TRY(m.alloc((void**)&t.d_w1_img, img.size() * 2));
        BCAD_CUDA_CHECK(cudaMemcpy(t.d_w1_img, img.data(), img.size() * 2, cudaMemcpyHostToDevice));
        if (!t.x3 && c1.Cin == 32 && c1.Cout == 64) {
            // pair layout for conv_fused2 (sm100_fused2.cu): the three dy taps of a (dx, chunk) are contiguous, highest dy first
            std::vector<uint16_t> pr((size_t)9 * chunks * c1.Cout * 8 + (size_t)2 * 2 * c1.Cout * 8, 0);
            for (int dx = 0; dx < 3; ++dx)
                for (int ch = 0; ch < chunks; ++ch)
                    for (int dy = 0; dy < 3; ++dy)
                        for (int f = 0; f < c1.Cout; ++f)
                            for (int e = 0; e < 8; ++e)
                                pr[((((size_t)dx * chunks + ch) * 3 + (2 - dy)) * c1.Cout + f) * 8 + e] =
                                    f2h(c1.h_w[((size_t)f * 9 + dy * 3 + dx) * c1.Cin + ch * 8 + e]);
            const size_t boff = (size_t)9 * chunks * c1.Cout * 8;
            for (int n = 0; n < 2 * c1.Cout; ++n) {                          // bias rows twice: rows n and n + Cout of an N = 128 operand
                const int f = n % c1.Cout;
                const float bhi = h2f(f2h(c1.h_b[f]));
                pr[boff + (size_t)n * 8 + 0] = f2h(bhi);
                pr[boff + (size_t)n * 8 + 1] = f2h(c1.h_b[f] - bhi);
            }
            if (!t.d_w1_pair) TP_TRY(m.alloc((void**)&t.d_w1_pair, pr.size() * 2));
            BCAD_CUDA_CHECK(cudaMemcpy(t.d_w1_pair, pr.data(), pr.size() * 2, cudaMemcpyHostToDevice));
        }
    }
    // ---- fc1: SW128 tiles [pixel][unit][128 B]; K index inside a tile = channel; S = per-channel column sums
    {
        const int npix = c1.Hp * c1.Wp, N = d0.out, C = c1.Cout;
        const int parts = t.x3 ? 2 : 1;                                      // x3: [pixel][hi|lo][unit][64]
        std::vector<uint16_t> tiles((size_t)npix * parts * N * 64);
        std::vector<double> S((size_t)N * C, 0.0);
        for (int u = 0; u < N; ++u) {
            const float* row = d0.h_w.data() + (size_t)u * d0.in;          // device (NHWC) column order: pixel*C + c
            for (int pp = 0; pp < npix; ++pp) {
                uint16_t* dst = tiles.data() + (((size_t)pp * parts) * N + u) * 64;
                for (int cidx = 0; cidx < C; ++cidx) {
                    const float v = row[(size_t)pp * C + cidx];
                    const int chunk = (cidx >> 3) ^ (u & 7);
                    const uint16_t q = f2h(v);
                    dst[chunk * 8 + (cidx & 7)] = q;
                    if (t.x3) {
                        dst[(size_t)N * 64 + chunk * 8 + (cidx & 7)] = f2h(v - h2f(q));
                        S[(size_t)u * C + cidx] += v;                        // the GEMM sees (almost) the fp32 weight
                    } else {
                        S[(size_t)u * C + cidx] += h2f(q);                   // S uses the fp16-rounded weights the GEMM sees
                    }
                }
            }
        }
        std::vector<float> Sf(S.begin(), S.end());
        if (!t.d_fc_w) TP_TRY(m.alloc((void**)&t.d_fc_w, tiles.size() * 2));
        if (!t.d_S) TP_TRY(m.alloc((void**)&t.d_S, Sf.size() * 4));
        BCAD_CUDA_CHECK(cudaMemcpy(t.d_fc_w, tiles.data(), tiles.size() * 2, cudaMemcpyHostToDevice));
        BCAD_CUDA_CHECK(cudaMemcpy(t.d_S, Sf.data(), Sf.size() * 4, cudaMemcpyHostToDevice));
    }
    // ---- tie-duplicating mode: fc1 transposed, as the W operand of the input-gradient GEMM g = dz1 . W1 on the tensor core
    //      (column block cb = 256 consecutive flat positions, K = units in blocks of 64; split hi/lo like every x3 operand)
    if (m.cfg.pool_ties != BCAD_TIES_FIRST && d0.in % 256 == 0 && d0.out % 64 == 0) {
        const int ncb = (int)(d0.in / 256), nkb = d0.out / 64;
        std::vector<uint16_t> tiles((size_t)ncb * nkb * 2 * 256 * 64);
        for (int cb = 0; cb < ncb; ++cb)
            for (int kb = 0; kb < nkb; ++kb) {
                uint16_t* hi = tiles.data() + (((size_t)cb * nkb + kb) * 2) * (256 * 64);
                uint16_t* lo = hi + 256 * 64;
                for (int c = 0; c < 256; ++c)
                    for (int j = 0; j < 64; ++j) {
                        const float v = d0.h_w[(size_t)(kb * 64 + j) * d0.in + (size_t)cb * 256 + c];
                        const uint16_t q = f2h(v);
                        const int pos = c * 64 + (((j >> 3) ^ (c & 7)) << 3) + (j & 7);
                        hi[pos] = q;
                        lo[pos] = f2h(v - h2f(q));
                    }
            }
        if (!t.d_fc_wT) TP_TRY(m.alloc((void**)&t.d_fc_wT, tiles.size() * 2));
        BCAD_CUDA_CHECK(cudaMemcpy(t.d_fc_wT, tiles.data(), tiles.size() * 2, cudaMemcpyHostToDevice));
        if (!t.dz_tiles) {
            const int m_pad = cdiv(mb, 128) * 128;
            TP_TRY(m.alloc((void**)&t.dz_tiles, (size_t)m_pad * d0.out * 2 * 2));
        }
    }
    // ---- workspace
    if (t.p1 == nullptr) {
        t.m_pad = cdiv(mb, 128) * 128;
        const int npix = c1.Hp * c1.Wp;
        const int m_tiles = t.m_pad / 128;
        int splits = cdiv(t.sms, m_tiles);
        if (splits > npix) splits = npix;
        t.kb_per_split = cdiv(npix, splits);
        t.fc_splits = cdiv(npix, t.kb_per_split);
        const size_t parts = t.x3 ? 2 : 1;
        TP_TRY(m.alloc((void**)&t.p1, parts * mb * c0.Hp * c0.Wp * c0.Cout * 2));
        TP_TRY(m.alloc((void**)&t.act, parts * mb * c1.Ho * c1.Wo * c1.Cout * 2));
        TP_TRY(m.alloc((void**)&t.fc_a, parts * t.m_pad * npix * 128));
        BCAD_CUDA_CHECK(cudaMemset(t.fc_a, 0, parts * t.m_pad * npix * 128));     // padding rows: finite zeros
        TP_TRY(m.alloc((void**)&t.fc_part, (size_t)t.fc_splits * t.m_pad * d0.out * 4));
        TP_TRY(m.alloc((void**)&t.alpha_raw, (size_t)TF_GROUP * mb * c1.Cout * 4));      // one [mb][C] slice per class of a tail group
    }
    return BCAD_OK;
}

void tensor_path_destroy(Model& m) {
    delete m.tp;
    m.tp = nullptr;
}

int tensor_forward_chunk(Model& m, const float* x, int n, bool explain, const int32_t* class_idx, int grad_mode, cudaStream_t s) {
    TensorPath& t = *m.tp;
    const ConvLayer& c0 = m.conv[0];
    const ConvLayer& c1 = m.conv[1];
    // both conv blocks in one persistent kernel when the shape allows (0.52 vs 0.25 + 0.35 ms at 512 x 256x256x1);
    // BCAD_TWO_CONV_KERNELS=1 forces the two-kernel path (profiling comparisons)
    // The choice is a property of the HANDLE (max_batch), not of the call, so that chunked == un-chunked and host call == device
    // call stay bit-identical: handles sized for fewer work items than SMs keep the two kernels, where the first block spreads
    // better on its own (0.216 vs 0.244 ms for a single image end to end).
    const int fuse_bands = cdiv(c1.Ho, c1.Ho < 64 ? cdiv(c1.Ho, 2) * 2 : 64);
    const bool fuse = !t.wide && t.d_w0_img != nullptr && conv_fused_supported(c0.Cin, c0.Cout, c1.Cout, c1.W, c1.Wo, t.x3) &&
                      (m.cfg.max_batch * fuse_bands >= t.sms || getenv("BCAD_FUSED_CONV") != nullptr) && getenv("BCAD_TWO_CONV_KERNELS") == nullptr;
    if (fuse) {
        FusedArgs f;
        f.x = x; f.w0_img = t.plain0 ? t.d_w0_plain : t.d_w0_img; f.plain0 = t.plain0 ? 1 : 0; f.w1_img = t.d_w1_img; f.act = t.act; f.pool_fc = t.fc_a;
        f.p1_out = m.cfg.keep_all_activations ? t.p1 : nullptr;          // the pooled first-block map normally never leaves the SM
        t.p1_valid = (f.p1_out != nullptr);
        f.B = n; f.H = c0.H; f.W = c0.W; f.H1 = c1.H; f.W1 = c1.W; f.Ho = c1.Ho; f.Wo = c1.Wo; f.Hp = c1.Hp; f.Wp = c1.Wp;
        f.pad = m.cfg.pad;
        f.band_rows = 64;
        if (f.band_rows > c1.Ho) f.band_rows = cdiv(c1.Ho, 2) * 2;
        f.bands = cdiv(c1.Ho, f.band_rows);
        f.alpha = m.cfg.alpha_conv;
        f.debug = 0;
        if (const char* dbg = getenv("BCAD_DEBUG_SKIP_STORES")) {      // timing experiments only (results are garbage)
            f.debug = atoi(dbg);
            if (f.debug & 1) f.act = nullptr;
            if (f.debug & 2) f.pool_fc = nullptr;
        }
        // second-generation kernel (patch-union first block, TMA input boxes) where its extra conditions hold; BCAD_FUSED_V1=1 keeps the first
        if (t.plain0 && t.d_w0_union != nullptr && t.d_w1_pair != nullptr && getenv("BCAD_FUSED_V1") == nullptr && conv_fused2_supported(x, c0.H, c0.W)) {
            f.w0_img = t.d_w0_union;
            f.w1_img = t.d_w1_pair;
            f.b0 = t.d_b0;
            f.xoff = (4 - m.cfg.pad % 4) % 4;                       // box start column -pad - xoff = a multiple of 4 floats
            // paired taps (N = 128 MMAs, 25 instead of 38 per row pair): 17 % faster second block on its own (0.233 vs 0.281 ms), but the whole
            // kernel is then bound by the teams / epilogue and, power-capped, measured 3 % SLOWER under sustained load (0.485 vs 0.469 ms,
            // profiles/r02_fused2_variants.md): opt-in
            if (getenv("BCAD_F2_PAIRED") == nullptr) f.debug |= 1024;
            if (getenv("BCAD_F2_NOSLEEP") == nullptr) f.debug |= 2048;      // loader warp backs off 64 ns between polling rounds (0.444-0.465 vs 0.469-0.470 ms sustained)
            if (const char* e = getenv("BCAD_F2_XOFF")) f.xoff = atoi(e);
            TP_LAUNCH(m, "conv01_fused_tcgen05", launch_conv_fused2(f, t.sms, s));
        } else
        TP_LAUNCH(m, "conv01_fused_tcgen05", launch_conv_fused(f, t.sms, s));
    } else {
    t.p1_valid = true;
    if (t.wide) {
        if (t.x3) TP_LAUNCH(m, "input_to_c8_hi_lo", launch_nhwc_to_c8_x3(x, t.x_c8, n, c0.H, c0.W, c0.Cin, t.cin_pad, s));
        else TP_LAUNCH(m, "input_to_c8", launch_nhwc_to_c8(x, t.x_c8, n, c0.H, c0.W, c0.Cin, t.cin_pad, s));
        const int parts = t.x3 ? 3 : 1;
        WideArgs w;
        w.in = t.x_c8; w.w_img = t.d_w0_wide; w.pool_c8 = t.p1;
        w.B = n; w.H = c0.H; w.W = c0.W; w.Ho = c0.Ho; w.Wo = c0.Wo; w.Hp = c0.Hp; w.Wp = c0.Wp; w.pad = m.cfg.pad;
        w.G = parts * t.groups; w.ybands = cdiv(c0.Ho, conv_wide_rows_per_band(c0.Cout)); w.xsegs = cdiv(c0.Wo, 128);
        w.alpha = m.cfg.alpha_conv;
        w.split_out = t.x3 ? 1 : 0;
        TP_LAUNCH(m, "conv0_wide_tcgen05", launch_conv_wide(w, parts * t.cin_pad, c0.Cout, t.sms, s));
    } else if (t.d_w0_img != nullptr && (t.x3 || getenv("BCAD_CONV0_CUDA_CORES") == nullptr))
        TP_LAUNCH(m, "conv0_first_tcgen05", launch_conv_first_tc(x, t.plain0 ? t.d_w0_plain : t.d_w0_img, t.p1, n, c0.H, c0.W, m.cfg.pad, c0.Cout, m.cfg.alpha_conv, t.x3, t.plain0, t.sms, s, m.n_dev));
    else
        TP_LAUNCH(m, "conv0_first_pool", launch_conv_first_pool(x, t.d_w0, t.d_b0, t.p1, n, c0.H, c0.W, m.cfg.pad, c0.Cout, m.cfg.alpha_conv, s));
    IgemmArgs a;
    a.in = t.p1; a.w_img = t.d_w1_img; a.act = t.act; a.pool_fc = t.fc_a; a.pool_c8 = nullptr;
    a.B = n; a.H = c1.H; a.W = c1.W; a.Ho = c1.Ho; a.Wo = c1.Wo; a.Hp = c1.Hp; a.Wp = c1.Wp; a.pad = m.cfg.pad;
    a.xsegs = cdiv(c1.Wo, 128);
    // rows per work item: 64 for big calls (2 halo rows per 64), fewer when the call would otherwise leave SMs idle (a single
    // image is 2 items at 64 rows, 64 items at 2) -- the banding does not change any result
    a.band_rows = 64;
    while (a.band_rows > 2 && (long long)n * cdiv(c1.Ho, a.band_rows) * a.xsegs < t.sms) a.band_rows -= 2;
    if (m.n_dev != nullptr && a.band_rows > 4) a.band_rows = 4;     // refinement twin: usually 1-3 of its slots are live -- spread each image
    if (a.band_rows > c1.Ho) a.band_rows = cdiv(c1.Ho, 2) * 2;
    a.bands = cdiv(c1.Ho, a.band_rows);
    a.alpha = m.cfg.alpha_conv;
    a.n_dev = m.n_dev;
    a.debug = 0;
    if (const char* dbg = getenv("BCAD_DEBUG_SKIP_STORES")) {      // timing experiments only (results are garbage)
        a.debug = atoi(dbg);
        if (a.debug & 1) a.act = nullptr;
        if (a.debug & 2) a.pool_fc = nullptr;
    }
    TP_LAUNCH(m, "conv1_igemm_tcgen05", launch_conv_igemm(a, t.x3 ? 2 * c1.Cin : c1.Cin, c1.Cout, t.x3, t.sms, s));
    }
    // fc1
    DenseLayer& d0 = m.dense[0];
    FcArgs f;
    f.a_tiles = t.fc_a; f.w_tiles = t.d_fc_w; f.partials = t.fc_part;
    f.N = d0.out; f.nkb = c1.Hp * c1.Wp; f.kb_per_split = t.kb_per_split; f.splits = t.fc_splits;
    f.m_tiles = cdiv(n, 128); f.m_pad = t.m_pad; f.x3 = t.x3 ? 1 : 0; f.ncb = 1; f.ld_out = 0; f.m_valid = 0; f.n_dev = m.n_dev;
    TP_LAUNCH(m, "fc1_splitk_tcgen05", launch_fc_splitk(f, s));
    if (m.fused_head) {
        // reduce + dense tail + class + (explain) backward to dz1 + alpha shortcut, one launch
        if (m.cfg.pool_ties != BCAD_TIES_FIRST)              // dz1 stays in dense[0].h for the fp32 tail; no alpha shortcut
            return launch_fused_head(&m, n, t.fc_part, t.fc_splits, (size_t)t.m_pad * d0.out, explain, class_idx, grad_mode,
                                     explain ? d0.h : nullptr, nullptr, 0, nullptr, s);
        return launch_fused_head(&m, n, t.fc_part, t.fc_splits, (size_t)t.m_pad * d0.out, explain, class_idx, grad_mode,
                                 nullptr, t.d_S, c1.Cout, t.alpha_raw, s);
    }
    const bool only = (m.dense.size() == 1);
    TP_LAUNCH(m, "fc1_reduce", launch_fc_reduce(t.fc_part, t.fc_splits, (size_t)t.m_pad * d0.out, d0.d_b, d0.z, only ? nullptr : d0.h,
                                                m.cfg.alpha_dense, n, d0.out, s));
    const float* in = d0.h;
    for (size_t j = 1; j < m.dense.size(); ++j) {
        DenseLayer& D = m.dense[j];
        const bool last = (j + 1 == m.dense.size());
        const int splits = std::min(D.splits, sgemm_pick_splits(n, D.out, D.in));
        TP_LAUNCH(m, "sgemm", launch_sgemm(in, D.d_w, m.partials, n, D.out, D.in, true, splits, s));
        TP_LAUNCH(m, "splitk_reduce", launch_splitk_reduce(m.partials, splits, D.d_b, D.z, last ? nullptr : D.h, m.cfg.alpha_dense, n, D.out, s));
        in = D.h;
    }
    TP_LAUNCH(m, "head", launch_head(m.dense.back().z, m.probs, m.cls, n, m.cfg.num_classes, m.cfg.head, s));
    return BCAD_OK;
}

// alpha_raw of one target class column (class_idx) into alpha_dst.  rerun_head: the chunk's dense head already ran for another class
static int tensor_alpha(Model& m, int n, const int32_t* class_idx, int grad_mode, float* alpha_dst, bool rerun_head, cudaStream_t s) {
    TensorPath& t = *m.tp;
    const ConvLayer& T = m.conv.back();
    if (m.cfg.pool_ties != BCAD_TIES_FIRST) {
        // tie-duplicating rule (the NumPy CNN): no alpha shortcut -- dz1 -> dense pooled gradient (fp32 GEMM with the fp32 fc1
        // weights) -> alpha with per-window tie counts read from the split activations; alpha_raw then feeds the usual tail
        if (!m.fused_head) TP_TRY(dense_backward(&m, n, class_idx, grad_mode, nullptr, s));          // leaves dz1 in dense[0].h
        else if (rerun_head) TP_TRY(relaunch_fused_head(&m, class_idx, nullptr, s));
        DenseLayer& D0 = m.dense[0];
        if (t.d_fc_wT != nullptr) {
            // g[b][col] = sum_u dz1[b][u] W1[u][col] on tcgen05: split operands, one CTA per (256-column block, 128-image tile)
            TP_LAUNCH(m, "dz1_to_tiles", launch_rows_to_fc_tiles_x3(D0.h, t.dz_tiles, n, D0.out, t.m_pad, s));
            FcArgs f;
            f.a_tiles = t.dz_tiles; f.w_tiles = t.d_fc_wT; f.partials = m.g_flat;
            f.N = 256; f.nkb = D0.out / 64; f.kb_per_split = f.nkb; f.splits = 1;
            f.m_tiles = cdiv(n, 128); f.m_pad = 0; f.x3 = 1; f.ncb = (int)(D0.in / 256); f.ld_out = (long long)D0.in; f.m_valid = n;
            TP_LAUNCH(m, "fc1_dgrad_tcgen05", launch_fc_splitk(f, s));
        } else {
            TP_LAUNCH(m, "fc1_dgrad_sgemm", launch_sgemm(D0.h, D0.d_w, m.g_flat, n, D0.in, D0.out, false, 1, s));
        }
        TP_LAUNCH(m, "alpha_ties_c8", launch_alpha_ties_c8(t.act, m.g_flat, alpha_dst, n, T.Ho, T.Wo, T.Cout, s));
    } else if (!m.fused_head) {
        // dense backward down to dz1 (left in dense[0].h); no fc1 dgrad GEMM, no dA
        TP_TRY(dense_backward(&m, n, class_idx, grad_mode, nullptr, s));
        const float* dz1 = (m.dense.size() > 1) ? m.dense[0].h : m.d_top;
        TP_LAUNCH(m, "alpha_shortcut_sgemm", launch_sgemm(dz1, t.d_S, alpha_dst, n, T.Cout, m.dense[0].out, false, 1, s));
    } else if (rerun_head) {
        TP_TRY(relaunch_fused_head(&m, class_idx, alpha_dst, s));                 // the fused head's alpha shortcut
    }
    return BCAD_OK;
}

int tensor_explain_chunk(Model& m, int n, const int32_t* class_idx, int grad_mode, float* heat, cudaStream_t s, int K, size_t col_ld,
                         size_t heat_stride) {
    TensorPath& t = *m.tp;
    const ConvLayer& T = m.conv.back();
    const float inv_hw = 1.0f / ((float)T.Ho * (float)T.Wo);
    const size_t hm = (size_t)m.heat_h * m.heat_w, slot = (size_t)m.cfg.max_batch * T.Cout;
    // The one-launch cluster tail needs about a CTA pair per SM to pay (one image's pair streams its 2-4 MB map at a single SM
    // pair's bandwidth: 73 us whatever the batch); handles sized for a few images (single requests, the refinement twin) take the
    // two-launch form, whose channel reduction spreads one image over 8 CTAs (16 images: 30 instead of 72 us).  A property of the
    // HANDLE, so that a given handle's results do not depend on how a batch is chunked.
    const bool small_handle = m.cfg.max_batch <= 32;
    const bool fused = !small_handle && tail_fused_supported(T.Ho, T.Wo, m.heat_h, m.heat_w, T.Cout) && getenv("BCAD_TAIL_TWO_KERNELS") == nullptr;
    // several classes: groups of TF_GROUP share one read of A in the fused tail; the two-launch form reads A once per class
    const int group = (fused && K > 1 && tail_fused_classes_supported(T.Ho, T.Wo, m.heat_h, m.heat_w, T.Cout)) ? TF_GROUP : 1;
    for (int k0 = 0; k0 < K; k0 += group) {
        const int g = std::min(group, K - k0);
        for (int j = 0; j < g; ++j) {
            const int k = k0 + j;
            TP_TRY(tensor_alpha(m, n, class_idx ? class_idx + k * col_ld : nullptr, grad_mode, t.alpha_raw + j * slot, k > 0, s));
        }
        float* hk = heat + k0 * hm;
        if (g > 1) {
            TP_LAUNCH(m, "tail_fused_classes", launch_tail_fused_classes(t.act, t.alpha_raw, slot, inv_hw, hk, heat_stride, n, T.Ho, T.Wo,
                                                                         m.heat_h, m.heat_w, T.Cout, t.x3, s, m.n_dev));
        } else if (fused) {
            TP_LAUNCH(m, "tail_fused", launch_tail_fused(t.act, t.alpha_raw, inv_hw, m.alpha, hk, n, T.Ho, T.Wo, m.heat_h, m.heat_w, T.Cout, t.x3, s, m.n_dev,
                                                         heat_stride));
        } else {
            TP_LAUNCH(m, "cam_c8", launch_cam_c8(t.act, t.alpha_raw, inv_hw, m.alpha, m.cam_lo, m.mm, n, T.Ho, T.Wo, T.Cout, m.cam_splits, t.x3, s, m.n_dev));
            TP_LAUNCH(m, "upsample_norm", launch_upsample_norm(m.cam_lo, m.mm, m.cam_splits, hk, n, T.Ho, T.Wo, m.heat_h, m.heat_w, s, m.n_dev,
                                                               heat_stride));
        }
    }
    return BCAD_OK;
}

int tensor_get_activation(Model& m, int kind, int index, int B, float* dst, cudaStream_t s) {
    TensorPath& t = *m.tp;
    if (kind == BCAD_T_CONV_OUT && index == 1) {
        const ConvLayer& L = m.conv[1];
        return launch_c8_to_nhwc(t.act, dst, B, L.Ho, L.Wo, L.Cout, t.x3, s);
    }
    if (kind == BCAD_T_POOL_OUT && index == 0) {
        if (!t.p1_valid) {
            set_error("get_tensor: the fused conv kernel keeps the pooled first-block map on chip; create the model with keep_all_activations=1 to have it written out");
            return BCAD_ERR_STATE;
        }
        const ConvLayer& L = m.conv[0];
        return launch_c8_to_nhwc(t.p1, dst, B, L.Hp, L.Wp, L.Cout, t.x3, s);
    }
    set_error("get_tensor: the tensor path does not materialise tensor (%d,%d); use BCAD_PREC_FP32 for full activation caches", kind, index);
    return BCAD_ERR_STATE;
}

}  // namespace bcad
