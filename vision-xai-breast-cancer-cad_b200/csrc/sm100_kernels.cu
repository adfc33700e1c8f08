// 16-bit tensor-core path (sm_100a; fp16 operands, fp32 accumulation): tcgen05.mma with TMEM accumulators, operands staged in shared memory by
// the bulk-copy (TMA) engine, warp-specialised persistent kernels.
//
// Device-internal layouts (all ours, chosen so every transfer is a contiguous bulk copy and every UMMA operand
// is a canonical K-major image with no data reshuffling):
//   "C8 planar" activations   X[b][y][c/8][x][8] fp16   -- one (row, channel-octet) plane is x-contiguous 16 B items
//   conv weights image        [tap*(Cin/8)+chunk][cout][8] fp16  -- no-swizzle core matrices (8 couts x 16 B)
//   fc1 A tiles (pooled act.) [b/128][pooled pixel][b%128][128 B, 16 B chunks XOR (row&7)]  -- SW128 K-major
//   fc1 W tiles               [pooled pixel][unit][128 B, chunks XOR (unit&7)]               -- SW128 K-major
//
// Reference semantics: conv+bias+LeakyReLU+2x2 max-pool (Classes/CNNModel.py:227-261, ADCNNM.py:48,76),
// dense z = W.flat + b (Classes/CNNModel.py:180); Grad-CAM channel reduction (pytorch_grad_cam, GRADCAM.py:64).
#include <stdlib.h>

#include "../../include/bcad.h"
#include "common.cuh"
#include "sm100.cuh"
#include "sm100_kernels.h"

namespace bcad {

using namespace sm100;

__device__ __forceinline__ uint32_t h2u(const __half2& h) { return *reinterpret_cast<const uint32_t*>(&h); }
__device__ __forceinline__ __half2 u2h(uint32_t v) { return *reinterpret_cast<const __half2*>(&v); }

// =====================================================================================================
// first conv block (Cin = 1, 3x3): CUDA cores, fused bias + LeakyReLU + 2x2 max-pool, fp16 C8-planar out.
// K = 9 is too skinny for the tensor core; the block is ~6 % of the network's MACs.
// block = 2 pooled rows x 128 pooled columns; thread = one pooled pixel, loops over channel octets.
// =====================================================================================================
template <int COUT>
__global__ void __launch_bounds__(256)
conv_first_pool_kernel(const float* __restrict__ x, const float* __restrict__ w /*[9][COUT]*/,
                       const float* __restrict__ bias, __half* __restrict__ out, int H, int W, int pad, int Hp,
                       int Wp, float alpha) {
    __shared__ __align__(16) float s_w[9 * COUT];
    __shared__ float s_b[COUT];
    for (int i = threadIdx.x; i < 9 * COUT; i += 256) s_w[i] = w[i];
    for (int i = threadIdx.x; i < COUT; i += 256) s_b[i] = bias[i];
    __syncthreads();
    const int b = blockIdx.z;
    const int px = blockIdx.x * 128 + (threadIdx.x & 127);
    const int py = blockIdx.y * 2 + (threadIdx.x >> 7);
    if (px >= Wp || py >= Hp) return;
    const float* xb = x + (size_t)b * H * W;
    float in[4][4];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int iy = 2 * py - pad + r;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int ix = 2 * px - pad + c;
            in[r][c] = (iy >= 0 && iy < H && ix >= 0 && ix < W) ? __ldg(xb + (size_t)iy * W + ix) : 0.f;
        }
    }
#pragma unroll 1
    for (int oc = 0; oc < COUT / 8; ++oc) {
        float acc[4][8];
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[q][j] = 0.f;
#pragma unroll
        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) {
                const float4 w0 = *reinterpret_cast<const float4*>(&s_w[(ky * 3 + kx) * COUT + oc * 8]);
                const float4 w1 = *reinterpret_cast<const float4*>(&s_w[(ky * 3 + kx) * COUT + oc * 8 + 4]);
                const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float v = in[(q >> 1) + ky][(q & 1) + kx];
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[q][j] = fmaf(v, wv[j], acc[q][j]);
                }
            }
        // max-pool commutes with the monotone bias + LeakyReLU (alpha >= 0): pool first, activate once
        uint32_t pk[4];
#pragma unroll
        for (int j = 0; j < 8; j += 2) {
            float m0 = fmaxf(fmaxf(acc[0][j], acc[1][j]), fmaxf(acc[2][j], acc[3][j])) + s_b[oc * 8 + j];
            float m1 = fmaxf(fmaxf(acc[0][j + 1], acc[1][j + 1]), fmaxf(acc[2][j + 1], acc[3][j + 1])) + s_b[oc * 8 + j + 1];
            pk[j >> 1] = pack_f16(leaky(m0, alpha), leaky(m1, alpha));
        }
        uint4* dst = reinterpret_cast<uint4*>(out) + (((size_t)b * Hp + py) * (COUT / 8) + oc) * Wp + px;
        *dst = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    }
}

int launch_conv_first_pool(const float* x, const float* w9c, const float* bias, __half* out, int B, int H, int W,
                           int pad, int Cout, float alpha, cudaStream_t s) {
    const int Ho = H + 2 * pad - 2, Wo = W + 2 * pad - 2, Hp = Ho / 2, Wp = Wo / 2;
    dim3 grid(cdiv(Wp, 128), cdiv(Hp, 2), B);
    switch (Cout) {
        case 16: conv_first_pool_kernel<16><<<grid, 256, 0, s>>>(x, w9c, bias, out, H, W, pad, Hp, Wp, alpha); break;
        case 32: conv_first_pool_kernel<32><<<grid, 256, 0, s>>>(x, w9c, bias, out, H, W, pad, Hp, Wp, alpha); break;
        case 64: conv_first_pool_kernel<64><<<grid, 256, 0, s>>>(x, w9c, bias, out, H, W, pad, Hp, Wp, alpha); break;
        default: set_error("conv_first_pool: Cout %d not supported (16/32/64)", Cout); return BCAD_ERR_INVALID;
    }
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// =====================================================================================================
// first conv block on the tensor core.  K = 9 taps is padded to 32 and the spare slots buy fp32-grade accuracy
// for free: with x = x_hi + x_lo and w = w_hi + w_lo (fp16 pairs),
//     A row = [x_hi(9) 1 | x_lo(9) 1 | x_hi(9) 0 0 0],   B row = [w_hi(9) b_hi | w_hi(9) b_lo | w_lo(9) 0 0 0]
// gives x_hi w_hi + x_lo w_hi + x_hi w_lo + b (every product exact in the fp32 accumulator; the dropped x_lo w_lo
// term is 2^-22 relative).  One CTA tile = 128 pooled pixels of one pooled row; the four members of each 2x2 pool
// window are four accumulators of the SAME TMEM lane, so pooling is three max ops per channel with no shuffles.
// The CUDA-core work left is the im2col row build (16 STS.128 / thread) and the pooled epilogue: ~4x fewer
// instructions than 1152 FFMAs per pooled pixel.  128-thread CTAs; DBUF: im2col image double-buffered, 3 CTAs per SM;
// !DBUF: one image, 4 CTAs per SM.
// =====================================================================================================
// PLAIN (the fp16 mode): operands as plain fp16 -- A row = [x(9) 1 1 0 0 0 0 0], B row = [w(9) b_hi b_lo 0 0 0 0 0], one K-step.
template <int COUT, bool SPLIT, bool DBUF, bool PLAIN>
__global__ void __launch_bounds__(128, DBUF ? 3 : 4)
conv_first_tc_kernel(const float* __restrict__ x, const uint8_t* __restrict__ w_img /*[4 or 2][COUT][16 B]*/,
                     __half* __restrict__ out, int B, int H, int W, int pad, int Hp, int Wp, float alpha, const int* __restrict__ n_dev) {
    if (n_dev != nullptr) {                       // live image count decided on the device (refine.cu)
        const int nd = *n_dev;
        if (nd <= 0) return;
        if (nd < B) B = nd;
    }
    extern __shared__ __align__(128) uint8_t smem[];
    uint8_t* s_a = smem;                          // (DBUF ? 2 : 1) buffers x 4 classes x [4 chunks][128 rows][16 B] = 32 KB each
    uint8_t* s_b = smem + (DBUF ? 2 : 1) * 32768;  // [4 chunks][COUT][16 B]
    __shared__ uint64_t bar;
    __shared__ uint32_t tmem_slot;
    const int tid = threadIdx.x, warp = tid >> 5;
    static_assert(!(PLAIN && SPLIT), "the fp16x3 mode keeps the hi/lo split");
    for (int i = tid; i < ((PLAIN ? 2 : 4) * COUT * 16) / 16; i += 128) reinterpret_cast<uint4*>(s_b)[i] = reinterpret_cast<const uint4*>(w_img)[i];
    if (tid == 0) {
        mbar_init(&bar, 1);
        fence_barrier_init();
    }
    if (warp == 0) {
        tmem_alloc(&tmem_slot, 4 * COUT);
        tmem_relinquish();
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const uint32_t lane_off = (uint32_t)(warp * 32) << 16;
    constexpr uint32_t idesc = make_idesc_f16(128, COUT);
    constexpr uint64_t a_tmpl = ((uint64_t)(2048 >> 4) << 16) | ((uint64_t)(128 >> 4) << 32) | ((uint64_t)1 << 46);
    constexpr uint64_t b_tmpl = ((uint64_t)((COUT * 16) >> 4) << 16) | ((uint64_t)(128 >> 4) << 32) | ((uint64_t)1 << 46);
    const uint64_t a_desc0 = a_tmpl | (uint64_t)((smem_u32(s_a) & 0x3FFFFu) >> 4);
    const uint64_t b_desc0 = b_tmpl | (uint64_t)((smem_u32(s_b) & 0x3FFFFu) >> 4);
    const bool max_form = alpha <= 1.f;
    const int xtiles = cdiv(Wp, 128);
    const int n_tiles = B * Hp * xtiles;
    uint32_t phase = 0;
    // input patch of a tile: 4 x 4 fp32 values per thread (zero outside the image); the loads of tile t+1 are
    // issued before the epilogue of tile t so their latency hides behind it
    // tile coordinates (image, pooled row, x tile) advance by gridDim.x tiles per iteration without divisions
    struct TileC { int b, py, xt; };
    const int G = gridDim.x;
    const int g_xt = G % xtiles, g_py = (G / xtiles) % Hp, g_b = G / (xtiles * Hp);
    auto advance = [&](TileC& t) {
        t.xt += g_xt;
        if (t.xt >= xtiles) { t.xt -= xtiles; ++t.py; }
        t.py += g_py;
        if (t.py >= Hp) { t.py -= Hp; ++t.b; }
        t.b += g_b;
    };
    auto load_patch = [&](const TileC& t, float (&v)[16]) {
        const int py = t.py, b = t.b;
        const int px = t.xt * 128 + tid;
        const float* xb = x + (size_t)b * H * W;
        const int iy0 = 2 * py - pad, ix0 = 2 * px - pad;
        if (iy0 >= 0 && iy0 + 3 < H && ix0 >= 0 && ix0 + 3 < W) {
            const float* p0 = xb + (size_t)iy0 * W + ix0;
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c) v[r * 4 + c] = __ldg(p0 + (size_t)r * W + c);
        } else {
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const int iy = iy0 + r, ix = ix0 + c;
                    v[r * 4 + c] = (iy >= 0 && iy < H && ix >= 0 && ix < W) ? __ldg(xb + (size_t)iy * W + ix) : 0.f;
                }
        }
    };
    // Software pipeline over tiles: the im2col image is double-buffered, so the rows of tile t+1 are built while the
    // MMAs of tile t run; one __syncthreads per tile.
    auto build = [&](int buf, const float (&patch)[16]) {
        // im2col rows of this thread's 2x2 pool window.  K slots (matching the weight image):
        //      [x(9) 1 | x_lo(9) 1 | x(9) 0 0 0]  -- cvt.rn.f16x2 turns an fp32 pair straight into one packed word
        float lo[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) lo[e] = PLAIN ? 0.f : patch[e] - __half2float(__float2half_rn(patch[e]));
#pragma unroll
        for (int q = 0; q < 4; ++q) {               // class q = (row parity, col parity) of the pool window
            const int qr = q >> 1, qc = q & 1;
            float xt[9], lt[9];
#pragma unroll
            for (int t = 0; t < 9; ++t) {
                const int pi = (qr + t / 3) * 4 + (qc + t % 3);
                xt[t] = patch[pi];
                lt[t] = lo[pi];
            }
            uint32_t wd[16];
            wd[0] = pack_f16(xt[0], xt[1]); wd[1] = pack_f16(xt[2], xt[3]); wd[2] = pack_f16(xt[4], xt[5]); wd[3] = pack_f16(xt[6], xt[7]);
            wd[4] = pack_f16(xt[8], 1.f);
            if constexpr (PLAIN) {
                wd[5] = 0x00003C00u;                // (1, 0): the b_lo slot
                wd[6] = wd[7] = 0u;
#pragma unroll
                for (int ch = 0; ch < 2; ++ch)
                    *reinterpret_cast<uint4*>(s_a + buf * 32768 + q * 8192 + ch * 2048 + tid * 16) =
                        make_uint4(wd[ch * 4], wd[ch * 4 + 1], wd[ch * 4 + 2], wd[ch * 4 + 3]);
                continue;
            }
            wd[5] = pack_f16(lt[0], lt[1]); wd[6] = pack_f16(lt[2], lt[3]); wd[7] = pack_f16(lt[4], lt[5]); wd[8] = pack_f16(lt[6], lt[7]);
            wd[9] = pack_f16(lt[8], 1.f);
            wd[10] = wd[0]; wd[11] = wd[1]; wd[12] = wd[2]; wd[13] = wd[3];
            wd[14] = wd[4] & 0x0000ffffu;           // (x8, 0)
            wd[15] = 0u;
#pragma unroll
            for (int ch = 0; ch < 4; ++ch)
                *reinterpret_cast<uint4*>(s_a + buf * 32768 + q * 8192 + ch * 2048 + tid * 16) =
                    make_uint4(wd[ch * 4], wd[ch * 4 + 1], wd[ch * 4 + 2], wd[ch * 4 + 3]);
        }
    };
    auto issue = [&](int buf) {
        if (warp == 0) {                            // warp-uniform; one elected lane issues (plain predicated UTCHMMA)
            const bool leader = elect_one();
            tc_fence_after();
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
                for (int ks = 0; ks < (PLAIN ? 1 : 2); ++ks)
                    umma_f16_if(leader, tmem + q * COUT, a_desc0 + (uint64_t)((buf * 32768 + q * 8192 + ks * 4096) >> 4),
                                b_desc0 + (uint64_t)((ks * 2 * COUT * 16) >> 4), idesc, ks);
            umma_commit_if(leader, &bar);
        }
    };
    auto epilogue = [&](const TileC& t) {
        const int py = t.py, b = t.b;
        const int px = t.xt * 128 + tid;
        // ---- epilogue: pool (3 max), LeakyReLU once, fp16 C8-planar store
#pragma unroll 1
        for (int c0 = 0; c0 < COUT; c0 += 16) {
            float v0[16], v1[16], v2[16], v3[16];
            tmem_ld16(tmem + lane_off + 0 * COUT + c0, v0);
            tmem_ld16(tmem + lane_off + 1 * COUT + c0, v1);
            tmem_ld16(tmem + lane_off + 2 * COUT + c0, v2);
            tmem_ld16(tmem + lane_off + 3 * COUT + c0, v3);
            tmem_ld_wait();
            if (px < Wp) {
#pragma unroll
                for (int cc = 0; cc < 2; ++cc) {
                    uint32_t pk[4];
#pragma unroll
                    for (int e = 0; e < 8; e += 2) {
                        const int k0 = cc * 8 + e;
                        float m0 = fmaxf(fmaxf(v0[k0], v1[k0]), fmaxf(v2[k0], v3[k0]));
                        float m1 = fmaxf(fmaxf(v0[k0 + 1], v1[k0 + 1]), fmaxf(v2[k0 + 1], v3[k0 + 1]));
                        m0 = max_form ? fmaxf(m0, alpha * m0) : leaky(m0, alpha);
                        m1 = max_form ? fmaxf(m1, alpha * m1) : leaky(m1, alpha);
                        pk[e >> 1] = pack_f16(m0, m1);
                    }
                    if constexpr (!SPLIT) {
                        uint4* dst = reinterpret_cast<uint4*>(out) + (((size_t)b * Hp + py) * (COUT / 8) + (c0 / 8 + cc)) * Wp + px;
                        *dst = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                    }
                }
                if constexpr (SPLIT) {
                    // fp16x3 mode: the pooled fp32 value goes out as hi + lo halves, as 2*COUT "virtual" channels
                    // (octets [hi 0..COUT/8) | lo 0..COUT/8)) of one C8-planar tensor
#pragma unroll
                    for (int cc = 0; cc < 2; ++cc) {
                        uint32_t ph[4], pl[4];
#pragma unroll
                        for (int e = 0; e < 8; e += 2) {
                            const int k0 = cc * 8 + e;
                            float m0 = fmaxf(fmaxf(v0[k0], v1[k0]), fmaxf(v2[k0], v3[k0]));
                            float m1 = fmaxf(fmaxf(v0[k0 + 1], v1[k0 + 1]), fmaxf(v2[k0 + 1], v3[k0 + 1]));
                            m0 = max_form ? fmaxf(m0, alpha * m0) : leaky(m0, alpha);
                            m1 = max_form ? fmaxf(m1, alpha * m1) : leaky(m1, alpha);
                            const __half2 h = __floats2half2_rn(m0, m1);
                            const float2 hf = __half22float2(h);
                            ph[e >> 1] = h2u(h);
                            pl[e >> 1] = pack_f16(m0 - hf.x, m1 - hf.y);
                        }
                        uint4* dh = reinterpret_cast<uint4*>(out) + (((size_t)b * Hp + py) * (2 * COUT / 8) + (c0 / 8 + cc)) * Wp + px;
                        *dh = make_uint4(ph[0], ph[1], ph[2], ph[3]);
                        *(dh + (size_t)(COUT / 8) * Wp) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
                    }
                }
            }
        }
    };
    float patch[16];
    int tile = blockIdx.x;
    TileC cur{tile / (xtiles * Hp), (tile / xtiles) % Hp, tile % xtiles};
    TileC nxt = cur;                                 // coordinates of the tile whose inputs `patch` holds
    if (tile < n_tiles) {
        load_patch(cur, patch);
        build(0, patch);
        fence_proxy_async();
        advance(nxt);
        if (tile + G < n_tiles) load_patch(nxt, patch);
        __syncthreads();
        issue(0);
    }
    for (int it = 0; tile < n_tiles; tile += G, ++it) {
        const int next = tile + G;
        if constexpr (DBUF) {
            if (next < n_tiles) {
                build((it + 1) & 1, patch);             // overlaps the MMAs of this tile
                fence_proxy_async();
                advance(nxt);
                if (next + G < n_tiles) load_patch(nxt, patch);          // inputs of tile t+2
            }
            mbar_wait(&bar, phase);
            phase ^= 1;
            tc_fence_after();
        } else {
            // one im2col buffer (a 4th CTA per SM instead): it is free again once this tile's MMAs have retired
            mbar_wait(&bar, phase);
            phase ^= 1;
            tc_fence_after();
            if (next < n_tiles) {
                build(0, patch);
                fence_proxy_async();
                advance(nxt);
                if (next + G < n_tiles) load_patch(nxt, patch);
            }
        }
        epilogue(cur);
        advance(cur);
        tc_fence_before();
        __syncthreads();                            // next image fully built; TMEM drained
        if (next < n_tiles) issue(DBUF ? ((it + 1) & 1) : 0);
    }
    if (warp == 0) tmem_dealloc(tmem, 4 * COUT);
}

template <int COUT, bool SPLIT, bool DBUF = true, bool PLAIN = false>
static int launch_conv_first_tc_t(const float* x, const uint8_t* w_img, __half* out, int B, int H, int W, int pad, int Hp,
                                  int Wp, float alpha, int grid, int smem, cudaStream_t s, const int* n_dev) {
    BCAD_CUDA_CHECK(cudaFuncSetAttribute(conv_first_tc_kernel<COUT, SPLIT, DBUF, PLAIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    conv_first_tc_kernel<COUT, SPLIT, DBUF, PLAIN><<<grid, 128, smem, s>>>(x, w_img, out, B, H, W, pad, Hp, Wp, alpha, n_dev);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

int launch_conv_first_tc(const float* x, const uint8_t* w_img, __half* out, int B, int H, int W, int pad, int Cout,
                         float alpha, bool split_hi_lo, bool plain, int sms, cudaStream_t s, const int* n_dev) {
    BCAD_REQUIRE(!(plain && split_hi_lo), "conv_first_tc: the hi/lo output split needs hi/lo operands");
    const int Ho = H + 2 * pad - 2, Wo = W + 2 * pad - 2, Hp = Ho / 2, Wp = Wo / 2;
    const int n_tiles = B * Hp * cdiv(Wp, 128);
    // 32 filters, fp16 mode: ONE im2col buffer and a 4th CTA per SM (TMEM allows 4 x 128 columns) measured 2.6 % faster than
    // double-buffering with 3 CTAs (0.254 vs 0.261 ms at 512 x 256x256)
    const bool single = (Cout == 32 && !split_hi_lo);
    const int smem = (single ? 1 : 2) * 32768 + 4 * Cout * 16;
    const int per_sm = Cout <= 32 ? (single ? 4 : 3) : 2;          // smem: 66 KB per CTA; TMEM: 4*Cout columns per CTA
    const int grid = n_tiles < sms * per_sm ? n_tiles : sms * per_sm;
    if (single && plain) return launch_conv_first_tc_t<32, false, false, true>(x, w_img, out, B, H, W, pad, Hp, Wp, alpha, grid, smem, s, n_dev);
    if (single) return launch_conv_first_tc_t<32, false, false>(x, w_img, out, B, H, W, pad, Hp, Wp, alpha, grid, smem, s, n_dev);
    if (Cout == 32 && split_hi_lo) return launch_conv_first_tc_t<32, true>(x, w_img, out, B, H, W, pad, Hp, Wp, alpha, grid, smem, s, n_dev);
    if (Cout == 64 && plain) return launch_conv_first_tc_t<64, false, true, true>(x, w_img, out, B, H, W, pad, Hp, Wp, alpha, grid, smem, s, n_dev);
    if (Cout == 64 && !split_hi_lo) return launch_conv_first_tc_t<64, false>(x, w_img, out, B, H, W, pad, Hp, Wp, alpha, grid, smem, s, n_dev);
    set_error("conv_first_tc: Cout %d (split=%d) not supported", Cout, (int)split_hi_lo);
    return BCAD_ERR_INVALID;
}

// =====================================================================================================
// 3x3 convolution as implicit GEMM on tcgen05 (Cin in {16,32,64}, Cout = 64, map width <= 128)
//
//   M = 128 consecutive pixels of one output row, N = Cout, K = 9 taps x Cin.
//   Input rows live in a shared-memory ring in C8-planar order (pixels 16 B apart), so the A operand of tap
//   (dy,dx) is just the ring row (y+dy) with the descriptor start address advanced by dx*16 bytes: no im2col
//   copy, every input row is fetched from L2/HBM exactly once per band.  Zero padding = two halo pixel slots
//   that are never written + a permanently-zero row slot.
//   Output rows are produced in pairs so the 2x2 max-pool happens in the epilogue (vertical max in registers,
//   horizontal max with one shuffle); accumulators are double-buffered in TMEM so the epilogue of pair p
//   overlaps the MMAs of pair p+1.
//   Warp roles: 0 = bulk-copy producer, 1 = MMA issuer, 2..9 = epilogue (TMEM lane quadrant = warp % 4; the two
//   warps of a quadrant split the channels, so every scheduler has two epilogue warps to hide latency).
// =====================================================================================================
#ifndef IG_STAGES_SMALL
#define IG_STAGES_SMALL 4
#endif
constexpr int IG_XP = 136;            // pixel slots per ring row (>= 128 + 2 halo; 137 / 140 measured identical: no bank effect)
constexpr int ig_stages(int cin) { return cin >= 64 ? 3 : IG_STAGES_SMALL; }   // ring stages of 2 input rows (smem budget)
constexpr int IG_THREADS = 320;         // producer warp, MMA warp, 8 epilogue warps (2 per scheduler)

template <int CIN, int COUT>
struct IgemmSmem {
    static constexpr int STAGES = ig_stages(CIN);
    static constexpr int CHUNKS = CIN / 8;
    static constexpr int LBO = IG_XP * 16;                 // bytes between channel octets of one row
    static constexpr int ROWB = CHUNKS * LBO;              // bytes per ring row
    static constexpr int WBYTES = 9 * CHUNKS * COUT * 16;  // weight image
    static constexpr int BIAS_TILE = 2 * COUT * 16;         // B operand of the bias K-step: rows {b_hi, b_lo, 0...}
    static constexpr int ONES_TILE = 2 * 128 * 16;          // A operand of the bias K-step: rows {1, 1, 0...}
    static constexpr int OFF_W = 0;                         // weight image followed by the bias tile (one bulk copy)
    static constexpr int OFF_ONES = OFF_W + WBYTES + BIAS_TILE;
    static constexpr int OFF_ZERO = OFF_ONES + ONES_TILE;
    static constexpr int OFF_RING = OFF_ZERO + ROWB;
    static constexpr int OFF_BAR = OFF_RING + STAGES * 2 * ROWB;
    // activation staging for bulk (TMA) stores: 2 accumulator buffers x 2 rows x (COUT/8) octets x 128 px x 16 B
    static constexpr bool STAGED = false;      // measured: the two extra epilogue barriers cost more than the 16 STG they save (0.371 vs 0.345 ms)
    static constexpr int STAGE_BYTES = 2 * (COUT / 8) * 128 * 16;
    static constexpr int OFF_STAGE = OFF_BAR + 256;
    static constexpr int TOTAL = OFF_STAGE + (STAGED ? 2 * STAGE_BYTES : 0);
};

template <int CIN, int COUT, bool X3>
__global__ void __launch_bounds__(IG_THREADS, 1) conv_igemm_kernel(IgemmArgs a) {
    int n_live = a.B;
    if (a.n_dev != nullptr) {                     // live image count decided on the device (refine.cu)
        const int nd = *a.n_dev;
        if (nd <= 0) return;
        if (nd < n_live) n_live = nd;
    }
    using L = IgemmSmem<CIN, COUT>;
    constexpr int IG_STAGES = L::STAGES;
    extern __shared__ __align__(1024) uint8_t smem[];
    uint8_t* s_w = smem + L::OFF_W;
    uint8_t* s_zero = smem + L::OFF_ZERO;
    uint8_t* s_ring = smem + L::OFF_RING;
    uint8_t* s_ones = smem + L::OFF_ONES;
    uint8_t* s_stage = smem + L::OFF_STAGE;
    constexpr bool STAGED = L::STAGED && !X3;
    (void)s_stage;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::OFF_BAR);
    uint64_t* full = bars;                       // [IG_STAGES] producer -> MMA
    uint64_t* empty = bars + IG_STAGES;          // [IG_STAGES] MMA -> producer
    uint64_t* tfull = bars + 2 * IG_STAGES;      // [2] MMA -> epilogue
    uint64_t* tempty = bars + 2 * IG_STAGES + 2; // [2] epilogue -> MMA
    uint64_t* wbar = bars + 2 * IG_STAGES + 4;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * IG_STAGES + 5);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    // ---- one-time setup: zero the halo slots + zero row, barriers, TMEM
    for (int i = tid; i < (L::ROWB * (1 + IG_STAGES * 2)) / 16; i += IG_THREADS)
        reinterpret_cast<uint4*>(s_zero)[i] = make_uint4(0, 0, 0, 0);
    for (int i = tid; i < L::ONES_TILE / 16; i += IG_THREADS)      // chunk 0: halves {1,1,0,0,0,0,0,0}; chunk 1: zeros
        reinterpret_cast<uint4*>(s_ones)[i] = (i < 128) ? make_uint4(0x3C003C00u, 0, 0, 0) : make_uint4(0, 0, 0, 0);
    if (tid == 0) {
        for (int i = 0; i < IG_STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 8); }
        mbar_init(wbar, 1);
        fence_barrier_init();
    }
    // accumulator columns per output row: COUT, or 2*COUT in the fp16x3 mode ([x.w_hi sums | x_hi.w_lo sums], added in the epilogue)
    constexpr int ACC = X3 ? 2 * COUT : COUT;
    if (warp == 0) {
        tmem_alloc(tmem_slot, 4 * ACC);
        tmem_relinquish();
    }
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    const int per_img = a.bands * a.xsegs;
    const int n_items = n_live * per_img;
    const int in_row_elems = L::CHUNKS * a.W * 8;          // fp16 elements per input row (all channel octets)

    if (warp == 0) {
        // ================================ producer ================================
        // (whole warp: lane 0 issues the bulk copies, the lanes zero the halo slots a segment leaves unwritten)
        {
            constexpr int WB = L::WBYTES + L::BIAS_TILE;
            if (lane == 0) {
                mbar_arrive_expect_tx(wbar, WB);
                for (int off = 0; off < WB; off += 16384)
                    bulk_g2s(s_w + off, a.w_img + off, min(16384, WB - off), wbar);
            }
            uint32_t g = 0;
            for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
                const int b = item / per_img, rem = item % per_img;
                const int band = rem / a.xsegs, x0 = (rem % a.xsegs) * 128;
                const int y0 = band * a.band_rows;
                const int nrows = min(a.band_rows, a.Ho - y0);
                const int nstages = (nrows + 1) / 2 + 1;
                // ring slot s holds input pixel x0 - pad + s; slots outside the image stay (or are made) zero
                const int s_lo = max(0, a.pad - x0), s_hi = min(130, a.W - x0 + a.pad);
                const bool zero_hi = (a.xsegs > 1) && (s_hi < 130);       // only a multi-segment map can leave stale pixels there
                const bool zero_lo = (a.xsegs > 1) && (s_lo > 0);
                const __half* inb = a.in + (size_t)b * a.H * in_row_elems + (size_t)(x0 - a.pad + s_lo) * 8;
                for (int q = 0; q < nstages; ++q, ++g) {
                    const uint32_t slot = g % IG_STAGES;
                    if (g >= IG_STAGES) mbar_wait(&empty[slot], ((g / IG_STAGES) - 1) & 1);
                    if (zero_hi || zero_lo) {
                        for (int i = lane; i < 2 * L::CHUNKS; i += 32) {
                            uint8_t* rowp = s_ring + (slot * 2 + (i / L::CHUNKS)) * L::ROWB + (i % L::CHUNKS) * L::LBO;
                            if (zero_lo) *reinterpret_cast<uint4*>(rowp) = make_uint4(0, 0, 0, 0);
                            if (zero_hi) *reinterpret_cast<uint4*>(rowp + s_hi * 16) = make_uint4(0, 0, 0, 0);
                        }
                        fence_proxy_async();
                        __syncwarp();
                    }
                    if (lane == 0) {
                        uint32_t bytes = 0;
                        for (int r = 0; r < 2; ++r) {
                            const int in_row = y0 - a.pad + 2 * q + r;
                            if (in_row >= 0 && in_row < a.H) bytes += L::CHUNKS * (s_hi - s_lo) * 16;
                        }
                        if (bytes) mbar_arrive_expect_tx(&full[slot], bytes);
                        else mbar_arrive(&full[slot]);
                        for (int r = 0; r < 2; ++r) {
                            const int in_row = y0 - a.pad + 2 * q + r;
                            if (in_row < 0 || in_row >= a.H) continue;
                            uint8_t* dst = s_ring + (slot * 2 + r) * L::ROWB + s_lo * 16;
                            const __half* src = inb + (size_t)in_row * in_row_elems;
                            for (int c = 0; c < L::CHUNKS; ++c)
                                bulk_g2s(dst + c * L::LBO, src + (size_t)c * a.W * 8, (s_hi - s_lo) * 16, &full[slot]);
                        }
                    }
                    __syncwarp();
                }
            }
        }
    } else if (warp == 1) {
        // ================================ MMA issuer ================================
        {   // warp-uniform loop; one elected lane issues the MMAs and commits
            const bool leader = elect_one();
            constexpr uint32_t idesc = make_idesc_f16(128, COUT);
            mbar_wait(wbar, 0);
            uint32_t g = 0, acc_it = 0;
            const uint32_t w_base = smem_u32(s_w), zero_base = smem_u32(s_zero), ring_base = smem_u32(s_ring);
            for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
                const int band = (item % per_img) / a.xsegs;
                const int y0 = band * a.band_rows;
                const int nrows = min(a.band_rows, a.Ho - y0);
                const int npairs = (nrows + 1) / 2;
                for (int p = 0; p < npairs; ++p, ++g, ++acc_it) {
                    if (p == 0) mbar_wait(&full[g % IG_STAGES], (g / IG_STAGES) & 1);
                    mbar_wait(&full[(g + 1) % IG_STAGES], ((g + 1) / IG_STAGES) & 1);
                    const uint32_t j = acc_it & 1;
                    if (acc_it >= 2) mbar_wait(&tempty[j], ((acc_it >> 1) - 1) & 1);
                    tc_fence_after();
                    // descriptor templates: only the 14-bit start-address field changes between MMAs, and all the
                    // per-tap offsets are compile-time constants after unrolling (the single issuing thread must
                    // spend fewer cycles per MMA than the tensor core does: 32)
                    constexpr uint32_t d_hi = (uint32_t)(128 >> 4) | (1u << 14);            // SBO = 128 B, descriptor version 1
                    constexpr uint32_t a_lo_t = (uint32_t)(L::LBO >> 4) << 16;              // LBO = octet pitch of a ring row
                    constexpr uint32_t b_lo_t = (uint32_t)((COUT * 16) >> 4) << 16;
                    const uint32_t b_lo0 = b_lo_t | ((w_base & 0x3FFFFu) >> 4);
                    const uint32_t ones_lo = ((uint32_t)((128 * 16) >> 4) << 16) | ((smem_u32(s_ones) & 0x3FFFFu) >> 4);
                    for (int r = 0; r < 2; ++r) {
                        if (2 * p + r >= nrows || (a.debug & 8)) break;     // debug bit 3: timing experiment without MMAs
                        const uint32_t d_tmem = tmem + j * (2 * ACC) + r * ACC;
                        // bias K-step: D = ones x {b_hi, b_lo} (initialises the accumulator with the fp32-exact bias); in the fp16x3
                        // mode the first N = 128 MMA initialises both column halves and the bias is accumulated last
                        if constexpr (!X3)
                            umma_f16_if(leader, d_tmem, desc64(ones_lo, d_hi), desc64(b_lo0 + (uint32_t)(L::WBYTES >> 4), d_hi), idesc, 0u);
#pragma unroll
                        for (int dy = 0; dy < 3; ++dy) {
                            const int i = 2 * p + r + dy;                    // band-local input row
                            const int in_row = y0 - a.pad + i;
                            uint32_t row_base;
                            if (in_row < 0 || in_row >= a.H) row_base = zero_base;
                            else row_base = ring_base + ((((g + (i >> 1) - p) % IG_STAGES) << 1) + (i & 1)) * L::ROWB;
                            const uint32_t a_lo0 = a_lo_t | ((row_base & 0x3FFFFu) >> 4);
#pragma unroll
                            for (int dx = 0; dx < 3; ++dx) {
                                if constexpr (!X3) {
#pragma unroll
                                    for (int ks = 0; ks < CIN / 16; ++ks)
                                        umma_f16_if(leader, d_tmem, desc64(a_lo0 + (uint32_t)((ks * 2 * L::LBO + dx * 16) >> 4), d_hi),
                                                  desc64(b_lo0 + (uint32_t)((((dy * 3 + dx) * L::CHUNKS + 2 * ks) * (COUT * 16)) >> 4), d_hi),
                                                  idesc, 1u);
                                } else {
                                    // fp16x3: input octets [x_hi (H) | x_lo (H)], weight octets per tap [w_hi (H) | w_lo (H)], H = CIN/16:
                                    //   x_hi.w_hi + x_lo.w_hi + x_hi.w_lo   (x_lo.w_lo ~ 2^-22 is dropped)
                                    // The weight image interleaves the halves per octet, [w_hi(c) | w_lo(c)] = 128 B-operand columns, so
                                    // x_hi takes both in ONE N = 128 MMA (columns [0, COUT) += x_hi.w_hi, [COUT, 2 COUT) += x_hi.w_lo:
                                    // 64 cycles instead of 2 x 48) and x_lo.w_hi is an N = 64 MMA over the first half of the same block.
                                    constexpr int HP = CIN / 32;               // octet PAIRS per half
                                    constexpr uint32_t idesc2 = make_idesc_f16(128, 2 * COUT);
                                    constexpr uint32_t b2_lo_t = (uint32_t)((2 * COUT * 16) >> 4) << 16;      // LBO: [hi | lo] blocks of consecutive octets
                                    const uint32_t b2_lo0 = b2_lo_t | ((w_base & 0x3FFFFu) >> 4);
#pragma unroll
                                    for (int kp = 0; kp < HP; ++kp) {
                                        const uint32_t boff = (uint32_t)(((((dy * 3 + dx) * (L::CHUNKS / 2) + 2 * kp) * 2) * (COUT * 16)) >> 4);
                                        umma_f16_if(leader, d_tmem, desc64(a_lo0 + (uint32_t)((kp * 2 * L::LBO + dx * 16) >> 4), d_hi),
                                                    desc64(b2_lo0 + boff, d_hi), idesc2, (dy | dx | kp) ? 1u : 0u);
                                        umma_f16_if(leader, d_tmem, desc64(a_lo0 + (uint32_t)(((HP + kp) * 2 * L::LBO + dx * 16) >> 4), d_hi),
                                                    desc64(b2_lo0 + boff, d_hi), idesc, 1u);
                                    }
                                }
                            }
                        }
                        if constexpr (X3)
                            umma_f16_if(leader, d_tmem, desc64(ones_lo, d_hi), desc64(b_lo0 + (uint32_t)(L::WBYTES >> 4), d_hi), idesc, 1u);
                    }
                    umma_commit_if(leader, &empty[g % IG_STAGES]);      // stage p is dead once these MMAs retire
                    umma_commit_if(leader, &tfull[j]);
                }
                umma_commit_if(leader, &empty[g % IG_STAGES]);          // the band's last stage
                ++g;
            }
        }
    } else {
        // ================================ epilogue (8 warps) ================================
        const int quad = warp & 3;
        const int half0 = (warp - 2) >> 2;              // which 32-channel half this warp owns
        const __half2 alpha2 = __float2half2_rn(a.alpha);
        const uint32_t lane_off = (uint32_t)(quad * 32) << 16;
        uint32_t acc_it = 0;
        for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
            const int b = item / per_img, rem = item % per_img;
            const int band = rem / a.xsegs;
            const int x = (rem % a.xsegs) * 128 + quad * 32 + lane;          // output pixel of this TMEM lane
            const int y0 = band * a.band_rows;
            const int nrows = min(a.band_rows, a.Ho - y0);
            const int npairs = (nrows + 1) / 2;
            for (int p = 0; p < npairs; ++p, ++acc_it) {
                const uint32_t j = acc_it & 1;
                mbar_wait(&tfull[j], (acc_it >> 1) & 1);
                tc_fence_after();
                if (a.debug & 4) {                         // timing experiment: epilogue does nothing
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&tempty[j]);
                    continue;
                }
                const int t0 = y0 + 2 * p;
                const bool has1 = (2 * p + 1 < nrows);
                const int py = t0 >> 1, px = x >> 1;
                const bool pool_ok = has1 && py < a.Hp && px < a.Wp && !(x & 1);
                if constexpr (X3) {
                    // fp16x3 epilogue: everything stays fp32 until the final hi/lo split
#pragma unroll 1
                    for (int half = half0; half < COUT / 32; half += 2) {
#pragma unroll 1
                        for (int sub = 0; sub < 2; ++sub) {                  // 16 channels at a time (register budget)
                            const int cbase = half * 32 + sub * 16;
                            float v0[16], v1[16], w0[16], w1[16];
                            tmem_ld16(tmem + lane_off + j * (2 * ACC) + cbase, v0);
                            tmem_ld16(tmem + lane_off + j * (2 * ACC) + COUT + cbase, w0);           // the x_hi.w_lo sums
                            tmem_ld16(tmem + lane_off + j * (2 * ACC) + ACC + cbase, v1);
                            tmem_ld16(tmem + lane_off + j * (2 * ACC) + ACC + COUT + cbase, w1);
                            tmem_ld_wait();
#pragma unroll
                            for (int q = 0; q < 16; ++q) {
                                v0[q] += w0[q];
                                v1[q] += w1[q];
                                v0[q] = fmaxf(v0[q], a.alpha * v0[q]);
                                v1[q] = fmaxf(v1[q], a.alpha * v1[q]);
                            }
                            auto split_store = [&](uint4* dst_hi, size_t lo_off, const float* v) {
                                const __half2 h0 = __floats2half2_rn(v[0], v[1]), h1 = __floats2half2_rn(v[2], v[3]);
                                const __half2 h2 = __floats2half2_rn(v[4], v[5]), h3 = __floats2half2_rn(v[6], v[7]);
                                const float2 f0 = __half22float2(h0), f1 = __half22float2(h1), f2 = __half22float2(h2), f3 = __half22float2(h3);
                                *dst_hi = make_uint4(h2u(h0), h2u(h1), h2u(h2), h2u(h3));
                                *(dst_hi + lo_off) = make_uint4(pack_f16(v[0] - f0.x, v[1] - f0.y), pack_f16(v[2] - f1.x, v[3] - f1.y),
                                                                pack_f16(v[4] - f2.x, v[5] - f2.y), pack_f16(v[6] - f3.x, v[7] - f3.y));
                            };
                            if (a.act != nullptr && x < a.Wo) {
#pragma unroll
                                for (int cc = 0; cc < 2; ++cc) {
                                    const int chunk = cbase / 8 + cc;
                                    // activations: 2*COUT virtual channels, octets [hi | lo]
                                    uint4* d0 = reinterpret_cast<uint4*>(a.act) + (((size_t)b * a.Ho + t0) * (2 * COUT / 8) + chunk) * a.Wo + x;
                                    split_store(d0, (size_t)(COUT / 8) * a.Wo, v0 + cc * 8);
                                    if (has1) split_store(d0 + (size_t)(2 * COUT / 8) * a.Wo, (size_t)(COUT / 8) * a.Wo, v1 + cc * 8);
                                }
                            }
#pragma unroll
                            for (int q = 0; q < 16; ++q) {
                                const float mv = fmaxf(v0[q], v1[q]);
                                v0[q] = fmaxf(mv, __shfl_xor_sync(0xffffffffu, mv, 1));
                            }
                            if (pool_ok && a.pool_fc != nullptr) {
                                // fc1 A tiles: [b/128][pooled pixel][hi|lo][b%128][128 B swizzled]
                                const int row = b & 127;
                                uint8_t* base = a.pool_fc + (((((size_t)(b >> 7) * a.Hp * a.Wp) + (size_t)py * a.Wp + px) * 2) * 128 + row) * 128;
#pragma unroll
                                for (int cc = 0; cc < 2; ++cc) {
                                    const int chunk = (cbase / 8 + cc) ^ (row & 7);
                                    split_store(reinterpret_cast<uint4*>(base + chunk * 16), (size_t)(128 * 128) / 16, v0 + cc * 8);
                                }
                            }
                        }
                    }
                } else {
                if constexpr (STAGED) {
                    // staging buffer j was last read by the bulk stores issued two pairs ago
                    if (tid == 64) bulk_wait_read<1>();
                    named_bar_sync(1, 256);
                }
#pragma unroll 1
                for (int half = half0; half < COUT / 32; half += 2) {
                    float v0[32], v1[32];
                    tmem_ld32(tmem + lane_off + j * (2 * COUT) + half * 32, v0);
                    tmem_ld32(tmem + lane_off + j * (2 * COUT) + COUT + half * 32, v1);
                    tmem_ld_wait();
                    // the bias is already in the accumulator; round to fp16 once, then LeakyReLU and the pool run on
                    // packed half2 (max commutes with the rounding; LeakyReLU(v) = max(v, alpha v), 0 <= alpha <= 1)
                    __half2 a0[16], a1[16];
#pragma unroll
                    for (int q = 0; q < 16; ++q) {
                        const __half2 h0 = __floats2half2_rn(v0[2 * q], v0[2 * q + 1]);
                        const __half2 h1 = __floats2half2_rn(v1[2 * q], v1[2 * q + 1]);
                        a0[q] = __hmax2(h0, __hmul2(h0, alpha2));
                        a1[q] = __hmax2(h1, __hmul2(h1, alpha2));
                    }
                    if constexpr (STAGED) {
                        // activations go to a shared-memory image of the two output rows ([row][octet][x][16 B], exactly
                        // their global layout) and leave with two bulk (TMA) stores per pair: 16 STS instead of 16 STG
                        if (a.act != nullptr && x < a.Wo) {
                            uint8_t* st = s_stage + j * L::STAGE_BYTES;
#pragma unroll
                            for (int cc = 0; cc < 4; ++cc) {
                                const int chunk = half * 4 + cc;
                                *reinterpret_cast<uint4*>(st + ((size_t)chunk * a.Wo + x) * 16) =
                                    make_uint4(h2u(a0[cc * 4]), h2u(a0[cc * 4 + 1]), h2u(a0[cc * 4 + 2]), h2u(a0[cc * 4 + 3]));
                                *reinterpret_cast<uint4*>(st + ((size_t)((COUT / 8) + chunk) * a.Wo + x) * 16) =
                                    make_uint4(h2u(a1[cc * 4]), h2u(a1[cc * 4 + 1]), h2u(a1[cc * 4 + 2]), h2u(a1[cc * 4 + 3]));
                            }
                        }
                    } else if (a.act != nullptr && x < a.Wo) {
#pragma unroll
                        for (int cc = 0; cc < 4; ++cc) {
                            const int chunk = half * 4 + cc;
                            uint4* d0 = reinterpret_cast<uint4*>(a.act) + (((size_t)b * a.Ho + t0) * (COUT / 8) + chunk) * a.Wo + x;
                            *d0 = make_uint4(h2u(a0[cc * 4]), h2u(a0[cc * 4 + 1]), h2u(a0[cc * 4 + 2]), h2u(a0[cc * 4 + 3]));
                            if (has1) {
                                uint4* d1 = d0 + (size_t)(COUT / 8) * a.Wo;
                                *d1 = make_uint4(h2u(a1[cc * 4]), h2u(a1[cc * 4 + 1]), h2u(a1[cc * 4 + 2]), h2u(a1[cc * 4 + 3]));
                            }
                        }
                    }
                    // 2x2 max-pool: vertical in registers, horizontal with the neighbouring lane
#pragma unroll
                    for (int q = 0; q < 16; ++q) {
                        const __half2 m = __hmax2(a0[q], a1[q]);
                        const uint32_t o = __shfl_xor_sync(0xffffffffu, h2u(m), 1);
                        a0[q] = __hmax2(m, *reinterpret_cast<const __half2*>(&o));
                    }
                    if (pool_ok) {
                        if (a.pool_fc != nullptr) {
                            // fc1 A-operand tile: [b/128][pooled pixel][b%128][128 B], chunk index XOR (row & 7)
                            const int row = b & 127;
                            uint8_t* base = a.pool_fc + ((((size_t)(b >> 7) * a.Hp * a.Wp) + (size_t)py * a.Wp + px) * 128 + row) * 128;
#pragma unroll
                            for (int cc = 0; cc < 4; ++cc) {
                                const int chunk = (half * 4 + cc) ^ (row & 7);
                                *reinterpret_cast<uint4*>(base + chunk * 16) =
                                    make_uint4(h2u(a0[cc * 4]), h2u(a0[cc * 4 + 1]), h2u(a0[cc * 4 + 2]), h2u(a0[cc * 4 + 3]));
                            }
                        }
                        if (a.pool_c8 != nullptr) {
#pragma unroll
                            for (int cc = 0; cc < 4; ++cc) {
                                const int chunk = half * 4 + cc;
                                uint4* d = reinterpret_cast<uint4*>(a.pool_c8) + (((size_t)b * a.Hp + py) * (COUT / 8) + chunk) * a.Wp + px;
                                *d = make_uint4(h2u(a0[cc * 4]), h2u(a0[cc * 4 + 1]), h2u(a0[cc * 4 + 2]), h2u(a0[cc * 4 + 3]));
                            }
                        }
                    }
                }
                if constexpr (!X3 && STAGED) {
                    if (a.act != nullptr) {
                        fence_proxy_async();                       // staged rows -> visible to the bulk-copy engine
                        named_bar_sync(1, 256);
                        if (tid == 64) {
                            const size_t row_bytes = (size_t)(COUT / 8) * a.Wo * 16;
                            uint8_t* gdst = reinterpret_cast<uint8_t*>(a.act) + ((size_t)b * a.Ho + t0) * row_bytes;
                            const uint8_t* st = s_stage + j * L::STAGE_BYTES;
                            bulk_s2g(gdst, st, (uint32_t)row_bytes);
                            if (has1) bulk_s2g(gdst + row_bytes, st + row_bytes, (uint32_t)row_bytes);
                            bulk_commit();
                        }
                    }
                }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&tempty[j]);
            }
        }
    }
    if (STAGED && tid == 64) bulk_wait<0>();         // staged rows must be read out before the CTA's smem goes away
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 4 * ACC);
}

template <int CIN, int COUT, bool X3>
static int launch_igemm_t(const IgemmArgs& a, int sms, cudaStream_t s) {
    using L = IgemmSmem<CIN, COUT>;
    BCAD_CUDA_CHECK(cudaFuncSetAttribute(conv_igemm_kernel<CIN, COUT, X3>, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL));
    const int items = a.B * a.bands * a.xsegs;
    const int grid = items < sms ? items : sms;
    conv_igemm_kernel<CIN, COUT, X3><<<grid, IG_THREADS, L::TOTAL, s>>>(a);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// Cin counts the channels the kernel sees: in fp16x3 mode that is 2 x the layer's channels (hi and lo octets)
int launch_conv_igemm(const IgemmArgs& a, int Cin, int Cout, bool x3, int sms, cudaStream_t s) {
    BCAD_REQUIRE(a.xsegs == cdiv(a.Wo, 128), "conv_igemm: xsegs must be ceil(Wo/128)");
    BCAD_REQUIRE(a.band_rows % 2 == 0, "conv_igemm: band_rows must be even");
    if (Cout == 64 && !x3) {
        if (Cin == 16) return launch_igemm_t<16, 64, false>(a, sms, s);
        if (Cin == 32) return launch_igemm_t<32, 64, false>(a, sms, s);
        if (Cin == 64) return launch_igemm_t<64, 64, false>(a, sms, s);
    }
    if (Cout == 64 && x3 && Cin == 64) return launch_igemm_t<64, 64, true>(a, sms, s);
    if (Cout == 32 && !x3 && Cin == 16) return launch_igemm_t<16, 32, false>(a, sms, s);      // tiny U-Net front, second conv (sm100_unet.cu)
    set_error("conv_igemm: Cin=%d Cout=%d x3=%d not supported", Cin, Cout, (int)x3);
    return BCAD_ERR_INVALID;
}

// =====================================================================================================
// fc1 as a split-K GEMM on tcgen05:  partial[split][m][n] = sum_{k in split} A[m][k] W[n][k]
//   CTA tile 128 (images) x N (units, <= 256) x 64 (one pooled pixel's channels) per k-block; both operands
//   arrive as ready-made SW128 tiles via one bulk copy each; 4-stage ring; warp roles as above.
// =====================================================================================================
constexpr int FC_STAGES = 4;
constexpr int FC_THREADS = 192;

__global__ void __launch_bounds__(FC_THREADS, 1) fc_splitk_kernel(FcArgs a) {
    if (a.n_dev != nullptr && *a.n_dev <= 0) return;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // dynamic smem base is 1024-aligned by declaration; SW128 tiles need it
    uint8_t* smem = smem_raw;
    const int a_tile = 128 * 128, w_tile = a.N * 128;
    const int nparts = a.x3 ? 2 : 1;                       // fp16x3: hi and lo tiles of both operands
    const int stage_bytes = nparts * (a_tile + w_tile);
    const int nst = a.x3 ? 2 : FC_STAGES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + nst * stage_bytes);
    uint64_t* full = bars;
    uint64_t* empty = bars + FC_STAGES;
    uint64_t* done = bars + 2 * FC_STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * FC_STAGES + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        for (int i = 0; i < FC_STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        mbar_init(done, 1);
        fence_barrier_init();
    }
    if (warp == 0) {
        tmem_alloc(tmem_slot, 256);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const int split = blockIdx.x, mt = blockIdx.y, cb = blockIdx.z;
    const int kb0 = split * a.kb_per_split, kb1 = min(a.nkb, kb0 + a.kb_per_split);
    const int nk = kb1 - kb0;

    if (warp == 0) {
        if (lane == 0) {
            for (int i = 0; i < nk; ++i) {
                const int st = i % nst;
                if (i >= nst) mbar_wait(&empty[st], ((i / nst) - 1) & 1);
                mbar_arrive_expect_tx(&full[st], stage_bytes);
                uint8_t* sa = smem + st * stage_bytes;
                const uint8_t* asrc = a.a_tiles + ((size_t)mt * a.nkb + kb0 + i) * (size_t)(nparts * a_tile);
                for (int off = 0; off < nparts * a_tile; off += 16384) bulk_g2s(sa + off, asrc + off, 16384, &full[st]);
                const uint8_t* wsrc = a.w_tiles + ((size_t)cb * a.nkb + kb0 + i) * (size_t)(nparts * w_tile);
                for (int off = 0; off < nparts * w_tile; off += 16384)
                    bulk_g2s(sa + nparts * a_tile + off, wsrc + off, min(16384, nparts * w_tile - off), &full[st]);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = make_idesc_f16(128, a.N);
            for (int i = 0; i < nk; ++i) {
                const int st = i % nst;
                mbar_wait(&full[st], (i / nst) & 1);
                tc_fence_after();
                const uint32_t sa = smem_u32(smem + st * stage_bytes), sw = sa + nparts * a_tile;
                // x3: A_hi.W_hi + A_lo.W_hi + A_hi.W_lo
                const int ngroups = a.x3 ? 3 : 1;
                for (int g3 = 0; g3 < ngroups; ++g3) {
                    const uint32_t sa_g = sa + (g3 == 1 ? a_tile : 0), sw_g = sw + (g3 == 2 ? w_tile : 0);
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint64_t ad = make_smem_desc(sa_g + k * 32, 16, 1024, LAYOUT_SW128);
                        const uint64_t bd = make_smem_desc(sw_g + k * 32, 16, 1024, LAYOUT_SW128);
                        umma_bf16(tmem, ad, bd, idesc, (i > 0 || k > 0 || g3 > 0) ? 1u : 0u);
                    }
                }
                umma_commit(&empty[st]);
            }
            umma_commit(done);
        }
    } else {
        const int quad = warp & 3;
        const int row = quad * 32 + lane;
        const size_t ld = a.ld_out > 0 ? (size_t)a.ld_out : (size_t)a.N;
        float* dst = a.partials + ((size_t)split * a.m_pad + (size_t)mt * 128 + row) * ld + (size_t)cb * a.N;
        const bool store = (a.m_valid <= 0) || (mt * 128 + row < a.m_valid);
        if (nk > 0) {
            mbar_wait(done, 0);
            tc_fence_after();
            for (int c0 = 0; c0 < a.N; c0 += 32) {
                float v[32];
                tmem_ld32(tmem + ((uint32_t)(quad * 32) << 16) + c0, v);
                tmem_ld_wait();
#pragma unroll
                for (int q = 0; q < 32; q += 4)
                    if (c0 + q < a.N && store)   // N is a multiple of 16, not necessarily of 32
                        *reinterpret_cast<float4*>(dst + c0 + q) = make_float4(v[q], v[q + 1], v[q + 2], v[q + 3]);
            }
        } else {
            for (int c0 = 0; c0 < a.N && store; c0 += 4) *reinterpret_cast<float4*>(dst + c0) = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 256);
}

int launch_fc_splitk(const FcArgs& a, cudaStream_t s) {
    BCAD_REQUIRE(a.N % 16 == 0 && a.N >= 16 && a.N <= 256, "fc_splitk: N=%d must be a multiple of 16 in 16..256", a.N);
    const int stage_bytes = (a.x3 ? 2 : 1) * (128 * 128 + a.N * 128);
    const int smem = (a.x3 ? 2 : FC_STAGES) * stage_bytes + 256;
    BCAD_CUDA_CHECK(cudaFuncSetAttribute(fc_splitk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    BCAD_REQUIRE(a.ncb <= 1 || a.splits == 1, "fc_splitk: column blocks need splits == 1");
    dim3 grid(a.splits, a.m_tiles, a.ncb > 1 ? a.ncb : 1);
    fc_splitk_kernel<<<grid, FC_THREADS, smem, s>>>(a);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// =====================================================================================================
// Grad-CAM channel weights of the PRE-activation target (the nn.Conv2d output that a hook on the reference torch CNN's last conv
// captures, ADCNNM.py:76) under first-index pooling, without the dense pooled gradient:
//   alpha_raw[b][k] = sum_q g[b][q][k] * (P[b][q][k] > 0 ? 1 : slope),     g[b][q][k] = sum_u dz1[b][u] W1[u][(q, k)]
// (only the window's first maximum receives g; LeakyReLU is monotone, so that element's z has the sign of the pooled P).
//   GEMM on tcgen05: M = 128 images, N = the 64 channels of one pooled pixel q, K = units.  A = dz1 tiles, resident for the CTA;
//   B = the fc1 forward tile of q ([unit][64 channels x 2 B], SW128) read MN-major -- no second copy of W1.
//   Epilogue: LeakyReLU' of each column from the pooled map (the fc1 A tiles: one 128-byte row per image and q), accumulated per
//   (image, channel) in registers over the CTA's range of q; partials [split][m_pad][64] -> alpha_preact_reduce (fixed order).
//   dz1 rows arrive scaled by 2^e and split into fp16 hi + lo parts (dz_rows_to_tiles): full precision whatever the gradient's
//   magnitude; the reduce undoes the scale exactly.  fp16: A_hi.W + A_lo.W (the W1 rounding the forward has is the only operand error);
//   fp16x3: A_hi.W_hi + A_lo.W_hi + A_hi.W_lo, the mask sign from hi + lo.
// Warp roles: 0 = bulk-copy producer, 1 = MMA issuer, 2..5 = epilogue (TMEM lane quadrant = warp % 4).
// =====================================================================================================
constexpr int PA_THREADS = 192;
constexpr int PA_ACC = 4;             // TMEM accumulator buffers of 64 columns: the epilogue of q overlaps the MMAs of q + 1 .. q + 3
constexpr int PA_MAXST = 4;           // W-tile ring stages (fewer when the resident dz1 tiles leave no room)

static int pa_nst(int units) {
    const int a_bytes = (units / 64) * 2 * 16384, w_bytes = units * 128;
    return std::min(PA_MAXST, (227 * 1024 - a_bytes - 256) / w_bytes);
}

__global__ void __launch_bounds__(PA_THREADS, 1) alpha_preact_kernel(PreactArgs a) {
    if (a.n_dev != nullptr && *a.n_dev <= 0) return;
    extern __shared__ __align__(1024) uint8_t smem[];
    const int parts = a.x3 ? 2 : 1;
    const int nkb = a.units / 64;
    const int a_bytes = nkb * 2 * 16384;           // resident dz1 tiles [kb][hi | lo][128 rows][128 B]
    const int w_bytes = a.units * 128;             // one W tile (q, part): [unit][64 channels]
    uint8_t* s_a = smem;
    uint8_t* s_w = smem + a_bytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(s_w + a.nst * w_bytes);
    uint64_t* full = bars;                         // [PA_MAXST] producer -> MMA
    uint64_t* empty = bars + PA_MAXST;             // [PA_MAXST] MMA -> producer
    uint64_t* tfull = bars + 2 * PA_MAXST;         // [PA_ACC] MMA -> epilogue
    uint64_t* tempty = tfull + PA_ACC;             // [PA_ACC] epilogue -> MMA (4 warps)
    uint64_t* abar = tempty + PA_ACC;              // resident A landed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(abar + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        for (int i = 0; i < PA_MAXST; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
        for (int i = 0; i < PA_ACC; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], 4); }
        mbar_init(abar, 1);
        fence_barrier_init();
    }
    if (warp == 0) {
        tmem_alloc(tmem_slot, 64 * PA_ACC);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const int mt = blockIdx.x, split = blockIdx.y;
    const int q0 = split * a.q_per_split, q1 = min(a.npix, q0 + a.q_per_split);
    const int nq = max(0, q1 - q0);

    if (warp == 0) {
        if (lane == 0) {
            mbar_arrive_expect_tx(abar, a_bytes);
            for (int off = 0; off < a_bytes; off += 16384)
                bulk_g2s(s_a + off, a.dz_tiles + (size_t)mt * a_bytes + off, 16384, abar);
            for (int i = 0; i < nq * parts; ++i) {
                const int st = i % a.nst, q = q0 + i / parts, p = i % parts;
                if (i >= a.nst) mbar_wait(&empty[st], ((i / a.nst) - 1) & 1);
                mbar_arrive_expect_tx(&full[st], w_bytes);
                const uint8_t* src = a.w_tiles + ((size_t)q * parts + p) * w_bytes;
                for (int off = 0; off < w_bytes; off += 16384)
                    bulk_g2s(s_w + st * w_bytes + off, src + off, min(16384, w_bytes - off), &full[st]);
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            // B MN-major (bit 16): the 64 channels of a unit are contiguous; SW128 atoms of 8 units x 128 B, SBO = 1024 B between them
            constexpr uint32_t idesc = (1u << 4) | (1u << 16) | ((uint32_t)(64 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
            const uint32_t sa = smem_u32(s_a);
            mbar_wait(abar, 0);
            for (int iq = 0; iq < nq; ++iq) {
                const int j = iq % PA_ACC;
                if (iq >= PA_ACC) mbar_wait(&tempty[j], ((iq / PA_ACC) - 1) & 1);
                tc_fence_after();
                uint32_t acc = 0;
                for (int p = 0; p < parts; ++p) {
                    const int i = iq * parts + p, st = i % a.nst;
                    mbar_wait(&full[st], (i / a.nst) & 1);
                    tc_fence_after();
                    const uint32_t sw = smem_u32(s_w + st * w_bytes);
                    const int na = (p == 0) ? 2 : 1;               // W (W_hi) meets A_hi and A_lo, W_lo meets A_hi
                    for (int ap = 0; ap < na; ++ap)
                        for (int kb = 0; kb < nkb; ++kb)
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                const uint64_t ad = make_smem_desc(sa + (kb * 2 + ap) * 16384 + k * 32, 16, 1024, LAYOUT_SW128);
                                const uint64_t bd = make_smem_desc(sw + kb * 8192 + k * 2048, 8192, 1024, LAYOUT_SW128);
                                umma_bf16(tmem + j * 64, ad, bd, idesc, acc);
                                acc = 1u;
                            }
                    umma_commit(&empty[st]);
                }
                umma_commit(&tfull[j]);
            }
        }
    } else {
        const int quad = warp & 3, row = quad * 32 + lane, sw = row & 7;
        const uint32_t lane_off = (uint32_t)(quad * 32) << 16;
        float acc[64];
#pragma unroll
        for (int c = 0; c < 64; ++c) acc[c] = 0.f;
        const uint8_t* mrow = a.mask_tiles + (size_t)mt * a.npix * parts * 16384 + (size_t)row * 128;
        for (int iq = 0; iq < nq; ++iq) {
            const int j = iq % PA_ACC;
            // LeakyReLU' of each channel at the window's maximum: bit c set <=> P > 0 (factor 1), else the slope
            const uint4* mh = reinterpret_cast<const uint4*>(mrow + (size_t)(q0 + iq) * parts * 16384);
            uint32_t pos0 = 0, pos1 = 0;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const uint4 h = ldg_stream_u4(mh + (c ^ sw));
                float2 f[4] = {unpack_f16(h.x), unpack_f16(h.y), unpack_f16(h.z), unpack_f16(h.w)};
                if (a.x3) {
                    const uint4 l = ldg_stream_u4(mh + 1024 + (c ^ sw));               // the lo tile, 16 KB further
                    const float2 g[4] = {unpack_f16(l.x), unpack_f16(l.y), unpack_f16(l.z), unpack_f16(l.w)};
#pragma unroll
                    for (int e = 0; e < 4; ++e) { f[e].x += g[e].x; f[e].y += g[e].y; }
                }
                uint32_t bits = 0;
#pragma unroll
                for (int e = 0; e < 4; ++e) bits |= ((f[e].x > 0.f) ? 1u : 0u) << (2 * e) | ((f[e].y > 0.f) ? 1u : 0u) << (2 * e + 1);
                if (c < 4) pos0 |= bits << (8 * c);
                else pos1 |= bits << (8 * (c - 4));
            }
            mbar_wait(&tfull[j], (iq / PA_ACC) & 1);
            tc_fence_after();
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                float d[32];
                tmem_ld32(tmem + lane_off + j * 64 + h * 32, d);
                tmem_ld_wait();
                const uint32_t pos = h ? pos1 : pos0;
#pragma unroll
                for (int c = 0; c < 32; ++c) acc[h * 32 + c] = fmaf(d[c], ((pos >> c) & 1u) ? 1.f : a.slope, acc[h * 32 + c]);
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[j]);
        }
        float4* dst = reinterpret_cast<float4*>(a.partials + ((size_t)split * a.m_pad + (size_t)mt * 128 + row) * 64);
#pragma unroll
        for (int c = 0; c < 16; ++c) dst[c] = make_float4(acc[4 * c], acc[4 * c + 1], acc[4 * c + 2], acc[4 * c + 3]);
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 64 * PA_ACC);
}

// alpha_raw[b][k] = 2^-e[b] * sum_s partial[s][b][k], splits in order
__global__ void alpha_preact_reduce_kernel(const float* __restrict__ part, int splits, size_t ld_split, const int* __restrict__ row_exp,
                                           float* __restrict__ alpha_raw, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * 64) return;
    float v = 0.f;
    for (int s = 0; s < splits; ++s) v += part[(size_t)s * ld_split + i];
    alpha_raw[i] = ldexpf(v, -row_exp[i / 64]);
}

bool alpha_preact_supported(int units, int C) { return C == 64 && units % 64 == 0 && units <= 256 && pa_nst(units) >= 2; }

int launch_alpha_preact(const PreactArgs& a0, int m_tiles, int splits, cudaStream_t s) {
    BCAD_REQUIRE(alpha_preact_supported(a0.units, 64), "alpha_preact: %d units (a multiple of 64 up to 256)", a0.units);
    PreactArgs a = a0;
    a.nst = pa_nst(a.units);
    const int smem = (a.units / 64) * 2 * 16384 + a.nst * a.units * 128 + 256;
    BCAD_CUDA_CHECK(cudaFuncSetAttribute(alpha_preact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    alpha_preact_kernel<<<dim3(m_tiles, splits), PA_THREADS, smem, s>>>(a);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

int launch_alpha_preact_reduce(const float* part, int splits, int m_pad, const int* row_exp, float* alpha_raw, int n, cudaStream_t s) {
    alpha_preact_reduce_kernel<<<cdiv(n * 64, 256), 256, 0, s>>>(part, splits, (size_t)m_pad * 64, row_exp, alpha_raw, n);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// dz1 rows [B][K] -> split fp16 SW128 A tiles as rows_to_fc_tiles_x3, each row first scaled by 2^e (exact; e -> row_exp) so that
// its largest magnitude lies in [2^14, 2^15): the hi part then carries 11 significant bits of the row's large elements for any
// gradient scale (a softmax gradient of a confident image can sit far below fp16's normal range).  One warp per row.
__global__ void __launch_bounds__(256) dz_rows_to_tiles_kernel(const float* __restrict__ src, uint8_t* __restrict__ tiles,
                                                               int* __restrict__ row_exp, int B, int K, int m_pad) {
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= m_pad) return;
    const int nkb = K / 64, items = nkb * 8;
    float mx = 0.f;
    for (int i = lane; i < items && row < B; i += 32) {
        const float4* p = reinterpret_cast<const float4*>(src + (size_t)row * K + i * 8);
        const float4 v0 = p[0], v1 = p[1];
        mx = fmaxf(mx, fmaxf(fmaxf(fmaxf(fabsf(v0.x), fabsf(v0.y)), fmaxf(fabsf(v0.z), fabsf(v0.w))),
                             fmaxf(fmaxf(fabsf(v1.x), fabsf(v1.y)), fmaxf(fabsf(v1.z), fabsf(v1.w)))));
    }
    mx = warp_max(mx);
    int e = 0;
    if (mx > 0.f && mx <= 3.4e38f) {
        int E;
        frexpf(mx, &E);
        e = 15 - E;
    }
    if (lane == 0) row_exp[row] = e;
    const int rr = row & 127;
    for (int i = lane; i < items; i += 32) {
        const int kb = i >> 3, ch = i & 7;
        float v[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) v[q] = (row < B) ? ldexpf(src[(size_t)row * K + i * 8 + q], e) : 0.f;
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const __half2 h = __floats2half2_rn(v[2 * q], v[2 * q + 1]);
            const float2 f = __half22float2(h);
            hi[q] = h2u(h);
            lo[q] = pack_f16(v[2 * q] - f.x, v[2 * q + 1] - f.y);
        }
        uint8_t* tile = tiles + (((size_t)(row >> 7) * nkb + kb) * 2) * (128 * 128);
        const int swz = (ch ^ (rr & 7)) * 16;
        *reinterpret_cast<uint4*>(tile + rr * 128 + swz) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4*>(tile + 128 * 128 + rr * 128 + swz) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    }
}

int launch_dz_rows_to_tiles(const float* src, uint8_t* tiles, int* row_exp, int B, int K, int m_pad, cudaStream_t s) {
    BCAD_REQUIRE(K % 64 == 0 && m_pad % 128 == 0, "dz_rows_to_tiles: K=%d m_pad=%d", K, m_pad);
    dz_rows_to_tiles_kernel<<<m_pad / 8, 256, 0, s>>>(src, tiles, row_exp, B, K, m_pad);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// fp32 rows [B][K] (K % 64 == 0) -> split fp16 SW128 A tiles [b/128][K/64][(hi|lo)][128][128 B]; rows >= B are zero
__global__ void rows_to_fc_tiles_x3_kernel(const float* __restrict__ src, uint8_t* __restrict__ tiles, int B, int K, int m_pad) {
    const int nkb = K / 64;
    const size_t total = (size_t)m_pad * nkb * 8;                 // (row, k-block, 16-byte chunk)
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int ch = (int)(i & 7);
        const size_t r = i >> 3;
        const int kb = (int)(r % nkb);
        const int row = (int)(r / nkb);
        float v[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = (row < B) ? src[(size_t)row * K + kb * 64 + ch * 8 + e] : 0.f;
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const __half2 h = __floats2half2_rn(v[2 * e], v[2 * e + 1]);
            const float2 f = __half22float2(h);
            hi[e] = h2u(h);
            lo[e] = pack_f16(v[2 * e] - f.x, v[2 * e + 1] - f.y);
        }
        const int rr = row & 127;
        uint8_t* tile = tiles + (((size_t)(row >> 7) * nkb + kb) * 2) * (128 * 128);
        const int sw = (ch ^ (rr & 7)) * 16;
        *reinterpret_cast<uint4*>(tile + rr * 128 + sw) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4*>(tile + 128 * 128 + rr * 128 + sw) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    }
}

int launch_rows_to_fc_tiles_x3(const float* src, uint8_t* tiles, int B, int K, int m_pad, cudaStream_t s) {
    BCAD_REQUIRE(K % 64 == 0 && m_pad % 128 == 0, "rows_to_fc_tiles: K=%d m_pad=%d", K, m_pad);
    const size_t total = (size_t)m_pad * (K / 64) * 8;
    rows_to_fc_tiles_x3_kernel<<<(int)std::min<size_t>(148 * 4, (total + 255) / 256), 256, 0, s>>>(src, tiles, B, K, m_pad);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// z[m][n] = sum_s partial[s][m][n] + bias[n] (fixed order), h = LeakyReLU(z); partial rows padded to m_pad
__global__ void fc_reduce_kernel(const float* __restrict__ part, int splits, size_t ld_split, const float* __restrict__ bias,
                                 float* __restrict__ z, float* __restrict__ h, float alpha, int M, int N) {
    const size_t total = (size_t)M * N;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        float v = 0.f;
        for (int s = 0; s < splits; ++s) v += part[(size_t)s * ld_split + i];
        v += __ldg(bias + (i % N));
        z[i] = v;
        if (h != nullptr) h[i] = leaky(v, alpha);
    }
}

int launch_fc_reduce(const float* part, int splits, size_t ld_split, const float* bias, float* z, float* h, float alpha,
                     int M, int N, cudaStream_t s) {
    const size_t total = (size_t)M * N;
    const int blocks = (int)min((size_t)2048, (total + 255) / 256);
    fc_reduce_kernel<<<blocks, 256, 0, s>>>(part, splits, ld_split, bias, z, h, alpha, M, N);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// =====================================================================================================
// Grad-CAM channel reduction on C8-planar fp16 activations: cam = ReLU(sum_k alpha_k A_k) + min/max partials
// grid (splits, B), 256 threads, thread = pixel; every load is a coalesced 16 B per lane.
// =====================================================================================================
template <bool X3, bool PRE>
__global__ void __launch_bounds__(256)
cam_c8_kernel(const __half* __restrict__ A, const float* __restrict__ alpha_raw, float scale,
              float* __restrict__ alpha_out, float* __restrict__ cam_lo, float* __restrict__ mm, int h, int w, int C,
              const int* __restrict__ n_dev, float inv_slope) {
    extern __shared__ float s_alpha[];
    __shared__ float s_min[8], s_max[8];
    const int b = blockIdx.y, split = blockIdx.x, splits = gridDim.x;
    if (n_dev != nullptr && b >= *n_dev) return;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const float t = alpha_raw[(size_t)b * C + c] * scale;
        s_alpha[c] = t;
        if (alpha_out != nullptr && split == 0) alpha_out[(size_t)b * C + c] = t;
    }
    __syncthreads();
    const int rows_per = cdiv(h, splits);
    const int y0 = split * rows_per, y1 = min(h, y0 + rows_per);
    const int chunks = C / 8;
    const int planes = X3 ? 2 * chunks : chunks;          // fp16x3: octets [hi | lo]
    float vmin = 3.4e38f, vmax = -3.4e38f;
    const uint4* base = reinterpret_cast<const uint4*>(A) + (size_t)b * h * planes * w;
    const int npix = (y1 - y0) * w;
    for (int i = threadIdx.x; i < npix; i += blockDim.x) {
        const int y = y0 + i / w, x = i % w;
        float acc = 0.f;
        const uint4* p = base + ((size_t)y * planes) * w + x;
        for (int c = 0; c < chunks; ++c) {
            const uint4 q = ldg_stream_u4(p + (size_t)c * w);
            const float* al = s_alpha + c * 8;
            float2 f0 = unpack_f16(q.x), f1 = unpack_f16(q.y), f2 = unpack_f16(q.z), f3 = unpack_f16(q.w);
            if constexpr (X3) {
                const uint4 ql = ldg_stream_u4(p + (size_t)(chunks + c) * w);
                const float2 g0 = unpack_f16(ql.x), g1 = unpack_f16(ql.y), g2 = unpack_f16(ql.z), g3 = unpack_f16(ql.w);
                f0.x += g0.x; f0.y += g0.y; f1.x += g1.x; f1.y += g1.y; f2.x += g2.x; f2.y += g2.y; f3.x += g3.x; f3.y += g3.y;
            }
            if constexpr (PRE) { f0 = unleaky2(f0, inv_slope); f1 = unleaky2(f1, inv_slope); f2 = unleaky2(f2, inv_slope); f3 = unleaky2(f3, inv_slope); }
            acc = fmaf(f0.x, al[0], acc); acc = fmaf(f0.y, al[1], acc);
            acc = fmaf(f1.x, al[2], acc); acc = fmaf(f1.y, al[3], acc);
            acc = fmaf(f2.x, al[4], acc); acc = fmaf(f2.y, al[5], acc);
            acc = fmaf(f3.x, al[6], acc); acc = fmaf(f3.y, al[7], acc);
        }
        acc = fmaxf(acc, 0.f);
        cam_lo[((size_t)b * h + y) * w + x] = acc;
        vmin = fminf(vmin, acc);
        vmax = fmaxf(vmax, acc);
    }
    vmin = warp_min(vmin);
    vmax = warp_max(vmax);
    if ((threadIdx.x & 31) == 0) { s_min[threadIdx.x >> 5] = vmin; s_max[threadIdx.x >> 5] = vmax; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int q = 1; q < 8; ++q) { vmin = fminf(vmin, s_min[q]); vmax = fmaxf(vmax, s_max[q]); }
        mm[((size_t)b * splits + split) * 2 + 0] = vmin;
        mm[((size_t)b * splits + split) * 2 + 1] = vmax;
    }
}

int launch_cam_c8(const __half* A, const float* alpha_raw, float scale, float* alpha_out, float* cam_lo, float* mm,
                  int B, int h, int w, int C, int splits, bool x3, cudaStream_t s, const int* n_dev, float inv_slope) {
    dim3 grid(splits, B);
    const size_t sm = C * sizeof(float);
    const bool pre = inv_slope > 0.f;
    if (x3 && pre) cam_c8_kernel<true, true><<<grid, 256, sm, s>>>(A, alpha_raw, scale, alpha_out, cam_lo, mm, h, w, C, n_dev, inv_slope);
    else if (x3) cam_c8_kernel<true, false><<<grid, 256, sm, s>>>(A, alpha_raw, scale, alpha_out, cam_lo, mm, h, w, C, n_dev, 0.f);
    else if (pre) cam_c8_kernel<false, true><<<grid, 256, sm, s>>>(A, alpha_raw, scale, alpha_out, cam_lo, mm, h, w, C, n_dev, inv_slope);
    else cam_c8_kernel<false, false><<<grid, 256, sm, s>>>(A, alpha_raw, scale, alpha_out, cam_lo, mm, h, w, C, n_dev, 0.f);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// Grad-CAM channel weights under the tie-duplicating pool rule, straight from the split (hi + lo) C8-planar activations:
//   alpha_raw[b][k] = sum over pool windows of g[b, window, k] * (number of window elements equal to the window maximum)
// (Classes/CNNModel.py:260,274-275: every tie receives the gradient; the dense map dA never exists).  g: fp32 NHWC pooled
// gradient [B][Hp][Wp][C].  One CTA per image, warp = channel octet (C = 64: 8 warps), lanes across windows; the activation value
// is hi + lo in fp32 -- the same number c8_to_nhwc_kernel reports, so the equality structure is the one the tests see.
__global__ void __launch_bounds__(256) alpha_ties_c8_kernel(const __half* __restrict__ A, const float* __restrict__ g,
                                                            float* __restrict__ alpha_raw, int h, int w, int C, float pre_slope) {
    const int octets = C / 8, planes = 2 * octets;
    const int Hp = h / 2, Wp = w / 2;
    const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const uint4* base = reinterpret_cast<const uint4*>(A) + (size_t)b * h * planes * w;
    const float* gb = g + (size_t)b * Hp * Wp * C;
    for (int o = warp; o < octets; o += nwarps) {
        float acc[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = 0.f;
        for (int wy = 0; wy < Hp; ++wy)
            for (int wx = lane; wx < Wp; wx += 32) {
                float v[4][8];
#pragma unroll
                for (int r = 0; r < 2; ++r)
#pragma unroll
                    for (int cx = 0; cx < 2; ++cx) {
                        const uint4* p = base + ((size_t)(2 * wy + r) * planes + o) * w + 2 * wx + cx;
                        const uint4 qh = ldg_stream_u4(p), ql = ldg_stream_u4(p + (size_t)octets * w);
                        const float2 h0 = unpack_f16(qh.x), h1 = unpack_f16(qh.y), h2 = unpack_f16(qh.z), h3 = unpack_f16(qh.w);
                        const float2 l0 = unpack_f16(ql.x), l1 = unpack_f16(ql.y), l2 = unpack_f16(ql.z), l3 = unpack_f16(ql.w);
                        float* d = v[r * 2 + cx];
                        d[0] = h0.x + l0.x; d[1] = h0.y + l0.y; d[2] = h1.x + l1.x; d[3] = h1.y + l1.y;
                        d[4] = h2.x + l2.x; d[5] = h2.y + l2.y; d[6] = h3.x + l3.x; d[7] = h3.y + l3.y;
                    }
                const float4 g0 = __ldg(reinterpret_cast<const float4*>(gb + ((size_t)wy * Wp + wx) * C + o * 8));
                const float4 g1 = __ldg(reinterpret_cast<const float4*>(gb + ((size_t)wy * Wp + wx) * C + o * 8) + 1);
                const float gv[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const float m = fmaxf(fmaxf(v[0][j], v[1][j]), fmaxf(v[2][j], v[3][j]));
                    const int cnt = (v[0][j] == m) + (v[1][j] == m) + (v[2][j] == m) + (v[3][j] == m);
                    float f = (float)cnt;
                    if (pre_slope >= 0.f && !(m > 0.f)) f *= pre_slope;       // every tie holds the window's value: one LeakyReLU'
                    acc[j] = fmaf(gv[j], f, acc[j]);
                }
            }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float t = warp_sum(acc[j]);
            if (lane == 0) alpha_raw[(size_t)b * C + o * 8 + j] = t;
        }
    }
}

int launch_alpha_ties_c8(const __half* A, const float* g, float* alpha_raw, int B, int h, int w, int C, cudaStream_t s, float pre_slope) {
    BCAD_REQUIRE(C % 8 == 0, "alpha_ties_c8: channel count %d", C);
    alpha_ties_c8_kernel<<<B, 256, 0, s>>>(A, g, alpha_raw, h, w, C, pre_slope);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// C8-planar fp16 [B][h][C/8][w][8] (fp16x3: octets [hi | lo]) -> NHWC fp32.  thread = (pixel, channel octet), octet fastest: a
// warp writes 1 KB of contiguous output and reads 64 contiguous bytes from each plane (inspection calls and the fp32 tail of the
// tie-duplicating mode)
__global__ void __launch_bounds__(256) c8_to_nhwc_kernel(const __half* __restrict__ src, float* __restrict__ dst, int w, int C, int x3,
                                                         size_t rows) {
    const int octets = C / 8, planes = (x3 ? 2 : 1) * octets;
    const size_t per_row = (size_t)octets * w, total = rows * per_row;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t row = i / per_row;
        const int rem = (int)(i - row * per_row);
        const int x = rem / octets, o = rem - x * octets;          // octet fastest: a warp writes 1 KB of contiguous NHWC floats
        const uint4* base = reinterpret_cast<const uint4*>(src) + (row * planes) * w;
        const uint4 q = ldg_stream_u4(base + (size_t)o * w + x);
        float2 f0 = unpack_f16(q.x), f1 = unpack_f16(q.y), f2 = unpack_f16(q.z), f3 = unpack_f16(q.w);
        if (x3) {
            const uint4 ql = ldg_stream_u4(base + (size_t)(octets + o) * w + x);
            const float2 g0 = unpack_f16(ql.x), g1 = unpack_f16(ql.y), g2 = unpack_f16(ql.z), g3 = unpack_f16(ql.w);
            f0.x += g0.x; f0.y += g0.y; f1.x += g1.x; f1.y += g1.y; f2.x += g2.x; f2.y += g2.y; f3.x += g3.x; f3.y += g3.y;
        }
        float4* out = reinterpret_cast<float4*>(dst + (row * w + x) * C + o * 8);
        out[0] = make_float4(f0.x, f0.y, f1.x, f1.y);
        out[1] = make_float4(f2.x, f2.y, f3.x, f3.y);
    }
}

int launch_c8_to_nhwc(const __half* src, float* dst, int B, int h, int w, int C, bool x3, cudaStream_t s) {
    const size_t total = (size_t)B * h * w * (C / 8);
    const int blocks = (int)min((size_t)148 * 16, (total + 255) / 256);
    c8_to_nhwc_kernel<<<blocks, 256, 0, s>>>(src, dst, w, C, x3 ? 1 : 0, (size_t)B * h);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

}  // namespace bcad
