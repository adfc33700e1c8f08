// Input-gradient saliency (explainability.py:44-78): the first conv block's input gradient, s = max_c |d_input| and its per-image
// min-max normalisation, for bcad_predict_saliency_classes.  The overlay kernel sits beside overlay_kernel in kernels_fp32.cu.
#include "common.cuh"
#include "kernels.h"

namespace bcad {

// ---------------------------------------------------------------------------------------------------------------------------------
// First block of the canonical shape (one input channel, 32 filters, 3x3, pad 0 or 1): pool backward + LeakyReLU' + input gradient in
// ONE pass.  The 32-channel full-resolution gradient dz0 is never written.
//   d_input[iy][ix] = sum_{ky,kx,f} dz0[iy - ky + pad][ix - kx + pad][f] * w[ky][kx][f]
// A pool window (2x2 outputs) touches a 4x4 input patch.  Per window, a warp (lane = filter) routes g to the window's maximum as
// conv0_bwd_fused_kernel does, forms its filter's 16 patch contributions, and sums them over the 32 filters with a 16-shuffle
// reduce-scatter (lane L ends with element L >> 1).  The patches of a CTA's windows go to shared memory; every input pixel then sums
// the (at most) four patches that cover it in a fixed order.  CTA = a tile of SC_TY x SC_TX windows plus one halo window row above and
// one column to the left; it owns the input pixels whose lower-right covering window lies in the tile.  No float atomics: the results
// are the same run to run.  Per-image min / max of s = |d_input| go through integer atomicMax on the bits of the non-negative values
// (exact); the minimum is kept as the maximum of the complemented bits so that both counters start at 0.
// ---------------------------------------------------------------------------------------------------------------------------------
constexpr int SC_TY = 8, SC_TX = 32, SC_WARPS = 8, SC_PITCH = 17;

__global__ void __launch_bounds__(32 * SC_WARPS) saliency_conv0_kernel(const float* __restrict__ g, const float* __restrict__ y,
                                                                      const float* __restrict__ w, int H, int W, int Ho, int Wo, int pad,
                                                                      int first_only, float alpha, float* __restrict__ d_input,
                                                                      float* __restrict__ sal, size_t out_stride, uint32_t* __restrict__ mm,
                                                                      int mm_ld) {
    __shared__ float s_p[(SC_TY + 1) * (SC_TX + 1) * SC_PITCH];
    const int Hp = Ho / 2, Wp = Wo / 2;
    const int b = blockIdx.z, wy0 = blockIdx.y * SC_TY, wx0 = blockIdx.x * SC_TX;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float wt[9];
#pragma unroll
    for (int t = 0; t < 9; ++t) wt[t] = __ldg(w + t * 32 + lane);              // packed [tap][Cin = 1][CoutPad = 32]
    const float* gb = g + (size_t)b * Hp * Wp * 32 + lane;
    const float* yb = y + (size_t)b * Ho * Wo * 32 + lane;
    for (int u = warp; u < (SC_TY + 1) * (SC_TX + 1); u += SC_WARPS) {
        const int wy = wy0 - 1 + u / (SC_TX + 1), wx = wx0 - 1 + u % (SC_TX + 1);
        float v = 0.f;
        if (wy >= 0 && wy < Hp && wx >= 0 && wx < Wp) {                        // warp-uniform
            const float gv = __ldg(gb + ((size_t)wy * Wp + wx) * 32);
            const float* y0 = yb + ((size_t)(2 * wy) * Wo + 2 * wx) * 32;
            const float a0 = __ldg(y0), a1 = __ldg(y0 + 32), a2 = __ldg(y0 + (size_t)Wo * 32), a3 = __ldg(y0 + (size_t)Wo * 32 + 32);
            const float m = fmaxf(fmaxf(a0, a1), fmaxf(a2, a3));
            bool s0 = (a0 == m), s1 = (a1 == m), s2 = (a2 == m), s3 = (a3 == m);
            if (first_only) { s1 = s1 && !s0; s2 = s2 && !(s0 || s1); s3 = s3 && !(s0 || s1 || s2); }
            float d[4];
            d[0] = (s0 ? gv : 0.f) * (a0 > 0.f ? 1.f : alpha);
            d[1] = (s1 ? gv : 0.f) * (a1 > 0.f ? 1.f : alpha);
            d[2] = (s2 ? gv : 0.f) * (a2 > 0.f ? 1.f : alpha);
            d[3] = (s3 ? gv : 0.f) * (a3 > 0.f ? 1.f : alpha);
            float pt[16];                                                        // patch row r = input row 2 wy - pad + r
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    float acc = 0.f;
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const int ky = r - (q >> 1), kx = c - (q & 1);
                        if (ky >= 0 && ky < 3 && kx >= 0 && kx < 3) acc = fmaf(d[q], wt[ky * 3 + kx], acc);
                    }
                    pt[r * 4 + c] = acc;
                }
            // reduce-scatter over the 32 lanes: each step halves the elements a lane keeps (8 + 4 + 2 + 1 shuffles), a last exchange
            // with the neighbour lane completes the sum (both lanes of a pair hold the same element)
#pragma unroll
            for (int half = 8, bit = 16; half >= 1; half >>= 1, bit >>= 1) {
                const bool hi = (lane & bit) != 0;
#pragma unroll
                for (int j = 0; j < half; ++j) {
                    const float mine = hi ? pt[half + j] : pt[j], other = hi ? pt[j] : pt[half + j];
                    pt[j] = mine + __shfl_xor_sync(0xffffffffu, other, bit);
                }
            }
            v = pt[0] + __shfl_xor_sync(0xffffffffu, pt[0], 1);
        }
        if ((lane & 1) == 0) s_p[u * SC_PITCH + (lane >> 1)] = v;
    }
    __syncthreads();
    // owned input pixels: rows whose covering windows are {q - 1, q}, q = (iy + pad) / 2 in [wy0, wy0 + SC_TY); the first tile row /
    // column also owns the leading border, the last one everything up to the image edge (windows outside the map contribute 0)
    const int iy_lo = wy0 == 0 ? 0 : 2 * wy0 - pad, ix_lo = wx0 == 0 ? 0 : 2 * wx0 - pad;
    const int iy_hi = wy0 + SC_TY >= Hp ? H : 2 * (wy0 + SC_TY) - pad, ix_hi = wx0 + SC_TX >= Wp ? W : 2 * (wx0 + SC_TX) - pad;
    const int iw = ix_hi - ix_lo, npx = (iy_hi - iy_lo) * iw;
    uint32_t vmax = 0u, vmin_c = 0u;
    float* db = d_input ? d_input + (size_t)b * out_stride : nullptr;
    float* sb = sal + (size_t)b * out_stride;
    for (int i = threadIdx.x; i < npx; i += blockDim.x) {
        const int iy = iy_lo + i / iw, ix = ix_lo + i % iw;
        const int qy = (iy + pad) >> 1, qx = (ix + pad) >> 1;
        float acc = 0.f;
#pragma unroll
        for (int t = 0; t < 4; ++t) {                                          // (q-1, q-1), (q-1, q), (q, q-1), (q, q)
            const int wy = qy - 1 + (t >> 1), wx = qx - 1 + (t & 1);
            if (wy >= 0 && wy < Hp && wx >= 0 && wx < Wp) {
                const int r = iy + pad - 2 * wy, c = ix + pad - 2 * wx;
                acc += s_p[((wy - wy0 + 1) * (SC_TX + 1) + (wx - wx0 + 1)) * SC_PITCH + r * 4 + c];
            }
        }
        const size_t o = (size_t)iy * W + ix;
        if (db) db[o] = acc;
        const float sv = fabsf(acc);
        sb[o] = sv;
        const uint32_t bits = __float_as_uint(sv);
        vmax = max(vmax, bits);
        vmin_c = max(vmin_c, ~bits);
    }
    vmax = __reduce_max_sync(0xffffffffu, vmax);
    vmin_c = __reduce_max_sync(0xffffffffu, vmin_c);
    if (lane == 0 && (vmax | vmin_c) != 0u) {
        atomicMax(mm + (size_t)b * mm_ld, vmax);
        atomicMax(mm + (size_t)b * mm_ld + 1, vmin_c);
    }
}

// Any other first block: its input gradient comes from conv_fp32 (d [n][HW][C]); s = max_c |d| per pixel, the per-image min / max as
// above, and d copied to the caller's strided [B][K][H][W][C] layout when wanted.
__global__ void saliency_absmax_kernel(const float* __restrict__ d, int hw, int C, float* __restrict__ d_input, float* __restrict__ sal,
                                       size_t out_stride, uint32_t* __restrict__ mm, int mm_ld) {
    const int b = blockIdx.y;
    const float* src = d + (size_t)b * hw * C;
    uint32_t vmax = 0u, vmin_c = 0u;
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < hw; p += gridDim.x * blockDim.x) {
        float sv = 0.f;
        for (int c = 0; c < C; ++c) {
            const float v = src[(size_t)p * C + c];
            sv = fmaxf(sv, fabsf(v));
            if (d_input) d_input[(size_t)b * out_stride * C + (size_t)p * C + c] = v;
        }
        sal[(size_t)b * out_stride + p] = sv;
        const uint32_t bits = __float_as_uint(sv);
        vmax = max(vmax, bits);
        vmin_c = max(vmin_c, ~bits);
    }
    vmax = __reduce_max_sync(0xffffffffu, vmax);
    vmin_c = __reduce_max_sync(0xffffffffu, vmin_c);
    if ((threadIdx.x & 31) == 0 && (vmax | vmin_c) != 0u) {
        atomicMax(mm + (size_t)b * mm_ld, vmax);
        atomicMax(mm + (size_t)b * mm_ld + 1, vmin_c);
    }
}

// (s - min s) / (max s - min s + 1e-8) in place, map m = image * K + class (explainability.py:73)
__global__ void saliency_norm_kernel(float* __restrict__ sal, int maps, int hw, const uint32_t* __restrict__ mm) {
    for (int map = blockIdx.y; map < maps; map += gridDim.y) {
        const float mx = __uint_as_float(mm[2 * map]), mn = __uint_as_float(~mm[2 * map + 1]);
        const float den = (mx - mn) + 1e-8f;
        float* sm = sal + (size_t)map * hw;
        for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < hw; p += gridDim.x * blockDim.x) sm[p] = (sm[p] - mn) / den;
    }
}

bool saliency_conv0_supported(int Cin, int Cout, int CoutPad, int k, int pad) {
    return Cin == 1 && Cout == 32 && CoutPad == 32 && k == 3 && (pad == 0 || pad == 1);
}

int launch_saliency_conv0(const float* g, const float* y, const float* w, int B, int H, int W, int Ho, int Wo, int pad, int first_only,
                          float alpha, float* d_input, float* sal, size_t out_stride, uint32_t* mm, int mm_ld, cudaStream_t s) {
    BCAD_REQUIRE(pad == 0 || pad == 1, "saliency_conv0: pad %d (0 or 1 supported)", pad);
    BCAD_REQUIRE(B <= 65535, "saliency_conv0: batch %d too large", B);
    const dim3 grid(cdiv(Wo / 2, SC_TX), cdiv(Ho / 2, SC_TY), B);
    saliency_conv0_kernel<<<grid, 32 * SC_WARPS, 0, s>>>(g, y, w, H, W, Ho, Wo, pad, first_only, alpha, d_input, sal, out_stride, mm, mm_ld);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

int launch_saliency_absmax(const float* d, int B, int hw, int C, float* d_input, float* sal, size_t out_stride, uint32_t* mm, int mm_ld,
                           cudaStream_t s) {
    const dim3 grid(std::min(cdiv(hw, 256), 64), B);
    saliency_absmax_kernel<<<grid, 256, 0, s>>>(d, hw, C, d_input, sal, out_stride, mm, mm_ld);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

int launch_saliency_norm(float* sal, int maps, int hw, const uint32_t* mm, cudaStream_t s) {
    const dim3 grid(std::min(cdiv(hw, 256), 64), std::min(maps, 65535));
    saliency_norm_kernel<<<grid, 256, 0, s>>>(sal, maps, hw, mm);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

}  // namespace bcad
