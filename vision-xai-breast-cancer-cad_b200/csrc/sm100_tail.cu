// Fused Grad-CAM tail of the tensor path: one thread-block CLUSTER of CL CTAs per image.
//
//   cam = ReLU(sum_k alpha_k A_k)            (HBM-bound: A is read exactly once, 16-byte coalesced streaming loads)
//   min-max -> bilinear resize (OpenCV order: horizontal, then vertical) -> min-max     (shared-memory bound)
//
// (pytorch_grad_cam semantics as restated in oracle/gradcam.py; call sites GRADCAM.py:53,64.)  Each CTA owns a band of the
// low-resolution rows: the low-resolution map never leaves shared memory; the per-band min/max pairs and the one halo row a
// band needs from the next one travel through distributed shared memory; and with ~105 KB of shared memory per CTA (CL = 2)
// two CTAs of different images share an SM, so the HBM phase of one overlaps the interpolation phase of the other.
// Arithmetic is the same sequence of fp32 operations as cam_c8_kernel + upsample_norm_sep_kernel (bit-identical maps).
//
// K target classes per launch (bcad_predict_explain_classes, profiling name tail_fused_classes): phase 1 streams every 16-byte
// octet of A once and keeps K fmaf chains per pixel, each in the channel order of the one-class kernel, so class k's map is
// bit-identical to a one-class launch with alpha_k.  The K low-resolution bands stay in shared memory; phases 2-3 run per class
// and reuse the one s_hr buffer.  Shared memory grows by (K - 1) * hh * w floats: at K = 2 on the canonical map (64 x 128 x 128
// -> 256 x 256) a 2-CTA cluster would need ~139 KB per CTA, one CTA per SM, and the HBM phase of one image could no longer
// hide behind the interpolation of another.  The K = 2 kernel therefore runs 4-CTA clusters of 256 threads (hh = 32: ~73 KB,
// three CTAs per SM); the 2 x 512 form at K = 2 has not been measured against it.  Measured at 512 x (64 x 128 x 128 -> 256 x 256),
// fp16, B200 at 1000 W: 0.348 ms for both classes against 0.226 ms for one (profiles/r03_multiclass_1gpu.json).  Larger K is cut
// into groups of TF_GROUP classes, each group one read of A.
#include <cooperative_groups.h>

#include "../../include/bcad.h"
#include "common.cuh"
#include "sm100_kernels.h"

namespace bcad {

namespace cg = cooperative_groups;


template <int NT>
__device__ __forceinline__ void tf_block_minmax(float& vmin, float& vmax, float* s_red) {
    vmin = warp_min(vmin);
    vmax = warp_max(vmax);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) { s_red[threadIdx.x >> 5] = vmin; s_red[32 + (threadIdx.x >> 5)] = vmax; }
    __syncthreads();
    vmin = s_red[0];
    vmax = s_red[32];
    for (int q = 1; q < NT / 32; ++q) { vmin = fminf(vmin, s_red[q]); vmax = fmaxf(vmax, s_red[32 + q]); }
}

// CL = CTAs per image (cluster size), NT = threads per CTA, K = target classes (alpha_raw + k * alpha_ld, the H x W map of class k
// of image b at out + b * out_stride + k * H * W)
// PRE: the pre-activation target, z = a > 0 ? a : a * inv_slope before the channel reduction (the post-activation instantiations are
// unchanged)
template <bool X3, int CL, int NT, int K, bool PRE>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(NT, 1024 / NT)
tail_fused_kernel(const __half* __restrict__ A, const float* __restrict__ alpha_raw, size_t alpha_ld, float scale, float* __restrict__ alpha_out,
                  float* __restrict__ out, size_t out_stride, int h, int w, int H, int W, int C, const int* __restrict__ n_dev, float inv_slope) {
    cg::cluster_group cluster = cg::this_cluster();
    const int rank = (int)cluster.block_rank();
    const int b = blockIdx.x / CL;
    if (n_dev != nullptr && b >= *n_dev) return;          // (every CTA of the image's cluster leaves together)
    constexpr int TF_THREADS = NT;
    extern __shared__ __align__(16) float sm[];
    __shared__ float s_red[64];
    __shared__ float s_mm[4 * K];             // per class: [0..1] min/max of my band of the cam, [2..3] of my band of the resized map
    __shared__ int s_cnt[CL];                 // output rows whose upper source row belongs to rank r
    const int hh = (h + CL - 1) / CL;         // rank r owns low-res rows [r * hh, min(h, (r + 1) * hh))
    const int r0 = min(h, rank * hh), nr = min(h, r0 + hh) - r0;
    int* s_x0 = reinterpret_cast<int*>(sm);
    int* s_x1 = s_x0 + W;
    float* s_fx = sm + 2 * W;
    int* s_y0 = reinterpret_cast<int*>(sm + 3 * W);
    int* s_y1 = s_y0 + H;
    float* s_fy = sm + 3 * W + 2 * H;
    const int cpad = (C + 3) & ~3;
    float* s_alpha = sm + 3 * W + 3 * H;      // [K][cpad]
    float* s_lo = s_alpha + K * cpad;         // [K][hh][w] my rows of the raw cam
    float* s_hr = s_lo + K * hh * w;          // [hh + 1][W] horizontally interpolated rows (+ the halo row)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = TF_THREADS / 32;

    if (tid < CL) s_cnt[tid] = 0;
#pragma unroll
    for (int k = 0; k < K; ++k)
        for (int c = tid; c < C; c += TF_THREADS) {
            const float t = alpha_raw[k * alpha_ld + (size_t)b * C + c] * scale;
            s_alpha[k * cpad + c] = t;
            if (alpha_out != nullptr && rank == 0) alpha_out[(size_t)b * C + c] = t;
        }
    __syncthreads();
    // coordinate tables: source coordinate in double, weight = float(frac) (oracle/gradcam.py, pinned to cv2)
    for (int d = tid; d < W + H; d += TF_THREADS) {
        const bool isx = d < W;
        const int dd = isx ? d : d - W;
        const int ns = isx ? w : h, nd = isx ? W : H;
        const double sc = ((double)dd + 0.5) * ((double)ns / (double)nd) - 0.5;
        int i0 = (int)floor(sc);
        float f = (float)(sc - (double)i0);
        if (i0 < 0) { i0 = 0; f = 0.f; }
        if (i0 >= ns - 1) { i0 = ns - 1; f = 0.f; }
        const int i1 = min(i0 + 1, ns - 1);
        if (isx) { s_x0[dd] = i0; s_x1[dd] = i1; s_fx[dd] = f; }
        else {
            s_y0[dd] = i0; s_y1[dd] = i1; s_fy[dd] = f;
            atomicAdd(&s_cnt[i0 / hh], 1);                // i0 is non-decreasing in dd: the counts give each rank's row range
        }
    }
    // ---- phase 1: channel reduction over my rows (one warp per row, lanes across pixels)
    const int chunks = C / 8;
    const int planes = X3 ? 2 * chunks : chunks;          // fp16x3: octets [hi | lo]
    const uint4* base = reinterpret_cast<const uint4*>(A) + (size_t)b * h * planes * w;
    float vmin[K], vmax[K];
#pragma unroll
    for (int k = 0; k < K; ++k) { vmin[k] = 3.4e38f; vmax[k] = -3.4e38f; }
    for (int lr = warp; lr < nr; lr += NW) {
        const uint4* prow = base + ((size_t)(r0 + lr) * planes) * w;
        for (int x = lane; x < w; x += 32) {
            float acc[K];
#pragma unroll
            for (int k = 0; k < K; ++k) acc[k] = 0.f;
            const uint4* p = prow + x;
            for (int c = 0; c < chunks; ++c) {
                const uint4 q = ldg_stream_u4(p + (size_t)c * w);
                float2 f0 = unpack_f16(q.x), f1 = unpack_f16(q.y), f2 = unpack_f16(q.z), f3 = unpack_f16(q.w);
                if constexpr (X3) {
                    const uint4 ql = ldg_stream_u4(p + (size_t)(chunks + c) * w);
                    const float2 g0 = unpack_f16(ql.x), g1 = unpack_f16(ql.y), g2 = unpack_f16(ql.z), g3 = unpack_f16(ql.w);
                    f0.x += g0.x; f0.y += g0.y; f1.x += g1.x; f1.y += g1.y; f2.x += g2.x; f2.y += g2.y; f3.x += g3.x; f3.y += g3.y;
                }
                if constexpr (PRE) { f0 = unleaky2(f0, inv_slope); f1 = unleaky2(f1, inv_slope); f2 = unleaky2(f2, inv_slope); f3 = unleaky2(f3, inv_slope); }
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    const float* al = s_alpha + k * cpad + c * 8;
                    float a = acc[k];
                    a = fmaf(f0.x, al[0], a); a = fmaf(f0.y, al[1], a);
                    a = fmaf(f1.x, al[2], a); a = fmaf(f1.y, al[3], a);
                    a = fmaf(f2.x, al[4], a); a = fmaf(f2.y, al[5], a);
                    a = fmaf(f3.x, al[6], a); a = fmaf(f3.y, al[7], a);
                    acc[k] = a;
                }
            }
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const float a = fmaxf(acc[k], 0.f);
                s_lo[(k * hh + lr) * w + x] = a;
                vmin[k] = fminf(vmin[k], a);
                vmax[k] = fmaxf(vmax[k], a);
            }
        }
    }
#pragma unroll
    for (int k = 0; k < K; ++k) {
        tf_block_minmax<NT>(vmin[k], vmax[k], s_red);
        if (tid == 0) { s_mm[4 * k] = vmin[k]; s_mm[4 * k + 1] = vmax[k]; }
    }
    cluster.sync();                                        // every band of the cam and its min/max are in shared memory
    int oy_lo = 0;
    for (int r = 0; r < rank; ++r) oy_lo += s_cnt[r];
    const int oy_hi = oy_lo + s_cnt[rank];
    const int nhr = nr + ((nr > 0 && r0 + nr < h) ? 1 : 0);
#pragma unroll
    for (int k = 0; k < K; ++k) {
    if (k > 0) __syncthreads();                            // the previous class's stores have finished reading s_hr
    float mn = vmin[k], mx = vmax[k];
#pragma unroll
    for (int r = 0; r < CL; ++r) {
        const float* pm = cluster.map_shared_rank(s_mm, r);
        mn = fminf(mn, pm[4 * k]);
        mx = fmaxf(mx, pm[4 * k + 1]);
    }
    const float* my_lo = s_lo + k * hh * w;
    const float* peer_lo = cluster.map_shared_rank(my_lo, min(rank + 1, CL - 1));    // first row of the next rank = my halo row
    const float inv = 1.f / (1e-7f + (mx - mn));
    // ---- phase 2: horizontal interpolation of my rows (+ the first row of the next rank, read through DSMEM)
    for (int lr = warp; lr < nhr; lr += NW) {
        const float* src = (lr < nr) ? my_lo + lr * w : peer_lo;
        float* dst = s_hr + lr * W;
#pragma unroll 4
        for (int ox = lane; ox < W; ox += 32) {
            const float fx = s_fx[ox];
            const float a0 = (src[s_x0[ox]] - mn) * inv, a1 = (src[s_x1[ox]] - mn) * inv;
            dst[ox] = a0 * (1.f - fx) + a1 * fx;
        }
    }
    __syncthreads();
    // ---- phase 3: vertical interpolation of my output rows, min-max, normalise, store
    float wmin = 3.4e38f, wmax = -3.4e38f;
    for (int oy = oy_lo + warp; oy < oy_hi; oy += NW) {
        const float fy = s_fy[oy], gy = 1.f - fy;
        const float* q0 = s_hr + (s_y0[oy] - r0) * W;
        const float* q1 = s_hr + (s_y1[oy] - r0) * W;
#pragma unroll 4
        for (int ox = lane; ox < W; ox += 32) {
            const float v = q0[ox] * gy + q1[ox] * fy;
            wmin = fminf(wmin, v);
            wmax = fmaxf(wmax, v);
        }
    }
    tf_block_minmax<NT>(wmin, wmax, s_red);
    if (tid == 0) { s_mm[4 * k + 2] = wmin; s_mm[4 * k + 3] = wmax; }
    cluster.sync();                                        // (also: the peer has finished reading my cam rows)
#pragma unroll
    for (int r = 0; r < CL; ++r) {
        const float* pm = cluster.map_shared_rank(s_mm, r);
        wmin = fminf(wmin, pm[4 * k + 2]);
        wmax = fmaxf(wmax, pm[4 * k + 3]);
    }
    const float inv2 = 1.f / (1e-7f + (wmax - wmin));      // x / d evaluated as x * (1/d), as upsample_norm_sep_kernel
    float* ob = out + (size_t)b * out_stride + (size_t)k * H * W;
    for (int oy = oy_lo + warp; oy < oy_hi; oy += NW) {
        const float fy = s_fy[oy], gy = 1.f - fy;
        const float* q0 = s_hr + (s_y0[oy] - r0) * W;
        const float* q1 = s_hr + (s_y1[oy] - r0) * W;
        float* orow = ob + (size_t)oy * W;
#pragma unroll 4
        for (int ox = lane; ox < W; ox += 32) orow[ox] = ((q0[ox] * gy + q1[ox] * fy) - wmin) * inv2;
    }
    }
    cluster.sync();                                        // my shared memory stays valid until the peer has read s_mm
}

// measured at 512 x (64 x 128 x 128 -> 256 x 256): 2 CTAs x 512 threads 0.227 ms, 4 CTAs x 256 threads 0.238 ms
// (cam_c8_kernel + upsample_norm_sep_kernel: 0.254 ms)
constexpr int TF_CL = 2, TF_NT = 512;
// K = 2 (see the header): 4 CTAs x 256 threads
constexpr int TF2_CL = 4, TF2_NT = 256;

static int tf_cl(int K) { return K == 1 ? TF_CL : TF2_CL; }

static size_t tail_fused_smem_k(int h, int w, int H, int W, int C, int K) {
    const int hh = (h + tf_cl(K) - 1) / tf_cl(K);
    return (size_t)(3 * W + 3 * H + K * ((C + 3) & ~3) + K * hh * w + (hh + 1) * W) * sizeof(float);
}

size_t tail_fused_smem(int h, int w, int H, int W, int C) { return tail_fused_smem_k(h, w, H, W, C, 1); }

bool tail_fused_supported(int h, int w, int H, int W, int C) {
    return C % 8 == 0 && tail_fused_smem(h, w, H, W, C) <= 200 * 1024;
}

bool tail_fused_classes_supported(int h, int w, int H, int W, int C) {
    return tail_fused_supported(h, w, H, W, C) && tail_fused_smem_k(h, w, H, W, C, TF_GROUP) <= 200 * 1024;
}

template <bool X3, int CL, int NT, int K, bool PRE>
static int launch_tf_t(const __half* A, const float* alpha_raw, size_t alpha_ld, float scale, float* alpha_out, float* out, size_t out_stride,
                       int B, int h, int w, int H, int W, int C, cudaStream_t s, const int* n_dev, float inv_slope) {
    const size_t smem = tail_fused_smem_k(h, w, H, W, C, K);
    BCAD_CUDA_CHECK(cudaFuncSetAttribute(tail_fused_kernel<X3, CL, NT, K, PRE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    tail_fused_kernel<X3, CL, NT, K, PRE><<<CL * B, NT, smem, s>>>(A, alpha_raw, alpha_ld, scale, alpha_out, out, out_stride, h, w, H, W, C, n_dev,
                                                                   inv_slope);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

template <bool X3, int CL, int NT, int K>
static int launch_tf(const __half* A, const float* alpha_raw, size_t alpha_ld, float scale, float* alpha_out, float* out, size_t out_stride,
                     int B, int h, int w, int H, int W, int C, cudaStream_t s, const int* n_dev, float inv_slope) {
    if (inv_slope > 0.f)
        return launch_tf_t<X3, CL, NT, K, true>(A, alpha_raw, alpha_ld, scale, alpha_out, out, out_stride, B, h, w, H, W, C, s, n_dev, inv_slope);
    return launch_tf_t<X3, CL, NT, K, false>(A, alpha_raw, alpha_ld, scale, alpha_out, out, out_stride, B, h, w, H, W, C, s, n_dev, 0.f);
}

int launch_tail_fused(const __half* A, const float* alpha_raw, float scale, float* alpha_out, float* out, int B, int h, int w,
                      int H, int W, int C, bool x3, cudaStream_t s, const int* n_dev, size_t out_stride, float inv_slope) {
    BCAD_REQUIRE(tail_fused_supported(h, w, H, W, C), "tail_fused: map %dx%d -> %dx%d does not fit in shared memory", h, w, H, W);
    const size_t os = out_stride ? out_stride : (size_t)H * W;
    if (x3) return launch_tf<true, TF_CL, TF_NT, 1>(A, alpha_raw, 0, scale, alpha_out, out, os, B, h, w, H, W, C, s, n_dev, inv_slope);
    return launch_tf<false, TF_CL, TF_NT, 1>(A, alpha_raw, 0, scale, alpha_out, out, os, B, h, w, H, W, C, s, n_dev, inv_slope);
}

int launch_tail_fused_classes(const __half* A, const float* alpha_raw, size_t alpha_ld, float scale, float* out, size_t out_stride, int B,
                              int h, int w, int H, int W, int C, bool x3, cudaStream_t s, const int* n_dev, float inv_slope) {
    BCAD_REQUIRE(tail_fused_classes_supported(h, w, H, W, C), "tail_fused_classes: map %dx%d -> %dx%d does not fit in shared memory", h, w, H, W);
    if (x3) return launch_tf<true, TF2_CL, TF2_NT, TF_GROUP>(A, alpha_raw, alpha_ld, scale, nullptr, out, out_stride, B, h, w, H, W, C, s, n_dev, inv_slope);
    return launch_tf<false, TF2_CL, TF2_NT, TF_GROUP>(A, alpha_raw, alpha_ld, scale, nullptr, out, out_stride, B, h, w, H, W, C, s, n_dev, inv_slope);
}

}  // namespace bcad
