// Small-margin refinement of the 16-bit tensor path (cfg.refine_margin): after the head of a chunk, the images whose two
// largest logits are closer than the margin are gathered, re-run through the split-operand (fp32-grade) kernels of a twin
// handle, and their results written back over the 16-bit ones -- all stream-ordered, no host round trip: the twin always
// runs a fixed number of slots and the device-side count decides which slots are written back.
// Why: north_star asks for predicted classes identical to the reference's (ADCNNM.py:72-78 logits, app.py:589 torch.max);
// the 16-bit logit error (~3e-3) flips the arg-max of an image whose margin is smaller than that.
#include "../../include/bcad.h"
#include "common.cuh"
#include "kernels.h"

namespace bcad {

// one CTA: ordered compaction of the flagged images (ascending index: the result does not depend on scheduling)
__global__ void __launch_bounds__(1024, 1)
refine_flag_kernel(const float* __restrict__ logits, int n, int nc, float margin, int cap, int32_t* __restrict__ idx,
                   int32_t* __restrict__ counters) {
    __shared__ int s_warp[32];
    __shared__ int s_base;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int b0 = 0; b0 < n; b0 += 1024) {
        const int b = b0 + tid;
        bool flag = false;
        if (b < n) {
            if (nc == 1) flag = fabsf(logits[b]) < margin;                  // single-logit head: distance to the decision threshold 0
            else {
                float m1 = -INFINITY, m2 = -INFINITY;
                for (int c = 0; c < nc; ++c) {
                    const float v = logits[(size_t)b * nc + c];
                    if (v > m1) { m2 = m1; m1 = v; }
                    else if (v > m2) m2 = v;
                }
                flag = !((m1 - m2) >= margin);                              // NaN logits are flagged too
            }
        }
        const unsigned bal = __ballot_sync(0xffffffffu, flag);
        if (lane == 0) s_warp[warp] = __popc(bal);
        __syncthreads();
        int before = s_base;
        for (int w = 0; w < warp; ++w) before += s_warp[w];
        const int pos = before + __popc(bal & ((1u << lane) - 1u));
        if (flag && pos < cap) idx[pos] = b;
        __syncthreads();
        if (tid == 0) {
            int tot = 0;
            for (int w = 0; w < 32; ++w) tot += s_warp[w];
            s_base += tot;
        }
        __syncthreads();
    }
    if (tid == 0) {
        const int total = s_base, kept = total < cap ? total : cap;
        counters[0] = kept;
        counters[1] += kept;
        counters[2] += total - kept;
    }
}

__global__ void __launch_bounds__(256)
refine_gather_kernel(const float* __restrict__ x, size_t img_elems, const int32_t* __restrict__ class_idx, const int32_t* __restrict__ idx,
                     const int32_t* __restrict__ counters, float* __restrict__ rx, int32_t* __restrict__ rcidx, int K) {
    const int slot = blockIdx.x;
    if (slot >= counters[0]) return;              // the twin's kernels only touch the first counters[0] slots
    const int src = idx[slot];
    const float* in = x + (size_t)src * img_elems;
    float* out = rx + (size_t)slot * img_elems;
    if (blockIdx.y == 0 && (int)threadIdx.x < K && class_idx != nullptr) rcidx[slot * K + threadIdx.x] = class_idx[src * K + threadIdx.x];
    const size_t per = (img_elems + gridDim.y - 1) / gridDim.y;
    const size_t lo = (size_t)blockIdx.y * per, hi = lo + per < img_elems ? lo + per : img_elems;
    if (((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & 15) == 0 && (lo & 3) == 0) {
        const size_t v_hi = lo + ((hi - lo) & ~(size_t)3);
        for (size_t i = lo + 4 * threadIdx.x; i < v_hi; i += 4 * blockDim.x)
            *reinterpret_cast<float4*>(out + i) = *reinterpret_cast<const float4*>(in + i);
        for (size_t i = v_hi + threadIdx.x; i < hi; i += blockDim.x) out[i] = in[i];
    } else {
        for (size_t i = lo + threadIdx.x; i < hi; i += blockDim.x) out[i] = in[i];
    }
}

__global__ void __launch_bounds__(256)
refine_scatter_kernel(RefineScatter a, const int32_t* __restrict__ idx, const int32_t* __restrict__ counters) {
    const int slot = blockIdx.x;
    if (slot >= counters[0]) return;
    const int dst = idx[slot];
    if (blockIdx.y == 0) {
        for (int j = 0; j < a.n_dense; ++j)
            for (int u = threadIdx.x; u < a.sizes[j]; u += blockDim.x)
                a.dst_z[j][(size_t)dst * a.sizes[j] + u] = a.src_z[j][(size_t)slot * a.sizes[j] + u];
        for (int c = threadIdx.x; c < a.nc; c += blockDim.x) a.dst_probs[(size_t)dst * a.nc + c] = a.src_probs[(size_t)slot * a.nc + c];
        if (threadIdx.x == 0) a.dst_cls[dst] = a.src_cls[slot];
    }
    if (a.dst_heat == nullptr) return;
    const float* in = a.src_heat + (size_t)slot * a.hm;
    float* out = a.dst_heat + (size_t)dst * a.hm;
    const size_t per = (a.hm + gridDim.y - 1) / gridDim.y;
    const size_t lo = (size_t)blockIdx.y * per, hi = lo + per < a.hm ? lo + per : a.hm;
    for (size_t i = lo + threadIdx.x; i < hi; i += blockDim.x) out[i] = in[i];
}

int launch_refine_flag(const float* logits, int n, int nc, float margin, int cap, int32_t* idx, int32_t* counters, cudaStream_t s) {
    refine_flag_kernel<<<1, 1024, 0, s>>>(logits, n, nc, margin, cap, idx, counters);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

static int copy_blocks(size_t elems) {
    const size_t b = (elems + 8191) / 8192;
    return (int)(b < 1 ? 1 : (b > 64 ? 64 : b));
}

int launch_refine_gather(const float* x, size_t img_elems, const int32_t* class_idx, const int32_t* idx, const int32_t* counters,
                         int slots, float* rx, int32_t* rcidx, cudaStream_t s, int K) {
    int by = copy_blocks(img_elems);
    while (by > 1 && (((img_elems + by - 1) / by) & 3)) --by;          // keep every block's range a multiple of 4 floats (vector path)
    refine_gather_kernel<<<dim3(slots, by), 256, 0, s>>>(x, img_elems, class_idx, idx, counters, rx, rcidx, K);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

int launch_refine_scatter(const RefineScatter& a, const int32_t* idx, const int32_t* counters, int slots, cudaStream_t s) {
    refine_scatter_kernel<<<dim3(slots, a.dst_heat ? copy_blocks(a.hm) : 1), 256, 0, s>>>(a, idx, counters);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

}  // namespace bcad
