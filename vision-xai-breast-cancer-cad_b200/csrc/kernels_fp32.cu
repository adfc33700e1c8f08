// fp32 CUDA-core kernels: the shape-generic path of libbcad (any ksize / channels / padding).
//
// Reference semantics implemented here (file:line under /root/reference):
//   conv + bias + LeakyReLU (strict ">")      Classes/CNNModel.py:227-240, ADCNNM.py:48,76
//   2x2/2 max-pool, floor dims                Classes/CNNModel.py:245-261
//   max-pool backward, ties ALL / FIRST       Classes/CNNModel.py:263-277 / nn.MaxPool2d autograd
//   dense  z = W.flat + b, LeakyReLU          Classes/CNNModel.py:177-189
//   softmax(clip +-50), /(sum+1e-12)          Classes/CNNModel.py:203-212
//   top gradient, dense backward              explainability.py:20-34
//   Grad-CAM tail                             pytorch_grad_cam (GRADCAM.py:53,64) -- see oracle/gradcam.py
#include "common.cuh"
#include "kernels.h"
#include "../../include/bcad.h"

namespace bcad {

// =====================================================================================================
// direct convolution, NHWC fp32, fused bias + LeakyReLU (+ 2x2 max-pool)
//   CTA tile 16 rows x 32 cols x 32 couts, 256 threads, thread tile 2 rows x 4 cols x 8 couts
//   (the 2x2 pool windows are thread-local), input channels staged through smem 8 at a time.
// =====================================================================================================
constexpr int CT_ROWS = 16, CT_COLS = 32, CT_COUT = 32, CT_CC = 8;

template <int K>
__global__ void __launch_bounds__(256, 2) conv_fp32_kernel(ConvArgs a, int tiles_x) {
    constexpr int PR = CT_ROWS + K - 1, PC = CT_COLS + K - 1;
    extern __shared__ float smem[];
    float* s_in = smem;                       // [CT_CC][PR][PC]
    float* s_w = smem + CT_CC * PR * PC;      // [K*K][CT_CC][32]

    const int tid = threadIdx.x;
    const int cg = tid & 3;                   // cout group: couts cg*8 .. cg*8+7 of this CTA's 32
    const int pg = tid >> 2;                  // pixel group
    const int tx = pg & 7, ty = pg >> 3;      // 8 x 8 groups of (2 rows x 4 cols)
    const int ox0 = (blockIdx.x % tiles_x) * CT_COLS, oy0 = (blockIdx.x / tiles_x) * CT_ROWS;
    const int co0 = blockIdx.y * CT_COUT;
    const int b = blockIdx.z;

    float acc[2][4][8];
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[r][c][j] = 0.f;

    const float* xb = a.x + (size_t)b * a.H * a.W * a.Cin;
    for (int c0 = 0; c0 < a.Cin; c0 += CT_CC) {
        const int cc = min(CT_CC, a.Cin - c0);
        __syncthreads();
        for (int i = tid; i < PR * PC * cc; i += 256) {
            const int ci = i % cc, rest = i / cc;
            const int pc = rest % PC, pr = rest / PC;
            const int iy = oy0 - a.pad + pr, ix = ox0 - a.pad + pc;
            float v = 0.f;
            if (iy >= 0 && iy < a.H && ix >= 0 && ix < a.W)
                v = __ldg(xb + ((size_t)iy * a.W + ix) * a.Cin + c0 + ci);
            s_in[(ci * PR + pr) * PC + pc] = v;
        }
        for (int i = tid; i < K * K * cc * 32; i += 256) {
            const int co = i & 31, rest = i >> 5;
            const int ci = rest % cc, tap = rest / cc;
            s_w[(tap * CT_CC + ci) * 32 + co] =
                __ldg(a.w + ((size_t)tap * a.Cin + c0 + ci) * a.CoutPad + co0 + co);
        }
        __syncthreads();
        for (int ci = 0; ci < cc; ++ci) {
            float win[K + 1][K + 3];
#pragma unroll
            for (int r = 0; r < K + 1; ++r)
#pragma unroll
                for (int c = 0; c < K + 3; ++c)
                    win[r][c] = s_in[(ci * PR + ty * 2 + r) * PC + tx * 4 + c];
#pragma unroll
            for (int ky = 0; ky < K; ++ky)
#pragma unroll
                for (int kx = 0; kx < K; ++kx) {
                    const float4* wp =
                        reinterpret_cast<const float4*>(s_w + ((ky * K + kx) * CT_CC + ci) * 32 + cg * 8);
                    const float4 w0 = wp[0], w1 = wp[1];
#pragma unroll
                    for (int r = 0; r < 2; ++r)
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const float v = win[r + ky][c + kx];
                            acc[r][c][0] = fmaf(v, w0.x, acc[r][c][0]);
                            acc[r][c][1] = fmaf(v, w0.y, acc[r][c][1]);
                            acc[r][c][2] = fmaf(v, w0.z, acc[r][c][2]);
                            acc[r][c][3] = fmaf(v, w0.w, acc[r][c][3]);
                            acc[r][c][4] = fmaf(v, w1.x, acc[r][c][4]);
                            acc[r][c][5] = fmaf(v, w1.y, acc[r][c][5]);
                            acc[r][c][6] = fmaf(v, w1.z, acc[r][c][6]);
                            acc[r][c][7] = fmaf(v, w1.w, acc[r][c][7]);
                        }
                }
        }
    }

    // ---- epilogue: bias + LeakyReLU, store y, thread-local 2x2 max-pool, store p
    const int cbase = co0 + cg * 8;
    float bias[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) bias[j] = __ldg(a.bias + cbase + j);
    const bool vec = (a.Cout % 4 == 0) && (cbase + 8 <= a.Cout);
#pragma unroll
    for (int r = 0; r < 2; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int oy = oy0 + ty * 2 + r, ox = ox0 + tx * 4 + c;
            const bool dead = (a.Hv > 0) && (oy >= a.Hv || ox >= a.Wv);     // zero border of the padded-size output
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[r][c][j] = dead ? 0.f : leaky(acc[r][c][j] + bias[j], a.alpha);
            if (a.y != nullptr && oy < a.Ho && ox < a.Wo) {
                float* dst = a.y + (((size_t)b * a.Ho + oy) * a.Wo + ox) * a.Cout + cbase;
                if (vec) {
                    reinterpret_cast<float4*>(dst)[0] = make_float4(acc[r][c][0], acc[r][c][1], acc[r][c][2], acc[r][c][3]);
                    reinterpret_cast<float4*>(dst)[1] = make_float4(acc[r][c][4], acc[r][c][5], acc[r][c][6], acc[r][c][7]);
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        if (cbase + j < a.Cout) dst[j] = acc[r][c][j];
                }
            }
        }
    if (a.p != nullptr) {
        const int py = (oy0 >> 1) + ty;
#pragma unroll
        for (int c2 = 0; c2 < 2; ++c2) {
            const int px = (ox0 >> 1) + tx * 2 + c2;
            if (py < a.Hp && px < a.Wp) {
                float m[8];
#pragma unroll
                for (int j = 0; j < 8; ++j)
                    m[j] = fmaxf(fmaxf(acc[0][2 * c2][j], acc[0][2 * c2 + 1][j]),
                                 fmaxf(acc[1][2 * c2][j], acc[1][2 * c2 + 1][j]));
                float* dst = a.p + (((size_t)b * a.Hp + py) * a.Wp + px) * a.Cout + cbase;
                if (vec) {
                    reinterpret_cast<float4*>(dst)[0] = make_float4(m[0], m[1], m[2], m[3]);
                    reinterpret_cast<float4*>(dst)[1] = make_float4(m[4], m[5], m[6], m[7]);
                } else {
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        if (cbase + j < a.Cout) dst[j] = m[j];
                }
            }
        }
    }
}

template <int K>
static int launch_conv_k(const ConvArgs& a, cudaStream_t s) {
    constexpr int PR = CT_ROWS + K - 1, PC = CT_COLS + K - 1;
    const size_t smem = (size_t)(CT_CC * PR * PC + K * K * CT_CC * 32) * sizeof(float);
    if (smem > 48 * 1024)   // per-device attribute; cheap enough to set on every launch of the large-k variants
        BCAD_CUDA_CHECK(cudaFuncSetAttribute(conv_fp32_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int tiles_x = cdiv(a.Wo, CT_COLS), tiles_y = cdiv(a.Ho, CT_ROWS);
    dim3 grid(tiles_x * tiles_y, a.CoutPad / CT_COUT, a.B);
    conv_fp32_kernel<K><<<grid, 256, smem, s>>>(a, tiles_x);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

int launch_conv_fp32(const ConvArgs& a, cudaStream_t s) {
    BCAD_REQUIRE(a.B <= 65535, "conv: batch chunk %d exceeds 65535", a.B);
    switch (a.ksize) {
        case 1: return launch_conv_k<1>(a, s);
        case 2: return launch_conv_k<2>(a, s);
        case 3: return launch_conv_k<3>(a, s);
        case 4: return launch_conv_k<4>(a, s);
        case 5: return launch_conv_k<5>(a, s);
        case 6: return launch_conv_k<6>(a, s);
        case 7: return launch_conv_k<7>(a, s);
        default:
            set_error("conv: ksize %d not supported (1..7)", a.ksize);
            return BCAD_ERR_INVALID;
    }
}

// =====================================================================================================
// SGEMM  C[M,N] = A[M,K] * B   (A row-major K-contiguous; B as [N,K] or [K,N]), split-K partials
//   128 x 128 x 8 tiles, 256 threads, 8x8 register tile split 4+4 so smem reads are conflict-free
// =====================================================================================================
constexpr int GM = 128, GN = 128, GK = 8, GLD = 132;

template <bool B_KMAJOR>
__global__ void __launch_bounds__(256, 2)
sgemm_kernel(const float* __restrict__ A, const float* __restrict__ Bm, float* __restrict__ C, int M, int N,
             int K, int k_per_split) {
    __shared__ __align__(16) float As[GK][GLD];
    __shared__ __align__(16) float Bs[GK][GLD];
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const int m0 = blockIdx.y * GM, n0 = blockIdx.x * GN;
    const int kbeg = blockIdx.z * k_per_split, kend = min(K, kbeg + k_per_split);

    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

    // K-major tile loader: 128 rows x 8 k; thread -> row tid/2, k-quad (tid&1)*4
    const int lrow = tid >> 1, lkq = (tid & 1) * 4;
    // N-major B loader: 8 k x 128 n; thread -> k tid/32, n-quad (tid&31)*4
    const int bk = tid >> 5, bnq = (tid & 31) * 4;
    const bool kvec = (K % 4 == 0), nvec = (N % 4 == 0);

    auto load_kmajor = [&](const float* P, int rows, int r0, int k0, float (&v)[4]) {
        const int r = r0 + lrow, k = k0 + lkq;
        v[0] = v[1] = v[2] = v[3] = 0.f;
        if (r < rows) {
            const float* src = P + (size_t)r * K + k;
            if (kvec && k + 4 <= kend) {
                const float4 t = __ldg(reinterpret_cast<const float4*>(src));
                v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (k + j < kend) v[j] = __ldg(src + j);
            }
        }
    };
    auto load_nmajor = [&](int k0, float (&v)[4]) {
        const int k = k0 + bk, n = n0 + bnq;
        v[0] = v[1] = v[2] = v[3] = 0.f;
        if (k < kend) {
            const float* src = Bm + (size_t)k * N + n;
            if (nvec && n + 4 <= N) {
                const float4 t = __ldg(reinterpret_cast<const float4*>(src));
                v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (n + j < N) v[j] = __ldg(src + j);
            }
        }
    };

    float ra[4], rb[4];
    if (kbeg < kend) {
        load_kmajor(A, M, m0, kbeg, ra);
        if (B_KMAJOR) load_kmajor(Bm, N, n0, kbeg, rb); else load_nmajor(kbeg, rb);
    }
    for (int k0 = kbeg; k0 < kend; k0 += GK) {
        __syncthreads();
#pragma unroll
        for (int j = 0; j < 4; ++j) As[lkq + j][lrow] = ra[j];
        if (B_KMAJOR) {
#pragma unroll
            for (int j = 0; j < 4; ++j) Bs[lkq + j][lrow] = rb[j];
        } else {
            *reinterpret_cast<float4*>(&Bs[bk][bnq]) = make_float4(rb[0], rb[1], rb[2], rb[3]);
        }
        __syncthreads();
        if (k0 + GK < kend) {   // prefetch the next tile into registers while computing this one
            load_kmajor(A, M, m0, k0 + GK, ra);
            if (B_KMAJOR) load_kmajor(Bm, N, n0, k0 + GK, rb); else load_nmajor(k0 + GK, rb);
        }
#pragma unroll
        for (int kk = 0; kk < GK; ++kk) {
            const float4 a0 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            const float4 a1 = *reinterpret_cast<const float4*>(&As[kk][ty * 4 + 64]);
            const float4 b0 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float4 b1 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4 + 64]);
            const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
    }
    float* Cz = C + (size_t)blockIdx.z * M * N;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int m = m0 + ty * 4 + (i & 3) + (i >> 2) * 64;
        if (m >= M) continue;
#pragma unroll
        for (int jh = 0; jh < 2; ++jh) {
            const int n = n0 + tx * 4 + jh * 64;
            float* dst = Cz + (size_t)m * N + n;
            if (nvec && n + 4 <= N) {
                *reinterpret_cast<float4*>(dst) = make_float4(acc[i][jh * 4], acc[i][jh * 4 + 1], acc[i][jh * 4 + 2], acc[i][jh * 4 + 3]);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (n + j < N) dst[j] = acc[i][jh * 4 + j];
            }
        }
    }
}

int sgemm_pick_splits(int M, int N, int K) {
    const int tiles = cdiv(M, GM) * cdiv(N, GN);
    int splits = 1;
    if (tiles < 296 && K >= 512) {
        splits = cdiv(296, tiles);
        const int max_splits = K / 256;
        if (splits > max_splits) splits = max_splits;
        if (splits < 1) splits = 1;
    }
    return splits;
}

int launch_sgemm(const float* A, const float* Bm, float* C, int M, int N, int K, bool b_kmajor, int splits,
                 cudaStream_t s) {
    int kps = cdiv(cdiv(K, splits), GK) * GK;
    dim3 grid(cdiv(N, GN), cdiv(M, GM), splits);
    BCAD_REQUIRE(grid.y <= 65535 && grid.z <= 65535, "sgemm: grid too large (M=%d splits=%d)", M, splits);
    if (b_kmajor) sgemm_kernel<true><<<grid, 256, 0, s>>>(A, Bm, C, M, N, K, kps);
    else sgemm_kernel<false><<<grid, 256, 0, s>>>(A, Bm, C, M, N, K, kps);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// z[m,n] = sum_s partial[s][m][n] + bias[n] (fixed order => run-to-run bit-stable); h = LeakyReLU(z)
__global__ void splitk_reduce_kernel(const float* __restrict__ part, int splits, const float* __restrict__ bias,
                                     float* __restrict__ z, float* __restrict__ h, float alpha, int M, int N) {
    const size_t total = (size_t)M * N;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        float v = 0.f;
        for (int s = 0; s < splits; ++s) v += part[(size_t)s * total + i];
        if (bias != nullptr) v += __ldg(bias + (i % N));
        if (z != nullptr) z[i] = v;
        if (h != nullptr) h[i] = leaky(v, alpha);
    }
}

int launch_splitk_reduce(const float* part, int splits, const float* bias, float* z, float* h, float alpha,
                         int M, int N, cudaStream_t s) {
    const size_t total = (size_t)M * N;
    const int blocks = (int)min((size_t)4096, (total + 255) / 256);
    splitk_reduce_kernel<<<blocks, 256, 0, s>>>(part, splits, bias, z, h, alpha, M, N);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// =====================================================================================================
// head: probabilities + class; top gradient; LeakyReLU' mask
// =====================================================================================================
__global__ void head_kernel(const float* __restrict__ logits, float* __restrict__ probs, int32_t* __restrict__ cls,
                            int B, int nc, int head) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const float* z = logits + (size_t)b * nc;
    // double arithmetic: the NumPy reference's softmax is float64 (Classes/CNNModel.py:205)
    double zmax = -1e300;
    for (int c = 0; c < nc; ++c) {
        double v = (double)z[c];
        if (head == BCAD_HEAD_SOFTMAX_CLIP) v = fmin(fmax(v, -50.0), 50.0);
        zmax = fmax(zmax, v);
    }
    double sum = 0.0;
    for (int c = 0; c < nc; ++c) {
        double v = (double)z[c];
        if (head == BCAD_HEAD_SOFTMAX_CLIP) v = fmin(fmax(v, -50.0), 50.0);
        sum += exp(v - zmax);
    }
    int best = 0;
    double best_v = -1e300;
    for (int c = 0; c < nc; ++c) {
        double v = (double)z[c];
        if (head == BCAD_HEAD_SOFTMAX_CLIP) v = fmin(fmax(v, -50.0), 50.0);
        double p = (head == BCAD_HEAD_SOFTMAX_CLIP) ? exp(v - zmax) / (sum + 1e-12) : exp(v - zmax) / sum;
        if (probs != nullptr) probs[(size_t)b * nc + c] = (float)p;
        // NumPy flavour: argmax(probs) (Classes/CNNModel.py:526); torch flavour: max(logits) (app.py:589)
        const double score = (head == BCAD_HEAD_SOFTMAX_CLIP) ? p : (double)z[c];
        if (score > best_v) { best_v = score; best = c; }
    }
    if (cls != nullptr) cls[b] = best;
}

int launch_head(const float* logits, float* probs, int32_t* cls, int B, int nc, int head, cudaStream_t s) {
    head_kernel<<<cdiv(B, 128), 128, 0, s>>>(logits, probs, cls, B, nc, head);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

__global__ void top_grad_kernel(const float* __restrict__ probs, const int32_t* __restrict__ cls,
                                const int32_t* __restrict__ class_idx, float* __restrict__ d_top, int B, int nc,
                                int grad_mode) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * nc) return;
    const int b = i / nc, c = i % nc;
    const int target = class_idx != nullptr ? class_idx[b] : cls[b];
    const float onehot = (c == target) ? 1.f : 0.f;
    d_top[i] = (grad_mode == BCAD_GRAD_LOGIT) ? onehot : probs[i] - onehot;
}

int launch_top_grad(const float* probs, const int32_t* cls, const int32_t* class_idx, float* d_top, int B, int nc,
                    int grad_mode, cudaStream_t s) {
    top_grad_kernel<<<cdiv(B * nc, 256), 256, 0, s>>>(probs, cls, class_idx, d_top, B, nc, grad_mode);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

__global__ void leaky_mask_mul_kernel(float* __restrict__ d, const float* __restrict__ z, float alpha, size_t n) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        d[i] *= (z[i] > 0.f ? 1.f : alpha);
}

int launch_leaky_mask_mul(float* d, const float* z, float alpha, int64_t n, cudaStream_t s) {
    const int blocks = (int)min((int64_t)148 * 16, (n + 255) / 256);
    leaky_mask_mul_kernel<<<blocks, 256, 0, s>>>(d, z, alpha, (size_t)n);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// =====================================================================================================
// max-pool backward: dy[window] = g * switch(window)
// =====================================================================================================
__global__ void unpool_kernel(const float* __restrict__ g, const float* __restrict__ y, float* __restrict__ dy,
                              int B, int Ho, int Wo, int C, int ties) {
    const int Hp = Ho / 2, Wp = Wo / 2;
    const int Hc = (Ho + 1) / 2, Wc = (Wo + 1) / 2;          // windows incl. the dropped odd row/col
    const size_t total = (size_t)B * Hc * Wc * C;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % C);
        size_t r = i / C;
        const int wx = (int)(r % Wc); r /= Wc;
        const int wy = (int)(r % Hc);
        const int b = (int)(r / Hc);
        const size_t ybase = ((size_t)b * Ho) * Wo * C + c;
        if (wy < Hp && wx < Wp) {
            const float gv = g[(((size_t)b * Hp + wy) * Wp + wx) * C + c];
            float v[4];
            size_t idx[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                idx[q] = ybase + ((size_t)(2 * wy + (q >> 1)) * Wo + (2 * wx + (q & 1))) * C;
                v[q] = y[idx[q]];
            }
            const float m = fmaxf(fmaxf(v[0], v[1]), fmaxf(v[2], v[3]));
            bool taken = false;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                bool sw = (v[q] == m);
                if (ties == BCAD_TIES_FIRST) { sw = sw && !taken; taken = taken || sw; }
                dy[idx[q]] = sw ? gv : 0.f;
            }
        } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int yy = 2 * wy + (q >> 1), xx = 2 * wx + (q & 1);
                if (yy < Ho && xx < Wo) dy[ybase + ((size_t)yy * Wo + xx) * C] = 0.f;
            }
        }
    }
}

int launch_unpool(const float* g, const float* y, float* dy, int B, int Ho, int Wo, int C, int ties, cudaStream_t s) {
    const size_t total = (size_t)B * ((Ho + 1) / 2) * ((Wo + 1) / 2) * C;
    const int blocks = (int)min((size_t)148 * 32, (total + 255) / 256);
    unpool_kernel<<<blocks, 256, 0, s>>>(g, y, dy, B, Ho, Wo, C, ties);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// =====================================================================================================
// Grad-CAM channel weights without materialising dA:
//   alpha_k * (h*w) = sum over pool windows of g[window,k] * (#elements the gradient is routed to)
//   (#routed = 1 for TIES_FIRST, number of maxima for TIES_ALL)
// grid (splits, B); block 256 = CL channel lanes x (256/CL) pixel lanes
// =====================================================================================================
// pre_slope >= 0: the target is the conv block's PRE-activation output (what a hook on the nn.Conv2d module captures,
// ADCNNM.py:76): the routed gradient is also multiplied by LeakyReLU'(z) at the maximum = (max > 0 ? 1 : pre_slope).
__global__ void alpha_from_pool_grad_kernel(const float* __restrict__ g, const float* __restrict__ y,
                                            float* __restrict__ alpha_part, int Ho, int Wo, int C, int ties,
                                            int CL, float pre_slope) {
    extern __shared__ float red[];                     // [256/CL][CL]
    const int Hp = Ho / 2, Wp = Wo / 2;
    const int b = blockIdx.y, split = blockIdx.x, splits = gridDim.x;
    const int cl = threadIdx.x % CL, pl = threadIdx.x / CL, PL = blockDim.x / CL;
    const int rows_per = cdiv(Hp, splits);
    const int r0 = split * rows_per, r1 = min(Hp, r0 + rows_per);
    for (int cb = 0; cb < C; cb += CL) {               // uniform trip count (barriers inside)
        const int c = cb + cl;
        float acc = 0.f;
        for (int wy = r0; wy < r1 && c < C; ++wy)
            for (int wx = pl; wx < Wp; wx += PL) {
                float gv = g[(((size_t)b * Hp + wy) * Wp + wx) * C + c];
                if (ties == BCAD_TIES_ALL || pre_slope >= 0.f) {
                    const float* yp = y + (((size_t)b * Ho + 2 * wy) * Wo + 2 * wx) * C + c;
                    const float v0 = yp[0], v1 = yp[C], v2 = yp[(size_t)Wo * C], v3 = yp[(size_t)Wo * C + C];
                    const float m = fmaxf(fmaxf(v0, v1), fmaxf(v2, v3));
                    if (ties == BCAD_TIES_ALL) gv *= (float)((v0 == m) + (v1 == m) + (v2 == m) + (v3 == m));
                    if (pre_slope >= 0.f && !(m > 0.f)) gv *= pre_slope;
                }
                acc += gv;
            }
        red[pl * CL + cl] = acc;
        __syncthreads();
        if (pl == 0 && c < C) {
            float t = 0.f;
            for (int q = 0; q < PL; ++q) t += red[q * CL + cl];
            alpha_part[((size_t)b * splits + split) * C + c] = t;
        }
        __syncthreads();
    }
}

int alpha_pool_splits(int Hp) { return Hp >= 32 ? 4 : 1; }

static int pick_channel_lanes(int C) {
    int cl = 1;
    while (cl < C && cl < 64) cl <<= 1;
    return cl;
}

int launch_alpha_from_pool_grad(const float* g, const float* y, float* alpha_part, int B, int Ho, int Wo, int C,
                                int ties, int splits, cudaStream_t s, float pre_slope) {
    const int CL = pick_channel_lanes(C);
    dim3 grid(splits, B);
    alpha_from_pool_grad_kernel<<<grid, 256, 256 * sizeof(float), s>>>(g, y, alpha_part, Ho, Wo, C, ties, CL, pre_slope);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// alpha partials from a dense gradient map dA [B,h,w,C] (fp32 or bf16): plain per-channel sums
template <typename T>
__global__ void alpha_from_dense_grad_kernel(const T* __restrict__ dA, float* __restrict__ alpha_part, int h, int w,
                                             int C, int CL) {
    extern __shared__ float red[];
    const int b = blockIdx.y, split = blockIdx.x, splits = gridDim.x;
    const int cl = threadIdx.x % CL, pl = threadIdx.x / CL, PL = blockDim.x / CL;
    const int npix = h * w;
    const int per = cdiv(npix, splits);
    const int p0 = split * per, p1 = min(npix, p0 + per);
    const T* base = dA + (size_t)b * npix * C;
    for (int cb = 0; cb < C; cb += CL) {               // uniform trip count (barriers inside)
        const int c = cb + cl;
        float acc = 0.f;
        for (int p = p0 + pl; p < p1 && c < C; p += PL) {
            if constexpr (sizeof(T) == 4) acc += base[(size_t)p * C + c];
            else acc += __bfloat162float(base[(size_t)p * C + c]);
        }
        red[pl * CL + cl] = acc;
        __syncthreads();
        if (pl == 0 && c < C) {
            float t = 0.f;
            for (int q = 0; q < PL; ++q) t += red[q * CL + cl];
            alpha_part[((size_t)b * splits + split) * C + c] = t;
        }
        __syncthreads();
    }
}

// vectorised variant: C % 4 == 0 (fp32) / C % 8 == 0 (bf16), 128-bit streaming loads
template <bool BF16>
__global__ void __launch_bounds__(256)
alpha_from_dense_grad_vec_kernel(const void* __restrict__ dA, float* __restrict__ alpha_part, int h, int w, int C) {
    constexpr int EPV = BF16 ? 8 : 4;                  // elements per 16-byte vector
    extern __shared__ float red[];                     // [256][EPV]
    const int b = blockIdx.y, split = blockIdx.x, splits = gridDim.x;
    const int npix = h * w;
    const int per = cdiv(npix, splits);
    const int p0 = split * per, p1 = min(npix, p0 + per);
    const int vpp = C / EPV;                           // vectors per pixel
    const size_t v0 = (size_t)p0 * vpp, v1 = (size_t)p1 * vpp;
    // thread t always sees the same channel group when 256 % vpp == 0; otherwise use the generic kernel
    const uint4* base = reinterpret_cast<const uint4*>(dA) + (size_t)b * npix * vpp;
    float acc[EPV];
#pragma unroll
    for (int j = 0; j < EPV; ++j) acc[j] = 0.f;
    for (size_t v = v0 + threadIdx.x; v < v1; v += 256) {
        const uint4 q = ldg_stream_u4(base + v);
        if constexpr (BF16) {
            acc[0] += bf16lo(q.x); acc[1] += bf16hi(q.x); acc[2] += bf16lo(q.y); acc[3] += bf16hi(q.y);
            acc[4] += bf16lo(q.z); acc[5] += bf16hi(q.z); acc[6] += bf16lo(q.w); acc[7] += bf16hi(q.w);
        } else {
            acc[0] += __uint_as_float(q.x); acc[1] += __uint_as_float(q.y);
            acc[2] += __uint_as_float(q.z); acc[3] += __uint_as_float(q.w);
        }
    }
#pragma unroll
    for (int j = 0; j < EPV; ++j) red[threadIdx.x * EPV + j] = acc[j];
    __syncthreads();
    // channel c is held by threads t with (v0 + t) % vpp == c / EPV
    for (int c = threadIdx.x; c < C; c += 256) {
        const int grp = c / EPV, j = c % EPV;
        const int first = (int)((grp + vpp - (v0 % vpp)) % vpp);
        float t = 0.f;
        for (int q = first; q < 256; q += vpp) t += red[q * EPV + j];
        alpha_part[((size_t)b * splits + split) * C + c] = t;
    }
}

int launch_alpha_from_dense_grad(const void* dA, int dtype, float* alpha_part, int B, int h, int w, int C, int splits,
                                 cudaStream_t s) {
    dim3 grid(splits, B);
    const int epv = dtype == 1 ? 8 : 4;
    if (C % epv == 0 && 256 % (C / epv) == 0) {
        if (dtype == 1) alpha_from_dense_grad_vec_kernel<true><<<grid, 256, 256 * 8 * sizeof(float), s>>>(dA, alpha_part, h, w, C);
        else alpha_from_dense_grad_vec_kernel<false><<<grid, 256, 256 * 4 * sizeof(float), s>>>(dA, alpha_part, h, w, C);
    } else {
        const int CL = pick_channel_lanes(C);
        if (dtype == 1)
            alpha_from_dense_grad_kernel<__nv_bfloat16><<<grid, 256, 256 * sizeof(float), s>>>(
                reinterpret_cast<const __nv_bfloat16*>(dA), alpha_part, h, w, C, CL);
        else
            alpha_from_dense_grad_kernel<float><<<grid, 256, 256 * sizeof(float), s>>>(
                reinterpret_cast<const float*>(dA), alpha_part, h, w, C, CL);
    }
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// =====================================================================================================
// cam_lo = ReLU(sum_k alpha_k A_k)  + per-CTA min/max partials
// grid (splits, B), 256 threads; LP lanes cooperate on one pixel with 128-bit loads
// =====================================================================================================
template <bool BF16>
__global__ void __launch_bounds__(256)
cam_kernel(const void* __restrict__ A, const float* __restrict__ alpha_part, int alpha_splits, float inv_hw,
           float* __restrict__ alpha_out, float* __restrict__ cam_lo, float* __restrict__ mm, int h, int w, int C,
           int LP, int vec, float inv_slope) {
    // inv_slope > 0 (fp32 maps only): A holds post-LeakyReLU values and the target is the PRE-activation map: z = a > 0 ? a : a / slope
    extern __shared__ float s_alpha[];                 // [C] then [16] reduction scratch
    __shared__ float s_min[8], s_max[8];
    const int b = blockIdx.y, split = blockIdx.x, splits = gridDim.x;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float t = 0.f;
        for (int q = 0; q < alpha_splits; ++q) t += alpha_part[((size_t)b * alpha_splits + q) * C + c];
        t *= inv_hw;
        s_alpha[c] = t;
        if (alpha_out != nullptr && split == 0) alpha_out[(size_t)b * C + c] = t;
    }
    __syncthreads();
    const int npix = h * w;
    const int per = cdiv(npix, splits);
    const int p0 = split * per, p1 = min(npix, p0 + per);
    float vmin = 3.4e38f, vmax = -3.4e38f;
    if (vec) {
        constexpr int EPV = BF16 ? 8 : 4;
        const int vpp = C / EPV;
        const int sub = threadIdx.x % LP, grp = threadIdx.x / LP, G = blockDim.x / LP;
        const uint4* base = reinterpret_cast<const uint4*>(A) + (size_t)b * npix * vpp;
        const int iters = cdiv_dev(p1 - p0, G);
        for (int it = 0; it < iters; ++it) {               // uniform trip count (shuffles inside)
            const int p = p0 + it * G + grp;
            float acc = 0.f;
            const bool live = p < p1;
            if (live)
                for (int v = sub; v < vpp; v += LP) {
                    const uint4 q = ldg_stream_u4(base + (size_t)p * vpp + v);
                    const float* al = s_alpha + v * EPV;
                    if constexpr (BF16) {
                        acc = fmaf(bf16lo(q.x), al[0], acc); acc = fmaf(bf16hi(q.x), al[1], acc);
                        acc = fmaf(bf16lo(q.y), al[2], acc); acc = fmaf(bf16hi(q.y), al[3], acc);
                        acc = fmaf(bf16lo(q.z), al[4], acc); acc = fmaf(bf16hi(q.z), al[5], acc);
                        acc = fmaf(bf16lo(q.w), al[6], acc); acc = fmaf(bf16hi(q.w), al[7], acc);
                    } else {
                        float a0 = __uint_as_float(q.x), a1 = __uint_as_float(q.y), a2 = __uint_as_float(q.z), a3 = __uint_as_float(q.w);
                        if (inv_slope > 0.f) {
                            a0 = a0 > 0.f ? a0 : a0 * inv_slope; a1 = a1 > 0.f ? a1 : a1 * inv_slope;
                            a2 = a2 > 0.f ? a2 : a2 * inv_slope; a3 = a3 > 0.f ? a3 : a3 * inv_slope;
                        }
                        acc = fmaf(a0, al[0], acc); acc = fmaf(a1, al[1], acc);
                        acc = fmaf(a2, al[2], acc); acc = fmaf(a3, al[3], acc);
                    }
                }
            for (int o = LP >> 1; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
            if (live && sub == 0) {
                acc = fmaxf(acc, 0.f);
                cam_lo[(size_t)b * npix + p] = acc;
                vmin = fminf(vmin, acc);
                vmax = fmaxf(vmax, acc);
            }
        }
    } else {
        for (int p = p0 + threadIdx.x; p < p1; p += blockDim.x) {
            float acc = 0.f;
            for (int c = 0; c < C; ++c) {
                float a;
                if (BF16) a = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(A)[((size_t)b * npix + p) * C + c]);
                else a = reinterpret_cast<const float*>(A)[((size_t)b * npix + p) * C + c];
                if (!BF16 && inv_slope > 0.f && !(a > 0.f)) a *= inv_slope;
                acc = fmaf(a, s_alpha[c], acc);
            }
            acc = fmaxf(acc, 0.f);
            cam_lo[(size_t)b * npix + p] = acc;
            vmin = fminf(vmin, acc);
            vmax = fmaxf(vmax, acc);
        }
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

int cam_splits(int h) { return h >= 64 ? 8 : (h >= 16 ? 2 : 1); }

int launch_cam(const void* A, int dtype, const float* alpha_part, int alpha_splits, float inv_hw, float* alpha_out,
               float* cam_lo, float* mm, int B, int h, int w, int C, int splits, cudaStream_t s, float inv_slope) {
    const int epv = dtype == 1 ? 8 : 4;
    const int vec = (C % epv == 0) ? 1 : 0;
    int LP = 1;
    if (vec) { while (LP < C / epv && LP < 32) LP <<= 1; }
    dim3 grid(splits, B);
    const size_t smem = (size_t)C * sizeof(float);
    if (dtype == 1) cam_kernel<true><<<grid, 256, smem, s>>>(A, alpha_part, alpha_splits, inv_hw, alpha_out, cam_lo, mm, h, w, C, LP, vec, 0.f);
    else cam_kernel<false><<<grid, 256, smem, s>>>(A, alpha_part, alpha_splits, inv_hw, alpha_out, cam_lo, mm, h, w, C, LP, vec, inv_slope);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// =====================================================================================================
// min-max -> bilinear (cv2.resize INTER_LINEAR) -> min-max.  One CTA per image; the low-res map
// lives in shared memory (falls back to global/L2 reads when it does not fit).
// =====================================================================================================
constexpr int UP_THREADS = 1024;

__device__ __forceinline__ void block_minmax(float& vmin, float& vmax, float* s_red) {
    vmin = warp_min(vmin);
    vmax = warp_max(vmax);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) { s_red[threadIdx.x >> 5] = vmin; s_red[32 + (threadIdx.x >> 5)] = vmax; }
    __syncthreads();
    const int nw = blockDim.x >> 5;
    vmin = s_red[0];
    vmax = s_red[32];
    for (int q = 1; q < nw; ++q) { vmin = fminf(vmin, s_red[q]); vmax = fmaxf(vmax, s_red[32 + q]); }
}

__global__ void __launch_bounds__(UP_THREADS)
upsample_norm_kernel(const float* __restrict__ cam_lo, const float* __restrict__ mm, int mm_splits,
                     float* __restrict__ out, size_t out_stride, int h, int w, int H, int W, int lo_in_smem) {
    extern __shared__ float sm[];
    __shared__ float s_red[64];
    // layout: x0[W] x1[W] fx[W] y0[H] y1[H] fy[H] (ints stored as float bits) then the low-res map
    int* s_x0 = reinterpret_cast<int*>(sm);
    int* s_x1 = s_x0 + W;
    float* s_fx = sm + 2 * W;
    int* s_y0 = reinterpret_cast<int*>(sm + 3 * W);
    int* s_y1 = s_y0 + H;
    float* s_fy = sm + 3 * W + 2 * H;
    float* s_lo = sm + 3 * W + 3 * H;
    const int b = blockIdx.x;
    const int tid = threadIdx.x;
    // coordinate tables: source coordinate in double, weight = float(frac) (oracle/gradcam.py, pinned to cv2)
    for (int d = tid; d < W + H; d += blockDim.x) {
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
        else { s_y0[dd] = i0; s_y1[dd] = i1; s_fy[dd] = f; }
    }
    float mn = 3.4e38f, mx = -3.4e38f;
    for (int q = 0; q < mm_splits; ++q) {
        mn = fminf(mn, mm[((size_t)b * mm_splits + q) * 2]);
        mx = fmaxf(mx, mm[((size_t)b * mm_splits + q) * 2 + 1]);
    }
    const float denom = 1e-7f + (mx - mn);
    const float* lo = cam_lo + (size_t)b * h * w;
    if (lo_in_smem) {
        for (int i = tid; i < h * w; i += blockDim.x) s_lo[i] = (lo[i] - mn) / denom;
    }
    __syncthreads();
    auto sample = [&](int oy, int ox) -> float {
        const int x0 = s_x0[ox], x1 = s_x1[ox], y0 = s_y0[oy], y1 = s_y1[oy];
        const float fx = s_fx[ox], fy = s_fy[oy];
        float a00, a01, a10, a11;
        if (lo_in_smem) {
            a00 = s_lo[y0 * w + x0]; a01 = s_lo[y0 * w + x1]; a10 = s_lo[y1 * w + x0]; a11 = s_lo[y1 * w + x1];
        } else {
            a00 = (lo[y0 * w + x0] - mn) / denom; a01 = (lo[y0 * w + x1] - mn) / denom;
            a10 = (lo[y1 * w + x0] - mn) / denom; a11 = (lo[y1 * w + x1] - mn) / denom;
        }
        const float top = a00 * (1.f - fx) + a01 * fx;       // horizontal pass first (OpenCV HResize)
        const float bot = a10 * (1.f - fx) + a11 * fx;
        return top * (1.f - fy) + bot * fy;
    };
    float vmin = 3.4e38f, vmax = -3.4e38f;
    const int npix = H * W;
    for (int i = tid; i < npix; i += blockDim.x) {
        const float v = sample(i / W, i % W);
        vmin = fminf(vmin, v);
        vmax = fmaxf(vmax, v);
    }
    block_minmax(vmin, vmax, s_red);
    const float denom2 = 1e-7f + (vmax - vmin);
    float* ob = out + (size_t)b * out_stride;
    for (int i = tid; i < npix; i += blockDim.x) ob[i] = (sample(i / W, i % W) - vmin) / denom2;
}

// Separable variant (the common case: everything fits in shared memory): the horizontally interpolated rows are
// built once (h x W floats, exactly OpenCV's HResize-then-VResize order), every output sample is then two
// shared-memory reads and one lerp; both min-max passes run over that.
__global__ void __launch_bounds__(UP_THREADS)
upsample_norm_sep_kernel(const float* __restrict__ cam_lo, const float* __restrict__ mm, int mm_splits,
                         float* __restrict__ out, size_t out_stride, int h, int w, int H, int W, const int* __restrict__ n_dev) {
    if (n_dev != nullptr && (int)blockIdx.x >= *n_dev) return;
    extern __shared__ float sm[];
    __shared__ float s_red[64];
    int* s_x0 = reinterpret_cast<int*>(sm);
    int* s_x1 = s_x0 + W;
    float* s_fx = sm + 2 * W;
    int* s_y0 = reinterpret_cast<int*>(sm + 3 * W);
    int* s_y1 = s_y0 + H;
    float* s_fy = sm + 3 * W + 2 * H;
    float* s_lo = sm + 3 * W + 3 * H;          // [h][w] normalised low-res map
    float* s_hr = s_lo + h * w;                // [h][W] horizontally interpolated rows
    const int b = blockIdx.x, tid = threadIdx.x;
    for (int d = tid; d < W + H; d += blockDim.x) {
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
        else { s_y0[dd] = i0 * W; s_y1[dd] = i1 * W; s_fy[dd] = f; }
    }
    float mn = 3.4e38f, mx = -3.4e38f;
    for (int q = 0; q < mm_splits; ++q) {
        mn = fminf(mn, mm[((size_t)b * mm_splits + q) * 2]);
        mx = fmaxf(mx, mm[((size_t)b * mm_splits + q) * 2 + 1]);
    }
    const float denom = 1e-7f + (mx - mn);
    const float* lo = cam_lo + (size_t)b * h * w;
    {
        const float inv = 1.f / denom;
        for (int i = tid; i < h * w; i += blockDim.x) s_lo[i] = (lo[i] - mn) * inv;
    }
    __syncthreads();
    // one warp per row, lanes across columns: the row's vertical taps are warp-uniform, the loops carry no index
    // arithmetic beyond +32, and every global store is a coalesced 128-byte line
    const int lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    for (int y = warp; y < h; y += nwarps) {
        const float* src = s_lo + y * w;
        float* dst = s_hr + y * W;
#pragma unroll 4
        for (int ox = lane; ox < W; ox += 32) {
            const float fx = s_fx[ox];
            dst[ox] = src[s_x0[ox]] * (1.f - fx) + src[s_x1[ox]] * fx;
        }
    }
    __syncthreads();
    float vmin = 3.4e38f, vmax = -3.4e38f;
    for (int oy = warp; oy < H; oy += nwarps) {
        const float fy = s_fy[oy], gy = 1.f - fy;
        const float* r0 = s_hr + s_y0[oy];
        const float* r1 = s_hr + s_y1[oy];
#pragma unroll 4
        for (int ox = lane; ox < W; ox += 32) {
            const float v = r0[ox] * gy + r1[ox] * fy;
            vmin = fminf(vmin, v);
            vmax = fmaxf(vmax, v);
        }
    }
    block_minmax(vmin, vmax, s_red);
    // x / d is evaluated as x * (1/d): within 1 ulp of the reference's true division
    const float inv2 = 1.f / (1e-7f + (vmax - vmin));
    float* ob = out + (size_t)b * out_stride;
    for (int oy = warp; oy < H; oy += nwarps) {
        const float fy = s_fy[oy], gy = 1.f - fy;
        const float* r0 = s_hr + s_y0[oy];
        const float* r1 = s_hr + s_y1[oy];
        float* orow = ob + (size_t)oy * W;
#pragma unroll 4
        for (int ox = lane; ox < W; ox += 32) orow[ox] = ((r0[ox] * gy + r1[ox] * fy) - vmin) * inv2;
    }
}

int launch_upsample_norm(const float* cam_lo, const float* mm, int mm_splits, float* out, int B, int h, int w, int H,
                         int W, cudaStream_t s, const int* n_dev, size_t out_stride) {
    if (out_stride == 0) out_stride = (size_t)H * W;
    const size_t tables = (size_t)(3 * W + 3 * H) * sizeof(float);
    const size_t lo_bytes = (size_t)h * w * sizeof(float), hr_bytes = (size_t)h * W * sizeof(float);
    if (tables + lo_bytes + hr_bytes <= 220 * 1024) {
        const size_t smem = tables + lo_bytes + hr_bytes;
        if (smem > 48 * 1024)
            BCAD_CUDA_CHECK(cudaFuncSetAttribute(upsample_norm_sep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
        upsample_norm_sep_kernel<<<B, UP_THREADS, smem, s>>>(cam_lo, mm, mm_splits, out, out_stride, h, w, H, W, n_dev);
        BCAD_CUDA_CHECK(cudaGetLastError());
        return BCAD_OK;
    }
    size_t smem = tables;
    int lo_in_smem = 0;
    if (smem + lo_bytes <= 200 * 1024) { smem += lo_bytes; lo_in_smem = 1; }
    BCAD_REQUIRE(smem <= 200 * 1024, "upsample: output %dx%d too large for the coordinate tables", H, W);
    if (smem > 48 * 1024)
        BCAD_CUDA_CHECK(cudaFuncSetAttribute(upsample_norm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    upsample_norm_kernel<<<B, UP_THREADS, smem, s>>>(cam_lo, mm, mm_splits, out, out_stride, h, w, H, W, lo_in_smem);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// =====================================================================================================
// small helpers of the tiny U-Net front (SURVEY 8 row f1)
// =====================================================================================================
__global__ void avg_pool_kernel(const float* __restrict__ x, float* __restrict__ out, int H, int W, int C, int pool,
                                int Hn, int Wn, size_t total) {
    const float inv = 1.f / (float)(pool * pool);
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % C);
        size_t r = i / C;
        const int j = (int)(r % Wn); r /= Wn;
        const int ii = (int)(r % Hn);
        const size_t b = r / Hn;
        float acc = 0.f;
        for (int u = 0; u < pool; ++u)
            for (int v = 0; v < pool; ++v) acc += x[((b * H + (size_t)ii * pool + u) * W + (size_t)j * pool + v) * C + c];
        out[i] = acc * inv;
    }
}

int launch_avg_pool(const float* x, float* out, int B, int H, int W, int C, int pool, cudaStream_t s) {
    const int Hn = H / pool, Wn = W / pool;
    const size_t total = (size_t)B * Hn * Wn * C;
    if (total == 0) return BCAD_OK;
    const int blocks = (int)min((size_t)148 * 8, (total + 255) / 256);
    avg_pool_kernel<<<blocks, 256, 0, s>>>(x, out, H, W, C, pool, Hn, Wn, total);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

__global__ void pad_conv_weights_kernel(const float* __restrict__ w, float* __restrict__ out, int rows, int Cout, int CoutPad) {
    const int total = rows * CoutPad;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int f = i % CoutPad, r = i / CoutPad;
        out[i] = f < Cout ? w[(size_t)r * Cout + f] : 0.f;
    }
}

int launch_pad_conv_weights(const float* w, float* out, int taps, int Cin, int Cout, int CoutPad, cudaStream_t s) {
    const int total = taps * Cin * CoutPad;
    pad_conv_weights_kernel<<<cdiv(total, 256), 256, 0, s>>>(w, out, taps * Cin, Cout, CoutPad);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// =====================================================================================================
// overlay: show_cam_on_image (JET LUT, 0.5/0.5 blend, /max, u8) + heatmap_uint8 (truncation)
// =====================================================================================================
__constant__ uint8_t c_jet_bgr[256 * 3] = {
#include "jet_lut.inc"
};

// One CTA per image.  The JET table sits in shared memory as the float heat values (the colour index differs from lane to lane, so
// constant memory would serialise every lookup); a thread handles 4 consecutive pixels: 16-byte loads of cam and image, one
// 12-byte store of RGB.  Pass 1: per-image maximum of the blend (+ heatmap_uint8); pass 2 (inputs come back from L2): scale, store.
__global__ void __launch_bounds__(1024)
overlay_kernel(const float* __restrict__ img01, const float* __restrict__ cam, int H, int W,
               uint8_t* __restrict__ overlay_rgb, uint8_t* __restrict__ heat_u8) {
    __shared__ float s_red[64];
    __shared__ float s_lut[256 * 3];                                       // RGB order, already / 255
    const int b = blockIdx.x, npix = H * W;
    for (int i = threadIdx.x; i < 768; i += blockDim.x) s_lut[i] = (float)c_jet_bgr[(i / 3) * 3 + (2 - i % 3)] / 255.f;   // BGR -> RGB
    __syncthreads();
    const float* ib = img01 + (size_t)b * npix;
    const float* cb = cam + (size_t)b * npix;
    const bool vec = (npix % 4 == 0) && ((reinterpret_cast<uintptr_t>(ib) | reinterpret_cast<uintptr_t>(cb)) % 16 == 0);
    const int n4 = vec ? npix / 4 : 0;
    float vmax = -3.4e38f, vmin = 0.f;
    auto blend_max = [&](float cv, float g) {
        const int li = (int)(uint8_t)(int)(255.f * cv);                   // np.uint8(255*cam): truncation
        const float* l = s_lut + li * 3;
        vmax = fmaxf(vmax, fmaxf(fmaxf(0.5f * l[0] + 0.5f * g, 0.5f * l[1] + 0.5f * g), 0.5f * l[2] + 0.5f * g));
    };
    for (int i = threadIdx.x; i < n4; i += blockDim.x) {
        const float4 c4 = __ldg(reinterpret_cast<const float4*>(cb) + i), g4 = __ldg(reinterpret_cast<const float4*>(ib) + i);
        blend_max(c4.x, g4.x); blend_max(c4.y, g4.y); blend_max(c4.z, g4.z); blend_max(c4.w, g4.w);
        if (heat_u8 != nullptr) {
            uchar4 o;
            o.x = (uint8_t)(int)(c4.x * 255.f); o.y = (uint8_t)(int)(c4.y * 255.f); o.z = (uint8_t)(int)(c4.z * 255.f); o.w = (uint8_t)(int)(c4.w * 255.f);
            reinterpret_cast<uchar4*>(heat_u8 + (size_t)b * npix)[i] = o;
        }
    }
    for (int i = n4 * 4 + threadIdx.x; i < npix; i += blockDim.x) {
        blend_max(cb[i], ib[i]);
        if (heat_u8 != nullptr) heat_u8[(size_t)b * npix + i] = (uint8_t)(int)(cb[i] * 255.f);
    }
    if (overlay_rgb == nullptr) return;
    block_minmax(vmin, vmax, s_red);
    auto rgb = [&](float cv, float g, uint8_t* o) {
        const int li = (int)(uint8_t)(int)(255.f * cv);
        const float* l = s_lut + li * 3;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) o[ch] = (uint8_t)(int)(255.f * ((0.5f * l[ch] + 0.5f * g) / vmax));
    };
    uint8_t* ob = overlay_rgb + (size_t)b * npix * 3;
    const bool vst = vec && (reinterpret_cast<uintptr_t>(ob) % 4 == 0);
    for (int i = threadIdx.x; i < n4; i += blockDim.x) {
        const float4 c4 = __ldg(reinterpret_cast<const float4*>(cb) + i), g4 = __ldg(reinterpret_cast<const float4*>(ib) + i);
        uint8_t o[12];
        rgb(c4.x, g4.x, o); rgb(c4.y, g4.y, o + 3); rgb(c4.z, g4.z, o + 6); rgb(c4.w, g4.w, o + 9);
        if (vst) {
            uint32_t* d = reinterpret_cast<uint32_t*>(ob + (size_t)i * 12);
#pragma unroll
            for (int q = 0; q < 3; ++q) d[q] = (uint32_t)o[4 * q] | ((uint32_t)o[4 * q + 1] << 8) | ((uint32_t)o[4 * q + 2] << 16) | ((uint32_t)o[4 * q + 3] << 24);
        } else {
#pragma unroll
            for (int q = 0; q < 12; ++q) ob[(size_t)i * 12 + q] = o[q];
        }
    }
    for (int i = n4 * 4 + threadIdx.x; i < npix; i += blockDim.x) rgb(cb[i], ib[i], ob + (size_t)i * 3);
}

// generate_saliency_overlay (explainability.py:74-77) for [B][K] saliency maps: heat = JET_BGR[uint8(s * 255)] (fp32 product,
// truncation), overlay = addWeighted(base, 0.5, heat, 0.5, 0).  OpenCV's 8-bit path rounds a * 0.5 + b * 0.5 half to even, i.e.
// (a + b) / 2 with an odd sum rounded to the even neighbour.  The base image (1 channel replicated, or BGR) is shared by an image's K maps.
__global__ void __launch_bounds__(256) saliency_overlay_kernel(const uint8_t* __restrict__ base, int base_c, const float* __restrict__ sal,
                                                               int K, size_t npix, size_t total, uint8_t* __restrict__ overlay,
                                                               uint8_t* __restrict__ heat) {
    __shared__ uint8_t s_lut[256 * 3];
    for (int i = threadIdx.x; i < 768; i += blockDim.x) s_lut[i] = c_jet_bgr[i];
    __syncthreads();
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {   // i = map * npix + p
        const size_t img = i / npix / K, p = i % npix;
        const int li = (int)(uint8_t)(int)(sal[i] * 255.f);
        const uint8_t* px = base + (img * npix + p) * base_c;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
            const int h = s_lut[li * 3 + ch];
            if (heat) heat[i * 3 + ch] = (uint8_t)h;
            if (overlay) {
                const int sum = px[base_c == 3 ? ch : 0] + h, q = sum >> 1;
                overlay[i * 3 + ch] = (uint8_t)(q + (sum & q & 1));
            }
        }
    }
}

// heatmap_uint8 = (cam * 255).astype(np.uint8)  (GRADCAM.py:70: truncation), 4 pixels per thread
__global__ void __launch_bounds__(256) heat_to_u8_kernel(const float* __restrict__ cam, uint8_t* __restrict__ out, size_t n) {
    const size_t n4 = n / 4;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
        const float4 v = ldg_stream(reinterpret_cast<const float4*>(cam) + i);
        uchar4 o;
        o.x = (uint8_t)(int)(v.x * 255.f); o.y = (uint8_t)(int)(v.y * 255.f); o.z = (uint8_t)(int)(v.z * 255.f); o.w = (uint8_t)(int)(v.w * 255.f);
        reinterpret_cast<uchar4*>(out)[i] = o;
    }
    for (size_t i = n4 * 4 + blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = (uint8_t)(int)(cam[i] * 255.f);
}

int launch_heat_to_u8(const float* cam, uint8_t* out, size_t n, cudaStream_t s) {
    const int blocks = (int)std::min<size_t>((size_t)148 * 8, (n / 4 + 255) / 256 + 1);
    heat_to_u8_kernel<<<blocks, 256, 0, s>>>(cam, out, n);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// 8-bit pixels -> the unit-range float32 image the CNN takes: x = float32(u8) / 255.0f, IEEE division (app.py:71
// `torch.tensor(resized, dtype=torch.float32) / 255.0`; GRADCAM.py:46 `img / 255.0`), 16 pixels per thread
__global__ void __launch_bounds__(256) u8_to_unit_kernel(const uint8_t* __restrict__ src, float* __restrict__ dst, size_t n) {
    const size_t n16 = n / 16;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) {
        const uint4 v = ldg_stream_u4(reinterpret_cast<const uint4*>(src) + i);
        const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float4 o;
            o.x = __fdiv_rn((float)(w[j] & 0xffu), 255.f);         o.y = __fdiv_rn((float)((w[j] >> 8) & 0xffu), 255.f);
            o.z = __fdiv_rn((float)((w[j] >> 16) & 0xffu), 255.f); o.w = __fdiv_rn((float)(w[j] >> 24), 255.f);
            reinterpret_cast<float4*>(dst)[i * 4 + j] = o;
        }
    }
    for (size_t i = n16 * 16 + blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = __fdiv_rn((float)src[i], 255.f);
}

int launch_u8_to_unit(const uint8_t* src, float* dst, size_t n, cudaStream_t s) {
    const int blocks = (int)std::min<size_t>((size_t)148 * 8, (n / 16 + 255) / 256 + 1);
    u8_to_unit_kernel<<<blocks, 256, 0, s>>>(src, dst, n);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// 8-bit grey image -> img01 = u8 / 255 (GRADCAM.py:46) and the CNN input: per-image standardisation (x - mean) / (std + 1e-8) as the
// reference prepares its CNN inputs (app.py:179-182), the single channel replicated to C.  mean / std from exact integer sums.
// img01 may be null (gray_resize_preprocess at the model's size: the overlay reads the 8-bit image itself).
__global__ void __launch_bounds__(512) gray_preprocess_kernel(const uint8_t* __restrict__ g8, float* __restrict__ img01, float* __restrict__ x,
                                                              int npix, int C, int standardise) {
    __shared__ unsigned long long s_sum[16], s_sq[16];
    __shared__ float s_mean, s_den;
    const int b = blockIdx.x, tid = threadIdx.x;
    const uint8_t* src = g8 + (size_t)b * npix;
    if (standardise) {
        unsigned long long sum = 0, sq = 0;
        if (npix % 4 == 0 && (reinterpret_cast<uintptr_t>(src) & 3) == 0) {
            unsigned s32 = 0, q32 = 0;                       // per thread <= npix / 512 * 255^2: fits 32 bits up to 33 M pixels
            for (int i = tid; i < npix / 4; i += 512) {
                const uchar4 q = reinterpret_cast<const uchar4*>(src)[i];
                s32 += q.x + q.y + q.z + q.w;
                q32 += q.x * q.x + q.y * q.y + q.z * q.z + q.w * q.w;
            }
            sum = s32; sq = q32;
        } else
        for (int i = tid; i < npix; i += 512) { const unsigned v = src[i]; sum += v; sq += v * v; }
        for (int o = 16; o > 0; o >>= 1) { sum += __shfl_xor_sync(0xffffffffu, sum, o); sq += __shfl_xor_sync(0xffffffffu, sq, o); }
        if ((tid & 31) == 0) { s_sum[tid >> 5] = sum; s_sq[tid >> 5] = sq; }
        __syncthreads();
        if (tid == 0) {
            unsigned long long ts = 0, tq = 0;
            for (int w = 0; w < 16; ++w) { ts += s_sum[w]; tq += s_sq[w]; }
            const double mean = (double)ts / (255.0 * npix);
            const double var = (double)tq / (65025.0 * npix) - mean * mean;
            s_mean = (float)mean;
            s_den = (float)sqrt(var > 0.0 ? var : 0.0) + 1e-8f;
        }
        __syncthreads();
    }
    const float mean = standardise ? s_mean : 0.f, den = standardise ? s_den : 1.f;
    float* ib = img01 + (size_t)b * npix;
    float* xb = x + (size_t)b * npix * C;
    if (C == 1 && npix % 4 == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(ib) | reinterpret_cast<uintptr_t>(xb)) & 15) == 0) {
        for (int i = tid; i < npix / 4; i += 512) {           // 4 pixels per thread: one 4-byte load, two 16-byte stores
            const uchar4 q = reinterpret_cast<const uchar4*>(src)[i];
            const float4 v = make_float4((float)q.x / 255.0f, (float)q.y / 255.0f, (float)q.z / 255.0f, (float)q.w / 255.0f);
            if (img01) reinterpret_cast<float4*>(ib)[i] = v;
            reinterpret_cast<float4*>(xb)[i] = standardise ? make_float4((v.x - mean) / den, (v.y - mean) / den, (v.z - mean) / den, (v.w - mean) / den) : v;
        }
        return;
    }
    for (int i = tid; i < npix; i += 512) {
        const float v = (float)src[i] / 255.0f;
        if (img01) ib[i] = v;
        const float xv = standardise ? (v - mean) / den : v;
        for (int c = 0; c < C; ++c) xb[(size_t)i * C + c] = xv;
    }
}

int launch_gray_preprocess(const uint8_t* g8, float* img01, float* x, int B, int npix, int C, int standardise, cudaStream_t s) {
    gray_preprocess_kernel<<<B, 512, 0, s>>>(g8, img01, x, npix, C, standardise);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

int launch_overlay(const float* img01, const float* cam, int B, int H, int W, uint8_t* overlay_rgb, uint8_t* heat_u8,
                   cudaStream_t s) {
    overlay_kernel<<<B, 1024, 0, s>>>(img01, cam, H, W, overlay_rgb, heat_u8);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

int launch_saliency_overlay(const uint8_t* base, int base_c, const float* sal, int B, int K, int npix, uint8_t* overlay, uint8_t* heat,
                            cudaStream_t s) {
    const size_t total = (size_t)B * K * npix;
    const int blocks = (int)std::min((size_t)148 * 16, (total + 255) / 256);
    saliency_overlay_kernel<<<blocks, 256, 0, s>>>(base, base_c, sal, K, (size_t)npix, total, overlay, heat);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// OpenCV's INTER_LINEAR source coordinate of destination index d (ns source, nd destination pixels): scale = 1 / (nd / ns) in double as
// cv::resize forms it, f = float((d + 0.5) * scale - 0.5) without FMA contraction, s = floor(f), f -= s.
__device__ __forceinline__ void cv_linear_coord(int d, int ns, int nd, int& s, float& f) {
    const double scale = 1.0 / ((double)nd / (double)ns);
    f = (float)__dsub_rn(__dmul_rn((double)d + 0.5, scale), 0.5);
    const float fl = floorf(f);
    s = (int)fl;
    f -= fl;
}

// generate_saliency_overlay (explainability.py:74-77) at the image's size for [B][K] model-size maps: the JET heat-map of the map
// (applyColorMap(uint8(s * 255)), built on the fly for the 2x2 source neighbourhood of each output pixel), cv2.resize of that 3-channel
// 8-bit image to img_h x img_w with OpenCV's fixed-point INTER_LINEAR (11-bit weights c = rint(w * 2048); columns clamp the coordinate at
// both borders, rows only their indices; vertical step ((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2, saturated), then
// addWeighted(grey3, 0.5, heat, 0.5, 0) with saliency_overlay_kernel's round-half-even blend.  The grey image is read once per pixel for
// all K maps.  CTA = SOR_ROWS output rows of SOR_THREADS x 4 consecutive pixels; a row's weights are warp-uniform.  The table comes
// from a global copy, 4 bytes per thread: read from constant memory, the divergent addresses serialise, and with many small CTAs that
// load cost more than the colouring (64 images at 512 x 512, K = 2: 0.40 ms with one-row CTAs and the constant table, 0.21 ms so; one
// B200 at a 1000 W limit).
constexpr int SOR_THREADS = 64, SOR_ROWS = 4;
__device__ __align__(4) uint8_t g_jet_bgr[256 * 3] = {
#include "jet_lut.inc"
};

template <int K>
__global__ void __launch_bounds__(SOR_THREADS * SOR_ROWS) saliency_overlay_resized_kernel(const uint8_t* __restrict__ g8,
                                                                                          const float* __restrict__ sal, int H, int W,
                                                                                          int hi, int wi, uint8_t* __restrict__ overlay,
                                                                                          uint8_t* __restrict__ heat) {
    __shared__ __align__(4) uint8_t s_lut[256 * 3];
    const int tid = threadIdx.y * SOR_THREADS + threadIdx.x;
    if (tid < 192) reinterpret_cast<uint32_t*>(s_lut)[tid] = __ldg(reinterpret_cast<const uint32_t*>(g_jet_bgr) + tid);
    __syncthreads();
    const int b = blockIdx.z, dy = blockIdx.y * SOR_ROWS + threadIdx.y, dx0 = (blockIdx.x * SOR_THREADS + threadIdx.x) * 4;
    if (dx0 >= wi || dy >= hi) return;
    int sy;
    float fy;
    cv_linear_coord(dy, H, hi, sy, fy);
    const int b0 = __float2int_rn((1.f - fy) * 2048.f), b1 = __float2int_rn(fy * 2048.f);
    const int y0 = min(max(sy, 0), H - 1), y1 = min(max(sy + 1, 0), H - 1);
    int x0[4], x1[4], c0[4], c1[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        int sx;
        float fx;
        cv_linear_coord(min(dx0 + j, wi - 1), W, wi, sx, fx);
        if (sx < 0) { fx = 0.f; sx = 0; }
        if (sx >= W - 1) { fx = 0.f; sx = W - 1; }
        x0[j] = sx;
        x1[j] = min(sx + 1, W - 1);
        c0[j] = __float2int_rn((1.f - fx) * 2048.f);
        c1[j] = __float2int_rn(fx * 2048.f);
    }
    const size_t hw = (size_t)hi * wi, px0 = (size_t)dy * wi + dx0;
    const int npx = min(4, wi - dx0);
    int g[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) g[j] = j < npx ? __ldg(g8 + (size_t)b * hw + px0 + j) : 0;
    const bool vst = npx == 4 && (wi & 3) == 0 && ((reinterpret_cast<uintptr_t>(overlay) | reinterpret_cast<uintptr_t>(heat)) & 3) == 0;
    auto lut_index = [](float v) { return 3 * (int)(uint8_t)(int)(v * 255.f); };
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const float* m = sal + ((size_t)b * K + k) * H * W;
        const float* r0 = m + (size_t)y0 * W;
        const float* r1 = m + (size_t)y1 * W;
        uint8_t hv[12], ov[12];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int i00 = lut_index(__ldg(r0 + x0[j])), i01 = lut_index(__ldg(r0 + x1[j]));
            const int i10 = lut_index(__ldg(r1 + x0[j])), i11 = lut_index(__ldg(r1 + x1[j]));
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
                const int h0 = s_lut[i00 + ch] * c0[j] + s_lut[i01 + ch] * c1[j];
                const int h1 = s_lut[i10 + ch] * c0[j] + s_lut[i11 + ch] * c1[j];
                const int v = min(max((((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2, 0), 255);
                const int sum = g[j] + v, q = sum >> 1;
                hv[3 * j + ch] = (uint8_t)v;
                ov[3 * j + ch] = (uint8_t)(q + (sum & q & 1));
            }
        }
        const size_t o = (((size_t)b * K + k) * hw + px0) * 3;
        if (vst) {
#pragma unroll
            for (int w = 0; w < 3; ++w) {
                if (heat) reinterpret_cast<uint32_t*>(heat + o)[w] = (uint32_t)hv[4 * w] | ((uint32_t)hv[4 * w + 1] << 8) |
                                                                      ((uint32_t)hv[4 * w + 2] << 16) | ((uint32_t)hv[4 * w + 3] << 24);
                if (overlay) reinterpret_cast<uint32_t*>(overlay + o)[w] = (uint32_t)ov[4 * w] | ((uint32_t)ov[4 * w + 1] << 8) |
                                                                            ((uint32_t)ov[4 * w + 2] << 16) | ((uint32_t)ov[4 * w + 3] << 24);
            }
        } else {
#pragma unroll
            for (int q = 0; q < 12; ++q) {
                if (q >= 3 * npx) break;
                if (heat) heat[o + q] = hv[q];
                if (overlay) overlay[o + q] = ov[q];
            }
        }
    }
}

int launch_saliency_overlay_resized(const uint8_t* g8, const float* sal, int B, int K, int H, int W, int hi, int wi, uint8_t* overlay,
                                    uint8_t* heat, cudaStream_t s) {
    if (hi == H && wi == W) return launch_saliency_overlay(g8, 1, sal, B, K, H * W, overlay, heat, s);   // cv2.resize to the same size copies
    const dim3 grid(cdiv(wi, 4 * SOR_THREADS), cdiv(hi, SOR_ROWS), B), block(SOR_THREADS, SOR_ROWS);
    switch (K) {
#define BCAD_SOR(k) case k: saliency_overlay_resized_kernel<k><<<grid, block, 0, s>>>(g8, sal, H, W, hi, wi, overlay, heat); break;
        BCAD_SOR(1) BCAD_SOR(2) BCAD_SOR(3) BCAD_SOR(4) BCAD_SOR(5) BCAD_SOR(6) BCAD_SOR(7) BCAD_SOR(8)
#undef BCAD_SOR
        default: set_error("saliency_overlay_resized: K=%d out of range 1..%d", K, BCAD_MAX_EXPLAIN_CLASSES); return BCAD_ERR_INVALID;
    }
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// =====================================================================================================
// The dual-class overlay call for grey images of any size (bcad_gradcam_overlays_classes_host)
// =====================================================================================================
// cv2.resize(u8 / 255.0f, (W, H), INTER_LINEAR) of one channel with the <= 4-channel arithmetic of bottleneck_resize_kernel
// (coordinate in double, weight = float(frac), no FMA contraction): the two kernels agree bit for bit.
__device__ __forceinline__ void resize_coord_d(int d, int ns, int nd, int& i0, int& i1, float& f) {
    const double sd = ((double)d + 0.5) * ((double)ns / (double)nd) - 0.5;
    i0 = (int)floor(sd);
    f = (float)(sd - (double)i0);
    if (i0 < 0) { i0 = 0; f = 0.f; }
    if (i0 >= ns - 1) { i0 = ns - 1; f = 0.f; }
    i1 = min(i0 + 1, ns - 1);
}

__device__ __forceinline__ float resize_gray_px(const uint8_t* __restrict__ src, int hi, int wi, int H, int W, int p) {
    int x0, x1, y0, y1;
    float fx, fy;
    resize_coord_d(p % W, wi, W, x0, x1, fx);
    resize_coord_d(p / W, hi, H, y0, y1, fy);
    auto at = [&](int y, int x) { return (float)__ldg(src + (size_t)y * wi + x) / 255.0f; };
    const float gx = __fsub_rn(1.f, fx), gy = __fsub_rn(1.f, fy);
    const float top = __fadd_rn(__fmul_rn(at(y0, x0), gx), __fmul_rn(at(y0, x1), fx));
    const float bot = __fadd_rn(__fmul_rn(at(y1, x0), gx), __fmul_rn(at(y1, x1), fx));
    return __fadd_rn(__fmul_rn(top, gy), __fmul_rn(bot, fy));
}

// One CTA per image.  Pass 1: resized pixels and their sum / sum of squares in float64, thread-strided then a fixed-order warp and
// block reduction (deterministic); pass 2 recomputes each pixel (four 8-bit reads) and stores (v - mean) / (std + 1e-8), or v.
constexpr int GRP_THREADS = 512;
__global__ void __launch_bounds__(GRP_THREADS) gray_resize_preprocess_kernel(const uint8_t* __restrict__ g8, float* __restrict__ x, int hi,
                                                                             int wi, int H, int W, int C, int standardise) {
    __shared__ double s_sum[GRP_THREADS / 32], s_sq[GRP_THREADS / 32];
    __shared__ float s_mean, s_den;
    const int b = blockIdx.x, tid = threadIdx.x, npix = H * W;
    const uint8_t* src = g8 + (size_t)b * hi * wi;
    if (standardise) {
        double sum = 0.0, sq = 0.0;
        for (int p = tid; p < npix; p += GRP_THREADS) {
            const double v = (double)resize_gray_px(src, hi, wi, H, W, p);
            sum += v;
            sq += v * v;
        }
        for (int o = 16; o > 0; o >>= 1) { sum += __shfl_xor_sync(0xffffffffu, sum, o); sq += __shfl_xor_sync(0xffffffffu, sq, o); }
        if ((tid & 31) == 0) { s_sum[tid >> 5] = sum; s_sq[tid >> 5] = sq; }
        __syncthreads();
        if (tid == 0) {
            double ts = 0.0, tq = 0.0;
            for (int w = 0; w < GRP_THREADS / 32; ++w) { ts += s_sum[w]; tq += s_sq[w]; }
            const double mean = ts / npix;
            const double var = tq / npix - mean * mean;
            s_mean = (float)mean;
            s_den = (float)sqrt(var > 0.0 ? var : 0.0) + 1e-8f;
        }
        __syncthreads();
    }
    const float mean = standardise ? s_mean : 0.f, den = standardise ? s_den : 1.f;
    float* xb = x + (size_t)b * npix * C;
    for (int p = tid; p < npix; p += GRP_THREADS) {
        const float v = resize_gray_px(src, hi, wi, H, W, p);
        const float xv = standardise ? (v - mean) / den : v;
        for (int c = 0; c < C; ++c) xb[(size_t)p * C + c] = xv;
    }
}

int launch_gray_resize_preprocess(const uint8_t* g8, float* x, int B, int hi, int wi, int H, int W, int C, int standardise, cudaStream_t s) {
    if (hi == H && wi == W) {
        // the model's own size: exactly gray_preprocess (exact integer sums), without its image-size float copy
        gray_preprocess_kernel<<<B, 512, 0, s>>>(g8, nullptr, x, H * W, C, standardise);
    } else {
        gray_resize_preprocess_kernel<<<B, GRP_THREADS, 0, s>>>(g8, x, hi, wi, H, W, C, standardise);
    }
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// overlay_kernel for the K maps of each grey image, reading the 8-bit image once per pixel for all of them: g = (float)q / 255.0f (the
// gray_preprocess expression), the same JET table, blend and two passes, so every map is byte for byte overlay_kernel on img01 = u8 / 255.
// One CTA per image; a thread takes 4 consecutive pixels: a 4-byte image load and a 16-byte cam load per map, 12-byte RGB stores.
template <int K>
__global__ void __launch_bounds__(1024)
overlay_classes_kernel(const uint8_t* __restrict__ g8, const float* __restrict__ cam, int npix, uint8_t* __restrict__ overlay_rgb,
                       uint8_t* __restrict__ heat_u8) {
    __shared__ float s_red[64];
    __shared__ float s_lut[256 * 3];                                       // RGB order, already / 255
    const int b = blockIdx.x;
    for (int i = threadIdx.x; i < 768; i += blockDim.x) s_lut[i] = (float)c_jet_bgr[(i / 3) * 3 + (2 - i % 3)] / 255.f;   // BGR -> RGB
    __syncthreads();
    const uint8_t* gb = g8 + (size_t)b * npix;
    const float* cb = cam + (size_t)b * K * npix;                          // map k at cb + k * npix
    const bool vec = (npix % 4 == 0) && (reinterpret_cast<uintptr_t>(gb) % 4 == 0) && (reinterpret_cast<uintptr_t>(cb) % 16 == 0);
    const int n4 = vec ? npix / 4 : 0;
    float vmax[K];
#pragma unroll
    for (int k = 0; k < K; ++k) vmax[k] = -3.4e38f;
    auto blend_max = [&](float& m, float cv, float g) {
        const int li = (int)(uint8_t)(int)(255.f * cv);                   // np.uint8(255*cam): truncation
        const float* l = s_lut + li * 3;
        m = fmaxf(m, fmaxf(fmaxf(0.5f * l[0] + 0.5f * g, 0.5f * l[1] + 0.5f * g), 0.5f * l[2] + 0.5f * g));
    };
    for (int i = threadIdx.x; i < n4; i += blockDim.x) {
        const uchar4 q = reinterpret_cast<const uchar4*>(gb)[i];
        const float4 g4 = make_float4((float)q.x / 255.0f, (float)q.y / 255.0f, (float)q.z / 255.0f, (float)q.w / 255.0f);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const float4 c4 = __ldg(reinterpret_cast<const float4*>(cb + (size_t)k * npix) + i);
            blend_max(vmax[k], c4.x, g4.x); blend_max(vmax[k], c4.y, g4.y); blend_max(vmax[k], c4.z, g4.z); blend_max(vmax[k], c4.w, g4.w);
            if (heat_u8 != nullptr) {
                uchar4 o;
                o.x = (uint8_t)(int)(c4.x * 255.f); o.y = (uint8_t)(int)(c4.y * 255.f); o.z = (uint8_t)(int)(c4.z * 255.f); o.w = (uint8_t)(int)(c4.w * 255.f);
                reinterpret_cast<uchar4*>(heat_u8 + ((size_t)b * K + k) * npix)[i] = o;
            }
        }
    }
    for (int i = n4 * 4 + threadIdx.x; i < npix; i += blockDim.x) {
        const float g = (float)gb[i] / 255.0f;
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const float cv = cb[(size_t)k * npix + i];
            blend_max(vmax[k], cv, g);
            if (heat_u8 != nullptr) heat_u8[((size_t)b * K + k) * npix + i] = (uint8_t)(int)(cv * 255.f);
        }
    }
    if (overlay_rgb == nullptr) return;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        float vmin = 0.f;
        block_minmax(vmin, vmax[k], s_red);
    }
    auto rgb = [&](float m, float cv, float g, uint8_t* o) {
        const int li = (int)(uint8_t)(int)(255.f * cv);
        const float* l = s_lut + li * 3;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) o[ch] = (uint8_t)(int)(255.f * ((0.5f * l[ch] + 0.5f * g) / m));
    };
    uint8_t* ob = overlay_rgb + (size_t)b * K * npix * 3;                  // map k at ob + k * npix * 3
    const bool vst = vec && (reinterpret_cast<uintptr_t>(ob) % 4 == 0);
    for (int i = threadIdx.x; i < n4; i += blockDim.x) {
        const uchar4 q = reinterpret_cast<const uchar4*>(gb)[i];
        const float4 g4 = make_float4((float)q.x / 255.0f, (float)q.y / 255.0f, (float)q.z / 255.0f, (float)q.w / 255.0f);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            const float4 c4 = __ldg(reinterpret_cast<const float4*>(cb + (size_t)k * npix) + i);
            uint8_t o[12];
            rgb(vmax[k], c4.x, g4.x, o); rgb(vmax[k], c4.y, g4.y, o + 3); rgb(vmax[k], c4.z, g4.z, o + 6); rgb(vmax[k], c4.w, g4.w, o + 9);
            uint8_t* d8 = ob + (size_t)k * npix * 3 + (size_t)i * 12;
            if (vst) {
                uint32_t* d = reinterpret_cast<uint32_t*>(d8);
#pragma unroll
                for (int w = 0; w < 3; ++w) d[w] = (uint32_t)o[4 * w] | ((uint32_t)o[4 * w + 1] << 8) | ((uint32_t)o[4 * w + 2] << 16) | ((uint32_t)o[4 * w + 3] << 24);
            } else {
#pragma unroll
                for (int w = 0; w < 12; ++w) d8[w] = o[w];
            }
        }
    }
    for (int i = n4 * 4 + threadIdx.x; i < npix; i += blockDim.x) {
        const float g = (float)gb[i] / 255.0f;
#pragma unroll
        for (int k = 0; k < K; ++k) rgb(vmax[k], cb[(size_t)k * npix + i], g, ob + ((size_t)k * npix + i) * 3);
    }
}

int launch_overlay_classes(const uint8_t* g8, const float* cam, int B, int K, int npix, uint8_t* overlay_rgb, uint8_t* heat_u8,
                           cudaStream_t s) {
    switch (K) {
#define BCAD_OVC(k) case k: overlay_classes_kernel<k><<<B, 1024, 0, s>>>(g8, cam, npix, overlay_rgb, heat_u8); break;
        BCAD_OVC(1) BCAD_OVC(2) BCAD_OVC(3) BCAD_OVC(4) BCAD_OVC(5) BCAD_OVC(6) BCAD_OVC(7) BCAD_OVC(8)
#undef BCAD_OVC
        default: set_error("overlay_classes: K=%d out of range 1..%d", K, BCAD_MAX_EXPLAIN_CLASSES); return BCAD_ERR_INVALID;
    }
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// =====================================================================================================
// process_bottleneck_features (app.py:466-489): [C,H,W] (or [H,W,C]) -> cv2.resize(INTER_LINEAR) -> [h,w,C].
// OpenCV's > 4-channel float path: source coordinate and weight in float32 (fx = (float)((dx+0.5)*scale-0.5); sx = floor;
// fx -= sx), horizontal pass then vertical, no FMA contraction (bit-exact against tests/golden/ref_bottleneck.npz);
// <= 4 channels: coordinate in double, weight = float(frac) as in the Grad-CAM tail.  thread = one output element, channel
// fastest so the HWC stores are coalesced (only 4 source pixels per output are ever read: the pass is tiny).
// =====================================================================================================
__global__ void __launch_bounds__(256) bottleneck_resize_kernel(const float* __restrict__ src, float* __restrict__ dst, int C, int H,
                                                                int W, int chw, int oh, int ow, size_t total) {
    const bool f32c = C > 4;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % C);
        size_t r = i / C;
        const int ox = (int)(r % ow);
        r /= ow;
        const int oy = (int)(r % oh);
        const size_t b = r / oh;
        auto coord = [&](int d, int ns, int nd, int& i0, int& i1, float& f) {
            const double sd = ((double)d + 0.5) * ((double)ns / (double)nd) - 0.5;
            if (f32c) {
                const float sf = (float)sd;
                const float fl = floorf(sf);
                i0 = (int)fl;
                f = __fsub_rn(sf, fl);
            } else {
                i0 = (int)floor(sd);
                f = (float)(sd - (double)i0);
            }
            if (i0 < 0) { i0 = 0; f = 0.f; }
            if (i0 >= ns - 1) { i0 = ns - 1; f = 0.f; }
            i1 = min(i0 + 1, ns - 1);
        };
        int x0, x1, y0, y1;
        float fx, fy;
        coord(ox, W, ow, x0, x1, fx);
        coord(oy, H, oh, y0, y1, fy);
        const float* sb = src + b * (size_t)C * H * W;
        auto at = [&](int y, int x) { return chw ? __ldg(sb + ((size_t)c * H + y) * W + x) : __ldg(sb + ((size_t)y * W + x) * C + c); };
        const float gx = __fsub_rn(1.f, fx), gy = __fsub_rn(1.f, fy);
        const float top = __fadd_rn(__fmul_rn(at(y0, x0), gx), __fmul_rn(at(y0, x1), fx));
        const float bot = __fadd_rn(__fmul_rn(at(y1, x0), gx), __fmul_rn(at(y1, x1), fx));
        dst[i] = __fadd_rn(__fmul_rn(top, gy), __fmul_rn(bot, fy));
    }
}

int launch_bottleneck_resize(const float* src, float* dst, int B, int C, int H, int W, int chw, int oh, int ow, cudaStream_t s) {
    const size_t total = (size_t)B * oh * ow * C;
    const int blocks = (int)std::min<size_t>((size_t)148 * 8, (total + 255) / 256);
    bottleneck_resize_kernel<<<blocks, 256, 0, s>>>(src, dst, C, H, W, chw, oh, ow, total);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

// =====================================================================================================
// fused dense head (one CTA per image): fc1 split-K reduce + bias + LeakyReLU, the remaining dense layers,
// probabilities / class, and -- when explaining -- the top gradient and the dense backward down to dz1
// plus the Grad-CAM channel weights through the alpha shortcut  alpha_raw[k] = sum_u dz1[u] S[u][k].
// Replaces ~12 tiny launches of the layer-by-layer path (explainability.py:20-34, Classes/CNNModel.py:177-212).
// =====================================================================================================
__global__ void __launch_bounds__(256) dense_head_kernel(HeadArgs a) {
    extern __shared__ __align__(16) float sh[];   // z of every layer, then activations / gradients scratch
    __shared__ int s_cls;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (a.n_dev != nullptr && b >= *a.n_dev) return;      // refinement twin: only the flagged images are live
    int off[BCAD_MAX_DENSE + 1];
    off[0] = 0;
    for (int j = 0; j < a.n_dense; ++j) off[j + 1] = off[j] + a.sizes[j];
    float* s_z = sh;                              // [sum sizes]
    float* s_v = sh + ((off[a.n_dense] + 3) & ~3); // activation vector of the current layer (max size), 16-byte aligned
    float* s_g = s_v + a.max_size;                // gradient vector (max size)
    // ---- layer 0: reduce the split-K partials in a fixed order
    const int n0 = a.sizes[0];
    for (int u = tid; u < n0; u += 256) {
        float v = 0.f;
        // fixed summation order; unrolled so that 8 partial loads are in flight (the kernel is a chain of L2 latencies)
#pragma unroll 8
        for (int sidx = 0; sidx < a.fc1_splits; ++sidx) v += a.fc1_part[(size_t)sidx * a.fc1_ld + (size_t)b * n0 + u];
        v += __ldg(a.bias[0] + u);
        s_z[u] = v;
        a.z[0][(size_t)b * n0 + u] = v;
        s_v[u] = (a.n_dense > 1) ? leaky(v, a.alpha) : v;
    }
    __syncthreads();
    // ---- layers 1..: one warp per output row, lanes across the input (coalesced weight reads)
    for (int j = 1; j < a.n_dense; ++j) {
        const int nin = a.sizes[j - 1], nout = a.sizes[j];
        const float* Wj = a.W[j];
        // four output rows at a time per warp (independent weight loads in flight); 16-byte loads when the row length allows
        const bool vec4 = (nin % 4 == 0);
        for (int v0 = warp * 4; v0 < nout; v0 += 32) {
            float acc[4] = {0.f, 0.f, 0.f, 0.f};
            if (vec4) {
                for (int u = lane * 4; u < nin; u += 128) {
                    const float4 x = *reinterpret_cast<const float4*>(s_v + u);
#pragma unroll
                    for (int r = 0; r < 4; ++r)
                        if (v0 + r < nout) {
                            const float4 w = __ldg(reinterpret_cast<const float4*>(Wj + (size_t)(v0 + r) * nin + u));
                            acc[r] = fmaf(w.x, x.x, fmaf(w.y, x.y, fmaf(w.z, x.z, fmaf(w.w, x.w, acc[r]))));
                        }
                }
            } else {
                for (int u = lane; u < nin; u += 32) {
                    const float x = s_v[u];
#pragma unroll
                    for (int r = 0; r < 4; ++r)
                        if (v0 + r < nout) acc[r] = fmaf(__ldg(Wj + (size_t)(v0 + r) * nin + u), x, acc[r]);
                }
            }
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const float t = warp_sum(acc[r]);
                if (lane == 0 && v0 + r < nout) {
                    const int v = v0 + r;
                    const float zz = t + __ldg(a.bias[j] + v);
                    s_z[off[j] + v] = zz;
                    a.z[j][(size_t)b * nout + v] = zz;
                }
            }
        }
        __syncthreads();
        for (int v = tid; v < nout; v += 256) s_v[v] = (j + 1 < a.n_dense) ? leaky(s_z[off[j] + v], a.alpha) : s_z[off[j] + v];
        __syncthreads();
    }
    // ---- probabilities + class (float64 like the NumPy reference)
    const int nc = a.sizes[a.n_dense - 1];
    const float* logit = s_z + off[a.n_dense - 1];
    if (tid == 0) {
        double zmax = -1e300;
        for (int c = 0; c < nc; ++c) {
            double v = (double)logit[c];
            if (a.head == BCAD_HEAD_SOFTMAX_CLIP) v = fmin(fmax(v, -50.0), 50.0);
            zmax = fmax(zmax, v);
        }
        double sum = 0.0;
        for (int c = 0; c < nc; ++c) {
            double v = (double)logit[c];
            if (a.head == BCAD_HEAD_SOFTMAX_CLIP) v = fmin(fmax(v, -50.0), 50.0);
            sum += exp(v - zmax);
        }
        int best = 0;
        double best_v = -1e300;
        for (int c = 0; c < nc; ++c) {
            double v = (double)logit[c];
            if (a.head == BCAD_HEAD_SOFTMAX_CLIP) v = fmin(fmax(v, -50.0), 50.0);
            const double p = (a.head == BCAD_HEAD_SOFTMAX_CLIP) ? exp(v - zmax) / (sum + 1e-12) : exp(v - zmax) / sum;
            a.probs[(size_t)b * nc + c] = (float)p;
            s_g[c] = (float)p;
            const double score = (a.head == BCAD_HEAD_SOFTMAX_CLIP) ? p : (double)logit[c];
            if (score > best_v) { best_v = score; best = c; }
        }
        a.cls[b] = best;
        s_cls = best;
    }
    __syncthreads();
    if (!a.explain) return;
    // ---- top gradient (explainability.py:21-22 / GRADCAM.py:64)
    const int target = a.class_idx != nullptr ? a.class_idx[b] : s_cls;
    for (int c = tid; c < nc; c += 256) {
        const float onehot = (c == target) ? 1.f : 0.f;
        s_g[c] = (a.grad_mode == BCAD_GRAD_LOGIT) ? onehot : s_g[c] - onehot;
    }
    __syncthreads();
    // ---- backward: d(h_{j-1}) = W_j^T dz_j, dz_{j-1} = d(h_{j-1}) * LeakyReLU'(z_{j-1})
    for (int j = a.n_dense - 1; j >= 1; --j) {
        const int nin = a.sizes[j - 1], nout = a.sizes[j];
        const float* Wj = a.W[j];
        if (nin == 256 && nout % 4 == 0) {
            // 64 column quads x 4 slices of the rows: 16-byte weight loads, partial sums combined in a fixed order
            const int uq = (tid & 63) * 4, part = tid >> 6, per = nout / 4;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
            for (int v = part * per; v < (part + 1) * per; ++v) {
                const float4 w = __ldg(reinterpret_cast<const float4*>(Wj + (size_t)v * nin + uq));
                const float gv = s_g[v];
                acc.x = fmaf(w.x, gv, acc.x); acc.y = fmaf(w.y, gv, acc.y); acc.z = fmaf(w.z, gv, acc.z); acc.w = fmaf(w.w, gv, acc.w);
            }
            __syncthreads();                               // s_g fully read
            float* s_p = s_v;                              // [4][256] partials need 4 * nin floats: s_v + s_g hold 2 * max_size
            if (part < 2) *reinterpret_cast<float4*>(s_p + part * 256 + uq) = acc;
            __syncthreads();
            if (part >= 2) {
                float4 t = *reinterpret_cast<const float4*>(s_p + (part - 2) * 256 + uq);
                t.x += acc.x; t.y += acc.y; t.z += acc.z; t.w += acc.w;
                *reinterpret_cast<float4*>(s_p + (part - 2) * 256 + uq) = t;
            }
            __syncthreads();
            {
                const int u = tid;
                const float t = s_p[u] + s_p[256 + u];
                __syncthreads();
                s_v[u] = t * (s_z[off[j - 1] + u] > 0.f ? 1.f : a.alpha);
            }
        } else {
            for (int u = tid; u < nin; u += 256) {
                float acc = 0.f;
#pragma unroll 8
                for (int v = 0; v < nout; ++v) acc = fmaf(__ldg(Wj + (size_t)v * nin + u), s_g[v], acc);   // coalesced over u
                s_v[u] = acc * (s_z[off[j - 1] + u] > 0.f ? 1.f : a.alpha);
            }
        }
        __syncthreads();
        for (int u = tid; u < nin; u += 256) s_g[u] = s_v[u];
        __syncthreads();
    }
    // s_g now holds dz of layer 0 (dz1)
    if (a.dz1 != nullptr)
        for (int u = tid; u < n0; u += 256) a.dz1[(size_t)b * n0 + u] = s_g[u];
    if (a.S != nullptr) {
        // alpha_raw[k] = sum_u dz1[u] S[u][k]: the u range is cut into `parts` slices so that all 256 threads work
        // (C is 64 on the tensor path); partial sums are combined in a fixed order
        if (a.C == 64 && n0 % 16 == 0 && a.max_size >= 256) {
            // 16 channel quads x 16 slices of u: 16-byte loads of S; the two slices of a warp meet by shuffle, the 8 warps in smem
            const int kq = (tid & 15) * 4, part = tid >> 4, per = n0 / 16;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
            for (int u = part * per; u < (part + 1) * per; ++u) {
                const float4 w = __ldg(reinterpret_cast<const float4*>(a.S + (size_t)u * 64 + kq));
                const float gv = s_g[u];
                acc.x = fmaf(w.x, gv, acc.x); acc.y = fmaf(w.y, gv, acc.y); acc.z = fmaf(w.z, gv, acc.z); acc.w = fmaf(w.w, gv, acc.w);
            }
            acc.x += __shfl_xor_sync(0xffffffffu, acc.x, 16); acc.y += __shfl_xor_sync(0xffffffffu, acc.y, 16);
            acc.z += __shfl_xor_sync(0xffffffffu, acc.z, 16); acc.w += __shfl_xor_sync(0xffffffffu, acc.w, 16);
            __syncthreads();                               // every thread has finished reading s_g
            if (lane < 16) *reinterpret_cast<float4*>(s_v + warp * 64 + kq) = acc;      // [8 warps][64]: 512 floats of scratch
            __syncthreads();
            if (tid < 64) {
                float t = 0.f;
#pragma unroll
                for (int q = 0; q < 8; ++q) t += s_v[q * 64 + tid];
                a.alpha_raw[(size_t)b * 64 + tid] = t;
            }
        } else {
            for (int k = tid; k < a.C; k += 256) {
                float acc = 0.f;
#pragma unroll 8
                for (int u = 0; u < n0; ++u) acc = fmaf(s_g[u], __ldg(a.S + (size_t)u * a.C + k), acc);
                a.alpha_raw[(size_t)b * a.C + k] = acc;
            }
        }
    }
}

__global__ void __launch_bounds__(256)
class_columns_kernel(const int32_t* __restrict__ rows, int K, int n, int32_t* __restrict__ cols, int ld) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n * K) return;
    const int b = i / K, k = i - b * K;
    cols[(size_t)k * ld + b] = rows != nullptr ? rows[i] : k;
}

int launch_class_columns(const int32_t* rows, int K, int n, int32_t* cols, int ld, cudaStream_t s) {
    class_columns_kernel<<<(n * K + 255) / 256, 256, 0, s>>>(rows, K, n, cols, ld);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

int launch_dense_head(const HeadArgs& a, int B, cudaStream_t s) {
    int total = 0;
    for (int j = 0; j < a.n_dense; ++j) total += a.sizes[j];
    const size_t smem = (size_t)(total + 4 + 2 * a.max_size) * sizeof(float);
    BCAD_REQUIRE(smem <= 48 * 1024, "dense head: layer sizes too large for the fused kernel (%zu bytes)", smem);
    dense_head_kernel<<<B, 256, smem, s>>>(a);
    BCAD_CUDA_CHECK(cudaGetLastError());
    return BCAD_OK;
}

}  // namespace bcad
