// Launchers of the 16-bit (fp16 operand) tensor path (sm100_kernels.cu).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace bcad {

int launch_conv_first_pool(const float* x, const float* w9c, const float* bias, __half* out, int B, int H, int W,
                           int pad, int Cout, float alpha, cudaStream_t s);

// tensor-core first conv: w_img = [4 chunks][Cout][8 halves] rows [w_hi(9) b_hi | w_hi(9) b_lo | w_lo(9) 0 0 0], or, with
// plain_operands (fp16 mode: no hi/lo split of image and weights), [2 chunks][Cout][8 halves] rows [w(9) b_hi b_lo 0 0 0 0 0]
// n_dev (nullable, also in the argument structs below): DEVICE pointer to the live image count of this launch -- the kernel works
// on min(B, *n_dev) images and returns at once when that is 0 (the refinement twin, refine.cu: the host does not know how many
// images were flagged)
int launch_conv_first_tc(const float* x, const uint8_t* w_img, __half* out, int B, int H, int W, int pad, int Cout,
                         float alpha, bool split_hi_lo, bool plain_operands, int sms, cudaStream_t s, const int* n_dev = nullptr);

struct IgemmArgs {
    const __half* in;      // C8 planar [B][H][Cin/8][W][8]
    const uint8_t* w_img;         // [9*(Cin/8)][Cout][16 B] weights, then the bias tile [2][Cout][16 B] rows {b_hi, b_lo, 0..}
    __half* act;           // C8 planar [B][Ho][Cout/8][Wo][8] post-activation, or nullptr
    uint8_t* pool_fc;             // pooled output as fc1 A tiles, or nullptr
    __half* pool_c8;       // pooled output C8 planar [B][Hp][Cout/8][Wp][8], or nullptr
    int B, H, W, Ho, Wo, Hp, Wp, pad;
    int bands, band_rows;         // row bands per image; output rows per band (even)
    int xsegs;                    // 128-pixel segments per row: work item = (image, band, segment)
    float alpha;
    int debug;                    // timing experiments only: 1 no act store, 2 no pool store, 4 empty epilogue, 8 no MMA
    const int* n_dev = nullptr;
};
int launch_conv_igemm(const IgemmArgs& a, int Cin, int Cout, bool x3, int sms, cudaStream_t s);

// first conv block with many input channels (sm100_wide.cu)
struct WideArgs {
    const __half* in;             // C8 planar [B][H][CinPad/8][W][8]
    const uint8_t* w_img;         // [G][9*(KC/8)][Cout][16 B] per channel group, then the bias tile [2][Cout][16 B]
    __half* pool_c8;              // pooled output C8 planar [B][Hp][Cout/8][Wp][8]
    int B, H, W, Ho, Wo, Hp, Wp, pad;
    int G;                        // channel groups of KC = conv_wide_group_channels(CinPad, Cout) channels
    int ybands, xsegs;            // bands of 256/Cout output rows, 128-pixel segments: work item = (image, band, segment)
    float alpha;
    int split_out = 0;            // fp16x3: the pooled fp32 value goes out as hi + lo halves, octets [hi 0..Cout/8) | lo 0..Cout/8)
};
int conv_wide_group_channels(int CinPad, int Cout);
int conv_wide_rows_per_band(int Cout);
int launch_conv_wide(const WideArgs& a, int CinPad, int Cout, int sms, cudaStream_t s);
int launch_nhwc_to_c8(const float* x, __half* out, int B, int H, int W, int C, int CinPad, cudaStream_t s);
// fp16x3: 3 * CinPad "virtual" channels, octets [x_hi | x_lo | x_hi]; against weight groups [w_hi | w_hi | w_lo] the plain kernel's
// fp32 accumulators then hold x_hi.w_hi + x_lo.w_hi + x_hi.w_lo
int launch_nhwc_to_c8_x3(const float* x, __half* out, int B, int H, int W, int C, int CinPad, cudaStream_t s);

// both conv blocks in one persistent kernel (sm100_fused.cu): Cin = 1 -> 32 -> 64 filters, fp16 mode, maps up to 128 px wide
struct FusedArgs {
    const float* x;               // fp32 [B][H][W]
    const uint8_t* w0_img;        // first-block image [4 chunks][32][16 B], or [2 chunks][32][16 B] with plain0 (as launch_conv_first_tc)
    int plain0;                   // first-block operands as plain fp16 (the fp16 mode) instead of hi/lo pairs
    const uint8_t* w1_img;        // second-block weight image + bias tile (as IgemmArgs::w_img; conv_fused2: the pair layout, see tensor_path.cu)
    const float* b0 = nullptr;    // conv_fused2 only: first-block bias fp32 [32]; w0_img is then the patch-union image [2 chunks][4 classes x 32][16 B]
    __half* act;                  // second-block activations, C8 planar, or nullptr
    uint8_t* pool_fc;             // pooled second-block output as fc1 A tiles, or nullptr
    __half* p1_out;               // optional copy of the pooled first-block output (C8 planar), nullptr = stays on chip
    int B, H, W;                  // input
    int H1, W1;                   // pooled first-block map = second-block input
    int Ho, Wo, Hp, Wp, pad;      // second-block output / pooled dims
    int bands, band_rows;
    float alpha;
    int debug;                    // timing experiments only: 1 no activation store, 2 no fc1-tile store, 16 first-block teams idle
    int xoff = 0;                 // conv_fused2 only: the input boxes start xoff columns left of -pad (16-byte aligned box starts)
};
bool conv_fused_supported(int Cin, int C0, int C1, int W1, int Wo1, bool x3);
int launch_conv_fused(const FusedArgs& a, int sms, cudaStream_t s);
// second generation (sm100_fused2.cu): patch-union first block (one MMA per tile), tensor-map TMA input boxes, three pipelined teams
bool conv_fused2_supported(const float* x, int H, int W);
int launch_conv_fused2(const FusedArgs& a, int sms, cudaStream_t s);

struct FcArgs {
    const uint8_t* a_tiles;       // [m_tiles][nkb][128][128 B] SW128
    const uint8_t* w_tiles;       // [nkb][N][128 B] SW128
    float* partials;              // [splits][m_pad][N]
    int N, nkb, kb_per_split, splits, m_tiles, m_pad;
    int x3;                       // fp16x3: tiles come as [hi][lo] pairs; A_hi.W_hi + A_lo.W_hi + A_hi.W_lo
    int ncb;                      // column blocks (grid.z): block cb reads w_tiles + cb * nkb tiles and writes columns [cb*N, +N); 0/1 = one
    long long ld_out;             // row stride of the output in floats; 0 = N (the split-K partial layout)
    int m_valid;                  // rows >= m_valid are not stored (0 = store all m_pad rows: the partial buffer is padded)
    const int* n_dev = nullptr;   // *n_dev == 0: nothing to do
};
// dz1 fp32 [B][K] -> fp16x3 A tiles [b/128][K/64][(hi|lo)][128][128 B, chunks XOR (row&7)] for the fc1 input-gradient GEMM
int launch_rows_to_fc_tiles_x3(const float* src, uint8_t* tiles, int B, int K, int m_pad, cudaStream_t s);
int launch_fc_splitk(const FcArgs& a, cudaStream_t s);
int launch_fc_reduce(const float* part, int splits, size_t ld_split, const float* bias, float* z, float* h, float alpha,
                     int M, int N, cudaStream_t s);

int launch_cam_c8(const __half* A, const float* alpha_raw, float scale, float* alpha_out, float* cam_lo, float* mm,
                  int B, int h, int w, int C, int splits, bool x3, cudaStream_t s, const int* n_dev = nullptr);
// fused tail (sm100_tail.cu): cam + min-max + bilinear + min-max, a 2-CTA cluster per image
bool tail_fused_supported(int h, int w, int H, int W, int C);
// out_stride: floats between the maps of consecutive images (0 = H * W)
int launch_tail_fused(const __half* A, const float* alpha_raw, float scale, float* alpha_out, float* out, int B, int h, int w,
                      int H, int W, int C, bool x3, cudaStream_t s, const int* n_dev = nullptr, size_t out_stride = 0);
// TF_GROUP target classes in one launch, one read of A: alpha of class k at alpha_raw + k * alpha_ld ([B][C] each), the map of class k
// of image b at out + b * out_stride + k * H * W; each bit-identical to a launch_tail_fused of that class
constexpr int TF_GROUP = 2;
bool tail_fused_classes_supported(int h, int w, int H, int W, int C);
int launch_tail_fused_classes(const __half* A, const float* alpha_raw, size_t alpha_ld, float scale, float* out, size_t out_stride, int B,
                              int h, int w, int H, int W, int C, bool x3, cudaStream_t s, const int* n_dev = nullptr);
// tie-duplicating rule on the fp16x3 path: alpha_raw[b][k] = sum_windows g * (#maxima in the window), A = split C8-planar activations
int launch_alpha_ties_c8(const __half* A, const float* g_pool, float* alpha_raw, int B, int h, int w, int C, cudaStream_t s);
int launch_c8_to_nhwc(const __half* src, float* dst, int B, int h, int w, int C, bool x3, cudaStream_t s);

}  // namespace bcad
