// Host-side helpers shared by the launchers: error reporting, launch counting, TMA descriptor encoding.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

namespace b2h {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);
int check_launch(const char* what);  // cudaGetLastError -> 0 / error code (+ message)

// 4-D NHWC-style bf16 tensor map, 128B swizzle. dims/strides listed innermost first; strides in BYTES for
// dims 1..3 (dim 0 is contiguous). box = {64 channels, box_w, box_h, 1}.
int make_tmap_4d(CUtensorMap* m, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t d3,
                 uint64_t s1, uint64_t s2, uint64_t s3, uint32_t box_w, uint32_t box_h);
// 2-D K-major bf16 matrix [rows][k] (pitch k elements), box = {64, box_rows}, 128B swizzle.
int make_tmap_2d(CUtensorMap* m, const void* base, uint64_t k, uint64_t rows, uint32_t box_rows);

// C channels of an NHWC bf16 tensor [N][H][W][pitch] (a channel slice when C < pitch).
inline int make_nhwc_map(CUtensorMap* m, const void* base, int C, int pitch, int N, int H, int W, uint32_t box_w,
                         uint32_t box_h) {
  const uint64_t s = static_cast<uint64_t>(pitch) * 2;
  return make_tmap_4d(m, base, C, W, H, N, s, s * W, s * W * H, box_w, box_h);
}
// The four pixel-shuffle sub-grids of a ConvTranspose2d(k2, s2) map: m[2i + j] is the H x W grid of canvas pixels
// (pad_top + 2h + i, pad_left + 2w + j), C channels, of the NHWC bf16 canvas [N][H2][W2][pitch].
int make_pixel_shuffle_maps(CUtensorMap m[4], const void* canvas, int C, int pitch, int N, int H, int W, int H2, int W2,
                            int pad_top, int pad_left, uint32_t box_w, uint32_t box_h);

#define B2_REQUIRE(cond, ...)        \
  do {                               \
    if (!(cond)) {                   \
      b2h::set_error(__VA_ARGS__);   \
      return 1;                      \
    }                                \
  } while (0)

inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// Kernel attributes (opt-in dynamic shared memory) are per device: each kernel instantiation keeps one bit per CUDA device
// in `configured` and opts in to `bytes` on its first launch there (a process may drive several GPUs). 0, or 2 + message.
template <class Kernel>
int opt_in_smem(Kernel* kern, int bytes, unsigned long long& configured, const char* what) {
  int dev = 0;
  cudaGetDevice(&dev);
  const unsigned long long bit = 1ull << (dev & 63);
  if (configured & bit) return 0;
  configured |= bit;
  const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e != cudaSuccess) {
    set_error("%s: cudaFuncSetAttribute(smem=%d): %s", what, bytes, cudaGetErrorString(e));
    return 2;
  }
  return 0;
}

// scale/shift (optional, [Cout] each): eval-mode BatchNorm + ReLU folded into the epilogue (stats_partial must be null)
// conv3_res.cu: persistent resident-weight 3x3 kernel for Cin in {64, 128}
bool conv3_res_applicable(int Cin, int Cout);
int conv3_res_stat_rows(int N, int H, int W, int Cin, int Cout);
int conv3_res_launch(const void* x, int x_cs, const void* w, void* y, int y_cs, float* stats_partial, int N, int H,
                     int W, int Cin, int Cout, cudaStream_t st, const float* scale = nullptr,
                     const float* shift = nullptr);
// ... with the BatchNorm-backward reduction of the consumer layer fused into the epilogue (backward-data, Cin = Cout = 64)
bool conv3_res_bnred_applicable(int Cin, int Cout);
int conv3_res_bnred_launch(const void* x, int x_cs, const void* w, void* y, int y_cs, const void* bn_y, int bn_y_cs,
                           const float* scale, const float* shift, const float* mean, const float* rstd, float* partial, int N,
                           int H, int W, int Cin, int Cout, cudaStream_t st);
// conv3_pair.cu: two CTA-pair kernels (tcgen05 cta_group::2, M = 256) on one skeleton. conv3_res2: the same layers as
// conv3_res with the weights resident; conv3_pair: weights streamed, for Cin >= 256
int conv3_res2_stat_rows(int N, int H, int W, int Cin, int Cout);
int conv3_res2_launch(const void* x, int x_cs, const void* w, void* y, int y_cs, float* stats_partial, int N, int H,
                      int W, int Cin, int Cout, cudaStream_t st, const float* scale = nullptr,
                     const float* shift = nullptr);
bool conv3_pair_applicable(int Cin, int Cout);
int conv3_pair_stat_rows(int N, int H, int W, int Cin, int Cout);
int conv3_pair_launch(const void* x, int x_cs, const void* w, void* y, int y_cs, float* stats_partial, int N, int H,
                      int W, int Cin, int Cout, cudaStream_t st, const float* scale = nullptr,
                     const float* shift = nullptr);
// ... as ConvTranspose2d(k2,s2) forward (scatter epilogue) and backward-data (4-map gather) for the shallow levels
bool convt_res_applicable(int Cin, int Cup);
int convt_res_fprop_launch(const void* x, int x_cs, const void* w_fprop, const float* bias, void* out, int out_cs, int N,
                           int H, int W, int Cin, int Cup, int H2, int W2, int pad_top, int pad_left, cudaStream_t st);
bool convt_res_dgrad_applicable(int Cin, int Cup);
int convt_res_dgrad_launch(const void* du, int du_cs, const void* w_dgrad, void* dx, int dx_cs, int N, int H, int W,
                           int Cin, int Cup, int H2, int W2, int pad_top, int pad_left, cudaStream_t st);
// the same kernel as a 1x1 convolution over a 64-channel input (inc.conv1 on its im2col'ed input, first_layer.cu)
int conv1x1_c64_stat_rows(int N, int H, int W, int Cout);
int conv1x1_c64_launch(const void* x, int x_cs, const void* w, void* y, int y_cs, float* stats_partial, int N, int H,
                       int W, int Cout, cudaStream_t st, const float* scale = nullptr,
                       const float* shift = nullptr);

// inc.conv1 from the fp32 NCHW input, im2col rows built in shared memory (conv3_res.cu RES_FIRST); w1 = [Cout][64] bf16
int conv3x3_first_launch(const float* x_nchw, const void* w1, void* y, int y_cs, float* stats_partial, int N, int H, int W,
                         int Cin, int Cout, cudaStream_t st, const float* scale = nullptr, const float* shift = nullptr);

// elementwise.cu: partial [rows][ncols] fp32 -> sums[ncols] fp64 (fixed order); out[c] = sum over rows of column col_lo + c
int reduce_partials_launch(const float* partial, long long rows, int ncols, double* sums, cudaStream_t st);
int partial_colsum_launch(const float* partial, long long rows, int row_pitch, int col_lo, int n, float* out, cudaStream_t st);

}  // namespace b2h
