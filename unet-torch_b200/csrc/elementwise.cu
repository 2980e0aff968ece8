// Bandwidth-bound kernels around the convolutions: BatchNorm2d statistics/affine, BN-apply + ReLU (+ 2x2 max
// pool with argmax position, + write-into-concat-buffer), their backward (reduce + apply, with the skip/pool
// gradient merge), and per-channel sums. Reference: Model.py:17-18,21-22 (BatchNorm2d, ReLU), :36,42 (MaxPool2d),
// :79 (torch.cat). All activation traffic is 128-bit (8 x bf16) per thread, channel-innermost (NHWC).
#include "../../include/b200unet.h"
#include "ew_common.cuh"
#include "host_common.h"

#include <cuda_bf16.h>
#include <stdlib.h>

namespace {

constexpr int EW_THREADS = 256;
constexpr int EW_MAX_BLOCKS = 148 * 8;

using namespace b2ew;

// Traversal direction of the three big elementwise passes (0 BN-apply forward, 1 BN-backward reduce, 2 BN-backward apply):
// alternating the direction between a producer and its consumer turns the tail the producer left in L2 into hits.
// B200UNET_EW_REV = three digits, 1 = back to front (default "000"). Measured on B200: no effect (22.5-22.9 ms per step for all
// eight combinations, inside run-to-run noise) - streaming kernels do not find the producer's tail in L2; kept as a knob.
int ew_rev(int which) {
  static int mask = -1;
  if (mask < 0) {
    const char* e = getenv("B200UNET_EW_REV");
    const char* d = (e != nullptr && e[0] && e[1] && e[2]) ? e : "000";
    mask = (d[0] == '1' ? 1 : 0) | (d[1] == '1' ? 2 : 0) | (d[2] == '1' ? 4 : 0);
  }
  return (mask >> which) & 1;
}

int ew_blocks(long long work_items) {
  long long b = (work_items + EW_THREADS - 1) / EW_THREADS;
  if (b > EW_MAX_BLOCKS) b = EW_MAX_BLOCKS;
  if (b < 1) b = 1;
  return static_cast<int>(b);
}

// ------------------------------------------------------------------------------------------ statistics
// partial [rows][ncols] fp32 -> sums[ncols] fp64. One block per 32 columns (32 row-lanes each, fixed summation order: no
// atomics, no memset, bit-reproducible).
__global__ void __launch_bounds__(1024) reduce_partials_kernel(const float* __restrict__ partial, long long rows, int ncols,
                                       double* __restrict__ sums) {
  __shared__ double sh[32][33];
  const int col = blockIdx.x * 32 + (threadIdx.x & 31);
  const int rl = threadIdx.x >> 5;
  double acc = 0.0;
  if (col < ncols) {
#pragma unroll 4
    for (long long r = rl; r < rows; r += 32) acc += static_cast<double>(__ldg(partial + r * ncols + col));
  }
  sh[rl][threadIdx.x & 31] = acc;
  __syncthreads();
  if (rl == 0 && col < ncols) {
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < 32; ++i) t += sh[i][threadIdx.x];
    sums[col] = t;
  }
}

int launch_reduce_partials(const float* partial, long long rows, int ncols, double* sums, cudaStream_t st) {
  reduce_partials_kernel<<<(ncols + 31) / 32, 1024, 0, st>>>(partial, rows, ncols, sums);
  return b2h::check_launch("reduce_partials");
}

// partial [rows][ncols] -> out [out_rows][ncols], out[b] = sum of the rows r = b (mod out_rows) in increasing order (fixed order,
// no atomics). The one-tile-per-CTA GEMM epilogues of the attention gates emit one statistics row per 128-pixel tile (131 072
// rows for a 32-channel map at 512^2): the finalisation kernels above run one block per 32 channels, so they get this
// machine-wide pre-reduction first.
__global__ void __launch_bounds__(256) fold_rows_kernel(const float* __restrict__ partial, long long rows, int ncols,
                                                        float* __restrict__ out, int out_rows) {
  __shared__ float sh[256];
  const int width = ncols < 256 ? ncols : 256;  // ncols is a power of two >= 2 or a multiple of 256
  const int lanes = 256 / width;
  const int cl = threadIdx.x % width, rl = threadIdx.x / width;
  for (int c0 = 0; c0 < ncols; c0 += width) {
    float acc = 0.f;
    if (rl < lanes)
      for (long long r = blockIdx.x + static_cast<long long>(out_rows) * rl; r < rows; r += static_cast<long long>(out_rows) * lanes)
        acc += __ldg(partial + r * ncols + c0 + cl);
    sh[threadIdx.x] = acc;
    __syncthreads();
    if (rl == 0) {
      float t = 0.f;
      for (int i = 0; i < lanes; ++i) t += sh[i * width + cl];
      out[static_cast<size_t>(blockIdx.x) * ncols + c0 + cl] = t;
    }
    __syncthreads();
  }
}

// The forward statistics path in ONE launch (single GPU): reduce the conv epilogue's partial rows [rows][2][C] (fp64, fixed
// order) and finalise BatchNorm2d for the block's 32 channels - mean, rstd, scale = gamma*rstd, shift = beta - mean*scale,
// running statistics (unbiased variance) and num_batches_tracked += 1 (Model.py:17,21). Replaces memset + reduce_partials +
// bn_finalize + a torch kernel for the counter: 4 launches per BatchNorm layer -> 1.
__global__ void __launch_bounds__(1024) bn_reduce_finalize_kernel(const float* __restrict__ partial, long long rows, int C,
                                                                  double count, const float* __restrict__ gamma,
                                                                  const float* __restrict__ beta, float eps, float momentum,
                                                                  float* running_mean, float* running_var,
                                                                  long long* num_batches, float* mean, float* rstd,
                                                                  float* scale, float* shift) {
  // 32 channels x 32 row-lanes: the loads of a lane are independent (latency-bound kernel: keep many in flight)
  __shared__ double sh[2][32][33];
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int rl = threadIdx.x >> 5;
  double a1 = 0.0, a2 = 0.0;
  if (c < C) {
#pragma unroll 4
    for (long long r = rl; r < rows; r += 32) {
      a1 += static_cast<double>(__ldg(partial + r * 2 * C + c));
      a2 += static_cast<double>(__ldg(partial + r * 2 * C + C + c));
    }
  }
  sh[0][rl][threadIdx.x & 31] = a1;
  sh[1][rl][threadIdx.x & 31] = a2;
  __syncthreads();
  if (blockIdx.x == 0 && threadIdx.x == 0 && num_batches != nullptr) *num_batches += 1;
  if (rl != 0 || c >= C) return;
  double s1 = 0.0, s2 = 0.0;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    s1 += sh[0][i][threadIdx.x];
    s2 += sh[1][i][threadIdx.x];
  }
  const double m = s1 / count;
  double var = s2 / count - m * m;
  if (var < 0.0) var = 0.0;
  const float mf = static_cast<float>(m);
  const float rs = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
  mean[c] = mf;
  rstd[c] = rs;
  const float sc = gamma[c] * rs;
  scale[c] = sc;
  shift[c] = beta[c] - mf * sc;
  if (running_mean != nullptr) {
    const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mf;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * static_cast<float>(unbiased);
  }
}

__global__ void bn_finalize_kernel(const double* __restrict__ sums, double count, const float* __restrict__ gamma,
                                   const float* __restrict__ beta, float eps, float momentum, float* running_mean,
                                   float* running_var, float* mean, float* rstd, float* scale, float* shift, int C) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double m = sums[c] / count;
  double var = sums[C + c] / count - m * m;
  if (var < 0.0) var = 0.0;
  const float mf = static_cast<float>(m);
  const float rs = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
  mean[c] = mf;
  rstd[c] = rs;
  const float sc = gamma[c] * rs;
  scale[c] = sc;
  shift[c] = beta[c] - mf * sc;
  if (running_mean != nullptr) {
    const double unbiased = count > 1.0 ? var * count / (count - 1.0) : var;
    running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mf;
    running_var[c] = (1.f - momentum) * running_var[c] + momentum * static_cast<float>(unbiased);
  }
}

__global__ void bn_eval_affine_kernel(const float* gamma, const float* beta, const float* rm, const float* rv, float eps,
                                      float* scale, float* shift, int C) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float sc = gamma[c] * (1.0f / sqrtf(rv[c] + eps));
  scale[c] = sc;
  shift[c] = beta[c] - rm[c] * sc;
}

__global__ void bn_eval_stats_kernel(const float* rm, const float* rv, float eps, float* mean, float* rstd, int C) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  mean[c] = rm[c];
  rstd[c] = 1.0f / sqrtf(rv[c] + eps);
}

// ------------------------------------------------------------------------------------------ pad strip
// nn.MaxPool2d(2) in floor mode (Model.py:36,42) leaves the last row of an odd-H map and the last column of an odd-W map out
// of every 2x2 window; on the way up, F.pad (Model.py:69-73) puts the same pixels of the concat buffer's upsampled half
// after the 2h'x2w' ConvTranspose2d output as zeros. Both are "the pad strip" of an [N][H][W] map: the pixels outside its
// leading 2*(H/2) x 2*(W/2) region, per image the bottom row (odd H) and then the right column above it (odd W).
__host__ __device__ __forceinline__ long long strip_pixels_per_image(int H, int W) {
  return static_cast<long long>(H & 1) * W + static_cast<long long>(W & 1) * (H & ~1);
}

// Strip work items (pixels x 8-channel groups) are counted in 32 bits (the host checks): 32-bit divisions stay inline, where
// 64-bit ones would call a subroutine and make the pooled backward kernels, at their 128-register cap, spill.
constexpr long long STRIP_MAX_ITEMS = 0x7fffffffLL - 148LL * 8 * EW_THREADS;

// NHWC pixel index of strip pixel s (0 <= s < N * strip_pixels_per_image)
__device__ __forceinline__ long long strip_pixel(int s, int H, int W) {
  const int per = static_cast<int>(strip_pixels_per_image(H, W));
  const int n = s / per;
  const int r = s - n * per;
  const int row = (H & 1) ? W : 0;
  if (r < row) return (static_cast<long long>(n) * H + H - 1) * W + r;
  return (static_cast<long long>(n) * H + (r - row)) * W + W - 1;
}

__global__ void __launch_bounds__(EW_THREADS) pad_strip_zero_kernel(__nv_bfloat16* __restrict__ x, int x_cs, int N, int H,
                                                                    int W, int C) {
  const int cgs = C >> 3;
  const int total = static_cast<int>(N * strip_pixels_per_image(H, W) * cgs);
  const int stride = gridDim.x * blockDim.x;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
    const int s = i / cgs;
    *reinterpret_cast<uint4*>(x + strip_pixel(s, H, W) * x_cs + (i - s * cgs) * 8) = make_uint4(0, 0, 0, 0);
  }
}

// out[c] -= sum over the pad strip of x[..., c] (fp64, fixed order). A block owns 32 channels (four 8-channel groups) and
// walks the strip with 64 pixel lanes; the lanes are summed in lane order.
constexpr int STRIP_LANES = 64;
__global__ void __launch_bounds__(256) pad_strip_sub_colsum_kernel(const __nv_bfloat16* __restrict__ x, int x_cs, int N,
                                                                   int H, int W, int C, float* __restrict__ out) {
  __shared__ double sh[STRIP_LANES][33];
  const int g = threadIdx.x & 3, lane = threadIdx.x >> 2;
  const int c0 = blockIdx.x * 32 + g * 8;
  const int pixels = static_cast<int>(N * strip_pixels_per_image(H, W));
  double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  if (c0 < C) {
    for (int s = lane; s < pixels; s += STRIP_LANES) {
      float f[8];
      unpack8(ldg128(x + strip_pixel(s, H, W) * x_cs + c0), f);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += static_cast<double>(f[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j) sh[lane][g * 8 + j] = acc[j];
  __syncthreads();
  if (threadIdx.x < 32 && blockIdx.x * 32 + static_cast<int>(threadIdx.x) < C) {
    double t = 0.0;
    for (int l = 0; l < STRIP_LANES; ++l) t += sh[l][threadIdx.x];
    const int c = blockIdx.x * 32 + threadIdx.x;
    out[c] = static_cast<float>(static_cast<double>(out[c]) - t);
  }
}

// ------------------------------------------------------------------------------------------ forward
// STRIP (with !POOL): the pixels are those of the pad strip (floor-mode pooling leaves them out of every window)
template <bool POOL, bool STRIP = false>
__global__ void __launch_bounds__(EW_THREADS) bn_relu_fwd_kernel(const __nv_bfloat16* __restrict__ y, int y_cs,
                                                                 const float* __restrict__ scale,
                                                                 const float* __restrict__ shift,
                                                                 __nv_bfloat16* __restrict__ a, int a_cs,
                                                                 __nv_bfloat16* __restrict__ pooled,
                                                                 uint8_t* __restrict__ pool_idx, int N, int H, int W,
                                                                 int C, int rev) {
  // rev: walk the tensor back to front. The producer (a conv kernel, front to back) leaves the TAIL of y in the 126 MB L2
  // and the consumer (the next conv, front to back) wants the HEAD of `a` there: a back-to-front pass gets both.
  const int cgs = C >> 3;  // 8-channel groups; divides blockDim, so a thread keeps its group across the loop
  const int cg = rev ? cgs - 1 - static_cast<int>(threadIdx.x % cgs) : static_cast<int>(threadIdx.x % cgs);
  float sc[8], sh[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    sc[i] = scale[cg * 8 + i];
    sh[i] = shift[cg * 8 + i];
  }
  const long long tid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  if (!POOL) {
    const long long total = (STRIP ? N * strip_pixels_per_image(H, W) : static_cast<long long>(N) * H * W) * cgs;
    constexpr int U = 4;  // independent 128-bit loads in flight per thread
    for (long long i0 = tid; i0 < total; i0 += stride * U) {
      uint4 raw[U];
      long long pix[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long i = i0 + u * stride;
        pix[u] = (rev ? total - 1 - i : i) / cgs;
        if (STRIP) pix[u] = strip_pixel(static_cast<int>(pix[u]), H, W);
        if (i < total) raw[u] = ldg128(y + pix[u] * y_cs + cg * 8);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (i0 + u * stride < total) {
          float f[8];
          unpack8(raw[u], f);
#pragma unroll
          for (int j = 0; j < 8; ++j) f[j] = fmaxf(fmaf(sc[j], f[j], sh[j]), 0.f);
          *reinterpret_cast<uint4*>(a + pix[u] * a_cs + cg * 8) = pack8(f);
        }
      }
    }
  } else {
    const int Hp = H >> 1, Wp = W >> 1;
    const long long total = static_cast<long long>(N) * Hp * Wp * cgs;
    for (long long i = tid; i < total; i += stride) {
      const long long pp = (rev ? total - 1 - i : i) / cgs;  // pooled pixel
      const int wp = static_cast<int>(pp % Wp);
      const int hp = static_cast<int>((pp / Wp) % Hp);
      const long long n = pp / (static_cast<long long>(Wp) * Hp);
      const long long p00 = (n * H + 2 * hp) * W + 2 * wp;
      float best[8];
      uint32_t bidx[8];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const long long pix = p00 + (k >> 1) * W + (k & 1);
        float f[8];
        unpack8(ldg128(y + pix * y_cs + cg * 8), f);
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = bf16_round(fmaxf(fmaf(sc[j], f[j], sh[j]), 0.f));
        *reinterpret_cast<uint4*>(a + pix * a_cs + cg * 8) = pack8(f);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          // nn.MaxPool2d: keep the first maximum in row-major window order; NaN wins
          if (k == 0 || f[j] > best[j] || f[j] != f[j]) {
            best[j] = f[j];
            bidx[j] = k;
          }
        }
      }
      *reinterpret_cast<uint4*>(pooled + pp * C + cg * 8) = pack8(best);
      if (pool_idx != nullptr) {
        uint2 pk;
        pk.x = bidx[0] | (bidx[1] << 8) | (bidx[2] << 16) | (bidx[3] << 24);
        pk.y = bidx[4] | (bidx[5] << 8) | (bidx[6] << 16) | (bidx[7] << 24);
        *reinterpret_cast<uint2*>(pool_idx + pp * C + cg * 8) = pk;
      }
    }
  }
}

// nn.MaxPool2d(2) alone (Model.py:36,42) over an NHWC bf16 tensor (possibly a channel slice): used by the inference path,
// where BatchNorm + ReLU already ran in the conv epilogue. Same window semantics as the fused kernel above (first maximum
// in row-major window order; NaN wins); position bytes optional.
__global__ void __launch_bounds__(EW_THREADS) maxpool_fwd_kernel(const __nv_bfloat16* __restrict__ a, int a_cs,
                                                                 __nv_bfloat16* __restrict__ pooled, int p_cs,
                                                                 uint8_t* __restrict__ pool_idx, int N, int H, int W, int C) {
  const int cgs = C >> 3;
  const int Hp = H >> 1, Wp = W >> 1;
  const long long total = static_cast<long long>(N) * Hp * Wp * cgs;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += stride) {
    const long long pp = i / cgs;
    const int cg = static_cast<int>(i - pp * cgs);
    const int wp = static_cast<int>(pp % Wp);
    const int hp = static_cast<int>((pp / Wp) % Hp);
    const long long n = pp / (static_cast<long long>(Wp) * Hp);
    const long long p00 = (n * H + 2 * hp) * W + 2 * wp;
    uint4 raw[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) raw[k] = ldg128(a + (p00 + (k >> 1) * W + (k & 1)) * a_cs + cg * 8);
    float best[8];
    uint32_t bidx[8];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float f[8];
      unpack8(raw[k], f);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        if (k == 0 || f[j] > best[j] || f[j] != f[j]) {
          best[j] = f[j];
          bidx[j] = k;
        }
      }
    }
    *reinterpret_cast<uint4*>(pooled + pp * p_cs + cg * 8) = pack8(best);
    if (pool_idx != nullptr) {
      uint2 pk;
      pk.x = bidx[0] | (bidx[1] << 8) | (bidx[2] << 16) | (bidx[3] << 24);
      pk.y = bidx[4] | (bidx[5] << 8) | (bidx[6] << 16) | (bidx[7] << 24);
      *reinterpret_cast<uint2*>(pool_idx + pp * C + cg * 8) = pk;
    }
  }
}

// ------------------------------------------------------------------------------------------ backward
// da for one pixel / channel group: (g1 + unpool(g_pool)) * [bn(y) > 0]
struct BwdSrc {
  const __nv_bfloat16* g1;
  int g1_cs;
  const __nv_bfloat16* gp;
  const uint8_t* pidx;
  const __nv_bfloat16* y;
  int y_cs;
};

// Raw 128-bit loads of one work item (one pixel, or one 2x2 pooling window), issued before any arithmetic so
// that several items' loads are in flight per thread.
template <bool POOL>
struct BwdRaw {
  static constexpr int NP = POOL ? 4 : 1;
  uint4 y[NP], g[NP], gp;
  uint2 idx;
  long long pix[NP];
};

// STRIP (with !POOL): item k is the k-th pixel of the pad strip
template <bool POOL, bool STRIP>
__device__ __forceinline__ void bwd_load(const BwdSrc& s, long long item, int cg, int C, int H, int W, BwdRaw<POOL>& r) {
  if (!POOL) {
    const long long pix = STRIP ? strip_pixel(static_cast<int>(item), H, W) : item;
    r.pix[0] = pix;
    r.y[0] = ldg128(s.y + pix * s.y_cs + cg * 8);
    r.g[0] = s.g1 != nullptr ? ldg128(s.g1 + pix * s.g1_cs + cg * 8) : make_uint4(0, 0, 0, 0);
  } else {
    const int Hp = H >> 1, Wp = W >> 1;
    const int wp = static_cast<int>(item % Wp);
    const int hp = static_cast<int>((item / Wp) % Hp);
    const long long n = item / (static_cast<long long>(Wp) * Hp);
    const long long p00 = (n * H + 2 * hp) * W + 2 * wp;
    r.gp = ldg128(s.gp + item * C + cg * 8);
    r.idx = __ldg(reinterpret_cast<const uint2*>(s.pidx + item * C + cg * 8));
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      r.pix[k] = p00 + (k >> 1) * W + (k & 1);
      r.y[k] = ldg128(s.y + r.pix[k] * s.y_cs + cg * 8);
      r.g[k] = s.g1 != nullptr ? ldg128(s.g1 + r.pix[k] * s.g1_cs + cg * 8) : make_uint4(0, 0, 0, 0);
    }
  }
}

template <bool POOL>
__device__ __forceinline__ void bwd_decode(const BwdRaw<POOL>& r, int k, const float (&sc)[8], const float (&sh)[8],
                                           float (&da)[8], float (&yv)[8]) {
  unpack8(r.y[k], yv);
  unpack8(r.g[k], da);
  if (POOL) {
    float gp[8];
    unpack8(r.gp, gp);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const uint32_t b = ((j < 4 ? r.idx.x : r.idx.y) >> (8 * (j & 3))) & 0xffu;
      if (b == static_cast<uint32_t>(k)) da[j] += gp[j];
    }
  }
#pragma unroll
  for (int j = 0; j < 8; ++j)
    if (!(fmaf(sc[j], yv[j], sh[j]) > 0.f)) da[j] = 0.f;
}

template <bool POOL, bool STRIP = false>
__global__ void __launch_bounds__(EW_THREADS, 2) bn_bwd_reduce_kernel(BwdSrc s, const float* __restrict__ scale,
                                                                      const float* __restrict__ shift,
                                                                      const float* __restrict__ mean,
                                                                      const float* __restrict__ rstd,
                                                                      float* __restrict__ partial, int N, int H, int W,
                                                                      int C, int rev) {
  constexpr int NP = POOL ? 4 : 1;
  constexpr int U = POOL ? 1 : 4;
  const int cgs = C >> 3;
  const int cg = rev ? cgs - 1 - static_cast<int>(threadIdx.x % cgs) : static_cast<int>(threadIdx.x % cgs);
  float sc[8], sh[8], s1[8], s2[8];  // s1 = sum da, s2 = sum da*y (turned into sum da*xhat at the end)
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    sc[i] = scale[cg * 8 + i];
    sh[i] = shift[cg * 8 + i];
    s1[i] = 0.f;
    s2[i] = 0.f;
  }
  const long long items = POOL    ? static_cast<long long>(N) * (H >> 1) * (W >> 1)
                          : STRIP ? N * strip_pixels_per_image(H, W)
                                  : static_cast<long long>(N) * H * W;
  const long long total = items * cgs;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i0 = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i0 < total; i0 += stride * U) {
    BwdRaw<POOL> raw[U];
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (i0 + u * stride < total)
        bwd_load<POOL, STRIP>(s, (rev ? total - 1 - (i0 + u * stride) : (i0 + u * stride)) / cgs, cg, C, H, W, raw[u]);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (i0 + u * stride < total) {
#pragma unroll
        for (int k = 0; k < NP; ++k) {
          float da[8], yv[8];
          bwd_decode<POOL>(raw[u], k, sc, sh, da, yv);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            s1[j] += da[j];
            s2[j] = fmaf(da[j], yv[j], s2[j]);
          }
        }
      }
    }
  }
  // block reduction across the threads that share a channel group
  __shared__ float sh_red[EW_THREADS][17];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    sh_red[threadIdx.x][j] = s1[j];
    sh_red[threadIdx.x][8 + j] = s2[j];
  }
  __syncthreads();
  for (int ch = threadIdx.x; ch < C; ch += blockDim.x) {
    const int g = ch >> 3, j = ch & 7;
    double a1 = 0.0, a2 = 0.0;
    for (int th = g; th < EW_THREADS; th += cgs) {
      a1 += static_cast<double>(sh_red[th][j]);
      a2 += static_cast<double>(sh_red[th][8 + j]);
    }
    // sum da*xhat = rstd * (sum da*y - mean * sum da)
    const double sx = static_cast<double>(rstd[ch]) * (a2 - static_cast<double>(mean[ch]) * a1);
    partial[static_cast<size_t>(blockIdx.x) * 2 * C + ch] = static_cast<float>(a1);
    partial[static_cast<size_t>(blockIdx.x) * 2 * C + C + ch] = static_cast<float>(sx);
  }
}

template <bool POOL, bool STRIP = false>
__global__ void __launch_bounds__(EW_THREADS, 2) bn_bwd_apply_kernel(BwdSrc s, const float* __restrict__ gamma,
                                                                     const float* __restrict__ scale,
                                                                     const float* __restrict__ shift,
                                                                     const float* __restrict__ mean,
                                                                     const float* __restrict__ rstd,
                                                                     const double* __restrict__ sums, double count,
                                                                     const double* __restrict__ sums_local,
                                                                     __nv_bfloat16* __restrict__ dy, int dy_cs,
                                                                     float* __restrict__ dgamma,
                                                                     float* __restrict__ dbeta, int N, int H, int W,
                                                                     int C, int rev) {
  constexpr int NP = POOL ? 4 : 1;
  constexpr int U = POOL ? 1 : 4;
  const int cgs = C >> 3;
  const int cg = rev ? cgs - 1 - static_cast<int>(threadIdx.x % cgs) : static_cast<int>(threadIdx.x % cgs);
  float sc[8], sh[8], k1[8], k2[8], k3[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int c = cg * 8 + i;
    sc[i] = scale[c];
    sh[i] = shift[c];
    const double g = gamma[c], r = rstd[c], m = mean[c];
    const double sda = sums[c] / count, sdx = sums[C + c] / count;
    // dy = g*r*(da - sda - xhat*sdx), xhat = (y - m)*r
    k1[i] = static_cast<float>(g * r);
    k2[i] = static_cast<float>(-g * r * r * sdx);
    k3[i] = static_cast<float>(-g * r * sda + g * r * r * m * sdx);
  }
  if (blockIdx.x == 0 && dgamma != nullptr) {
    const double* sl = sums_local != nullptr ? sums_local : sums;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      dbeta[c] = static_cast<float>(sl[c]);
      dgamma[c] = static_cast<float>(sl[C + c]);
    }
  }
  const long long items = POOL    ? static_cast<long long>(N) * (H >> 1) * (W >> 1)
                          : STRIP ? N * strip_pixels_per_image(H, W)
                                  : static_cast<long long>(N) * H * W;
  const long long total = items * cgs;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i0 = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i0 < total; i0 += stride * U) {
    BwdRaw<POOL> raw[U];
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (i0 + u * stride < total)
        bwd_load<POOL, STRIP>(s, (rev ? total - 1 - (i0 + u * stride) : (i0 + u * stride)) / cgs, cg, C, H, W, raw[u]);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (i0 + u * stride < total) {
#pragma unroll
        for (int k = 0; k < NP; ++k) {
          float da[8], yv[8], o[8];
          bwd_decode<POOL>(raw[u], k, sc, sh, da, yv);
#pragma unroll
          for (int j = 0; j < 8; ++j) o[j] = fmaf(k1[j], da[j], fmaf(k2[j], yv[j], k3[j]));
          *reinterpret_cast<uint4*>(dy + raw[u].pix[k] * dy_cs + cg * 8) = pack8(o);
        }
      }
    }
  }
}

__global__ void __launch_bounds__(EW_THREADS) channel_sum_kernel(const __nv_bfloat16* __restrict__ x, int x_cs,
                                                                 float* __restrict__ partial, long long pixels, int C) {
  const int cgs = C >> 3;
  const int cg = threadIdx.x % cgs;
  float s1[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  const long long total = pixels * cgs;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += stride) {
    float f[8];
    unpack8(ldg128(x + (i / cgs) * x_cs + cg * 8), f);
#pragma unroll
    for (int j = 0; j < 8; ++j) s1[j] += f[j];
  }
  __shared__ float sh_red[EW_THREADS][9];
#pragma unroll
  for (int j = 0; j < 8; ++j) sh_red[threadIdx.x][j] = s1[j];
  __syncthreads();
  for (int ch = threadIdx.x; ch < C; ch += blockDim.x) {
    const int g = ch >> 3, j = ch & 7;
    float acc = 0.f;
    for (int th = g; th < EW_THREADS; th += cgs) acc += sh_red[th][j];
    partial[static_cast<size_t>(blockIdx.x) * C + ch] = acc;
  }
}

// out[c] = sum over rows of partial[r][col_lo + c] (fp64 accumulation, fixed order): per-channel sums taken from the
// statistics rows a convolution epilogue already produced (ConvTranspose2d bias gradient, Model.py:56).
__global__ void partial_colsum_kernel(const float* __restrict__ partial, long long rows, int row_pitch, int col_lo, int n,
                                      float* __restrict__ out) {
  __shared__ double sh[8][32];
  const int c = blockIdx.x * 32 + (threadIdx.x & 31);
  const int rl = threadIdx.x >> 5;
  double acc = 0.0;
  if (c < n)
    for (long long r = rl; r < rows; r += 8) acc += static_cast<double>(partial[r * row_pitch + col_lo + c]);
  sh[rl][threadIdx.x & 31] = acc;
  __syncthreads();
  if (rl == 0 && c < n) {
    double t = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += sh[i][threadIdx.x];
    out[c] = static_cast<float>(t);
  }
}

// ------------------------------------------------------------------------------------------ channel-slice copy / sum
// A network with two decoders over one encoder (UNet_multitask, Model.py:172-250) needs the skip activations in a second
// concat buffer and the sum of the two decoders' gradients on the way back: out = a (+ b) over a channel slice of NHWC
// buffers with independent pixel pitches. out may alias a. fp32 sum, one bf16 rounding.
template <bool ADD>
__global__ void __launch_bounds__(EW_THREADS) slice_copy_add_kernel(const __nv_bfloat16* __restrict__ a, int a_cs,
                                                                    const __nv_bfloat16* __restrict__ b, int b_cs,
                                                                    __nv_bfloat16* __restrict__ out, int out_cs,
                                                                    long long pixels, int C) {
  const int cgs = C >> 3;
  const long long total = pixels * cgs;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += stride) {
    const long long p = i / cgs;
    const int c = static_cast<int>(i - p * cgs) * 8;
    uint4 v = ldg128(a + p * a_cs + c);
    if (ADD) {
      float fa[8], fb[8];
      unpack8(v, fa);
      unpack8(ldg128(b + p * b_cs + c), fb);
#pragma unroll
      for (int j = 0; j < 8; ++j) fa[j] += fb[j];
      v = pack8(fa);
    }
    *reinterpret_cast<uint4*>(out + p * out_cs + c) = v;
  }
}

__global__ void double_to_float_kernel(const double* in, float* out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = static_cast<float>(in[i]);
}

bool ok_channels(int C) { return C >= 64 && C <= 2048 && (C & (C - 1)) == 0; }

// The backward kernels keep 100-128 registers per thread, i.e. two resident blocks per SM: a grid of 148 x 8 blocks runs
// as four waves, each paying its own ramp-up, block reduction and tail (ncu: bn_bwd_reduce at 4.9 TB/s, 24 % warps
// active). One wave of exactly-resident blocks that loop longer removes that. B200UNET_BWD_BLOCKS_PER_SM overrides (8 =
// the former grid).
int bwd_blocks_for(long long items, int C) {
  static int per_sm = 0;
  if (per_sm == 0) {
    const char* e = getenv("B200UNET_BWD_BLOCKS_PER_SM");
    per_sm = e != nullptr ? atoi(e) : 2;
    if (per_sm < 1 || per_sm > 8) per_sm = 2;
  }
  const int b = ew_blocks(items * (C / 8));
  return b < 148 * per_sm ? b : 148 * per_sm;
}

int bwd_blocks(int N, int H, int W, int C, bool pool) {
  return bwd_blocks_for(pool ? static_cast<long long>(N) * (H / 2) * (W / 2) : static_cast<long long>(N) * H * W, C);
}

// floor-mode pooled passes: the pad strip runs as a second, unpooled launch over its pixels (none at even H and W, where
// the pooled kernels are exactly those of the even-size path)
long long floor_strip_pixels(bool floor_mode, bool pool, int N, int H, int W) {
  return floor_mode && pool ? N * strip_pixels_per_image(H, W) : 0;
}

}  // namespace

namespace b2h {
int reduce_partials_launch(const float* partial, long long rows, int ncols, double* sums, cudaStream_t st) {
  return launch_reduce_partials(partial, rows, ncols, sums, st);
}
int partial_colsum_launch(const float* partial, long long rows, int row_pitch, int col_lo, int n, float* out, cudaStream_t st) {
  partial_colsum_kernel<<<(n + 31) / 32, 256, 0, st>>>(partial, rows, row_pitch, col_lo, n, out);
  return check_launch("partial_colsum");
}
}  // namespace b2h

extern "C" {

int b200unet_bn_reduce_partials(const float* stats_partial, int64_t mtiles, int C, double* sums, b200_stream_t stream) {
  return launch_reduce_partials(stats_partial, mtiles, 2 * C, sums, static_cast<cudaStream_t>(stream));
}

int b200unet_fold_rows(const float* partial, int64_t rows, int ncols, float* out, int out_rows, b200_stream_t stream) {
  B2_REQUIRE(partial && out && rows > 0 && out_rows > 0 && out_rows <= rows, "fold_rows: bad arguments (rows=%lld out_rows=%d)",
             static_cast<long long>(rows), out_rows);
  B2_REQUIRE(ncols >= 2 && ((ncols <= 256 && (ncols & (ncols - 1)) == 0) || ncols % 256 == 0),
             "fold_rows: ncols=%d must be a power of two in [2, 256] or a multiple of 256", ncols);
  fold_rows_kernel<<<out_rows, 256, 0, static_cast<cudaStream_t>(stream)>>>(partial, rows, ncols, out, out_rows);
  return b2h::check_launch("fold_rows");
}

int b200unet_bn_finalize(const double* sums, double count, const float* gamma, const float* beta, float eps,
                         float momentum, float* running_mean, float* running_var, float* mean, float* rstd, float* scale,
                         float* shift, int C, b200_stream_t stream) {
  bn_finalize_kernel<<<(C + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(
      sums, count, gamma, beta, eps, momentum, running_mean, running_var, mean, rstd, scale, shift, C);
  return b2h::check_launch("bn_finalize");
}

int b200unet_bn_reduce_finalize(const float* stats_partial, int64_t rows, int C, double count, const float* gamma,
                                const float* beta, float eps, float momentum, float* running_mean, float* running_var,
                                int64_t* num_batches_tracked, float* mean, float* rstd, float* scale, float* shift,
                                b200_stream_t stream) {
  B2_REQUIRE(stats_partial && gamma && beta && mean && rstd && scale && shift && rows > 0 && C > 0 && count > 0,
             "bn_reduce_finalize: bad arguments");
  B2_REQUIRE((running_mean == nullptr) == (running_var == nullptr), "bn_reduce_finalize: running_mean / running_var go together");
  bn_reduce_finalize_kernel<<<(C + 31) / 32, 1024, 0, static_cast<cudaStream_t>(stream)>>>(
      stats_partial, rows, C, count, gamma, beta, eps, momentum, running_mean, running_var,
      reinterpret_cast<long long*>(num_batches_tracked), mean, rstd, scale, shift);
  return b2h::check_launch("bn_reduce_finalize");
}

int b200unet_bn_eval_affine(const float* gamma, const float* beta, const float* running_mean, const float* running_var,
                            float eps, float* scale, float* shift, int C, b200_stream_t stream) {
  B2_REQUIRE(running_mean && running_var, "bn_eval_affine: null running statistics (BatchNorm2d(track_running_stats=False))");
  B2_REQUIRE(gamma && beta && scale && shift && C > 0, "bn_eval_affine: null argument");
  bn_eval_affine_kernel<<<(C + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(gamma, beta, running_mean,
                                                                                      running_var, eps, scale, shift, C);
  return b2h::check_launch("bn_eval_affine");
}

int b200unet_bn_eval_stats(const float* running_mean, const float* running_var, float eps, float* mean, float* rstd, int C,
                           b200_stream_t stream) {
  B2_REQUIRE(running_mean && running_var && mean && rstd && C > 0, "bn_eval_stats: null argument");
  bn_eval_stats_kernel<<<(C + 127) / 128, 128, 0, static_cast<cudaStream_t>(stream)>>>(running_mean, running_var, eps, mean,
                                                                                     rstd, C);
  return b2h::check_launch("bn_eval_stats");
}

}  // extern "C"

namespace {

int bn_relu_fwd_impl(const void* y, int y_cs, const float* scale, const float* shift, void* a, int a_cs, void* pooled,
                     uint8_t* pool_idx, int N, int H, int W, int C, bool floor_mode, b200_stream_t stream) {
  B2_REQUIRE(ok_channels(C), "bn_relu_fwd: C=%d must be a power of two in [64, 2048]", C);
  B2_REQUIRE(y_cs % 8 == 0 && a_cs % 8 == 0, "bn_relu_fwd: pitches must be multiples of 8");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const auto* yy = static_cast<const __nv_bfloat16*>(y);
  auto* aa = static_cast<__nv_bfloat16*>(a);
  static int fwd_per_sm = 0;  // B200UNET_FWD_BLOCKS_PER_SM: grid cap of the BN-apply pass in resident blocks per SM (default 8)
  if (fwd_per_sm == 0) {
    const char* e = getenv("B200UNET_FWD_BLOCKS_PER_SM");
    fwd_per_sm = e != nullptr ? atoi(e) : 8;
    if (fwd_per_sm < 1 || fwd_per_sm > 8) fwd_per_sm = 8;
  }
  if (pooled == nullptr) {
    int blocks = ew_blocks(static_cast<long long>(N) * H * W * (C / 8));
    if (blocks > 148 * fwd_per_sm) blocks = 148 * fwd_per_sm;
    bn_relu_fwd_kernel<false><<<blocks, EW_THREADS, 0, st>>>(yy, y_cs, scale, shift, aa, a_cs, nullptr, nullptr, N, H, W, C,
                                                             ew_rev(0));
  } else {
    if (!floor_mode) B2_REQUIRE(H % 2 == 0 && W % 2 == 0, "bn_relu_fwd(pool): H=%d W=%d must be even", H, W);
    int blocks = ew_blocks(static_cast<long long>(N) * (H / 2) * (W / 2) * (C / 8));
    if (blocks > 148 * fwd_per_sm) blocks = 148 * fwd_per_sm;
    bn_relu_fwd_kernel<true><<<blocks, EW_THREADS, 0, st>>>(yy, y_cs, scale, shift, aa, a_cs,
                                                            static_cast<__nv_bfloat16*>(pooled), pool_idx, N, H, W, C,
                                                            ew_rev(0));
    if (const long long strip = floor_strip_pixels(floor_mode, true, N, H, W)) {
      if (int e = b2h::check_launch("bn_relu_fwd")) return e;
      int sb = ew_blocks(strip * (C / 8));
      if (sb > 148 * fwd_per_sm) sb = 148 * fwd_per_sm;
      bn_relu_fwd_kernel<false, true><<<sb, EW_THREADS, 0, st>>>(yy, y_cs, scale, shift, aa, a_cs, nullptr, nullptr, N, H, W,
                                                                 C, ew_rev(0));
    }
  }
  return b2h::check_launch("bn_relu_fwd");
}

int bn_relu_bwd_reduce_rows_impl(const void* g1, int g1_cs, const void* g_pool, const uint8_t* pool_idx, const void* y,
                                 int y_cs, const float* scale, const float* shift, const float* mean, const float* rstd,
                                 float* partial, int* rows_out, int N, int H, int W, int C, bool floor_mode,
                                 b200_stream_t stream) {
  B2_REQUIRE(ok_channels(C), "bn_relu_bwd_reduce: C=%d must be a power of two in [64, 2048]", C);
  B2_REQUIRE(g1 != nullptr || g_pool != nullptr, "bn_relu_bwd_reduce: no gradient source");
  B2_REQUIRE(y && scale && shift && mean && rstd && partial && rows_out,
             "bn_relu_bwd_reduce: null argument (eval-mode forwards must save mean/rstd: b200unet_bn_eval_stats)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  BwdSrc s{static_cast<const __nv_bfloat16*>(g1), g1_cs, static_cast<const __nv_bfloat16*>(g_pool), pool_idx,
           static_cast<const __nv_bfloat16*>(y), y_cs};
  const bool pool = g_pool != nullptr;
  if (pool) B2_REQUIRE((floor_mode || (H % 2 == 0 && W % 2 == 0)) && pool_idx != nullptr, "bn_relu_bwd_reduce(pool): bad arguments");
  const int blocks = bwd_blocks(N, H, W, C, pool);
  if (pool)
    bn_bwd_reduce_kernel<true><<<blocks, EW_THREADS, 0, st>>>(s, scale, shift, mean, rstd, partial, N, H, W, C, ew_rev(1));
  else
    bn_bwd_reduce_kernel<false><<<blocks, EW_THREADS, 0, st>>>(s, scale, shift, mean, rstd, partial, N, H, W, C, ew_rev(1));
  *rows_out = blocks;
  if (const long long strip = floor_strip_pixels(floor_mode, pool, N, H, W)) {
    // the strip's partial rows follow the windows'. Each launch is capped at 148 x per_sm <= EW_MAX_BLOCKS blocks
    // (B200UNET_BWD_BLOCKS_PER_SM up to 8), so the two together need up to 2 x EW_MAX_BLOCKS rows: what
    // b200unet_bn_bwd_workspace_floats sizes for when H or W is odd
    if (int e = b2h::check_launch("bn_relu_bwd_reduce")) return e;
    const int sb = bwd_blocks_for(strip, C);
    bn_bwd_reduce_kernel<false, true><<<sb, EW_THREADS, 0, st>>>(s, scale, shift, mean, rstd,
                                                                 partial + static_cast<size_t>(blocks) * 2 * C, N, H, W, C,
                                                                 ew_rev(1));
    *rows_out = blocks + sb;
  }
  return b2h::check_launch("bn_relu_bwd_reduce");
}

int bn_relu_bwd_apply_impl(const void* g1, int g1_cs, const void* g_pool, const uint8_t* pool_idx, const void* y, int y_cs,
                           const float* gamma, const float* scale, const float* shift, const float* mean, const float* rstd,
                           const double* sums, double count, const double* sums_local, void* dy, int dy_cs, float* dgamma,
                           float* dbeta, int N, int H, int W, int C, bool floor_mode, b200_stream_t stream) {
  B2_REQUIRE(ok_channels(C), "bn_relu_bwd_apply: C=%d must be a power of two in [64, 2048]", C);
  B2_REQUIRE(g1 != nullptr || g_pool != nullptr, "bn_relu_bwd_apply: no gradient source");
  B2_REQUIRE(y && gamma && scale && shift && mean && rstd && sums && dy,
             "bn_relu_bwd_apply: null argument (eval-mode forwards must save mean/rstd: b200unet_bn_eval_stats)");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  BwdSrc s{static_cast<const __nv_bfloat16*>(g1), g1_cs, static_cast<const __nv_bfloat16*>(g_pool), pool_idx,
           static_cast<const __nv_bfloat16*>(y), y_cs};
  const bool pool = g_pool != nullptr;
  if (pool) B2_REQUIRE((floor_mode || (H % 2 == 0 && W % 2 == 0)) && pool_idx != nullptr, "bn_relu_bwd_apply(pool): bad arguments");
  const int blocks = bwd_blocks(N, H, W, C, pool);
  if (pool)
    bn_bwd_apply_kernel<true><<<blocks, EW_THREADS, 0, st>>>(s, gamma, scale, shift, mean, rstd, sums, count, sums_local,
                                                             static_cast<__nv_bfloat16*>(dy), dy_cs, dgamma, dbeta, N, H,
                                                             W, C, ew_rev(2));
  else
    bn_bwd_apply_kernel<false><<<blocks, EW_THREADS, 0, st>>>(s, gamma, scale, shift, mean, rstd, sums, count, sums_local,
                                                              static_cast<__nv_bfloat16*>(dy), dy_cs, dgamma, dbeta, N,
                                                              H, W, C, ew_rev(2));
  if (const long long strip = floor_strip_pixels(floor_mode, pool, N, H, W)) {
    if (int e = b2h::check_launch("bn_relu_bwd_apply")) return e;
    bn_bwd_apply_kernel<false, true><<<bwd_blocks_for(strip, C), EW_THREADS, 0, st>>>(
        s, gamma, scale, shift, mean, rstd, sums, count, sums_local, static_cast<__nv_bfloat16*>(dy), dy_cs, nullptr, nullptr,
        N, H, W, C, ew_rev(2));
  }
  return b2h::check_launch("bn_relu_bwd_apply");
}

int maxpool2x2_fwd_impl(const void* a, int a_cs, void* pooled, int p_cs, uint8_t* pool_idx, int N, int H, int W, int C,
                        bool floor_mode, b200_stream_t stream) {
  B2_REQUIRE(C > 0 && C % 8 == 0 && a_cs % 8 == 0 && p_cs % 8 == 0 && a_cs >= C && p_cs >= C,
             "maxpool2x2_fwd: C=%d and the pitches (%d, %d) must be multiples of 8 with pitch >= C", C, a_cs, p_cs);
  if (floor_mode)
    B2_REQUIRE(N > 0 && H >= 2 && W >= 2, "maxpool2x2_fwd: N=%d H=%d W=%d: the map must be at least 2x2", N, H, W);
  else
    B2_REQUIRE(N > 0 && H >= 2 && W >= 2 && H % 2 == 0 && W % 2 == 0, "maxpool2x2_fwd: H=%d W=%d must be even and >= 2", H, W);
  const int blocks = ew_blocks(static_cast<long long>(N) * (H / 2) * (W / 2) * (C / 8));
  maxpool_fwd_kernel<<<blocks, EW_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(a), a_cs, static_cast<__nv_bfloat16*>(pooled), p_cs, pool_idx, N, H, W, C);
  return b2h::check_launch("maxpool2x2_fwd");
}

// what the floor-mode entry points check on top of the shared implementations: the map is at least 2x2 when pooled, and
// every pitch holds the channels (a pooled call reads 2x2 windows and writes [N][H/2][W/2][C] unchecked)
int floor_pool_args(const char* what, bool pooled, int N, int H, int W, int C, int y_cs, const void* g1, int g1_cs, int out_cs) {
  B2_REQUIRE(N > 0 && H > 0 && W > 0, "%s: empty map N=%d H=%d W=%d", what, N, H, W);
  B2_REQUIRE(N * strip_pixels_per_image(H, W) * (C / 8) <= STRIP_MAX_ITEMS, "%s: pad strip too large", what);
  B2_REQUIRE(!pooled || (H >= 2 && W >= 2), "%s(pool): H=%d W=%d: the map must be at least 2x2", what, H, W);
  B2_REQUIRE(y_cs >= C && y_cs % 8 == 0 && out_cs >= C && out_cs % 8 == 0 && (g1 == nullptr || (g1_cs >= C && g1_cs % 8 == 0)),
             "%s: pixel pitches (%d, %d, %d) must be multiples of 8 and >= C=%d", what, y_cs, g1 == nullptr ? 0 : g1_cs, out_cs, C);
  return 0;
}

int strip_args(const char* what, const void* x, int x_cs, int N, int H, int W, int C) {
  B2_REQUIRE(x != nullptr, "%s: null tensor", what);
  B2_REQUIRE(N > 0 && H > 0 && W > 0, "%s: empty map N=%d H=%d W=%d", what, N, H, W);
  B2_REQUIRE(C > 0 && C % 8 == 0 && x_cs % 8 == 0 && x_cs >= C,
             "%s: C=%d and the pixel pitch %d must be multiples of 8 with pitch >= C", what, C, x_cs);
  B2_REQUIRE(reinterpret_cast<uintptr_t>(x) % 16 == 0, "%s: the slice must start on a 16-byte boundary", what);
  B2_REQUIRE(N * strip_pixels_per_image(H, W) * (C / 8) <= STRIP_MAX_ITEMS, "%s: pad strip too large", what);
  return 0;
}

}  // namespace

extern "C" {

int b200unet_bn_relu_fwd(const void* y, int y_cs, const float* scale, const float* shift, void* a, int a_cs, void* pooled,
                         uint8_t* pool_idx, int N, int H, int W, int C, b200_stream_t stream) {
  return bn_relu_fwd_impl(y, y_cs, scale, shift, a, a_cs, pooled, pool_idx, N, H, W, C, false, stream);
}

int b200unet_bn_relu_fwd_floor(const void* y, int y_cs, const float* scale, const float* shift, void* a, int a_cs,
                               void* pooled, uint8_t* pool_idx, int N, int H, int W, int C, b200_stream_t stream) {
  B2_REQUIRE(y && scale && shift && a, "bn_relu_fwd_floor: null argument");
  B2_REQUIRE(pooled != nullptr || pool_idx == nullptr, "bn_relu_fwd_floor: pool_idx without pooled");
  if (int e = floor_pool_args("bn_relu_fwd_floor", pooled != nullptr, N, H, W, C, y_cs, nullptr, 0, a_cs)) return e;
  return bn_relu_fwd_impl(y, y_cs, scale, shift, a, a_cs, pooled, pool_idx, N, H, W, C, true, stream);
}

int64_t b200unet_bn_bwd_workspace_floats(int N, int H, int W, int C) {
  (void)N;
  // odd H or W: a floor-mode pooled reduce writes the pad strip's partial rows after the windows' (two launches)
  const int launches = strip_pixels_per_image(H, W) > 0 ? 2 : 1;
  return static_cast<int64_t>(launches) * EW_MAX_BLOCKS * 2 * C;
}

int b200unet_bn_relu_bwd_reduce(const void* g1, int g1_cs, const void* g_pool, const uint8_t* pool_idx, const void* y,
                                int y_cs, const float* scale, const float* shift, const float* mean, const float* rstd,
                                float* partial, double* sums, int N, int H, int W, int C, b200_stream_t stream) {
  B2_REQUIRE(sums != nullptr, "bn_relu_bwd_reduce: null sums");
  int rows = 0;
  if (int e = b200unet_bn_relu_bwd_reduce_rows(g1, g1_cs, g_pool, pool_idx, y, y_cs, scale, shift, mean, rstd, partial, &rows, N,
                                               H, W, C, stream))
    return e;
  return launch_reduce_partials(partial, rows, 2 * C, sums, static_cast<cudaStream_t>(stream));
}

int b200unet_bn_relu_bwd_reduce_rows(const void* g1, int g1_cs, const void* g_pool, const uint8_t* pool_idx, const void* y,
                                     int y_cs, const float* scale, const float* shift, const float* mean, const float* rstd,
                                     float* partial, int* rows_out, int N, int H, int W, int C, b200_stream_t stream) {
  return bn_relu_bwd_reduce_rows_impl(g1, g1_cs, g_pool, pool_idx, y, y_cs, scale, shift, mean, rstd, partial, rows_out, N, H,
                                      W, C, false, stream);
}

int b200unet_bn_relu_bwd_apply(const void* g1, int g1_cs, const void* g_pool, const uint8_t* pool_idx, const void* y,
                               int y_cs, const float* gamma, const float* scale, const float* shift, const float* mean,
                               const float* rstd, const double* sums, double count, const double* sums_local, void* dy,
                               int dy_cs, float* dgamma, float* dbeta, int N, int H, int W, int C, b200_stream_t stream) {
  return bn_relu_bwd_apply_impl(g1, g1_cs, g_pool, pool_idx, y, y_cs, gamma, scale, shift, mean, rstd, sums, count, sums_local,
                                dy, dy_cs, dgamma, dbeta, N, H, W, C, false, stream);
}

int b200unet_bn_relu_bwd_reduce_rows_floor(const void* g1, int g1_cs, const void* g_pool, const uint8_t* pool_idx,
                                           const void* y, int y_cs, const float* scale, const float* shift, const float* mean,
                                           const float* rstd, float* partial, int* rows_out, int N, int H, int W, int C,
                                           b200_stream_t stream) {
  B2_REQUIRE(g_pool == nullptr || pool_idx != nullptr, "bn_relu_bwd_reduce_floor(pool): a pooled gradient needs pool_idx");
  if (int e = floor_pool_args("bn_relu_bwd_reduce_floor", g_pool != nullptr, N, H, W, C, y_cs, g1, g1_cs, y_cs)) return e;
  return bn_relu_bwd_reduce_rows_impl(g1, g1_cs, g_pool, pool_idx, y, y_cs, scale, shift, mean, rstd, partial, rows_out, N, H,
                                      W, C, true, stream);
}

int b200unet_bn_relu_bwd_reduce_floor(const void* g1, int g1_cs, const void* g_pool, const uint8_t* pool_idx, const void* y,
                                      int y_cs, const float* scale, const float* shift, const float* mean, const float* rstd,
                                      float* partial, double* sums, int N, int H, int W, int C, b200_stream_t stream) {
  B2_REQUIRE(sums != nullptr, "bn_relu_bwd_reduce_floor: null sums");
  int rows = 0;
  if (int e = b200unet_bn_relu_bwd_reduce_rows_floor(g1, g1_cs, g_pool, pool_idx, y, y_cs, scale, shift, mean, rstd, partial,
                                                     &rows, N, H, W, C, stream))
    return e;
  return launch_reduce_partials(partial, rows, 2 * C, sums, static_cast<cudaStream_t>(stream));
}

int b200unet_bn_relu_bwd_apply_floor(const void* g1, int g1_cs, const void* g_pool, const uint8_t* pool_idx, const void* y,
                                     int y_cs, const float* gamma, const float* scale, const float* shift, const float* mean,
                                     const float* rstd, const double* sums, double count, const double* sums_local, void* dy,
                                     int dy_cs, float* dgamma, float* dbeta, int N, int H, int W, int C,
                                     b200_stream_t stream) {
  B2_REQUIRE(g_pool == nullptr || pool_idx != nullptr, "bn_relu_bwd_apply_floor(pool): a pooled gradient needs pool_idx");
  if (int e = floor_pool_args("bn_relu_bwd_apply_floor", g_pool != nullptr, N, H, W, C, y_cs, g1, g1_cs, dy_cs)) return e;
  return bn_relu_bwd_apply_impl(g1, g1_cs, g_pool, pool_idx, y, y_cs, gamma, scale, shift, mean, rstd, sums, count, sums_local,
                                dy, dy_cs, dgamma, dbeta, N, H, W, C, true, stream);
}

int b200unet_partial_colsum(const float* partial, int64_t rows, int row_pitch, int col_lo, int n, float* out,
                            b200_stream_t stream) {
  B2_REQUIRE(rows > 0 && n > 0 && col_lo >= 0 && col_lo + n <= row_pitch, "partial_colsum: bad column range");
  partial_colsum_kernel<<<(n + 31) / 32, 256, 0, static_cast<cudaStream_t>(stream)>>>(partial, rows, row_pitch, col_lo, n, out);
  return b2h::check_launch("partial_colsum");
}

int64_t b200unet_channel_sum_workspace_floats(int C) { return static_cast<int64_t>(EW_MAX_BLOCKS) * C + 2 * C; }

int b200unet_channel_sum(const void* x, int x_cs, float* workspace, float* out, int64_t pixels, int C,
                         b200_stream_t stream) {
  B2_REQUIRE(ok_channels(C), "channel_sum: C=%d must be a power of two in [64, 2048]", C);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int blocks = ew_blocks(pixels * (C / 8));
  channel_sum_kernel<<<blocks, EW_THREADS, 0, st>>>(static_cast<const __nv_bfloat16*>(x), x_cs, workspace, pixels, C);
  if (int e = b2h::check_launch("channel_sum")) return e;
  // fp64 accumulator lives at the (8-byte aligned) tail of the workspace
  double* acc = reinterpret_cast<double*>(workspace + static_cast<size_t>(EW_MAX_BLOCKS) * C);
  if (int e = launch_reduce_partials(workspace, blocks, C, acc, st)) return e;
  double_to_float_kernel<<<(C + 127) / 128, 128, 0, st>>>(acc, out, C);
  return b2h::check_launch("channel_sum_cast");
}

int b200unet_maxpool2x2_fwd(const void* a, int a_cs, void* pooled, int p_cs, uint8_t* pool_idx, int N, int H, int W, int C,
                            b200_stream_t stream) {
  return maxpool2x2_fwd_impl(a, a_cs, pooled, p_cs, pool_idx, N, H, W, C, false, stream);
}

int b200unet_maxpool2x2_fwd_floor(const void* a, int a_cs, void* pooled, int p_cs, uint8_t* pool_idx, int N, int H, int W,
                                  int C, b200_stream_t stream) {
  B2_REQUIRE(a && pooled, "maxpool2x2_fwd_floor: null argument");
  return maxpool2x2_fwd_impl(a, a_cs, pooled, p_cs, pool_idx, N, H, W, C, true, stream);
}

int b200unet_pad_strip_zero(void* x, int x_cs, int N, int H, int W, int C, b200_stream_t stream) {
  if (int e = strip_args("pad_strip_zero", x, x_cs, N, H, W, C)) return e;
  const long long items = N * strip_pixels_per_image(H, W) * (C / 8);
  if (items == 0) return 0;
  pad_strip_zero_kernel<<<ew_blocks(items), EW_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<__nv_bfloat16*>(x), x_cs, N, H, W, C);
  return b2h::check_launch("pad_strip_zero");
}

int b200unet_pad_strip_sub_colsum(const void* x, int x_cs, int N, int H, int W, int C, float* out, b200_stream_t stream) {
  if (int e = strip_args("pad_strip_sub_colsum", x, x_cs, N, H, W, C)) return e;
  B2_REQUIRE(out != nullptr, "pad_strip_sub_colsum: null out");
  if (strip_pixels_per_image(H, W) == 0) return 0;
  pad_strip_sub_colsum_kernel<<<(C + 31) / 32, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(x), x_cs, N, H, W, C, out);
  return b2h::check_launch("pad_strip_sub_colsum");
}

int b200unet_nhwc_copy(const void* src, int src_cs, void* dst, int dst_cs, int64_t pixels, int C, b200_stream_t stream) {
  B2_REQUIRE(C > 0 && C % 8 == 0 && src_cs % 8 == 0 && dst_cs % 8 == 0 && src_cs >= C && dst_cs >= C,
             "nhwc_copy: C=%d and the pixel pitches (%d, %d) must be multiples of 8 with pitch >= C", C, src_cs, dst_cs);
  B2_REQUIRE(pixels > 0, "nhwc_copy: empty tensor");
  slice_copy_add_kernel<false><<<ew_blocks(pixels * (C / 8)), EW_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(src), src_cs, nullptr, 0, static_cast<__nv_bfloat16*>(dst), dst_cs, pixels, C);
  return b2h::check_launch("nhwc_copy");
}

int b200unet_nhwc_add(const void* a, int a_cs, const void* b, int b_cs, void* out, int out_cs, int64_t pixels, int C,
                      b200_stream_t stream) {
  B2_REQUIRE(C > 0 && C % 8 == 0 && a_cs % 8 == 0 && b_cs % 8 == 0 && out_cs % 8 == 0 && a_cs >= C && b_cs >= C && out_cs >= C,
             "nhwc_add: C=%d and the pixel pitches (%d, %d, %d) must be multiples of 8 with pitch >= C", C, a_cs, b_cs, out_cs);
  B2_REQUIRE(pixels > 0, "nhwc_add: empty tensor");
  slice_copy_add_kernel<true><<<ew_blocks(pixels * (C / 8)), EW_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __nv_bfloat16*>(a), a_cs, static_cast<const __nv_bfloat16*>(b), b_cs,
      static_cast<__nv_bfloat16*>(out), out_cs, pixels, C);
  return b2h::check_launch("nhwc_add");
}

}  // extern "C"
