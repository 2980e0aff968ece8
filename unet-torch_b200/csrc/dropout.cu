// nn.Dropout (Model.py:34-39 after MaxPool2d in Down, :80-81 after the concat in Up) as one in-place element-wise pass over
// a channel slice of an NHWC bf16 buffer. The mask is a counter-based function of (seed, site, element index) only
// (DESIGN.md §4): forward and backward regenerate it independently, so nothing is stored and a captured CUDA graph that
// reads the seed through a device pointer draws a new mask on every replay. For the element with NHWC index
// e = ((n*H + h)*W + w)*C_site + c of the site tensor:
//   r = Philox4x32-10(counter = (lo32(e/4), hi32(e/4), site, 0), key = (lo32(seed), hi32(seed)))
//   out = r[e % 4] < threshold ? bf16(float(x) * scale) : 0
#include "../../include/b200unet.h"
#include "ew_common.cuh"
#include "host_common.h"

#include <cuda_bf16.h>

namespace {

using namespace b2ew;

constexpr int DROP_THREADS = 256;
constexpr int DROP_MAX_BLOCKS = 148 * 8;

// Random123's Philox4x32-10 (Salmon et al., SC'11): ten rounds of two 32x32 -> 64-bit products, key bumped after each.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += 0x9E3779B9u;
    k.y += 0xBB67AE85u;
  }
  return c;
}

__device__ __forceinline__ uint4 philox_at(unsigned long long q, uint32_t site, uint2 key) {
  return philox4x32_10(make_uint4(static_cast<uint32_t>(q), static_cast<uint32_t>(q >> 32), site, 0u), key);
}

// keep[j] for the elements e0 .. e0 + 7: two Philox calls when e0 is a multiple of 4 (every site of the network), three
// otherwise. The word index is a compile-time constant in each branch, so w[] stays in registers.
__device__ __forceinline__ void keep8(unsigned long long e0, uint32_t site, uint2 key, uint32_t threshold, bool (&keep)[8]) {
  const unsigned long long q = e0 >> 2;
  const int off = static_cast<int>(e0 & 3);
  uint32_t w[12];
  const uint4 r0 = philox_at(q, site, key), r1 = philox_at(q + 1, site, key);
  w[0] = r0.x; w[1] = r0.y; w[2] = r0.z; w[3] = r0.w;
  w[4] = r1.x; w[5] = r1.y; w[6] = r1.z; w[7] = r1.w;
  if (off == 0) {
#pragma unroll
    for (int j = 0; j < 8; ++j) keep[j] = w[j] < threshold;
    return;
  }
  const uint4 r2 = philox_at(q + 2, site, key);
  w[8] = r2.x; w[9] = r2.y; w[10] = r2.z; w[11] = r2.w;
  if (off == 1) {
#pragma unroll
    for (int j = 0; j < 8; ++j) keep[j] = w[j + 1] < threshold;
  } else if (off == 2) {
#pragma unroll
    for (int j = 0; j < 8; ++j) keep[j] = w[j + 2] < threshold;
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) keep[j] = w[j + 3] < threshold;
  }
}

struct DropArgs {
  __nv_bfloat16* x;           // channel c_lo of the site tensor, pixel pitch x_cs
  long long pixels;           // N * H * W
  int x_cs, c_site, c_lo, nc;
  uint32_t site, threshold;
  float scale;
  const long long* seed;      // one int64 on the device
  float* partial;             // [gridDim.x][sum_n] per-block sums of the output channels [sum_lo, sum_lo + sum_n), or null
  int sum_lo, sum_n;
};

// Thread t owns the 8-channel group g of pixel row r of its block (cgs = nc / 8 groups per pixel; 256 / cgs rows per block,
// one row that loops over the groups when cgs > 256). A thread keeps its group for the whole grid-stride loop, so the
// per-block sums are per-thread fp32 sums reduced in a fixed order: no atomics, bit-reproducible for a given shape.
template <bool SUMS>
__global__ void __launch_bounds__(DROP_THREADS) dropout_mul_kernel(const DropArgs a) {
  const int cgs = a.nc >> 3;
  const int rpb = cgs >= DROP_THREADS ? 1 : DROP_THREADS / cgs;
  const int r = cgs >= DROP_THREADS ? 0 : static_cast<int>(threadIdx.x) / cgs;
  const int g0 = cgs >= DROP_THREADS ? static_cast<int>(threadIdx.x) : static_cast<int>(threadIdx.x) % cgs;
  const unsigned long long seed = static_cast<unsigned long long>(*a.seed);
  const uint2 key = make_uint2(static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (r < rpb) {
    for (long long p = static_cast<long long>(blockIdx.x) * rpb + r; p < a.pixels; p += static_cast<long long>(gridDim.x) * rpb) {
      for (int g = g0; g < cgs; g += DROP_THREADS) {
        uint4* ptr = reinterpret_cast<uint4*>(a.x + p * a.x_cs + g * 8);
        float f[8];
        unpack8(*ptr, f);
        bool keep[8];
        keep8(static_cast<unsigned long long>(p) * a.c_site + a.c_lo + g * 8, a.site, key, a.threshold, keep);
#pragma unroll
        for (int j = 0; j < 8; ++j) f[j] = keep[j] ? bf16_round(f[j] * a.scale) : 0.f;
        *ptr = pack8(f);
        if (SUMS) {
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[j] += f[j];
        }
      }
    }
  }
  if (SUMS) {
    __shared__ float sh[DROP_THREADS][9];
#pragma unroll
    for (int j = 0; j < 8; ++j) sh[threadIdx.x][j] = acc[j];
    __syncthreads();
    for (int i = threadIdx.x; i < a.sum_n; i += DROP_THREADS) {
      const int c = a.sum_lo + i;
      float s = 0.f;
      for (int rr = 0; rr < rpb; ++rr) s += sh[rr * cgs + (c >> 3)][c & 7];
      a.partial[static_cast<size_t>(blockIdx.x) * a.sum_n + i] = s;
    }
  }
}

int drop_blocks(long long pixels, int nc) {
  const int cgs = nc / 8;
  const long long rpb = cgs >= DROP_THREADS ? 1 : DROP_THREADS / cgs;
  long long b = (pixels + rpb - 1) / rpb;
  if (b > DROP_MAX_BLOCKS) b = DROP_MAX_BLOCKS;
  if (b < 1) b = 1;
  return static_cast<int>(b);
}

}  // namespace

extern "C" {

int b200unet_dropout_partial_rows(int N, int H, int W, int nc) {
  if (N <= 0 || H <= 0 || W <= 0 || nc <= 0 || nc % 8) return 0;
  return drop_blocks(static_cast<long long>(N) * H * W, nc);
}

int b200unet_dropout_mul(void* x, int x_cs, int N, int H, int W, int C_site, int c_lo, int nc, int site, const int64_t* seed,
                         int64_t threshold, float scale, float* partial, int sum_lo, int sum_n, b200_stream_t stream) {
  B2_REQUIRE(x != nullptr && seed != nullptr, "dropout_mul: null tensor or seed");
  B2_REQUIRE(N > 0 && H > 0 && W > 0, "dropout_mul: empty tensor (N=%d H=%d W=%d)", N, H, W);
  B2_REQUIRE(nc > 0 && nc % 8 == 0 && x_cs % 8 == 0 && x_cs >= nc,
             "dropout_mul: nc=%d and the pixel pitch %d must be multiples of 8 with pitch >= nc", nc, x_cs);
  B2_REQUIRE(reinterpret_cast<uintptr_t>(x) % 16 == 0, "dropout_mul: the slice must start on a 16-byte boundary");
  B2_REQUIRE(c_lo >= 0 && c_lo + nc <= C_site, "dropout_mul: channels [%d, %d) outside the site's %d", c_lo, c_lo + nc, C_site);
  B2_REQUIRE(site >= 0 && threshold >= 0 && threshold <= 0xffffffffLL, "dropout_mul: bad site %d or threshold", site);
  const long long pixels = static_cast<long long>(N) * H * W;
  DropArgs a{static_cast<__nv_bfloat16*>(x), pixels, x_cs, C_site, c_lo, nc, static_cast<uint32_t>(site),
             static_cast<uint32_t>(threshold), scale, reinterpret_cast<const long long*>(seed), partial, sum_lo, sum_n};
  const int blocks = drop_blocks(pixels, nc);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (partial != nullptr) {
    B2_REQUIRE(nc <= 8 * DROP_THREADS, "dropout_mul: channel sums need nc <= %d (got %d)", 8 * DROP_THREADS, nc);
    B2_REQUIRE(sum_n > 0 && sum_lo >= 0 && sum_lo + sum_n <= nc, "dropout_mul: sum range [%d, %d) outside the slice's %d",
               sum_lo, sum_lo + sum_n, nc);
    dropout_mul_kernel<true><<<blocks, DROP_THREADS, 0, st>>>(a);
  } else {
    dropout_mul_kernel<false><<<blocks, DROP_THREADS, 0, st>>>(a);
  }
  return b2h::check_launch("dropout_mul");
}

}  // extern "C"
