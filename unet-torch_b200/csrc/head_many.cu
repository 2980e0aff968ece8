// OutConv (nn.Conv2d(C, n_classes, 1), Model.py:86-92) and its inference epilogues for 1..256 classes. The heads of
// small.cu / edge.cu are compiled once per class count up to 8 and stay the path there; these kernels walk the classes in
// compile-time chunks of b2head::CHUNK over zero-padded weight rows (head_common.cuh), so the class count is a run-time
// argument without per-class predicates. Cin is 64 or 128 (the networks' base widths), a compile-time KC = Cin / 64.
#include "../../include/b200unet.h"
#include "host_common.h"
#include "head_common.cuh"

#include <cuda_bf16.h>

namespace {

using b2head::CHUNK;
using b2head::MANY_MAXC;
using b2head::STAGE_BYTES_PER_WARP;
using b2head::pad_classes;

constexpr int MAX_SMEM = 227 * 1024;
constexpr int MAX_BLOCKS = 148 * 8;

__device__ __forceinline__ uint32_t pack2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

// dynamic shared memory: weights [np][Cin], bias [np], one staging tile per warp, then `extra` bytes per warp
struct ManySmem {
  float* w;
  float* b;
  uint32_t* stage;
  char* extra;
};
template <int KC>
__device__ __forceinline__ ManySmem many_smem(float* smem, int ncls, int extra_per_warp) {
  const int np = pad_classes(ncls);
  const int warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
  ManySmem s;
  s.w = smem;
  s.b = smem + np * KC * 64;
  char* stages = reinterpret_cast<char*>(s.b + np);
  s.stage = reinterpret_cast<uint32_t*>(stages + warp * STAGE_BYTES_PER_WARP);
  s.extra = stages + warps * STAGE_BYTES_PER_WARP + warp * extra_per_warp;
  return s;
}

// ---------------------------------------------------------------------------------------------- forward
// two blocks per SM at Cin = 64 (at most 128 registers)
template <int KC>
__global__ void __launch_bounds__(256, 3 - KC) head_many_fprop_kernel(const __nv_bfloat16* __restrict__ a, int a_cs,
                                                              const float* __restrict__ w, const float* __restrict__ bias,
                                                              float* __restrict__ z, long long P, long long HW, int ncls) {
  extern __shared__ __align__(16) float smem[];
  const ManySmem s = many_smem<KC>(smem, ncls, 0);
  b2head::load_weights_padded(s.w, s.b, w, bias, KC * 64, ncls);
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long warps = static_cast<long long>(gridDim.x) * (blockDim.x >> 5);
  for (long long g = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); g * 32 < P; g += warps) {
    uint4 row[KC * 8];
    b2head::load_rows_warp32<KC>(a, a_cs, s.stage, g * 32, P, row);
    const long long p = g * 32 + lane;
    if (p >= P) continue;
    const long long n = p / HW, hw = p - n * HW;
    float* out = z + n * ncls * HW + hw;
    int j0 = 0;
    for (; j0 + CHUNK <= ncls; j0 += CHUNK) {
      float zc[CHUNK];
      b2head::logits_chunk<KC>(row, s.w, s.b, j0, zc);
#pragma unroll
      for (int j = 0; j < CHUNK; ++j) out[(j0 + j) * HW] = zc[j];
    }
    if (j0 < ncls) {
      float zc[CHUNK];
      b2head::logits_chunk<KC>(row, s.w, s.b, j0, zc);
#pragma unroll
      for (int j = 0; j < CHUNK; ++j)
        if (j0 + j < ncls) out[(j0 + j) * HW] = zc[j];
    }
  }
}

// ---------------------------------------------------------------------------------------------- mask / density
// The softmax -> first-maximum argmax of softmax_argmax_many_kernel (loss.cu) on logits parked in shared memory
// ([np][32] per warp): max, then sum_j expf(z_j - max) in class order, then p_j = expf(z_j - max) / sum; a NaN
// probability wins over a number, the first maximum wins a tie. Same operations, so the same mask as the two-kernel path.
template <int KC>
__global__ void __launch_bounds__(256) head_many_mask_kernel(const __nv_bfloat16* __restrict__ a, int a_cs,
                                                             const float* __restrict__ w, const float* __restrict__ bias,
                                                             uint8_t* __restrict__ mask, long long P, int ncls) {
  extern __shared__ __align__(16) float smem[];
  const int np = pad_classes(ncls);
  const ManySmem s = many_smem<KC>(smem, ncls, np * 32 * 4);
  float* zs = reinterpret_cast<float*>(s.extra);
  b2head::load_weights_padded(s.w, s.b, w, bias, KC * 64, ncls);
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long warps = static_cast<long long>(gridDim.x) * (blockDim.x >> 5);
  for (long long g = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5); g * 32 < P; g += warps) {
    uint4 row[KC * 8];
    b2head::load_rows_warp32<KC>(a, a_cs, s.stage, g * 32, P, row);
    for (int j0 = 0; j0 < ncls; j0 += CHUNK) {
      float zc[CHUNK];
      b2head::logits_chunk<KC>(row, s.w, s.b, j0, zc);
#pragma unroll
      for (int j = 0; j < CHUNK; ++j) zs[(j0 + j) * 32 + lane] = zc[j];
    }
    const long long p = g * 32 + lane;
    if (p >= P) continue;
    float m = -INFINITY;
#pragma unroll 8
    for (int j = 0; j < ncls; ++j) m = fmaxf(m, zs[j * 32 + lane]);
    float sum = 0.f;
#pragma unroll 8
    for (int j = 0; j < ncls; ++j) sum += expf(zs[j * 32 + lane] - m);
    int best = 0;
    float bv = expf(zs[lane] - m) / sum;
#pragma unroll 8
    for (int j = 1; j < ncls; ++j) {
      const float pj = expf(zs[j * 32 + lane] - m) / sum;
      if (pj > bv || (pj != pj && bv == bv)) {
        bv = pj;
        best = j;
      }
    }
    mask[p] = static_cast<uint8_t>(best);
  }
}

// OutConv + F.relu + division by `divisor` -> fp32 NCHW maps, and per-(image, class) fp64 sums of the stored values. Per
// chunk the warp folds its 32 lanes (fixed shuffle tree) into a per-warp fp64 row in shared memory; the block adds the
// warps' rows in order and one atomic per class joins the blocks of an image (as head_density does).
template <int KC>
__global__ void __launch_bounds__(256) head_many_density_kernel(const __nv_bfloat16* __restrict__ a, int a_cs,
                                                                const float* __restrict__ w, const float* __restrict__ bias,
                                                                float* __restrict__ out, double* __restrict__ counts,
                                                                long long HW, int blocks_per_image, int ncls, float divisor) {
  extern __shared__ __align__(16) float smem[];
  const int np = pad_classes(ncls);
  const ManySmem s = many_smem<KC>(smem, ncls, np * 8);
  double* red = reinterpret_cast<double*>(s.extra);
  b2head::load_weights_padded(s.w, s.b, w, bias, KC * 64, ncls);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  for (int j = lane; j < np; j += 32) red[j] = 0.0;
  __syncthreads();
  const int n = blockIdx.x / blocks_per_image, b = blockIdx.x % blocks_per_image;
  const __nv_bfloat16* src = a + static_cast<long long>(n) * HW * a_cs;
  float* dst = out + static_cast<long long>(n) * ncls * HW;
  for (long long g = static_cast<long long>(b) * nwarps + warp; g * 32 < HW; g += static_cast<long long>(blocks_per_image) * nwarps) {
    uint4 row[KC * 8];
    b2head::load_rows_warp32<KC>(src, a_cs, s.stage, g * 32, HW, row);
    const long long hw = g * 32 + lane;
    const bool live = hw < HW;
    for (int j0 = 0; j0 < ncls; j0 += CHUNK) {
      float zc[CHUNK];
      b2head::logits_chunk<KC>(row, s.w, s.b, j0, zc);
      double part[CHUNK];
#pragma unroll
      for (int j = 0; j < CHUNK; ++j) {
        // F.relu keeps NaN; fmaxf would drop it
        const float r = (zc[j] > 0.f || zc[j] != zc[j]) ? zc[j] : 0.f;
        const float v = r / divisor;
        part[j] = 0.0;
        if (live && j0 + j < ncls) {
          dst[(j0 + j) * HW + hw] = v;
          part[j] = static_cast<double>(v);
        }
      }
      if (counts == nullptr) continue;
#pragma unroll
      for (int j = 0; j < CHUNK; ++j) {
        double v = part[j];
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (lane == 0) red[j0 + j] += v;
      }
    }
  }
  if (counts == nullptr) return;
  __syncthreads();
  for (int j = threadIdx.x; j < ncls; j += blockDim.x) {
    double t = 0.0;
    for (int wv = 0; wv < nwarps; ++wv) t += red[(wv - warp) * np + j];  // red is this warp's row
    atomicAdd(counts + static_cast<long long>(n) * ncls + j, t);
  }
}

// ---------------------------------------------------------------------------------------------- backward
// da[p][c] = bf16(sum_j dz[j][p] w[j][c]), classes in order (fmaf from 0, as head_bwd_kernel). Thread = (pixel pair,
// 8-channel group cg); per class chunk the block stages dz[CHUNK][T] for its tile of T pixels.
template <int KC>
__global__ void __launch_bounds__(256) head_many_dgrad_kernel(const float* __restrict__ dz, const float* __restrict__ w,
                                                              __nv_bfloat16* __restrict__ da, int da_cs, long long P,
                                                              long long HW, int ncls) {
  constexpr int Cin = KC * 64, CGS = Cin / 8, PPB = 256 / CGS, T = 2 * PPB;
  extern __shared__ __align__(16) float smem[];
  const int np = pad_classes(ncls);
  float* wsm = smem;                 // [np][Cin], zero rows past ncls
  float* dzs = smem + np * Cin;      // [CHUNK][T]
  for (int i = threadIdx.x; i < np * Cin; i += blockDim.x) wsm[i] = (i < ncls * Cin) ? w[i] : 0.f;
  const int cg = threadIdx.x % CGS, pl = threadIdx.x / CGS;
  const long long ntiles = (P + T - 1) / T;
  for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const long long p0 = tile * T;
    float o[2][8];
#pragma unroll
    for (int u = 0; u < 2; ++u)
#pragma unroll
      for (int i = 0; i < 8; ++i) o[u][i] = 0.f;
    for (int j0 = 0; j0 < ncls; j0 += CHUNK) {
      __syncthreads();  // weights loaded / the previous chunk's reads of dzs are done
      for (int e = threadIdx.x; e < CHUNK * T; e += blockDim.x) {
        const int j = e / T, lp = e % T;
        const long long p = p0 + lp;
        const long long n = p / HW, hw = p - n * HW;
        dzs[e] = (p < P && j0 + j < ncls) ? __ldg(dz + (n * ncls + j0 + j) * HW + hw) : 0.f;
      }
      __syncthreads();
#pragma unroll
      for (int j = 0; j < CHUNK; ++j) {
        const float4 w0 = *reinterpret_cast<const float4*>(wsm + (j0 + j) * Cin + cg * 8);
        const float4 w1 = *reinterpret_cast<const float4*>(wsm + (j0 + j) * Cin + cg * 8 + 4);
        const float wr[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const float g = dzs[j * T + u * PPB + pl];
#pragma unroll
          for (int i = 0; i < 8; ++i) o[u][i] = fmaf(g, wr[i], o[u][i]);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const long long p = p0 + u * PPB + pl;
      if (p < P)
        *reinterpret_cast<uint4*>(da + p * da_cs + cg * 8) =
            make_uint4(pack2(o[u][0], o[u][1]), pack2(o[u][2], o[u][3]), pack2(o[u][4], o[u][5]), pack2(o[u][6], o[u][7]));
    }
  }
}

// dW / db partials of one class chunk (blockIdx.x % nchunks) over the tiles of one pixel slice (blockIdx.x / nchunks):
// the blocks of one slice run side by side, so the activation tile they all read comes from L2 after the first.
// partial layout [slice][np][Cin + 1], last column = bias gradient; fp32 in registers, one fixed-order block reduction.
template <int KC>
__global__ void __launch_bounds__(256) head_many_wgrad_kernel(const float* __restrict__ dz, const __nv_bfloat16* __restrict__ a,
                                                              int a_cs, float* __restrict__ partial, long long P, long long HW,
                                                              int ncls, int nchunks) {
  constexpr int Cin = KC * 64, CGS = Cin / 8, PPB = 256 / CGS;
  __shared__ float dzs[CHUNK][256];
  __shared__ float sh[256][9];
  const int np = pad_classes(ncls);
  const int chunk = blockIdx.x % nchunks, slice = blockIdx.x / nchunks, slices = gridDim.x / nchunks;
  const int j0 = chunk * CHUNK;
  const int cg = threadIdx.x % CGS, pl = threadIdx.x / CGS;
  float dwacc[CHUNK][8], dbacc[CHUNK];
#pragma unroll
  for (int j = 0; j < CHUNK; ++j) {
    dbacc[j] = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) dwacc[j][i] = 0.f;
  }
  const long long ntiles = (P + 255) / 256;
  for (long long tile = slice; tile < ntiles; tile += slices) {
    const long long p0 = tile * 256;
    __syncthreads();
    {
      const long long p = p0 + threadIdx.x;
      const long long n = p / HW, hw = p - n * HW;
#pragma unroll
      for (int j = 0; j < CHUNK; ++j)
        dzs[j][threadIdx.x] = (p < P && j0 + j < ncls) ? __ldg(dz + (n * ncls + j0 + j) * HW + hw) : 0.f;
    }
    __syncthreads();
    for (int it0 = 0; it0 < CGS; it0 += 4) {
      uint4 raw[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const long long p = p0 + (it0 + u) * PPB + pl;
        raw[u] = (p < P) ? __ldg(reinterpret_cast<const uint4*>(a + p * a_cs + cg * 8)) : make_uint4(0, 0, 0, 0);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int lp = (it0 + u) * PPB + pl;
        float f[8];
        b2head::unpack8(raw[u], f);
#pragma unroll
        for (int j = 0; j < CHUNK; ++j) {
          const float g = dzs[j][lp];
          dbacc[j] += g;
#pragma unroll
          for (int i = 0; i < 8; ++i) dwacc[j][i] = fmaf(g, f[i], dwacc[j][i]);
        }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < CHUNK; ++j) {
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; ++i) sh[threadIdx.x][i] = dwacc[j][i];
    sh[threadIdx.x][8] = (cg == 0) ? dbacc[j] : 0.f;
    __syncthreads();
    float* dst = partial + (static_cast<size_t>(slice) * np + j0 + j) * (Cin + 1);
    for (int c = threadIdx.x; c <= Cin; c += blockDim.x) {
      float t = 0.f;
      if (c < Cin) {
        const int g = c >> 3, i = c & 7;
        for (int l = 0; l < PPB; ++l) t += sh[l * CGS + g][i];
      } else {
        for (int l = 0; l < 256; ++l) t += sh[l][8];
      }
      dst[c] = t;
    }
  }
}

// dw[j][c] / db[j] = sum over slices of the partials (fp64, slice order)
__global__ void head_many_reduce_kernel(const float* __restrict__ partial, int slices, int np, int Cin, int ncls,
                                        float* __restrict__ dw, float* __restrict__ db) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= ncls * (Cin + 1)) return;
  const size_t pitch = static_cast<size_t>(np) * (Cin + 1);
  double acc = 0.0;
  for (int r = 0; r < slices; ++r) acc += static_cast<double>(partial[r * pitch + col]);
  const int j = col / (Cin + 1), c = col % (Cin + 1);
  if (c < Cin) dw[j * Cin + c] = static_cast<float>(acc);
  else db[j] = static_cast<float>(acc);
}

int wgrad_slices(long long P, int ncls) {
  const int nchunks = pad_classes(ncls) / CHUNK;
  long long s = (P + 255) / 256, cap = (148 * 4 + nchunks - 1) / nchunks;
  if (s > cap) s = cap;
  return static_cast<int>(s < 1 ? 1 : s);
}

// warps per block of a kernel whose per-warp shared memory is a staging tile + extra bytes (at most 8, at least 1)
int many_warps(int Cin, int ncls, int extra_per_warp) {
  const int fixed = pad_classes(ncls) * (Cin + 1) * 4;
  int wv = (MAX_SMEM - fixed) / (STAGE_BYTES_PER_WARP + extra_per_warp);
  return wv > 8 ? 8 : wv;
}

template <class K>
int launch_opt_in(K* kern, unsigned long long& configured, const char* what) {
  return b2h::opt_in_smem(kern, MAX_SMEM, configured, what);
}

#define B2_MANY_ARGS(what)                                                                                               \
  B2_REQUIRE(ncls >= 1 && ncls <= MANY_MAXC, what ": n_classes=%d must be in [1,%d]", ncls, MANY_MAXC);                 \
  B2_REQUIRE(Cin == 64 || Cin == 128, what ": Cin=%d must be 64 or 128", Cin);                                           \
  B2_REQUIRE(N > 0 && H > 0 && W > 0, what ": empty input (N=%d, H=%d, W=%d)", N, H, W)

}  // namespace

extern "C" {

int b200unet_head_many_fprop(const void* a, int a_cs, const float* w, const float* bias, float* logits_nchw, int N, int H,
                             int W, int Cin, int ncls, b200_stream_t stream) {
  B2_MANY_ARGS("head_many_fprop");
  B2_REQUIRE(a && w && bias && logits_nchw, "head_many_fprop: null pointer");
  B2_REQUIRE(a_cs % 8 == 0 && a_cs >= Cin, "head_many_fprop: pixel pitch %d must be a multiple of 8 and >= Cin", a_cs);
  static unsigned long long cfg[2] = {0, 0};
  const long long P = static_cast<long long>(N) * H * W;
  long long blocks = (P + 255) / 256;
  if (blocks > MAX_BLOCKS) blocks = MAX_BLOCKS;
  const int smem = b2head::many_smem_bytes(Cin, ncls, 8);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const auto* ap = static_cast<const __nv_bfloat16*>(a);
  if (Cin == 64) {
    if (int e = launch_opt_in(head_many_fprop_kernel<1>, cfg[0], "head_many_fprop")) return e;
    head_many_fprop_kernel<1><<<static_cast<int>(blocks), 256, smem, st>>>(ap, a_cs, w, bias, logits_nchw, P,
                                                                           static_cast<long long>(H) * W, ncls);
  } else {
    if (int e = launch_opt_in(head_many_fprop_kernel<2>, cfg[1], "head_many_fprop")) return e;
    head_many_fprop_kernel<2><<<static_cast<int>(blocks), 256, smem, st>>>(ap, a_cs, w, bias, logits_nchw, P,
                                                                           static_cast<long long>(H) * W, ncls);
  }
  return b2h::check_launch("head_many_fprop");
}

int64_t b200unet_head_many_bwd_workspace_floats(int N, int H, int W, int Cin, int ncls) {
  if (ncls < 1 || ncls > MANY_MAXC || Cin < 1) return 0;
  return static_cast<int64_t>(wgrad_slices(static_cast<long long>(N) * H * W, ncls)) * pad_classes(ncls) * (Cin + 1);
}

int b200unet_head_many_bwd(const float* dz_nchw, const void* a, int a_cs, const float* w, void* da, int da_cs, float* partial,
                           float* dw, float* db, int N, int H, int W, int Cin, int ncls, b200_stream_t stream) {
  B2_MANY_ARGS("head_many_bwd");
  B2_REQUIRE(dz_nchw && a && w && da && partial && dw && db, "head_many_bwd: null pointer");
  B2_REQUIRE(a_cs % 8 == 0 && da_cs % 8 == 0 && a_cs >= Cin && da_cs >= Cin,
             "head_many_bwd: pixel pitches %d / %d must be multiples of 8 and >= Cin", a_cs, da_cs);
  static unsigned long long cfg[2] = {0, 0};
  const long long P = static_cast<long long>(N) * H * W, HW = static_cast<long long>(H) * W;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int np = pad_classes(ncls), nchunks = np / CHUNK;
  const int slices = wgrad_slices(P, ncls);
  const auto* ap = static_cast<const __nv_bfloat16*>(a);
  auto* dap = static_cast<__nv_bfloat16*>(da);
  const long long T = 2 * (256 / (Cin / 8));
  long long blocks = (P + T - 1) / T;
  if (blocks > MAX_BLOCKS) blocks = MAX_BLOCKS;
  const int smem = (np * Cin + CHUNK * static_cast<int>(T)) * 4;
  if (Cin == 64) {
    if (int e = launch_opt_in(head_many_dgrad_kernel<1>, cfg[0], "head_many_bwd")) return e;
    head_many_dgrad_kernel<1><<<static_cast<int>(blocks), 256, smem, st>>>(dz_nchw, w, dap, da_cs, P, HW, ncls);
    if (int e = b2h::check_launch("head_many_dgrad")) return e;
    head_many_wgrad_kernel<1><<<slices * nchunks, 256, 0, st>>>(dz_nchw, ap, a_cs, partial, P, HW, ncls, nchunks);
  } else {
    if (int e = launch_opt_in(head_many_dgrad_kernel<2>, cfg[1], "head_many_bwd")) return e;
    head_many_dgrad_kernel<2><<<static_cast<int>(blocks), 256, smem, st>>>(dz_nchw, w, dap, da_cs, P, HW, ncls);
    if (int e = b2h::check_launch("head_many_dgrad")) return e;
    head_many_wgrad_kernel<2><<<slices * nchunks, 256, 0, st>>>(dz_nchw, ap, a_cs, partial, P, HW, ncls, nchunks);
  }
  if (int e = b2h::check_launch("head_many_wgrad")) return e;
  const int ncols = ncls * (Cin + 1);
  head_many_reduce_kernel<<<(ncols + 127) / 128, 128, 0, st>>>(partial, slices, np, Cin, ncls, dw, db);
  return b2h::check_launch("head_many_reduce");
}

int b200unet_head_many_mask(const void* a, int a_cs, const float* w, const float* bias, uint8_t* mask, int N, int H, int W,
                            int Cin, int ncls, b200_stream_t stream) {
  B2_MANY_ARGS("head_many_mask");
  B2_REQUIRE(a && w && bias && mask, "head_many_mask: null pointer");
  B2_REQUIRE(a_cs % 8 == 0 && a_cs >= Cin, "head_many_mask: pixel pitch %d must be a multiple of 8 and >= Cin", a_cs);
  static unsigned long long cfg[2] = {0, 0};
  const int extra = pad_classes(ncls) * 32 * 4;
  const int warps = many_warps(Cin, ncls, extra);
  const int smem = pad_classes(ncls) * (Cin + 1) * 4 + warps * (STAGE_BYTES_PER_WARP + extra);
  const long long P = static_cast<long long>(N) * H * W;
  long long blocks = (P + warps * 32 - 1) / (warps * 32);
  if (blocks > MAX_BLOCKS) blocks = MAX_BLOCKS;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const auto* ap = static_cast<const __nv_bfloat16*>(a);
  if (Cin == 64) {
    if (int e = launch_opt_in(head_many_mask_kernel<1>, cfg[0], "head_many_mask")) return e;
    head_many_mask_kernel<1><<<static_cast<int>(blocks), warps * 32, smem, st>>>(ap, a_cs, w, bias, mask, P, ncls);
  } else {
    if (int e = launch_opt_in(head_many_mask_kernel<2>, cfg[1], "head_many_mask")) return e;
    head_many_mask_kernel<2><<<static_cast<int>(blocks), warps * 32, smem, st>>>(ap, a_cs, w, bias, mask, P, ncls);
  }
  return b2h::check_launch("head_many_mask");
}

int b200unet_head_many_density(const void* a, int a_cs, const float* w, const float* bias, float* out_nchw, double* counts,
                               int N, int H, int W, int Cin, int ncls, float divisor, b200_stream_t stream) {
  B2_MANY_ARGS("head_many_density");
  B2_REQUIRE(a && w && bias && out_nchw, "head_many_density: null pointer");
  B2_REQUIRE(a_cs % 8 == 0 && a_cs >= Cin, "head_many_density: pixel pitch %d must be a multiple of 8 and >= Cin", a_cs);
  static unsigned long long cfg[2] = {0, 0};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long HW = static_cast<long long>(H) * W;
  if (counts != nullptr) {
    cudaError_t e = cudaMemsetAsync(counts, 0, sizeof(double) * N * ncls, st);
    if (e != cudaSuccess) {
      b2h::set_error("head_many_density memset: %s", cudaGetErrorString(e));
      return 2;
    }
  }
  const int extra = pad_classes(ncls) * 8;
  const int warps = many_warps(Cin, ncls, extra);
  const int smem = pad_classes(ncls) * (Cin + 1) * 4 + warps * (STAGE_BYTES_PER_WARP + extra);
  long long bpi = (148 * 8 + N - 1) / N;
  const long long cap = (HW + warps * 32 - 1) / (warps * 32);
  if (bpi > cap) bpi = cap;
  const auto* ap = static_cast<const __nv_bfloat16*>(a);
  if (Cin == 64) {
    if (int e = launch_opt_in(head_many_density_kernel<1>, cfg[0], "head_many_density")) return e;
    head_many_density_kernel<1><<<static_cast<int>(N * bpi), warps * 32, smem, st>>>(ap, a_cs, w, bias, out_nchw, counts, HW,
                                                                                      static_cast<int>(bpi), ncls, divisor);
  } else {
    if (int e = launch_opt_in(head_many_density_kernel<2>, cfg[1], "head_many_density")) return e;
    head_many_density_kernel<2><<<static_cast<int>(N * bpi), warps * 32, smem, st>>>(ap, a_cs, w, bias, out_nchw, counts, HW,
                                                                                      static_cast<int>(bpi), ncls, divisor);
  }
  return b2h::check_launch("head_many_density");
}

}  // extern "C"
