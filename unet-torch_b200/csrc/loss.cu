// Fused loss kernels (reference loss.py:442-516 calc_loss, loss.py:215-251 DiceLoss) and the inference
// softmax -> argmax head (reference test_mc3serousv5.py:880-881). One read of logits + labels per pass,
// warp-shuffle + shared-memory block reduction, fp64 cross-block accumulation.
//   'dice_bce_mc' : L = 0.5 * CE + 0.5 * Dice,   CE = -(1/P) sum_pix log p[target]
//                   Dice = (1/C) sum_c (1 - (2 I_c + s) / (Z_c + Y_c + s)),  I = sum p_c t_c, Z = sum p_c^2,
//                   Y = sum t_c^2 over the whole batch, s = 1e-5, p = softmax(logits), t = one-hot(target).
#include "../../include/b200unet.h"
#include "host_common.h"

namespace {

constexpr int MAXC = 8;
// every accumulated scalar lives in its own 128-byte line: fp64 atomics from ~1200 blocks to the SAME line serialise
// (25 scalars in 2 lines cost ~100 us), spread over 25 lines they take a few us
constexpr int SUM_STRIDE = 16;
constexpr int SUM_SLOTS = 1 + 3 * MAXC;
constexpr int LOSS_THREADS = 256;
constexpr int LOSS_MAX_BLOCKS = 148 * 8;

template <int NV>
__device__ __forceinline__ void block_reduce_atomic(float (&v)[NV], int nv, double* dst) {
  __shared__ float sh[LOSS_THREADS / 32][NV];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    float x = v[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if (lane == 0) sh[warp][i] = x;
  }
  __syncthreads();
  if (threadIdx.x < nv) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < LOSS_THREADS / 32; ++w) t += static_cast<double>(sh[w][threadIdx.x]);
    atomicAdd(dst + threadIdx.x * SUM_STRIDE, t);
  }
}

__device__ __forceinline__ void softmax_px(const float* __restrict__ z, long long base, long long HW, int ncls,
                                           float (&p)[MAXC], float& m, float& lse) {
  float zz[MAXC];
  m = -INFINITY;
#pragma unroll
  for (int j = 0; j < MAXC; ++j)
    if (j < ncls) {
      zz[j] = __ldg(z + base + j * HW);
      m = fmaxf(m, zz[j]);
    }
  float sum = 0.f;
#pragma unroll
  for (int j = 0; j < MAXC; ++j)
    if (j < ncls) {
      p[j] = expf(zz[j] - m);
      sum += p[j];
    }
#pragma unroll
  for (int j = 0; j < MAXC; ++j)
    if (j < ncls) p[j] = p[j] / sum;
  lse = logf(sum);
}

// The training-loss kernels are compiled per class count (all loops over classes unroll, no run-time predicates) and walk
// V = 4 consecutive pixels of one image per thread with 128-bit loads / stores (V = 1 when H*W is not a multiple of 4):
// the run-time-ncls scalar version spent 130 us on 50 MB (instruction-bound); same per-pixel arithmetic, so same bits.
template <int NCLS>
__device__ __forceinline__ void softmax_n(const float (&zz)[NCLS], float (&p)[NCLS], float& m, float& lse) {
  m = -INFINITY;
#pragma unroll
  for (int j = 0; j < NCLS; ++j) m = fmaxf(m, zz[j]);
  float sum = 0.f;
#pragma unroll
  for (int j = 0; j < NCLS; ++j) {
    p[j] = expf(zz[j] - m);
    sum += p[j];
  }
#pragma unroll
  for (int j = 0; j < NCLS; ++j) p[j] = p[j] / sum;
  lse = logf(sum);
}

template <int V>
__device__ __forceinline__ void load_v(const float* __restrict__ src, float (&dst)[V]) {
  if (V == 4) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(src));
    dst[0] = t.x; dst[1] = t.y; dst[2] = t.z; dst[V - 1] = t.w;
  } else {
    dst[0] = __ldg(src);
  }
}

template <int NCLS, int V>
__global__ void __launch_bounds__(LOSS_THREADS) ce_dice_fwd_kernel(const float* __restrict__ z,
                                                                   const float* __restrict__ target,
                                                                   double* __restrict__ sums, int* __restrict__ err,
                                                                   long long groups, long long HW) {
  constexpr int NA = 1 + 3 * NCLS;
  float acc[NA];
#pragma unroll
  for (int i = 0; i < NA; ++i) acc[i] = 0.f;
  const long long HWv = HW / V;
  for (long long g = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; g < groups;
       g += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long n = g / HWv, hw = (g - n * HWv) * V;
    const long long base = n * NCLS * HW + hw;
    float zz[NCLS][V], tt[V];
#pragma unroll
    for (int j = 0; j < NCLS; ++j) load_v<V>(z + base + j * HW, zz[j]);
    load_v<V>(target + n * HW + hw, tt);
#pragma unroll
    for (int v = 0; v < V; ++v) {
      float zp[NCLS], p[NCLS], m, lse;
#pragma unroll
      for (int j = 0; j < NCLS; ++j) zp[j] = zz[j][v];
      softmax_n<NCLS>(zp, p, m, lse);
      const float t = tt[v];
      const long long ti = static_cast<long long>(t);  // .long(): truncation toward zero
      if (ti < 0 || ti >= NCLS) {
        *err = 1;
      } else {
        float zt = zp[0];
#pragma unroll
        for (int j = 1; j < NCLS; ++j) zt = (ti == j) ? zp[j] : zt;
        acc[0] += -(zt - m - lse);
      }
#pragma unroll
      for (int j = 0; j < NCLS; ++j) {
        const float oh = (t == static_cast<float>(j)) ? 1.f : 0.f;  // _one_hot_encoder: target == j
        acc[1 + j] = fmaf(p[j], oh, acc[1 + j]);
        acc[1 + NCLS + j] = fmaf(p[j], p[j], acc[1 + NCLS + j]);
        acc[1 + 2 * NCLS + j] += oh;
      }
    }
  }
  // block reduction; slot of accumulator i in the MAXC-strided sums layout [CE, I[MAXC], Z[MAXC], Y[MAXC]]
  __shared__ float sh[LOSS_THREADS / 32][NA];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < NA; ++i) {
    float x = acc[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    if (lane == 0) sh[warp][i] = x;
  }
  __syncthreads();
  if (threadIdx.x < NA) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < LOSS_THREADS / 32; ++w) t += static_cast<double>(sh[w][threadIdx.x]);
    const int i = threadIdx.x;
    const int slot = i == 0 ? 0 : 1 + ((i - 1) / NCLS) * MAXC + (i - 1) % NCLS;
    atomicAdd(sums + slot * SUM_STRIDE, t);
  }
}

// sums layout inside the kernels: [CE, I[MAXC], Z[MAXC], Y[MAXC]] (fixed MAXC stride)
__global__ void ce_dice_finalize_kernel(const double* __restrict__ sums, float* __restrict__ loss_out, double P,
                                        int ncls, int mode) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  const double ce = sums[0] / P;
  double dice = 0.0;
  const double s = 1e-5;
  for (int j = 0; j < ncls; ++j) {
    // reference arithmetic is fp32; reproduce its rounding points on the large sums
    const float I = static_cast<float>(sums[(1 + j) * SUM_STRIDE]);
    const float Z = static_cast<float>(sums[(1 + MAXC + j) * SUM_STRIDE]);
    const float Y = static_cast<float>(sums[(1 + 2 * MAXC + j) * SUM_STRIDE]);
    const float d = 1.f - (2.f * I + static_cast<float>(s)) / (Z + Y + static_cast<float>(s));
    dice += static_cast<double>(d);
  }
  dice /= ncls;
  loss_out[1] = static_cast<float>(ce);
  loss_out[2] = static_cast<float>(dice);
  loss_out[0] = (mode == 0) ? 0.5f * static_cast<float>(ce) + 0.5f * static_cast<float>(dice) : static_cast<float>(ce);
}

template <int NCLS, int V>
__global__ void __launch_bounds__(LOSS_THREADS) ce_dice_bwd_kernel(const float* __restrict__ z,
                                                                   const float* __restrict__ target,
                                                                   const double* __restrict__ sums,
                                                                   const float* __restrict__ grad_out,
                                                                   float* __restrict__ dz, long long groups, long long HW,
                                                                   long long P, int mode) {
  const float go = grad_out[0];
  const float w_ce = (mode == 0 ? 0.5f : 1.f) / static_cast<float>(P);
  const float w_dice = (mode == 0) ? 0.5f : 0.f;
  float cN[NCLS], cD[NCLS];  // g_j = a_j * t_j + b_j * p_j,  a_j = -(2/C)/D_j,  b_j = (2/C) N_j / D_j^2
#pragma unroll
  for (int j = 0; j < NCLS; ++j) {
    const double N = 2.0 * sums[(1 + j) * SUM_STRIDE] + 1e-5;
    const double D = sums[(1 + MAXC + j) * SUM_STRIDE] + sums[(1 + 2 * MAXC + j) * SUM_STRIDE] + 1e-5;
    cN[j] = static_cast<float>(-(2.0 / NCLS) / D);
    cD[j] = static_cast<float>((2.0 / NCLS) * N / (D * D));
  }
  const long long HWv = HW / V;
  for (long long gi = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; gi < groups;
       gi += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long n = gi / HWv, hw = (gi - n * HWv) * V;
    const long long base = n * NCLS * HW + hw;
    float zz[NCLS][V], tt[V], out[NCLS][V];
#pragma unroll
    for (int j = 0; j < NCLS; ++j) load_v<V>(z + base + j * HW, zz[j]);
    load_v<V>(target + n * HW + hw, tt);
#pragma unroll
    for (int v = 0; v < V; ++v) {
      float zp[NCLS], p[NCLS], m, lse;
#pragma unroll
      for (int j = 0; j < NCLS; ++j) zp[j] = zz[j][v];
      softmax_n<NCLS>(zp, p, m, lse);
      const float t = tt[v];
      const long long ti = static_cast<long long>(t);
      float g[NCLS], dot = 0.f;
#pragma unroll
      for (int j = 0; j < NCLS; ++j) {
        const float oh = (t == static_cast<float>(j)) ? 1.f : 0.f;
        g[j] = cN[j] * oh + cD[j] * p[j];
        dot = fmaf(p[j], g[j], dot);
      }
#pragma unroll
      for (int j = 0; j < NCLS; ++j) {
        const float tce = (ti == j) ? 1.f : 0.f;
        const float d = w_ce * (p[j] - tce) + w_dice * p[j] * (g[j] - dot);
        out[j][v] = go * d;
      }
    }
#pragma unroll
    for (int j = 0; j < NCLS; ++j) {
      if (V == 4)
        *reinterpret_cast<float4*>(dz + base + j * HW) = make_float4(out[j][0], out[j][1], out[j][2], out[j][V - 1]);
      else
        dz[base + j * HW] = out[j][0];
    }
  }
}

__global__ void __launch_bounds__(LOSS_THREADS) mse_fwd_kernel(const float* __restrict__ pred,
                                                               const float* __restrict__ target,
                                                               double* __restrict__ sum, long long n, int relu_input) {
  float acc[1] = {0.f};
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float p = __ldg(pred + i);
    if (relu_input) p = fmaxf(p, 0.f);
    const float d = p - __ldg(target + i);
    acc[0] = fmaf(d, d, acc[0]);
  }
  block_reduce_atomic<1>(acc, 1, sum);
}
__global__ void mse_finalize_kernel(const double* sum, float* loss_out, double n) {
  if (threadIdx.x == 0 && blockIdx.x == 0) loss_out[0] = static_cast<float>(sum[0] / n);
}
__global__ void __launch_bounds__(LOSS_THREADS) mse_bwd_kernel(const float* __restrict__ pred,
                                                               const float* __restrict__ target,
                                                               const float* __restrict__ grad_out,
                                                               float* __restrict__ dpred, long long n, int relu_input) {
  const float k = grad_out[0] * 2.f / static_cast<float>(n);
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float o = __ldg(pred + i);
    const float p = relu_input ? fmaxf(o, 0.f) : o;
    float d = k * (p - __ldg(target + i));
    if (relu_input && !(o > 0.f)) d = 0.f;
    dpred[i] = d;
  }
}

// torch.softmax(dim=1) in fp32 followed by torch.argmax(dim=1): probabilities that round to the same float tie,
// and the first maximum wins, so the softmax is reproduced rather than shortcut to argmax(logits).
__global__ void __launch_bounds__(LOSS_THREADS) softmax_argmax_kernel(const float* __restrict__ z,
                                                                      long long* __restrict__ mask, long long P,
                                                                      long long HW, int ncls) {
  for (long long px = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; px < P;
       px += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long n = px / HW, hw = px - n * HW;
    float p[MAXC], m, lse;
    softmax_px(z, n * ncls * HW + hw, HW, ncls, p, m, lse);
    int best = 0;
    float bv = p[0];
#pragma unroll
    for (int j = 1; j < MAXC; ++j)
      if (j < ncls && (p[j] > bv || (p[j] != p[j] && bv == bv))) {
        bv = p[j];
        best = j;
      }
    mask[px] = best;
  }
}

// ---------------------------------------------------------------------------------------------- more than MAXC classes
// The instances above are compiled per class count up to MAXC and stay the path there. Past it the classes are a run-time
// count walked in passes over the pixel's logits (each pass a loop unrolled by MANY_CHUNK, so no per-class predicates; the
// pixel's logits are re-read from L1): max, then sum_j expf(z_j - max), then the per-class terms. The per-class Dice sums
// cannot live in registers, so each warp folds a chunk's 3 x MANY_CHUNK values over its lanes through a transposed
// shared-memory tile into its own fp32 row [I[np], Z[np], Y[np]] in global memory (one lane per slot, so the row size does
// not bound the class count); the block adds its warps' rows in order into an fp64 row of `part` (one per block), and the
// rows are summed in block order: deterministic, no atomics.
// sums layout for ncls > MAXC: [CE, I[ncls], Z[ncls], Y[ncls]] (S = 1 + 3 ncls doubles), the backward's Dice coefficients
// [cN[ncls], cD[ncls]], then forward-only scratch: part[LOSS_MAX_BLOCKS][S] and the warps' fp32 rows
// [LOSS_MAX_BLOCKS][LOSS_THREADS / 32][3 np]. The backward reads the first many_saved(ncls) doubles only.
constexpr int MANY_CHUNK = 8;
constexpr int MANY_TILE = 3 * MANY_CHUNK * 33;  // per-warp transposed tile [3 * MANY_CHUNK][33] floats

__host__ __device__ inline int many_pad(int ncls) { return (ncls + MANY_CHUNK - 1) / MANY_CHUNK * MANY_CHUNK; }
__host__ __device__ inline int many_slots(int ncls) { return 1 + 3 * ncls; }
inline long long many_saved(int ncls) { return many_slots(ncls) + 2ll * ncls; }
// doubles taken by the warps' fp32 rows
inline long long many_warp_rows_doubles(int ncls) { return static_cast<long long>(LOSS_MAX_BLOCKS) * (LOSS_THREADS / 32) * 3 * many_pad(ncls) / 2; }

// max and sum_j expf(z_j - max) of V pixels (class stride HW)
template <int V>
__device__ __forceinline__ void softmax_stats_many(const float* __restrict__ z, long long HW, int ncls, float (&m)[V],
                                                   float (&s)[V]) {
#pragma unroll
  for (int v = 0; v < V; ++v) m[v] = -INFINITY, s[v] = 0.f;
#pragma unroll MANY_CHUNK
  for (int j = 0; j < ncls; ++j) {
    float zz[V];
    load_v<V>(z + j * HW, zz);
#pragma unroll
    for (int v = 0; v < V; ++v) m[v] = fmaxf(m[v], zz[v]);
  }
#pragma unroll MANY_CHUNK
  for (int j = 0; j < ncls; ++j) {
    float zz[V];
    load_v<V>(z + j * HW, zz);
#pragma unroll
    for (int v = 0; v < V; ++v) s[v] += expf(zz[v] - m[v]);
  }
}

// Dice terms of classes j0 .. j0 + MANY_CHUNK - 1 for V pixels, summed over V; TAIL: classes past ncls count as zero
template <int V, bool TAIL>
__device__ __forceinline__ void dice_chunk(const float* __restrict__ z, long long HW, int ncls, int j0, const float (&m)[V],
                                           const float (&inv)[V], const float (&tt)[V], bool live, float (&r)[3 * MANY_CHUNK]) {
#pragma unroll
  for (int j = 0; j < MANY_CHUNK; ++j) {
    float I = 0.f, Z = 0.f, Y = 0.f;
    if (!TAIL || j0 + j < ncls) {
      float zz[V];
      load_v<V>(z + (j0 + j) * HW, zz);
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const float p = expf(zz[v] - m[v]) * inv[v];
        const float oh = (tt[v] == static_cast<float>(j0 + j)) ? 1.f : 0.f;
        I = fmaf(p, oh, I);
        Z = fmaf(p, p, Z);
        Y += oh;
      }
    }
    r[j] = live ? I : 0.f;
    r[MANY_CHUNK + j] = live ? Z : 0.f;
    r[2 * MANY_CHUNK + j] = live ? Y : 0.f;
  }
}

template <int V>
__global__ void __launch_bounds__(LOSS_THREADS) ce_dice_fwd_many_kernel(const float* __restrict__ z,
                                                                        const float* __restrict__ target,
                                                                        double* __restrict__ part, float* __restrict__ rows,
                                                                        int* __restrict__ err, long long groups, long long HW,
                                                                        int ncls) {
  __shared__ float tiles[LOSS_THREADS / 32][MANY_TILE];
  const int np = many_pad(ncls);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* tile = tiles[warp];
  float* acc = rows + static_cast<size_t>(blockIdx.x) * (LOSS_THREADS / 32) * 3 * np;  // this block's [warps][3 np]
  float* wacc = acc + warp * 3 * np;
  for (int i = lane; i < 3 * np; i += 32) wacc[i] = 0.f;
  __syncwarp();
  float ce = 0.f;
  const long long HWv = HW / V;
  // warp-uniform trip count: every lane takes part in the transposed reductions
  for (long long g0 = static_cast<long long>(blockIdx.x) * blockDim.x + warp * 32; g0 < groups;
       g0 += static_cast<long long>(gridDim.x) * blockDim.x) {
    const bool live = g0 + lane < groups;
    const long long g = live ? g0 + lane : groups - 1;
    const long long n = g / HWv, hw = (g - n * HWv) * V;
    const float* zp = z + n * ncls * HW + hw;
    float tt[V], m[V], s[V], inv[V];
    load_v<V>(target + n * HW + hw, tt);
    softmax_stats_many<V>(zp, HW, ncls, m, s);
#pragma unroll
    for (int v = 0; v < V; ++v) {
      inv[v] = 1.f / s[v];
      const long long ti = static_cast<long long>(tt[v]);  // .long(): truncation toward zero
      if (!live) continue;
      if (ti < 0 || ti >= ncls) {
        *err = 1;
      } else {
        ce += -(__ldg(zp + ti * HW + v) - m[v] - logf(s[v]));
      }
    }
    for (int j0 = 0; j0 < ncls; j0 += MANY_CHUNK) {
      float r[3 * MANY_CHUNK];
      if (j0 + MANY_CHUNK <= ncls) dice_chunk<V, false>(zp, HW, ncls, j0, m, inv, tt, live, r);
      else dice_chunk<V, true>(zp, HW, ncls, j0, m, inv, tt, live, r);
#pragma unroll
      for (int i = 0; i < 3 * MANY_CHUNK; ++i) tile[i * 33 + lane] = r[i];
      __syncwarp();
      if (lane < 3 * MANY_CHUNK) {
        float t = 0.f;
#pragma unroll 8
        for (int l = 0; l < 32; ++l) t += tile[lane * 33 + l];
        wacc[(lane / MANY_CHUNK) * np + j0 + lane % MANY_CHUNK] += t;
      }
      __syncwarp();
    }
  }
  // block: CE through the warp tree, the class sums warp by warp in order; one fp64 row per block
  __shared__ float shce[LOSS_THREADS / 32];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ce += __shfl_xor_sync(0xffffffffu, ce, o);
  if (lane == 0) shce[warp] = ce;
  __syncthreads();
  double* row = part + static_cast<size_t>(blockIdx.x) * many_slots(ncls);
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int wv = 0; wv < LOSS_THREADS / 32; ++wv) t += static_cast<double>(shce[wv]);
    row[0] = t;
  }
  for (int i = threadIdx.x; i < 3 * ncls; i += blockDim.x) {
    const int k = i / ncls, j = i - k * ncls;
    double t = 0.0;
    for (int wv = 0; wv < LOSS_THREADS / 32; ++wv) t += static_cast<double>(acc[wv * 3 * np + k * np + j]);
    row[1 + i] = t;
  }
}

// sums[c] = sum over the blocks' rows of column c (block order), c < S
__global__ void ce_dice_rows_kernel(const double* __restrict__ part, int rows, int S, double* __restrict__ sums) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= S) return;
  double t = 0.0;
  for (int r = 0; r < rows; ++r) t += part[static_cast<size_t>(r) * S + c];
  sums[c] = t;
}

// ce_dice_finalize_kernel on the [CE, I[ncls], Z[ncls], Y[ncls]] layout; also the backward's per-class Dice coefficients
// coef = [cN[ncls], cD[ncls]] (g_j = cN_j t_j + cD_j p_j, the same arithmetic as ce_dice_bwd_kernel)
__global__ void ce_dice_finalize_many_kernel(const double* __restrict__ sums, double* __restrict__ coef,
                                             float* __restrict__ loss_out, double P, int ncls, int mode) {
  for (int j = threadIdx.x; j < ncls; j += blockDim.x) {
    const double N = 2.0 * sums[1 + j] + 1e-5;
    const double D = sums[1 + ncls + j] + sums[1 + 2 * ncls + j] + 1e-5;
    coef[j] = -(2.0 / ncls) / D;
    coef[ncls + j] = (2.0 / ncls) * N / (D * D);
  }
  if (threadIdx.x != 0) return;
  const double ce = sums[0] / P;
  double dice = 0.0;
  const double s = 1e-5;
  for (int j = 0; j < ncls; ++j) {
    const float I = static_cast<float>(sums[1 + j]);
    const float Z = static_cast<float>(sums[1 + ncls + j]);
    const float Y = static_cast<float>(sums[1 + 2 * ncls + j]);
    const float d = 1.f - (2.f * I + static_cast<float>(s)) / (Z + Y + static_cast<float>(s));
    dice += static_cast<double>(d);
  }
  dice /= ncls;
  loss_out[1] = static_cast<float>(ce);
  loss_out[2] = static_cast<float>(dice);
  loss_out[0] = (mode == 0) ? 0.5f * static_cast<float>(ce) + 0.5f * static_cast<float>(dice) : static_cast<float>(ce);
}

// ce_dice_bwd_kernel for any class count: per pixel group four passes over its logits (max, sum, dot = sum_j p_j g_j,
// store), the per-class Dice coefficients read from the forward's `sums` (the same value for every thread: L1 broadcasts).
template <int V>
__global__ void __launch_bounds__(LOSS_THREADS) ce_dice_bwd_many_kernel(const float* __restrict__ z,
                                                                        const float* __restrict__ target,
                                                                        const double* __restrict__ sums,
                                                                        const float* __restrict__ grad_out,
                                                                        float* __restrict__ dz, long long groups,
                                                                        long long HW, long long P, int ncls, int mode) {
  const double* cN = sums + many_slots(ncls);  // g_j = cN_j * t_j + cD_j * p_j
  const double* cD = cN + ncls;
  const float go = grad_out[0];
  const float w_ce = (mode == 0 ? 0.5f : 1.f) / static_cast<float>(P);
  const float w_dice = (mode == 0) ? 0.5f : 0.f;
  const long long HWv = HW / V;
  for (long long gi = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; gi < groups;
       gi += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long n = gi / HWv, hw = (gi - n * HWv) * V;
    const float* zp = z + n * ncls * HW + hw;
    float* dp = dz + n * ncls * HW + hw;
    float tt[V], m[V], s[V], inv[V], dot[V];
    load_v<V>(target + n * HW + hw, tt);
    softmax_stats_many<V>(zp, HW, ncls, m, s);
#pragma unroll
    for (int v = 0; v < V; ++v) inv[v] = 1.f / s[v], dot[v] = 0.f;
#pragma unroll MANY_CHUNK
    for (int j = 0; j < ncls; ++j) {
      float zz[V];
      load_v<V>(zp + j * HW, zz);
      const float a = static_cast<float>(__ldg(cN + j)), b = static_cast<float>(__ldg(cD + j));
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const float p = expf(zz[v] - m[v]) * inv[v];
        const float oh = (tt[v] == static_cast<float>(j)) ? 1.f : 0.f;
        dot[v] = fmaf(p, a * oh + b * p, dot[v]);
      }
    }
#pragma unroll MANY_CHUNK
    for (int j = 0; j < ncls; ++j) {
      float zz[V], out[V];
      load_v<V>(zp + j * HW, zz);
      const float a = static_cast<float>(__ldg(cN + j)), b = static_cast<float>(__ldg(cD + j));
#pragma unroll
      for (int v = 0; v < V; ++v) {
        const float p = expf(zz[v] - m[v]) * inv[v];
        const float oh = (tt[v] == static_cast<float>(j)) ? 1.f : 0.f;
        const float tce = (static_cast<long long>(tt[v]) == j) ? 1.f : 0.f;
        out[v] = go * (w_ce * (p - tce) + w_dice * p * (a * oh + b * p - dot[v]));
      }
      if (V == 4)
        *reinterpret_cast<float4*>(dp + j * HW) = make_float4(out[0], out[1], out[2], out[V - 1]);
      else
        dp[j * HW] = out[0];
    }
  }
}

// softmax_argmax_kernel for any class count: max, sum in class order, then the first maximum of expf(z_j - max) / sum
__global__ void __launch_bounds__(LOSS_THREADS) softmax_argmax_many_kernel(const float* __restrict__ z,
                                                                           long long* __restrict__ mask, long long P,
                                                                           long long HW, int ncls) {
  for (long long px = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; px < P;
       px += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long n = px / HW, hw = px - n * HW;
    const float* zp = z + n * ncls * HW + hw;
    float m[1], s[1];
    softmax_stats_many<1>(zp, HW, ncls, m, s);
    int best = 0;
    float bv = expf(__ldg(zp) - m[0]) / s[0];
#pragma unroll MANY_CHUNK
    for (int j = 1; j < ncls; ++j) {
      const float pj = expf(__ldg(zp + j * HW) - m[0]) / s[0];
      if (pj > bv || (pj != pj && bv == bv)) {
        bv = pj;
        best = j;
      }
    }
    mask[px] = best;
  }
}

int loss_blocks(long long n) {
  long long b = (n + LOSS_THREADS - 1) / LOSS_THREADS;
  if (b > LOSS_MAX_BLOCKS) b = LOSS_MAX_BLOCKS;
  return static_cast<int>(b < 1 ? 1 : b);
}

int ce_dice_fwd_many(const float* logits, const float* target, double* sums, float* loss_out, int* err_flag, long long P,
                     int ncls, long long HW, int mode, cudaStream_t st) {
  const int S = many_slots(ncls);
  double* part = sums + many_saved(ncls);
  float* rows = reinterpret_cast<float*>(part + static_cast<size_t>(LOSS_MAX_BLOCKS) * S);
  cudaMemsetAsync(err_flag, 0, sizeof(int), st);
  const bool vec = (HW % 4 == 0) && (reinterpret_cast<uintptr_t>(logits) % 16 == 0) && (reinterpret_cast<uintptr_t>(target) % 16 == 0);
  const long long groups = vec ? P / 4 : P;
  const int blocks = loss_blocks(groups);
  if (vec)
    ce_dice_fwd_many_kernel<4><<<blocks, LOSS_THREADS, 0, st>>>(logits, target, part, rows, err_flag, groups, HW, ncls);
  else
    ce_dice_fwd_many_kernel<1><<<blocks, LOSS_THREADS, 0, st>>>(logits, target, part, rows, err_flag, groups, HW, ncls);
  if (int e = b2h::check_launch("loss_ce_dice_fwd")) return e;
  ce_dice_rows_kernel<<<(S + 127) / 128, 128, 0, st>>>(part, blocks, S, sums);
  if (int e = b2h::check_launch("loss_ce_dice_rows")) return e;
  ce_dice_finalize_many_kernel<<<1, 256, 0, st>>>(sums, sums + S, loss_out, static_cast<double>(P), ncls, mode);
  return b2h::check_launch("loss_ce_dice_finalize");
}

}  // namespace

extern "C" {

// `sums` must hold b200unet_loss_sums_doubles() doubles: [CE, I[8], Z[8], Y[8]], one scalar per 128-byte line.
int b200unet_loss_sums_doubles(void) { return SUM_SLOTS * SUM_STRIDE; }

// the size for a given class count: the layout above up to 8 classes; past it the many-class layout (sums, backward
// coefficients, forward-only scratch)
int64_t b200unet_loss_sums_doubles_n(int ncls) {
  if (ncls < 1) return 0;
  if (ncls <= MAXC) return SUM_SLOTS * SUM_STRIDE;
  return many_saved(ncls) + static_cast<int64_t>(LOSS_MAX_BLOCKS) * many_slots(ncls) + many_warp_rows_doubles(ncls);
}

// the leading doubles of `sums` that the backward reads (a caller may keep only these between forward and backward)
int64_t b200unet_loss_sums_saved_doubles_n(int ncls) {
  if (ncls < 1) return 0;
  return ncls <= MAXC ? SUM_SLOTS * SUM_STRIDE : many_saved(ncls);
}

int b200unet_loss_ce_dice_fwd(const float* logits, const float* target, double* sums, float* loss_out, int* err_flag,
                              int N, int ncls, int64_t HW, int mode, b200_stream_t stream) {
  B2_REQUIRE(ncls >= 1, "loss_ce_dice_fwd: n_classes=%d must be >= 1", ncls);
  B2_REQUIRE(mode == 0 || mode == 1, "loss_ce_dice_fwd: bad mode %d", mode);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long P = static_cast<long long>(N) * HW;
  if (ncls > MAXC) return ce_dice_fwd_many(logits, target, sums, loss_out, err_flag, P, ncls, HW, mode, st);
  cudaMemsetAsync(sums, 0, sizeof(double) * SUM_SLOTS * SUM_STRIDE, st);
  cudaMemsetAsync(err_flag, 0, sizeof(int), st);
  const bool vec = (HW % 4 == 0) && (reinterpret_cast<uintptr_t>(logits) % 16 == 0) && (reinterpret_cast<uintptr_t>(target) % 16 == 0);
  const long long groups = vec ? P / 4 : P;
#define B2_CE_FWD(NC)                                                                                                  \
  case NC:                                                                                                            \
    if (vec)                                                                                                          \
      ce_dice_fwd_kernel<NC, 4><<<loss_blocks(groups), LOSS_THREADS, 0, st>>>(logits, target, sums, err_flag, groups, HW); \
    else                                                                                                              \
      ce_dice_fwd_kernel<NC, 1><<<loss_blocks(groups), LOSS_THREADS, 0, st>>>(logits, target, sums, err_flag, groups, HW); \
    break;
  switch (ncls) { B2_CE_FWD(1) B2_CE_FWD(2) B2_CE_FWD(3) B2_CE_FWD(4) B2_CE_FWD(5) B2_CE_FWD(6) B2_CE_FWD(7) B2_CE_FWD(8) }
#undef B2_CE_FWD
  if (int e = b2h::check_launch("loss_ce_dice_fwd")) return e;
  ce_dice_finalize_kernel<<<1, 32, 0, st>>>(sums, loss_out, static_cast<double>(P), ncls, mode);
  return b2h::check_launch("loss_ce_dice_finalize");
}

int b200unet_loss_ce_dice_bwd(const float* logits, const float* target, const double* sums, const float* grad_out,
                              float* dlogits, int N, int ncls, int64_t HW, int mode, b200_stream_t stream) {
  B2_REQUIRE(ncls >= 1, "loss_ce_dice_bwd: n_classes=%d must be >= 1", ncls);
  const long long P = static_cast<long long>(N) * HW;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool vec = (HW % 4 == 0) && (reinterpret_cast<uintptr_t>(logits) % 16 == 0) &&
                   (reinterpret_cast<uintptr_t>(target) % 16 == 0) && (reinterpret_cast<uintptr_t>(dlogits) % 16 == 0);
  const long long groups = vec ? P / 4 : P;
  if (ncls > MAXC) {
    if (vec)
      ce_dice_bwd_many_kernel<4><<<loss_blocks(groups), LOSS_THREADS, 0, st>>>(logits, target, sums, grad_out, dlogits,
                                                                              groups, HW, P, ncls, mode);
    else
      ce_dice_bwd_many_kernel<1><<<loss_blocks(groups), LOSS_THREADS, 0, st>>>(logits, target, sums, grad_out, dlogits,
                                                                              groups, HW, P, ncls, mode);
    return b2h::check_launch("loss_ce_dice_bwd");
  }
#define B2_CE_BWD(NC)                                                                                                   \
  case NC:                                                                                                             \
    if (vec)                                                                                                           \
      ce_dice_bwd_kernel<NC, 4><<<loss_blocks(groups), LOSS_THREADS, 0, st>>>(logits, target, sums, grad_out, dlogits,   \
                                                                              groups, HW, P, mode);                    \
    else                                                                                                               \
      ce_dice_bwd_kernel<NC, 1><<<loss_blocks(groups), LOSS_THREADS, 0, st>>>(logits, target, sums, grad_out, dlogits,   \
                                                                              groups, HW, P, mode);                    \
    break;
  switch (ncls) { B2_CE_BWD(1) B2_CE_BWD(2) B2_CE_BWD(3) B2_CE_BWD(4) B2_CE_BWD(5) B2_CE_BWD(6) B2_CE_BWD(7) B2_CE_BWD(8) }
#undef B2_CE_BWD
  return b2h::check_launch("loss_ce_dice_bwd");
}

int b200unet_mse_fwd(const float* pred, const float* target, double* sum, float* loss_out, int64_t n, int relu_input,
                     b200_stream_t stream) {
  B2_REQUIRE(n > 0, "mse_fwd: empty input");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  cudaMemsetAsync(sum, 0, sizeof(double), st);
  mse_fwd_kernel<<<loss_blocks(n), LOSS_THREADS, 0, st>>>(pred, target, sum, n, relu_input);
  if (int e = b2h::check_launch("mse_fwd")) return e;
  mse_finalize_kernel<<<1, 32, 0, st>>>(sum, loss_out, static_cast<double>(n));
  return b2h::check_launch("mse_finalize");
}

int b200unet_mse_bwd(const float* pred, const float* target, const float* grad_out, float* dpred, int64_t n,
                     int relu_input, b200_stream_t stream) {
  mse_bwd_kernel<<<loss_blocks(n), LOSS_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(pred, target, grad_out, dpred, n,
                                                                                     relu_input);
  return b2h::check_launch("mse_bwd");
}

int b200unet_softmax_argmax(const float* logits, int64_t* mask, int N, int ncls, int64_t HW, b200_stream_t stream) {
  B2_REQUIRE(ncls >= 1, "softmax_argmax: n_classes=%d must be >= 1", ncls);
  const long long P = static_cast<long long>(N) * HW;
  if (ncls > MAXC) {
    softmax_argmax_many_kernel<<<loss_blocks(P), LOSS_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
        logits, reinterpret_cast<long long*>(mask), P, HW, ncls);
    return b2h::check_launch("softmax_argmax");
  }
  softmax_argmax_kernel<<<loss_blocks(P), LOSS_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      logits, reinterpret_cast<long long*>(mask), P, HW, ncls);
  return b2h::check_launch("softmax_argmax");
}

}  // extern "C"
