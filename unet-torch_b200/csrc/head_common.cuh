// OutConv (nn.Conv2d(C, n_classes, 1), Model.py:86-92) shared by the training head (small.cu) and the fused inference
// heads (edge.cu), so that all of them produce bit-identical logits.
//
// A warp takes 32 consecutive pixels per pass. One thread per pixel reading its own 128-byte row touches 32 different
// lines per load instruction, so the rows are first STAGED through shared memory: per 64-channel chunk the warp issues 8
// fully coalesced 512-byte loads (lane l, load i -> 16-byte element i*32 + l of the 4 KB block), stores them into a
// padded [32][144 B] tile, and each lane then reads back its own pixel row (16-byte reads at a 144-byte stride are
// conflict-free) and accumulates the dot products sequentially over the channels (fixed order -> deterministic).
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

namespace b2head {

constexpr int MAXC = 8;
constexpr int ROW_WORDS = 36;                        // 128 B of bf16 + 16 B pad, in 32-bit words
constexpr int STAGE_BYTES_PER_WARP = 32 * ROW_WORDS * 4;

__host__ __device__ inline int smem_bytes(int Cin, int ncls, int warps) {
  return ((ncls * Cin * 4 + 15) / 16) * 16 + warps * STAGE_BYTES_PER_WARP;
}
__device__ __forceinline__ void load_weights(float* wsm, const float* __restrict__ w, int Cin, int ncls) {
  for (int i = threadIdx.x; i < ncls * Cin; i += blockDim.x) wsm[i] = w[i];  // [ncls][Cin]
}
// this warp's staging tile inside the dynamic shared memory that starts with the weights
__device__ __forceinline__ uint32_t* warp_stage(float* wsm, int Cin, int ncls) {
  char* base = reinterpret_cast<char*>(wsm) + ((ncls * Cin * 4 + 15) / 16) * 16;
  return reinterpret_cast<uint32_t*>(base + (threadIdx.x >> 5) * STAGE_BYTES_PER_WARP);
}

__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    f[2 * i] = __uint_as_float(w[i] << 16);
    f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
  }
}

// z[j] (j < NCLS) of pixel p0 + lane (rows >= P are read as zero: callers do not store them). The whole warp must call.
// Compiled per class count: with a run-time count the 64 x ncls FMAs per pixel carry predicates and the kernels were
// issue-bound at 35-45 % of the HBM rate.
template <int NCLS>
__device__ __forceinline__ void logits_warp32_n(const __nv_bfloat16* __restrict__ a, int a_cs, const float* wsm,
                                                uint32_t* stage, const float* __restrict__ bias, long long p0, long long P,
                                                int Cin, float (&z)[MAXC]) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int j = 0; j < MAXC; ++j) z[j] = (j < NCLS) ? __ldg(bias + j) : 0.f;
  for (int c0 = 0; c0 < Cin; c0 += 64) {
    uint4 v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {  // element e = i*32 + lane of the block: pixel e >> 3, 16-byte group e & 7
      const int e = i * 32 + lane;
      const long long p = p0 + (e >> 3);
      v[i] = (p < P) ? __ldg(reinterpret_cast<const uint4*>(a + p * a_cs + c0 + (e & 7) * 8)) : make_uint4(0, 0, 0, 0);
    }
    __syncwarp();  // the previous chunk's reads of the tile are done
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int e = i * 32 + lane;
      *reinterpret_cast<uint4*>(stage + (e >> 3) * ROW_WORDS + (e & 7) * 4) = v[i];
    }
    __syncwarp();
#pragma unroll
    for (int c8 = 0; c8 < 8; ++c8) {
      float f[8];
      unpack8(*reinterpret_cast<const uint4*>(stage + lane * ROW_WORDS + c8 * 4), f);
#pragma unroll
      for (int j = 0; j < NCLS; ++j) {
        {
          // 128-bit broadcast reads (Cin % 64 == 0 keeps every row 16-byte aligned): the scalar form issues 64 x ncls
          // shared-memory loads per pixel and is bound by the load/store pipe, not by HBM
          const float4 w0 = *reinterpret_cast<const float4*>(wsm + j * Cin + c0 + c8 * 8);
          const float4 w1 = *reinterpret_cast<const float4*>(wsm + j * Cin + c0 + c8 * 8 + 4);
          float t = z[j];
          t = fmaf(f[0], w0.x, t);
          t = fmaf(f[1], w0.y, t);
          t = fmaf(f[2], w0.z, t);
          t = fmaf(f[3], w0.w, t);
          t = fmaf(f[4], w1.x, t);
          t = fmaf(f[5], w1.y, t);
          t = fmaf(f[6], w1.z, t);
          t = fmaf(f[7], w1.w, t);
          z[j] = t;
        }
      }
    }
  }
  __syncwarp();
}

// run-time class count -> the compiled instance (warp-uniform switch, once per 32 pixels)
__device__ __forceinline__ void logits_warp32(const __nv_bfloat16* __restrict__ a, int a_cs, const float* wsm,
                                              uint32_t* stage, const float* __restrict__ bias, long long p0, long long P,
                                              int Cin, int ncls, float (&z)[MAXC]) {
  switch (ncls) {
    case 1: logits_warp32_n<1>(a, a_cs, wsm, stage, bias, p0, P, Cin, z); break;
    case 2: logits_warp32_n<2>(a, a_cs, wsm, stage, bias, p0, P, Cin, z); break;
    case 3: logits_warp32_n<3>(a, a_cs, wsm, stage, bias, p0, P, Cin, z); break;
    case 4: logits_warp32_n<4>(a, a_cs, wsm, stage, bias, p0, P, Cin, z); break;
    case 5: logits_warp32_n<5>(a, a_cs, wsm, stage, bias, p0, P, Cin, z); break;
    case 6: logits_warp32_n<6>(a, a_cs, wsm, stage, bias, p0, P, Cin, z); break;
    case 7: logits_warp32_n<7>(a, a_cs, wsm, stage, bias, p0, P, Cin, z); break;
    default: logits_warp32_n<8>(a, a_cs, wsm, stage, bias, p0, P, Cin, z); break;
  }
}

// ---- more than MAXC classes (head_many.cu). Each lane keeps its pixel's KC x 64 channels (packed bf16) in registers and
// the classes are walked in compile-time chunks of CHUNK over zero-padded weight / bias rows in shared memory, so no FMA
// carries a class predicate. Every logit is still bias, then fmaf over the channels in order: the same bits as
// logits_warp32_n at the same class count.
constexpr int CHUNK = 8;
constexpr int MANY_MAXC = 256;

__host__ __device__ inline int pad_classes(int ncls) { return (ncls + CHUNK - 1) / CHUNK * CHUNK; }
// [pad_classes][Cin] weights, [pad_classes] bias, then one staging tile per warp
__host__ __device__ inline int many_smem_bytes(int Cin, int ncls, int warps) {
  return pad_classes(ncls) * (Cin + 1) * 4 + warps * STAGE_BYTES_PER_WARP;
}
__device__ __forceinline__ void load_weights_padded(float* wsm, float* bsm, const float* __restrict__ w,
                                                    const float* __restrict__ bias, int Cin, int ncls) {
  const int np = pad_classes(ncls);
  for (int i = threadIdx.x; i < np * Cin; i += blockDim.x) wsm[i] = (i < ncls * Cin) ? w[i] : 0.f;
  for (int j = threadIdx.x; j < np; j += blockDim.x) bsm[j] = (j < ncls) ? bias[j] : 0.f;
}

// Rows p0 + lane (rows >= P read as zero) -> row[] of this lane. The whole warp must call.
template <int KC>
__device__ __forceinline__ void load_rows_warp32(const __nv_bfloat16* __restrict__ a, int a_cs, uint32_t* stage,
                                                 long long p0, long long P, uint4 (&row)[KC * 8]) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int kc = 0; kc < KC; ++kc) {
    uint4 v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int e = i * 32 + lane;
      const long long p = p0 + (e >> 3);
      v[i] = (p < P) ? __ldg(reinterpret_cast<const uint4*>(a + p * a_cs + kc * 64 + (e & 7) * 8)) : make_uint4(0, 0, 0, 0);
    }
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int e = i * 32 + lane;
      *reinterpret_cast<uint4*>(stage + (e >> 3) * ROW_WORDS + (e & 7) * 4) = v[i];
    }
    __syncwarp();
#pragma unroll
    for (int c8 = 0; c8 < 8; ++c8) row[kc * 8 + c8] = *reinterpret_cast<const uint4*>(stage + lane * ROW_WORDS + c8 * 4);
  }
  __syncwarp();
}

// z[j] = logit of class j0 + j of this lane's row, j < CHUNK (padded classes give 0)
template <int KC>
__device__ __forceinline__ void logits_chunk(const uint4 (&row)[KC * 8], const float* wsm, const float* bsm, int j0,
                                             float (&z)[CHUNK]) {
  constexpr int Cin = KC * 64;
#pragma unroll
  for (int j = 0; j < CHUNK; ++j) z[j] = bsm[j0 + j];
#pragma unroll
  for (int c8 = 0; c8 < KC * 8; ++c8) {
    float f[8];
    unpack8(row[c8], f);
#pragma unroll
    for (int j = 0; j < CHUNK; ++j) {
      const float4 w0 = *reinterpret_cast<const float4*>(wsm + (j0 + j) * Cin + c8 * 8);
      const float4 w1 = *reinterpret_cast<const float4*>(wsm + (j0 + j) * Cin + c8 * 8 + 4);
      float t = z[j];
      t = fmaf(f[0], w0.x, t);
      t = fmaf(f[1], w0.y, t);
      t = fmaf(f[2], w0.z, t);
      t = fmaf(f[3], w0.w, t);
      t = fmaf(f[4], w1.x, t);
      t = fmaf(f[5], w1.y, t);
      t = fmaf(f[6], w1.z, t);
      t = fmaf(f[7], w1.w, t);
      z[j] = t;
    }
  }
}

}  // namespace b2head
