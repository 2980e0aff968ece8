// tcgen05 weight-gradient kernels: the reduction runs over PIXELS, so both operands are MN-major in smem
// (NHWC tiles: pixels are rows = K, channels contiguous = M / N).
//   KIND_CONV3  dW[k][r][s][c] = sum_{n,h,w} dy[n,h,w,k] * x[n,h+r-1,w+s-1,c]     (nn.Conv2d backward-weight)
//   KIND_UP     dW[ci][d][i][j] = sum_{n,h,w} x[n,h,w,ci] * du[n,2h+i,2w+j,d]      (nn.ConvTranspose2d k2 s2)
//   KIND_PLAIN  dW[k][j]        = sum_{n,h,w} dy[n,h,w,k] * col[n,h,w,j]            (inc.conv1 on its im2col'ed input)
//   KIND_FIRST  the same with the im2col rows col[.][c*9+r*3+s] = x[n,c,h+r-1,w+s-1] built in shared memory from the fp32
//               NCHW network input by the four (otherwise idle) epilogue warps - no im2col tensor in HBM (first_tile.cuh)
// A CTA owns a 128 (A-side channels) x BNC (B-side channels) x TAPS accumulator set in TMEM and streams a
// contiguous range of 8x16 pixel tiles through a TMA ring (split-K over pixels across CTAs). For the 3x3 case
// a CTA handles one horizontal tap s; its x tile carries two halo rows and the three vertical taps r are
// descriptor offsets of r*16 pixel rows. fp32 partials go to a workspace and a second kernel reduces the splits
// in a fixed order (deterministic) into the parameter's own layout.
#include "../../include/b200unet.h"
#include "host_common.h"
#include "first_tile.cuh"
#include "tc_common.cuh"

#include <stdlib.h>

namespace {

using namespace b2;

constexpr int TH = 8, TW = 16, BM = TH * TW;
enum { KIND_CONV3 = 0, KIND_UP = 1, KIND_PLAIN = 2, KIND_FIRST = 3 };

struct WgradArgs {
  CUtensorMap tmA;     // A-side activations (conv3: dy, up: x)
  CUtensorMap tmB[4];  // B-side (conv3: x [0]; up: du, one strided map per (i,j))
  int tiles_w, tiles_h, tiles_total;
  int mtiles, ntiles, splits;
  int Ca, Cb;          // channel counts of the A and B side
  float* partial;      // [splits][Ca][TAPS_TOTAL][Cb]
  const float* x_nchw;  // KIND_FIRST: fp32 NCHW network input
  int H, W;
};

template <int KIND, int BNC, int CIN = 0>
struct WPlan {
  static constexpr int TAPS = (KIND == KIND_CONV3) ? 3 : (KIND == KIND_UP ? 4 : 1);        // accumulators per CTA
  static constexpr int TAPS_TOTAL = (KIND == KIND_CONV3) ? 9 : (KIND == KIND_UP ? 4 : 1);  // taps in the partial layout
  static constexpr int A_BYTES = 2 * BM * 128;                     // two 64-channel boxes
  static constexpr int B_BOX = (KIND == KIND_CONV3) ? (TH + 2) * TW * 128 : BM * 128;
  static constexpr int B_BYTES = (KIND == KIND_UP ? 4 : 1) * (BNC / 64) * B_BOX;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int NS = (227 * 1024 - 2048) / STAGE_BYTES;
  static constexpr int BAR_OFF = NS * STAGE_BYTES;
  static constexpr int TOTAL = BAR_OFF + 256 + 1024;
  static constexpr int TMEM_COLS = (TAPS * BNC <= 256) ? 256 : 512;
  static_assert(TAPS * BNC <= 512, "accumulators exceed TMEM");
  static_assert(NS >= 2, "need at least a double buffer");
};

// warps: 0 TMA producer, 1 MMA issuer, 2-5 epilogue (KIND_FIRST: also im2col builders of the even tiles); KIND_FIRST adds
// warps 6-9, the builders of the odd tiles
constexpr int wgrad_threads(int kind) { return kind == 3 /* KIND_FIRST */ ? 320 : 192; }

template <int KIND, int BNC, int CIN = 0>
__global__ void __launch_bounds__(wgrad_threads(KIND), 1) wgrad_kernel(const __grid_constant__ WgradArgs args) {
  using P = WPlan<KIND, BNC>;
  static_assert(KIND != KIND_FIRST || (BNC == 64 && CIN >= 1 && CIN <= 7), "KIND_FIRST: 64 im2col columns");
  constexpr int NS = P::NS;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bars = smem_base + P::BAR_OFF;
  auto full = [&](int i) { return bars + 8u * i; };
  auto empty = [&](int i) { return bars + 8u * (NS + i); };
  const uint32_t acc_full = bars + 8u * (2 * NS);
  const uint32_t tmem_slot = acc_full + 8;
  volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + P::BAR_OFF + 8 * (2 * NS) + 8);

  const int warp = warp_idx_uniform(), lane = threadIdx.x & 31;

  // CTA -> (m tile, n tile, horizontal tap, split)
  int b = blockIdx.x;
  const int mt = b % args.mtiles; b /= args.mtiles;
  const int nt = b % args.ntiles; b /= args.ntiles;
  int s = 0;
  if (KIND == KIND_CONV3) { s = b % 3; b /= 3; }
  const int z = b;
  const int m0 = mt * 128, n0 = nt * BNC;
  const int t_begin = static_cast<int>(static_cast<long long>(args.tiles_total) * z / args.splits);
  const int t_end = static_cast<int>(static_cast<long long>(args.tiles_total) * (z + 1) / args.splits);

  if (warp == 0 && elect_one_sync()) {
    prefetch_tmap(&args.tmA);
    prefetch_tmap(&args.tmB[0]);
    for (int i = 0; i < NS; ++i) {
      mbar_init(full(i), KIND == KIND_FIRST ? 5 : 1);  // FIRST: the TMA producer + one arrival per builder warp
      mbar_init(empty(i), 1);
    }
    mbar_init(acc_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, P::TMEM_COLS);
  if (KIND == KIND_FIRST) {  // columns >= 9*CIN of the B tiles stay zero for the whole launch
    for (int i = 0; i < NS; ++i)
      b2first::zero_smem(smem_base + i * P::STAGE_BYTES + P::A_BYTES, P::B_BYTES, threadIdx.x, wgrad_threads(KIND));
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;

  if (warp == 0) {
    if (elect_one_sync()) {
      int st = 0, ph = 0;
      for (int t = t_begin; t < t_end; ++t) {
        const int twi = t % args.tiles_w;
        const int thi = (t / args.tiles_w) % args.tiles_h;
        const int img = t / (args.tiles_w * args.tiles_h);
        const int h0 = thi * TH, w0 = twi * TW;
        mbar_wait(empty(st), ph ^ 1);
        mbar_arrive_expect_tx(full(st), KIND == KIND_FIRST ? P::A_BYTES : P::STAGE_BYTES);
        const uint32_t sA = smem_base + st * P::STAGE_BYTES;
        const uint32_t sB = sA + P::A_BYTES;
        tma_load_4d(sA, &args.tmA, full(st), m0, w0, h0, img);
        tma_load_4d(sA + BM * 128, &args.tmA, full(st), m0 + 64, w0, h0, img);
        if (KIND == KIND_FIRST) {
          // B is built by warps 2-5
        } else if (KIND == KIND_CONV3) {
#pragma unroll
          for (int j = 0; j < BNC / 64; ++j)
            tma_load_4d(sB + j * P::B_BOX, &args.tmB[0], full(st), n0 + 64 * j, w0 + s - 1, h0 - 1, img);
        } else {
#pragma unroll
          for (int ij = 0; ij < P::TAPS; ++ij)
#pragma unroll
            for (int j = 0; j < BNC / 64; ++j)
              tma_load_4d(sB + (ij * (BNC / 64) + j) * P::B_BOX, &args.tmB[ij], full(st), n0 + 64 * j, w0, h0, img);
        }
        if (++st == NS) { st = 0; ph ^= 1; }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (elect_one_sync()) {
      constexpr uint32_t idesc = umma_idesc_bf16(128, BNC, 1, 1);
      constexpr uint32_t d_hi = umma_desc_hi_sw128(1024);
      int st = 0, ph = 0;
      uint32_t acc = 0;
      for (int t = t_begin; t < t_end; ++t) {
        mbar_wait(full(st), ph);
        tc_fence_after();
        const uint32_t sA = smem_base + st * P::STAGE_BYTES;
        const uint32_t sB = sA + P::A_BYTES;
#pragma unroll
        for (int k = 0; k < BM / 16; ++k) {
          const uint32_t a_lo = umma_desc_lo(sA + k * 2048, BM * 128);
#pragma unroll
          for (int tap = 0; tap < P::TAPS; ++tap) {
            uint32_t bb;
            if (KIND == KIND_CONV3) bb = sB + (k * 16 + tap * TW) * 128;
            else bb = sB + tap * (BNC / 64) * P::B_BOX + k * 2048;
            umma_bf16_lh(tmem_base + tap * BNC, a_lo, d_hi, umma_desc_lo(bb, P::B_BOX), d_hi, idesc, acc);
          }
          acc = 1;
        }
        umma_commit(empty(st));
        if (++st == NS) { st = 0; ph ^= 1; }
      }
      umma_commit(acc_full);
    }
    __syncwarp();
  } else {
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    const int ka = m0 + row;
    const bool second_builders = KIND == KIND_FIRST && warp >= 6;
    if (KIND == KIND_FIRST) {
      // im2col builders during the main loop: two groups of 128 threads alternate tiles; thread `row` of a group owns pixel
      // row `row` of its 8 x 16 tiles (tile row row >> 4, column row & 15 - the order a {64, 16, 8} TMA box would have).
      // The loads are issued before the wait for the stage.
      constexpr int CI = CIN > 0 ? CIN : 1;
      const int tiles_img = args.tiles_w * args.tiles_h;
#pragma unroll 1
      for (int i = second_builders ? 1 : 0; t_begin + i < t_end; i += 2) {
        const int t = t_begin + i, st = i % NS, ph = (i / NS) & 1;
        if (t + 8 < t_end)
          b2first::prefetch_tile_l2<CI, TH, TW>(args.x_nchw, (t + 8) / tiles_img, (((t + 8) / args.tiles_w) % args.tiles_h) * TH,
                                                ((t + 8) % args.tiles_w) * TW, args.H, args.W, row);
        b2first::Row<CI> r;
        b2first::load_row<CI>(args.x_nchw, t / tiles_img, ((t / args.tiles_w) % args.tiles_h) * TH + (row >> 4),
                              (t % args.tiles_w) * TW + (row & 15), args.H, args.W, r);
        mbar_wait(empty(st), ph ^ 1);
        b2first::store_row<CI>(smem_base + st * P::STAGE_BYTES + P::A_BYTES, row, r);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(full(st));
      }
    }
    if (!second_builders) {
    mbar_wait(acc_full, 0);
    tc_fence_after();
#pragma unroll 1
    for (int tap = 0; tap < P::TAPS; ++tap) {
      const int tapidx = (KIND == KIND_CONV3) ? tap * 3 + s : tap;
      float* dst = args.partial +
                   ((static_cast<size_t>(z) * args.Ca + ka) * P::TAPS_TOTAL + tapidx) * static_cast<size_t>(args.Cb) + n0;
#pragma unroll 1
      for (int c = 0; c < BNC / 32; ++c) {
        uint32_t v[32];
        tmem_ld32(tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + tap * BNC + c * 32, v);
        tmem_ld_wait();
        if (ka < args.Ca) {
          float4* d4 = reinterpret_cast<float4*>(dst + c * 32);
#pragma unroll
          for (int j = 0; j < 8; ++j)
            d4[j] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]),
                                __uint_as_float(v[4 * j + 3]));
        }
      }
    }
    tc_fence_before();
    }  // !second_builders
  }
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, P::TMEM_COLS);
}

// partial [Z][K][9][C] -> dw OIHW [K][C][3][3]. Block = one k x 64 channels: the 9 x 64 sums are read as nine coalesced
// 256-byte rows per split, transposed through smem and written as one contiguous 576-float run of the OIHW tensor.
__global__ void __launch_bounds__(192) reduce_conv3_kernel(const float* __restrict__ partial, float* __restrict__ dw, int Z,
                                                           int K, int C) {
  __shared__ float t[9][65];
  const int c0 = blockIdx.x * 64, k = blockIdx.y;
  const size_t total = static_cast<size_t>(K) * 9 * C;
  for (int idx = threadIdx.x; idx < 576; idx += 192) {
    const int rs = idx >> 6, cc = idx & 63;
    const float* p = partial + (static_cast<size_t>(k) * 9 + rs) * C + c0 + cc;
    float acc = 0.f;
    for (int z = 0; z < Z; ++z) acc += p[z * total];
    t[rs][cc] = acc;
  }
  __syncthreads();
  float* out = dw + (static_cast<size_t>(k) * C + c0) * 9;
  for (int idx = threadIdx.x; idx < 576; idx += 192) {
    const int cc = idx / 9, rs = idx - cc * 9;
    out[idx] = t[rs][cc];
  }
}
// partial [Z][Cin][4][Cup] -> dw [Cin][Cup][2][2]
__global__ void reduce_up_kernel(const float* __restrict__ partial, float* __restrict__ dw, int Z, int Cin, int Cup) {
  const size_t total = static_cast<size_t>(Cin) * 4 * Cup;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    float acc = 0.f;
    for (int z = 0; z < Z; ++z) acc += partial[z * total + i];
    const int d = static_cast<int>(i % Cup);
    const int ij = static_cast<int>((i / Cup) % 4);
    const size_t ci = i / (static_cast<size_t>(Cup) * 4);
    dw[(ci * Cup + d) * 4 + ij] = acc;
  }
}

// partial [Z][Ka][pitch] -> dw [K][T] (the first K <= Ka rows and T <= pitch columns are real: inc.conv1's OIHW gradient
// flattened as [k][c*9 + r*3 + s]; a 1x1 convolution whose output channels were padded to a multiple of 64)
__global__ void reduce_plain_kernel(const float* __restrict__ partial, float* __restrict__ dw, int Z, int Ka, int K, int T,
                                    int pitch) {
  const int total = K * T;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int k = i / T, j = i - k * T;
    float acc = 0.f;
    for (int z = 0; z < Z; ++z) acc += partial[(static_cast<size_t>(z) * Ka + k) * pitch + j];
    dw[i] = acc;
  }
}

// ---- weight preparation (fp32 parameter -> bf16 GEMM operands)
__global__ void prep_conv3_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ wf,
                                  __nv_bfloat16* __restrict__ wd, int K, int C) {
  const size_t total = static_cast<size_t>(K) * C * 9;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    // i indexes the fprop operand [k][rs][c]
    const int c = static_cast<int>(i % C);
    const int rs = static_cast<int>((i / C) % 9);
    const size_t k = i / (static_cast<size_t>(C) * 9);
    const __nv_bfloat16 v = __float2bfloat16_rn(w[(k * C + c) * 9 + rs]);
    if (wf) wf[i] = v;
    if (wd) wd[(static_cast<size_t>(c) * 9 + (8 - rs)) * K + k] = v;
  }
}
__global__ void prep_up_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ wf,
                               __nv_bfloat16* __restrict__ wd, int Cin, int Cup) {
  const size_t total = static_cast<size_t>(Cin) * Cup * 4;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    // i indexes the fprop operand [(ij, d)][ci]
    const int ci = static_cast<int>(i % Cin);
    const int d = static_cast<int>((i / Cin) % Cup);
    const int ij = static_cast<int>(i / (static_cast<size_t>(Cin) * Cup));
    const __nv_bfloat16 v = __float2bfloat16_rn(w[(static_cast<size_t>(ci) * Cup + d) * 4 + ij]);
    if (wf) wf[i] = v;
    if (wd) wd[static_cast<size_t>(ci) * 4 * Cup + static_cast<size_t>(ij) * Cup + d] = v;
  }
}

int conv3_bnc(int Cin) { return (Cin % 128 == 0) ? 128 : 64; }

// Split-K factor over the pixel tiles. One CTA per SM (the TMA ring takes ~200 KB), so the launch runs in
// ceil(ctas / 148) waves: pick the split whose last wave is fullest (e.g. 96 base CTAs -> z = 3 -> 288 CTAs = 1.95
// waves instead of 0.65), preferring fewer splits (less partial traffic) on ties.
int pick_splits(int base_ctas, int tiles_total) {
  const int sms = 148;
  int best_z = 1;
  double best_eff = 0.0;
  for (int z = 1; z <= tiles_total; ++z) {
    const int ctas = base_ctas * z;
    if (z > 1 && ctas > 4 * sms) break;
    const int waves = (ctas + sms - 1) / sms;
    const double eff = static_cast<double>(ctas) / (waves * sms);
    if (eff > best_eff + 0.02) {
      best_eff = eff;
      best_z = z;
    }
  }
  return best_z;
}

template <int KIND, int BNC, int CIN = 0>
int launch_wgrad(const WgradArgs& a, cudaStream_t st) {
  using P = WPlan<KIND, BNC>;
  static unsigned long long configured = 0;
  auto kern = wgrad_kernel<KIND, BNC, CIN>;
  if (int e = b2h::opt_in_smem(kern, P::TOTAL, configured, "wgrad")) return e;
  const int grid = a.mtiles * a.ntiles * (KIND == KIND_CONV3 ? 3 : 1) * a.splits;
  kern<<<grid, wgrad_threads(KIND), P::TOTAL, st>>>(a);
  return b2h::check_launch("wgrad");
}


// ---------------------------------------------------------------------------------------------------------------------
// Cout = 64 layers (inc.conv2, up4.conv1, up4.conv2 at 512^2: 20 % of the wgrad FLOPs). With dy on the M side half of
// every 128-row MMA would be idle, so the roles are swapped: M = x channels, N = the 64 dy channels.
// A CTA covers the three vertical taps of one horizontal shift s (grid x3) of its pixel tiles from ONE x tile with a full
// halo (10 rows x 18 pixels): a K step is the 16 pixels of one tile row, i.e. 16 consecutive 128-byte rows of the halo tile
// starting at pixel row (k + r) * 18 + s - any start works because the swizzle is a function of the absolute address
// (tests/test_gpu_probe.py). One x + one dy tile per 8x16 pixels instead of three of each keeps the kernel off the L2->SM
// limit it hit with one CTA per horizontal tap (ncu: 3.4x the tensor bytes, 58 % tensor-pipe active).
// CB = 2 (Cin = 128, the only instantiation): M = 128 x channels, one MMA per tap; 9 accumulators of 64 columns would need
// 576 TMEM columns, hence one s per CTA and 3 accumulators. Cin = 64 runs wgrad_swap3_kernel below.
// Partials: [z][tap][Cin][64].
template <int CB>
struct WSPlan {
  static_assert(CB == 2, "Cin = 128: two 64-channel x boxes per stage");
  static constexpr int HW_ = TW + 2;                       // halo tile width in pixels
  static constexpr int X_BOX = (TH + 2) * HW_ * 128;       // 23040
  // + two spare halo rows: not read, kept so the stage layout stays the one the kernel was measured with
  static constexpr int X_BOX_PAD = (X_BOX + 2 * HW_ * 128 + 1023) / 1024 * 1024;
  static constexpr int Y_BOX = BM * 128;                   // 16384
  static constexpr int STAGE = CB * X_BOX_PAD + Y_BOX;
  static constexpr int NS_MAX = (227 * 1024 - 2048) / STAGE;
  static constexpr int NS = NS_MAX > 5 ? 5 : NS_MAX;
  static constexpr int NACC = 3;
  static constexpr int TMEM_COLS = 256;
  static constexpr int BAR_OFF = NS * STAGE;
  static constexpr int TOTAL = BAR_OFF + 256 + 1024;
};

template <int CB>
__global__ void __launch_bounds__(192, 1) wgrad_swap_kernel(const __grid_constant__ WgradArgs args) {
  using P = WSPlan<CB>;
  constexpr int NS = P::NS, HW_ = P::HW_;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bars = smem_base + P::BAR_OFF;
  auto full = [&](int i) { return bars + 8u * i; };
  auto empty = [&](int i) { return bars + 8u * (NS + i); };
  const uint32_t acc_full = bars + 8u * (2 * NS);
  const uint32_t tmem_slot = acc_full + 8;
  volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + P::BAR_OFF + 8 * (2 * NS) + 8);
  const int warp = warp_idx_uniform(), lane = threadIdx.x & 31;
  const int s_cta = static_cast<int>(blockIdx.x % 3);
  const int z = static_cast<int>(blockIdx.x / 3);
  const int t_begin = static_cast<int>(static_cast<long long>(args.tiles_total) * z / args.splits);
  const int t_end = static_cast<int>(static_cast<long long>(args.tiles_total) * (z + 1) / args.splits);

  if (warp == 0 && elect_one_sync()) {
    prefetch_tmap(&args.tmA);
    prefetch_tmap(&args.tmB[0]);
    for (int i = 0; i < NS; ++i) {
      mbar_init(full(i), 1);
      mbar_init(empty(i), 1);
    }
    mbar_init(acc_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, P::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;

  if (warp == 0) {
    if (elect_one_sync()) {
      int st = 0, ph = 0;
      for (int t = t_begin; t < t_end; ++t) {
        const int twi = t % args.tiles_w;
        const int thi = (t / args.tiles_w) % args.tiles_h;
        const int img = t / (args.tiles_w * args.tiles_h);
        const int h0 = thi * TH, w0 = twi * TW;
        mbar_wait(empty(st), ph ^ 1);
        mbar_arrive_expect_tx(full(st), CB * P::X_BOX + P::Y_BOX);
        const uint32_t sX = smem_base + st * P::STAGE;
#pragma unroll
        for (int cb = 0; cb < CB; ++cb)
          tma_load_4d(sX + cb * P::X_BOX_PAD, &args.tmB[0], full(st), cb * 64, w0 - 1, h0 - 1, img);  // x, full halo
        tma_load_4d(sX + CB * P::X_BOX_PAD, &args.tmA, full(st), 0, w0, h0, img);                      // dy
        if (++st == NS) { st = 0; ph ^= 1; }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (elect_one_sync()) {
      constexpr uint32_t idesc = umma_idesc_bf16(128, 64, 1, 1);
      constexpr uint32_t d_hi = umma_desc_hi_sw128(1024);
      int st = 0, ph = 0;
      uint32_t acc = 0;
      for (int t = t_begin; t < t_end; ++t) {
        mbar_wait(full(st), ph);
        tc_fence_after();
        const uint32_t sX = smem_base + st * P::STAGE;
        const uint32_t sY = sX + CB * P::X_BOX_PAD;
#pragma unroll
        for (int k = 0; k < BM / 16; ++k) {  // 16 pixels (one tile row) per MMA
          const uint32_t b_lo = umma_desc_lo(sY + k * 2048, P::Y_BOX);
#pragma unroll
          for (int r = 0; r < 3; ++r)
            umma_bf16_lh(tmem_base + r * 64, umma_desc_lo(sX + ((k + r) * HW_ + s_cta) * 128, P::X_BOX_PAD), d_hi, b_lo,
                         d_hi, idesc, acc);
          acc = 1;
        }
        umma_commit(empty(st));
        if (++st == NS) { st = 0; ph ^= 1; }
      }
      umma_commit(acc_full);
    }
    __syncwarp();
  } else {
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    mbar_wait(acc_full, 0);
    tc_fence_after();
    const int Cin = args.Cb;
#pragma unroll 1
    for (int a = 0; a < P::NACC; ++a) {
      const int r = a, s = s_cta, c = row;
      float* dst = args.partial + ((static_cast<size_t>(z) * 9 + (r * 3 + s)) * Cin + c) * 64;
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        uint32_t v[32];
        tmem_ld32(tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + a * 64 + h * 32, v);
        tmem_ld_wait();
        float4* d4 = reinterpret_cast<float4*>(dst + h * 32);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          d4[j] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]),
                              __uint_as_float(v[4 * j + 3]));
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, P::TMEM_COLS);
}

// ---------------------------------------------------------------------------------------------------------------------
// Cin = Cout = 64 (inc.conv2, up4.conv2 at 512^2): the THREE HORIZONTAL TAPS STACKED ON N.
// With only the vertical taps stacked on M (a second 64-row block of the MN-major A descriptor one halo row further down),
// a 16-pixel K step is six 128x64x16 MMAs; each reads 4 KB (A) + 2 KB (B) of shared memory per 32 tensor cycles = 192 B/clk
// against the 128 B/clk the SM delivers (ncu: 51 % of the bf16 peak, tensor pipe 58 %). Here the dy operand carries a
// one-pixel horizontal halo and its MN-major descriptor takes N = 192 = three 64-channel blocks ONE PIXEL (LBO = 128 B)
// apart: block b is "dy shifted by b pixels", i.e. tap s = 2 - b, because
//     dW[k,c,r,s] = sum_q x[q + (r-1, 0), c] * dy[q + (0, 1-s), k]          (the sum re-indexed by the x pixel q).
// With the two vertical taps stacked on M as before (LBO = one x row = 2048 B) a K step is TWO 128x192x16 MMAs (taps
// (0..1, 0..2) and (2..3, 0..2), r = 3 discarded): 4 KB + 6 KB per 96 cycles = 107 B/clk - no longer bound by shared memory.
// x tile: {64 ch, 16, 8 + 2 rows} (vertical halo only); dy tile: {64 ch, 16 + 2, 8}. Partials as wgrad_swap_kernel.
struct WS3Plan {
  static constexpr int X_BOX = (TH + 2) * TW * 128;                       // 20480
  static constexpr int X_PAD = ((TH + 3) * TW * 128 + 1023) / 1024 * 1024;  // + the junk row tap r = 3 touches
  static constexpr int Y_BOX = TH * (TW + 2) * 128;                       // 18432
  static constexpr int Y_PAD = (Y_BOX + 2 * 128 + 1023) / 1024 * 1024;    // + the two pixels block b = 2 reads past the last row
  static constexpr int STAGE = X_PAD + Y_PAD;
  static constexpr int NS_MAX = (227 * 1024 - 2048) / STAGE;
  static constexpr int NS = NS_MAX > 5 ? 5 : NS_MAX;
  static constexpr int BAR_OFF = NS * STAGE;
  static constexpr int TOTAL = BAR_OFF + 256 + 1024;
};

__global__ void __launch_bounds__(192, 1) wgrad_swap3_kernel(const __grid_constant__ WgradArgs args) {
  using P = WS3Plan;
  constexpr int NS = P::NS;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bars = smem_base + P::BAR_OFF;
  auto full = [&](int i) { return bars + 8u * i; };
  auto empty = [&](int i) { return bars + 8u * (NS + i); };
  const uint32_t acc_full = bars + 8u * (2 * NS);
  const uint32_t tmem_slot = acc_full + 8;
  volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + P::BAR_OFF + 8 * (2 * NS) + 8);
  const int warp = warp_idx_uniform(), lane = threadIdx.x & 31;
  const int z = static_cast<int>(blockIdx.x);
  const int t_begin = static_cast<int>(static_cast<long long>(args.tiles_total) * z / args.splits);
  const int t_end = static_cast<int>(static_cast<long long>(args.tiles_total) * (z + 1) / args.splits);

  if (warp == 0 && elect_one_sync()) {
    prefetch_tmap(&args.tmA);
    prefetch_tmap(&args.tmB[0]);
    for (int i = 0; i < NS; ++i) {
      mbar_init(full(i), 1);
      mbar_init(empty(i), 1);
    }
    mbar_init(acc_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;

  if (warp == 0) {
    if (elect_one_sync()) {
      int st = 0, ph = 0;
      for (int t = t_begin; t < t_end; ++t) {
        const int twi = t % args.tiles_w;
        const int thi = (t / args.tiles_w) % args.tiles_h;
        const int img = t / (args.tiles_w * args.tiles_h);
        const int h0 = thi * TH, w0 = twi * TW;
        mbar_wait(empty(st), ph ^ 1);
        mbar_arrive_expect_tx(full(st), P::X_BOX + P::Y_BOX);
        const uint32_t sX = smem_base + st * P::STAGE;
        tma_load_4d(sX, &args.tmB[0], full(st), 0, w0, h0 - 1, img);            // x, vertical halo
        tma_load_4d(sX + P::X_PAD, &args.tmA, full(st), 0, w0 - 1, h0, img);    // dy, horizontal halo
        if (++st == NS) { st = 0; ph ^= 1; }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (elect_one_sync()) {
      constexpr uint32_t idesc = umma_idesc_bf16(128, 192, 1, 1);
      constexpr uint32_t d_hi = umma_desc_hi_sw128(1024);
      int st = 0, ph = 0;
      uint32_t acc = 0;
      for (int t = t_begin; t < t_end; ++t) {
        mbar_wait(full(st), ph);
        tc_fence_after();
        const uint32_t sX = smem_base + st * P::STAGE;
        const uint32_t sY = sX + P::X_PAD;
#pragma unroll
        for (int k = 0; k < TH; ++k) {  // one tile row = 16 x pixels per K step
          // B: dy pixels (k, j + b), b = 0..2 <-> tap s = 2 - b; consecutive blocks one pixel (128 B) apart
          const uint32_t b_lo = umma_desc_lo(sY + (k * (TW + 2)) * 128, 128);
#pragma unroll
          for (int pr = 0; pr < 2; ++pr)  // A: x rows (k + 2 pr) and (k + 2 pr + 1) of the vertical-halo tile, 64 channels each
            umma_bf16_lh(tmem_base + pr * 192, umma_desc_lo(sX + ((k + 2 * pr) * TW) * 128, TW * 128), d_hi, b_lo, d_hi, idesc, acc);
          acc = 1;
        }
        umma_commit(empty(st));
        if (++st == NS) { st = 0; ph ^= 1; }
      }
      umma_commit(acc_full);
    }
    __syncwarp();
  } else {
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    mbar_wait(acc_full, 0);
    tc_fence_after();
    const int Cin = args.Cb;
#pragma unroll 1
    for (int a = 0; a < 6; ++a) {
      const int pr = a / 3, b = a - pr * 3;
      const int r = 2 * pr + (row >> 6), s = 2 - b, c = row & 63;
      float* dst = args.partial + ((static_cast<size_t>(z) * 9 + (r * 3 + s)) * Cin + c) * 64;
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        uint32_t v[32];
        tmem_ld32(tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + pr * 192 + b * 64 + h * 32, v);
        tmem_ld_wait();
        if (r < 3) {
          float4* d4 = reinterpret_cast<float4*>(dst + h * 32);
#pragma unroll
          for (int j = 0; j < 8; ++j)
            d4[j] = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]),
                                __uint_as_float(v[4 * j + 3]));
        }
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

int launch_wgrad_swap3(const WgradArgs& a, cudaStream_t st) {
  static unsigned long long configured = 0;
  if (int e = b2h::opt_in_smem(wgrad_swap3_kernel, WS3Plan::TOTAL, configured, "wgrad_swap3")) return e;
  wgrad_swap3_kernel<<<a.splits, 192, WS3Plan::TOTAL, st>>>(a);
  return b2h::check_launch("wgrad_swap3");
}

// partial [Z][9][C][64] -> dw OIHW [64][C][3][3]
__global__ void reduce_conv3_swapped_kernel(const float* __restrict__ partial, float* __restrict__ dw, int Z, int C) {
  const int total = 9 * C * 64;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    float acc = 0.f;
    for (int z = 0; z < Z; ++z) acc += partial[static_cast<size_t>(z) * total + i];
    const int k = i & 63, c = (i >> 6) % C, rs = i / (64 * C);
    dw[(static_cast<size_t>(k) * C + c) * 9 + rs] = acc;
  }
}

int launch_wgrad_swap(const WgradArgs& a, cudaStream_t st) {
  using P = WSPlan<2>;
  static unsigned long long configured = 0;
  if (int e = b2h::opt_in_smem(wgrad_swap_kernel<2>, P::TOTAL, configured, "wgrad_swap")) return e;
  wgrad_swap_kernel<2><<<3 * a.splits, 192, P::TOTAL, st>>>(a);
  return b2h::check_launch("wgrad_swap");
}

bool use_swap(int Cin, int Cout) {
  static int off = -1;
  if (off < 0) {
    const char* e = getenv("B200UNET_NO_WGRAD_SWAP");
    off = (e && atoi(e) != 0) ? 1 : 0;
  }
  return !off && Cout == 64 && (Cin == 64 || Cin == 128);
}

// Pixel-tile fields and CTA grid of wgrad_kernel<KIND_UP / KIND_PLAIN / KIND_FIRST, 64> over N x H x W: 128 A-side x 64
// B-side channels per CTA, split over the pixel tiles; every optional pointer null, tensor maps to be encoded by the caller.
WgradArgs wgrad_args(int N, int H, int W, int Ca, int Cb, float* partial) {
  WgradArgs a = {};
  a.tiles_w = b2h::ceil_div(W, TW);
  a.tiles_h = b2h::ceil_div(H, TH);
  a.tiles_total = N * a.tiles_w * a.tiles_h;
  a.mtiles = b2h::ceil_div(Ca, 128);
  a.ntiles = Cb / 64;
  a.splits = pick_splits(a.mtiles * a.ntiles, a.tiles_total);
  a.Ca = Ca;
  a.Cb = Cb;
  a.partial = partial;
  a.H = H;
  a.W = W;
  return a;
}

// the 3x3 weight gradient: A = dy (Cout), B = x (Cin). wgrad_kernel and wgrad_swap_kernel run one horizontal tap per CTA
// (grid x3), wgrad_swap3_kernel all nine
WgradArgs conv3_wgrad_args(int N, int H, int W, int Cin, int Cout, float* partial) {
  WgradArgs a = wgrad_args(N, H, W, Cout, Cin, partial);
  if (use_swap(Cin, Cout)) {
    a.mtiles = 1;
    a.ntiles = 1;
    a.splits = pick_splits(Cin == 64 ? 1 : 3, a.tiles_total);
  } else {
    a.ntiles = Cin / conv3_bnc(Cin);
    a.splits = pick_splits(a.mtiles * a.ntiles * 3, a.tiles_total);
  }
  return a;
}

}  // namespace

extern "C" {

int b200unet_prep_conv3x3_weight(const float* w_oihw, void* w_fprop, void* w_dgrad, int K, int C, b200_stream_t stream) {
  const size_t total = static_cast<size_t>(K) * C * 9;
  const int blocks = static_cast<int>((total + 255) / 256 < 148 * 8 ? (total + 255) / 256 : 148 * 8);
  prep_conv3_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      w_oihw, static_cast<__nv_bfloat16*>(w_fprop), static_cast<__nv_bfloat16*>(w_dgrad), K, C);
  return b2h::check_launch("prep_conv3x3_weight");
}

int b200unet_prep_convt2x2_weight(const float* w, void* w_fprop, void* w_dgrad, int Cin, int Cup, b200_stream_t stream) {
  const size_t total = static_cast<size_t>(Cin) * Cup * 4;
  const int blocks = static_cast<int>((total + 255) / 256 < 148 * 8 ? (total + 255) / 256 : 148 * 8);
  prep_up_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(
      w, static_cast<__nv_bfloat16*>(w_fprop), static_cast<__nv_bfloat16*>(w_dgrad), Cin, Cup);
  return b2h::check_launch("prep_convt2x2_weight");
}

int64_t b200unet_conv3x3_wgrad_workspace_floats(int N, int H, int W, int Cin, int Cout) {
  return static_cast<int64_t>(conv3_wgrad_args(N, H, W, Cin, Cout, nullptr).splits) * Cout * 9 * Cin;
}

int b200unet_conv3x3_wgrad(const void* x, int x_cs, const void* dy, int dy_cs, float* partial, float* dw_oihw, int N,
                           int H, int W, int Cin, int Cout, b200_stream_t stream) {
  B2_REQUIRE(Cin % 64 == 0 && Cout % 64 == 0, "conv3x3_wgrad: Cin (%d) and Cout (%d) must be multiples of 64", Cin, Cout);
  B2_REQUIRE(x_cs % 8 == 0 && dy_cs % 8 == 0, "conv3x3_wgrad: pitches must be multiples of 8");
  WgradArgs a = conv3_wgrad_args(N, H, W, Cin, Cout, partial);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool swap = use_swap(Cin, Cout), swap3 = swap && Cin == 64;
  // halos: x vertical (split-tap kernel, swap3) or full (swap); dy none, or horizontal for swap3 (taps stacked on N)
  if (int e = b2h::make_nhwc_map(&a.tmA, dy, Cout, dy_cs, N, H, W, swap3 ? TW + 2 : TW, TH)) return e;
  if (int e = b2h::make_nhwc_map(&a.tmB[0], x, Cin, x_cs, N, H, W, swap && !swap3 ? TW + 2 : TW, TH + 2)) return e;
  if (swap) {
    if (int e = swap3 ? launch_wgrad_swap3(a, st) : launch_wgrad_swap(a, st)) return e;
    reduce_conv3_swapped_kernel<<<b2h::ceil_div(9 * Cin * 64, 256), 256, 0, st>>>(partial, dw_oihw, a.splits, Cin);
    return b2h::check_launch("conv3x3_wgrad_reduce");
  }
  int e = (conv3_bnc(Cin) == 128) ? launch_wgrad<KIND_CONV3, 128>(a, st) : launch_wgrad<KIND_CONV3, 64>(a, st);
  if (e) return e;
  reduce_conv3_kernel<<<dim3(Cin / 64, Cout), 192, 0, st>>>(partial, dw_oihw, a.splits, Cout, Cin);
  return b2h::check_launch("conv3x3_wgrad_reduce");
}

int64_t b200unet_convt2x2_wgrad_workspace_floats(int N, int H, int W, int Cin, int Cup) {
  return static_cast<int64_t>(wgrad_args(N, H, W, Cin, Cup, nullptr).splits) * Cin * 4 * Cup;
}

int b200unet_convt2x2_wgrad(const void* x, int x_cs, const void* du, int du_cs, float* partial, float* dw, int N, int H,
                            int W, int Cin, int Cup, int H2, int W2, int pad_top, int pad_left, b200_stream_t stream) {
  B2_REQUIRE(Cin % 64 == 0 && Cup % 64 == 0, "convt2x2_wgrad: Cin (%d) and Cup (%d) must be multiples of 64", Cin, Cup);
  B2_REQUIRE(pad_top >= 0 && pad_left >= 0 && 2 * H + pad_top <= H2 && 2 * W + pad_left <= W2, "convt2x2_wgrad: bad canvas");
  B2_REQUIRE(x_cs % 8 == 0 && du_cs % 8 == 0, "convt2x2_wgrad: pitches must be multiples of 8");
  WgradArgs a = wgrad_args(N, H, W, Cin, Cup, partial);
  if (int e = b2h::make_nhwc_map(&a.tmA, x, Cin, x_cs, N, H, W, TW, TH)) return e;
  if (int e = b2h::make_pixel_shuffle_maps(a.tmB, du, Cup, du_cs, N, H, W, H2, W2, pad_top, pad_left, TW, TH)) return e;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int e = launch_wgrad<KIND_UP, 64>(a, st)) return e;
  const size_t total = static_cast<size_t>(Cin) * 4 * Cup;
  const int blocks = static_cast<int>((total + 255) / 256 < 148 * 8 ? (total + 255) / 256 : 148 * 8);
  reduce_up_kernel<<<blocks, 256, 0, st>>>(partial, dw, a.splits, Cin, Cup);
  return b2h::check_launch("convt2x2_wgrad_reduce");
}

int64_t b200unet_conv1x1_c64_wgrad_workspace_floats(int N, int H, int W, int Cout) {
  return static_cast<int64_t>(wgrad_args(N, H, W, Cout, 64, nullptr).splits) * Cout * 64;
}

int b200unet_conv1x1_c64_wgrad(const void* col, int col_cs, const void* dy, int dy_cs, float* partial, float* dw, int N,
                               int H, int W, int T, int Cout, b200_stream_t stream) {
  B2_REQUIRE(Cout % 64 == 0 && T >= 1 && T <= 64, "conv1x1_c64_wgrad: Cout=%d must be a multiple of 64 and T=%d in [1,64]", Cout, T);
  B2_REQUIRE(col_cs % 8 == 0 && dy_cs % 8 == 0 && col_cs >= 64, "conv1x1_c64_wgrad: bad pitches");
  WgradArgs a = wgrad_args(N, H, W, Cout, 64, partial);
  if (int e = b2h::make_nhwc_map(&a.tmA, dy, Cout, dy_cs, N, H, W, TW, TH)) return e;
  if (int e = b2h::make_nhwc_map(&a.tmB[0], col, 64, col_cs, N, H, W, TW, TH)) return e;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int e = launch_wgrad<KIND_PLAIN, 64>(a, st)) return e;
  reduce_plain_kernel<<<b2h::ceil_div(Cout * T, 256), 256, 0, st>>>(partial, dw, a.splits, Cout, Cout, T, 64);
  return b2h::check_launch("conv1x1_c64_wgrad_reduce");
}

int64_t b200unet_conv1x1_wgrad_workspace_floats(int N, int H, int W, int Cin, int Cout) {
  return static_cast<int64_t>(wgrad_args(N, H, W, Cout, Cin, nullptr).splits) * Cout * Cin;
}

int b200unet_conv1x1_wgrad(const void* x, int x_cs, const void* dy, int dy_cs, float* partial, float* dw, int N, int H, int W,
                           int Cin, int Cout, int Cout_real, b200_stream_t stream) {
  B2_REQUIRE(x && dy && partial && dw, "conv1x1_wgrad: null argument");
  B2_REQUIRE(Cin % 64 == 0 && Cout % 64 == 0 && Cout_real >= 1 && Cout_real <= Cout,
             "conv1x1_wgrad: Cin=%d and Cout=%d must be multiples of 64, Cout_real=%d in [1, Cout]", Cin, Cout, Cout_real);
  B2_REQUIRE(x_cs % 8 == 0 && dy_cs % 8 == 0 && x_cs >= Cin && dy_cs >= Cout, "conv1x1_wgrad: bad pitches");
  WgradArgs a = wgrad_args(N, H, W, Cout, Cin, partial);
  if (int e = b2h::make_nhwc_map(&a.tmA, dy, Cout, dy_cs, N, H, W, TW, TH)) return e;
  if (int e = b2h::make_nhwc_map(&a.tmB[0], x, Cin, x_cs, N, H, W, TW, TH)) return e;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (int e = launch_wgrad<KIND_PLAIN, 64>(a, st)) return e;
  const int total = Cout_real * Cin;
  reduce_plain_kernel<<<b2h::ceil_div(total, 256) < 148 * 8 ? b2h::ceil_div(total, 256) : 148 * 8, 256, 0, st>>>(
      partial, dw, a.splits, Cout, Cout_real, Cin, Cin);
  return b2h::check_launch("conv1x1_wgrad_reduce");
}

int64_t b200unet_conv3x3_first_tc_wgrad_workspace_floats(int N, int H, int W, int Cout) {
  return b200unet_conv1x1_c64_wgrad_workspace_floats(N, H, W, Cout);
}

int b200unet_conv3x3_first_tc_wgrad(const float* x_nchw, const void* dy, int dy_cs, float* partial, float* dw_oihw, int N, int H,
                                    int W, int Cin, int Cout, b200_stream_t stream) {
  B2_REQUIRE(Cin >= 1 && Cin <= 7 && Cout % 64 == 0 && Cout > 0, "conv3x3_first_tc_wgrad: Cin=%d must be in [1,7], Cout=%d a multiple of 64", Cin, Cout);
  B2_REQUIRE(x_nchw && dy && partial && dw_oihw && dy_cs % 8 == 0 && dy_cs >= Cout, "conv3x3_first_tc_wgrad: bad arguments");
  WgradArgs a = wgrad_args(N, H, W, Cout, 64, partial);
  a.x_nchw = x_nchw;
  if (int e = b2h::make_nhwc_map(&a.tmA, dy, Cout, dy_cs, N, H, W, TW, TH)) return e;
  a.tmB[0] = a.tmA;  // unused (prefetch target only)
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int e = 1;
  switch (Cin) {
    case 1: e = launch_wgrad<KIND_FIRST, 64, 1>(a, st); break;
    case 2: e = launch_wgrad<KIND_FIRST, 64, 2>(a, st); break;
    case 3: e = launch_wgrad<KIND_FIRST, 64, 3>(a, st); break;
    case 4: e = launch_wgrad<KIND_FIRST, 64, 4>(a, st); break;
    case 5: e = launch_wgrad<KIND_FIRST, 64, 5>(a, st); break;
    case 6: e = launch_wgrad<KIND_FIRST, 64, 6>(a, st); break;
    case 7: e = launch_wgrad<KIND_FIRST, 64, 7>(a, st); break;
  }
  if (e) return e;
  const int T = Cin * 9;
  reduce_plain_kernel<<<b2h::ceil_div(Cout * T, 256), 256, 0, st>>>(partial, dw_oihw, a.splits, Cout, Cout, T, 64);
  return b2h::check_launch("conv3x3_first_tc_wgrad_reduce");
}

}  // extern "C"
