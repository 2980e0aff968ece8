// Persistent tcgen05 implicit-GEMM for the 3x3 convolutions with few input channels (Cin = 64 or 128), i.e. the
// high-resolution levels of the U-Net where the reduction is short (K = 9*Cin <= 1152) and per-tile overheads and
// operand re-fetches, not arithmetic, bound a one-tile-per-CTA kernel (nn.Conv2d fprop / dgrad, reference
// Model.py:15-16,19-20: inc.conv2, down1.*, up3.conv2, up4.* and the matching backward-data passes).
//
//   * One CTA per SM, alive for the whole launch. Its BN-channel slice of the weights (all 9 taps, all of Cin:
//     <= 144 KiB of bf16) is TMA-loaded into shared memory ONCE and stays resident.
//   * Pixel tile = 16 rows x 8 columns = 128 pixels = UMMA M. Per 64-channel block ONE halo tile of 18 x 10 pixels
//     (128 B per pixel, 128B-swizzled by TMA, out-of-bounds = conv zero padding) is loaded; the 9 taps are UMMA
//     shared-memory descriptors into that tile: start = (r*10 + s) pixel rows, 8-row groups 10 pixels (1280 B) apart.
//     The tensor core applies the swizzle on absolute smem address bits, so neither the start nor the group stride
//     has to be a multiple of the 1024-byte swizzle atom (tests/test_gpu_probe.py checks this on the device).
//     => 1.4 activation tile loads per K block instead of 9 (im2col) or 3.75 (igemm.cu).
//   * Two accumulator buffers in TMEM: the MMA warp runs tile i+1 while the epilogue warps drain tile i
//     (tcgen05.ld -> bf16 -> swizzled smem staging -> TMA store) and accumulate the BatchNorm statistics
//     (Model.py:17,21) of the STORED bf16 values in registers; one partial row per CTA at the end.
#include "../../include/b200unet.h"
#include "host_common.h"
#include "first_tile.cuh"
#include "tc_common.cuh"

namespace {

using namespace b2;

constexpr int RTH = 16, RTW = 8;                      // output pixel tile
constexpr int OUT_CHUNK = 128 * 128;                  // 128 pixels x 64 channels bf16

// TAPS = 9: 3x3 conv, input tile carries a one-pixel halo. TAPS = 1: 1x1 conv (plain GEMM over pixels), used for
// inc.conv1 on its im2col'ed input (first_layer.cu).
template <int TAPS>
struct TileGeom {
  static constexpr int HALO = (TAPS == 9) ? 1 : 0;
  static constexpr int IN_H = RTH + 2 * HALO, IN_W = RTW + 2 * HALO;
  static constexpr int A_BOX_BYTES = IN_H * IN_W * 128;  // 23040 for 3x3
  static constexpr int A_STAGE = (A_BOX_BYTES + 1023) / 1024 * 1024;
};

struct ResArgs {
  CUtensorMap tmA[4];  // activations; [1..3] only for the 4-map gather (ConvTranspose2d backward-data)
  CUtensorMap tmW;
  CUtensorMap tmO[4];  // output; [1..3] only for the pixel-shuffle scatter (ConvTranspose2d forward)
  int tiles_w, tiles_h, tiles_total;
  int H, W;
  int ncols;          // GEMM N (all output columns)
  int ntiles_n;       // ncols / BN
  int workers;        // CTAs per channel slice (grid = workers * ntiles_n)
  int cup;            // UP: output channels per (i,j) sub-position
  float* stats;       // [workers][2][ncols] or null
  const float* bias;  // UP: [cup] or null
  const float* scale;  // CONV: eval-mode BatchNorm + ReLU folded into the epilogue: [ncols] each, or null
  const float* shift;
  const float* x_nchw;  // FIRST: the fp32 NCHW network input the im2col rows are built from
  // BNRED (backward-data launches whose output is the gradient g at a BatchNorm+ReLU output): the pre-BN tensor y of THAT
  // BatchNorm and its affine / statistics; `stats` then receives [workers][2][ncols] = (sum da, sum da*xhat), da = g*[bn(y) > 0]
  CUtensorMap tmY;
  const float* bn_mean;
  const float* bn_rstd;
};

// What the GEMM is:            A operand per K block                      epilogue
//   RES_CONV (TAPS 9 or 1)      tmA[0], channel block cb                   one output map, BN statistics
//   RES_UP     (TAPS 1)         tmA[0], channel block cb                   + bias, one strided output map per (i,j)
//   RES_GATHER (TAPS 1)         tmA[ij], K block kb = ij * (KB/4) + cb     one output map
//   RES_FIRST  (TAPS 1, KB 1)   im2col rows of the fp32 NCHW input built   one output map, BN statistics
//                               in shared memory by 8 builder warps (first_tile.cuh): inc.conv1 without an HBM im2col
enum { RES_CONV = 0, RES_UP = 1, RES_GATHER = 2, RES_FIRST = 3 };

// epilogue groups per CTA (see the comment at res_threads below)
constexpr int res_epi_groups(int ob) { return ob == 2 ? 2 : 1; }

template <int BN, int KB, int NA, int OB, int TAPS, int KIND = RES_CONV, bool BNRED = false>
struct ResPlan {
  static constexpr int A_STAGE = TileGeom<TAPS>::A_STAGE;
  static constexpr int W_BYTES = TAPS * KB * BN * 128;
  static constexpr int A_OFF = W_BYTES;
  static constexpr int OUT_OFF = A_OFF + NA * A_STAGE;
  static constexpr int OUT_BYTES = OB * (BN / 64) * OUT_CHUNK;
  static constexpr int Y_OFF = OUT_OFF + OUT_BYTES;                      // BNRED: one y tile per epilogue group
  static constexpr int Y_BYTES = BNRED ? 2 * (BN / 64) * OUT_CHUNK : 0;
  static constexpr int BAR_OFF = Y_OFF + Y_BYTES;
  static constexpr int TOTAL = BAR_OFF + 256 + 1024 /* alignment slack */;
  static_assert(TOTAL <= 227 * 1024, "shared memory plan exceeds 227 KiB");
  static_assert(res_epi_groups(OB) * 4 * 2 * BN * 4 <= OUT_BYTES, "final statistics reduction aliases the staging buffer");
};

// Epilogue groups. With few output channels per tile (BN = 64) the main loop of a tile is short (1x1: 4 MMAs, 3x3 over 64
// channels: 36) and ONE group of four epilogue warps (tcgen05.ld -> bf16 -> staging -> TMA store -> BatchNorm statistics,
// ~1.15 us per tile) was the bottleneck: every BN = 64 kernel ran at exactly that rate whatever its K (64->64 3x3: 1.26 us
// per tile = 54-57 % tensor pipe). Instantiations with two staging buffers (OB = 2) therefore run TWO epilogue groups that
// alternate tiles: group g drains TMEM buffer g into staging buffer g.
// warps: 0 TMA producer, 1 MMA issuer, then 4 epilogue warps per group; RES_FIRST appends two groups of four im2col builders
constexpr int res_threads(int kind, int ob) { return 64 + 128 * res_epi_groups(ob) + (kind == RES_FIRST ? 256 : 0); }

template <int BN, int KB, int NA, int OB, int TAPS, int KIND = RES_CONV, int CIN = 0, bool BNRED = false>
__global__ void __launch_bounds__(res_threads(KIND, OB), 1) conv3_res_kernel(const __grid_constant__ ResArgs args) {
  using P = ResPlan<BN, KB, NA, OB, TAPS, KIND, BNRED>;
  static_assert(!BNRED || (KIND == RES_CONV && OB == 2), "BNRED: conv epilogue with one staging buffer per epilogue group");
  static_assert(KIND != RES_FIRST || (TAPS == 1 && KB == 1 && CIN >= 1 && CIN <= 7), "RES_FIRST: one K block of im2col rows");
  static_assert(KIND == RES_CONV || TAPS == 1, "the transposed-convolution GEMMs have no spatial taps");
  static_assert(KIND != RES_GATHER || KB % 4 == 0, "gather: K blocks split evenly over the four (i,j) maps");
  using G = TileGeom<TAPS>;
  constexpr int A_STAGE = G::A_STAGE, A_BOX_BYTES = G::A_BOX_BYTES, IN_W = G::IN_W;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t sW = smem_base;
  const uint32_t sA = smem_base + P::A_OFF;
  const uint32_t sO = smem_base + P::OUT_OFF;
  const uint32_t bars = smem_base + P::BAR_OFF;
  const uint32_t W_full = bars;
  auto A_full = [&](int i) { return bars + 8u * (1 + i); };
  auto A_empty = [&](int i) { return bars + 8u * (1 + NA + i); };
  auto T_full = [&](int i) { return bars + 8u * (1 + 2 * NA + i); };
  auto T_empty = [&](int i) { return bars + 8u * (3 + 2 * NA + i); };
  const uint32_t tmem_slot = bars + 8u * (5 + 2 * NA);
  volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + P::BAR_OFF + 8 * (5 + 2 * NA));
  auto Y_full = [&](int i) { return bars + 8u * (6 + 2 * NA + i); };
  auto Y_empty = [&](int i) { return bars + 8u * (8 + 2 * NA + i); };
  const uint32_t sY = smem_base + P::Y_OFF;

  constexpr int EG = res_epi_groups(OB);
  const int warp = warp_idx_uniform();
  const int lane = threadIdx.x & 31;
  const int nt = blockIdx.x % args.ntiles_n;
  const int pw = blockIdx.x / args.ntiles_n;
  const int n0 = nt * BN;
  const int ntiles_mine = (args.tiles_total - pw + args.workers - 1) / args.workers;  // tiles pw, pw+workers, ...

  if (warp == 0 && elect_one_sync()) {
    prefetch_tmap(&args.tmA[0]);
    prefetch_tmap(&args.tmW);
    prefetch_tmap(&args.tmO[0]);
    mbar_init(W_full, 1);
    for (int i = 0; i < NA; ++i) {
      mbar_init(A_full(i), KIND == RES_FIRST ? 4 : 1);  // FIRST: one arrival per builder warp of the tile's group
      mbar_init(A_empty(i), 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(T_full(i), 1);
      mbar_init(T_empty(i), 4);  // one arrival per epilogue warp
      if (BNRED) {
        mbar_init(Y_full(i), 1);
        mbar_init(Y_empty(i), 4);
      }
    }
    if (BNRED) prefetch_tmap(&args.tmY);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 2 * BN);
  if (KIND == RES_FIRST) {  // columns >= 9*CIN of every im2col row stay zero for the whole launch
    b2first::zero_smem(sA, NA * A_STAGE, threadIdx.x, res_threads(KIND, OB));
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;

  auto tile_coords = [&](int j, int& img, int& h0, int& w0) {
    const int t = pw + j * args.workers;
    const int twi = t % args.tiles_w;
    const int thi = (t / args.tiles_w) % args.tiles_h;
    img = t / (args.tiles_w * args.tiles_h);
    h0 = thi * RTH;
    w0 = twi * RTW;
  };

  if (warp == 0) {
    // ================================================================= TMA producer
    if (elect_one_sync()) {
      mbar_arrive_expect_tx(W_full, P::W_BYTES);
#pragma unroll 1
      for (int tap = 0; tap < TAPS; ++tap)
#pragma unroll
        for (int cb = 0; cb < KB; ++cb)
          tma_load_2d(sW + (tap * KB + cb) * (BN * 128), &args.tmW, W_full, (tap * KB + cb) * 64, n0);
      int sa = 0, pa = 0;
#pragma unroll 1
      for (int j = 0; j < (KIND == RES_FIRST ? 0 : ntiles_mine); ++j) {
        int img, h0, w0;
        tile_coords(j, img, h0, w0);
#pragma unroll 1
        for (int cb = 0; cb < KB; ++cb) {
          mbar_wait(A_empty(sa), pa ^ 1);
          mbar_arrive_expect_tx(A_full(sa), A_BOX_BYTES);
          if (KIND == RES_GATHER)
            tma_load_4d(sA + sa * A_STAGE, &args.tmA[cb / (KB / 4)], A_full(sa), (cb % (KB / 4)) * 64, w0, h0, img);
          else
            tma_load_4d(sA + sa * A_STAGE, &args.tmA[0], A_full(sa), cb * 64, w0 - G::HALO, h0 - G::HALO, img);
          if (++sa == NA) { sa = 0; pa ^= 1; }
        }
        if (BNRED) {  // the consumer BatchNorm's pre-activation tile of the same pixels / channels, for the epilogue
          const int buf = j & 1;
          mbar_wait(Y_empty(buf), ((j >> 1) & 1) ^ 1);
          mbar_arrive_expect_tx(Y_full(buf), (BN / 64) * OUT_CHUNK);
#pragma unroll
          for (int q = 0; q < BN / 64; ++q)
            tma_load_4d(sY + (buf * (BN / 64) + q) * OUT_CHUNK, &args.tmY, Y_full(buf), n0 + q * 64, w0, h0, img);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ================================================================= MMA issuer
    if (elect_one_sync()) {
      constexpr uint32_t idesc = umma_idesc_bf16(128, BN, 0, 0);
      constexpr uint32_t a_hi = umma_desc_hi_sw128(IN_W * 128), b_hi = umma_desc_hi_sw128(1024);
      const uint32_t w_lo = umma_desc_lo(sW, 16);
      mbar_wait(W_full, 0);
      tc_fence_after();
      int sa = 0, pa = 0;
#pragma unroll 1
      for (int j = 0; j < ntiles_mine; ++j) {
        const int buf = j & 1;
        mbar_wait(T_empty(buf), ((j >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * BN;
        uint32_t acc = 0;
#pragma unroll(KB <= 2 ? KB : 1)
        for (int cb = 0; cb < KB; ++cb) {
          mbar_wait(A_full(sa), pa);
          tc_fence_after();
          const uint32_t a_lo = umma_desc_lo(sA + sa * A_STAGE, 16);
#pragma unroll
          for (int tap = 0; tap < TAPS; ++tap) {
            // descriptor low words step in 16-byte units: tap (r,s) = (r*10+s) pixel rows of 128 B, K step = 32 B
            const uint32_t a_tap = a_lo + ((tap / 3) * IN_W + (tap % 3)) * 8;
            const uint32_t b_tap = w_lo + (tap * KB + cb) * (BN * 8);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              umma_bf16_lh(d_tmem, a_tap + 2 * k, a_hi, b_tap + 2 * k, b_hi, idesc, acc);
              acc = 1;
            }
          }
          umma_commit(A_empty(sa));
          if (++sa == NA) { sa = 0; pa ^= 1; }
        }
        umma_commit(T_full(buf));
      }
    }
    __syncwarp();
  } else if (KIND == RES_FIRST && warp >= 2 + 4 * EG) {
    // ================================================================= im2col builders (2 groups x 4 warps)
    // Group g builds the tiles j = g, g + 2, ...: thread r of the group owns pixel row r of the 16 x 8 tile (row r >> 3,
    // column r & 7 - the order a {64, 8, 16} TMA box would have). The 9*CIN loads of a row are issued before the wait for
    // the stage, so two tiles' worth of loads are in flight per CTA.
    const int bt = threadIdx.x - 32 * (2 + 4 * EG);
    const int grp = bt >> 7, r = bt & 127;
    constexpr int CI = CIN > 0 ? CIN : 1;
#pragma unroll 1
    for (int j = grp; j < ntiles_mine; j += 2) {
      const int sa = j % NA, pa = (j / NA) & 1;
      int img, h0, w0;
      if (j + 8 < ntiles_mine) {  // pull the input lines of a tile four rounds ahead into L2
        tile_coords(j + 8, img, h0, w0);
        b2first::prefetch_tile_l2<CI, RTH, RTW>(args.x_nchw, img, h0, w0, args.H, args.W, r);
      }
      tile_coords(j, img, h0, w0);
      b2first::Row<CI> row;  // the loads are issued before the wait for the stage: two tiles' worth in flight per CTA
      b2first::load_row<CI>(args.x_nchw, img, h0 + (r >> 3), w0 + (r & 7), args.H, args.W, row);
      mbar_wait(A_empty(sa), pa ^ 1);
      b2first::store_row<CI>(sA + sa * A_STAGE, r, row);
      fence_proxy_async_smem();  // generic-proxy stores -> visible to the tensor core (async proxy)
      __syncwarp();
      if (lane == 0) mbar_arrive(A_full(sa));
    }
  } else if (warp >= 2 && warp < 2 + 4 * EG) {
    // ================================================================= epilogue (EG groups of 4 warps = 128 threads)
    const int eg = (warp - 2) >> 2;     // group: takes the tiles j = eg, eg + EG, ...
    const int quad = warp & 3;          // TMEM lanes [32*quad, 32*quad+32)
    const int row = quad * 32 + lane;   // pixel of the tile: (row >> 3, row & 7)
    const int et = (threadIdx.x - 64) & 127;  // 0..127 inside the group
    const int gbar = 1 + eg;            // named barrier of the group
    const int cp = et & 31, rq = et >> 5;  // statistics: channel pair within a 64-channel chunk, 32-row quarter
    const bool want_stats = args.stats != nullptr;
    float s1[BN / 64][2], s2[BN / 64][2];
#pragma unroll
    for (int q = 0; q < BN / 64; ++q) s1[q][0] = s1[q][1] = s2[q][0] = s2[q][1] = 0.f;
    float bsc[BN / 64][2], bsh[BN / 64][2];  // BNRED: scale / shift of this thread's channel pair
    if (BNRED) {
#pragma unroll
      for (int q = 0; q < BN / 64; ++q)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          bsc[q][e] = __ldg(args.scale + n0 + q * 64 + cp * 2 + e);
          bsh[q][e] = __ldg(args.shift + n0 + q * 64 + cp * 2 + e);
        }
    }

#pragma unroll 1
    for (int j = eg; j < ntiles_mine; j += EG) {
      const int buf = j & 1;
      const uint32_t stage = sO + (OB == 1 ? 0 : (j & 1)) * ((BN / 64) * OUT_CHUNK);
      int img, h0, w0;
      tile_coords(j, img, h0, w0);
      mbar_wait(T_full(buf), (j >> 1) & 1);
      tc_fence_after();
#pragma unroll
      for (int q = 0; q < BN / 64; ++q) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
          uint32_t v[32];
          tmem_ld32(tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + buf * BN + q * 64 + half * 32, v);
          tmem_ld_wait();
          if (!BNRED && (KIND == RES_CONV || KIND == RES_FIRST) && args.scale != nullptr)
            affine_relu32(v, args.scale + n0 + q * 64 + half * 32, args.shift + n0 + q * 64 + half * 32);
          if (KIND == RES_UP && args.bias != nullptr) {
            const float* bp = args.bias + (n0 + q * 64 + half * 32) % args.cup;
#pragma unroll
            for (int jj = 0; jj < 32; ++jj) v[jj] = __float_as_uint(__uint_as_float(v[jj]) + __ldg(bp + jj));
          }
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const uint32_t p0 = pack_bf16x2(__uint_as_float(v[8 * t + 0]), __uint_as_float(v[8 * t + 1]));
            const uint32_t p1 = pack_bf16x2(__uint_as_float(v[8 * t + 2]), __uint_as_float(v[8 * t + 3]));
            const uint32_t p2 = pack_bf16x2(__uint_as_float(v[8 * t + 4]), __uint_as_float(v[8 * t + 5]));
            const uint32_t p3 = pack_bf16x2(__uint_as_float(v[8 * t + 6]), __uint_as_float(v[8 * t + 7]));
            const uint32_t chunk = static_cast<uint32_t>(half * 4 + t) ^ (row & 7);
            const uint32_t addr = stage + q * OUT_CHUNK + row * 128 + chunk * 16;
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(p0), "r"(p1), "r"(p2), "r"(p3)
                         : "memory");
          }
        }
      }
      // accumulator buffer drained: hand it back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(T_empty(buf));
      fence_proxy_async_smem();
      asm volatile("bar.sync %0, 128;" ::"r"(gbar) : "memory");
      if (et == 0) {
#pragma unroll
        for (int q = 0; q < BN / 64; ++q) {
          if (KIND == RES_UP) {  // column block -> (i,j) sub-position -> its strided (pixel-shuffle) output map
            const int col = n0 + q * 64, ij = col / args.cup;
            tma_store_4d(&args.tmO[ij], stage + q * OUT_CHUNK, col - ij * args.cup, w0, h0, img);
          } else {
            tma_store_4d(&args.tmO[0], stage + q * OUT_CHUNK, n0 + q * 64, w0, h0, img);
          }
        }
        tma_store_commit();
      }
      if (want_stats) {
        const bool full = (h0 + RTH <= args.H) && (w0 + RTW <= args.W);
        if (BNRED) {
          mbar_wait(Y_full(buf), (j >> 1) & 1);
        }
#pragma unroll
        for (int q = 0; q < BN / 64; ++q) {
          const uint32_t base = stage + q * OUT_CHUNK + (cp & 3) * 4;
          const uint32_t ybase = sY + (buf * (BN / 64) + q) * OUT_CHUNK + (cp & 3) * 4;
#pragma unroll 8
          for (int i = 0; i < 32; ++i) {
            const int r = rq * 32 + i;
            const uint32_t off = r * 128 + ((static_cast<uint32_t>(cp >> 2) ^ (r & 7)) << 4);
            uint32_t u;
            asm volatile("ld.shared.b32 %0, [%1];" : "=r"(u) : "r"(base + off));
            float x0 = __uint_as_float(u << 16), x1 = __uint_as_float(u & 0xffff0000u);
            if (!full && !((h0 + (r >> 3) < args.H) && (w0 + (r & 7) < args.W))) x0 = x1 = 0.f;
            if (BNRED) {
              // the stored gradient g, masked by the ReLU of the consumer BatchNorm: da = g * [scale*y + shift > 0];
              // accumulates (sum da, sum da*y) - turned into (sum da, sum da*xhat) once per CTA below
              uint32_t uy;
              asm volatile("ld.shared.b32 %0, [%1];" : "=r"(uy) : "r"(ybase + off));
              const float y0 = __uint_as_float(uy << 16), y1 = __uint_as_float(uy & 0xffff0000u);
              if (!(fmaf(bsc[q][0], y0, bsh[q][0]) > 0.f)) x0 = 0.f;
              if (!(fmaf(bsc[q][1], y1, bsh[q][1]) > 0.f)) x1 = 0.f;
              s1[q][0] += x0;
              s1[q][1] += x1;
              s2[q][0] = fmaf(x0, y0, s2[q][0]);
              s2[q][1] = fmaf(x1, y1, s2[q][1]);
            } else {
              s1[q][0] += x0;
              s1[q][1] += x1;
              s2[q][0] = fmaf(x0, x0, s2[q][0]);
              s2[q][1] = fmaf(x1, x1, s2[q][1]);
            }
          }
        }
        if (BNRED) {
          __syncwarp();
          if (lane == 0) mbar_arrive(Y_empty(buf));
        }
      }
      // the group's staging buffer is free again once its store has read it (by then the statistics pass above is done too)
      if (et == 0) tma_store_wait_read0();
      asm volatile("bar.sync %0, 128;" ::"r"(gbar) : "memory");
    }
    if (EG == 2) asm volatile("bar.sync 3, 256;" ::: "memory");  // both groups' stores have read the staging buffers
    if (want_stats) {
      // cross-quarter reduction through the (now idle) staging buffer: red[rq][stat][BN]
      float* red = reinterpret_cast<float*>(smem_gen + P::OUT_OFF);
#pragma unroll
      for (int q = 0; q < BN / 64; ++q) {
        red[((eg * 4 + rq) * 2 + 0) * BN + q * 64 + cp * 2 + 0] = s1[q][0];
        red[((eg * 4 + rq) * 2 + 0) * BN + q * 64 + cp * 2 + 1] = s1[q][1];
        red[((eg * 4 + rq) * 2 + 1) * BN + q * 64 + cp * 2 + 0] = s2[q][0];
        red[((eg * 4 + rq) * 2 + 1) * BN + q * 64 + cp * 2 + 1] = s2[q][1];
      }
      if (EG == 2) asm volatile("bar.sync 3, 256;" ::: "memory");
      else asm volatile("bar.sync 1, 128;" ::: "memory");
      float* dst = args.stats + static_cast<size_t>(pw) * 2 * args.ncols + n0;
      for (int i = et + eg * 128; i < 2 * BN; i += 128 * EG) {
        const int stat = i / BN, ch = i - stat * BN;
        float t = 0.f;
#pragma unroll
        for (int part = 0; part < 4 * EG; ++part) t += red[(part * 2 + stat) * BN + ch];  // fixed order: reproducible
        if (BNRED && stat == 1) {  // sum da*y -> sum da*xhat = rstd * (sum da*y - mean * sum da)
          float t0 = 0.f;
#pragma unroll
          for (int part = 0; part < 4 * EG; ++part) t0 += red[(part * 2 + 0) * BN + ch];
          t = static_cast<float>(static_cast<double>(__ldg(args.bn_rstd + n0 + ch)) *
                                 (static_cast<double>(t) - static_cast<double>(__ldg(args.bn_mean + n0 + ch)) * static_cast<double>(t0)));
        }
        dst[stat * args.ncols + ch] = t;
      }
    }
    tc_fence_before();
  }

  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 2 * BN);
}

template <int BN, int KB, int NA, int OB, int TAPS, int KIND = RES_CONV, int CIN = 0, bool BNRED = false>
int launch_res(const ResArgs& a, cudaStream_t st) {
  using P = ResPlan<BN, KB, NA, OB, TAPS, KIND, BNRED>;
  static unsigned long long configured = 0;
  auto kern = conv3_res_kernel<BN, KB, NA, OB, TAPS, KIND, CIN, BNRED>;
  if (int e = b2h::opt_in_smem(kern, P::TOTAL, configured, "conv3_res")) return e;
  kern<<<a.workers * a.ntiles_n, res_threads(KIND, OB), P::TOTAL, st>>>(a);
  return b2h::check_launch("conv3_res");
}

// SMs the persistent grids fill
int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
  }
  return n;
}

}  // namespace

namespace b2h {

bool conv3_res_applicable(int Cin, int Cout) {
  return (Cin == 64 || Cin == 128) && Cout % 64 == 0;
}

static int res_bn(int Cin, int Cout) { return (Cin == 64 && Cout % 128 == 0) ? 128 : 64; }

// Geometry of a persistent launch over an N x H x W pixel grid with ncols GEMM columns in bn-wide channel slices (shared by
// the launchers and the statistics-row queries); one column group, every optional pointer null, tensor maps to be encoded
// by the caller.
static ResArgs res_args(int N, int H, int W, int ncols, int bn) {
  ResArgs a = {};
  a.tiles_w = ceil_div(W, RTW);
  a.tiles_h = ceil_div(H, RTH);
  a.tiles_total = N * a.tiles_w * a.tiles_h;
  a.H = H;
  a.W = W;
  a.ncols = ncols;
  a.cup = ncols;
  a.ntiles_n = ncols / bn;
  a.workers = num_sms() / a.ntiles_n;
  if (a.workers < 1) a.workers = 1;
  if (a.workers > a.tiles_total) a.workers = a.tiles_total;
  return a;
}

int conv3_res_stat_rows(int N, int H, int W, int Cin, int Cout) { return res_args(N, H, W, Cout, res_bn(Cin, Cout)).workers; }

// BatchNorm-backward reduction fused into a backward-data launch (Cin = Cout = 64: the level-0 layers, where the separate
// reduce pass reads 1.07 GB): bn_y = pre-BN tensor of the BatchNorm whose OUTPUT gradient this launch produces.
bool conv3_res_bnred_applicable(int Cin, int Cout) { return Cin == 64 && Cout == 64; }

int conv3_res_bnred_launch(const void* x, int x_cs, const void* w, void* y, int y_cs, const void* bn_y, int bn_y_cs,
                           const float* scale, const float* shift, const float* mean, const float* rstd, float* partial, int N,
                           int H, int W, int Cin, int Cout, cudaStream_t st) {
  ResArgs a = res_args(N, H, W, Cout, 64);
  a.stats = partial;
  a.scale = scale;
  a.shift = shift;
  a.bn_mean = mean;
  a.bn_rstd = rstd;
  if (int e = make_nhwc_map(&a.tmA[0], x, Cin, x_cs, N, H, W, TileGeom<9>::IN_W, TileGeom<9>::IN_H)) return e;
  if (int e = make_tmap_2d(&a.tmW, w, static_cast<uint64_t>(9) * Cin, Cout, 64)) return e;
  if (int e = make_nhwc_map(&a.tmO[0], y, Cout, y_cs, N, H, W, RTW, RTH)) return e;
  if (int e = make_nhwc_map(&a.tmY, bn_y, Cout, bn_y_cs, N, H, W, RTW, RTH)) return e;
  return launch_res<64, 1, 3, 2, 9, RES_CONV, 0, true>(a, st);
}

int conv3_res_launch(const void* x, int x_cs, const void* w, void* y, int y_cs, float* stats_partial, int N, int H,
                     int W, int Cin, int Cout, cudaStream_t st, const float* scale,
                     const float* shift) {
  const int bn = res_bn(Cin, Cout);
  ResArgs a = res_args(N, H, W, Cout, bn);
  a.stats = stats_partial;
  a.scale = scale;
  a.shift = shift;
  if (int e = make_nhwc_map(&a.tmA[0], x, Cin, x_cs, N, H, W, TileGeom<9>::IN_W, TileGeom<9>::IN_H)) return e;
  if (int e = make_tmap_2d(&a.tmW, w, static_cast<uint64_t>(9) * Cin, Cout, bn)) return e;
  if (int e = make_nhwc_map(&a.tmO[0], y, Cout, y_cs, N, H, W, RTW, RTH)) return e;
  if (Cin == 64 && bn == 64) return launch_res<64, 1, 4, 2, 9>(a, st);
  if (Cin == 64 && bn == 128) return launch_res<128, 1, 2, 1, 9>(a, st);
  return launch_res<64, 2, 2, 2, 9>(a, st);
}

// 1x1 convolution of a 64-channel NHWC tensor (the im2col'ed network input) with a [Cout][64] bf16 operand.
int conv1x1_c64_stat_rows(int N, int H, int W, int Cout) { return res_args(N, H, W, Cout, 64).workers; }

int conv1x1_c64_launch(const void* x, int x_cs, const void* w, void* y, int y_cs, float* stats_partial, int N, int H,
                       int W, int Cout, cudaStream_t st, const float* scale,
                     const float* shift) {
  ResArgs a = res_args(N, H, W, Cout, 64);
  a.stats = stats_partial;
  a.scale = scale;
  a.shift = shift;
  if (int e = make_nhwc_map(&a.tmA[0], x, 64, x_cs, N, H, W, RTW, RTH)) return e;
  if (int e = make_tmap_2d(&a.tmW, w, 64, Cout, 64)) return e;
  if (int e = make_nhwc_map(&a.tmO[0], y, Cout, y_cs, N, H, W, RTW, RTH)) return e;
  return launch_res<64, 1, 4, 2, 1>(a, st);
}

// inc.conv1 straight from the fp32 NCHW network input: the im2col rows are built in shared memory (RES_FIRST).
int conv3x3_first_launch(const float* x_nchw, const void* w1, void* y, int y_cs, float* stats_partial, int N, int H, int W,
                         int Cin, int Cout, cudaStream_t st, const float* scale, const float* shift) {
  ResArgs a = res_args(N, H, W, Cout, 64);
  a.stats = stats_partial;
  a.scale = scale;
  a.shift = shift;
  a.x_nchw = x_nchw;
  if (int e = make_tmap_2d(&a.tmW, w1, 64, Cout, 64)) return e;
  if (int e = make_nhwc_map(&a.tmO[0], y, Cout, y_cs, N, H, W, RTW, RTH)) return e;
  a.tmA[0] = a.tmO[0];  // unused by RES_FIRST (prefetch target only)
  switch (Cin) {
    case 1: return launch_res<64, 1, 4, 2, 1, RES_FIRST, 1>(a, st);
    case 2: return launch_res<64, 1, 4, 2, 1, RES_FIRST, 2>(a, st);
    case 3: return launch_res<64, 1, 4, 2, 1, RES_FIRST, 3>(a, st);
    case 4: return launch_res<64, 1, 4, 2, 1, RES_FIRST, 4>(a, st);
    case 5: return launch_res<64, 1, 4, 2, 1, RES_FIRST, 5>(a, st);
    case 6: return launch_res<64, 1, 4, 2, 1, RES_FIRST, 6>(a, st);
    case 7: return launch_res<64, 1, 4, 2, 1, RES_FIRST, 7>(a, st);
  }
  b2h::set_error("conv3x3_first: Cin=%d must be in [1,7]", Cin);
  return 1;
}

// ---- ConvTranspose2d(k2,s2) forward as a resident-weight GEMM with the pixel-shuffle scatter epilogue.
// Applicable while a BN-column slice of the [4*Cup][Cin] operand fits next to the activation ring and every CTA's
// activation re-reads stay cheap: Cin <= 512 (up2/up3/up4 of the U-Net; up1 streams through igemm.cu).
bool convt_res_applicable(int Cin, int Cup) { return (Cin == 128 || Cin == 256 || Cin == 512) && Cup == Cin / 2; }

int convt_res_fprop_launch(const void* x, int x_cs, const void* w_fprop, const float* bias, void* out, int out_cs, int N,
                           int H, int W, int Cin, int Cup, int H2, int W2, int pad_top, int pad_left, cudaStream_t st) {
  const int bn = (Cin == 128) ? 256 : 128;
  ResArgs a = res_args(N, H, W, 4 * Cup, bn);
  a.cup = Cup;
  a.bias = bias;
  if (int e = make_nhwc_map(&a.tmA[0], x, Cin, x_cs, N, H, W, RTW, RTH)) return e;
  if (int e = make_tmap_2d(&a.tmW, w_fprop, Cin, static_cast<uint64_t>(4) * Cup, bn)) return e;
  if (int e = make_pixel_shuffle_maps(a.tmO, out, Cup, out_cs, N, H, W, H2, W2, pad_top, pad_left, RTW, RTH)) return e;
  if (Cin == 128) return launch_res<256, 2, 4, 1, 1, RES_UP>(a, st);
  if (Cin == 256) return launch_res<128, 4, 4, 1, 1, RES_UP>(a, st);
  return launch_res<128, 8, 3, 1, 1, RES_UP>(a, st);
}

// ---- its backward-data: dx[p][ci] = sum_{ij,d} du[2h+i, 2w+j][d] W[ci][ij*Cup + d]; four strided gathers on the A side.
bool convt_res_dgrad_applicable(int Cin, int Cup) { return (Cin == 128 || Cin == 256) && Cup == Cin / 2; }

int convt_res_dgrad_launch(const void* du, int du_cs, const void* w_dgrad, void* dx, int dx_cs, int N, int H, int W,
                           int Cin, int Cup, int H2, int W2, int pad_top, int pad_left, cudaStream_t st) {
  ResArgs a = res_args(N, H, W, Cin, 128);
  if (int e = make_pixel_shuffle_maps(a.tmA, du, Cup, du_cs, N, H, W, H2, W2, pad_top, pad_left, RTW, RTH)) return e;
  if (int e = make_tmap_2d(&a.tmW, w_dgrad, static_cast<uint64_t>(4) * Cup, Cin, 128)) return e;
  if (int e = make_nhwc_map(&a.tmO[0], dx, Cin, dx_cs, N, H, W, RTW, RTH)) return e;
  if (Cin == 128) return launch_res<128, 4, 4, 1, 1, RES_GATHER>(a, st);
  return launch_res<128, 8, 3, 1, 1, RES_GATHER>(a, st);
}

}  // namespace b2h
