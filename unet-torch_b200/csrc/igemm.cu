// tcgen05 implicit-GEMM kernel for the dense contractions of the U-Net whose reduction runs over channels:
//   MODE_CONV3   nn.Conv2d 3x3 pad 1 fprop and dgrad        (reference Model.py:15-16,19-20)
//   MODE_UP      nn.ConvTranspose2d(k2,s2) fprop + bias     (reference Model.py:56-57,66), scatter epilogue
//   MODE_GATHER4 its backward-data (4 strided gathers)
//
// One CTA computes a 128-pixel (8 x 16 patch of one image) x BN-channel output tile:
//   warp 0   TMA producer   : NHWC bf16 activation tiles (4-D tensor maps, halo rows/cols zero-filled by TMA
//                             out-of-bounds handling) and K-major weight tiles, 128B-swizzled into smem rings
//   warp 1   MMA issuer     : tcgen05.mma kind::f16 (bf16 x bf16 -> fp32 in TMEM), one elected thread
//   warps 2-5 epilogue      : tcgen05.ld -> (+bias) -> bf16 -> swizzled smem staging -> TMA store; per-channel
//                             sum / sum-of-squares of the stored tile for BatchNorm (Model.py:17,21)
// For the 3x3 case an activation tile is loaded once per horizontal tap s with two halo rows, and the three
// vertical taps r are UMMA descriptor offsets of r*16 rows (= r*2048 B, swizzle-atom aligned) into that tile,
// so A traffic is 3.75 tile loads per K block instead of 9.
#include "../../include/b200unet.h"
#include "host_common.h"
#include "tc_common.cuh"

#include <stdlib.h>

namespace {

using namespace b2;

constexpr int TH = 8, TW = 16, BM = TH * TW;  // pixel tile
enum { MODE_CONV3 = 0, MODE_UP = 1, MODE_GATHER4 = 2 };

struct IgemmArgs {
  CUtensorMap tmA[4];
  CUtensorMap tmB;
  CUtensorMap tmO[4];
  int tiles_w, tiles_h;  // pixel tiles per image
  int H, W;              // pixel grid of the GEMM M dimension
  int kblocks;           // channels per tap / 64
  int ktap;              // channels per tap (K extent of one tap in the weight matrix)
  int ncols;             // GEMM N (all output channels)
  int ntiles_n;          // ncols / BN
  int cup;               // MODE_UP: channels per (i,j) group of the N dimension
  int stat_c;            // channels of a statistics row (<= cup: a gate whose channels were padded to 64 keeps its real count)
  float* stats;          // [mtiles][2][ncols] or null
  const float* bias;     // MODE_UP: [cup] or null
  const float* scale;    // MODE_CONV3: eval-mode BatchNorm + ReLU folded into the epilogue: [ncols] each, or null
  const float* shift;
};

template <int MODE>
struct ModeTraits {
  static constexpr int TAPS = (MODE == MODE_CONV3) ? 3 : 1;                    // B tiles per A tile
  static constexpr int A_ROWS = (MODE == MODE_CONV3) ? (TH + 2) * TW : BM;     // pixels per A tile
  static constexpr int A_BYTES = A_ROWS * 128;
};

template <int MODE, int BN, int NA, int NB>
struct SmemPlan {
  static constexpr int A_BYTES = ModeTraits<MODE>::A_BYTES;
  static constexpr int B_BYTES = BN * 128;
  static constexpr int RING_BYTES = NA * A_BYTES + NB * B_BYTES;
  static constexpr int STAGE_OUT_BYTES = (BN / 64) * BM * 128;
  static_assert(STAGE_OUT_BYTES <= RING_BYTES, "epilogue staging must fit in the (idle) rings");
  static constexpr int BAR_OFF = RING_BYTES;                // barriers, tmem pointer
  static constexpr int RED_OFF = BAR_OFF + 256;             // float red[2][2][BN]
  static constexpr int TOTAL = RED_OFF + 2 * 2 * BN * 4 + 1024 /* alignment slack */;
};

template <int MODE, int BN, int NA, int NB>
__global__ void __launch_bounds__(192) igemm_kernel(const __grid_constant__ IgemmArgs args) {
  using Plan = SmemPlan<MODE, BN, NA, NB>;
  constexpr int TAPS = ModeTraits<MODE>::TAPS;
  constexpr int A_BYTES = Plan::A_BYTES, B_BYTES = Plan::B_BYTES;

  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t sA = smem_base;
  const uint32_t sB = smem_base + NA * A_BYTES;
  const uint32_t bars = smem_base + Plan::BAR_OFF;
  auto A_full = [&](int i) { return bars + 8u * i; };
  auto A_empty = [&](int i) { return bars + 8u * (NA + i); };
  auto B_full = [&](int i) { return bars + 8u * (2 * NA + i); };
  auto B_empty = [&](int i) { return bars + 8u * (2 * NA + NB + i); };
  const uint32_t acc_full = bars + 8u * (2 * NA + 2 * NB);
  const uint32_t tmem_slot = acc_full + 8;
  volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + Plan::BAR_OFF + 8 * (2 * NA + 2 * NB) + 8);
  float* red = reinterpret_cast<float*>(smem_gen + Plan::RED_OFF);

  const int warp = warp_idx_uniform();
  const int lane = threadIdx.x & 31;

  // ---- tile coordinates
  const int nt = blockIdx.x % args.ntiles_n;
  const int mt = blockIdx.x / args.ntiles_n;
  const int twi = mt % args.tiles_w;
  const int thi = (mt / args.tiles_w) % args.tiles_h;
  const int img = mt / (args.tiles_w * args.tiles_h);
  const int h0 = thi * TH, w0 = twi * TW;
  const int n0 = nt * BN;

  const int ngroups = (MODE == MODE_CONV3) ? args.kblocks * 3 : (MODE == MODE_GATHER4 ? args.kblocks * 4 : args.kblocks);

  // ---- one-time setup
  if (warp == 0 && elect_one_sync()) {
    prefetch_tmap(&args.tmA[0]);
    prefetch_tmap(&args.tmB);
    prefetch_tmap(&args.tmO[0]);
    for (int i = 0; i < NA; ++i) {
      mbar_init(A_full(i), 1);
      mbar_init(A_empty(i), 1);
    }
    for (int i = 0; i < NB; ++i) {
      mbar_init(B_full(i), 1);
      mbar_init(B_empty(i), 1);
    }
    mbar_init(acc_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, BN);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;

  if (warp == 0) {
    // ================================================================= TMA producer
    if (elect_one_sync()) {
      int sa = 0, pa = 0, sb = 0, pb = 0;
      for (int g = 0; g < ngroups; ++g) {
        int cb, s = 0, ij = 0;
        if (MODE == MODE_CONV3) {
          cb = g / 3;
          s = g - cb * 3;
        } else if (MODE == MODE_GATHER4) {
          ij = g / args.kblocks;
          cb = g - ij * args.kblocks;
        } else {
          cb = g;
        }
        mbar_wait(A_empty(sa), pa ^ 1);
        mbar_arrive_expect_tx(A_full(sa), A_BYTES);
        if (MODE == MODE_CONV3)
          tma_load_4d(sA + sa * A_BYTES, &args.tmA[0], A_full(sa), cb * 64, w0 + s - 1, h0 - 1, img);
        else
          tma_load_4d(sA + sa * A_BYTES, &args.tmA[ij], A_full(sa), cb * 64, w0, h0, img);
        if (++sa == NA) { sa = 0; pa ^= 1; }
#pragma unroll
        for (int t = 0; t < TAPS; ++t) {
          int kc;
          if (MODE == MODE_CONV3) kc = (t * 3 + s) * args.ktap + cb * 64;
          else if (MODE == MODE_GATHER4) kc = ij * args.ktap + cb * 64;
          else kc = cb * 64;
          mbar_wait(B_empty(sb), pb ^ 1);
          mbar_arrive_expect_tx(B_full(sb), B_BYTES);
          tma_load_2d(sB + sb * B_BYTES, &args.tmB, B_full(sb), kc, n0);
          if (++sb == NB) { sb = 0; pb ^= 1; }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ================================================================= MMA issuer
    if (elect_one_sync()) {
      constexpr uint32_t idesc = umma_idesc_bf16(BM, BN, 0, 0);
      constexpr uint32_t d_hi = umma_desc_hi_sw128(1024);
      int sa = 0, pa = 0, sb = 0, pb = 0;
      uint32_t acc = 0;
      for (int g = 0; g < ngroups; ++g) {
        mbar_wait(A_full(sa), pa);
        tc_fence_after();
#pragma unroll
        for (int t = 0; t < TAPS; ++t) {
          mbar_wait(B_full(sb), pb);
          tc_fence_after();
          const uint32_t a_lo = umma_desc_lo(sA + sa * A_BYTES + (MODE == MODE_CONV3 ? t * TW * 128 : 0), 16);
          const uint32_t b_lo = umma_desc_lo(sB + sb * B_BYTES, 16);
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            umma_bf16_lh(tmem_base, a_lo + 2 * k, d_hi, b_lo + 2 * k, d_hi, idesc, acc);
            acc = 1;
          }
          umma_commit(B_empty(sb));
          if (++sb == NB) { sb = 0; pb ^= 1; }
        }
        umma_commit(A_empty(sa));
        if (++sa == NA) { sa = 0; pa ^= 1; }
      }
      umma_commit(acc_full);
    }
    __syncwarp();
  } else {
    // ================================================================= epilogue (4 warps, 128 threads)
    const int quad = warp & 3;  // TMEM lanes [32*quad, 32*quad+32) are the ones this warp may read
    const int row = quad * 32 + lane;
    const int et = threadIdx.x - 64;  // 0..127
    mbar_wait(acc_full, 0);
    tc_fence_after();
    const uint32_t stage = smem_base;  // rings are idle now: alias them as the output staging buffer
#pragma unroll 1
    for (int q = 0; q < BN / 64; ++q) {
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        uint32_t v[32];
        tmem_ld32(tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + q * 64 + half * 32, v);
        tmem_ld_wait();
        if (MODE == MODE_CONV3 && args.scale != nullptr)
          affine_relu32(v, args.scale + n0 + q * 64 + half * 32, args.shift + n0 + q * 64 + half * 32);
        if (MODE == MODE_UP && args.bias != nullptr) {
          const int cbase = (n0 + q * 64 + half * 32) % args.cup;
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __ldg(args.bias + cbase + j));
        }
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          uint4 pk;
          pk.x = pack_bf16x2(__uint_as_float(v[8 * t + 0]), __uint_as_float(v[8 * t + 1]));
          pk.y = pack_bf16x2(__uint_as_float(v[8 * t + 2]), __uint_as_float(v[8 * t + 3]));
          pk.z = pack_bf16x2(__uint_as_float(v[8 * t + 4]), __uint_as_float(v[8 * t + 5]));
          pk.w = pack_bf16x2(__uint_as_float(v[8 * t + 6]), __uint_as_float(v[8 * t + 7]));
          const uint32_t chunk = static_cast<uint32_t>(half * 4 + t) ^ (row & 7);
          const uint32_t addr = stage + q * (BM * 128) + row * 128 + chunk * 16;
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(pk.x), "r"(pk.y), "r"(pk.z), "r"(pk.w)
                       : "memory");
        }
      }
    }
    tc_fence_before();
    fence_proxy_async_smem();
    asm volatile("bar.sync 1, 128;" ::: "memory");
    if (et == 0) {
      for (int q = 0; q < BN / 64; ++q) {
        if (MODE == MODE_UP) {
          const int col = n0 + q * 64;  // a tile may span several (i,j) sub-positions: one output map per chunk
          const int ij = col / args.cup;
          tma_store_4d(&args.tmO[ij], stage + q * (BM * 128), col - ij * args.cup, w0, h0, img);
        } else {
          tma_store_4d(&args.tmO[0], stage + q * (BM * 128), n0 + q * 64, w0, h0, img);
        }
      }
      tma_store_commit();
    }
    if (MODE != MODE_GATHER4 && args.stats != nullptr) {
      // per-channel sum and sum of squares over the valid pixels of this tile, from the bf16 values stored. Row layout
      // [m tile][column group][2][cup]: one group for a convolution, the four (i,j) sub-positions for ConvTranspose2d
      const int c = et & 63, hf = et >> 6;
#pragma unroll 1
      for (int q = 0; q < BN / 64; ++q) {
        float s1 = 0.f, s2 = 0.f;
        const uint32_t base = stage + q * (BM * 128);
#pragma unroll 8
        for (int i = 0; i < 64; ++i) {
          const int r = hf * 64 + i;
          const bool valid = (h0 + r / TW < args.H) && (w0 + (r % TW) < args.W);
          uint16_t u;
          const uint32_t addr = base + r * 128 + ((static_cast<uint32_t>(c >> 3) ^ (r & 7)) << 4) + (c & 7) * 2;
          asm volatile("ld.shared.u16 %0, [%1];" : "=h"(u) : "r"(addr));
          const float x = valid ? __uint_as_float(static_cast<uint32_t>(u) << 16) : 0.f;
          s1 += x;
          s2 = fmaf(x, x, s2);
        }
        red[(hf * 2 + 0) * BN + q * 64 + c] = s1;
        red[(hf * 2 + 1) * BN + q * 64 + c] = s2;
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
      const int groups = args.ncols / args.cup;
      for (int ch = et; ch < BN; ch += 128) {
        const int col = n0 + ch, g = col / args.cup, cc = col - g * args.cup;
        if (cc >= args.stat_c) continue;
        float* dst = args.stats + (static_cast<size_t>(mt) * groups + g) * 2 * args.stat_c;
        dst[cc] = red[0 * BN + ch] + red[2 * BN + ch];
        dst[args.stat_c + cc] = red[1 * BN + ch] + red[3 * BN + ch];
      }
    }
    if (et == 0) tma_store_wait_read0();
    __syncwarp();
  }

  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, BN);
}

// ----------------------------------------------------------------------------------------------- host side
// Geometry of a launch over an H x W pixel grid, K = ktap per tap, ncols GEMM columns in groups of cup (statistics rows of
// cup channels); every optional pointer null, tensor maps to be encoded by the caller.
IgemmArgs igemm_args(int H, int W, int ktap, int ncols, int cup) {
  IgemmArgs a = {};
  a.tiles_w = b2h::ceil_div(W, TW);
  a.tiles_h = b2h::ceil_div(H, TH);
  a.H = H;
  a.W = W;
  a.kblocks = ktap / 64;
  a.ktap = ktap;
  a.ncols = ncols;
  a.cup = cup;
  a.stat_c = cup;
  return a;
}

template <int MODE, int BN, int NA, int NB>
int launch_t(const IgemmArgs& a, int N, cudaStream_t st) {
  using Plan = SmemPlan<MODE, BN, NA, NB>;
  static unsigned long long configured = 0;
  auto kern = igemm_kernel<MODE, BN, NA, NB>;
  if (int e = b2h::opt_in_smem(kern, Plan::TOTAL, configured, "igemm")) return e;
  const long long grid = static_cast<long long>(N) * a.tiles_w * a.tiles_h * a.ntiles_n;
  kern<<<static_cast<unsigned>(grid), 192, Plan::TOTAL, st>>>(a);
  return b2h::check_launch("igemm");
}

// BN = 256 only for the ConvTranspose2d forward (all four (i,j) sub-positions of 64 channels per CTA)
template <int MODE>
int launch_mode(IgemmArgs& a, int bn, int N, cudaStream_t st) {
  a.ntiles_n = a.ncols / bn;
  if (bn == 64) return launch_t<MODE, 64, 3, 6>(a, N, st);
  if (bn == 128) return launch_t<MODE, 128, 2, 4>(a, N, st);
  if constexpr (MODE == MODE_UP) {
    if (bn == 256) return launch_t<MODE, 256, 3, 4>(a, N, st);
  }
  b2h::set_error("igemm: bad BN %d", bn);
  return 1;
}

int pick_bn(int ncols) { return ncols % 128 == 0 ? 128 : 64; }

// Kernel-selection overrides: -1 = automatic (measured rules below), 0 = off, 1 = forced on. Initialised from the
// environment (B200UNET_NO_RES, B200UNET_RES2, B200UNET_PAIR), changeable at run time with b200unet_set_kernel_choice.
int g_opt_res = -2, g_opt_res2 = -2, g_opt_pair = -2;
int opt_from_env(const char* name, bool invert) {
  const char* e = getenv(name);
  if (!e) return -1;
  const int v = atoi(e) != 0 ? 1 : 0;
  return invert ? 1 - v : v;
}
void init_opts() {
  if (g_opt_res == -2) g_opt_res = opt_from_env("B200UNET_NO_RES", true);
  if (g_opt_res2 == -2) g_opt_res2 = opt_from_env("B200UNET_RES2", false);
  if (g_opt_pair == -2) g_opt_pair = opt_from_env("B200UNET_PAIR", false);
}

bool use_resident(int Cin, int Cout) {
  init_opts();
  return g_opt_res != 0 && b2h::conv3_res_applicable(Cin, Cout);
}

enum class Conv3Path { RESIDENT, RESIDENT_PAIRS, STREAMING_PAIRS, IGEMM };

// The kernel a 3x3 convolution runs on. The launch and the statistics-row queries all read this one decision, so a buffer
// sized from a query always matches the kernel that fills it.
Conv3Path conv3_path(int N, int H, int W, int Cin, int Cout) {
  init_opts();
  if (use_resident(Cin, Cout)) {
    // CTA pairs (conv3_res2_kernel, conv3_pair.cu) for the resident-weight layers. Measured on B200 (profiles/): pairs win
    // 25-35 % when a tile carries two K blocks (Cin = 128: 128->128, 128->256 and 128->64 up to 256^2), and lose when the
    // per-tile MMA burst is short (Cin = 64) or for 128->64 at 512^2 and above, where the cluster-wide barrier round trip per
    // tile is exposed. B200UNET_RES2=0 / 1 forces the choice off / on for every resident-weight layer.
    bool pairs;
    if (g_opt_res2 >= 0) pairs = g_opt_res2 == 1;
    else pairs = Cin == 128 && (Cout >= 128 || static_cast<long long>(N) * H * W <= 16ll * 256 * 256);
    return pairs ? Conv3Path::RESIDENT_PAIRS : Conv3Path::RESIDENT;
  }
  // streaming CTA-pair kernel (conv3_pair.cu) for the deep layers; B200UNET_PAIR=0 keeps the one-tile-per-CTA igemm
  if (g_opt_pair != 0 && b2h::conv3_pair_applicable(Cin, Cout)) return Conv3Path::STREAMING_PAIRS;
  return Conv3Path::IGEMM;
}

// conv3x3 dispatch shared by the training entry point (BN statistics epilogue) and the eval entry point (BatchNorm + ReLU
// folded into the epilogue: scale/shift per output channel)
int conv3x3_dispatch(const void* x, int x_cs, const void* w, void* y, int y_cs, float* stats_partial, const float* scale,
                     const float* shift, int N, int H, int W, int Cin, int Cout, b200_stream_t stream) {
  B2_REQUIRE(Cin % 64 == 0 && Cout % 64 == 0, "conv3x3_igemm: Cin (%d) and Cout (%d) must be multiples of 64", Cin, Cout);
  B2_REQUIRE(N > 0 && H > 0 && W > 0, "conv3x3_igemm: empty tensor");
  B2_REQUIRE(x_cs >= Cin && y_cs >= Cout && x_cs % 8 == 0 && y_cs % 8 == 0, "conv3x3_igemm: bad pitches %d %d", x_cs, y_cs);
  const cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (conv3_path(N, H, W, Cin, Cout)) {
    case Conv3Path::RESIDENT:
      return b2h::conv3_res_launch(x, x_cs, w, y, y_cs, stats_partial, N, H, W, Cin, Cout, st, scale, shift);
    case Conv3Path::RESIDENT_PAIRS:
      return b2h::conv3_res2_launch(x, x_cs, w, y, y_cs, stats_partial, N, H, W, Cin, Cout, st, scale, shift);
    case Conv3Path::STREAMING_PAIRS:
      return b2h::conv3_pair_launch(x, x_cs, w, y, y_cs, stats_partial, N, H, W, Cin, Cout, st, scale, shift);
    case Conv3Path::IGEMM:
      break;
  }
  IgemmArgs a = igemm_args(H, W, Cin, Cout, Cout);
  a.stats = stats_partial;
  a.scale = scale;
  a.shift = shift;
  const int bn = pick_bn(Cout);
  if (int e = b2h::make_nhwc_map(&a.tmA[0], x, Cin, x_cs, N, H, W, TW, TH + 2)) return e;
  if (int e = b2h::make_tmap_2d(&a.tmB, w, static_cast<uint64_t>(9) * Cin, Cout, bn)) return e;
  if (int e = b2h::make_nhwc_map(&a.tmO[0], y, Cout, y_cs, N, H, W, TW, TH)) return e;
  return launch_mode<MODE_CONV3>(a, bn, N, st);
}

int convt2x2_fprop_impl(const void* x, int x_cs, const void* w_fprop, const float* bias, void* out, int out_cs, float* stats,
                        int stat_c, int N, int H, int W, int Cin, int Cup, int H2, int W2, int pad_top, int pad_left,
                        b200_stream_t stream) {
  B2_REQUIRE(Cin % 64 == 0 && Cup % 64 == 0, "convt2x2_fprop: Cin (%d) and Cup (%d) must be multiples of 64", Cin, Cup);
  B2_REQUIRE(pad_top >= 0 && pad_left >= 0 && 2 * H + pad_top <= H2 && 2 * W + pad_left <= W2,
             "convt2x2_fprop: upsampled map (%dx%d)+pad(%d,%d) does not fit canvas %dx%d", 2 * H, 2 * W, pad_top, pad_left, H2, W2);
  B2_REQUIRE(x_cs % 8 == 0 && out_cs % 8 == 0, "convt2x2_fprop: pitches must be multiples of 8");
  if (stats == nullptr && use_resident(64, 64) && b2h::convt_res_applicable(Cin, Cup))
    return b2h::convt_res_fprop_launch(x, x_cs, w_fprop, bias, out, out_cs, N, H, W, Cin, Cup, H2, W2, pad_top, pad_left,
                                       static_cast<cudaStream_t>(stream));
  IgemmArgs a = igemm_args(H, W, Cin, 4 * Cup, Cup);
  a.stat_c = stat_c;
  a.stats = stats;
  a.bias = bias;
  const int bn = 256;  // all four (i,j) sub-positions of 64 channels per CTA
  if (int e = b2h::make_nhwc_map(&a.tmA[0], x, Cin, x_cs, N, H, W, TW, TH)) return e;
  if (int e = b2h::make_tmap_2d(&a.tmB, w_fprop, Cin, static_cast<uint64_t>(4) * Cup, bn)) return e;
  if (int e = b2h::make_pixel_shuffle_maps(a.tmO, out, Cup, out_cs, N, H, W, H2, W2, pad_top, pad_left, TW, TH)) return e;
  return launch_mode<MODE_UP>(a, bn, N, static_cast<cudaStream_t>(stream));
}


}  // namespace

extern "C" {

int b200unet_conv3x3_igemm(const void* x, int x_cs, const void* w, void* y, int y_cs, float* stats_partial, int N,
                           int H, int W, int Cin, int Cout, b200_stream_t stream) {
  return conv3x3_dispatch(x, x_cs, w, y, y_cs, stats_partial, nullptr, nullptr, N, H, W, Cin, Cout, stream);
}

int b200unet_conv3x3_bn_relu_igemm(const void* x, int x_cs, const void* w, const float* scale, const float* shift, void* a,
                                   int a_cs, int N, int H, int W, int Cin, int Cout, b200_stream_t stream) {
  B2_REQUIRE(scale != nullptr && shift != nullptr, "conv3x3_bn_relu_igemm: scale and shift are required");
  B2_REQUIRE(reinterpret_cast<uintptr_t>(scale) % 16 == 0 && reinterpret_cast<uintptr_t>(shift) % 16 == 0,
             "conv3x3_bn_relu_igemm: scale/shift must be 16-byte aligned");
  return conv3x3_dispatch(x, x_cs, w, a, a_cs, nullptr, scale, shift, N, H, W, Cin, Cout, stream);
}

int b200unet_conv3x3_dgrad_bnred_rows(int N, int H, int W, int Cin, int Cout) {
  if (!(conv3_path(N, H, W, Cin, Cout) == Conv3Path::RESIDENT && b2h::conv3_res_bnred_applicable(Cin, Cout))) return 0;
  static int off = -1;
  if (off < 0) {
    const char* e = getenv("B200UNET_NO_BNRED");
    off = (e != nullptr && atoi(e) != 0) ? 1 : 0;
  }
  return off ? 0 : b2h::conv3_res_stat_rows(N, H, W, Cin, Cout);
}

int b200unet_conv3x3_igemm_bnred(const void* x, int x_cs, const void* w, void* y, int y_cs, const void* bn_y, int bn_y_cs,
                                 const float* scale, const float* shift, const float* mean, const float* rstd,
                                 float* partial, int N, int H, int W, int Cin, int Cout, b200_stream_t stream) {
  B2_REQUIRE(b200unet_conv3x3_dgrad_bnred_rows(N, H, W, Cin, Cout) > 0,
             "conv3x3_igemm_bnred: no fused form for Cin=%d Cout=%d at %dx%d (query b200unet_conv3x3_dgrad_bnred_rows first)", Cin,
             Cout, H, W);
  B2_REQUIRE(x && w && y && bn_y && scale && shift && mean && rstd && partial, "conv3x3_igemm_bnred: null argument");
  B2_REQUIRE(x_cs % 8 == 0 && y_cs % 8 == 0 && bn_y_cs % 8 == 0 && bn_y_cs >= Cout, "conv3x3_igemm_bnred: bad pitches");
  return b2h::conv3_res_bnred_launch(x, x_cs, w, y, y_cs, bn_y, bn_y_cs, scale, shift, mean, rstd, partial, N, H, W, Cin, Cout,
                                     static_cast<cudaStream_t>(stream));
}

int b200unet_set_kernel_choice(int resident, int resident_pairs, int streaming_pairs) {
  B2_REQUIRE(resident >= -1 && resident <= 1 && resident_pairs >= -1 && resident_pairs <= 1 && streaming_pairs >= -1 &&
                 streaming_pairs <= 1,
             "set_kernel_choice: each argument is -1 (automatic), 0 (off) or 1 (on)");
  g_opt_res = resident;
  g_opt_res2 = resident_pairs;
  g_opt_pair = streaming_pairs;
  return 0;
}

int b200unet_conv3x3_stat_rows(int N, int H, int W, int Cin, int Cout) {
  switch (conv3_path(N, H, W, Cin, Cout)) {
    case Conv3Path::RESIDENT: return b2h::conv3_res_stat_rows(N, H, W, Cin, Cout);
    case Conv3Path::RESIDENT_PAIRS: return b2h::conv3_res2_stat_rows(N, H, W, Cin, Cout);
    case Conv3Path::STREAMING_PAIRS: return b2h::conv3_pair_stat_rows(N, H, W, Cin, Cout);
    case Conv3Path::IGEMM: break;
  }
  return N * b2h::ceil_div(H, TH) * b2h::ceil_div(W, TW);
}

int b200unet_convt2x2_fprop(const void* x, int x_cs, const void* w_fprop, const float* bias, void* out, int out_cs,
                            int N, int H, int W, int Cin, int Cup, int H2, int W2, int pad_top, int pad_left,
                            b200_stream_t stream) {
  return convt2x2_fprop_impl(x, x_cs, w_fprop, bias, out, out_cs, nullptr, Cup, N, H, W, Cin, Cup, H2, W2, pad_top, pad_left, stream);
}

int b200unet_convt2x2_stat_rows(int N, int H, int W) { return 4 * N * b2h::ceil_div(H, TH) * b2h::ceil_div(W, TW); }

int b200unet_convt2x2_fprop_stats(const void* x, int x_cs, const void* w_fprop, const float* bias, void* out, int out_cs,
                                  float* stats_partial, int stat_channels, int N, int H, int W, int Cin, int Cup, int H2,
                                  int W2, int pad_top, int pad_left, b200_stream_t stream) {
  B2_REQUIRE(stats_partial != nullptr, "convt2x2_fprop_stats: stats_partial is required (b200unet_convt2x2_stat_rows x 2 x stat_channels floats)");
  B2_REQUIRE(stat_channels >= 1 && stat_channels <= Cup, "convt2x2_fprop_stats: stat_channels=%d must be in [1, Cup]", stat_channels);
  return convt2x2_fprop_impl(x, x_cs, w_fprop, bias, out, out_cs, stats_partial, stat_channels, N, H, W, Cin, Cup, H2, W2, pad_top,
                             pad_left, stream);
}

int b200unet_conv1x1_stat_rows(int N, int H, int W) { return N * b2h::ceil_div(H, TH) * b2h::ceil_div(W, TW); }

int b200unet_conv1x1_fprop(const void* x, int x_cs, const void* w, const float* bias, void* y, int y_cs, float* stats_partial,
                           int stat_channels, int N, int H, int W, int Cin, int Cout, b200_stream_t stream) {
  B2_REQUIRE(x && w && y, "conv1x1_fprop: null argument");
  B2_REQUIRE(stats_partial == nullptr || (stat_channels >= 1 && stat_channels <= Cout), "conv1x1_fprop: stat_channels=%d must be in [1, Cout]", stat_channels);
  B2_REQUIRE(Cin % 64 == 0 && Cout % 64 == 0, "conv1x1_fprop: Cin (%d) and Cout (%d) must be multiples of 64", Cin, Cout);
  B2_REQUIRE(N > 0 && H > 0 && W > 0, "conv1x1_fprop: empty tensor");
  B2_REQUIRE(x_cs >= Cin && y_cs >= Cout && x_cs % 8 == 0 && y_cs % 8 == 0, "conv1x1_fprop: bad pitches %d %d", x_cs, y_cs);
  // K = 64 without bias / statistics (the backward-data of a 64-wide gate): one K block per 128-pixel tile is all prologue for
  // a one-tile-per-CTA launch - the persistent resident-weight kernel streams the tiles instead
  if (Cin == 64 && bias == nullptr && stats_partial == nullptr && use_resident(64, 64))
    return b2h::conv1x1_c64_launch(x, x_cs, w, y, y_cs, nullptr, N, H, W, Cout, static_cast<cudaStream_t>(stream));
  // one column group: the scatter epilogue of the ConvTranspose2d mode degenerates to a plain NHWC store
  IgemmArgs a = igemm_args(H, W, Cin, Cout, Cout);
  a.stat_c = stat_channels;
  a.stats = stats_partial;
  a.bias = bias;
  const int bn = pick_bn(Cout);
  if (int e = b2h::make_nhwc_map(&a.tmA[0], x, Cin, x_cs, N, H, W, TW, TH)) return e;
  if (int e = b2h::make_tmap_2d(&a.tmB, w, Cin, Cout, bn)) return e;
  if (int e = b2h::make_nhwc_map(&a.tmO[0], y, Cout, y_cs, N, H, W, TW, TH)) return e;
  return launch_mode<MODE_UP>(a, bn, N, static_cast<cudaStream_t>(stream));
}


int b200unet_convt2x2_dgrad(const void* du, int du_cs, const void* w_dgrad, void* dx, int dx_cs, int N, int H, int W,
                            int Cin, int Cup, int H2, int W2, int pad_top, int pad_left, b200_stream_t stream) {
  B2_REQUIRE(Cin % 64 == 0 && Cup % 64 == 0, "convt2x2_dgrad: Cin (%d) and Cup (%d) must be multiples of 64", Cin, Cup);
  B2_REQUIRE(pad_top >= 0 && pad_left >= 0 && 2 * H + pad_top <= H2 && 2 * W + pad_left <= W2, "convt2x2_dgrad: bad canvas");
  B2_REQUIRE(du_cs % 8 == 0 && dx_cs % 8 == 0, "convt2x2_dgrad: pitches must be multiples of 8");
  if (use_resident(64, 64) && b2h::convt_res_dgrad_applicable(Cin, Cup))
    return b2h::convt_res_dgrad_launch(du, du_cs, w_dgrad, dx, dx_cs, N, H, W, Cin, Cup, H2, W2, pad_top, pad_left,
                                       static_cast<cudaStream_t>(stream));
  IgemmArgs a = igemm_args(H, W, Cup, Cin, Cin);
  const int bn = pick_bn(Cin);
  if (int e = b2h::make_pixel_shuffle_maps(a.tmA, du, Cup, du_cs, N, H, W, H2, W2, pad_top, pad_left, TW, TH)) return e;
  if (int e = b2h::make_tmap_2d(&a.tmB, w_dgrad, static_cast<uint64_t>(4) * Cup, Cin, bn)) return e;
  if (int e = b2h::make_nhwc_map(&a.tmO[0], dx, Cin, dx_cs, N, H, W, TW, TH)) return e;
  return launch_mode<MODE_GATHER4>(a, bn, N, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
