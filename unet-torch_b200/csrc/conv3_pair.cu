// CTA-pair (tcgen05 cta_group::2) persistent 3x3 implicit GEMMs (nn.Conv2d fprop and dgrad, reference
// Model.py:15-16,19-20). Two kernels on one skeleton that differ only in how the weights reach shared memory:
//  * conv3_res2_kernel<BN, KB, NA, OB>: weights RESIDENT, for the layers of conv3_res.cu's resident-weight kernel
//    (Cin = 64 / 128). All 9 x KB weight tiles of the CTA's BN/2 rows are loaded once, behind one barrier.
//  * conv3_pair_kernel<BN, NA, NB, OB>: weights STREAMED, for the deep levels (Cin >= 256: down2.conv2 ... up3.conv1),
//    where a channel slice of the weights no longer fits in shared memory. They pass through a second TMA ring at tap
//    granularity: per K block and CTA 23 KB of activations + 9 x (BN/2 rows x 128 B) of weights. With BN = 256 that is
//    170 KB of L2->SM traffic per 36 MMAs of 128 cycles (37 B/clk/SM; igemm.cu: 90 B/clk) and 64 B/clk of
//    shared-memory operand reads (igemm.cu: 128).
//
// Why pairs: with one CTA per MMA an N = 64 tile reads 6 KB of shared-memory operands per 32-cycle MMA (192 B/clk, over
// the 128 B/clk an SM can deliver) and Cin = 128 layers cannot keep more than a 64-column weight slice resident. A pair
// issues ONE M = 256 MMA for two adjacent 16x8 pixel tiles: each CTA supplies its own 128 activation rows and only HALF
// of the weight rows (BN/2), so the resident slice per CTA halves (N = 128 fits for Cin = 128) and shared-memory reads
// per MMA cycle drop to 96-160 B/clk. The MMA instruction count per FLOP halves as well.
//
// Persistent pairs walk a static tile-pair schedule; per 64-channel block one 18x10 halo tile is loaded and the 9 taps
// are descriptor offsets into it; two TMEM accumulator buffers. Roles per CTA (192 threads): warp 0 TMA producer (its
// own activation halo tiles, its half of the weights; completion bytes are credited to the LEADER's barriers), warp 1
// MMA issuer (leader CTA only), warps 2-5 epilogue (each CTA drains its own 128 TMEM lanes: bf16 -> swizzled staging ->
// TMA store, BatchNorm statistics in registers).
// Barriers: B_full (weights) / A_full[NA] / T_empty[2] live in the leader (remote TMA complete_tx / remote arrives);
// B_empty (streamed weights) / A_empty[NA] / T_full[2] exist in both CTAs and are signalled by multicast tcgen05.commit.
#include "../../include/b200unet.h"
#include "host_common.h"
#include "tc_common.cuh"

namespace {

using namespace b2;

constexpr int RTH = 16, RTW = 8;
constexpr int IN_H = RTH + 2, IN_W = RTW + 2;
constexpr int A_BOX_BYTES = IN_H * IN_W * 128;                    // 23040
constexpr int A_STAGE = (A_BOX_BYTES + 1023) / 1024 * 1024;       // 23552
constexpr int OUT_CHUNK = 128 * 128;

struct PairArgs {
  CUtensorMap tmA, tmW, tmO;
  int tiles_w, tiles_h, tiles_total;
  int H, W;
  int ncols;     // Cout
  int ntiles_n;  // Cout / BN
  int workers;   // CTA pairs per channel slice (grid = 2 * workers * ntiles_n)
  int kblocks;   // Cin / 64 (streamed weights; the resident kernel has it as a template parameter)
  int ktap;      // Cin (K extent of one tap in the weight operand; streamed weights)
  float* stats;  // [2 * workers][2][ncols] or null
  const float* scale;  // eval-mode BatchNorm + ReLU folded into the epilogue: [ncols] each, or null
  const float* shift;
};

// Shared-memory plans: byte offsets from the 1024-aligned base, barriers in 8-byte slots from BAR_OFF. A_full[NA] and
// A_empty[NA] start at slot A_BAR, T_full[2], T_empty[2] and the TMEM address at slot T_BAR, the weight barriers at B_BAR.
template <int BN_, int KB_, int NA_, int OB_>
struct Res2Plan {  // resident: 9 x KB weight tiles at B_OFF, one barrier B_full(0)
  static constexpr bool RESIDENT = true;
  static constexpr int BN = BN_, KB = KB_, NA = NA_, NB = 0, OB = OB_;
  static constexpr int B_STAGE = (BN / 2) * 128;  // one weight tile: BN/2 rows x 64 channels
  static constexpr int B_BYTES = 9 * KB * B_STAGE;
  static constexpr int B_OFF = 0;
  static constexpr int A_OFF = B_BYTES;
  static constexpr int OUT_OFF = A_OFF + NA * A_STAGE;
  static constexpr int BAR_OFF = OUT_OFF + OB * (BN / 64) * OUT_CHUNK;
  static constexpr int TOTAL = BAR_OFF + 256 + 1024;
  static constexpr int B_BAR = 0, A_BAR = 1, T_BAR = 1 + 2 * NA;
  static_assert(B_BYTES % 1024 == 0, "weight tiles must stay 1024-byte aligned");
};

template <int BN_, int NA_, int NB_, int OB_>
struct PairPlan {  // streamed: an NB-stage ring of (one tap, one 64-channel block) weight tiles, B_full[NB] / B_empty[NB]
  static constexpr bool RESIDENT = false;
  static constexpr int BN = BN_, KB = 0, NA = NA_, NB = NB_, OB = OB_;
  static constexpr int B_STAGE = (BN / 2) * 128;  // one weight tile: BN/2 rows x 64 channels
  static constexpr int A_OFF = 0;
  static constexpr int B_OFF = NA * A_STAGE;
  static constexpr int OUT_OFF = B_OFF + NB * B_STAGE;
  static constexpr int BAR_OFF = OUT_OFF + OB * (BN / 64) * OUT_CHUNK;
  static constexpr int TOTAL = BAR_OFF + 512 + 1024;
  static constexpr int A_BAR = 0, B_BAR = 2 * NA, T_BAR = 2 * NA + 2 * NB;
};

template <class P>
__device__ __forceinline__ void conv3_pair_body(const PairArgs& args) {
  constexpr int BN = P::BN, NA = P::NA, NB = P::NB, OB = P::OB;
  constexpr int BH = BN / 2;  // weight rows this CTA supplies
  static_assert(P::TOTAL <= 227 * 1024, "shared memory plan exceeds 227 KiB");
  static_assert(4 * 2 * BN * 4 <= OB * (BN / 64) * OUT_CHUNK, "final statistics reduction aliases the staging buffer");
  extern __shared__ uint8_t smem_raw[];
  // both CTAs must use IDENTICAL smem offsets (operand descriptors and barrier offsets are shared by the pair)
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t sA = smem_base + P::A_OFF;
  const uint32_t sB = smem_base + P::B_OFF;
  const uint32_t sO = smem_base + P::OUT_OFF;
  const uint32_t bars = smem_base + P::BAR_OFF;
  auto A_full = [&](int i) { return bars + 8u * (P::A_BAR + i); };
  auto A_empty = [&](int i) { return bars + 8u * (P::A_BAR + NA + i); };
  auto B_full = [&](int i) { return bars + 8u * (P::B_BAR + i); };
  auto B_empty = [&](int i) { return bars + 8u * (P::B_BAR + NB + i); };
  auto T_full = [&](int i) { return bars + 8u * (P::T_BAR + i); };
  auto T_empty = [&](int i) { return bars + 8u * (P::T_BAR + 2 + i); };
  const uint32_t tmem_slot = bars + 8u * (P::T_BAR + 4);
  volatile uint32_t* tmem_slot_gen = reinterpret_cast<volatile uint32_t*>(smem_gen + P::BAR_OFF + 8 * (P::T_BAR + 4));
  const int KB = P::RESIDENT ? P::KB : args.kblocks;

  const int warp = warp_idx_uniform();
  const int lane = threadIdx.x & 31;
  const uint32_t crank = cluster_ctarank();  // 0 = leader
  const int cluster = blockIdx.x >> 1;
  const int nt = cluster % args.ntiles_n;
  const int pw = cluster / args.ntiles_n;
  const int n0 = nt * BN;
  const int pairs_total = (args.tiles_total + 1) >> 1;
  const int npairs_mine = (pairs_total - pw + args.workers - 1) / args.workers;  // tile pairs pw, pw+workers, ...

  if (warp == 0 && elect_one_sync()) {
    prefetch_tmap(&args.tmA);
    prefetch_tmap(&args.tmW);
    prefetch_tmap(&args.tmO);
    if constexpr (P::RESIDENT) mbar_init(B_full(0), 1);
    for (int i = 0; i < NA; ++i) {
      mbar_init(A_full(i), 1);   // the leader's arrive.expect_tx; bytes arrive from both CTAs
      mbar_init(A_empty(i), 1);  // multicast commit
    }
    if constexpr (!P::RESIDENT) {
      for (int i = 0; i < NB; ++i) {
        mbar_init(B_full(i), 1);
        mbar_init(B_empty(i), 1);
      }
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(T_full(i), 1);   // multicast commit
      mbar_init(T_empty(i), 8);  // 4 epilogue warps x 2 CTAs (used in the leader only)
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc_2cta(tmem_slot, 2 * BN);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // peer barriers are initialised before any remote arrive / complete_tx can reach them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_gen;

  auto tile_coords = [&](int j, int& img, int& h0, int& w0) {
    const int t = 2 * (pw + j * args.workers) + static_cast<int>(crank);  // may be == tiles_total (odd count): TMA clips
    const int twi = t % args.tiles_w;
    const int thi = (t / args.tiles_w) % args.tiles_h;
    img = t / (args.tiles_w * args.tiles_h);
    h0 = thi * RTH;
    w0 = twi * RTW;
  };

  if (warp == 0) {
    // ================================================================= TMA producer (both CTAs)
    if (elect_one_sync()) {
      if constexpr (P::RESIDENT) {
        const uint32_t B_full_l = mapa_cluster(B_full(0), 0);
        if (crank == 0) mbar_arrive_expect_tx(B_full(0), 2 * P::B_BYTES);
#pragma unroll 1
        for (int tap = 0; tap < 9; ++tap)
#pragma unroll
          for (int cb = 0; cb < KB; ++cb)
            tma_load_2d_2cta(sB + (tap * KB + cb) * P::B_STAGE, &args.tmW, B_full_l, (tap * KB + cb) * 64,
                             n0 + static_cast<int>(crank) * BH);
      }
      int sa = 0, pa = 0, sb = 0, pb = 0;
#pragma unroll 1
      for (int j = 0; j < npairs_mine; ++j) {
        int img, h0, w0;
        tile_coords(j, img, h0, w0);
#pragma unroll 1
        for (int cb = 0; cb < KB; ++cb) {
          mbar_wait(A_empty(sa), pa ^ 1);
          if (crank == 0) mbar_arrive_expect_tx(A_full(sa), 2 * A_BOX_BYTES);
          tma_load_4d_2cta(sA + sa * A_STAGE, &args.tmA, mapa_cluster(A_full(sa), 0), cb * 64, w0 - 1, h0 - 1, img);
          if (++sa == NA) { sa = 0; pa ^= 1; }
          if constexpr (!P::RESIDENT) {
#pragma unroll 1
            for (int tap = 0; tap < 9; ++tap) {
              mbar_wait(B_empty(sb), pb ^ 1);
              if (crank == 0) mbar_arrive_expect_tx(B_full(sb), 2 * P::B_STAGE);
              tma_load_2d_2cta(sB + sb * P::B_STAGE, &args.tmW, mapa_cluster(B_full(sb), 0), tap * args.ktap + cb * 64,
                               n0 + static_cast<int>(crank) * BH);
              if (++sb == NB) { sb = 0; pb ^= 1; }
            }
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ================================================================= MMA issuer (leader only)
    if (crank == 0 && elect_one_sync()) {
      constexpr uint32_t idesc = umma_idesc_bf16(256, BN, 0, 0);
      constexpr uint32_t a_hi = umma_desc_hi_sw128(IN_W * 128), b_hi = umma_desc_hi_sw128(1024);
      const uint32_t w_lo = umma_desc_lo(sB, 16);  // resident weights: tile (tap, cb) at w_lo + (tap * KB + cb) * (BH * 8)
      if constexpr (P::RESIDENT) {
        mbar_wait(B_full(0), 0);
        tc_fence_after();
      }
      int sa = 0, pa = 0, sb = 0, pb = 0;
#pragma unroll 1
      for (int j = 0; j < npairs_mine; ++j) {
        const int buf = j & 1;
        mbar_wait(T_empty(buf), ((j >> 1) & 1) ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * BN;
        uint32_t acc = 0;
#pragma unroll(P::RESIDENT && P::KB <= 2 ? P::KB : 1)
        for (int cb = 0; cb < KB; ++cb) {
          mbar_wait(A_full(sa), pa);
          tc_fence_after();
          const uint32_t a_lo = umma_desc_lo(sA + sa * A_STAGE, 16);
#pragma unroll
          for (int tap = 0; tap < 9; ++tap) {
            if constexpr (!P::RESIDENT) {
              mbar_wait(B_full(sb), pb);
              tc_fence_after();
            }
            const uint32_t a_tap = a_lo + ((tap / 3) * IN_W + (tap % 3)) * 8;
            const uint32_t b_tap = P::RESIDENT ? w_lo + (tap * KB + cb) * (BH * 8) : umma_desc_lo(sB + sb * P::B_STAGE, 16);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              umma_bf16_lh_2cta(d_tmem, a_tap + 2 * k, a_hi, b_tap + 2 * k, b_hi, idesc, acc);
              acc = 1;
            }
            if constexpr (!P::RESIDENT) {
              umma_commit_2cta(B_empty(sb));  // frees the weight stage in BOTH CTAs
              if (++sb == NB) { sb = 0; pb ^= 1; }
            }
          }
          umma_commit_2cta(A_empty(sa));  // frees the activation stage in BOTH CTAs
          if (++sa == NA) { sa = 0; pa ^= 1; }
        }
        umma_commit_2cta(T_full(buf));  // accumulator ready: both CTAs' epilogues
      }
    }
    __syncwarp();
  } else {
    // ================================================================= epilogue (both CTAs, 4 warps each)
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    const int et = threadIdx.x - 64;
    const int cp = et & 31, rq = et >> 5;
    const bool want_stats = args.stats != nullptr;
    float s1[BN / 64][2], s2[BN / 64][2];
#pragma unroll
    for (int q = 0; q < BN / 64; ++q) s1[q][0] = s1[q][1] = s2[q][0] = s2[q][1] = 0.f;
    const uint32_t T_empty_l0 = mapa_cluster(T_empty(0), 0), T_empty_l1 = mapa_cluster(T_empty(1), 0);

#pragma unroll 1
    for (int j = 0; j < npairs_mine; ++j) {
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
          if (args.scale != nullptr) affine_relu32(v, args.scale + n0 + q * 64 + half * 32, args.shift + n0 + q * 64 + half * 32);
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
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(buf ? T_empty_l1 : T_empty_l0);  // hand the buffer back to the leader's MMA warp
      fence_proxy_async_smem();
      if (OB == 2 && et == 0) tma_store_wait_read0();
      asm volatile("bar.sync 1, 128;" ::: "memory");
      if (et == 0) {
#pragma unroll
        for (int q = 0; q < BN / 64; ++q) tma_store_4d(&args.tmO, stage + q * OUT_CHUNK, n0 + q * 64, w0, h0, img);
        tma_store_commit();
      }
      if (want_stats) {
        // img >= N (the odd tile of the last pair) contributes nothing: its accumulators are zero (TMA zero fill)
        const bool full = (h0 + RTH <= args.H) && (w0 + RTW <= args.W);
#pragma unroll
        for (int q = 0; q < BN / 64; ++q) {
          const uint32_t base = stage + q * OUT_CHUNK + (cp & 3) * 4;
#pragma unroll 8
          for (int i = 0; i < 32; ++i) {
            const int r = rq * 32 + i;
            uint32_t u;
            asm volatile("ld.shared.b32 %0, [%1];"
                         : "=r"(u)
                         : "r"(base + r * 128 + ((static_cast<uint32_t>(cp >> 2) ^ (r & 7)) << 4)));
            float x0 = __uint_as_float(u << 16), x1 = __uint_as_float(u & 0xffff0000u);
            if (!full && !((h0 + (r >> 3) < args.H) && (w0 + (r & 7) < args.W))) x0 = x1 = 0.f;
            s1[q][0] += x0;
            s1[q][1] += x1;
            s2[q][0] = fmaf(x0, x0, s2[q][0]);
            s2[q][1] = fmaf(x1, x1, s2[q][1]);
          }
        }
      }
      if (OB == 1) {
        if (et == 0) tma_store_wait_read0();
        asm volatile("bar.sync 1, 128;" ::: "memory");
      }
    }
    if (et == 0) tma_store_wait_read0();
    asm volatile("bar.sync 1, 128;" ::: "memory");
    if (want_stats) {
      float* red = reinterpret_cast<float*>(smem_gen + P::OUT_OFF);
#pragma unroll
      for (int q = 0; q < BN / 64; ++q) {
        red[(rq * 2 + 0) * BN + q * 64 + cp * 2 + 0] = s1[q][0];
        red[(rq * 2 + 0) * BN + q * 64 + cp * 2 + 1] = s1[q][1];
        red[(rq * 2 + 1) * BN + q * 64 + cp * 2 + 0] = s2[q][0];
        red[(rq * 2 + 1) * BN + q * 64 + cp * 2 + 1] = s2[q][1];
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");
      float* dst = args.stats + (static_cast<size_t>(pw) * 2 + crank) * 2 * args.ncols + n0;
      for (int i = et; i < 2 * BN; i += 128) {
        const int stat = i / BN, ch = i - stat * BN;
        dst[stat * args.ncols + ch] = red[(0 * 2 + stat) * BN + ch] + red[(1 * 2 + stat) * BN + ch] +
                                      red[(2 * 2 + stat) * BN + ch] + red[(3 * 2 + stat) * BN + ch];
      }
    }
    tc_fence_before();
  }

  __syncthreads();
  cluster_sync_all();  // nobody leaves (or frees TMEM) while the peer may still touch this CTA's smem / barriers
  if (warp == 1) tmem_dealloc_2cta(tmem_base, 2 * BN);
}

template <int BN, int KB, int NA, int OB>
__global__ void __launch_bounds__(192, 1) conv3_res2_kernel(const __grid_constant__ PairArgs args) {
  conv3_pair_body<Res2Plan<BN, KB, NA, OB>>(args);
}

template <int BN, int NA, int NB, int OB>
__global__ void __launch_bounds__(192, 1) conv3_pair_kernel(const __grid_constant__ PairArgs args) {
  conv3_pair_body<PairPlan<BN, NA, NB, OB>>(args);
}

using PairKernel = void (*)(PairArgs);

// kern must be the kernel instantiation of plan P (P::TOTAL bytes of dynamic shared memory)
template <class P>
int launch_pair(PairKernel kern, const PairArgs& a, cudaStream_t st) {
  const char* name = P::RESIDENT ? "conv3_res2" : "conv3_pair";
  static unsigned long long configured = 0;
  if (int e = b2h::opt_in_smem(kern, P::TOTAL, configured, name)) return e;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * a.workers * a.ntiles_n);
  cfg.blockDim = dim3(192);
  cfg.dynamicSmemBytes = P::TOTAL;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, a);
  if (e != cudaSuccess) {
    b2h::set_error("%s launch: %s", name, cudaGetErrorString(e));
    return 2;
  }
  return b2h::check_launch(name);
}

// Number of CTA pairs that can be resident at once (one CTA per SM, both CTAs of a pair in one TPC): the persistent
// schedule is static, so the grid must not exceed it. Queried once per kernel, with its largest shared-memory variant.
template <class P>
int max_pairs(PairKernel kern) {
  static int n = 0;
  if (n == 0) {
    int got = 0;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * 74);
    cfg.blockDim = dim3(192);
    cfg.dynamicSmemBytes = P::TOTAL;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, P::TOTAL) == cudaSuccess &&
        cudaOccupancyMaxActiveClusters(&got, kern, &cfg) == cudaSuccess && got > 0)
      n = got;
    else
      n = 64;  // conservative
    cudaGetLastError();
  }
  return n;
}

int res2_max_pairs() { return max_pairs<Res2Plan<128, 2, 2, 1>>(conv3_res2_kernel<128, 2, 2, 1>); }
int pair_max_pairs() { return max_pairs<PairPlan<256, 2, 6, 1>>(conv3_pair_kernel<256, 2, 6, 1>); }

}  // namespace

namespace b2h {

static int res2_bn(int Cout) { return (Cout % 128 == 0) ? 128 : 64; }
static int pair_bn(int Cout) { return (Cout % 256 == 0) ? 256 : 128; }

// max_pairs: CTA pairs resident at once for the kernel that will run
static void pair_geometry(int N, int H, int W, int Cout, int bn, int max_pairs, int* ntn, int* workers, int* tiles) {
  *ntn = Cout / bn;
  *tiles = N * ceil_div(H, RTH) * ceil_div(W, RTW);
  const int pairs = (*tiles + 1) / 2;
  int w = max_pairs / *ntn;
  if (w < 1) w = 1;
  if (w > pairs) w = pairs;
  *workers = w;
}

static int pair_stat_rows(int N, int H, int W, int Cout, int bn, int max_pairs) {
  int ntn, workers, tiles;
  pair_geometry(N, H, W, Cout, bn, max_pairs, &ntn, &workers, &tiles);
  return 2 * workers;
}

// Arguments of either kernel; tensor-map encoding failures return their error code.
static int pair_args(PairArgs* a, const void* x, int x_cs, const void* w, void* y, int y_cs, float* stats_partial, int N,
                     int H, int W, int Cin, int Cout, int bn, int max_pairs, const float* scale, const float* shift) {
  pair_geometry(N, H, W, Cout, bn, max_pairs, &a->ntiles_n, &a->workers, &a->tiles_total);
  a->tiles_w = ceil_div(W, RTW);
  a->tiles_h = ceil_div(H, RTH);
  a->H = H;
  a->W = W;
  a->ncols = Cout;
  a->kblocks = Cin / 64;
  a->ktap = Cin;
  a->stats = stats_partial;
  a->scale = scale;
  a->shift = shift;
  if (int e = make_nhwc_map(&a->tmA, x, Cin, x_cs, N, H, W, IN_W, IN_H)) return e;
  if (int e = make_tmap_2d(&a->tmW, w, static_cast<uint64_t>(9) * Cin, Cout, bn / 2)) return e;
  return make_nhwc_map(&a->tmO, y, Cout, y_cs, N, H, W, RTW, RTH);
}

int conv3_res2_stat_rows(int N, int H, int W, int Cin, int Cout) {
  (void)Cin;
  return pair_stat_rows(N, H, W, Cout, res2_bn(Cout), res2_max_pairs());
}

int conv3_res2_launch(const void* x, int x_cs, const void* w, void* y, int y_cs, float* stats_partial, int N, int H,
                      int W, int Cin, int Cout, cudaStream_t st, const float* scale,
                     const float* shift) {
  const int bn = res2_bn(Cout);
  PairArgs a;
  if (int e = pair_args(&a, x, x_cs, w, y, y_cs, stats_partial, N, H, W, Cin, Cout, bn, res2_max_pairs(), scale, shift))
    return e;
  if (Cin == 64 && bn == 64) return launch_pair<Res2Plan<64, 1, 4, 2>>(conv3_res2_kernel<64, 1, 4, 2>, a, st);
  if (Cin == 64 && bn == 128) return launch_pair<Res2Plan<128, 1, 3, 2>>(conv3_res2_kernel<128, 1, 3, 2>, a, st);
  if (Cin == 128 && bn == 64) return launch_pair<Res2Plan<64, 2, 4, 2>>(conv3_res2_kernel<64, 2, 4, 2>, a, st);
  return launch_pair<Res2Plan<128, 2, 2, 1>>(conv3_res2_kernel<128, 2, 2, 1>, a, st);
}

bool conv3_pair_applicable(int Cin, int Cout) { return Cin >= 256 && Cin % 64 == 0 && Cout % 128 == 0; }

int conv3_pair_stat_rows(int N, int H, int W, int Cin, int Cout) {
  (void)Cin;
  return pair_stat_rows(N, H, W, Cout, pair_bn(Cout), pair_max_pairs());
}

int conv3_pair_launch(const void* x, int x_cs, const void* w, void* y, int y_cs, float* stats_partial, int N, int H,
                      int W, int Cin, int Cout, cudaStream_t st, const float* scale,
                     const float* shift) {
  const int bn = pair_bn(Cout);
  PairArgs a;
  if (int e = pair_args(&a, x, x_cs, w, y, y_cs, stats_partial, N, H, W, Cin, Cout, bn, pair_max_pairs(), scale, shift))
    return e;
  if (bn == 256) return launch_pair<PairPlan<256, 2, 6, 1>>(conv3_pair_kernel<256, 2, 6, 1>, a, st);
  return launch_pair<PairPlan<128, 3, 8, 2>>(conv3_pair_kernel<128, 3, 8, 2>, a, st);
}

}  // namespace b2h
