// Library-level entry points: version, error string, launch counter, tensor-map encoding.
#include <atomic>
#include <mutex>
#include <string.h>

#include "../../include/b200unet.h"
#include "host_common.h"

namespace b2h {

static thread_local char g_err[512] = "";
static std::atomic<int64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return 2;
  }
  count_launch();
  return 0;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

int make_tmap_4d(CUtensorMap* m, const void* base, uint64_t d0, uint64_t d1, uint64_t d2, uint64_t d3, uint64_t s1,
                 uint64_t s2, uint64_t s3, uint32_t box_w, uint32_t box_h) {
  EncodeTiledFn enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled unavailable (no CUDA driver?)");
    return 3;
  }
  if ((reinterpret_cast<uintptr_t>(base) & 15) || (s1 & 15) || (s2 & 15) || (s3 & 15)) {
    set_error("tensor map: base/strides must be 16-byte aligned (base=%p s1=%llu s2=%llu s3=%llu)", base,
              (unsigned long long)s1, (unsigned long long)s2, (unsigned long long)s3);
    return 3;
  }
  cuuint64_t dims[4] = {d0, d1, d2, d3};
  cuuint64_t strides[3] = {s1, s2, s3};
  cuuint32_t box[4] = {64, box_w, box_h, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(4d) failed: %d (dims %llu %llu %llu %llu strides %llu %llu %llu box %u %u)",
              (int)r, (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2,
              (unsigned long long)d3, (unsigned long long)s1, (unsigned long long)s2, (unsigned long long)s3, box_w,
              box_h);
    return 3;
  }
  return 0;
}

int make_pixel_shuffle_maps(CUtensorMap m[4], const void* canvas, int C, int pitch, int N, int H, int W, int H2, int W2,
                            int pad_top, int pad_left, uint32_t box_w, uint32_t box_h) {
  const uint64_t s = static_cast<uint64_t>(pitch) * 2;
  for (int ij = 0; ij < 4; ++ij) {
    const int i = ij >> 1, j = ij & 1;
    const uint8_t* base = static_cast<const uint8_t*>(canvas) + (static_cast<uint64_t>(pad_top + i) * W2 + pad_left + j) * s;
    if (int e = make_tmap_4d(&m[ij], base, C, W, H, N, 2 * s, 2 * s * W2, s * W2 * H2, box_w, box_h)) return e;
  }
  return 0;
}

int make_tmap_2d(CUtensorMap* m, const void* base, uint64_t k, uint64_t rows, uint32_t box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled unavailable (no CUDA driver?)");
    return 3;
  }
  if ((reinterpret_cast<uintptr_t>(base) & 15) || ((k * 2) & 15)) {
    set_error("tensor map 2d: base/pitch must be 16-byte aligned");
    return 3;
  }
  cuuint64_t dims[2] = {k, rows};
  cuuint64_t strides[1] = {k * 2};
  cuuint32_t box[2] = {64, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(2d) failed: %d (k %llu rows %llu box_rows %u)", (int)r,
              (unsigned long long)k, (unsigned long long)rows, box_rows);
    return 3;
  }
  return 0;
}

}  // namespace b2h

extern "C" {
int b200unet_version(void) { return 100; }
const char* b200unet_last_error(void) { return b2h::g_err; }
int64_t b200unet_launch_count(void) { return b2h::g_launches.load(); }
int b200unet_tile_h(void) { return 8; }
int b200unet_tile_w(void) { return 16; }
}
