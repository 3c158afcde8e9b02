// runtime.cu -- error plumbing, launch counter, device queries and TMA
// descriptor encoding (driver entry point fetched through cudart, so the
// library has no link-time dependency on libcuda and loads on a CPU-only box).
#include <atomic>
#include <cstdlib>
#include <mutex>

#include "common.h"

namespace vb {

namespace {
thread_local std::string g_last_error;
std::atomic<int64_t> g_launches{0};

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode = nullptr;
std::once_flag g_encode_once;
typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t, const cuuint32_t*,
                                   CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeIm2colFn g_encode_im2col = nullptr;
std::once_flag g_encode_im2col_once;
}  // namespace

void set_error(const std::string& msg) { g_last_error = msg; }
const std::string& last_error_ref() { return g_last_error; }

int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}
int cuda_fail(cudaError_t e, const char* what) {
  g_last_error = std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")";
  return VITB200_ERR_CUDA;
}
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
int64_t launch_count() { return g_launches.load(std::memory_order_relaxed); }

bool pdl_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("VITB200_PDL");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}

int sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

static bool load_encoder() {
  std::call_once(g_encode_once, [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) ==
            cudaSuccess && q == cudaDriverEntryPointSuccess)
      g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  });
  return g_encode != nullptr;
}

static CUtensorMapDataType tmap_type(int dt) {
  return dt == VITB200_DT_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
         : dt == VITB200_DT_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
         : dt == VITB200_DT_E4M3 ? CU_TENSOR_MAP_DATA_TYPE_UINT8     // E4M3 codes: TMA only moves the bytes
                                : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
}

int make_tmap_2d(CUtensorMap* out, const void* base, int64_t rows, int64_t cols, int64_t ld,
                 int box_rows, int dt, int box_bytes) {
  if (!load_encoder()) return fail(VITB200_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
  const int esz = dt == VITB200_DT_F32 ? 4 : (dt == VITB200_DT_E4M3 ? 1 : 2);
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (ld * esz) % 16 != 0)
    return fail(VITB200_ERR_INVALID, "TMA operand must be 16-byte aligned with a 16-byte row pitch");
  if (box_rows < 1 || box_rows > 256) return fail(VITB200_ERR_INVALID, "TMA box rows out of range");
  if (box_bytes != 128 && box_bytes != 64) return fail(VITB200_ERR_INVALID, "TMA box width must be 64 or 128 bytes");
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstride[1] = {static_cast<cuuint64_t>(ld) * esz};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(box_bytes / esz), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1u, 1u};
  CUresult r = g_encode(out, tmap_type(dt), 2, const_cast<void*>(base), gdim, gstride, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, box_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(VITB200_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult " + std::to_string(int(r)));
  return 0;
}

// [batch, rows, cols] 16-bit tensor (cols contiguous): box = [1, box_rows, 64 cols], 128-byte swizzle.
// Rows >= `rows` of an image are out of bounds for that image: zero-filled on load, clipped on store.
int make_tmap_3d_16(CUtensorMap* out, const void* base, int64_t batch, int64_t rows, int64_t cols,
                    int64_t ld, int box_rows, int dt) {
  if (!load_encoder()) return fail(VITB200_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable");
  if ((reinterpret_cast<uintptr_t>(base) & 15) != 0 || (ld * 2) % 16 != 0)
    return fail(VITB200_ERR_INVALID, "TMA operand must be 16-byte aligned with a 16-byte row pitch");
  if (box_rows < 1 || box_rows > 256) return fail(VITB200_ERR_INVALID, "TMA box rows out of range");
  cuuint64_t gdim[3] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows), static_cast<cuuint64_t>(batch)};
  cuuint64_t gstride[2] = {static_cast<cuuint64_t>(ld) * 2, static_cast<cuuint64_t>(ld) * 2 * static_cast<cuuint64_t>(rows)};
  cuuint32_t box[3] = {64u, static_cast<cuuint32_t>(box_rows), 1u};
  cuuint32_t estr[3] = {1u, 1u, 1u};
  CUresult r = g_encode(out, tmap_type(dt), 3, const_cast<void*>(base), gdim, gstride, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(VITB200_ERR_CUDA, "cuTensorMapEncodeTiled(3d) failed with CUresult " + std::to_string(int(r)));
  return 0;
}

// The patch rearrange of vit.py:146 as an im2col-mode TMA map (patch_tc.cu header).  NHWC fp32 images [batch, H, W, C] are
// described as the 5-D "NDHWC" tensor [batch, gh, ph, gw, pw*C]: depth = the patch row hh, height = the row p1 inside a
// patch, width = the patch column ww, channels = the pw*C contiguous floats of one patch row.  The filter is ph x 1 x 1
// (all of H, nothing else), so the box of filter origins is {w in [0, gw), h = 0, d in [0, gh)} and consecutive "pixels"
// are consecutive patches (ww fastest, then hh, then the image).  One load = `pixels` patches x pw*C floats of patch row
// h_off, dense.  (A 4-D map with an H traversal stride of ph is the obvious form, but TMA traversal strides stop at 8.)
int make_tmap_im2col_patches(CUtensorMap* out, const float* images, int64_t batch, int H, int W, int C, int ph, int pw,
                             int pixels) {
  std::call_once(g_encode_im2col_once, [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &fn, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      g_encode_im2col = reinterpret_cast<EncodeIm2colFn>(fn);
  });
  if (!g_encode_im2col) return fail(VITB200_ERR_CUDA, "cuTensorMapEncodeIm2col entry point unavailable");
  const int run = pw * C;
  if ((reinterpret_cast<uintptr_t>(images) & 15) != 0 || (run * 4) % 16 != 0 || run > 256 || pixels < 1 || pixels > 1024 ||
      ph < 1 || ph > 16 || pw < 1 || H % ph != 0 || W % pw != 0)
    return fail(VITB200_ERR_INVALID, "im2col patch map: unsupported geometry (pw*C*4 a multiple of 16 bytes, ph <= 16)");
  const int gw = W / pw, gh = H / ph;
  cuuint64_t gdim[5] = {cuuint64_t(run), cuuint64_t(gw), cuuint64_t(ph), cuuint64_t(gh), cuuint64_t(batch)};
  cuuint64_t gstride[4] = {cuuint64_t(run) * 4, cuuint64_t(W) * C * 4, cuuint64_t(ph) * W * C * 4, cuuint64_t(H) * W * C * 4};
  int lower[3] = {0, 0, 0};               // {W, H, D}
  int upper[3] = {0, -(ph - 1), 0};       // the filter covers all ph rows of H: its only origin is h = 0
  cuuint32_t estr[5] = {1u, 1u, 1u, 1u, 1u};
  CUresult r = g_encode_im2col(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, const_cast<float*>(images), gdim, gstride, lower,
                               upper, cuuint32_t(run), cuuint32_t(pixels), estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS)
    return fail(VITB200_ERR_CUDA, "cuTensorMapEncodeIm2col failed with CUresult " + std::to_string(int(r)));
  return 0;
}

}  // namespace vb
