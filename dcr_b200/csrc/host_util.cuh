// Host-side helpers shared by the .cu translation units: error capture for the C ABI, the driver entry point
// for tensor-map encoding (no link-time dependency on libcuda), SM count cache.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <string>

namespace dcr {

// last error message, per host thread (returned by dcr_last_error()).
std::string& last_error_storage();
int set_error(int code, const char* fmt, ...);

#define DCR_CUDA_CHECK(expr)                                                                           \
  do {                                                                                                 \
    cudaError_t _e = (expr);                                                                           \
    if (_e != cudaSuccess)                                                                             \
      return ::dcr::set_error(-2, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)

#define DCR_REQUIRE(cond, ...)                        \
  do {                                                \
    if (!(cond)) return ::dcr::set_error(-1, __VA_ARGS__); \
  } while (0)

struct DeviceInfo {
  int device = -1;
  int num_sms = 0;
  int cc_major = 0, cc_minor = 0;
  size_t max_smem_optin = 0;
};
// cumulative number of kernels this library has launched (all threads)
void count_launch(int n = 1);
long long launch_count();

// Tuning switches are honoured ONLY when DCR_B200_TUNING=1 is set in the environment: a stray variable cannot change
// what a benchmark or a test runs.  Each one selects a variant that gives the same results as the default path, and a
// GPU test uses each one to compare that variant against the default: DCR_GEMM_CG2, DCR_GEMM_TILE_ORDER and
// DCR_CONV_NO_HALO (conv_gemm.cu, conv3x3_halo.cu), DCR_POOL_GENERIC (pool_norm.cu), DCR_NO_BLOCK_FUSION
// (bottleneck_fuse.cu) and DCR_SIM_RESCORE_BLOCK (sim_topk.cu).
bool tuning_enabled();
int tuning_int(const char* name, int dflt);
bool tuning_flag(const char* name);   // true when tuning is enabled and the variable is set (to anything)

// cached per current device; returns nullptr and sets the error on failure
const DeviceInfo* device_info();

// 2-D row-major bf16 tensor [rows, cols] (cols contiguous), box = [box_rows, box_cols], 128-byte swizzle.
// box_cols * 2 bytes must be 128.
int make_tmap_2d_bf16(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint64_t row_stride_elems,
                      uint32_t box_rows, uint32_t box_cols);

// im2col tensor map over an NHWC bf16 activation tensor (see conv_gemm.cu)
// stride_w/h/n: element strides of the (possibly overlapping-window) NHWC view; 0 = dense
// 4-D tiled map over an NHWC bf16 tensor (dims C, W, H, N; `pixel_stride` elements between pixels), box = 64 channels x
// box_w x box_h x 1 image, 128B swizzle, out-of-bounds elements read as zero / are not written.
int make_tmap_nhwc_box_bf16(CUtensorMap* out, const void* base, int n, int h, int w, int c, long long pixel_stride,
                            uint32_t box_w, uint32_t box_h);
int make_tmap_im2col_bf16(CUtensorMap* out, const void* base, int n, int h, int w, int c, int pad_h, int pad_w,
                          int kh, int kw, int stride, int channels_per_pixel, int pixels_per_column,
                          long long stride_w = 0, long long stride_h = 0, long long stride_n = 0);

}  // namespace dcr
