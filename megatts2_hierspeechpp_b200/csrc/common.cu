// Error reporting, version and device probe of the hsv C-ABI.
#include <stdarg.h>
#include <string.h>
#include "hsv_common.cuh"

namespace hsv {
int g_pdl = 1;
static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
}  // namespace hsv

extern "C" int hsv_version(void) { return HSV_VERSION; }

// bring-up switch (not part of the drop-in contract): 0 disables programmatic dependent launch
extern "C" int hsv_set_pdl(int on) {
  hsv::g_pdl = on ? 1 : 0;
  return HSV_OK;
}

extern "C" const char *hsv_last_error(void) { return hsv::g_err; }

extern "C" int hsv_device_supported(void) {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  int major = 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return major == 10 ? 1 : 0;
}

extern "C" int64_t hsv_blk16_rows(int64_t L) { return hsv::blk16_rows(L); }

namespace hsv {
int g_last_launch[4][16] = {};

void note_mha_launch(int kernel, int D, int out_mode, int has_lens, int has_valid_len, int prescale, int kv16, int q16,
                     int key_tiles, dim3 grid) {
  const int v[LAST_MHA_N - 1] = {kernel, D, out_mode, has_lens, has_valid_len, prescale ? 1 : 0, kv16, q16, key_tiles,
                                 (int)grid.x, (int)grid.y, (int)grid.z};
  int *last = g_last_launch[2];
  for (int i = 0; i < LAST_MHA_N - 1; ++i) last[i] = v[i];
  ++last[LAST_MHA_N - 1];
}

void note_direct_launch(int kernel, int flags, int has_valid_len, dim3 grid) {
  const int v[LAST_DIRECT_N - 1] = {kernel, flags, has_valid_len, (int)grid.x, (int)grid.y, (int)grid.z};
  int *last = g_last_launch[3];
  for (int i = 0; i < LAST_DIRECT_N - 1; ++i) last[i] = v[i];
  ++last[LAST_DIRECT_N - 1];
}
}

extern "C" int hsv_last_launch_config(int family, int *out, int n) {
  HSV_REQUIRE(family >= 0 && family <= 3,
              "last_launch_config: family must be 0 (conv), 1 (activation), 2 (attention) or 3 (CUDA-core conv), got %d",
              family);
  HSV_REQUIRE(n >= 0 && (out || n == 0), "last_launch_config: null output");
  const int have_n[4] = {hsv::LAST_CONV_N, hsv::LAST_ACT_N, hsv::LAST_MHA_N, hsv::LAST_DIRECT_N};
  const int have = have_n[family];
  for (int i = 0; i < n && i < have; ++i) out[i] = hsv::g_last_launch[family][i];
  return have;
}
