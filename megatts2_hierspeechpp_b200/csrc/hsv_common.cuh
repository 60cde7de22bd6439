// Shared helpers for the hsv kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include "hsv.h"

#ifdef __CUDA_ARCH__
#if __CUDA_ARCH__ < 1000
#error "hsv kernels are written for sm_100a (Blackwell B200) only"
#endif
#endif

namespace hsv {

void set_error(const char *fmt, ...);

inline int check_launch(const char *what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return HSV_ERR_CUDA;
  }
  return HSV_OK;
}

#define HSV_REQUIRE(cond, ...)        \
  do {                                \
    if (!(cond)) {                    \
      hsv::set_error(__VA_ARGS__);    \
      return HSV_ERR_ARG;             \
    }                                 \
  } while (0)

// 12-tap kaiser-sinc filter, cutoff 0.25, half-width 0.3 (alias_free_torch/filter.py:28-57);
// fp32 values as stored in both bundled checkpoints (SURVEY.md §A.2).  Symmetric: f[j] == f[11-j].
#define HSV_F0 0.0020289647f
#define HSV_F1 0.0093894657f
#define HSV_F2 (-0.0255434588f)
#define HSV_F3 (-0.0576573834f)
#define HSV_F4 0.1285725832f
#define HSV_F5 0.4432097971f

__host__ __device__ inline int64_t blk16_rows(int64_t L) {
  return 2 * (int64_t)HSV_BLK_PAD + ((L + HSV_BLK_ROUND - 1) / HSV_BLK_ROUND) * HSV_BLK_ROUND;
}

// ---- tensor-core operand layout ("blk16" buffers) ----
// fp16 [B][C/CW][Lp][CW], CW = 64 / 32 / 16 channels per row (128 / 64 / 32-byte rows); the 16-byte units of a
// row are XOR-swizzled with the row index exactly as tcgen05's K-major SWIZZLE_128B / 64B / 32B shared-memory
// layouts expect (byte-offset bits [4,7) ^= bits [7,10) & mask), so that a span of rows that starts at a
// multiple of 8 rows, copied linearly (1-D bulk TMA) to a 1024-byte aligned shared address, IS the canonical
// swizzled operand tile.
__host__ __device__ inline int blk_cw(int C) { return (C % 64 == 0) ? 64 : ((C % 32 == 0) ? 32 : 16); }
// byte offset (within the whole tensor) of the 16-byte unit holding channels [c0, c0+8) of padded row r
__host__ __device__ inline int64_t blk_unit_offset(int cw, int64_t Lp, int C, int64_t b, int c0, int64_t r) {
  const int rowbytes = cw * 2;
  const int chunk = c0 / cw, u = (c0 - chunk * cw) >> 3;
  const int64_t base = (b * (C / cw) + chunk) * Lp * rowbytes;
  const uint64_t lin = (uint64_t)r * rowbytes + (uint64_t)u * 16;
  const uint64_t mask = (uint64_t)((cw >> 3) - 1);  // 7 / 3 / 1
  return base + (int64_t)(lin ^ (((lin >> 7) & mask) << 4));
}

inline cudaStream_t as_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }

// Programmatic dependent launch (PDL): a kernel launched with the attribute may start while its
// predecessor in the stream is still running; it must execute pdl_wait() before touching any memory
// the predecessor reads or writes.  Work that only depends on static data (weights, parameters,
// barrier/TMEM set-up) goes before the wait and overlaps the predecessor's tail.
extern int g_pdl;  // 0 = plain stream order (bring-up switch), 1 = PDL on the act/conv kernels
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// What the most recent host-side launch decision of a kernel family chose (hsv_last_launch_config, common.cu):
// [0] = the tcgen05 conv (conv_umma.cu), [1] = the fused activation (act1d.cu), [2] = attention (mha_mma.cu and the
// fp32 kernel of frame_ops.cu), [3] = the CUDA-core convs of conv_direct.cu.  Process-global bookkeeping, written just
// before the launch; it never changes what is launched.
constexpr int LAST_CONV_N = 15, LAST_ACT_N = 5, LAST_MHA_N = 13, LAST_DIRECT_N = 7;
extern int g_last_launch[4][16];
// family 2: kernel (0 tensor-core, 1 fp32 CUDA-core), D, out_mode, lens, valid_len, prescale, kv16 (16-byte K / V tile
// copies), q16 (16-byte Q tile copies), key tiles, grid x / y / z; then the running launch count
void note_mha_launch(int kernel, int D, int out_mode, int has_lens, int has_valid_len, int prescale, int kv16, int q16,
                     int key_tiles, dim3 grid);
// family 3: kernel (0 vecdot, 1 rowdot, 2 thin_vec, 3 thin_smem, 4 thin, 5 tiled, 6 ConvTranspose direct), flags (the
// ConvTranspose: HSV_CONV_ADD_OUT when it adds), valid_len given, grid x / y / z; then the running launch count
void note_direct_launch(int kernel, int flags, int has_valid_len, dim3 grid);

}  // namespace hsv
