// The step AFTER the waveform path (SURVEY.md §8f3): peak-normalise and quantise to int16 PCM on the device,
// so the device->host copy moves 2 bytes per sample instead of 4 and the host does no arithmetic.
//
// Replaces (reference, bit-exact in fp32 operation order):
//   inference_plm.py:183-188       audio / abs(audio).max() * 32767.0 * s         (s = 0.999 or the prompt's peak)
//   inference_speechsr.py:39-41    audio / abs(audio).max() * 0.999 * 32767.0
//   followed by .cpu().numpy().astype('int16')   (C cast: truncation toward zero)
#include "hsv_common.cuh"

namespace {

// max |x| per row.  Non-negative fp32 order == unsigned order of the bit patterns, so atomicMax on the bits is
// exact and order-independent; NaN has the largest pattern and therefore propagates like torch.max does.
__global__ void absmax_kernel(const float *__restrict__ x, unsigned int *__restrict__ peak_bits, int64_t L) {
  const int row = blockIdx.y;
  const float *xr = x + (int64_t)row * L;
  unsigned int m = 0u;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < L; i += (int64_t)gridDim.x * blockDim.x) {
    const unsigned int b = __float_as_uint(fabsf(xr[i]));
    m = b > m ? b : m;
  }
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned int t = __shfl_xor_sync(0xffffffffu, m, o);
    m = t > m ? t : m;
  }
  if ((threadIdx.x & 31) == 0 && m) atomicMax(peak_bits + row, m);
}

// ROW_S2: s2 = s2_row[row] (one prompt peak per utterance), else the scalar s2
template <bool ROW_S2>
__global__ void pcm16_kernel(const float *__restrict__ x, const unsigned int *__restrict__ peak_bits,
                             int16_t *__restrict__ out, int64_t L, int peak_stride, float s1, float s2,
                             const float *__restrict__ s2_row) {
  const int row = blockIdx.y;
  const float peak = __uint_as_float(peak_bits[row * peak_stride]);
  if (ROW_S2) s2 = __ldg(s2_row + row);
  const float *xr = x + (int64_t)row * L;
  int16_t *orow = out + (int64_t)row * L;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < L; i += (int64_t)gridDim.x * blockDim.x) {
    // IEEE division and two separately rounded multiplications, left to right, as the reference evaluates it
    const float v = __fmul_rn(__fmul_rn(__fdiv_rn(xr[i], peak), s1), s2);
    int q = (int)v;                      // truncation toward zero == numpy astype('int16') in range
    q = q > 32767 ? 32767 : (q < -32768 ? -32768 : q);
    orow[i] = (int16_t)q;
  }
}

__global__ void rowmax_kernel(unsigned int *peak_bits, int rows) {
  // global peak (the reference normalises the whole tensor): fold all rows into row 0
  unsigned int m = 0u;
  for (int i = threadIdx.x; i < rows; i += blockDim.x) m = peak_bits[i] > m ? peak_bits[i] : m;
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned int t = __shfl_xor_sync(0xffffffffu, m, o);
    m = t > m ? t : m;
  }
  if (threadIdx.x == 0) peak_bits[0] = m;
}

}  // namespace

static int peak_norm_pcm16(const float *x, int16_t *out, float *peak_ws, int rows, int64_t L, float s1, float s2,
                           const float *s2_row, int per_row, void *stream) {
  if (rows == 0 || L == 0) return HSV_OK;  // empty batch / sequence
  HSV_REQUIRE(x && out && peak_ws, "peak_norm_pcm16: null pointer");
  HSV_REQUIRE(rows > 0 && rows <= 65535 && L > 0, "peak_norm_pcm16: bad shape rows=%d L=%lld", rows, (long long)L);
  cudaStream_t st = hsv::as_stream(stream);
  unsigned int *bits = reinterpret_cast<unsigned int *>(peak_ws);
  cudaError_t e = cudaMemsetAsync(bits, 0, sizeof(unsigned int) * rows, st);
  if (e != cudaSuccess) {
    cudaGetLastError();
    hsv::set_error("peak_norm_pcm16: memset failed: %s", cudaGetErrorString(e));
    return HSV_ERR_CUDA;
  }
  int gx = (int)((L + 256 * 8 - 1) / (256 * 8));
  gx = gx < 1 ? 1 : (gx > 148 * 8 ? 148 * 8 : gx);
  absmax_kernel<<<dim3(gx, rows), 256, 0, st>>>(x, bits, L);
  if (!per_row && rows > 1) rowmax_kernel<<<1, 32, 0, st>>>(bits, rows);
  if (s2_row)
    pcm16_kernel<true><<<dim3(gx, rows), 256, 0, st>>>(x, bits, out, L, 1, s1, s2, s2_row);
  else
    pcm16_kernel<false><<<dim3(gx, rows), 256, 0, st>>>(x, bits, out, L, per_row ? 1 : 0, s1, s2, nullptr);
  return hsv::check_launch("peak_norm_pcm16");
}

extern "C" int hsv_peak_norm_pcm16(const float *x, int16_t *out, float *peak_ws, int rows, int64_t L, float s1,
                                   float s2, int per_row, void *stream) {
  return peak_norm_pcm16(x, out, peak_ws, rows, L, s1, s2, nullptr, per_row, stream);
}

extern "C" int hsv_peak_norm_pcm16_rows(const float *x, int16_t *out, float *peak_ws, int rows, int64_t L, float s1,
                                        const float *s2, void *stream) {
  HSV_REQUIRE(s2 || rows == 0 || L == 0, "peak_norm_pcm16_rows: null s2");
  return peak_norm_pcm16(x, out, peak_ws, rows, L, s1, 0.f, s2, 1, stream);
}
