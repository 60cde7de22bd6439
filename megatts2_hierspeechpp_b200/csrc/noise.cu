// Seeded Gaussian noise of the per-item synthesizer batches: each request carries its own 64-bit seed, and the noise
// at (item b, channel c, frame t) is a function of (seed[b], c, t) alone -- not of the batch size, the padded length,
// the item's position or length, or whether the launch is replayed from a CUDA graph.  So an item of a per-item batch
// draws exactly the noise of its own batch-1 call, and no host-side generator or [B, C, T] noise tensor is needed.
//
// Generator: Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC'11; the Random123
// constants), key = the seed's two 32-bit halves, counter = (t >> 2, c, draw, 0).  Its four output words become four
// normals by Box-Muller, frame t taking normal t & 3.  This is the project's own bit pattern, not torch's randn stream.
//   u(w)       = ((w >> 8) | 1) * 2^-24       odd multiples of 2^-24: exact in fp32 and strictly inside (0, 1)
//   n0, n1     = sqrt(-2 log u(w0)) * (cos, sin)(2 pi u(w1))
//   n2, n3     = sqrt(-2 log u(w2)) * (cos, sin)(2 pi u(w3))
// with logf, sqrtf and sincospif (|n| <= sqrt(48 ln 2) ~= 5.77).
#include "hsv_common.cuh"

namespace {

constexpr int NOISE_THREADS = 128;   // one thread per group of 4 frames of one (item, channel) row
constexpr uint32_t DRAW_SAMPLE = 0;  // draw id of the noise that multiplies exp(logs_p)

__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) {
      k0 += 0x9E3779B9u;
      k1 += 0xBB67AE85u;
    }
    const uint32_t lo0 = 0xD2511F53u * ctr.x, hi0 = __umulhi(0xD2511F53u, ctr.x);
    const uint32_t lo1 = 0xCD9E8D57u * ctr.z, hi1 = __umulhi(0xCD9E8D57u, ctr.z);
    ctr = make_uint4(hi1 ^ ctr.y ^ k0, lo1, hi0 ^ ctr.w ^ k1, lo0);
  }
  return ctr;
}

__device__ __forceinline__ float unit_open(uint32_t w) { return (float)((w >> 8) | 1u) * 0x1p-24f; }

// the four normals of frame group g (frames 4g .. 4g+3) of channel c under seed
__device__ __forceinline__ void seeded_normal4(uint64_t seed, int c, int64_t g, uint32_t draw, float n[4]) {
  const uint4 w = philox4x32_10(make_uint4((uint32_t)g, (uint32_t)c, draw, 0u), (uint32_t)seed, (uint32_t)(seed >> 32));
  float s0, c0, s1, c1;
  const float r0 = sqrtf(-2.0f * logf(unit_open(w.x)));
  sincospif(2.0f * unit_open(w.y), &s0, &c0);
  const float r1 = sqrtf(-2.0f * logf(unit_open(w.z)));
  sincospif(2.0f * unit_open(w.w), &s1, &c1);
  n[0] = r0 * c0;
  n[1] = r0 * s0;
  n[2] = r1 * c1;
  n[3] = r1 * s1;
}

__device__ __forceinline__ int64_t item_frames(const int32_t *vlen, int b, int64_t T) {
  if (!vlen) return T;
  const int64_t n = __ldg(vlen + b);
  return n < 0 ? 0 : (n > T ? T : n);
}

// out [B, C, T] = the seeded normals, 0 at t >= valid_len[b]
__global__ void __launch_bounds__(NOISE_THREADS) seeded_normal_kernel(const int64_t *__restrict__ seeds,
                                                                      float *__restrict__ out, int C, int64_t T,
                                                                      const int32_t *__restrict__ vlen) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, t0 = 4 * g;
  if (t0 >= T) return;
  const int c = blockIdx.y, b = blockIdx.z;
  const int64_t n = item_frames(vlen, b, T);
  float v[4] = {0.f, 0.f, 0.f, 0.f};
  if (t0 < n) seeded_normal4((uint64_t)__ldg(seeds + b), c, g, DRAW_SAMPLE, v);
  float *o = out + ((int64_t)b * C + c) * T;
#pragma unroll
  for (int j = 0; j < 4; ++j)
    if (t0 + j < T) o[t0 + j] = t0 + j < n ? v[j] : 0.f;
}

// z = (m + noise * exp(logs) * s[b]) past-length-masked, stats = [B, 2C, T] (m | logs).  SEEDED: the noise is generated
// here (seeded_normal_kernel's values, never stored); else it is read from eps [B, C, T].
template <bool SEEDED>
__global__ void __launch_bounds__(NOISE_THREADS) sample_kernel(const float *__restrict__ stats,
                                                               const float *__restrict__ eps,
                                                               const int64_t *__restrict__ seeds,
                                                               const float *__restrict__ s_vec, float s,
                                                               const int32_t *__restrict__ vlen, float *__restrict__ out,
                                                               int C, int64_t T) {
  const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, t0 = 4 * g;
  if (t0 >= T) return;
  const int c = blockIdx.y, b = blockIdx.z;
  const int64_t n = item_frames(vlen, b, T);
  const float sb = s_vec ? __ldg(s_vec + b) : s;
  float nz[4] = {0.f, 0.f, 0.f, 0.f};
  if (SEEDED && t0 < n) seeded_normal4((uint64_t)__ldg(seeds + b), c, g, DRAW_SAMPLE, nz);
  const float *m = stats + ((int64_t)b * 2 * C + c) * T, *lg = m + (int64_t)C * T;
  const int64_t row = ((int64_t)b * C + c) * T;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int64_t t = t0 + j;
    if (t >= T) break;
    float z = 0.f;
    if (t < n) {
      const float e = SEEDED ? nz[j] : __ldg(eps + row + t);
      // frame_op's OP_SAMPLE expression in its order, with expf (its mask is 1 here): the same bits
      z = __ldg(m + t) + (e * expf(__ldg(lg + t))) * sb;
    }
    out[row + t] = z;
  }
}

inline dim3 noise_grid(int B, int C, int64_t T) {
  const int64_t groups = (T + 3) / 4;
  return dim3((unsigned)((groups + NOISE_THREADS - 1) / NOISE_THREADS), (unsigned)C, (unsigned)B);
}

}  // namespace

// the frame group index is the counter's 32-bit word 0
#define HSV_NOISE_SHAPE_OK(B, C, T) ((B) > 0 && (B) <= 65535 && (C) > 0 && (C) <= 65535 && (T) > 0 && (T) <= ((int64_t)1 << 34))

extern "C" int hsv_seeded_normal(const int64_t *seeds, float *out, int B, int C, int64_t T, const int32_t *valid_len,
                                 void *stream) {
  if (B == 0 || C == 0 || T == 0) return HSV_OK;
  HSV_REQUIRE(seeds && out, "seeded_normal: null pointer");
  HSV_REQUIRE(HSV_NOISE_SHAPE_OK(B, C, T), "seeded_normal: bad shape B=%d C=%d T=%lld", B, C, (long long)T);
  seeded_normal_kernel<<<noise_grid(B, C, T), NOISE_THREADS, 0, hsv::as_stream(stream)>>>(seeds, out, C, T, valid_len);
  return hsv::check_launch("seeded_normal");
}

extern "C" int hsv_sample_ragged(const float *stats, const float *eps, const int64_t *seeds, const float *noise_scale,
                                 float s, const int32_t *valid_len, float *out, int B, int C, int64_t T, void *stream) {
  if (B == 0 || C == 0 || T == 0) return HSV_OK;
  HSV_REQUIRE(stats && out, "sample_ragged: null pointer");
  HSV_REQUIRE(!eps != !seeds, "sample_ragged: exactly one of eps and seeds");
  HSV_REQUIRE(HSV_NOISE_SHAPE_OK(B, C, T), "sample_ragged: bad shape B=%d C=%d T=%lld", B, C, (long long)T);
  const dim3 grid = noise_grid(B, C, T);
  cudaStream_t st = hsv::as_stream(stream);
  if (seeds)
    sample_kernel<true><<<grid, NOISE_THREADS, 0, st>>>(stats, nullptr, seeds, noise_scale, s, valid_len, out, C, T);
  else
    sample_kernel<false><<<grid, NOISE_THREADS, 0, st>>>(stats, eps, nullptr, noise_scale, s, valid_len, out, C, T);
  return hsv::check_launch("sample_ragged");
}
