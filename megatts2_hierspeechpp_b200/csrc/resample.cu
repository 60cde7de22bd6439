// The step BEFORE SpeechSR (inference_speechsr.py:28-34): torchaudio's kaiser-windowed sinc resampler
// (functional.resample(x, orig, new, resampling_method="kaiser_window")) of a ragged batch, one rate and one valid
// length per item, on the device.
//
// Item b has rate r with o : n = r : new (reduced), a filter table t[n][K], K = 2 width + o, and output
//   y[f n + p] = sum_{k < K} t[p][k] x[f o + k - width],   x = 0 outside [0, L_b)
// for the first n_out outputs (torchaudio's count, see the kernel).  The table is stored transposed, [K][n], so a
// warp's consecutive outputs (consecutive phases p of one frame) read consecutive table words; it stays in global
// memory (L2-resident, up to 1.2 MB per rate).
//
// A block computes 256 consecutive outputs of one item.  It stages the input window those outputs read -- whole frames,
// (f_hi - f_lo) o + K samples -- in shared memory, zero outside [0, L_b), so nothing past L_b is read.  Each output is
// summed by one thread in a fixed order (four interleaved fp32 FMA chains over k mod 4, then (a0 + a1) + (a2 + a3)),
// which depends on K alone: never on B, the padding, the tile or the item's position.
#include "hsv_common.cuh"

namespace {

constexpr int RS_THREADS = 256;      // outputs per block
constexpr int RS_MAX_DESC = 16;
constexpr int RS_MAX_WINDOW = 12288; // staged input samples per block (48 KB of shared memory)

struct RateDesc {
  int rate, o, n, width, K, offset;
};
struct RateSet {
  RateDesc d[RS_MAX_DESC];
  int count;
};

__device__ __forceinline__ float in_sample(const float *x, int64_t i) { return x[i]; }
// int16 PCM as torchaudio.load returns it: s / 32768, exact in fp32
__device__ __forceinline__ float in_sample(const int16_t *x, int64_t i) { return (float)x[i] * (1.0f / 32768.0f); }

template <typename TIn>
__global__ void __launch_bounds__(RS_THREADS)
    resample_kernel(const TIn *__restrict__ x, const int32_t *__restrict__ rate, const int32_t *__restrict__ valid_len,
                    const float *__restrict__ table, const RateSet rs, int new_freq, float *__restrict__ out,
                    int32_t *__restrict__ n_out, int64_t T, int64_t T_out) {
  extern __shared__ float xs[];
  const int b = blockIdx.y;
  const int r = __ldg(rate + b);
  RateDesc d = {0, 0, 0, 0, 0, 0};
  bool found = false;
#pragma unroll
  for (int i = 0; i < RS_MAX_DESC; ++i) {   // constant indices: the descriptor stays in registers
    if (i < rs.count && rs.d[i].rate == r) {
      d = rs.d[i];
      found = true;
    }
  }
  int64_t L = __ldg(valid_len + b);
  L = L < 0 ? 0 : (L > T ? T : L);
  const bool copy = found && r == new_freq;
  int64_t ne = 0;
  if (copy) {
    ne = L;
  } else if (found) {
    // torchaudio's count: ceil(torch.as_tensor(n * L / o)), i.e. the fp64 quotient rounded to fp32 (the default dtype),
    // capped at the (L / o + 1) n outputs its conv1d produces.  One below the exact ceiling for some L >= ~2^17.
    const int64_t c = (int64_t)ceilf(__double2float_rn((double)((int64_t)d.n * L) / (double)d.o));
    const int64_t full = (L / d.o + 1) * d.n;
    ne = c < full ? c : full;
  }
  ne = ne < T_out ? ne : T_out;
  if (blockIdx.x == 0 && threadIdx.x == 0) n_out[b] = (int32_t)ne;

  const TIn *xb = x + (int64_t)b * T;
  float *yb = out + (int64_t)b * T_out;
  const int64_t j0 = (int64_t)blockIdx.x * RS_THREADS;
  const int64_t j = j0 + threadIdx.x;
  if (copy || j0 >= ne) {   // block-uniform: bit-for-bit copy, or nothing but zeros
    if (j < T_out) yb[j] = j < ne ? in_sample(xb, j) : 0.f;
    return;
  }
  const int o = d.o, n = d.n, K = d.K;
  const int64_t j_last = (j0 + RS_THREADS < ne ? j0 + RS_THREADS : ne) - 1;
  const int64_t f_lo = j0 / n;
  const int64_t s0 = f_lo * o - d.width;
  const int win = (int)(j_last / n - f_lo) * o + K;
  for (int i = threadIdx.x; i < win; i += RS_THREADS) {
    const int64_t g = s0 + i;
    xs[i] = (g >= 0 && g < L) ? in_sample(xb, g) : 0.f;
  }
  __syncthreads();
  if (j >= T_out) return;
  if (j >= ne) {
    yb[j] = 0.f;
    return;
  }
  const int64_t f = j / n;
  const int p = (int)(j - f * n);
  const float *xp = xs + (int)(f - f_lo) * o;
  const float *tp = table + d.offset + p;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  int k = 0;
  for (; k + 4 <= K; k += 4) {
    a0 = fmaf(__ldg(tp + (k + 0) * n), xp[k + 0], a0);
    a1 = fmaf(__ldg(tp + (k + 1) * n), xp[k + 1], a1);
    a2 = fmaf(__ldg(tp + (k + 2) * n), xp[k + 2], a2);
    a3 = fmaf(__ldg(tp + (k + 3) * n), xp[k + 3], a3);
  }
  for (; k < K; ++k) a0 = fmaf(__ldg(tp + k * n), xp[k], a0);
  yb[j] = (a0 + a1) + (a2 + a3);
}

}  // namespace

extern "C" int hsv_resample_ragged(const void *x, int x_int16, const int32_t *rate, const int32_t *valid_len,
                                   const float *table, int64_t table_len, const int32_t *host_desc, int n_desc,
                                   int new_freq, float *out, int32_t *n_out, int B, int64_t T, int64_t T_out,
                                   void *stream) {
  HSV_REQUIRE(host_desc, "resample_ragged: null host_desc");
  HSV_REQUIRE(n_desc >= 1 && n_desc <= RS_MAX_DESC, "resample_ragged: n_desc = %d outside [1, %d]", n_desc,
              RS_MAX_DESC);
  HSV_REQUIRE(new_freq > 0, "resample_ragged: new_freq = %d", new_freq);
  HSV_REQUIRE(table_len >= 0 && (table || table_len == 0), "resample_ragged: null table");
  RateSet rs = {};
  rs.count = n_desc;
  int smem_floats = 0;
  for (int i = 0; i < n_desc; ++i) {
    const int32_t *s = host_desc + 6 * i;
    RateDesc d = {s[0], s[1], s[2], s[3], s[4], s[5]};
    HSV_REQUIRE(d.rate > 0, "resample_ragged: descriptor %d: rate %d", i, d.rate);
    for (int q = 0; q < i; ++q) HSV_REQUIRE(rs.d[q].rate != d.rate, "resample_ragged: rate %d listed twice", d.rate);
    if (d.rate == new_freq) {
      HSV_REQUIRE(d.o == 1 && d.n == 1 && d.width == 0 && d.K == 0,
                  "resample_ragged: descriptor %d: the copy entry (rate == new_freq) must be {rate, 1, 1, 0, 0, *}", i);
    } else {
      HSV_REQUIRE(d.o >= 1 && d.n >= 1 && d.width >= 1 && d.K == 2 * d.width + d.o,
                  "resample_ragged: descriptor %d: need o, n, width >= 1 and K == 2 width + o", i);
      HSV_REQUIRE(d.offset >= 0 && (int64_t)d.offset + (int64_t)d.K * d.n <= table_len,
                  "resample_ragged: descriptor %d: table [%d][%d] at %d outside the %lld-float table", i, d.K, d.n,
                  d.offset, (long long)table_len);
      const int64_t w = (int64_t)((RS_THREADS - 1) / d.n + 1) * d.o + d.K;
      HSV_REQUIRE(w <= RS_MAX_WINDOW, "resample_ragged: rate %d -> %d needs a %lld-sample window (max %d)", d.rate,
                  new_freq, (long long)w, RS_MAX_WINDOW);
      smem_floats = (int)w > smem_floats ? (int)w : smem_floats;
    }
    rs.d[i] = d;
  }
  HSV_REQUIRE(x_int16 == 0 || x_int16 == 1, "resample_ragged: x_int16 must be 0 or 1");
  HSV_REQUIRE(B >= 0 && B <= 65535 && T >= 1 && T <= INT32_MAX && T_out >= 1 && T_out <= INT32_MAX,
              "resample_ragged: bad shape B=%d T=%lld T_out=%lld", B, (long long)T, (long long)T_out);
  if (B == 0) return HSV_OK;
  HSV_REQUIRE(x && rate && valid_len && out && n_out, "resample_ragged: null pointer");
  const dim3 grid((unsigned)((T_out + RS_THREADS - 1) / RS_THREADS), (unsigned)B);
  const size_t smem = sizeof(float) * (size_t)smem_floats;
  cudaStream_t st = hsv::as_stream(stream);
  if (x_int16)
    resample_kernel<int16_t><<<grid, RS_THREADS, smem, st>>>(static_cast<const int16_t *>(x), rate, valid_len, table,
                                                             rs, new_freq, out, n_out, T, T_out);
  else
    resample_kernel<float><<<grid, RS_THREADS, smem, st>>>(static_cast<const float *>(x), rate, valid_len, table, rs,
                                                           new_freq, out, n_out, T, T_out);
  return hsv::check_launch("resample_ragged");
}
