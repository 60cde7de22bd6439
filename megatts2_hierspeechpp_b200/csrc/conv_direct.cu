// fp32 CUDA-core kernels for the small / odd-shaped ops of the path:
//   conv1d_direct            conv_pre, cond, proj, DBlock convs, conv_post(+tanh)
//   conv_transpose1d_direct  ups[i] as u polyphase stride-1 convs
//   sr_pre_interp            SpeechSR conv_pre (Cin=1) fused with the linear interpolation
//   nearest_gather, add3_bcast, weight_norm_fold, pack_blk16, interp_linear_table
// These carry < 6 % of the path's FLOPs (SURVEY.md §8a); the dense AMP convs run on tcgen05
// (conv_umma.cu).
#include "hsv_common.cuh"

namespace {

constexpr int CI = 8;        // input channels per shared-memory chunk
constexpr int KMAX = 16;     // max taps
constexpr int HALO_MAX = 64; // max (k-1)*d

// ------------------------------------------------------------------------------------------
// tiled conv1d: CTA = TCO out channels x TT time steps, thread = 4 co x 4 t
// ------------------------------------------------------------------------------------------
template <int TCO, int TT>
__global__ void __launch_bounds__((TCO / 4) * (TT / 4))
conv1d_tiled_kernel(const float *__restrict__ x, const float *__restrict__ w, const float *__restrict__ bias,
                    float *__restrict__ out, int Cin, int Cout, int64_t Lin, int64_t Lout, int k, int d,
                    int pad, int flags) {
  constexpr int NTHR = (TCO / 4) * (TT / 4);
  constexpr int LT = TT / 4;  // lanes along time
  __shared__ float x_s[CI][TT + HALO_MAX];
  __shared__ float w_s[CI * KMAX][TCO + 1];

  const int tid = threadIdx.x;
  const int tt = tid % LT, tco = tid / LT;
  const int64_t t0 = (int64_t)blockIdx.x * TT;
  const int co0 = blockIdx.y * TCO;
  const int b = blockIdx.z;
  const int span = TT + (k - 1) * d;

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int q = 0; q < 4; ++q) acc[i][q] = 0.f;

  for (int ci0 = 0; ci0 < Cin; ci0 += CI) {
    for (int idx = tid; idx < CI * span; idx += NTHR) {
      const int ci = idx / span, pp = idx - ci * span;
      const int64_t t = t0 - pad + pp;
      float v = 0.f;
      if (ci0 + ci < Cin && t >= 0 && t < Lin) {
        v = __ldg(x + ((int64_t)b * Cin + ci0 + ci) * Lin + t);
        if (flags & HSV_CONV_LRELU_IN) v = v > 0.f ? v : 0.1f * v;
        if (flags & HSV_CONV_LRELU001_IN) v = v > 0.f ? v : 0.01f * v;
        if (flags & HSV_CONV_SILU_IN) v = v / (1.f + expf(-v));
      }
      x_s[ci][pp] = v;
    }
    const int cik = CI * k;
    for (int idx = tid; idx < TCO * cik; idx += NTHR) {
      const int co = idx / cik, r = idx - co * cik;  // r = ci*k + j, contiguous in global
      const int ci = r / k;
      float v = 0.f;
      if (co0 + co < Cout && ci0 + ci < Cin) v = __ldg(w + ((int64_t)(co0 + co) * Cin + ci0) * k + r);
      w_s[r][co] = v;
    }
    __syncthreads();
#pragma unroll 1
    for (int ci = 0; ci < CI; ++ci) {
      for (int j = 0; j < k; ++j) {
        float wv[4], xv[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) wv[i] = w_s[ci * k + j][tco * 4 + i];
#pragma unroll
        for (int q = 0; q < 4; ++q) xv[q] = x_s[ci][tt + LT * q + j * d];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int q = 0; q < 4; ++q) acc[i][q] = fmaf(wv[i], xv[q], acc[i][q]);
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int co = co0 + tco * 4 + i;
    if (co >= Cout) continue;
    const float bv = bias ? __ldg(bias + co) : 0.f;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int64_t t = t0 + tt + LT * q;
      if (t >= Lout) continue;
      float v = acc[i][q] + bv;
      if (flags & HSV_CONV_TANH) v = tanhf(v);
      float *o = out + ((int64_t)b * Cout + co) * Lout + t;
      if (flags & HSV_CONV_ADD_OUT) v += *o;
      *o = v;
    }
  }
}

// One output of a very short sequence (cond(g): Lin == Lout == 1): one warp per output element, lanes split the
// Cin*k products, shuffle reduction.  xb = the batch item's [Cin] rows of stride ldx, of which [0, Lin) are read;
// every lane returns the sum, lane 0 stores out = epilogue(sum).
__device__ __forceinline__ void rowdot_out(const float *__restrict__ xb, const float *__restrict__ w,
                                           const float *__restrict__ bias, float *o, int Cin, int64_t ldx,
                                           int64_t Lin, int k, int d, int pad, int co, int64_t t, int flags,
                                           int lane) {
  float acc = 0.f;
  for (int r = lane; r < Cin * k; r += 32) {
    const int ci = r / k, j = r - ci * k;
    const int64_t ts = t - pad + (int64_t)j * d;
    if (ts >= 0 && ts < Lin) {
      float v = __ldg(xb + (int64_t)ci * ldx + ts);
      if (flags & HSV_CONV_LRELU_IN) v = v > 0.f ? v : 0.1f * v;
      if (flags & HSV_CONV_LRELU001_IN) v = v > 0.f ? v : 0.01f * v;
      if (flags & HSV_CONV_SILU_IN) v = v / (1.f + expf(-v));
      acc = fmaf(__ldg(w + (int64_t)co * Cin * k + r), v, acc);
    }
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) {
    if (bias) acc += __ldg(bias + co);
    if (flags & HSV_CONV_TANH) acc = tanhf(acc);
    if (flags & HSV_CONV_ADD_OUT) acc += *o;
    *o = acc;
  }
}

// Ragged batch item of the thin kernels (Lout == Lin, pad 3, k 7): valid length of item b, clamped to [0, Lin).
__device__ __forceinline__ int64_t thin_valid_len(const int32_t *valid_len, int b, int64_t Lin) {
  if (!valid_len) return Lin;
  const int v = __ldg(valid_len + b);
  return v < 0 ? 0 : (v > Lin ? Lin : v);
}

// An item of at most 8 valid steps is computed the way hsv_conv1d_direct computes it alone (Lout <= 8: the warp
// reduction above, a different summation order from the thin kernels), so it stays bit-identical to its own run.
// CTA 0 of the item computes the Lv * Cout outputs, every CTA zeroes its part of [Lv, Lout).
__device__ __forceinline__ void thin_short_item(const float *__restrict__ x, const float *__restrict__ w,
                                                const float *__restrict__ bias, float *__restrict__ out, int b, int Cin, int Cout, int64_t Lin,
                                                int64_t Lv, int flags, int64_t t0, int TT) {
  const int lane = threadIdx.x & 31, nw = blockDim.x >> 5, wid = threadIdx.x >> 5;
  if (blockIdx.x == 0) {
    for (int q = wid; q < Cout * (int)Lv; q += nw) {
      const int co = q / (int)Lv, t = q - co * (int)Lv;
      rowdot_out(x + (int64_t)b * Cin * Lin, w, bias, out + ((int64_t)b * Cout + co) * Lin + t, Cin, Lin, Lv, 7, 1,
                 3, co, t, flags, lane);
    }
  }
  for (int q = threadIdx.x; q < Cout * TT; q += blockDim.x) {
    const int co = q / TT;
    const int64_t t = t0 + (q - co * TT);
    if (t >= Lv && t < Lin) out[((int64_t)b * Cout + co) * Lin + t] = 0.f;
  }
}

// thin conv for Cout <= 4 and d == 1 (conv_post 16|32|64 -> 1, k=7).  CTA = TT consecutive outputs of one batch
// row: the input window of CC channels is staged in shared memory with coalesced, independent loads (the previous
// version walked the channels serially from global memory: 20 us for the [16,160000] conv_post of the batch-1
// vocoder, a dependent-load chain), then every thread produces 2 outputs per output channel from a register window
// of K+1 samples per input channel.  Accumulation order (ci outer, tap inner, fmaf) as before.
// valid_len (K == 7, Lout == Lin only): item b reads x[t < Lv] (the rest as 0) and writes 0 at t >= Lv.
template <int K>
struct ThinSmem {
  static constexpr int TT = 512, CC = 16, W = TT + K - 1, WP = (W + 3) & ~3;
};

// body of conv1d_thin_smem_kernel, inlined with valid_len == nullptr (the full-length path, constant-folded) and without
template <int K>
__device__ __forceinline__ void thin_smem_body(float (*__restrict__ xs)[ThinSmem<K>::WP], float (*__restrict__ ws)[16 * K],
                                               const float *__restrict__ x, const float *__restrict__ w,
                                               const float *__restrict__ bias, float *__restrict__ out,
                                               const int32_t *__restrict__ valid_len, int Cin, int Cout, int64_t Lin,
                                               int64_t Lout, int pad, int flags) {
  constexpr int TT = ThinSmem<K>::TT, CC = ThinSmem<K>::CC, W = ThinSmem<K>::W;
  const int tid = threadIdx.x;
  const int b = blockIdx.y;
  const int64_t t0 = (int64_t)blockIdx.x * TT;
  const int64_t Lv = thin_valid_len(valid_len, b, Lin);
  if (valid_len && Lv <= 8) {
    thin_short_item(x, w, bias, out, b, Cin, Cout, Lin, Lv, flags, t0, TT);
    return;
  }
  float acc[4][2];
#pragma unroll
  for (int co = 0; co < 4; ++co) acc[co][0] = acc[co][1] = 0.f;
  for (int c0 = 0; c0 < Cin; c0 += CC) {
    const int nc = min(CC, Cin - c0);
    if (c0) __syncthreads();
    // all loads of a batch are issued before the first store (independent L2 round trips, not a chain)
    constexpr int NB = 11;
    for (int i0 = tid; i0 < nc * W; i0 += 256 * NB) {
      float v[NB];
#pragma unroll
      for (int q = 0; q < NB; ++q) {
        const int idx = i0 + 256 * q;
        const int c = idx / W, pp = idx - c * W;
        const int64_t ts = t0 - pad + pp;
        v[q] = (idx < nc * W && ts >= 0 && ts < Lv) ? __ldg(x + ((int64_t)b * Cin + c0 + c) * Lin + ts) : 0.f;
      }
#pragma unroll
      for (int q = 0; q < NB; ++q) {
        const int idx = i0 + 256 * q;
        const int c = idx / W, pp = idx - c * W;
        float u = v[q];
        if (flags & HSV_CONV_LRELU_IN) u = u > 0.f ? u : 0.1f * u;
        if (flags & HSV_CONV_LRELU001_IN) u = u > 0.f ? u : 0.01f * u;
        if (flags & HSV_CONV_SILU_IN) u = u / (1.f + expf(-u));
        if (idx < nc * W) xs[c][pp] = u;
      }
    }
    for (int idx = tid; idx < Cout * nc * K; idx += 256) {
      const int co = idx / (nc * K), r = idx - co * (nc * K);
      ws[co][r] = __ldg(w + ((int64_t)co * Cin + c0) * K + r);
    }
    __syncthreads();
    for (int c = 0; c < nc; ++c) {
      float xv[K + 1];
#pragma unroll
      for (int j = 0; j < K + 1; j += 2) {
        const float2 v2 = *reinterpret_cast<const float2 *>(&xs[c][2 * tid + j]);
        xv[j] = v2.x;
        if (j + 1 < K + 1) xv[j + 1] = v2.y;
      }
#pragma unroll
      for (int co = 0; co < 4; ++co) {
        if (co < Cout) {
#pragma unroll
          for (int j = 0; j < K; ++j) {
            const float wj = ws[co][c * K + j];
            acc[co][0] = fmaf(wj, xv[j], acc[co][0]);
            acc[co][1] = fmaf(wj, xv[j + 1], acc[co][1]);
          }
        }
      }
    }
  }
#pragma unroll
  for (int co = 0; co < 4; ++co) {
    if (co >= Cout) break;
    const float bv = bias ? __ldg(bias + co) : 0.f;
    float *o = out + ((int64_t)b * Cout + co) * Lout + t0 + 2 * tid;
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      if (t0 + 2 * tid + r < Lout) {
        float v = acc[co][r] + bv;
        if (flags & HSV_CONV_TANH) v = tanhf(v);
        if (flags & HSV_CONV_ADD_OUT) v += o[r];
        o[r] = valid_len && t0 + 2 * tid + r >= Lv ? 0.f : v;
      }
    }
  }
}

template <int K>
__global__ void __launch_bounds__(256) conv1d_thin_smem_kernel(const float *__restrict__ x, const float *__restrict__ w,
                                                               const float *__restrict__ bias, float *__restrict__ out,
                                                               const int32_t *__restrict__ valid_len, int Cin,
                                                               int Cout, int64_t Lin, int64_t Lout, int pad,
                                                               int flags) {
  __shared__ __align__(16) float xs[ThinSmem<K>::CC][ThinSmem<K>::WP];
  __shared__ float ws[4][ThinSmem<K>::CC * K];
  if (valid_len)
    thin_smem_body<K>(xs, ws, x, w, bias, out, valid_len, Cin, Cout, Lin, Lout, pad, flags);
  else
    thin_smem_body<K>(xs, ws, x, w, bias, out, nullptr, Cin, Cout, Lin, Lout, pad, flags);
}

// The same for 16-byte aligned tensors with Lin % 4 == 0 and pad == 3 (every conv_post of the path): the window is staged with
// float4 loads from t0 - 4 (a float4 is entirely inside or outside [0, Lin)), one warp per channel row, no index
// division; every thread produces 4 outputs per output channel from three LDS.128 of inputs and two of weights per input
// channel.  SpeechSR48 conv_post at batch 16 ([16,32,480000]): 577 us (scalar staging) / 364 us (the round-1 kernel) -> see
// DESIGN.md §4; ~224 FMAs per output make it FMA-issue-bound once the staging is out of the way.
// valid_len: as conv1d_thin_smem_kernel, except that a float4 straddling Lv is loaded whole and its lanes >= Lv are
// zeroed in shared memory before use.
constexpr int THIN_VEC_WP = 4 * (512 / 4 + 2);   // window = [t0 - 4, t0 + TT + 4)

// body of conv1d_thin_vec_kernel, inlined with valid_len == nullptr (the full-length path, constant-folded) and without
__device__ __forceinline__ void thin_vec_body(float (*__restrict__ xs)[THIN_VEC_WP], float (*__restrict__ ws)[16][8],
                                              const float *__restrict__ x, const float *__restrict__ w,
                                              const float *__restrict__ bias, float *__restrict__ out,
                                              const int32_t *__restrict__ valid_len, int Cin, int Cout, int64_t Lin,
                                              int64_t Lout, int flags) {
  constexpr int K = 7, TT = 512, CC = 16, W4 = TT / 4 + 2;
  const int tid = threadIdx.x, lane = tid & 31, wrp = tid >> 5;
  const int b = blockIdx.y;
  const int64_t t0 = (int64_t)blockIdx.x * TT;
  const int64_t Lv = thin_valid_len(valid_len, b, Lin);
  if (valid_len && Lv <= 8) {
    thin_short_item(x, w, bias, out, b, Cin, Cout, Lin, Lv, flags, t0, TT);
    return;
  }
  // window float4 that straddles Lv (-1: none; Lin % 4 == 0, so only a ragged item has one)
  const int p4v = valid_len && (Lv & 3) && Lv > t0 - 4 && Lv < t0 + TT + 4 ? (int)((Lv - (t0 - 4)) >> 2) : -1;
  float acc[4][4];
#pragma unroll
  for (int co = 0; co < 4; ++co) acc[co][0] = acc[co][1] = acc[co][2] = acc[co][3] = 0.f;
  for (int c0 = 0; c0 < Cin; c0 += CC) {
    const int nc = min(CC, Cin - c0);
    if (c0) __syncthreads();
    // ---- staging: warp wrp takes channels wrp, wrp + 4, ...; lane takes float4s lane, lane + 32, ... ----
    float4 v[(CC / 4) * 5];
#pragma unroll
    for (int cc = 0; cc < CC / 4; ++cc) {
      const int c = wrp + 4 * cc;
      const float *row = x + ((int64_t)b * Cin + c0 + c) * Lin + (t0 - 4);
#pragma unroll
      for (int i = 0; i < 5; ++i) {
        const int p4 = lane + 32 * i;
        const int64_t ts = t0 - 4 + 4 * (int64_t)p4;
        v[cc * 5 + i] = (c < nc && p4 < W4 && ts >= 0 && ts < Lv) ? __ldg(reinterpret_cast<const float4 *>(row) + p4)
                                                                   : make_float4(0.f, 0.f, 0.f, 0.f);
      }
    }
#pragma unroll
    for (int cc = 0; cc < CC / 4; ++cc) {
      const int c = wrp + 4 * cc;
#pragma unroll
      for (int i = 0; i < 5; ++i) {
        const int p4 = lane + 32 * i;
        float4 u = v[cc * 5 + i];
        if (flags & (HSV_CONV_LRELU_IN | HSV_CONV_LRELU001_IN | HSV_CONV_SILU_IN)) {
          float *e = reinterpret_cast<float *>(&u);
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            if (flags & HSV_CONV_LRELU_IN) e[q] = e[q] > 0.f ? e[q] : 0.1f * e[q];
            if (flags & HSV_CONV_LRELU001_IN) e[q] = e[q] > 0.f ? e[q] : 0.01f * e[q];
            if (flags & HSV_CONV_SILU_IN) e[q] = e[q] / (1.f + expf(-e[q]));
          }
        }
        if (c < nc && p4 < W4) *reinterpret_cast<float4 *>(&xs[c][4 * p4]) = u;
      }
    }
    if (p4v >= 0 && (p4v & 31) == lane) {
      // the float4 that straddles Lv was staged by this thread: zero its steps >= Lv
#pragma unroll
      for (int cc = 0; cc < CC / 4; ++cc)
        if (wrp + 4 * cc < nc)
          for (int q = (int)(Lv & 3); q < 4; ++q) xs[wrp + 4 * cc][4 * p4v + q] = 0.f;
    }
    for (int idx = tid; idx < 4 * CC * 8; idx += 128) {
      const int co = idx / (CC * 8), r = idx - co * (CC * 8), c = r >> 3, j = r & 7;
      ws[co][c][j] = (co < Cout && c < nc && j < K) ? __ldg(w + ((int64_t)co * Cin + c0 + c) * K + j) : 0.f;
    }
    __syncthreads();
    // ---- outputs o = 4 tid .. 4 tid + 3: input index (window-relative) o + 1 + j ----
    for (int c = 0; c < nc; ++c) {
      float xv[12];
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        const float4 a = *reinterpret_cast<const float4 *>(&xs[c][4 * tid + 4 * q]);
        xv[4 * q] = a.x; xv[4 * q + 1] = a.y; xv[4 * q + 2] = a.z; xv[4 * q + 3] = a.w;
      }
#pragma unroll
      for (int co = 0; co < 4; ++co) {
        if (co < Cout) {
          const float4 w0 = *reinterpret_cast<const float4 *>(&ws[co][c][0]);
          const float4 w1 = *reinterpret_cast<const float4 *>(&ws[co][c][4]);
          const float wj[7] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z};
#pragma unroll
          for (int j = 0; j < K; ++j)
#pragma unroll
            for (int r = 0; r < 4; ++r) acc[co][r] = fmaf(wj[j], xv[r + 1 + j], acc[co][r]);
        }
      }
    }
  }
#pragma unroll
  for (int co = 0; co < 4; ++co) {
    if (co >= Cout) break;
    const float bv = bias ? __ldg(bias + co) : 0.f;
    const int64_t t = t0 + 4 * tid;
    if (t >= Lout) continue;
    float *o = out + ((int64_t)b * Cout + co) * Lout + t;    // Lout == Lin: % 4 == 0, 16-byte aligned
    float4 r4 = make_float4(acc[co][0] + bv, acc[co][1] + bv, acc[co][2] + bv, acc[co][3] + bv);
    if (flags & HSV_CONV_TANH) {
      r4.x = tanhf(r4.x); r4.y = tanhf(r4.y); r4.z = tanhf(r4.z); r4.w = tanhf(r4.w);
    }
    if (flags & HSV_CONV_ADD_OUT) {
      const float4 prev = *reinterpret_cast<const float4 *>(o);
      r4.x += prev.x; r4.y += prev.y; r4.z += prev.z; r4.w += prev.w;
    }
    if (valid_len && t + 4 > Lv) {
      r4.x = t < Lv ? r4.x : 0.f;
      r4.y = t + 1 < Lv ? r4.y : 0.f;
      r4.z = t + 2 < Lv ? r4.z : 0.f;
      r4.w = t + 3 < Lv ? r4.w : 0.f;
    }
    *reinterpret_cast<float4 *>(o) = r4;
  }
}

__global__ void __launch_bounds__(128) conv1d_thin_vec_kernel(const float *__restrict__ x, const float *__restrict__ w,
                                                              const float *__restrict__ bias, float *__restrict__ out,
                                                              const int32_t *__restrict__ valid_len, int Cin,
                                                              int Cout, int64_t Lin, int64_t Lout, int flags) {
  __shared__ __align__(16) float xs[16][THIN_VEC_WP];
  __shared__ __align__(16) float ws[4][16][8];
  if (valid_len)
    thin_vec_body(xs, ws, x, w, bias, out, valid_len, Cin, Cout, Lin, Lout, flags);
  else
    thin_vec_body(xs, ws, x, w, bias, out, nullptr, Cin, Cout, Lin, Lout, flags);
}

// generic thin conv (any k, d): one thread per (b, t)
__global__ void conv1d_thin_kernel(const float *__restrict__ x, const float *__restrict__ w,
                                   const float *__restrict__ bias, float *__restrict__ out, int B, int Cin,
                                   int Cout, int64_t Lin, int64_t Lout, int k, int d, int pad, int flags) {
  const int64_t n = (int64_t)B * Lout;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(i / Lout);
    const int64_t t = i - (int64_t)b * Lout;
    for (int co = 0; co < Cout; ++co) {
      float acc = 0.f;
      for (int ci = 0; ci < Cin; ++ci) {
        const float *xr = x + ((int64_t)b * Cin + ci) * Lin;
        const float *wr = w + ((int64_t)co * Cin + ci) * k;
        for (int j = 0; j < k; ++j) {
          const int64_t ts = t - pad + (int64_t)j * d;
          if (ts >= 0 && ts < Lin) {
            float v = __ldg(xr + ts);
            if (flags & HSV_CONV_LRELU_IN) v = v > 0.f ? v : 0.1f * v;
            if (flags & HSV_CONV_LRELU001_IN) v = v > 0.f ? v : 0.01f * v;
            if (flags & HSV_CONV_SILU_IN) v = v / (1.f + expf(-v));
            acc = fmaf(__ldg(wr + j), v, acc);
          }
        }
      }
      if (bias) acc += __ldg(bias + co);
      if (flags & HSV_CONV_TANH) acc = tanhf(acc);
      float *o = out + ((int64_t)b * Cout + co) * Lout + t;
      if (flags & HSV_CONV_ADD_OUT) acc += *o;
      *o = acc;
    }
  }
}

// very short sequences (cond(g): Lin == Lout == 1): see rowdot_out
__global__ void conv1d_rowdot_kernel(const float *__restrict__ x, const float *__restrict__ w,
                                     const float *__restrict__ bias, float *__restrict__ out, int B, int Cin,
                                     int Cout, int64_t Lin, int64_t Lout, int k, int d, int pad, int flags) {
  const int lane = threadIdx.x & 31;
  const int64_t nout = (int64_t)B * Cout * Lout;
  const int64_t wid = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (wid >= nout) return;
  const int64_t t = wid % Lout;
  const int co = (int)((wid / Lout) % Cout);
  const int b = (int)(wid / (Lout * Cout));
  rowdot_out(x + (int64_t)b * Cin * Lin, w, bias, out + ((int64_t)b * Cout + co) * Lout + t, Cin, Lin, Lin, k, d, pad,
             co, t, flags, lane);
}

// the same for a per-utterance vector (k == 1, Lin == Lout == 1, Cin % 4 == 0: cond(g), adaLN, cond_layer): float4
// loads, all of a lane's weight loads issued before the first FMA (the scalar loop above is a chain of dependent
// DRAM round trips when the weights are cold: 9 us for 512 x 256)
__global__ void conv1d_vecdot_kernel(const float *__restrict__ x, const float *__restrict__ w,
                                     const float *__restrict__ bias, float *__restrict__ out, int B, int Cin,
                                     int Cout, int flags) {
  const int lane = threadIdx.x & 31;
  const int64_t wid = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
  if (wid >= (int64_t)B * Cout) return;
  const int co = (int)(wid % Cout);
  const int b = (int)(wid / Cout);
  const float4 *w4 = reinterpret_cast<const float4 *>(w + (int64_t)co * Cin);
  const float4 *x4 = reinterpret_cast<const float4 *>(x + (int64_t)b * Cin);
  const int n4 = Cin >> 2;
  float acc = 0.f;
  for (int r0 = lane; r0 < n4; r0 += 128) {
    float4 wv[4], xv[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int r = r0 + 32 * q;
      wv[q] = r < n4 ? __ldg(w4 + r) : make_float4(0.f, 0.f, 0.f, 0.f);
      xv[q] = r < n4 ? __ldg(x4 + r) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float v[4] = {xv[q].x, xv[q].y, xv[q].z, xv[q].w};
      const float ww[4] = {wv[q].x, wv[q].y, wv[q].z, wv[q].w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        if (flags & HSV_CONV_LRELU_IN) v[e] = v[e] > 0.f ? v[e] : 0.1f * v[e];
        if (flags & HSV_CONV_LRELU001_IN) v[e] = v[e] > 0.f ? v[e] : 0.01f * v[e];
        if (flags & HSV_CONV_SILU_IN) v[e] = v[e] / (1.f + expf(-v[e]));
        acc = fmaf(ww[e], v[e], acc);
      }
    }
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) {
    if (bias) acc += __ldg(bias + co);
    if (flags & HSV_CONV_TANH) acc = tanhf(acc);
    float *o = out + (int64_t)b * Cout + co;
    if (flags & HSV_CONV_ADD_OUT) acc += *o;
    *o = acc;
  }
}

// ------------------------------------------------------------------------------------------
// ConvTranspose1d, polyphase: output phase rho = o mod u is a stride-1 conv over the input rows
//   o = u*q + rho,  r = (rho+p) mod u,  c = (rho+p) div u,  taps j = r + i*u reading x[q + c - i]
// ------------------------------------------------------------------------------------------
template <int TCO, int TT>
__global__ void __launch_bounds__((TCO / 4) * (TT / 4))
conv_transpose1d_kernel(const float *__restrict__ x, const float *__restrict__ w,
                        const float *__restrict__ bias, const float *__restrict__ add,
                        float *__restrict__ out, int Cin, int Cout, int64_t Lin, int k, int u, int nco_tiles) {
  constexpr int NTHR = (TCO / 4) * (TT / 4);
  constexpr int LT = TT / 4;
  constexpr int XH = 8;  // taps per phase <= ceil(k/u) <= 4; window halo
  __shared__ float x_s[CI][TT + 2 * XH];
  __shared__ float w_s[CI * 4][TCO + 1];

  const int tid = threadIdx.x;
  const int tt = tid % LT, tco = tid / LT;
  const int64_t q0 = (int64_t)blockIdx.x * TT;
  const int rho = blockIdx.y / nco_tiles;
  const int co0 = (blockIdx.y % nco_tiles) * TCO;
  const int b = blockIdx.z;
  const int p = (k - u) / 2;
  const int r = (rho + p) % u, c = (rho + p) / u;
  const int ntaps = (k - r + u - 1) / u;  // taps j = r + i*u < k
  const int64_t Lout = (int64_t)u * Lin;

  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int qq = 0; qq < 4; ++qq) acc[i][qq] = 0.f;

  for (int ci0 = 0; ci0 < Cin; ci0 += CI) {
    // x_s[ci][pp] = x[q0 - XH + pp]
    for (int idx = tid; idx < CI * (TT + 2 * XH); idx += NTHR) {
      const int ci = idx / (TT + 2 * XH), pp = idx - ci * (TT + 2 * XH);
      const int64_t t = q0 - XH + pp;
      float v = 0.f;
      if (ci0 + ci < Cin && t >= 0 && t < Lin) v = __ldg(x + ((int64_t)b * Cin + ci0 + ci) * Lin + t);
      x_s[ci][pp] = v;
    }
    // w_s[ci*ntaps + i][co] = W[ci0+ci][co0+co][r + i*u]      (W is [Cin, Cout, k])
    for (int idx = tid; idx < CI * ntaps * TCO; idx += NTHR) {
      const int i = idx % ntaps;
      const int co = (idx / ntaps) % TCO;
      const int ci = idx / (ntaps * TCO);
      float v = 0.f;
      if (ci0 + ci < Cin && co0 + co < Cout)
        v = __ldg(w + ((int64_t)(ci0 + ci) * Cout + co0 + co) * k + r + i * u);
      w_s[ci * ntaps + i][co] = v;
    }
    __syncthreads();
#pragma unroll 1
    for (int ci = 0; ci < CI; ++ci) {
      for (int i = 0; i < ntaps; ++i) {
        float wv[4], xv[4];
#pragma unroll
        for (int ii = 0; ii < 4; ++ii) wv[ii] = w_s[ci * ntaps + i][tco * 4 + ii];
#pragma unroll
        for (int qq = 0; qq < 4; ++qq) xv[qq] = x_s[ci][XH + tt + LT * qq + c - i];
#pragma unroll
        for (int ii = 0; ii < 4; ++ii)
#pragma unroll
          for (int qq = 0; qq < 4; ++qq) acc[ii][qq] = fmaf(wv[ii], xv[qq], acc[ii][qq]);
      }
    }
    __syncthreads();
  }
#pragma unroll
  for (int ii = 0; ii < 4; ++ii) {
    const int co = co0 + tco * 4 + ii;
    if (co >= Cout) continue;
    const float bv = bias ? __ldg(bias + co) : 0.f;
#pragma unroll
    for (int qq = 0; qq < 4; ++qq) {
      const int64_t q = q0 + tt + LT * qq;
      if (q >= Lin) continue;
      const int64_t off = ((int64_t)b * Cout + co) * Lout + q * u + rho;
      float v = acc[ii][qq] + bv;
      if (add) v += __ldg(add + off);
      out[off] = v;
    }
  }
}

// ------------------------------------------------------------------------------------------
// SpeechSR front: conv_pre (Cin=1,k=7,pad=3) + linear interpolation (align_corners=False)
// ATen upsample_linear1d (CUDA): src = scale*(dst+0.5)-0.5 clamped at 0, evaluated in fp32 with
// nvcc's default contraction (one FMA);  out = (1-lam)*v[i0] + lam*v[i1].
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void lin_src(int64_t dst, float scale, int64_t Lin, int &i0, int &i1, float &lam) {
  float src = __fmaf_rn(scale, (float)dst + 0.5f, -0.5f);
  src = src < 0.f ? 0.f : src;
  int a = (int)src;
  if (a > Lin - 1) a = (int)(Lin - 1);
  i0 = a;
  i1 = a + (a < Lin - 1 ? 1 : 0);
  lam = src - (float)a;
}

// vl_in / vl_out (nullable): per-item valid lengths; item b is then interpolated from Lin_b to Lout_b samples (its
// own scale, bit-identical to a call with Lin = Lin_b, Lout = Lout_b) and its outputs at t >= Lout_b are 0.
__global__ void sr_pre_interp_kernel(const float *__restrict__ x, const float *__restrict__ w,
                                     const float *__restrict__ bias, float *__restrict__ out,
                                     const int32_t *__restrict__ vl_in, const int32_t *__restrict__ vl_out, int B,
                                     int C, int64_t Lin, int64_t Lout, float scale) {
  const int64_t n = (int64_t)B * Lout;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(i / Lout);
    const int64_t t = i - (int64_t)b * Lout;
    const float *xr = x + (int64_t)b * Lin;
    int64_t Li = Lin;
    float sc = scale;
    if (vl_in || vl_out) {
      const int vi = vl_in ? __ldg(vl_in + b) : (int)Lin, vo = vl_out ? __ldg(vl_out + b) : (int)Lout;
      Li = vi < 0 ? 0 : (vi > Lin ? Lin : vi);
      const int64_t Lo = vo < 0 ? 0 : (vo > Lout ? Lout : vo);
      if (t >= Lo || Li == 0) {
        for (int c = 0; c < C; ++c) out[((int64_t)b * C + c) * Lout + t] = 0.f;
        continue;
      }
      sc = (float)Li / (float)Lo;
    }
    int i0, i1;
    float lam;
    lin_src(t, sc, Li, i0, i1, lam);
    float xa[7], xb[7];
#pragma unroll
    for (int j = 0; j < 7; ++j) {
      const int64_t ta = (int64_t)i0 - 3 + j, tb = (int64_t)i1 - 3 + j;
      xa[j] = (ta >= 0 && ta < Li) ? __ldg(xr + ta) : 0.f;
      xb[j] = (tb >= 0 && tb < Li) ? __ldg(xr + tb) : 0.f;
    }
    const float w0 = 1.0f - lam, w1 = lam;
    for (int c = 0; c < C; ++c) {
      float va = 0.f, vb = 0.f;
#pragma unroll
      for (int j = 0; j < 7; ++j) {
        const float wj = __ldg(w + c * 7 + j);
        va = fmaf(wj, xa[j], va);
        vb = fmaf(wj, xb[j], vb);
      }
      const float bv = bias ? __ldg(bias + c) : 0.f;
      va += bv;
      vb += bv;
      out[((int64_t)b * C + c) * Lout + t] = w0 * va + w1 * vb;
    }
  }
}

// Streaming windows: item b is the window x[b, :vl_in[b]] of a longer stream, starting at the stream's input sample
// org[b].in and output sample org[b].out.  Output t of the window is the stream's output org.out + t: i0 / i1 / lambda
// come from that global index and the stream's constant scale (down / up, which is what (float)L / (float)Lout rounds
// to for every L the stream accepts), the Lin - 1 clamp uses the stream's total length org[b].total only when it is
// known (>= 0, the stream's last window), and conv_pre taps outside the window read 0.  Where every tap of an output
// lies inside the window (or at the stream's own edges), it equals the full-length kernel on the whole stream.
struct StreamOrigin {
  int64_t in, out, total;
};
static_assert(sizeof(StreamOrigin) == 3 * sizeof(int64_t), "origin rows are int64 [B, 3]");

__global__ void sr_pre_interp_stream_kernel(const float *__restrict__ x, const float *__restrict__ w,
                                            const float *__restrict__ bias, float *__restrict__ out,
                                            const int32_t *__restrict__ vl_in, const int32_t *__restrict__ vl_out,
                                            const StreamOrigin *__restrict__ org, int B, int C, int64_t Lin,
                                            int64_t Lout, float scale) {
  const int64_t n = (int64_t)B * Lout;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int b = (int)(i / Lout);
    const int64_t t = i - (int64_t)b * Lout;
    const int vi = __ldg(vl_in + b), vo = __ldg(vl_out + b);
    const int64_t Li = vi < 0 ? 0 : (vi > Lin ? Lin : vi);
    const int64_t Lo = vo < 0 ? 0 : (vo > Lout ? Lout : vo);
    if (t >= Lo || Li == 0) {
      for (int c = 0; c < C; ++c) out[((int64_t)b * C + c) * Lout + t] = 0.f;
      continue;
    }
    const StreamOrigin o = org[b];
    int i0, i1;
    float lam;
    lin_src(o.out + t, scale, o.total >= 0 ? o.total : INT64_MAX, i0, i1, lam);
    const float *xr = x + (int64_t)b * Lin;
    float xa[7], xb[7];
#pragma unroll
    for (int j = 0; j < 7; ++j) {
      const int64_t ta = (int64_t)i0 - 3 + j - o.in, tb = (int64_t)i1 - 3 + j - o.in;   // window-relative taps
      xa[j] = (ta >= 0 && ta < Li) ? __ldg(xr + ta) : 0.f;
      xb[j] = (tb >= 0 && tb < Li) ? __ldg(xr + tb) : 0.f;
    }
    const float w0 = 1.0f - lam, w1 = lam;
    for (int c = 0; c < C; ++c) {
      float va = 0.f, vb = 0.f;
#pragma unroll
      for (int j = 0; j < 7; ++j) {
        const float wj = __ldg(w + c * 7 + j);
        va = fmaf(wj, xa[j], va);
        vb = fmaf(wj, xb[j], vb);
      }
      const float bv = bias ? __ldg(bias + c) : 0.f;
      va += bv;
      vb += bv;
      out[((int64_t)b * C + c) * Lout + t] = w0 * va + w1 * vb;
    }
  }
}

__global__ void interp_table_kernel(int64_t Lin, int64_t Lout, float scale, int32_t *__restrict__ i0,
                                    int32_t *__restrict__ i1, float *__restrict__ lam) {
  for (int64_t t = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; t < Lout; t += (int64_t)gridDim.x * blockDim.x) {
    int a, b;
    float l;
    lin_src(t, scale, Lin, a, b, l);
    i0[t] = a;
    i1[t] = b;
    lam[t] = l;
  }
}

__global__ void nearest_gather_kernel(const float *__restrict__ x, float *__restrict__ out, int64_t rows,
                                      int64_t Lin, int64_t Lout, float scale) {
  const int64_t n = rows * Lout;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / Lout, t = i - r * Lout;
    int64_t s = (int64_t)floorf((float)t * scale);
    if (s > Lin - 1) s = Lin - 1;
    out[i] = __ldg(x + r * Lin + s);
  }
}

__global__ void add3_bcast_kernel(const float *__restrict__ a, const float *__restrict__ b,
                                  const float *__restrict__ bc, float *__restrict__ out, int64_t rows, int64_t L) {
  const int64_t n = rows * L;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float v = a[i];
    if (b) v += b[i];
    if (bc) v += __ldg(bc + i / L);
    out[i] = v;
  }
}

// w[r, :] = v[r, :] * (g[r] / ||v[r, :]||_2)   one CTA per row
__global__ void weight_norm_fold_kernel(const float *__restrict__ v, const float *__restrict__ g,
                                        float *__restrict__ w, int inner) {
  __shared__ float red[32];
  const int r = blockIdx.x;
  const float *vr = v + (int64_t)r * inner;
  float s = 0.f;
  for (int i = threadIdx.x; i < inner; i += blockDim.x) {
    const float t = vr[i];
    s = fmaf(t, t, s);
  }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    s = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.f;
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (threadIdx.x == 0) red[0] = g[r] / sqrtf(s);
  }
  __syncthreads();
  const float sc = red[0];
  for (int i = threadIdx.x; i < inner; i += blockDim.x) w[(int64_t)r * inner + i] = vr[i] * sc;
}

// fp32 [B,C,L] -> fp16 blk16; one thread per (b, chunk, t)
// x2 / x3 (nullable): further addends, summed in the fixed order (x + x2) + x3 before the scale -- the consumer-side
// sum over the resblocks of a stage (each resblock stream writes its own tensor; no chained accumulation)
// grid = (time blocks, channel groups of 8, batch): no index division (a flat index cost two 64-bit divisions per thread,
// as many instructions as the rest of the kernel)
// valid_len (nullable): rows t >= valid_len[b] of item b are written as zero without reading x
__global__ void __launch_bounds__(256) pack_blk16_kernel(const float *__restrict__ x, const float *__restrict__ x2,
                                                         const float *__restrict__ x3,
                                                         const int32_t *__restrict__ valid_len, uint4 *__restrict__ out,
                                                         int C, int64_t L, int64_t Lp, int lrelu, float sc, int cw) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= L) return;
  const int q = blockIdx.y, bb = blockIdx.z;
  if (valid_len && t >= __ldg(valid_len + bb)) {
    *reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(out) + hsv::blk_unit_offset(cw, Lp, C, bb, 8 * q, HSV_BLK_PAD + t)) =
        make_uint4(0u, 0u, 0u, 0u);
    return;
  }
  const int64_t off = ((int64_t)bb * C + 8 * q) * L + t;
  const float *xr = x + off;
  float v[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) v[e] = __ldg(xr + e * L);
  if (x2) {
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] += __ldg(x2 + off + e * L);
  }
  if (x3) {
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] += __ldg(x3 + off + e * L);
  }
  __half2 h[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    float v0 = v[2 * e] * sc, v1 = v[2 * e + 1] * sc;
    if (lrelu) {
      v0 = v0 > 0.f ? v0 : 0.1f * v0;
      v1 = v1 > 0.f ? v1 : 0.1f * v1;
    }
    h[e] = __floats2half2_rn(v0, v1);
  }
  *reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(out) +
                             hsv::blk_unit_offset(cw, Lp, C, bb, 8 * q, HSV_BLK_PAD + t)) = *reinterpret_cast<uint4 *>(h);
}

// inverse of pack_blk16 (test / debugging aid): blk16 -> fp32 [B,C,L]
__global__ void unpack_blk16_kernel(const uint4 *__restrict__ in, float *__restrict__ x, int B, int C, int64_t L,
                                    int64_t Lp, int cw) {
  const int nch = C >> 3;
  const int64_t n = (int64_t)B * nch * L;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t bq = i / L, t = i - bq * L;
    const int64_t bb = bq / nch;
    const int c0 = (int)(bq - bb * nch) * 8;
    const uint4 v = *reinterpret_cast<const uint4 *>(reinterpret_cast<const uint8_t *>(in) +
                                                     hsv::blk_unit_offset(cw, Lp, C, bb, c0, HSV_BLK_PAD + t));
    const __half *h = reinterpret_cast<const __half *>(&v);
    float *xr = x + bq * 8 * L + t;
#pragma unroll
    for (int e = 0; e < 8; ++e) xr[e * L] = __half2float(h[e]);
  }
}

// operand health of a blk16 buffer (debugging aid): stats[0] += number of non-finite fp16 values (an fp32 value
// beyond +-65504 became inf when the operand was produced), stats[1] = max |value| as float bits (atomicMax on the
// non-negative bit pattern)
__global__ void blk16_stats_kernel(const uint4 *__restrict__ in, unsigned int *__restrict__ stats, int B, int C,
                                   int64_t L, int64_t Lp, int cw) {
  const int nch = C >> 3;
  const int64_t n = (int64_t)B * nch * L;
  unsigned int bad = 0, mx = 0;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t bq = i / L, t = i - bq * L;
    const int64_t bb = bq / nch;
    const int c0 = (int)(bq - bb * nch) * 8;
    const uint4 v = *reinterpret_cast<const uint4 *>(reinterpret_cast<const uint8_t *>(in) +
                                                     hsv::blk_unit_offset(cw, Lp, C, bb, c0, HSV_BLK_PAD + t));
    const unsigned short *h = reinterpret_cast<const unsigned short *>(&v);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const unsigned int a = h[e] & 0x7fffu;
      if (a >= 0x7c00u) ++bad;                                   // inf / nan
      else mx = max(mx, __float_as_uint(__half2float(__ushort_as_half((unsigned short)a))));
    }
  }
  for (int o = 16; o; o >>= 1) {
    bad += __shfl_xor_sync(0xffffffffu, bad, o);
    mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) {
    if (bad) atomicAdd(stats, bad);
    atomicMax(stats + 1, mx);
  }
}

inline int grid_for(int64_t n, int threads) {
  int64_t b = (n + threads - 1) / threads;
  const int64_t cap = 148 * 32;
  return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace

extern "C" int hsv_conv1d_direct(const float *x, const float *w, const float *bias, float *out, int B, int Cin,
                                 int Cout, int64_t Lin, int64_t Lout, int k, int d, int pad, int flags,
                                 void *stream) {
  return hsv_conv1d_direct_ragged(x, w, bias, nullptr, out, B, Cin, Cout, Lin, Lout, k, d, pad, flags, stream);
}

extern "C" int hsv_conv1d_direct_ragged(const float *x, const float *w, const float *bias, const int32_t *valid_len,
                                        float *out, int B, int Cin, int Cout, int64_t Lin, int64_t Lout, int k, int d,
                                        int pad, int flags, void *stream) {
  if (B == 0 || Lout <= 0) return HSV_OK;  // empty batch / sequence
  HSV_REQUIRE(x && w && out, "conv1d_direct: null pointer");
  HSV_REQUIRE(Cin > 0 && Cout > 0 && k >= 1 && k <= KMAX && d >= 1, "conv1d_direct: bad shape");
  HSV_REQUIRE((k - 1) * d <= HALO_MAX, "conv1d_direct: (k-1)*d=%d exceeds %d", (k - 1) * d, HALO_MAX);
  HSV_REQUIRE(Lout == Lin + 2 * (int64_t)pad - (int64_t)d * (k - 1), "conv1d_direct: Lout mismatch");
  HSV_REQUIRE(!valid_len || (Cout <= 4 && k == 7 && d == 1 && pad == 3),
              "conv1d_direct: valid lengths need Cout <= 4, k = 7, d = 1, Lout == Lin (Cout=%d k=%d d=%d pad=%d)",
              Cout, k, d, pad);
  if (B == 0 || Lout <= 0) return HSV_OK;
  cudaStream_t st = hsv::as_stream(stream);
  if (k == 1 && Lin == 1 && pad == 0 && (Cin & 3) == 0 && ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(w)) & 15) == 0) {
    const int64_t nwarps = (int64_t)B * Cout;
    HSV_REQUIRE(nwarps * 32 / 256 + 1 < (1ll << 31), "conv1d_direct: grid too large");
    hsv::note_direct_launch(0, flags, 0, dim3((unsigned)((nwarps * 32 + 255) / 256)));
    conv1d_vecdot_kernel<<<(unsigned)((nwarps * 32 + 255) / 256), 256, 0, st>>>(x, w, bias, out, B, Cin, Cout, flags);
  } else if (Lout <= 8 && !valid_len) {   // (with valid_len, short items take the warp reduction inside the thin kernels)
    const int64_t nwarps = (int64_t)B * Cout * Lout;
    HSV_REQUIRE(nwarps * 32 / 256 + 1 < (1ll << 31), "conv1d_direct: grid too large");
    hsv::note_direct_launch(1, flags, 0, dim3((unsigned)((nwarps * 32 + 255) / 256)));
    conv1d_rowdot_kernel<<<(unsigned)((nwarps * 32 + 255) / 256), 256, 0, st>>>(x, w, bias, out, B, Cin, Cout, Lin,
                                                                               Lout, k, d, pad, flags);
  } else if (Cout <= 4 && d == 1 && k == 7) {
    HSV_REQUIRE(B <= 65535, "conv1d_direct: grid too large");
    dim3 grid((unsigned)((Lout + 511) / 512), (unsigned)B);
    const bool vec = pad == 3 && (Lin & 3) == 0 && Lout == Lin &&
                     ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
    hsv::note_direct_launch(vec ? 2 : 3, flags, valid_len != nullptr, grid);
    if (vec) conv1d_thin_vec_kernel<<<grid, 128, 0, st>>>(x, w, bias, out, valid_len, Cin, Cout, Lin, Lout, flags);
    else conv1d_thin_smem_kernel<7><<<grid, 256, 0, st>>>(x, w, bias, out, valid_len, Cin, Cout, Lin, Lout, pad, flags);
  } else if (Cout <= 4) {
    hsv::note_direct_launch(4, flags, 0, dim3((unsigned)grid_for((int64_t)B * Lout, 256)));
    conv1d_thin_kernel<<<grid_for((int64_t)B * Lout, 256), 256, 0, st>>>(x, w, bias, out, B, Cin, Cout, Lin,
                                                                        Lout, k, d, pad, flags);
  } else {
    constexpr int TCO = 32, TT = 64;
    HSV_REQUIRE(B <= 65535 && (Cout + TCO - 1) / TCO <= 65535, "conv1d_direct: grid too large");
    dim3 grid((unsigned)((Lout + TT - 1) / TT), (unsigned)((Cout + TCO - 1) / TCO), (unsigned)B);
    hsv::note_direct_launch(5, flags, 0, grid);
    conv1d_tiled_kernel<TCO, TT><<<grid, (TCO / 4) * (TT / 4), 0, st>>>(x, w, bias, out, Cin, Cout, Lin, Lout, k,
                                                                       d, pad, flags);
  }
  return hsv::check_launch("conv1d_direct");
}

extern "C" int hsv_conv_transpose1d_direct(const float *x, const float *w, const float *bias, const float *add,
                                           float *out, int B, int Cin, int Cout, int64_t Lin, int k, int u,
                                           void *stream) {
  if (B == 0 || Lin == 0) return HSV_OK;
  HSV_REQUIRE(x && w && out, "conv_transpose1d: null pointer");
  HSV_REQUIRE(Cin > 0 && Cout > 0 && u >= 1 && k >= u && k <= KMAX, "conv_transpose1d: bad shape k=%d u=%d", k, u);
  HSV_REQUIRE((k + u - 1) / u <= 4, "conv_transpose1d: more than 4 taps per phase");
  // L_out = (Lin-1)*u - 2p + k must equal u*Lin  (true for all five (k,u) pairs of the path)
  HSV_REQUIRE(k - 2 * ((k - u) / 2) == u, "conv_transpose1d: (k,u)=(%d,%d) does not give L_out = u*L_in", k, u);
  if (B == 0 || Lin == 0) return HSV_OK;
  constexpr int TCO = 32, TT = 64;
  const int nco = (Cout + TCO - 1) / TCO;
  HSV_REQUIRE(B <= 65535 && (int64_t)nco * u <= 65535, "conv_transpose1d: grid too large");
  dim3 grid((unsigned)((Lin + TT - 1) / TT), (unsigned)(nco * u), (unsigned)B);
  hsv::note_direct_launch(6, add ? HSV_CONV_ADD_OUT : 0, 0, grid);   // flags: the add operand as ADD_OUT
  conv_transpose1d_kernel<TCO, TT><<<grid, (TCO / 4) * (TT / 4), 0, hsv::as_stream(stream)>>>(
      x, w, bias, add, out, Cin, Cout, Lin, k, u, nco);
  return hsv::check_launch("conv_transpose1d_direct");
}

extern "C" int hsv_sr_pre_interp(const float *x, const float *w, const float *bias, float *out, int B, int C,
                                 int64_t Lin, int64_t Lout, void *stream) {
  return hsv_sr_pre_interp_ragged(x, w, bias, nullptr, nullptr, out, B, C, Lin, Lout, stream);
}

extern "C" int hsv_sr_pre_interp_ragged(const float *x, const float *w, const float *bias, const int32_t *valid_len_in,
                                        const int32_t *valid_len_out, float *out, int B, int C, int64_t Lin,
                                        int64_t Lout, void *stream) {
  if (B == 0) return HSV_OK;
  HSV_REQUIRE(x && w && out, "sr_pre_interp: null pointer");
  HSV_REQUIRE(C > 0 && Lin > 0 && Lout > 0, "sr_pre_interp: bad shape");
  if (B == 0) return HSV_OK;
  const float scale = (float)Lin / (float)Lout;  // ATen area_pixel_compute_scale, align_corners=False
  sr_pre_interp_kernel<<<grid_for((int64_t)B * Lout, 256), 256, 0, hsv::as_stream(stream)>>>(
      x, w, bias, out, valid_len_in, valid_len_out, B, C, Lin, Lout, scale);
  return hsv::check_launch("sr_pre_interp");
}

extern "C" int hsv_sr_pre_interp_stream(const float *x, const float *w, const float *bias, const int32_t *valid_len_in,
                                        const int32_t *valid_len_out, const int64_t *origin, float *out, int B, int C,
                                        int64_t Lin, int64_t Lout, int up, int down, void *stream) {
  if (B == 0) return HSV_OK;
  HSV_REQUIRE(x && w && out && valid_len_in && valid_len_out && origin, "sr_pre_interp_stream: null pointer");
  HSV_REQUIRE(C > 0 && Lin > 0 && Lout > 0, "sr_pre_interp_stream: bad shape");
  HSV_REQUIRE((up == 3 && down == 1) || (up == 3 && down == 2), "sr_pre_interp_stream: ratio must be 3/1 or 3/2");
  const float scale = (float)down / (float)up;   // == (float)L / (float)(L * up / down) for L * up < 2^24, (L % down) == 0
  sr_pre_interp_stream_kernel<<<grid_for((int64_t)B * Lout, 256), 256, 0, hsv::as_stream(stream)>>>(
      x, w, bias, out, valid_len_in, valid_len_out, reinterpret_cast<const StreamOrigin *>(origin), B, C, Lin, Lout,
      scale);
  return hsv::check_launch("sr_pre_interp_stream");
}

extern "C" int hsv_interp_linear_table(int64_t Lin, int64_t Lout, int32_t *i0, int32_t *i1, float *lam,
                                       void *stream) {
  HSV_REQUIRE(i0 && i1 && lam && Lin > 0 && Lout > 0, "interp_linear_table: bad argument");
  const float scale = (float)Lin / (float)Lout;
  interp_table_kernel<<<grid_for(Lout, 256), 256, 0, hsv::as_stream(stream)>>>(Lin, Lout, scale, i0, i1, lam);
  return hsv::check_launch("interp_linear_table");
}

extern "C" int hsv_nearest_gather(const float *x, float *out, int rows, int64_t Lin, int64_t Lout, void *stream) {
  if (rows == 0) return HSV_OK;
  HSV_REQUIRE(x && out && rows >= 0 && Lin > 0 && Lout > 0, "nearest_gather: bad argument");
  if (rows == 0) return HSV_OK;
  const float scale = (float)Lin / (float)Lout;  // ATen compute_scales_value
  nearest_gather_kernel<<<grid_for((int64_t)rows * Lout, 256), 256, 0, hsv::as_stream(stream)>>>(x, out, rows,
                                                                                                 Lin, Lout, scale);
  return hsv::check_launch("nearest_gather");
}

extern "C" int hsv_add3_bcast(const float *a, const float *b, const float *bc, float *out, int rows, int64_t L,
                              void *stream) {
  if (rows == 0 || L == 0) return HSV_OK;
  HSV_REQUIRE(a && out && rows >= 0 && L >= 0, "add3_bcast: bad argument");
  if (rows == 0 || L == 0) return HSV_OK;
  add3_bcast_kernel<<<grid_for((int64_t)rows * L, 256), 256, 0, hsv::as_stream(stream)>>>(a, b, bc, out, rows, L);
  return hsv::check_launch("add3_bcast");
}

extern "C" int hsv_weight_norm_fold(const float *v, const float *g, float *w, int n0, int inner, void *stream) {
  HSV_REQUIRE(v && g && w && n0 > 0 && inner > 0, "weight_norm_fold: bad argument");
  weight_norm_fold_kernel<<<n0, 256, 0, hsv::as_stream(stream)>>>(v, g, w, inner);
  return hsv::check_launch("weight_norm_fold");
}

namespace {
// the three pack entry points share one launch; `name` prefixes their argument errors
int pack_blk16_launch(const char *name, const float *x1, const float *x2, const float *x3, const int32_t *valid_len,
                      void *out, int B, int C, int64_t L, int lrelu, float in_scale, void *stream) {
  if (B == 0 || L == 0) return HSV_OK;
  HSV_REQUIRE(x1 && out, "%s: null pointer", name);
  HSV_REQUIRE(x2 || !x3, "%s: x3 without x2", name);
  HSV_REQUIRE(C > 0 && C % 16 == 0, "%s: C %% 16 != 0 (C=%d)", name, C);
  HSV_REQUIRE(B <= 65535 && C / 8 <= 65535, "%s: grid too large", name);
  pack_blk16_kernel<<<dim3((unsigned)((L + 255) / 256), (unsigned)(C / 8), (unsigned)B), 256, 0, hsv::as_stream(stream)>>>(
      x1, x2, x3, valid_len, reinterpret_cast<uint4 *>(out), C, L, hsv::blk16_rows(L), lrelu, in_scale,
      hsv::blk_cw(C));
  return hsv::check_launch(name);
}
}  // namespace

extern "C" int hsv_pack_blk16(const float *x, void *out, int B, int C, int64_t L, int lrelu, float in_scale,
                              void *stream) {
  return pack_blk16_launch("pack_blk16", x, nullptr, nullptr, nullptr, out, B, C, L, lrelu, in_scale, stream);
}

extern "C" int hsv_pack_blk16_sum3(const float *x1, const float *x2, const float *x3, void *out, int B, int C,
                                   int64_t L, int lrelu, float in_scale, void *stream) {
  return pack_blk16_launch("pack_blk16_sum3", x1, x2, x3, nullptr, out, B, C, L, lrelu, in_scale, stream);
}

extern "C" int hsv_pack_blk16_sum3_ragged(const float *x1, const float *x2, const float *x3, const int32_t *valid_len,
                                          void *out, int B, int C, int64_t L, int lrelu, float in_scale, void *stream) {
  return pack_blk16_launch("pack_blk16_sum3_ragged", x1, x2, x3, valid_len, out, B, C, L, lrelu, in_scale, stream);
}

extern "C" int hsv_unpack_blk16(const void *in, float *x, int B, int C, int64_t L, void *stream) {
  if (B == 0 || L == 0) return HSV_OK;
  HSV_REQUIRE(in && x, "unpack_blk16: null pointer");
  HSV_REQUIRE(C > 0 && C % 16 == 0, "unpack_blk16: C %% 16 != 0 (C=%d)", C);
  unpack_blk16_kernel<<<grid_for((int64_t)B * (C / 8) * L, 256), 256, 0, hsv::as_stream(stream)>>>(
      reinterpret_cast<const uint4 *>(in), x, B, C, L, hsv::blk16_rows(L), hsv::blk_cw(C));
  return hsv::check_launch("unpack_blk16");
}

extern "C" int hsv_blk16_stats(const void *in, void *stats, int B, int C, int64_t L, void *stream) {
  if (B == 0 || L == 0) return HSV_OK;
  HSV_REQUIRE(in && stats, "blk16_stats: null pointer");
  HSV_REQUIRE(C > 0 && C % 16 == 0, "blk16_stats: C %% 16 != 0 (C=%d)", C);
  blk16_stats_kernel<<<grid_for((int64_t)B * (C / 8) * L, 256), 256, 0, hsv::as_stream(stream)>>>(
      reinterpret_cast<const uint4 *>(in), reinterpret_cast<unsigned int *>(stats), B, C, L, hsv::blk16_rows(L),
      hsv::blk_cw(C));
  return hsv::check_launch("blk16_stats");
}
