// Frame-rate (50 Hz) operators of the step BEFORE the vocoder (SURVEY.md §8f2): the pieces of StyleEncoder,
// PosteriorSFEncoder (three WaveNet stacks) and the reverse coupling flows (DiT blocks) that are not convolutions.
// The convolutions / Linear layers themselves run on the tcgen05 kernel (conv_umma.cu) through the operand packers
// below.  All tensors are fp32 [B, C, T] (the reference's layout; T ~ 50 frames per second), so these kernels are
// small, HBM/L2-bound element-wise or row-reduction kernels on CUDA cores; what matters is that each reference
// expression becomes ONE launch instead of 3-9 ATen kernels, and that the whole front is CUDA-graph capturable.
//
// Reference expressions (paths relative to the reference root):
//   gate      commons.fused_add_tanh_sigmoid_multiply            commons.py:108-114   (WN, modules.py:158-165)
//   wn_res    x = (x + res) * mask ; output += skip               modules.py:167-174
//   ln_mod    modulate(LayerNorm(x) [* mask], shift, scale)       modules.py:346-347, 405-410 (eps 1e-6, no affine)
//   mha       softmax(q k^T / sqrt(d)) v                          timm 0.6.13 Attention; attentions.py:157-188
//   gate_add  x + gate[b,c] * y * mask                            modules.py:408-409
//   couple    x1 = (x1 - m) * mask        (mean_only, reverse)    modules.py:484-487
//   sample    z = (m + eps * exp(logs) * noise_scale) * mask      hierspeechpp_speechsynthesizer.py:201, 687
//   glu_res   x + y1 * sigmoid(y2)                                styleencoder.py:25-31
//   mish      x * tanh(softplus(x))                               styleencoder.py:6-10
//   flip      torch.flip(x, [1])                                  modules.py:270-277
//   mean      x.sum(2) / mask.sum(2)                              styleencoder.py:91-99
#include "hsv_common.cuh"

namespace {

inline int grid_for(int64_t n, int threads) {
  int64_t b = (n + threads - 1) / threads;
  const int64_t cap = 148 * 32;
  return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

__device__ __forceinline__ float sigmoidf_(float v) { return 1.0f / (1.0f + expf(-v)); }
__device__ __forceinline__ float gelu_tanh(float v) {
  // F.gelu(approximate="tanh"): 0.5 x (1 + tanh(sqrt(2/pi) (x + 0.044715 x^3)))
  const float k = 0.7978845608028654f;
  return 0.5f * v * (1.0f + tanhf(k * (v + 0.044715f * v * v * v)));
}
__device__ __forceinline__ float mishf(float v) {
  // F.softplus (beta 1, threshold 20) then tanh
  const float sp = v > 20.f ? v : log1pf(expf(v));
  return v * tanhf(sp);
}

// ---- operand packers: fp32 [B, Cin, T] -> fp16 blk16 [C] with a fused activation --------------------------------
// mode 0: x * mask            mode 1: tanh(x[c] + bc[c]) * sigmoid(x[C+c] + bc[C+c])   (x has 2C channels, bc [B,2C])
// mode 2: gelu_tanh(x) * mask mode 3: mish(x) * mask
__global__ void pack_act_kernel(const float *__restrict__ x, const float *__restrict__ bc, const float *__restrict__ mask,
                                uint4 *__restrict__ out, int B, int C, int64_t L, int64_t Lp, int cw, int mode, int cin) {
  // cin = channels per batch item of x (>= C, or >= 2C for the gate): a channel prefix of a wider tensor can be packed
  // grid = (time blocks, channel groups of 8, batch): no index division
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < L) {
    const int64_t bb = blockIdx.z;
    const int c0 = blockIdx.y * 8;
    const float mk = mask ? __ldg(mask + bb * L + t) : 1.f;
    const float *xr = x + (bb * cin + c0) * L + t;
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      const float a = __ldg(xr + (int64_t)e * L);
      if (mode == 1) {
        const float g = __ldg(xr + (int64_t)(C + e) * L);
        const float ba = bc ? __ldg(bc + bb * 2 * C + c0 + e) : 0.f, bg = bc ? __ldg(bc + bb * 2 * C + C + c0 + e) : 0.f;
        v[e] = tanhf(a + ba) * sigmoidf_(g + bg);
      } else if (mode == 2) {
        v[e] = gelu_tanh(a) * mk;
      } else if (mode == 3) {
        v[e] = mishf(a) * mk;
      } else {
        v[e] = a * mk;
      }
    }
    __half2 h[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) h[e] = __floats2half2_rn(v[2 * e], v[2 * e + 1]);
    *reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(out) +
                               hsv::blk_unit_offset(cw, Lp, C, bb, c0, HSV_BLK_PAD + t)) = *reinterpret_cast<uint4 *>(h);
  }
}

// WN layer tail fused with the next layer's operand pack (modules.py:167-174 + the PACK of in_layers[i+1]):
//   x = (x + rs[:, :C]) * mask  (in place, fp32: the residual stream)   output += rs[:, C:]   blk = fp16(x)
__global__ void wn_res_pack_kernel(float *__restrict__ x, const float *__restrict__ rs, const float *__restrict__ mask,
                                   float *__restrict__ output, uint4 *__restrict__ blk, int B, int C, int64_t L,
                                   int64_t Lp, int cw) {
  const int nch = C >> 3;
  const int64_t n = (int64_t)B * nch * L;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t bq = i / L, t = i - bq * L;
    const int64_t bb = bq / nch;
    const int c0 = (int)(bq - bb * nch) * 8;
    const float mk = mask ? __ldg(mask + bb * L + t) : 1.f;
    float *xr = x + (bb * C + c0) * L + t, *orow = output + (bb * C + c0) * L + t;
    const float *rr = rs + (bb * 2 * C + c0) * L + t;
    // all 32 loads first (x and output are updated in place: interleaved with the stores the compiler must keep them in
    // program order, a chain of 8 dependent round trips)
    float xv[8], ov[8], rv[8], sv[8], v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      xv[e] = xr[(int64_t)e * L];
      ov[e] = orow[(int64_t)e * L];
      rv[e] = __ldg(rr + (int64_t)e * L);
      sv[e] = __ldg(rr + (int64_t)(C + e) * L);
    }
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      v[e] = (xv[e] + rv[e]) * mk;
      xr[(int64_t)e * L] = v[e];
      orow[(int64_t)e * L] = ov[e] + sv[e];
    }
    __half2 h[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) h[e] = __floats2half2_rn(v[2 * e], v[2 * e + 1]);
    *reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(blk) +
                               hsv::blk_unit_offset(cw, Lp, C, bb, c0, HSV_BLK_PAD + t)) = *reinterpret_cast<uint4 *>(h);
  }
}

// LayerNorm over channels (no affine) -> optional mask -> modulate -> fp16 blk16.  CTA = 32 time steps x 8 channel
// groups; thread (tx, g) owns the C/8 consecutive channels of group g at step tx (C % 64 == 0: whole 16-byte units).
// With y != nullptr the preceding gated residual update is fused in (modules.py:408-409): x = x + gate[b,c] * y * mask is
// written back to x (fp32, in place) and the normalisation runs on the new x.
// ZROWS: operand rows where mask == 0 are written as zero (HSV_LN_ZERO_MASKED; a separate instantiation, so the
// other launches run none of it)
template <int CPT, bool ZROWS>   // channels per thread = C / 8
__global__ void __launch_bounds__(256) ln_mod_kernel(float *x, const float *__restrict__ y, const float *__restrict__ gate,
                                                     int64_t gate_stride, const float *__restrict__ shift,
                                                     const float *__restrict__ scale, const float *__restrict__ mask,
                                                     uint4 *__restrict__ out, int C, int64_t L, int64_t Lp, int cw,
                                                     float eps, int inmask, int premask, int64_t mod_stride) {
  __shared__ float red[8][33];
  const int tx = threadIdx.x & 31, g = threadIdx.x >> 5;
  const int b = blockIdx.y;
  const int64_t t = (int64_t)blockIdx.x * 32 + tx;
  const bool ok = t < L;
  const float mk = (mask && ok) ? __ldg(mask + (int64_t)b * L + t) : 1.f;
  float v[CPT];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < CPT; ++i) v[i] = ok ? x[((int64_t)b * C + g * CPT + i) * L + t] : 0.f;
  if (y) {
    float yv[CPT];
#pragma unroll
    for (int i = 0; i < CPT; ++i) yv[i] = ok ? __ldg(y + ((int64_t)b * C + g * CPT + i) * L + t) : 0.f;
#pragma unroll
    for (int i = 0; i < CPT; ++i) {
      v[i] = v[i] + (__ldg(gate + (int64_t)b * gate_stride + g * CPT + i) * yv[i]) * mk;
      if (ok) x[((int64_t)b * C + g * CPT + i) * L + t] = v[i];
    }
  }
#pragma unroll
  for (int i = 0; i < CPT; ++i) {
    if (inmask) v[i] *= mk;
    s += v[i];
  }
  red[g][tx] = s;
  __syncthreads();
  float mean = 0.f;
#pragma unroll
  for (int q = 0; q < 8; ++q) mean += red[q][tx];
  mean /= (float)C;
  __syncthreads();
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < CPT; ++i) {
    const float d = v[i] - mean;
    ss += d * d;
  }
  red[g][tx] = ss;
  __syncthreads();
  float var = 0.f;
#pragma unroll
  for (int q = 0; q < 8; ++q) var += red[q][tx];
  const float rstd = rsqrtf(var / (float)C + eps);
  if (!ok) return;
  if (ZROWS && mk == 0.f) {               // rows past an item of a ragged batch: the zero padding of its own run
#pragma unroll
    for (int u = 0; u < CPT / 8; ++u)
      *reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(out) +
                                 hsv::blk_unit_offset(cw, Lp, C, b, g * CPT + u * 8, HSV_BLK_PAD + t)) = make_uint4(0, 0, 0, 0);
    return;
  }
  const float pm = (premask & 1) ? mk : 1.f;
#pragma unroll
  for (int u = 0; u < CPT / 8; ++u) {
    __half2 h[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      float o[2];
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        const int c = g * CPT + u * 8 + 2 * e + q;
        const float nrm = (v[u * 8 + 2 * e + q] - mean) * rstd * pm;
        o[q] = nrm * (1.f + __ldg(scale + (int64_t)b * mod_stride + c)) + __ldg(shift + (int64_t)b * mod_stride + c);
      }
      h[e] = __floats2half2_rn(o[0], o[1]);
    }
    *reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(out) +
                               hsv::blk_unit_offset(cw, Lp, C, b, g * CPT + u * 8, HSV_BLK_PAD + t)) =
        *reinterpret_cast<uint4 *>(h);
  }
}

// ---- element-wise fp32 ops on [B, C, T] ---------------------------------------------------------------------------
enum { OP_WN_RES = 1, OP_WN_LAST = 2, OP_GATE_ADD = 3, OP_COUPLE = 4, OP_SAMPLE = 5, OP_MASK = 6, OP_ADD = 7,
       OP_GLU_RES = 8, OP_MISH = 9, OP_FLIP = 10, OP_ADD_BCAST = 11 };

// (a / out / out2 may alias: several ops update a tensor in place)
__global__ void frame_op_kernel(int op, const float *a, const float *__restrict__ b2, const float *__restrict__ c2,
                                const float *__restrict__ mask, float *out, float *out2, int B, int C, int64_t L,
                                float s, int64_t cstride) {
  // grid = (time blocks, channels, batch): no index division
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < L) {
    const int c = blockIdx.y;
    const int64_t bb = blockIdx.z;
    const int64_t i = (bb * C + c) * L + t;
    const float mk = mask ? __ldg(mask + bb * L + t) : 1.f;
    switch (op) {
      case OP_WN_RES: {   // a = x [B,C,T] (updated in place through out), b2 = rs [B,2C,T], out2 = output accumulator
        const float res = __ldg(b2 + (bb * 2 * C + c) * L + t), skip = __ldg(b2 + (bb * 2 * C + C + c) * L + t);
        out[i] = (a[i] + res) * mk;
        out2[i] = out2[i] + skip;
        break;
      }
      case OP_WN_LAST:    // out2 = (output + rs) * mask, b2 = rs [B,C,T]
        out2[i] = (out2[i] + __ldg(b2 + i)) * mk;
        break;
      case OP_GATE_ADD:   // out = a + gate[b, c] * b2 * mask; c2 = gate base, cstride = batch stride of the gate vector
        out[i] = a[i] + (__ldg(c2 + bb * cstride + c) * __ldg(b2 + i)) * mk;
        break;
      case OP_COUPLE:     // a = x [B,2C,T]: channels [C, 2C) become (x1 - m) * mask, b2 = m [B,C,T]; in place via out
        out[(bb * 2 * C + C + c) * L + t] = (a[(bb * 2 * C + C + c) * L + t] - __ldg(b2 + i)) * mk;
        break;
      case OP_SAMPLE: {   // a = stats [B,2C,T] (m | logs), b2 = eps [B,C,T]: out = (m + eps * exp(logs) * s) * mask
        const float m = __ldg(a + (bb * 2 * C + c) * L + t), lg = __ldg(a + (bb * 2 * C + C + c) * L + t);
        out[i] = (m + (__ldg(b2 + i) * expf(lg)) * s) * mk;
        break;
      }
      case OP_MASK:
        out[i] = a[i] * mk;
        break;
      case OP_ADD:
        out[i] = (a[i] + __ldg(b2 + i)) * mk;
        break;
      case OP_GLU_RES: {  // a = x [B,C,T], b2 = y [B,2C,T]: out = x + y1 * sigmoid(y2)
        const float y1 = __ldg(b2 + (bb * 2 * C + c) * L + t), y2 = __ldg(b2 + (bb * 2 * C + C + c) * L + t);
        out[i] = (a[i] + y1 * sigmoidf_(y2)) * mk;
        break;
      }
      case OP_MISH:
        out[i] = mishf(a[i]) * mk;
        break;
      case OP_FLIP:
        out[i] = __ldg(a + (bb * C + (C - 1 - c)) * L + t);
        break;
      case OP_ADD_BCAST:  // out = (a + c2[b, c]) * mask
        out[i] = (a[i] + __ldg(c2 + bb * cstride + c)) * mk;
        break;
    }
  }
}

// ---- multi-head attention, fp32, online softmax -------------------------------------------------------------------
// q, k, v: channel-major [heads*D, T] per batch item (time contiguous), batch strides in elements; out [B, heads*D, Tq].
// CTA = 4 warps, each warp owns RW query rows of one (batch, head) outright (no cross-warp traffic); keys in tiles of
// 64, double-buffered with cp.async (16-byte copies: the channel-major layout IS the [d][t] layout both products
// want, so a tile is 2*D row segments of 256 bytes).
//   S = Q K^T : lane = 2 keys, RW rows -> per d one broadcast LDS of the rows + one LDS.64 of the keys, 2*RW FMAs
//   softmax   : a row's 64 scores live in the 32 lanes of its warp -> shuffles
//   O += P V  : lane = dims {lane, lane+32, ...}, four keys per step: one LDS.128 of V per dim (16-byte chunks of a
//               V row XOR-swizzled with d, so the 8 lanes of a quarter-warp hit 8 different chunks) and 4*RW
//               broadcast P values -> 4*RW*D/32 FMAs per 3-4 shared loads
constexpr int MHA_K = 64, MHA_THREADS = 128;

__device__ __forceinline__ void cp_async16(void *dst, const void *src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

template <int D, int RW>
__global__ void __launch_bounds__(MHA_THREADS) mha_kernel(const float *__restrict__ q, const float *__restrict__ k,
                                                          const float *__restrict__ v, float *__restrict__ out,
                                                          const int *__restrict__ lens, int Tq, int Tk, int64_t qbs,
                                                          int64_t kbs, int64_t vbs, int heads, float scale, int prescale,
                                                          int fast) {
  constexpr int QT = 4 * RW;            // query rows per CTA
  constexpr int DL = D / 32;            // output dims per lane
  constexpr int TILE = D * MHA_K;       // floats per K (or V) tile
  extern __shared__ __align__(16) float sm[];
  float *Qs = sm;                       // [D][QT]
  float *KV = Qs + D * QT;              // 2 stages x (K tile [D][64], V tile [D][64] chunk-swizzled)
  float *Ps = KV + 4 * TILE;            // [4 warps][MHA_K][RW]
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * QT;
  const float *qb = q + (int64_t)b * qbs + (int64_t)h * D * Tq;
  const float *kb = k + (int64_t)b * kbs + (int64_t)h * D * Tk;
  const float *vb = v + (int64_t)b * vbs + (int64_t)h * D * Tk;
  const int len = lens ? lens[b] : 0x7fffffff;
  const int ntiles = (Tk + MHA_K - 1) / MHA_K;

  auto load_tile = [&](int t, int stage) {
    float *Kd = KV + stage * 2 * TILE, *Vd = Kd + TILE;
    const int k0 = t * MHA_K;
    if (fast && k0 + MHA_K <= Tk) {
      for (int c = tid; c < D * 16; c += MHA_THREADS) {          // 16-byte chunks: 16 per row
        const int d = c >> 4, ch = c & 15;
        cp_async16(Kd + d * MHA_K + ch * 4, kb + (int64_t)d * Tk + k0 + ch * 4);
        cp_async16(Vd + d * MHA_K + ((ch ^ (d & 15)) << 2), vb + (int64_t)d * Tk + k0 + ch * 4);
      }
    } else {                                                     // ragged last tile / unaligned tensors
      for (int idx = tid; idx < TILE; idx += MHA_THREADS) {
        const int d = idx / MHA_K, j = idx - d * MHA_K;
        const bool okj = k0 + j < Tk;
        Kd[idx] = okj ? __ldg(kb + (int64_t)d * Tk + k0 + j) : 0.f;
        Vd[d * MHA_K + ((((j >> 2) ^ (d & 15)) << 2) | (j & 3))] = okj ? __ldg(vb + (int64_t)d * Tk + k0 + j) : 0.f;
      }
    }
    cp_async_commit();
  };

  load_tile(0, 0);
  for (int idx = tid; idx < D * QT; idx += MHA_THREADS) {
    const int d = idx / QT, i = idx - d * QT;
    const float val = (q0 + i < Tq) ? __ldg(qb + (int64_t)d * Tq + q0 + i) : 0.f;
    Qs[idx] = prescale ? val * scale : val;
  }
  float m_run[RW], l_run[RW], acc[RW][DL];
#pragma unroll
  for (int r = 0; r < RW; ++r) {
    m_run[r] = -INFINITY;
    l_run[r] = 0.f;
#pragma unroll
    for (int j = 0; j < DL; ++j) acc[r][j] = 0.f;
  }
  float *Pw = Ps + w * MHA_K * RW;
  for (int t = 0; t < ntiles; ++t) {
    const int k0 = t * MHA_K;
    if (t + 1 < ntiles) {
      load_tile(t + 1, (t + 1) & 1);     // its buffer was released by the barrier at the end of iteration t - 1
      cp_async_wait<1>();
    } else {
      cp_async_wait<0>();
    }
    __syncthreads();
    const float *Ks = KV + (t & 1) * 2 * TILE, *Vs = Ks + TILE;
    // ---- S: RW rows x 2 keys per lane ----
    float s0[RW], s1[RW];
#pragma unroll
    for (int r = 0; r < RW; ++r) s0[r] = s1[r] = 0.f;
#pragma unroll 8
    for (int d = 0; d < D; ++d) {
      const float2 kk = *reinterpret_cast<const float2 *>(Ks + d * MHA_K + 2 * lane);
      float qq[RW];
      if (RW == 4) {
        const float4 tq = *reinterpret_cast<const float4 *>(Qs + d * QT + 4 * w);
        qq[0] = tq.x; qq[1] = tq.y; qq[2 % RW] = tq.z; qq[3 % RW] = tq.w;
      } else {
        const float2 tq = *reinterpret_cast<const float2 *>(Qs + d * QT + 2 * w);
        qq[0] = tq.x; qq[1 % RW] = tq.y;
      }
#pragma unroll
      for (int r = 0; r < RW; ++r) {
        s0[r] = fmaf(qq[r], kk.x, s0[r]);
        s1[r] = fmaf(qq[r], kk.y, s1[r]);
      }
    }
    // ---- online softmax per row (a row = one warp's 64 values) ----
    const int j0 = k0 + 2 * lane, j1 = j0 + 1;
#pragma unroll
    for (int r = 0; r < RW; ++r) {
      const int qi = q0 + RW * w + r;
      float a = prescale ? s0[r] : s0[r] * scale, c = prescale ? s1[r] : s1[r] * scale;
      if (lens && (qi >= len || j0 >= len)) a = -1e4f;     // masked_fill(mask == 0, -1e4)
      if (lens && (qi >= len || j1 >= len)) c = -1e4f;
      if (j0 >= Tk) a = -INFINITY;                         // padding of the last key tile
      if (j1 >= Tk) c = -INFINITY;
      float mx = fmaxf(a, c);
#pragma unroll
      for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      const float m_new = fmaxf(m_run[r], mx);
      const float corr = expf(m_run[r] - m_new);
      const float p0 = expf(a - m_new), p1 = expf(c - m_new);
      float sum = p0 + p1;
#pragma unroll
      for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
      l_run[r] = l_run[r] * corr + sum;
      m_run[r] = m_new;
#pragma unroll
      for (int j = 0; j < DL; ++j) acc[r][j] *= corr;
      *reinterpret_cast<float2 *>(Pw + r * MHA_K + 2 * lane) = make_float2(p0, p1);      // Pw[r][key]
    }
    __syncwarp();
    // ---- O += P V, four keys per step ----
#pragma unroll 2
    for (int j4 = 0; j4 < MHA_K / 4; ++j4) {
      float4 pp[RW];
#pragma unroll
      for (int r = 0; r < RW; ++r) pp[r] = *reinterpret_cast<const float4 *>(Pw + r * MHA_K + 4 * j4);   // broadcast
#pragma unroll
      for (int e = 0; e < DL; ++e) {
        const int d = lane + 32 * e;
        const float4 vv = *reinterpret_cast<const float4 *>(Vs + d * MHA_K + ((j4 ^ (d & 15)) << 2));
#pragma unroll
        for (int r = 0; r < RW; ++r) {
          acc[r][e] = fmaf(pp[r].x, vv.x, acc[r][e]);
          acc[r][e] = fmaf(pp[r].y, vv.y, acc[r][e]);
          acc[r][e] = fmaf(pp[r].z, vv.z, acc[r][e]);
          acc[r][e] = fmaf(pp[r].w, vv.w, acc[r][e]);
        }
      }
    }
    __syncthreads();     // this stage's K / V may be overwritten by the load issued in the next iteration
  }
  float *ob = out + ((int64_t)b * heads + h) * D * Tq;
#pragma unroll
  for (int r = 0; r < RW; ++r) {
    const int qi = q0 + RW * w + r;
    if (qi < Tq) {
      const float inv = 1.0f / l_run[r];
#pragma unroll
      for (int e = 0; e < DL; ++e) ob[(int64_t)(lane + 32 * e) * Tq + qi] = acc[r][e] * inv;
    }
  }
}

template <int D, int RW>
int mha_launch(const float *q, const float *k, const float *v, float *out, const int *lens, int B, int heads, int Tq,
               int Tk, int64_t qbs, int64_t kbs, int64_t vbs, float scale, int prescale, cudaStream_t st) {
  constexpr int QT = 4 * RW;
  const size_t smem = sizeof(float) * (D * QT + 4 * D * MHA_K + 4 * MHA_K * RW);
  static bool done = false;
  if (!done) {
    cudaError_t e = cudaFuncSetAttribute(mha_kernel<D, RW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      cudaGetLastError();
      hsv::set_error("mha: cudaFuncSetAttribute(%zu): %s", smem, cudaGetErrorString(e));
      return HSV_ERR_CUDA;
    }
    done = true;
  }
  // 16-byte cp.async needs every K / V row segment aligned: Tk % 4 == 0, aligned bases and batch strides
  auto al = [](const void *p_) { return (reinterpret_cast<uintptr_t>(p_) & 15) == 0; };
  const int fast = (Tk % 4 == 0) && al(k) && al(v) && (kbs % 4 == 0) && (vbs % 4 == 0);
  dim3 grid((unsigned)((Tq + QT - 1) / QT), (unsigned)heads, (unsigned)B);
  hsv::note_mha_launch(1, D, 0, lens != nullptr, 0, prescale, fast, 0, (Tk + MHA_K - 1) / MHA_K, grid);
  mha_kernel<D, RW><<<grid, MHA_THREADS, smem, st>>>(q, k, v, out, lens, Tq, Tk, qbs, kbs, vbs, heads, scale, prescale, fast);
  return hsv::check_launch("mha");
}

// Conv1d with ONE input channel and a stride (PosteriorSFEncoder.pre_filter: Conv1d(1, 192, 9, stride 4, padding 4),
// hierspeechpp_speechsynthesizer.py:187,196): out[b, co, t] = bias[co] + sum_j w[co, j] * x[b, t*stride + j - pad]
// VLEN: item b is its first vlen[b] output frames and stride * vlen[b] input samples (the rest of its input is the
// conv's zero padding and is never read, its output there is 0)
template <bool VLEN>
__global__ void conv1d_c1_strided_kernel(const float *__restrict__ x, const float *__restrict__ w,
                                         const float *__restrict__ bias, const float *__restrict__ mask,
                                         const int *__restrict__ vlen, float *__restrict__ out, int B, int Cout,
                                         int64_t Lin, int64_t Lout, int k, int stride, int pad) {
  const int64_t n = (int64_t)B * Cout * Lout;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t bc = i / Lout, t = i - bc * Lout;
    const int64_t bb = bc / Cout;
    const int co = (int)(bc - bb * Cout);
    int64_t lin = Lin;
    if (VLEN) {
      const int64_t nv = min((int64_t)max(__ldg(vlen + bb), 0), Lout);
      if (t >= nv) {
        out[i] = 0.f;
        continue;
      }
      lin = min(nv * stride, Lin);
    }
    float acc = 0.f;
    for (int j = 0; j < k; ++j) {
      const int64_t s = t * stride + j - pad;
      if (s >= 0 && s < lin) acc = fmaf(__ldg(w + co * k + j), __ldg(x + bb * Lin + s), acc);
    }
    acc += bias ? __ldg(bias + co) : 0.f;
    out[i] = acc * (mask ? __ldg(mask + bb * Lout + t) : 1.f);
  }
}

// out[b, c] = sum_t x[b, c, t] / denom[b]   (StyleEncoder.temporal_avg_pool: the sum runs over ALL frames)
// VLEN: the sum of item b runs over t < vlen[b] only, in the order of its own launch with L = vlen[b]
template <bool VLEN>
__global__ void masked_mean_kernel(const float *__restrict__ x, const int *__restrict__ vlen, float *__restrict__ out,
                                   int C, int64_t L) {
  const int64_t row = blockIdx.x;            // b * C + c
  const int64_t n = VLEN ? min((int64_t)max(__ldg(vlen + row / C), 0), L) : L;
  float s = 0.f;
  for (int64_t t = threadIdx.x; t < n; t += blockDim.x) s += __ldg(x + row * L + t);
  __shared__ float red[32];
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) tot += red[i];
    out[row] = tot;
  }
}
__global__ void mean_div_kernel(float *__restrict__ out, const float *__restrict__ mask, const int *__restrict__ vlen,
                                int C, int64_t L) {
  const int b = blockIdx.x;
  __shared__ float len_s;
  if (threadIdx.x == 0) {
    float l = 0.f;
    if (vlen) {                              // an item's own run: a mask of n ones sums to n exactly (n < 2^24)
      l = (float)min((int64_t)max(vlen[b], 0), L);
    } else {
      for (int64_t t = 0; t < L; ++t) l += mask ? mask[(int64_t)b * L + t] : 1.f;
    }
    len_s = l;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) out[(int64_t)b * C + c] = out[(int64_t)b * C + c] / len_s;
}

}  // namespace

extern "C" int hsv_pack_blk16_act(const float *x, const float *bcast, const float *mask, void *out, int B, int C,
                                  int64_t L, int mode, int x_channels, void *stream) {
  if (B == 0 || L == 0) return HSV_OK;
  HSV_REQUIRE(x && out, "pack_blk16_act: null pointer");
  HSV_REQUIRE(C > 0 && C % 16 == 0 && mode >= 0 && mode <= 3, "pack_blk16_act: bad C=%d / mode=%d", C, mode);
  HSV_REQUIRE(x_channels >= (mode == 1 ? 2 * C : C), "pack_blk16_act: x has %d channels, needs %d", x_channels,
              mode == 1 ? 2 * C : C);
  HSV_REQUIRE(B <= 65535 && C / 8 <= 65535, "pack_blk16_act: grid too large");
  pack_act_kernel<<<dim3((unsigned)((L + 127) / 128), (unsigned)(C / 8), (unsigned)B), 128, 0, hsv::as_stream(stream)>>>(
      x, bcast, mask, reinterpret_cast<uint4 *>(out), B, C, L, hsv::blk16_rows(L), hsv::blk_cw(C), mode, x_channels);
  return hsv::check_launch("pack_blk16_act");
}

extern "C" int hsv_wn_res_pack(float *x, const float *rs, const float *mask, float *output, void *blk, int B, int C,
                               int64_t L, void *stream) {
  if (B == 0 || L == 0) return HSV_OK;
  HSV_REQUIRE(x && rs && output && blk, "wn_res_pack: null pointer");
  HSV_REQUIRE(C > 0 && C % 16 == 0, "wn_res_pack: C %% 16 != 0 (C=%d)", C);
  wn_res_pack_kernel<<<grid_for((int64_t)B * (C / 8) * L, 256), 256, 0, hsv::as_stream(stream)>>>(
      x, rs, mask, output, reinterpret_cast<uint4 *>(blk), B, C, L, hsv::blk16_rows(L), hsv::blk_cw(C));
  return hsv::check_launch("wn_res_pack");
}

static int ln_mod_launch(float *x, const float *y, const float *gate, int64_t gate_stride, const float *shift,
                         const float *scale, const float *mask, void *out, int B, int C, int64_t L, float eps, int inmask,
                         int premask, int64_t mod_stride, void *stream, const char *what) {
  if (B == 0 || L == 0) return HSV_OK;
  HSV_REQUIRE(x && shift && scale && out, "%s: null pointer", what);
  HSV_REQUIRE(C == 192 || C == 256 || C == 128 || C == 64, "%s: C must be 64, 128, 192 or 256 (C=%d)", what, C);
  HSV_REQUIRE(B <= 65535, "%s: batch too large", what);
  HSV_REQUIRE(!(premask & HSV_LN_ZERO_MASKED) || mask, "%s: zeroing masked rows needs a mask", what);
  dim3 grid((unsigned)((L + 31) / 32), (unsigned)B);
  cudaStream_t st = hsv::as_stream(stream);
  uint4 *o = reinterpret_cast<uint4 *>(out);
  const int64_t Lp = hsv::blk16_rows(L);
  const int cw = hsv::blk_cw(C);
#define HSV_LN(CPT)                                                                                                       \
  if (premask & HSV_LN_ZERO_MASKED)                                                                                         \
    ln_mod_kernel<CPT, true><<<grid, 256, 0, st>>>(x, y, gate, gate_stride, shift, scale, mask, o, C, L, Lp, cw, eps, inmask, \
                                                   premask, mod_stride);                                                    \
  else                                                                                                                      \
    ln_mod_kernel<CPT, false><<<grid, 256, 0, st>>>(x, y, gate, gate_stride, shift, scale, mask, o, C, L, Lp, cw, eps, inmask, \
                                                    premask, mod_stride)
  if (C == 192) {
    HSV_LN(24);
  } else if (C == 256) {
    HSV_LN(32);
  } else if (C == 128) {
    HSV_LN(16);
  } else {
    HSV_LN(8);
  }
#undef HSV_LN
  return hsv::check_launch(what);
}

extern "C" int hsv_ln_mod_blk16(const float *x, const float *shift, const float *scale, const float *mask, void *out,
                                int B, int C, int64_t L, float eps, int inmask, int premask, int64_t mod_stride,
                                void *stream) {
  return ln_mod_launch(const_cast<float *>(x), nullptr, nullptr, 0, shift, scale, mask, out, B, C, L, eps, inmask, premask,
                       mod_stride, stream, "ln_mod_blk16");   // y == nullptr: x is only read
}

extern "C" int hsv_gate_ln_mod_blk16(float *x, const float *y, const float *gate, int64_t gate_stride, const float *shift,
                                     const float *scale, const float *mask, void *out, int B, int C, int64_t L, float eps,
                                     int premask, int64_t mod_stride, void *stream) {
  HSV_REQUIRE(y && gate, "gate_ln_mod_blk16: null pointer");
  return ln_mod_launch(x, y, gate, gate_stride, shift, scale, mask, out, B, C, L, eps, 0, premask, mod_stride, stream,
                       "gate_ln_mod_blk16");
}

extern "C" int hsv_frame_op(int op, const float *a, const float *b, const float *c, const float *mask, float *out,
                            float *out2, int B, int C, int64_t L, float s, int64_t cstride, void *stream) {
  if (B == 0 || L == 0 || C == 0) return HSV_OK;
  HSV_REQUIRE(op >= OP_WN_RES && op <= OP_ADD_BCAST, "frame_op: unknown op %d", op);
  HSV_REQUIRE(a || op == OP_WN_LAST, "frame_op: null input");
  HSV_REQUIRE(B <= 65535 && C <= 65535, "frame_op: grid too large");
  const int th = L >= 256 ? 256 : 128;
  frame_op_kernel<<<dim3((unsigned)((L + th - 1) / th), (unsigned)C, (unsigned)B), th, 0, hsv::as_stream(stream)>>>(
      op, a, b, c, mask, out, out2, B, C, L, s, cstride);
  return hsv::check_launch("frame_op");
}

namespace hsv {
int mha_mma_launch(const float *q, const float *k, const float *v, void *out, int blk, const int *lens, const int *vlen,
                   int B, int heads, int D, int Tq, int Tk, int64_t qbs, int64_t kbs, int64_t vbs, float scale,
                   int prescale, cudaStream_t st);
}
static int g_mha_variant = 0;   // 0: tensor cores (mha_mma.cu), 1: the fp32 CUDA-core kernel of this file (test hook)
extern "C" int hsv_set_mha_variant(int v) {
  g_mha_variant = v;
  return HSV_OK;
}

extern "C" int hsv_mha_ragged(const float *q, const float *k, const float *v, void *out, int out_mode, const int *lens,
                              const int32_t *valid_len, int B, int heads, int D, int Tq, int Tk, int64_t q_bstride,
                              int64_t k_bstride, int64_t v_bstride, float scale, int prescale_q, void *stream) {
  const char *what = out_mode ? "mha_blk16" : "mha";
  if (B == 0 || Tq == 0) return HSV_OK;
  HSV_REQUIRE(q && k && v && out, "%s: null pointer", what);
  HSV_REQUIRE(D == 96 || D == 128 || D == 64, "%s: head dim must be 64, 96 or 128 (D=%d)", what, D);
  HSV_REQUIRE(Tk > 0 && heads > 0 && heads <= (out_mode ? 32767 : 65535) && B <= 65535 && (heads * D) % 16 == 0,
              "%s: bad shape", what);
  HSV_REQUIRE(out_mode == 0 || out_mode == 1, "%s: out_mode %d", what, out_mode);
  HSV_REQUIRE(!valid_len || (!lens && Tq == Tk), "%s: valid_len is self-attention per item (Tq == Tk, no lens)", what);
  HSV_REQUIRE(!valid_len || g_mha_variant == 0, "%s: the fp32 CUDA-core variant takes no valid_len", what);
  cudaStream_t st = hsv::as_stream(stream);
  if (g_mha_variant == 0 || out_mode) {
    const int rc = hsv::mha_mma_launch(q, k, v, out, out_mode, lens, valid_len, B, heads, D, Tq, Tk, q_bstride, k_bstride,
                                       v_bstride, scale, prescale_q, st);
    if (rc != 1) return rc;
  }
  float *o = reinterpret_cast<float *>(out);
  // few (batch, head, query tile) items: 8-row tiles spread the work over more SMs
  const bool small = (int64_t)B * heads * ((Tq + 15) / 16) < 148;
#define HSV_MHA(DD)                                                                                               \
  return small ? mha_launch<DD, 2>(q, k, v, o, lens, B, heads, Tq, Tk, q_bstride, k_bstride, v_bstride, scale,   \
                                   prescale_q, st)                                                                 \
               : mha_launch<DD, 4>(q, k, v, o, lens, B, heads, Tq, Tk, q_bstride, k_bstride, v_bstride, scale,   \
                                   prescale_q, st)
  if (D == 96) { HSV_MHA(96); }
  if (D == 128) { HSV_MHA(128); }
  HSV_MHA(64);
#undef HSV_MHA
}

extern "C" int hsv_mha(const float *q, const float *k, const float *v, float *out, const int *lens, int B, int heads,
                       int D, int Tq, int Tk, int64_t q_bstride, int64_t k_bstride, int64_t v_bstride, float scale,
                       int prescale_q, void *stream) {
  return hsv_mha_ragged(q, k, v, out, 0, lens, nullptr, B, heads, D, Tq, Tk, q_bstride, k_bstride, v_bstride, scale,
                        prescale_q, stream);
}

extern "C" int hsv_mha_blk16(const float *q, const float *k, const float *v, void *out_blk16, const int *lens, int B,
                             int heads, int D, int Tq, int Tk, int64_t q_bstride, int64_t k_bstride, int64_t v_bstride,
                             float scale, int prescale_q, void *stream) {
  return hsv_mha_ragged(q, k, v, out_blk16, 1, lens, nullptr, B, heads, D, Tq, Tk, q_bstride, k_bstride, v_bstride, scale,
                        prescale_q, stream);
}

extern "C" int hsv_conv1d_c1_strided_ragged(const float *x, const float *w, const float *bias, const float *mask,
                                            const int32_t *valid_len, float *out, int B, int Cout, int64_t Lin,
                                            int64_t Lout, int k, int stride, int pad, void *stream) {
  if (B == 0 || Lout == 0) return HSV_OK;
  HSV_REQUIRE(x && w && out && k >= 1 && stride >= 1 && pad >= 0, "conv1d_c1_strided: bad arguments");
  const int grid = grid_for((int64_t)B * Cout * Lout, 256);
  cudaStream_t st = hsv::as_stream(stream);
  if (valid_len)
    conv1d_c1_strided_kernel<true><<<grid, 256, 0, st>>>(x, w, bias, mask, valid_len, out, B, Cout, Lin, Lout, k, stride,
                                                         pad);
  else
    conv1d_c1_strided_kernel<false><<<grid, 256, 0, st>>>(x, w, bias, mask, nullptr, out, B, Cout, Lin, Lout, k, stride,
                                                          pad);
  return hsv::check_launch("conv1d_c1_strided");
}

extern "C" int hsv_conv1d_c1_strided(const float *x, const float *w, const float *bias, const float *mask, float *out,
                                     int B, int Cout, int64_t Lin, int64_t Lout, int k, int stride, int pad,
                                     void *stream) {
  return hsv_conv1d_c1_strided_ragged(x, w, bias, mask, nullptr, out, B, Cout, Lin, Lout, k, stride, pad, stream);
}

extern "C" int hsv_masked_mean_ragged(const float *x, const float *mask, const int32_t *valid_len, float *out, int B,
                                      int C, int64_t L, void *stream) {
  if (B == 0 || C == 0) return HSV_OK;
  HSV_REQUIRE(x && out && L > 0, "masked_mean: bad arguments");
  cudaStream_t st = hsv::as_stream(stream);
  if (valid_len) masked_mean_kernel<true><<<(unsigned)(B * C), 128, 0, st>>>(x, valid_len, out, C, L);
  else masked_mean_kernel<false><<<(unsigned)(B * C), 128, 0, st>>>(x, nullptr, out, C, L);
  mean_div_kernel<<<B, 128, 0, st>>>(out, mask, valid_len, C, L);
  return hsv::check_launch("masked_mean");
}

extern "C" int hsv_masked_mean(const float *x, const float *mask, float *out, int B, int C, int64_t L, void *stream) {
  return hsv_masked_mean_ragged(x, mask, nullptr, out, B, C, L, stream);
}
