// Fused anti-aliased activation: UpSample1d(x2 kaiser-sinc) -> SnakeBeta -> DownSample1d(x2).
//
// Replaces alias_free_torch/act.py:23-27 (9 ATen kernels and three 2x-rate
// temporaries per call in the reference) with ONE kernel that reads x once and
// writes the result once.  Closed form (SURVEY.md §A.1), f = 12 symmetric taps:
//   y[2m-1] = 2*sum_i f[2i]  *x[clamp(m+2-i)]      (odd 2x sample)
//   y[2m]   = 2*sum_i f[2i+1]*x[clamp(m+2-i)]      (even 2x sample)
//   z[n]    = y[n] + 1/(exp(beta)+1e-9) * sin(y[n]*exp(alpha))^2
//   out[t]  = sum_j f[j]*z[clamp2L(2t+j-5)]
// x is edge-replicated on the 1x grid, z on the 2x grid (the *activated* edge
// sample is replicated, resample.py:28 / filter.py:90).
//
// Mapping: a CTA owns ROWS=8 channel rows x TILE=RUNS*R time steps.  The x tile
// (+-5 halo, clamped) is staged in shared memory with coalesced loads; each
// thread then walks a run of R consecutive outputs with the 2x signal living
// only in registers (a ring of six (odd,even) z pairs), so no 2x-rate value
// ever touches shared or global memory.  R is odd and the row pitch is
// 4 (mod 32) words, which makes every shared access of the walk conflict-free.
// Results are staged in shared memory and written back coalesced, either as
// fp32 [B,C,L] or as the fp16 "blk16" tensor-core operand layout.
//
// Ragged batches: with valid_len, row b is a sequence of Lv = valid_len[b]
// steps stored with row stride L.  Lv takes the place of L in every clamp and
// edge test, x at t >= Lv is never read, and outputs at Lv <= t < L are 0, so
// the first Lv outputs equal those of the same row run alone at L = Lv.
#include "act_core.cuh"

namespace hsv {
int act1d_mma_launch(const float *x, void *out, const float *alpha, const float *beta, int B, int C, int64_t L,
                     float sc, cudaStream_t st);
}

namespace {

using namespace hsv_act;

// The kernel body, inlined twice by act1d_kernel: once with valid_len == nullptr (constant-folded: the full-length
// path compiles to the code it had before lengths existed) and once for ragged batches.
template <int R, int OUT_MODE>
__device__ __forceinline__ void act1d_body(float *__restrict__ x_s, float *__restrict__ o_s, uint64_t &bar,
                                           const float *__restrict__ x, void *__restrict__ outp,
                                           const float *__restrict__ alpha, const float *__restrict__ beta,
                                           const int32_t *__restrict__ valid_len, int C, int64_t L, int64_t nrows,
                                           int ntiles, int64_t Lp, float sc, int cw) {
  using K = Cfg<R>;

  const int tid = threadIdx.x;
  int tile, ch;        // time tile; channel of this thread's row
  int64_t row0;        // first of the CTA's 8 (b, channel) rows
  const int c = tid % ROWS, run = tid / ROWS;
  if (OUT_MODE == 1) {
    // swizzled operand output: grid = (tiles x units-per-chunk, chunks, batch), no divisions.  The cw/8 CTAs that
    // fill the 16-byte units of the same operand rows are adjacent in launch order, so their partial-sector
    // writes meet in L2.
    const int lgu = cw == 64 ? 3 : (cw == 32 ? 2 : 1);  // log2(units per chunk)
    tile = (int)(blockIdx.x >> lgu);
    const int c0 = (int)blockIdx.y * cw + (int)(blockIdx.x & ((1u << lgu) - 1u)) * 8;
    row0 = (int64_t)blockIdx.z * C + c0;
    ch = c0 + c;
  } else {
    tile = blockIdx.x % ntiles;
    row0 = (int64_t)(blockIdx.x / ntiles) * ROWS;
    ch = (int)((row0 + c) % C);
  }
  const int64_t t0 = (int64_t)tile * K::TILE;
  const int64_t row = row0 + c;
  // PDL: let the next kernel start its prologue now; parameters are static, so load them before waiting
  // for the producer of x
  hsv::pdl_launch_dependents();
  float al = 0.f, be = 0.f;
  if (row < nrows) {
    al = __ldg(alpha + ch);
    be = __ldg(beta + ch);
  }
  hsv::pdl_wait();
  // valid lengths are data of the forward (not static): read after the wait
  // valid length of this thread's row (32-bit: one register across the kernel; with valid_len == nullptr every use
  // below folds to L)
  int lv = 0;
  if (valid_len && row < nrows) {
    const int v = __ldg(valid_len + (OUT_MODE == 1 ? (int64_t)blockIdx.z : row / C));
    lv = v < 0 ? 0 : (v > L ? (int)L : v);
  } else if (valid_len) {
    lv = (int)L;
  }
  const int64_t Lv = valid_len ? (int64_t)lv : L;

  // ---- stage the x tile ----
  // interior tiles of 16-byte-aligned rows: one 1-D bulk TMA copy per row (no issue slots, no registers);
  // edge tiles / unaligned rows: plain loads with the replicate clamp of the 1x grid.
  // lanes 0..7 of every warp hold the valid lengths of rows 0..7 (c == lane % 8); with valid_len the tile must lie
  // inside every row's valid part
  bool fast = ((L & 3) == 0) && t0 >= K::XOFF && t0 + K::TILE + K::XOFF <= L && row0 + ROWS <= nrows &&
              ((reinterpret_cast<uintptr_t>(x) & 15) == 0);
  if (valid_len) fast = __all_sync(0xffffffffu, t0 + K::TILE + K::XOFF <= Lv) && fast;
  if (fast) {
    const uint32_t bar_a = static_cast<uint32_t>(__cvta_generic_to_shared(&bar));
    if (tid == 0) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a));
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    constexpr uint32_t ROW_BYTES = (K::TILE + 2 * K::XOFF) * 4;
    if (tid == 0)
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"(ROW_BYTES * ROWS)
                   : "memory");
    if (tid < ROWS) {
      const float *src = x + (row0 + tid) * L + (t0 - K::XOFF);
      const uint32_t dst = static_cast<uint32_t>(__cvta_generic_to_shared(x_s + tid * K::PITCH));
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                   "l"(src), "r"(ROW_BYTES), "r"(bar_a)
                   : "memory");
    }
    uint32_t ok = 0;
    while (!ok) {
      asm volatile(
          "{\n\t"
          ".reg .pred p;\n\t"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\t"
          "selp.u32 %0, 1, 0, p;\n\t"
          "}"
          : "=r"(ok)
          : "r"(bar_a)
          : "memory");
    }
  } else {
    // all loads of a thread are issued before the first store (one exposed memory latency, not one per row)
    constexpr int NLD = (ROWS * K::XW + NT - 1) / NT;
    float v[NLD];
#pragma unroll
    for (int i = 0; i < NLD; ++i) {
      const int idx = tid + NT * i;
      const int cc = idx / K::XW, p = idx - cc * K::XW;
      const int64_t rw = row0 + cc;
      const int64_t t = t0 - K::XOFF + p;
      const int Lm1 = (valid_len ? __shfl_sync(0xffffffffu, (int)Lv, cc & (ROWS - 1)) : (int)L) - 1;
      const int tc = t < 0 ? 0 : (t > Lm1 ? Lm1 : (int)t);
      v[i] = (idx < ROWS * K::XW && rw < nrows && Lm1 >= 0) ? __ldg(x + rw * L + tc) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < NLD; ++i) {
      const int idx = tid + NT * i;
      const int cc = idx / K::XW, p = idx - cc * K::XW;
      if (idx < ROWS * K::XW) x_s[cc * K::PITCH + p] = v[i];
    }
    __syncthreads();
  }

  const int64_t ta = t0 + (int64_t)run * R;
  float outv[R];
  const bool active = row < nrows && ta < L;
  if (row < nrows && ta < Lv) {
    const float *xw = x_s + c * K::PITCH + run * R + (K::XOFF - 5);
    act_run<R>(xw, outv, al, be, ta, Lv, x + row * L, sc);
  }

  // ---- stage results, write back coalesced ----
  if (OUT_MODE == 0) {
    if (active) {
      float *o = o_s + c * K::OPITCH + run * R;
      if (valid_len && ta + R > Lv) {   // the run reaches past the row's valid part: zero tail
#pragma unroll
        for (int j = 0; j < R; ++j) o[j] = ta + j < Lv ? outv[j] : 0.f;
      } else {
#pragma unroll
        for (int j = 0; j < R; ++j) o[j] = outv[j];
      }
    }
    __syncthreads();
    float *out = reinterpret_cast<float *>(outp);
    for (int idx = tid; idx < ROWS * K::TILE; idx += NT) {
      const int cc = idx / K::TILE, p = idx - cc * K::TILE;
      const int64_t r = row0 + cc, t = t0 + p;
      if (r < nrows && t < L) out[r * L + t] = o_s[cc * K::OPITCH + p];
    }
  } else {
    __half *o_h = reinterpret_cast<__half *>(o_s);  // [TILE][8]
    if (active) {
      if (valid_len && ta + R > Lv) {
#pragma unroll
        for (int j = 0; j < R; ++j) o_h[(run * R + j) * 8 + c] = __float2half_rn(ta + j < Lv ? outv[j] : 0.f);
      } else {
#pragma unroll
        for (int j = 0; j < R; ++j) o_h[(run * R + j) * 8 + c] = __float2half_rn(outv[j]);
      }
    }
    __syncthreads();
    // rows row0..row0+7 are one 8-channel unit of one batch item (C % 8 == 0)
    const uint4 *src = reinterpret_cast<const uint4 *>(o_s);
    // the swizzled offset is shifts and xors (cw is a power of two)
    const int lg = cw == 64 ? 7 : (cw == 32 ? 6 : 5);              // log2(row bytes)
    const uint32_t mask = (uint32_t)(cw >> 3) - 1u;
    const uint32_t ub = (blockIdx.x & mask) << 4;                  // byte offset of this CTA's unit in a row
    uint8_t *base = reinterpret_cast<uint8_t *>(outp) + (((int64_t)blockIdx.z * gridDim.y + blockIdx.y) * Lp << lg);
    const uint64_t r0 = (uint64_t)(HSV_BLK_PAD + t0);
    for (int p = tid; p < K::TILE; p += NT) {
      if (t0 + p < L) {
        const uint64_t lin = ((r0 + (uint64_t)p) << lg) + ub;
        *reinterpret_cast<uint4 *>(base + (lin ^ (((lin >> 7) & mask) << 4))) = src[p];
      }
    }
  }
}

template <int R, int OUT_MODE>
// 7 CTAs per SM need <= 72 registers: the fp16-operand kernels (both bodies inlined) meet it only with the bound, the
// fp32-output ones without it (with it, R = 25 spills)
__global__ void __launch_bounds__(NT, OUT_MODE == 1 ? 7 : 0) act1d_kernel(const float *__restrict__ x, void *__restrict__ outp,
                                                   const float *__restrict__ alpha,
                                                   const float *__restrict__ beta,
                                                   const int32_t *__restrict__ valid_len, int C, int64_t L,
                                                   int64_t nrows, int ntiles, int64_t Lp, float sc, int cw) {
  using K = Cfg<R>;
  // x_s[c][p] holds x[row0+c][t0 - XOFF + p]; XOFF = 8 keeps the tile start 16-byte aligned for TMA
  __shared__ __align__(16) float x_s[ROWS * K::PITCH];
  __shared__ __align__(16) float o_s[OUT_MODE == 0 ? ROWS * K::OPITCH : K::TILE * 4];
  __shared__ __align__(8) uint64_t bar;
  if (valid_len)
    act1d_body<R, OUT_MODE>(x_s, o_s, bar, x, outp, alpha, beta, valid_len, C, L, nrows, ntiles, Lp, sc, cw);
  else
    act1d_body<R, OUT_MODE>(x_s, o_s, bar, x, outp, alpha, beta, nullptr, C, L, nrows, ntiles, Lp, sc, cw);
}

int g_act_run = 0;      // bring-up aid: force the run length (17 or 25); 0 = automatic
#ifndef HSV_ACT_MMA_AUTO
#define HSV_ACT_MMA_AUTO 0   // policy of variant 0 (auto): 1 = tensor-core kernel for L >= 256 (set once it wins on B200)
#endif
int g_act_mma = 0;      // fp16-operand output: 0 = auto, 1 = CUDA-core kernel (act1d.cu), 2 = tensor-core kernel (act1d_mma.cu)

// hsv_last_launch_config, family 1: run length R (0 for the tensor-core kernel), act1d_mma ran, out_mode, valid_len
// given, launch count
void note_launch(int R, int mma, int out_mode, int has_valid_len) {
  int *last = hsv::g_last_launch[1];
  last[0] = R;
  last[1] = mma;
  last[2] = out_mode;
  last[3] = has_valid_len;
  ++last[4];
}

template <int R, int OUT_MODE>
int launch(const float *x, void *out, const float *alpha, const float *beta, const int32_t *valid_len, int B, int C,
           int64_t L, float sc, cudaStream_t st) {
  using K = Cfg<R>;
  const int64_t nrows = (int64_t)B * C;
  const int64_t ntiles = (L + K::TILE - 1) / K::TILE;
  const int64_t ngrp = (nrows + ROWS - 1) / ROWS;
  const int64_t nblk = ntiles * ngrp;
  HSV_REQUIRE(nblk < (1ll << 31) && ntiles < (1ll << 31), "act1d: grid too large");
  cudaLaunchConfig_t cfg = {};
  if (OUT_MODE == 1) {
    const int cwl = hsv::blk_cw(C);
    HSV_REQUIRE(ntiles * (cwl / 8) < (1ll << 31) && C / cwl <= 65535 && B <= 65535, "act1d: grid too large");
    cfg.gridDim = dim3((unsigned)(ntiles * (cwl / 8)), (unsigned)(C / cwl), (unsigned)B);
  } else {
    cfg.gridDim = dim3((unsigned)nblk);
  }
  cfg.blockDim = dim3(NT);
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = hsv::g_pdl ? 1 : 0;
  const int nt_i = (int)ntiles;
  const int64_t Lp = hsv::blk16_rows(L);
  const int cw = OUT_MODE == 1 ? hsv::blk_cw(C) : 0;
  note_launch(R, 0, OUT_MODE, valid_len != nullptr);
  cudaError_t e = cudaLaunchKernelEx(&cfg, act1d_kernel<R, OUT_MODE>, x, out, alpha, beta, valid_len, C, L, nrows, nt_i, Lp,
                                     sc, cw);
  if (e != cudaSuccess) {
    cudaGetLastError();
    hsv::set_error("act1d_snakebeta: launch failed: %s", cudaGetErrorString(e));
    return HSV_ERR_CUDA;
  }
  return hsv::check_launch("act1d_snakebeta");
}

}  // namespace

// bring-up aid (forced run length, bits 8..15); not part of the drop-in contract
extern "C" int hsv_set_act_variant(int v) {
  g_act_run = v >> 8;  // bits 8..: forced run length
  g_act_mma = v & 3;   // bits 0..1: tensor-core variant policy (0 auto, 1 off, 2 forced)
  return HSV_OK;
}

extern "C" int hsv_act1d_snakebeta(const float *x, void *out, const float *alpha, const float *beta, int B,
                                   int C, int64_t L, int out_mode, float in_scale, void *stream) {
  return hsv_act1d_snakebeta_ragged(x, out, alpha, beta, nullptr, B, C, L, out_mode, in_scale, stream);
}

extern "C" int hsv_act1d_snakebeta_ragged(const float *x, void *out, const float *alpha, const float *beta,
                                          const int32_t *valid_len, int B, int C, int64_t L, int out_mode,
                                          float in_scale, void *stream) {
  if (B == 0 || L == 0) return HSV_OK;  // empty batch / sequence
  HSV_REQUIRE(x && out && alpha && beta, "act1d: null pointer");
  HSV_REQUIRE(B >= 0 && C > 0 && L >= 0, "act1d: bad shape B=%d C=%d L=%lld", B, C, (long long)L);
  HSV_REQUIRE(out_mode == 0 || out_mode == 1, "act1d: out_mode must be 0 (fp32 NCL) or 1 (fp16 blk16)");
  if (B == 0 || L == 0) return HSV_OK;
  cudaStream_t st = hsv::as_stream(stream);
  // Run length per thread R (a CTA covers 8 rows x 16 R steps; every thread also evaluates a 5-step halo): longer runs
  // waste less on the halo (R = 25: 1.2x redundant 2x-rate work, 3.97 TB/s on [16,32,480000] vs 3.06 for R = 17), shorter
  // runs give more CTAs.  Seven CTAs fit an SM (66 registers), so the launch runs in ceil(CTAs / (148 x 7)) waves of
  // ~(R + 5) steps each: pick the R that minimises waves x (R + 5).  This matters at batch 1: the three late stages of
  // the vocoder are 2.56 M elements each = 1180 CTAs at R = 17, i.e. 1.14 waves (7.6 us); R = 21 fits one wave.
  const int64_t groups = ((int64_t)B * C + ROWS - 1) / ROWS;
  int R = 17;
  if (g_act_run) {
    R = g_act_run;
  } else {
    int64_t best = -1;
    // R = 9: only for launches that leave most SMs empty at R = 17 (the SourceNetwork / early stages at batch 1: 64
    // CTAs): twice the CTAs, half the serial work per thread
    static const bool no_r9 = getenv("HSV_ACT_NO_R9") != nullptr;   // A/B switch
    const bool tiny = !no_r9 && groups * ((L + 17 * RUNS - 1) / (17 * RUNS)) < 148;
    for (int cand : {9, 17, 21, 25}) {
      if (cand == 9 && !tiny) continue;
      const int64_t ctas = groups * ((L + cand * RUNS - 1) / (cand * RUNS));
      const int64_t waves = (ctas + 148 * 7 - 1) / (148 * 7);
      // many waves: the halo overhead decides (cost per element ~ (R + 5) / R); few: the wave count does
      const int64_t cost = waves * (cand + 5) * 1000 / (waves >= 4 ? cand : 1) / (waves >= 4 ? waves : 1);
      if (best < 0 || cost < best) {
        best = cost;
        R = cand;
      }
    }
  }
  HSV_REQUIRE(R == 9 || R == 17 || R == 21 || R == 25, "act1d: run length must be 9, 17, 21 or 25");
  if (out_mode == 0)
    return R == 25 ? launch<25, 0>(x, out, alpha, beta, valid_len, B, C, L, in_scale, st)
                   : (R == 21 ? launch<21, 0>(x, out, alpha, beta, valid_len, B, C, L, in_scale, st)
                              : (R == 17 ? launch<17, 0>(x, out, alpha, beta, valid_len, B, C, L, in_scale, st)
                                         : launch<9, 0>(x, out, alpha, beta, valid_len, B, C, L, in_scale, st)));
  HSV_REQUIRE(C % 16 == 0, "act1d: blk16 output needs C %% 16 == 0 (C=%d)", C);
  // tensor-core FIR variant (act1d_mma.cu): every shape with at least half a tile of work per row; the CUDA-core
  // kernel keeps the tiny sequences (its tiles are 8 x 272 instead of 8 x 512)
  HSV_REQUIRE(!(valid_len && g_act_mma == 2), "act1d: the forced tensor-core variant takes no valid lengths");
  if (g_act_mma == 2 || (g_act_mma == 0 && HSV_ACT_MMA_AUTO && L >= 256 && !valid_len)) {
    const int rc = hsv::act1d_mma_launch(x, out, alpha, beta, B, C, L, in_scale, st);
    if (rc != 1) {
      note_launch(0, 1, 1, 0);
      return rc;
    }
    HSV_REQUIRE(g_act_mma != 2, "act1d: shape not eligible for the forced tensor-core variant");
  }
  return R == 25 ? launch<25, 1>(x, out, alpha, beta, valid_len, B, C, L, in_scale, st)
                 : (R == 21 ? launch<21, 1>(x, out, alpha, beta, valid_len, B, C, L, in_scale, st)
                            : (R == 17 ? launch<17, 1>(x, out, alpha, beta, valid_len, B, C, L, in_scale, st)
                                       : launch<9, 1>(x, out, alpha, beta, valid_len, B, C, L, in_scale, st)));
}
