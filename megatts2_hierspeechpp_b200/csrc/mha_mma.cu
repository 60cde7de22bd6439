// Multi-head attention of the step before the vocoder (timm Attention inside DiTConVBlock, modules.py:390-411; the
// StyleEncoder's MultiHeadAttention, styleencoder.py:61-66 / attentions.py:152-190) on the tensor cores.
//
// The problem is tiny (T = 500 frames, 2 heads, D = 96: 0.1 GFLOP) and ran as a latency chain on the FP32 pipe (31 us per
// call x 24 calls = the largest single item of the synthesizer call).  Here:
//   * a CLUSTER of 2 CTAs = 16 query rows of one (batch, head); its 2 x 4 warps SPLIT THE KEYS (tiles of 16 keys,
//     warp j of 8 takes tiles j, j+8, ...) with private online-softmax state (flash-decoding): every warp has 1/8 of
//     the serial work and there is no barrier inside the key loop.  The warps of a CTA merge through shared memory,
//     CTA 1 hands its merged (m, l, O) to CTA 0 through distributed shared memory, CTA 0 stores.  64 (q-tile, head)
//     items become 128 CTAs: one wave on the 148 SMs.
//   * products on mma.sync.m16n8k16 (f16 x f16 -> f32).  The LOGITS keep fp32-level accuracy: Q and K are split into
//     fp16 hi + fp16 lo and Q K^T is three MMAs (hi*hi + hi*lo + lo*hi; the dropped lo*lo term is 2^-22 relative) --
//     softmax turns an absolute logit error into a relative weight error, and real checkpoints have large logits.
//     P V uses plain fp16 operands (P in [0, 1], V rounded once; fp32 accumulate): the same rounding the very next op
//     (the tcgen05 proj conv's operand pack) applies to the result anyway.  mma.sync is the right tool here: a
//     16 x 16 x 96 tile per step is far below what a tcgen05 M = 128 tile needs.
//   * K / V tiles stream global -> shared with 16-byte cp.async, double-buffered per warp, in the tensors' own
//     channel-major fp32 layout ([d][t]: exactly the "col" B operand of Q K^T and of P V); fragments are converted
//     to hi/lo fp16 in registers, each element once (a warp owns its tiles).  Pitches 20 / 24 words make every
//     fragment load bank-conflict free.
#include <cooperative_groups.h>

#include "hsv_common.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int KT = 16;          // keys per warp tile
constexpr int QT = 16;          // query rows per CTA
constexpr int KP = 20;          // K stage pitch (words):  (2c * KP + g) mod 32 distinct for c < 4, g < 8
constexpr int VP = 24;          // V stage pitch (words):  (g * VP + 2c) distinct within a half-warp (LDS.64)
constexpr int NWARP = 4;
constexpr int NSPLIT = 2;      // CTAs per cluster (key split across CTAs)

__device__ __forceinline__ void cp16(void *dst, const void *src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src)
               : "memory");
}
__device__ __forceinline__ void cp_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// fp32 pair -> (hi, lo) fp16 pairs packed for an MMA register
__device__ __forceinline__ void split2(float x, float y, uint32_t &hi, uint32_t &lo) {
  const __half2 h = __floats2half2_rn(x, y);
  const float2 hf = __half22float2(h);
  const __half2 l = __floats2half2_rn(x - hf.x, y - hf.y);
  hi = *reinterpret_cast<const uint32_t *>(&h);
  lo = *reinterpret_cast<const uint32_t *>(&l);
}

__device__ __forceinline__ uint32_t pack2(float x, float y) {
  const __half2 h = __floats2half2_rn(x, y);
  return *reinterpret_cast<const uint32_t *>(&h);
}

__device__ __forceinline__ void mma16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// BLK: the result is written as the fp16 blk16 operand of the following proj conv (out = blk16 buffer of heads*D channels)
// instead of fp32 [B, heads*D, Tq]
// VLEN: per-item lengths (self-attention of a ragged batch): item b has n = vlen[b] queries and keys, stored with the row
// pitches Tq / Tk.  It runs exactly as its own launch with Tq = Tk = n (same key tiles, same zero fill and -inf past n),
// and its rows [n, Tq) are written as zero; a query tile wholly past n does no key work.
template <int D, bool BLK, bool VLEN>
__global__ void __cluster_dims__(1, NSPLIT, 1) __launch_bounds__(32 * NWARP)
mha_mma_kernel(const float *__restrict__ q, const float *__restrict__ k, const float *__restrict__ v, void *__restrict__ out,
               const int *__restrict__ lens, const int *__restrict__ vlen, int Tq, int Tk, int64_t qbs, int64_t kbs,
               int64_t vbs, int heads, float scale, int prescale, int fast) {
  constexpr int KS = D / 16;                      // k-steps of Q K^T
  constexpr int NT = D / 8;                       // n-tiles of P V
  constexpr int STAGE = D * (KP + VP);            // words per (K, V) stage of one warp
  extern __shared__ __align__(16) float sm[];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int g = lane >> 2, c = lane & 3;
  cg::cluster_group cluster = cg::this_cluster();
  const int split = (int)(blockIdx.y % NSPLIT);   // == cluster.block_rank() for cluster dims (1, NSPLIT, 1)
  const int b = blockIdx.z, h = blockIdx.y / NSPLIT, q0 = blockIdx.x * QT;
  const int jw = split * NWARP + w;               // this warp's index among the cluster's key streams
  constexpr int NJ = NWARP * NSPLIT;
  const float *qb = q + (int64_t)b * qbs + (int64_t)h * D * Tq;
  const float *kb = k + (int64_t)b * kbs + (int64_t)h * D * Tk;
  const float *vb = v + (int64_t)b * vbs + (int64_t)h * D * Tk;
  const int len = lens ? lens[b] : 0x7fffffff;
  // logical query / key counts of this item (the row pitches stay Tq / Tk)
  const int nv = VLEN ? min(max(vlen[b], 0), min(Tq, Tk)) : 0;
  const int tq = VLEN ? nv : Tq, tk = VLEN ? nv : Tk;
  const int ntiles = (tk + KT - 1) / KT;
  float *my = sm + w * 2 * STAGE;                 // this warp's two stages

  // merged values per thread.  fp32 output: value i = (d, r) with rows fastest (64-byte segments of a channel row);
  // blk16 output: a thread owns whole 16-byte units (8 consecutive channels of one row): unit u = tid + 128 * (i / 8)
  constexpr int NUNIT = QT * D / 8;
  constexpr int PER = BLK ? 8 * ((NUNIT + 32 * NWARP - 1) / (32 * NWARP)) : QT * D / (32 * NWARP);
  auto where = [&](int i, int &d, int &r) -> bool {
    if (BLK) {
      const int u = tid + 32 * NWARP * (i >> 3);
      d = 8 * (u / QT) + (i & 7);
      r = u % QT;
      return u < NUNIT;
    }
    const int idx = tid + 32 * NWARP * i;
    d = idx / QT;
    r = idx - d * QT;
    return true;
  };
  // CTA 0's store of the tile's rows [q0, min(q0 + QT, Tq))
  auto store = [&](const float (&accv)[PER]) {
    if (BLK) {
      const int C = heads * D;
      const int cw = hsv::blk_cw(C);
      const int64_t Lp = hsv::blk16_rows(Tq);
#pragma unroll
      for (int j = 0; j < PER / 8; ++j) {
        int d, r;
        if (!where(8 * j, d, r) || q0 + r >= Tq) continue;
        __half2 hh[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) hh[e] = __floats2half2_rn(accv[8 * j + 2 * e], accv[8 * j + 2 * e + 1]);
        *reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(out) +
                                   hsv::blk_unit_offset(cw, Lp, C, b, h * D + d, HSV_BLK_PAD + q0 + r)) =
            *reinterpret_cast<uint4 *>(hh);
      }
    } else {
      float *ob = reinterpret_cast<float *>(out) + ((int64_t)b * heads + h) * D * Tq;
#pragma unroll
      for (int i = 0; i < PER; ++i) {
        int d, r;
        where(i, d, r);
        if (q0 + r < Tq) ob[(int64_t)d * Tq + q0 + r] = accv[i];
      }
    }
  };
  if (VLEN && q0 >= tq) {                         // every row of the tile is past the item: zero rows, no key work
    if (split == 0) {
      float zero[PER];
#pragma unroll
      for (int i = 0; i < PER; ++i) zero[i] = 0.f;
      store(zero);
    }
    return;                                       // both CTAs of the cluster leave here (same q0, same b)
  }

  // per-lane constants of the tile copy: chunk ch = lane + 32 i  ->  d = (lane >> 2) + 8 i, 4 keys at (lane & 3) * 4
  const int ld_d0 = lane >> 2, ld_x4 = (lane & 3) * 4;
  const float *ld_k = kb + (int64_t)ld_d0 * Tk + ld_x4, *ld_v = vb + (int64_t)ld_d0 * Tk + ld_x4;
  const uint32_t ld_sk = (uint32_t)__cvta_generic_to_shared(my + ld_d0 * KP + ld_x4);
  const uint32_t ld_sv = (uint32_t)__cvta_generic_to_shared(my + D * KP + ld_d0 * VP + ld_x4);
  const int64_t ld_step = (int64_t)8 * Tk;
  auto load_tile = [&](int t, int stage) {
    const int k0 = t * KT;
    if (fast && k0 + KT <= tk) {
      const float *gk = ld_k + k0, *gv = ld_v + k0;
      const uint32_t sk = ld_sk + stage * (STAGE * 4), sv = ld_sv + stage * (STAGE * 4);
#pragma unroll
      for (int i = 0; i < D / 8; ++i) {                           // 16-byte chunks: 4 per row, 8 rows per step
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sk + i * (8 * KP * 4)), "l"(gk) : "memory");
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sv + i * (8 * VP * 4)), "l"(gv) : "memory");
        gk += ld_step;
        gv += ld_step;
      }
    } else {
      // ragged last tile / Tk % 4 != 0 / unaligned tensors: 4-byte cp.async with zero fill past Tk (src-size 0) -- still
      // asynchronous (a plain load -> store loop here was a chain of L2 round trips: 29 us for the StyleEncoder's T = 150)
      const uint32_t sk0 = (uint32_t)__cvta_generic_to_shared(my + stage * STAGE);
      const uint32_t sv0 = sk0 + D * KP * 4;
      const int j = lane & (KT - 1), dq = lane / KT;             // 16 keys x 2 rows per warp step
      const int ok = (k0 + j < tk) ? 4 : 0;
      const int64_t col = ok ? k0 + j : 0;                       // keep the (unused) source address in bounds
#pragma unroll 8
      for (int d = dq; d < D; d += 32 / KT) {
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(sk0 + (d * KP + j) * 4),
                     "l"(kb + (int64_t)d * Tk + col), "r"(ok) : "memory");
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(sv0 + (d * VP + j) * 4),
                     "l"(vb + (int64_t)d * Tk + col), "r"(ok) : "memory");
      }
    }
    cp_commit();
  };

  // ---- Q tile [D][16 rows] -> shared (cp.async, same [d][t] form as a K tile), then the first K / V tile ----
  float *Qs = sm + NWARP * 2 * STAGE + QT * (D + 1) + 2 * QT;     // behind the peer's landing zone; pitch KP
  {
    const bool qfast = (Tq % 4 == 0) && q0 + QT <= tq && ((reinterpret_cast<uintptr_t>(q) & 15) == 0) && (qbs % 4 == 0);
    if (qfast) {
      for (int ch = tid; ch < D * 4; ch += 32 * NWARP) {
        const int d = ch >> 2, x4 = (ch & 3) * 4;
        cp16(Qs + d * KP + x4, qb + (int64_t)d * Tq + q0 + x4);
      }
    } else {                                                     // ragged / unaligned: 4-byte copies, zero fill past Tq
      const uint32_t sq0 = (uint32_t)__cvta_generic_to_shared(Qs);
      const int r = tid & (QT - 1);
      const int ok = (q0 + r < tq) ? 4 : 0;
      const int64_t col = ok ? q0 + r : 0;
#pragma unroll 4
      for (int d = tid / QT; d < D; d += 32 * NWARP / QT)
        asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(sq0 + (d * KP + r) * 4),
                     "l"(qb + (int64_t)d * Tq + col), "r"(ok) : "memory");
    }
    cp_commit();
  }
  if (jw < ntiles) load_tile(jw, 0);
  else cp_commit();                                // keep the group count uniform
  cp_wait<1>();                                    // this thread's Q chunks have landed (tile 0 may still be in flight)
  __syncthreads();

  // ---- Q fragments (hi, lo), rows g and g + 8 of the CTA's 16, all D: built once ----
  uint32_t qh[KS][4], ql[KS][4];
  {
    const float sq = prescale ? scale : 1.f;
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
      const float *qp = Qs + (16 * ks + 2 * c) * KP + g;          // A[m = row][k = d]: Qs[d][row]
      split2(qp[0] * sq, qp[KP] * sq, qh[ks][0], ql[ks][0]);              // a0: row g,     d 2c, 2c+1
      split2(qp[8] * sq, qp[KP + 8] * sq, qh[ks][1], ql[ks][1]);          // a1: row g + 8
      split2(qp[8 * KP] * sq, qp[9 * KP] * sq, qh[ks][2], ql[ks][2]);     // a2: row g,     d 2c+8, 2c+9
      split2(qp[8 * KP + 8] * sq, qp[9 * KP + 8] * sq, qh[ks][3], ql[ks][3]);   // a3: row g + 8
    }
  }

  float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};   // rows g, g + 8 (partial over this warp's keys)
  float o[NT][4];
#pragma unroll
  for (int nt = 0; nt < NT; ++nt) o[nt][0] = o[nt][1] = o[nt][2] = o[nt][3] = 0.f;

  int it = 0;
  for (int t = jw; t < ntiles; t += NJ, ++it) {
    if (t + NJ < ntiles) {
      load_tile(t + NJ, (it + 1) & 1);          // the other stage was released by the __syncwarp ending iteration it-1
      cp_wait<1>();
    } else {
      cp_wait<0>();
    }
    __syncwarp();
    const float *Ks = my + (it & 1) * STAGE, *Vs = Ks + D * KP;
    const int k0 = t * KT;

    // ---- S = Q K^T : 16 rows x 16 keys = two n-tiles ----
    float s[2][4];
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) s[nt][0] = s[nt][1] = s[nt][2] = s[nt][3] = 0.f;
#pragma unroll
    for (int ks = 0; ks < KS; ++ks) {
#pragma unroll
      for (int nt = 0; nt < 2; ++nt) {
        const float *kp = Ks + (16 * ks + 2 * c) * KP + nt * 8 + g;     // B[k = d][n = key]
        uint32_t bh0, bl0, bh1, bl1;
        split2(kp[0], kp[KP], bh0, bl0);
        split2(kp[8 * KP], kp[9 * KP], bh1, bl1);
        mma16816(s[nt], qh[ks], bh0, bh1);
        mma16816(s[nt], qh[ks], bl0, bl1);
        mma16816(s[nt], ql[ks], bh0, bh1);
      }
    }
    // ---- masks, online softmax (row g: regs 0, 1; row g + 8: regs 2, 3; keys nt*8 + 2c + {0, 1}) ----
    float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int j = k0 + nt * 8 + 2 * c + (e & 1);
        const int qi = q0 + g + 8 * (e >> 1);
        float a = prescale ? s[nt][e] : s[nt][e] * scale;
        if (lens && (qi >= len || j >= len)) a = -1e4f;      // masked_fill(mask == 0, -1e4)
        if (j >= tk) a = -INFINITY;                          // padding of the last key tile
        s[nt][e] = a;
        mx[e >> 1] = fmaxf(mx[e >> 1], a);
      }
    float corr[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
      mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
      const float m_new = fmaxf(m_run[r], mx[r]);            // finite: a tile always holds at least one key < Tk
      corr[r] = __expf(m_run[r] - m_new);
      m_run[r] = m_new;
    }
    float sum[2] = {0.f, 0.f};
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float p = __expf(s[nt][e] - m_run[e >> 1]);
        s[nt][e] = p;
        sum[e >> 1] += p;
      }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      sum[r] += __shfl_xor_sync(0xffffffffu, sum[r], 1);
      sum[r] += __shfl_xor_sync(0xffffffffu, sum[r], 2);
      l_run[r] = l_run[r] * corr[r] + sum[r];
    }
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      o[nt][0] *= corr[0];
      o[nt][1] *= corr[0];
      o[nt][2] *= corr[1];
      o[nt][3] *= corr[1];
    }
    // ---- O += P V : P's accumulator fragments ARE the A fragments of a k = 16 step (plain fp16 operands) ----
    uint32_t ph[4];
    ph[0] = pack2(s[0][0], s[0][1]);              // row g,     keys 2c, 2c+1
    ph[1] = pack2(s[0][2], s[0][3]);              // row g + 8
    ph[2] = pack2(s[1][0], s[1][1]);              // row g,     keys 2c+8, 2c+9
    ph[3] = pack2(s[1][2], s[1][3]);              // row g + 8
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      const float *vp = Vs + (nt * 8 + g) * VP + 2 * c;                 // B[k = key][n = d]
      const float2 v0 = *reinterpret_cast<const float2 *>(vp);
      const float2 v1 = *reinterpret_cast<const float2 *>(vp + 8);
      mma16816(o[nt], ph, pack2(v0.x, v0.y), pack2(v1.x, v1.y));
    }
    __syncwarp();      // every lane is done with this stage before the next iteration's load overwrites it
  }

  // ---- merge: warps of a CTA through shared memory, CTA 1 -> CTA 0 through distributed shared memory ----
  __syncthreads();                                  // all stages are dead: reuse the front of shared memory
  float *Om = sm;                                   // [NWARP][QT][D + 1]
  float *Mm = Om + NWARP * QT * (D + 1);            // [NWARP][QT]
  float *Lm = Mm + NWARP * QT;
  float *Ro = sm + NWARP * 2 * STAGE;               // landing zone for the peer CTA (never aliases a stage): [QT][D + 1]
  float *Rm = Ro + QT * (D + 1);                    // [QT], [QT]
  float *Rl = Rm + QT;
  {
    float *ow = Om + w * QT * (D + 1);
#pragma unroll
    for (int nt = 0; nt < NT; ++nt) {
      const int d = nt * 8 + 2 * c;
      ow[g * (D + 1) + d] = o[nt][0];
      ow[g * (D + 1) + d + 1] = o[nt][1];
      ow[(g + 8) * (D + 1) + d] = o[nt][2];
      ow[(g + 8) * (D + 1) + d + 1] = o[nt][3];
    }
    if (c == 0) {
      Mm[w * QT + g] = m_run[0];
      Mm[w * QT + g + 8] = m_run[1];
      Lm[w * QT + g] = l_run[0];
      Lm[w * QT + g + 8] = l_run[1];
    }
  }
  __syncthreads();
  // per (row, warp) weights exp(m_w - m) and the CTA's (m, l): 64 threads, once
  float *Fm = Lm + NWARP * QT;                      // [NWARP][QT] weights, then [QT] m, [QT] l
  float *Cm = Fm + NWARP * QT, *Cl = Cm + QT;
  if (tid < QT) {
    const int r = tid;
    float m = Mm[r];
#pragma unroll
    for (int ww = 1; ww < NWARP; ++ww) m = fmaxf(m, Mm[ww * QT + r]);
    float l = 0.f;
#pragma unroll
    for (int ww = 0; ww < NWARP; ++ww) {
      const float mw = Mm[ww * QT + r];
      const float f = mw == -INFINITY ? 0.f : __expf(mw - m);  // a warp that saw no tile contributes nothing
      Fm[ww * QT + r] = f;
      l = fmaf(Lm[ww * QT + r], f, l);
    }
    Cm[r] = m;
    Cl[r] = l;
  }
  __syncthreads();
  float accv[PER];
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    int d, r;
    float acc = 0.f;
    if (where(i, d, r)) {
#pragma unroll
      for (int ww = 0; ww < NWARP; ++ww) acc = fmaf(Om[(ww * QT + r) * (D + 1) + d], Fm[ww * QT + r], acc);
    }
    accv[i] = acc;
  }
  if (split != 0) {                                 // hand (m, l, O) to CTA 0 of the cluster
    float *po = cluster.map_shared_rank(Ro, 0), *pm = cluster.map_shared_rank(Rm, 0), *pl = cluster.map_shared_rank(Rl, 0);
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      int d, r;
      if (where(i, d, r)) po[r * (D + 1) + d] = accv[i];
    }
    if (tid < QT) {
      pm[tid] = Cm[tid];
      pl[tid] = Cl[tid];
    }
  }
  cluster.sync();                                   // release / acquire over the cluster: the peer's stores are visible
  if (split != 0) return;
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    int d, r;
    if (!where(i, d, r)) continue;
    const float m0 = Cm[r], m1 = Rm[r];
    const float m = fmaxf(m0, m1);                   // CTA 0 always holds tile 0: finite
    const float f0 = __expf(m0 - m), f1 = m1 == -INFINITY ? 0.f : __expf(m1 - m);
    const float l = fmaf(Cl[r], f0, Rl[r] * f1);
    accv[i] = fmaf(accv[i], f0, Ro[r * (D + 1) + d] * f1) / l;
    if (VLEN && q0 + r >= tq) accv[i] = 0.f;       // rows past the item
  }
  store(accv);
}

template <int D, bool BLK, bool VLEN>
int launch(const float *q, const float *k, const float *v, void *out, const int *lens, const int *vlen, int B, int heads,
           int Tq, int Tk, int64_t qbs, int64_t kbs, int64_t vbs, float scale, int prescale, cudaStream_t st) {
  static_assert((QT * D) % (32 * NWARP) == 0 && D % 8 == 0, "merge mapping");
  const size_t stages = sizeof(float) * NWARP * 2 * D * (KP + VP);           // >= the CTA-level merge area that reuses it
  const size_t smem = stages + sizeof(float) * (QT * (D + 1) + 2 * QT + D * KP);   // + the peer's landing zone + Q tile
  static bool done = false;
  if (!done) {
    cudaError_t e = cudaFuncSetAttribute(mha_mma_kernel<D, BLK, VLEN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) {
      cudaGetLastError();
      hsv::set_error("mha_mma: cudaFuncSetAttribute(%zu): %s", smem, cudaGetErrorString(e));
      return HSV_ERR_CUDA;
    }
    done = true;
  }
  auto al = [](const void *p_) { return (reinterpret_cast<uintptr_t>(p_) & 15) == 0; };
  const int fast = (Tk % 4 == 0) && al(k) && al(v) && (kbs % 4 == 0) && (vbs % 4 == 0);
  dim3 grid((unsigned)((Tq + QT - 1) / QT), (unsigned)(heads * NSPLIT), (unsigned)B);   // cluster dims (1, NSPLIT, 1)
  hsv::note_mha_launch(0, D, BLK, lens != nullptr, VLEN, prescale, fast,
                       (Tq % 4 == 0) && al(q) && (qbs % 4 == 0),   // the Q tile's 16-byte copies (full tiles only)
                       (Tk + KT - 1) / KT, grid);
  mha_mma_kernel<D, BLK, VLEN><<<grid, 32 * NWARP, smem, st>>>(q, k, v, out, lens, vlen, Tq, Tk, qbs, kbs, vbs, heads,
                                                             scale, prescale, fast);
  return hsv::check_launch("mha_mma");
}

}  // namespace

namespace hsv {
// returns 1 when the shape is not taken by this kernel (the caller falls back to the fp32 CUDA-core kernel).
// blk != 0: ``out`` is the fp16 blk16 operand buffer of heads*D channels x Tq rows (zero padding rows untouched).
// vlen != nullptr: per-item lengths (mha_mma_kernel's VLEN); a separate instantiation, so a launch without them runs
// none of that code.
int mha_mma_launch(const float *q, const float *k, const float *v, void *out, int blk, const int *lens, const int *vlen,
                   int B, int heads, int D, int Tq, int Tk, int64_t qbs, int64_t kbs, int64_t vbs, float scale,
                   int prescale, cudaStream_t st) {
#define HSV_MHA_MMA(DD)                                                                                              \
  if (vlen)                                                                                                          \
    return blk ? launch<DD, true, true>(q, k, v, out, lens, vlen, B, heads, Tq, Tk, qbs, kbs, vbs, scale, prescale, st) \
               : launch<DD, false, true>(q, k, v, out, lens, vlen, B, heads, Tq, Tk, qbs, kbs, vbs, scale, prescale, st); \
  return blk ? launch<DD, true, false>(q, k, v, out, lens, nullptr, B, heads, Tq, Tk, qbs, kbs, vbs, scale, prescale, st) \
             : launch<DD, false, false>(q, k, v, out, lens, nullptr, B, heads, Tq, Tk, qbs, kbs, vbs, scale, prescale, st)
  if (D == 96) { HSV_MHA_MMA(96); }
  if (D == 128) { HSV_MHA_MMA(128); }
  if (D == 64) { HSV_MHA_MMA(64); }
#undef HSV_MHA_MMA
  return 1;
}
}  // namespace hsv
