// Dense Conv1d / ConvTranspose1d as a tcgen05 / TMEM implicit GEMM (sm_100a), swizzled operands.
//
// Replaces the weight-normed convolutions of the reference's waveform path
//   * AMPBlock convs    hierspeechpp_speechsynthesizer.py:349-364,380-384; speechsr24k/speechsr.py:21-36,52-56
//   * conv_pre / proj / DBlock convs   hierspeechpp_speechsynthesizer.py:401,426,321-325
//   * ups[i] ConvTranspose1d           hierspeechpp_speechsynthesizer.py:404-408,434
// with one kernel.  Both are "sum over taps of a row-shifted [rows x Cin] x [Cin x Cout] product":
//   conv1d      out[t]       = b + sum_j  W[:, :, j]        a[t + (j-(k-1)/2) d]
//   convT phase out[u q + r] = b + sum_i  W[:, :, r' + i u] a[q + c - i]      (r' = (r+p) mod u, c = (r+p) div u)
// GEMM view per CTA:  D[M = 128 rows, N = n_tile out channels] += A_tap[128 x 16] * W_tap[16 x n_tile]
// over all channel chunks, taps and 16-channel K-steps; fp16 operands, fp32 accumulation in TMEM.
//
// Operand staging.  Activations arrive in the swizzled "blk16" layout written by the fused activation kernel
// (or hsv_pack_blk16): fp16 [B][Cin/CW][Lp][CW], CW = 64/32/16 channels per row, zero rows around every
// sequence, 16-byte units XOR-swizzled with the row index (hsv_common.cuh).  A time tile (+halo, start rounded
// down to a multiple of 8 rows) of one chunk is ONE contiguous span, fetched with a 1-D bulk TMA copy to a
// 1024-byte aligned shared address: that IS tcgen05's K-major SWIZZLE_128B/64B/32B canonical layout (row pitch
// = swizzle width, SBO = 8 rows).  Because the swizzle is a function of the shared-memory address bits, the
// operand of a tap is the SAME tile with the descriptor start address advanced by the tap's row offset: the
// halo is loaded once and reused by all taps; zero padding comes from the zero rows of the layout.
// Weights are pre-packed per (phase, n-tile) as a stream of [chunk][tap] blocks of n_tile rows x CW channels in
// the same swizzled K-major form, streamed through a ring of shared stages by bulk TMA copies.
//
// Roles (128 threads): warp0/lane0 TMA producer, warp1/lane0 MMA issuer, warp2 TMEM alloc/free, then all
// four warps run the epilogue: tcgen05.ld (lane = row), + bias, + residual, store fp32 [B,C,L] (for
// stride-1 outputs a warp stores 32 consecutive time steps of one channel = 128 B coalesced) and
// optionally accumulate the sum over resblocks.
#include "act_core.cuh"
#include "umma_common.cuh"

namespace {

using namespace hsv_umma;

constexpr int TILE_M = HSV_UMMA_TILE_M;  // 128
constexpr int MAX_STAGES = 4;
constexpr int MAX_PHASES = 8;
constexpr int MAX_TAPS = 16;
constexpr int MAX_CHUNKS = 16;

struct TapTable {
  int nphase;
  int out_stride;
  int ntaps[MAX_PHASES];
  int out_off[MAX_PHASES];
  int8_t row_off[MAX_PHASES][MAX_TAPS];  // input row offset of the tap relative to the output row
  int8_t wj[MAX_PHASES][MAX_TAPS];       // which tap of the weight tensor
  int h_lo, h_hi;                        // rows needed before / after the tile
};

struct Params {
  const uint8_t *a;   // swizzled blk16 activations
  const uint8_t *w;   // packed weights
  const float *bias;
  const float *residual;
  float *out;
  float *acc;
  int acc_mode;
  int Cin, Cout;
  int64_t L, Lp, Lout;
  int n_tile, nco_tiles;
  int ntiles;
  int B;             // batch (persistent variant: tiles are enumerated over (b, n-tile, row tile))
  int resident;      // persistent variant: 1 = all weight blocks stay in shared memory (loaded once per CTA)
  int nabuf;         // persistent variant: A-tile buffers (2 = double-buffered, 1 when two do not fit: C = 256)
  int msub;          // 128-row sub-tiles per CTA (1, 2 or 4): every weight K-step feeds msub MMAs
  int cw;            // channels per operand row (64 / 32 / 16)
  int nchunks;       // Cin / cw
  int a_bchunks;     // operand chunks between batch items of A (nchunks, more when A is a channel range of a wider buffer)
  int R;             // rows per chunk of the shared A tile = 128*msub + hlo8 + h_hi
  int hlo8;          // halo rows before the tile, rounded up to a multiple of 8 (swizzle phase alignment)
  uint32_t a_pitch;  // bytes between chunks of the shared A tile (multiple of 1024)
  int G;             // weight blocks ([chunk][tap] units) per ring stage
  int nrounds_ph[MAX_PHASES];  // ceil(nchunks * ntaps[ph] / G) per phase
  int stages;
  uint32_t tmem_cols;
  int vec_epi;       // 1: float4 epilogue (stride-1 output, Lout % 4 == 0, 16-byte aligned tensors)
  int tap_step;      // row offset between consecutive taps of a phase (taps are an arithmetic progression)
  // activation-producing variant (RR > 0): the A tile is computed in the CTA from the fp32 tensor fx
  const float *fx;     // [B, Cin, L] fp32 input of Activation1d
  const float *alpha;  // [Cin] log-scale SnakeBeta parameters
  const float *beta;
  float in_scale;
  uint32_t x_off;      // byte offset (from the aligned shared base) of the two fp32 staging buffers
  // operand-writing epilogue (hsv_conv1d_umma_blk16): the result goes out as the fp16 blk16 operand of the NEXT conv
  void *out_blk;          // nullptr = the fp32 epilogues below
  int blk_mode;           // 0 none, 1 WN gate (column pairs), 2 gelu_tanh, 3 leaky_relu(0.1), 4 WN layer tail
  int blk_C;              // channels of the output buffer (Cout; Cout / 2 for the gate and the WN tail)
  const float *blk_bc;    // [B][Cout] vector added before the activation (batch stride blk_bcs), or nullptr
  int64_t blk_bcs;
  const float *blk_mask;  // [B][L] frame mask applied to the result, or nullptr
  float *blk_x;           // mode 4 (WN layer tail): residual stream [B][Cout/2][L], updated in place
  float *blk_acc;         // mode 4: skip accumulator [B][Cout/2][L], updated in place
  int debug;
  long long *trace;  // bring-up: clock64 stamps of CTA (0,0,0) (hsv_set_umma_trace), else nullptr
  TapTable tt;
};

__device__ __forceinline__ void stamp(const Params &p, int slot) {
  if (p.trace == nullptr) return;
  if ((blockIdx.x | blockIdx.y | blockIdx.z) == 0) p.trace[slot] = clock64();
  // a CTA from the middle of the grid (steady state, loaded memory system): slots 16..
  if (blockIdx.x == gridDim.x / 2 && blockIdx.y == 0 && blockIdx.z == gridDim.z / 2 && gridDim.x * gridDim.z > 1)
    p.trace[16 + slot] = clock64();
}

// The KS K-steps (16 channels = 32 bytes each) of one [chunk][tap] weight block on one 128-row sub-tile, issued by
// the elected lane of a converged warp.  lo words: start>>4 | LBO; +2 per K-step (32 bytes); hi word shared.
template <int KS>
__device__ __forceinline__ void issue_ksteps(uint32_t tmem, uint32_t a_lo, uint32_t b_lo, uint32_t hi, uint32_t idesc,
                                             uint32_t not_first) {
  if constexpr (KS == 4) {
    asm volatile(
        "{\n\t"
        ".reg .pred pe, pa, pt;\n\t"
        ".reg .b64 da, db;\n\t"
        ".reg .b32 al, bl;\n\t"
        "elect.sync _|pe, 0xffffffff;\n\t"
        "setp.ne.b32 pa, %5, 0;\n\t"
        "setp.eq.b32 pt, 0, 0;\n\t"
        "mov.b64 da, {%1, %3};\n\t"
        "mov.b64 db, {%2, %3};\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, pa;\n\t"
        "add.u32 al, %1, 2;\n\t"
        "add.u32 bl, %2, 2;\n\t"
        "mov.b64 da, {al, %3};\n\t"
        "mov.b64 db, {bl, %3};\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, pt;\n\t"
        "add.u32 al, %1, 4;\n\t"
        "add.u32 bl, %2, 4;\n\t"
        "mov.b64 da, {al, %3};\n\t"
        "mov.b64 db, {bl, %3};\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, pt;\n\t"
        "add.u32 al, %1, 6;\n\t"
        "add.u32 bl, %2, 6;\n\t"
        "mov.b64 da, {al, %3};\n\t"
        "mov.b64 db, {bl, %3};\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, pt;\n\t"
        "}" ::"r"(tmem),
        "r"(a_lo), "r"(b_lo), "r"(hi), "r"(idesc), "r"(not_first)
        : "memory");
  } else if constexpr (KS == 2) {
    asm volatile(
        "{\n\t"
        ".reg .pred pe, pa, pt;\n\t"
        ".reg .b64 da, db;\n\t"
        ".reg .b32 al, bl;\n\t"
        "elect.sync _|pe, 0xffffffff;\n\t"
        "setp.ne.b32 pa, %5, 0;\n\t"
        "setp.eq.b32 pt, 0, 0;\n\t"
        "mov.b64 da, {%1, %3};\n\t"
        "mov.b64 db, {%2, %3};\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, pa;\n\t"
        "add.u32 al, %1, 2;\n\t"
        "add.u32 bl, %2, 2;\n\t"
        "mov.b64 da, {al, %3};\n\t"
        "mov.b64 db, {bl, %3};\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, pt;\n\t"
        "}" ::"r"(tmem),
        "r"(a_lo), "r"(b_lo), "r"(hi), "r"(idesc), "r"(not_first)
        : "memory");
  } else {
    asm volatile(
        "{\n\t"
        ".reg .pred pe, pa;\n\t"
        ".reg .b64 da, db;\n\t"
        "elect.sync _|pe, 0xffffffff;\n\t"
        "setp.ne.b32 pa, %5, 0;\n\t"
        "mov.b64 da, {%1, %3};\n\t"
        "mov.b64 db, {%2, %3};\n\t"
        "@pe tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, pa;\n\t"
        "}" ::"r"(tmem),
        "r"(a_lo), "r"(b_lo), "r"(hi), "r"(idesc), "r"(not_first)
        : "memory");
  }
}
struct MmaCtx {
  uint32_t tmem, hi, idesc, n_tile, sub16;
  uint32_t a_first;     // lo word of the first tap's A descriptor in chunk 0
  uint32_t a_step16;    // row offset between consecutive taps (16-byte units, may be "negative")
  uint32_t a_pitch16, w_lo0, stage16, blk16;
  uint32_t bar_wf, bar_we, bar_a, bar_acc;
  int nrounds, nblocks, G, stages, ntaps;
};

// The MMA issue loop of one CTA: every value is warp-uniform and the whole warp walks it.
template <int KS, int MSUB>
__device__ __forceinline__ void mma_loop(const MmaCtx &m) {
  int stage = 0, c = 0, j = 0;
  uint32_t parity = 0, not_first = 0;
  uint32_t a_chunk = m.a_first, a_lo = m.a_first;
  for (int rnd = 0; rnd < m.nrounds; ++rnd) {
    mbar_wait_warp(m.bar_wf + 8 * stage, parity);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const int nb = min(m.G, m.nblocks - rnd * m.G);
    uint32_t b_lo = m.w_lo0 + (uint32_t)stage * m.stage16;
    for (int g = 0; g < nb; ++g) {
      if (j == 0) {
        mbar_wait_warp(m.bar_a + 8 * c, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      }
#pragma unroll
      for (int sub = 0; sub < MSUB; ++sub)  // the same weight block feeds every 128-row sub-tile
        issue_ksteps<KS>(m.tmem + (uint32_t)sub * m.n_tile, a_lo + (uint32_t)sub * m.sub16, b_lo, m.hi, m.idesc,
                         not_first);
      not_first = 1u;
      b_lo += m.blk16;
      a_lo += m.a_step16;
      if (++j == m.ntaps) {
        j = 0;
        ++c;
        a_chunk += m.a_pitch16;
        a_lo = a_chunk;
      }
    }
    umma_commit_elect(m.bar_we + 8 * stage);  // the stage is free once these MMAs have read it
    if (++stage == m.stages) {
      stage = 0;
      parity ^= 1u;
    }
  }
  umma_commit_elect(m.bar_acc);
}

// bars: [0] acc_full, [1 .. 1+MAX_CHUNKS) a_full[chunk], then w_full[S], w_empty[S]
constexpr int BAR_A = 1, BAR_WF = 1 + MAX_CHUNKS, BAR_WE = BAR_WF + MAX_STAGES, NBARS = BAR_WE + MAX_STAGES;

// RR == 0: A tile = bulk copies of the pre-activated fp16 operand tensor (p.a).
// RR  > 0: activation-producing variant (whole-layer fusion, SURVEY.md §8f1): the CTA evaluates the fused
//          Activation1d (act_core.cuh; 8 channels x 16 runs of RR rows per pass, the mapping of act1d.cu) on the
//          fp32 input and writes the fp16 results straight into the swizzled shared A tile -- the operand never
//          exists in HBM.  Single-chunk inputs only (Cin = cw <= 64), n_tile = Cout (no recomputation).
// NW = warps per CTA: 4, or 8 for the wide variants -- warps 4..7 only take part in the epilogue (two warps per
// TMEM lane quarter, alternating 16-column units), which is a chain of ~180 dependent instructions per unit for
// a lone warp per scheduler.
// BLK = the operand-writing epilogue is compiled in (its own instantiations: the fp32 variants of the vocoder's hot path
// keep their register budget -- with the extra path in the same kernel the 80-register narrow variant spilled 52 bytes)
template <int MSUB, int MINB, bool SMALLN, int RR, int NW, bool BLK = false>
__global__ void __launch_bounds__(32 * NW, MINB) conv_umma_kernel(const __grid_constant__ Params p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bars[NBARS + 2];
  __shared__ uint32_t tmem_base_s;
  __shared__ float bias_s[256];

  // canonical (shuffled) warp index: tells ptxas the role branches are warp-uniform
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int tile = blockIdx.x, b = blockIdx.z;
  // (phase, n-tile) of this CTA and its ring rounds without integer divisions: both are host-known per launch / phase
  // (the two divisions were 6 % of the instructions of a streaming C = 32 tile)
  int ph, nt;
  if (p.tt.nphase == 1) {
    ph = 0;
    nt = blockIdx.y;
  } else if (p.nco_tiles == 1) {
    ph = blockIdx.y;
    nt = 0;
  } else {
    ph = blockIdx.y / p.nco_tiles;
    nt = blockIdx.y - ph * p.nco_tiles;
  }
  const int ntaps = p.tt.ntaps[ph];
  const int nblocks = p.nchunks * ntaps;          // [chunk][tap] weight blocks of this (phase, n-tile)
  const int nrounds = p.nrounds_ph[ph];           // ring rounds = ceil(nblocks / G)
  const uint32_t rowbytes = (uint32_t)p.cw * 2u;
  const uint32_t a_chunk_bytes = (uint32_t)p.R * rowbytes;
  const uint32_t blk_bytes = (uint32_t)p.n_tile * rowbytes;
  const uint32_t stage_bytes = blk_bytes * (uint32_t)p.G;

  // swizzled tiles want 1024-byte aligned shared addresses: align by hand (1 KB slack is budgeted by the host)
  const uint32_t a_s = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t w_s = a_s + p.a_pitch * (uint32_t)p.nchunks;
  const uint32_t bar0 = smem_u32(&bars[0]);
  const uint32_t bar_acc = bar0, bar_a = bar0 + 8 * BAR_A, bar_wf = bar0 + 8 * BAR_WF, bar_we = bar0 + 8 * BAR_WE;

  if (threadIdx.x == 0) stamp(p, 0);

  // weight stream of this (phase, n-tile)
  int64_t blk0 = 0;  // first weight block in the packed stream
  for (int q = 0; q < ph; ++q) blk0 += (int64_t)p.tt.ntaps[q] * p.nchunks * p.nco_tiles;
  blk0 += (int64_t)nt * nblocks;
  const uint8_t *wsrc = p.w + blk0 * blk_bytes;
  auto load_w = [&](int rnd, int s) {
    const int nb = min(p.G, nblocks - rnd * p.G);
    const uint32_t bytes = blk_bytes * (uint32_t)nb;
    mbar_expect_tx(bar_wf + 8 * s, bytes);
    bulk_g2s(w_s + s * stage_bytes, wsrc + (int64_t)rnd * stage_bytes, bytes, bar_wf + 8 * s);
  };
  const int npre = nrounds < p.stages ? nrounds : p.stages;

  if (threadIdx.x == 0) {
    mbar_init(bar_acc, 1);
    for (int c = 0; c < p.nchunks; ++c) mbar_init(bar_a + 8 * c, 1);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(bar_wf + 8 * s, 1);
      mbar_init(bar_we + 8 * s, 1);
    }
    if (RR > 0) {
      mbar_init(bar0 + 8 * NBARS, 1);
      mbar_init(bar0 + 8 * (NBARS + 1), 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                     smem_u32(&tmem_base_s)),
                 "r"(p.tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  // bias of this n-tile (static data): loaded to registers now, parked in shared memory at the start of the
  // epilogue (its global latency must not sit in front of the set-up barrier), read there as broadcast LDS
  // instead of 16 dependent global loads per 16-column unit
  constexpr int NBR = 256 / (32 * NW);
  float bias_r[NBR];
#pragma unroll
  for (int q = 0; q < NBR; ++q) {
    const int i = threadIdx.x + 32 * NW * q;
    bias_r[q] = (p.bias && i < p.n_tile) ? __ldg(p.bias + nt * p.n_tile + i) : 0.f;
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = tmem_base_s;
  // PDL: the next kernel may begin its prologue.  Triggered only AFTER this CTA owns its TMEM columns: a dependent
  // CTA that became resident earlier could take the columns and then park in griddepcontrol.wait -- which only
  // returns when this grid has finished -- while this CTA blocks in tcgen05.alloc.
  hsv::pdl_launch_dependents();
  if (threadIdx.x == 0) {
    stamp(p, 1);
    // weights are static data: fill the ring before waiting for the kernel that produces the activations
    // (issuing a bulk copy costs the thread a few hundred cycles: measured ~900 cycles for 4 stages)
    for (int rnd = 0; rnd < npre; ++rnd) load_w(rnd, rnd);
    stamp(p, 10);
  }
  hsv::pdl_wait();  // activations / residual / out / acc belong to predecessor kernels
  if (threadIdx.x == 0) stamp(p, 2);

  // ---- epilogue addressing + EARLY residual prefetch (float4 path) ----
  // Every warp issues the residual loads of its first PF units NOW, before its role loop: warps 0 and 1 used to
  // issue them only after producing / issuing (ncu: 23 % of the stall samples sat on the first use).
  constexpr int PF = 2;   // residual prefetch depth (units).  4 was measured too (136 registers): no gain at batch
                          // 16 (C=128, k=11: 82.0 vs 83.6 us) and one CTA per SM less for the n_tile = 64 variant
  constexpr int PFG = 2;  // the generic (scalar) path
  const int co0 = nt * p.n_tile;
  const int64_t cs = p.Lout;  // channel stride
  const int64_t chan_base = ((int64_t)b * p.Cout + co0) * p.Lout + p.tt.out_off[ph];
  const int nchk = p.n_tile >> 4;
  const int nunits = MSUB * nchk;
  const bool has_res = p.residual != nullptr;
  constexpr int NH = NW / 4;                 // warps per TMEM lane quarter
  const int wq = warp & 3, half = warp >> 2;  // lane quarter (rows 32*wq..), and which of its NH unit streams
  const int cq = lane >> 3, i4 = (lane & 7) << 2;
  const int64_t t_warp = (int64_t)tile * MSUB * TILE_M + wq * 32 + i4;  // first row of this lane's float4 (sub 0)
  const int64_t lane_off = chan_base + (int64_t)cq * cs + t_warp;
  const int64_t cs4b = 16 * cs;                                   // 4 channels, in bytes
  const int64_t unit_b = 64 * cs;                                 // 16 channels, in bytes
  const int64_t wrap_b = 4 * ((int64_t)TILE_M - (int64_t)p.n_tile * cs);  // next sub-tile, first unit (bytes)
  const char *res_b = has_res ? reinterpret_cast<const char *>(p.residual + lane_off) : nullptr;  // unit u + PF
  // (sub, chunk) walkers over this warp's unit stream (units half, half + NH, ...): advance by one unit
  auto advance = [&](int &u, int &sub, int &ch, int64_t &off, bool &ok) {
    ++u;
    off += unit_b;
    if constexpr (MSUB == 1) {
      ++ch;                      // one sub-tile: the units are the 16-column chunks, nothing wraps
    } else {
      if (++ch == nchk) {
        ch = 0;
        ++sub;
        off += wrap_b;
        ok = t_warp + (int64_t)sub * TILE_M < p.L;
      }
    }
  };
  int nxt_sub = 0, nxt_ch = 0, nxt_u = 0;   // the unit being prefetched
  int64_t nxt_b = 0;
  bool nxt_ok = t_warp < p.L;               // L % 4 == 0: a float4 is all-valid or all-invalid
  if (NH > 1 && half) advance(nxt_u, nxt_sub, nxt_ch, nxt_b, nxt_ok);
  float4 res[PF][4];
#pragma unroll
  for (int q = 0; q < PF; ++q)
#pragma unroll
    for (int ps = 0; ps < 4; ++ps) res[q][ps] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (p.vec_epi) {
#pragma unroll
    for (int q = 0; q < PF; ++q) {
      // warp-uniform guard: without a residual (every first conv of a half-layer) or past the last unit nothing is
      // computed at all (the predicated form cost ~6 instructions per dead load)
      if (has_res && nxt_u < nunits) {
#pragma unroll
        for (int ps = 0; ps < 4; ++ps)
          res[q][ps] = nxt_ok ? *reinterpret_cast<const float4 *>(res_b + nxt_b + ps * cs4b) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int h = 0; h < NH; ++h) advance(nxt_u, nxt_sub, nxt_ch, nxt_b, nxt_ok);
    }
  }

  if constexpr (RR > 0) {
    // ---------------- activation producer: all 128 threads ----------------
    using K = hsv_act::Cfg<RR>;
    const uint32_t bar_x = bar0 + 8 * NBARS;                      // two staging barriers
    uint8_t *smem_al = smem_raw + (a_s - smem_u32(smem_raw));     // generic pointer to the aligned base
    float *xs = reinterpret_cast<float *>(smem_al + p.x_off);     // [2][8][PITCH]
    const int tid = threadIdx.x;
    const int c = tid % hsv_act::ROWS, run = tid / hsv_act::ROWS;
    const int64_t t_first = (int64_t)tile * TILE_M * MSUB - p.hlo8;   // time of A-tile row 0 (multiple of 8)
    const int ngroups = p.Cin >> 3;
    const bool fast = ((p.L & 3) == 0) && t_first >= K::XOFF && t_first + K::TILE + K::XOFF <= p.L &&
                      ((reinterpret_cast<uintptr_t>(p.fx) & 15) == 0);
    constexpr uint32_t ROW_BYTES = (uint32_t)K::XW * 4u;
    auto issue = [&](int g) {   // TMA staging of group g (fast tiles): one bulk copy per channel row
      const uint32_t bar = bar_x + 8 * (g & 1);
      if (tid == 0) mbar_expect_tx(bar, ROW_BYTES * hsv_act::ROWS);
      if (tid < hsv_act::ROWS) {
        const float *src = p.fx + ((int64_t)b * p.Cin + g * 8 + tid) * p.L + (t_first - K::XOFF);
        bulk_g2s(smem_u32(xs + (g & 1) * (hsv_act::ROWS * K::PITCH) + tid * K::PITCH), src, ROW_BYTES, bar);
      }
    };
    if (fast) issue(0);
    const int64_t ta = t_first + (int64_t)run * RR;
    const bool need = run * RR < p.R && ta < p.L && ta + RR > 0;     // this run holds rows of the A tile inside [0, L)
    float al = __ldg(p.alpha + c), be = __ldg(p.beta + c);
    for (int g = 0; g < ngroups; ++g) {
      float *xb = xs + (g & 1) * (hsv_act::ROWS * K::PITCH);
      const float al_g = al, be_g = be;
      if (g + 1 < ngroups) {
        al = __ldg(p.alpha + (g + 1) * 8 + c);
        be = __ldg(p.beta + (g + 1) * 8 + c);
      }
      if (fast) {
        if (g + 1 < ngroups) issue(g + 1);   // its buffer was released by the barrier that ended pass g - 1
        mbar_wait(bar_x + 8 * (g & 1), (uint32_t)(g >> 1) & 1u);
      } else {
        // tiles touching either end of the sequence (or unaligned tensors): clamped loads, all issued before
        // the first store
        constexpr int NLD = (hsv_act::ROWS * K::XW + 127) / 128;
        const int Lm1 = (int)(p.L - 1);
        float v[NLD];
#pragma unroll
        for (int i = 0; i < NLD; ++i) {
          const int idx = tid + 128 * i;
          const int cc = idx / K::XW, pp = idx - cc * K::XW;
          const int64_t t = t_first - K::XOFF + pp;
          const int tc = t < 0 ? 0 : (t > Lm1 ? Lm1 : (int)t);
          v[i] = idx < hsv_act::ROWS * K::XW ? __ldg(p.fx + ((int64_t)b * p.Cin + g * 8 + cc) * p.L + tc) : 0.f;
        }
#pragma unroll
        for (int i = 0; i < NLD; ++i) {
          const int idx = tid + 128 * i;
          const int cc = idx / K::XW, pp = idx - cc * K::XW;
          if (idx < hsv_act::ROWS * K::XW) xb[cc * K::PITCH + pp] = v[i];
        }
        __syncthreads();
      }
      if (run * RR < p.R) {
        float outv[RR];
        if (need) {
          const float *xw = xb + c * K::PITCH + run * RR + (K::XOFF - 5);
          hsv_act::act_run<RR>(xw, outv, al_g, be_g, ta, p.L, p.fx + ((int64_t)b * p.Cin + g * 8 + c) * p.L,
                                     p.in_scale);
        }
        // fp16 into the swizzled A tile: row = run*RR + j, 16-byte unit g, half c; rows outside [0, L) are the
        // conv's zero padding
        const uint32_t swz_mask = (uint32_t)(p.cw >> 3) - 1u;
#pragma unroll
        for (int j = 0; j < RR; ++j) {
          const int rowt = run * RR + j;
          const int64_t t = ta + j;
          const float val = (need && t >= 0 && t < p.L) ? outv[j] : 0.f;
          if (rowt < p.R) {
            const uint32_t lin = (uint32_t)rowt * rowbytes + (uint32_t)g * 16u;
            const uint32_t addr = a_s + (lin ^ (((lin >> 7) & swz_mask) << 4)) + (uint32_t)c * 2u;
            const unsigned short hbits = __half_as_ushort(__float2half_rn(val));
            asm volatile("st.shared.b16 [%0], %1;" ::"r"(addr), "h"(hbits) : "memory");
          }
        }
      }
      // generic-proxy writes of the A tile must be visible to the tensor core (async proxy)
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncthreads();  // staging buffer reusable; after the last pass: the A tile is complete
    }
    if (threadIdx.x == 0) {
      asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar_a) : "memory");  // A chunk 0 "landed"
      stamp(p, 4);
    }
  }

  if (warp == 0 && lane == 0) {
    // ---------------- TMA producer ----------------
    if constexpr (RR == 0) {
      const int64_t row0 = (int64_t)HSV_BLK_PAD + (int64_t)tile * TILE_M * MSUB - p.hlo8;  // multiple of 8
      for (int c = 0; c < p.nchunks; ++c) {
        const uint8_t *src = p.a + ((int64_t)(b * p.a_bchunks + c) * p.Lp + row0) * rowbytes;   // B * a_bchunks < 2^31
        mbar_expect_tx(bar_a + 8 * c, a_chunk_bytes);
        bulk_g2s(a_s + c * p.a_pitch, src, a_chunk_bytes, bar_a + 8 * c);
      }
    }
    int s = 0;
    uint32_t par = 0;
    for (int rnd = npre; rnd < nrounds; ++rnd) {  // ring slot s was last used by round rnd - stages
      mbar_wait(bar_we + 8 * s, par);
      load_w(rnd, s);
      if (++s == p.stages) {
        s = 0;
        par ^= 1u;
      }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer ----------------
    // The whole warp walks the loop with warp-uniform values; only the elected lane issues.  The tensor pipe
    // retires a 128 x N x 16 MMA every N/2 cycles, so every dependent scalar instruction in this chain is
    // directly visible (measured: 28 SASS instructions per MMA = 236 cycles per MMA, 4x the pipe time).
    MmaCtx m;
    m.tmem = tmem;
    // InstrDescriptor: D=F32 (1<<4), A=B=F16 (0), K-major both, N>>3 at [17,23), M>>4 at [24,29)
    m.idesc = (1u << 4) | ((uint32_t)(p.n_tile >> 3) << 17) | ((uint32_t)(TILE_M >> 4) << 24);
    // SmemDescriptor (cute::UMMA::SmemDescriptor): lo = start>>4 [0,14) | LBO>>4 [16,30) (=1, unused for swizzled
    // K-major); hi = SBO>>4 [0,14) (8 rows) | version=1 [14,16) | base_offset [17,20) = 0 | layout [29,32).
    // base_offset stays 0 for row-shifted starts: the swizzle is a function of the absolute shared address
    // (verified on B200: tools/umma_diag.py).
    const uint32_t layout = p.cw == 64 ? 2u : (p.cw == 32 ? 4u : 6u);  // SWIZZLE_128B / 64B / 32B
    m.hi = ((8u * rowbytes) >> 4) | (1u << 14) | (layout << 29);
    const uint32_t row16 = rowbytes >> 4;
    m.n_tile = (uint32_t)p.n_tile;
    m.sub16 = (uint32_t)TILE_M * row16;
    // 16-byte-unit addresses stay below 2^14 (228 KB of shared memory), so adding offsets never carries out
    // of the 14-bit start-address field.  Taps are an arithmetic progression of row offsets (host-checked).
    m.a_first = ((1u << 16) | ((a_s & 0x3FFFFu) >> 4)) + (uint32_t)((p.hlo8 + p.tt.row_off[ph][0]) * (int)row16);
    m.a_step16 = (uint32_t)(p.tap_step * (int)row16);
    m.a_pitch16 = p.a_pitch >> 4;
    m.w_lo0 = (1u << 16) | ((w_s & 0x3FFFFu) >> 4);
    m.stage16 = stage_bytes >> 4;
    m.blk16 = blk_bytes >> 4;
    m.bar_wf = bar_wf; m.bar_we = bar_we; m.bar_a = bar_a; m.bar_acc = bar_acc;
    m.nrounds = nrounds; m.nblocks = nblocks; m.G = p.G; m.stages = p.stages; m.ntaps = ntaps;
    // broadcast from lane 0: marks every loop input as warp-uniform for ptxas (uniform registers, no R2UR per MMA)
    {
      uint32_t *f = reinterpret_cast<uint32_t *>(&m);
#pragma unroll
      for (int q = 0; q < (int)(sizeof(MmaCtx) / 4); ++q) f[q] = __shfl_sync(0xffffffffu, f[q], 0);
    }
    if (p.cw == 64) mma_loop<4, MSUB>(m);
    else if (p.cw == 32) mma_loop<2, MSUB>(m);
    else mma_loop<1, MSUB>(m);
    if (lane == 0) stamp(p, 5);
    __syncwarp();
  }

  // ---------------- epilogue: all 4 warps ----------------
  // Units of (sub-tile, 16 columns).  tcgen05.ld gives every lane ONE time row x 16 channels; stored straight to
  // [B,C,L] that is 16 scalar accesses per lane per tensor with 64-bit address math each -- measured ~1000 cycles
  // per unit of pure issue time for a lone warp per scheduler, as long as the whole MMA phase.  So each warp
  // transposes the unit through a private 2 KB shared buffer ([16 ch][32 rows]) and then moves float4s: lane =
  // (channel c = lane/8 + 4*pass, rows 4*(lane%8)..+3): one LDS.128 + one LDG.128 (residual, prefetched PF units
  // ahead in registers, first PF before the accumulator wait) + one STG.128 per 4 elements.
  // out may alias residual (same offsets): loads of a unit always precede its stores.
  __syncwarp();
#pragma unroll
  for (int q = 0; q < NBR; ++q) bias_s[threadIdx.x + 32 * NW * q] = bias_r[q];
  if (threadIdx.x == 0) stamp(p, 6);
  const uint32_t trow = tmem + ((uint32_t)(wq * 32) << 16);
  if (BLK && p.out_blk) {
    // Operand-writing epilogue.  tcgen05.ld gives a lane one time row x 16 consecutive output channels: exactly two
    // 16-byte units of the blk16 layout ([row][8 channels]) -- no transpose.  The WN gate pairs columns: the host packs
    // in_layers' output channels as [8 tanh | 8 sigmoid] groups, so a 16-column unit yields 8 gate outputs = one unit.
    const int64_t row_base = (int64_t)tile * MSUB * TILE_M + wq * 32 + lane;
    const int cwo = hsv::blk_cw(p.blk_C);
    uint8_t *ob = reinterpret_cast<uint8_t *>(p.out_blk);
    const float *bcv = p.blk_bc ? p.blk_bc + (int64_t)b * p.blk_bcs + co0 : nullptr;
    __syncthreads();  // bias_s complete
    mbar_wait(bar_acc, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    __syncwarp();
#pragma unroll 1
    for (int u = half ? nunits : 0; u < nunits; ++u) {   // warps 4..7 (NW = 8) sit this path out
      const int sub = u / nchk, c0 = (u - sub * nchk) << 4;
      const int64_t t = row_base + (int64_t)sub * TILE_M;
      uint32_t r[16];
      tmem_ld16(trow + (uint32_t)(sub * p.n_tile + c0), r);
      if (t < p.L) {
        const float mk = p.blk_mask ? __ldg(p.blk_mask + (int64_t)b * p.L + t) : 1.f;
        float v[16];
#pragma unroll
        for (int c = 0; c < 16; ++c) v[c] = __uint_as_float(r[c]) + bias_s[c0 + c] + (bcv ? __ldg(bcv + c0 + c) : 0.f);
        if (p.blk_mode == 4) {
          // WN layer tail (modules.py:167-174): columns [0, H) are the residual branch: x = (x + rs) * mask in place, and
          // the new x IS the next in_layer's operand; columns [H, 2H) are the skip branch: output += rs.  H % n_tile == 0,
          // so a CTA is entirely on one side.  For a fixed channel consecutive lanes are consecutive frames: coalesced.
          const int H = p.blk_C;
          const int cb = co0 + c0;
          if (cb < H) {
            float *xp = p.blk_x + ((int64_t)b * H + cb) * p.L + t;
            float xv[16];
#pragma unroll
            for (int c = 0; c < 16; ++c) xv[c] = xp[(int64_t)c * p.L];
#pragma unroll
            for (int c = 0; c < 16; ++c) {
              xv[c] = (xv[c] + v[c]) * mk;
              xp[(int64_t)c * p.L] = xv[c];
            }
#pragma unroll
            for (int q8 = 0; q8 < 2; ++q8) {
              __half2 hh[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) hh[e] = __floats2half2_rn(xv[8 * q8 + 2 * e], xv[8 * q8 + 2 * e + 1]);
              *reinterpret_cast<uint4 *>(ob + hsv::blk_unit_offset(cwo, p.Lp, H, b, cb + 8 * q8, HSV_BLK_PAD + t)) =
                  *reinterpret_cast<uint4 *>(hh);
            }
          } else {
            float *op = p.blk_acc + ((int64_t)b * H + (cb - H)) * p.L + t;
            float ov[16];
#pragma unroll
            for (int c = 0; c < 16; ++c) ov[c] = op[(int64_t)c * p.L];
#pragma unroll
            for (int c = 0; c < 16; ++c) op[(int64_t)c * p.L] = ov[c] + v[c];
          }
        } else if (p.blk_mode == 1) {
          __half2 hh[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float g0 = tanhf(v[2 * e]) * (1.0f / (1.0f + expf(-v[8 + 2 * e])));
            const float g1 = tanhf(v[2 * e + 1]) * (1.0f / (1.0f + expf(-v[9 + 2 * e])));
            hh[e] = __floats2half2_rn(g0 * mk, g1 * mk);
          }
          *reinterpret_cast<uint4 *>(ob + hsv::blk_unit_offset(cwo, p.Lp, p.blk_C, b, (co0 + c0) >> 1, HSV_BLK_PAD + t)) =
              *reinterpret_cast<uint4 *>(hh);
        } else {
#pragma unroll
          for (int c = 0; c < 16; ++c) {
            float a = v[c];
            if (p.blk_mode == 2) {
              const float kk = 0.7978845608028654f;
              a = 0.5f * a * (1.0f + tanhf(kk * (a + 0.044715f * a * a * a)));
            } else if (p.blk_mode == 3) {
              a = a > 0.f ? a : 0.1f * a;
            }
            v[c] = a * mk;
          }
#pragma unroll
          for (int q8 = 0; q8 < 2; ++q8) {
            __half2 hh[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) hh[e] = __floats2half2_rn(v[8 * q8 + 2 * e], v[8 * q8 + 2 * e + 1]);
            *reinterpret_cast<uint4 *>(ob + hsv::blk_unit_offset(cwo, p.Lp, p.blk_C, b, co0 + c0 + 8 * q8, HSV_BLK_PAD + t)) =
                *reinterpret_cast<uint4 *>(hh);
          }
        }
      }
    }
  } else if (p.vec_epi) {
    // the A tile / weight ring are idle once the accumulator is complete: reuse 2 KB per warp as staging
    const uint32_t stg = a_s + (uint32_t)warp * 2048u;
    const uint32_t stg_w = stg + (uint32_t)lane * 4u;                       // [c][lane]
    const uint32_t stg_r = stg + (uint32_t)(cq * 32 + i4) * 4u;             // [cq + 4*pass][i4 .. i4+3]
    // exactly one destination on this path (host-checked): out, or acc written (mode 1) / accumulated (mode 2)
    char *dst_b = reinterpret_cast<char *>((p.out ? p.out : p.acc) + lane_off);
    const bool is_red = !p.out && p.acc_mode == 2;
    int64_t cur_b = 0;  // byte offset of the current unit relative to the per-lane bases
    int cur_sub = 0, cur_ch = 0, cur_u = 0;
    bool cur_ok = t_warp < p.L;
    if (NH > 1 && half) advance(cur_u, cur_sub, cur_ch, cur_b, cur_ok);
    __syncthreads();  // bias_s complete (every warp is past its role loop here; the MMAs are in flight)
    mbar_wait(bar_acc, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    __syncwarp();
    if (threadIdx.x == 0) stamp(p, 7);
#pragma unroll 1
    for (int u0 = half; u0 < nunits; u0 += PF * NH) {
#pragma unroll
      for (int q = 0; q < PF; ++q) {
        if (u0 + q * NH < nunits) {
          uint32_t r[16];
          tmem_ld16(trow + (uint32_t)(cur_sub * p.n_tile + (cur_ch << 4)), r);
#pragma unroll
          for (int c = 0; c < 16; ++c)
            asm volatile("st.shared.b32 [%0], %1;" ::"r"(stg_w + (uint32_t)c * 128u), "r"(r[c]) : "memory");
          __syncwarp();
          const bool refill = has_res && nxt_u < nunits;   // warp-uniform: is there a unit u + PF to prefetch for?
          const float *bias_u = bias_s + (cur_ch << 4) + cq;
#pragma unroll
          for (int ps = 0; ps < 4; ++ps) {
            float4 a;
            asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                         : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w)
                         : "r"(stg_r + (uint32_t)ps * 512u)
                         : "memory");
            const float bch = bias_u[ps * 4];
            const float4 rr = res[q][ps];
            a.x = (a.x + bch) + rr.x;  // (conv + bias) + residual: the reference's order
            a.y = (a.y + bch) + rr.y;
            a.z = (a.z + bch) + rr.z;
            a.w = (a.w + bch) + rr.w;
            // refill this ring slot (unit u + PF) before this unit's stores
            if (refill)
              res[q][ps] = nxt_ok ? *reinterpret_cast<const float4 *>(res_b + nxt_b + ps * cs4b)
                                  : make_float4(0.f, 0.f, 0.f, 0.f);
            if (cur_ok) {
              char *o = dst_b + cur_b + ps * cs4b;
              // red.global.add: no read, one add per element per kernel -> deterministic given stream order
              if (is_red)
                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(o), "f"(a.x), "f"(a.y), "f"(a.z), "f"(a.w)
                             : "memory");
              else
                *reinterpret_cast<float4 *>(o) = a;
            }
          }
          __syncwarp();  // the staging buffer is rewritten by the next unit
#pragma unroll
          for (int h = 0; h < NH; ++h) {
            advance(cur_u, cur_sub, cur_ch, cur_b, cur_ok);
            advance(nxt_u, nxt_sub, nxt_ch, nxt_b, nxt_ok);
          }
        }
      }
    }
  } else {
    // generic path (strided ConvTranspose1d phases, L % 4 != 0, unaligned tensors): lane = row, scalar accesses
    const int64_t row_base = (int64_t)tile * MSUB * TILE_M + wq * 32 + lane;  // GEMM row of sub-tile 0
    auto unit_ptr = [&](int u, int64_t &off, bool &ok) {
      const int sub = u / nchk, c0 = (u - sub * nchk) << 4;
      const int64_t t = row_base + (int64_t)sub * TILE_M;
      ok = t < p.L;
      off = chan_base + (int64_t)p.tt.out_stride * t + (int64_t)c0 * cs;
    };
    // (addresses walk by pointer increments: `off + c * cs` per element was 16 64-bit multiply-adds per unit and made this
    // path -- every ConvTranspose1d of the vocoder -- issue-bound: 1 575 instructions per warp for 32 outputs per lane)
    float res[PFG][16];
#pragma unroll
    for (int q = 0; q < PFG; ++q)
#pragma unroll
      for (int c = 0; c < 16; ++c) res[q][c] = 0.f;
    if (has_res && half == 0) {
#pragma unroll
      for (int q = 0; q < PFG; ++q) {
        int64_t off; bool ok;
        unit_ptr(q < nunits ? q : 0, off, ok);
        if (ok && q < nunits) {
          const float *rp = p.residual + off;
#pragma unroll
          for (int c = 0; c < 16; ++c, rp += cs) res[q][c] = *rp;
        }
      }
    }
    __syncthreads();  // bias_s complete (every warp is past its role loop here; the MMAs are in flight)
    mbar_wait(bar_acc, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    __syncwarp();
    if (threadIdx.x == 0) stamp(p, 7);
#pragma unroll 1
    for (int u0 = half ? nunits : 0; u0 < nunits; u0 += PFG) {  // warps 4..7 (NW = 8) sit this path out
#pragma unroll
      for (int q = 0; q < PFG; ++q) {
        const int u = u0 + q;
        if (u < nunits) {
          const int sub = u / nchk, c0 = (u - sub * nchk) << 4;
          int64_t off; bool valid;
          unit_ptr(u, off, valid);
          uint32_t r[16];
          tmem_ld16(trow + (uint32_t)(sub * p.n_tile + c0), r);
          float v[16];
#pragma unroll
          for (int c = 0; c < 16; ++c) v[c] = (__uint_as_float(r[c]) + bias_s[c0 + c]) + res[q][c];  // reference order
          if (has_res) {
            int64_t offn; bool okn;
            unit_ptr(u + PFG < nunits ? u + PFG : u, offn, okn);
            okn = okn && u + PFG < nunits;
            const float *rp = p.residual + offn;
#pragma unroll
            for (int c = 0; c < 16; ++c, rp += cs) res[q][c] = okn ? *rp : 0.f;
          }
          if (valid) {
            if (p.acc_mode == 1) {
              float *ap = p.acc + off;
#pragma unroll
              for (int c = 0; c < 16; ++c, ap += cs) *ap = v[c];
            } else if (p.acc_mode == 2) {
              float *ap = p.acc + off;
#pragma unroll
              for (int c = 0; c < 16; ++c, ap += cs) atomicAdd(ap, v[c]);
            }
            if (p.out) {
              float *op = p.out + off;
#pragma unroll
              for (int c = 0; c < 16; ++c, op += cs) *op = v[c];
            }
          }
        }
      }
    }
  }
  if (threadIdx.x == 0) stamp(p, 8);
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (threadIdx.x == 0) stamp(p, 9);
  if (warp == 2) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(p.tmem_cols)
                 : "memory");
  }
}

// ------------------------------------------------------------------------------------------------------------
// Persistent variant for the wide layers (n_tile >= 128) at batch scale.
// One CTA per SM walks its share of the (batch, n-tile, 128-row tile) list; the three roles run concurrently on
// DIFFERENT tiles: warp 0 streams the A tile of tile i+1 and the weights of tile i, warp 1 issues the MMAs of
// tile i into TMEM buffer i & 1, warps 2..5 drain tile i-1 from the other TMEM buffer (float4 epilogue).  The
// tensor pipe therefore never waits for a prologue or an epilogue (ncu on the one-tile-per-CTA kernel at C=128,
// batch 16: two co-resident CTAs, tensor pipe 36-48 % busy, the rest is their load / drain phases).
// Restrictions: stride-1 conv, MSUB = 1, float4 epilogue.  The A tile is double-buffered when two fit (C = 128),
// else single (C = 256: the next tile is staged after this tile's MMAs).  Measured at batch 16: C = 128 k=3 49.1
// -> 38.0 us, k=7 60.2 -> 51.3, k=11 74.3 -> 64.3 us (897 TFLOP/s); C = 256 k=3 25.5 -> 23.1 us, k=7 38.1 -> 33.3,
// k=11 50.5 -> 46.0 us (1003 TFLOP/s = 73 % of the measured sustained bf16 peak); C = 64 (weights resident in shared
// memory) k=11 103.7 -> 79.0 us.  C <= 32 loses (two units per tile leave half the epilogue warps idle).
// ------------------------------------------------------------------------------------------------------------
constexpr int PB_ACC_F = 0, PB_ACC_E = 2, PB_A_F = 4, PB_A_E = 6, PB_WF = 8, PB_WE = PB_WF + MAX_STAGES,
              PB_N = PB_WE + MAX_STAGES;

// EPW = epilogue warps per TMEM lane quarter: the drain of a tile is a chain of global round trips, so it takes
// many warps (each with its own units of 16 columns, residual prefetched before the accumulator is complete)
// to keep up with the MMAs of the next tile (measured: 4 warps in all -> 2300 cycles per unit under load).
template <int EPW>
__global__ void __launch_bounds__(64 + 128 * EPW, 1) conv_umma_persist_kernel(const __grid_constant__ Params p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bars[PB_N];
  __shared__ uint32_t tmem_base_s;

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int ntaps = p.tt.ntaps[0];
  const int nblocks = p.nchunks * ntaps;
  const int nrounds = (nblocks + p.G - 1) / p.G;
  const uint32_t rowbytes = (uint32_t)p.cw * 2u;
  const uint32_t a_chunk_bytes = (uint32_t)p.R * rowbytes;
  const uint32_t a_tile_bytes = p.a_pitch * (uint32_t)p.nchunks;
  const uint32_t blk_bytes = (uint32_t)p.n_tile * rowbytes;
  const uint32_t stage_bytes = blk_bytes * (uint32_t)p.G;
  const uint32_t a_s = (smem_u32(smem_raw) + 1023u) & ~1023u;       // one or two A tiles
  const uint32_t w_s = a_s + (uint32_t)p.nabuf * a_tile_bytes;       // weight ring
  const bool a2 = p.nabuf == 2;
  const uint32_t stg_s = w_s + (uint32_t)p.stages * stage_bytes;     // 2 KB of epilogue staging per warp
  const uint32_t bar0 = smem_u32(&bars[0]);
  const int total = p.ntiles * p.nco_tiles * p.B;                    // tiles of the launch
  const int my_n = (total - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;  // tiles of this CTA

  if (threadIdx.x == 0) {
    mbar_init(bar0 + 8 * (PB_ACC_F + 0), 1); mbar_init(bar0 + 8 * (PB_ACC_F + 1), 1);
    mbar_init(bar0 + 8 * (PB_ACC_E + 0), 128 * EPW); mbar_init(bar0 + 8 * (PB_ACC_E + 1), 128 * EPW);
    mbar_init(bar0 + 8 * (PB_A_F + 0), 1); mbar_init(bar0 + 8 * (PB_A_F + 1), 1);
    mbar_init(bar0 + 8 * (PB_A_E + 0), 1); mbar_init(bar0 + 8 * (PB_A_E + 1), 1);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(bar0 + 8 * (PB_WF + s), 1);
      mbar_init(bar0 + 8 * (PB_WE + s), 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)),
                 "r"(p.tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = tmem_base_s;
  hsv::pdl_launch_dependents();  // after the TMEM allocation (see conv_umma_kernel)
  hsv::pdl_wait();

  auto tile_coords = [&](int i, int &b, int &nt, int &tile) {
    const int lin = (int)blockIdx.x + i * (int)gridDim.x;
    tile = lin % p.ntiles;
    const int r = lin / p.ntiles;
    nt = r % p.nco_tiles;
    b = r / p.nco_tiles;
  };

  if (warp == 0) {
    // ---------------- TMA producer (one lane) ----------------
    if (lane == 0) {
      auto load_a = [&](int i) {
        int b, nt, tile;
        tile_coords(i, b, nt, tile);
        const int buf = a2 ? (i & 1) : 0, use = a2 ? (i >> 1) : i;   // use-th fill of this buffer
        if (use >= 1) mbar_wait(bar0 + 8 * (PB_A_E + buf), (uint32_t)(use - 1) & 1u);
        const int64_t row0 = (int64_t)HSV_BLK_PAD + (int64_t)tile * TILE_M - p.hlo8;
        mbar_expect_tx(bar0 + 8 * (PB_A_F + buf), a_chunk_bytes * (uint32_t)p.nchunks);
        for (int c = 0; c < p.nchunks; ++c) {
          const uint8_t *src = p.a + (((int64_t)b * p.a_bchunks + c) * p.Lp + row0) * rowbytes;
          bulk_g2s(a_s + buf * a_tile_bytes + c * p.a_pitch, src, a_chunk_bytes, bar0 + 8 * (PB_A_F + buf));
        }
      };
      int it = 0, ws = 0;
      uint32_t wpar = 0;
      if (my_n > 0) load_a(0);
      for (int i = 0; i < my_n; ++i) {
        int b, nt, tile;
        tile_coords(i, b, nt, tile);
        const uint8_t *wsrc = p.w + (int64_t)nt * nblocks * blk_bytes;
        if (a2 && i + 1 < my_n) load_a(i + 1);  // one tile ahead of the MMAs
        for (int rnd = 0; rnd < nrounds && !(p.resident && i > 0); ++rnd, ++it) {  // resident: first tile only
          if (it >= p.stages) mbar_wait(bar0 + 8 * (PB_WE + ws), wpar ^ 1u);
          const int nb = min(p.G, nblocks - rnd * p.G);
          const uint32_t bytes = blk_bytes * (uint32_t)nb;
          mbar_expect_tx(bar0 + 8 * (PB_WF + ws), bytes);
          bulk_g2s(w_s + ws * stage_bytes, wsrc + (int64_t)rnd * stage_bytes, bytes, bar0 + 8 * (PB_WF + ws));
          if (++ws == p.stages) {
            ws = 0;
            wpar ^= 1u;
          }
        }
        // single A buffer: the next tile can only be staged once this tile's MMAs have read it (its weights are
        // all issued by now, so the wait inside load_a cannot deadlock)
        if (!a2 && i + 1 < my_n) load_a(i + 1);
      }
    }
  } else if (warp == 1) {
    // ---------------- MMA issuer (whole warp walks, elected lane issues) ----------------
    const uint32_t idesc = (1u << 4) | ((uint32_t)(p.n_tile >> 3) << 17) | ((uint32_t)(TILE_M >> 4) << 24);
    const uint32_t layout = p.cw == 64 ? 2u : (p.cw == 32 ? 4u : 6u);
    const uint32_t hi = ((8u * rowbytes) >> 4) | (1u << 14) | (layout << 29);
    const uint32_t row16 = rowbytes >> 4;
    const uint32_t a_lo00 = ((1u << 16) | ((a_s & 0x3FFFFu) >> 4)) + (uint32_t)((p.hlo8 + p.tt.row_off[0][0]) * (int)row16);
    const uint32_t a_step16 = (uint32_t)(p.tap_step * (int)row16);
    const uint32_t a_pitch16 = p.a_pitch >> 4, a_tile16 = a_tile_bytes >> 4;
    const uint32_t w_lo0 = (1u << 16) | ((w_s & 0x3FFFFu) >> 4);
    const uint32_t stage16 = stage_bytes >> 4, blk16 = blk_bytes >> 4;
    int ws = 0;
    uint32_t wpar = 0;
    for (int i = 0; i < my_n; ++i) {
      const int buf = i & 1;                                            // TMEM accumulator buffer
      const int abuf = a2 ? buf : 0, ause = a2 ? (i >> 1) : i;          // A-tile buffer and its use count
      if (i >= 2) mbar_wait_warp(bar0 + 8 * (PB_ACC_E + buf), (uint32_t)((i >> 1) - 1) & 1u);  // TMEM buffer drained
      mbar_wait_warp(bar0 + 8 * (PB_A_F + abuf), (uint32_t)ause & 1u);                         // A tile landed
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint32_t tacc = tmem + (uint32_t)(buf * p.n_tile);
      uint32_t a_chunk = a_lo00 + (uint32_t)abuf * a_tile16, a_lo = a_chunk, not_first = 0;
      int j = 0;
      for (int rnd = 0; rnd < nrounds; ++rnd) {
        if (!(p.resident && i > 0)) {  // resident weights: landed once, never recycled
          mbar_wait_warp(bar0 + 8 * (PB_WF + ws), wpar);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        }
        const int nb = min(p.G, nblocks - rnd * p.G);
        uint32_t b_lo = w_lo0 + (uint32_t)ws * stage16;
        for (int g = 0; g < nb; ++g) {
          if (p.cw == 64) issue_ksteps<4>(tacc, a_lo, b_lo, hi, idesc, not_first);
          else if (p.cw == 32) issue_ksteps<2>(tacc, a_lo, b_lo, hi, idesc, not_first);
          else issue_ksteps<1>(tacc, a_lo, b_lo, hi, idesc, not_first);
          not_first = 1u;
          b_lo += blk16;
          a_lo += a_step16;
          if (++j == ntaps) {
            j = 0;
            a_chunk += a_pitch16;
            a_lo = a_chunk;
          }
        }
        if (!p.resident) {
          umma_commit_elect(bar0 + 8 * (PB_WE + ws));
          if (++ws == p.stages) {
            ws = 0;
            wpar ^= 1u;
          }
        }
      }
      umma_commit_elect(bar0 + 8 * (PB_A_E + abuf));   // the A buffer may be refilled
      umma_commit_elect(bar0 + 8 * (PB_ACC_F + buf));  // the accumulator is complete
    }
  } else {
    // ---------------- epilogue: warps 2.. (TMEM lane quarter = warp & 3, unit stream = (warp - 2) / 4) ----------
    const int wq = warp & 3, strm = (warp - 2) >> 2;
    const int cq = lane >> 3, i4 = (lane & 7) << 2;
    const int64_t cs = p.Lout;
    const int64_t cs4b = 16 * cs, unit_b = 64 * cs;
    const int nchk = p.n_tile >> 4;
    const bool has_res = p.residual != nullptr;
    const bool is_red = !p.out && p.acc_mode == 2;
    const uint32_t stg = stg_s + (uint32_t)(warp - 2) * 2048u;
    const uint32_t stg_w = stg + (uint32_t)lane * 4u;
    const uint32_t stg_r = stg + (uint32_t)(cq * 32 + i4) * 4u;
    constexpr int PF = 2;   // in units of this warp's stream (units strm, strm + EPW, ...)
    for (int i = 0; i < my_n; ++i) {
      int b, nt, tile;
      tile_coords(i, b, nt, tile);
      const int buf = i & 1;
      const int co0 = nt * p.n_tile;
      const int64_t t_warp = (int64_t)tile * TILE_M + wq * 32 + i4;
      const bool ok_rows = t_warp < p.L;
      const int64_t lane_off = ((int64_t)b * p.Cout + co0 + cq) * p.Lout + t_warp;
      const char *res_b = has_res ? reinterpret_cast<const char *>(p.residual + lane_off) : nullptr;
      char *dst_b = reinterpret_cast<char *>((p.out ? p.out : p.acc) + lane_off);
      float4 res[PF][4];
#pragma unroll
      for (int q = 0; q < PF; ++q) {
        const int u = strm + q * EPW;
        const bool ok = ok_rows && has_res && u < nchk;
#pragma unroll
        for (int ps = 0; ps < 4; ++ps)
          res[q][ps] = ok ? *reinterpret_cast<const float4 *>(res_b + (int64_t)u * unit_b + ps * cs4b)
                          : make_float4(0.f, 0.f, 0.f, 0.f);
      }
      mbar_wait(bar0 + 8 * (PB_ACC_F + buf), (uint32_t)(i >> 1) & 1u);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      __syncwarp();
      const uint32_t trow = tmem + ((uint32_t)(wq * 32) << 16) + (uint32_t)(buf * p.n_tile);
#pragma unroll 1
      for (int u0 = strm; u0 < nchk; u0 += PF * EPW) {
#pragma unroll
        for (int q = 0; q < PF; ++q) {
          const int u = u0 + q * EPW;
          if (u < nchk) {
            uint32_t r[16];
            tmem_ld16(trow + (uint32_t)(u << 4), r);
#pragma unroll
            for (int c = 0; c < 16; ++c)
              asm volatile("st.shared.b32 [%0], %1;" ::"r"(stg_w + (uint32_t)c * 128u), "r"(r[c]) : "memory");
            __syncwarp();
            const bool okn = ok_rows && has_res && u + PF * EPW < nchk;
#pragma unroll
            for (int ps = 0; ps < 4; ++ps) {
              float4 a;
              asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
                           : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w)
                           : "r"(stg_r + (uint32_t)ps * 512u)
                           : "memory");
              const float bch = p.bias ? __ldg(p.bias + co0 + (u << 4) + ps * 4 + cq) : 0.f;
              const float4 rr = res[q][ps];
              a.x = (a.x + bch) + rr.x;  // (conv + bias) + residual: the reference's order
              a.y = (a.y + bch) + rr.y;
              a.z = (a.z + bch) + rr.z;
              a.w = (a.w + bch) + rr.w;
              res[q][ps] = okn ? *reinterpret_cast<const float4 *>(res_b + (int64_t)(u + PF * EPW) * unit_b + ps * cs4b)
                               : make_float4(0.f, 0.f, 0.f, 0.f);
              if (ok_rows) {
                char *o = dst_b + (int64_t)u * unit_b + ps * cs4b;
                if (is_red)
                  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(o), "f"(a.x), "f"(a.y), "f"(a.z), "f"(a.w)
                               : "memory");
                else
                  *reinterpret_cast<float4 *>(o) = a;
              }
            }
            __syncwarp();
          }
        }
      }
      // this TMEM buffer may be overwritten by the MMAs of tile i + 2
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar0 + 8 * (PB_ACC_E + buf)) : "memory");
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 1) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(p.tmem_cols) : "memory");
  }
}

int g_host_debug = 0;
int g_persist = 1;  // persistent variant for eligible launches (hsv_set_umma_debug bit 6 turns it off)

constexpr int PERSIST_EPW = 4;

// hsv_last_launch_config, family 0: kind (0 one-tile, 1 persistent, 2 fused activation, 3 operand-writing epilogue),
// msub, warps per CTA, vec_epi, nphase, n_tile, stages, G, resident, nabuf, grid x / y / z, blk_mode (kind 3 only, else
// 0), running launch count
void note_launch(int kind, const Params &p, int warps, dim3 grid) {
  const bool persist = kind == 1;  // resident / nabuf are only set (and read) by the persistent variant
  const int v[hsv::LAST_CONV_N - 1] = {kind, p.msub, warps, p.vec_epi, p.tt.nphase, p.n_tile, p.stages, p.G,
                                       persist ? p.resident : 0, persist ? p.nabuf : 0, (int)grid.x, (int)grid.y,
                                       (int)grid.z, kind == 3 ? p.blk_mode : 0};
  int *last = hsv::g_last_launch[0];
  for (int i = 0; i < hsv::LAST_CONV_N - 1; ++i) last[i] = v[i];
  ++last[hsv::LAST_CONV_N - 1];
}

int launch_persist(Params p, int B, cudaStream_t st, const char *what) {
  static int max_dyn[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  if (max_dyn[dev] == 0) {
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, conv_umma_persist_kernel<PERSIST_EPW>);
    int want = 227 * 1024 - (e == cudaSuccess ? (int)fa.sharedSizeBytes : 1024);
    want &= ~1023;
    if (e == cudaSuccess) e = cudaFuncSetAttribute(conv_umma_persist_kernel<PERSIST_EPW>, cudaFuncAttributeMaxDynamicSharedMemorySize, want);
    if (e != cudaSuccess) {
      cudaGetLastError();
      hsv::set_error("%s: cudaFuncSetAttribute(%d): %s", what, want, cudaGetErrorString(e));
      return HSV_ERR_CUDA;
    }
    max_dyn[dev] = want;
  }
  p.B = B;
  p.stages = MAX_STAGES;
  // two A tiles when they leave room for a 3-stage ring of 16 KB, else one (C = 256: 92 KB per tile)
  p.nabuf = 1024 + 2 * (size_t)p.a_pitch * p.nchunks + 4 * PERSIST_EPW * 2048 + 3 * 16384 <= (size_t)max_dyn[dev] ? 2 : 1;
  // weights resident in shared memory (one stage holding every block, loaded once per CTA) when the whole set of
  // one n-tile fits next to the A tiles: the C <= 64 layers (<= 90 KB), whose weight stream per 128-row tile would
  // otherwise need more L2->SM bandwidth than the MMAs leave time for
  p.resident = 0;
  {
    const size_t wall = (size_t)p.nchunks * p.tt.ntaps[0] * p.n_tile * p.cw * 2;
    const size_t fixed = 1024 + p.nabuf * (size_t)p.a_pitch * p.nchunks + 4 * PERSIST_EPW * 2048;
    if (p.nco_tiles == 1 && wall < (1u << 20) && fixed + wall <= (size_t)max_dyn[dev] && !(g_host_debug & 2)) {
      p.resident = 1;
      p.G = p.nchunks * p.tt.ntaps[0];
      p.stages = 1;
    }
  }
  // weight-ring stage: 32 KB when three of them fit next to the two A tiles (one elected thread issues every
  // bulk copy of the CTA: fewer, larger copies), else the 16 KB of the one-tile kernel
  {
    const int blk_bytes = p.n_tile * p.cw * 2;
    const int nblk = p.nchunks * p.tt.ntaps[0];
    int g32 = 32768 / blk_bytes;
    g32 = g32 < 1 ? 1 : (g32 > nblk ? nblk : g32);
    const size_t fixed = 1024 + p.nabuf * (size_t)p.a_pitch * p.nchunks + 4 * PERSIST_EPW * 2048;
    // (measured at C=128, batch 16: k=11 70.8 -> 64.3 us = 897 TFLOP/s, k=7 53.9 -> 51.3 us; short K loops prefer
    //  four small stages: k=3 38.0 vs 47.1 us)
    if (!p.resident && !(g_host_debug & 1) && nblk >= 12 && g32 > p.G &&
        fixed + 3 * (size_t)g32 * blk_bytes <= (size_t)max_dyn[dev])
      p.G = g32;
  }
  const size_t stage_bytes = (size_t)p.G * p.n_tile * p.cw * 2;
  size_t smem = 1024 + p.nabuf * (size_t)p.a_pitch * p.nchunks + 4 * PERSIST_EPW * 2048;
  while (!p.resident && p.stages > 3 && smem + p.stages * stage_bytes > (size_t)max_dyn[dev]) p.stages--;
  smem += p.stages * stage_bytes;
  if (smem > (size_t)max_dyn[dev]) return 1;  // not eligible: fall back to the one-tile-per-CTA kernel
  uint32_t cols = 32;
  while ((int)cols < 2 * p.n_tile) cols <<= 1;
  p.tmem_cols = cols;
  const int total = p.ntiles * p.nco_tiles * B;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(total < 148 ? total : 148));
  cfg.blockDim = dim3(64 + 128 * PERSIST_EPW);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = hsv::g_pdl ? 1 : 0;
  note_launch(1, p, 2 + 4 * PERSIST_EPW, cfg.gridDim);
  cudaError_t e = cudaLaunchKernelEx(&cfg, conv_umma_persist_kernel<PERSIST_EPW>, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    hsv::set_error("%s: launch failed: %s", what, cudaGetErrorString(e));
    return HSV_ERR_CUDA;
  }
  return hsv::check_launch(what);
}

// Packed weight stream: [phase][n-tile][chunk][tap] blocks of n_tile rows x cw channels (fp16, K-major, swizzled
// relative to the block start):  W(co = nt*n_tile + n, ci = chunk*cw + 8*u + e, tap wj[ph][ti]) at byte
// swz(n*rowbytes + 16*u) + 2*e of its block.  Element strides (s_co, s_ci) select Conv1d [Cout,Cin,k] or
// ConvTranspose1d [Cin,Cout,k] weights.
__global__ void pack_weight_kernel(const float *__restrict__ w, __half *__restrict__ out, int Cout, int Cin,
                                   int n_tile, int cw, int64_t s_co, int64_t s_ci, const TapTable tt) {
  const int nchunks = Cin / cw;
  const int nco = Cout / n_tile;
  const int blk_elems = n_tile * cw;
  const uint32_t rowbytes = (uint32_t)cw * 2u, mask = (uint32_t)(cw >> 3) - 1u;
  int64_t ph_base = 0;  // in blocks
  for (int ph = 0; ph < tt.nphase; ++ph) {
    const int nt_ph = tt.ntaps[ph];
    const int64_t cnt = (int64_t)nco * nchunks * nt_ph * blk_elems;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < cnt; i += (int64_t)gridDim.x * blockDim.x) {
      int64_t r = i;
      const int cil = (int)(r % cw); r /= cw;       // channel within the chunk
      const int n = (int)(r % n_tile); r /= n_tile;
      const int ti = (int)(r % nt_ph); r /= nt_ph;
      const int chunk = (int)(r % nchunks); r /= nchunks;
      const int nt = (int)r;
      const int co = nt * n_tile + n, ci = chunk * cw + cil;
      const uint32_t lin = (uint32_t)n * rowbytes + (uint32_t)(cil >> 3) * 16u;
      const uint32_t phys = (lin ^ (((lin >> 7) & mask) << 4)) + 2u * (uint32_t)(cil & 7);
      const int64_t blk = ph_base + ((int64_t)nt * nchunks + chunk) * nt_ph + ti;
      out[blk * blk_elems + (phys >> 1)] = __float2half_rn(w[co * s_co + ci * s_ci + tt.wj[ph][ti]]);
    }
    ph_base += (int64_t)nco * nchunks * nt_ph;
  }
}

TapTable conv_taps(int k, int d) {
  TapTable tt = {};
  tt.nphase = 1;
  tt.out_stride = 1;
  tt.ntaps[0] = k;
  const int h = ((k - 1) / 2) * d;
  for (int j = 0; j < k; ++j) {
    tt.row_off[0][j] = (int8_t)((j - (k - 1) / 2) * d);
    tt.wj[0][j] = (int8_t)j;
  }
  tt.h_lo = h;
  tt.h_hi = h;
  return tt;
}

// ConvTranspose1d(k, stride u, padding p=(k-u)/2): output phase rho = o mod u reads input rows q + c - i
// through taps j = r + i*u, r = (rho+p) mod u, c = (rho+p) div u   (SURVEY.md §A.3)
TapTable convT_taps(int k, int u) {
  TapTable tt = {};
  tt.nphase = u;
  tt.out_stride = u;
  const int p = (k - u) / 2;
  int lo = 0, hi = 0;
  for (int rho = 0; rho < u; ++rho) {
    const int r = (rho + p) % u, c = (rho + p) / u;
    int n = 0;
    for (int j = r; j < k; j += u, ++n) {
      tt.row_off[rho][n] = (int8_t)(c - n);
      tt.wj[rho][n] = (int8_t)j;
      if (c - n < lo) lo = c - n;
      if (c - n > hi) hi = c - n;
    }
    tt.ntaps[rho] = n;
    tt.out_off[rho] = rho;
  }
  tt.h_lo = -lo;
  tt.h_hi = hi;
  return tt;
}

long long *g_trace = nullptr;
int g_msub_override = 0;  // bring-up aid: force the sub-tiles per CTA (0 = automatic)

template <int MSUB, int MINB, bool SMALLN, int RR = 0, int NW = 4, bool BLK = false>
int launch_variant(const Params &p, dim3 grid, size_t smem, cudaStream_t st, const char *what) {
  // opt-in dynamic shared memory: 227 KB per block minus the kernel's static shared memory
  static int max_dyn[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  if (max_dyn[dev] == 0) {
    cudaFuncAttributes fa;
    cudaError_t e = cudaFuncGetAttributes(&fa, conv_umma_kernel<MSUB, MINB, SMALLN, RR, NW, BLK>);
    int want = 227 * 1024 - (e == cudaSuccess ? (int)fa.sharedSizeBytes : 1024);
    want &= ~1023;
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(conv_umma_kernel<MSUB, MINB, SMALLN, RR, NW, BLK>, cudaFuncAttributeMaxDynamicSharedMemorySize, want);
    if (e != cudaSuccess) {
      cudaGetLastError();  // clear
      hsv::set_error("%s: cudaFuncSetAttribute(%d): %s", what, want, cudaGetErrorString(e));
      return HSV_ERR_CUDA;
    }
    max_dyn[dev] = want;
  }
  HSV_REQUIRE(smem <= (size_t)max_dyn[dev], "%s: shared memory %zu B exceeds %d B (Cin=%d)", what, smem,
              max_dyn[dev], p.Cin);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = dim3(32 * NW);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = hsv::g_pdl ? 1 : 0;
  note_launch(RR > 0 ? 2 : (BLK ? 3 : 0), p, NW, grid);
  cudaError_t e = cudaLaunchKernelEx(&cfg, conv_umma_kernel<MSUB, MINB, SMALLN, RR, NW, BLK>, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    hsv::set_error("%s: launch failed: %s", what, cudaGetErrorString(e));
    return HSV_ERR_CUDA;
  }
  return hsv::check_launch(what);
}

struct FusedAct {  // activation-producing variant: fp32 input of Activation1d instead of the fp16 operand tensor
  const float *x, *alpha, *beta;
  float in_scale;
};

struct BlkOut {    // operand-writing epilogue (see Params)
  void *out;
  int mode, C;
  const float *bc;
  int64_t bcs;
  const float *mask;
  float *x, *acc;  // mode 4
};

int launch(const TapTable &tt, const void *a_blk16, const void *w_packed, const float *bias,
           const float *residual, float *out, float *acc, int acc_mode, int B, int Cin, int Cout, int64_t L,
           int64_t Lout, int n_tile, cudaStream_t st, const char *what, const FusedAct *fa = nullptr,
           const BlkOut *bo = nullptr, int64_t a_bchunks = 0) {
  Params p;
  p.out_blk = bo ? bo->out : nullptr;
  p.blk_mode = bo ? bo->mode : 0;
  p.blk_C = bo ? bo->C : 0;
  p.blk_bc = bo ? bo->bc : nullptr;
  p.blk_bcs = bo ? bo->bcs : 0;
  p.blk_mask = bo ? bo->mask : nullptr;
  p.blk_x = bo ? bo->x : nullptr;
  p.blk_acc = bo ? bo->acc : nullptr;
  p.fx = fa ? fa->x : nullptr;
  p.alpha = fa ? fa->alpha : nullptr;
  p.beta = fa ? fa->beta : nullptr;
  p.in_scale = fa ? fa->in_scale : 1.f;
  p.x_off = 0;
  p.a = reinterpret_cast<const uint8_t *>(a_blk16);
  p.w = reinterpret_cast<const uint8_t *>(w_packed);
  p.bias = bias; p.residual = residual; p.out = out; p.acc = acc;
  p.acc_mode = acc_mode;
  p.Cin = Cin; p.Cout = Cout; p.L = L; p.Lp = hsv::blk16_rows(L); p.Lout = Lout;
  p.n_tile = n_tile; p.nco_tiles = Cout / n_tile;
  p.cw = hsv::blk_cw(Cin);
  p.nchunks = Cin / p.cw;
  p.a_bchunks = (int)(a_bchunks > 0 ? a_bchunks : p.nchunks);
  HSV_REQUIRE((int64_t)B * p.a_bchunks < (int64_t)1 << 31, "%s: batch x operand chunks too large", what);
  HSV_REQUIRE(p.nchunks <= MAX_CHUNKS, "%s: Cin=%d needs %d operand chunks (max %d)", what, Cin, p.nchunks, MAX_CHUNKS);
  const int rowbytes = p.cw * 2;
  p.hlo8 = (tt.h_lo + 7) & ~7;
  HSV_REQUIRE(p.hlo8 <= HSV_BLK_PAD && tt.h_hi <= HSV_BLK_PAD, "%s: halo (%d,%d) exceeds blk16 padding %d", what,
              tt.h_lo, tt.h_hi, HSV_BLK_PAD);
  const int ntiles128 = (int)((L + TILE_M - 1) / TILE_M);
  const int blk_bytes = n_tile * rowbytes;
  // sub-tiles per CTA (measured policy, tools/microbench4.py on B200): msub = 2 shares every weight block between
  // two 128-row MMAs and halves the per-row prologue/weight traffic, but doubles the A tile.  It pays for
  // compute-heavy layers (Cin * taps >= 512) when the grid is large and either the tile is narrow (n_tile <= 64)
  // or msub = 1 could not keep two CTAs per SM anyway (C = 256: 535 -> 746 TFLOP/s); where msub = 1 fits two
  // CTAs with a 3-stage ring it is better (C = 128: 690 vs 466 TFLOP/s), and so it is for the HBM-bound k = 3 layers.
  int msub = 1;
  const int64_t ctas1 = (int64_t)ntiles128 * p.nco_tiles * tt.nphase * B;
  int max_taps = 0;
  for (int q = 0; q < tt.nphase; ++q) max_taps = tt.ntaps[q] > max_taps ? tt.ntaps[q] : max_taps;
  if (Cin * max_taps >= 512 && ctas1 >= 2 * 148) {
    const size_t stage1 = (size_t)(16384 / blk_bytes > 0 ? 16384 / blk_bytes : 1) * blk_bytes;
    const size_t a1 = ((((size_t)(TILE_M + p.hlo8 + tt.h_hi) * rowbytes) + 1023) & ~(size_t)1023) * p.nchunks;
    if (1024 + a1 + 3 * stage1 > 113 * 1024) msub = 2;              // one CTA per SM either way (C = 256)
    else if (n_tile <= 64 && ctas1 >= 2 * 148 * 2) msub = 2;
  }
  // C = 16 streaming layers: a 128-row tile moves only 20 KB, the per-CTA prologue dominates -> 512-row tiles
  // (3.5 -> 5.4 TB/s at batch 16, 8.7 -> 6.5 us at batch 1 on [16, 160000])
  if (n_tile <= 16 && ctas1 >= 2 * 148 * 2) msub = 4;
  // C = 32 streaming layers at batch scale (SpeechSR48 batch 16: 60 000 128-row tiles): the ~1 800 set-up / addressing
  // instructions of a tile are paid once per 512 rows instead of once per 128 -- 16.8 -> 16.0 ms per step (A/B on one box);
  // small grids (batch 1: 625 tiles) keep 128-row tiles, there the CTA count matters more
  if (n_tile <= 32 && ctas1 >= 16 * 148) msub = 4;
  if (g_msub_override > 0) msub = g_msub_override;
  if (msub == 3) msub = 2;
  // persistent variant (opt-in): one 128-row tile at a time per CTA, roles overlapped across tiles
  auto al16e = [](const void *q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  const bool force_persist = (g_host_debug & 128) != 0;  // tests: any size / tile width
  const bool want_persist = g_persist && !fa && !bo && tt.nphase == 1 && tt.out_stride == 1 &&
                            (force_persist || (n_tile >= 128 && ctas1 >= 2 * 148) || (n_tile == 64 && Cout == 64 && ctas1 >= 4 * 148)) &&
                            (Lout % 4) == 0 && al16e(residual) && al16e(out) && al16e(acc) &&
                            ((out != nullptr) != (acc_mode != 0));
  if (want_persist || bo) msub = 1;
  if (fa) msub = 2;  // 256-row tiles: the activation's 5-row run halo and the conv halo are amortised over more rows
  auto a_bytes_for = [&](int ms) {
    const size_t per = (((size_t)(TILE_M * ms + p.hlo8 + tt.h_hi) * rowbytes) + 1023) & ~(size_t)1023;
    return per * p.nchunks;
  };
  while (!fa && msub > 1 &&
         (msub * n_tile > 512 || msub > ntiles128 || a_bytes_for(msub) + 2 * (size_t)blk_bytes > 200 * 1024))
    msub >>= 1;
  p.msub = msub;
  p.ntiles = (ntiles128 + msub - 1) / msub;
  p.R = TILE_M * msub + p.hlo8 + tt.h_hi;
  p.a_pitch = (uint32_t)((((size_t)p.R * rowbytes) + 1023) & ~(size_t)1023);
  p.tt = tt;
  p.tap_step = 0;
  for (int q = 0; q < tt.nphase; ++q)
    for (int j = 1; j < tt.ntaps[q]; ++j) {
      const int st = tt.row_off[q][j] - tt.row_off[q][j - 1];
      HSV_REQUIRE(p.tap_step == 0 || st == p.tap_step, "%s: taps are not an arithmetic progression", what);
      p.tap_step = st;
    }
  int max_blocks = 0;
  for (int q = 0; q < tt.nphase; ++q) max_blocks = tt.ntaps[q] * p.nchunks > max_blocks ? tt.ntaps[q] * p.nchunks : max_blocks;
  // ring stage = G blocks, about 16 KB (32 KB when the grid is small and each CTA is alone on its SM; 8 KB for
  // the narrow streaming layers, which want 8 co-resident CTAs per SM)
  const int64_t total_ctas = (int64_t)p.ntiles * p.nco_tiles * tt.nphase * B;
  int G = (n_tile <= 32 ? 8192 : (total_ctas <= 148 ? 32768 : 16384)) / blk_bytes;
  if (G < 1) G = 1;
  if (G > max_blocks) G = max_blocks;
  p.G = G;
  for (int q = 0; q < MAX_PHASES; ++q) p.nrounds_ph[q] = q < tt.nphase ? (p.nchunks * tt.ntaps[q] + G - 1) / G : 0;
  const int nrounds = (max_blocks + G - 1) / G;
  p.stages = nrounds < MAX_STAGES ? nrounds : MAX_STAGES;
  uint32_t cols = 32;
  while ((int)cols < n_tile * msub) cols <<= 1;
  p.tmem_cols = cols;
  p.debug = g_host_debug;
  p.trace = g_trace;
  auto al16 = [](const void *q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  p.vec_epi = tt.out_stride == 1 && (Lout % 4) == 0 && al16(residual) && al16(out) && al16(acc) &&
              ((out != nullptr) != (acc_mode != 0)) && !(g_host_debug & 16);

  if (want_persist && p.msub == 1 && p.vec_epi) {
    const int rc = launch_persist(p, B, st, what);
    if (rc != 1) return rc;  // 1 = does not fit (A tile too large to double-buffer): one-tile-per-CTA kernel below
  }
  const size_t a_bytes = (size_t)p.a_pitch * p.nchunks;
  // shared-memory budget: leave room for as many co-resident CTAs per SM as the grid can use (they hide
  // each other's prologue / epilogue latency), down to a 2-stage weight ring
  // 8-warp CTAs (two epilogue warps per TMEM lane quarter) for n_tile >= 128 only: measured +7 % on the C=128/256
  // layers at batch 16 (722 -> 770 TFLOP/s), but -20 % on n_tile = 64 (two CTAs per SM instead of four) and on
  // the 512-row C=16 tiles
  const bool w8 = !(g_host_debug & 32) && !fa && !bo && n_tile >= 128;
  const int minb = n_tile <= 32 && msub == 1 ? 6 : (w8 ? 2 : (n_tile <= 64 ? 4 : 2));
  int want = (int)((total_ctas + 147) / 148);
  want = want < 1 ? 1 : (want > minb ? minb : want);
  const size_t budget = (size_t)(226 * 1024) / want - 1024;
  const size_t stage_bytes = (size_t)G * blk_bytes;
  size_t smem = 1024 + a_bytes + (size_t)p.stages * stage_bytes;
  while (smem > budget && p.stages > 2) {
    p.stages--;
    smem = 1024 + a_bytes + (size_t)p.stages * stage_bytes;
  }
  if (smem < 1024 + 16384) smem = 1024 + 16384;  // the epilogue stages 2 KB per warp in the (then idle) operand area
  int rr = 0;
  if (fa) {
    // run length of the in-CTA activation: 16 runs must cover the A tile (256 + halo rows)
    rr = p.R <= 16 * 17 ? 17 : 20;
    HSV_REQUIRE(p.R <= 16 * rr && p.nchunks == 1 && p.nco_tiles == 1 && tt.nphase == 1 && msub == 2 && n_tile <= 256,
                "%s: shape not supported by the activation-producing variant (Cin=%d Cout=%d n_tile=%d rows=%d)", what,
                Cin, Cout, n_tile, p.R);
    const size_t pitch = rr == 17 ? hsv_act::Cfg<17>::PITCH : hsv_act::Cfg<20>::PITCH;
    smem = (smem + 15) & ~(size_t)15;
    p.x_off = (uint32_t)(smem - 1024);
    smem += 2 * hsv_act::ROWS * pitch * sizeof(float);
  }
  HSV_REQUIRE(B <= 65535 && (int64_t)p.nco_tiles * tt.nphase <= 65535, "%s: grid too large", what);
  dim3 grid((unsigned)p.ntiles, (unsigned)(p.nco_tiles * tt.nphase), (unsigned)B);
  if (fa) {
    if (rr == 17) return launch_variant<2, 3, false, 17, 4>(p, grid, smem, st, what);
    return launch_variant<2, 3, false, 20, 4>(p, grid, smem, st, what);
  }
  // small n_tile = HBM/latency-bound streaming layers: they want many co-resident CTAs (register cap 80);
  // large n_tile = few fat CTAs per SM anyway
  // wide tiles (>= 4 units of 16 columns per CTA) run 8 warps: two epilogue warps per TMEM lane quarter
  if (bo) {   // operand-writing epilogue: 128-row tiles, 4 warps
    HSV_REQUIRE(p.msub == 1, "%s: the operand-writing epilogue runs 128-row tiles", what);
    if (n_tile <= 32) return launch_variant<1, 6, true, 0, 4, true>(p, grid, smem, st, what);
    if (n_tile <= 64) return launch_variant<1, 4, false, 0, 4, true>(p, grid, smem, st, what);
    return launch_variant<1, 2, false, 0, 4, true>(p, grid, smem, st, what);
  }
  if (p.msub == 1) {
    if (n_tile <= 32) return launch_variant<1, 6, true>(p, grid, smem, st, what);
    if (w8) return launch_variant<1, 2, false, 0, 8>(p, grid, smem, st, what);
    if (n_tile <= 64) return launch_variant<1, 4, false>(p, grid, smem, st, what);
    return launch_variant<1, 2, false>(p, grid, smem, st, what);
  }
  if (p.msub == 2) {
    if (w8) return launch_variant<2, 2, false, 0, 8>(p, grid, smem, st, what);
    return launch_variant<2, 2, false>(p, grid, smem, st, what);
  }
  return launch_variant<4, 1, false>(p, grid, smem, st, what);
}

int check_common(const char *what, const void *a, const void *w, int Cin, int Cout, int n_tile) {
  HSV_REQUIRE(a && w, "%s: null operand", what);
  HSV_REQUIRE(Cin > 0 && Cin % 16 == 0, "%s: Cin %% 16 != 0 (Cin=%d)", what, Cin);
  HSV_REQUIRE(n_tile >= 16 && n_tile <= 256 && n_tile % 16 == 0 && Cout % n_tile == 0,
              "%s: bad n_tile=%d for Cout=%d", what, n_tile, Cout);
  return HSV_OK;
}

int pack(const float *w, void *packed, int Cout, int Cin, int k, int n_tile, int64_t s_co, int64_t s_ci,
         const TapTable &tt, cudaStream_t st, const char *what) {
  const int64_t total = (int64_t)Cout * Cin * k;
  const int blocks = (int)((total + 255) / 256 < 2048 ? (total + 255) / 256 : 2048);
  pack_weight_kernel<<<blocks, 256, 0, st>>>(w, reinterpret_cast<__half *>(packed), Cout, Cin, n_tile,
                                             hsv::blk_cw(Cin), s_co, s_ci, tt);
  return hsv::check_launch(what);
}

}  // namespace

// bring-up aid only; not part of the drop-in contract.
//   bit 0: persistent variant keeps 16 KB weight-ring stages, bit 1: ... never keeps the weights resident, bit 2: skip the epilogue's global stores, bit 3: skip its TMEM loads, bit 4: force the scalar epilogue,
//   bit 5: 4-warp CTAs for the wide variants too, bit 6: persistent variant off,
//   bit 7: persistent variant for every launch it can run (tests);
//   bits 24..26: forced sub-tiles per CTA.
extern "C" int hsv_set_umma_debug(int flags) {
  g_host_debug = flags & 0xff;
  g_persist = ((flags >> 6) & 1) ? 0 : 1;
  if (flags & 128) g_persist = 1;
  g_msub_override = (flags >> 24) & 0x7;
  return HSV_OK;
}

// bring-up aid: device buffer of >= 16 int64 that CTA (0,0,0) of every conv launch stamps with clock64() at its
// phase boundaries (nullptr = off)
extern "C" int hsv_set_umma_trace(void *dev_buf) {
  g_trace = reinterpret_cast<long long *>(dev_buf);
  return HSV_OK;
}

extern "C" int hsv_pack_conv_weight(const float *w, void *packed, int Cout, int Cin, int k, int n_tile,
                                    void *stream) {
  if (int rc = check_common("pack_conv_weight", w, packed, Cin, Cout, n_tile)) return rc;
  HSV_REQUIRE(k >= 1 && k <= MAX_TAPS && (k & 1), "pack_conv_weight: k=%d (odd, <= %d)", k, MAX_TAPS);
  return pack(w, packed, Cout, Cin, k, n_tile, (int64_t)Cin * k, k, conv_taps(k, 1), hsv::as_stream(stream),
              "pack_conv_weight");
}

extern "C" int hsv_pack_convT_weight(const float *w, void *packed, int Cin, int Cout, int k, int u, int n_tile,
                                     void *stream) {
  if (int rc = check_common("pack_convT_weight", w, packed, Cin, Cout, n_tile)) return rc;
  HSV_REQUIRE(u >= 1 && u <= MAX_PHASES && k >= u && k <= MAX_TAPS && k - 2 * ((k - u) / 2) == u,
              "pack_convT_weight: unsupported (k,u)=(%d,%d)", k, u);
  return pack(w, packed, Cout, Cin, k, n_tile, k, (int64_t)Cout * k, convT_taps(k, u), hsv::as_stream(stream),
              "pack_convT_weight");
}

extern "C" int hsv_conv1d_umma_astride(const void *a_blk16, int64_t a_bchunks, const void *w_packed, const float *bias,
                                       const float *residual, float *out, float *acc, int acc_mode, int B, int Cin,
                                       int Cout, int64_t L, int k, int d, int n_tile, void *stream) {
  if (B == 0 || L == 0) return HSV_OK;  // empty batch / sequence
  if (int rc = check_common("conv1d_umma", a_blk16, w_packed, Cin, Cout, n_tile)) return rc;
  HSV_REQUIRE(a_bchunks == 0 || (a_bchunks >= Cin / hsv::blk_cw(Cin) && a_bchunks <= 65535),
              "conv1d_umma: A batch stride of %lld chunks outside [%d (Cin=%d), 65535]", (long long)a_bchunks,
              Cin / hsv::blk_cw(Cin), Cin);
  HSV_REQUIRE(k >= 1 && k <= MAX_TAPS && (k & 1) && d >= 1, "conv1d_umma: k must be odd and <= %d (k=%d d=%d)",
              MAX_TAPS, k, d);
  HSV_REQUIRE(((k - 1) / 2) * d <= HSV_BLK_PAD, "conv1d_umma: halo %d exceeds blk16 padding %d",
              ((k - 1) / 2) * d, HSV_BLK_PAD);
  HSV_REQUIRE(acc_mode >= 0 && acc_mode <= 2 && (acc_mode == 0 || acc), "conv1d_umma: bad acc_mode/acc");
  HSV_REQUIRE(out || acc_mode, "conv1d_umma: no output");
  return launch(conv_taps(k, d), a_blk16, w_packed, bias, residual, out, acc, acc_mode, B, Cin, Cout, L, L, n_tile,
                hsv::as_stream(stream), "conv1d_umma", nullptr, nullptr, a_bchunks);
}

extern "C" int hsv_conv1d_umma(const void *a_blk16, const void *w_packed, const float *bias,
                               const float *residual, float *out, float *acc, int acc_mode, float /*acc_div: reserved*/,
                               int B, int Cin, int Cout, int64_t L, int k, int d, int n_tile, void *stream) {
  return hsv_conv1d_umma_astride(a_blk16, 0, w_packed, bias, residual, out, acc, acc_mode, B, Cin, Cout, L, k, d, n_tile,
                                 stream);
}

extern "C" int hsv_conv1d_umma_blk16(const void *a_blk16, const void *w_packed, const float *bias, void *out_blk16, int mode,
                                     const float *bc, int64_t bc_stride, const float *mask, int B, int Cin, int Cout,
                                     int64_t L, int k, int d, int n_tile, void *stream) {
  if (B == 0 || L == 0) return HSV_OK;  // empty batch / sequence
  if (int rc = check_common("conv1d_umma_blk16", a_blk16, w_packed, Cin, Cout, n_tile)) return rc;
  HSV_REQUIRE(out_blk16 && out_blk16 != a_blk16, "conv1d_umma_blk16: bad output buffer");
  HSV_REQUIRE(mode >= 0 && mode <= 3, "conv1d_umma_blk16: mode %d", mode);
  HSV_REQUIRE(mode != 1 || Cout % 32 == 0, "conv1d_umma_blk16: the gate needs Cout %% 32 == 0 (Cout=%d)", Cout);
  HSV_REQUIRE(k >= 1 && k <= MAX_TAPS && (k & 1) && d >= 1, "conv1d_umma_blk16: k must be odd and <= %d (k=%d d=%d)",
              MAX_TAPS, k, d);
  HSV_REQUIRE(((k - 1) / 2) * d <= HSV_BLK_PAD, "conv1d_umma_blk16: halo %d exceeds blk16 padding %d", ((k - 1) / 2) * d,
              HSV_BLK_PAD);
  const BlkOut bo = {out_blk16, mode, mode == 1 ? Cout / 2 : Cout, bc, bc_stride, mask, nullptr, nullptr};
  return launch(conv_taps(k, d), a_blk16, w_packed, bias, nullptr, nullptr, nullptr, 0, B, Cin, Cout, L, L, n_tile,
                hsv::as_stream(stream), "conv1d_umma_blk16", nullptr, &bo);
}

extern "C" int hsv_conv1d_umma_wn_tail(const void *a_blk16, const void *w_packed, const float *bias, float *x, float *output,
                                       const float *mask, void *next_blk16, int B, int Cin, int H, int64_t L, int n_tile,
                                       void *stream) {
  if (B == 0 || L == 0) return HSV_OK;
  if (int rc = check_common("conv1d_umma_wn_tail", a_blk16, w_packed, Cin, 2 * H, n_tile)) return rc;
  HSV_REQUIRE(x && output && next_blk16 && next_blk16 != a_blk16, "conv1d_umma_wn_tail: null / aliased buffer");
  HSV_REQUIRE(H % n_tile == 0, "conv1d_umma_wn_tail: H=%d must be a multiple of n_tile=%d", H, n_tile);
  const BlkOut bo = {next_blk16, 4, H, nullptr, 0, mask, x, output};
  return launch(conv_taps(1, 1), a_blk16, w_packed, bias, nullptr, nullptr, nullptr, 0, B, Cin, 2 * H, L, L, n_tile,
                hsv::as_stream(stream), "conv1d_umma_wn_tail", nullptr, &bo);
}

extern "C" int hsv_act_conv1d_umma(const float *x, const float *alpha, const float *beta, float in_scale,
                                   const void *w_packed, const float *bias, const float *residual, float *out,
                                   float *acc, int acc_mode, int B, int Cin, int Cout, int64_t L, int k, int d,
                                   void *stream) {
  if (B == 0 || L == 0) return HSV_OK;  // empty batch / sequence
  HSV_REQUIRE(x && alpha && beta, "act_conv1d_umma: null pointer");
  HSV_REQUIRE(Cin == 16 || Cin == 32 || Cin == 64, "act_conv1d_umma: Cin must be 16, 32 or 64 (Cin=%d)", Cin);
  if (int rc = check_common("act_conv1d_umma", x, w_packed, Cin, Cout, Cout)) return rc;
  HSV_REQUIRE(k >= 1 && k <= MAX_TAPS && (k & 1) && d >= 1, "act_conv1d_umma: k must be odd and <= %d (k=%d d=%d)",
              MAX_TAPS, k, d);
  HSV_REQUIRE(((k - 1) / 2) * d <= HSV_BLK_PAD, "act_conv1d_umma: halo %d exceeds %d", ((k - 1) / 2) * d, HSV_BLK_PAD);
  HSV_REQUIRE(acc_mode >= 0 && acc_mode <= 2 && (acc_mode == 0 || acc), "act_conv1d_umma: bad acc_mode/acc");
  HSV_REQUIRE(out || acc_mode, "act_conv1d_umma: no output");
  HSV_REQUIRE(out != x && acc != x, "act_conv1d_umma: the output must not alias the activation input");
  const FusedAct fa = {x, alpha, beta, in_scale};
  return launch(conv_taps(k, d), x, w_packed, bias, residual, out, acc, acc_mode, B, Cin, Cout, L, L, Cout,
                hsv::as_stream(stream), "act_conv1d_umma", &fa);
}

extern "C" int hsv_conv_transpose1d_umma(const void *a_blk16, const void *w_packed, const float *bias,
                                         const float *add, float *out, int B, int Cin, int Cout, int64_t Lin,
                                         int k, int u, int n_tile, void *stream) {
  if (B == 0 || Lin == 0) return HSV_OK;
  if (int rc = check_common("conv_transpose1d_umma", a_blk16, w_packed, Cin, Cout, n_tile)) return rc;
  HSV_REQUIRE(u >= 1 && u <= MAX_PHASES && k >= u && k <= MAX_TAPS && k - 2 * ((k - u) / 2) == u,
              "conv_transpose1d_umma: unsupported (k,u)=(%d,%d)", k, u);
  HSV_REQUIRE(out, "conv_transpose1d_umma: no output");
  return launch(convT_taps(k, u), a_blk16, w_packed, bias, add, out, nullptr, 0, B, Cin, Cout, Lin,
                (int64_t)u * Lin, n_tile, hsv::as_stream(stream), "conv_transpose1d_umma");
}
