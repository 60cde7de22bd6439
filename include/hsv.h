/*
 * hsv.h — C-ABI of the B200 (sm_100a) waveform-generation kernels.
 *
 * The reference (liuhuang31/Megatts2_HierSpeechpp) is pure Python/PyTorch and
 * has no FFI for this path; its "operator interface" is the set of ATen calls
 * made by the nn.Modules on the hot path.  Each entry point below replaces one
 * such call group and cites it (paths relative to the reference root).  The
 * Python host side (megatts2_hierspeechpp_b200/) binds these with ctypes and
 * mirrors the reference's nn.Module classes on top (see INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers and sizes only; all pointers are DEVICE pointers unless
 *     named host_*; the caller (PyTorch) owns every buffer, nothing is
 *     allocated or freed here;
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on
 *     that stream, does no host synchronisation and is CUDA-graph capturable;
 *   - return value 0 = success, negative = error (hsv_last_error() gives the
 *     message, thread-local);
 *   - activations are fp32, layout [B, C, L] contiguous ("NCL", the
 *     reference's layout) unless stated otherwise;
 *   - "blk16" is the tensor-core operand layout produced by the activation
 *     kernel and consumed by hsv_conv1d_umma: fp16 [B][C/CW][Lp][CW], CW = 64
 *     (C % 64 == 0), else 32 (C % 32 == 0), else 16 channels per row, with
 *     Lp = HSV_BLK_PAD + roundup(L,HSV_BLK_ROUND) + HSV_BLK_PAD rows per (b, chunk);
 *     within the buffer of one (b, chunk) the 16-byte unit at linear byte offset
 *     o is stored at o ^ (((o >> 7) & (CW/8 - 1)) << 4)  -- tcgen05's K-major
 *     SWIZZLE_128B/64B/32B pattern, so a linear (1-D bulk TMA) copy of a row span
 *     into 1024-byte aligned shared memory is a ready MMA operand tile.  Rows
 *     outside [HSV_BLK_PAD, HSV_BLK_PAD+L) must be zero (they implement the
 *     conv's zero padding) and are never written.  Treat the buffer as opaque:
 *     hsv_pack_blk16 / hsv_unpack_blk16 convert from / to fp32 [B,C,L].
 */
#ifndef HSV_H_
#define HSV_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HSV_VERSION 100
#define HSV_BLK_PAD 32          /* zero rows before/after each blk16 sequence */
#define HSV_UMMA_TILE_M 128     /* rows of one tcgen05 accumulator tile */
#define HSV_BLK_ROUND 512       /* blk16 sequences are padded to a multiple of this many rows (max CTA tile) */

/* error codes */
#define HSV_OK 0
#define HSV_ERR_ARG (-1)        /* bad argument / unsupported shape */
#define HSV_ERR_CUDA (-2)       /* CUDA runtime error at launch */

int hsv_version(void);
const char *hsv_last_error(void);
/* 1 if the running device is compute capability 10.x (tcgen05 capable). */
int hsv_device_supported(void);

/* Rows per (b, chunk) of a blk16 buffer for sequence length L. */
int64_t hsv_blk16_rows(int64_t L);

/* Test hook, read-only: which kernel variant the most recent host-side launch decision of a family chose.
 * Process-global (like the bring-up switches); it never changes what is launched.  Copies min(n, count) ints to
 * out and returns count (negative on a bad argument).
 *   family 0, tcgen05 conv (count 15): kind (0 one-tile, 1 persistent, 2 fused activation, 3 operand-writing
 *             epilogue), msub, warps per CTA, vec_epi (float4 epilogue), nphase, n_tile, stages, G (weight blocks
 *             per ring stage), resident, nabuf (persistent only, else 0), grid x, y, z, blk_mode (kind 3: the
 *             hsv_conv1d_umma_blk16 mode 0-3, 4 = hsv_conv1d_umma_wn_tail; else 0), launches so far
 *   family 1, Activation1d (count 5): run length R (0 when the tensor-core kernel ran), act1d_mma ran, out_mode,
 *             valid_len given (hsv_act1d_snakebeta_ragged with lengths), launches so far
 *   family 2, attention (count 13): kernel (0 tensor-core, 1 fp32 CUDA-core), D, out_mode, lens given, valid_len
 *             given, prescale, kv16 (K / V tiles copied in 16-byte chunks: Tk % 4 == 0, 16-byte aligned k and v,
 *             batch strides % 4 == 0), q16 (tensor-core kernel: Q tiles copied in 16-byte chunks: Tq % 4 == 0,
 *             16-byte aligned q, q batch stride % 4 == 0; 0 for the fp32 kernel), key tiles, grid x, y, z, launches
 *             so far
 *   family 3, CUDA-core conv (hsv_conv1d_direct[_ragged], hsv_conv_transpose1d_direct; count 7): kernel (0 vecdot,
 *             1 rowdot, 2 thin_vec, 3 thin_smem, 4 thin, 5 tiled, 6 ConvTranspose direct), flags (HSV_CONV_*; for
 *             the ConvTranspose HSV_CONV_ADD_OUT when `add` is given, else 0), valid_len given, grid x, y, z,
 *             launches so far.  A call that launches nothing (B = 0, Lout <= 0 or Lin = 0) leaves it unchanged. */
int hsv_last_launch_config(int family, int *out, int n);

/* ---- Activation1d(SnakeBeta): alias_free_torch/act.py:23-27 =
 * UpSample1d (resample.py:25-32) o SnakeBeta (activations.py:107-119, log-scale
 * alpha/beta) o DownSample1d (resample.py:46-48 -> filter.py:86-94), with the
 * fixed 12-tap kaiser-sinc filter (filter.py:28-57) — ONE fused kernel.
 *   x      [B,C,L] fp32
 *   alpha, beta [C] fp32 (log scale, as stored in the state_dict)
 *   out_mode 0: out = fp32 [B,C,L]
 *   out_mode 1: out = fp16 blk16 (C % 16 == 0), rows per chunk = hsv_blk16_rows(L)
 *   in_scale    x is multiplied by this first (1/num_kernels: the "xs / self.num_kernels" of
 *               hierspeechpp_speechsynthesizer.py:446 when x is the un-normalised sum over resblocks)
 */
int hsv_act1d_snakebeta(const float *x, void *out, const float *alpha, const float *beta,
                        int B, int C, int64_t L, int out_mode, float in_scale, void *stream);
/* The same for a ragged batch (utterances of different lengths padded to L):
 *   valid_len [B] int32, device (NULL = L for every item); values are clamped to [0, L] on the device.
 * Item b is a sequence of Lv = valid_len[b] steps stored with row stride L: x at t >= Lv is never read, the
 * edge replication happens at Lv, and outputs at Lv <= t < L are written as 0 (both out modes), so out[b, :, :Lv]
 * equals, bit for bit, the call on that item alone with L = Lv.  Returns HSV_ERR_ARG when the tensor-core variant
 * is forced (hsv_set_act_variant), which takes no lengths. */
int hsv_act1d_snakebeta_ragged(const float *x, void *out, const float *alpha, const float *beta,
                               const int32_t *valid_len, int B, int C, int64_t L, int out_mode, float in_scale,
                               void *stream);

/* ---- weight norm fold: torch._weight_norm(v, g, dim=0) as applied by the
 * forward pre-hook of torch.nn.utils.weight_norm on every conv of the path
 * (hierspeechpp_speechsynthesizer.py:401,406,349-364; speechsr.py:21-36,73).
 *   v [n0, inner], g [n0]  ->  w [n0, inner] = v * g / ||v||_2(row)
 */
int hsv_weight_norm_fold(const float *v, const float *g, float *w, int n0, int inner, void *stream);

/* ---- pack a folded Conv1d weight [Cout,Cin,k] fp32 into the tcgen05 B-operand
 * stream: fp16 [Cout/n_tile][Cin/CW][k] blocks of n_tile rows x CW channels
 * (K-major, swizzled like blk16).  Cin % 16 == 0, Cout % n_tile == 0,
 * n_tile % 16 == 0, n_tile <= 256.  Size: Cout*Cin*k halves.
 */
int hsv_pack_conv_weight(const float *w, void *packed, int Cout, int Cin, int k, int n_tile, void *stream);

/* ---- dilated 'same' Conv1d as a tcgen05/TMEM implicit GEMM:
 * the AMPBlock convs (hierspeechpp_speechsynthesizer.py:349-364,380-384;
 * speechsr24k/speechsr.py:21-36,52-56): F.conv1d(x, w, b, dilation=d,
 * padding=(k*d-d)/2), fp16 operands, fp32 accumulation, fused epilogue.
 *   a_blk16   fp16 blk16 activations (B*Cin*Lp halves)
 *   w_packed  from hsv_pack_conv_weight (same n_tile)
 *   bias      [Cout] fp32 or NULL
 *   residual  [B,Cout,L] fp32 or NULL     (v = acc + bias + residual)
 *   out       [B,Cout,L] fp32 or NULL     (out = v; may alias residual)
 *   acc       [B,Cout,L] fp32 or NULL, acc_mode: 0 none, 1 acc = v, 2 acc += v (sum over
 *             resblocks, hierspeechpp_speechsynthesizer.py:440-445; the division by
 *             num_kernels (:446) is the consumer's in_scale).  acc_div is reserved (pass 1).
 */
int hsv_conv1d_umma(const void *a_blk16, const void *w_packed, const float *bias,
                    const float *residual, float *out, float *acc, int acc_mode, float acc_div,
                    int B, int Cin, int Cout, int64_t L, int k, int d, int n_tile, void *stream);
/* The same with an explicit batch stride of the operand: a_bchunks = operand chunks (CW channels x
 * hsv_blk16_rows(L) rows each) from one batch item to the next (0 = Cin / CW, a dense buffer).  A channel
 * range [c0, c0 + Cin) of a wider blk16 buffer with the same CW is then read in place at any batch size:
 * a_blk16 = the buffer + the byte offset of chunk c0 / CW of item 0, a_bchunks = the wider buffer's chunks
 * per item (split-K passes over one packed operand).  Results equal a dense copy of the range, bit for bit. */
int hsv_conv1d_umma_astride(const void *a_blk16, int64_t a_bchunks, const void *w_packed, const float *bias,
                            const float *residual, float *out, float *acc, int acc_mode, int B, int Cin, int Cout,
                            int64_t L, int k, int d, int n_tile, void *stream);

/* hsv_conv1d_umma_blk16: the same convolution with an OPERAND-WRITING epilogue: (conv + bias + bc[b]) -> activation ->
 * * mask -> fp16 blk16 buffer that the next hsv_conv1d_umma reads (no fp32 round trip, no pack launch).
 *   mode 0: none;  2: gelu_tanh (FFN_Conv, modules.py:382-388);  3: leaky_relu(0.1);
 *   mode 1: the WN gate tanh(a) * sigmoid(b) (commons.py:108-114): the caller packs the weights / bias / bc with the
 *           output channels ordered as groups of [8 tanh | 8 sigmoid] (channels 8j..8j+7 then H+8j..H+8j+7), the
 *           output buffer has Cout / 2 channels.
 *   bc: [B][Cout] (batch stride bc_stride) added before the activation, or NULL; mask: [B][L] or NULL. */
int hsv_conv1d_umma_blk16(const void *a_blk16, const void *w_packed, const float *bias, void *out_blk16, int mode,
                          const float *bc, int64_t bc_stride, const float *mask, int B, int Cin, int Cout, int64_t L, int k,
                          int d, int n_tile, void *stream);

/* hsv_conv1d_umma_wn_tail: a WN layer's res_skip 1x1 conv (Cin -> 2H) with the layer tail in its epilogue (modules.py:167-174):
 * x = (x + rs[:, :H]) * mask in place, output += rs[:, H:] in place, and the new x written as the next in_layer's fp16
 * blk16 operand.  H must be a multiple of n_tile. */
int hsv_conv1d_umma_wn_tail(const void *a_blk16, const void *w_packed, const float *bias, float *x, float *output,
                            const float *mask, void *next_blk16, int B, int Cin, int H, int64_t L, int n_tile, void *stream);

/* ---- whole AMP half-layer (SURVEY.md §8f1): Activation1d(SnakeBeta) followed by the dilated Conv1d,
 *   xt = conv(Activation1d(x * in_scale))            (hierspeechpp_speechsynthesizer.py:380-384)
 * in ONE kernel: the CTA evaluates the fused activation on the fp32 input and writes the fp16 operand
 * straight into the shared-memory MMA tile, so the operand never exists in HBM.  Same arithmetic as
 * hsv_act1d_snakebeta(out_mode 1) + hsv_conv1d_umma (bit-identical results).
 *   x [B,Cin,L] fp32, Cin in {16, 32, 64}; w_packed from hsv_pack_conv_weight with n_tile = Cout (<= 256);
 *   bias / residual / out / acc / acc_mode as hsv_conv1d_umma; out and acc must not alias x
 *   (other CTAs still read x's halo); residual may alias out.
 */
int hsv_act_conv1d_umma(const float *x, const float *alpha, const float *beta, float in_scale,
                        const void *w_packed, const float *bias, const float *residual, float *out,
                        float *acc, int acc_mode, int B, int Cin, int Cout, int64_t L, int k, int d,
                        void *stream);

/* ---- ConvTranspose1d (ups[i], hierspeechpp_speechsynthesizer.py:404-408,434) on the same
 * tcgen05 kernel: the u output phases are u stride-1 convolutions over the input rows
 * (SURVEY.md §A.3), each an N-tile group of one launch.
 *   hsv_pack_convT_weight: w [Cin,Cout,k] fp32 (folded) -> fp16 [phase][Cout/n_tile][Cin/CW][taps] blocks
 *   hsv_conv_transpose1d_umma: a_blk16 (rows per chunk = hsv_blk16_rows(Lin)) -> out [B,Cout,u*Lin] fp32,
 *   out = convT + bias (+ add, same shape as out: proj(pitch) at stage 0, :436-438).
 *   stride u <= 8, padding (k-u)/2, k - 2*((k-u)/2) == u (true for every (k,u) on the path).
 */
int hsv_pack_convT_weight(const float *w, void *packed, int Cin, int Cout, int k, int u, int n_tile, void *stream);
int hsv_conv_transpose1d_umma(const void *a_blk16, const void *w_packed, const float *bias, const float *add,
                              float *out, int B, int Cin, int Cout, int64_t Lin, int k, int u, int n_tile,
                              void *stream);

/* ---- generic fp32 Conv1d (stride 1, zero padding `pad`, dilation d) on CUDA
 * cores, for the small/odd-shaped convs of the path: conv_pre, cond, proj,
 * DBlock convs, conv_post (+tanh) (hierspeechpp_speechsynthesizer.py:401,
 * 421-426,430,437,449-450; speechsr.py:106-107).
 *   x [B,Cin,Lin], w [Cout,Cin,k], bias [Cout] or NULL -> out [B,Cout,Lout],
 *   Lout = Lin + 2*pad - d*(k-1).
 *   flags: HSV_CONV_LRELU_IN  apply leaky_relu(0.1) to x first (DBlock :336-337)
 *          HSV_CONV_TANH      tanh on the result (Generator :450)
 *          HSV_CONV_ADD_OUT   out += result instead of out = result
 */
#define HSV_CONV_LRELU_IN 1
#define HSV_CONV_TANH 2
#define HSV_CONV_ADD_OUT 4
#define HSV_CONV_SILU_IN 8      /* apply SiLU to x first (adaLN / cond_block, modules.py:402, hierspeechpp_speechsynthesizer.py:70) */
#define HSV_CONV_LRELU001_IN 16 /* apply leaky_relu(0.01) to x first (PitchPredictor, ttv_v1/t2w2v_transformer.py:456) */
int hsv_conv1d_direct(const float *x, const float *w, const float *bias, float *out,
                      int B, int Cin, int Cout, int64_t Lin, int64_t Lout, int k, int d, int pad,
                      int flags, void *stream);
/* The same for a ragged batch: valid_len [B] int32, device (NULL = as hsv_conv1d_direct), clamped to [0, Lin].
 * Item b uses x at t < valid_len[b] only (the rest counts as 0: values there never reach the result, though the float4
 * staging of aligned rows may load the 16 bytes that straddle valid_len[b]) and writes 0 at t >= valid_len[b]; its first valid_len[b]
 * outputs equal, bit for bit, hsv_conv1d_direct on that item alone with Lin = Lout = valid_len[b].  With valid_len,
 * only the conv_post shape is supported (Cout <= 4, k = 7, d = 1, pad = 3, Lout == Lin); others return HSV_ERR_ARG. */
int hsv_conv1d_direct_ragged(const float *x, const float *w, const float *bias, const int32_t *valid_len, float *out,
                             int B, int Cin, int Cout, int64_t Lin, int64_t Lout, int k, int d, int pad, int flags,
                             void *stream);

/* ---- ConvTranspose1d (ups[i], hierspeechpp_speechsynthesizer.py:404-408,434):
 *   x [B,Cin,Lin], w [Cin,Cout,k] (folded), bias [Cout] -> out [B,Cout,u*Lin],
 *   stride u, padding (k-u)/2, output_padding 0.  add [B,Cout,u*Lin] or NULL is
 *   added to the result (proj(pitch) at stage 0, :436-438).
 */
int hsv_conv_transpose1d_direct(const float *x, const float *w, const float *bias, const float *add,
                                float *out, int B, int Cin, int Cout, int64_t Lin, int k, int u,
                                void *stream);

/* ---- SpeechSR front end: conv_pre (Cin=1, k=7, pad 3; speechsr.py:90) followed
 * by F.interpolate(mode='linear', align_corners=False) to Lout (speechsr.py:96),
 * fused.  x [B,1,Lin], w [C,1,7], bias [C] -> out [B,C,Lout].
 * Source index math in fp32 exactly as ATen's CUDA kernel (SURVEY.md §A.5).
 */
int hsv_sr_pre_interp(const float *x, const float *w, const float *bias, float *out,
                      int B, int C, int64_t Lin, int64_t Lout, void *stream);
/* The same for a ragged batch: valid_len_in [B] / valid_len_out [B] int32, device (each NULL = Lin / Lout), clamped
 * to [0, Lin] / [0, Lout].  Item b is interpolated from Lin_b to Lout_b samples with its own scale
 * (float)Lin_b / (float)Lout_b, conv_pre's zero padding sits at Lin_b, and outputs at t >= Lout_b are 0: out[b, :, :Lout_b]
 * equals, bit for bit, hsv_sr_pre_interp on that item alone with Lin = Lin_b, Lout = Lout_b. */
int hsv_sr_pre_interp_ragged(const float *x, const float *w, const float *bias, const int32_t *valid_len_in,
                             const int32_t *valid_len_out, float *out, int B, int C, int64_t Lin, int64_t Lout,
                             void *stream);

/* Streaming windows (hsv.SpeechSRStream): item b is a window x[b, 0, :valid_len_in[b]] of a longer stream, whose input
 * sample 0 is the stream's sample origin[b, 0] and whose output sample 0 is the stream's output origin[b, 1]; origin
 * [B, 3] int64, device.  Output t of the window is computed for the stream's output index origin[b, 1] + t with the
 * stream's constant scale (float)down / (float)up (up / down = 3 / 1 or 3 / 2, the ratio Lout / Lin), the Lin - 1
 * clamp at the stream's total length origin[b, 2] when that is >= 0 (no clamp when it is -1), and conv_pre taps
 * outside the window read 0; outputs at t >= valid_len_out[b] are 0.  An output whose taps all lie inside the window
 * (or at the stream's own edges) equals, bit for bit, hsv_sr_pre_interp on the whole stream, provided the stream's
 * length L has up * L < 2^24 and is a multiple of down. */
int hsv_sr_pre_interp_stream(const float *x, const float *w, const float *bias, const int32_t *valid_len_in,
                             const int32_t *valid_len_out, const int64_t *origin, float *out, int B, int C,
                             int64_t Lin, int64_t Lout, int up, int down, void *stream);

/* Per-step bookkeeping of S concurrent SpeechSR streams (all device memory, nothing read back).
 * State: hist [S, H] fp32 (the last min(received, H) input samples of each slot, right-aligned) and state [S, 3] int64
 * (samples received, output samples emitted, stream open), zero-initialised.  Inputs: x_new [S, N] fp32, n_new [S]
 * int32 (valid samples of x_new per slot), start / end [S] int32 flags (a new stream begins in this slot / this is its
 * last chunk).  A slot request is ignored (the slot stays as it was and emits nothing) when n_new < 0, n_new > N,
 * n_new % down != 0, or when it carries samples or an end while no stream is open and start is not set.
 * Window: writes win [S, H + N] (history then new samples), the windows' valid lengths in / out (0 for slots with
 * nothing to emit), origin [S, 3] for hsv_sr_pre_interp_stream and a plan [S, 6] int64 for the emit launch; state
 * and hist are only read.  The stream's first (received * up / down - lookahead) outputs are final before its end,
 * all of them at its end. */
int hsv_sr_stream_window(const float *x_new, const int32_t *n_new, const int32_t *start, const int32_t *end,
                         const float *hist, const int64_t *state, float *win, int32_t *valid_len_in,
                         int32_t *valid_len_out, int64_t *origin, int64_t *plan, int S, int N, int H, int up, int down,
                         int lookahead, void *stream);
/* Emit: y [S, Lout] (the windows' SpeechSR outputs, Lout = (H + N) * up / down) -> out [S, cap] (each slot's newly final
 * outputs, then zeros) and n_out [S] int32; advances hist and state (a slot closed by end is reset). */
int hsv_sr_stream_emit(const float *y, const float *win, const int64_t *origin, const int64_t *plan, float *hist,
                       int64_t *state, float *out, int32_t *n_out, int S, int H, int W, int64_t Lout, int cap,
                       void *stream);

/* Index probe for the bit-exact part of the parity contract: writes, for each
 * dst in [0,Lout): i0, i1 (int32) and lambda (fp32) of the linear interpolation. */
int hsv_interp_linear_table(int64_t Lin, int64_t Lout, int32_t *i0, int32_t *i1, float *lam, void *stream);

/* ---- nearest-neighbour down-sampling gather of DBlock
 * (F.interpolate(x, size=L//factor), hierspeechpp_speechsynthesizer.py:329-334):
 * out[b,c,t] = x[b,c,min(floor(t*scale), Lin-1)], scale = (float)Lin/Lout. */
int hsv_nearest_gather(const float *x, float *out, int rows, int64_t Lin, int64_t Lout, void *stream);

/* out[i] = a[i] + b[i] + c[row(i)] ... small fused adds used at the stage-0 join
 * (x = conv_pre(x) + downs(pitch) + cond(g), :430): out = a + b + bc[b,c,0]. */
int hsv_add3_bcast(const float *a, const float *b, const float *bc, float *out,
                   int rows, int64_t L, void *stream);

/* fp32 [B,C,L] * in_scale -> fp16 blk16 (optional leaky_relu(0.1) first); C % 16 == 0. */
int hsv_pack_blk16(const float *x, void *out, int B, int C, int64_t L, int lrelu, float in_scale, void *stream);
/* the same with the operand = ((x1 + x2) + x3) * in_scale (x2, x3 nullable): the sum over the resblocks of a stage
 * (hierspeechpp_speechsynthesizer.py:440-446) taken by the consumer, each resblock writing its own tensor. */
int hsv_pack_blk16_sum3(const float *x1, const float *x2, const float *x3, void *out, int B, int C, int64_t L,
                        int lrelu, float in_scale, void *stream);
/* the same for a ragged batch: valid_len [B] int32, device (NULL = L for every item); rows t >= valid_len[b] of item
 * b are written as zero without reading x (the zero padding of the item's own run). */
int hsv_pack_blk16_sum3_ragged(const float *x1, const float *x2, const float *x3, const int32_t *valid_len, void *out,
                               int B, int C, int64_t L, int lrelu, float in_scale, void *stream);
/* inverse (tests / debugging): fp16 blk16 -> fp32 [B,C,L]. */
int hsv_unpack_blk16(const void *in, float *x, int B, int C, int64_t L, void *stream);
/* operand health (debugging aid; the reference keeps fp32 everywhere, the tensor-core operands here are fp16):
 * stats[0] (uint32) += number of non-finite values in the valid rows of a blk16 buffer (an activation beyond
 * +-65504 saturates to inf when the operand is produced), stats[1] (float bits, non-negative) = max(stats[1],
 * max |finite value|).  The caller zeroes stats[2] first. */
int hsv_blk16_stats(const void *in, void *stats, int B, int C, int64_t L, void *stream);

/* ---- the step after the path (SURVEY.md §8f3): peak-normalise + int16 quantise on the device.
 * Replaces inference_plm.py:183-188 (audio / abs(audio).max() * 32767.0 * s) and
 * inference_speechsr.py:39-41 (audio / abs(audio).max() * 0.999 * 32767.0), each followed by
 * .cpu().numpy().astype('int16'):  out = trunc(((x / peak) * s1) * s2), fp32, operations rounded
 * separately in that order (bit-exact with the reference), saturated to int16.
 *   x [rows, L] fp32, out [rows, L] int16, peak_ws [rows] fp32 workspace (receives the peaks)
 *   per_row 0: peak = max |x| over the whole tensor (the reference's semantics, one utterance);
 *           1: one peak per row (batched utterances are normalised independently).
 */
int hsv_peak_norm_pcm16(const float *x, int16_t *out, float *peak_ws, int rows, int64_t L, float s1, float s2,
                        int per_row, void *stream);
/* the same with one peak and one s2 per row: s2 [rows] fp32, device (the prompt peak of each utterance,
 * inference_plm.py:183-188 with scale_norm="prompt").  Row b equals hsv_peak_norm_pcm16 of row b alone with s2[b]. */
int hsv_peak_norm_pcm16_rows(const float *x, int16_t *out, float *peak_ws, int rows, int64_t L, float s1,
                             const float *s2, void *stream);

/* ---- the step before SpeechSR (inference_speechsr.py:28-34): torchaudio.functional.resample(x, orig, new_freq,
 * resampling_method="kaiser_window") (lowpass_filter_width 6, rolloff 0.99, beta 14.769656459379492) of a ragged batch
 * with one rate per item (csrc/resample.cu).
 *   x          [B, T] fp32 (x_int16 = 0) or int16 PCM (x_int16 = 1, read as (float)s * (1.0f / 32768), exact)
 *   rate       [B] int32, device: each item's sample rate
 *   valid_len  [B] int32, device: each item's input samples, clamped to [0, T]; x[b, t >= valid_len[b]] is never
 *              read and counts as zero, as torchaudio's padding does
 *   host_desc  [n_desc][6] int32, HOST (1 <= n_desc <= 16, distinct rates): {rate, o, n, width, K, offset} with
 *              o : n = rate : new_freq reduced, K = 2 width + o, the item's filter stored transposed as
 *              table[offset + k * n + p] = torchaudio's kernel[p, 0, k] (fp32).  The entry of rate == new_freq is the
 *              copy {new_freq, 1, 1, 0, 0, 0}: its items are copied (converted, for int16), bit for bit.
 *   table      [table_len] fp32, device (may be NULL when table_len == 0)
 *   out        [B, T_out] fp32, n_out [B] int32, device
 * Item b's first n_out[b] = min(N_b, T_out) outputs, N_b = min(ceil((float)((double)(n L_b) / o)), (L_b / o + 1) n)
 * (torchaudio's output count: its ceil(torch.as_tensor(n * L / o)) rounds the quotient to fp32), are y[f n + p] = sum_{k < K} t[p][k] x[f o + k -
 * width], summed in an order that depends on K alone, so they equal, bit for bit, the item's own call with B = 1 and
 * no padding; the rest of its row is 0.  An item whose rate has no descriptor gets n_out = 0 and zeros;
 * nothing else is checked on the device.  Argument errors (descriptors, shapes, a rate ratio whose 256 outputs need
 * more than 12288 staged input samples) are reported before any CUDA call. */
int hsv_resample_ragged(const void *x, int x_int16, const int32_t *rate, const int32_t *valid_len, const float *table,
                        int64_t table_len, const int32_t *host_desc, int n_desc, int new_freq, float *out,
                        int32_t *n_out, int B, int64_t T, int64_t T_out, void *stream);

/* ---- frame-rate operators of the step BEFORE the vocoder (SURVEY.md §8f2; csrc/frame_ops.cu).  fp32 [B,C,T] tensors,
 * mask = [B,T] (1 = valid frame, may be NULL), blk16 outputs feed hsv_conv1d_umma.
 *
 * hsv_pack_blk16_act: operand packer with a fused activation.
 *   mode 0: x * mask;  1: tanh(x[c] + bc[c]) * sigmoid(x[C+c] + bc[C+c]) (x [B,2C,T], bc [B,2C] or NULL: WN gate,
 *   commons.py:108-114);  2: gelu_tanh(x) * mask (FFN_Conv, modules.py:382-388);  3: mish(x) * mask (styleencoder.py:6-10)
 *   x_channels = channels per batch item of x (a channel prefix of a wider tensor can be packed).
 * hsv_ln_mod_blk16: LayerNorm over channels (eps, no affine) [* mask] -> x*(1+scale[b,c]) + shift[b,c] (modules.py:346,
 *   405-410); inmask: x*mask first; premask bit 0: normalised*mask before the modulation, bit 1 (HSV_LN_ZERO_MASKED):
 *   operand rows where mask == 0 are written as zero (the rows past an item of a ragged batch, which its own run
 *   does not have: a following k > 1 conv then sees its zero padding); mod_stride = batch stride of shift/scale.
 * hsv_frame_op: element-wise ops (op codes in csrc/frame_ops.cu): 1 wn_res, 2 wn_last, 3 gate_add, 4 couple, 5 sample,
 *   6 mask, 7 add, 8 glu_res, 9 mish, 10 flip, 11 add_bcast.
 * hsv_mha: softmax(q k^T * scale) v per (batch, head); q/k/v channel-major [heads*D, T] with batch strides (so the fused
 *   qkv tensor of timm's Attention can be addressed in place); lens [B] int32 or NULL = masked_fill(-1e4) of
 *   attentions.py:174-175 for prefix masks; prescale_q: scale q before the product (attentions.py:164) or the scores
 *   after it (timm).
 * hsv_conv1d_c1_strided: Conv1d(1, Cout, k, stride, pad) * mask (PosteriorSFEncoder.pre_filter, :187,196).
 * hsv_masked_mean: out[b,c] = sum_t x[b,c,t] / sum_t mask[b,t] (styleencoder.py:91-99: the sum runs over all frames). */
int hsv_pack_blk16_act(const float *x, const float *bcast, const float *mask, void *out, int B, int C, int64_t L,
                       int mode, int x_channels, void *stream);
/* WN layer tail + the next layer's operand pack in one pass (modules.py:167-174): x = (x + rs[:, :C]) * mask in place,
 * output += rs[:, C:], blk = fp16 blk16 operand of the new x.  rs is [B, 2C, T]. */
int hsv_wn_res_pack(float *x, const float *rs, const float *mask, float *output, void *blk, int B, int C, int64_t L,
                    void *stream);
#define HSV_LN_ZERO_MASKED 2
int hsv_ln_mod_blk16(const float *x, const float *shift, const float *scale, const float *mask, void *out, int B, int C,
                     int64_t L, float eps, int inmask, int premask, int64_t mod_stride, void *stream);
/* hsv_gate_ln_mod_blk16: x = x + gate[b,c] * y * mask (in place, modules.py:408-409) fused with hsv_ln_mod_blk16 of the new x:
 * the gated residual update of a DiT block and the LayerNorm/modulate/pack that follows it, one pass. */
int hsv_gate_ln_mod_blk16(float *x, const float *y, const float *gate, int64_t gate_stride, const float *shift,
                          const float *scale, const float *mask, void *out, int B, int C, int64_t L, float eps, int premask,
                          int64_t mod_stride, void *stream);
int hsv_frame_op(int op, const float *a, const float *b, const float *c, const float *mask, float *out, float *out2,
                 int B, int C, int64_t L, float s, int64_t cstride, void *stream);
int hsv_mha(const float *q, const float *k, const float *v, float *out, const int *lens, int B, int heads, int D, int Tq,
            int Tk, int64_t q_bstride, int64_t k_bstride, int64_t v_bstride, float scale, int prescale_q, void *stream);
/* the same (tensor-core kernel only), the result written as the fp16 blk16 operand [heads*D channels, Tq rows] of the
 * projection conv that follows (timm Attention.proj): saves the fp32 round trip and the pack launch. */
int hsv_mha_blk16(const float *q, const float *k, const float *v, void *out_blk16, const int *lens, int B, int heads, int D,
                  int Tq, int Tk, int64_t q_bstride, int64_t k_bstride, int64_t v_bstride, float scale, int prescale_q,
                  void *stream);
/* hsv_mha (out_mode 0) / hsv_mha_blk16 (out_mode 1) for a ragged batch of self-attention (Tq == Tk, lens NULL):
 *   valid_len [B] int32, device (NULL = as hsv_mha / hsv_mha_blk16), clamped to [0, Tk].  Item b has n = valid_len[b]
 *   queries and keys stored with row pitch Tk; it runs as its own launch with Tq = Tk = n (keys past n are never read
 *   and weigh nothing), so out[b, :, :n] equals that launch bit for bit, and its rows [n, Tq) are written as 0 in
 *   both out modes.  Unlike lens (masked_fill(-1e4) over the padded length), the padding does not take part at all.
 *   Tensor-core kernel only: returns HSV_ERR_ARG with valid_len under hsv_set_mha_variant(1). */
int hsv_mha_ragged(const float *q, const float *k, const float *v, void *out, int out_mode, const int *lens,
                   const int32_t *valid_len, int B, int heads, int D, int Tq, int Tk, int64_t q_bstride,
                   int64_t k_bstride, int64_t v_bstride, float scale, int prescale_q, void *stream);
/* test hook: 0 = tensor-core attention (csrc/mha_mma.cu, default), 1 = the fp32 CUDA-core kernel. Process-global. */
int hsv_set_mha_variant(int v);
int hsv_conv1d_c1_strided(const float *x, const float *w, const float *bias, const float *mask, float *out, int B,
                          int Cout, int64_t Lin, int64_t Lout, int k, int stride, int pad, void *stream);
/* the same for a ragged batch: valid_len [B] int32, device (NULL = as above), in OUTPUT frames, clamped to [0, Lout].
 * Item b reads x[b, 0, :stride * valid_len[b]] only (samples past it are the conv's zero padding, as in its own run with
 * Lin = stride * valid_len[b]) and writes 0 at t >= valid_len[b]. */
int hsv_conv1d_c1_strided_ragged(const float *x, const float *w, const float *bias, const float *mask,
                                 const int32_t *valid_len, float *out, int B, int Cout, int64_t Lin, int64_t Lout, int k,
                                 int stride, int pad, void *stream);
int hsv_masked_mean(const float *x, const float *mask, float *out, int B, int C, int64_t L, void *stream);
/* the same for a ragged batch: valid_len [B] int32, device (NULL = as above), clamped to [0, L].  Item b sums
 * x[b, c, :valid_len[b]] in the order of its own call with L = valid_len[b] (and an all-ones mask) and divides by
 * valid_len[b]; mask is not read. */
int hsv_masked_mean_ragged(const float *x, const float *mask, const int32_t *valid_len, float *out, int B, int C,
                           int64_t L, void *stream);

/* ---- seeded noise of per-item batches (csrc/noise.cu).  The value at (item b, channel c, frame t) depends on
 * (seeds[b], c, t) only: Philox4x32-10 keyed by the 64-bit seed, counter (t >> 2, c, 0, 0), Box-Muller normal t & 3.
 * This is the project's own bit pattern, not torch's randn stream.  seeds [B] int64, valid_len [B] int32 (NULL = T),
 * both device; 1 <= T <= 2^34.
 * hsv_seeded_normal: out [B, C, T] fp32 = the normals, 0 at t >= valid_len[b].
 * hsv_sample_ragged: out [B, C, T] = m + n * exp(logs) * s_b with stats [B, 2C, T] = (m | logs), in the operation order
 *   and with the expf of hsv_frame_op's sample op (so its output equals that op fed with the same noise and mask 1);
 *   0 at t >= valid_len[b], where nothing is read or generated.  n: generated in registers from seeds (eps NULL) or
 *   read from eps [B, C, T] (seeds NULL); s_b = noise_scale[b] ([B] fp32, device) or s when noise_scale is NULL. */
int hsv_seeded_normal(const int64_t *seeds, float *out, int B, int C, int64_t T, const int32_t *valid_len, void *stream);
int hsv_sample_ragged(const float *stats, const float *eps, const int64_t *seeds, const float *noise_scale, float s,
                      const int32_t *valid_len, float *out, int B, int C, int64_t T, void *stream);

/* ---- f0-driven harmonic sine source (BASELINE.json north_star item 3; NSF / HiFTNet-style SineGen -- the
 * reference repository has no counterpart on this path, SURVEY.md §0.3).  The phase accumulator is 64-bit fixed point
 * (2^64 = one cycle): the cumulative sum is exact integer arithmetic, so a 30 s utterance does not drift.
 *   f0        [B, T] fp32, Hz per frame (<= 0: unvoiced, the phase holds)
 *   out       [B, harmonics, T*hop] fp32 = amp * voiced * sin(2 pi (h+1) phase[n]),  phase[n] = sum_{k<=n} f0[k/hop]/sr
 *   uv        [B, T*hop] fp32 voiced mask (may be NULL)
 *   workspace hsv_sinegen_workspace(B, T, hop) bytes
 */
int64_t hsv_sinegen_workspace(int B, int64_t T, int hop);
int hsv_sinegen(const float *f0, float *out, float *uv, void *workspace, int B, int64_t T, int hop,
                float sample_rate, int harmonics, float amp, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* HSV_H_ */
