// Streaming SpeechSR: the per-step bookkeeping of S concurrent streams, entirely on the device.
//
// Each slot keeps the last H input samples of its stream (hist, right-aligned) and three counters (state: samples
// received, output samples emitted, stream open).  A step is three parts:
//   hsv_sr_stream_window   builds every slot's window = its history + its new samples, applies start / end, and
//                          writes the window's valid lengths, origins and emit range (nothing of the state changes);
//   (the ragged SpeechSR kernels run on the windows: hsv_sr_pre_interp_stream, Activation1d, tcgen05 convs, conv_post)
//   hsv_sr_stream_emit     copies each slot's final outputs, writes n_out and advances the state.
// A slot whose step carries nothing (n_new = 0, no flag) or is invalid (see hsv.h) changes nothing, so an all-idle
// step leaves the whole state bit for bit as it was.
#include "hsv_common.cuh"

namespace {

// plan row of a slot (int64 [S, 6]), written by the window launch, read by the emit launch
enum { P_EMIT0 = 0, P_EMIT1, P_RECV1, P_WLEN, P_OPEN1, P_UPDATE, P_N };
// state row (int64 [S, 3])
enum { S_RECV = 0, S_EMIT, S_OPEN, S_N };

struct SlotPlan {
  int64_t o_in, o_out, total, emit0, emit1, recv1, wlen, hlen;
  bool open1, update, active;
};

__device__ __forceinline__ SlotPlan plan_slot(const int64_t *st, int n, bool start, bool end, int N, int H, int up,
                                              int down, int lookahead) {
  const bool open = st[S_OPEN] != 0;
  // invalid requests leave the slot idle: more than N samples, a sample count the ratio cannot take, samples or an end
  // for a slot with no open stream
  if (n < 0 || n > N || (n % down) != 0 || (!open && !start && (n > 0 || end))) {
    n = 0;
    start = end = false;
  }
  SlotPlan p;
  const int64_t recv0 = start ? 0 : st[S_RECV];
  p.emit0 = start ? 0 : st[S_EMIT];
  p.hlen = recv0 < H ? recv0 : H;
  p.o_in = recv0 - p.hlen;
  p.o_out = p.o_in * up / down;
  p.recv1 = recv0 + n;
  p.wlen = p.hlen + n;
  const bool live = open || start;
  const int64_t full = p.recv1 * up / down;
  if (!live) {
    p.emit1 = p.emit0;
  } else if (end) {
    p.emit1 = full;
  } else {
    const int64_t e = full - lookahead;
    p.emit1 = e > p.emit0 ? e : p.emit0;
  }
  p.total = end ? p.recv1 : -1;
  p.open1 = live && !end;
  p.update = start || end || n > 0;
  p.active = p.emit1 > p.emit0;
  return p;
}

__global__ void sr_stream_window_kernel(const float *__restrict__ x_new, const int32_t *__restrict__ n_new,
                                        const int32_t *__restrict__ start, const int32_t *__restrict__ end,
                                        const float *__restrict__ hist, const int64_t *__restrict__ state,
                                        float *__restrict__ win, int32_t *__restrict__ vin, int32_t *__restrict__ vout,
                                        int64_t *__restrict__ origin, int64_t *__restrict__ plan, int N, int H, int W,
                                        int up, int down, int lookahead) {
  const int b = blockIdx.y;
  const SlotPlan p = plan_slot(state + (int64_t)b * S_N, __ldg(n_new + b), __ldg(start + b) != 0, __ldg(end + b) != 0,
                               N, H, up, down, lookahead);
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < W; k += gridDim.x * blockDim.x) {
    float v = 0.f;
    if (k < p.hlen) v = hist[(int64_t)b * H + (H - p.hlen) + k];
    else if (k < p.wlen) v = x_new[(int64_t)b * N + (k - p.hlen)];
    win[(int64_t)b * W + k] = v;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    // slots with nothing to emit take no work in the ragged launches
    const int32_t wl = p.active ? (int32_t)p.wlen : 0;
    vin[b] = wl;
    vout[b] = (int32_t)((int64_t)wl * up / down);
    int64_t *o = origin + (int64_t)b * 3;
    o[0] = p.o_in;
    o[1] = p.o_out;
    o[2] = p.total;
    int64_t *q = plan + (int64_t)b * P_N;
    q[P_EMIT0] = p.emit0;
    q[P_EMIT1] = p.emit1;
    q[P_RECV1] = p.recv1;
    q[P_WLEN] = p.wlen;
    q[P_OPEN1] = p.open1;
    q[P_UPDATE] = p.update;
  }
}

__global__ void sr_stream_emit_kernel(const float *__restrict__ y, const float *__restrict__ win,
                                      const int64_t *__restrict__ origin, const int64_t *__restrict__ plan,
                                      float *__restrict__ hist, int64_t *__restrict__ state, float *__restrict__ out,
                                      int32_t *__restrict__ n_out, int H, int W, int64_t Lout, int cap) {
  const int b = blockIdx.y;
  const int64_t *q = plan + (int64_t)b * P_N;
  const int64_t emit0 = q[P_EMIT0], ne = q[P_EMIT1] - emit0, wlen = q[P_WLEN];
  const int64_t first = emit0 - origin[(int64_t)b * 3 + 1];   // window-relative index of the first final output
  const bool update = q[P_UPDATE] != 0, open1 = q[P_OPEN1] != 0;
  const int64_t recv1 = q[P_RECV1];
  const int64_t h1 = recv1 < H ? recv1 : H;
  const int span = cap > H ? cap : H;
  for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < span; k += gridDim.x * blockDim.x) {
    if (k < cap) out[(int64_t)b * cap + k] = k < ne ? y[(int64_t)b * Lout + first + k] : 0.f;
    // the history keeps the last h1 samples of the stream (the window's last h1); a closed slot keeps none
    if (update && open1 && k < h1) hist[(int64_t)b * H + (H - h1) + k] = win[(int64_t)b * W + (wlen - h1) + k];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    n_out[b] = (int32_t)ne;
    if (update) {
      int64_t *s = state + (int64_t)b * S_N;
      s[S_RECV] = open1 ? recv1 : 0;
      s[S_EMIT] = open1 ? q[P_EMIT1] : 0;
      s[S_OPEN] = open1;
    }
  }
}

}  // namespace

extern "C" int hsv_sr_stream_window(const float *x_new, const int32_t *n_new, const int32_t *start, const int32_t *end,
                                    const float *hist, const int64_t *state, float *win, int32_t *valid_len_in,
                                    int32_t *valid_len_out, int64_t *origin, int64_t *plan, int S, int N, int H,
                                    int up, int down, int lookahead, void *stream) {
  if (S == 0) return HSV_OK;
  HSV_REQUIRE(x_new && n_new && start && end && hist && state && win && valid_len_in && valid_len_out && origin && plan,
              "sr_stream_window: null pointer");
  HSV_REQUIRE(S > 0 && S <= 65535 && N > 0 && H > 0 && lookahead >= 0, "sr_stream_window: bad shape");
  HSV_REQUIRE((up == 3 && down == 1) || (up == 3 && down == 2), "sr_stream_window: ratio must be 3/1 or 3/2");
  HSV_REQUIRE(H % down == 0, "sr_stream_window: history %d not a multiple of %d", H, down);
  const int W = H + N;
  dim3 grid((unsigned)((W + 255) / 256), (unsigned)S);
  sr_stream_window_kernel<<<grid, 256, 0, hsv::as_stream(stream)>>>(x_new, n_new, start, end, hist, state, win,
                                                                    valid_len_in, valid_len_out, origin, plan, N, H, W,
                                                                    up, down, lookahead);
  return hsv::check_launch("sr_stream_window");
}

extern "C" int hsv_sr_stream_emit(const float *y, const float *win, const int64_t *origin, const int64_t *plan,
                                  float *hist, int64_t *state, float *out, int32_t *n_out, int S, int H, int W,
                                  int64_t Lout, int cap, void *stream) {
  if (S == 0) return HSV_OK;
  HSV_REQUIRE(y && win && origin && plan && hist && state && out && n_out, "sr_stream_emit: null pointer");
  HSV_REQUIRE(S > 0 && S <= 65535 && H > 0 && W > H && Lout > 0 && cap > 0, "sr_stream_emit: bad shape");
  const int span = cap > H ? cap : H;
  dim3 grid((unsigned)((span + 255) / 256), (unsigned)S);
  sr_stream_emit_kernel<<<grid, 256, 0, hsv::as_stream(stream)>>>(y, win, origin, plan, hist, state, out, n_out, H, W,
                                                                  Lout, cap);
  return hsv::check_launch("sr_stream_emit");
}
