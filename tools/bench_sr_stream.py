"""Steady-state step time of streaming SpeechSR (``SpeechSRStream``): S concurrent 16 kHz streams fed 20 ms (320-sample)
chunks, one graph replay per step, timed with CUDA events after a warm-up.

Reports, per rate and S: the time per step, the streams sustained in real time (S x 20 ms / step time) and the recompute
overhead against offline SpeechSR on the same audio, from shapes: every step runs the stack over each slot's window of
history + chunk input samples, the offline call over the chunk alone.

    python tools/bench_sr_stream.py [--slots 1 64 256 1024] [--steps 200] [--warmup 20] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power = q.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def bench(hsv, which, S, N, steps, warmup):
    from conftest import golden_sd
    m = (hsv.SpeechSR24 if which == 24 else hsv.SpeechSR48)(100, 40, **hsv.SR_CFG)
    m.load_state_dict(golden_sd(f"speechsr{which}_state.npz"), strict=True)
    m = m.to("cuda").eval()
    st = hsv.SpeechSRStream(m, S, N)
    dev = torch.device("cuda")
    gen = torch.Generator(device=dev).manual_seed(S + which)
    xs = [torch.randn(S, N, device=dev, generator=gen) * 0.2 for _ in range(8)]
    n_new = torch.full((S,), N, dtype=torch.int32, device=dev)
    one = torch.ones(S, dtype=torch.int32, device=dev)
    zero = torch.zeros(S, dtype=torch.int32, device=dev)
    st.step(xs[0], n_new, one, zero)                       # every slot opens a stream
    for i in range(warmup):
        st.step(xs[i % 8], n_new, zero, zero)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for i in range(steps):
        st.step(xs[i % 8], n_new, zero, zero)
    t1.record()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / steps
    up, down = st.ratio
    chunk_ms = 1000.0 * N / 16000
    return {
        "rate_khz": which, "slots": S, "chunk": N, "history": st.history, "lookahead_out": st.lookahead,
        "step_ms": round(ms, 4), "realtime_streams": round(S * chunk_ms / ms, 1),
        # output samples the stack computes per step over those it emits (offline computes exactly the emitted ones)
        "recompute_overhead": round((st.history + N) / N, 3),
        "captures": st.captures,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--slots", type=int, nargs="+", default=[1, 64, 256, 1024])
    ap.add_argument("--chunk", type=int, default=320)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_sr_stream: needs a CUDA device")
    import megatts2_hierspeechpp_b200 as hsv
    card, power = _card()
    rows = []
    for which in (48, 24):
        for S in a.slots:
            r = bench(hsv, which, S, a.chunk, a.steps, a.warmup)
            r.update(card=card, power_limit=power)
            print(json.dumps(r), flush=True)
            rows.append(r)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
