"""Voice-conversion job where every request has its own seed, noise_scale and denoise_ratio: one batch-1 call per
request vs per-item batches with the seeds and controls passed as device tensors.

    python tools/bench_vc_controls.py [--utts 128] [--tmin 100] [--tmax 1000] [--pmin 100] [--pmax 300]
                                      [--max-batch 16] [--frame-multiple 50] [--prompt-multiple 50]
                                      [--parallel-blocks 1] [--reps 3]

The job is tools/bench_synth_ragged.py's (torch generator seeded 1111: lengths, prompt lengths, then per request a
noise_scale uniform in [0.2, 0.8], a denoise_ratio uniform in [0, 1] and a seed in [0, 2^63 - 1); inputs
``synthetic.synthesizer_inputs(T_i, Tm_i, seed=1111 + i)``, weights ``synthetic.synthesizer_sd(1234)``).

(a) what a caller can do without per-item controls: one batch-1 ``voice_conversion_noise_control(..., per_item=True)``
    per request through ``CudaGraphRunner(capture_after=2)`` with that request's Python-float controls and
    ``eps = ops.seeded_normal(seed)``.  The floats are baked into each captured graph, so the runner is keyed on them
    too; each timed pass uses a fresh runner (the untimed pass loads modules and folds weights).
(b) ``runtime.ragged_prompt_batches`` micro-batches with ``per_item=True`` and ``seed=`` / ``noise_scale=`` /
    ``denoise_ratio=`` as [B] device tensors through ONE ``CudaGraphRunner``: the untimed pass captures one graph per
    padded (B, T, Tm), the timed passes replay it for whatever controls the batch carries.

Every waveform is compared between (a) and (b) with ``torch.equal``.  Prints one JSON line with the card's name and
power limit.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import megatts2_hierspeechpp_b200 as hsv  # noqa: E402
from megatts2_hierspeechpp_b200 import ops, synthetic  # noqa: E402
from megatts2_hierspeechpp_b200.runtime import CudaGraphRunner, ragged_prompt_batches  # noqa: E402
from bench_ragged import power_limit_w, timed  # noqa: E402

HOP, SR = 320, 16000


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--utts", type=int, default=128)
    ap.add_argument("--tmin", type=int, default=100)
    ap.add_argument("--tmax", type=int, default=1000)
    ap.add_argument("--pmin", type=int, default=100)
    ap.add_argument("--pmax", type=int, default=300)
    ap.add_argument("--max-batch", type=int, default=16)
    ap.add_argument("--frame-multiple", type=int, default=50)
    ap.add_argument("--prompt-multiple", type=int, default=50)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--parallel-blocks", type=int, default=1, help="multi-stream mode (bench.py's default: 1)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_vc_controls.py needs a CUDA device")
    dev = torch.device("cuda:0")

    gen = torch.Generator().manual_seed(1111)
    n = args.utts
    lengths = torch.randint(args.tmin, args.tmax + 1, (n,), generator=gen).tolist()
    prompts = torch.randint(args.pmin, args.pmax + 1, (n,), generator=gen).tolist()
    noise_scale = (torch.rand(n, generator=gen) * 0.6 + 0.2).tolist()             # exact fp32 values
    denoise = torch.rand(n, generator=gen, dtype=torch.float64).tolist()
    seeds = torch.randint(0, (1 << 63) - 1, (n,), generator=gen, dtype=torch.int64).tolist()
    ins = [[t.to(dev) for t in synthetic.synthesizer_inputs(T, Tm, seed=1111 + i)]
           for i, (T, Tm) in enumerate(zip(lengths, prompts))]          # w2v [1,1024,T], f0 [1,1,4T], mel [2,80,Tm]
    model = hsv.HierSpeechSynthesizer()
    model.load_state_dict(synthetic.synthesizer_sd(1234), strict=True)
    model.to(dev).eval()
    for m in model.modules():
        if hasattr(m, "parallel_blocks"):
            m.parallel_blocks = bool(args.parallel_blocks)
    a_len = [(torch.tensor([T], dtype=torch.int32, device=dev), torch.tensor([Tm, Tm], dtype=torch.int32, device=dev))
             for T, Tm in zip(lengths, prompts)]
    a_seed = [torch.tensor([s], dtype=torch.int64, device=dev) for s in seeds]

    # (a) one batch-1 call per request; its scalars are part of what a graph bakes in, so they key the runner
    class PerControls:
        def __init__(self):
            self.runners = {}

        def __call__(self, i, *xs):
            key = (noise_scale[i], denoise[i])
            if key not in self.runners:
                def one(w2v, f0, mel, ln, ln2, seed, ns=key[0], r=key[1]):
                    return model.voice_conversion_noise_control(w2v, ln, mel, ln2, f0, ns, False, r, per_item=True,
                                                                eps=ops.seeded_normal(seed, 192, w2v.shape[-1]))
                self.runners[key] = CudaGraphRunner(one, capture_after=2)
            return self.runners[key](*xs)

        @property
        def captures(self):
            return sum(r.captures for r in self.runners.values())

    def run_a(runner):
        return {i: runner(i, w2v, f0, mel, ln, ln2, a_seed[i]).clone()
                for i, ((w2v, f0, mel), (ln, ln2)) in enumerate(zip(ins, a_len))}

    # (b) per-item micro-batches, seeds and controls as device tensors
    batches = ragged_prompt_batches(range(n), lengths, prompts, args.max_batch, args.frame_multiple,
                                    args.prompt_multiple)
    b_in = []
    for ids, Tp, Tmp in batches:
        B = len(ids)
        src = torch.zeros(B, 1024, Tp, device=dev)
        f0 = torch.zeros(B, 1, 4 * Tp, device=dev)
        mel = torch.zeros(2 * B, 80, Tmp, device=dev)
        for j, i in enumerate(ids):
            T, Tm = lengths[i], prompts[i]
            src[j, :, :T] = ins[i][0][0]
            f0[j, :, :4 * T] = ins[i][1][0]
            mel[j, :, :Tm] = ins[i][2][0]
            mel[B + j, :, :Tm] = ins[i][2][1]
        vl = torch.tensor([lengths[i] for i in ids], dtype=torch.int32, device=dev)
        tl = torch.tensor([prompts[i] for i in ids] * 2, dtype=torch.int32, device=dev)
        sd = torch.tensor([seeds[i] for i in ids], dtype=torch.int64, device=dev)
        ns = torch.tensor([noise_scale[i] for i in ids], dtype=torch.float32, device=dev)
        r = torch.tensor([denoise[i] for i in ids], dtype=torch.float64, device=dev)
        b_in.append((src, f0, mel, vl, tl, sd, ns, r))

    def batch(src, f0, mel, vl, tl, sd, ns, r):
        return model.voice_conversion_noise_control(src, vl, mel, tl, f0, ns, False, r, per_item=True, seed=sd)

    runner_b = CudaGraphRunner(batch)

    def run_b():
        res = {}
        for (ids, _, _), xs in zip(batches, b_in):
            w = runner_b(*xs)
            for j, i in enumerate(ids):
                res[i] = w[j, :, :lengths[i] * HOP].clone()
        return res

    with torch.no_grad():
        run_a(PerControls())                                     # untimed
        torch.cuda.synchronize()
        runners_a = []

        def fresh_a():
            runners_a.append(PerControls())
            return run_a(runners_a[-1])

        ms_a, out_a = timed(fresh_a, args.reps)
        run_b()                                                  # untimed: captures
        torch.cuda.synchronize()
        cap_b0 = runner_b.captures
        ms_b, out_b = timed(run_b, args.reps)
        cap_b_timed = runner_b.captures - cap_b0
        tails_zero = True
        for (ids, _, _), xs in zip(batches, b_in):
            w = runner_b(*xs)
            tails_zero &= all(bool((w[j, :, lengths[i] * HOP:] == 0).all()) for j, i in enumerate(ids))

    mismatches = sum(0 if torch.equal(out_a[i][0], out_b[i]) else 1 for i in range(n))
    audio_s = sum(lengths) * HOP / SR
    padded = sum(len(ids) * Tp for ids, Tp, _ in batches)

    def summary(ms):
        med = statistics.median(ms)
        return {"ms_per_job": round(med, 2), "ms_all": [round(m, 2) for m in ms],
                "audio_s_per_s": round(audio_s / (med / 1e3), 1)}

    line = {
        "tool": "bench_vc_controls",
        "device": torch.cuda.get_device_name(0),
        "power_limit_w": power_limit_w(),
        "job": {"utterances": n, "frames": [args.tmin, args.tmax], "prompt_frames": [args.pmin, args.pmax],
                "seed": 1111, "noise_scale": [0.2, 0.8], "denoise_ratio": [0.0, 1.0], "audio_s": round(audio_s, 2),
                "max_batch": args.max_batch, "parallel_blocks": bool(args.parallel_blocks)},
        "a_batch1": {**summary(ms_a), "calls": n, "captures_timed": sum(r.captures for r in runners_a)},
        "b_per_item": {**summary(ms_b), "micro_batches": len(batches), "frame_multiple": args.frame_multiple,
                       "prompt_multiple": args.prompt_multiple,
                       "graph_shapes": len({(len(ids), Tp, Tmp) for ids, Tp, Tmp in batches}),
                       "graphs_captured": runner_b.captures, "captures_timed": cap_b_timed,
                       "padded_frame_fraction": round(1 - sum(lengths) / padded, 4), "tails_zero": tails_zero},
        "speedup_b_over_a": round(statistics.median(ms_a) / statistics.median(ms_b), 3),
        "mismatches": mismatches,
    }
    print(json.dumps(line), flush=True)
    if mismatches or cap_b_timed or not tails_zero:
        sys.exit(1)


if __name__ == "__main__":
    main()
