"""Variable-length text-to-speech job on one GPU: one batch-1 call per utterance vs per-item batches.

    python tools/bench_tts_ragged.py [--utts 128] [--tmin 100] [--tmax 1000] [--pmin 100] [--pmax 300]
                                     [--max-batch 16] [--frame-multiple 50] [--prompt-multiple 50]
                                     [--parallel-blocks 1] [--reps 3] [--profile DIR]

The job: ``--utts`` utterances with T uniform in [tmin, tmax] frames and a prompt of Tm uniform in [pmin, pmax] frames
(torch generator seeded 1111).  Utterance i's flow output z, its style vector g (``synthetic.ttv_tail_inputs(1, T_i,
seed=1111 + i)``) and its prompt pair (``synthetic.synthesizer_inputs(T_i, Tm_i, seed=1111 + i)``, prompt and denoised
twin of the same length) run through the text-to-speech chain of inference.py:158-167: ``TTVTail`` (weights
``synthetic.ttv_tail_sd(3456)``) -> ``voice_conversion_noise_control(w2v, ..., pitch, noise_scale=0.333,
denoise_ratio=0.3)`` (weights ``synthetic.synthesizer_sd(1234)``).  Utterance i's noise is what the batch-1 call draws
after ``torch.manual_seed(1111 + i)`` (its second draw): (a) reseeds before each call, (b) passes those draws as
explicit per-item ``eps``.

(a) one batch-1 call per utterance through ``CudaGraphRunner(capture_after=2)``, the setting INTEGRATION.md recommends
    for variable lengths.  Each timed pass uses a fresh runner, as a stream of one-off lengths would see it (the untimed
    pass loads modules and folds weights).
(b) ``runtime.ragged_prompt_batches`` micro-batches, each one captured graph of the whole chain:
    ``TTVTail(..., lengths=)`` -> ``voice_conversion_noise_control(..., per_item=True, eps=)``.  The untimed pass
    captures one graph per padded (B, T, Tm), the timed passes replay.

Batch inputs are assembled on the device before timing; per-utterance outputs are sliced and cloned inside it.  Every
waveform is compared between (a) and (b) with ``torch.equal``.  Prints one JSON line.  ``--profile DIR``: instead, one
``torch.profiler`` pass of (b) (after the untimed one) with a kernel table and a trace written under DIR.
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
from megatts2_hierspeechpp_b200 import synthetic  # noqa: E402
from megatts2_hierspeechpp_b200.runtime import CudaGraphRunner, ragged_prompt_batches  # noqa: E402
from bench_ragged import power_limit_w, timed  # noqa: E402

HOP, SR = 320, 16000
NOISE_SCALE, DENOISE = 0.333, 0.3


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
    ap.add_argument("--profile", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_tts_ragged.py needs a CUDA device")
    dev = torch.device("cuda:0")

    gen = torch.Generator().manual_seed(1111)
    lengths = torch.randint(args.tmin, args.tmax + 1, (args.utts,), generator=gen).tolist()
    prompts = torch.randint(args.pmin, args.pmax + 1, (args.utts,), generator=gen).tolist()
    ins = []                                                     # z [1,256,T], g [1,256,1], mel [2,80,Tm]
    for i, (T, Tm) in enumerate(zip(lengths, prompts)):
        z, _, g = synthetic.ttv_tail_inputs(1, T, seed=1111 + i)
        ins.append((z.to(dev), g.to(dev), synthetic.synthesizer_inputs(T, Tm, seed=1111 + i)[2].to(dev)))
    eps = []
    for i, T in enumerate(lengths):
        torch.manual_seed(1111 + i)
        eps.append([torch.randn(1, 192, T, device=dev) for _ in range(2)][1])
    tail = hsv.TTVTail()
    tail.load_state_dict(synthetic.ttv_tail_sd(3456), strict=True)
    tail.to(dev).eval()
    syn = hsv.HierSpeechSynthesizer()
    syn.load_state_dict(synthetic.synthesizer_sd(1234), strict=True)
    syn.to(dev).eval()
    for m in list(tail.modules()) + list(syn.modules()):
        if hasattr(m, "parallel_blocks"):
            m.parallel_blocks = bool(args.parallel_blocks)
    a_in = [(torch.ones(1, 1, T, device=dev), torch.LongTensor([T]).to(dev), torch.LongTensor([Tm, Tm]).to(dev))
            for T, Tm in zip(lengths, prompts)]

    # (a) one batch-1 call per utterance
    def run_a(runner):
        res = {}
        for i, ((z, g, mel), (mask, ln, ln2)) in enumerate(zip(ins, a_in)):
            torch.manual_seed(1111 + i)
            res[i] = runner(z, mask, g, mel, ln, ln2).clone()
        return res

    def one(z, mask, g, mel, ln, ln2):
        w2v, pitch = tail(z, mask, g)
        return syn.voice_conversion_noise_control(w2v, ln, mel, ln2, pitch, NOISE_SCALE, False, DENOISE)

    # (b) per-item micro-batches
    batches = ragged_prompt_batches(range(args.utts), lengths, prompts, args.max_batch, args.frame_multiple,
                                    args.prompt_multiple)
    b_in = []
    for ids, Tp, Tmp in batches:
        B = len(ids)
        z = torch.zeros(B, 256, Tp, device=dev)
        g = torch.cat([ins[i][1] for i in ids])
        mel = torch.zeros(2 * B, 80, Tmp, device=dev)
        ep = torch.zeros(B, 192, Tp, device=dev)
        for j, i in enumerate(ids):
            T, Tm = lengths[i], prompts[i]
            z[j, :, :T] = ins[i][0][0]
            mel[j, :, :Tm] = ins[i][2][0]
            mel[B + j, :, :Tm] = ins[i][2][1]
            ep[j, :, :T] = eps[i][0]
        vl = torch.tensor([lengths[i] for i in ids], dtype=torch.int32, device=dev)
        tl = torch.tensor([prompts[i] for i in ids] * 2, dtype=torch.int32, device=dev)
        b_in.append((z, g, mel, vl, tl, ep))

    def batch(z, g, mel, vl, tl, ep):
        w2v, pitch = tail(z, None, g, lengths=vl)
        return syn.voice_conversion_noise_control(w2v, vl, mel, tl, pitch, NOISE_SCALE, False, DENOISE, per_item=True,
                                                  eps=ep)

    runner_b = CudaGraphRunner(batch)

    def run_b():
        res = {}
        for (ids, _, _), xs in zip(batches, b_in):
            w = runner_b(*xs)
            for j, i in enumerate(ids):
                res[i] = w[j, :, :lengths[i] * HOP].clone()
        return res

    with torch.no_grad():
        if args.profile:
            run_b()
            torch.cuda.synchronize()
            os.makedirs(args.profile, exist_ok=True)
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
                run_b()
                torch.cuda.synchronize()
            table = prof.key_averages().table(sort_by="cuda_time_total", row_limit=40)
            with open(os.path.join(args.profile, "tts_ragged_kernels.txt"), "w") as f:
                f.write(table)
            prof.export_chrome_trace(os.path.join(args.profile, "tts_ragged.pt.trace.json"))
            print(table)
            return
        run_a(CudaGraphRunner(one, capture_after=2))            # untimed
        torch.cuda.synchronize()
        runners_a = []

        def fresh_a():
            runners_a.append(CudaGraphRunner(one, capture_after=2))
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

    mismatches = sum(0 if torch.equal(out_a[i][0], out_b[i]) else 1 for i in range(args.utts))
    audio_s = sum(lengths) * HOP / SR
    padded = sum(len(ids) * Tp for ids, Tp, _ in batches)

    def summary(ms):
        med = statistics.median(ms)
        return {"ms_per_job": round(med, 2), "ms_all": [round(m, 2) for m in ms],
                "audio_s_per_s": round(audio_s / (med / 1e3), 1)}

    line = {
        "tool": "bench_tts_ragged",
        "device": torch.cuda.get_device_name(0),
        "power_limit_w": power_limit_w(),
        "job": {"utterances": args.utts, "frames": [args.tmin, args.tmax], "prompt_frames": [args.pmin, args.pmax],
                "seed": 1111, "audio_s": round(audio_s, 2), "max_batch": args.max_batch,
                "parallel_blocks": bool(args.parallel_blocks)},
        "a_batch1": {**summary(ms_a), "calls": args.utts, "captures_timed": sum(r.captures for r in runners_a)},
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
