"""SpeechSR48 on a job of mixed-rate int16 requests: where the resampling to 16 kHz runs, and what it costs.

Job: ``--requests`` (256) requests, rates drawn from {16, 22.05, 24, 32, 44.1, 48} kHz, lengths uniform in 2-15 s, int16
audio (tones + noise) in pinned host memory, fixed seed.  Every arm cuts the same micro-batches
(``resample.audio_batches``: by 16 kHz length, at most ``--max-batch`` each) and runs SpeechSR48 with ragged ``lengths=``
through one ``CudaGraphRunner``; they differ in the step before it:

  (a) torchaudio ``resample(..., "kaiser_window")`` per request on the CPU (all host threads), H2D of fp32 16 kHz audio;
  (b) H2D of int16, torchaudio on the GPU per request (eager), the results packed into the padded batch;
  (c) ``hsv.SpeechSRAudio``: H2D of the padded int16 batch, one graph per micro-batch (resampler + SpeechSR).

Reports per arm the job time (host clock around work that ends in a device synchronise; median of ``--reps`` timed
passes after an untimed one that captures every graph), useful audio-seconds per second and host CPU time (process
time, all threads); the largest difference between the outputs of (a) and (c) (and (b) and (c)); and, in a separate pass,
the resampler kernel alone by CUDA events per source rate with its FLOPs (2 K per output) and bytes from shapes.  The card
name and power limit are read in the same run.

    python tools/bench_sr_any_rate.py [--requests 256] [--max-batch 16] [--reps 3] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

RATES = (16000, 22050, 24000, 32000, 44100, 48000)


def _card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                            "-i", "0"], capture_output=True, text=True, timeout=30)
        power, clock = [v.strip() for v in q.stdout.strip().split(",")]
    except (OSError, subprocess.SubprocessError, ValueError):
        power, clock = "unknown", "unknown"
    return name, power, clock


class _RaggedSR(torch.nn.Module):
    """``sr(x, lengths=lengths)`` with the lengths positional, as ``CudaGraphRunner`` passes graph inputs."""

    def __init__(self, sr):
        super().__init__()
        self.sr = sr

    def forward(self, x, lengths):
        return self.sr(x, lengths=lengths)


def make_job(n, seed):
    rng = np.random.default_rng(seed)
    rates = [int(r) for r in rng.choice(RATES, n)]
    lengths = [int(rng.uniform(2.0, 15.0) * r) for r in rates]
    audio = []
    for r, L in zip(rates, lengths):
        t = np.arange(L) / r
        x = 0.3 * np.sin(2 * np.pi * rng.uniform(100, 400) * t) + 0.1 * np.sin(2 * np.pi * rng.uniform(2e3, 7e3) * t)
        x += 0.03 * rng.standard_normal(L)
        audio.append(torch.from_numpy(np.round(x * 32767).clip(-32768, 32767).astype(np.int16)).pin_memory())
    return rates, lengths, audio


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--requests", type=int, default=256)
    ap.add_argument("--max-batch", type=int, default=16)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--kernel-iters", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_sr_any_rate: needs a CUDA device")
    import torchaudio
    import megatts2_hierspeechpp_b200 as hsv
    from megatts2_hierspeechpp_b200 import resample as RS
    from conftest import golden_sd
    warnings.filterwarnings("ignore", message=".*resampling method name is being deprecated.*")
    dev = torch.device("cuda")
    card, power, clock = _card()
    sr = hsv.SpeechSR48(100, 40, **hsv.SR_CFG)
    sr.load_state_dict(golden_sd("speechsr48_state.npz"), strict=True)
    sr = sr.to(dev).eval()
    rates, lengths, audio = make_job(a.requests, a.seed)
    n16 = RS.resampled_lengths(rates, lengths)
    batches = RS.audio_batches(rates, lengths, a.max_batch)
    audio_s = sum(n / 16000 for n in n16)
    sr_runner = hsv.CudaGraphRunner(_RaggedSR(sr))
    chain = hsv.SpeechSRAudio(sr)
    chain_runner = hsv.CudaGraphRunner(chain)

    def sr_batches(wav16):
        """The shared SpeechSR step: wav16[i] = 16 kHz fp32 audio of request i (host or device)."""
        outs = {}
        for ids, _, out_len in batches:
            pinned = wav16[ids[0]].device.type == "cpu"
            buf = torch.zeros(len(ids), 1, out_len, pin_memory=pinned,
                              device="cpu" if pinned else dev)
            for k, i in enumerate(ids):
                buf[k, 0, :wav16[i].numel()] = wav16[i]
            x = buf.to(dev, non_blocking=True)
            ln = torch.tensor([n16[i] for i in ids], dtype=torch.int32).to(dev)
            y = sr_runner(x, ln)
            for k, i in enumerate(ids):
                outs[i] = y[k, 0, :3 * n16[i]].clone()
        return outs

    def arm_a():
        wav = [torchaudio.functional.resample(x.float() / 32768.0, r, 16000, resampling_method="kaiser_window")
               if r != 16000 else x.float() / 32768.0 for x, r in zip(audio, rates)]
        return sr_batches(wav)

    def arm_b():
        wav = []
        for x, r in zip(audio, rates):
            xg = x.to(dev, non_blocking=True).float() / 32768.0
            wav.append(torchaudio.functional.resample(xg, r, 16000, resampling_method="kaiser_window")
                       if r != 16000 else xg)
        return sr_batches(wav)

    def arm_c():
        outs = {}
        for ids, T, out_len in batches:
            buf = torch.zeros(len(ids), T, dtype=torch.int16, pin_memory=True)
            for k, i in enumerate(ids):
                buf[k, :lengths[i]] = audio[i]
            x = buf.to(dev, non_blocking=True)
            rl = torch.tensor([[rates[i] for i in ids], [lengths[i] for i in ids]], dtype=torch.int32).to(dev)
            y, _ = chain_runner(x, rl[0], rl[1], out_len=out_len)
            for k, i in enumerate(ids):
                outs[i] = y[k, 0, :3 * n16[i]].clone()
        return outs

    results, outputs = {}, {}
    for name, fn in (("a_torchaudio_cpu", arm_a), ("b_torchaudio_gpu", arm_b), ("c_speechsr_audio", arm_c)):
        with torch.no_grad():
            outputs[name] = fn()                   # untimed: captures every graph, warms every path
            torch.cuda.synchronize()
            ms, cpu = [], []
            for _ in range(a.reps):
                c0, t0 = time.process_time(), time.perf_counter()
                fn()
                torch.cuda.synchronize()
                ms.append(1000 * (time.perf_counter() - t0))
                cpu.append(1000 * (time.process_time() - c0))
        results[name] = {"job_ms": round(statistics.median(ms), 2), "job_ms_all": [round(v, 2) for v in ms],
                         "audio_s_per_s": round(audio_s / (statistics.median(ms) / 1000), 1),
                         "host_cpu_ms": round(statistics.median(cpu), 1)}
        print(json.dumps({"arm": name, **results[name]}), flush=True)

    def max_diff(p, q):
        return max(float((outputs[p][i] - outputs[q][i]).abs().max()) for i in range(a.requests))

    diffs = {"a_vs_c_max_abs": max_diff("a_torchaudio_cpu", "c_speechsr_audio"),
             "b_vs_c_max_abs": max_diff("b_torchaudio_gpu", "c_speechsr_audio")}
    print(json.dumps(diffs), flush=True)

    # the resampler kernel alone: 16 items of 10 s per source rate, CUDA events around --kernel-iters launches
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    kern = []
    for r in RATES[1:]:
        m = RS.Resample((r,)).to(dev)
        o, n, width = RS.ratio(r, 16000)
        K = 2 * width + o
        B, L = 16, 10 * r
        x = torch.randint(-30000, 30000, (B, L), dtype=torch.int16, device=dev)
        rt = torch.full((B,), r, dtype=torch.int32, device=dev)
        lt = torch.full((B,), L, dtype=torch.int32, device=dev)
        nout = RS.resampled_lengths([r], [L])[0]
        for _ in range(3):
            m(x, rt, lt, out_len=nout)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(a.kernel_iters):
            m(x, rt, lt, out_len=nout)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / a.kernel_iters
        flops = 2.0 * K * nout * B
        nbytes = 2.0 * B * L + 4.0 * B * nout + 4.0 * K * n        # int16 in, fp32 out, the table once
        row = {"rate": r, "K": K, "B": B, "seconds": 10, "kernel_ms": round(ms, 4),
               "gflop_s": round(flops / ms / 1e6, 1), "gb_s": round(nbytes / ms / 1e6, 1)}
        if clock != "unknown":
            hz = float(clock) * 1e6
            # each FMA loads one table word (L1) and one staged sample (shared memory): two 128-byte warp loads per 32
            # FMAs, so the load pipe (128 B / clk / SM) allows 16 FMA / clk / SM against 128 for the FMA pipe
            row["fma_pipe_min_ms"] = round(flops / (sms * 128 * 2 * hz) * 1e3, 4)
            row["load_pipe_min_ms"] = round(flops / (sms * 16 * 2 * hz) * 1e3, 4)
            row["hbm_min_ms"] = round(nbytes / 7.7e12 * 1e3, 4)
            row["bound"] = max(("fma_pipe", row["fma_pipe_min_ms"]), ("load_pipe", row["load_pipe_min_ms"]),
                               ("hbm", row["hbm_min_ms"]), key=lambda kv: kv[1])[0]
        kern.append(row)
        print(json.dumps(row), flush=True)

    summary = {"card": card, "power_limit_w": power, "max_sm_clock_mhz": clock, "host_threads": torch.get_num_threads(),
               "host_cpus": os.cpu_count(), "requests": a.requests, "micro_batches": len(batches),
               "audio_s_16k": round(audio_s, 1), "arms": results, **diffs, "kernel": kern}
    print(json.dumps({k: v for k, v in summary.items() if k != "kernel"}), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(summary, f, indent=1)


if __name__ == "__main__":
    main()
