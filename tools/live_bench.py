"""Live multi-stream front-end benchmark (LiveStreams / kws_live_push), next to the existing window paths.

    python tools/live_bench.py [--streams 1,148,1024,8192] [--push-ms 10,100] [--dtypes float32,int16]
                               [--models res15,cnn-trad-fpool3] [--seconds 2] [--reps 3] [--profile-calls 50]
                               [--out FILE]

For every S, push length and sample type (1 s windows, 10 ms shift) it reports, per push of S x n samples:
  live_ms       front-end alone: LiveStreams.push into a preallocated buffer (the four launches of kws_live_push)
  <model>_ms    LiveStreams.push(chunk, model): front-end + the model on the S K new windows (bf16)
  batch_ms      the existing path on the same windows: compute_mfccs_batch on the S K materialised windows
  stream_ms     the existing path on the same windows: compute_mfccs_stream, one call per stream, K windows each
  windows_per_s S K / live_ms
  h2d_B_per_window  host->device bytes per window: the push's new samples (live) against a whole window (batch)
  live_kernel_ms, batch_kernel_ms  the same calls' kernel time alone: the sum of their kernels' durations per call,
                from torch.profiler (CUDA activity only) over a separate loop of --profile-calls calls
  live_regime   "host" when live_kernel_ms < 0.7 live_ms (the GPU waits for the Python loop: live_ms is the host's
                launch rate, not front-end time), else "device"
Times (*_ms) are device times from CUDA events around a loop of calls that runs for --seconds (after warm-up), median
over --reps repetitions, with the spread (max - min) / median.  Events around a loop include the gaps between
launches; the kernel times do not.  Inputs are device resident.  The device name and power limit are read (nvidia-smi,
query only) and printed in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import honk2_b200  # noqa: E402
from honk2_b200 import AudioProcessor, LiveStreams  # noqa: E402

W, H = 16000, 160


def device_line():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "nvidia-smi: n/a"
    except (OSError, subprocess.TimeoutExpired):
        return "nvidia-smi: n/a"


def timed(fn, seconds, reps):
    """Median / spread of the per-call device time (ms) of fn over loops that run for about `seconds`."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(10):
        fn()
    torch.cuda.synchronize()
    n = max(10, int(seconds / max((time.perf_counter() - t) / 10, 1e-6)))
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b) / n)
    med = float(np.median(ms))
    return med, (max(ms) - min(ms)) / med, n


def kernel_ms(fn, calls):
    """Summed duration of the kernels fn launches, per call (torch.profiler, CUDA activity only)."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    us = sum(e.time_range.elapsed_us() for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)
    if us == 0:   # builds that attach kernels to their launching CPU events only
        us = sum(getattr(e, "self_device_time_total", 0) for e in prof.key_averages())
    return us / calls / 1000.0


def main():
    ap_ = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap_.add_argument("--streams", default="1,148,1024,8192")
    ap_.add_argument("--push-ms", default="10,100")
    ap_.add_argument("--dtypes", default="float32,int16")
    ap_.add_argument("--models", default="res15,cnn-trad-fpool3", help="bf16 models run after the front-end ('' = none)")
    ap_.add_argument("--seconds", type=float, default=2.0)
    ap_.add_argument("--reps", type=int, default=3)
    ap_.add_argument("--profile-calls", type=int, default=50)
    ap_.add_argument("--out", default=None, help="also write the JSON lines here")
    args = ap_.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("live_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    header = {"device": device_line(), "torch_device": torch.cuda.get_device_name(dev), "window": W, "shift": H,
              "seconds": args.seconds, "reps": args.reps}
    print(json.dumps(header), flush=True)
    lines = [header]
    ap = AudioProcessor()
    models = {}
    for name in [m for m in args.models.split(",") if m]:
        models[name] = honk2_b200.build_model(name, precision="bf16").to(dev)
    gen = torch.Generator(device=dev).manual_seed(0)
    for S in [int(s) for s in args.streams.split(",")]:
        for push_ms in [int(p) for p in args.push_ms.split(",")]:
            n = 16 * push_ms
            K = n // H
            for dtype in args.dtypes.split(","):
                pcm16 = dtype == "int16"
                x = torch.rand((S, n), generator=gen, device=dev) * 2 - 1
                chunk = (x * 32767).to(torch.int16) if pcm16 else x
                live = LiveStreams(ap, S, W, H, max_push=n, device=dev)
                out = torch.empty((S, K, 101, 40), device=dev)
                for _ in range(W // n + 2):          # past the warm-up: every slot valid
                    live.push(chunk, out=out)
                row = {"S": S, "push_ms": push_ms, "n": n, "K": K, "dtype": dtype, "windows_per_push": S * K,
                       "h2d_B_per_window": {"live": H * chunk.element_size(), "batch": W * chunk.element_size()}}
                row["live_ms"], row["live_spread"], row["live_pushes"] = timed(
                    lambda: live.push(chunk, out=out), args.seconds, args.reps)
                row["windows_per_s"] = S * K / (row["live_ms"] * 1e-3)
                row["live_kernel_ms"] = kernel_ms(lambda: live.push(chunk, out=out), args.profile_calls)
                row["live_regime"] = "host" if row["live_kernel_ms"] < 0.7 * row["live_ms"] else "device"
                with torch.no_grad():
                    for name, m in models.items():
                        ms, spread, _ = timed(lambda: live.push(chunk, m, out=out), args.seconds, args.reps)
                        row[f"{name}_ms"], row[f"{name}_spread"] = ms, spread
                        row[f"{name}_windows_per_s"] = S * K / (ms * 1e-3)
                # the existing paths on the same S K windows
                seg = (torch.rand((S, W + n), generator=gen, device=dev) * 2 - 1)
                seg = (seg * 32767).to(torch.int16) if pcm16 else seg
                wins = seg.unfold(1, W, H)[:, :K].reshape(S * K, W).contiguous()   # the K windows of each row
                bout = torch.empty((S * K, 101, 40), device=dev)
                row["batch_ms"], row["batch_spread"], _ = timed(lambda: ap.compute_mfccs_batch(wins, out=bout),
                                                                args.seconds, args.reps)
                row["batch_kernel_ms"] = kernel_ms(lambda: ap.compute_mfccs_batch(wins, out=bout), args.profile_calls)
                streams = [seg[s] for s in range(S)]   # W + n samples: exactly K windows each
                sout = bout.view(S, K, 101, 40)

                def per_stream():
                    for s in range(S):
                        ap.compute_mfccs_stream(streams[s], W, H, out=sout[s])
                row["stream_ms"], row["stream_spread"], _ = timed(per_stream, args.seconds, args.reps)
                print(json.dumps(row), flush=True)
                lines.append(row)
                del live, out, wins, bout, seg, streams, sout
                torch.cuda.empty_cache()
    print(json.dumps({"device": device_line()}), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            for ln in lines:
                f.write(json.dumps(ln) + "\n")


if __name__ == "__main__":
    main()
