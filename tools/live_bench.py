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

    python tools/live_bench.py --ragged [--streams 148,1024,8192] [--models res15,cnn-trad-fpool3]
                                        [--model-streams 8192] [--seconds 1] [--reps 3] [--out FILE]

runs the ragged-push leg instead (LiveStreams.push_ragged against LiveStreams.push; 1 s windows, 10 ms shift).  The two
paths run on two states fed the same audio and are timed alternately in the same loop of repetitions:
  aligned   every stream brings 160 samples, float32 and int16: ragged_ms / uniform_ms per push and their kernel time
            (torch.profiler, all device activity of a call, the ragged push's small host->device copy included)
  jitter    per push and stream a length drawn from {0, 160, 320, 1024} with probabilities (0.5, 0.3, 0.13, 0.07), mean
            161 samples (float32): ragged_ms against a uniform 160-sample push, and the windows per push
  model     push_ragged(x, model) against push(x, model), bf16, at --model-streams streams: during the warm-up of fresh
            streams (the 99 pushes of 160 samples before the first window completes: the uniform push runs the model on
            S all-zero slots, the ragged push on none) and in the steady state (both run it on S windows)

    python tools/live_bench.py --cnn [--streams 148,1024,8192] [--push-ms 10,100] [--dtypes float32,int16]
                                     [--kernel-only] [--seconds 2] [--reps 3] [--profile-calls 20] [--out FILE]

runs the live CNN leg instead: LiveCNN.push(chunk) against LiveStreams.push(chunk, model) on cnn-trad-fpool3 in bf16
(1 s windows, 10 ms shift), two states fed the same chunk past the warm-up, timed alternately in the same loop of
repetitions (cnn_ms, streams_model_ms, their spreads and ratio).  With --kernel-only it reports instead, from
torch.profiler in a loop of --profile-calls calls per path, the summed kernel time per push of each path
(cnn_kernel_ms, streams_model_kernel_ms); run it as a separate invocation so that tracing does not slow the timed
loops.

    python tools/live_bench.py --cnn --ragged [--streams 148,1024,8192] [--push-ms 10,100] [--kernel-only]
                                              [--seconds 2] [--reps 3] [--profile-calls 20] [--out FILE]

runs the live CNN's ragged-push leg: cnn-trad-fpool3 in bf16 (1 s windows, 10 ms shift), float32 samples, states fed
the same audio past the warm-up and timed alternately in the same loop of repetitions.
  aligned   every stream brings the push's n samples: LiveCNN.push_ragged (cnn_ragged_ms), LiveStreams.push_ragged(x,
            lengths, model) (streams_model_ms, the route without LiveCNN's row sharing) and LiveCNN.push (cnn_uniform_ms)
  jitter    the --ragged leg's jittered lengths (10 ms only), which LiveCNN.push cannot take: cnn_ragged_ms against
            streams_model_ms, and the windows per push
With --kernel-only the same rows report the summed kernel time per push of each path (torch.profiler, *_kernel_ms).
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
from honk2_b200 import AudioProcessor, LiveCNN, LiveStreams  # noqa: E402
from honk2_b200.streaming import ragged_push_plan  # noqa: E402

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


def timed_pair(fa, fb, seconds, reps):
    """timed() of two calls, their repetitions alternating: (median_a, spread_a), (median_b, spread_b)."""
    return timed_group((fa, fb), seconds, reps)


def timed_group(fns, seconds, reps):
    """timed() of several calls, their repetitions alternating: ((median, spread) of each)."""
    loops = []
    for fn in fns:
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        t = time.perf_counter()
        for _ in range(10):
            fn()
        torch.cuda.synchronize()
        loops.append(max(10, int(seconds / max((time.perf_counter() - t) / 10, 1e-6))))
    ms = tuple([] for _ in fns)
    for _ in range(reps):
        for i, fn in enumerate(fns):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(loops[i]):
                fn()
            b.record()
            b.synchronize()
            ms[i].append(a.elapsed_time(b) / loops[i])
    return tuple((float(np.median(m)), (max(m) - min(m)) / float(np.median(m))) for m in ms)


def ragged_leg(args, dev, ap, models):
    """The --ragged leg (see the module doc); returns its JSON lines."""
    lines = []
    rng = np.random.default_rng(0)
    gen = torch.Generator(device=dev).manual_seed(0)

    def emit(row):
        print(json.dumps(row), flush=True)
        lines.append(row)

    for S in [int(s) for s in args.streams.split(",")]:
        max_push = 1600
        n160 = np.full(S, H, dtype=np.int64)
        for dtype in args.dtypes.split(","):
            x = torch.rand((S, H), generator=gen, device=dev) * 2 - 1
            chunk = (x * 32767).to(torch.int16) if dtype == "int16" else x
            flat = chunk.reshape(-1)
            uni = LiveStreams(ap, S, W, H, max_push, device=dev)
            rag = LiveStreams(ap, S, W, H, max_push, device=dev)
            out_u = torch.empty((S, 1, 101, 40), device=dev)
            out_r = torch.empty((S, 101, 40), device=dev)
            for _ in range(W // H + 1):                # past the warm-up: S windows per push
                uni.push(chunk, out=out_u)
                rag.push_ragged(flat, n160, out=out_r)
            fu = lambda: uni.push(chunk, out=out_u)            # noqa: E731
            fr = lambda: rag.push_ragged(flat, n160, out=out_r)  # noqa: E731
            (u_ms, u_sp), (r_ms, r_sp) = timed_pair(fu, fr, args.seconds, args.reps)
            emit({"leg": "aligned", "S": S, "dtype": dtype, "windows_per_push": S, "uniform_ms": u_ms,
                  "uniform_spread": u_sp, "ragged_ms": r_ms, "ragged_spread": r_sp,
                  "uniform_kernel_ms": kernel_ms(fu, args.profile_calls),
                  "ragged_kernel_ms": kernel_ms(fr, args.profile_calls)})
            del uni, rag
            torch.cuda.empty_cache()
        # jittered lengths: a fixed cycle of 64 pushes, the same for every repetition
        cycle = jitter_cycle(S, rng)
        pool = torch.rand(S * max_push, generator=gen, device=dev) * 2 - 1
        x = torch.rand((S, H), generator=gen, device=dev) * 2 - 1
        uni = LiveStreams(ap, S, W, H, max_push, device=dev)
        rag = LiveStreams(ap, S, W, H, max_push, device=dev)
        out_u = torch.empty((S, 1, 101, 40), device=dev)
        out_r = torch.empty((S * 7, 101, 40), device=dev)   # >= sum(ceil(n / 160)) for n <= 1024
        for i in range(2 * W // 160):
            n = cycle[i % 64]
            rag.push_ragged(pool[:int(n.sum())], n, out=out_r)
            uni.push(x, out=out_u)
        state = {"i": 0}

        def fr():
            n = cycle[state["i"] % 64]
            state["i"] += 1
            rag.push_ragged(pool[:int(n.sum())], n, out=out_r)
        fu = lambda: uni.push(x, out=out_u)   # noqa: E731
        (u_ms, u_sp), (r_ms, r_sp) = timed_pair(fu, fr, args.seconds, args.reps)
        seen = rag.samples_seen.numpy()
        wins = []
        for n in cycle:                       # windows per push over the cycle, from the host plan
            wins.append(len(ragged_push_plan(seen, n, W, H).stream_ids))
            seen = seen + n
        emit({"leg": "jitter", "S": S, "dtype": "float32", "mean_samples": float(np.mean([c.mean() for c in cycle])),
              "mean_windows_per_push": float(np.mean(wins)), "uniform160_ms": u_ms, "uniform160_spread": u_sp,
              "ragged_ms": r_ms, "ragged_spread": r_sp, "uniform160_kernel_ms": kernel_ms(fu, args.profile_calls),
              "ragged_kernel_ms": kernel_ms(fr, 64)})
        del uni, rag, pool
        torch.cuda.empty_cache()

    # models: warm-up and steady state
    S = args.model_streams
    n160 = np.full(S, H, dtype=np.int64)
    x = torch.rand((S, H), generator=gen, device=dev) * 2 - 1
    flat = x.reshape(-1)
    uni = LiveStreams(ap, S, W, H, 1600, device=dev)
    rag = LiveStreams(ap, S, W, H, 1600, device=dev)
    n_warm = -(-W // H) - 1    # pushes of a fresh stream before its first window completes
    everyone = np.arange(S)
    with torch.no_grad():
        for name, m in models.items():
            fu = lambda: uni.push(x, m)                    # noqa: E731
            fr = lambda: rag.push_ragged(flat, n160, m)    # noqa: E731
            for _ in range(n_warm + 2):
                fu()
                fr()
            (u_ms, u_sp), (r_ms, r_sp) = timed_pair(fu, fr, args.seconds, args.reps)
            ms = ([], [])
            for _ in range(args.reps):
                for i, (st, fn) in enumerate(((uni, fu), (rag, fr))):
                    st.reset(everyone)   # fresh streams: the next n_warm pushes complete no window
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    for _ in range(n_warm):
                        fn()
                    b.record()
                    b.synchronize()
                    ms[i].append(a.elapsed_time(b) / n_warm)
            med = [float(np.median(v)) for v in ms]
            emit({"leg": "model", "model": name, "precision": "bf16", "S": S,
                  "warmup_uniform_ms": med[0], "warmup_uniform_spread": (max(ms[0]) - min(ms[0])) / med[0],
                  "warmup_ragged_ms": med[1], "warmup_ragged_spread": (max(ms[1]) - min(ms[1])) / med[1],
                  "steady_uniform_ms": u_ms, "steady_uniform_spread": u_sp,
                  "steady_ragged_ms": r_ms, "steady_ragged_spread": r_sp})
    return lines


def cnn_leg(args, dev, ap):
    """The --cnn leg (see the module doc); returns its JSON lines."""
    lines = []
    gen = torch.Generator(device=dev).manual_seed(0)
    m = honk2_b200.build_model("cnn-trad-fpool3", precision="bf16").to(dev)
    for S in [int(s) for s in args.streams.split(",")]:
        for push_ms in [int(p) for p in args.push_ms.split(",")]:
            n = 16 * push_ms
            K = n // H
            for dtype in args.dtypes.split(","):
                x = torch.rand((S, n), generator=gen, device=dev) * 2 - 1
                chunk = (x * 32767).to(torch.int16) if dtype == "int16" else x
                lc = LiveCNN(m, S, W, H, max_push=n, audio_processor=ap, device=dev)
                ls = LiveStreams(ap, S, W, H, max_push=n, device=dev)
                out_c = torch.empty((S, K, 12), device=dev)
                feats = torch.empty((S, K, 101, 40), device=dev)
                fc = lambda: lc.push(chunk, out=out_c)            # noqa: E731
                fs = lambda: ls.push(chunk, m, out=feats)         # noqa: E731
                with torch.no_grad():
                    for _ in range(W // n + 2):                   # past the warm-up: every slot valid
                        fc()
                        fs()
                    row = {"leg": "cnn", "model": "cnn-trad-fpool3", "precision": "bf16", "S": S, "push_ms": push_ms,
                           "K": K, "dtype": dtype, "windows_per_push": S * K}
                    if args.kernel_only:
                        row["cnn_kernel_ms"] = kernel_ms(fc, args.profile_calls)
                        row["streams_model_kernel_ms"] = kernel_ms(fs, args.profile_calls)
                    else:
                        (c_ms, c_sp), (s_ms, s_sp) = timed_pair(fc, fs, args.seconds, args.reps)
                        row.update({"cnn_ms": c_ms, "cnn_spread": c_sp, "streams_model_ms": s_ms,
                                    "streams_model_spread": s_sp, "speedup": s_ms / c_ms})
                print(json.dumps(row), flush=True)
                lines.append(row)
                del lc, ls, out_c, feats
                torch.cuda.empty_cache()
    return lines


def jitter_cycle(S, rng):
    """The --ragged leg's jittered lengths: a fixed cycle of 64 pushes, lengths from {0, 160, 320, 1024}."""
    choices = np.array([0, 160, 320, 1024])
    return [rng.choice(choices, size=S, p=[0.5, 0.3, 0.13, 0.07]).astype(np.int64) for _ in range(64)]


def cnn_ragged_leg(args, dev, ap):
    """The --cnn --ragged leg (see the module doc); returns its JSON lines."""
    lines = []
    rng = np.random.default_rng(0)
    gen = torch.Generator(device=dev).manual_seed(0)
    m = honk2_b200.build_model("cnn-trad-fpool3", precision="bf16").to(dev)

    def measure(row, paths):
        names = list(paths)
        if args.kernel_only:
            for k in names:
                row[f"{k}_kernel_ms"] = kernel_ms(paths[k], args.profile_calls)
        else:
            for k, (ms, sp) in zip(names, timed_group([paths[k] for k in names], args.seconds, args.reps)):
                row[f"{k}_ms"], row[f"{k}_spread"] = ms, sp
        print(json.dumps(row), flush=True)
        lines.append(row)

    with torch.no_grad():
        for S in [int(s) for s in args.streams.split(",")]:
            for push_ms in [int(p) for p in args.push_ms.split(",")]:
                n = 16 * push_ms
                K = n // H
                x = torch.rand((S, n), generator=gen, device=dev) * 2 - 1
                flat = x.reshape(-1)
                lengths = np.full(S, n, dtype=np.int64)
                rag = LiveCNN(m, S, W, H, max_push=n, audio_processor=ap, device=dev)
                uni = LiveCNN(m, S, W, H, max_push=n, audio_processor=ap, device=dev)
                ls = LiveStreams(ap, S, W, H, max_push=n, device=dev)
                out_r = torch.empty((S * K, 12), device=dev)
                out_u = torch.empty((S, K, 12), device=dev)
                feats = torch.empty((S * K, 101, 40), device=dev)
                paths = {"cnn_ragged": lambda: rag.push_ragged(flat, lengths, out=out_r),
                         "streams_model": lambda: ls.push_ragged(flat, lengths, m, out=feats),
                         "cnn_uniform": lambda: uni.push(x, out=out_u)}
                for _ in range(W // n + 2):                   # past the warm-up: every stream completes K windows
                    for f in paths.values():
                        f()
                measure({"leg": "cnn_aligned", "model": "cnn-trad-fpool3", "precision": "bf16", "S": S,
                         "push_ms": push_ms, "dtype": "float32", "windows_per_push": S * K}, paths)
                del rag, uni, ls, out_r, out_u, feats, paths
                torch.cuda.empty_cache()
            if 10 not in [int(p) for p in args.push_ms.split(",")]:
                continue
            cycle = jitter_cycle(S, rng)
            max_push = 1600
            pool = torch.rand(S * max_push, generator=gen, device=dev) * 2 - 1
            rag = LiveCNN(m, S, W, H, max_push=max_push, audio_processor=ap, device=dev)
            ls = LiveStreams(ap, S, W, H, max_push=max_push, device=dev)
            out_r = torch.empty((S * 7, 12), device=dev)       # >= sum(ceil(n / 160)) for n <= 1024
            feats = torch.empty((S * 7, 101, 40), device=dev)
            state = {"r": 0, "s": 0}

            def step(key, fn):
                def call():
                    nn = cycle[state[key] % 64]
                    state[key] += 1
                    fn(pool[:int(nn.sum())], nn)
                return call
            paths = {"cnn_ragged": step("r", lambda v, nn: rag.push_ragged(v, nn, out=out_r)),
                     "streams_model": step("s", lambda v, nn: ls.push_ragged(v, nn, m, out=feats))}
            for _ in range(2 * W // 160):
                for f in paths.values():
                    f()
            seen = rag.samples_seen.numpy()
            wins = []
            for nn in cycle:
                wins.append(len(ragged_push_plan(seen, nn, W, H).stream_ids))
                seen = seen + nn
            measure({"leg": "cnn_jitter", "model": "cnn-trad-fpool3", "precision": "bf16", "S": S, "dtype": "float32",
                     "mean_samples": float(np.mean([c.mean() for c in cycle])),
                     "mean_windows_per_push": float(np.mean(wins))}, paths)
            del rag, ls, out_r, feats, pool, paths
            torch.cuda.empty_cache()
    return lines


def cnn_ragged_table(lines):
    """The --cnn --ragged leg's lines as text tables."""
    kern = any("cnn_ragged_kernel_ms" in r for r in lines)
    suf = "_kernel_ms" if kern else "_ms"
    out = [f"cnn-trad-fpool3 bf16, {'kernel ' if kern else ''}ms per push" + ("" if kern else " (spread)")]

    def cell(r, k):
        return f"{r[k + suf]:>9.3f}" + ("" if kern else f" ({100 * r[k + '_spread']:4.1f}%)")
    rows = [r for r in lines if r.get("leg") == "cnn_aligned"]
    if rows:
        out.append("aligned pushes: LiveCNN.push_ragged, LiveStreams.push_ragged(x, lengths, model), LiveCNN.push")
        out.append(f"{'S':>6} {'push':>6} {'cnn_ragged':>18} {'streams+model':>18} {'cnn_uniform':>18} "
                   f"{'model/ragged':>13} {'ragged/uniform':>15}")
        for r in rows:
            out.append(f"{r['S']:>6} {r['push_ms']:>4}ms {cell(r, 'cnn_ragged'):>18} {cell(r, 'streams_model'):>18} "
                       f"{cell(r, 'cnn_uniform'):>18} {r['streams_model' + suf] / r['cnn_ragged' + suf]:>13.2f} "
                       f"{r['cnn_ragged' + suf] / r['cnn_uniform' + suf]:>15.2f}")
    rows = [r for r in lines if r.get("leg") == "cnn_jitter"]
    if rows:
        out.append("jittered pushes (lengths from {0, 160, 320, 1024}), which LiveCNN.push cannot take")
        out.append(f"{'S':>6} {'samples':>8} {'windows':>8} {'cnn_ragged':>18} {'streams+model':>18} {'model/ragged':>13}")
        for r in rows:
            out.append(f"{r['S']:>6} {r['mean_samples']:>8.1f} {r['mean_windows_per_push']:>8.1f} "
                       f"{cell(r, 'cnn_ragged'):>18} {cell(r, 'streams_model'):>18} "
                       f"{r['streams_model' + suf] / r['cnn_ragged' + suf]:>13.2f}")
    return "\n".join(out)


def cnn_table(lines):
    """The --cnn leg's lines as a text table."""
    rows = [r for r in lines if r.get("leg") == "cnn"]
    out = ["cnn-trad-fpool3 bf16, ms per push: LiveCNN.push against LiveStreams.push(chunk, model)"]
    if rows and "cnn_ms" in rows[0]:
        out.append(f"{'S':>6} {'push':>6} {'dtype':>8} {'LiveCNN':>18} {'LiveStreams+model':>20} {'speedup':>8}")
        for r in rows:
            out.append(f"{r['S']:>6} {r['push_ms']:>4}ms {r['dtype']:>8} {r['cnn_ms']:>9.3f} "
                       f"({100 * r['cnn_spread']:.1f}%) {r['streams_model_ms']:>11.3f} "
                       f"({100 * r['streams_model_spread']:.1f}%) {r['speedup']:>8.2f}")
    elif rows:
        out.append(f"{'S':>6} {'push':>6} {'dtype':>8} {'LiveCNN kernels':>16} {'LiveStreams+model kernels':>26}")
        for r in rows:
            out.append(f"{r['S']:>6} {r['push_ms']:>4}ms {r['dtype']:>8} {r['cnn_kernel_ms']:>16.3f} "
                       f"{r['streams_model_kernel_ms']:>26.3f}")
    return "\n".join(out)


def ragged_table(lines):
    """The --ragged leg's lines as text tables."""
    out = []
    rows = [r for r in lines if r.get("leg") == "aligned"]
    if rows:
        out.append("aligned 10 ms pushes (every stream 160 samples): ms per push, [kernel ms], (spread)")
        out.append(f"{'S':>6} {'dtype':>8} {'uniform':>20} {'ragged':>20} {'ragged/uniform':>15}")
        for r in rows:
            out.append(f"{r['S']:>6} {r['dtype']:>8} {r['uniform_ms']:>7.4f} [{r['uniform_kernel_ms']:.4f}] "
                       f"({100 * r['uniform_spread']:.1f}%) {r['ragged_ms']:>7.4f} [{r['ragged_kernel_ms']:.4f}] "
                       f"({100 * r['ragged_spread']:.1f}%) {r['ragged_ms'] / r['uniform_ms']:>8.2f} "
                       f"[{r['ragged_kernel_ms'] / r['uniform_kernel_ms']:.2f}]")
    rows = [r for r in lines if r.get("leg") == "jitter"]
    if rows:
        out.append("jittered pushes (lengths from {0, 160, 320, 1024}) against uniform 160-sample pushes")
        out.append(f"{'S':>6} {'samples':>8} {'windows':>8} {'uniform160':>20} {'ragged':>20}")
        for r in rows:
            out.append(f"{r['S']:>6} {r['mean_samples']:>8.1f} {r['mean_windows_per_push']:>8.1f} "
                       f"{r['uniform160_ms']:>7.4f} [{r['uniform160_kernel_ms']:.4f}] "
                       f"({100 * r['uniform160_spread']:.1f}%) {r['ragged_ms']:>7.4f} [{r['ragged_kernel_ms']:.4f}] "
                       f"({100 * r['ragged_spread']:.1f}%)")
    rows = [r for r in lines if r.get("leg") == "model"]
    if rows:
        out.append("with a model (bf16), ms per push (spread): warm-up of fresh streams, steady state")
        out.append(f"{'model':>16} {'S':>6} {'warm-up uniform':>18} {'warm-up ragged':>18} {'steady uniform':>18} "
                   f"{'steady ragged':>18}")
        for r in rows:
            out.append(f"{r['model']:>16} {r['S']:>6} " + " ".join(
                f"{r[k + '_ms']:>10.3f} ({100 * r[k + '_spread']:.1f}%)"
                for k in ("warmup_uniform", "warmup_ragged", "steady_uniform", "steady_ragged")))
    return "\n".join(out)


def main():
    ap_ = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap_.add_argument("--ragged", action="store_true", help="run the ragged-push leg instead")
    ap_.add_argument("--cnn", action="store_true", help="run the live CNN leg instead")
    ap_.add_argument("--kernel-only", action="store_true", help="--cnn: kernel times from torch.profiler only")
    ap_.add_argument("--model-streams", type=int, default=8192, help="streams of the ragged leg's model runs")
    ap_.add_argument("--streams", default=None, help="default 1,148,1024,8192 (--ragged: 148,1024,8192)")
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
    if args.cnn and args.ragged:
        args.streams = args.streams or "148,1024,8192"
        lines += cnn_ragged_leg(args, dev, ap)
        lines.append({"device": device_line()})
        print(json.dumps(lines[-1]), flush=True)
        table = cnn_ragged_table(lines)
        print(table, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(f"# tools/live_bench.py {' '.join(sys.argv[1:])}\n# device: {header['device']}\n")
                f.write("\n".join("# " + ln for ln in table.splitlines()) + "\n")
                for ln in lines:
                    f.write(json.dumps(ln) + "\n")
        return
    if args.cnn:
        args.streams = args.streams or "148,1024,8192"
        lines += cnn_leg(args, dev, ap)
        lines.append({"device": device_line()})
        print(json.dumps(lines[-1]), flush=True)
        table = cnn_table(lines)
        print(table, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(f"# tools/live_bench.py {' '.join(sys.argv[1:])}\n# device: {header['device']}\n")
                f.write("\n".join("# " + ln for ln in table.splitlines()) + "\n")
                for ln in lines:
                    f.write(json.dumps(ln) + "\n")
        return
    models = {}
    for name in [m for m in args.models.split(",") if m]:
        models[name] = honk2_b200.build_model(name, precision="bf16").to(dev)
    if args.ragged:
        args.streams = args.streams or "148,1024,8192"
        lines += ragged_leg(args, dev, ap, models)
        lines.append({"device": device_line()})
        print(json.dumps(lines[-1]), flush=True)
        table = ragged_table(lines)
        print(table, flush=True)
        if args.out:
            with open(args.out, "w") as f:
                f.write(f"# tools/live_bench.py {' '.join(sys.argv[1:])}\n# device: {header['device']}\n")
                f.write("\n".join("# " + ln for ln in table.splitlines()) + "\n")
                for ln in lines:
                    f.write(json.dumps(ln) + "\n")
        return
    args.streams = args.streams or "1,148,1024,8192"
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
