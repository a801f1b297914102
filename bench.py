#!/usr/bin/env python
"""Headline benchmark: res15 utterances/second, 1 s @ 16 kHz clips, waveform -> MFCC -> logits
(BASELINE.json `metric`; workload = `configs[1]`, res15 at batch 8192 per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--model res15] [--precision bf16|bf16x3|fp32]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # the reference algorithm on the host CPU cores
    python bench.py ... --dump-outputs DIR    # also write the last timed step's logits as DIR/*.npy

One "step" = one pass of the hot path over one batch of synthetic waveforms per GPU.
  value     whole-job utterances/s with the waveforms already resident in HBM (device-timed, CUDA events, max over
            ranks); N > 1 is weak scaling (8192 utterances per GPU) and includes the per-step exchange: ONE NCCL
            all-gather of [logits | correct,total] blocks (honk2_b200.dist.LogitsGather).  `strong_scaling` (N > 1)
            repeats the measurement with the 8192 utterances split over the ranks.
  e2e       same metric through the public API (evaluate.HostPipeline -> model.forward_wave) with HOST buffers:
            pinned waveforms copied host->device and logits copied device->host inside the timed region, every step's
            result guarded by a CUDA event before its buffer is reused.
  roofline  the dominant kernel: algorithmic FLOPs per launch / its average launch duration, measured with CUDA events
            around every launch in a second pass over the same K steps; bound and peak follow the path that ran
            (tensor pipe for the tcgen05 modes, FFMA for the fp32 CUDA-core mode).
  parity    max logit error and argmax agreement of the TIMED precision against the fp32 CUDA-core path (pinned to the
            reference modules by the GPU tests) on >= 8192 synthetic utterances, with an output layer calibrated so that
            the classes are spread (honk2_b200.parity).
  parity_mode  the same measurements for the other tensor-core precision (bf16x3 when the headline runs bf16): the
            mode that meets the fp32 tolerance, driver-visible next to the headline.
  other_configs  the other BASELINE.json configurations (res8, res26, res15-narrow, cnn-trad-fpool3, res15 in fp32, res15
            on 9 s clips), --steps device-resident steps each with their own roofline object, so that one driver run sees them.
  e2e_pcm16 the e2e path fed with int16 PCM host buffers (the wav files' own sample format; bit-identical logits).
  cpu_baseline  the oracle port (oracle/: the reference algorithm in numpy / PyTorch-CPU fp32) timed on this host's
            cores on a bounded sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "res15 utterances/sec (1s 16kHz, MFCC+forward)"
UNIT = "utterances/s"
N_SAMPLES = 16000
FLOPS_PER_UTT = {  # SURVEY.md section 8d / BASELINE.md section 3 (2*MAC, padded taps counted)
    "res15": 1.917627e9, "res8": 0.074351e9, "res26": 0.878073e9, "res15_narrow": 0.342657e9,
    "res8_narrow": 0.014053e9, "res26_narrow": 0.157334e9, "cnn-trad-fpool3": 0.249187e9,
}


DATA = "synthetic (broadband noise clips rounded to 16-bit PCM, s / 32768: what librosa hands the reference for a 16-bit wav)"


def pcm_round(w):
    """float32 clips -> the nearest 16-bit PCM clips, still as float32 (s / 32768, exact).  Both arms, the fp32 and the
    int16 e2e paths then process IDENTICAL samples."""
    return (np.clip(np.round(w * 32768.0), -32768, 32767) / 32768.0).astype(np.float32)


def committed_traffic(kernel_path, batch, precision):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture of the same command
    (profiles/*traffic*.json; the newest record whose kernel, precision and batch match), or None."""
    import glob
    best = None
    for f in sorted(glob.glob(os.path.join(ROOT, "profiles", "*traffic*.json"))):
        try:
            d = json.load(open(f))
        except Exception:
            continue
        if kernel_path in d.get("kernel", "") and d.get("batch_per_launch") == batch and \
                d.get("precision", "bf16") == precision:
            best = d
    return None if best is None else {"dram_bytes_per_launch": best["dram_bytes_per_launch"], "source": best.get("source")}


def dump_outputs(path, arrays, limit=64 << 20):
    """Write each array (name -> tensor) as float32 `path/<name>.npy`, so that two builds can be compared output for output.
    An array larger than its share of `limit` bytes is cut to a fixed, seeded sample of its rows (the same rows on every
    run with the same arguments)."""
    os.makedirs(path, exist_ok=True)
    share = limit // len(arrays)
    for name, t in arrays.items():
        a = torch.as_tensor(t).detach().float().cpu().numpy()
        if a.nbytes > share:
            keep = share // (a.nbytes // a.shape[0])
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], keep, replace=False))]
        np.save(os.path.join(path, name + ".npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "sm_max_mhz": d.get("sm_max_mhz", 1965.0), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "sm_max_mhz": 1965.0,
            "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        # started BEFORE the warm-up (nvidia-smi needs ~0.3 s to produce its first row) and sampled every 20 ms; every
        # row is tagged with the host time it arrived at, stop() keeps the rows that fall inside the timed region
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "20"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self, window=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows, note = [r for _, r in self.rows], None
        if window is not None:
            t0, t1 = window
            inside = [r for t, r in self.rows if t0 <= t <= t1 + 0.03]
            if inside:
                rows = inside
            else:   # region shorter than the sampling period: nearest rows (the GPU is under the same load in the warm-up)
                rows = [r for t, r in self.rows if t0 - 0.25 <= t <= t1 + 0.25]
                note = "no sample fell inside the timed region; rows within 0.25 s of it"
        for r in rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except ValueError:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        out = {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
               "reasons": sorted(reasons), "samples": len(sm)}
        if note:
            out["note"] = note
        return out


# ---------------------------------------------------------------------------------------------------------------------
# the reference arm: the reference algorithm on the host cores.  Imports oracle/ only -- never the product package.

def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import bench_ref
    ref = bench_ref.CpuReference(args.model)
    batch = args.ref_batch
    # the synthetic waveforms are made BEFORE the timed region (the GPU arm's are resident before its region too)
    waves = [pcm_round(bench_ref.broadband(batch, N=N_SAMPLES, seed=1000 + i)) for i in range(args.warmup + args.steps)]
    for i in range(args.warmup):
        ref.step(waves[i])
    t_fe = t_model = 0.0
    t0 = time.perf_counter()
    for i in range(args.steps):
        a, b, logits = ref.step(waves[args.warmup + i])
        t_fe += a; t_model += b
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logits": logits})
    value = batch * args.steps / dt
    sample = (f"each step is a bounded sample of the workload: {batch} of its {args.batch} synthetic {N_SAMPLES / 16000:g} s clips "
              f"(the reference's own configured batch size), {args.steps} steps: numpy restatement of compute_mfccs per "
              f"sample + PyTorch-CPU fp32 restatement of {args.model} forward; front-end {t_fe:.2f} s, model {t_model:.2f} s")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": DATA,
            # the SAME workload as the GPU arm (its `config`); `sample_per_step` is what one timed step of this arm covers
            "config": dict(workload_config(args, args.batch), sample_per_step=batch),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": ref.cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


def workload_config(args, batch):
    secs, frames = N_SAMPLES / 16000.0, 1 + N_SAMPLES // 160
    return {"workload": f"{args.model} inference, {batch} synthetic {secs:g} s / 16 kHz clips per GPU per step, "
                        f"waveform -> {frames}x40 MFCC -> logits (12 GSC classes), random-init weights (seed of the config)",
            "model_config": args.model, "batch_per_gpu": batch, "clip_samples": N_SAMPLES,
            "l2": "inputs larger than L2 (%.0f MB of waveforms per GPU per step, two alternating sets)" % (batch * N_SAMPLES * 4 / 1e6)}


# ---------------------------------------------------------------------------------------------------------------------

def roofline_for(prof, precision, pk, B, K):
    """`roofline` object of the dominant kernel from a per-launch profile pass."""
    if prof is None or prof["conv_launches"] <= 0:
        return None
    flops_per_launch = prof["conv_flops_per_launch"]
    avg_s = prof["conv_ms"] / prof["conv_launches"] / 1e3
    achieved = flops_per_launch / avg_s / 1e12
    if precision == "fp32":
        # CUDA-core path: 148 SMs x 128 FP32 lanes x 2 FLOP at the maximum SM clock
        peak = 148 * 128 * 2 * pk["sm_max_mhz"] * 1e6 / 1e12
        bound, peak_src, burst = "ffma", "148 SMs x 128 lanes x 2 x %.0f MHz (nominal FP32 FMA rate)" % pk["sm_max_mhz"], peak
    else:
        peak, burst = pk["bf16_tflops_sustained"], pk["bf16_tflops"]
        bound, peak_src = "tensor", pk["source"] + " (sustained bf16)"
    tr = committed_traffic(prof.get("kernel_path", "?"), B, precision)
    roof = {"bound": bound, "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
            "traffic": None if tr is None else tr["dram_bytes_per_launch"],
            "traffic_source": None if tr is None else tr["source"],
            "frac_of_burst_peak": achieved / burst,
            "kernel": prof["conv_kernel"], "launches": prof["conv_launches"],
            "avg_launch_ms": prof["conv_ms"] / prof["conv_launches"], "peak_source": peak_src,
            "share_of_step": prof["conv_ms"] / max(prof["total_ms"], 1e-9),
            "frontend_ms_per_step": prof["frontend_ms"] / K, "other_ms_per_step": prof["other_ms"] / K}
    if precision == "bf16x3":
        roof["note"] = ("algorithmic FLOPs are the fp32 network's; this mode issues three bf16 MMAs per product, so "
                        "the tensor pipe does 3x the counted work")
        roof["tensor_pipe_frac_of_burst_peak"] = 3 * achieved / burst
    return roof


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="res15")
    ap.add_argument("--precision", default=None, choices=["fp32", "bf16", "bf16x3"])
    ap.add_argument("--batch", type=int, default=8192)
    ap.add_argument("--clip-samples", type=int, default=16000,
                    help="samples per clip (16000 = the headline 1 s clips; 144000 = the hey_snips-shaped 9 s clips of config 5)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: weak = --batch utterances per GPU (default), strong = --batch utterances in total")
    ap.add_argument("--chunk", type=int, default=0)
    ap.add_argument("--lanes", type=int, default=0, help="concurrent chunk streams of the layer-per-launch path (0 = library default)")
    ap.add_argument("--ref-batch", type=int, default=64)
    ap.add_argument("--e2e-sub-batch", type=int, default=4096)
    ap.add_argument("--e2e-slots", type=int, default=3)
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-second-mode", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true",
                    help="skip the short device-resident runs of the other BASELINE.json configurations (`other_configs`)")
    ap.add_argument("--gpu-eager-bar", action="store_true",
                    help="also time the PyTorch-eager (cuDNN) forward of the reference architecture on this GPU (SURVEY 8d)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the logits of the last timed step as DIR/<name>.npy (float32; rank 0): logits (device-"
                         "resident path), e2e_logits and e2e_pcm16_logits (host-buffer paths); --impl reference: logits")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)
    global N_SAMPLES
    N_SAMPLES = args.clip_samples

    if args.impl == "reference":
        run_reference_arm(args)
        return
    if args.lanes:
        os.environ["HONK2_TC_LANES"] = str(args.lanes)

    import honk2_b200
    from honk2_b200 import AudioProcessor, numa, parity, synth
    from honk2_b200 import dist as kdist
    from honk2_b200.evaluate import HostPipeline
    from honk2_b200.metric import Acc
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU path (use --impl reference for the CPU arm)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # pinned host buffers allocated below land on the NUMA node of this rank's GPU (first touch)
    numa_info = numa.bind_to_gpu_node(local) if world > 1 else {"bound": False, "why": "single process"}
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    precision = args.precision or os.environ.get("HONK2_BENCH_PRECISION", "bf16")
    model = honk2_b200.build_model(args.model, precision=precision).to(dev)
    if args.chunk:
        model.chunk = {p: args.chunk for p in ("fp32", "bf16", "bf16x3")}
    fe = AudioProcessor()
    B_cfg = args.batch
    B = B_cfg if args.scaling == "weak" else -(-B_cfg // world)     # utterances per GPU per step
    K, W = args.steps, max(args.warmup, 3)

    # synthetic data: two distinct batches (each 524 MB > L2), device resident for `value`
    n_sets = 2
    host_sets = [torch.from_numpy(pcm_round(synth.broadband(B_cfg, N=N_SAMPLES, seed=100 * rank + s))).pin_memory() for s in range(n_sets)]
    host_f32 = host_sets
    dev_sets = [h.to(dev) for h in host_sets]
    targets = torch.randint(0, model.n_labels, (B_cfg,), device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        t = torch.tensor([ms], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed_device(per_gpu, steps, warm):
        """`steps` device-resident steps of `per_gpu` utterances per GPU: forward_wave straight into the gather buffer,
        accuracy counted on the device into the same buffer, one collective.
        -> (ms max over ranks, launches, host time window, logits of the last step)."""
        gather = kdist.LogitsGather(per_gpu * world, model.n_labels, dev)
        acc = Acc(counts=gather.counts)
        tg = targets[:per_gpu]

        def step(i):
            model.forward_wave(dev_sets[i % n_sets][:per_gpu], fe, out=gather.logits)
            acc.accumulate(gather.logits, tg)
            if world > 1:
                gather.exchange()

        for i in range(warm):
            step(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches = 0
        th0 = time.perf_counter()
        e0.record()
        for i in range(steps):
            step(i)
            launches += model.last_launches(dev) + 1          # front-end + network (+ tail) launches, + the accuracy kernel
        e1.record()
        barrier()
        th1 = time.perf_counter()
        return max_over_ranks(e0.elapsed_time(e1)), launches, (th0, th1), gather.logits

    def timed_e2e(per_gpu, steps, hosts=None):
        """pinned host waveforms -> H2D -> forward_wave -> logits D2H, pipelined; every step's result is complete (event)
        before its host buffer is handed out again.  `hosts`: other pinned host batches (the int16 PCM form).
        -> (ms max over ranks, host logits of the last step)."""
        host_sets = hosts if hosts is not None else host_f32
        pipe = HostPipeline(model, fe, N_SAMPLES, sub_batch=min(args.e2e_sub_batch, per_gpu), device=dev,
                            slots=args.e2e_slots, dtype=host_sets[0].dtype)
        outs = [torch.empty((per_gpu, model.n_labels), dtype=torch.float32).pin_memory() for _ in range(2)]
        pending = [None, None]

        def step(i):
            j = i & 1
            if pending[j] is not None:
                pending[j].synchronize()                       # the caller reads / reuses outs[j] only after this
            pending[j] = pipe(host_sets[i % n_sets][:per_gpu], outs[j], sync=False)

        for i in range(2):
            step(i)
        for ev in pending:
            ev.synchronize()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            step(i)
        e1.record()
        for ev in pending:
            ev.synchronize()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)), outs[(steps - 1) & 1]

    with torch.no_grad():
        sampler = ClockSampler(local)
        if rank == 0:
            sampler.start()
        ms, launches, window, logits = timed_device(B, K, W)
        clocks = sampler.stop(window) if rank == 0 else None
        value = B * world * K / (ms / 1e3)
        ms_e2e, logits_e2e = timed_e2e(B, K)
        e2e_value = B * world * K / (ms_e2e / 1e3)
        # the same end-to-end path fed with 16-bit PCM samples, the format of the wav files behind the reference's
        # datasets (librosa returns float32(s / 32768) for them): half the host->device bytes, bit-identical logits
        host_pcm = [(h * 32768.0).round().clamp(-32768, 32767).to(torch.int16).pin_memory() for h in host_f32]
        ms_e2e_pcm, logits_e2e_pcm = timed_e2e(B, K, hosts=host_pcm)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"logits": logits, "e2e_logits": logits_e2e,
                                             "e2e_pcm16_logits": logits_e2e_pcm})
        # (the clips are 16-bit PCM already, see pcm_round: the two paths must agree bit for bit)
        n_chk = min(B, 1024)
        pcm_same = bool(torch.equal(model.forward_wave(host_pcm[0][:n_chk].to(dev), fe),
                                    model.forward_wave(dev_sets[0][:n_chk], fe)))
        del host_pcm

        strong = None
        if world > 1 and args.scaling == "weak":
            per = -(-B_cfg // world)
            ms_s = timed_device(per, K, W)[0]
            ms_s_e2e = timed_e2e(per, K)[0]
            strong = {"total_batch": per * world, "batch_per_gpu": per, "value": per * world * K / (ms_s / 1e3),
                      "ms_per_step": ms_s / K, "e2e_value": per * world * K / (ms_s_e2e / 1e3), "unit": UNIT,
                      "note": "the 8192-utterance batch of the headline configuration split over the ranks "
                              "(persistent kernel: %.1f utterances per SM per step)" % (per / 148.0)}

        # ---- roofline of the dominant kernel: per-launch events in a second pass over K steps
        prof = honk2_b200.profile_layers(model, fe, [d[:B] for d in dev_sets], K) if rank == 0 else None

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk = peaks()
    roof = roofline_for(prof, precision, pk, B, K)

    # ---- parity of the timed mode (and of the second mode) against the fp32 path, calibrated diverse-class weights
    par = second = None
    if args.model in FLOPS_PER_UTT and not args.model.startswith("cnn") and N_SAMPLES == 16000:
        with torch.no_grad():
            pw = torch.cat([dev_sets[0][:8192], torch.from_numpy(synth.speechlike(1024, seed=9)).to(dev)])
            if not args.no_parity or not args.no_second_mode:
                cal = fe.compute_mfccs_batch(torch.from_numpy(synth.speechlike(256, seed=21)).to(dev))
                cm = parity.calibrated_model(args.model, cal, precision=precision)
            if not args.no_parity and precision != "fp32":
                par = parity.parity_report(cm, fe, pw, precision)
                par["inputs"] = "8192 broadband + 1024 speech-like synthetic clips; hardened weights, output layer calibrated on 256 clips"
            other = {"bf16": "bf16x3", "bf16x3": "bf16"}.get(precision)
            if other is not None and world == 1 and not args.no_second_mode:
                model.precision = other
                try:
                    ms2 = timed_device(B, K, W)[0]
                    ms2_e2e = timed_e2e(B, K)[0]
                    prof2 = honk2_b200.profile_layers(model, fe, [d[:B] for d in dev_sets], K)
                    second = {"precision": other, "value": B * K / (ms2 / 1e3), "unit": UNIT, "ms_per_step": ms2 / K,
                              "e2e": {"value": B * K / (ms2_e2e / 1e3), "unit": UNIT, "ms_per_step": ms2_e2e / K},
                              "roofline": roofline_for(prof2, other, pk, B, K),
                              "parity": parity.parity_report(cm, fe, pw, other)}
                finally:
                    model.precision = precision

    if args.model.startswith("cnn") and precision != "fp32" and not args.no_parity and N_SAMPLES == 16000:
        # CNN family: hardened weights (no global-mean layer to calibrate on); the timed mode against the fp32 CUDA-core path
        with torch.no_grad():
            pw = torch.cat([dev_sets[0][:8192], torch.from_numpy(synth.speechlike(1024, seed=9)).to(dev)])
            cm = honk2_b200.build_model(args.model, precision=precision)
            synth.harden_(cm.state_dict())
            cm = cm.to(dev)
            par = parity.parity_report(cm, fe, pw, precision)
            par["inputs"] = "8192 broadband + 1024 speech-like synthetic clips; hardened weights"

    # ---- the other BASELINE.json configurations, device-resident, a few steps each, in the same driver-visible line
    others = None
    if world == 1 and not args.no_other_configs and args.model == "res15" and N_SAMPLES == 16000:
        others = []
        plan = [("res8", "bf16", 8192, 16000, "configs[0] on the GPU"), ("res15", "fp32", 2048, 16000, "configs[1], fp32 half"),
                ("res15", "bf16x3", 8192, 16000, "configs[1], fp32-grade tensor-core mode"),
                ("res26", "bf16", 8192, 16000, "configs[2]"), ("res15_narrow", "bf16", 8192, 16000, "configs[2]"),
                ("res15_narrow", "fp32", 2048, 16000, "configs[2], CUDA-core path"),
                ("cnn-trad-fpool3", "bf16", 8192, 16000, "configs[3]"),
                ("cnn-trad-fpool3", "fp32", 4096, 16000, "configs[3], CUDA-core parity mode"),
                ("res15", "bf16", 1024, 144000, "configs[4], one GPU's view: hey_snips-shaped 9 s clips"),
                ("hey_snips_res26", "bf16", 256, 144000, "configs[2], the deep dilated stack (24 layers, dilation <= 128) at its own 901x40 shape")]
        for name, prec, nb, ns, tag in plan:
            if prec == precision and name == args.model and ns == N_SAMPLES:
                continue
            if second is not None and name == args.model and prec == second["precision"] and ns == N_SAMPLES:
                continue   # already in `parity_mode`
            try:
                with torch.no_grad():
                    mo = honk2_b200.build_model(name, precision=prec).to(dev)
                    # the resident synthetic waveforms again (no host-side generation): 1 s clips as they are, the 9 s clips
                    # cut from the two sets laid end to end (synthetic broadband noise either way)
                    if ns == N_SAMPLES:
                        ws = [d[:nb] for d in dev_sets]
                    else:
                        flat = torch.cat([d.reshape(-1) for d in dev_sets])
                        ws = [flat[o:o + nb * ns].view(nb, ns) for o in (0, 8000)]
                    out = torch.empty((nb, mo.n_labels), dtype=torch.float32, device=dev)
                    for i in range(3):
                        mo.forward_wave(ws[i & 1], fe, out=out)
                    torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for i in range(K):
                        mo.forward_wave(ws[i & 1], fe, out=out)
                    e1.record()
                    torch.cuda.synchronize()
                    ms_o = e0.elapsed_time(e1)
                    pr = honk2_b200.profile_layers(mo, fe, ws, K)
                    rf = roofline_for(pr, prec, pk, nb, K)
                    others.append({"model": name, "precision": prec, "batch": nb, "clip_samples": ns, "baseline_config": tag,
                                   "value": nb * K / (ms_o / 1e3), "unit": UNIT, "ms_per_step": ms_o / K, "steps": K,
                                   "roofline": None if rf is None else {k: rf[k] for k in (
                                       "bound", "achieved", "peak", "unit", "frac", "frac_of_burst_peak", "kernel",
                                       "avg_launch_ms", "share_of_step", "frontend_ms_per_step")}})
                    del mo, ws, out
                    flat = None
                    torch.cuda.empty_cache()
            except Exception as exc:   # one configuration failing must not lose the headline line
                others.append({"model": name, "precision": prec, "batch": nb, "clip_samples": ns, "error": repr(exc)[:300]})

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        from oracle import bench_ref
        ref = bench_ref.CpuReference(args.model)
        ref.step(pcm_round(bench_ref.broadband(8, N=N_SAMPLES, seed=1)))
        n, t_cpu, fe_s, mo_s = 0, 0.0, 0.0, 0.0
        while t_cpu < args.cpu_seconds and n < 64 * 64:
            waves = pcm_round(bench_ref.broadband(args.ref_batch, N=N_SAMPLES, seed=3000 + n))
            t0 = time.perf_counter()
            a, b, _ = ref.step(waves)
            t_cpu += time.perf_counter() - t0
            fe_s += a; mo_s += b
            n += args.ref_batch
        cpu = {"value": n / t_cpu, "unit": UNIT, "cores": ref.cores, "kind": "port",
               "sample": f"{n} synthetic {N_SAMPLES / 16000:g} s clips in batches of {args.ref_batch}: numpy compute_mfccs "
                         f"restatement per sample ({fe_s:.1f} s) + PyTorch-CPU fp32 {args.model} forward ({mo_s:.1f} s)"}

    eager = None
    if args.gpu_eager_bar and world == 1:
        from oracle import bench_ref
        eager = bench_ref.gpu_eager_bar(args.model, batch=min(B, 1024 if N_SAMPLES == 16000 else 64), T=1 + N_SAMPLES // 160)

    # ---- streaming windows (SURVEY 8f-1), reported next to the headline: B windows of 1 s at a 10 ms shift
    # (gsc_dev_config.json:62-63) from one resident stream; front-end alone and front-end + network.
    streaming = None
    if world == 1 and N_SAMPLES == 16000:
        with torch.no_grad():
            stream = torch.from_numpy(synth.broadband(1, N=B * 160 + N_SAMPLES, seed=77)[0]).to(dev)
            feats_s = torch.empty((B, fe.n_frames(N_SAMPLES), fe.n_mels), dtype=torch.float32, device=dev)

            def timed(fn, reps=K):
                for _ in range(2):
                    fn()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                a.record()
                for _ in range(reps):
                    fn()
                b.record()
                torch.cuda.synchronize()
                return a.elapsed_time(b) / reps

            ms_fe_stream = timed(lambda: fe.compute_mfccs_stream(stream, N_SAMPLES, 160, out=feats_s))
            ms_fe_batch = timed(lambda: fe.compute_mfccs_batch(dev_sets[0][:B], out=feats_s))
            ms_all = timed(lambda: model(fe.compute_mfccs_stream(stream, N_SAMPLES, 160, out=feats_s)))
            streaming = {"windows_per_step": B, "window_samples": N_SAMPLES, "shift_samples": 160,
                         "frontend_ms_shared_frames": ms_fe_stream, "frontend_ms_per_window_batch": ms_fe_batch,
                         "windows_per_s_frontend_plus_network": B / (ms_all / 1e3)}

    # front-end kernel against ITS roofline (HBM): 64 000 B in + 16 160 B out per 1 s utterance (SURVEY 8d)
    fe_roof = None
    if prof is not None and prof["frontend_ms"] > 0:
        fe_bytes = B * (N_SAMPLES * 4 + (1 + N_SAMPLES // 160) * 40 * 4)
        gbs = fe_bytes / (prof["frontend_ms"] / K / 1e3) / 1e9
        fe_roof = {"bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": gbs / pk["hbm_gbs"],
                   "kernel": "mfcc_kernel", "ms_per_launch": prof["frontend_ms"] / K}
        # what actually limits it (committed `ncu --set full` record of the same kernel): the SM, not HBM
        try:
            rec = json.load(open(os.path.join(ROOT, "profiles", "r2_mfcc_ncu.json")))
            fe_roof["limiter"] = {"lsu_wavefronts_pct_of_peak": rec.get("lsu_wavefronts_pct_of_peak"),
                                  "issue_slots_busy_pct": rec.get("issue_slots_busy_pct"),
                                  "dram_gb_per_s": rec.get("dram_gb_per_s_under_ncu"), "source": rec.get("source"),
                                  "note": "instruction / shared-memory bound (240-point FFT in registers + one exchange per frame)"}
        except Exception:
            pass

    dtype = {"bf16": "bf16", "bf16x3": "bf16 (split hi+lo pairs, 3 MMAs per product, fp32 accumulate)", "fp32": "f32"}[precision]
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None,
            "dtype": dtype, "data": DATA,
            "config": dict(workload_config(args, B), precision=precision, parallelism=f"dp{world}",
                           exchange="one all-gather of [logits | correct,total] per step" if world > 1 else "none",
                           e2e_pipeline=f"{args.e2e_slots} staging slots x {min(args.e2e_sub_batch, B)} clips"),
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": B * N_SAMPLES * 4,
                    "d2h_bytes_per_step": B * model.n_labels * 4, "ms_per_step": ms_e2e / K},
            "e2e_pcm16": {"value": B * world * K / (ms_e2e_pcm / 1e3), "unit": UNIT, "h2d_bytes_per_step": B * N_SAMPLES * 2,
                          "d2h_bytes_per_step": B * model.n_labels * 4, "ms_per_step": ms_e2e_pcm / K,
                          "logits_bit_identical_to_f32_path": pcm_same,
                          "note": "the SAME clips handed over as int16 PCM host buffers (the wav files' sample format) through "
                                  "kws_model_forward_wave_pcm16: half the host->device bytes"},
            "gpu_launches": launches, "roofline": roof, "frontend_roofline": fe_roof, "parity": par,
            "parity_mode": second, "cpu_baseline": cpu, "gpu_eager_bar": eager, "streaming_windows": streaming,
            "strong_scaling": strong, "numa": numa_info, "other_configs": others,
            "tensor_frac_of_burst_peak_whole_step": FLOPS_PER_UTT.get(args.model, 0) * value / world / 1e12 / pk["bf16_tflops"]}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
