#!/usr/bin/env python
"""Benchmark of the DDSP synthesis hot path on B200 (BASELINE.json metric / configs[1]).

A "step" is one pass of the hot path over one batch of synthetic decoder outputs:
controls -> harmonic bank + filtered noise -> reverb -> multi-scale spectral loss -> backward to the
synth parameters (decoder.py:106-125 + train.py:92-103,129 of the reference, without the control
network).  Workload: 16 kHz, block 160, 100 harmonics, 65 noise bands, 4 s, batch 64 sharded over
the N GPUs (strong scaling), reverb 16000 taps, 6 STFT scales.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload train|bulk]
                    [--dump-outputs DIR]
    torchrun --nproc-per-node N bench.py --gpus N ...     (one rank per GPU)

Prints ONE JSON line (rank 0).  `value` = audio samples/s of forward+backward with inputs resident
in HBM (CUDA events, max over ranks); `e2e` = the same through pinned host buffers with the H2D
copies and the loss read-back inside the timed region; `roofline` = the dominant kernel against its
binding roof; `parity` = this run's audio and loss against the float64 oracle (outside the timed
region); `cpu_baseline` = the unmodified reference (oracle/_ref) on this box's host cores;
`configs` = the other BASELINE.json configurations (full model step, batch-16 forward, realtime
latency, autoencoder, bulk-render slice).  `--impl reference` times only the reference's CPU path and
imports nothing of the product.  `--workload bulk` is configs[3]: forward only, 1024 voices per GPU
(weak scaling, no collective).
"""
from __future__ import annotations

import argparse
import importlib.util
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "DDSP synth audio samples/sec (fwd+bwd)"
UNIT = "samples/s"
WORKLOAD = dict(sample_rate=16000, block_size=160, n_harmonic=100, n_bands=65, frames=400, batch=64,
                reverb_length=16000, scales=(4096, 2048, 1024, 512, 256, 128), overlap=0.75)
WORKLOAD_NAME = ("configs[1]: synth hot path fwd+bwd with multiscale_fft loss, 16 kHz, block 160, "
                 "100 harmonics, 65 bands, 4 s, batch 64 sharded over N GPUs, reverb 16000 taps")
BULK_NAME = ("configs[3]: bulk render, 48 kHz, block 512, 256 harmonics, 65 bands, 4 s, 1 s learned-IR reverb, forward, "
             "1024 voices per GPU (8192 over 8), no cross-GPU traffic")


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=100, help="steps of every timed loop")
    p.add_argument("--warmup", type=int, default=10)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--workload", default="train", choices=["train", "bulk"])
    p.add_argument("--no-graph", action="store_true", help="launch eagerly instead of replaying a CUDA graph")
    p.add_argument("--cpu-batch", type=int, default=16, help="voices in the bounded cpu_baseline sample of the B200 arm")
    p.add_argument("--skip-cpu", action="store_true")
    p.add_argument("--global-batch", type=int, default=WORKLOAD["batch"],
                   help="experiments only: the benchmark config is batch 64 (BASELINE.json configs[1])")
    p.add_argument("--skip-kernels", action="store_true")
    p.add_argument("--e2e-sets", type=int, default=3,
                   help="static input sets (each with its own captured graph) of the end-to-end loop: sets - 1 batches in flight")
    p.add_argument("--allreduce-outside", action="store_true",
                   help="N>1: queue the gradient all-reduce after the graph instead of inside it (A/B of the overlap)")
    p.add_argument("--skip-configs", action="store_true", help="do not measure the other BASELINE.json configurations")
    p.add_argument("--skip-parity", action="store_true")
    p.add_argument("--bulk-voices", type=int, default=1024, help="voices per GPU of --workload bulk")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="after the timed steps, write what the last one computed (audio, loss, gradients; rank 0's voices) "
                        "as DIR/<name>.npy in float32, so that two builds can be compared output for output")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "train"):
        p.error("--dump-outputs writes the outputs of --impl b200 --workload train")
    return args


def shapes_module():
    """ddsp_pytorch_b200/shapes.py loaded by path: pure Python, does not import the package (no native library is
    mapped into a process that only runs the reference arm)."""
    name = "b200_bench_shapes"
    if name in sys.modules:
        return sys.modules[name]
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, "ddsp_pytorch_b200", "shapes.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


# ------------------------------------------------------------------------------------------ CPU arm
def cpu_reverb_state(shapes, seed=0):
    g = torch.Generator().manual_seed(seed)
    L = shapes.reverb_length
    return {"noise": (torch.rand(L, generator=g) * 2 - 1).unsqueeze(-1), "decay": torch.tensor(5.0),
            "wet": torch.tensor(0.0), "t": (torch.arange(L) / shapes.sample_rate).reshape(1, -1, 1)}


class CpuArm:
    """The reference's CPU implementation of the step on `batch` voices of the benchmark shapes: the unmodified
    reference from oracle/_ref (kind "reference") when it is in place, else the oracle port (kind "port")."""

    def __init__(self, batch):
        sm = shapes_module()
        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        w = dict(WORKLOAD)
        w["batch"] = batch
        self.shapes = sm.SynthShapes(**w)
        self.host = sm.synthetic_inputs(self.shapes, seed=0)
        rs = cpu_reverb_state(self.shapes)
        from oracle import ref_step
        if ref_step.available():
            self.kind = "reference"
            self.impl = ref_step.ReferenceStep(self.shapes, rs)
            self.fn = lambda: self.impl.step(self.host)
        else:
            from oracle import ddsp_oracle as orc
            self.kind = "port"
            h, s = self.host, self.shapes
            self.fn = lambda: orc.synth_train_step(h["amp_raw"], h["dist_raw"], h["mag_raw"], h["pitch"], h["noise"],
                                                   h["target"], s.block_size, s.sample_rate, dict(rs), list(s.scales),
                                                   s.overlap)

    def time(self, steps, warmup):
        for _ in range(warmup):
            self.fn()
        times = []
        for _ in range(steps):
            t0 = time.perf_counter()
            self.fn()
            times.append(time.perf_counter() - t0)
        return times


def run_reference(args, rank):
    """--impl reference: the reference's own CPU path, all host threads, on as many of the 64 voices per step as
    keep the whole run within a few minutes (all 64 on the GPU boxes' hosts).  Nothing of the product is imported."""
    if rank != 0:
        return
    total_steps = max(1, args.steps + args.warmup)
    budget = 240.0 / total_steps                                  # seconds one step may take
    probe = CpuArm(4)
    t4 = min(probe.time(2, 1))
    batch = WORKLOAD["batch"]
    while batch > 2 and t4 * batch / 4 > budget:
        batch //= 2
    arm = CpuArm(batch)
    times = arm.time(args.steps, args.warmup)
    total = sum(times)
    value = batch * arm.shapes.samples * len(times) / total
    same = batch == WORKLOAD["batch"]
    sample = (f"all {batch} voices per step" if same else f"{batch} of 64 voices per step (same shapes)") + \
        f", float32, {arm.cores} threads, " + ("unmodified reference code from oracle/_ref" if arm.kind == "reference"
                                               else "oracle port (oracle/_ref not present)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": {"workload": WORKLOAD_NAME, "per_step_sample": sample, "same_config": same},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": arm.cores, "kind": arm.kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "product_modules_imported": sorted(m for m in sys.modules if m.startswith("ddsp_pytorch_b200")),
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
               0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz, self.ok = [], set(), None, False
        self._stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False
        self.t = threading.Thread(target=self._loop, daemon=True)

    def _loop(self):
        while not self._stop.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                bits = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for b, name in self.REASONS.items():
                    if bits & b and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def __enter__(self):
        if self.ok:
            self.t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self.ok:
            self.t.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": []}
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2], "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------------------ B200 arm
def event_time(fn, iters, warmup, flush=None):
    """Average device time of fn() over iters, CUDA events on the current stream, L2 flushed between."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    total = 0.0
    for _ in range(iters):
        if flush is not None:
            flush()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        total += a.elapsed_time(b)
    return total / iters          # ms


def load_peaks():
    peaks = {"hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk):
        with open(pk) as f:
            peaks = json.load(f)
        peaks["source"] = "MEASURED_PEAKS.json (burst copy bandwidth)"
    return peaks


class near_gpu:
    """Context manager: run the body with the process bound to the CPUs NVML lists as local to the GPU, so that pinned
    host buffers allocated (first touched) inside land on the GPU's NUMA node.  Best effort: any failure leaves the
    affinity alone."""

    def __init__(self, dev):
        self.dev, self.saved = dev, None

    def __enter__(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            props = torch.cuda.get_device_properties(self.dev)
            uuid = getattr(props, "uuid", None)
            h = pynvml.nvmlDeviceGetHandleByUUID(f"GPU-{uuid}") if uuid is not None else \
                pynvml.nvmlDeviceGetHandleByIndex(self.dev.index or 0)
            words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
            cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (w >> b) & 1}
            allowed = os.sched_getaffinity(0)
            if cpus & allowed and (cpus & allowed) != allowed:
                self.saved = allowed
                os.sched_setaffinity(0, cpus & allowed)
        except Exception:
            self.saved = None
        return self

    def __exit__(self, *a):
        if self.saved is not None:
            os.sched_setaffinity(0, self.saved)


def h2d_rate(block, step, flush):
    """The host link alone: the step's pinned input block copied into the idle input set, nothing else running."""
    dst = step._pair[1]["flat"]
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    ts = []
    with torch.cuda.stream(s):
        for _ in range(16):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(s)
            dst.copy_(block, non_blocking=True)
            b.record(s)
            b.synchronize()
            ts.append(a.elapsed_time(b))
    ms = sorted(ts)[len(ts) // 2]
    nbytes = block.numel() * block.element_size()
    return {"ms_per_batch": ms, "gb_per_s": nbytes / (ms * 1e-3) / 1e9, "ms_min": min(ts), "ms_max": max(ts), "copies": len(ts),
            "note": "host->device copy of one step's inputs on an otherwise idle GPU; when this exceeds ms_per_step of "
                    "the device-timed value, e2e is bound by the host link, not by the kernels"}


def ncu_traffic(key):
    """DRAM bytes per launch from the committed ncu --set full capture (profiles/r02_ncu_traffic.json), or None."""
    p = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
    if not os.path.exists(p):
        return None, None
    with open(p) as f:
        d = json.load(f)
    e = d.get(key)
    return (e["dram_bytes"], e.get("note")) if e else (None, None)


def kernel_table(step, shapes, flush, peaks):
    """Per-kernel device time (events, L2 flushed) and roofline fraction for the stages of the path."""
    import math
    ops = torch.ops.ddsp_b200
    i = {k: v.detach() for k, v in step.inputs.items()}
    B, T, bs, H, NB, N = shapes.batch, shapes.frames, shapes.block_size, shapes.n_harmonic, shapes.n_bands, shapes.samples
    sr = float(shapes.sample_rate)
    amps, dist, w = ops.harmonic_controls_fwd(i["amp_raw"], i["dist_raw"], i["pitch"], sr, True)
    audio, _, phi, delta = ops.harmonic_fwd(i["pitch"], w, bs, sr, None)
    g = torch.randn_like(audio)
    sig2 = audio.squeeze(-1).contiguous()
    imp = step.reverb.build_impulse().detach().reshape(1, -1)
    from ddsp_pytorch_b200.functions import hann_window_like_reference
    windows = torch.cat([hann_window_like_reference(s, audio.device) for s in shapes.scales])
    clk = (peaks.get("sm_max_mhz") or 1965.0) * 1e6
    fma_peak = 148 * 128 * clk                      # FP32 lanes x clock: FMAs (or adds, or muls) per second
    hs = B * N * H                                  # harmonic-samples
    rows = []

    def add(name, fn, alg_bytes=None, fma_ops=None, note=""):
        ms = event_time(fn, 20, 3, flush)
        r = {"kernel": name, "ms": ms}
        if alg_bytes is not None:
            r.update(bound="hbm", achieved=alg_bytes / (ms * 1e-3) / 1e9, peak=peaks["hbm_gbs"], unit="GB/s")
        if fma_ops is not None:
            r.update(bound="fp32", achieved=fma_ops / (ms * 1e-3) / 1e12, peak=fma_peak / 1e12, unit="TFMA/s")
        r["frac"] = r["achieved"] / r["peak"]
        r["note"] = note
        rows.append(r)

    # the step's own form of K1: get_controls rides in the bank's prologue, its backward in the backward's epilogue
    # (phase scan included in the forward's time, as in the op)
    add("K0+K1 harmonic_raw_fwd (controls + oscillator bank)",
        lambda: ops.harmonic_raw_fwd(i["amp_raw"], i["dist_raw"], i["pitch"], bs, sr, None), fma_ops=2 * hs,
        note="SURVEY 8d: 2 FMA per harmonic-sample (recurrence + weighted sum) vs 148 SM x 128 lanes x max clock")
    add("K0+K1 harmonic_raw_bwd (oscillator bank + controls backward)",
        lambda: ops.harmonic_raw_bwd(g, i["amp_raw"], i["dist_raw"], i["pitch"], phi, delta, bs, sr), fma_ops=2 * hs)
    add("K1 harmonic_frames_fwd (bank alone, weights given)", lambda: ops.harmonic_fwd(i["pitch"], w, bs, sr, None), fma_ops=2 * hs)
    add("K1 harmonic_frames_bwd (bank alone, d weights)", lambda: ops.harmonic_bwd(g, w, phi, delta, bs, sr, False), fma_ops=2 * hs)
    add("K2 filtered_noise_fwd", lambda: ops.noise_fwd(i["mag_raw"], i["noise"], audio, True, -5.0), alg_bytes=4 * B * T * (NB + 3 * bs))
    add("K2 filtered_noise_bwd", lambda: ops.noise_bwd(g, i["noise"], i["mag_raw"], NB, True, -5.0), alg_bytes=4 * B * T * (NB + 2 * bs))
    kept = ops.fftconv_fwd(sig2, imp, True)
    add("K3 reverb fftconv_fwd", lambda: ops.fftconv_fwd(sig2, imp, True), alg_bytes=4 * (2 * B * N + imp.numel()))
    add("K3 reverb fftconv_bwd (transforms kept by fwd)", lambda: ops.fftconv_bwd(sig2, sig2, imp, kept[1], kept[2], True, True),
        alg_bytes=4 * (3 * B * N + 2 * imp.numel()))
    # K4L: FP32-pipe bound (ncu: profiles/).  Algorithmic flops = 5 n log2 n per complex FFT, one forward per frame
    # (rec + i*target) and one inverse per frame pair; HBM view (SURVEY 8d: read rec + target, write grad) beside it.
    fft_flops = 0.0
    for s_ in shapes.scales:
        hop = int(s_ * (1 - shapes.overlap))
        fft_flops += 1.5 * (1 + N // hop) * 5.0 * s_ * math.log2(s_)
    fft_flops *= B
    # shared-memory bytes the transform needs (DESIGN 3.4): 16 B per point and Stockham exchange (forward: two lanes of
    # a 16 B entry = 8 B per frame sample and direction), mirror exchange 8, gradient exchange 4, inverse at half the
    # forward's count, overlap-add carry and run heads in thread-private strips 3
    smem_bytes = 0.0
    for s_ in shapes.scales:
        hop = int(s_ * (1 - shapes.overlap))
        stages = 2 if s_ <= 256 else 3
        per_point = 16 * (stages - 1) + 8 + 4 + 8 * (stages - 1) + 3
        smem_bytes += (1 + N // hop) * s_ * per_point
    smem_bytes *= B
    smem_peak = 148 * 128 * clk / 1e9                 # GB/s: 128 B per clock per SM
    ms = event_time(lambda: ops.mss_loss_fwd(i["target"], sig2, list(shapes.scales), shapes.overlap, windows, True), 20, 3, flush)
    rows.append({"kernel": "K4L mss_loss fwd+grad (all scales in one launch + finalize + combine)", "ms": ms, "bound": "fp32",
                 "achieved": fft_flops / (ms * 1e-3) / 1e12, "peak": 2 * fma_peak / 1e12, "unit": "TFLOP/s",
                 "frac": fft_flops / (ms * 1e-3) / (2 * fma_peak),
                 "note": "FFT butterflies only (5 n log2 n, 7.0 GFLOP/step at batch 64) against 2 x 128 lanes x 148 SMs x max clock",
                 "smem": {"achieved": smem_bytes / (ms * 1e-3) / 1e9, "peak": smem_peak, "unit": "GB/s",
                          "frac": smem_bytes / (ms * 1e-3) / 1e9 / smem_peak,
                          "note": "shared-memory bytes of the Stockham exchanges, the mirror exchanges and the overlap-add carry "
                                  "against 128 B/clk/SM; the transform phases run at 76 % of it (DESIGN 3.4), the bin maths and "
                                  "sample loads do not overlap with them"},
                 "hbm": {"achieved": 4 * 3 * B * N / (ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                         "frac": 4 * 3 * B * N / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                         "note": "SURVEY 8d's HBM view: read rec + target, write grad (12 B per sample)"}})
    add("K0 harmonic_controls_fwd (standalone op; inside K1's launch in the step)", lambda: ops.harmonic_controls_fwd(i["amp_raw"], i["dist_raw"], i["pitch"], sr, True),
        alg_bytes=4 * B * T * (2 * H + 3))
    return rows


DUMP_BYTES = 60 << 20          # array data of --dump-outputs: with the .npy headers, under 64 MB in all


def step_outputs(step):
    """What a caller of SynthStep.run() receives: the audio, the loss and the gradient of every leaf."""
    leaves = ("amp_raw", "dist_raw", "mag_raw", "reverb_noise", "reverb_decay", "reverb_wet")
    return {"signal": step.signal, "loss": step.loss, **{"grad_" + n: g for n, g in zip(leaves, step.grads)}}


def dump_outputs(out_dir, outputs, batch):
    """Writes each output as out_dir/<name>.npy in float32.  Past DUMP_BYTES the per-voice outputs keep the same fixed,
    seeded subset of voices, whose indices go to voices.npy."""
    import numpy as np
    arrays = {k: v.detach().float().cpu().numpy() for k, v in outputs.items()}
    per_voice = [k for k in ("signal", "grad_amp_raw", "grad_dist_raw", "grad_mag_raw") if k in arrays]
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_BYTES:
        voice_bytes = sum(arrays[k].nbytes for k in per_voice) // batch
        keep = (DUMP_BYTES - total + voice_bytes * batch - 8 * batch) // voice_bytes
        assert keep >= 1, "a single voice's outputs exceed the dump budget"
        idx = np.sort(np.random.default_rng(0).choice(batch, keep, replace=False))
        arrays = {k: a[idx] if k in per_voice else a for k, a in arrays.items()}
        arrays["voices"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def parity_check(step, shapes, host, dev):
    """This run against the float64 oracle, outside the timed region: (a) the first two voices of the benchmark-shape
    step's audio, (b) a two-voice step (same kernels, same reverb) for audio, loss and the reverb-parameter gradients."""
    from oracle import ddsp_oracle as orc
    from ddsp_pytorch_b200.hotpath import SynthShapes, SynthStep
    n = min(2, shapes.batch)
    rp = {k: v.detach().double().cpu() for k, v in step.reverb.state_dict().items()}
    d = {k: v[:n].double() for k, v in host.items()}
    out = orc.synth_chain(d["amp_raw"], d["dist_raw"], d["mag_raw"], d["pitch"], d["noise"], shapes.block_size,
                          shapes.sample_rate, rp)
    ref_sig = out["signal"]
    with step.local_only():                      # this check runs on rank 0 alone: no collective
        step.run()
    torch.cuda.synchronize()
    audio_bench = float((step.signal[:n].detach().double().cpu() - ref_sig).abs().max())
    small = SynthShapes(**{**shapes.__dict__, "batch": n})
    s2 = SynthStep(small, dev, reverb_state=step.reverb.state_dict())
    s2.load_inputs({k: v[:n].contiguous() for k, v in host.items()}, non_blocking=False)
    s2.run()
    torch.cuda.synchronize()
    ref_loss = float(orc.mss_loss(d["target"], ref_sig.squeeze(-1), list(shapes.scales), shapes.overlap))
    return {"against": "float64 oracle (oracle/ddsp_oracle.py), 2-voice slice of the benchmark inputs",
            "audio_max_abs_bench_shape": audio_bench,
            "audio_max_abs_2_voices": float((s2.signal.detach().double().cpu() - ref_sig).abs().max()),
            "audio_peak": float(ref_sig.abs().max()),
            "loss_rel_2_voices": abs(float(s2.loss) - ref_loss) / abs(ref_loss),
            "tolerance": {"audio_max_abs": 1e-4, "loss_rel": 1e-5},
            "ok": bool(audio_bench <= 1e-4 and abs(float(s2.loss) - ref_loss) <= 1e-5 * abs(ref_loss))}


def other_configs(dev):
    """The other BASELINE.json configurations, measured in this process (rank 0, one GPU)."""
    from ddsp_pytorch_b200 import workloads as W
    out = {}
    for name, fn in (("model_step", lambda: W.model_step(64)), ("fwd_b16", W.forward_b16), ("realtime", W.realtime_latency),
                     ("autoencoder", lambda: W.model_step(16, autoencoder=True)), ("bulk_render", lambda: W.bulk_render(256, 128))):
        try:
            out[name] = fn()
        except Exception as e:                       # a sub-measurement must not lose the headline line
            out[name] = {"error": f"{type(e).__name__}: {e}"}
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
    return out


def init_dist(world, dev):
    if world <= 1:
        return None
    # keep stdout to the single JSON line: NCCL writes its version banner (and, at INFO, its topology lines) to
    # stdout unless it is given a file; whoever asked for NCCL_DEBUG output still gets it, on stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"            # level VERSION prints the banner to stdout whatever the file
    import torch.distributed as dist
    dist.init_process_group("nccl", device_id=dev)
    return dist


def run_bulk(args, rank, world):
    """configs[3]: every rank renders its own `bulk-voices` voices, forward only; weak scaling, no collective."""
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = init_dist(world, dev)
    import ctypes
    import ddsp_pytorch_b200  # noqa: F401
    from ddsp_pytorch_b200._lib import core_library
    from ddsp_pytorch_b200.workloads import BulkRenderer
    lib = core_library()
    lib.ddsp_b200_launch_count.restype = ctypes.c_uint64
    chunk = 128
    voices = args.bulk_voices
    r = BulkRenderer(chunk, dev, seed=100 + rank)
    c0 = lib.ddsp_b200_launch_count()
    r.render(voices)
    launches = int(lib.ddsp_b200_launch_count() - c0)

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    steps = args.steps
    for _ in range(min(args.warmup, 3)):
        r.render(voices)
    barrier()
    with ClockSampler(local) as clocks:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            r.render(voices)                  # 1024 voices x 768 KB of output each: far larger than L2
        b.record()
        barrier()
    tt = torch.tensor([a.elapsed_time(b)], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    total_ms = float(tt)
    samples = voices * world * r.N
    # end to end: frame-rate controls from pinned host memory per chunk, rendered audio back to pinned host memory
    hin = {k: v.pin_memory() for k, v in r.host.items() if k != "target" and k != "noise"}
    hout = torch.empty(chunk, r.N, pin_memory=True)
    h2d = sum(v.numel() * 4 for v in hin.values())

    def e2e_once():
        for _ in range(voices // chunk):
            for k, v in hin.items():
                r.inp[k].copy_(v, non_blocking=True)
            hout.copy_(r.render_chunk(), non_blocking=True)
        torch.cuda.synchronize()

    e2e_once()
    barrier()
    t0 = time.perf_counter()
    e2e_once()
    barrier()
    te = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    if rank == 0:
        peaks = load_peaks()
        clk = (peaks.get("sm_max_mhz") or 1965.0) * 1e6
        hs = voices * r.N * r.H
        ms_h = event_time(lambda: torch.ops.ddsp_b200.harmonic_fwd(
            r.inp["pitch"], torch.ops.ddsp_b200.harmonic_controls_fwd(r.inp["amp_raw"], r.inp["dist_raw"], r.inp["pitch"],
                                                                      float(r.SR), True)[2], r.BS, float(r.SR), None), 5, 2)
        line = {"metric": "DDSP synth audio samples/sec (fwd)", "value": samples * steps / (total_ms * 1e-3), "unit": UNIT,
                "n_gpus": world, "steps": steps, "warmup": min(args.warmup, 3), "ms_per_step": total_ms / steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": {"workload": BULK_NAME, "voices_per_gpu": voices, "chunk": chunk, "samples_per_voice": r.N,
                           "parallelism": f"voices sharded x{world}, no collective", "l2": "outputs of one step (786 MB) exceed L2"},
                "e2e": {"value": samples / float(te), "unit": UNIT, "h2d_bytes_per_step": h2d * (voices // chunk) * world,
                        "d2h_bytes_per_step": 4 * voices * r.N * world, "ms_per_step": 1e3 * float(te)},
                "gpu_launches": launches,
                "roofline": {"kernel": "K1 harmonic_frames_fwd (one chunk incl. controls)", "bound": "fp32",
                             "achieved": 2 * chunk * r.N * r.H / (ms_h * 1e-3) / 1e12, "peak": 148 * 128 * clk / 1e12, "unit": "TFMA/s",
                             "frac": 2 * chunk * r.N * r.H / (ms_h * 1e-3) / (148 * 128 * clk), "traffic": None, "ms": ms_h,
                             "note": "SURVEY 8d: 2 FMA per harmonic-sample against 148 SMs x 128 lanes x max clock"},
                "harmonic_samples_per_s": hs * world * steps / (total_ms * 1e-3), "clocks": clocks.summary()}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def run_b200(args, rank, world):
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = init_dist(world, dev)

    import ddsp_pytorch_b200  # noqa: F401  (fails loudly without the native libraries)
    from ddsp_pytorch_b200._lib import core_library
    from ddsp_pytorch_b200.hotpath import SynthShapes, SynthStep, synthetic_inputs
    import ctypes
    lib = core_library()
    lib.ddsp_b200_launch_count.restype = ctypes.c_uint64

    w = dict(WORKLOAD)
    w["batch"] = args.global_batch
    assert w["batch"] % world == 0, "the global batch must divide over the GPUs"
    w["batch"] //= world
    shapes = SynthShapes(**w)
    torch.manual_seed(0)
    step = SynthStep(shapes, dev)
    host_cpu = synthetic_inputs(shapes, seed=100 + rank)
    host = {k: v.pin_memory() for k, v in host_cpu.items()}
    h2d = step.load_inputs(host)
    torch.cuda.synchronize()

    # parameter gradients (reverb.noise/decay/wet) are averaged across ranks: the only collective
    params = list(step.reverb.parameters())
    n_param = sum(p.numel() for p in params)

    c0 = lib.ddsp_b200_launch_count()
    step.run()
    launches = int(lib.ddsp_b200_launch_count() - c0)
    use_graph = not args.no_graph
    graph_note = "CUDA graph replay"
    if dist is not None:
        # the reverb's backward comes first; its packed parameter gradients are averaged by one NCCL all-reduce on a
        # communication stream, a node of the same graph, while the synthesisers' backward runs
        step.enable_grad_allreduce(dist, in_step=not args.allreduce_outside)
        graph_note += (" + one eager NCCL all-reduce (AVG) launch on the packed parameter gradients" if args.allreduce_outside
                       else ", the NCCL all-reduce (AVG) of the packed parameter gradients is a node of the graph, "
                            "overlapped with the synthesisers' backward")
    outputs = None                                  # the captured step's output buffers, rewritten by every replay
    if use_graph:
        try:
            step.capture(forward_only=False)
            outputs = step_outputs(step)
            step.capture(forward_only=True)
        except Exception as e:                      # stay measurable: fall back to eager launches
            use_graph = False
            outputs = None
            graph_note = f"eager (graph capture failed: {type(e).__name__})"
            torch.cuda.synchronize()
    else:
        graph_note = "eager"
    run_step = (lambda: step.replay()) if use_graph else step.run
    run_fwd = (lambda: step.replay(True)) if use_graph else step.run_forward

    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB of L2
    flush = lambda: flush_buf.zero_()

    def full_step():
        run_step()
        step.allreduce_grads()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        flush()
        full_step()
    barrier()
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    with ClockSampler(local) as clocks:
        t_wall = time.perf_counter()
        for k in range(args.steps):
            flush()
            starts[k].record()
            full_step()
            ends[k].record()
        barrier()
        t_wall = time.perf_counter() - t_wall
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outputs if outputs is not None else step_outputs(step), shapes.batch)
    total_ms = sum(a.elapsed_time(b) for a, b in zip(starts, ends))
    tt = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    total_ms = float(tt)
    samples_per_step = args.global_batch * shapes.samples           # whole job, all ranks
    value = samples_per_step * args.steps / (total_ms * 1e-3)

    # forward only (the "fwd" half of the metric)
    fwd_ms = event_time(run_fwd, args.steps, 3, flush)
    tf = torch.tensor([fwd_ms], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(tf, op=dist.ReduceOp.MAX)
    fwd_ms = float(tf)

    # end to end through the public API with HOST buffers: every step's inputs travel from pinned host memory into
    # the idle one of two static input sets (copy engine, while the previous step computes), the step is one graph
    # launch on that set, and its loss is read back to the host (the read of step k is waited for after step k+1 has
    # been queued, so the host never stalls the device).  Falls back to the staged variant without graphs.
    barrier()
    e2e_steps = args.steps
    hosts = [host, {k: v.clone().pin_memory() for k, v in host.items()}]
    paired = use_graph
    link = None
    if paired:
        step.capture_pair(sets=args.e2e_sets)
        with near_gpu(dev):                                 # first touch on the GPU's NUMA node
            hosts = [step.pack_host(h) for h in hosts]      # one pinned block per batch: one H2D copy per step
        link = h2d_rate(hosts[0], step, flush)

    fed_bytes = [h2d]

    def e2e_loop(n):
        last = 0.0
        if paired:
            # up to sets - 1 batches are in flight ahead of the running step; the loss of a step is read sets - 1 steps
            # after it was queued (the host never stalls the device, the device never waits for the host's next call)
            from collections import deque
            ahead = args.e2e_sets - 1
            pending, fed = deque(), 0
            while fed < min(ahead, n):
                fed_bytes[0] = step.feed(hosts[fed & 1])
                fed += 1
            for k in range(n):
                cur = step.step_fed()
                step.allreduce_grads()
                step.loss_to_host(cur)
                if fed < n:
                    step.feed(hosts[fed & 1])                    # H2D of a later batch, overlapped
                    fed += 1
                pending.append(cur)
                if len(pending) > ahead:
                    last = step.read_loss(pending.popleft())     # D2H of an earlier step's result
            while pending:
                last = step.read_loss(pending.popleft())
            return last
        step.prefetch(hosts[0])
        for k in range(n):
            step.step_prefetched()
            step.allreduce_grads()
            step.prefetch(hosts[(k + 1) & 1])
            last = float(step.loss.detach())
        return last

    # three timed loops of e2e_steps steps each, the median is reported (the host link's share of a step differs from
    # loop to loop on some boxes; all three are kept in the JSON)
    e2e_loop(3)
    loop_s = []
    for _ in range(3):
        barrier()
        t0 = time.perf_counter()
        loss_host = e2e_loop(e2e_steps)
        barrier()
        tl = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(tl, op=dist.ReduceOp.MAX)
        loop_s.append(float(tl))
    te = torch.tensor([sorted(loop_s)[1]], device=dev, dtype=torch.float64)
    e2e_value = samples_per_step * e2e_steps / float(te)

    if rank == 0:
        peaks = load_peaks()
        kernels, roof = [], None
        if not args.skip_kernels:
            kernels = kernel_table(step, shapes, flush, peaks)
            top = max(kernels, key=lambda r: r["ms"])
            traffic, tnote = ncu_traffic("K4L" if top["kernel"].startswith("K4L") else top["kernel"])
            roof = {"kernel": top["kernel"], "bound": top["bound"], "achieved": top["achieved"], "peak": top["peak"],
                    "unit": top["unit"], "frac": top["frac"], "traffic": traffic, "ms": top["ms"],
                    "peak_source": ("148 SMs x 128 FP32 lanes x 2 flop x max SM clock (MEASURED_PEAKS.json has no FP32 entry; "
                                    "tools/probes/fp32_pace_probe.cu measured 120 of 128 lanes/clk/SM)") if top["bound"] == "fp32"
                    else peaks["source"]}
            if tnote:
                roof["traffic_note"] = tnote
            if "hbm" in top:
                roof["hbm"] = top["hbm"]
            if "smem" in top:
                roof["smem"] = top["smem"]
        parity = None
        if not args.skip_parity:
            try:
                parity = parity_check(step, shapes, host_cpu, dev)
            except Exception as e:
                parity = {"error": f"{type(e).__name__}: {e}", "ok": False}
        cpu = None
        if world == 1 and not args.skip_cpu:
            arm = CpuArm(args.cpu_batch)
            times = arm.time(3, 1)
            best = min(times)
            cpu = {"value": args.cpu_batch * arm.shapes.samples / best, "unit": UNIT, "cores": arm.cores, "kind": arm.kind,
                   "sample": f"{args.cpu_batch} of 64 voices, same shapes, float32 torch CPU, best of 3 ("
                             + ("unmodified reference from oracle/_ref" if arm.kind == "reference" else "oracle port") + ")",
                   "ms_per_sample_step": best * 1e3}
        configs = None
        if world == 1 and not args.skip_configs:
            configs = other_configs(dev)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD_NAME, "global_batch": args.global_batch, "per_gpu_batch": shapes.batch,
                       "samples_per_voice": shapes.samples, "parallelism": f"voices sharded x{world}, NCCL "
                       f"all-reduce of {n_param} reverb-parameter grads" if world > 1 else "single GPU",
                       "l2": "256 MiB memset between timed steps (outside the event pairs)",
                       "launch": graph_note},
            "fwd": {"value": samples_per_step / (fwd_ms * 1e-3), "unit": UNIT, "ms_per_step": fwd_ms},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": fed_bytes[0] * world, "d2h_bytes_per_step": 4 * world,
                    "ms_per_step": 1e3 * float(te) / e2e_steps, "loss": loss_host, "h2d_link": link,
                    "loops_ms_per_step": [1e3 * t / e2e_steps for t in loop_s], "steps_per_loop": e2e_steps,
                    "how": f"pinned host -> H2D on the copy stream straight into an idle one of {args.e2e_sets} static input sets "
                           f"({args.e2e_sets - 1} batches in flight ahead of the step) -> one graph launch per step -> loss D2H read "
                           f"every step (waited for {args.e2e_sets - 1} steps later); wall clock between synchronisations, median of three loops"},
            "gpu_launches": launches, "roofline": roof, "parity": parity, "kernels": kernels, "cpu_baseline": cpu,
            "configs": configs, "clocks": clocks.summary(), "wall_s_timed_loop": t_wall,
        }
        print(json.dumps(line), flush=True)
    if dist is not None:
        step.release_graphs()                        # the graphs hold NCCL nodes: they go before the communicator
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device: there is no CPU fallback for the kernels")
    if args.workload == "bulk":
        run_bulk(args, rank, world)
    else:
        run_b200(args, rank, world)


if __name__ == "__main__":
    main()
