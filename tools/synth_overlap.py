#!/usr/bin/env python
"""Does the filtered noise run beside the oscillator bank?  The step of bench.py (batch 64) in three layouts:

  two_stream : FilteredNoiseFused on the side stream, HarmonicFromRaw on the current stream (the fallback layout)
  pair_k1    : SynthPair, the noise kernel as 1 persistent CTA per SM, the bank its programmatic dependent
  pair_k2    : the same with 2 noise CTAs per SM

1. Timing: full step and forward-only graph replays, CUDA events around each replay, the L2 overwritten (256 MiB
   memset) before each one as bench.py does; the layouts alternate round by round in one process.
2. Trace (a separate run, the profiler slows the host): torch.profiler over graph replays of each layout; per
   direction the start and end of the bank and noise kernels relative to the earlier of the two, and their overlap.

    python tools/synth_overlap.py [--rounds 5] [--steps 50] [--out profiles/synth_overlap.json]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

LAYOUTS = {"two_stream": None, "pair_k1": 1, "pair_k2": 2}
KERNELS = {"fwd": ("harmonic_frames_fwd_x2_kernel", "filtered_noise2_fwd_kernel"),
           "bwd": ("harmonic_frames_bwd_w_x2_kernel", "filtered_noise2_bwd_kernel")}


def make_steps(dev):
    from ddsp_pytorch_b200.hotpath import SynthShapes, SynthStep, synthetic_inputs
    sys.path.insert(0, ROOT)
    from bench import WORKLOAD
    shapes = SynthShapes(**WORKLOAD)
    host = {k: v.pin_memory() for k, v in synthetic_inputs(shapes, seed=100).items()}
    steps = {}
    for name, ctas in LAYOUTS.items():
        torch.manual_seed(0)
        st = SynthStep(shapes, dev)
        st._pair_ctas = ctas
        st.load_inputs(host)
        st.capture(forward_only=False)
        st.capture(forward_only=True)
        steps[name] = st
    return shapes, steps


def timed(fn, n, flush):
    ms = []
    for _ in range(n):
        flush()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return ms


def trace(steps, replays):
    from torch.profiler import ProfilerActivity, profile
    out = {}
    for name, st in steps.items():
        for _ in range(3):
            st.replay()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
            for _ in range(replays):
                st.replay()
                torch.cuda.synchronize()
        evs = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        res = {}
        for d, (bank_name, noise_name) in KERNELS.items():
            bank = sorted((e.time_range.start, e.time_range.end) for e in evs if bank_name in e.name)
            noise = sorted((e.time_range.start, e.time_range.end) for e in evs if noise_name in e.name)
            rows = []
            for (b0, b1), (n0, n1) in zip(bank, noise):
                t0 = min(b0, n0)
                ov = max(0.0, min(b1, n1) - max(b0, n0))
                rows.append({"bank_us": [b0 - t0, b1 - t0], "noise_us": [n0 - t0, n1 - t0], "overlap_us": ov,
                             "both_us": max(b1, n1) - t0, "overlap_of_noise": ov / max(n1 - n0, 1e-9)})
            if not rows:
                res[d] = {"error": f"no {bank_name} / {noise_name} kernels in the trace ({len(evs)} device events)"}
                continue
            mid = sorted(rows, key=lambda r: r["both_us"])[len(rows) // 2]
            res[d] = {"replays": len(rows), "median_replay": mid,
                      "overlap_of_noise_median": statistics.median(r["overlap_of_noise"] for r in rows)}
        out[name] = res
    return out


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--rounds", type=int, default=5)
    p.add_argument("--steps", type=int, default=50, help="timed replays per layout and round")
    p.add_argument("--replays", type=int, default=10, help="traced replays per layout")
    p.add_argument("--out", default=os.path.join(ROOT, "profiles", "synth_overlap.json"))
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("synth_overlap.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    import ddsp_pytorch_b200  # noqa: F401
    shapes, steps = make_steps(dev)
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    flush = flush_buf.zero_
    for st in steps.values():                                    # warm every graph
        timed(st.replay, 5, flush)
        timed(lambda: st.replay(True), 5, flush)
    rounds = {n: {"step_ms": [], "fwd_ms": []} for n in steps}
    for _ in range(args.rounds):
        for name, st in steps.items():
            rounds[name]["step_ms"].append(statistics.mean(timed(st.replay, args.steps, flush)))
            rounds[name]["fwd_ms"].append(statistics.mean(timed(lambda: st.replay(True), args.steps, flush)))
    timing = {n: {**r, "step_ms_median": statistics.median(r["step_ms"]), "fwd_ms_median": statistics.median(r["fwd_ms"]),
                  "step_spread_ms": max(r["step_ms"]) - min(r["step_ms"]),
                  "fwd_spread_ms": max(r["fwd_ms"]) - min(r["fwd_ms"])} for n, r in rounds.items()}
    traced = trace(steps, args.replays)
    props = torch.cuda.get_device_properties(dev)
    clocks = None
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(0)
        clocks = {"power_limit_w": pynvml.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0,
                  "sm_max_mhz": pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)}
    except Exception as e:                                       # the card name still identifies the run
        clocks = {"error": f"{type(e).__name__}: {e}"}
    res = {"gpu": props.name, **clocks, "workload": f"bench.py step, batch {shapes.batch}, graph replay",
           "how": f"{args.rounds} rounds x {args.steps} replays per layout, layouts alternating; mean per round, "
                  "median over rounds; L2 overwritten before every replay. Trace: torch.profiler, separate run, "
                  f"{args.replays} replays per layout, times in us from the earlier of the two kernels",
           "timing": timing, "trace": traced}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    for n in steps:
        t = timing[n]
        ov = {d: traced[n][d].get("overlap_of_noise_median") for d in KERNELS}
        print(f"{n:11s} step {t['step_ms_median']:.4f} ms (spread {t['step_spread_ms']:.4f})  fwd {t['fwd_ms_median']:.4f} ms "
              f"(spread {t['fwd_spread_ms']:.4f})  overlap/noise fwd {ov['fwd']} bwd {ov['bwd']}")


if __name__ == "__main__":
    main()
