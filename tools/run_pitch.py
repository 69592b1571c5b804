"""YIN pitch kernel (csrc/pitch.cu) against a float32 torch composition of the same definition on the same device:
reflect pad + ``unfold`` frames, ``rfft`` / ``irfft`` for the correlation, ``cumsum`` for the energies and the
cumulative mean, then the threshold / global-minimum decision and the parabolic shift in torch ops.  CUDA events
around back-to-back warm calls, blocks of the two alternating, median of the blocks.  Inputs are reused across calls
(L2 is warm where the signal fits in it: 16 MB at batch 64, not at 256 x 192 000 = 197 MB).

Each shape is also checked: the share of frames where the two float32 paths choose periods more than 0.01 samples
apart (a threshold or trough decision taken the other way; random inputs have many close calls) and the largest
period difference over the others.  The op's throughput is given as the FFT flops of its form (two L-point complex
transforms per frame, 5 L log2 L each) over its time, and as a share of the FP32 peak at the card's maximum SM clock
(148 SMs x 128 lanes x 2 flops per FMA).

    python tools/run_pitch.py [--out profiles/pitch.json]
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ddsp_pytorch_b200  # noqa: E402,F401
from ddsp_pytorch_b200 import core  # noqa: E402

ops = torch.ops.ddsp_b200
CALLS, BLOCKS = 20, 9
L, FMIN, FMAX, THRESHOLD = 2048, 50.0, 2000.0, 0.1
SHAPES = [(1, 64000, 16000, 160), (64, 64000, 16000, 160), (256, 192000, 48000, 480)]
FLT_MIN = torch.finfo(torch.float32).tiny


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def max_sm_clock_hz(rec):
    try:
        return float(rec["nvidia_smi"].split(",")[2].strip().split()[0]) * 1e6
    except (IndexError, ValueError):
        return float("nan")


def time_block(fn):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(CALLS):
        fn()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) * 1e3 / CALLS          # us per call


def composed(x, sr, hop, pmin, pmax):
    W = L // 2
    frames = F.pad(x[:, None], (W, W), mode="reflect")[:, 0].unfold(-1, L, hop)[:, :x.shape[1] // hop]
    acf = torch.fft.irfft(torch.fft.rfft(frames, L) * torch.fft.rfft(frames[..., 1:W + 1].flip(-1), L), L)
    en = torch.cumsum(frames.square(), -1)
    en = en[..., W:W + pmax + 1] - en[..., :pmax + 1]                     # E(tau), tau = 0 .. pmax
    d = (en[..., :1] + en - 2 * acf[..., W:W + pmax + 1]).clamp_min(0)
    cm = torch.cumsum(d[..., 1:], -1) / torch.arange(1, pmax + 1, device=x.device)
    y = d[..., pmin:] / (cm[..., pmin - 1:] + FLT_MIN)
    trough = torch.zeros_like(y, dtype=torch.bool)
    trough[..., 1:-1] = (y[..., 1:-1] < y[..., :-2]) & (y[..., 1:-1] <= y[..., 2:])
    trough[..., 0] = y[..., 0] < y[..., 1]
    cand = trough & (y < THRESHOLD)
    idx = torch.where(cand.any(-1), cand.to(torch.uint8).argmax(-1), y.argmin(-1))
    n = y.shape[-1]
    y0 = y.gather(-1, idx[..., None])[..., 0]
    yp = y.gather(-1, (idx + 1).clamp_max(n - 1)[..., None])[..., 0]
    ym = y.gather(-1, (idx - 1).clamp_min(0)[..., None])[..., 0]
    a, b = yp + ym - 2 * y0, (yp - ym) / 2
    inner = (idx > 0) & (idx < n - 1) & (b.abs() < a.abs())
    shift = torch.where(inner, -b / torch.where(inner, a, torch.ones_like(a)), torch.zeros_like(a))
    return sr / (pmin + idx + shift), y0


def run(B, N, sr, hop, peak):
    g = torch.Generator().manual_seed(B + N + hop)
    t = torch.arange(N, dtype=torch.float64) / sr
    f0 = 80 + 800 * torch.rand(B, 1, generator=g, dtype=torch.float64)
    tone = sum(torch.sin(2 * math.pi * k * f0 * t + 6.28 * torch.rand(B, 1, generator=g, dtype=torch.float64)) / k
               for k in range(1, 9))
    x = (0.3 * tone + 1e-3 * torch.randn(B, N, generator=g, dtype=torch.float64)).float().cuda()
    pmin, pmax = core._yin_periods(sr, FMIN, FMAX, L)
    fns = {
        "op": lambda: ops.pitch_yin_fwd(x, L, hop, pmin, pmax, float(sr), THRESHOLD),
        "composed": lambda: composed(x, sr, hop, pmin, pmax),
    }
    fo, _ = fns["op"]()
    fc, _ = fns["composed"]()
    dp = (sr / fo.double() - sr / fc.double()).abs()
    flips = dp > 1e-2
    for fn in fns.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in fns}
    for _ in range(BLOCKS):
        for k, fn in fns.items():
            times[k].append(time_block(fn))
    med = {k: sorted(v)[BLOCKS // 2] for k, v in times.items()}
    frames = B * (N // hop)
    flops = frames * 2 * 5 * L * math.log2(L)
    tflops = flops / (med["op"] * 1e-6) / 1e12
    return {"B": B, "N": N, "sample_rate": sr, "hop": hop, "frame_length": L, "fmin": FMIN, "fmax": FMAX,
            "periods": [pmin, pmax], "frames": frames,
            **{f"{k}_us": round(v, 1) for k, v in med.items()},
            "speedup": round(med["composed"] / med["op"], 2),
            "op_frames_per_us": round(frames / med["op"], 1),
            "op_fft_tflops": round(tflops, 2), "op_share_of_fp32_peak": round(tflops * 1e12 / peak, 3),
            "op_spread_us": [round(min(times["op"]), 1), round(max(times["op"]), 1)],
            "composed_spread_us": [round(min(times["composed"]), 1), round(max(times["composed"]), 1)],
            "frames_with_period_diff_above_0.01": int(flips.sum()),
            "max_period_diff_other_frames": float(dp[~flips].max()) if (~flips).any() else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "run_pitch.py measures on the GPU"
    head = dict(card(), calls_per_block=CALLS, blocks=BLOCKS,
                composed="reflect pad + unfold, rfft x rfft -> irfft, cumsum energies and mean, decision and "
                         "parabola in torch ops (float32)",
                l2="inputs reused across calls: warm where the signal fits the 126 MB L2")
    peak = 148 * 128 * 2 * max_sm_clock_hz(head)
    head["fp32_peak_tflops"] = round(peak / 1e12, 1)
    lines = [head]
    for shape in SHAPES:
        lines.append(run(*shape, peak))
        print(json.dumps(lines[-1]), flush=True)
    text = "\n".join(json.dumps(line) for line in lines)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
