"""Streaming reverb kernel (csrc/conv_stream.cu) against the composition of existing kernels that computes the same
buffer: fftconv_fwd(cat([history, x]), h)[..., L-1:] with history_out = cat(...)[..., N:] (both slices are views, no
copy is charged to the composition).  CUDA events around 50 back-to-back calls, blocks of the two alternating, median
of the blocks.  Inputs are reused across calls: L2 is warm.  That is the realistic case: a realtime working set (the
impulse, the history and one buffer, under 1 MB at 1 x 1024 x 48000) stays in the 126 MB L2 from one buffer to the
next.  Each shape is also checked: both results against each other, relative to the output's peak.

    python tools/run_conv_stream.py [--out FILE]           one JSON line per shape, plus a header line
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ddsp_pytorch_b200  # noqa: E402,F401

ops = torch.ops.ddsp_b200
CALLS, BLOCKS = 50, 12


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def time_block(fn):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(CALLS):
        fn()
    stop.record()
    stop.synchronize()
    return start.elapsed_time(stop) * 1e3 / CALLS          # us per call


def run(B, N, L):
    g = torch.Generator().manual_seed(B * 7 + N + L)
    x = torch.randn(B, N, generator=g).cuda()
    h = (torch.randn(L, generator=g) * torch.exp(-torch.arange(L) / (L / 4))).cuda()
    hist = torch.randn(B, L - 1, generator=g).cuda()
    h2 = h.view(1, L)

    def stream():
        return ops.conv_stream_fwd(x, h, hist)

    def composed():
        u = torch.cat([hist, x], 1)
        return ops.fftconv_fwd(u, h2, False)[0][:, L - 1:], u[:, N:]

    ys, hs = stream()
    yc, hc = composed()
    peak = float(yc.abs().max())
    agree = float((ys - yc).abs().max()) / peak
    assert torch.equal(hs, hc) and agree < 1e-4, (B, N, L, agree)
    for _ in range(5):
        stream(), composed()
    torch.cuda.synchronize()
    ts, tc = [], []
    for _ in range(BLOCKS):
        ts.append(time_block(stream))
        tc.append(time_block(composed))
    ts.sort(), tc.sort()
    s_us, c_us = ts[BLOCKS // 2], tc[BLOCKS // 2]
    return {"B": B, "N": N, "L": L, "stream_us": round(s_us, 2), "composed_us": round(c_us, 2),
            "speedup": round(c_us / s_us, 2), "stream_gfma_per_s": round(B * N * L / s_us / 1e3, 1),
            "stream_spread_us": [round(ts[0], 2), round(ts[-1], 2)],
            "composed_spread_us": [round(tc[0], 2), round(tc[-1], 2)], "max_rel_diff": agree}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "run_conv_stream.py measures on the GPU"
    lines = [dict(card(), l2="warm (inputs reused across calls; the realtime working set stays in L2)",
                  calls_per_block=CALLS, blocks=BLOCKS,
                  composed="cat([history, x]) + fftconv_fwd (kernel spectrum included, as in the realtime export)")]
    for L in (16000, 48000):
        for B in (1, 8):
            for N in (256, 1024, 4096):
                lines.append(run(B, N, L))
    text = "\n".join(json.dumps(line) for line in lines)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
