"""Feature kernel (csrc/features.cu) against the composed torch path that computes the same features on the same
device: torch.stft(center=True, pad_mode="reflect") with the periodic Hann window, then abs / log / A-weighting / mean
for the loudness, and power / mel matmul / dB / per-row top_db clamp / DCT matmul for the MFCC.  CUDA events around
back-to-back warm calls, blocks of the two alternating, median of the blocks.  Inputs are reused across calls (L2 is
warm where the signal fits in it: 16 MB at batch 64, not at 256 x 192 000 = 197 MB).  Each shape is also checked: the
two results against each other.  Last, the dataset tool's throughput (audio seconds per second, wall clock including
the memory-mapped reads and the .npy writes) on a 1024-example synthetic set of 4 s examples.

    python tools/run_features.py [--out profiles/features.json]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import ddsp_pytorch_b200  # noqa: E402,F401
from ddsp_pytorch_b200 import functions as F  # noqa: E402

ops = torch.ops.ddsp_b200
CALLS, BLOCKS = 20, 9
N_FFT, N_MFCC = 2048, 30
SHAPES = [(1, 64000, 16000, 160), (64, 64000, 16000, 160), (256, 192000, 48000, 480)]


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


def composed(x, sr, hop, window, a_weight, mel_dense, dct, mfcc=True):
    spec = torch.stft(x, N_FFT, hop, window=window, center=True, pad_mode="reflect", return_complex=True).abs()
    loud = (torch.log(spec + 1e-7) + a_weight[:, None]).mean(1)
    if not mfcc:
        return loud, None
    db = 10 * torch.log10((mel_dense @ spec.square()).clamp_min(1e-10))
    db = torch.maximum(db, db.amax((1, 2), keepdim=True) - 80)
    return loud, (dct @ db).transpose(1, 2)


def run(B, N, sr, hop):
    g = torch.Generator().manual_seed(B + N + hop)
    x = (0.3 * torch.randn(B, N, generator=g)).cuda()
    window, a_weight, mel, dct_t = F.feature_tables(sr, N_FFT, N_MFCC, x.device)
    mel_dense = torch.from_numpy(F.mel_filterbank(sr, N_FFT)).float().cuda()
    dct = torch.from_numpy(F.dct_matrix(N_MFCC)).float().cuda()
    fns = {
        "op": lambda: ops.features_fwd(x, window, a_weight, mel, dct_t, N_FFT, hop, True),
        "op_loudness_only": lambda: ops.features_fwd(x, window, a_weight, mel, dct_t, N_FFT, hop, False),
        "composed": lambda: composed(x, sr, hop, window, a_weight, mel_dense, dct),
        "composed_loudness_only": lambda: composed(x, sr, hop, window, a_weight, mel_dense, dct, False),
    }
    lo, mo = fns["op"]()
    lc, mc = fns["composed"]()
    d_loud, d_mfcc = float((lo - lc).abs().max()), float((mo - mc).abs().max())
    for fn in fns.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in fns}
    for _ in range(BLOCKS):
        for k, fn in fns.items():
            times[k].append(time_block(fn))
    med = {k: sorted(v)[BLOCKS // 2] for k, v in times.items()}
    frames = B * (1 + N // hop)
    return {"B": B, "N": N, "sample_rate": sr, "hop": hop, "n_fft": N_FFT, "n_mfcc": N_MFCC, "frames": frames,
            **{f"{k}_us": round(v, 1) for k, v in med.items()},
            "speedup": round(med["composed"] / med["op"], 2),
            "speedup_loudness_only": round(med["composed_loudness_only"] / med["op_loudness_only"], 2),
            "op_frames_per_us": round(frames / med["op"], 1),
            "op_spread_us": [round(min(times["op"]), 1), round(max(times["op"]), 1)],
            "composed_spread_us": [round(min(times["composed"]), 1), round(max(times["composed"]), 1)],
            "max_abs_diff_loudness": d_loud, "max_abs_diff_mfcc": d_mfcc}


def tool_throughput(n=1024):
    import extract_features
    from ddsp_pytorch_b200.train import write_synthetic_dataset
    with tempfile.TemporaryDirectory() as d:
        write_synthetic_dataset(d, n, seconds=4.0)
        extract_features.extract(d, 16000, 160, overwrite=True)                 # warm-up: module load, tables
        best = None
        for _ in range(3):
            rec = extract_features.extract(d, 16000, 160, overwrite=True)
            best = rec if best is None or rec["wall_s"] < best["wall_s"] else best
    return {"tool": "tools/extract_features.py --batch 256", "examples": n, "audio_seconds": best["audio_seconds"],
            "wall_s": best["wall_s"], "audio_seconds_per_s": best["audio_seconds_per_s"],
            "note": "best of 3 runs after one warm-up; page cache warm (the set was just written)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "run_features.py measures on the GPU"
    lines = [dict(card(), calls_per_block=CALLS, blocks=BLOCKS,
                  composed="torch.stft(center, reflect) + abs/log/A/mean; power, mel matmul, dB, per-row clamp, DCT matmul",
                  l2="inputs reused across calls: warm where the signal fits the 126 MB L2")]
    for shape in SHAPES:
        lines.append(run(*shape))
        print(json.dumps(lines[-1]), flush=True)
    lines.append(tool_throughput())
    text = "\n".join(json.dumps(line) for line in lines)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
