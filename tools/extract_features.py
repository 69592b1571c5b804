"""Write the signal-processing features of a dataset from its signals, on the GPU.

A dataset directory in the reference's format holds ``signals.npy`` (n, N), ``pitchs.npy`` (n, T),
``loudness.npy`` (n, T) and ``mfccs.npy`` (n, T+1, n_mfcc), T = N // block_size (``ddsp/data.py:13-16``).  This tool
memory-maps ``signals.npy``, runs it through ``core.extract_features`` (csrc/features.cu) in batches and writes
``loudness.npy`` and ``mfccs.npy`` as float32, the layout ``train.NpyDataset`` reads.  With ``--pitch`` it also writes
``pitchs.npy`` (n, T) from the same batches, by YIN (``core.extract_pitch_yin``, csrc/pitch.cu) over fmin .. fmax;
without it ``pitchs.npy`` is left as it is.

    python tools/extract_features.py --data DIR --sample-rate 16000 --block-size 160 [--n-mfcc 30] [--batch 256]
                                     [--pitch [--fmin 50] [--fmax 2000]] [--overwrite]

Existing feature files are only replaced with ``--overwrite``.  Prints one JSON line: examples, audio seconds, wall
time, card name and power limit.
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
from ddsp_pytorch_b200 import core  # noqa: E402


def card() -> dict:
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True).stdout.strip().splitlines()
    except OSError:
        q = []
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def extract(data, sample_rate: int, block_size: int, n_mfcc: int = 30, batch: int = 256, overwrite: bool = False,
            n_fft: int = 2048, pitch: bool = False, fmin: float = 50.0, fmax: float = 2000.0) -> dict:
    """Compute and write ``loudness.npy`` / ``mfccs.npy`` (and ``pitchs.npy`` with ``pitch``) under ``data``; returns
    the JSON record."""
    if not torch.cuda.is_available():
        raise RuntimeError("extract_features runs on a CUDA device")
    names = ("loudness", "mfccs", "pitchs") if pitch else ("loudness", "mfccs")
    outs = {name: os.path.join(data, name + ".npy") for name in names}
    existing = [p for p in outs.values() if os.path.exists(p)]
    if existing and not overwrite:
        raise FileExistsError(f"{', '.join(existing)} exist; pass --overwrite to replace them")
    if pitch:
        core._yin_periods(sample_rate, fmin, fmax)             # a bad range fails before any file is opened
    signals = np.load(os.path.join(data, "signals.npy"), mmap_mode="r")
    if signals.ndim != 2:
        raise ValueError(f"signals.npy must be (examples, samples), got {signals.shape}")
    n, length = signals.shape
    frames = length // block_size
    dev = torch.device("cuda")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    # written to temporary names first, so that an interrupted run never leaves a half-written feature file behind
    tmp = {k: p + ".partial.npy" for k, p in outs.items()}
    loud_out = np.lib.format.open_memmap(tmp["loudness"], mode="w+", dtype=np.float32, shape=(n, frames))
    mfcc_out = np.lib.format.open_memmap(tmp["mfccs"], mode="w+", dtype=np.float32, shape=(n, frames + 1, n_mfcc))
    pitch_out = (np.lib.format.open_memmap(tmp["pitchs"], mode="w+", dtype=np.float32, shape=(n, frames))
                 if pitch else None)
    with torch.no_grad():
        for lo in range(0, n, batch):
            hi = min(n, lo + batch)
            x = torch.from_numpy(np.array(signals[lo:hi], dtype=np.float32)).pin_memory()
            xd = x.to(dev, non_blocking=True)
            loud, mfcc = core.extract_features(xd, sample_rate, block_size, n_mfcc=n_mfcc, n_fft=n_fft)
            loud_out[lo:hi] = loud.cpu().numpy()
            mfcc_out[lo:hi] = mfcc.cpu().numpy()
            if pitch:
                pitch_out[lo:hi] = core.extract_pitch_yin(xd, sample_rate, block_size, fmin, fmax)[0].cpu().numpy()
    for out in (loud_out, mfcc_out, pitch_out):
        if out is not None:
            out.flush()
    del loud_out, mfcc_out, pitch_out
    for k in outs:
        os.replace(tmp[k], outs[k])
    wall = time.perf_counter() - t0
    seconds = n * length / sample_rate
    return dict(card(), examples=n, audio_seconds=round(seconds, 3), wall_s=round(wall, 4),
                audio_seconds_per_s=round(seconds / wall, 1), sample_rate=sample_rate, block_size=block_size,
                n_mfcc=n_mfcc, n_fft=n_fft, batch=batch, **({"pitch_fmin": fmin, "pitch_fmax": fmax} if pitch else {}))


def main(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--data", required=True, help="dataset directory holding signals.npy")
    ap.add_argument("--sample-rate", type=int, required=True)
    ap.add_argument("--block-size", type=int, required=True, help="hop between frames, in samples")
    ap.add_argument("--n-mfcc", type=int, default=30)
    ap.add_argument("--batch", type=int, default=256, help="examples per call of the kernel")
    ap.add_argument("--pitch", action="store_true", help="also write pitchs.npy, by YIN")
    ap.add_argument("--fmin", type=float, default=50.0, help="lowest pitch YIN looks for, in Hz")
    ap.add_argument("--fmax", type=float, default=2000.0, help="highest pitch YIN looks for, in Hz")
    ap.add_argument("--overwrite", action="store_true", help="replace existing loudness.npy / mfccs.npy / pitchs.npy")
    a = ap.parse_args(argv)
    try:
        rec = extract(a.data, a.sample_rate, a.block_size, a.n_mfcc, a.batch, a.overwrite, pitch=a.pitch,
                      fmin=a.fmin, fmax=a.fmax)
    except FileExistsError as e:
        sys.exit(f"extract_features: {e}")
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
