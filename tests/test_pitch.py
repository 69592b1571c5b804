"""Dataset pitch by YIN: csrc/pitch.cu, its C ABI, the torch op, ``core.extract_pitch_yin`` and
``tools/extract_features.py --pitch``.  The GPU results are held against a float64 numpy oracle written here from the
definition (librosa.yin with the frames of the loudness: reflect padding of L/2, window W = L/2, the difference
function by its direct sum, the cumulative mean normalisation, the threshold / global-minimum decision and the
parabolic shift).

YIN's decisions are discontinuous: a lag is chosen by comparisons of y against the threshold and its neighbours, and
a float32 computation may take the other branch wherever the oracle's margin is tiny.  So the parity test compares
only *decided* frames, whose decisions keep a margin of DELTA in the oracle (DELTA is far above the float32 error of
y, ~1e-6), and asserts how many frames that is."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOOL = os.path.join(ROOT, "tools", "extract_features.py")
FLT_MIN = float(np.finfo(np.float32).tiny)
DELTA = 1e-4
FMIN, FMAX, THRESHOLD = 50.0, 2000.0, 0.1


@pytest.fixture(scope="module")
def pkg():
    import ddsp_pytorch_b200
    return ddsp_pytorch_b200


# ---------------------------------------------------------------------------------------------------- oracle
def periods(sr, fmin, fmax, L):
    return max(int(np.floor(sr / fmax)), 1), min(int(np.ceil(sr / fmin)), L - L // 2 - 1)


def frames_of(x, L, hop):
    """(N,) -> (N // hop, L): the signal reflect-padded by L/2, frame f = padded[f hop : f hop + L]"""
    p = np.pad(np.asarray(x, np.float64), L // 2, mode="reflect")
    return p[np.arange(len(x) // hop)[:, None] * hop + np.arange(L)[None, :]]


def diff_direct(fr, pmax):
    """d(tau) = sum_{j=1..W} (x[j] - x[j+tau])^2, tau = 0 .. pmax, float64"""
    W = fr.shape[1] // 2
    a = fr[:, 1:W + 1]
    d = np.empty((fr.shape[0], pmax + 1))
    for tau in range(pmax + 1):
        e = a - fr[:, 1 + tau:W + 1 + tau]
        d[:, tau] = np.einsum("ij,ij->i", e, e)
    return d


def diff_fft(fr, pmax):
    """librosa 0.10's form of the same: E(0) + E(tau) - 2 acf(tau), by FFTs and cumulative sums, float64"""
    L = fr.shape[1]
    W = L // 2
    a = np.fft.rfft(fr, L, axis=-1)
    b = np.fft.rfft(fr[:, W:0:-1], L, axis=-1)
    acf = np.fft.irfft(a * b, L, axis=-1)[:, W:]
    en = np.cumsum(fr ** 2, axis=-1)
    en = en[:, W:] - en[:, :-W]
    return (en[:, :1] + en - 2 * acf)[:, :pmax + 1]


def normalised(d, pmin, pmax):
    """y(tau), tau = pmin .. pmax"""
    cm = np.cumsum(d[:, 1:pmax + 1], axis=1) / np.arange(1, pmax + 1)
    return d[:, pmin:pmax + 1] / (cm[:, pmin - 1:pmax] + FLT_MIN)


def choose(y, thr):
    """index into the lag range of the first trough below thr, else of the first global minimum; and whether a
    trough was found"""
    tr = np.zeros_like(y, bool)
    tr[:, 1:-1] = (y[:, 1:-1] < y[:, :-2]) & (y[:, 1:-1] <= y[:, 2:])
    tr[:, 0] = y[:, 0] < y[:, 1]
    tt = tr & (y < thr)
    found = tt.any(1)
    return np.where(found, tt.argmax(1), y.argmin(1)), found


def oracle(x, sr, L, hop, fmin=FMIN, fmax=FMAX, thr=THRESHOLD):
    """one row (N,) -> dict of f0, aperiodicity, integer lag, parabolic shift and the decided mask, per frame"""
    pmin, pmax = periods(sr, fmin, fmax, L)
    y = normalised(np.maximum(diff_direct(frames_of(x, L, hop), pmax), 0.0), pmin, pmax)
    idx, found = choose(y, thr)
    n = y.shape[1]
    r = np.arange(len(idx))
    shift = np.zeros(len(idx))
    inner = (idx > 0) & (idx < n - 1)
    i, ri = idx[inner], r[inner]
    a = y[ri, i + 1] + y[ri, i - 1] - 2 * y[ri, i]
    b = (y[ri, i + 1] - y[ri, i - 1]) / 2
    shift[inner] = np.where(np.abs(b) >= np.abs(a), 0.0, -b / np.where(a == 0, 1.0, a))
    # decided: the lag does not move with the threshold by +-DELTA, no two neighbouring y up to lag + 1 are within
    # DELTA of each other, and on the global-minimum path the runner-up is more than DELTA above the minimum
    lo, _ = choose(y, thr - DELTA)
    hi, _ = choose(y, thr + DELTA)
    decided = (lo == idx) & (hi == idx)
    for f in range(len(idx)):
        if np.abs(np.diff(y[f, :idx[f] + 2])).min() <= DELTA:
            decided[f] = False
        if not found[f]:
            s = np.sort(y[f])
            decided[f] &= s[1] - s[0] > DELTA
    lag = pmin + idx
    return dict(f0=sr / (lag + shift), ap=y[r, idx], lag=lag, shift=shift, decided=decided)


def tone_signal(B, N, sr, seed, floor=True):
    """harmonic tones with envelopes, an exactly silent stretch and, unless floor=False, a -60 dB noise floor outside
    the silence (the signals of test_features.py)"""
    rng = np.random.default_rng(seed)
    t = np.arange(N) / sr
    x = np.zeros((B, N))
    for b in range(B):
        f0 = rng.uniform(80, 900)
        env = 0.05 + 0.45 * (0.5 + 0.5 * np.sin(2 * np.pi * rng.uniform(0.5, 3) * t + rng.uniform(0, 6.28)))
        tone = sum(np.sin(2 * np.pi * k * f0 * t + rng.uniform(0, 6.28)) / k for k in range(1, 12) if k * f0 < sr / 2)
        x[b] = env * tone / 3
        if floor:
            x[b] += 1e-3 * rng.standard_normal(N)
        s0 = int(rng.uniform(0.3, 0.5) * N)
        x[b, s0:s0 + N // 4] = 0.0
    return x.astype(np.float32)


def steady_tones(f0s, N, sr, seed):
    """steady harmonic tones (1/k amplitudes up to Nyquist), no silence, a -60 dB floor"""
    rng = np.random.default_rng(seed)
    t = np.arange(N) / sr
    x = np.zeros((len(f0s), N))
    for b, f0 in enumerate(f0s):
        tone = sum(np.sin(2 * np.pi * k * f0 * t + rng.uniform(0, 6.28)) / k for k in range(1, 12) if k * f0 < sr / 2)
        x[b] = 0.3 * tone + 1e-3 * rng.standard_normal(N)
    return x.astype(np.float32)


def cents(a, b):
    return 1200 * np.abs(np.log2(np.asarray(a, np.float64) / np.asarray(b, np.float64)))


# ---------------------------------------------------------------------------------------------------- CPU
def test_direct_sum_equals_fft_form():
    """The oracle's direct sum is librosa's E(0) + E(tau) - 2 acf(tau): the window starts at frame sample 1."""
    rng = np.random.default_rng(3)
    for L, pmax in ((256, 127), (2048, 1023), (4096, 441)):
        fr = rng.standard_normal((6, L))
        d1, d2 = diff_direct(fr, pmax), diff_fft(fr, pmax)
        assert np.abs(d1 - d2).max() <= 1e-12 * np.abs(d1).max(), L


def test_argument_errors_do_not_need_a_gpu(pkg):
    from ddsp_pytorch_b200._lib import core_library
    lib = core_library()
    vp, i32, i64, f32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float
    fwd = lib.ddsp_b200_pitch_yin_fwd
    fwd.restype = i32
    fwd.argtypes = [vp, vp, vp, vp, i32, i64, i32, i32, i32, i32, f32, f32, vp]
    p = ctypes.c_void_p(0x1000)          # never dereferenced: the arguments are rejected before any launch
    ok = (2, 16000, 2048, 160, 8, 320, 16000.0, 0.1)     # B, N, L, hop, min_period, max_period, sr, threshold

    def call(ptrs, sizes=ok):
        return fwd(*ptrs, *sizes, None)

    for i in range(4):                                   # signal, stage twiddles, f0, aperiodicity
        ptrs = [p] * 4
        ptrs[i] = None
        assert call(ptrs) == -1, i
    bad = [(0, 16000, 2048, 160, 8, 320, 16000.0, 0.1), (65536, 16000, 2048, 160, 8, 320, 16000.0, 0.1),    # B
           (2, 1024, 2048, 160, 8, 320, 16000.0, 0.1), (2, 1 << 30, 2048, 160, 8, 320, 16000.0, 0.1),       # N
           (2, 16000, 2000, 160, 8, 320, 16000.0, 0.1), (2, 16000, 128, 16, 8, 50, 16000.0, 0.1),            # L
           (2, 16000, 8192, 160, 8, 320, 16000.0, 0.1),
           (2, 16000, 2048, 0, 8, 320, 16000.0, 0.1), (2, 16000, 2048, -3, 8, 320, 16000.0, 0.1),            # hop
           (2, 16000, 2048, 160, 0, 320, 16000.0, 0.1),                                                      # min_period
           (2, 16000, 2048, 160, 8, 1024, 16000.0, 0.1), (2, 16000, 256, 160, 8, 128, 16000.0, 0.1),         # max_period > L-W-1
           (2, 16000, 2048, 160, 8, 9, 16000.0, 0.1), (2, 16000, 2048, 160, 300, 200, 16000.0, 0.1),         # < min + 2
           (2, 16000, 2048, 160, 8, 320, 16000.0, float("nan")), (2, 16000, 2048, 160, 8, 320, 16000.0, float("inf"))]
    for sizes in bad:
        assert call([p] * 4, sizes) == -1, sizes


def test_op_registered_without_cpu_kernel(pkg):
    assert hasattr(torch.ops.ddsp_b200, "pitch_yin_fwd")
    with pytest.raises((RuntimeError, NotImplementedError)):
        torch.ops.ddsp_b200.pitch_yin_fwd(torch.zeros(1, 4000), 2048, 160, 8, 320, 16000.0, 0.1)
    with pytest.raises((RuntimeError, NotImplementedError)):
        pkg.extract_pitch_yin(torch.zeros(1, 4000), 16000, 160, FMIN, FMAX)


def test_extract_pitch_yin_is_exported_forward_only_and_checks_its_range(pkg):
    import inspect
    import ddsp
    assert "extract_pitch_yin" in pkg.core.__all__ and ddsp.extract_pitch_yin is pkg.core.extract_pitch_yin
    assert list(inspect.signature(pkg.extract_pitch_yin).parameters) == [
        "signal", "sample_rate", "block_size", "fmin", "fmax", "frame_length", "threshold"]
    x = torch.zeros(1, 4000, requires_grad=True)
    with pytest.raises(RuntimeError, match="no backward"):
        pkg.extract_pitch_yin(x, 16000, 160, FMIN, FMAX)
    z = torch.zeros(4000)
    for fmin, fmax in [(0.0, 2000.0), (-5.0, 2000.0), (300.0, 300.0), (500.0, 400.0), (50.0, 8000.5)]:
        with pytest.raises(ValueError):
            pkg.extract_pitch_yin(z, 16000, 160, fmin, fmax)
    with pytest.raises(ValueError, match="empty"):
        pkg.extract_pitch_yin(z, 16000, 160, 7000.0, 8000.0)             # lags 2 .. 3
    with pytest.raises(ValueError, match="empty"):
        pkg.extract_pitch_yin(z, 16000, 160, 100.0, 126.5, frame_length=256)   # lags 126 .. 127
    assert pkg.core._yin_periods(16000, FMIN, FMAX) == (8, 320)
    assert pkg.core._yin_periods(48000, FMIN, FMAX) == (24, 960)
    assert pkg.core._yin_periods(16000, 20.0, 2000.0, 1024) == (8, 511)


def test_oracle_on_a_tone():
    sr, L, hop = 16000, 2048, 160
    x = steady_tones([220.0], 16000, sr, seed=1)[0]
    o = oracle(x, sr, L, hop)
    mid = slice(L // 2 // hop + 1, -(L // 2 // hop + 1))
    assert cents(o["f0"][mid], 220.0).max() <= 1.0 and o["decided"][mid].all()


# ---------------------------------------------------------------------------------------------------- GPU
# (sr, L, hop, B, N, floor): N not a multiple of hop; B in {1, 3, 64}; the minimum share of decided frames
# (the oracle decides 77-84 % of the frames of these inputs)
PARITY = [
    (16000, 2048, 160, 3, 16077, True, 0.7),
    (16000, 2048, 160, 3, 16077, False, 0.7),
    (48000, 2048, 480, 1, 48100, True, 0.7),
    (22050, 4096, 441, 3, 22350, True, 0.7),
    (16000, 1024, 64, 64, 8005, True, 0.7),
]


@pytest.mark.gpu
@pytest.mark.parametrize("sr,L,hop,B,N,floor,share", PARITY)
def test_parity_on_decided_frames(pkg, sr, L, hop, B, N, floor, share):
    x = tone_signal(B, N, sr, seed=L + hop + B, floor=floor)
    f0, ap = pkg.extract_pitch_yin(torch.from_numpy(x).cuda(), sr, hop, FMIN, FMAX, frame_length=L)
    assert f0.shape == (B, N // hop) and ap.shape == (B, N // hop)
    f0, ap = f0.double().cpu().numpy(), ap.double().cpu().numpy()
    decided = total = 0
    worst_p = worst_ap = 0.0
    for b in range(B):
        o = oracle(x[b], sr, L, hop)
        m = o["decided"]
        per, per_o = sr / f0[b], sr / o["f0"]
        assert np.array_equal(np.rint(per[m] - o["shift"][m]).astype(int), o["lag"][m]), b
        if m.any():
            worst_p = max(worst_p, float(np.abs(per - per_o)[m].max()))
            worst_ap = max(worst_ap, float(np.abs(ap[b] - o["ap"])[m].max()))
        decided += int(m.sum())
        total += m.size
    print(f"\nsr {sr} L {L} hop {hop} B {B} floor {floor}: decided {decided} of {total}; "
          f"worst period diff {worst_p:.2e} samples, aperiodicity {worst_ap:.2e}")
    assert decided >= share * total, (decided, total)
    assert worst_p <= 2e-3 and worst_ap <= 1e-4, (worst_p, worst_ap)


@pytest.mark.gpu
@pytest.mark.parametrize("sr,L,fmin,fmax", [(16000, 2048, 50.0, 2000.0), (22050, 1024, 50.0, 1000.0),
                                            (48000, 256, 400.0, 8000.0)])
def test_all_zero_rows_closed_form(pkg, sr, L, fmin, fmax):
    pmin, _ = periods(sr, fmin, fmax, L)
    f0, ap = pkg.extract_pitch_yin(torch.zeros(3, 5000, device="cuda"), sr, 100, fmin, fmax, frame_length=L)
    assert f0.shape == (3, 50)
    assert (f0.cpu().numpy() == np.float32(sr / pmin)).all()
    assert (ap.cpu().numpy() == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("sr,L,hop", [(16000, 2048, 160), (48000, 2048, 480)])
def test_steady_tones_within_3_cents(pkg, sr, L, hop):
    """Against the true pitch, on frames at least L/2 from the ends: within 3 cents wherever the period is 20 samples
    or more.  Shorter periods are bounded by the definition, not the kernel: the parabola through y at three integer
    lags is off by up to 6.7 cents for 880 Hz at 16 kHz (an 18.2-sample period) in float64 too.  So every tone is
    also held to the float64 oracle, within 0.1 cents."""
    f0s = [80.0, 123.4, 196.0, 261.6, 333.3, 440.0, 555.0, 698.5, 880.0, 1000.0]
    N = sr
    x = steady_tones(f0s, N, sr, seed=sr)
    f0, _ = pkg.extract_pitch_yin(torch.from_numpy(x).cuda(), sr, hop, FMIN, FMAX, frame_length=L)
    f0 = f0.cpu().numpy()
    centre = np.arange(N // hop) * hop
    keep = (centre >= L // 2) & (centre + L // 2 <= N)                 # frames at least L/2 from the ends
    worst = worst_o = 0.0
    for b, f in enumerate(f0s):
        err = cents(f0[b, keep], f).max()
        err_o = cents(f0[b, keep], oracle(x[b], sr, L, hop)["f0"][keep]).max()
        if sr / f >= 20:
            worst = max(worst, err)
            assert err <= 3.0, (f, err)
        worst_o = max(worst_o, err_o)
        assert err_o <= 0.1, (f, err_o)
    print(f"\nsteady tones at {sr} Hz: {worst:.2f} cents from the truth (periods >= 20), {worst_o:.3f} from the oracle")


@pytest.mark.gpu
def test_synthetic_dataset_pitch(pkg, tmp_path):
    from ddsp_pytorch_b200.train import write_synthetic_dataset
    data = write_synthetic_dataset(tmp_path / "ds", 8, seconds=1.0)
    sig, truth = np.load(data / "signals.npy"), np.load(data / "pitchs.npy")
    f0, _ = pkg.extract_pitch_yin(torch.from_numpy(sig).cuda(), 16000, 160, FMIN, FMAX)
    assert f0.shape == truth.shape
    err = cents(f0.cpu().numpy()[:, 7:-7], truth[:, 7:-7])         # edge frames can be an octave off (reflection)
    print(f"\nsynthetic dataset: median {np.median(err):.2f} cents, max {err.max():.2f}")
    assert np.median(err) <= 15.0 and err.max() <= 30.0


@pytest.mark.gpu
@pytest.mark.parametrize("sr,L,hop", [(16000, 2048, 160), (16000, 256, 1), (22050, 4096, 441)])
def test_deterministic_and_independent_of_batch(pkg, sr, L, hop):
    x = torch.from_numpy(tone_signal(64, 6000 if hop == 1 else 24000, sr, seed=11)).cuda()
    fmin = 200.0 if L == 256 else FMIN
    f1, a1 = pkg.extract_pitch_yin(x, sr, hop, fmin, FMAX, frame_length=L)
    f2, a2 = pkg.extract_pitch_yin(x, sr, hop, fmin, FMAX, frame_length=L)
    assert torch.equal(f1, f2) and torch.equal(a1, a2)
    for lo, hi in ((0, 1), (37, 38), (63, 64), (5, 22)):
        fb, ab = pkg.extract_pitch_yin(x[lo:hi], sr, hop, fmin, FMAX, frame_length=L)
        assert torch.equal(fb, f1[lo:hi]) and torch.equal(ab, a1[lo:hi])
    fo, ao = pkg.extract_pitch_yin(x[37], sr, hop, fmin, FMAX, frame_length=L)       # (N,) input
    assert torch.equal(fo, f1[37]) and torch.equal(ao, a1[37])


@pytest.mark.gpu
def test_tool_writes_pitch_the_harness_reads(tmp_path):
    import json
    from ddsp_pytorch_b200 import core
    from ddsp_pytorch_b200.models.decoder import DDSPDecoder
    from ddsp_pytorch_b200.train import NpyDataset, write_synthetic_dataset
    data = write_synthetic_dataset(tmp_path / "ds", 8, seconds=1.0)
    cmd = [sys.executable, TOOL, "--data", str(data), "--sample-rate", "16000", "--block-size", "160", "--batch", "3",
           "--pitch"]
    refused = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert refused.returncode != 0 and "--overwrite" in refused.stderr
    res = subprocess.run(cmd + ["--overwrite"], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    rec = json.loads(res.stdout.strip().splitlines()[-1])
    assert rec["examples"] == 8 and rec["pitch_fmin"] == FMIN and rec["pitch_fmax"] == FMAX
    pitch = np.load(data / "pitchs.npy")
    assert pitch.shape == (8, 100) and pitch.dtype == np.float32
    assert not any(p.name.endswith(".partial.npy") for p in data.iterdir())
    sig = torch.from_numpy(np.load(data / "signals.npy")).cuda()
    assert np.array_equal(pitch, core.extract_pitch_yin(sig, 16000, 160, FMIN, FMAX)[0].cpu().numpy())
    ds = NpyDataset(data)
    batch = {k: v.cuda() for k, v in ds.batch(np.arange(8)).items()}
    assert torch.equal(batch["pitch"].reshape(8, 100).cpu(), torch.from_numpy(pitch))
    torch.manual_seed(0)
    model = DDSPDecoder(hidden_size=64, n_harmonic=16, n_bands=65, sample_rate=16000, block_size=160,
                        has_reverb=True).cuda()
    with torch.no_grad():
        out = model(batch)
    assert out["signal"].shape == (8, 100 * 160, 1) and torch.isfinite(out["signal"]).all()
