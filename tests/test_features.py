"""Dataset features: A-weighted loudness and MFCCs from one pass of csrc/features.cu, its C ABI, the torch op,
``core.extract_loudness`` / ``core.extract_features`` and ``tools/extract_features.py``.  The GPU results are held
against a float64 numpy oracle written here from the formulas (reflect padding, ``np.fft.rfft``, librosa's
A-weighting, Slaney mel bands, power_to_db with top_db = 80 per row, DCT-II ortho)."""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOOL = os.path.join(ROOT, "tools", "extract_features.py")


@pytest.fixture(scope="module")
def pkg():
    import ddsp_pytorch_b200
    return ddsp_pytorch_b200


# ---------------------------------------------------------------------------------------------------- CPU
def test_argument_errors_do_not_need_a_gpu(pkg):
    from ddsp_pytorch_b200._lib import core_library
    lib = core_library()
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64
    fwd = lib.ddsp_b200_features_fwd
    fwd.restype = i32
    fwd.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i64, i32, i32, i32, vp]
    size = lib.ddsp_b200_features_scratch
    size.restype, size.argtypes = i64, [i32, i64, i32, i32, i32]
    p = ctypes.c_void_p(0x1000)          # never dereferenced: the arguments are rejected before any launch
    ok = (2, 16000, 2048, 160, 30)       # B, N, n_fft, hop, n_mfcc

    def call(ptrs, sizes=ok):
        return fwd(*ptrs, *sizes, None)

    full = [p] * 9
    for i in (0, 1, 2):                                  # signal, window, stage twiddles
        ptrs = list(full)
        ptrs[i] = None
        assert call(ptrs) == -1, i
    for i in (4, 5, 8):                                  # mel table, dct, scratch: needed for the MFCC
        ptrs = list(full)
        ptrs[i] = None
        assert call(ptrs) == -1, i
    assert call([p, p, p, None, p, p, p, p, p]) == -1    # A table with a loudness output
    assert call([p, p, p, p, p, p, None, None, p]) == -1  # no output at all
    bad = [(0, 16000, 2048, 160, 30), (65536, 16000, 2048, 160, 30),        # B
           (2, 1024, 2048, 160, 30), (2, 1 << 30, 2048, 160, 30),           # N <= n_fft/2, N >= 2^30
           (2, 16000, 2000, 160, 30), (2, 16000, 128, 16, 30), (2, 16000, 8192, 160, 30),   # n_fft
           (2, 16000, 2048, 0, 30), (2, 16000, 2048, -5, 30),              # hop
           (2, 16000, 2048, 160, 0), (2, 16000, 2048, 160, 129)]           # n_mfcc
    for sizes in bad:
        assert call(full, sizes) == -1, sizes
        assert size(*sizes) == -1, sizes
    assert size(*ok) > 2 * (1 + 16000 // 160) * 128 - 1
    assert size(1, 129, 256, 1, 1) > 0 and size(65535, 3000, 4096, 4096, 128) > 0


def test_op_registered_without_cpu_kernel(pkg):
    from ddsp_pytorch_b200 import functions as F
    assert hasattr(torch.ops.ddsp_b200, "features_fwd")
    window, a, mel, dct = F.feature_tables(16000, 256, 13, "cpu")
    with pytest.raises((RuntimeError, NotImplementedError)):
        torch.ops.ddsp_b200.features_fwd(torch.zeros(1, 1000), window, a, mel, dct, 256, 64, True)
    with pytest.raises((RuntimeError, NotImplementedError)):
        pkg.extract_features(torch.zeros(1, 1000), 16000, 64, n_mfcc=13, n_fft=256)


def test_extract_features_is_exported_and_forward_only(pkg):
    import ddsp
    assert "extract_features" in pkg.core.__all__ and ddsp.extract_features is pkg.core.extract_features
    x = torch.zeros(1, 4000, requires_grad=True)
    with pytest.raises(RuntimeError, match="no backward"):
        pkg.extract_features(x, 16000, 160)
    with pytest.raises(RuntimeError, match="no backward"):
        pkg.core._features(x, 16000, 160, 2048, 1, False, "extract_loudness")


@pytest.mark.parametrize("sr,n_fft", [(16000, 2048), (48000, 2048), (44100, 1024)])
def test_filterbank_matches_torchaudio(sr, n_fft):
    import torchaudio.functional as AF
    from ddsp_pytorch_b200 import functions as F
    ours = F.mel_filterbank(sr, n_fft)
    ref = AF.melscale_fbanks(n_fft // 2 + 1, 0.0, sr / 2, 128, sr, norm="slaney", mel_scale="slaney").double().T.numpy()
    assert ours.shape == (128, n_fft // 2 + 1)
    assert np.abs(ours - ref).max() <= 1e-6
    # the compact table the kernel reads holds the same weights
    tab = F.mel_band_table(ours)
    first, count, offset = tab[:128].astype(int), tab[128:256].astype(int), tab[256:384].astype(int)
    dense = np.zeros_like(ours)
    for j in range(128):
        dense[j, first[j]:first[j] + count[j]] = tab[384 + offset[j]:384 + offset[j] + count[j]]
    assert np.abs(dense - ours).max() <= 1e-7 * ours.max()
    assert count.min() >= 1 and tab.size == 384 + count.sum()


def test_a_weighting_spot_values():
    from ddsp_pytorch_b200 import functions as F
    a = F.a_weighting_db([0.0, 100.0, 1000.0, 10000.0])
    assert a[0] == -80.0
    assert np.allclose(a[1:], [-19.1424, 0.0003, -2.4914], atol=1e-4)


def test_dct_table_matches_scipy():
    from scipy.fft import dct
    from ddsp_pytorch_b200 import functions as F
    ref = dct(np.eye(128), type=2, norm="ortho", axis=0)
    assert np.abs(F.dct_matrix(128) - ref).max() <= 1e-12
    assert np.array_equal(F.dct_matrix(30), F.dct_matrix(128)[:30])


# ---------------------------------------------------------------------------------------------------- oracle
def oracle(x, sr, n_fft, hop, n_mfcc):
    """float64 loudness (B, F) over all F = 1 + N // hop frames and MFCC (B, F, n_mfcc)"""
    from scipy.fft import dct
    from ddsp_pytorch_b200 import functions as F
    x = np.asarray(x, np.float64)
    pad = np.pad(x, ((0, 0), (n_fft // 2, n_fft // 2)), mode="reflect")
    frames = 1 + x.shape[1] // hop
    window = torch.hann_window(n_fft).double().numpy()      # the float32 table the kernel reads
    a = F.a_weighting_db(np.arange(n_fft // 2 + 1) * sr / n_fft)
    mel_fb = F.mel_filterbank(sr, n_fft)
    loud = np.empty((x.shape[0], frames))
    db = np.empty((x.shape[0], frames, 128))
    step = max(1, 4096 // hop)
    for f0 in range(0, frames, step):                       # in slices: hop 1 would need N x n_fft at once
        f1 = min(frames, f0 + step)
        idx = np.arange(f0, f1)[:, None] * hop + np.arange(n_fft)[None, :]
        spec = np.fft.rfft(pad[:, idx] * window, axis=-1)
        mag = np.abs(spec)
        loud[:, f0:f1] = np.mean(np.log(mag + 1e-7) + a, -1)
        db[:, f0:f1] = 10 * np.log10(np.maximum(1e-10, (mag ** 2) @ mel_fb.T))
    db = np.maximum(db, db.max(axis=(1, 2), keepdims=True) - 80.0)
    return loud, dct(db, type=2, norm="ortho", axis=-1)[..., :n_mfcc]


def torch_composed(x, sr, n_fft, hop, n_mfcc):
    """the same features from float32 torch.stft + matmuls (for comparison only)"""
    from ddsp_pytorch_b200 import functions as F
    window, a, _, _ = F.feature_tables(sr, n_fft, n_mfcc, x.device)
    spec = torch.stft(x, n_fft, hop, window=window, center=True, pad_mode="reflect", return_complex=True).abs()
    loud = (torch.log(spec + 1e-7) + a[:, None]).mean(1)
    mel = torch.from_numpy(F.mel_filterbank(sr, n_fft)).float().to(x.device) @ spec ** 2
    db = 10 * torch.log10(mel.clamp_min(1e-10))
    db = torch.maximum(db, db.amax((1, 2), keepdim=True) - 80)
    dct = torch.from_numpy(F.dct_matrix(n_mfcc)).float().to(x.device)
    return loud, (dct @ db).transpose(1, 2)


def tone_signal(B, N, sr, seed, floor=True):
    """harmonic tones with envelopes, an exactly silent stretch (so that the top_db clamp acts) and, unless
    floor=False, a -60 dB noise floor outside the silence"""
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



# (sr, n_fft, hop, B, N, n_mfcc): N not a multiple of hop everywhere; B in {1, 3, 64}; n_mfcc in {13, 30, 128}
CASES = [
    (16000, 2048, 160, 3, 16077, 30),
    (48000, 2048, 512, 1, 48100, 13),
    (16000, 1024, 64, 64, 8005, 128),
    (22050, 4096, 441, 3, 22350, 30),
    (16000, 256, 1, 3, 1501, 13),
]


# ---------------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("sr,n_fft,hop,B,N,n_mfcc", CASES)
def test_features_match_float64_oracle(pkg, sr, n_fft, hop, B, N, n_mfcc):
    x = tone_signal(B, N, sr, seed=n_fft + hop)
    loud_ref, mfcc_ref = oracle(x, sr, n_fft, hop, n_mfcc)
    xd = torch.from_numpy(x).cuda()
    loud, mfcc = pkg.extract_features(xd, sr, hop, n_mfcc=n_mfcc, n_fft=n_fft)
    assert loud.shape == (B, N // hop) and mfcc.shape == (B, 1 + N // hop, n_mfcc)
    e_loud = float(np.abs(loud.double().cpu().numpy() - loud_ref[:, :-1]).max())
    e_mfcc = float(np.abs(mfcc.double().cpu().numpy() - mfcc_ref).max())
    tl, tm = torch_composed(xd, sr, n_fft, hop, n_mfcc)
    c_loud = float(np.abs(tl.double().cpu().numpy() - loud_ref).max())
    c_mfcc = float(np.abs(tm.double().cpu().numpy() - mfcc_ref).max())
    print(f"\nsr {sr} n_fft {n_fft} hop {hop}: kernel loudness {e_loud:.2e} mfcc {e_mfcc:.2e}; "
          f"float32 torch.stft composition loudness {c_loud:.2e} mfcc {c_mfcc:.2e}")
    # At n_fft 256 and hop 1 every sample offset of the silence's edges starts a frame, among them frames that hold
    # 2 or 3 windowed edge samples: their spectra have nulls near 1e-7, where the float32 rounding of any FFT moves
    # ln(|X| + 1e-7).  Only 129 bins average it out.  The float32 torch.stft composition deviates as much (2.3e-4).
    loud_bar = 5e-4 if (n_fft, hop) == (256, 1) else 1e-4
    assert e_loud <= loud_bar and e_mfcc <= 1e-3, (e_loud, e_mfcc)


@pytest.mark.gpu
def test_pure_tones_without_floor(pkg):
    """Pure tones with no noise floor: most bins hold only the window's sidelobes, down near 1e-7 where
    ln(|X| + 1e-7) turns FFT rounding (~1e-7 of the frame's norm) into errors of order 1 per bin, and the mel bands
    there sit close to the top_db floor.  So the bars are looser here; the silence and the tones' bins agree as above."""
    sr, n_fft, hop = 16000, 2048, 160
    x = tone_signal(3, 16077, sr, seed=5, floor=False)
    loud_ref, mfcc_ref = oracle(x, sr, n_fft, hop, 30)
    loud, mfcc = pkg.extract_features(torch.from_numpy(x).cuda(), sr, hop, n_mfcc=30, n_fft=n_fft)
    e_loud = float(np.abs(loud.double().cpu().numpy() - loud_ref[:, :-1]).max())
    e_mfcc = float(np.abs(mfcc.double().cpu().numpy() - mfcc_ref).max())
    print(f"\npure tones: loudness {e_loud:.2e} mfcc {e_mfcc:.2e}")
    assert e_loud <= 2e-2 and e_mfcc <= 2e-1, (e_loud, e_mfcc)


@pytest.mark.gpu
@pytest.mark.parametrize("n_fft,hop", [(2048, 160), (256, 3)])
def test_all_zero_rows_closed_form(pkg, n_fft, hop):
    from ddsp_pytorch_b200 import functions as F
    sr = 16000
    loud, mfcc = pkg.extract_features(torch.zeros(2, 4000, device="cuda"), sr, hop, n_mfcc=30, n_fft=n_fft)
    a = F.a_weighting_db(np.arange(n_fft // 2 + 1) * sr / n_fft).astype(np.float32).astype(np.float64)
    assert np.abs(loud.double().cpu().numpy() - (np.log(1e-7) + a.mean())).max() <= 1e-4
    m = mfcc.double().cpu().numpy()
    assert np.abs(m[..., 0] + 100 * np.sqrt(128)).max() <= 1e-3
    assert np.abs(m[..., 1:]).max() <= 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("sr,n_fft,hop", [(16000, 2048, 160), (16000, 256, 1), (22050, 4096, 441)])
def test_deterministic_and_independent_of_batch(pkg, sr, n_fft, hop):
    x = torch.from_numpy(tone_signal(64, 6000 if hop == 1 else 24000, sr, seed=11)).cuda()
    l1, m1 = pkg.extract_features(x, sr, hop, n_mfcc=30, n_fft=n_fft)
    l2, m2 = pkg.extract_features(x, sr, hop, n_mfcc=30, n_fft=n_fft)
    assert torch.equal(l1, l2) and torch.equal(m1, m2)
    for b in (0, 37, 63):
        lb, mb = pkg.extract_features(x[b:b + 1], sr, hop, n_mfcc=30, n_fft=n_fft)
        assert torch.equal(lb[0], l1[b]) and torch.equal(mb[0], m1[b])
        l1d, m1d = pkg.extract_features(x[b], sr, hop, n_mfcc=30, n_fft=n_fft)       # (N,) input
        assert torch.equal(l1d, l1[b]) and torch.equal(m1d, m1[b])


@pytest.mark.gpu
def test_extract_loudness_on_cuda_tensors(pkg):
    sr, hop = 16000, 160
    x = torch.from_numpy(tone_signal(3, 16077, sr, seed=2)).cuda()
    loud = pkg.extract_loudness(x, sr, hop)
    assert loud.shape == (3, 16077 // hop) and loud.is_cuda
    assert torch.equal(loud, pkg.extract_features(x, sr, hop)[0])
    one = pkg.extract_loudness(x[1], sr, hop, 1024)
    assert one.shape == (16077 // hop,)
    assert torch.equal(one, pkg.extract_features(x[1:2], sr, hop, n_fft=1024)[0][0])


@pytest.mark.gpu
def test_tool_writes_a_dataset_the_harness_reads(tmp_path):
    from ddsp_pytorch_b200 import core
    from ddsp_pytorch_b200.models.encoder import DDSPAutoencoder
    from ddsp_pytorch_b200.train import NpyDataset, write_synthetic_dataset
    data = write_synthetic_dataset(tmp_path / "ds", 8, seconds=1.0)
    pitch_before = np.load(data / "pitchs.npy")
    cmd = [sys.executable, TOOL, "--data", str(data), "--sample-rate", "16000", "--block-size", "160", "--batch", "3"]
    refused = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert refused.returncode != 0 and "--overwrite" in refused.stderr
    res = subprocess.run(cmd + ["--overwrite"], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr
    import json
    rec = json.loads(res.stdout.strip().splitlines()[-1])
    assert rec["examples"] == 8 and rec["audio_seconds"] == 8.0 and "nvidia_smi" in rec
    assert np.array_equal(np.load(data / "pitchs.npy"), pitch_before)
    ds = NpyDataset(data)
    T = 100
    assert ds.loudness.shape == (8, T) and ds.mfccs.shape == (8, T + 1, 30)
    assert ds.loudness.dtype == np.float32 and ds.mfccs.dtype == np.float32
    sig = torch.from_numpy(np.array(ds.signals[[1, 6]])).cuda()
    loud, mfcc = core.extract_features(sig, 16000, 160)
    assert np.array_equal(np.asarray(ds.loudness[[1, 6]]), loud.cpu().numpy())
    assert np.array_equal(np.asarray(ds.mfccs[[1, 6]]), mfcc.cpu().numpy())
    batch = {k: v.cuda() for k, v in ds.batch(np.arange(8)).items()}
    assert batch["mfcc"].shape == (8, T, 30)
    torch.manual_seed(0)
    model = DDSPAutoencoder(hidden_size=64, n_harmonic=16, n_bands=65, sample_rate=16000, block_size=160,
                            has_reverb=True).cuda()
    with torch.no_grad():
        out = model(batch)
    assert out["signal"].shape == (8, T * 160, 1) and torch.isfinite(out["signal"]).all()
    assert torch.isfinite(out["z"]).all()
