"""Streaming reverb: the direct-form convolution with caller-owned history (csrc/conv_stream.cu), its C ABI, torch op,
``core.convolve_stream`` and the ``streaming_reverb`` realtime export, down to the C++ host.  Played buffer by buffer,
the stream must equal one causal convolution of the whole signal, and the training path's ``Reverb.forward``."""
import ctypes
import json
import math
import os
import subprocess

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "realtime", "ddsp_host")


@pytest.fixture(scope="module")
def pkg():
    import ddsp_pytorch_b200
    return ddsp_pytorch_b200


def _model(seed=0, **kw):
    import ddsp_pytorch_b200  # noqa: F401
    from ddsp_pytorch_b200.models.decoder import DDSPDecoder
    torch.manual_seed(seed)
    cfg = dict(hidden_size=32, n_harmonic=16, n_bands=65, sample_rate=48000, block_size=512, has_reverb=True)
    cfg.update(kw)
    return DDSPDecoder(**cfg)


def _silence_noise(model):
    """the noise branch's magnitudes at the scale function's floor (1e-7): the audio is all but deterministic"""
    with torch.no_grad():
        model.noise_proj.weight.zero_()
        model.noise_proj.bias.fill_(-60.0)
    return model


def _full_conv(x, h):
    """float64 causal convolution of each row of x with h, truncated to the signal length"""
    from scipy.signal import fftconvolve
    x = np.asarray(x, np.float64)
    h = np.asarray(h, np.float64).reshape(1, -1)
    return fftconvolve(x, h, axes=-1)[:, :x.shape[1]]


# ---------------------------------------------------------------------------------------------------- CPU
def test_argument_errors_do_not_need_a_gpu(pkg):
    from ddsp_pytorch_b200._lib import core_library
    lib = core_library()
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64
    fwd = lib.ddsp_b200_conv_stream_fwd
    fwd.restype = i32
    fwd.argtypes = [vp, vp, vp, vp, vp, i32, i64, i32, vp, vp]
    size = lib.ddsp_b200_conv_stream_scratch
    size.restype, size.argtypes = i64, [i32, i64, i32]
    p = ctypes.c_void_p(0x1000)          # never dereferenced: the arguments are rejected before any launch
    assert fwd(None, p, p, p, p, 1, 1024, 48000, p, None) == -1          # null signal
    assert fwd(p, None, p, p, p, 1, 1024, 48000, p, None) == -1          # null kernel
    assert fwd(p, p, None, p, p, 1, 1024, 48000, p, None) == -1          # null history with L > 1
    assert fwd(p, p, p, None, p, 1, 1024, 48000, p, None) == -1          # null output
    assert fwd(p, p, p, p, None, 1, 1024, 48000, p, None) == -1          # null history_out
    assert fwd(p, p, p, p, p, 1, 0, 48000, p, None) == -1                # N = 0
    assert fwd(p, p, p, p, p, 1, 1024, 0, p, None) == -1                 # L = 0
    assert fwd(p, p, p, p, p, 0, 1024, 48000, p, None) == -1             # B = 0
    assert size(1, 0, 48000) == -1 and size(1, 1024, 0) == -1 and size(0, 1024, 48000) == -1
    assert size(1, 1024, 48000) > 0                                     # realtime shape: chunk sums in scratch
    assert fwd(p, p, p, p, p, 1, 1024, 48000, None, None) == -1          # ... so NULL scratch is refused
    assert size(1, 1024, 37) == 0                                       # one chunk of taps: no scratch


def test_op_registered_without_cpu_kernel(pkg):
    assert hasattr(torch.ops.ddsp_b200, "conv_stream_fwd")
    with pytest.raises((RuntimeError, NotImplementedError)):
        torch.ops.ddsp_b200.conv_stream_fwd(torch.zeros(1, 8), torch.zeros(4), torch.zeros(1, 3))


def test_convolve_stream_is_forward_only(pkg):
    x = torch.zeros(1, 8, requires_grad=True)
    with pytest.raises(RuntimeError, match="no backward"):
        pkg.convolve_stream(x, torch.zeros(4))


def test_streaming_export_scripts_on_cpu(tmp_path):
    from ddsp_pytorch_b200.export import export_torchscript
    model = _model()
    path = os.path.join(tmp_path, "rt_reverb.ts")
    export_torchscript(model, path, mean_loudness=-30.0, std_loudness=12.0, realtime=True, streaming_reverb=True)
    loaded = torch.jit.load(path)
    graph = str(loaded.inlined_graph)
    for op in ("conv_stream_fwd", "reverb_impulse_fwd", "noise_fwd"):
        assert "ddsp_b200::" + op in graph
    assert "fftconv_fwd" not in graph
    buffers = dict(loaded.named_buffers())
    assert tuple(buffers["reverb_history"].shape) == (1, model.reverb.length - 1)
    assert {"cache_gru", "phase"} <= set(buffers)
    loaded.reset()
    # the dry realtime export keeps its graph and buffers
    export_torchscript(model, os.path.join(tmp_path, "rt.ts"), realtime=True)
    dry = torch.jit.load(os.path.join(tmp_path, "rt.ts"))
    assert "conv_stream_fwd" not in str(dry.inlined_graph)
    assert "reverb_history" not in dict(dry.named_buffers())


def test_streaming_reverb_needs_realtime_and_a_reverb(tmp_path):
    from ddsp_pytorch_b200.export import export_torchscript
    with pytest.raises(ValueError):
        export_torchscript(_model(), os.path.join(tmp_path, "a.ts"), realtime=False, streaming_reverb=True)
    with pytest.raises(ValueError):
        export_torchscript(_model(has_reverb=False), os.path.join(tmp_path, "b.ts"), realtime=True,
                           streaming_reverb=True)


# ---------------------------------------------------------------------------------------------------- GPU
TOTAL = 9000
CHUNKINGS = {
    "1024": [1024] * (TOTAL // 1024) + [TOTAL % 1024],
    "160": [160] * (TOTAL // 160) + [TOTAL % 160],
    "irregular": [1, 3, 1000, 4097, TOTAL - 5101],
}


def _stream(x, h, sizes):
    from ddsp_pytorch_b200 import core
    outs, hist, pos = [], None, 0
    with torch.no_grad():
        for n in sizes:
            y, hist = core.convolve_stream(x[:, pos:pos + n].contiguous(), h, hist)
            outs.append(y)
            pos += n
    return torch.cat(outs, 1), hist


@pytest.mark.gpu
@pytest.mark.parametrize("L", [1, 2, 37, 4000, 16000, 48000])
@pytest.mark.parametrize("chunking", sorted(CHUNKINGS))
def test_stream_matches_float64_convolution(pkg, L, chunking):
    g = torch.Generator().manual_seed(L)
    x = torch.randn(3, TOTAL, generator=g)
    h = torch.randn(L, generator=g) * torch.exp(-torch.arange(L) / max(L / 4, 1.0))
    got, hist = _stream(x.cuda(), h.cuda(), CHUNKINGS[chunking])
    ref = _full_conv(x.numpy(), h.numpy())
    peak = float(np.abs(ref).max())
    err = float(np.abs(got.double().cpu().numpy() - ref).max())
    assert err <= 1e-5 * peak, (err, peak)
    want = torch.zeros(3, L - 1)
    keep = min(L - 1, TOTAL)
    if keep:
        want[:, L - 1 - keep:] = x[:, TOTAL - keep:]
    assert torch.equal(hist.cpu(), want)          # the last L-1 inputs, bit for bit, zeros before the first


@pytest.mark.gpu
@pytest.mark.parametrize("sample_rate", [16000, 48000])
def test_stream_matches_training_reverb(pkg, sample_rate):
    from ddsp_pytorch_b200.models.modules import Reverb
    torch.manual_seed(3)
    reverb = Reverb(sample_rate, sample_rate).cuda()
    g = torch.Generator().manual_seed(4)
    n = 1024 * (sample_rate * 5 // 4 // 1024 + 2)          # longer than the impulse: every tap is used
    x = torch.randn(2, n, 1, generator=g).cuda()
    with torch.no_grad():
        whole = reverb(x).squeeze(-1)
        impulse = reverb.build_impulse()
    got, _ = _stream(x.squeeze(-1), impulse, [1024] * (n // 1024))
    peak = float(whole.abs().max())
    assert float((got - whole).abs().max()) <= 1e-5 * peak


@pytest.mark.gpu
@pytest.mark.parametrize("B,N,L", [(1, 1024, 48000), (3, 1000, 16000), (2, 4097, 37)])
def test_stream_is_deterministic(pkg, B, N, L):
    g = torch.Generator().manual_seed(9)
    x, h = torch.randn(B, N, generator=g).cuda(), torch.randn(L, generator=g).cuda()
    hist = torch.randn(B, L - 1, generator=g).cuda()
    y1, h1 = pkg.convolve_stream(x, h, hist)
    y2, h2 = pkg.convolve_stream(x, h, hist)
    assert torch.equal(y1, y2) and torch.equal(h1, h2)


def _buffers(n_buf, n=1024):
    i = torch.arange(n_buf * n, dtype=torch.float32)
    pitch = (220.0 + 20.0 * torch.sin(0.001 * i)).view(1, -1, 1).cuda()
    loud = torch.full((1, n_buf * n, 1), -25.0).cuda()
    return pitch, loud


@pytest.mark.gpu
def test_streaming_export_equals_dry_export_convolved(tmp_path):
    from ddsp_pytorch_b200.export import export_torchscript
    model = _silence_noise(_model(seed=2)).cuda().eval()
    export_torchscript(model, os.path.join(tmp_path, "dry.ts"), realtime=True)
    export_torchscript(model, os.path.join(tmp_path, "wet.ts"), realtime=True, streaming_reverb=True)
    dry = torch.jit.load(os.path.join(tmp_path, "dry.ts")).cuda()
    wet = torch.jit.load(os.path.join(tmp_path, "wet.ts")).cuda()
    pitch, loud = _buffers(4)
    a, b = [], []
    with torch.no_grad():
        for k in range(4):
            s = slice(k * 1024, (k + 1) * 1024)
            torch.manual_seed(100 + k)                  # the same noise draw in both exports
            a.append(dry(pitch[:, s], loud[:, s]))
            torch.manual_seed(100 + k)
            b.append(wet(pitch[:, s], loud[:, s]))
        impulse = model.reverb.build_impulse().reshape(-1)
    ref = _full_conv(torch.cat(a, 1).squeeze(-1).double().cpu().numpy(), impulse.double().cpu().numpy())
    got = torch.cat(b, 1).squeeze(-1).double().cpu().numpy()
    peak = float(np.abs(ref).max())
    assert peak > 0 and float(np.abs(got - ref).max()) <= 2e-5 * peak
    wet.reset()
    with torch.no_grad():
        torch.manual_seed(100)
        again = wet(pitch[:, :1024], loud[:, :1024])
    assert torch.equal(again, b[0])


@pytest.mark.gpu
def test_cpp_host_streams_the_reverb(tmp_path):
    import ddsp_pytorch_b200  # noqa: F401
    from ddsp_pytorch_b200._lib import TORCH_PATH
    from ddsp_pytorch_b200.export import export_torchscript
    from ddsp_pytorch_b200.models.decoder import DDSPDecoder
    torch.manual_seed(4)
    model = _silence_noise(DDSPDecoder(hidden_size=64, n_harmonic=32, n_bands=65, sample_rate=48000, block_size=512,
                                       has_reverb=True)).cuda().eval()
    path = os.path.join(tmp_path, "rt_reverb.ts")
    export_torchscript(model, path, mean_loudness=-30.0, std_loudness=10.0, realtime=True, streaming_reverb=True)
    buffers, n = 6, 1024
    res = subprocess.run([HOST, TORCH_PATH, path, str(buffers), str(n)], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr
    got = json.loads(res.stdout.strip().splitlines()[-1])
    rt = torch.jit.load(path).cuda()                   # the same stream through the scripted module in Python
    checksum, peak = 0.0, 0.0
    with torch.no_grad():
        for b in range(buffers + 2):
            i = torch.arange(b * n, (b + 1) * n, dtype=torch.float32)
            pitch = (220.0 + 20.0 * torch.sin(0.001 * i)).view(1, n, 1).cuda()
            loud = torch.full((1, n, 1), -25.0).cuda()
            y = rt(pitch, loud).double().cpu()
            checksum += float(y.sum())
            peak = max(peak, float(y.abs().max()))
    assert math.isclose(got["peak"], peak, rel_tol=1e-4, abs_tol=1e-6)
    assert abs(got["checksum"] - checksum) <= 1e-3 * max(1.0, abs(checksum)) + 1e-2
    assert got["worst_ms"] < 21.3, "1024 samples at 48 kHz leave 21.3 ms per buffer"
