"""torch.autograd.Function wrappers around the ddsp_b200:: custom ops.

Each Function pairs a ``*_fwd`` op with its hand-written ``*_bwd`` op (SURVEY 8a row a13).  The
backward kernels are not differentiable again (``once_differentiable``).  Scripted / C++ inference
calls the ``*_fwd`` ops directly and never touches this file.
"""
from __future__ import annotations

from typing import List, Optional, Sequence

import numpy as np
import torch
from torch.autograd.function import once_differentiable

from ._lib import get_ops

_ops = get_ops()

_WINDOWS = {}


def hann_window_like_reference(n_fft: int, device) -> torch.Tensor:
    """core.py:35 builds the window with ``torch.hann_window(s)`` on the CPU in float32 and then
    moves it; doing the same keeps the window bit-identical to the reference's."""
    key = (int(n_fft), str(device))
    w = _WINDOWS.get(key)
    if w is None:
        w = torch.hann_window(int(n_fft)).to(device)
        _WINDOWS[key] = w
    return w


_WINDOW_SETS = {}


def hann_windows_like_reference(scales: Sequence[int], device) -> torch.Tensor:
    """The scales' windows back to back (the layout ``mss_loss_fwd`` takes), built once per (scales, device)."""
    key = (tuple(int(s) for s in scales), str(device))
    w = _WINDOW_SETS.get(key)
    if w is None:
        w = torch.cat([hann_window_like_reference(s, device) for s in key[0]])
        _WINDOW_SETS[key] = w
    return w


# ---- constant tables of the feature extractor (csrc/features.cu), built in float64 on the host ----------------------
N_MELS = 128


def a_weighting_db(freqs) -> np.ndarray:
    """librosa's ``A_weighting`` (min_db = -80) in dB at ``freqs`` Hz, float64."""
    f2 = np.asarray(freqs, np.float64) ** 2
    c = np.array([12194.217, 20.598997, 107.65265, 737.86223]) ** 2
    with np.errstate(divide="ignore"):
        a = 2.0 + 20.0 * (np.log10(c[0]) + 2 * np.log10(f2) - np.log10(f2 + c[0]) - np.log10(f2 + c[1])
                          - 0.5 * np.log10(f2 + c[2]) - 0.5 * np.log10(f2 + c[3]))
    return np.maximum(-80.0, a)


def _hz_to_mel(f):
    """Slaney mel scale (librosa ``htk=False``): linear below 1 kHz, logarithmic above."""
    f = np.asarray(f, np.float64)
    logstep = np.log(6.4) / 27.0
    return np.where(f >= 1000.0, 15.0 + np.log(np.maximum(f, 1e-300) / 1000.0) / logstep, f / (200.0 / 3))


def _mel_to_hz(m):
    m = np.asarray(m, np.float64)
    logstep = np.log(6.4) / 27.0
    return np.where(m >= 15.0, 1000.0 * np.exp(logstep * (m - 15.0)), m * (200.0 / 3))


def mel_filterbank(sample_rate: float, n_fft: int, n_mels: int = N_MELS) -> np.ndarray:
    """``librosa.filters.mel(sr, n_fft, n_mels, fmin=0, fmax=sr/2, htk=False, norm="slaney")``: (n_mels, n_fft/2+1)
    float64 triangles on the Slaney mel scale, each scaled to unit area (2 / its width in Hz)."""
    fft_freqs = np.linspace(0.0, sample_rate / 2, 1 + n_fft // 2)
    mel_f = _mel_to_hz(np.linspace(_hz_to_mel(0.0), _hz_to_mel(sample_rate / 2), n_mels + 2))
    fdiff = np.diff(mel_f)
    ramps = mel_f[:, None] - fft_freqs[None, :]
    lower = -ramps[:-2] / fdiff[:-1, None]
    upper = ramps[2:] / fdiff[1:, None]
    weights = np.maximum(0.0, np.minimum(lower, upper))
    return weights * (2.0 / (mel_f[2:] - mel_f[:-2]))[:, None]


def mel_band_table(weights: np.ndarray) -> np.ndarray:
    """The compact band table the kernel reads: first bin, bin count and weight offset of each band (as floats, exact
    below 2^24), then every band's nonzero run of weights back to back.  float32."""
    n_mels = weights.shape[0]
    first, count, offset, runs, pos = [], [], [], [], 0
    for row in weights:
        nz = np.nonzero(row)[0]
        lo, hi = (int(nz[0]), int(nz[-1]) + 1) if nz.size else (0, 0)
        first.append(lo)
        count.append(hi - lo)
        offset.append(pos)
        runs.append(row[lo:hi])
        pos += hi - lo
    head = np.array([first, count, offset], np.float64).reshape(3 * n_mels)
    return np.concatenate([head] + runs).astype(np.float32)


def dct_matrix(n_mfcc: int, n_mels: int = N_MELS) -> np.ndarray:
    """DCT-II with ``norm="ortho"``, the first n_mfcc rows: (n_mfcc, n_mels) float64."""
    i = np.arange(n_mfcc, dtype=np.float64)[:, None]
    j = np.arange(n_mels, dtype=np.float64)[None, :]
    d = np.cos(np.pi * i * (2 * j + 1) / (2 * n_mels)) * np.sqrt(2.0 / n_mels)
    d[0] *= np.sqrt(0.5)
    return d


_FEATURE_TABLES = {}


def feature_tables(sample_rate: float, n_fft: int, n_mfcc: int, device):
    """(window, a_weight, mel_table, dct (128, n_mfcc)) for ``features_fwd``, built once per
    (sample_rate, n_fft, n_mfcc, device)."""
    key = (float(sample_rate), int(n_fft), int(n_mfcc), str(device))
    tabs = _FEATURE_TABLES.get(key)
    if tabs is None:
        sr, n_fft = key[0], key[1]
        freqs = np.arange(n_fft // 2 + 1, dtype=np.float64) * sr / n_fft
        tabs = (hann_window_like_reference(n_fft, device),
                torch.from_numpy(a_weighting_db(freqs).astype(np.float32)).to(device),
                torch.from_numpy(mel_band_table(mel_filterbank(sr, n_fft))).to(device),
                torch.from_numpy(np.ascontiguousarray(dct_matrix(key[2]).T).astype(np.float32)).to(device))
        _FEATURE_TABLES[key] = tabs
    return tabs


class ScaleFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        ctx.save_for_backward(x)
        return _ops.scale_function_fwd(x)

    @staticmethod
    @once_differentiable
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        return _ops.scale_function_bwd(x, dy).view_as(x)


class RemoveAboveNyquist(torch.autograd.Function):
    @staticmethod
    def forward(ctx, amplitudes, f0, sample_rate):
        ctx.save_for_backward(f0)
        ctx.sample_rate = float(sample_rate)
        return _ops.remove_above_nyquist(amplitudes, f0, ctx.sample_rate)

    @staticmethod
    @once_differentiable
    def backward(ctx, dy):
        (f0,) = ctx.saved_tensors            # the mask has no gradient w.r.t. f0 (core.py:73)
        return _ops.remove_above_nyquist(dy, f0, ctx.sample_rate), None, None


class HarmonicControls(torch.autograd.Function):
    """modules.py:44-67 fused: (amp_raw, dist_raw, f0) -> (amplitudes, normalised distribution)."""

    @staticmethod
    def forward(ctx, amp_raw, dist_raw, f0, sample_rate):
        ctx.save_for_backward(amp_raw, dist_raw, f0)
        ctx.sample_rate = float(sample_rate)
        amps, dist, _ = _ops.harmonic_controls_fwd(amp_raw, dist_raw, f0, ctx.sample_rate, False)
        return amps, dist

    @staticmethod
    @once_differentiable
    def backward(ctx, d_amps, d_dist):
        amp_raw, dist_raw, f0 = ctx.saved_tensors
        da, dd = _ops.harmonic_controls_bwd(amp_raw, dist_raw, f0, d_amps, d_dist, None, ctx.sample_rate)
        return da.view_as(amp_raw), dd.view_as(dist_raw), None, None


class HarmonicControlsWeights(torch.autograd.Function):
    """get_controls + the in-place ``distribution *= amplitudes`` of HarmonicSynth.forward
    (modules.py:44-67,73) in one launch: -> (amplitudes, distribution, weights = distribution*amplitudes)."""

    @staticmethod
    def forward(ctx, amp_raw, dist_raw, f0, sample_rate):
        ctx.save_for_backward(amp_raw, dist_raw, f0)
        ctx.sample_rate = float(sample_rate)
        ctx.set_materialize_grads(False)
        return _ops.harmonic_controls_fwd(amp_raw, dist_raw, f0, ctx.sample_rate, True)

    @staticmethod
    @once_differentiable
    def backward(ctx, d_amps, d_dist, d_weights):
        amp_raw, dist_raw, f0 = ctx.saved_tensors
        da, dd = _ops.harmonic_controls_bwd(amp_raw, dist_raw, f0, d_amps, d_dist, d_weights, ctx.sample_rate)
        return da.view_as(amp_raw), dd.view_as(dist_raw), None, None


class HarmonicFrames(torch.autograd.Function):
    """modules.py:69-80 fused: frame-rate f0 (B,T,1) and weights (B,T,H) -> audio (B,T*bs,1)."""

    @staticmethod
    def forward(ctx, f0, weights, block_size, sample_rate, phase0):
        audio, phase_end, phi, delta = _ops.harmonic_fwd(f0, weights, int(block_size),
                                                         float(sample_rate), phase0)
        ctx.save_for_backward(weights, phi, delta)
        ctx.cfg = (int(block_size), float(sample_rate), f0.shape)
        ctx.mark_non_differentiable(phase_end)
        return audio, phase_end

    @staticmethod
    @once_differentiable
    def backward(ctx, g_audio, _g_phase):
        weights, phi, delta = ctx.saved_tensors
        bs, sr, f0_shape = ctx.cfg
        need_f0 = ctx.needs_input_grad[0]
        dw, df0 = _ops.harmonic_bwd(g_audio, weights, phi, delta, bs, sr, need_f0)
        return (df0.view(f0_shape) if need_f0 else None), dw, None, None, None


class HarmonicFromRaw(torch.autograd.Function):
    """decoder.py:106-110 + modules.py:44-80 in ONE launch per direction: the control net's raw outputs go straight
    into the oscillator bank, whose prologue applies get_controls (scale_function, Nyquist mask, normalise) and the
    in-place ``distribution *= amplitudes``; the backward's epilogue takes the weight gradients through the controls'
    backward.  ``first`` = the projection output (B,T,H+1) with ``dist_raw=None`` (read and differentiated in place, no
    slicing copies), or amp_raw (B,T,1) with dist_raw (B,T,H).
    -> (audio (B,T*bs,1), phase_end (B), amplitudes (B,T,1), weights (B,T,H))."""

    @staticmethod
    def forward(ctx, first, dist_raw, f0, block_size, sample_rate, phase0):
        audio, phase_end, phi, delta, amps, weights = _ops.harmonic_raw_fwd(
            first, dist_raw, f0, int(block_size), float(sample_rate), phase0)
        ctx.save_for_backward(first, dist_raw, f0, phi, delta)
        ctx.cfg = (int(block_size), float(sample_rate))
        ctx.mark_non_differentiable(phase_end)
        ctx.set_materialize_grads(False)
        return audio, phase_end, amps, weights

    @staticmethod
    @once_differentiable
    def backward(ctx, g_audio, _g_phase, g_amps, g_weights):
        first, dist_raw, f0, phi, delta = ctx.saved_tensors
        bs, sr = ctx.cfg
        joint = dist_raw is None
        if g_audio is None:
            g_audio = torch.zeros(f0.shape[0], f0.shape[1] * bs, 1, device=f0.device, dtype=f0.dtype)
        if g_amps is None and g_weights is None:
            d0, d1 = _ops.harmonic_raw_bwd(g_audio, first, dist_raw, f0, phi, delta, bs, sr)
            return d0, (None if joint else d1), None, None, None, None
        # someone differentiates the returned controls as well (never the reference's training loop): two launches
        a_raw = first[..., :1] if joint else first
        d_raw = first[..., 1:] if joint else dist_raw
        amps, _, weights = _ops.harmonic_controls_fwd(a_raw, d_raw, f0, sr, True)
        dw, _ = _ops.harmonic_bwd(g_audio, weights, phi, delta, bs, sr, False)
        if g_weights is not None:
            dw = dw + g_weights
        da, dd = _ops.harmonic_controls_bwd(a_raw, d_raw, f0, g_amps, None, dw, sr)
        if joint:
            return torch.cat([da.view_as(a_raw), dd.view_as(d_raw)], -1), None, None, None, None, None
        return da.view_as(first), dd.view_as(dist_raw), None, None, None, None


class HarmonicAudioRate(torch.autograd.Function):
    """core.py:136-141: f0 (B,N,1), amplitudes (B,N,H) at audio rate -> (B,N,1)."""

    @staticmethod
    def forward(ctx, f0, amplitudes, sample_rate):
        audio, phase = _ops.harmonic_ar_fwd(f0, amplitudes, float(sample_rate))
        ctx.save_for_backward(amplitudes, phase)
        ctx.cfg = (float(sample_rate), f0.shape)
        return audio

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        amplitudes, phase = ctx.saved_tensors
        sr, f0_shape = ctx.cfg
        need_f0 = ctx.needs_input_grad[0]
        da, df0 = _ops.harmonic_ar_bwd(g, amplitudes, phase, sr, need_f0)
        return (df0.view(f0_shape) if need_f0 else None), da, None


class AmpToImpulseResponse(torch.autograd.Function):
    @staticmethod
    def forward(ctx, amp, target_size):
        ctx.n_bands = amp.shape[-1]
        return _ops.amp_to_ir_fwd(amp, int(target_size))

    @staticmethod
    @once_differentiable
    def backward(ctx, d_ir):
        return _ops.amp_to_ir_bwd(d_ir, ctx.n_bands), None


class FilteredNoise(torch.autograd.Function):
    """modules.py:116-128 fused, noise passed in: magnitudes (B,T,NB), noise (B,T,bs) -> (B,T*bs,1)."""

    @staticmethod
    def forward(ctx, magnitudes, noise):
        ctx.save_for_backward(noise)
        ctx.n_bands = magnitudes.shape[-1]
        return _ops.noise_fwd(magnitudes, noise, None, False, 0.0)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        (noise,) = ctx.saved_tensors
        return _ops.noise_bwd(g, noise, None, ctx.n_bands, False, 0.0), None   # the draw has no gradient


class FilteredNoiseFused(torch.autograd.Function):
    """get_controls + forward + the mix of decoder.py:115-121 in one launch:
    scale_function(raw + bias) -> IR -> FIR of the noise draw -> + ``add`` (the harmonic audio)."""

    @staticmethod
    def forward(ctx, magnitudes_raw, noise, add, bias):
        ctx.save_for_backward(magnitudes_raw, noise)
        ctx.bias = float(bias)
        return _ops.noise_fwd(magnitudes_raw, noise, add, True, ctx.bias)

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        raw, noise = ctx.saved_tensors
        d_raw = _ops.noise_bwd(g, noise, raw, raw.shape[-1], True, ctx.bias)
        return d_raw, None, (g if ctx.needs_input_grad[2] else None), None


class FFTConvolve(torch.autograd.Function):
    """core.py:169-176 on 2-D (rows, n) operands; kernel rows 1 (shared) or equal to signal rows.
    When a gradient will be needed the forward keeps the transform of the signal and the kernel spectrum
    (32 MB + 1 MB at config 2) so the backward does not recompute them.  ``hspec`` = the kernel's spectrum from
    ``fftconv_spectrum`` when the caller computed it ahead of time.  ``signal2``: convolve ``signal + signal2`` (the sum
    is formed while the first pass loads its input: decoder.py:121's ``harmonic + noise`` without its own launch);
    both summands receive the same gradient."""

    @staticmethod
    def forward(ctx, signal, kernel, hspec=None, signal2=None):
        need = list(ctx.needs_input_grad) + [False] * 4           # apply() may be called with 2, 3 or 4 arguments
        keep = bool(need[0] or need[1] or (signal2 is not None and need[3]))
        out, work_x, hspec = _ops.fftconv_fwd(signal, kernel, keep, hspec, signal2)
        ctx.save_for_backward(signal, kernel, work_x, hspec)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        signal, kernel, work_x, hspec = ctx.saved_tensors
        n = len(ctx.needs_input_grad)
        need = list(ctx.needs_input_grad) + [False] * 4
        wx, hs = (work_x if work_x.numel() else None), (hspec if hspec.numel() else None)
        part = _FFTCONV_PART[0]
        if part is None:
            ds, dk = _ops.fftconv_bwd(g, signal, kernel, wx, hs, need[0] or need[3], need[1])
        elif part == "kernel":
            # first of two calls over the same grad_output: the kernel gradient only; the transform of g is kept
            _, dk, ctx._work_g = _ops.fftconv_bwd_parts(g, signal, kernel, wx, hs, None, False, need[1])
            ctx._work_g_key = (g.data_ptr(), g._version)
            ds = None
        else:
            kept = getattr(ctx, "_work_g", None)
            if kept is not None and ctx._work_g_key != (g.data_ptr(), g._version):
                kept = None
            ds, _, _ = _ops.fftconv_bwd_parts(g, signal, kernel, wx, hs, kept, need[0] or need[3], False)
            ctx._work_g = None                        # filtered in place by the call above
            dk = None
        grads = ((ds if need[0] else None), (dk if need[1] else None), None, (ds if need[3] else None))
        return grads[:n]


_FFTCONV_PART = [None]


class fftconv_backward_part:
    """Context manager for callers that take FFTConvolve's two gradients in two ``autograd.grad`` calls over the same
    grad_output (``retain_graph=True`` on the first): ``"kernel"`` computes the kernel gradient only and keeps the
    transform of grad_output, ``"signal"`` reuses it for the signal gradient.  The data-parallel step does this to have
    the reverb parameters' all-reduce in flight during the rest of the backward (hotpath.SynthStep)."""

    def __init__(self, part: str):
        assert part in ("kernel", "signal")
        self.part = part

    def __enter__(self):
        self.saved = _FFTCONV_PART[0]
        _FFTCONV_PART[0] = self.part

    def __exit__(self, *a):
        _FFTCONV_PART[0] = self.saved


class ReverbImpulse(torch.autograd.Function):
    """modules.py:21-26: (noise (L,1), decay, wet, t (1,L,1)) -> impulse (1,L,1)."""

    @staticmethod
    def forward(ctx, noise, decay, wet, t):
        ctx.save_for_backward(noise, decay, wet, t)
        return _ops.reverb_impulse_fwd(noise, decay, wet, t)

    @staticmethod
    @once_differentiable
    def backward(ctx, d_imp):
        noise, decay, wet, t = ctx.saved_tensors
        dn, dd, dw = _ops.reverb_impulse_bwd(d_imp, noise, decay, wet, t)
        return dn.view_as(noise), dd.view_as(decay), dw.view_as(wet), None


class Linear3x(torch.autograd.Function):
    """``F.linear`` (core.py:122-129's nn.Linear layers, the GRU input projection, decoder.py:86-87's
    projections) on the tcgen05 tensor cores with float32-class accuracy (csrc/gemm3x.cu).  All three GEMMs of a
    layer take the same kernel, and every matrix is split into its bf16 parts exactly once: x and W in the
    forward (kept for the backward), dy in the backward; y = x W^T reads them K-major, dx = dy W reads W
    MN-major, dW = dy^T x reads dy and x MN-major -- no transposed copies."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        x2 = x.reshape(-1, x.shape[-1]).contiguous()
        m, k = x2.shape
        n = weight.shape[0]
        xs = _ops.gemm3x_split(x2, False)
        ws = _ops.gemm3x_split(weight.contiguous(), False)
        ctx.save_for_backward(xs if ctx.needs_input_grad[1] else None, ws if ctx.needs_input_grad[0] else None)
        ctx.has_bias = bias is not None
        ctx.mnk = (m, n, k)
        return _ops.gemm3x_mm(xs, ws, m, n, k, bias, False, False).view(*x.shape[:-1], n)

    @staticmethod
    @once_differentiable
    def backward(ctx, dy):
        xs, ws = ctx.saved_tensors
        m, n, k = ctx.mnk
        dy2 = dy.reshape(m, n).contiguous()
        dx = dw = db = None
        if ctx.has_bias and ctx.needs_input_grad[2]:
            dys, db = _ops.gemm3x_split_colsum(dy2)          # the bias gradient rides on the split of dy
        else:
            dys = _ops.gemm3x_split(dy2, False)
        if ctx.needs_input_grad[0]:          # (m, n) x (n, k): dy K-major, W (n rows = contraction) MN-major
            dx = _ops.gemm3x_mm(dys, ws, m, k, n, None, False, True).view(*dy.shape[:-1], k)
        if ctx.needs_input_grad[1]:          # (n, m) x (m, k): both stored with the contraction (rows) outermost
            dw = _ops.gemm3x_mm(dys, xs, n, k, m, None, True, True)
        return dx, dw, db


class LayerNormLeakyReLU(torch.autograd.Function):
    """leaky_relu(layer_norm(x)) over the last dimension in one pass each way (csrc/layernorm.cu):
    core.py:122-129's LayerNorm -> LeakyReLU pair."""

    @staticmethod
    def forward(ctx, x, weight, bias, eps, slope):
        x = x.contiguous()
        y, stats = _ops.ln_lrelu_fwd(x, weight, bias, eps, slope, any(ctx.needs_input_grad[:3]))
        ctx.save_for_backward(x, weight, bias, stats)
        ctx.slope = slope
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, dy):
        x, weight, bias, stats = ctx.saved_tensors
        dx, dg, db = _ops.ln_lrelu_bwd(dy.contiguous(), x, weight, bias, stats, ctx.slope)
        return dx, dg, db, None, None


class GRURecurrence(torch.autograd.Function):
    """The time loop of core.py:132-133's nn.GRU (one layer, batch_first) as one cluster-persistent launch.
    gi (B,T,3H) = x W_ih^T + b_ih is computed by the caller (a cuBLAS GEMM autograd differentiates);
    returns every hidden state (B,T,H).  Backward: one reverse-time launch for the gate gradients, then
    dW_hh / db_hh as GEMM / reduction over them."""

    @staticmethod
    def forward(ctx, gi, weight_hh, bias_hh, h0):
        need = any(ctx.needs_input_grad)
        y, gates = _ops.gru_fwd(gi, weight_hh, bias_hh, h0, need)
        ctx.save_for_backward(weight_hh, y, h0, gates)
        return y

    @staticmethod
    @once_differentiable
    def backward(ctx, dy):
        weight_hh, y, h0, gates = ctx.saved_tensors
        B, T, H = y.shape
        dgi, dgh, dh0 = _ops.gru_bwd(dy, None, weight_hh, y, h0, gates)
        d_w = d_b = None
        if ctx.needs_input_grad[1]:
            h_prev = torch.empty_like(y)
            h_prev[:, 1:] = y[:, :-1]
            if h0 is None:
                h_prev[:, 0].zero_()
            else:
                h_prev[:, 0] = h0.reshape(B, H)
            dghs, d_b = _ops.gemm3x_split_colsum(dgh.reshape(B * T, 3 * H))     # db_hh rides on the split
            d_w = _ops.gemm3x_mm(dghs, _ops.gemm3x_split(h_prev.reshape(B * T, H), False), 3 * H, H, B * T, None,
                                 True, True)
        elif ctx.needs_input_grad[2]:
            d_b = dgh.sum((0, 1))
        d_h0 = None
        if h0 is not None and ctx.needs_input_grad[3]:
            d_h0 = dh0.view_as(h0)
        return (dgi if ctx.needs_input_grad[0] else None), d_w, d_b, d_h0


class StftMag(torch.autograd.Function):
    """One scale of core.py:27-41: signal (B,N) -> |STFT| (B, s/2+1, 1+N//hop)."""

    @staticmethod
    def forward(ctx, signal, n_fft, hop):
        window = hann_window_like_reference(n_fft, signal.device)
        ctx.save_for_backward(signal, window)
        ctx.cfg = (int(n_fft), int(hop))
        return _ops.stft_mag_fwd(signal, window, int(n_fft), int(hop))

    @staticmethod
    @once_differentiable
    def backward(ctx, d_mag):
        signal, window = ctx.saved_tensors
        n_fft, hop = ctx.cfg
        return _ops.stft_mag_bwd(signal, d_mag, window, n_fft, hop), None, None


class MultiScaleSpectralLoss(torch.autograd.Function):
    """train.py:70-76 over core.py:27-41, fused: (target (B,N), rec (B,N)) -> scalar loss.
    The gradient w.r.t. rec is produced by the forward launch itself (same FFTs); backward only
    scales it.  target gets no gradient (train.py feeds data there)."""

    @staticmethod
    def forward(ctx, target, rec, scales, overlap):
        scales = [int(s) for s in scales]
        windows = hann_windows_like_reference(scales, rec.device)
        need = bool(ctx.needs_input_grad[1])
        loss, d_rec = _ops.mss_loss_fwd(target, rec, scales, float(overlap), windows, need)
        if need:
            ctx.save_for_backward(d_rec)
        ctx.rec_shape = rec.shape
        return loss

    @staticmethod
    @once_differentiable
    def backward(ctx, g):
        (d_rec,) = ctx.saved_tensors
        return None, (d_rec * g).view(ctx.rec_shape), None, None
