"""The DDSP DSP core with the reference's function signatures (ddsp/core.py), running on the
hand-written sm_100a kernels.

Every hot function of the reference module is here under the same name and argument list, so
``ddsp.<name>`` call sites (modules.py:33,53-56,74-78,113,117,125; train.py:92-103) keep working:

    safe_log  multiscale_fft  upsample  remove_above_nyquist  scale_function
    harmonic_synth  amp_to_impulse_response  fft_convolve

plus the non-hot helpers that must stay importable (mean_std_loudness, resample, extract_loudness,
extract_pitch, mlp, gru).  Tensors must be CUDA float32: there is no CPU implementation of the
kernels and a CPU tensor raises from the dispatcher.  Additions that have no counterpart in the
reference are marked "extension".
"""
from __future__ import annotations

import math
from typing import List, Optional, Sequence

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import functions as _F

__all__ = [
    "safe_log", "mean_std_loudness", "multiscale_fft", "resample", "upsample", "remove_above_nyquist",
    "scale_function", "extract_loudness", "extract_pitch", "mlp", "gru", "harmonic_synth",
    "amp_to_impulse_response", "fft_convolve",
    "harmonic_synth_frames", "filtered_noise", "multiscale_spectral_loss", "convolve_stream", "extract_features",
    "extract_pitch_yin",
]


def safe_log(x):
    """ddsp/core.py:10-11."""
    return torch.log(x + 1e-7)


@torch.no_grad()
def mean_std_loudness(dataset):
    """ddsp/core.py:14-24: running mean of the per-batch loudness mean / std (host side)."""
    mean, std = 0.0, 0.0
    for count, batch in enumerate(dataset, start=1):
        loud = batch["loudness"]
        mean += (loud.mean().item() - mean) / count
        std += (loud.std().item() - std) / count
    return mean, std


def multiscale_fft(signal, scales: Sequence[int], overlap: float) -> List[torch.Tensor]:
    """ddsp/core.py:27-41: |STFT| of ``signal`` (B,N) at every scale, hop = int(s*(1-overlap)).
    Returns a list of (B, s/2+1, 1+N//hop) tensors, differentiable w.r.t. ``signal``."""
    squeeze = signal.dim() == 1
    sig = signal.unsqueeze(0) if squeeze else signal
    out = []
    for s in scales:
        mag = _F.StftMag.apply(sig, int(s), int(s * (1 - overlap)))
        out.append(mag[0] if squeeze else mag)
    return out


def resample(x, factor: int):
    """ddsp/core.py:44-61 (unused by the reference itself): zero-stuff by ``factor`` and smooth with
    a Hann kernel of 2*factor taps.  Kept for import compatibility; stock torch ops."""
    b, t, c = x.shape
    rows = x.permute(0, 2, 1).reshape(b * c, 1, t)
    stuffed = rows.new_zeros(b * c, 1, t * factor)
    stuffed[..., ::factor] = rows
    stuffed[..., -1:] = rows[..., -1:]
    kernel = torch.hann_window(2 * factor, dtype=x.dtype, device=x.device).view(1, 1, -1)
    smooth = nn.functional.conv1d(nn.functional.pad(stuffed, [factor, factor]), kernel)[..., :-1]
    return smooth.reshape(b, c, t * factor).permute(0, 2, 1)


def upsample(signal, factor):
    """ddsp/core.py:64-67: nearest-neighbour hold, (B,T,C) -> (B,T*factor,C).  F.interpolate's default
    mode is 'nearest', i.e. exactly repeat_interleave (SURVEY 0.3).  Inside the model this tensor
    is never materialised: HarmonicSynth.forward calls the fused frame-rate kernel instead."""
    return signal.repeat_interleave(int(factor), dim=1)


def remove_above_nyquist(amplitudes, f0, sample_rate):
    """ddsp/core.py:70-74."""
    return _F.RemoveAboveNyquist.apply(amplitudes, f0, float(sample_rate))


def scale_function(x):
    """ddsp/core.py:77-78."""
    return _F.ScaleFunction.apply(x)


def _feature_rows(signal, name: str):
    if torch.is_grad_enabled() and signal.requires_grad:
        raise RuntimeError(f"{name} has no backward: call it under torch.no_grad() or on a detached tensor")
    if signal.dim() not in (1, 2):
        raise ValueError(f"{name}: signal must be (N,) or (B, N), got {tuple(signal.shape)}")
    return signal.unsqueeze(0) if signal.dim() == 1 else signal


def _features(signal, sample_rate, block_size: int, n_fft: int, n_mfcc: int, mfcc: bool, name: str):
    rows = _feature_rows(signal, name)
    window, a_weight, mel, dct = _F.feature_tables(sample_rate, n_fft, n_mfcc, signal.device)
    loud, coeffs = _F._ops.features_fwd(rows, window, a_weight, mel, dct, int(n_fft), int(block_size), mfcc)
    if signal.dim() == 1:
        return loud[0], (coeffs[0] if mfcc else coeffs)
    return loud, coeffs


def extract_loudness(signal, sample_rate, block_size, n_fft=2048):
    """ddsp/core.py:81-97: A-weighted loudness, mean over bins of log(|STFT| + 1e-7) + A_weighting, one value per
    block.  A CUDA float32 tensor (N,) or (B, N) runs on the feature kernel (csrc/features.cu) and returns
    (..., N // block_size); anything else takes the reference's numpy + librosa code (offline preprocessing)."""
    if isinstance(signal, torch.Tensor) and signal.is_cuda and signal.dtype == torch.float32 and signal.dim() in (1, 2):
        loud, _ = _features(signal, sample_rate, block_size, n_fft, 1, False, "extract_loudness")
        return loud[..., :-1]
    import numpy as np
    import librosa as li
    spec = li.stft(signal, n_fft=n_fft, hop_length=block_size, win_length=n_fft, center=True)
    spec = np.log(abs(spec) + 1e-7)
    weight = li.A_weighting(li.fft_frequencies(sr=sample_rate, n_fft=n_fft))
    return np.mean(spec + weight.reshape(-1, 1), 0)[..., :-1]


def extract_pitch(signal, sample_rate, block_size):
    """ddsp/core.py:100-119 (offline preprocessing with CREPE; out of the hot path)."""
    import numpy as np
    import crepe
    length = signal.shape[-1] // block_size
    f0 = crepe.predict(signal, sample_rate, step_size=int(1000 * block_size / sample_rate),
                       verbose=1, center=True, viterbi=True)[1].reshape(-1)[:-1]
    if f0.shape[-1] != length:
        f0 = np.interp(np.linspace(0, 1, length, endpoint=False),
                       np.linspace(0, 1, f0.shape[-1], endpoint=False), f0)
    return f0


LINEAR3X_MIN_ROWS = 1        # every CUDA float32 call runs on the kernel (the realtime path's 2-row calls included)


class Linear(nn.Linear):
    """``nn.Linear`` (same parameters, state_dict keys and call) whose three GEMMs run on the tcgen05
    tensor cores with float32-class accuracy (csrc/gemm3x.cu, split-bf16) instead of cuBLAS's SIMT SGEMM.
    Every CUDA float32 call takes the kernel, whatever the row count and fan-in (the decoder's first layers have fan-in 1,
    the realtime path 2 rows); only non-CUDA / non-float32 inputs (the CPU tests) take the stock path."""

    __constants__ = ["in_features", "out_features", "min_rows"]

    def __init__(self, in_features: int, out_features: int, bias: bool = True):
        super().__init__(in_features, out_features, bias)
        self.min_rows: int = LINEAR3X_MIN_ROWS

    def forward(self, input: torch.Tensor) -> torch.Tensor:      # noqa: A002
        rows = input.numel() // max(1, input.shape[-1])
        fast = input.is_cuda and input.dtype == torch.float32 and rows >= self.min_rows
        if torch.jit.is_scripting():
            if fast:
                x2 = input.reshape(-1, self.in_features).contiguous()
                y = torch.ops.ddsp_b200.gemm3x_mm(torch.ops.ddsp_b200.gemm3x_split(x2, False),
                                                  torch.ops.ddsp_b200.gemm3x_split(self.weight, False),
                                                  x2.shape[0], self.out_features, self.in_features, self.bias,
                                                  False, False)
                return y.view(input.shape[:-1] + [self.out_features])
            return F.linear(input, self.weight, self.bias)
        if fast:
            return _F.Linear3x.apply(input, self.weight, self.bias)
        return F.linear(input, self.weight, self.bias)


class LayerNormLeakyReLU(nn.LayerNorm):
    """``nn.LayerNorm`` (same parameters and state_dict keys) that also applies the LeakyReLU which follows it
    in every MLP block, as one kernel each way (csrc/layernorm.cu).  Widths other than 128/256/384/512 and
    non-CUDA inputs compose the two stock ops."""

    __constants__ = ["normalized_shape", "eps", "elementwise_affine", "negative_slope", "fused"]

    def __init__(self, normalized_shape: int, negative_slope: float = 0.01):
        super().__init__(normalized_shape)
        self.negative_slope: float = negative_slope
        self.fused: bool = normalized_shape % 128 == 0 and 128 <= normalized_shape <= 512

    def forward(self, input: torch.Tensor) -> torch.Tensor:      # noqa: A002
        if self.fused and input.is_cuda and input.dtype == torch.float32:
            if torch.jit.is_scripting():
                return torch.ops.ddsp_b200.ln_lrelu_fwd(input, self.weight, self.bias, self.eps,
                                                        self.negative_slope, False)[0]
            return _F.LayerNormLeakyReLU.apply(input, self.weight, self.bias, self.eps, self.negative_slope)
        return F.leaky_relu(F.layer_norm(input, self.normalized_shape, self.weight, self.bias, self.eps),
                            self.negative_slope)


class FusedIntoLayerNorm(nn.Identity):
    """Placeholder at the Sequential index where the reference has ``nn.LeakyReLU`` (the activation is applied
    by the preceding LayerNormLeakyReLU), so that state_dict keys keep the reference's numbering."""


def mlp(in_size, hidden_size, n_layers):
    """ddsp/core.py:122-129: n_layers x (Linear, LayerNorm, LeakyReLU); same Sequential indices so
    state_dict keys match the reference's checkpoints."""
    sizes = [in_size] + [hidden_size] * n_layers
    layers = []
    for a, b in zip(sizes[:-1], sizes[1:]):
        layers += [Linear(a, b), LayerNormLeakyReLU(b), FusedIntoLayerNorm()]
    return nn.Sequential(*layers)


class ClusterGRU(nn.GRU):
    """``nn.GRU`` (same parameters, state_dict keys and call signature) whose recurrence runs as one
    cluster-persistent launch (csrc/gru.cu) instead of cuDNN's two launches per time step.  Used when the
    layer has the shape the reference's decoder and encoder build (one layer, batch_first, hidden 512) and the
    input is CUDA float32.  Any batch: above one pass of the resident clusters (70 voices on a B200) the kernel
    itself loops over groups of voices.  Other hidden sizes (the reference never builds one) and non-CUDA inputs
    take the stock path of the base class."""

    def _cluster_path(self, x, hx) -> bool:
        return (isinstance(x, torch.Tensor) and x.is_cuda and x.dtype == torch.float32 and x.dim() == 3
                and self.num_layers == 1 and not self.bidirectional and self.batch_first and self.bias
                and self.proj_size == 0 and not torch.jit.is_scripting()
                and x.shape[0] > 0 and int(_F._ops.gru_supported(self.hidden_size)) > 0)

    def forward(self, input, hx=None):      # noqa: A002 (nn.GRU's argument name)
        if not self._cluster_path(input, hx):
            return super().forward(input, hx)
        if input.shape[0] * input.shape[1] >= LINEAR3X_MIN_ROWS:
            gi = _F.Linear3x.apply(input, self.weight_ih_l0, self.bias_ih_l0)
        else:
            gi = F.linear(input, self.weight_ih_l0, self.bias_ih_l0)
        h0 = None
        if hx is not None:
            h0 = hx.expand(1, input.shape[0], self.hidden_size)[0].contiguous()
        y = _F.GRURecurrence.apply(gi, self.weight_hh_l0, self.bias_hh_l0, h0)
        return y, y[:, -1].unsqueeze(0)


def to_stock_layers(module: nn.Module) -> nn.Module:
    """Replace, in place, this file's control-net layers by the stock ``torch.nn`` ones the reference builds
    (same parameters, same state_dict keys): the A/B switch of the parity tests, ``tools/model_step.py`` and
    ``train.py --stock-control-net``."""
    for name, child in list(module.named_children()):
        if isinstance(child, Linear):
            new = nn.Linear(child.in_features, child.out_features, bias=child.bias is not None)
        elif isinstance(child, LayerNormLeakyReLU):
            new = nn.LayerNorm(child.normalized_shape, eps=child.eps)
        elif isinstance(child, FusedIntoLayerNorm):
            setattr(module, name, nn.LeakyReLU())
            continue
        elif isinstance(child, ClusterGRU):
            new = nn.GRU(child.input_size, child.hidden_size, batch_first=True)
        else:
            to_stock_layers(child)
            continue
        new = new.to(next(child.parameters()).device)
        new.load_state_dict(child.state_dict())
        setattr(module, name, new)
    return module


def gru(n_input, hidden_size):
    """ddsp/core.py:132-133."""
    return ClusterGRU(n_input * hidden_size, hidden_size, batch_first=True)


def harmonic_synth(f0, amplitudes, sample_rate):
    """ddsp/core.py:136-141, generic audio-rate signature: f0 (B,N,1), amplitudes (B,N,H) -> (B,N,1)."""
    return _F.HarmonicAudioRate.apply(f0, amplitudes, float(sample_rate))


def amp_to_impulse_response(amp, target_size):
    """ddsp/core.py:144-166."""
    return _F.AmpToImpulseResponse.apply(amp, int(target_size))


def fft_convolve(signal, kernel):
    """ddsp/core.py:169-176: causal convolution truncated to the signal length, last dim; leading
    dims broadcast like the reference's rfft product."""
    n = signal.shape[-1]
    lead = torch.broadcast_shapes(signal.shape[:-1], kernel.shape[:-1])
    rows = 1
    for d in lead:
        rows *= d
    sig2 = signal.expand(*lead, n).reshape(rows, n)
    k_rows = 1
    for d in kernel.shape[:-1]:
        k_rows *= d
    if k_rows == 1:
        ker2 = kernel.reshape(1, kernel.shape[-1])
    else:
        ker2 = kernel.expand(*lead, kernel.shape[-1]).reshape(rows, kernel.shape[-1])
    return _F.FFTConvolve.apply(sig2, ker2).reshape(*lead, n)


# ------------------------------------------------------------------------------------ extensions
def harmonic_synth_frames(f0, weights, block_size: int, sample_rate, phase0: Optional[torch.Tensor] = None):
    """Extension: the fused form of ``harmonic_synth(upsample(f0), upsample(weights))`` that
    HarmonicSynth.forward uses.  f0 (B,T,1), weights (B,T,H) -> (audio (B,T*block,1), phase_end (B)).
    ``phase0`` / ``phase_end`` carry the oscillator phase (turns, float64) across streaming calls."""
    return _F.HarmonicFrames.apply(f0, weights, int(block_size), float(sample_rate), phase0)


def harmonic_raw_supported(n_harmonic: int, block_size: int) -> bool:
    return bool(_F._ops.harmonic_raw_supported(int(n_harmonic), int(block_size)))


def harmonic_synth_from_raw(first, dist_raw, f0, block_size: int, sample_rate, phase0: Optional[torch.Tensor] = None):
    """Extension: ``HarmonicSynth.get_controls`` + ``HarmonicSynth.forward`` (modules.py:44-80) on the control net's raw
    outputs in one launch.  ``first`` = the projection output (B,T,H+1) and ``dist_raw=None``, or amp_raw (B,T,1) and
    dist_raw (B,T,H).  -> (audio, phase_end, amplitudes, weights = normalised distribution x amplitudes)."""
    return _F.HarmonicFromRaw.apply(first, dist_raw, f0, int(block_size), float(sample_rate), phase0)


def filtered_noise(magnitudes, noise):
    """Extension: FilteredNoise.forward with the uniform(-1,1) draw passed in (B,T,block)."""
    return _F.FilteredNoise.apply(magnitudes, noise)


def convolve_stream(signal, kernel, history: Optional[torch.Tensor] = None):
    """Extension: one buffer of a causal convolution that continues across calls (Reverb.forward, modules.py:28-35,
    played buffer by buffer).  signal (B,N), kernel with L taps (L elements, e.g. (L,) or (1,L) or the reverb's
    (1,L,1) impulse), history (B,L-1) = the previous L-1 input samples, oldest first; None = silence before.
    -> (out (B,N), history (B,L-1) for the next call).  out[b,n] = sum_k kernel[k] * [history | signal][b, L-1+n-k].
    Direct form, B*N*L FMA.  Forward only: inputs that require grad raise under grad mode."""
    L = kernel.numel()
    if history is None:
        history = signal.new_zeros(signal.shape[0], max(L - 1, 0))
    if torch.is_grad_enabled() and any(t.requires_grad for t in (signal, kernel, history)):
        raise RuntimeError("convolve_stream has no backward: call it under torch.no_grad() or on detached tensors")
    return _F._ops.conv_stream_fwd(signal, kernel, history)


def extract_features(signal, sample_rate, block_size, n_mfcc=30, n_fft=2048):
    """Extension: the two signal-processing features of a dataset from one pass of the feature kernel over a CUDA
    float32 signal (N,) or (B, N): -> (loudness (..., N // block_size) as ``extract_loudness``,
    mfcc (..., 1 + N // block_size, n_mfcc) as ``librosa.feature.mfcc(y, sr, n_mfcc=n_mfcc, n_fft=n_fft,
    hop_length=block_size)`` with its defaults: 128 Slaney mel bands, power_to_db with top_db = 80 per row,
    DCT-II ortho; the layout of ``mfccs.npy``).  Forward only: an input that requires grad raises under grad mode."""
    if not 1 <= int(n_mfcc) <= _F.N_MELS:
        raise ValueError(f"extract_features: n_mfcc must be in 1..{_F.N_MELS}, got {n_mfcc}")
    loud, mfcc = _features(signal, sample_rate, block_size, n_fft, int(n_mfcc), True, "extract_features")
    return loud[..., :-1], mfcc


def _yin_periods(sample_rate, fmin, fmax, frame_length: int = 2048):
    """The lag range of ``extract_pitch_yin``, in samples, as librosa.yin derives it:
    (max(floor(sr / fmax), 1), min(ceil(sr / fmin), frame_length - frame_length // 2 - 1))."""
    sr, fmin, fmax = float(sample_rate), float(fmin), float(fmax)
    if not fmin > 0.0:
        raise ValueError(f"extract_pitch_yin: fmin must be > 0, got {fmin}")
    if not fmin < fmax:
        raise ValueError(f"extract_pitch_yin: fmin ({fmin}) must be below fmax ({fmax})")
    if fmax > sr / 2:
        raise ValueError(f"extract_pitch_yin: fmax ({fmax}) is above the Nyquist frequency ({sr / 2})")
    L = int(frame_length)
    min_period = max(int(math.floor(sr / fmax)), 1)
    max_period = min(int(math.ceil(sr / fmin)), L - L // 2 - 1)
    if max_period < min_period + 2:
        raise ValueError(f"extract_pitch_yin: the lag range {min_period}..{max_period} of fmin {fmin}, fmax {fmax} at "
                         f"frame_length {L} is empty (it needs three lags at least)")
    return min_period, max_period


def extract_pitch_yin(signal, sample_rate, block_size, fmin, fmax, frame_length=2048, threshold=0.1):
    """Extension: the pitch of a CUDA float32 signal (N,) or (B, N) by YIN (csrc/pitch.cu), one value per block like
    ``extract_pitch`` and ``extract_loudness``: -> (f0 (..., N // block_size) in Hz, aperiodicity (..., N // block_size)).
    librosa.yin's definition with the frames of ``extract_loudness`` (reflect padding of frame_length/2, window
    frame_length/2): the first trough of the cumulative mean normalised difference below ``threshold``, else its
    global minimum, refined by a parabola.  The aperiodicity is the normalised difference at the chosen lag (YIN's
    voicing measure: small for periodic frames).  No smoothing: unvoiced frames take the global minimum, and an
    all-zero frame gives f0 = sample_rate / floor(sample_rate / fmax) with aperiodicity 0, as in librosa.
    Forward only: an input that requires grad raises under grad mode."""
    rows = _feature_rows(signal, "extract_pitch_yin")
    min_period, max_period = _yin_periods(sample_rate, fmin, fmax, frame_length)
    f0, ap = _F._ops.pitch_yin_fwd(rows, int(frame_length), int(block_size), min_period, max_period,
                                   float(sample_rate), float(threshold))
    if signal.dim() == 1:
        return f0[0], ap[0]
    return f0, ap


def multiscale_spectral_loss(target, rec, scales: Sequence[int], overlap: float):
    """Extension: train.py:70-76 applied to multiscale_fft(target), multiscale_fft(rec), as one fused
    op (the magnitude lists are never written to HBM).  Differentiable w.r.t. ``rec`` only."""
    return _F.MultiScaleSpectralLoss.apply(target, rec, [int(s) for s in scales], float(overlap))
