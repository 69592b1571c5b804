"""TorchScript export of a trained decoder for the realtime host (SURVEY 8f rank 1).

The reference's ``export.py`` does not run in its fork (SURVEY 3.3: stale attribute names, ``**kwargs``
in the scripted path, ``realtime_forward`` not exported).  This module provides the capability it was
meant to give: a scripted module with the reference's calling convention
(``export.py:33-40``: ``forward(pitch, loudness)`` with audio-rate (B, N, 1) inputs, loudness standardised
with the dataset mean/std, inputs strided to frame rate by ``block_size``) whose graph calls the
``ddsp_b200::*_fwd`` custom ops directly -- inference needs no autograd wrappers, matching the
``torch::NoGradGuard`` of ``ddsp_model.cpp:34``.

Streaming state lives in buffers: the GRU hidden state (``cache_gru``, as the reference) and the
oscillator phase (``phase``: the reference registers it at decoder.py:99 and never uses it, so every
1024-sample buffer restarted the phase at zero).  A realtime export is dry by default; with
``streaming_reverb=True`` it also plays the trained reverb, carrying the last L-1 samples of the reverb's input
in ``reverb_history`` so that the impulse's tail runs on into the following buffers.  The C++ host must load
``libddsp_b200_torch.so`` before ``torch::jit::load`` (INTEGRATION.md section 4).
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn as nn

from ._lib import get_ops
from .models.decoder import DDSPDecoder


class ScriptDDSP(nn.Module):
    # compile-time constants: the scripted graph only contains the branches that are taken
    __constants__ = ["block_size", "sample_rate", "reverb_length", "has_reverb", "realtime", "device_noise",
                     "mean_loudness", "std_loudness", "noise_bias", "cluster_gru", "streaming_reverb"]

    def __init__(self, ddsp: DDSPDecoder, mean_loudness: float, std_loudness: float, realtime: bool = True,
                 device_noise: bool = True, streaming_reverb: bool = False):
        super().__init__()
        if streaming_reverb and not (realtime and ddsp.has_reverb):
            raise ValueError("streaming_reverb needs realtime=True and a model built with has_reverb=True")
        dec = ddsp.decoder
        assert not dec.add_z, "export covers the f0 + loudness decoder (config.yaml's single-inst-decoder)"
        self.f0_mlp = dec.f0_mlp
        self.loudness_mlp = dec.loudness_mlp
        # a stock nn.GRU holds the weights in the scripted module (ClusterGRU's forward is Python-side
        # dispatch); the graph calls ddsp_b200::gru_fwd on them when the kernel covers the layer
        self.gru = nn.GRU(dec.gru.input_size, dec.gru.hidden_size, batch_first=True)
        self.gru.load_state_dict(dec.gru.state_dict())
        self.gru.to(dec.cache_gru.device)
        self.cluster_gru: bool = bool(dec.cache_gru.is_cuda and get_ops().gru_supported(dec.gru.hidden_size) > 0)
        self.out_mlp = dec.out_mlp
        self.harmonic_proj = ddsp.harmonic_proj
        self.noise_proj = ddsp.noise_proj
        self.register_buffer("cache_gru", torch.zeros_like(dec.cache_gru))
        self.register_buffer("phase", torch.zeros(1, dtype=torch.float64))
        self.register_buffer("reverb_noise", ddsp.reverb.noise.detach().clone())
        self.register_buffer("reverb_decay", ddsp.reverb.decay.detach().clone())
        self.register_buffer("reverb_wet", ddsp.reverb.wet.detach().clone())
        self.register_buffer("reverb_t", ddsp.reverb.t.detach().clone())
        self.block_size: int = int(ddsp.block_size)
        self.sample_rate: float = float(ddsp.sample_rate)
        self.reverb_length: int = int(ddsp.reverb.length)
        self.has_reverb: bool = bool(ddsp.has_reverb) and not realtime     # the host convolves (patches/example.pd)
        # realtime reverb: the last L-1 samples of the reverb's input, batch 1 like cache_gru and phase
        self.streaming_reverb: bool = bool(streaming_reverb)
        if self.streaming_reverb:
            self.register_buffer("reverb_history", torch.zeros(1, self.reverb_length - 1,
                                                               device=ddsp.reverb.noise.device))
        self.realtime: bool = realtime
        self.device_noise: bool = device_noise
        self.mean_loudness: float = float(mean_loudness)
        self.std_loudness: float = float(std_loudness)
        self.noise_bias: float = float(ddsp.noise_synth.initial_bias)
        self.fused_controls: bool = bool(torch.ops.ddsp_b200.harmonic_raw_supported(
            int(ddsp.harmonic_proj.out_features) - 1, self.block_size))

    def forward(self, pitch: torch.Tensor, loudness: torch.Tensor) -> torch.Tensor:
        """pitch, loudness: (B, N, 1) at audio rate, N a multiple of block_size -> audio (B, N, 1)."""
        loudness = (loudness - self.mean_loudness) / self.std_loudness
        f0 = pitch[:, ::self.block_size].contiguous()
        ld = loudness[:, ::self.block_size].contiguous()
        hidden = torch.cat([self.f0_mlp(f0), self.loudness_mlp(ld)], -1)
        if self.cluster_gru:
            gi = torch.nn.functional.linear(hidden, self.gru.weight_ih_l0, self.gru.bias_ih_l0)
            h0: Optional[torch.Tensor] = None
            if self.realtime:
                h0 = self.cache_gru.expand(1, hidden.shape[0], hidden.shape[2] // 2)[0].contiguous()
            gru_out = torch.ops.ddsp_b200.gru_fwd(gi, self.gru.weight_hh_l0, self.gru.bias_hh_l0, h0, False)[0]
            if self.realtime:
                self.cache_gru.copy_(gru_out[:1, -1:])
        elif self.realtime:
            gru_out, cache = self.gru(hidden, self.cache_gru)
            self.cache_gru.copy_(cache)
        else:
            gru_out = self.gru(hidden)[0]
        hidden = self.out_mlp(torch.cat([gru_out, f0, ld], -1))

        param = self.harmonic_proj(hidden)
        phase0: Optional[torch.Tensor] = None
        if self.realtime:
            phase0 = self.phase.expand(f0.shape[0]).contiguous()
        if self.fused_controls:      # get_controls inside the oscillator bank's launch, param read in place
            audio, phase_end, phi, delta, amps, weights = torch.ops.ddsp_b200.harmonic_raw_fwd(
                param, None, f0, self.block_size, self.sample_rate, phase0)
        else:
            amps, dist, weights = torch.ops.ddsp_b200.harmonic_controls_fwd(
                param[..., :1], param[..., 1:], f0, self.sample_rate, True)
            audio, phase_end, phi, delta = torch.ops.ddsp_b200.harmonic_fwd(
                f0, weights, self.block_size, self.sample_rate, phase0)
        if self.realtime:
            self.phase.copy_(phase_end[:1])

        mags = self.noise_proj(hidden)
        if self.device_noise:
            noise = torch.rand(mags.shape[0], mags.shape[1], self.block_size, device=mags.device) * 2 - 1
        else:       # modules.py:119-123: CPU generator, then moved
            noise = torch.rand(mags.shape[0], mags.shape[1], self.block_size).to(mags) * 2 - 1
        signal = torch.ops.ddsp_b200.noise_fwd(mags, noise, audio, True, self.noise_bias)

        if self.has_reverb:
            impulse = torch.ops.ddsp_b200.reverb_impulse_fwd(self.reverb_noise, self.reverb_decay, self.reverb_wet,
                                                             self.reverb_t)
            taps = min(signal.shape[1], self.reverb_length)
            kernel = impulse.reshape(1, self.reverb_length)[:, :taps]
            signal = torch.ops.ddsp_b200.fftconv_fwd(signal.squeeze(-1), kernel, False)[0].unsqueeze(-1)
        if self.streaming_reverb:
            impulse = torch.ops.ddsp_b200.reverb_impulse_fwd(self.reverb_noise, self.reverb_decay, self.reverb_wet,
                                                             self.reverb_t)
            history = self.reverb_history.expand(signal.shape[0], self.reverb_length - 1).contiguous()
            wet, history = torch.ops.ddsp_b200.conv_stream_fwd(signal.squeeze(-1), impulse, history)
            self.reverb_history.copy_(history[:1])
            signal = wet.unsqueeze(-1)
        return signal

    @torch.jit.export
    def reset(self):
        """Forget the streaming state (GRU cache, oscillator phase and, when streamed, the reverb's input)."""
        self.cache_gru.zero_()
        self.phase.zero_()
        if self.streaming_reverb:
            self.reverb_history.zero_()


def export_torchscript(model: DDSPDecoder, path: str, mean_loudness: float = 0.0, std_loudness: float = 1.0,
                       realtime: bool = True, device_noise: bool = True,
                       streaming_reverb: bool = False) -> torch.jit.ScriptModule:
    """export.py:55-65: script the wrapper and save it to ``path`` (a ``.ts`` file).  ``streaming_reverb``
    (realtime exports of a model with ``has_reverb`` only): play the trained reverb, its tail carried across calls."""
    wrapper = ScriptDDSP(model.eval(), mean_loudness, std_loudness, realtime, device_noise, streaming_reverb).eval()
    scripted = torch.jit.script(wrapper)
    torch.jit.save(scripted, path)
    return scripted
