"""GPU parity tests: the sm_100a kernels (through the TORCH_LIBRARY shim -> C ABI) against the CPU
oracle evaluated in float64 and against the golden vectors made from the real reference.

Tolerances (BASELINE.json north_star): audio <= 1e-4 max abs; gradients <= 1e-3 relative, per op
with a fixed grad_output (never end to end, SURVEY 0.5); the MSS-loss gradient is judged against
the reference float32 path's own deviation recorded in the fixture.
"""
import math

import numpy as np
import pytest
import torch

from conftest import load_golden

pytestmark = pytest.mark.gpu

AUDIO_TOL = 1e-4
GRAD_REL = 1e-3


@pytest.fixture(scope="module")
def ddsp():
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    import ddsp_pytorch_b200 as pkg
    return pkg


@pytest.fixture(scope="module")
def orc():
    from oracle import ddsp_oracle
    return ddsp_oracle


def dev(a, grad=False):
    t = torch.as_tensor(np.asarray(a), dtype=torch.float32).cuda()
    return t.requires_grad_(True) if grad else t


def t64(a, grad=False):
    t = torch.as_tensor(np.asarray(a), dtype=torch.float64)
    return t.requires_grad_(True) if grad else t


def _ref64(ref):
    if isinstance(ref, torch.Tensor):
        return ref.detach().double().cpu()
    return torch.as_tensor(np.asarray(ref)).double()


def max_abs(got, ref):
    return float((got.detach().double().cpu() - _ref64(ref)).abs().max())


def rel_err(got, ref):
    ref = _ref64(ref)
    return float((got.detach().double().cpu() - ref).norm() / ref.norm().clamp_min(1e-30))


def assert_audio(got, ref, tol=AUDIO_TOL):
    e = max_abs(got, ref)
    assert e <= tol, f"max abs error {e:.3e} > {tol:.1e}"


def assert_grad(got, ref, tol=GRAD_REL):
    e = rel_err(got, ref)
    assert e <= tol, f"relative error {e:.3e} > {tol:.1e}"


SYNTH = ["synth_c1_small", "synth_c3_buffer", "synth_h100"]


# ------------------------------------------------------------------------------- a1, a2, a3
def test_scale_function(ddsp, orc):
    x = torch.linspace(-30, 30, 4001, dtype=torch.float64).requires_grad_(True)
    y = orc.scale_function(x)
    go = torch.randn(4001, dtype=torch.float64, generator=torch.Generator().manual_seed(0))
    (y * go).sum().backward()
    xd = dev(x.detach(), grad=True)
    yd = ddsp.scale_function(xd)
    assert float(((yd.double().cpu() - y.detach()).abs() / y.detach()).max()) < 5e-6
    (yd * dev(go)).sum().backward()
    assert_grad(xd.grad, x.grad, 1e-5)


def test_remove_above_nyquist_mask_is_float32_exact(ddsp, orc):
    g = torch.Generator().manual_seed(1)
    f0 = (torch.rand(3, 50, 1, generator=g) * 700 + 60)
    f0[0, 0, 0] = 8000.0 / 7          # k*f0 lands next to Nyquist: the float32 product must decide
    amp = torch.rand(3, 50, 40, generator=g)
    ref = orc.remove_above_nyquist(amp, f0, 16000)             # float32 reference arithmetic
    got = ddsp.remove_above_nyquist(amp.cuda(), f0.cuda(), 16000)
    assert torch.equal(got.cpu(), ref), "mask must match the float32 reference bit for bit"
    a = amp.cuda().requires_grad_(True)
    ddsp.remove_above_nyquist(a, f0.cuda(), 16000).sum().backward()
    assert torch.equal(a.grad.cpu(), orc.remove_above_nyquist(torch.ones_like(amp), f0, 16000))


@pytest.mark.parametrize("name", SYNTH)
def test_harmonic_controls(ddsp, orc, name):
    g = load_golden(name)
    sr = int(g["sr"])
    from ddsp_pytorch_b200.models.modules import HarmonicSynth
    hs = HarmonicSynth(int(g["bs"]), sr)
    a, d = dev(g["amp_raw"], True), dev(g["dist_raw"], True)
    c = hs.get_controls(a, d, dev(g["f0"]))
    assert max_abs(c["amplitudes"], g["amps"]) < 2e-6
    assert max_abs(c["harmonic_distribution"], g["dist"]) < 2e-6
    # per-op gradient with a fixed grad_output, against float64 autograd of the oracle
    gen = torch.Generator().manual_seed(5)
    ga = torch.randn(g["amps"].shape, generator=gen, dtype=torch.float64)
    gd = torch.randn(g["dist"].shape, generator=gen, dtype=torch.float64)
    a64, d64 = t64(g["amp_raw"], True), t64(g["dist_raw"], True)
    c64 = orc.harmonic_controls(a64, d64, t64(g["f0"]), sr)
    ((c64["amplitudes"] * ga).sum() + (c64["harmonic_distribution"] * gd).sum()).backward()
    ((c["amplitudes"] * dev(ga)).sum() + (c["harmonic_distribution"] * dev(gd)).sum()).backward()
    assert_grad(a.grad, a64.grad, 1e-4)
    assert_grad(d.grad, d64.grad, 1e-4)


# ------------------------------------------------------------------------------- a4, a5, a6
@pytest.mark.parametrize("name", SYNTH)
def test_harmonic_frames_golden(ddsp, name):
    g = load_golden(name)
    bs, sr = int(g["bs"]), int(g["sr"])
    w = dev(g["dist"] * g["amps"], True)
    f0 = dev(g["f0"], True)
    audio, _ = ddsp.harmonic_synth_frames(f0, w, bs, sr)
    assert_audio(audio, g["harm"])
    # the reference's own float32 path deviates more than we do from float64
    assert max_abs(audio, g["harm"]) <= max(float(g["dev32_harm"]), 2e-5)
    (audio * dev(g["g_harm"])).sum().backward()
    # d weights: golden holds grads w.r.t. the raw controls; compare d_weights against the oracle
    from oracle import ddsp_oracle as orc
    w64 = t64(g["dist"] * g["amps"], True)
    f64 = t64(g["f0"], True)
    y64 = orc.harmonic_synth(orc.upsample(f64, bs), orc.upsample(w64, bs), sr)
    (y64 * t64(g["g_harm"])).sum().backward()
    assert_grad(w.grad, w64.grad)
    assert_grad(f0.grad, f64.grad)
    assert_grad(f0.grad, g["d_f0"])


def test_harmonic_module_chain_grads(ddsp):
    """controls -> in-place scaling -> fused synth, gradients w.r.t. the raw decoder outputs."""
    g = load_golden("synth_c1_small")
    from ddsp_pytorch_b200.models.modules import HarmonicSynth
    hs = HarmonicSynth(int(g["bs"]), int(g["sr"]))
    a, d = dev(g["amp_raw"], True), dev(g["dist_raw"], True)
    c = hs.get_controls(a, d, dev(g["f0"]))
    y = hs(**c)
    assert_audio(y, g["harm"])
    # SURVEY 3.2: after forward the dict holds distribution x amplitude
    assert max_abs(c["harmonic_distribution"], g["dist"] * g["amps"]) < 2e-6
    (y * dev(g["g_harm"])).sum().backward()
    assert_grad(a.grad, g["d_amp_raw"])
    assert_grad(d.grad, g["d_dist_raw"])


def test_harmonic_frames_config1_shapes(ddsp, orc):
    """B=2 slice of config 1 (16 kHz, block 160, 100 harmonics, 4 s) against the float64 oracle."""
    gen = torch.Generator().manual_seed(3)
    B, T, bs, H, sr = 2, 400, 160, 100, 16000
    f0 = torch.rand(B, T, 1, generator=gen) * 700 + 80
    w = torch.rand(B, T, H, generator=gen) * (2.0 / H)
    ref = orc.harmonic_synth(orc.upsample(f0.double(), bs), orc.upsample(w.double(), bs), sr)
    got, phase_end = ddsp.harmonic_synth_frames(f0.cuda(), w.cuda(), bs, sr)
    assert_audio(got, ref)
    ref32 = orc.harmonic_synth(orc.upsample(f0, bs), orc.upsample(w, bs), sr)
    assert max_abs(got, ref) < max_abs(ref32, ref), "must beat the reference's float32 phase error"
    turns = (f0.double()[..., 0] / sr).sum(1) * bs
    d = (phase_end.cpu() - (turns - turns.floor())).abs()
    assert float(torch.minimum(d, 1 - d).max()) < 1e-9


def test_harmonic_frames_config4_shapes_and_reseed(ddsp, orc):
    """48 kHz, block 512, 256 harmonics (crosses the recurrence re-seed at harmonic 129); and 2000 harmonics at
    block 160, a weight table too large for 16 frames per CTA (the forward takes fewer frames per CTA)."""
    gen = torch.Generator().manual_seed(4)
    for B, T, bs, H, sr in ((1, 24, 512, 256, 48000), (1, 20, 160, 2000, 16000)):
        f0 = torch.rand(B, T, 1, generator=gen) * 120 + 40
        w = torch.rand(B, T, H, generator=gen) * (2.0 / H)
        ref = orc.harmonic_synth(orc.upsample(f0.double(), bs), orc.upsample(w.double(), bs), sr)
        wd = w.cuda().requires_grad_(True)
        got, _ = ddsp.harmonic_synth_frames(f0.cuda(), wd, bs, sr)
        assert_audio(got, ref)
        go = torch.randn(B, T * bs, 1, generator=gen)
        (got * go.cuda()).sum().backward()
        w64 = w.double().requires_grad_(True)
        y = orc.harmonic_synth(orc.upsample(f0.double(), bs), orc.upsample(w64, bs), sr)
        (y * go.double()).sum().backward()
        assert_grad(wd.grad, w64.grad)


def test_harmonic_frames_odd_block_and_streaming(ddsp, orc):
    """block sizes that are not multiples of 4 / 2, and phase carry across two calls."""
    gen = torch.Generator().manual_seed(6)
    for bs in (6, 50, 37):
        B, T, H, sr = 2, 9, 7, 8000
        f0 = torch.rand(B, T, 1, generator=gen) * 300 + 50
        w = torch.rand(B, T, H, generator=gen)
        ref = orc.harmonic_synth(orc.upsample(f0.double(), bs), orc.upsample(w.double(), bs), sr)
        got, _ = ddsp.harmonic_synth_frames(f0.cuda(), w.cuda(), bs, sr)
        assert_audio(got, ref, 2e-5 * H)
        a, pe = ddsp.harmonic_synth_frames(f0[:, :4].cuda(), w[:, :4].cuda(), bs, sr)
        b, _ = ddsp.harmonic_synth_frames(f0[:, 4:].cuda(), w[:, 4:].cuda(), bs, sr, pe)
        assert_audio(torch.cat([a, b], 1), ref, 2e-5 * H)


def test_harmonic_audio_rate_golden(ddsp):
    g = load_golden("harmonic_audio_rate")
    f0, amps = dev(g["f0"], True), dev(g["amps"], True)
    y = ddsp.harmonic_synth(f0, amps, int(g["sr"]))
    assert y.shape == g["y"].shape
    assert_audio(y, g["y"])
    (y * dev(g["go"])).sum().backward()
    assert_grad(amps.grad, g["d_amps"])
    assert_grad(f0.grad, g["d_f0"])


def test_harmonic_audio_rate_equals_frames(ddsp):
    gen = torch.Generator().manual_seed(7)
    B, T, bs, H, sr = 2, 20, 160, 100, 16000
    f0 = (torch.rand(B, T, 1, generator=gen) * 700 + 80).cuda()
    w = (torch.rand(B, T, H, generator=gen) / H).cuda()
    a, _ = ddsp.harmonic_synth_frames(f0, w, bs, sr)
    b = ddsp.harmonic_synth(ddsp.upsample(f0, bs), ddsp.upsample(w, bs), sr)
    assert max_abs(a, b.cpu()) < 2e-5


# ------------------------------------------------------------------------------- a7, a8, a9
@pytest.mark.parametrize("name", SYNTH)
def test_filtered_noise_golden(ddsp, name):
    g = load_golden(name)
    from ddsp_pytorch_b200.models.modules import FilteredNoise
    fn = FilteredNoise(int(g["bs"]), int(g["NB"]))
    m = dev(g["mag_raw"], True)
    mags = fn.get_controls(m)["magnitudes"]
    assert max_abs(mags, g["mags"]) < 1e-6
    y = fn(mags, noise=dev(g["noise"]))
    assert y.shape == g["nz"].shape
    assert_audio(y, g["nz"], 1e-6)
    (y * dev(g["g_noise"])).sum().backward()
    assert_grad(m.grad, g["d_mag_raw"])


def test_filtered_noise_draw_matches_reference_generator(ddsp, orc):
    from ddsp_pytorch_b200.models.modules import FilteredNoise
    fn = FilteredNoise(160, 65)
    mags = torch.rand(2, 5, 65).cuda()
    torch.manual_seed(123)
    y = fn(mags)
    torch.manual_seed(123)
    noise = orc.draw_noise(2, 5, 160)
    ref = orc.filtered_noise(mags.double().cpu(), noise.double(), 160)
    assert_audio(y, ref, 1e-6)


def test_amp_to_impulse_response_golden(ddsp):
    g = load_golden("impulse_response")
    for tag in "abcd":
        amp = dev(g[f"{tag}_amp"], True)
        ir = ddsp.amp_to_impulse_response(amp, int(g[f"{tag}_ts"]))
        assert ir.shape == g[f"{tag}_ir"].shape
        assert_audio(ir, g[f"{tag}_ir"], 1e-6)
        (ir * dev(g[f"{tag}_go"])).sum().backward()
        assert_grad(amp.grad, g[f"{tag}_damp"], 1e-4)


def test_fft_convolve_golden(ddsp):
    g = load_golden("fft_convolve")
    for tag in "abc":
        s, k = dev(g[f"{tag}_s"], True), dev(g[f"{tag}_k"], True)
        y = ddsp.fft_convolve(s, k)
        assert y.shape == g[f"{tag}_y"].shape
        scale = max(1.0, float(np.abs(g[f"{tag}_y"]).max()))
        assert_audio(y, g[f"{tag}_y"], 2e-5 * scale)
        (y * dev(g[f"{tag}_go"])).sum().backward()
        assert_grad(s.grad, g[f"{tag}_ds"], 1e-4)
        assert_grad(k.grad, g[f"{tag}_dk"], 1e-4)


# ------------------------------------------------------------------------------- a10
@pytest.mark.parametrize("name", ["reverb_pad", "reverb_crop"])
def test_reverb_golden(ddsp, name):
    g = load_golden(name)
    from ddsp_pytorch_b200.models.modules import Reverb
    rv = Reverb(int(g["L"]), int(g["sr"]))
    rv.load_state_dict({"noise": torch.as_tensor(g["noise"]).float(), "decay": torch.as_tensor(g["decay"]).float(),
                        "wet": torch.as_tensor(g["wet"]).float(), "t": torch.as_tensor(g["t"]).float()})
    rv.cuda()
    assert max_abs(rv.build_impulse(), g["impulse"]) < 1e-6
    x = dev(g["x"], True)
    y = rv(x)
    assert y.shape == g["y"].shape
    assert_audio(y, g["y"], 2e-5 * max(1.0, float(np.abs(g["y"]).max())))
    (y * dev(g["go"])).sum().backward()
    assert_grad(x.grad, g["d_x"], 1e-4)
    assert_grad(rv.noise.grad, g["d_noise"], 1e-4)
    assert abs(float(rv.decay.grad) - float(g["d_decay"])) <= 1e-3 * abs(float(g["d_decay"])) + 1e-6
    assert abs(float(rv.wet.grad) - float(g["d_wet"])) <= 1e-3 * abs(float(g["d_wet"])) + 1e-6


def test_reverb_config1_shapes(ddsp, orc):
    """L = sr = 16000 taps over 4 s, B = 3 (odd: exercises the unpaired voice)."""
    torch.manual_seed(0)
    from ddsp_pytorch_b200.models.modules import Reverb
    rv = Reverb(16000, 16000, initial_wet=1.0, initial_decay=3.0)
    x = torch.randn(3, 64000, 1) * 0.1
    ref = orc.reverb(x.double(), rv.noise.detach().double(), rv.decay.detach().double(),
                     rv.wet.detach().double(), rv.t.double())
    y = rv.cuda()(x.cuda())
    assert_audio(y, ref, 1e-4)


# ------------------------------------------------------------------------------- a11, a12
@pytest.mark.parametrize("name", ["mss_full_scales", "mss_small"])
def test_multiscale_fft_golden(ddsp, name):
    g = load_golden(name)
    scales, ov = [int(s) for s in g["scales"]], float(g["overlap"])
    rec = dev(g["rec"], True)
    mags = ddsp.multiscale_fft(rec, scales, ov)
    for s, m in zip(scales, mags):
        assert m.shape == g[f"mag_rec_{s}"].shape
        assert_audio(m, g[f"mag_rec_{s}"], 2e-6)
        (gr,) = torch.autograd.grad((m * dev(g[f"go_{s}"])).sum(), rec, retain_graph=True)
        assert_grad(gr, g[f"d_rec_{s}"], 1e-4)


@pytest.mark.parametrize("name", ["mss_full_scales", "mss_small"])
def test_mss_loss_fused_golden(ddsp, name):
    g = load_golden(name)
    scales, ov = [int(s) for s in g["scales"]], float(g["overlap"])
    rec = dev(g["rec"], True)
    loss = ddsp.multiscale_spectral_loss(dev(g["tgt"]), rec, scales, ov)
    assert abs(float(loss) - float(g["loss"])) <= 2e-6 * abs(float(g["loss"]))
    loss.backward()
    # L1 sign ties: the reference's own float32 gradient is this far from float64 (SURVEY 8c)
    bound = max(GRAD_REL, 1.5 * float(g["dev32_d_rec_rel"]))
    assert_grad(rec.grad, g["d_rec"], bound)
    # list API + train.py's loss give the same number
    mt = ddsp.multiscale_fft(dev(g["tgt"]), scales, ov)
    mr = ddsp.multiscale_fft(rec.detach(), scales, ov)
    l2 = sum((a - b).abs().mean() + (ddsp.safe_log(a) - ddsp.safe_log(b)).abs().mean() for a, b in zip(mt, mr))
    assert abs(float(l2) - float(g["loss"])) <= 2e-6 * abs(float(g["loss"]))


def test_mss_loss_config_shapes_and_determinism(ddsp, orc):
    gen = torch.Generator().manual_seed(11)
    B, N = 2, 64000
    scales, ov = [4096, 2048, 1024, 512, 256, 128], 0.75
    tgt = 0.1 * torch.randn(B, N, generator=gen)
    rec = 0.1 * torch.randn(B, N, generator=gen)
    r64 = rec.double().requires_grad_(True)
    ref = orc.mss_loss(tgt.double(), r64, scales, ov)
    ref.backward()
    r = rec.cuda().requires_grad_(True)
    loss = ddsp.multiscale_spectral_loss(tgt.cuda(), r, scales, ov)
    loss.backward()
    assert abs(float(loss) - float(ref)) <= 5e-6 * abs(float(ref))
    r32 = rec.clone().requires_grad_(True)
    orc.mss_loss(tgt, r32, scales, ov).backward()
    ref32_dev = float((r32.grad.double() - r64.grad).norm() / r64.grad.norm())
    assert_grad(r.grad, r64.grad, max(GRAD_REL, 1.5 * ref32_dev))
    r2 = rec.cuda().requires_grad_(True)
    loss2 = ddsp.multiscale_spectral_loss(tgt.cuda(), r2, scales, ov)
    loss2.backward()
    assert torch.equal(loss, loss2) and torch.equal(r.grad, r2.grad), "no atomics: bit-reproducible"


# ------------------------------------------------------------------------------- a14 models
@pytest.mark.parametrize("name,cls", [("model_decoder", "DDSPDecoder"), ("model_autoencoder", "DDSPAutoencoder")])
def test_model_forward_matches_reference(ddsp, name, cls):
    g = load_golden(name)
    from ddsp_pytorch_b200.models import decoder, encoder
    ctor = getattr(decoder, cls, None) or getattr(encoder, cls)
    model = ctor(hidden_size=16, n_harmonic=12, n_bands=65, sample_rate=16000, block_size=160, has_reverb=True)
    sd = {k[3:]: torch.as_tensor(v) for k, v in g.items() if k.startswith("sd_")}
    assert set(sd) == set(model.state_dict()), "state_dict keys must equal the reference's"
    model.load_state_dict(sd)
    model.cuda()
    batch = {k[3:]: torch.as_tensor(v).cuda() for k, v in g.items() if k.startswith("in_")}
    torch.manual_seed(int(g["noise_seed"]))
    out = model(batch)
    for key in ["signal", "noise", "harmonic_audio"]:
        assert out[key].shape == g["out_" + key].shape
        assert_audio(out[key], g["out_" + key], 1e-4)
    assert max_abs(out["harmonic_ctrls"]["harmonic_distribution"], g["out_harmonic_distribution"]) < 1e-5
    assert max_abs(out["noise_ctrls"]["magnitudes"], g["out_magnitudes"]) < 1e-5
    assert set(out) >= {"f0", "loudness", "signal", "noise", "harmonic_audio", "noise_ctrls", "harmonic_ctrls"}
    out["signal"].square().mean().backward()
    assert all(p.grad is not None and torch.isfinite(p.grad).all() for n, p in model.named_parameters()
               if not n.startswith("decoder.z") or True)


# ------------------------------------------------------------------------------- C ABI, direct
def test_c_abi_direct_call(ddsp):
    import ctypes
    from ddsp_pytorch_b200._lib import core_library
    lib = core_library()
    x = torch.linspace(-4, 4, 1000).cuda()
    y = torch.empty_like(x)
    fn = lib.ddsp_b200_scale_function_fwd
    fn.restype = ctypes.c_int
    fn.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]
    st = torch.cuda.current_stream().cuda_stream
    assert fn(x.data_ptr(), y.data_ptr(), x.numel(), st) == 0
    torch.cuda.synchronize()
    ref = 2 * torch.sigmoid(x.double().cpu()) ** math.log(10) + 1e-7
    assert max_abs(y, ref) < 1e-6
    assert fn(None, y.data_ptr(), 3, st) == -1, "argument errors are negative status codes"


def test_no_cpu_fallback(ddsp):
    with pytest.raises((RuntimeError, NotImplementedError)):
        ddsp.scale_function(torch.zeros(4))


# ------------------------------------------------------------------------------- fused hot path
def test_fused_controls_and_noise_match_unfused(ddsp):
    from ddsp_pytorch_b200 import functions as F_
    g = load_golden("synth_c1_small")
    sr, bs = int(g["sr"]), int(g["bs"])
    f0 = dev(g["f0"])
    a1, d1 = dev(g["amp_raw"], True), dev(g["dist_raw"], True)
    a2, d2 = dev(g["amp_raw"], True), dev(g["dist_raw"], True)
    amps, dist = F_.HarmonicControls.apply(a1, d1, f0, float(sr))
    w_ref = dist * amps
    _, _, w = F_.HarmonicControlsWeights.apply(a2, d2, f0, float(sr))
    assert max_abs(w, w_ref.detach().cpu()) < 1e-7
    go = torch.randn_like(w)
    (w_ref * go).sum().backward()
    (w * go).sum().backward()
    assert_grad(a2.grad, a1.grad.cpu(), 1e-5)
    assert_grad(d2.grad, d1.grad.cpu(), 1e-5)
    # noise: scale_function(raw - 5) + FIR + add, against the separate ops
    m1, m2 = dev(g["mag_raw"], True), dev(g["mag_raw"], True)
    noise = dev(g["noise"])
    harm = dev(g["harm"], True)
    harm2 = dev(g["harm"], True)
    y_ref = ddsp.filtered_noise(ddsp.scale_function(m1 + (-5.0)), noise) + harm
    y = F_.FilteredNoiseFused.apply(m2, noise, harm2, -5.0)
    assert max_abs(y, y_ref.detach().cpu()) < 1e-6
    go = torch.randn_like(y)
    (y_ref * go).sum().backward()
    (y * go).sum().backward()
    assert_grad(m2.grad, m1.grad.cpu(), 1e-5)
    assert torch.equal(harm2.grad, harm.grad)


@pytest.mark.parametrize("B,T,bs,H", [(3, 37, 160, 100), (2, 5, 512, 64), (1, 2, 128, 7), (2, 19, 160, 256)])
def test_controls_fused_into_the_oscillator_bank(ddsp, B, T, bs, H):
    """decoder.py:106-110 + modules.py:44-80 in one launch per direction (SURVEY 8f rank 3): the projection output
    goes straight into the bank.  Same arithmetic as the two-launch path, so audio, controls and gradients are equal
    bit for bit -- for the projection form (param (B,T,H+1) read and differentiated in place) and the split form."""
    from ddsp_pytorch_b200 import functions as F_
    assert ddsp.core.harmonic_raw_supported(H, bs)
    gen = torch.Generator().manual_seed(B * 1000 + T)
    sr = 16000.0
    param0 = torch.randn(B, T, H + 1, generator=gen).cuda()
    f0 = (80 + 700 * torch.rand(B, T, 1, generator=gen)).cuda()
    go = torch.randn(B, T * bs, 1, generator=gen).cuda()
    # reference: the two-launch path on slices of the projection
    p1 = param0.clone().requires_grad_(True)
    amps1, _, w1 = F_.HarmonicControlsWeights.apply(p1[..., :1], p1[..., 1:], f0, sr)
    y1, pe1 = ddsp.core.harmonic_synth_frames(f0, w1, bs, sr)
    (y1 * go).sum().backward()
    # projection form
    p2 = param0.clone().requires_grad_(True)
    y2, pe2, amps2, w2 = ddsp.core.harmonic_synth_from_raw(p2, None, f0, bs, sr)
    (y2 * go).sum().backward()
    assert torch.equal(y2, y1) and torch.equal(pe2, pe1) and torch.equal(amps2, amps1) and torch.equal(w2, w1)
    assert torch.equal(p2.grad, p1.grad)
    # split form (the hot path's leaves)
    a3 = param0[..., :1].clone().requires_grad_(True)
    d3 = param0[..., 1:].clone().requires_grad_(True)
    y3, _, amps3, w3 = ddsp.core.harmonic_synth_from_raw(a3, d3, f0, bs, sr)
    (y3 * go).sum().backward()
    assert torch.equal(y3, y1) and torch.equal(amps3, amps1) and torch.equal(w3, w1)
    assert torch.equal(a3.grad, p1.grad[..., :1]) and torch.equal(d3.grad, p1.grad[..., 1:])
    # gradients through the returned controls too (not the training loop's case): the two-launch backward
    p4 = param0.clone().requires_grad_(True)
    y4, _, amps4, w4 = ddsp.core.harmonic_synth_from_raw(p4, None, f0, bs, sr)
    ga, gw = torch.randn_like(amps4), torch.randn_like(w4)
    ((y4 * go).sum() + (amps4 * ga).sum() + (w4 * gw).sum()).backward()
    p5 = param0.clone().requires_grad_(True)
    amps5, _, w5 = F_.HarmonicControlsWeights.apply(p5[..., :1], p5[..., 1:], f0, sr)
    y5, _ = ddsp.core.harmonic_synth_frames(f0, w5, bs, sr)
    ((y5 * go).sum() + (amps5 * ga).sum() + (w5 * gw).sum()).backward()
    assert_grad(p4.grad, p5.grad, 1e-5)
    # streaming phase carry
    ph = torch.rand(B, generator=gen).double().cuda()
    ya, pea, _, _ = ddsp.core.harmonic_synth_from_raw(param0, None, f0, bs, sr, ph)
    yb, peb = ddsp.core.harmonic_synth_frames(f0, w1.detach(), bs, sr, ph)
    assert torch.equal(ya, yb) and torch.equal(pea, peb)


def test_model_uses_the_fused_controls_and_matches_the_two_launch_path(ddsp):
    """DDSPDecoder._synthesize goes through HarmonicSynth.synthesize; the returned harmonic_ctrls dict holds what the
    reference's holds after forward (distribution already scaled by the amplitudes, modules.py:73)."""
    from ddsp_pytorch_b200.models.modules import HarmonicSynth
    hs = HarmonicSynth(160, 16000)
    gen = torch.Generator().manual_seed(5)
    param = torch.randn(2, 30, 101, generator=gen).cuda().requires_grad_(True)
    f0 = (100 + 400 * torch.rand(2, 30, 1, generator=gen)).cuda()
    audio, ctrls = hs.synthesize(param, f0)
    ref_ctrls = hs.get_controls(param[..., :1], param[..., 1:], f0)
    ref_audio = hs(**ref_ctrls)
    assert torch.equal(audio, ref_audio)
    assert torch.equal(ctrls["amplitudes"], ref_ctrls["amplitudes"])
    assert torch.equal(ctrls["harmonic_distribution"], ref_ctrls["harmonic_distribution"])     # mutated in place by forward
    assert ctrls["f0"] is f0


def test_hotpath_step_against_oracle(ddsp, orc):
    """SynthStep (the benchmarked callable): audio, loss and every gradient against the float64 oracle,
    eager and CUDA-graph replay."""
    from ddsp_pytorch_b200.hotpath import SynthShapes, SynthStep, synthetic_inputs
    shapes = SynthShapes(batch=3, frames=30, block_size=160, n_harmonic=100, n_bands=65, sample_rate=16000,
                         reverb_length=2000, scales=(1024, 512, 256, 128), overlap=0.75)
    torch.manual_seed(0)
    step = SynthStep(shapes, "cuda")
    with torch.no_grad():
        step.reverb.wet.fill_(0.7)
        step.reverb.decay.fill_(3.0)
    host = synthetic_inputs(shapes, seed=5)
    step.load_inputs(host)
    step.run()
    rp = {k: v.detach().double().cpu() for k, v in step.reverb.state_dict().items()}
    d = {k: v.double() for k, v in host.items()}
    loss64, grads64 = orc.synth_train_step(d["amp_raw"], d["dist_raw"], d["mag_raw"], d["pitch"], d["noise"],
                                           d["target"], shapes.block_size, shapes.sample_rate, rp,
                                           list(shapes.scales), shapes.overlap)
    out64 = orc.synth_chain(d["amp_raw"], d["dist_raw"], d["mag_raw"], d["pitch"], d["noise"], shapes.block_size,
                            shapes.sample_rate, rp)
    assert_audio(step.signal, out64["signal"])
    assert abs(float(step.loss) - float(loss64)) <= 1e-5 * abs(float(loss64))
    # End-to-end gradients cross the L1 sign ties of the loss (a float32 magnitude that differs from the
    # target's by less than its rounding error flips a +-1), which the chain then spreads over every
    # control: SURVEY 0.5 measured ~100 % for the reference's own float32 path.  This is a wiring check;
    # the per-op gradient tests above carry the 1e-3 bar.
    for got, ref in zip(step.grads, grads64):
        assert rel_err(got.reshape(ref.shape), ref) < 0.1
    eager = [g_.clone() for g_ in step.grads]
    eager_loss = step.loss.clone()
    step.capture()
    step.replay()
    torch.cuda.synchronize()
    assert torch.equal(step.loss, eager_loss)
    for a, b in zip(step.grads, eager):
        assert torch.equal(a, b), "graph replay must reproduce the eager step bit for bit"
    # host-fed, prefetched execution gives the same numbers
    pinned = {k: v.pin_memory() for k, v in host.items()}
    step.prefetch(pinned)
    step.step_prefetched()
    torch.cuda.synchronize()
    assert torch.equal(step.loss, eager_loss)
    # double-buffered host feeding (two input sets, one graph each, no device-side copies): both sets reproduce it
    step.capture_pair()
    for _ in range(3):
        step.feed(pinned)
        k = step.step_fed()
        step.loss_to_host(k)
        assert step.read_loss(k) == float(eager_loss)
        for a, b in zip(step.grads, eager):
            assert torch.equal(a, b)


def test_data_parallel_step_matches_the_plain_step():
    """SURVEY 8e: with the gradient all-reduce enabled the backward is cut in two (reverb first, then the collective on
    a communication stream, a node of the captured graph, beside the synthesisers' backward).  On a one-rank NCCL
    group the average is the identity, so eager and replayed gradients must equal the plain step's bit for bit."""
    import torch.distributed as dist
    from ddsp_pytorch_b200.hotpath import SynthShapes, SynthStep, synthetic_inputs
    shapes = SynthShapes(batch=2, frames=30, block_size=160, n_harmonic=100, n_bands=65, sample_rate=16000,
                         reverb_length=2000, scales=(1024, 512, 256, 128), overlap=0.75)
    torch.manual_seed(0)
    step = SynthStep(shapes, "cuda")
    step.load_inputs(synthetic_inputs(shapes, seed=9))
    step.run()
    plain = [g_.clone() for g_ in step.grads]
    plain_loss = step.loss.clone()
    created = not dist.is_initialized()
    if created:
        dist.init_process_group("nccl", init_method="tcp://127.0.0.1:29741", rank=0, world_size=1,
                                device_id=torch.device("cuda", torch.cuda.current_device()))
    try:
        step.enable_grad_allreduce(dist)
        step.run()
        torch.cuda.synchronize()
        assert torch.equal(step.loss, plain_loss)
        for a, b in zip(step.grads, plain):
            assert torch.equal(a.reshape(b.shape), b)
        step.capture()
        for _ in range(2):
            step.replay()
        torch.cuda.synchronize()
        for a, b in zip(step.grads, plain):
            assert torch.equal(a.reshape(b.shape), b)
        with step.local_only():                      # no collective: what a single rank may call on its own
            step.run()
        torch.cuda.synchronize()
        for a, b in zip(step.grads, plain):
            assert torch.equal(a.reshape(b.shape), b)
    finally:
        step.release_graphs()
        if created:
            dist.destroy_process_group()


# ------------------------------------------------------------------------------- edge cases
@pytest.mark.parametrize("B,T,bs,H,NB", [(1, 1, 128, 1, 65), (2, 3, 128, 7, 65), (1, 5, 256, 33, 33),
                                           (3, 2, 64, 13, 9), (1, 2, 160, 101, 65)])
def test_ragged_shapes_forward_backward(ddsp, orc, B, T, bs, H, NB):
    """Single frame / single harmonic, harmonic counts that are not multiples of 4, block == filter size,
    other band counts: module chain against the float64 oracle, forward and gradients."""
    from ddsp_pytorch_b200.models.modules import FilteredNoise, HarmonicSynth
    sr = 16000
    gen = torch.Generator().manual_seed(B * 1000 + T * 100 + H)
    amp = torch.randn(B, T, 1, generator=gen)
    dist = torch.randn(B, T, H, generator=gen)
    mag = torch.randn(B, T, NB, generator=gen)
    f0 = torch.rand(B, T, 1, generator=gen) * 500 + 60
    noise = torch.rand(B, T, bs, generator=gen) * 2 - 1
    go = torch.randn(B, T * bs, 1, generator=gen)
    # oracle
    a64, d64, m64 = (t.double().requires_grad_(True) for t in (amp, dist, mag))
    out = orc.synth_chain(a64, d64, m64, f0.double(), noise.double(), bs, sr, None)
    (out["signal"] * go.double()).sum().backward()
    # kernels
    a, d, m = (t.cuda().requires_grad_(True) for t in (amp, dist, mag))
    hs, fn = HarmonicSynth(bs, sr), FilteredNoise(bs, NB)
    c = hs.get_controls(a, d, f0.cuda())
    sig = hs(**c) + fn(fn.get_controls(m)["magnitudes"], noise=noise.cuda())
    assert_audio(sig, out["signal"])
    (sig * go.cuda()).sum().backward()
    assert_grad(a.grad, a64.grad)
    assert_grad(d.grad, d64.grad)
    assert_grad(m.grad, m64.grad)


def test_non_contiguous_and_strided_inputs(ddsp, orc):
    """decoder.py:107-108 hands the synth strided slices of one projection (param[..., :1], param[..., 1:])."""
    gen = torch.Generator().manual_seed(21)
    B, T, H, bs, sr = 2, 6, 12, 160, 16000
    param = torch.randn(B, T, H + 1, generator=gen)
    f0 = torch.rand(B, T, 1, generator=gen) * 300 + 100
    from ddsp_pytorch_b200.models.modules import HarmonicSynth
    hs = HarmonicSynth(bs, sr)
    p = param.cuda().requires_grad_(True)
    c = hs.get_controls(p[..., :1], p[..., 1:], f0.cuda())
    y = hs(**c)
    p64 = param.double().requires_grad_(True)
    c64 = orc.harmonic_controls(p64[..., :1], p64[..., 1:], f0.double(), sr)
    y64 = orc.harmonic_synth_frames(c64["amplitudes"], c64["harmonic_distribution"], f0.double(), bs, sr)
    assert_audio(y, y64)
    go = torch.randn(y64.shape, generator=gen)
    (y * go.cuda()).sum().backward()
    (y64 * go.double()).sum().backward()
    assert_grad(p.grad, p64.grad)


def test_unsupported_shapes_fail_loudly(ddsp):
    """Shapes outside what the kernels implement raise (no silent fallback)."""
    with pytest.raises(RuntimeError):           # block smaller than the 128-tap noise filter
        ddsp.filtered_noise(torch.rand(1, 2, 65).cuda(), torch.rand(1, 2, 64).cuda())
    with pytest.raises(RuntimeError):           # reflect padding needs n_fft/2 < N, as torch.stft
        ddsp.multiscale_fft(torch.rand(1, 100).cuda(), [512], 0.75)
    with pytest.raises(RuntimeError):           # float64 is the oracle's job
        ddsp.scale_function(torch.zeros(4, dtype=torch.float64).cuda())
    with pytest.raises(RuntimeError):           # one frame's duplicated weights exceed shared memory
        ddsp.harmonic_synth_frames(torch.full((1, 1, 1), 100.0).cuda(), torch.rand(1, 1, 30000).cuda(), 160, 16000)


def test_large_amplitude_and_extreme_pitch(ddsp, orc):
    """f0 near 0, near and above Nyquist, and loud controls: masks, folding and the recurrence hold."""
    B, T, bs, H, sr = 1, 8, 160, 64, 16000
    f0 = torch.tensor([0.5, 20.0, 7999.0, 8001.0, 15999.0, 3999.9, 125.0, 4000.0]).view(1, T, 1)
    gen = torch.Generator().manual_seed(33)
    w = torch.rand(B, T, H, generator=gen)
    ref = orc.harmonic_synth(orc.upsample(f0.double(), bs), orc.upsample(w.double(), bs), sr)
    got, _ = ddsp.harmonic_synth_frames(f0.cuda(), w.cuda(), bs, sr)
    # sum of weights is ~32 here (not normalised): scale the 1e-4 bar accordingly
    assert_audio(got, ref, 1e-4 * float(w.sum(-1).max()) / 2)


def test_empty_batch(ddsp):
    """Zero voices / zero frames flow through the synth ops like any other shape (nothing is launched)."""
    from ddsp_pytorch_b200.models.modules import FilteredNoise, HarmonicSynth
    hs, fn = HarmonicSynth(160, 16000), FilteredNoise(160, 65)
    for B, T in ((0, 4), (2, 0)):
        a = torch.zeros(B, T, 1, device="cuda", requires_grad=True)
        d = torch.zeros(B, T, 8, device="cuda", requires_grad=True)
        m = torch.zeros(B, T, 65, device="cuda", requires_grad=True)
        c = hs.get_controls(a, d, torch.zeros(B, T, 1, device="cuda"))
        y = hs(**c) + fn(fn.get_controls(m)["magnitudes"])
        assert y.shape == (B, T * 160, 1)
        y.sum().backward()
        assert d.grad.shape == d.shape and m.grad.shape == m.shape
