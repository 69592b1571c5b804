// TORCH_LIBRARY shim over the C ABI of libddsp_b200.so (include/ddsp_b200.h).
//
// This file is plumbing only: it checks tensors (CUDA, float32, contiguous), allocates outputs
// and workspaces with torch's caching allocator, takes the current CUDA stream and calls the
// extern "C" entry points.  A non-zero status becomes a c10::Error (Python RuntimeError).  The
// ops are registered for the CUDA dispatch key only: there is no CPU implementation and a CPU
// tensor fails loudly in the dispatcher.  The schemas are visible to eager Python, to
// torch.jit.script and to libtorch C++ (the realtime ddsp~ host dlopen()s this library before
// torch::jit::load, INTEGRATION.md).
#include <ATen/ATen.h>
#include <ATen/cuda/CUDAContext.h>
#include <ATen/cuda/CUDAEvent.h>
#include <c10/cuda/CUDAGuard.h>
#include <c10/cuda/CUDAStream.h>
#include <torch/library.h>

#include <map>
#include <mutex>
#include <tuple>
#include <vector>

#include "ddsp_b200.h"

namespace {

using at::Tensor;

void check(int status, const char *what) {
    TORCH_CHECK(status == DDSP_B200_OK, "ddsp_b200::", what, " failed: ", ddsp_b200_strerror(status),
                " (status ", status, ")");
}

Tensor prep(const Tensor &t, const char *name) {
    TORCH_CHECK(t.is_cuda(), "ddsp_b200: ", name, " must be a CUDA tensor (no CPU fallback exists)");
    TORCH_CHECK(t.scalar_type() == at::kFloat, "ddsp_b200: ", name, " must be float32, got ",
                t.scalar_type());
    return t.contiguous();
}

void *cur_stream() { return (void *)at::cuda::getCurrentCUDAStream().stream(); }
const float *fp(const Tensor &t) { return t.data_ptr<float>(); }
float *fpm(Tensor &t) { return t.data_ptr<float>(); }

// A constant table is built once per (device, size) by whichever thread and stream asks first, and is then
// handed to every other thread and stream from the cache.  So the build must not be part of a CUDA graph capture
// (the tensor would live in the graph's private pool) and must be complete before the cache publishes it.
void finish_table_build(const char *what) {
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    cudaStream_t st = at::cuda::getCurrentCUDAStream().stream();
    TORCH_CHECK(cudaStreamIsCapturing(st, &cap) == cudaSuccess && cap == cudaStreamCaptureStatusNone,
                "ddsp_b200: constant table '", what, "' would be built inside a CUDA graph capture; run the op "
                "once eagerly (warm-up) before capturing");
    TORCH_CHECK(cudaStreamSynchronize(st) == cudaSuccess, "ddsp_b200: building table '", what, "' failed");
}

// Caller-owned constant tables, created lazily per (device, size); safe from any thread.
Tensor twiddle_table(const at::Device &dev, int64_t n) {
    static std::mutex mu;
    static std::map<std::pair<int, int64_t>, Tensor> cache;
    std::lock_guard<std::mutex> lock(mu);
    auto key = std::make_pair((int)dev.index(), n);
    auto it = cache.find(key);
    if (it != cache.end()) return it->second;
    Tensor t = at::empty({n, 2}, at::TensorOptions().device(dev).dtype(at::kFloat));
    check(ddsp_b200_twiddle_table(fpm(t), (int)n, cur_stream()), "twiddle_table");
    finish_table_build("twiddle_table");
    cache[key] = t;
    return t;
}

Tensor stage_twiddle_table(const at::Device &dev, int64_t n_fft) {
    static std::mutex mu;
    static std::map<std::pair<int, int64_t>, Tensor> cache;
    std::lock_guard<std::mutex> lock(mu);
    auto key = std::make_pair((int)dev.index(), n_fft);
    auto it = cache.find(key);
    if (it != cache.end()) return it->second;
    const int64_t n = ddsp_b200_fft_stage_twiddles_size((int)n_fft);
    Tensor t;
    if (n > 0) {
        t = at::empty({n, 2}, at::TensorOptions().device(dev).dtype(at::kFloat));
        check(ddsp_b200_fft_stage_twiddles(fpm(t), (int)n_fft, cur_stream()), "stft_stage_twiddles");
        finish_table_build("fft_stage_twiddles");
    }
    cache[key] = t;
    return t;
}

Tensor noise_design_table(const at::Device &dev, int64_t NB) {
    static std::mutex mu;
    static std::map<std::pair<int, int64_t>, Tensor> cache;
    std::lock_guard<std::mutex> lock(mu);
    auto key = std::make_pair((int)dev.index(), NB);
    auto it = cache.find(key);
    if (it != cache.end()) return it->second;
    Tensor t = at::empty({ddsp_b200_noise_design_size((int)NB)}, at::TensorOptions().device(dev).dtype(at::kFloat));
    check(ddsp_b200_noise_design_table(fpm(t), (int)NB, cur_stream()), "noise_design_table");
    finish_table_build("noise_design_table");
    cache[key] = t;
    return t;
}

// ---------------------------------------------------------------------------------------- a1-a3
Tensor scale_function_fwd(const Tensor &x_) {
    Tensor x = prep(x_, "x");
    c10::cuda::CUDAGuard guard(x.device());
    Tensor y = at::empty_like(x);
    check(ddsp_b200_scale_function_fwd(fp(x), fpm(y), x.numel(), cur_stream()), "scale_function_fwd");
    return y;
}

Tensor scale_function_bwd(const Tensor &x_, const Tensor &dy_) {
    Tensor x = prep(x_, "x"), dy = prep(dy_, "dy");
    TORCH_CHECK(x.numel() == dy.numel(), "scale_function_bwd: size mismatch");
    c10::cuda::CUDAGuard guard(x.device());
    Tensor dx = at::empty_like(x);
    check(ddsp_b200_scale_function_bwd(fp(x), fp(dy), fpm(dx), x.numel(), cur_stream()),
          "scale_function_bwd");
    return dx;
}

Tensor remove_above_nyquist(const Tensor &amp_, const Tensor &f0_, double sample_rate) {
    Tensor amp = prep(amp_, "amplitudes"), f0 = prep(f0_, "f0");
    TORCH_CHECK(amp.dim() >= 1 && f0.numel() * amp.size(-1) == amp.numel(),
                "remove_above_nyquist: f0 must have one value per row of amplitudes");
    c10::cuda::CUDAGuard guard(amp.device());
    Tensor out = at::empty_like(amp);
    check(ddsp_b200_remove_above_nyquist(fp(amp), fp(f0), fpm(out), f0.numel(), (int)amp.size(-1),
                                         (float)sample_rate, cur_stream()),
          "remove_above_nyquist");
    return out;
}

Tensor opt_prep(const c10::optional<Tensor> &t, const char *name) {
    return (t.has_value() && t->defined()) ? prep(*t, name) : Tensor();
}
const float *opt_fp(const Tensor &t) { return t.defined() ? t.data_ptr<float>() : nullptr; }

// (amps, dist, weights = dist*amps)
std::tuple<Tensor, Tensor, Tensor> harmonic_controls_fwd(const Tensor &amp_raw_, const Tensor &dist_raw_,
                                                         const Tensor &f0_, double sample_rate,
                                                         bool with_weights) {
    Tensor a = prep(amp_raw_, "amplitudes"), d = prep(dist_raw_, "harmonic_distribution"),
           f = prep(f0_, "f0");
    const int64_t H = d.size(-1), rows = d.numel() / H;
    TORCH_CHECK(a.numel() == rows && f.numel() == rows, "harmonic_controls: shape mismatch");
    c10::cuda::CUDAGuard guard(d.device());
    Tensor amps = at::empty_like(a), dist = at::empty_like(d);
    Tensor weights = with_weights ? at::empty_like(d) : at::empty({0}, d.options());
    check(ddsp_b200_harmonic_controls_fwd(fp(a), fp(d), fp(f), fpm(amps), fpm(dist),
                                          with_weights ? fpm(weights) : nullptr, rows, (int)H,
                                          (float)sample_rate, cur_stream()),
          "harmonic_controls_fwd");
    return {amps, dist, weights};
}

std::tuple<Tensor, Tensor> harmonic_controls_bwd(const Tensor &amp_raw_, const Tensor &dist_raw_,
                                                 const Tensor &f0_, const c10::optional<Tensor> &d_amps_,
                                                 const c10::optional<Tensor> &d_dist_,
                                                 const c10::optional<Tensor> &d_weights_,
                                                 double sample_rate) {
    Tensor a = prep(amp_raw_, "amplitudes"), d = prep(dist_raw_, "harmonic_distribution"),
           f = prep(f0_, "f0");
    Tensor ga = opt_prep(d_amps_, "d_amps"), gd = opt_prep(d_dist_, "d_dist"),
           gw = opt_prep(d_weights_, "d_weights");
    const int64_t H = d.size(-1), rows = d.numel() / H;
    TORCH_CHECK(a.numel() == rows && f.numel() == rows && (!ga.defined() || ga.numel() == rows) &&
                    (!gd.defined() || gd.numel() == d.numel()) && (!gw.defined() || gw.numel() == d.numel()),
                "harmonic_controls_bwd: shape mismatch");
    c10::cuda::CUDAGuard guard(d.device());
    Tensor da = at::empty_like(a), dd = at::empty_like(d);
    check(ddsp_b200_harmonic_controls_bwd(fp(a), fp(d), fp(f), opt_fp(ga), opt_fp(gd), opt_fp(gw), fpm(da),
                                          fpm(dd), rows, (int)H, (float)sample_rate, cur_stream()),
          "harmonic_controls_bwd");
    return {da, dd};
}

// ---------------------------------------------------------------------------------------- a4-a6
// f0 (B,T,1), weights (B,T,H) -> audio (B,T*bs,1), phase_end (B) float64 turns,
// phi/delta (B,T) int64 views of the Q0.64 phase workspace (kept for the backward).
std::tuple<Tensor, Tensor, Tensor, Tensor> harmonic_fwd(const Tensor &f0_, const Tensor &weights_,
                                                        int64_t block_size, double sample_rate,
                                                        const c10::optional<Tensor> &phase0_) {
    Tensor f0 = prep(f0_, "f0"), w = prep(weights_, "weights");
    TORCH_CHECK(w.dim() == 3, "harmonic_fwd: weights must be (B,T,H)");
    const int64_t B = w.size(0), T = w.size(1), H = w.size(2);
    TORCH_CHECK(f0.numel() == B * T, "harmonic_fwd: f0 must be (B,T,1)");
    c10::cuda::CUDAGuard guard(w.device());
    auto opt64 = w.options().dtype(at::kLong);
    Tensor phi = at::empty({B, T}, opt64), delta = at::empty({B, T}, opt64);
    Tensor phase_end = at::empty({B}, w.options().dtype(at::kDouble));
    Tensor audio = at::empty({B, T * block_size, 1}, w.options());
    if (B == 0 || T == 0) return {audio, phase_end.zero_(), phi, delta};      // empty batch: nothing to launch
    const double *p0 = nullptr;
    Tensor phase0;
    if (phase0_.has_value() && phase0_->defined()) {
        phase0 = phase0_->contiguous();
        TORCH_CHECK(phase0.is_cuda() && phase0.scalar_type() == at::kDouble && phase0.numel() == B,
                    "harmonic_fwd: phase0 must be a CUDA float64 tensor of B turns");
        p0 = phase0.data_ptr<double>();
    }
    check(ddsp_b200_phase_scan(fp(f0), p0, (uint64_t *)phi.data_ptr<int64_t>(),
                               (uint64_t *)delta.data_ptr<int64_t>(), phase_end.data_ptr<double>(),
                               (int)B, (int)T, (int)block_size, sample_rate, cur_stream()),
          "phase_scan");
    check(ddsp_b200_harmonic_frames_fwd(fp(w), (const uint64_t *)phi.data_ptr<int64_t>(),
                                        (const uint64_t *)delta.data_ptr<int64_t>(), fpm(audio), (int)B,
                                        (int)T, (int)H, (int)block_size, cur_stream()),
          "harmonic_frames_fwd");
    return {audio, phase_end, phi, delta};
}

std::tuple<Tensor, Tensor> harmonic_bwd(const Tensor &g_, const Tensor &weights_, const Tensor &phi,
                                        const Tensor &delta, int64_t block_size, double sample_rate,
                                        bool need_f0) {
    Tensor g = prep(g_, "grad_audio"), w = prep(weights_, "weights");
    const int64_t B = w.size(0), T = w.size(1), H = w.size(2);
    TORCH_CHECK(g.numel() == B * T * block_size, "harmonic_bwd: grad shape mismatch");
    TORCH_CHECK(phi.is_cuda() && phi.scalar_type() == at::kLong && phi.is_contiguous() &&
                    delta.is_cuda() && delta.scalar_type() == at::kLong && delta.is_contiguous() &&
                    phi.numel() == B * T && delta.numel() == B * T,
                "harmonic_bwd: bad phase workspace");
    c10::cuda::CUDAGuard guard(w.device());
    Tensor dw = at::empty_like(w);
    if (B == 0 || T == 0) return {dw, at::empty({B, T, 1}, w.options())};
    const uint64_t *ph = (const uint64_t *)phi.data_ptr<int64_t>();
    const uint64_t *dl = (const uint64_t *)delta.data_ptr<int64_t>();
    check(ddsp_b200_harmonic_frames_bwd_weights(fp(g), ph, dl, fpm(dw), (int)B, (int)T, (int)H,
                                                (int)block_size, cur_stream()),
          "harmonic_frames_bwd_weights");
    Tensor df0;
    if (need_f0) {
        df0 = at::empty({B, T, 1}, w.options());
        Tensor scratch = at::empty({B, T, 2}, w.options());
        check(ddsp_b200_harmonic_frames_bwd_f0(fp(g), fp(w), ph, dl, fpm(scratch), fpm(df0), (int)B, (int)T,
                                               (int)H, (int)block_size, sample_rate, cur_stream()),
              "harmonic_frames_bwd_f0");
    } else {
        df0 = at::empty({0}, w.options());
    }
    return {dw, df0};
}

// ---------------------------------------------------------------------------------------- a3 + a6 in one launch
// decoder.py:106-110 -> modules.py:44-80: the projection's raw outputs go straight into the oscillator bank.
// `first` is either the projection output param (B,T,H+1) with dist_raw absent (amplitude = column 0, distribution =
// columns 1..H, read in place), or amp_raw (B,T,1) with dist_raw (B,T,H).
int64_t harmonic_raw_supported(int64_t H, int64_t block_size) {
    return ddsp_b200_harmonic_frames_raw_supported((int)H, (int)block_size);
}

struct RawViews {
    Tensor first, dist;
    const float *amp, *dst;
    int64_t amp_stride, dist_stride, B, T, H;
    bool joint;
};

RawViews raw_views(const Tensor &first_, const c10::optional<Tensor> &dist_raw_) {
    RawViews v;
    v.first = prep(first_, "amplitudes / projection");
    v.joint = !(dist_raw_.has_value() && dist_raw_->defined());
    TORCH_CHECK(v.first.dim() == 3, "harmonic_raw: expected (B,T,.) tensors");
    v.B = v.first.size(0);
    v.T = v.first.size(1);
    if (v.joint) {
        v.H = v.first.size(2) - 1;
        TORCH_CHECK(v.H >= 1, "harmonic_raw: the projection must be (B,T,H+1)");
        v.amp = fp(v.first);
        v.dst = v.amp + 1;
        v.amp_stride = v.dist_stride = v.H + 1;
    } else {
        v.dist = prep(*dist_raw_, "harmonic_distribution");
        TORCH_CHECK(v.dist.dim() == 3 && v.dist.size(0) == v.B && v.dist.size(1) == v.T && v.first.size(2) == 1,
                    "harmonic_raw: amplitudes (B,T,1) and harmonic_distribution (B,T,H) expected");
        v.H = v.dist.size(2);
        v.amp = fp(v.first);
        v.dst = fp(v.dist);
        v.amp_stride = 1;
        v.dist_stride = v.H;
    }
    return v;
}

std::tuple<Tensor, Tensor, Tensor, Tensor, Tensor, Tensor> harmonic_raw_fwd(
    const Tensor &first_, const c10::optional<Tensor> &dist_raw_, const Tensor &f0_, int64_t block_size,
    double sample_rate, const c10::optional<Tensor> &phase0_) {
    RawViews v = raw_views(first_, dist_raw_);
    Tensor f0 = prep(f0_, "f0");
    const int64_t B = v.B, T = v.T, H = v.H;
    TORCH_CHECK(f0.numel() == B * T, "harmonic_raw_fwd: f0 must be (B,T,1)");
    c10::cuda::CUDAGuard guard(f0.device());
    auto opt = f0.options();
    Tensor phi = at::empty({B, T}, opt.dtype(at::kLong)), delta = at::empty({B, T}, opt.dtype(at::kLong));
    Tensor phase_end = at::empty({B}, opt.dtype(at::kDouble));
    Tensor audio = at::empty({B, T * block_size, 1}, opt);
    Tensor amps = at::empty({B, T, 1}, opt), weights = at::empty({B, T, H}, opt);
    if (B == 0 || T == 0) return {audio, phase_end.zero_(), phi, delta, amps, weights};
    const double *p0 = nullptr;
    Tensor phase0;
    if (phase0_.has_value() && phase0_->defined()) {
        phase0 = phase0_->contiguous();
        TORCH_CHECK(phase0.is_cuda() && phase0.scalar_type() == at::kDouble && phase0.numel() == B,
                    "harmonic_raw_fwd: phase0 must be a CUDA float64 tensor of B turns");
        p0 = phase0.data_ptr<double>();
    }
    // phase scan, controls and oscillator bank in one launch
    check(ddsp_b200_harmonic_frames_raw_scan_fwd(v.amp, v.amp_stride, v.dst, v.dist_stride, fp(f0), p0,
                                                 (uint64_t *)phi.data_ptr<int64_t>(),
                                                 (uint64_t *)delta.data_ptr<int64_t>(), phase_end.data_ptr<double>(),
                                                 fpm(amps), fpm(weights), fpm(audio), (int)B, (int)T, (int)H,
                                                 (int)block_size, sample_rate, cur_stream()),
          "harmonic_frames_raw_scan_fwd");
    return {audio, phase_end, phi, delta, amps, weights};
}

// joint (projection) form: (d_param (B,T,H+1), empty); split form: (d_amp_raw (B,T,1), d_dist_raw (B,T,H))
std::tuple<Tensor, Tensor> harmonic_raw_bwd(const Tensor &g_, const Tensor &first_,
                                            const c10::optional<Tensor> &dist_raw_, const Tensor &f0_,
                                            const Tensor &phi, const Tensor &delta, int64_t block_size,
                                            double sample_rate) {
    RawViews v = raw_views(first_, dist_raw_);
    Tensor g = prep(g_, "grad_audio"), f0 = prep(f0_, "f0");
    const int64_t B = v.B, T = v.T, H = v.H;
    TORCH_CHECK(g.numel() == B * T * block_size && f0.numel() == B * T, "harmonic_raw_bwd: shape mismatch");
    TORCH_CHECK(phi.is_cuda() && phi.scalar_type() == at::kLong && phi.is_contiguous() &&
                    delta.is_cuda() && delta.scalar_type() == at::kLong && delta.is_contiguous() &&
                    phi.numel() == B * T && delta.numel() == B * T,
                "harmonic_raw_bwd: bad phase workspace");
    c10::cuda::CUDAGuard guard(g.device());
    Tensor d0, d1;
    float *da, *dd;
    int64_t das, dds;
    if (v.joint) {
        d0 = at::empty({B, T, H + 1}, g.options());
        d1 = at::empty({0}, g.options());
        da = fpm(d0);
        dd = da + 1;
        das = dds = H + 1;
    } else {
        d0 = at::empty({B, T, 1}, g.options());
        d1 = at::empty({B, T, H}, g.options());
        da = fpm(d0);
        dd = fpm(d1);
        das = 1;
        dds = H;
    }
    if (B == 0 || T == 0) return {d0, d1};
    check(ddsp_b200_harmonic_frames_raw_bwd(fp(g), v.amp, v.amp_stride, v.dst, v.dist_stride, fp(f0),
                                            (const uint64_t *)phi.data_ptr<int64_t>(),
                                            (const uint64_t *)delta.data_ptr<int64_t>(), da, das, dd, dds, (int)B,
                                            (int)T, (int)H, (int)block_size, (float)sample_rate, cur_stream()),
          "harmonic_frames_raw_bwd");
    return {d0, d1};
}

// ---------------------------------------------------------------------------------------- a5 generic
std::tuple<Tensor, Tensor> harmonic_ar_fwd(const Tensor &f0_, const Tensor &amps_, double sample_rate) {
    Tensor f0 = prep(f0_, "f0"), a = prep(amps_, "amplitudes");
    TORCH_CHECK(a.dim() == 3, "harmonic_synth: amplitudes must be (B,N,H)");
    const int64_t B = a.size(0), N = a.size(1), H = a.size(2);
    TORCH_CHECK(f0.numel() == B * N, "harmonic_synth: f0 must be (B,N,1)");
    c10::cuda::CUDAGuard guard(a.device());
    Tensor phase = at::empty({B, N}, a.options().dtype(at::kLong));
    Tensor audio = at::empty({B, N, 1}, a.options());
    check(ddsp_b200_phase_scan_audio_rate(fp(f0), (uint64_t *)phase.data_ptr<int64_t>(), (int)B, N,
                                          sample_rate, cur_stream()),
          "phase_scan_audio_rate");
    check(ddsp_b200_harmonic_audio_rate_fwd(fp(a), (const uint64_t *)phase.data_ptr<int64_t>(), fpm(audio),
                                            (int)B, N, (int)H, cur_stream()),
          "harmonic_audio_rate_fwd");
    return {audio, phase};
}

std::tuple<Tensor, Tensor> harmonic_ar_bwd(const Tensor &g_, const Tensor &amps_, const Tensor &phase,
                                           double sample_rate, bool need_f0) {
    Tensor g = prep(g_, "grad_audio"), a = prep(amps_, "amplitudes");
    const int64_t B = a.size(0), N = a.size(1), H = a.size(2);
    TORCH_CHECK(g.numel() == B * N && phase.numel() == B * N && phase.scalar_type() == at::kLong &&
                    phase.is_cuda() && phase.is_contiguous(),
                "harmonic_synth backward: shape mismatch");
    c10::cuda::CUDAGuard guard(a.device());
    Tensor da = at::empty_like(a);
    Tensor df0 = need_f0 ? at::empty({B, N, 1}, a.options()) : at::empty({0}, a.options());
    Tensor dphi = need_f0 ? at::empty({B, N}, a.options()) : Tensor();
    check(ddsp_b200_harmonic_audio_rate_bwd(fp(g), fp(a), (const uint64_t *)phase.data_ptr<int64_t>(),
                                            fpm(da), need_f0 ? fpm(dphi) : nullptr,
                                            need_f0 ? fpm(df0) : nullptr, (int)B, N, (int)H, sample_rate,
                                            cur_stream()),
          "harmonic_audio_rate_bwd");
    return {da, df0};
}

// ---------------------------------------------------------------------------------------- a7, a8
Tensor amp_to_ir_fwd(const Tensor &amp_, int64_t target) {
    Tensor amp = prep(amp_, "amp");
    const int64_t NB = amp.size(-1), rows = amp.numel() / NB;
    c10::cuda::CUDAGuard guard(amp.device());
    auto shape = amp.sizes().vec();
    shape.back() = target;
    Tensor ir = at::empty(shape, amp.options());
    check(ddsp_b200_amp_to_ir_fwd(fp(amp), fpm(ir), rows, (int)NB, (int)target, cur_stream()),
          "amp_to_ir_fwd");
    return ir;
}

Tensor amp_to_ir_bwd(const Tensor &d_ir_, int64_t NB) {
    Tensor d_ir = prep(d_ir_, "d_ir");
    const int64_t target = d_ir.size(-1), rows = d_ir.numel() / target;
    c10::cuda::CUDAGuard guard(d_ir.device());
    auto shape = d_ir.sizes().vec();
    shape.back() = NB;
    Tensor d_amp = at::empty(shape, d_ir.options());
    check(ddsp_b200_amp_to_ir_bwd(fp(d_ir), fpm(d_amp), rows, (int)NB, (int)target, cur_stream()),
          "amp_to_ir_bwd");
    return d_amp;
}

Tensor noise_fwd(const Tensor &mags_, const Tensor &noise_, const c10::optional<Tensor> &add_, bool apply_scale,
                 double bias) {
    Tensor mags = prep(mags_, "magnitudes"), noise = prep(noise_, "noise"), add = opt_prep(add_, "add");
    TORCH_CHECK(mags.dim() == 3 && noise.dim() == 3 && mags.size(0) == noise.size(0) &&
                    mags.size(1) == noise.size(1),
                "filtered noise: magnitudes (B,T,NB) and noise (B,T,block) expected");
    const int64_t B = mags.size(0), T = mags.size(1), NB = mags.size(2), bs = noise.size(2);
    TORCH_CHECK(!add.defined() || add.numel() == B * T * bs, "filtered noise: `add` must be (B,T*block,1)");
    c10::cuda::CUDAGuard guard(mags.device());
    Tensor out = at::empty({B, T * bs, 1}, mags.options());
    if (B * T == 0) return out;
    Tensor design = noise_design_table(mags.device(), NB);
    check(ddsp_b200_filtered_noise_fwd(fp(mags), fp(noise), opt_fp(add), fp(design), fpm(out), B * T, (int)NB,
                                       (int)bs, apply_scale, (float)bias, cur_stream()),
          "filtered_noise_fwd");
    return out;
}

Tensor noise_bwd(const Tensor &g_, const Tensor &noise_, const c10::optional<Tensor> &mags_raw_, int64_t NB,
                 bool apply_scale, double bias) {
    Tensor g = prep(g_, "grad_out"), noise = prep(noise_, "noise"), raw = opt_prep(mags_raw_, "mags_raw");
    const int64_t B = noise.size(0), T = noise.size(1), bs = noise.size(2);
    TORCH_CHECK(g.numel() == B * T * bs, "filtered noise backward: shape mismatch");
    TORCH_CHECK(!apply_scale || (raw.defined() && raw.numel() == B * T * NB),
                "filtered noise backward: raw magnitudes needed when the scale function is fused");
    c10::cuda::CUDAGuard guard(noise.device());
    Tensor d_mags = at::empty({B, T, NB}, noise.options());
    if (B * T == 0) return d_mags;
    Tensor design = noise_design_table(noise.device(), NB);
    check(ddsp_b200_filtered_noise_bwd(fp(g), fp(noise), opt_fp(raw), fp(design), fpm(d_mags), B * T, (int)NB,
                                       (int)bs, apply_scale, (float)bias, cur_stream()),
          "filtered_noise_bwd");
    return d_mags;
}

// ---------------------------------------------------------------------------------------- a9, a10
struct ConvPlan {
    int n1, n2;
    int64_t n;
    Tensor tw, st1, st2;       // W_n table and the stage tables of the two sub-transforms
};

ConvPlan conv_plan(const at::Device &dev, int64_t min_len) {
    ConvPlan p;
    check(ddsp_b200_conv_plan(min_len, &p.n1, &p.n2), "conv_plan");
    p.n = (int64_t)p.n1 * p.n2;
    p.tw = twiddle_table(dev, p.n);
    p.st1 = stage_twiddle_table(dev, p.n1);
    p.st2 = stage_twiddle_table(dev, p.n2);
    return p;
}

// signal (R,n), kernel (Rk,Lk) with Rk in {1,R}: out[r,i] = sum_{j<=i} signal[r,j] kernel[rk,i-j]
// keep != 0 also returns the column-transformed signal and the kernel spectrum for the backward pass
// spectrum of the convolution kernel in the layout the row passes multiply with (four-step [k1][k2]); depends on the
// signal length only through the transform size.  Separate op so that a caller can compute it early / on another stream
// (hotpath.py: the reverb's spectrum only depends on the reverb parameters, not on the audio).
Tensor fftconv_spectrum(const Tensor &kernel_, int64_t n_signal) {
    Tensor ker = prep(kernel_, "kernel");
    TORCH_CHECK(ker.dim() == 2 && n_signal > 0, "fftconv_spectrum: 2-D (rows, length) kernel expected");
    const int64_t Rk = ker.size(0), Lk = ker.size(1);
    c10::cuda::CUDAGuard guard(ker.device());
    const int64_t Lc = std::min(Lk, n_signal);          // taps beyond the signal length never matter
    Tensor kc = Lc == Lk ? ker : ker.narrow(1, 0, Lc).contiguous();
    ConvPlan p = conv_plan(ker.device(), n_signal + Lc - 1);
    void *st = cur_stream();
    Tensor hspec = at::empty({Rk, p.n, 2}, ker.options());
    check(ddsp_b200_fft4_cols_fwd(fp(kc), Rk, Lc, 0, fpm(hspec), fp(p.tw), opt_fp(p.st1), p.n1, p.n2, st), "fft4_cols_fwd(h)");
    check(ddsp_b200_fft4_rows_spectrum(fpm(hspec), Rk, fp(p.tw), fp(p.st2), p.n1, p.n2, st), "fft4_rows_spectrum");
    return hspec;
}

std::tuple<Tensor, Tensor, Tensor> fftconv_fwd(const Tensor &signal_, const Tensor &kernel_, bool keep,
                                               const c10::optional<Tensor> &hspec_,
                                               const c10::optional<Tensor> &signal2_) {
    Tensor sig = prep(signal_, "signal"), ker = prep(kernel_, "kernel");
    Tensor sig2 = opt_prep(signal2_, "signal2");                  // convolve signal + signal2
    TORCH_CHECK(!sig2.defined() || sig2.sizes() == sig.sizes(), "fftconv: signal2 must have the signal's shape");
    TORCH_CHECK(sig.dim() == 2 && ker.dim() == 2, "fftconv: 2-D (rows, length) tensors expected");
    const int64_t R = sig.size(0), n = sig.size(1), Rk = ker.size(0), Lk = ker.size(1);
    TORCH_CHECK(Rk == 1 || Rk == R, "fftconv: kernel rows must be 1 or match the signal rows");
    c10::cuda::CUDAGuard guard(sig.device());
    Tensor out = at::empty_like(sig);
    Tensor none = at::empty({0}, sig.options());
    if (R == 0 || n == 0) return {out, none, none};
    const int64_t Lc = std::min(Lk, n);                 // taps beyond the signal length never matter
    ConvPlan p = conv_plan(sig.device(), n + Lc - 1);
    const int pair = Rk == 1;
    const int64_t slots = pair ? (R + 1) / 2 : R;
    void *st = cur_stream();
    Tensor hspec;
    if (hspec_.has_value() && hspec_->defined()) {
        hspec = prep(*hspec_, "hspec");
        TORCH_CHECK(hspec.numel() == Rk * p.n * 2, "fftconv: hspec does not belong to this kernel / signal length");
    } else {
        hspec = fftconv_spectrum(ker, n);
    }
    Tensor work = at::empty({slots, p.n, 2}, sig.options());
    check(ddsp_b200_fft4_cols_fwd_sum(fp(sig), opt_fp(sig2), R, n, pair, fpm(work), fp(p.tw), opt_fp(p.st1), p.n1, p.n2, st),
          "fft4_cols_fwd(x)");
    Tensor filtered = keep ? at::empty_like(work) : work;
    check(ddsp_b200_fft4_rows_filter(fp(work), fpm(filtered), slots, fp(hspec), pair ? 0 : p.n, 0, fp(p.tw), fp(p.st2),
                                     p.n1, p.n2, st),
          "fft4_rows_filter");
    check(ddsp_b200_fft4_cols_inv(fp(filtered), fpm(out), R, n, pair, opt_fp(p.st1), p.n1, p.n2, st), "fft4_cols_inv");
    if (keep) return {out, work, hspec};
    return {out, none, none};
}

// The two gradients can be taken in two calls (the data-parallel step wants the kernel gradient first, so that its
// all-reduce is in flight while the signal gradient and everything upstream of it is computed): `work_g_` = the
// transform of grad_out returned by an earlier call; the signal-gradient chain filters it in place, so it is valid for
// further calls only as long as need_signal was false.
std::tuple<Tensor, Tensor, Tensor> fftconv_bwd_parts(const Tensor &g_, const Tensor &signal_, const Tensor &kernel_,
                                                     const c10::optional<Tensor> &work_x_,
                                                     const c10::optional<Tensor> &hspec_,
                                                     const c10::optional<Tensor> &work_g_, bool need_signal,
                                                     bool need_kernel) {
    Tensor g = prep(g_, "grad_out"), sig = prep(signal_, "signal"), ker = prep(kernel_, "kernel");
    const int64_t R = sig.size(0), n = sig.size(1), Rk = ker.size(0), Lk = ker.size(1);
    TORCH_CHECK(g.dim() == 2 && g.size(0) == R && g.size(1) == n, "fftconv backward: grad shape mismatch");
    c10::cuda::CUDAGuard guard(sig.device());
    Tensor d_sig = need_signal ? at::empty_like(sig) : at::empty({0}, sig.options());
    Tensor d_ker = need_kernel ? at::zeros_like(ker) : at::empty({0}, sig.options());
    if (R == 0 || n == 0 || (!need_signal && !need_kernel)) return {d_sig, d_ker, at::empty({0}, sig.options())};
    const int64_t Lc = std::min(Lk, n);
    Tensor kc = Lc == Lk ? ker : ker.narrow(1, 0, Lc).contiguous();
    ConvPlan p = conv_plan(sig.device(), n + Lc - 1);
    const int pair = Rk == 1;
    const int64_t slots = pair ? (R + 1) / 2 : R;
    auto main_stream = at::cuda::getCurrentCUDAStream();
    void *st = (void *)main_stream.stream();
    // d_kernel and d_signal are independent after the transform of g: the kernel-gradient chain runs on a
    // pool stream (it only reads work_g), the signal-gradient chain (which filters work_g in place) waits
    // for the correlation to have consumed work_g.
    const bool fork = need_kernel && need_signal;
    at::cuda::CUDAStream side = fork ? at::cuda::getStreamFromPool(false, sig.device().index()) : main_stream;
    void *ss = (void *)side.stream();
    // the correlation's scratch (partial spectra + row counters) is allocated up front and its counters are zeroed on the
    // side stream while the transform of g runs on the main stream: no zeroing launch on the backward's critical path
    Tensor scratch;
    int counters_zeroed = 0;
    if (need_kernel) {
        scratch = at::empty({ddsp_b200_fft4_correlate_splits_plan(slots, pair, p.n1, p.n2), p.n, 2}, sig.options());
        const int64_t coff = ddsp_b200_fft4_correlate_counter_offset(slots, pair, p.n1, p.n2);
        if (fork && coff >= 0) {
            at::cuda::CUDAEvent begun;
            begun.record(main_stream);
            begun.block(side);
            c10::cuda::CUDAStreamGuard sg(side);
            scratch.view({-1}).narrow(0, coff, p.n1).zero_();
            counters_zeroed = 1;
        }
    }
    Tensor work_g;
    if (work_g_.has_value() && work_g_->defined() && work_g_->numel() == slots * p.n * 2) {
        work_g = *work_g_;
        TORCH_CHECK(work_g.is_cuda() && work_g.scalar_type() == at::kFloat && work_g.is_contiguous(),
                    "fftconv backward: bad work_g");
    } else {
        work_g = at::empty({slots, p.n, 2}, sig.options());
        check(ddsp_b200_fft4_cols_fwd(fp(g), R, n, pair, fpm(work_g), fp(p.tw), opt_fp(p.st1), p.n1, p.n2, st), "fft4_cols_fwd(g)");
    }
    // transforms kept by the forward pass (FFTConvolve saves them) are reused instead of recomputed
    Tensor hspec = (hspec_.has_value() && hspec_->defined() && hspec_->numel() == Rk * p.n * 2) ? *hspec_ : Tensor();
    Tensor saved_x = (work_x_.has_value() && work_x_->defined() && work_x_->numel() == slots * p.n * 2) ? *work_x_ : Tensor();
    if (need_signal && !hspec.defined()) {
        hspec = at::empty({Rk, p.n, 2}, sig.options());
        check(ddsp_b200_fft4_cols_fwd(fp(kc), Rk, Lc, 0, fpm(hspec), fp(p.tw), opt_fp(p.st1), p.n1, p.n2, st), "fft4_cols_fwd(h)");
        check(ddsp_b200_fft4_rows_spectrum(fpm(hspec), Rk, fp(p.tw), fp(p.st2), p.n1, p.n2, st), "fft4_rows_spectrum");
    }
    at::cuda::CUDAEvent corr_done;
    if (need_kernel) {
        if (fork) {
            at::cuda::CUDAEvent g_ready;
            g_ready.record(main_stream);
            g_ready.block(side);
        }
        Tensor work_x = saved_x;
        if (!work_x.defined()) {
            work_x = at::empty({slots, p.n, 2}, sig.options());
            check(ddsp_b200_fft4_cols_fwd(fp(sig), R, n, pair, fpm(work_x), fp(p.tw), opt_fp(p.st1), p.n1, p.n2, ss),
                  "fft4_cols_fwd(x)");
        }
        Tensor corr = at::empty({Rk, p.n, 2}, sig.options());
        check(ddsp_b200_fft4_rows_correlate_ex(fp(work_g), fp(work_x), slots, pair, fpm(scratch), fpm(corr),
                                               fp(p.tw), fp(p.st2), p.n1, p.n2, counters_zeroed, ss),
              "fft4_rows_correlate");
        if (fork) corr_done.record(side);
        Tensor dk = Lc == Lk ? d_ker : at::empty({Rk, Lc}, sig.options());
        check(ddsp_b200_fft4_cols_inv(fp(corr), fpm(dk), Rk, Lc, 0, opt_fp(p.st1), p.n1, p.n2, ss), "fft4_cols_inv(dh)");
        if (Lc != Lk) {
            c10::cuda::CUDAStreamGuard sg(side);
            d_ker.narrow(1, 0, Lc).copy_(dk);
        }
        // (temporaries are released after the join below, i.e. ordered after their last use)
    }
    if (need_signal) {
        if (fork) corr_done.block(main_stream);          // work_g is filtered in place below
        check(ddsp_b200_fft4_rows_filter(fp(work_g), fpm(work_g), slots, fp(hspec), pair ? 0 : p.n, 1, fp(p.tw), fp(p.st2),
                                         p.n1, p.n2, st),
              "fft4_rows_filter(conj)");
        check(ddsp_b200_fft4_cols_inv(fp(work_g), fpm(d_sig), R, n, pair, opt_fp(p.st1), p.n1, p.n2, st),
              "fft4_cols_inv(dx)");
    }
    if (fork) {
        at::cuda::CUDAEvent join;
        join.record(side);
        join.block(main_stream);
    }
    return {d_sig, d_ker, work_g};
}

std::tuple<Tensor, Tensor> fftconv_bwd(const Tensor &g, const Tensor &signal, const Tensor &kernel,
                                       const c10::optional<Tensor> &work_x, const c10::optional<Tensor> &hspec,
                                       bool need_signal, bool need_kernel) {
    auto r = fftconv_bwd_parts(g, signal, kernel, work_x, hspec, c10::nullopt, need_signal, need_kernel);
    return {std::get<0>(r), std::get<1>(r)};
}

Tensor reverb_impulse_fwd(const Tensor &noise_, const Tensor &decay_, const Tensor &wet_, const Tensor &t_) {
    Tensor noise = prep(noise_, "noise"), decay = prep(decay_, "decay"), wet = prep(wet_, "wet"),
           t = prep(t_, "t");
    const int64_t L = noise.numel();
    TORCH_CHECK(t.numel() == L && decay.numel() == 1 && wet.numel() == 1, "reverb impulse: shape mismatch");
    c10::cuda::CUDAGuard guard(noise.device());
    Tensor imp = at::empty({1, L, 1}, noise.options());
    check(ddsp_b200_reverb_impulse_fwd(fp(noise), fp(decay), fp(wet), fp(t), fpm(imp), (int)L, cur_stream()),
          "reverb_impulse_fwd");
    return imp;
}

std::tuple<Tensor, Tensor, Tensor> reverb_impulse_bwd(const Tensor &d_imp_, const Tensor &noise_,
                                                      const Tensor &decay_, const Tensor &wet_,
                                                      const Tensor &t_) {
    Tensor d_imp = prep(d_imp_, "d_impulse"), noise = prep(noise_, "noise"), decay = prep(decay_, "decay"),
           wet = prep(wet_, "wet"), t = prep(t_, "t");
    const int64_t L = noise.numel();
    TORCH_CHECK(d_imp.numel() <= L, "reverb impulse backward: d_impulse longer than the impulse");
    c10::cuda::CUDAGuard guard(noise.device());
    Tensor dn = at::empty_like(noise), dd = at::empty_like(decay), dw = at::empty_like(wet);
    Tensor scratch = at::empty({ddsp_b200_reverb_impulse_bwd_scratch() / 8}, noise.options().dtype(at::kDouble));
    check(ddsp_b200_reverb_impulse_bwd(fp(d_imp), (int)d_imp.numel(), fp(noise), fp(decay), fp(wet), fp(t),
                                       fpm(dn), fpm(dd), fpm(dw), (int)L, scratch.data_ptr(), cur_stream()),
          "reverb_impulse_bwd");
    return {dn, dd, dw};
}

// ---------------------------------------------------------------------------------------- a10s streaming reverb
// signal (B,N), kernel with L taps (any shape of L elements), history (B,L-1) -> (y (B,N), history_out (B,L-1))
std::tuple<Tensor, Tensor> conv_stream_fwd(const Tensor &signal_, const Tensor &kernel_, const Tensor &history_) {
    Tensor sig = prep(signal_, "signal"), ker = prep(kernel_, "kernel"), hist = prep(history_, "history");
    TORCH_CHECK(sig.dim() == 2 && sig.size(0) >= 1 && sig.size(1) >= 1, "conv_stream: signal must be (B,N), B, N >= 1");
    const int64_t B = sig.size(0), N = sig.size(1), L = ker.numel();
    TORCH_CHECK(L >= 1 && L <= INT32_MAX && B <= INT32_MAX, "conv_stream: the kernel needs 1 .. 2^31-1 taps");
    TORCH_CHECK(hist.dim() == 2 && hist.size(0) == B && hist.size(1) == L - 1, "conv_stream: history must be (B, L-1) = (",
                B, ", ", L - 1, "), got ", hist.sizes());
    TORCH_CHECK(ker.device() == sig.device() && hist.device() == sig.device(), "conv_stream: tensors on different devices");
    c10::cuda::CUDAGuard guard(sig.device());
    Tensor y = at::empty_like(sig), hist_out = at::empty_like(hist);
    const int64_t ns = ddsp_b200_conv_stream_scratch((int)B, N, (int)L);       // sizes checked above: >= 0
    Tensor scratch = ns > 0 ? at::empty({ns}, sig.options()) : Tensor();
    check(ddsp_b200_conv_stream_fwd(fp(sig), fp(ker), L > 1 ? fp(hist) : nullptr, fpm(y),
                                    L > 1 ? fpm(hist_out) : nullptr, (int)B, N, (int)L,
                                    ns > 0 ? fpm(scratch) : nullptr, cur_stream()),
          "conv_stream_fwd");
    return {y, hist_out};
}

// ---------------------------------------------------------------------------------------- f1 dataset features
// signal (B,N) -> (loudness (B,F), mfcc (B,F,n_mfcc) or an empty tensor when mfcc is false), F = 1 + N/hop.
// a_weight (n_fft/2+1), mel_table (the compact band table of the C ABI), dct (128, n_mfcc): functions.feature_tables.
std::tuple<Tensor, Tensor> features_fwd(const Tensor &signal_, const Tensor &window_, const Tensor &a_weight_,
                                        const Tensor &mel_table_, const Tensor &dct_, int64_t n_fft, int64_t hop,
                                        bool mfcc) {
    Tensor sig = prep(signal_, "signal"), win = prep(window_, "window"), aw = prep(a_weight_, "a_weight");
    Tensor mel = prep(mel_table_, "mel_table"), dct = prep(dct_, "dct");
    TORCH_CHECK(sig.dim() == 2, "features: signal must be (B,N)");
    TORCH_CHECK(win.numel() == n_fft && aw.numel() == n_fft / 2 + 1, "features: window (n_fft) and a_weight (n_fft/2+1) expected");
    TORCH_CHECK(dct.dim() == 2 && dct.size(0) == 128, "features: dct must be (128, n_mfcc)");
    TORCH_CHECK(mel.numel() >= 384, "features: mel_table is shorter than its header");
    for (const Tensor *t : {&win, &aw, &mel, &dct})
        TORCH_CHECK(t->device() == sig.device(), "features: tensors on different devices");
    const int64_t B = sig.size(0), N = sig.size(1), n_mfcc = dct.size(1);
    TORCH_CHECK(B <= INT32_MAX && n_fft <= 4096 && hop >= 1 && hop <= INT32_MAX, "features: unsupported sizes");
    c10::cuda::CUDAGuard guard(sig.device());
    const int64_t ns = ddsp_b200_features_scratch((int)B, N, (int)n_fft, (int)hop, (int)n_mfcc);
    TORCH_CHECK(ns > 0, "features: unsupported sizes (B ", B, ", N ", N, ", n_fft ", n_fft, ", hop ", hop,
                ", n_mfcc ", n_mfcc, ")");
    const int64_t F = 1 + N / hop;
    Tensor loud = at::empty({B, F}, sig.options());
    Tensor out = at::empty({mfcc ? B : 0, F, n_mfcc}, sig.options());
    Tensor scratch = mfcc ? at::empty({ns}, sig.options()) : Tensor();
    Tensor stw = stage_twiddle_table(sig.device(), n_fft);
    check(ddsp_b200_features_fwd(fp(sig), fp(win), fp(stw), fp(aw), fp(mel), fp(dct), fpm(loud),
                                 mfcc ? fpm(out) : nullptr, mfcc ? fpm(scratch) : nullptr, (int)B, N, (int)n_fft,
                                 (int)hop, (int)n_mfcc, cur_stream()),
          "features_fwd");
    return {loud, out};
}

// ---------------------------------------------------------------------------------------- f1 dataset pitch (YIN)
// signal (B,N) -> (f0 (B,F), aperiodicity (B,F)), F = N/hop; the periods come from core.extract_pitch_yin.
std::tuple<Tensor, Tensor> pitch_yin_fwd(const Tensor &signal_, int64_t frame_length, int64_t hop, int64_t min_period,
                                         int64_t max_period, double sample_rate, double threshold) {
    Tensor sig = prep(signal_, "signal");
    TORCH_CHECK(sig.dim() == 2, "pitch_yin: signal must be (B,N)");
    const int64_t B = sig.size(0), N = sig.size(1);
    TORCH_CHECK(B >= 1 && B <= 65535 && frame_length >= 256 && frame_length <= 4096 &&
                    (frame_length & (frame_length - 1)) == 0 && hop >= 1 && hop <= INT32_MAX && min_period >= 1 &&
                    max_period <= frame_length / 2 - 1 && max_period >= min_period + 2,
                "pitch_yin: unsupported sizes (B ", B, ", frame_length ", frame_length, ", hop ", hop, ", periods ",
                min_period, "..", max_period, ")");
    c10::cuda::CUDAGuard guard(sig.device());
    const int64_t F = N / hop;
    Tensor f0 = at::empty({B, F}, sig.options()), ap = at::empty({B, F}, sig.options());
    Tensor stw = stage_twiddle_table(sig.device(), frame_length);
    check(ddsp_b200_pitch_yin_fwd(fp(sig), fp(stw), fpm(f0), fpm(ap), (int)B, N, (int)frame_length, (int)hop,
                                  (int)min_period, (int)max_period, (float)sample_rate, (float)threshold, cur_stream()),
          "pitch_yin_fwd");
    return {f0, ap};
}

// ---------------------------------------------------------------------------------------- a11, a12
int64_t pow2_ge(int64_t v) {
    int64_t p = 1;
    while (p < v) p <<= 1;
    return p;
}

Tensor stft_mag_fwd(const Tensor &signal_, const Tensor &window_, int64_t n_fft, int64_t hop) {
    Tensor sig = prep(signal_, "signal"), win = prep(window_, "window");
    TORCH_CHECK(sig.dim() == 2 && win.numel() == n_fft, "stft_mag: signal (B,N) and window (n_fft) expected");
    const int64_t B = sig.size(0), N = sig.size(1);
    c10::cuda::CUDAGuard guard(sig.device());
    Tensor tw = twiddle_table(sig.device(), std::max<int64_t>(4096, n_fft));
    Tensor mag = at::empty({B, n_fft / 2 + 1, 1 + N / hop}, sig.options());
    Tensor stw = stage_twiddle_table(sig.device(), n_fft);
    check(ddsp_b200_stft_mag_fwd(fp(sig), fp(win), fp(tw), (int)tw.size(0), stw.defined() ? fp(stw) : nullptr, fpm(mag),
                                 (int)B, N, (int)n_fft, (int)hop, cur_stream()),
          "stft_mag_fwd");
    return mag;
}

Tensor stft_mag_bwd(const Tensor &signal_, const Tensor &d_mag_, const Tensor &window_, int64_t n_fft,
                    int64_t hop) {
    Tensor sig = prep(signal_, "signal"), gm = prep(d_mag_, "d_mag"), win = prep(window_, "window");
    const int64_t B = sig.size(0), N = sig.size(1);
    TORCH_CHECK(gm.numel() == B * (n_fft / 2 + 1) * (1 + N / hop), "stft_mag backward: shape mismatch");
    c10::cuda::CUDAGuard guard(sig.device());
    Tensor tw = twiddle_table(sig.device(), std::max<int64_t>(4096, n_fft));
    Tensor d_sig = at::empty_like(sig);
    Tensor edge = at::empty({B, n_fft}, sig.options());
    void *st = cur_stream();
    Tensor stw = stage_twiddle_table(sig.device(), n_fft);
    check(ddsp_b200_stft_mag_bwd(fp(sig), fp(gm), fp(win), fp(tw), (int)tw.size(0), stw.defined() ? fp(stw) : nullptr,
                                 fpm(d_sig), fpm(edge), (int)B, N, (int)n_fft, (int)hop, 0, st),
          "stft_mag_bwd");
    const int sc = (int)n_fft;
    check(ddsp_b200_stft_fold_edges(fp(edge), fpm(d_sig), (int)B, N, &sc, 1, st), "stft_fold_edges");
    return d_sig;
}

// target, rec (B,N); windows = the float32 hann windows of every scale, concatenated.
// Returns (loss[], d_rec (B,N) for unit upstream gradient, or an empty tensor).
std::tuple<Tensor, Tensor> mss_loss_fwd(const Tensor &target_, const Tensor &rec_, at::IntArrayRef scales,
                                        double overlap, const Tensor &windows_, bool need_grad) {
    Tensor tgt = prep(target_, "target"), rec = prep(rec_, "rec"), win = prep(windows_, "windows");
    TORCH_CHECK(tgt.dim() == 2 && rec.sizes() == tgt.sizes(), "mss_loss: target and rec must both be (B,N)");
    const int64_t B = rec.size(0), N = rec.size(1);
    const int ns = (int)scales.size();
    TORCH_CHECK(ns >= 1 && ns <= 8, "mss_loss: 1..8 scales supported");
    std::vector<int> sc(ns), hp(ns);
    int64_t wsum = 0, tiles = 0, esum = 0, smax = 0;
    for (int i = 0; i < ns; ++i) {
        sc[i] = (int)scales[i];
        hp[i] = (int)((double)scales[i] * (1.0 - overlap));     // int(s * (1 - overlap)), core.py:33
        const int64_t t = ddsp_b200_mss_tiles((int)B, N, sc[i], hp[i]);
        TORCH_CHECK(t > 0, "mss_loss: scale ", sc[i], " with hop ", hp[i], " unsupported for N=", N);
        tiles += t * B;
        wsum += sc[i];
        esum += B * sc[i];
        smax = std::max<int64_t>(smax, sc[i]);
    }
    TORCH_CHECK(win.numel() == wsum, "mss_loss: windows must hold sum(scales) values");
    c10::cuda::CUDAGuard guard(rec.device());
    if (ddsp_b200_mss_fused_supported(sc.data(), hp.data(), ns)) {
        // the reference's setting (overlap 0.75): every scale in one launch
        int64_t ws_floats = 0, part_floats = 0;
        check(ddsp_b200_mss_fused_sizes((int)B, N, sc.data(), ns, &ws_floats, &part_floats), "mss_fused_sizes");
        std::vector<Tensor> tables;
        std::vector<const float *> tabs;
        for (int i = 0; i < ns; ++i) {
            tables.push_back(stage_twiddle_table(rec.device(), sc[i]));
            tabs.push_back(fp(tables.back()));
        }
        Tensor partial = at::empty({part_floats}, rec.options());
        Tensor loss = at::empty({}, rec.options());
        Tensor d_rec = need_grad ? at::empty_like(rec) : at::empty({0}, rec.options());
        Tensor ws = need_grad ? at::empty({ws_floats}, rec.options()) : Tensor();
        check(ddsp_b200_mss_fused(fp(tgt), fp(rec), fp(win), tabs.data(), need_grad ? fpm(ws) : nullptr, fpm(partial),
                                  need_grad ? fpm(d_rec) : nullptr, fpm(loss), (int)B, N, sc.data(), ns, cur_stream()),
              "mss_fused");
        return {loss, d_rec};
    }
    Tensor tw = twiddle_table(rec.device(), std::max<int64_t>(4096, pow2_ge(smax)));
    Tensor partial = at::empty({tiles, 2}, rec.options());
    Tensor loss = at::empty({}, rec.options());
    Tensor d_rec = need_grad ? at::empty_like(rec) : at::empty({0}, rec.options());
    Tensor edge = need_grad ? at::empty({esum}, rec.options()) : Tensor();
    // The scales are independent (own partials, own gradient buffer): fork them over pool streams so
    // these latency-bound launches overlap, join before the finish kernel.  Captured as graph branches.
    Tensor d_scales = need_grad ? at::empty({ns, B, N}, rec.options()) : Tensor();
    auto main_stream = at::cuda::getCurrentCUDAStream();
    // constant tables are built (first use only) on the main stream BEFORE the fork, so that the side
    // streams are ordered after their initialisation
    std::vector<Tensor> stage_tables;
    for (int i = 0; i < ns; ++i) stage_tables.push_back(stage_twiddle_table(rec.device(), sc[i]));
    std::vector<at::cuda::CUDAStream> streams;
    streams.push_back(main_stream);
    for (int i = 1; i < ns; ++i) streams.push_back(at::cuda::getStreamFromPool(false, rec.device().index()));
    at::cuda::CUDAEvent fork;
    fork.record(main_stream);
    for (int i = 1; i < ns; ++i) fork.block(streams[i]);
    int64_t woff = 0, poff = 0, eoff = 0;
    for (int i = 0; i < ns; ++i) {
        const Tensor &stw = stage_tables[i];
        check(ddsp_b200_mss_scale(fp(tgt), fp(rec), fp(win) + woff, fp(tw), (int)tw.size(0),
                                  stw.defined() ? fp(stw) : nullptr, fpm(partial) + 2 * poff,
                                  need_grad ? fpm(d_scales) + (int64_t)i * B * N : nullptr,
                                  need_grad ? fpm(edge) + eoff : nullptr, (int)B, N, sc[i], hp[i], 0,
                                  (void *)streams[i].stream()),
              "mss_scale");
        woff += sc[i];
        poff += ddsp_b200_mss_tiles((int)B, N, sc[i], hp[i]) * B;
        eoff += B * sc[i];
    }
    for (int i = 1; i < ns; ++i) {
        at::cuda::CUDAEvent join;
        join.record(streams[i]);
        join.block(main_stream);
    }
    check(ddsp_b200_mss_finish(fp(partial), need_grad ? fp(edge) : nullptr, need_grad ? fp(d_scales) : nullptr,
                               need_grad ? fpm(d_rec) : nullptr, fpm(loss), (int)B, N, sc.data(), hp.data(), ns,
                               (void *)main_stream.stream()),
          "mss_finish");
    return {loss, d_rec};
}

// ---------------------------------------------------------------------------------------- f3 GRU
// voices one pass of the resident clusters covers (0: such clusters cannot run here, or hidden != 512);
// above it the cluster kernel needs a second pass over time and the library recurrence wins
int64_t gru_supported(int64_t hidden) {
    if (hidden != 512) return 0;
    const int clusters = ddsp_b200_gru_resident_clusters();
    return clusters > 0 ? (int64_t)clusters * 10 : 0;
}

// gi (B,T,3H) = x W_ih^T + b_ih; returns (y (B,T,H), gates (B,T,4H) or empty)
std::tuple<Tensor, Tensor> gru_fwd(const Tensor &gi_, const Tensor &w_hh_, const Tensor &b_hh_,
                                   const c10::optional<Tensor> &h0_, bool save_gates) {
    Tensor gi = prep(gi_, "gi"), w = prep(w_hh_, "weight_hh"), b = prep(b_hh_, "bias_hh"), h0 = opt_prep(h0_, "h0");
    TORCH_CHECK(gi.dim() == 3 && gi.size(2) % 3 == 0, "gru_fwd: gi must be (B,T,3H)");
    const int64_t B = gi.size(0), T = gi.size(1), H = gi.size(2) / 3;
    TORCH_CHECK(w.numel() == 3 * H * H && b.numel() == 3 * H && (!h0.defined() || h0.numel() == B * H),
                "gru_fwd: weight / bias / h0 shape mismatch");
    c10::cuda::CUDAGuard guard(gi.device());
    Tensor y = at::empty({B, T, H}, gi.options());
    Tensor gates = save_gates ? at::empty({B, T, 4 * H}, gi.options()) : at::empty({0}, gi.options());
    if (B == 0 || T == 0) return {y, gates};
    check(ddsp_b200_gru_fwd(fp(gi), fp(w), fp(b), opt_fp(h0), fpm(y), save_gates ? fpm(gates) : nullptr, (int)B,
                            (int)T, (int)H, cur_stream()),
          "gru_fwd");
    return {y, gates};
}

// returns (dgi, dgh, dh0)
std::tuple<Tensor, Tensor, Tensor> gru_bwd(const Tensor &dy_, const c10::optional<Tensor> &dhT_, const Tensor &w_hh_,
                                           const Tensor &y_, const c10::optional<Tensor> &h0_, const Tensor &gates_) {
    Tensor dy = prep(dy_, "dy"), w = prep(w_hh_, "weight_hh"), y = prep(y_, "y"), gates = prep(gates_, "gates");
    Tensor dhT = opt_prep(dhT_, "dhT"), h0 = opt_prep(h0_, "h0");
    const int64_t B = y.size(0), T = y.size(1), H = y.size(2);
    TORCH_CHECK(dy.numel() == y.numel() && gates.numel() == 4 * y.numel(), "gru_bwd: shape mismatch");
    c10::cuda::CUDAGuard guard(y.device());
    Tensor dgi = at::empty({B, T, 3 * H}, y.options()), dgh = at::empty({B, T, 3 * H}, y.options());
    Tensor dh0 = at::empty({B, H}, y.options());
    if (B == 0 || T == 0) return {dgi, dgh, dh0.zero_()};
    check(ddsp_b200_gru_bwd(fp(dy), opt_fp(dhT), fp(w), fp(y), opt_fp(h0), fp(gates), fpm(dgi), fpm(dgh), fpm(dh0),
                            (int)B, (int)T, (int)H, cur_stream()),
          "gru_bwd");
    return {dgi, dgh, dh0};
}

// ---------------------------------------------------------------------------------------- f3 GEMM
// x (rows, cols) contiguous -> split operand (3 * Rp, ld) bf16: part p in rows [p Rp, p Rp + R).
// transpose = false: R = rows, Rp = R rounded up to 64 with zero rows (usable K-major and MN-major);
// transpose = true: operand of x^T, R = cols, Rp = R (K-major use only).
Tensor gemm3x_split(const Tensor &x_, bool transpose) {
    Tensor x = prep(x_, "x");
    TORCH_CHECK(x.dim() == 2, "gemm3x_split: x must be 2-D");
    const int64_t rows = x.size(0), cols = x.size(1);
    const int64_t R = transpose ? cols : rows, K = transpose ? rows : cols;
    const int64_t Rp = transpose ? R : (R + 63) / 64 * 64;
    c10::cuda::CUDAGuard guard(x.device());
    Tensor out = at::empty({3 * Rp, ddsp_b200_gemm3x_ld(K)}, x.options().dtype(at::kBFloat16));
    if (rows == 0 || cols == 0) return out.zero_();
    check(ddsp_b200_gemm3x_split(fp(x), rows, cols, cols, transpose ? 1 : 0, out.data_ptr(), Rp, cur_stream()), "gemm3x_split");
    return out;
}

// non-transposed gemm3x_split that also returns the column sums of x: (operand, colsum (cols))
std::tuple<Tensor, Tensor> gemm3x_split_colsum(const Tensor &x_) {
    Tensor x = prep(x_, "x");
    TORCH_CHECK(x.dim() == 2, "gemm3x_split_colsum: x must be 2-D");
    const int64_t rows = x.size(0), cols = x.size(1), Rp = (rows + 63) / 64 * 64;
    c10::cuda::CUDAGuard guard(x.device());
    Tensor out = at::empty({3 * Rp, ddsp_b200_gemm3x_ld(cols)}, x.options().dtype(at::kBFloat16));
    Tensor colsum = at::empty({cols}, x.options());
    if (rows == 0 || cols == 0) return {out.zero_(), colsum.zero_()};
    Tensor partial = at::empty({ddsp_b200_gemm3x_colsum_scratch(Rp, cols)}, x.options());
    check(ddsp_b200_gemm3x_split_colsum(fp(x), rows, cols, cols, out.data_ptr(), Rp, fpm(colsum), fpm(partial), cur_stream()),
          "gemm3x_split_colsum");
    return {out, colsum};
}

// x (rows, cols) -> (split operand of x, split operand of x^T) from one pass over x
std::tuple<Tensor, Tensor> gemm3x_split_both(const Tensor &x_) {
    Tensor x = prep(x_, "x");
    TORCH_CHECK(x.dim() == 2, "gemm3x_split_both: x must be 2-D");
    const int64_t rows = x.size(0), cols = x.size(1);
    c10::cuda::CUDAGuard guard(x.device());
    Tensor out = at::empty({3 * rows, ddsp_b200_gemm3x_ld(cols)}, x.options().dtype(at::kBFloat16));
    Tensor out_t = at::empty({3 * cols, ddsp_b200_gemm3x_ld(rows)}, x.options().dtype(at::kBFloat16));
    if (rows == 0 || cols == 0) return {out.zero_(), out_t.zero_()};
    check(ddsp_b200_gemm3x_split_both(fp(x), rows, cols, cols, out.data_ptr(), rows, out_t.data_ptr(), cols, cur_stream()),
          "gemm3x_split_both");
    return {out, out_t};
}

// a, b split operands (gemm3x_split) -> A B^T + bias (M, N) float32 with A logically M x K, B logically N x K;
// x_mn = false: the operand tensor is (rows = M or N) x K; true: K x (M or N) as split from a non-transposed matrix
Tensor gemm3x_mm(const Tensor &a, const Tensor &b, int64_t M, int64_t N, int64_t K, const c10::optional<Tensor> &bias_,
                 bool a_mn, bool b_mn) {
    Tensor bias = opt_prep(bias_, "bias");
    TORCH_CHECK(a.is_cuda() && b.is_cuda() && a.scalar_type() == at::kBFloat16 && b.scalar_type() == at::kBFloat16 &&
                    a.is_contiguous() && b.is_contiguous() && a.dim() == 2 && b.dim() == 2 && a.size(0) % 3 == 0 &&
                    b.size(0) % 3 == 0,
                "gemm3x_mm: operands must be gemm3x_split outputs");
    const int64_t a_pr = a.size(0) / 3, b_pr = b.size(0) / 3;
    TORCH_CHECK(a_mn ? (a_pr >= K && a_pr % 64 == 0 && a.size(1) >= M) : (a_pr >= M && a.size(1) >= K),
                "gemm3x_mm: operand a does not hold an ", M, " x ", K, " matrix in the stated orientation");
    TORCH_CHECK(b_mn ? (b_pr >= K && b_pr % 64 == 0 && b.size(1) >= N) : (b_pr >= N && b.size(1) >= K),
                "gemm3x_mm: operand b does not hold an ", N, " x ", K, " matrix in the stated orientation");
    TORCH_CHECK(!bias.defined() || bias.numel() == N, "gemm3x_mm: bias must have N entries");
    c10::cuda::CUDAGuard guard(a.device());
    auto fopt = a.options().dtype(at::kFloat);
    Tensor c = at::empty({M, N}, fopt);
    if (M == 0 || N == 0) return c;
    if (K == 0) return bias.defined() ? c.copy_(bias.expand({M, N})) : c.zero_();
    const int splits = ddsp_b200_gemm3x_splits((int)M, (int)N, (int)K);
    Tensor ws = splits > 1 ? at::empty({splits, M, N}, fopt) : Tensor();
    check(ddsp_b200_gemm3x(a.data_ptr(), a_pr, a.size(1), a_mn ? 1 : 0, b.data_ptr(), b_pr, b.size(1), b_mn ? 1 : 0,
                           opt_fp(bias), fpm(c), N, (int)M, (int)N, (int)K, splits > 1 ? fpm(ws) : nullptr, cur_stream()),
          "gemm3x_mm");
    return c;
}

// ---------------------------------------------------------------------------------------- f3 LayerNorm
int64_t ln_lrelu_supported(int64_t n) { return n % 128 == 0 && n >= 128 && n <= 512; }

// x (..., N) -> (y, stats (rows, 2) or empty)
std::tuple<Tensor, Tensor> ln_lrelu_fwd(const Tensor &x_, const Tensor &gamma_, const Tensor &beta_, double eps,
                                        double slope, bool save_stats) {
    Tensor x = prep(x_, "x"), gamma = prep(gamma_, "weight"), beta = prep(beta_, "bias");
    const int64_t N = x.size(-1), rows = N ? x.numel() / N : 0;
    TORCH_CHECK(gamma.numel() == N && beta.numel() == N, "ln_lrelu_fwd: weight / bias must have N entries");
    c10::cuda::CUDAGuard guard(x.device());
    Tensor y = at::empty_like(x);
    Tensor stats = save_stats ? at::empty({rows, 2}, x.options()) : at::empty({0}, x.options());
    check(ddsp_b200_ln_lrelu_fwd(fp(x), fp(gamma), fp(beta), fpm(y), save_stats ? fpm(stats) : nullptr, rows, (int)N,
                                 (float)eps, (float)slope, cur_stream()),
          "ln_lrelu_fwd");
    return {y, stats};
}

// -> (dx, d_gamma, d_beta)
std::tuple<Tensor, Tensor, Tensor> ln_lrelu_bwd(const Tensor &dy_, const Tensor &x_, const Tensor &gamma_,
                                                const Tensor &beta_, const Tensor &stats_, double slope) {
    Tensor dy = prep(dy_, "dy"), x = prep(x_, "x"), gamma = prep(gamma_, "weight"), beta = prep(beta_, "bias");
    Tensor stats = prep(stats_, "stats");
    const int64_t N = x.size(-1), rows = N ? x.numel() / N : 0;
    TORCH_CHECK(dy.numel() == x.numel() && stats.numel() == 2 * rows, "ln_lrelu_bwd: shape mismatch");
    c10::cuda::CUDAGuard guard(x.device());
    Tensor dx = at::empty_like(x), dg = at::empty({N}, x.options()), db = at::empty({N}, x.options());
    if (rows == 0) return {dx, dg.zero_(), db.zero_()};
    Tensor partial = at::empty({ddsp_b200_ln_lrelu_slots(rows), 2 * N}, x.options());
    check(ddsp_b200_ln_lrelu_bwd(fp(dy), fp(x), fp(gamma), fp(beta), fp(stats), fpm(dx), fpm(dg), fpm(db), fpm(partial),
                                 rows, (int)N, (float)slope, cur_stream()),
          "ln_lrelu_bwd");
    return {dx, dg, db};
}

int64_t abi_version() { return ddsp_b200_abi_version(); }

}  // namespace

TORCH_LIBRARY(ddsp_b200, m) {
    m.def("abi_version() -> int", abi_version);
    m.def("gru_supported(int hidden) -> int", gru_supported);
    m.def("ln_lrelu_supported(int n) -> int", ln_lrelu_supported);
    m.def("ln_lrelu_fwd(Tensor x, Tensor weight, Tensor bias, float eps, float slope, bool save_stats) -> (Tensor, Tensor)");
    m.def("ln_lrelu_bwd(Tensor dy, Tensor x, Tensor weight, Tensor bias, Tensor stats, float slope) -> (Tensor, Tensor, Tensor)");
    m.def("gemm3x_split(Tensor x, bool transpose) -> Tensor");
    m.def("gemm3x_split_both(Tensor x) -> (Tensor, Tensor)");
    m.def("gemm3x_split_colsum(Tensor x) -> (Tensor, Tensor)");
    m.def("gemm3x_mm(Tensor a, Tensor b, int M, int N, int K, Tensor? bias, bool a_mn, bool b_mn) -> Tensor");
    m.def("gru_fwd(Tensor gi, Tensor weight_hh, Tensor bias_hh, Tensor? h0, bool save_gates) -> (Tensor, Tensor)");
    m.def("gru_bwd(Tensor dy, Tensor? dhT, Tensor weight_hh, Tensor y, Tensor? h0, Tensor gates) -> (Tensor, Tensor, Tensor)");
    m.def("scale_function_fwd(Tensor x) -> Tensor");
    m.def("scale_function_bwd(Tensor x, Tensor dy) -> Tensor");
    m.def("remove_above_nyquist(Tensor amplitudes, Tensor f0, float sample_rate) -> Tensor");
    m.def("harmonic_controls_fwd(Tensor amplitudes, Tensor harmonic_distribution, Tensor f0, float sample_rate, bool with_weights) -> (Tensor, Tensor, Tensor)");
    m.def("harmonic_controls_bwd(Tensor amplitudes, Tensor harmonic_distribution, Tensor f0, Tensor? d_amps, Tensor? d_dist, Tensor? d_weights, float sample_rate) -> (Tensor, Tensor)");
    m.def("harmonic_fwd(Tensor f0, Tensor weights, int block_size, float sample_rate, Tensor? phase0) -> (Tensor, Tensor, Tensor, Tensor)");
    m.def("harmonic_bwd(Tensor grad_audio, Tensor weights, Tensor phi, Tensor delta, int block_size, float sample_rate, bool need_f0) -> (Tensor, Tensor)");
    m.def("harmonic_raw_supported(int n_harmonic, int block_size) -> int", harmonic_raw_supported);
    m.def("harmonic_raw_fwd(Tensor first, Tensor? dist_raw, Tensor f0, int block_size, float sample_rate, Tensor? phase0) -> (Tensor, Tensor, Tensor, Tensor, Tensor, Tensor)");
    m.def("harmonic_raw_bwd(Tensor grad_audio, Tensor first, Tensor? dist_raw, Tensor f0, Tensor phi, Tensor delta, int block_size, float sample_rate) -> (Tensor, Tensor)");
    m.def("harmonic_ar_fwd(Tensor f0, Tensor amplitudes, float sample_rate) -> (Tensor, Tensor)");
    m.def("harmonic_ar_bwd(Tensor grad_audio, Tensor amplitudes, Tensor phase, float sample_rate, bool need_f0) -> (Tensor, Tensor)");
    m.def("amp_to_ir_fwd(Tensor amp, int target_size) -> Tensor");
    m.def("amp_to_ir_bwd(Tensor d_ir, int n_bands) -> Tensor");
    m.def("noise_fwd(Tensor magnitudes, Tensor noise, Tensor? add, bool apply_scale, float bias) -> Tensor");
    m.def("noise_bwd(Tensor grad_out, Tensor noise, Tensor? magnitudes_raw, int n_bands, bool apply_scale, float bias) -> Tensor");
    m.def("fftconv_spectrum(Tensor kernel, int n_signal) -> Tensor");
    m.def("fftconv_fwd(Tensor signal, Tensor kernel, bool keep_transforms, Tensor? hspec=None, Tensor? signal2=None) -> (Tensor, Tensor, Tensor)");
    m.def("fftconv_bwd(Tensor grad_out, Tensor signal, Tensor kernel, Tensor? work_x, Tensor? hspec, bool need_signal, bool need_kernel) -> (Tensor, Tensor)");
    m.def("fftconv_bwd_parts(Tensor grad_out, Tensor signal, Tensor kernel, Tensor? work_x, Tensor? hspec, Tensor? work_g, bool need_signal, bool need_kernel) -> (Tensor, Tensor, Tensor)");
    m.def("reverb_impulse_fwd(Tensor noise, Tensor decay, Tensor wet, Tensor t) -> Tensor");
    m.def("reverb_impulse_bwd(Tensor d_impulse, Tensor noise, Tensor decay, Tensor wet, Tensor t) -> (Tensor, Tensor, Tensor)");
    m.def("conv_stream_fwd(Tensor signal, Tensor kernel, Tensor history) -> (Tensor, Tensor)");
    m.def("features_fwd(Tensor signal, Tensor window, Tensor a_weight, Tensor mel_table, Tensor dct, int n_fft, int hop, bool mfcc) -> (Tensor, Tensor)");
    m.def("pitch_yin_fwd(Tensor signal, int frame_length, int hop, int min_period, int max_period, float sample_rate, float threshold) -> (Tensor, Tensor)");
    m.def("stft_mag_fwd(Tensor signal, Tensor window, int n_fft, int hop) -> Tensor");
    m.def("stft_mag_bwd(Tensor signal, Tensor d_mag, Tensor window, int n_fft, int hop) -> Tensor");
    m.def("mss_loss_fwd(Tensor target, Tensor rec, int[] scales, float overlap, Tensor windows, bool need_grad) -> (Tensor, Tensor)");
}

TORCH_LIBRARY_IMPL(ddsp_b200, CUDA, m) {
    m.impl("ln_lrelu_fwd", ln_lrelu_fwd);
    m.impl("ln_lrelu_bwd", ln_lrelu_bwd);
    m.impl("gemm3x_split", gemm3x_split);
    m.impl("gemm3x_split_both", gemm3x_split_both);
    m.impl("gemm3x_split_colsum", gemm3x_split_colsum);
    m.impl("gemm3x_mm", gemm3x_mm);
    m.impl("gru_fwd", gru_fwd);
    m.impl("gru_bwd", gru_bwd);
    m.impl("scale_function_fwd", scale_function_fwd);
    m.impl("scale_function_bwd", scale_function_bwd);
    m.impl("remove_above_nyquist", remove_above_nyquist);
    m.impl("harmonic_controls_fwd", harmonic_controls_fwd);
    m.impl("harmonic_controls_bwd", harmonic_controls_bwd);
    m.impl("harmonic_fwd", harmonic_fwd);
    m.impl("harmonic_bwd", harmonic_bwd);
    m.impl("harmonic_raw_fwd", harmonic_raw_fwd);
    m.impl("harmonic_raw_bwd", harmonic_raw_bwd);
    m.impl("harmonic_ar_fwd", harmonic_ar_fwd);
    m.impl("harmonic_ar_bwd", harmonic_ar_bwd);
    m.impl("amp_to_ir_fwd", amp_to_ir_fwd);
    m.impl("amp_to_ir_bwd", amp_to_ir_bwd);
    m.impl("noise_fwd", noise_fwd);
    m.impl("noise_bwd", noise_bwd);
    m.impl("fftconv_spectrum", fftconv_spectrum);
    m.impl("fftconv_fwd", fftconv_fwd);
    m.impl("fftconv_bwd", fftconv_bwd);
    m.impl("fftconv_bwd_parts", fftconv_bwd_parts);
    m.impl("reverb_impulse_fwd", reverb_impulse_fwd);
    m.impl("reverb_impulse_bwd", reverb_impulse_bwd);
    m.impl("conv_stream_fwd", conv_stream_fwd);
    m.impl("features_fwd", features_fwd);
    m.impl("pitch_yin_fwd", pitch_yin_fwd);
    m.impl("stft_mag_fwd", stft_mag_fwd);
    m.impl("stft_mag_bwd", stft_mag_bwd);
    m.impl("mss_loss_fwd", mss_loss_fwd);
}
