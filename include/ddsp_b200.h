/*
 * ddsp_b200.h -- C ABI of libddsp_b200.so: the DDSP synthesis hot path as hand-written
 * sm_100a CUDA kernels.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  The reference
 * (hugofloresgarcia/ddsp_pytorch) has no native code on this path: every entry point below
 * replaces a chain of eager ATen calls in the reference's Python, cited per function as
 * <file>:<lines> relative to the reference tree.  The TORCH_LIBRARY shim
 * (ddsp_pytorch_b200/csrc/torch_ops.cpp) is the only in-repo caller; INTEGRATION.md shows the
 * ctypes / libtorch bindings a maintainer of the reference would add.
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is a DEVICE pointer to contiguous float32
 *    (or the stated type) on the current CUDA device; nothing here allocates or frees device
 *    memory or keeps state -- workspaces and constant tables are caller-owned;
 *  - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *  - return value: 0 = launched; < 0 = argument error (DDSP_B200_E*); > 0 = cudaError_t of the
 *    failed launch.  Nothing throws or aborts across this boundary;
 *  - B = voices, T = frames, bs = block_size (samples per frame), N = T*bs, H = harmonics,
 *    NB = noise bands, L = reverb taps.
 */
#ifndef DDSP_B200_H
#define DDSP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DDSP_B200_OK 0
#define DDSP_B200_EINVAL (-1)      /* bad size / null pointer */
#define DDSP_B200_EUNSUPPORTED (-2) /* shape outside what the kernels implement */

int ddsp_b200_abi_version(void);
const char *ddsp_b200_strerror(int status);
/* kernels launched through this library since it was loaded (diagnostic counter) */
uint64_t ddsp_b200_launch_count(void);

/* ---- a1  scale_function: 2*sigmoid(x)^ln10 + 1e-7            (ddsp/core.py:77-78) ---------- */
int ddsp_b200_scale_function_fwd(const float *x, float *y, int64_t n, void *stream);
/* dx = dy * dy/dx, recomputed from x */
int ddsp_b200_scale_function_bwd(const float *x, const float *dy, float *dx, int64_t n, void *stream);

/* ---- a2  remove_above_nyquist                                 (ddsp/core.py:70-74) ---------- */
/* out[r,k] = amp[r,k] * ((f0[r]*(k+1) < sample_rate/2) + 1e-4f);  rows = B*T.  With `grad` != 0
 * the same call is the backward (amp := dy, out := dx): the mask does not depend on amp.       */
int ddsp_b200_remove_above_nyquist(const float *amp, const float *f0, float *out, int64_t rows,
                                   int H, float sample_rate, void *stream);

/* ---- a3  HarmonicSynth.get_controls, fused          (ddsp/models/modules.py:44-67) ---------- */
/* amp_raw[rows], dist_raw[rows,H], f0[rows]  ->  amps[rows] = scale(amp_raw),
 * dist[rows,H] = normalise(scale(dist_raw) * nyquist_mask) and, if weights != NULL,
 * weights[rows,H] = dist * amps (the in-place product of HarmonicSynth.forward, modules.py:73).
 * Backward: any of d_amps / d_dist / d_weights may be NULL (= zero upstream gradient).          */
int ddsp_b200_harmonic_controls_fwd(const float *amp_raw, const float *dist_raw, const float *f0,
                                    float *amps, float *dist, float *weights, int64_t rows, int H,
                                    float sample_rate, void *stream);
int ddsp_b200_harmonic_controls_bwd(const float *amp_raw, const float *dist_raw, const float *f0,
                                    const float *d_amps, const float *d_dist, const float *d_weights,
                                    float *d_amp_raw, float *d_dist_raw, int64_t rows, int H,
                                    float sample_rate, void *stream);

/* ---- a4+a5+a6  HarmonicSynth.forward, fused         (ddsp/models/modules.py:69-80,
 *                upsample ddsp/core.py:64-67, harmonic_synth ddsp/core.py:136-141) ------------ */
/* Phase workspace: phi[B*T], delta[B*T] uint64 = phase at the start of each frame and phase
 * increment per sample, in turns as Q0.64 fixed point.  phase0[B] (may be NULL = 0) and
 * phase_end[B] (may be NULL) are turns in [0,1) as double: the streaming carry (SURVEY 3.3). */
/* Host-side evaluation of the per-sample phase increment the scans use: frac(f0 / sample_rate) as Q0.64, the exact
 * product of the float32 pitch and the double 1/sample_rate, truncated (integer arithmetic, no device needed). */
uint64_t ddsp_b200_pitch_to_q64(float f0, double sample_rate);
int ddsp_b200_phase_scan(const float *f0, const double *phase0, uint64_t *phi, uint64_t *delta,
                         double *phase_end, int B, int T, int block_size, double sample_rate,
                         void *stream);
/* weights[B,T,H] = harmonic_distribution * amplitudes;  audio[B, T*bs].  Any block_size; H <= 25 596 (one frame's
 * weights, duplicated, in shared memory), else DDSP_B200_EUNSUPPORTED. */
int ddsp_b200_harmonic_frames_fwd(const float *weights, const uint64_t *phi, const uint64_t *delta,
                                  float *audio, int B, int T, int H, int block_size, void *stream);
/* d_weights[B,T,H] = sum over the frame's samples of g * sin(k*phase). */
int ddsp_b200_harmonic_frames_bwd_weights(const float *g_audio, const uint64_t *phi,
                                          const uint64_t *delta, float *d_weights, int B, int T,
                                          int H, int block_size, void *stream);
/* d_f0[B,T] (only when f0 requires grad).  scratch: float[2*B*T]. */
int ddsp_b200_harmonic_frames_bwd_f0(const float *g_audio, const float *weights,
                                     const uint64_t *phi, const uint64_t *delta, float *scratch,
                                     float *d_f0, int B, int T, int H, int block_size,
                                     double sample_rate, void *stream);

/* ---- a3+a6 in one launch: projection outputs -> controls -> audio   (ddsp/models/decoder.py:106-110,
 *      ddsp/models/modules.py:44-67,73 get_controls + the in-place product, modules.py:69-80 forward) -------------
 * The control net's raw outputs go straight into the oscillator bank: the bank's prologue applies scale_function,
 * the Nyquist mask and the normalisation to the CTA's frame rows (bit-identical to ddsp_b200_harmonic_controls_fwd),
 * and the backward's epilogue takes the weight gradients through the controls' backward.  amp_raw / dist_raw (and
 * their gradients) are rows of amp_stride / dist_stride floats, so views into the (rows, H+1) output of
 * decoder.py:106 `harmonic_proj` are read and written in place (amp_raw = param, stride H+1; dist_raw = param + 1).
 * Outputs: amps[B*T], weights[B*T,H] (what the reference's harmonic_ctrls dict holds after forward), audio[B,T*bs].
 * H <= 256 and block_size % 4 == 0 (ddsp_b200_harmonic_frames_raw_supported), else DDSP_B200_EUNSUPPORTED: use the
 * two-launch path above.                                                                                          */
int ddsp_b200_harmonic_frames_raw_supported(int H, int block_size);
int ddsp_b200_harmonic_frames_raw_fwd(const float *amp_raw, int64_t amp_stride, const float *dist_raw,
                                      int64_t dist_stride, const float *f0, const uint64_t *phi,
                                      const uint64_t *delta, float *amps, float *weights, float *audio, int B,
                                      int T, int H, int block_size, float sample_rate, void *stream);
/* The same with the phase scan inside the launch: phi / delta are OUTPUTS here (kept for the backward), phase0 (may be
 * NULL) and phase_end (may be NULL) as in ddsp_b200_phase_scan; same bits as scan + ddsp_b200_harmonic_frames_raw_fwd. */
int ddsp_b200_harmonic_frames_raw_scan_fwd(const float *amp_raw, int64_t amp_stride, const float *dist_raw,
                                           int64_t dist_stride, const float *f0, const double *phase0, uint64_t *phi,
                                           uint64_t *delta, double *phase_end, float *amps, float *weights,
                                           float *audio, int B, int T, int H, int block_size, double sample_rate,
                                           void *stream);
int ddsp_b200_harmonic_frames_raw_bwd(const float *g_audio, const float *amp_raw, int64_t amp_stride,
                                      const float *dist_raw, int64_t dist_stride, const float *f0,
                                      const uint64_t *phi, const uint64_t *delta, float *d_amp_raw,
                                      int64_t d_amp_stride, float *d_dist_raw, int64_t d_dist_stride, int B, int T,
                                      int H, int block_size, float sample_rate, void *stream);

/* ---- a5  harmonic_synth at audio rate (generic signature)    (ddsp/core.py:136-141) -------- */
/* f0[B,N], amps[B,N,H] -> audio[B,N];  phase[B*N] uint64 workspace (Q0.64 turns, inclusive). */
int ddsp_b200_phase_scan_audio_rate(const float *f0, uint64_t *phase, int B, int64_t N,
                                    double sample_rate, void *stream);
int ddsp_b200_harmonic_audio_rate_fwd(const float *amps, const uint64_t *phase, float *audio, int B,
                                      int64_t N, int H, void *stream);
/* d_amps[B,N,H] and, if d_f0 != NULL, d_f0[B,N] (dphi[B*N] float workspace needed then). */
int ddsp_b200_harmonic_audio_rate_bwd(const float *g_audio, const float *amps,
                                      const uint64_t *phase, float *d_amps, float *dphi,
                                      float *d_f0, int B, int64_t N, int H, double sample_rate,
                                      void *stream);

/* ---- a7  amp_to_impulse_response                             (ddsp/core.py:144-166) -------- */
/* amp[rows,NB] -> ir[rows,target]: irfft (size 2(NB-1)), roll, periodic Hann, pad/crop, roll back */
int ddsp_b200_amp_to_ir_fwd(const float *amp, float *ir, int64_t rows, int NB, int target,
                            void *stream);
int ddsp_b200_amp_to_ir_bwd(const float *d_ir, float *d_amp, int64_t rows, int NB, int target,
                            void *stream);

/* ---- a7+a8+a9  FilteredNoise.forward, fused        (ddsp/models/modules.py:116-128) -------- */
/* mags[rows,NB], noise[rows,bs] (the uniform(-1,1) draw, an INPUT) -> out[rows*bs]; rows = B*T;
 * requires bs >= 2(NB-1), bs % 4 == 0, (NB-1) % 4 == 0.
 * apply_scale != 0: `mags` are the raw noise_proj outputs and FilteredNoise.get_controls
 *   (modules.py:111-114: scale_function(raw + bias)) is applied inside the kernel.
 * add != NULL: out = filtered noise + add[rows*bs] (decoder.py:121: harmonic + noise).
 * Backward: d_mags w.r.t. what `mags` was (raw when apply_scale, which then needs mags_raw).      */
/* design: the constant IR-design matrix of ddsp_b200_noise_design_table(NB) (caller-owned; NULL selects
 * the first-generation kernels that rebuild the cosine sums per frame).                           */
int64_t ddsp_b200_noise_design_size(int NB);                       /* floats */
int ddsp_b200_noise_design_table(float *table, int NB, void *stream);
int ddsp_b200_filtered_noise_fwd(const float *mags, const float *noise, const float *add,
                                 const float *design, float *out, int64_t rows, int NB, int block_size,
                                 int apply_scale, float bias, void *stream);
int ddsp_b200_filtered_noise_bwd(const float *g_out, const float *noise, const float *mags_raw,
                                 const float *design, float *d_mags, int64_t rows, int NB,
                                 int block_size, int apply_scale, float bias, void *stream);

/* ---- a3+a6 beside a7+a8+a9: the oscillator bank and the filtered noise as one pair of launches ------------------
 * ddsp_b200_harmonic_frames_raw_scan_fwd and ddsp_b200_filtered_noise_fwd (apply_scale = 1, add = NULL) in one call,
 * and their backward (ddsp_b200_filtered_noise_bwd with apply_scale = 1, ddsp_b200_harmonic_frames_raw_bwd); same
 * arguments, same bits.  The noise kernel runs as a fixed number of persistent CTAs per SM and the bank is launched
 * as its programmatic dependent on the same stream, so the two run on every SM at once (the bank is bound by the FMA
 * pipe, the noise by shared-memory wavefronts).  Work queued on `stream` after the call waits for both kernels.
 * event: a cudaEvent_t created by the caller (cudaEventDisableTiming), recorded and waited for on `stream` inside the
 * call; one call at a time per event.  ctas_per_sm: noise CTAs per SM (1 or 2; 0 = the library's choice per direction).
 * Supported when the bank takes the scan inside its launch and every noise CTA gets at least one full sweep of rows
 * (ddsp_b200_synth_pair_supported); else DDSP_B200_EUNSUPPORTED: use the two entry points on two streams.       */
int ddsp_b200_synth_pair_supported(int B, int T, int H, int NB, int block_size, int ctas_per_sm);
int ddsp_b200_synth_pair_fwd(const float *amp_raw, int64_t amp_stride, const float *dist_raw, int64_t dist_stride,
                             const float *f0, const double *phase0, uint64_t *phi, uint64_t *delta, double *phase_end,
                             float *amps, float *weights, float *audio, const float *mags_raw, const float *noise,
                             const float *design, float *noise_out, int B, int T, int H, int NB, int block_size,
                             double sample_rate, float bias, int ctas_per_sm, void *event, void *stream);
int ddsp_b200_synth_pair_bwd(const float *g_audio, const float *g_noise, const float *amp_raw, int64_t amp_stride,
                             const float *dist_raw, int64_t dist_stride, const float *f0, const uint64_t *phi,
                             const uint64_t *delta, float *d_amp_raw, int64_t d_amp_stride, float *d_dist_raw,
                             int64_t d_dist_stride, const float *mags_raw, const float *noise, const float *design,
                             float *d_mags, int B, int T, int H, int NB, int block_size, float sample_rate, float bias,
                             int ctas_per_sm, void *event, void *stream);

/* ---- FFT tables (caller-owned constant tables) --------------------------------------------- */
/* table[m] = (cos, -sin)(2*pi*m/n), m in [0,n): n float2 = 2n floats; n a power of two.  One
 * table of size n serves every transform whose size divides n (read with stride n/size).       */
int ddsp_b200_twiddle_table(float *table, int n, void *stream);
/* per-size constant table of the register-tiled FFT (ddsp_pytorch_b200/csrc/regfft.cuh), sizes
 * 64..4096: `size` float2 entries, laid out per stage as [r-1][k] so a warp reads them coalesced. */
int64_t ddsp_b200_fft_stage_twiddles_size(int n_fft);
int ddsp_b200_fft_stage_twiddles(float *table, int n_fft, void *stream);

/* ---- a9 / a10  long FFT convolution = fft_convolve            (ddsp/core.py:169-176),
 *                used by Reverb.forward                (ddsp/models/modules.py:28-35) ---------- */
/* The reference pads to 2N and calls rfft/irfft; the result is the causal convolution truncated
 * to the signal length, so any transform length n >= N + L - 1 is equivalent.  The transform is a
 * four-step FFT of n = n1*n2 points held as `work[slot][k1][k2]` float2 (frequency k = k1 + n1*k2);
 * spectra are multiplied in that layout and never transposed.  With `pair` != 0 a slot carries two
 * real rows (re = row 2p, im = row 2p+1): a real filter acts on both parts independently.
 * The host side composes (ddsp_pytorch_b200/csrc/torch_ops.cpp: fftconv_fwd / fftconv_bwd):
 *   y  = cols_inv( rows_filter( cols_fwd(x),  H ) )            H = rows_spectrum(cols_fwd(h))
 *   dx = cols_inv( rows_filter( cols_fwd(g),  H, conj ) )
 *   dh = cols_inv( rows_correlate( cols_fwd(g), cols_fwd(x), reduce ) )                         */
int ddsp_b200_conv_plan(int64_t min_len, int *n1, int *n2);          /* host only: n1*n2 >= min_len */
/* twiddle: ddsp_b200_twiddle_table of size n1*n2; stage1 / stage2: ddsp_b200_fft_stage_twiddles of
 * size n1 / n2 (constant tables of the register-tiled sub-transforms).                            */
int ddsp_b200_fft4_cols_fwd(const float *x /*[rows,len]*/, int64_t rows, int64_t len, int pair,
                            float *work, const float *twiddle, const float *stage1, int n1, int n2,
                            void *stream);
/* the same for x + x2 (x2 may be NULL): the mix `harmonic + noise` of decoder.py:121 rides in the reverb's first pass */
int ddsp_b200_fft4_cols_fwd_sum(const float *x, const float *x2, int64_t rows, int64_t len, int pair, float *work,
                                const float *twiddle, const float *stage1, int n1, int n2, void *stream);
int ddsp_b200_fft4_cols_inv(const float *work, float *out /*[rows,len]*/, int64_t rows, int64_t len,
                            int pair, const float *stage1, int n1, int n2, void *stream);
int ddsp_b200_fft4_rows_spectrum(float *work, int64_t slots, const float *twiddle, const float *stage2,
                                 int n1, int n2, void *stream);
/* h_slot_stride in complex elements between the filter spectra of successive slots (0 = shared);
 * dst may be `work` itself (in place) or a second buffer (keeps `work` = the transform of x for the
 * backward pass).                                                                                 */
int ddsp_b200_fft4_rows_filter(const float *work, float *dst, int64_t slots, const float *hspec,
                               int64_t h_slot_stride, int conj_h, const float *twiddle,
                               const float *stage2, int n1, int n2, void *stream);
/* out = rows of IFFT( FFT(g) * conj(FFT(x)) ), summed over slots into one slot when reduce != 0.
 * scratch: ddsp_b200_fft4_correlate_splits_plan(slots, reduce, n1, n2) * n1*n2 complex: the partial spectra and, on
 * the 5-smooth plans with reduce != 0, one more plane for the row counters of the in-launch finish (zeroed by the
 * call, or by the caller: ddsp_b200_fft4_rows_correlate_ex).  ddsp_b200_fft4_correlate_splits is the plan-independent upper bound.                                      */
int64_t ddsp_b200_fft4_correlate_splits(int64_t slots, int reduce);
int64_t ddsp_b200_fft4_correlate_splits_plan(int64_t slots, int reduce, int n1, int n2);   /* the same, for a given plan */
int ddsp_b200_fft4_rows_correlate(const float *work_g, const float *work_x, int64_t slots, int reduce,
                                  float *scratch, float *out, const float *twiddle, const float *stage2,
                                  int n1, int n2, void *stream);
/* The same for a caller that zeroed the row counters itself, off the critical path: n1 ints at float offset
 * ddsp_b200_fft4_correlate_counter_offset(...) of scratch (-1: this plan has no counters).  The launch leaves them zero. */
int64_t ddsp_b200_fft4_correlate_counter_offset(int64_t slots, int reduce, int n1, int n2);
int ddsp_b200_fft4_rows_correlate_ex(const float *work_g, const float *work_x, int64_t slots, int reduce,
                                     float *scratch, float *out, const float *twiddle, const float *stage2,
                                     int n1, int n2, int counters_zeroed, void *stream);

/* ---- a10  Reverb.build_impulse                       (ddsp/models/modules.py:21-26) -------- */
/* impulse[l] = noise[l]*exp(-softplus(-decay)*t[l]*500)*sigmoid(wet), impulse[0] = 1; l < L.
 * decay, wet: device scalars; t: the module's (float32) time buffer.                            */
int ddsp_b200_reverb_impulse_fwd(const float *noise, const float *decay, const float *wet,
                                 const float *t, float *impulse, int L, void *stream);
/* d_noise[L], d_decay[1], d_wet[1] from d_impulse[0..Lvalid) (taps >= Lvalid were cropped).
 * scratch: ddsp_b200_reverb_impulse_bwd_scratch() BYTES, 8-byte aligned (per-block partial sums in double).  */
int64_t ddsp_b200_reverb_impulse_bwd_scratch(void);
int ddsp_b200_reverb_impulse_bwd(const float *d_impulse, int Lvalid, const float *noise,
                                 const float *decay, const float *wet, const float *t,
                                 float *d_noise, float *d_decay, float *d_wet, int L, void *scratch, void *stream);

/* ---- a10s  streaming reverb: Reverb.forward buffer by buffer     (ddsp/models/modules.py:28-35) ------
 * modules.py:28-35 convolves one whole signal and crops the impulse to its length; played in buffers, the tail
 * of each buffer is lost.  Here the previous L-1 input samples of each voice are carried by the caller:
 *   u = [history | x] (B, L-1+N, oldest first);  y[b,n] = sum_{k<L} h[k] * u[b, L-1+n-k];
 *   history_out[b] = the last L-1 samples of u[b]  (a separate buffer from history: both are read and written by
 *   the same launch).  Zeros in history = silence before the first call.
 * x[B,N], h[L] (one impulse for all voices), history / history_out [B,L-1] (may be NULL when L == 1), y[B,N].
 * Direct form on the CUDA cores, B*N*L FMA (1 x 1024 x 48000 = 49 M per buffer); deterministic, no atomics.
 * scratch: ddsp_b200_conv_stream_scratch(B, N, L) floats (the taps' chunk sums; 0 = none needed, may be NULL). */
int64_t ddsp_b200_conv_stream_scratch(int B, int64_t N, int L);
int ddsp_b200_conv_stream_fwd(const float *x, const float *h, const float *history, float *y, float *history_out,
                              int B, int64_t N, int L, float *scratch, void *stream);

/* ---- f1  dataset features: A-weighted loudness and MFCCs  (ddsp/core.py:81-97, librosa.feature.mfcc defaults) --
 * signal[B,N] -> F = 1 + N/hop frames of the unnormalised STFT (reflect padding of n_fft/2 on each side, periodic
 * Hann window[n_fft]), bins k = 0 .. n_fft/2.
 *   loudness[B,F]  = mean over k of ln(|X[k]| + 1e-7) + a_weight[k]           (a_weight: A-weighting in dB, n_fft/2+1)
 *   mfcc[B,F,n_mfcc]: P = |X|^2, mel = 128 Slaney bands of P, dB = 10 log10(max(1e-10, mel)) clamped per row to
 *                    its maximum - 80, then dct[128][n_mfcc] (the DCT-II ortho matrix, transposed) applied to dB.
 * mel_table: floats [0,128) first bin, [128,256) bin count, [256,384) offset of the band's weights past the
 * header, then the weights back to back.  stage_twiddle: ddsp_b200_fft_stage_twiddles(n_fft).
 * loudness or mfcc may be NULL (not both); without mfcc, mel_table / dct / scratch may be NULL and one launch runs.
 * scratch: ddsp_b200_features_scratch(...) floats.  n_fft a power of two in 256..4096, 1 <= hop <= 2^30,
 * n_fft/2 < N < 2^30, 1 <= n_mfcc <= 128, 1 <= B <= 65535, else DDSP_B200_EINVAL (both functions).
 * Deterministic: sums in a fixed order, a row's output does not depend on the batch it is computed in.         */
int64_t ddsp_b200_features_scratch(int B, int64_t N, int n_fft, int hop, int n_mfcc);
int ddsp_b200_features_fwd(const float *signal, const float *window, const float *stage_twiddle, const float *a_weight,
                           const float *mel_table, const float *dct, float *loudness, float *mfcc, float *scratch,
                           int B, int64_t N, int n_fft, int hop, int n_mfcc, void *stream);

/* ---- f1  dataset pitch: YIN  (replaces ddsp/core.py:100-119, CREPE; librosa.yin's definition) --------------------
 * signal[B,N] -> N/hop frames x of L = frame_length samples (reflect padding of L/2 on each side, frame f starts at
 * f*hop of the padded signal: the frames of the loudness), W = L/2.  For tau = 0 .. max_period:
 *   d(tau) = max(0, sum_{j=1..W} (x[j] - x[j+tau])^2)      (computed as E(0) + E(tau) - 2 acf(tau) by one FFT pair)
 *   y(tau) = d(tau) / (sum_{k=1..tau} d(k) / tau + FLT_MIN),   tau in [min_period, max_period]
 * lag = the first trough of y (y(tau) < y(tau-1) and y(tau) <= y(tau+1); at min_period y < y(tau+1); never at
 * max_period) with y < threshold, else the first global minimum of y.  Parabolic shift s = -b/a through y(lag-1),
 * y(lag), y(lag+1) (a = y+ + y- - 2y, b = (y+ - y-)/2; 0 at either end of the range or when |b| >= |a|).
 *   f0[B, N/hop] = sample_rate / (lag + s)          aperiodicity[B, N/hop] = y(lag)
 * An all-zero frame has y == 0 and no trough: f0 = sample_rate / min_period, aperiodicity 0.
 * stage_twiddle: ddsp_b200_fft_stage_twiddles(frame_length).  DDSP_B200_EINVAL before any launch unless
 * 1 <= B <= 65535, L/2 < N < 2^30, L a power of two in 256..4096, hop >= 1, min_period >= 1,
 * min_period + 2 <= max_period <= L - W - 1, threshold finite, and no pointer NULL.
 * Deterministic: fixed-order sums, no atomics; a row's output does not depend on the batch it is computed in.    */
int ddsp_b200_pitch_yin_fwd(const float *signal, const float *stage_twiddle, float *f0, float *aperiodicity, int B,
                            int64_t N, int frame_length, int hop, int min_period, int max_period, float sample_rate,
                            float threshold, void *stream);

/* ---- a11  multiscale_fft, one scale                           (ddsp/core.py:27-41) --------- */
/* signal[B,N] -> mag[B, n_fft/2+1, frames], frames = 1 + N/hop (centred, reflect padded, periodic
 * Hann, normalised).  window[n_fft] is the float32 torch.hann_window(n_fft) the reference builds on
 * the CPU; twiddle is a table of size n_tab (a multiple of n_fft).                              */
/* stage_twiddle: ddsp_b200_fft_stage_twiddles(n_fft) selects the register-tiled FFT (64..4096);
 * NULL falls back to the generic radix-4 kernels driven by `twiddle`.                             */
int ddsp_b200_stft_mag_fwd(const float *signal, const float *window, const float *twiddle, int n_tab,
                           const float *stage_twiddle, float *mag, int B, int64_t N, int n_fft, int hop,
                           void *stream);
/* d_signal[B,N] (=, or += when accumulate) from d_mag; the gradient of the reflect padding goes to
 * edge[B, n_fft] and is folded in by ddsp_b200_stft_fold_edges.                                 */
int ddsp_b200_stft_mag_bwd(const float *signal, const float *d_mag, const float *window,
                           const float *twiddle, int n_tab, const float *stage_twiddle, float *d_signal,
                           float *edge, int B, int64_t N, int n_fft, int hop, int accumulate,
                           void *stream);
/* edge holds the blocks of `n_scales` scales back to back: [scale][B][n_fft]; scales: HOST array */
int ddsp_b200_stft_fold_edges(const float *edge, float *d_signal, int B, int64_t N,
                              const int *scales, int n_scales, void *stream);

/* ---- a11+a12  multiscale spectral loss, fused                 (train.py:70-76,92-103) ------ */
/* Per scale: CTA tiles of one voice; partial[] receives 2 floats per CTA (sum |Sx-Sy|, sum
 * |log(Sx+1e-7)-log(Sy+1e-7)|), ddsp_b200_mss_tiles(B,N,n_fft,hop)*B CTAs.  If d_rec != NULL the same
 * launch also produces d(loss)/d(rec) for unit upstream gradient (= or += into d_rec[B,N], reflect
 * padding part into edge[B,n_fft]).  ddsp_b200_mss_finish reduces the partials of all scales to
 * loss[0] (layout: scales back to back) and folds the edges.  scales/hops: HOST arrays.
 * The per-scale launches are independent of each other when each gets its own d_rec buffer.      */
int64_t ddsp_b200_mss_tiles(int B, int64_t N, int n_fft, int hop);   /* tiles per voice (depends on B) */
/* stage_twiddle: the table above for n_fft (may be NULL outside 64..4096, where `twiddle` is used) */
int ddsp_b200_mss_scale(const float *target, const float *rec, const float *window,
                        const float *twiddle, int n_tab, const float *stage_twiddle, float *partial,
                        float *d_rec, float *edge, int B, int64_t N, int n_fft, int hop, int accumulate,
                        void *stream);
/* d_rec_scales != NULL: the scales wrote their gradients to separate buffers [n_scales][B][N] (so
 * their launches may overlap on different streams); finish sums them in scale order and folds.   */
int ddsp_b200_mss_finish(const float *partial, const float *edge, const float *d_rec_scales,
                         float *d_rec, float *loss, int B, int64_t N, const int *scales,
                         const int *hops, int n_scales, void *stream);

/* ---- a11+a12+a13, all scales in one launch  (ddsp/core.py:27-41 + train.py:70-76,92-103 + backward) ----
 * The fused loss for the reference's setting hop = n_fft/4 (overlap 0.75), n_fft = 64..4096 powers of two
 * (mss_fused_supported says whether a scale list qualifies; anything else goes through mss_scale/mss_finish).
 * One launch covers every (scale, voice, tile of frames): each frame is transformed once, rec and target are
 * read once per scale from L2, the per-scale gradients meet in `workspace` and a second small launch sums
 * them in scale order and folds the reflect padding into d_rec (deterministic, no atomics).
 *   windows        : the scales' windows back to back (sum(scales) floats), as for mss_scale
 *   stage_twiddles : n_scales device pointers (host array), table i = ddsp_b200_fft_stage_twiddles(scales[i])
 *   workspace / partial : caller-owned scratch of the sizes mss_fused_sizes returns (floats); partial is
 *                    needed always, workspace only with d_rec
 *   d_rec == NULL  : loss only.                                                                       */
int ddsp_b200_mss_fused_supported(const int *scales, const int *hops, int n_scales);
int ddsp_b200_mss_fused_sizes(int B, int64_t N, const int *scales, int n_scales, int64_t *workspace_floats,
                              int64_t *partial_floats);
/* plan of scale `which`: out8 = {frames, hop, frames per tile, tiles per voice, thread groups per CTA, frames per
 * run, first frame slot past the last tile, floats per voice of the scale's gradient plane}                      */
int ddsp_b200_mss_fused_plan(int B, int64_t N, const int *scales, int n_scales, int which, int64_t *out8);
int ddsp_b200_mss_fused(const float *target, const float *rec, const float *windows,
                        const float *const *stage_twiddles, float *workspace, float *partial, float *d_rec,
                        float *loss, int B, int64_t N, const int *scales, int n_scales, void *stream);

/* ---- f3 (next row)  GRU recurrence of the control net  (ddsp/core.py:132-133, decoder.py:40,59,65) --- */
/* The cuDNN GRU the reference calls runs one SGEMM + one element-wise launch per time step.  Here the
 * recurrence is one launch: 16-CTA clusters keep W_hh (3H x H fp32) in distributed shared memory.
 * H must be 512; PyTorch gate order (r, z, n).  gi[B,T,3H] = x W_ih^T + b_ih (a library GEMM, caller).
 * fwd: y[B,T,H] = h_1..h_T; gates[B,T,4H] = r, z, n, W_hn h + b_hn (NULL for inference); h0 may be NULL.
 * bwd: dgi, dgh [B,T,3H] gradients of gi and of gh = W_hh h + b_hh; dh0[B,H]; dhT = gradient of the
 * last hidden state (may be NULL).  Returns DDSP_B200_EUNSUPPORTED where such clusters cannot run.  */
int ddsp_b200_gru_resident_clusters(void);
int ddsp_b200_gru_fwd(const float *gi, const float *w_hh, const float *b_hh, const float *h0, float *y,
                      float *gates, int B, int T, int H, void *stream);
int ddsp_b200_gru_bwd(const float *dy, const float *dhT, const float *w_hh, const float *y, const float *h0,
                      const float *gates, float *dgi, float *dgh, float *dh0, int B, int T, int H,
                      void *stream);

/* ---- f3 (next row)  fp32-accurate GEMM on the tcgen05 tensor cores for the control net's nn.Linear layers
 * and the GRU projections (ddsp/core.py:122-133, decoder.py:40-68,86-87; torch runs them as SIMT SGEMM).
 * Operands are split once into three bf16 parts x = b0 + b1 + b2 (exact); C = sum of the six leading part
 * products with fp32 accumulation (tensor memory, promoted to registers every 64 values of K).
 * gemm3x_ld(K): padded column count of a split operand.  gemm3x_split: x (rows x cols, row pitch ld) ->
 * out[3 * part_rows][gemm3x_ld(K)] bf16: part p in rows [p * part_rows, p * part_rows + R), K padding zeroed;
 * transpose = 0: operand = x (R = rows, K = cols); 1: operand = x^T (R = cols, K = rows).
 * gemm3x_split_both: the operands of x and of x^T from one read of x.  gemm3x_split_colsum: gemm3x_split
 * (transpose = 0) that also returns the column sums of x (bias gradient when x = dy; deterministic).
 * gemm3x: C[M][N] (row pitch ldc) = A B^T + bias (bias may be NULL), A logically M x K, B logically N x K.
 * Each operand is a split matrix (parts x_part_rows rows apart, row pitch x_ld elements) stored K-major
 * (x_mn = 0: rows = M or N, columns = K) or MN-major (x_mn = 1: rows = K, columns = M or N; x_part_rows a
 * multiple of 64 with rows K..x_part_rows zero, which gemm3x_split writes when given such a part_rows), so a
 * matrix split once serves y = x W^T, dx = dy W and dW = dy^T x without transposed copies.
 * gemm3x_splits: K splits used for a shape; when > 1 pass workspace of splits * M * N floats.             */
int64_t ddsp_b200_gemm3x_ld(int64_t k);
int ddsp_b200_gemm3x_splits(int M, int N, int K);
int ddsp_b200_gemm3x_split(const float *x, int64_t rows, int64_t cols, int64_t ld, int transpose, void *out,
                           int64_t part_rows, void *stream);
int64_t ddsp_b200_gemm3x_colsum_scratch(int64_t part_rows, int64_t cols);
int ddsp_b200_gemm3x_split_colsum(const float *x, int64_t rows, int64_t cols, int64_t ld, void *out,
                                  int64_t part_rows, float *colsum, float *partial, void *stream);
int ddsp_b200_gemm3x_split_both(const float *x, int64_t rows, int64_t cols, int64_t ld, void *out,
                                int64_t part_rows, void *out_t, int64_t part_rows_t, void *stream);
int ddsp_b200_gemm3x(const void *a, int64_t a_part_rows, int64_t a_ld, int a_mn, const void *b,
                     int64_t b_part_rows, int64_t b_ld, int b_mn, const float *bias, float *c, int64_t ldc, int M,
                     int N, int K, float *workspace, void *stream);

/* ---- f3 (next row)  LayerNorm + LeakyReLU of the MLP blocks in one pass (ddsp/core.py:122-129) ------
 * y = leaky_relu(layer_norm(x; gamma, beta, eps), slope) over rows of N = 128, 256, 384 or 512 floats;
 * stats[rows][2] = mean, rstd kept for the backward (NULL for inference).  bwd: dx, d_gamma, d_beta;
 * partial = ln_lrelu_slots(rows) * 2 * N floats of scratch (deterministic two-level column sums).        */
int ddsp_b200_ln_lrelu_slots(int64_t rows);
int ddsp_b200_ln_lrelu_fwd(const float *x, const float *gamma, const float *beta, float *y, float *stats,
                           int64_t rows, int N, float eps, float slope, void *stream);
int ddsp_b200_ln_lrelu_bwd(const float *dy, const float *x, const float *gamma, const float *beta,
                           const float *stats, float *dx, float *d_gamma, float *d_beta, float *partial,
                           int64_t rows, int N, float slope, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* DDSP_B200_H */
