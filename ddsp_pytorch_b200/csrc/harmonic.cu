// K1: harmonic oscillator bank (SURVEY 8a rows a4, a5, a6 and their backward).
//
// Reference path replaced (all eager ATen, each streaming a (B,N,H) float32 tensor):
//   ddsp/models/modules.py:69-80   HarmonicSynth.forward  (upsample x2, harmonic_synth)
//   ddsp/core.py:64-67             upsample = nearest hold of a frame for block_size samples
//   ddsp/core.py:136-141           harmonic_synth = cumsum phase, sin(k*phase) bank, weighted sum
//
// Design (DESIGN.md section 3.1).  Only frame-rate controls are read and only audio is written.
//  * phase: Q0.64 turns.  phi[t] = phase before the first sample of frame t, delta[t] = per-sample
//    increment; sample j of frame t has phase phi[t] + (j+1)*delta[t]  (inclusive cumsum).
//  * forward: one thread owns 4 consecutive samples of one frame (a frame of bs samples is ceil(bs/4)
//    such groups; the last one is masked when 4 does not divide bs) and walks the harmonics with a
//    Reinsch sine recurrence in packed FP32 (FFMA2 / FADD2, two samples per register pair) + 1 FFMA2
//    for the weighted sum; the frame's H weights sit in shared memory duplicated (A, A), one LDS.128
//    per 2 harmonics per 4 samples.  The phase is folded to |psi| <= pi/2 where the recurrence is
//    stable; the fold's sign (-1)^k goes to two accumulators (odd / even harmonics).
//  * backward (d weights): one thread owns (frame, harmonic pair, chunk of samples) and walks TIME with
//    the same recurrence (the frame's phase increment is constant), so the reduction over the
//    frame's samples is a private accumulation; g is broadcast from shared memory.
#include <cmath>
#include <cstring>

#include "common.cuh"

namespace {

constexpr int kReseed = 128;   // harmonics (fwd) between exact re-seeds of the recurrence
constexpr int kChunk = 128;    // samples (bwd) per recurrence run

// ------------------------------------------------------------------------------------------
// Phase scan at frame rate: one CTA per voice.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t turns_to_q64(double turns) {
    turns -= floor(turns);
    return __double2ull_rz(turns * 18446744073709551616.0);
}

// Phase increment per sample of a float32 pitch, frac(f0 / sr) in Q0.64, in INTEGER arithmetic (no FP64 instructions in
// the scans: every CTA of the oscillator bank converts the voice's earlier frames, the audio-rate scan converts every
// sample).  f0 = m * 2^e with a 24-bit m; k = (1/sr as a double) * 2^104 as a 128-bit integer (53 significant bits:
// exact); delta = (m * k) >> (40 - e) mod 2^64 = the EXACT product truncated -- the double form rounds the product to
// 53 bits first, so this is the more accurate of the two; tests/test_abi_cpu.py checks the host build of this function
// against exact rationals.  (Device time of the bank at config 2 is the same with either form.)
struct PhaseK { uint64_t hi, lo; double inv_sr; };
static PhaseK make_phase_k(double inv_sr) {
    PhaseK k{0, 0, inv_sr};
    int ex = 0;
    const double fr = frexp(inv_sr, &ex);                       // inv_sr = fr * 2^ex, fr in [0.5, 1)
    const uint64_t mant = (uint64_t)ldexp(fr, 53);              // exact 53-bit integer
    const int sh = 104 + ex - 53;                               // k = mant << sh
    if (inv_sr > 0 && sh >= 0 && sh < 64 && (sh == 0 || (mant >> (64 - sh)) < (1ull << 40))) {
        k.lo = mant << sh;
        k.hi = sh == 0 ? 0 : mant >> (64 - sh);
    }                                                           // else hi = lo = 0: the kernels take the double form
    return k;
}
__host__ __device__ __forceinline__ uint64_t pitch_to_q64(float f0, const PhaseK k) {
#ifdef __CUDA_ARCH__
    if (k.hi == 0 && k.lo == 0) return turns_to_q64((double)f0 * k.inv_sr);
    const uint32_t bits = __float_as_uint(f0);
#else
    uint32_t bits;                                              // host build: the same integer arithmetic, for the CPU test
    memcpy(&bits, &f0, sizeof bits);
    if (k.hi == 0 && k.lo == 0) return 0;
#endif
    const int ex = (int)((bits >> 23) & 0xffu);
    if (ex == 0) return 0;                                      // zero / denormal pitch
    const uint64_t m = (uint64_t)((bits & 0x7fffffu) | 0x800000u);
    const int sh = 40 - (ex - 150);                             // right shift of the 128-bit product
    uint64_t d = 0;
    if (sh >= 0 && sh < 128) {
        const uint64_t p0 = m * k.lo;
#ifdef __CUDA_ARCH__
        const uint64_t p1 = __umul64hi(m, k.lo) + m * k.hi;     // m < 2^24, k.hi < 2^40: no overflow
#else
        const uint64_t p1 = (uint64_t)(((unsigned __int128)m * k.lo) >> 64) + m * k.hi;
#endif
        d = sh == 0 ? p0 : sh < 64 ? (p0 >> sh) | (p1 << (64 - sh)) : sh == 64 ? p1 : p1 >> (sh - 64);
    }
    return (bits >> 31) ? 0ull - d : d;                          // a negative pitch runs the phase backwards
}

constexpr int kScanThreads = 256;

__global__ void __launch_bounds__(kScanThreads)
phase_scan_kernel(const float *__restrict__ f0, const double *__restrict__ phase0,
                  uint64_t *__restrict__ phi, uint64_t *__restrict__ delta,
                  double *__restrict__ phase_end, int T, int block_size, const PhaseK pk) {
    __shared__ uint64_t tot[kScanThreads];
    const int b = blockIdx.x;
    const int tid = threadIdx.x;
    const int per = (T + kScanThreads - 1) / kScanThreads;
    const int lo = min(tid * per, T), hi = min(lo + per, T);
    const float *f = f0 + (size_t)b * T;
    uint64_t sum = 0;
    for (int t = lo; t < hi; ++t) {
        uint64_t d = pitch_to_q64(f[t], pk);
        delta[(size_t)b * T + t] = d;
        sum += d * (uint64_t)block_size;
    }
    tot[tid] = sum;
    __syncthreads();
    uint64_t run = phase0 ? turns_to_q64(phase0[b]) : 0ull;
    for (int i = 0; i < tid; ++i) run += tot[i];
    for (int t = lo; t < hi; ++t) {
        phi[(size_t)b * T + t] = run;
        run += delta[(size_t)b * T + t] * (uint64_t)block_size;
    }
    if (phase_end && tid == kScanThreads - 1) {
        // last thread's `run` is the total only if it owns the tail; recompute from totals
        uint64_t total = phase0 ? turns_to_q64(phase0[b]) : 0ull;
        for (int i = 0; i < kScanThreads; ++i) total += tot[i];
        phase_end[b] = (double)total * 5.421010862427522e-20;   // * 2^-64
    }
}

// ------------------------------------------------------------------------------------------
// Forward.  CTA = FR consecutive frames of one voice; work item = (frame, group of 4 consecutive samples), packed FP32
// (sm_100 FFMA2 / FADD2: one instruction works on a register pair holding two floats).  The group's two sample pairs
// keep the recurrence state (s, d, u) and the two accumulators in 64-bit registers, weights sit in shared memory already
// duplicated (A, A) so one LDS.128 feeds two harmonics.  Per harmonic and 4 samples: 6 packed math instructions.
// ------------------------------------------------------------------------------------------
constexpr int kFwdThreads = 128;
constexpr int kFwdMaxThreads = 640;   // one sweep of a 16-frame, 160-sample tile (small batches)

// RAW: the CTA's weights are not read but computed from the control net's raw outputs in the prologue --
// HarmonicSynth.get_controls (modules.py:44-67: scale_function on both, Nyquist mask, normalise) and the in-place
// `distribution *= amplitudes` of modules.py:73, with the arithmetic of controls_fwd_kernel (bit-identical results);
// one warp per frame row.  Amplitudes and weights are also written out (the model returns them as harmonic_ctrls).
struct RawControls {
    const float *amp_raw, *dist_raw, *f0;    // rows of amp_stride / dist_stride floats (views into the projection)
    long long amp_stride, dist_stride;
    float nyq;
    float *amps, *weights;                   // [B*T], [B*T][H]
    // scan != 0: the CTA also does the phase scan for its frames (phase_scan_kernel's integer arithmetic: exact and
    // associative, so the same bits) and writes phi / delta for the backward; phase0 / phase_end as in the scan
    int scan, block_size;
    PhaseK pk;
    const double *phase0;
    double *phase_end;
    uint64_t *phi_out, *delta_out;
};

// (64 registers: eight 128-thread CTAs per SM.  The prologue's scan and controls would otherwise raise the count to 74
// = six CTAs; __maxnreg__ and __launch_bounds__ exclude each other, 640 threads x 64 registers fit the register file)
template <bool RAW>
__global__ void __maxnreg__(64)
harmonic_frames_fwd_x2_kernel(const float *__restrict__ weights, const uint64_t *__restrict__ phi,
                              const uint64_t *__restrict__ delta, float *__restrict__ audio, int T,
                              int H, int Hp, int bs, int FR, const RawControls rc) {
    extern __shared__ __align__(16) float smem[];
    float2 *w2 = reinterpret_cast<float2 *>(smem);                         // [FR][Hp] of (A, A)
    uint64_t *sphi = reinterpret_cast<uint64_t *>(w2 + (size_t)FR * Hp);   // [FR]
    uint64_t *sdel = sphi + FR;

    const int b = blockIdx.y;
    const int t0 = blockIdx.x * FR;
    const int nfr = min(FR, T - t0);
    const int tid = threadIdx.x;
    const int nthr = blockDim.x;                          // kFwdThreads, or more when the grid alone cannot fill the GPU
    if (RAW) {
        // phase A, every thread busy: v = scale_function(raw) * mask per (frame, harmonic), parked in the weight table
        for (int i = tid; i < nfr * H; i += nthr) {
            const int f = i / H, k = i - f * H;
            const size_t row = (size_t)b * T + t0 + f;
            const float v = ddsp_scale_fn(rc.dist_raw[row * rc.dist_stride + k]) * ddsp_nyquist_mask(rc.f0[row], k + 1, rc.nyq);
            w2[f * Hp + k].x = v;
        }
        __syncthreads();
        // phase B, one warp per frame row: normalise (controls_fwd_kernel's summation order), scale by the amplitude
        const int lane = tid & 31;
        constexpr int kKeepF = 8;                          // H <= 256 (the host falls back to the two-launch path above)
        for (int f = tid >> 5; f < nfr; f += nthr >> 5) {
            const size_t row = (size_t)b * T + t0 + f;
            float vk[kKeepF];
            float sum = 0.f;
#pragma unroll
            for (int i = 0; i < kKeepF; ++i) {
                const int k = lane + 32 * i;
                vk[i] = k < H ? w2[f * Hp + k].x : 0.f;
                sum += vk[i];
            }
            sum = ddsp_warp_sum(sum);
            const float amp = ddsp_scale_fn(rc.amp_raw[row * rc.amp_stride]);
#pragma unroll
            for (int i = 0; i < kKeepF; ++i) {
                const int k = lane + 32 * i;
                if (k < Hp) {
                    float a = 0.f;
                    if (k < H) {
                        const float n = vk[i] / sum;
                        a = n * amp;                       // modules.py:73: distribution *= amplitudes
                        rc.weights[row * H + k] = a;
                    }
                    w2[f * Hp + k] = make_float2(a, a);
                }
            }
            if (lane == 0) rc.amps[row] = amp;
        }
    } else {
        const float *wg = weights + ((size_t)b * T + t0) * H;
        for (int i = tid; i < nfr * Hp; i += nthr) {
            const int f = i / Hp, k = i - f * Hp;
            const float a = k < H ? __ldg(wg + (size_t)f * H + k) : 0.f;
            w2[i] = make_float2(a, a);
        }
    }
    if (RAW && rc.scan) {
        // phase before the CTA's first frame = phase0 + block * (sum of the increments of every earlier frame)
        __shared__ uint64_t wsum[kFwdMaxThreads / 32];
        const float *fv = rc.f0 + (size_t)b * T;
        uint64_t part = 0;
        for (int t = tid; t < t0; t += nthr) part += pitch_to_q64(fv[t], rc.pk);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        if ((tid & 31) == 0) wsum[tid >> 5] = part;
        if (tid < nfr) sdel[tid] = pitch_to_q64(fv[t0 + tid], rc.pk);
        __syncthreads();
        if (tid == 0) {
            uint64_t run = rc.phase0 ? turns_to_q64(rc.phase0[b]) : 0ull;
            for (int i = 0; i < (nthr >> 5); ++i) run += wsum[i] * (uint64_t)rc.block_size;
            for (int f = 0; f < nfr; ++f) {
                sphi[f] = run;
                run += sdel[f] * (uint64_t)rc.block_size;
            }
            if (rc.phase_end && t0 + nfr == T) rc.phase_end[b] = (double)run * 5.421010862427522e-20;   // * 2^-64
        }
        __syncthreads();
        if (tid < nfr) {
            rc.phi_out[(size_t)b * T + t0 + tid] = sphi[tid];
            rc.delta_out[(size_t)b * T + t0 + tid] = sdel[tid];
        }
    } else {
        if (tid < nfr) {
            sphi[tid] = phi[(size_t)b * T + t0 + tid];
            sdel[tid] = delta[(size_t)b * T + t0 + tid];
        }
        __syncthreads();
    }

    const int G = (bs + 3) >> 2;                          // groups per frame (4 | bs: item it = the CTA's samples 4it..4it+3)
    float *out = audio + ((size_t)b * T + t0) * bs;
    for (int it = tid; it < nfr * G; it += nthr) {
        const int f = it / G;
        const int j0 = 4 * (it - f * G);
        const uint64_t ph = sphi[f], dl = sdel[f];
        const ulonglong2 *wr = reinterpret_cast<const ulonglong2 *>(w2 + (size_t)f * Hp);   // 2 harmonics each

        float q[4], ch[4], s0[4], u0[4];
        int flip[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const uint64_t p = ph + (uint64_t)(j0 + e + 1) * dl;
            const float x = ddsp_fold_quarter(p, &flip[e]) * DDSP_PI_F;
            const float sh = ddsp_sin_q(x);
            ch[e] = ddsp_cos_q(x);
            q[e] = 2.f * sh;
            u0[e] = -q[e] * q[e];
            s0[e] = q[e] * ch[e];
        }
        uint64_t sA = pk2(s0[0], s0[1]), sB = pk2(s0[2], s0[3]);
        uint64_t dA = sA, dB = sB;
        const uint64_t uA = pk2(u0[0], u0[1]), uB = pk2(u0[2], u0[3]);
        uint64_t aeA = 0, aeB = 0, aoA = 0, aoB = 0;                       // (+0.f, +0.f)
        for (int k0 = 0; k0 < Hp; k0 += kReseed) {
            if (k0 > 0) {
                float sn[4], dn[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const uint64_t p = ph + (uint64_t)(j0 + e + 1) * dl;
                    const uint32_t r = (uint32_t)(((p >> 62) + 1) >> 1);
                    const uint64_t psi = p - ((uint64_t)r << 63);
                    const float a = ddsp_turns_signed((uint64_t)(k0 + 1) * psi) * DDSP_2PI_F;
                    float sk, ck;
                    __sincosf(a, &sk, &ck);
                    sn[e] = sk;
                    dn[e] = q[e] * fmaf(ck, ch[e], sk * (0.5f * q[e]));
                }
                sA = pk2(sn[0], sn[1]); sB = pk2(sn[2], sn[3]);
                dA = pk2(dn[0], dn[1]); dB = pk2(dn[2], dn[3]);
            }
            const int kend = min(k0 + kReseed, Hp);
            for (int k = k0; k < kend; k += 4) {
                const ulonglong2 a01 = wr[k >> 1], a23 = wr[(k >> 1) + 1];
                // harmonic k+1 (odd)
                aoA = fma2(a01.x, sA, aoA); aoB = fma2(a01.x, sB, aoB);
                dA = fma2(uA, sA, dA); dB = fma2(uB, sB, dB); sA = add2(sA, dA); sB = add2(sB, dB);
                // harmonic k+2 (even)
                aeA = fma2(a01.y, sA, aeA); aeB = fma2(a01.y, sB, aeB);
                dA = fma2(uA, sA, dA); dB = fma2(uB, sB, dB); sA = add2(sA, dA); sB = add2(sB, dB);
                aoA = fma2(a23.x, sA, aoA); aoB = fma2(a23.x, sB, aoB);
                dA = fma2(uA, sA, dA); dB = fma2(uB, sB, dB); sA = add2(sA, dA); sB = add2(sB, dB);
                aeA = fma2(a23.y, sA, aeA); aeB = fma2(a23.y, sB, aeB);
                dA = fma2(uA, sA, dA); dB = fma2(uB, sB, dB); sA = add2(sA, dA); sB = add2(sB, dB);
            }
        }
        float ae[4], ao[4];
        unpk2(aeA, ae[0], ae[1]); unpk2(aeB, ae[2], ae[3]);
        unpk2(aoA, ao[0], ao[1]); unpk2(aoB, ao[2], ao[3]);
        float y[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) y[e] = flip[e] ? ae[e] - ao[e] : ae[e] + ao[e];
        float *o = out + (size_t)f * bs + j0;
        if ((bs & 3) == 0) {
            *reinterpret_cast<float4 *>(o) = make_float4(y[0], y[1], y[2], y[3]);
        } else {                                          // frames start unaligned; the last group is masked
#pragma unroll
            for (int e = 0; e < 4; ++e)
                if (j0 + e < bs) o[e] = y[e];
        }
    }
}

// ------------------------------------------------------------------------------------------
// Backward w.r.t. weights.  CTA = FR frames of one voice; work item = (chunk, frame, harmonic pair).
// ------------------------------------------------------------------------------------------
constexpr int kBwdThreads = 256;

// Packed FP32: one thread walks time for TWO harmonics (k, k+1) held in a register pair; g is staged
// duplicated (g, g) so the packed FFMA2 needs no per-step packing.
// RAW: the chunk partials are not written out as d_weights but taken through the backward of the controls
// (controls_bwd_kernel's arithmetic with d_amps = d_dist = 0) in the epilogue, one warp per frame row: the gradient
// arrives at the control net's raw outputs in the same launch.
struct RawControlsGrad {
    const float *amp_raw, *dist_raw, *f0;
    long long amp_stride, dist_stride;
    float nyq;
    float *d_amp_raw, *d_dist_raw;           // rows of damp_stride / ddist_stride floats
    long long damp_stride, ddist_stride;
};

template <bool RAW>
__global__ void __launch_bounds__(kBwdThreads)
harmonic_frames_bwd_w_x2_kernel(const float *__restrict__ g_audio, const uint64_t *__restrict__ phi,
                                const uint64_t *__restrict__ delta, float *__restrict__ d_weights,
                                int T, int H, int bs, int FR, int nchunk, int clen, const RawControlsGrad rc) {
    extern __shared__ __align__(16) float smem[];
    float2 *g2 = reinterpret_cast<float2 *>(smem);                       // [FR*bs] of (g, g)
    float *part = smem + 2 * (((size_t)FR * bs + 1) & ~(size_t)1);       // [nchunk][FR][H]
    const int b = blockIdx.y;
    const int t0 = blockIdx.x * FR;
    const int nfr = min(FR, T - t0);
    const int tid = threadIdx.x;
    const int HP2 = (H + 1) >> 1;                                        // harmonic pairs

    const float *gg = g_audio + ((size_t)b * T + t0) * bs;
    for (int i = tid; i < nfr * bs; i += kBwdThreads) {
        const float v = __ldg(gg + i);
        g2[i] = make_float2(v, v);
    }
    __syncthreads();

    const int items = nchunk * nfr * HP2;
    for (int it = tid; it < items; it += kBwdThreads) {
        const int kp = it % HP2;
        const int fc = it / HP2;
        const int f = fc % nfr;
        const int c = fc / nfr;
        const int jlo = c * clen, jhi = min(jlo + clen, bs);
        const uint64_t ph = phi[(size_t)b * T + t0 + f], dl = delta[(size_t)b * T + t0 + f];
        float s0[2], d0[2], u0[2];
        uint32_t rr[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const uint64_t kk = (uint64_t)(2 * kp + e + 1);
            const uint64_t alpha = kk * dl;
            const uint32_t r = (uint32_t)(((alpha >> 62) + 1) >> 1);
            const uint64_t af = alpha - ((uint64_t)r << 63);
            const float q = 2.f * ddsp_sin_q(ddsp_turns_signed(af) * DDSP_PI_F);
            const uint64_t th = kk * (ph + (uint64_t)(jlo + 1) * dl);
            rr[e] = r & 1u;
            u0[e] = -q * q;
            s0[e] = __sinf(ddsp_turns_signed(th) * DDSP_2PI_F);
            d0[e] = q * __cosf(ddsp_turns_signed(th - (uint64_t)((int64_t)af >> 1)) * DDSP_2PI_F);
        }
        uint64_t sP = pk2(s0[0], s0[1]), dP = pk2(d0[0], d0[1]);
        const uint64_t uP = pk2(u0[0], u0[1]);
        uint64_t a0 = 0, a1 = 0;                        // even / odd sample offsets from jlo
        const uint64_t *gp = reinterpret_cast<const uint64_t *>(g2 + (size_t)f * bs);
        int j = jlo;
        for (; j + 1 < jhi; j += 2) {
            a0 = fma2(gp[j], sP, a0);
            dP = fma2(uP, sP, dP); sP = add2(sP, dP);
            a1 = fma2(gp[j + 1], sP, a1);
            dP = fma2(uP, sP, dP); sP = add2(sP, dP);
        }
        if (j < jhi) a0 = fma2(gp[j], sP, a0);
        float e0[2], e1[2];
        unpk2(a0, e0[0], e0[1]);
        unpk2(a1, e1[0], e1[1]);
        float *dst = part + ((size_t)c * nfr + f) * H + 2 * kp;
        dst[0] = rr[0] ? e0[0] - e1[0] : e0[0] + e1[0];
        if (2 * kp + 1 < H) dst[1] = rr[1] ? e0[1] - e1[1] : e0[1] + e1[1];
    }
    __syncthreads();
    if (RAW) {
        // phase A, every thread busy: per (frame, harmonic) the chunk sum, scale_function's value and derivative
        // (the expensive part), parked as  part[0] = d weight,  sv = v = fn * mask,  sd = mask * fn'
        float *sv = part + (size_t)nchunk * nfr * H;                     // [nfr][H]   (extra shared memory of the RAW launch)
        float *sd = sv + (size_t)FR * H;
        for (int i = tid; i < nfr * H; i += kBwdThreads) {
            const int f = i / H, k = i - f * H;
            const size_t row = (size_t)b * T + t0 + f;
            float dwk = 0.f;
            for (int c = 0; c < nchunk; ++c) dwk += part[(size_t)c * nfr * H + i];
            float fn, gr;
            ddsp_scale_fn_grad(rc.dist_raw[row * rc.dist_stride + k], &fn, &gr);
            const float mask = ddsp_nyquist_mask(rc.f0[row], k + 1, rc.nyq);
            part[i] = dwk;
            sv[i] = fn * mask;
            sd[i] = mask * gr;
        }
        __syncthreads();
        // phase B, one warp per frame row: the normalisation's three sums and the outputs (controls_bwd_kernel's
        // arithmetic and summation order)
        const int lane = tid & 31;
        constexpr int kKeep = 8;                                         // H <= 256
        for (int f = tid >> 5; f < nfr; f += kBwdThreads >> 5) {
            const size_t row = (size_t)b * T + t0 + f;
            float amp, amp_grad;
            ddsp_scale_fn_grad(rc.amp_raw[row * rc.amp_stride], &amp, &amp_grad);
            // n_k = v_k / S;  g_k = d_weights_k * amp;  dv_k = (g_k - sum_j g_j n_j) / S;  d amp = sum_k d_weights_k n_k
            float gk[kKeep];
            float sum = 0.f, dot = 0.f, wdot = 0.f;
#pragma unroll
            for (int i = 0; i < kKeep; ++i) {
                const int k = lane + 32 * i;
                gk[i] = 0.f;
                if (k < H) {
                    const float dwk = part[f * H + k], v = sv[f * H + k];
                    const float g = dwk * amp;
                    sum += v;
                    dot = fmaf(g, v, dot);
                    wdot = fmaf(dwk, v, wdot);
                    gk[i] = g;
                }
            }
            sum = ddsp_warp_sum(sum);
            const float inv = 1.f / sum;
            dot = ddsp_warp_sum(dot) * inv;
            wdot = ddsp_warp_sum(wdot) * inv;
            float *out = rc.d_dist_raw + row * rc.ddist_stride;
#pragma unroll
            for (int i = 0; i < kKeep; ++i) {
                const int k = lane + 32 * i;
                if (k < H) out[k] = (gk[i] - dot) * inv * sd[f * H + k];
            }
            if (lane == 0) rc.d_amp_raw[row * rc.damp_stride] = wdot * amp_grad;
        }
        return;
    }
    float *dw = d_weights + ((size_t)b * T + t0) * H;
    for (int i = tid; i < nfr * H; i += kBwdThreads) {
        float acc = 0.f;
        for (int c = 0; c < nchunk; ++c) acc += part[(size_t)c * nfr * H + i];
        dw[i] = acc;
    }
}

// ------------------------------------------------------------------------------------------
// Backward w.r.t. f0 (only when f0 requires grad): per frame S0 = sum dphi, S1 = sum (j+1) dphi,
// dphi_n = g_n * sum_k k w_k cos(k phase_n); then d f0[t] = 2 pi/sr (S1[t] + bs * sum_{t'>t} S0[t']).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kFwdThreads)
harmonic_frames_dphi_kernel(const float *__restrict__ g_audio, const float *__restrict__ weights,
                            const uint64_t *__restrict__ phi, const uint64_t *__restrict__ delta,
                            float *__restrict__ s01, int T, int H, int bs) {
    extern __shared__ __align__(16) float smem[];
    float *w = smem;                                   // [H] pre-multiplied by k
    __shared__ float red0[kFwdThreads / 32], red1[kFwdThreads / 32];
    const int b = blockIdx.y, t = blockIdx.x, tid = threadIdx.x;
    for (int k = tid; k < H; k += kFwdThreads)
        w[k] = weights[((size_t)b * T + t) * H + k] * (float)(k + 1);
    __syncthreads();
    const uint64_t ph = phi[(size_t)b * T + t], dl = delta[(size_t)b * T + t];
    const float *g = g_audio + ((size_t)b * T + t) * bs;
    float s0 = 0.f, s1 = 0.f;
    for (int j = tid; j < bs; j += kFwdThreads) {
        const uint64_t p = ph + (uint64_t)(j + 1) * dl;
        int flip;
        const float x = ddsp_fold_quarter(p, &flip) * DDSP_PI_F;
        const float sh = ddsp_sin_q(x), chh = ddsp_cos_q(x);
        const float q = 2.f * sh;
        // cosine via the same recurrence: c_1 = cos(psi) = 1 - 2 sin^2(psi/2), e_1 = c_1 - c_0
        ddsp_osc o;
        o.u = -q * q;
        o.d = 0.5f * o.u;
        o.s = 1.f + o.d;
        float ae = 0.f, ao = 0.f;
        for (int k0 = 0; k0 < H; k0 += kReseed) {
            if (k0 > 0) {
                uint32_t r = (uint32_t)(((p >> 62) + 1) >> 1);
                uint64_t psi = p - ((uint64_t)r << 63);
                float a = ddsp_turns_signed((uint64_t)(k0 + 1) * psi) * DDSP_2PI_F;
                float sk, ck;
                __sincosf(a, &sk, &ck);
                o.s = ck;
                // c_k - c_{k-1} = -2 sin(psi/2) sin((k-1/2) psi)
                o.d = -q * fmaf(sk, chh, -ck * (0.5f * q));
            }
            const int kend = min(k0 + kReseed, H);
            for (int k = k0; k < kend; ++k) {
                if (k & 1) ae = fmaf(w[k], o.s, ae); else ao = fmaf(w[k], o.s, ao);
                o.step();
            }
        }
        const float dphi = g[j] * (flip ? ae - ao : ae + ao);
        s0 += dphi;
        s1 = fmaf((float)(j + 1), dphi, s1);
    }
    s0 = ddsp_warp_sum(s0);
    s1 = ddsp_warp_sum(s1);
    if ((tid & 31) == 0) { red0[tid >> 5] = s0; red1[tid >> 5] = s1; }
    __syncthreads();
    if (tid == 0) {
        float a = 0.f, c = 0.f;
        for (int i = 0; i < kFwdThreads / 32; ++i) { a += red0[i]; c += red1[i]; }
        s01[((size_t)b * T + t) * 2 + 0] = a;
        s01[((size_t)b * T + t) * 2 + 1] = c;
    }
}

// one thread per voice: suffix sum over frames (T is a few hundred; only runs if f0 needs grad)
__global__ void harmonic_frames_df0_scan_kernel(const float *__restrict__ s01,
                                                float *__restrict__ d_f0, int B, int T, int bs,
                                                double scale) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    double suffix = 0.0;
    for (int t = T - 1; t >= 0; --t) {
        const double s0 = s01[((size_t)b * T + t) * 2 + 0];
        const double s1 = s01[((size_t)b * T + t) * 2 + 1];
        d_f0[(size_t)b * T + t] = (float)(scale * (s1 + (double)bs * suffix));
        suffix += s0;
    }
}

// ------------------------------------------------------------------------------------------
// Audio-rate generic harmonic_synth (core.py:136-141): per-sample f0 and amplitudes.
// ------------------------------------------------------------------------------------------
constexpr int kArThreads = 256;

__global__ void __launch_bounds__(kArThreads)
phase_scan_audio_rate_kernel(const float *__restrict__ f0, uint64_t *__restrict__ phase, int64_t N,
                             const PhaseK pk) {
    __shared__ uint64_t tot[kArThreads];
    const int b = blockIdx.x, tid = threadIdx.x;
    const int64_t per = (N + kArThreads - 1) / kArThreads;
    const int64_t lo = min((int64_t)tid * per, N), hi = min(lo + per, N);
    const float *f = f0 + (size_t)b * N;
    uint64_t *p = phase + (size_t)b * N;
    uint64_t sum = 0;
    for (int64_t n = lo; n < hi; ++n) {
        sum += pitch_to_q64(f[n], pk);
        p[n] = sum;                                   // inclusive within the chunk
    }
    tot[tid] = sum;
    __syncthreads();
    uint64_t base = 0;
    for (int i = 0; i < tid; ++i) base += tot[i];
    for (int64_t n = lo; n < hi; ++n) p[n] += base;
}

constexpr int kArTile = 128;   // samples per CTA (one per thread), harmonics staged 32 at a time

template <bool BWD>
__global__ void __launch_bounds__(kArTile)
harmonic_audio_rate_kernel(const float *__restrict__ amps, const uint64_t *__restrict__ phase,
                           const float *__restrict__ g_audio, float *__restrict__ audio,
                           float *__restrict__ d_amps, float *__restrict__ dphi, int64_t N, int H) {
    __shared__ float tile[kArTile][33];
    const int b = blockIdx.y, tid = threadIdx.x;
    const int64_t n0 = (int64_t)blockIdx.x * kArTile;
    const int64_t n = n0 + tid;
    const bool live = n < N;
    const int rows = (int)min((int64_t)kArTile, N - n0);
    const uint64_t p = live ? phase[(size_t)b * N + n] : 0ull;
    int flip;
    const float x = ddsp_fold_quarter(p, &flip) * DDSP_PI_F;
    const float sh = ddsp_sin_q(x), chh = ddsp_cos_q(x);
    const float q = 2.f * sh;
    const uint32_t r = (uint32_t)(((p >> 62) + 1) >> 1);
    const uint64_t psi = p - ((uint64_t)r << 63);
    const float g = (BWD && live) ? g_audio[(size_t)b * N + n] : 0.f;
    float acc = 0.f, dacc = 0.f;
    const float *abase = amps + ((size_t)b * N + n0) * H;
    float *dbase = BWD ? d_amps + ((size_t)b * N + n0) * H : nullptr;
    const int warp = tid >> 5, lane = tid & 31;
    for (int k0 = 0; k0 < H; k0 += 32) {
        const int kn = min(32, H - k0);
        __syncthreads();
        // coalesced staging: each warp loads whole 32-harmonic runs of successive samples
        for (int rr = warp; rr < rows; rr += kArTile / 32)
            tile[rr][lane] = lane < kn ? __ldg(abase + (size_t)rr * H + k0 + lane) : 0.f;
        __syncthreads();
        // exact seed at harmonic k0+1 (every 32 harmonics)
        float a = ddsp_turns_signed((uint64_t)(k0 + 1) * psi) * DDSP_2PI_F;
        float sk, ck;
        if (k0 == 0) { sk = q * chh; ck = fmaf(-0.5f * q, q, 1.f); }
        else __sincosf(a, &sk, &ck);
        ddsp_osc os, oc;
        os.u = oc.u = -q * q;
        os.s = sk;
        os.d = q * fmaf(ck, chh, sk * (0.5f * q));
        oc.s = ck;
        oc.d = -q * fmaf(sk, chh, -ck * (0.5f * q));
        for (int k = 0; k < kn; ++k) {
            const float sgn = (flip && !((k0 + k) & 1)) ? -1.f : 1.f;   // (-1)^(k+1) for harmonic k0+k+1
            const float a_k = tile[tid][k];
            const float sv = sgn * os.s;
            if (!BWD) {
                acc = fmaf(a_k, sv, acc);
            } else {
                tile[tid][k] = g * sv;                                  // d_amps, staged for a coalesced store
                dacc = fmaf(a_k * (float)(k0 + k + 1), sgn * oc.s, dacc);
                oc.step();
            }
            os.step();
        }
        if (BWD) {
            __syncthreads();
            for (int rr = warp; rr < rows; rr += kArTile / 32)
                if (lane < kn) dbase[(size_t)rr * H + k0 + lane] = tile[rr][lane];
        }
    }
    if (live) {
        if (!BWD) audio[(size_t)b * N + n] = acc;
        else if (dphi) dphi[(size_t)b * N + n] = g * dacc;
    }
}

// d_f0[n] = 2 pi / sr * sum_{m >= n} dphi[m]  (reverse inclusive scan), one CTA per voice
__global__ void __launch_bounds__(kArThreads)
audio_rate_df0_kernel(const float *__restrict__ dphi, float *__restrict__ d_f0, int64_t N,
                      double scale) {
    __shared__ double tot[kArThreads];
    const int b = blockIdx.x, tid = threadIdx.x;
    const int64_t per = (N + kArThreads - 1) / kArThreads;
    const int64_t lo = min((int64_t)tid * per, N), hi = min(lo + per, N);
    const float *d = dphi + (size_t)b * N;
    double sum = 0.0;
    for (int64_t n = lo; n < hi; ++n) sum += d[n];
    tot[tid] = sum;
    __syncthreads();
    double suffix = 0.0;
    for (int i = tid + 1; i < kArThreads; ++i) suffix += tot[i];
    for (int64_t n = hi - 1; n >= lo; --n) {
        suffix += d[n];
        d_f0[(size_t)b * N + n] = (float)(scale * suffix);
    }
}

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
// the integer phase increment evaluated on the HOST (same source as the kernels): frac(f0 / sample_rate) in Q0.64
extern "C" uint64_t ddsp_b200_pitch_to_q64(float f0, double sample_rate) {
    return pitch_to_q64(f0, make_phase_k(1.0 / sample_rate));
}

extern "C" int ddsp_b200_phase_scan(const float *f0, const double *phase0, uint64_t *phi,
                                    uint64_t *delta, double *phase_end, int B, int T,
                                    int block_size, double sample_rate, void *stream) {
    DDSP_REQUIRE(f0 && phi && delta && B > 0 && T > 0 && block_size > 0 && sample_rate > 0);
    phase_scan_kernel<<<B, kScanThreads, 0, (cudaStream_t)stream>>>(
        f0, phase0, phi, delta, phase_end, T, block_size, make_phase_k(1.0 / sample_rate));
    return ddsp_launch_status();
}

// frames per CTA: the smallest count that makes the CTA's samples a whole number of
// (threads x 4) sweeps, so no thread idles in the last sweep (bs=160 -> 16 frames, 512 -> 1)
static int frames_per_cta(int bs, int T, int sweep, int cap) {
    int fr = 1;
    while (fr < cap && (fr * bs) % sweep != 0) ++fr;
    if ((fr * bs) % sweep != 0) fr = (sweep + bs - 1) / bs;
    if (fr > T) fr = T;
    return fr < 1 ? 1 : fr;
}

// shared by the two forward entry points; rc = nullptr: weights are read, else computed in the prologue
// programmatic: launched as the programmatic dependent of the kernel before it on `st` (the synth pair)
static int launch_frames_fwd(const float *weights, const RawControls *rc, const uint64_t *phi, const uint64_t *delta,
                             float *audio, int B, int T, int H, int block_size, cudaStream_t st,
                             bool programmatic = false) {
    const int bs = block_size;
    const int bsp = (bs + 3) & ~3;                                      // frame length in whole groups of 4 samples
    const int Hp = (H + 3) & ~3;
    int fr = frames_per_cta(bsp, T, kFwdThreads * 4, 32);
    auto bytes = [&](int fr_) { return 2 * (size_t)fr_ * Hp * sizeof(float) + 2 * (size_t)fr_ * sizeof(uint64_t); };
    while (bytes(fr) > 200 * 1024 && fr > 1) fr = (fr + 1) / 2;
    const size_t smem = bytes(fr);
    // one frame's (A, A) table must fit: H <= 25 596, far above the harmonics the Nyquist mask keeps at 1 Hz / 48 kHz
    if (smem > 200 * 1024) return DDSP_B200_EUNSUPPORTED;
    if (rc && H > 256) return DDSP_B200_EUNSUPPORTED;
    dim3 grid((T + fr - 1) / fr, B);
    // few voices (strong scaling leaves 8 per GPU, realtime 1): the grid alone leaves most warp slots empty, so
    // the CTA takes more threads = fewer sweeps per thread, until about 16 warps per SM are in flight
    int threads = kFwdThreads;
    const long long ctas = (long long)grid.x * grid.y;
    const int max_useful = (int)(((long long)fr * bsp / 4 + 31) / 32 * 32);         // one sweep covers the tile
    while (threads < kFwdMaxThreads && threads < max_useful && ctas * (threads / 32) < 16ll * DDSP_SM_COUNT)
        threads += kFwdThreads;
    if (threads > max_useful) threads = max_useful > kFwdThreads ? max_useful : kFwdThreads;
    if (threads > kFwdMaxThreads) threads = kFwdMaxThreads;
    auto kernel = rc ? harmonic_frames_fwd_x2_kernel<true> : harmonic_frames_fwd_x2_kernel<false>;
    if (smem > 48 * 1024) cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (programmatic)
        return ddsp_launch_programmatic(kernel, grid, dim3(threads), smem, st, weights, phi, delta, audio, T, H, Hp, bs,
                                        fr, rc ? *rc : RawControls{});
    kernel<<<grid, threads, smem, st>>>(weights, phi, delta, audio, T, H, Hp, bs, fr, rc ? *rc : RawControls{});
    return ddsp_launch_status();
}

extern "C" int ddsp_b200_harmonic_frames_fwd(const float *weights, const uint64_t *phi,
                                             const uint64_t *delta, float *audio, int B, int T,
                                             int H, int block_size, void *stream) {
    DDSP_REQUIRE(weights && phi && delta && audio && B > 0 && T > 0 && H > 0 && block_size > 0);
    DDSP_REQUIRE(B <= 65535);
    return launch_frames_fwd(weights, nullptr, phi, delta, audio, B, T, H, block_size, (cudaStream_t)stream);
}

extern "C" int ddsp_b200_harmonic_frames_raw_supported(int H, int block_size) {
    const int Hp = (H + 3) & ~3;
    const int fr = frames_per_cta(block_size, 1 << 30, kFwdThreads * 4, 32);
    return H >= 1 && H <= 256 && block_size > 0 && block_size % 4 == 0 &&
           2 * (size_t)fr * Hp * sizeof(float) + 2 * (size_t)fr * sizeof(uint64_t) <= 200 * 1024;
}

extern "C" int ddsp_b200_harmonic_frames_raw_fwd(const float *amp_raw, int64_t amp_stride, const float *dist_raw,
                                                 int64_t dist_stride, const float *f0, const uint64_t *phi,
                                                 const uint64_t *delta, float *amps, float *weights, float *audio,
                                                 int B, int T, int H, int block_size, float sample_rate,
                                                 void *stream) {
    DDSP_REQUIRE(amp_raw && dist_raw && f0 && phi && delta && amps && weights && audio);
    DDSP_REQUIRE(B > 0 && B <= 65535 && T > 0 && H > 0 && block_size > 0 && amp_stride >= 1 && dist_stride >= H);
    if (!ddsp_b200_harmonic_frames_raw_supported(H, block_size)) return DDSP_B200_EUNSUPPORTED;
    RawControls rc{amp_raw, dist_raw, f0, amp_stride, dist_stride, sample_rate * 0.5f, amps, weights,
                   0, block_size, PhaseK{0, 0, 0.0}, nullptr, nullptr, nullptr, nullptr};
    return launch_frames_fwd(nullptr, &rc, phi, delta, audio, B, T, H, block_size, (cudaStream_t)stream);
}

extern "C" int ddsp_b200_harmonic_frames_raw_scan_fwd(const float *amp_raw, int64_t amp_stride, const float *dist_raw,
                                                      int64_t dist_stride, const float *f0, const double *phase0,
                                                      uint64_t *phi, uint64_t *delta, double *phase_end, float *amps,
                                                      float *weights, float *audio, int B, int T, int H,
                                                      int block_size, double sample_rate, void *stream) {
    DDSP_REQUIRE(amp_raw && dist_raw && f0 && phi && delta && amps && weights && audio);
    DDSP_REQUIRE(B > 0 && B <= 65535 && T > 0 && H > 0 && block_size > 0 && amp_stride >= 1 && dist_stride >= H);
    DDSP_REQUIRE(sample_rate > 0);
    if (!ddsp_b200_harmonic_frames_raw_supported(H, block_size)) return DDSP_B200_EUNSUPPORTED;
    // every CTA of a voice redoes the scan over the voice's earlier frames: fine for 25 CTAs of 16 frames (config 2),
    // not for 375 CTAs of one 512-sample frame (config 4), which take the scan as its own launch
    const int fr = frames_per_cta(block_size, T, kFwdThreads * 4, 32);
    if ((T + fr - 1) / fr > 64) {
        phase_scan_kernel<<<B, kScanThreads, 0, (cudaStream_t)stream>>>(f0, phase0, phi, delta, phase_end, T, block_size,
                                                                       make_phase_k(1.0 / sample_rate));
        int s = ddsp_launch_status();
        if (s) return s;
        return ddsp_b200_harmonic_frames_raw_fwd(amp_raw, amp_stride, dist_raw, dist_stride, f0, phi, delta, amps,
                                                 weights, audio, B, T, H, block_size, (float)sample_rate, stream);
    }
    RawControls rc{amp_raw, dist_raw, f0, amp_stride, dist_stride, (float)sample_rate * 0.5f, amps, weights,
                   1, block_size, make_phase_k(1.0 / sample_rate), phase0, phase_end, phi, delta};
    return launch_frames_fwd(nullptr, &rc, phi, delta, audio, B, T, H, block_size, (cudaStream_t)stream);
}

// The synth pair takes the bank with the scan inside the launch only: a separate scan launch would be the noise
// kernel's dependent instead, and the bank would wait for the noise to finish.
bool ddsp_pair_bank_supported(int T, int H, int block_size) {
    if (T < 1 || !ddsp_b200_harmonic_frames_raw_supported(H, block_size)) return false;
    const int fr = frames_per_cta(block_size, T, kFwdThreads * 4, 32);
    return (T + fr - 1) / fr <= 64;
}

int ddsp_pair_bank_fwd(const float *amp_raw, int64_t amp_stride, const float *dist_raw, int64_t dist_stride,
                       const float *f0, const double *phase0, uint64_t *phi, uint64_t *delta, double *phase_end,
                       float *amps, float *weights, float *audio, int B, int T, int H, int block_size,
                       double sample_rate, cudaStream_t st) {
    DDSP_REQUIRE(amp_raw && dist_raw && f0 && phi && delta && amps && weights && audio);
    DDSP_REQUIRE(B > 0 && B <= 65535 && T > 0 && H > 0 && block_size > 0 && amp_stride >= 1 && dist_stride >= H);
    DDSP_REQUIRE(sample_rate > 0);
    if (!ddsp_pair_bank_supported(T, H, block_size)) return DDSP_B200_EUNSUPPORTED;
    RawControls rc{amp_raw, dist_raw, f0, amp_stride, dist_stride, (float)sample_rate * 0.5f, amps, weights,
                   1, block_size, make_phase_k(1.0 / sample_rate), phase0, phase_end, phi, delta};
    return launch_frames_fwd(nullptr, &rc, phi, delta, audio, B, T, H, block_size, st, true);
}

static int launch_frames_bwd(const float *g_audio, const uint64_t *phi, const uint64_t *delta, float *d_weights,
                             const RawControlsGrad *rc, int B, int T, int H, int block_size, cudaStream_t st,
                             bool programmatic = false) {
    const int bs = block_size;
    const int nchunk = (bs + kChunk - 1) / kChunk;
    const int clen = (((bs + nchunk - 1) / nchunk) + 1) & ~1;   // even, so chunk parity is uniform
    const int per_frame = nchunk * ((H + 1) / 2);                  // work items per frame
    // enough (chunk, frame, harmonic pair) items for >= 4 sweeps of the CTA
    int fr = (4 * kBwdThreads + per_frame - 1) / per_frame;
    if (fr > T) fr = T;
    if (fr < 1) fr = 1;
    auto bytes = [&](int fr_) {
        const size_t gsz = 2 * (((size_t)fr_ * bs + 1) & ~(size_t)1);
        return (gsz + (size_t)nchunk * fr_ * H + (rc ? 2 * (size_t)fr_ * H : 0)) * sizeof(float);
    };
    while (bytes(fr) > 200 * 1024 && fr > 1) fr = (fr + 1) / 2;
    const size_t smem = bytes(fr);
    if (smem > 200 * 1024) return DDSP_B200_EUNSUPPORTED;
    if (rc && H > 256) return DDSP_B200_EUNSUPPORTED;
    dim3 grid((T + fr - 1) / fr, B);
    auto kernel = rc ? harmonic_frames_bwd_w_x2_kernel<true> : harmonic_frames_bwd_w_x2_kernel<false>;
    if (smem > 48 * 1024) cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (programmatic)
        return ddsp_launch_programmatic(kernel, grid, dim3(kBwdThreads), smem, st, g_audio, phi, delta, d_weights, T, H,
                                        bs, fr, nchunk, clen, rc ? *rc : RawControlsGrad{});
    kernel<<<grid, kBwdThreads, smem, st>>>(g_audio, phi, delta, d_weights, T, H, bs, fr, nchunk, clen,
                                            rc ? *rc : RawControlsGrad{});
    return ddsp_launch_status();
}

extern "C" int ddsp_b200_harmonic_frames_bwd_weights(const float *g_audio, const uint64_t *phi,
                                                     const uint64_t *delta, float *d_weights, int B,
                                                     int T, int H, int block_size, void *stream) {
    DDSP_REQUIRE(g_audio && phi && delta && d_weights && B > 0 && T > 0 && H > 0 && block_size > 0);
    DDSP_REQUIRE(B <= 65535);
    return launch_frames_bwd(g_audio, phi, delta, d_weights, nullptr, B, T, H, block_size, (cudaStream_t)stream);
}

extern "C" int ddsp_b200_harmonic_frames_raw_bwd(const float *g_audio, const float *amp_raw, int64_t amp_stride,
                                                 const float *dist_raw, int64_t dist_stride, const float *f0,
                                                 const uint64_t *phi, const uint64_t *delta, float *d_amp_raw,
                                                 int64_t d_amp_stride, float *d_dist_raw, int64_t d_dist_stride,
                                                 int B, int T, int H, int block_size, float sample_rate,
                                                 void *stream) {
    DDSP_REQUIRE(g_audio && amp_raw && dist_raw && f0 && phi && delta && d_amp_raw && d_dist_raw);
    DDSP_REQUIRE(B > 0 && B <= 65535 && T > 0 && H > 0 && block_size > 0);
    DDSP_REQUIRE(amp_stride >= 1 && dist_stride >= H && d_amp_stride >= 1 && d_dist_stride >= H);
    RawControlsGrad rc{amp_raw, dist_raw, f0, amp_stride, dist_stride, sample_rate * 0.5f,
                       d_amp_raw, d_dist_raw, d_amp_stride, d_dist_stride};
    return launch_frames_bwd(g_audio, phi, delta, nullptr, &rc, B, T, H, block_size, (cudaStream_t)stream);
}

int ddsp_pair_bank_bwd(const float *g_audio, const float *amp_raw, int64_t amp_stride, const float *dist_raw,
                       int64_t dist_stride, const float *f0, const uint64_t *phi, const uint64_t *delta,
                       float *d_amp_raw, int64_t d_amp_stride, float *d_dist_raw, int64_t d_dist_stride, int B, int T,
                       int H, int block_size, float sample_rate, cudaStream_t st) {
    DDSP_REQUIRE(g_audio && amp_raw && dist_raw && f0 && phi && delta && d_amp_raw && d_dist_raw);
    DDSP_REQUIRE(B > 0 && B <= 65535 && T > 0 && H > 0 && block_size > 0);
    DDSP_REQUIRE(amp_stride >= 1 && dist_stride >= H && d_amp_stride >= 1 && d_dist_stride >= H);
    RawControlsGrad rc{amp_raw, dist_raw, f0, amp_stride, dist_stride, sample_rate * 0.5f,
                       d_amp_raw, d_dist_raw, d_amp_stride, d_dist_stride};
    return launch_frames_bwd(g_audio, phi, delta, nullptr, &rc, B, T, H, block_size, st, true);
}

extern "C" int ddsp_b200_harmonic_frames_bwd_f0(const float *g_audio, const float *weights,
                                                const uint64_t *phi, const uint64_t *delta,
                                                float *scratch, float *d_f0, int B, int T, int H,
                                                int block_size, double sample_rate, void *stream) {
    DDSP_REQUIRE(g_audio && weights && phi && delta && scratch && d_f0);
    DDSP_REQUIRE(B > 0 && B <= 65535 && T > 0 && H > 0 && block_size > 0 && sample_rate > 0);
    if ((size_t)H * sizeof(float) > 40 * 1024) return DDSP_B200_EUNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    harmonic_frames_dphi_kernel<<<dim3(T, B), kFwdThreads, (size_t)H * sizeof(float), st>>>(
        g_audio, weights, phi, delta, scratch, T, H, block_size);
    int s = ddsp_launch_status();
    if (s) return s;
    harmonic_frames_df0_scan_kernel<<<(B + 63) / 64, 64, 0, st>>>(
        scratch, d_f0, B, T, block_size, 6.283185307179586476925 / sample_rate);
    return ddsp_launch_status();
}

extern "C" int ddsp_b200_phase_scan_audio_rate(const float *f0, uint64_t *phase, int B, int64_t N,
                                               double sample_rate, void *stream) {
    DDSP_REQUIRE(f0 && phase && B > 0 && N > 0 && sample_rate > 0);
    phase_scan_audio_rate_kernel<<<B, kArThreads, 0, (cudaStream_t)stream>>>(f0, phase, N,
                                                                              make_phase_k(1.0 / sample_rate));
    return ddsp_launch_status();
}

extern "C" int ddsp_b200_harmonic_audio_rate_fwd(const float *amps, const uint64_t *phase,
                                                 float *audio, int B, int64_t N, int H,
                                                 void *stream) {
    DDSP_REQUIRE(amps && phase && audio && B > 0 && B <= 65535 && N > 0 && H > 0);
    dim3 grid((unsigned)ddsp_ceil_div(N, kArTile), B);
    harmonic_audio_rate_kernel<false><<<grid, kArTile, 0, (cudaStream_t)stream>>>(
        amps, phase, nullptr, audio, nullptr, nullptr, N, H);
    return ddsp_launch_status();
}

extern "C" int ddsp_b200_harmonic_audio_rate_bwd(const float *g_audio, const float *amps,
                                                 const uint64_t *phase, float *d_amps, float *dphi,
                                                 float *d_f0, int B, int64_t N, int H,
                                                 double sample_rate, void *stream) {
    DDSP_REQUIRE(g_audio && amps && phase && d_amps && B > 0 && B <= 65535 && N > 0 && H > 0);
    DDSP_REQUIRE(!d_f0 || dphi);
    cudaStream_t st = (cudaStream_t)stream;
    dim3 grid((unsigned)ddsp_ceil_div(N, kArTile), B);
    harmonic_audio_rate_kernel<true><<<grid, kArTile, 0, st>>>(amps, phase, g_audio, nullptr,
                                                               d_amps, d_f0 ? dphi : nullptr, N, H);
    int s = ddsp_launch_status();
    if (s || !d_f0) return s;
    audio_rate_df0_kernel<<<B, kArThreads, 0, st>>>(dphi, d_f0, N,
                                                    6.283185307179586476925 / sample_rate);
    return ddsp_launch_status();
}
