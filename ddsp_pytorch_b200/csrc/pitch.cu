// K6: pitch of a dataset's signals by YIN (librosa.yin's definition; SURVEY 8f, the reference's CREPE preprocessing).
//
// Reference path replaced:
//   ddsp/core.py:100-119  extract_pitch: CREPE (a TensorFlow network with Viterbi smoothing), one f0 per block
//
// Frames: the signal reflect-padded by L/2 on each side, frame f = padded[f*hop, f*hop + L), f < N / hop (the
// frames of extract_loudness, DESIGN.md 3.8).  With W = L/2 and x the frame:
//   d(tau) = sum_{j=1..W} (x[j] - x[j+tau])^2 = E(0) + E(tau) - 2 acf(tau),   tau = 0 .. max_period
//   E(tau) = sum_{j=tau+1..tau+W} x[j]^2,  acf(tau) = sum_{j=1..W} x[j] x[j+tau]          (d clamped at 0)
//   y(tau) = d(tau) / (sum_{k=1..tau} d(k) / tau + FLT_MIN),                              tau = min_period .. max_period
// The lag is the first trough of y below the threshold (else the first global minimum of y), refined by a parabola
// through its neighbours; f0 = sr / (lag + shift), aperiodicity = y(lag).
//
// One launch, one CTA per (tile of frames, row); the frames never go to HBM.  Per batch of G frames, each frame is
// one L-point complex FFT of the register-tiled kind (regfft.cuh) with the frame in the real part and its reversed
// window x[W], x[W-1] .. x[1] in the imaginary part.  The two spectra X, R come apart by the mirror bins, and their
// product is  X[k] R[k] = (Z[k]^2 - conj(Z[-k])^2) / 4i,  so one inverse transform gives the linear correlation
// acf(tau) at output W + tau (no wrap-around reaches it: tau <= L - W - 1).  Each frame has a transform of its own, so
// its rounding error scales with its own energy and a silent frame comes out exact.  Then one warp per frame:
//   energies: chunk sums of x^2 in double, a warp scan, and a walk over each lane's chunk (fixed order);
//   the cumulative mean of d: the same, in double (a float32 running sum, simulated on the parity tests' signals,
//   moves y by up to 7.7e-6 relative: no lag changed there, but double costs one add per lag and takes that error
//   out of every threshold and trough comparison);
//   the first qualifying trough: a warp min over each lane's first candidate; the first global minimum: a warp
//   min over (value, lag).
// No atomics: outputs are bit-identical from run to run, and a row's result does not depend on its batch or tile.
#include <cfloat>
#include <climits>
#include <cmath>

#include "common.cuh"
#include "regfft.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;

template <int LG>
struct YinCfg {
    using P = regfft::Plan<LG>;
    static constexpr int L = P::N, W = L / 2;
    static constexpr int G = (kThreads / P::T) > 16 ? 16 : (kThreads / P::T);   // frames (transforms) per batch
    static constexpr int K = L / 64;            // lags per lane in the epilogue (32 lanes cover 0 .. W-1)
    static constexpr int XS = L + L / K;        // a frame's samples, one float of padding per K (conflict-free walks)
    static constexpr int DS = W + W / K;        // d, then y, per lag
    static constexpr size_t SMEM = (size_t)G * P::PITCH * sizeof(float2) + (size_t)G * (XS + DS) * sizeof(float);
};

template <int K> __device__ __forceinline__ int padk(int j) { return j + j / K; }

__device__ __forceinline__ int reflect_index(int m, int n) {
    m = m < 0 ? -m : m;
    return m >= n ? 2 * (n - 1) - m : m;
}

__device__ __forceinline__ double warp_scan_incl(double v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double u = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += u;
    }
    return v;
}
__device__ __forceinline__ double warp_excl(double incl, int lane) {
    const double u = __shfl_up_sync(0xffffffffu, incl, 1);
    return lane ? u : 0.0;
}

template <int LG>
__global__ void __launch_bounds__(kThreads, 2)
pitch_yin_kernel(const float *__restrict__ signal, const float2 *__restrict__ tw, float *__restrict__ f0_out,
                 float *__restrict__ ap_out, int64_t n, int hop, int frames, int tile_frames, int pmin, int pmax,
                 float sample_rate, float threshold) {
    using namespace regfft;
    using P = Plan<LG>;
    using C = YinCfg<LG>;
    constexpr int L = P::N, T = P::T, G = C::G, PITCH = P::PITCH, W = C::W, K = C::K;
    extern __shared__ __align__(16) float smem[];
    float2 *buf = reinterpret_cast<float2 *>(smem);                          // [G][PITCH]  transforms
    float *xs = reinterpret_cast<float *>(buf + (size_t)G * PITCH);          // [G][XS]     frame samples
    float *dv = xs + (size_t)G * C::XS;                                     // [G][DS]     acf -> d -> y

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int grp = tid / T, t = tid - grp * T;
    const bool act = grp < G;
    const int b = blockIdx.y;
    const int fa = blockIdx.x * tile_frames;
    const int fe = min(fa + tile_frames, frames);
    const float *x = signal + (size_t)b * n;
    const int Ni = (int)n;
    const int nl = pmax + 1;

    for (int fb = fa; fb < fe; fb += G) {
        __syncthreads();                                                     // previous batch consumed
        float2 v[16];
        float2 *bg = buf + (size_t)grp * PITCH;
        if (act) {
            // stage 0 straight from global memory: x[j] + i x[W - j] (j < W), x[j] (j >= W)
            const int f = fb + grp;
            const bool has = f < fe;
            const int start = f * hop - W;
            const bool inner = start >= 0 && (int64_t)start + L <= n;
            float *xq = xs + (size_t)grp * C::XS;
#pragma unroll
            for (int r = 0; r < 16; ++r) {
                const int j = t + r * T;
                float re = 0.f, im = 0.f;
                if (has) {
                    re = __ldg(x + (inner ? start + j : reflect_index(start + j, Ni)));
                    if (r < 8) im = __ldg(x + (inner ? start + W - j : reflect_index(start + W - j, Ni)));
                }
                xq[padk<K>(j)] = re;
                v[r] = make_float2(re, im);
            }
            stage_compute_store<LG, 0, false>(v, bg, t, tw);
        }
        __syncthreads();
        if (act) stage_load<LG, 1>(v, bg, t);
        __syncthreads();
        if (act) stage_compute_store<LG, 1, false>(v, bg, t, tw);
        if (P::STAGES == 3) {
            __syncthreads();
            if (act) stage_load<LG, 2>(v, bg, t);
            __syncthreads();
            if (act) stage_compute_store<LG, 2, false>(v, bg, t, tw);
        }
        __syncthreads();

        // u[k] = Z[k]^2 - conj(Z[-k])^2 = 4i X[k] R[k]: the input of the inverse transform's stage 0
        if (act) {
#pragma unroll
            for (int r = 0; r < 16; ++r) {
                const int j = t + r * T;
                const float2 a = bg[pad16(j)];
                float2 c = bg[pad16((L - j) & (L - 1))];
                c.y = -c.y;
                v[r] = c_mul(c_add(a, c), c_sub(a, c));
            }
        }
        __syncthreads();
        if (act) stage_compute_store<LG, 0, true>(v, bg, t, tw);
        __syncthreads();
        if (act) stage_load<LG, 1>(v, bg, t);
        __syncthreads();
        if (act) stage_compute_store<LG, 1, true>(v, bg, t, tw);
        if (P::STAGES == 3) {
            __syncthreads();
            if (act) stage_load<LG, 2>(v, bg, t);
            __syncthreads();
            if (act) stage_compute_store<LG, 2, true>(v, bg, t, tw);
        }
        __syncthreads();

        // acf(tau) = Re(IFFT(u / 4i))[W + tau] / L = Im(IFFT(u))[W + tau] / (4L): exact power-of-two scaling
        for (int idx = tid; idx < G * nl; idx += kThreads) {
            const int q = idx / nl, tau = idx - q * nl;
            dv[(size_t)q * C::DS + padk<K>(tau)] = buf[(size_t)q * PITCH + pad16(W + tau)].y * (0.25f / (float)L);
        }
        __syncthreads();

        // one warp per frame; lane l owns lags [lK, lK + K) and, for the energies, samples [lK, lK + K) and
        // [lK + W, lK + W + K)
        for (int q = warp; q < G; q += kWarps) {
            const int f = fb + q;
            if (f >= fe) break;
            const float *xq = xs + (size_t)q * C::XS;
            float *dq = dv + (size_t)q * C::DS;
            const int lo = lane * K;
            const int hi = min(lo + K - 1, pmax);                            // last lag of this lane (hi < lo: none)

            double s0 = 0.0, s1 = 0.0;
#pragma unroll 4
            for (int i = 0; i < K; ++i) {
                const double a = xq[padk<K>(lo + i)], c = xq[padk<K>(lo + W + i)];
                s0 = fma(a, a, s0);
                s1 = fma(c, c, s1);
            }
            const double c0 = warp_scan_incl(s0, lane), c1 = warp_scan_incl(s1, lane);
            const double head = __shfl_sync(0xffffffffu, c0, 31);             // sum_{j<W} x[j]^2
            double ea = warp_excl(c0, lane);                                 // sum_{j<lo} x[j]^2
            double eb = head + warp_excl(c1, lane);                          // sum_{j<lo+W} x[j]^2
            const double x0 = xq[padk<K>(0)], xw = xq[padk<K>(W)];
            const double e0 = fma(xw, xw, head) - fma(x0, x0, 0.0);        // E(0), the same expression as lane 0's

            // d(tau) in place of acf(tau), and the lane's sum of d(1 ..)
            double ds = 0.0;
            for (int tau = lo; tau <= hi; ++tau) {
                const double a = xq[padk<K>(tau)], c = xq[padk<K>(tau + W)];
                ea = fma(a, a, ea);                                          // sum_{j<=tau} x[j]^2
                eb = fma(c, c, eb);                                          // sum_{j<=tau+W} x[j]^2
                const double acf = dq[padk<K>(tau)];
                const float d = (float)fmax(e0 + (eb - ea) - 2.0 * acf, 0.0);
                dq[padk<K>(tau)] = d;
                if (tau >= 1) ds += d;
            }
            // y(tau) in place of d(tau), over the lag range
            double run = warp_excl(warp_scan_incl(ds, lane), lane);
            for (int tau = lo; tau <= hi; ++tau) {
                const float d = dq[padk<K>(tau)];
                if (tau >= 1) run += d;
                if (tau >= pmin) dq[padk<K>(tau)] = (float)((double)d / (run / (double)tau + (double)FLT_MIN));
            }
            __syncwarp();

            // first trough below the threshold; first global minimum
            int first = INT_MAX, arg = INT_MAX;
            float best = INFINITY;
            for (int tau = max(lo, pmin); tau <= hi; ++tau) {
                const float yv = dq[padk<K>(tau)];
                if (yv < best) {
                    best = yv;
                    arg = tau;
                }
                if (first == INT_MAX && yv < threshold && tau < pmax) {
                    const float yn = dq[padk<K>(tau + 1)];
                    const bool trough = tau == pmin ? yv < yn : (yv < dq[padk<K>(tau - 1)] && yv <= yn);
                    if (trough) first = tau;
                }
            }
            first = (int)__reduce_min_sync(0xffffffffu, (unsigned)first);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const float ob = __shfl_xor_sync(0xffffffffu, best, o);
                const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
                if (ob < best || (ob == best && oa < arg)) {
                    best = ob;
                    arg = oa;
                }
            }
            if (lane == 0) {
                const int lag = first != INT_MAX ? first : (arg != INT_MAX ? arg : pmin);
                const float yl = dq[padk<K>(lag)];
                double shift = 0.0;
                if (lag > pmin && lag < pmax) {
                    const double yp = dq[padk<K>(lag + 1)], ym = dq[padk<K>(lag - 1)];
                    const double a = yp + ym - 2.0 * (double)yl, bb = (yp - ym) * 0.5;
                    if (fabs(bb) < fabs(a)) shift = -bb / a;
                }
                const size_t o = (size_t)b * frames + f;
                f0_out[o] = (float)((double)sample_rate / ((double)lag + shift));
                ap_out[o] = yl;
            }
        }
    }
}

struct YinPlan {
    int lg, frames, tile_frames, tiles;
};

int yin_plan(int B, int64_t N, int L, int hop, int pmin, int pmax, float threshold, YinPlan *p) {
    if (B < 1 || B > 65535 || L < 256 || L > 4096 || (L & (L - 1))) return DDSP_B200_EINVAL;
    if (N <= L / 2 || N >= (1ll << 30) || hop < 1) return DDSP_B200_EINVAL;
    if (pmin < 1 || pmax > L - L / 2 - 1 || pmax < pmin + 2 || !std::isfinite(threshold)) return DDSP_B200_EINVAL;
    p->lg = 0;
    while ((1 << p->lg) < L) ++p->lg;
    p->frames = (int)(N / hop);
    const int T = L / 16;
    const int nf = kThreads / T > 16 ? 16 : kThreads / T;              // frames per batch
    // frames per tile, a whole number of batches: up to 4 batches, fewer while the grid is short of 4 CTAs per SM
    int batches = 4;
    while (batches > 1 && (int64_t)ddsp_ceil_div(p->frames, (int64_t)batches * nf) * B < 4 * DDSP_SM_COUNT) batches >>= 1;
    p->tile_frames = batches * nf;
    p->tiles = (int)ddsp_ceil_div(p->frames, p->tile_frames);
    return DDSP_B200_OK;
}

template <int LG>
int launch_yin(const float *signal, const float *stage_tw, float *f0, float *ap, int B, int64_t N, int hop, int pmin,
               int pmax, float sample_rate, float threshold, const YinPlan &p, cudaStream_t st) {
    constexpr size_t smem = YinCfg<LG>::SMEM;
    cudaError_t e = cudaFuncSetAttribute(pitch_yin_kernel<LG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    pitch_yin_kernel<LG><<<dim3(p.tiles, B), kThreads, smem, st>>>(
        signal, reinterpret_cast<const float2 *>(stage_tw), f0, ap, N, hop, p.frames, p.tile_frames, pmin, pmax,
        sample_rate, threshold);
    return ddsp_launch_status();
}

}  // namespace

extern "C" int ddsp_b200_pitch_yin_fwd(const float *signal, const float *stage_twiddle, float *f0,
                                       float *aperiodicity, int B, int64_t N, int frame_length, int hop,
                                       int min_period, int max_period, float sample_rate, float threshold,
                                       void *stream) {
    DDSP_REQUIRE(signal && stage_twiddle && f0 && aperiodicity);
    YinPlan p;
    int s = yin_plan(B, N, frame_length, hop, min_period, max_period, threshold, &p);
    if (s) return s;
    if (p.frames == 0) return DDSP_B200_OK;                             // hop > N: no whole block, nothing to do
    cudaStream_t st = (cudaStream_t)stream;
    switch (p.lg) {
        case 8: return launch_yin<8>(signal, stage_twiddle, f0, aperiodicity, B, N, hop, min_period, max_period, sample_rate, threshold, p, st);
        case 9: return launch_yin<9>(signal, stage_twiddle, f0, aperiodicity, B, N, hop, min_period, max_period, sample_rate, threshold, p, st);
        case 10: return launch_yin<10>(signal, stage_twiddle, f0, aperiodicity, B, N, hop, min_period, max_period, sample_rate, threshold, p, st);
        case 11: return launch_yin<11>(signal, stage_twiddle, f0, aperiodicity, B, N, hop, min_period, max_period, sample_rate, threshold, p, st);
        case 12: return launch_yin<12>(signal, stage_twiddle, f0, aperiodicity, B, N, hop, min_period, max_period, sample_rate, threshold, p, st);
        default: return DDSP_B200_EINVAL;
    }
}
