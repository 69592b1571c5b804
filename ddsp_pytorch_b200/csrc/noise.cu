// K2: filtered-noise branch (SURVEY 8a rows a7, a8, a9-per-frame and their backward).
//
// Reference path replaced:
//   ddsp/core.py:144-166            amp_to_impulse_response  irfft(128) -> roll -> hann -> pad -> roll
//   ddsp/models/modules.py:116-128  FilteredNoise.forward    IR, uniform noise, fft_convolve, reshape
//   ddsp/core.py:169-176            fft_convolve             rfft/irfft of size 2*block per frame
//
// What the maths is (oracle/closed_form.py: fir_taps, filtered_noise).  With F = 2(NB-1), half = F/2
//   h[n]   = (m_0 + (-1)^n m_{NB-1} + 2 sum_{k=1}^{NB-2} m_k cos(2 pi k n / F)) / F     (irfft, even)
//   IR[d]             = h[d]      * w[d+half]   d = 0..half-1        (w = periodic Hann(F))
//   IR[bs-half+e]     = h[half-e] * w[e]        e = 1..half-1
// and fft_convolve is the causal convolution truncated to the frame: only 2*half-1 = 127 taps are
// non-zero whatever the block size, so the per-frame FFTs (3 of size 2*bs) are replaced by a direct
// FIR from shared memory; the IR never goes to HBM.  Algorithmic HBM bytes: 4*(NB + 2*bs) per frame.
#include "common.cuh"

namespace {

constexpr int kNoiseThreads = 128;

// h[0..half] from mags[0..NB) for one row, cooperatively by `nthr` threads (tid in [0,nthr)).
// Uses cos(2 pi k (half-n)/F) = (-1)^k cos(2 pi k n/F): thread n produces h[n] and h[half-n].
// `ct` is a shared cos table ct[i] = cos(2 pi i / F), i in [0,F).
__device__ __forceinline__ void ir_design_row(const float *m, const float *ct, float *h, int NB,
                                              int tid, int nthr) {
    const int half = NB - 1, F = 2 * half;
    const float invF = 1.f / (float)F;
    for (int n = tid; 2 * n <= half; n += nthr) {
        float ev = 0.f, od = 0.f;
        int idx = 0;                                  // (k*n) mod F
        for (int k = 0; k < NB; ++k) {
            const float ck = (k == 0 || k == half) ? 1.f : 2.f;
            const float t = ck * m[k] * ct[idx];
            if (k & 1) od += t; else ev += t;
            idx += n;
            if (idx >= F) idx -= F;
        }
        h[n] = (ev + od) * invF;
        h[half - n] = (ev - od) * invF;               // same value twice when 2n == half
    }
}

// adjoint of ir_design_row: dm[k] = c_k/F * sum_{n=0}^{half} dh[n] cos(2 pi k n / F)
__device__ __forceinline__ void ir_design_row_bwd(const float *dh, const float *ct, float *dm, int NB,
                                                  int tid, int nthr) {
    const int half = NB - 1, F = 2 * half;
    const float invF = 1.f / (float)F;
    for (int k = tid; k < NB; k += nthr) {
        float acc = 0.f;
        int idx = 0;
        for (int n = 0; n <= half; ++n) {
            acc = fmaf(dh[n], ct[idx], acc);
            idx += k;
            if (idx >= F) idx -= F;
        }
        dm[k] = acc * invF * ((k == 0 || k == half) ? 1.f : 2.f);
    }
}

__device__ __forceinline__ float hann_periodic(int i, int F) {
    return 0.5f - 0.5f * cospif(2.f * (float)i / (float)F);
}

// ---------------------------------------------------------------------------------------------
// a7 standalone: amp[rows,NB] -> ir[rows,target], any target (pad or crop).
//   ir[i] = g'[(i+half) mod target],  g'[j] = (j < min(F,target)) ? h[(j-half) mod F] * w[j] : 0
// ---------------------------------------------------------------------------------------------
template <bool BWD>
__global__ void __launch_bounds__(kNoiseThreads)
amp_to_ir_kernel(const float *__restrict__ in, float *__restrict__ out, int64_t rows, int NB,
                 int target) {
    extern __shared__ __align__(16) float smem[];
    const int half = NB - 1, F = 2 * half;
    float *ct = smem;                // [F]
    float *m = ct + F;               // [NB]   mags (fwd) / d_amp staging (bwd)
    float *h = m + NB;               // [half+1]
    const int tid = threadIdx.x;
    for (int i = tid; i < F; i += kNoiseThreads) ct[i] = cospif(2.f * (float)i / (float)F);
    const int lim = min(F, target);
    for (int64_t row = blockIdx.x; row < rows; row += gridDim.x) {
        __syncthreads();
        if (!BWD) {
            for (int k = tid; k < NB; k += kNoiseThreads) m[k] = in[row * NB + k];
            __syncthreads();
            ir_design_row(m, ct, h, NB, tid, kNoiseThreads);
            __syncthreads();
            for (int i = tid; i < target; i += kNoiseThreads) {
                int j = i + half;
                j = j % target;
                float v = 0.f;
                if (j < lim) {
                    int n = j - half;
                    if (n < 0) n += F;
                    n = min(n, F - n);
                    v = h[n] * hann_periodic(j, F);
                }
                out[row * target + i] = v;
            }
        } else {
            for (int n = tid; n <= half; n += kNoiseThreads) h[n] = 0.f;
            __syncthreads();
            for (int i = tid; i < target; i += kNoiseThreads) {
                int j = (i + half) % target;
                if (j < lim) {
                    int n = j - half;
                    if (n < 0) n += F;
                    n = min(n, F - n);
                    atomicAdd(&h[n], in[row * target + i] * hann_periodic(j, F));  // <= 2 adds per slot
                }
            }
            __syncthreads();
            ir_design_row_bwd(h, ct, m, NB, tid, kNoiseThreads);
            __syncthreads();
            for (int k = tid; k < NB; k += kNoiseThreads) out[row * NB + k] = m[k];
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Fused FilteredNoise.forward.  CTA processes RPC rows (frames) at once; QT = bs/4 threads per row,
// each thread owns 4 consecutive outputs and slides a register window over the noise.
// Shared layout per row: m[NBp] | h[HP] | taps[F] (causal | far) | xs[half + bs] | ys[bs]
// ---------------------------------------------------------------------------------------------
struct NoiseLayout {
    int NBp, HP, F, half, bs, stride;
    __host__ __device__ NoiseLayout(int NB, int bs_) {
        half = NB - 1; F = 2 * half; bs = bs_;
        NBp = (NB + 3) & ~3; HP = (half + 1 + 3) & ~3;
        stride = NBp + HP + F + (half + bs) + bs;
        stride = (stride + 3) & ~3;
    }
    __host__ __device__ int m() const { return 0; }
    __host__ __device__ int h() const { return NBp; }
    __host__ __device__ int taps() const { return NBp + HP; }
    __host__ __device__ int xs() const { return NBp + HP + F; }
    __host__ __device__ int ys() const { return NBp + HP + F + half + bs; }
};

__global__ void __launch_bounds__(kNoiseThreads)
filtered_noise_fwd_kernel(const float *__restrict__ mags, const float *__restrict__ noise,
                          const float *__restrict__ add, float *__restrict__ out, int64_t rows, int NB,
                          int bs, int RPC, int apply_scale, float bias) {
    extern __shared__ __align__(16) float smem[];
    const NoiseLayout L(NB, bs);
    const int half = L.half, F = L.F;
    float *ct = smem;                                   // [F] cos table, then per-row areas
    float *rowbase = smem + ((F + 3) & ~3);
    const int tid = threadIdx.x;
    for (int i = tid; i < F; i += kNoiseThreads) ct[i] = cospif(2.f * (float)i / (float)F);

    const int QT = bs >> 2;                             // threads per row in the FIR phase
    for (int64_t r0 = (int64_t)blockIdx.x * RPC; r0 < rows; r0 += (int64_t)gridDim.x * RPC) {
        const int nr = (int)min((int64_t)RPC, rows - r0);
        __syncthreads();
        // ---- stage mags and noise (coalesced over the CTA's rows)
        for (int i = tid; i < nr * NB; i += kNoiseThreads) {
            const int r = i / NB, k = i - r * NB;
            const float m = __ldg(mags + (r0 + r) * NB + k);
            // modules.py:111-114 folded in: magnitudes = scale_function(raw + initial_bias)
            rowbase[r * L.stride + L.m() + k] = apply_scale ? ddsp_scale_fn(m + bias) : m;
        }
        for (int i = tid; i < nr * (half + bs); i += kNoiseThreads) {
            const int r = i / (half + bs), j = i - r * (half + bs);
            rowbase[r * L.stride + L.xs() + j] = j < half ? 0.f : __ldg(noise + (r0 + r) * bs + (j - half));
        }
        __syncthreads();
        // ---- IR design: split the CTA's threads over the rows
        {
            const int per = kNoiseThreads / nr;
            const int r = tid / per, t = tid - r * per;
            if (r < nr) {
                float *rb = rowbase + r * L.stride;
                ir_design_row(rb + L.m(), ct, rb + L.h(), NB, t, per);
            }
        }
        __syncthreads();
        for (int i = tid; i < nr * F; i += kNoiseThreads) {
            const int r = i / F, d = i - r * F;
            float *rb = rowbase + r * L.stride;
            const float *h = rb + L.h();
            // taps[0..half) causal, taps[half..F) far (far[0] = 0 because w[0] = 0)
            rb[L.taps() + d] = d < half ? h[d] * hann_periodic(d + half, F)
                                        : h[F - d] * hann_periodic(d - half, F);
        }
        __syncthreads();
        // ---- main FIR: y[i..i+3] = sum_d causal[d] * x[i-d]
        for (int w = tid; w < nr * QT; w += kNoiseThreads) {
            const int r = w / QT, i = (w - r * QT) * 4;
            const float *rb = rowbase + r * L.stride;
            const float4 *c4 = reinterpret_cast<const float4 *>(rb + L.taps());
            const float *xs = rb + L.xs() + half + i;        // xs[-d] = x[i-d], zero padded below 0
            float y0 = 0.f, y1 = 0.f, y2 = 0.f, y3 = 0.f;
            float4 hi = *reinterpret_cast<const float4 *>(xs);   // x[i..i+3]
            for (int d = 0; d < half; d += 4) {
                const float4 lo = *reinterpret_cast<const float4 *>(xs - d - 4);   // x[i-d-4..i-d-1]
                const float4 c = c4[d >> 2];
                // tap d   : x[i-d+r]      = hi.{x,y,z,w}
                y0 = fmaf(c.x, hi.x, y0); y1 = fmaf(c.x, hi.y, y1); y2 = fmaf(c.x, hi.z, y2); y3 = fmaf(c.x, hi.w, y3);
                // tap d+1 : x[i-d-1+r]    = lo.w, hi.x, hi.y, hi.z
                y0 = fmaf(c.y, lo.w, y0); y1 = fmaf(c.y, hi.x, y1); y2 = fmaf(c.y, hi.y, y2); y3 = fmaf(c.y, hi.z, y3);
                // tap d+2
                y0 = fmaf(c.z, lo.z, y0); y1 = fmaf(c.z, lo.w, y1); y2 = fmaf(c.z, hi.x, y2); y3 = fmaf(c.z, hi.y, y3);
                // tap d+3
                y0 = fmaf(c.w, lo.y, y0); y1 = fmaf(c.w, lo.z, y1); y2 = fmaf(c.w, lo.w, y2); y3 = fmaf(c.w, hi.x, y3);
                hi = lo;
            }
            *reinterpret_cast<float4 *>(const_cast<float *>(rb) + L.ys() + i) = make_float4(y0, y1, y2, y3);
        }
        __syncthreads();
        // ---- far taps: y[bs-half+t] += sum_{e=1}^{t} far[e] * x[t-e],  t = 1..half-1
        for (int w = tid; w < nr * half; w += kNoiseThreads) {
            const int r = w / half, t = w - r * half;
            float *rb = rowbase + r * L.stride;
            const float *far = rb + L.taps() + half;
            const float *x = rb + L.xs() + half;
            float acc = 0.f;
            for (int e = 1; e <= t; ++e) acc = fmaf(far[e], x[t - e], acc);
            rb[L.ys() + bs - half + t] += acc;
        }
        __syncthreads();
        for (int i = tid; i < nr * bs; i += kNoiseThreads) {
            const int r = i / bs, j = i - r * bs;
            float y = rowbase[r * L.stride + L.ys() + j];
            if (add) y += __ldg(add + (r0 + r) * bs + j);       // decoder.py:121: harmonic + noise
            out[(r0 + r) * bs + j] = y;
        }
    }
}

// Backward: d_mags from g (grad of the frame's output) and the same noise.
//   d causal[d] = sum_{i>=d} g[i] x[i-d];  d far[e] = sum_{t>=e} g[bs-half+t] x[t-e]
// ys area is reused for g; taps area receives d taps; h area receives dh.
__global__ void __launch_bounds__(kNoiseThreads)
filtered_noise_bwd_kernel(const float *__restrict__ g_out, const float *__restrict__ noise,
                          const float *__restrict__ mags_raw, float *__restrict__ d_mags, int64_t rows,
                          int NB, int bs, int RPC, int apply_scale, float bias) {
    extern __shared__ __align__(16) float smem[];
    const NoiseLayout L(NB, bs);
    const int half = L.half, F = L.F;
    float *ct = smem;
    float *rowbase = smem + ((F + 3) & ~3);
    const int tid = threadIdx.x;
    for (int i = tid; i < F; i += kNoiseThreads) ct[i] = cospif(2.f * (float)i / (float)F);

    for (int64_t r0 = (int64_t)blockIdx.x * RPC; r0 < rows; r0 += (int64_t)gridDim.x * RPC) {
        const int nr = (int)min((int64_t)RPC, rows - r0);
        __syncthreads();
        for (int i = tid; i < nr * (half + bs); i += kNoiseThreads) {
            const int r = i / (half + bs), j = i - r * (half + bs);
            rowbase[r * L.stride + L.xs() + j] = j < half ? 0.f : __ldg(noise + (r0 + r) * bs + (j - half));
        }
        for (int i = tid; i < nr * bs; i += kNoiseThreads) {
            const int r = i / bs, j = i - r * bs;
            rowbase[r * L.stride + L.ys() + j] = __ldg(g_out + (r0 + r) * bs + j);
        }
        __syncthreads();
        // d taps: one thread per (row, tap); causal taps walk the whole frame, far taps a triangle
        for (int w = tid; w < nr * F; w += kNoiseThreads) {
            const int r = w / F, d = w - r * F;
            float *rb = rowbase + r * L.stride;
            const float *g = rb + L.ys();
            const float *x = rb + L.xs() + half;             // x[-1..-half] are zeros
            float a0 = 0.f, a1 = 0.f;
            if (d < half) {
                int i = 0;
                for (; i + 1 < bs; i += 2) {
                    a0 = fmaf(g[i], x[i - d], a0);
                    a1 = fmaf(g[i + 1], x[i + 1 - d], a1);
                }
                if (i < bs) a0 = fmaf(g[i], x[i - d], a0);
            } else {
                const int e = d - half;
                if (e >= 1)
                    for (int t = e; t < half; ++t) a0 = fmaf(g[bs - half + t], x[t - e], a0);
            }
            rb[L.taps() + d] = a0 + a1;
        }
        __syncthreads();
        // dh[n] = d causal[n] w[n+half] (n < half)  +  d far[half-n] w[half-n] (1 <= half-n < half)
        for (int w = tid; w < nr * (half + 1); w += kNoiseThreads) {
            const int r = w / (half + 1), n = w - r * (half + 1);
            float *rb = rowbase + r * L.stride;
            const float *dt = rb + L.taps();
            float v = 0.f;
            if (n < half) v = dt[n] * hann_periodic(n + half, F);
            const int e = half - n;
            if (e >= 1 && e < half) v = fmaf(dt[half + e], hann_periodic(e, F), v);
            rb[L.h() + n] = v;
        }
        __syncthreads();
        {
            const int per = kNoiseThreads / nr;
            const int r = tid / per, t = tid - r * per;
            if (r < nr) {
                float *rb = rowbase + r * L.stride;
                ir_design_row_bwd(rb + L.h(), ct, rb + L.m(), NB, t, per);
            }
        }
        __syncthreads();
        for (int i = tid; i < nr * NB; i += kNoiseThreads) {
            const int r = i / NB, k = i - r * NB;
            float d = rowbase[r * L.stride + L.m() + k];
            if (apply_scale) d *= ddsp_scale_grad(__ldg(mags_raw + (r0 + r) * NB + k) + bias);
            d_mags[(r0 + r) * NB + k] = d;
        }
    }
}

// =============================================================================================
// Second generation of the fused kernels.  The IR design is linear in the magnitudes with a CONSTANT
// matrix:  taps[j] = sum_k m[k] * D[k][j],  j < F  (j < half: causal tap j, window folded in;
// j >= half: far tap e = j - half).  D (NB x F, 33 KB for 65 bands) comes from a caller-owned table
// (ddsp_b200_noise_design_table) and sits in shared memory; a sweep of RPC frames is then
//   A  stage magnitudes (+ scale_function) and noise          B  taps = M x D   (register-tiled matmul)
//   C  64-tap FIRs (main + far) with a register sliding window   D  coalesced store (+ mix-in)
// with every thread busy in every phase and 3 barriers per sweep.  Backward mirrors it:
//   d taps = correlation (same sliding-window kernel), d m = d taps x D^T (table holds D^T too).
// =============================================================================================
constexpr int kN2Threads = 256;

__global__ void noise_design_kernel(float *__restrict__ tab, int NB) {
    // tab = D[NB][F] followed by Dt[F][NBq], NBq = NB rounded up to 4
    const int half = NB - 1, F = 2 * half, NBq = (NB + 3) & ~3;
    const int total = NB * F;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int k = i / F, j = i - k * F;
        const int n = j < half ? j : half - (j - half);          // h index feeding this tap
        const int wi = j < half ? j + half : j - half;           // window index
        const double ck = (k == 0 || k == half) ? 1.0 : 2.0;
        const double c = ck * cospi(2.0 * (double)((k * n) % F) / F) / F;
        const double w = 0.5 - 0.5 * cospi(2.0 * (double)wi / F);
        const float v = (float)(c * w);
        tab[i] = v;
        tab[(size_t)total + (size_t)j * NBq + k] = v;
    }
    // zero the padding columns of Dt
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < F * (NBq - NB); i += gridDim.x * blockDim.x) {
        const int j = i / (NBq - NB), k = NB + i % (NBq - NB);
        tab[(size_t)total + (size_t)j * NBq + k] = 0.f;
    }
}

// y[0..3] = sum_{d < ntaps} taps[d] * x[-d + 0..3]   (x points at sample i; x[-1..-ntaps] must be readable)
__device__ __forceinline__ float4 fir4(const float4 *__restrict__ t4, const float *x, int ntaps) {
    float y0 = 0.f, y1 = 0.f, y2 = 0.f, y3 = 0.f;
    float4 hi = *reinterpret_cast<const float4 *>(x);
    for (int d = 0; d < ntaps; d += 4) {
        const float4 lo = *reinterpret_cast<const float4 *>(x - d - 4);
        const float4 c = t4[d >> 2];
        y0 = fmaf(c.x, hi.x, y0); y1 = fmaf(c.x, hi.y, y1); y2 = fmaf(c.x, hi.z, y2); y3 = fmaf(c.x, hi.w, y3);
        y0 = fmaf(c.y, lo.w, y0); y1 = fmaf(c.y, hi.x, y1); y2 = fmaf(c.y, hi.y, y2); y3 = fmaf(c.y, hi.z, y3);
        y0 = fmaf(c.z, lo.z, y0); y1 = fmaf(c.z, lo.w, y1); y2 = fmaf(c.z, hi.x, y2); y3 = fmaf(c.z, hi.y, y3);
        y0 = fmaf(c.w, lo.y, y0); y1 = fmaf(c.w, lo.z, y1); y2 = fmaf(c.w, lo.w, y2); y3 = fmaf(c.w, hi.x, y3);
        hi = lo;
    }
    return make_float4(y0, y1, y2, y3);
}

// a[0..3] = sum_{i < len, step 4} g[i..i+3] (x) x[i - d - 0..3]: gradient of taps d..d+3
__device__ __forceinline__ float4 corr4(const float *g, const float *x, int d, int len) {
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
    float4 lo = *reinterpret_cast<const float4 *>(x - d - 4);
    for (int i = 0; i < len; i += 4) {
        const float4 hi = *reinterpret_cast<const float4 *>(x + i - d);
        const float4 gv = *reinterpret_cast<const float4 *>(g + i);
        a0 = fmaf(gv.x, hi.x, a0); a0 = fmaf(gv.y, hi.y, a0); a0 = fmaf(gv.z, hi.z, a0); a0 = fmaf(gv.w, hi.w, a0);
        a1 = fmaf(gv.x, lo.w, a1); a1 = fmaf(gv.y, hi.x, a1); a1 = fmaf(gv.z, hi.y, a1); a1 = fmaf(gv.w, hi.z, a1);
        a2 = fmaf(gv.x, lo.z, a2); a2 = fmaf(gv.y, lo.w, a2); a2 = fmaf(gv.z, hi.x, a2); a2 = fmaf(gv.w, hi.y, a2);
        a3 = fmaf(gv.x, lo.y, a3); a3 = fmaf(gv.y, lo.z, a3); a3 = fmaf(gv.z, lo.w, a3); a3 = fmaf(gv.w, hi.x, a3);
        lo = hi;
    }
    return make_float4(a0, a1, a2, a3);
}

struct Noise2Layout {         // per-row shared areas of the second-generation kernels (floats)
    int half, F, NBq, bs, xs_len, stride;
    __host__ __device__ Noise2Layout(int NB, int bs_) {
        half = NB - 1; F = 2 * half; NBq = (NB + 3) & ~3; bs = bs_;
        xs_len = half + bs;                         // `half` zeros in front of the frame
        stride = NBq + F + xs_len + bs + half;      // m | taps | xs | ys (fwd) or g (bwd) | yf
    }
    __host__ __device__ int m() const { return 0; }
    __host__ __device__ int taps() const { return NBq; }
    __host__ __device__ int xs() const { return NBq + F; }
    __host__ __device__ int ys() const { return NBq + F + xs_len; }
    __host__ __device__ int yf() const { return NBq + F + xs_len + bs; }
};

// PAIR: launched first of the synth pair (ddsp_b200_synth_pair_fwd / _bwd); the oscillator bank is its programmatic
// dependent and is dispatched beside it as soon as every CTA has started here
template <bool PAIR>
__global__ void __launch_bounds__(kN2Threads)
filtered_noise2_fwd_kernel(const float *__restrict__ mags, const float *__restrict__ noise,
                           const float *__restrict__ add, const float *__restrict__ design,
                           float *__restrict__ out, int64_t rows, int NB, int bs, int RPC, int apply_scale,
                           float bias) {
    if (PAIR) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    extern __shared__ __align__(16) float smem[];
    const Noise2Layout L(NB, bs);
    const int half = L.half, F = L.F;
    float *D = smem;                                     // [NB][F]
    float *rowbase = D + NB * F;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    constexpr int NW = kN2Threads / 32;
    for (int i = tid; i < NB * F / 4; i += kN2Threads)
        reinterpret_cast<float4 *>(D)[i] = __ldg(reinterpret_cast<const float4 *>(design) + i);

    const int QM = bs >> 2, QF = half >> 2;              // main / far output quads per row
    for (int64_t r0 = (int64_t)blockIdx.x * RPC; r0 < rows; r0 += (int64_t)gridDim.x * RPC) {
        const int nr = (int)min((int64_t)RPC, rows - r0);
        __syncthreads();
        // ---- A: stage (one warp per row, lanes along the row: coalesced, no index division)
        for (int r = warp; r < nr; r += NW) {
            float *rb = rowbase + r * L.stride;
            const float *mg = mags + (r0 + r) * NB;
            for (int k = lane; k < NB; k += 32) {
                const float m = __ldg(mg + k);
                rb[L.m() + k] = apply_scale ? ddsp_scale_fn(m + bias) : m;
            }
            for (int j = lane; j < half; j += 32) rb[L.xs() + j] = 0.f;
            const float4 *nz = reinterpret_cast<const float4 *>(noise + (r0 + r) * bs);
            float4 *xs4 = reinterpret_cast<float4 *>(rb + L.xs() + half);
            for (int j = lane; j < QM; j += 32) xs4[j] = __ldg(nz + j);
        }
        __syncthreads();
        // ---- B: taps[r][4c..4c+3] for two rows at a time = sum_k m[r][k] * D[k][...]
        //      (lanes take consecutive 16-byte columns of D: conflict-free)
        for (int it = tid; it < ((nr + 1) >> 1) * (F / 4); it += kN2Threads) {
            const int rp = it / (F / 4), c = it - rp * (F / 4);
            const int ra = 2 * rp, rb_ = min(2 * rp + 1, nr - 1);
            const float *ma = rowbase + ra * L.stride + L.m();
            const float *mb = rowbase + rb_ * L.stride + L.m();
            const float4 *d4 = reinterpret_cast<const float4 *>(D) + c;
            float4 a = make_float4(0.f, 0.f, 0.f, 0.f), e = a;
#define DDSP_N2_MAC(X, Y, U)                                                                                  \
    a.x = fmaf(X, U.x, a.x); a.y = fmaf(X, U.y, a.y); a.z = fmaf(X, U.z, a.z); a.w = fmaf(X, U.w, a.w);      \
    e.x = fmaf(Y, U.x, e.x); e.y = fmaf(Y, U.y, e.y); e.z = fmaf(Y, U.z, e.z); e.w = fmaf(Y, U.w, e.w);
            // four magnitudes of both rows per LDS.128 (NB - 1 is a multiple of 4), same summation order as one by one
            for (int k = 0; k < NB - 1; k += 4) {
                const float4 xa = *reinterpret_cast<const float4 *>(ma + k);
                const float4 xb = *reinterpret_cast<const float4 *>(mb + k);
                const float4 u0 = d4[k * (F / 4)], u1 = d4[(k + 1) * (F / 4)];
                const float4 u2 = d4[(k + 2) * (F / 4)], u3 = d4[(k + 3) * (F / 4)];
                DDSP_N2_MAC(xa.x, xb.x, u0)
                DDSP_N2_MAC(xa.y, xb.y, u1)
                DDSP_N2_MAC(xa.z, xb.z, u2)
                DDSP_N2_MAC(xa.w, xb.w, u3)
            }
            {
                const float4 u = d4[(NB - 1) * (F / 4)];
                const float x = ma[NB - 1], y = mb[NB - 1];
                DDSP_N2_MAC(x, y, u)
            }
#undef DDSP_N2_MAC
            reinterpret_cast<float4 *>(rowbase + ra * L.stride + L.taps())[c] = a;
            if (rb_ != ra) reinterpret_cast<float4 *>(rowbase + rb_ * L.stride + L.taps())[c] = e;
        }
        __syncthreads();
        // ---- C: main FIR (causal taps) over the frame, then far FIR over its first `half` samples; the two
        //      kinds of work item are laid out one after the other so that warps do not mix them
        const int nmain = nr * QM;
        for (int it = tid; it < nmain + nr * QF; it += kN2Threads) {
            if (it < nmain) {
                const int r = it / QM, q = it - r * QM;
                float *rb = rowbase + r * L.stride;
                const float4 y = fir4(reinterpret_cast<const float4 *>(rb + L.taps()), rb + L.xs() + half + 4 * q, half);
                *reinterpret_cast<float4 *>(rb + L.ys() + 4 * q) = y;
            } else {
                const int i2 = it - nmain;
                const int r = i2 / QF, qq = i2 - r * QF;
                float *rb = rowbase + r * L.stride;
                const float4 y = fir4(reinterpret_cast<const float4 *>(rb + L.taps()) + QF,
                                      rb + L.xs() + half + 4 * qq, half);
                *reinterpret_cast<float4 *>(rb + L.yf() + 4 * qq) = y;
            }
        }
        __syncthreads();
        // ---- D: out = main + far (last `half` samples) (+ add), one warp per row, float4
        for (int r = warp; r < nr; r += NW) {
            const float *rb = rowbase + r * L.stride;
            const float4 *ys4 = reinterpret_cast<const float4 *>(rb + L.ys());
            const float4 *yf4 = reinterpret_cast<const float4 *>(rb + L.yf());
            const float4 *ad4 = add ? reinterpret_cast<const float4 *>(add + (r0 + r) * bs) : nullptr;
            float4 *o4 = reinterpret_cast<float4 *>(out + (r0 + r) * bs);
            for (int j = lane; j < QM; j += 32) {
                float4 y = ys4[j];
                if (j >= QM - QF) {
                    const float4 f = yf4[j - (QM - QF)];
                    y.x += f.x; y.y += f.y; y.z += f.z; y.w += f.w;
                }
                if (ad4) {
                    const float4 f = __ldg(ad4 + j);
                    y.x += f.x; y.y += f.y; y.z += f.z; y.w += f.w;
                }
                o4[j] = y;
            }
        }
    }
}

template <bool PAIR>
__global__ void __launch_bounds__(kN2Threads)
filtered_noise2_bwd_kernel(const float *__restrict__ g_out, const float *__restrict__ noise,
                           const float *__restrict__ mags_raw, const float *__restrict__ design,
                           float *__restrict__ d_mags, int64_t rows, int NB, int bs, int RPC,
                           int apply_scale, float bias) {
    if (PAIR) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    extern __shared__ __align__(16) float smem[];
    const Noise2Layout L(NB, bs);
    const int half = L.half, F = L.F, NBq = L.NBq;
    float *Dt = smem;                                    // [F][NBq]
    float *rowbase = Dt + F * NBq;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    constexpr int NW = kN2Threads / 32;
    const float *dt_src = design + (size_t)NB * F;
    for (int i = tid; i < F * NBq / 4; i += kN2Threads)
        reinterpret_cast<float4 *>(Dt)[i] = __ldg(reinterpret_cast<const float4 *>(dt_src) + i);
    const int QM = bs >> 2;

    for (int64_t r0 = (int64_t)blockIdx.x * RPC; r0 < rows; r0 += (int64_t)gridDim.x * RPC) {
        const int nr = (int)min((int64_t)RPC, rows - r0);
        __syncthreads();
        for (int r = warp; r < nr; r += NW) {
            float *rb = rowbase + r * L.stride;
            for (int j = lane; j < half; j += 32) rb[L.xs() + j] = 0.f;
            const float4 *nz = reinterpret_cast<const float4 *>(noise + (r0 + r) * bs);
            const float4 *gz = reinterpret_cast<const float4 *>(g_out + (r0 + r) * bs);
            float4 *xs4 = reinterpret_cast<float4 *>(rb + L.xs() + half);
            float4 *g4 = reinterpret_cast<float4 *>(rb + L.ys());
            for (int j = lane; j < QM; j += 32) {
                xs4[j] = __ldg(nz + j);
                g4[j] = __ldg(gz + j);
            }
        }
        __syncthreads();
        // ---- d taps: causal taps correlate the whole frame (long items first), far taps its last `half`
        const int ncausal = nr * (half / 4);
        for (int it = tid; it < 2 * ncausal; it += kN2Threads) {
            const bool far = it >= ncausal;
            const int i2 = far ? it - ncausal : it;
            const int r = i2 / (half / 4), tg = i2 - r * (half / 4);
            float *rb = rowbase + r * L.stride;
            const float *x = rb + L.xs() + half;
            const float4 a = far ? corr4(rb + L.ys() + bs - half, x, 4 * tg, half) : corr4(rb + L.ys(), x, 4 * tg, bs);
            *reinterpret_cast<float4 *>(rb + L.taps() + (far ? half : 0) + 4 * tg) = a;
        }
        __syncthreads();
        // ---- d m[r][4kg..] = sum_j dtaps[r][j] * Dt[j][...], two rows per thread and four taps per LDS.128
        //      (F is a multiple of 4; same summation order as one by one)
        for (int it = tid; it < ((nr + 1) >> 1) * (NBq / 4); it += kN2Threads) {
            const int rp = it / (NBq / 4), kg = it - rp * (NBq / 4);
            const int ra = 2 * rp, rb_ = min(2 * rp + 1, nr - 1);
            const float *ta = rowbase + ra * L.stride + L.taps();
            const float *tb = rowbase + rb_ * L.stride + L.taps();
            const float4 *d4 = reinterpret_cast<const float4 *>(Dt) + kg;
            float4 a = make_float4(0.f, 0.f, 0.f, 0.f), e = a;
#define DDSP_N2_MAC(X, Y, U)                                                                                  \
    a.x = fmaf(X, U.x, a.x); a.y = fmaf(X, U.y, a.y); a.z = fmaf(X, U.z, a.z); a.w = fmaf(X, U.w, a.w);      \
    e.x = fmaf(Y, U.x, e.x); e.y = fmaf(Y, U.y, e.y); e.z = fmaf(Y, U.z, e.z); e.w = fmaf(Y, U.w, e.w);
            for (int j = 0; j < F; j += 4) {
                const float4 xa = *reinterpret_cast<const float4 *>(ta + j);
                const float4 xb = *reinterpret_cast<const float4 *>(tb + j);
                const float4 u0 = d4[j * (NBq / 4)], u1 = d4[(j + 1) * (NBq / 4)];
                const float4 u2 = d4[(j + 2) * (NBq / 4)], u3 = d4[(j + 3) * (NBq / 4)];
                DDSP_N2_MAC(xa.x, xb.x, u0)
                DDSP_N2_MAC(xa.y, xb.y, u1)
                DDSP_N2_MAC(xa.z, xb.z, u2)
                DDSP_N2_MAC(xa.w, xb.w, u3)
            }
#undef DDSP_N2_MAC
#pragma unroll
            for (int h2 = 0; h2 < 2; ++h2) {
                if (h2 == 1 && rb_ == ra) break;
                const int r = h2 ? rb_ : ra;
                const float4 acc = h2 ? e : a;
                const float av[4] = {acc.x, acc.y, acc.z, acc.w};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int k = 4 * kg + q;
                    if (k < NB) {
                        float d = av[q];
                        if (apply_scale) d *= ddsp_scale_grad(__ldg(mags_raw + (r0 + r) * NB + k) + bias);
                        d_mags[(r0 + r) * NB + k] = d;
                    }
                }
            }
        }
    }
}

inline int noise_rows_per_cta(int bs) {
    int rpc = (kNoiseThreads * 4) / bs;
    if (rpc < 1) rpc = 1;
    if (rpc > 8) rpc = 8;
    return rpc;
}

}  // namespace

extern "C" int ddsp_b200_amp_to_ir_fwd(const float *amp, float *ir, int64_t rows, int NB, int target,
                                       void *stream) {
    DDSP_REQUIRE(amp && ir && rows >= 0 && NB >= 2 && target >= 1);
    if (rows == 0) return DDSP_B200_OK;
    const size_t smem = (size_t)(2 * (NB - 1) + NB + NB) * sizeof(float);
    if (smem > 48 * 1024) return DDSP_B200_EUNSUPPORTED;
    const int grid = (int)(rows < DDSP_SM_COUNT * 16 ? rows : DDSP_SM_COUNT * 16);
    amp_to_ir_kernel<false><<<grid, kNoiseThreads, smem, (cudaStream_t)stream>>>(amp, ir, rows, NB,
                                                                                 target);
    return ddsp_launch_status();
}

extern "C" int ddsp_b200_amp_to_ir_bwd(const float *d_ir, float *d_amp, int64_t rows, int NB,
                                       int target, void *stream) {
    DDSP_REQUIRE(d_ir && d_amp && rows >= 0 && NB >= 2 && target >= 1);
    if (rows == 0) return DDSP_B200_OK;
    const size_t smem = (size_t)(2 * (NB - 1) + NB + NB) * sizeof(float);
    if (smem > 48 * 1024) return DDSP_B200_EUNSUPPORTED;
    const int grid = (int)(rows < DDSP_SM_COUNT * 16 ? rows : DDSP_SM_COUNT * 16);
    amp_to_ir_kernel<true><<<grid, kNoiseThreads, smem, (cudaStream_t)stream>>>(d_ir, d_amp, rows,
                                                                                NB, target);
    return ddsp_launch_status();
}

static int noise_launch_cfg(int64_t rows, int NB, int bs, int *rpc, size_t *smem, int *grid) {
    if (NB < 3 || (NB - 1) % 4 != 0) return DDSP_B200_EUNSUPPORTED;     // half % 4 == 0 for LDS.128 taps
    if (bs % 4 != 0 || bs < 2 * (NB - 1)) return DDSP_B200_EUNSUPPORTED;  // see header
    *rpc = noise_rows_per_cta(bs);
    const NoiseLayout L(NB, bs);
    *smem = ((size_t)((L.F + 3) & ~3) + (size_t)*rpc * L.stride) * sizeof(float);
    if (*smem > 200 * 1024) return DDSP_B200_EUNSUPPORTED;
    const int64_t ctas = ddsp_ceil_div(rows, *rpc);
    *grid = (int)(ctas < DDSP_SM_COUNT * 8 ? ctas : DDSP_SM_COUNT * 8);
    return DDSP_B200_OK;
}

// second generation: needs the design table and (NB-1) % 4 == 0, bs % 4 == 0, bs >= F; rows per sweep
// chosen so that two or three CTAs share an SM
static bool noise2_cfg(int64_t rows, int NB, int bs, bool bwd, int *rpc, size_t *smem, int *grid) {
    if (NB < 5 || (NB - 1) % 4 != 0 || bs % 4 != 0 || bs < 2 * (NB - 1)) return false;
    const Noise2Layout L(NB, bs);
    const size_t fixed = (bwd ? (size_t)L.F * L.NBq : (size_t)NB * L.F) * sizeof(float);
    int r = 16;
    while (r > 1 && fixed + (size_t)r * L.stride * sizeof(float) > 75 * 1024) r >>= 1;
    *smem = fixed + (size_t)r * L.stride * sizeof(float);
    if (*smem > 200 * 1024) return false;
    *rpc = r;
    const int64_t ctas = ddsp_ceil_div(rows, r);
    *grid = (int)(ctas < DDSP_SM_COUNT * 3 ? ctas : DDSP_SM_COUNT * 3);
    return true;
}

// The synth pair (ddsp_b200_synth_pair_fwd / _bwd): exactly k persistent CTAs per SM, launched before the oscillator
// bank, whose CTAs take the rest of each SM.  The k CTAs keep at most half of the SM's shared memory, and every CTA
// gets at least one full sweep of RPC rows (fewer rows: the pair does not apply).  A row's arithmetic does not depend
// on RPC or on the grid, so the pair computes the same bits as the standalone launch.
constexpr int kPairCtasFwd = 1, kPairCtasBwd = 2;        // per SM; chosen with tools/synth_overlap.py

static bool noise2_pair_cfg(int64_t rows, int NB, int bs, bool bwd, int k, int *rpc, size_t *smem, int *grid) {
    if (k < 1 || k > 2 || NB < 5 || (NB - 1) % 4 != 0 || bs % 4 != 0 || bs < 2 * (NB - 1)) return false;
    const Noise2Layout L(NB, bs);
    const size_t fixed = (bwd ? (size_t)L.F * L.NBq : (size_t)NB * L.F) * sizeof(float);
    const size_t budget = (size_t)112 * 1024 / k;
    int r = 16;
    while (r > 1 && fixed + (size_t)r * L.stride * sizeof(float) > budget) r >>= 1;
    *smem = fixed + (size_t)r * L.stride * sizeof(float);
    if (*smem > budget || rows < (int64_t)k * DDSP_SM_COUNT * r) return false;
    *rpc = r;
    *grid = k * DDSP_SM_COUNT;
    return true;
}

extern "C" int64_t ddsp_b200_noise_design_size(int NB) {
    if (NB < 2) return 0;
    const int F = 2 * (NB - 1), NBq = (NB + 3) & ~3;
    return (int64_t)NB * F + (int64_t)F * NBq;
}

extern "C" int ddsp_b200_noise_design_table(float *table, int NB, void *stream) {
    DDSP_REQUIRE(table && NB >= 2);
    noise_design_kernel<<<64, 256, 0, (cudaStream_t)stream>>>(table, NB);
    return ddsp_launch_status();
}

extern "C" int ddsp_b200_filtered_noise_fwd(const float *mags, const float *noise, const float *add,
                                            const float *design, float *out, int64_t rows, int NB,
                                            int block_size, int apply_scale, float bias, void *stream) {
    DDSP_REQUIRE(mags && noise && out && rows >= 0);
    if (rows == 0) return DDSP_B200_OK;
    int rpc, grid;
    size_t smem;
    if (design && noise2_cfg(rows, NB, block_size, false, &rpc, &smem, &grid)) {
        if (smem > 48 * 1024)
            cudaFuncSetAttribute(filtered_noise2_fwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)smem);
        filtered_noise2_fwd_kernel<false><<<grid, kN2Threads, smem, (cudaStream_t)stream>>>(
            mags, noise, add, design, out, rows, NB, block_size, rpc, apply_scale, bias);
        return ddsp_launch_status();
    }
    int s = noise_launch_cfg(rows, NB, block_size, &rpc, &smem, &grid);
    if (s) return s;
    if (smem > 48 * 1024)
        cudaFuncSetAttribute(filtered_noise_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)smem);
    filtered_noise_fwd_kernel<<<grid, kNoiseThreads, smem, (cudaStream_t)stream>>>(
        mags, noise, add, out, rows, NB, block_size, rpc, apply_scale, bias);
    return ddsp_launch_status();
}

extern "C" int ddsp_b200_filtered_noise_bwd(const float *g_out, const float *noise,
                                            const float *mags_raw, const float *design, float *d_mags,
                                            int64_t rows, int NB, int block_size, int apply_scale,
                                            float bias, void *stream) {
    DDSP_REQUIRE(g_out && noise && d_mags && rows >= 0 && (!apply_scale || mags_raw));
    if (rows == 0) return DDSP_B200_OK;
    int rpc, grid;
    size_t smem;
    if (design && noise2_cfg(rows, NB, block_size, true, &rpc, &smem, &grid)) {
        if (smem > 48 * 1024)
            cudaFuncSetAttribute(filtered_noise2_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)smem);
        filtered_noise2_bwd_kernel<false><<<grid, kN2Threads, smem, (cudaStream_t)stream>>>(
            g_out, noise, mags_raw, design, d_mags, rows, NB, block_size, rpc, apply_scale, bias);
        return ddsp_launch_status();
    }
    int s = noise_launch_cfg(rows, NB, block_size, &rpc, &smem, &grid);
    if (s) return s;
    if (smem > 48 * 1024)
        cudaFuncSetAttribute(filtered_noise_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             (int)smem);
    filtered_noise_bwd_kernel<<<grid, kNoiseThreads, smem, (cudaStream_t)stream>>>(
        g_out, noise, mags_raw, d_mags, rows, NB, block_size, rpc, apply_scale, bias);
    return ddsp_launch_status();
}

extern "C" int ddsp_b200_synth_pair_supported(int B, int T, int H, int NB, int block_size, int ctas_per_sm) {
    if (B < 1 || B > 65535 || T < 1 || ctas_per_sm < 0 || ctas_per_sm > 2) return 0;
    if (!ddsp_pair_bank_supported(T, H, block_size)) return 0;
    const int64_t rows = (int64_t)B * T;
    int rpc, grid;
    size_t smem;
    return noise2_pair_cfg(rows, NB, block_size, false, ctas_per_sm ? ctas_per_sm : kPairCtasFwd, &rpc, &smem, &grid) &&
           noise2_pair_cfg(rows, NB, block_size, true, ctas_per_sm ? ctas_per_sm : kPairCtasBwd, &rpc, &smem, &grid);
}

// The noise kernel's shared-memory carveout is set to the largest, so that the SM configuration it is dispatched with
// also has room for the bank's CTAs.
template <typename K>
static void pair_noise_attributes(K kernel, size_t smem) {
    cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
}

// The noise's consumer (the reverb's first pass in the forward, the end of the step in the backward) comes after
// this call on `stream`.  The bank is the noise kernel's programmatic dependent, and that edge does not make "bank
// finished" imply "noise finished": `event` is recorded after the noise launch and waited for after the bank's, so
// that everything queued later also waits for the noise kernel to complete.
static int pair_join(int status, cudaEvent_t event, cudaStream_t st) {
    if (status) return status;
    const cudaError_t e = cudaStreamWaitEvent(st, event, 0);
    return e == cudaSuccess ? DDSP_B200_OK : (int)e;
}

extern "C" int ddsp_b200_synth_pair_fwd(const float *amp_raw, int64_t amp_stride, const float *dist_raw,
                                        int64_t dist_stride, const float *f0, const double *phase0, uint64_t *phi,
                                        uint64_t *delta, double *phase_end, float *amps, float *weights, float *audio,
                                        const float *mags_raw, const float *noise, const float *design,
                                        float *noise_out, int B, int T, int H, int NB, int block_size,
                                        double sample_rate, float bias, int ctas_per_sm, void *event, void *stream) {
    DDSP_REQUIRE(mags_raw && noise && design && noise_out && event && B > 0 && T > 0 && sample_rate > 0);
    if (!ddsp_b200_synth_pair_supported(B, T, H, NB, block_size, ctas_per_sm)) return DDSP_B200_EUNSUPPORTED;
    const int64_t rows = (int64_t)B * T;
    int rpc, grid;
    size_t smem;
    noise2_pair_cfg(rows, NB, block_size, false, ctas_per_sm ? ctas_per_sm : kPairCtasFwd, &rpc, &smem, &grid);
    cudaStream_t st = (cudaStream_t)stream;
    pair_noise_attributes(filtered_noise2_fwd_kernel<true>, smem);
    filtered_noise2_fwd_kernel<true><<<grid, kN2Threads, smem, st>>>(mags_raw, noise, nullptr, design, noise_out, rows,
                                                                     NB, block_size, rpc, 1, bias);
    int s = ddsp_launch_status();
    if (s) return s;
    const cudaError_t e = cudaEventRecord((cudaEvent_t)event, st);
    if (e != cudaSuccess) return (int)e;
    s = ddsp_pair_bank_fwd(amp_raw, amp_stride, dist_raw, dist_stride, f0, phase0, phi, delta, phase_end, amps, weights,
                           audio, B, T, H, block_size, sample_rate, st);
    return pair_join(s, (cudaEvent_t)event, st);
}

extern "C" int ddsp_b200_synth_pair_bwd(const float *g_audio, const float *g_noise, const float *amp_raw,
                                        int64_t amp_stride, const float *dist_raw, int64_t dist_stride, const float *f0,
                                        const uint64_t *phi, const uint64_t *delta, float *d_amp_raw,
                                        int64_t d_amp_stride, float *d_dist_raw, int64_t d_dist_stride,
                                        const float *mags_raw, const float *noise, const float *design, float *d_mags,
                                        int B, int T, int H, int NB, int block_size, float sample_rate, float bias,
                                        int ctas_per_sm, void *event, void *stream) {
    DDSP_REQUIRE(g_noise && mags_raw && noise && design && d_mags && event && B > 0 && T > 0);
    if (!ddsp_b200_synth_pair_supported(B, T, H, NB, block_size, ctas_per_sm)) return DDSP_B200_EUNSUPPORTED;
    const int64_t rows = (int64_t)B * T;
    int rpc, grid;
    size_t smem;
    noise2_pair_cfg(rows, NB, block_size, true, ctas_per_sm ? ctas_per_sm : kPairCtasBwd, &rpc, &smem, &grid);
    cudaStream_t st = (cudaStream_t)stream;
    pair_noise_attributes(filtered_noise2_bwd_kernel<true>, smem);
    filtered_noise2_bwd_kernel<true><<<grid, kN2Threads, smem, st>>>(g_noise, noise, mags_raw, design, d_mags, rows, NB,
                                                                     block_size, rpc, 1, bias);
    int s = ddsp_launch_status();
    if (s) return s;
    const cudaError_t e = cudaEventRecord((cudaEvent_t)event, st);
    if (e != cudaSuccess) return (int)e;
    s = ddsp_pair_bank_bwd(g_audio, amp_raw, amp_stride, dist_raw, dist_stride, f0, phi, delta, d_amp_raw, d_amp_stride,
                           d_dist_raw, d_dist_stride, B, T, H, block_size, sample_rate, st);
    return pair_join(s, (cudaEvent_t)event, st);
}
