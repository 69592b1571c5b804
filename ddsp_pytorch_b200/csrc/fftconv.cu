// K3: long FFT convolution (SURVEY 8a rows a9 generic, a10 reverb, and their backward).
//
// Reference path replaced:
//   ddsp/core.py:169-176          fft_convolve: pad to 2N, rfft x2, complex multiply, irfft, slice
//   ddsp/models/modules.py:21-35  Reverb.build_impulse / forward (IR padded to the signal, fft_convolve)
// i.e. three cuFFT launches of length 2N = 128000 / 384000 (non power of two) plus pads and slices.
//
// fft_convolve is a causal linear convolution truncated to the signal length (SURVEY 0.4), so any
// transform length n >= N + L - 1 gives the same result.  We use n = n1*n2 = 2^17 / 2^18 and the
// four-step decomposition with both factors' sub-FFTs in shared memory:
//   i = i1*n2 + i2  (time),  k = k1 + n1*k2  (frequency)
//   A: column FFTs over i1 (n1 points, CW adjacent columns per CTA) * W_n^(i2*k1)   -> work[k1][i2]
//   B: row FFT over i2 (n2 points) -> spectrum row k1; multiply by the filter spectrum (same
//      layout, never transposed); inverse row FFT; * W_n^(-i2*k1)                    (one kernel)
//   C: inverse column FFTs over k1, scale 1/n, write the first N samples
// Two real voices ride in one complex transform (re = voice 2p, im = voice 2p+1): a real filter acts
// on both parts independently, so no Hermitian untangling is ever needed.  For the gradient of the
// filter, sum_pairs G_p * conj(X_p) has the wanted cross-correlation in its real part.
#include <atomic>

#include "fft.cuh"
#include "regfft.cuh"

namespace {

using namespace regfft;

// Columns per CTA in the column passes: 16 adjacent columns = 64 B runs of the real inputs and
// 128 B runs of the complex work buffer; a column transform uses n1/16 threads, so a CTA has n1 threads.
constexpr int kCols = 16;
constexpr int kRowThreads = 256;      // row passes: 256/(n2/16) rows per CTA

__global__ void twiddle_kernel(float2 *__restrict__ tab, int n) {
    const int m = blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= n) return;
    double s, c;
    sincospi(2.0 * (double)m / (double)n, &s, &c);
    tab[m] = make_float2((float)c, (float)(-s));
}

// The inter-step twiddle W_n^(a*b) for one fixed a (a column index or a row index) and b = 0..len-1 is
// served from two small shared tables: W^(a*b) = hi[b >> 4] * lo[b & 15],  hi[j] = W^(16 a j), lo[j] = W^(a j)
// (one extra rounding instead of a scattered read of the n-entry table per element).
struct StepTwiddle {
    const float2 *hi, *lo;
    __device__ __forceinline__ float2 at(int b, bool conj) const {
        const float2 h = hi[b >> 4], l = lo[b & 15];
        float2 w = make_float2(h.x * l.x - h.y * l.y, h.x * l.y + h.y * l.x);
        if (conj) w.y = -w.y;
        return w;
    }
};

// fill hi[0..len/16), lo[0..16) for fixed a; a*b < n for all b < len (a < other factor)
__device__ __forceinline__ void fill_step_twiddle(float2 *hi, float2 *lo, const float2 *__restrict__ twn,
                                                  int a, int len, int t, int nthr) {
    for (int j = t; j < len / 16; j += nthr) hi[j] = __ldg(twn + (size_t)a * 16 * j);
    for (int j = t; j < 16; j += nthr) lo[j] = __ldg(twn + (size_t)a * j);
}

template <int LG, bool INV>
__device__ __forceinline__ void mid_stages(float2 (&x)[16], float2 *buf, int t, const float2 *__restrict__ stw,
                                           bool act) {
    // stages 1 .. last-1 (i.e. stage 1 of a 3-stage transform), each: sync, load, sync, compute+store
    if (Plan<LG>::STAGES == 3) {
        __syncthreads();
        if (act) stage_load<LG, 1>(x, buf, t);
        __syncthreads();
        if (act) stage_compute_store<LG, 1, INV>(x, buf, t, stw);
    }
    __syncthreads();
    if (act) stage_load<LG, Plan<LG>::STAGES - 1>(x, buf, t);
    __syncthreads();
}

// ---- A: real rows -> column FFT over i1 -> * W_n^(i2 k1) -> work[slot][k1][i2] -------------------
template <int LG1>
__global__ void __launch_bounds__((1 << LG1))
cols_fwd_kernel(const float *__restrict__ x, const float *__restrict__ x2, int64_t rows, int64_t len, int pair,
                float2 *__restrict__ work,
                const float2 *__restrict__ twn, const float2 *__restrict__ stw, int n2) {
    using P = Plan<LG1>;
    constexpr int n1 = P::N, T = P::T, PITCH = P::PITCH + 1;     // odd pitch: the 16 columns hit 16 banks
    extern __shared__ __align__(16) float smem[];
    float2 *bufs = reinterpret_cast<float2 *>(smem);              // [kCols][PITCH]
    float2 *thi = bufs + kCols * PITCH;                           // [kCols][n1/16]
    float2 *tlo = thi + kCols * (n1 / 16);                        // [kCols][16]
    const int tid = threadIdx.x, c = tid & (kCols - 1), t = tid >> 4;
    const int64_t p = blockIdx.y;
    const int col = blockIdx.x * kCols + c;
    const int64_t rre = pair ? 2 * p : p, rim = pair ? 2 * p + 1 : rows;
    const float *xr = x + rre * len;
    const float *xi = rim < rows ? x + rim * len : nullptr;
    fill_step_twiddle(thi + c * (n1 / 16), tlo + c * 16, twn, col, n1, t, T);
    float2 v[16];
#pragma unroll
    for (int r = 0; r < 16; ++r) {
        const int64_t pos = (int64_t)(t + r * T) * n2 + col;
        v[r] = make_float2(0.f, 0.f);
        if (pos < len) {
            v[r].x = __ldg(xr + pos);
            if (xi) v[r].y = __ldg(xi + pos);
            if (x2) {                                   // transform of x + x2 (decoder.py:121: harmonic + noise)
                v[r].x += __ldg(x2 + rre * len + pos);
                if (xi) v[r].y += __ldg(x2 + rim * len + pos);
            }
        }
    }
    float2 *buf = bufs + c * PITCH;
    stage_compute_store<LG1, 0, false>(v, buf, t, stw);
    mid_stages<LG1, false>(v, buf, t, stw, true);
    const StepTwiddle st{thi + c * (n1 / 16), tlo + c * 16};
    float2 *w = work + (size_t)p * n1 * n2 + col;
    stage_compute_sink<LG1, P::STAGES - 1, false>(v, t, stw, [&](int k1, float2 val) {
        w[(size_t)k1 * n2] = c_mul(val, st.at(k1, false));
    });
}

// ---- C: work[slot][k1][i2] -> inverse column FFT over k1 -> real rows, scaled 1/n ------------------
template <int LG1>
__global__ void __launch_bounds__((1 << LG1))
cols_inv_kernel(const float2 *__restrict__ work, float *__restrict__ out, int64_t rows, int64_t len, int pair,
                const float2 *__restrict__ stw, int n2) {
    using P = Plan<LG1>;
    constexpr int n1 = P::N, T = P::T, PITCH = P::PITCH + 1;
    extern __shared__ __align__(16) float smem[];
    float2 *bufs = reinterpret_cast<float2 *>(smem);
    const int tid = threadIdx.x, c = tid & (kCols - 1), t = tid >> 4;
    const int64_t p = blockIdx.y;
    const int col = blockIdx.x * kCols + c;
    const float2 *w = work + (size_t)p * n1 * n2 + col;
    float2 v[16];
#pragma unroll
    for (int r = 0; r < 16; ++r) v[r] = w[(size_t)(t + r * T) * n2];
    float2 *buf = bufs + c * PITCH;
    stage_compute_store<LG1, 0, true>(v, buf, t, stw);
    mid_stages<LG1, true>(v, buf, t, stw, true);
    const float sc = 1.0f / ((float)n1 * (float)n2);
    const int64_t rre = pair ? 2 * p : p, rim = pair ? 2 * p + 1 : rows;
    float *yr = out + rre * len;
    float *yi = rim < rows ? out + rim * len : nullptr;
    stage_compute_sink<LG1, P::STAGES - 1, true>(v, t, stw, [&](int i1, float2 val) {
        const int64_t pos = (int64_t)i1 * n2 + col;
        if (pos < len) {
            yr[pos] = val.x * sc;
            if (yi) yi[pos] = val.y * sc;
        }
    });
}

// ---- B: row passes.  A CTA works on ROWS = 256/(n2/16) consecutive rows k1 of one slot. ----------------
template <int LG2> struct RowCfg {
    using P = Plan<LG2>;
    static constexpr int ROWS = kRowThreads / P::T;
};

// MODE 0 spectrum: row FFT, write.   MODE 1 filter: row FFT, * H (or conj H), inverse row FFT,
// * W_n^(-i2 k1), write in place.
// TWIN: the inter-step twiddle W_n^(i2 k1) of the FORWARD direction is applied here, while the row is loaded (the
// direct column pass of the 5-smooth lengths writes plain DFT outputs); otherwise the column pass already applied it.
template <int LG2, int MODE, bool TWIN>
__global__ void __launch_bounds__(kRowThreads)
rows_kernel(const float2 *src_work, float2 *dst_work, const float2 *__restrict__ hspec, int64_t h_slot_stride,
            int conj_h, const float2 *__restrict__ twn, const float2 *__restrict__ stw, int n1) {
    using P = Plan<LG2>;
    constexpr int n2 = P::N, T = P::T, PITCH = P::PITCH, ROWS = RowCfg<LG2>::ROWS;
    extern __shared__ __align__(16) float smem[];
    float2 *bufs = reinterpret_cast<float2 *>(smem);              // [ROWS][PITCH]
    float2 *thi = bufs + ROWS * PITCH;                            // [ROWS][n2/16]
    float2 *tlo = thi + ROWS * (n2 / 16);                         // [ROWS][16]
    const int tid = threadIdx.x, g = tid / T, t = tid - g * T;
    const int k1 = blockIdx.x * ROWS + g;
    const int64_t p = blockIdx.y;
    const float2 *row_in = src_work + ((size_t)p * n1 + k1) * n2;
    float2 *row = dst_work + ((size_t)p * n1 + k1) * n2;       // may alias row_in (in-place): read fully first
    float2 *buf = bufs + g * PITCH;
    if (MODE == 1 || TWIN) fill_step_twiddle(thi + g * (n2 / 16), tlo + g * 16, twn, k1, n2, t, T);
    float2 v[16];
#pragma unroll
    for (int r = 0; r < 16; ++r) v[r] = row_in[t + r * T];
    if (TWIN) {
        __syncthreads();                                   // the row's twiddle tables are filled
        const StepTwiddle sti{thi + g * (n2 / 16), tlo + g * 16};
#pragma unroll
        for (int r = 0; r < 16; ++r) v[r] = c_mul(v[r], sti.at(t + r * T, false));
    }
    stage_compute_store<LG2, 0, false>(v, buf, t, stw);
    mid_stages<LG2, false>(v, buf, t, stw, true);
    if (MODE == 0) {
        stage_compute_sink<LG2, P::STAGES - 1, false>(v, t, stw, [&](int k2, float2 val) { row[k2] = val; });
        return;
    }
    const float2 *h = hspec + (size_t)p * h_slot_stride + (size_t)k1 * n2;
    stage_compute_sink<LG2, P::STAGES - 1, false>(v, t, stw, [&](int k2, float2 val) {
        float2 hv = __ldg(h + k2);
        if (conj_h) hv.y = -hv.y;
        buf[pad16(k2)] = c_mul(val, hv);
    });
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 16; ++r) v[r] = buf[pad16(t + r * T)];
    __syncthreads();
    stage_compute_store<LG2, 0, true>(v, buf, t, stw);
    mid_stages<LG2, true>(v, buf, t, stw, true);
    const StepTwiddle st{thi + g * (n2 / 16), tlo + g * 16};
    stage_compute_sink<LG2, P::STAGES - 1, true>(v, t, stw, [&](int i2, float2 val) {
        row[i2] = c_mul(val, st.at(i2, true));
    });
}

// Correlation, phase 1: partial[split][k1][k2] = sum over the slots of this split of
// FFT_row(G)[k2] * conj(FFT_row(X)[k2]).  The accumulator lives in registers (same positions as the
// last stage's outputs).
// FINISH (one row per CTA, TWIN): the last of a row's `nsplit` CTAs to arrive (a counter per row, which it resets)
// also does phase 2 for that row -- sum of the partial spectra in split order (so the result does not depend on which
// CTA came last), inverse row transform, inter-step twiddle -- instead of a second, 20-CTA launch on the critical path
// of the reverb's backward.
template <int LG2, bool TWIN, bool FINISH = false>
__global__ void __launch_bounds__(kRowThreads)
rows_corr_kernel(const float2 *__restrict__ work_g, const float2 *__restrict__ work_x, int64_t slots,
                 int nsplit, float2 *partial, const float2 *__restrict__ twn,
                 const float2 *__restrict__ stw, int n1, float2 *__restrict__ final_out = nullptr,
                 int *__restrict__ counters = nullptr) {
    using P = Plan<LG2>;
    constexpr int n2 = P::N, T = P::T, PITCH = P::PITCH, ROWS = RowCfg<LG2>::ROWS;
    constexpr int R = Stage<LG2, P::STAGES - 1>::R, M = 16 / R;
    extern __shared__ __align__(16) float smem[];
    float2 *bufs = reinterpret_cast<float2 *>(smem);              // [ROWS][PITCH]
    const int tid = threadIdx.x, g = tid / T, t = tid - g * T;
    const int k1 = blockIdx.x * ROWS + g;
    const int split = blockIdx.y;
    float2 *buf = bufs + g * PITCH;
    float2 *thi = bufs + ROWS * PITCH;                            // [ROWS][n2/16]   (TWIN only)
    float2 *tlo = thi + ROWS * (n2 / 16);                         // [ROWS][16]
    float2 acc[16];
#pragma unroll
    for (int r = 0; r < 16; ++r) acc[r] = make_float2(0.f, 0.f);
    float2 v[16], win[16];
    if (TWIN) {
        fill_step_twiddle(thi + g * (n2 / 16), tlo + g * 16, twn, k1, n2, t, T);
        __syncthreads();
        const StepTwiddle sti{thi + g * (n2 / 16), tlo + g * 16};
#pragma unroll
        for (int r = 0; r < 16; ++r) win[r] = sti.at(t + r * T, false);
    }
    for (int64_t p = split; p < slots; p += nsplit) {
        const float2 *rg = work_g + ((size_t)p * n1 + k1) * n2;
        const float2 *rx = work_x + ((size_t)p * n1 + k1) * n2;
        // spectrum of the G row into shared memory
#pragma unroll
        for (int r = 0; r < 16; ++r) v[r] = TWIN ? c_mul(rg[t + r * T], win[r]) : rg[t + r * T];
        __syncthreads();                                  // previous slot's spectrum fully consumed
        stage_compute_store<LG2, 0, false>(v, buf, t, stw);
        mid_stages<LG2, false>(v, buf, t, stw, true);
        stage_compute_store<LG2, P::STAGES - 1, false>(v, buf, t, stw);
        __syncthreads();
        // this thread's part of the G spectrum (the positions its last stage produces), to registers
        float2 gs[16];
#pragma unroll
        for (int m = 0; m < M; ++m)
#pragma unroll
            for (int r = 0; r < R; ++r)
                gs[m * R + r] = buf[pad16(stage_out_index<LG2, P::STAGES - 1>(t, m, r))];
        // spectrum of the X row, consumed straight from the last stage's registers
#pragma unroll
        for (int r = 0; r < 16; ++r) v[r] = TWIN ? c_mul(rx[t + r * T], win[r]) : rx[t + r * T];
        __syncthreads();
        stage_compute_store<LG2, 0, false>(v, buf, t, stw);
        mid_stages<LG2, false>(v, buf, t, stw, true);
        stage_compute_regs<LG2, P::STAGES - 1, false>(v, t, stw);
#pragma unroll
        for (int i = 0; i < 16; ++i) {                       // g * conj(x)
            acc[i].x += gs[i].x * v[i].x + gs[i].y * v[i].y;
            acc[i].y += gs[i].y * v[i].x - gs[i].x * v[i].y;
        }
    }
    float2 *out = partial + ((size_t)split * n1 + k1) * n2;
#pragma unroll
    for (int m = 0; m < M; ++m)
#pragma unroll
        for (int r = 0; r < R; ++r) out[stage_out_index<LG2, P::STAGES - 1>(t, m, r)] = acc[m * R + r];
    if (FINISH) {
        static_assert(!FINISH || (ROWS == 1 && TWIN), "fused finish: one row per CTA, twiddles in shared memory");
        __shared__ int is_last;
        __threadfence();                                   // this CTA's partial spectrum is visible device-wide
        __syncthreads();
        if (tid == 0) {
            const int old = atomicAdd(&counters[k1], 1);
            is_last = old == nsplit - 1;
            if (is_last) counters[k1] = 0;                 // ready for the next launch on this workspace
        }
        __syncthreads();
        if (!is_last) return;
        __threadfence();
#pragma unroll
        for (int r = 0; r < 16; ++r) v[r] = make_float2(0.f, 0.f);
        for (int sp = 0; sp < nsplit; ++sp) {
            const float2 *src = partial + ((size_t)sp * n1 + k1) * n2;
#pragma unroll
            for (int r = 0; r < 16; ++r) v[r] = c_add(v[r], __ldcg(src + t + r * T));
        }
        stage_compute_store<LG2, 0, true>(v, buf, t, stw);
        mid_stages<LG2, true>(v, buf, t, stw, true);
        const StepTwiddle st{thi + g * (n2 / 16), tlo + g * 16};
        float2 *row = final_out + (size_t)k1 * n2;
        stage_compute_sink<LG2, P::STAGES - 1, true>(v, t, stw, [&](int i2, float2 val) {
            row[i2] = c_mul(val, st.at(i2, true));
        });
    }
}

__global__ void zero_ints_kernel(int *p, int n) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) p[i] = 0;
}

// Correlation, phase 2: out[o][k1] = IFFT_row(sum of `nsum` partial spectra) * W_n^(-i2 k1)
template <int LG2>
__global__ void __launch_bounds__(kRowThreads)
rows_corr_finish_kernel(const float2 *__restrict__ partial, int nsum, float2 *__restrict__ out,
                        const float2 *__restrict__ twn, const float2 *__restrict__ stw, int n1) {
    using P = Plan<LG2>;
    constexpr int n2 = P::N, T = P::T, PITCH = P::PITCH, ROWS = RowCfg<LG2>::ROWS;
    extern __shared__ __align__(16) float smem[];
    float2 *bufs = reinterpret_cast<float2 *>(smem);
    float2 *thi = bufs + ROWS * PITCH;
    float2 *tlo = thi + ROWS * (n2 / 16);
    const int tid = threadIdx.x, g = tid / T, t = tid - g * T;
    const int k1 = blockIdx.x * ROWS + g;
    const int64_t o = blockIdx.y;
    float2 *buf = bufs + g * PITCH;
    fill_step_twiddle(thi + g * (n2 / 16), tlo + g * 16, twn, k1, n2, t, T);
    float2 v[16];
#pragma unroll
    for (int r = 0; r < 16; ++r) v[r] = make_float2(0.f, 0.f);
    for (int s = 0; s < nsum; ++s) {
        const float2 *src = partial + (((size_t)o * nsum + s) * n1 + k1) * n2;
#pragma unroll
        for (int r = 0; r < 16; ++r) v[r] = c_add(v[r], src[t + r * T]);
    }
    stage_compute_store<LG2, 0, true>(v, buf, t, stw);
    mid_stages<LG2, true>(v, buf, t, stw, true);
    const StepTwiddle st{thi + g * (n2 / 16), tlo + g * 16};
    float2 *row = out + ((size_t)o * n1 + k1) * n2;
    stage_compute_sink<LG2, P::STAGES - 1, true>(v, t, stw, [&](int i2, float2 val) {
        row[i2] = c_mul(val, st.at(i2, true));
    });
}


// ---- Column passes of the 5-smooth transform lengths n = N1 * n2, N1 = 20 or 24 (n2 = 4096) -------------------
// fft_convolve only needs n >= N + L - 1.  The power of two above 79 999 (config 2: N = 64000, L = 16000) is 131 072;
// 20 * 4096 = 81 920 does the same job with 0.625x the data in every pass.  The N1-point column DFT is small enough to
// be done directly in registers, one thread per column: fully coalesced rows in, rows out, no shared memory, no
// barriers; the inter-step twiddle moves to the row pass (TWIN above).  Only the first ceil(len / n2) input rows of the
// forward pass are non-zero and only that many output rows of the inverse pass are kept.
template <int N1> struct DirectTw;
template <> struct DirectTw<20> {
    static __host__ __device__ constexpr float c(int j) { constexpr float t[20] = {1.0f, 0.951056516f, 0.809016994f, 0.587785252f, 0.309016994f, 6.123234e-17f, -0.309016994f, -0.587785252f, -0.809016994f, -0.951056516f, -1.0f, -0.951056516f, -0.809016994f, -0.587785252f, -0.309016994f, -1.8369702e-16f, 0.309016994f, 0.587785252f, 0.809016994f, 0.951056516f}; return t[j]; }
    static __host__ __device__ constexpr float s(int j) { constexpr float t[20] = {0.0f, 0.309016994f, 0.587785252f, 0.809016994f, 0.951056516f, 1.0f, 0.951056516f, 0.809016994f, 0.587785252f, 0.309016994f, 1.2246468e-16f, -0.309016994f, -0.587785252f, -0.809016994f, -0.951056516f, -1.0f, -0.951056516f, -0.809016994f, -0.587785252f, -0.309016994f}; return t[j]; }
};
template <> struct DirectTw<24> {
    static __host__ __device__ constexpr float c(int j) { constexpr float t[24] = {1.0f, 0.965925826f, 0.866025404f, 0.707106781f, 0.5f, 0.258819045f, 6.123234e-17f, -0.258819045f, -0.5f, -0.707106781f, -0.866025404f, -0.965925826f, -1.0f, -0.965925826f, -0.866025404f, -0.707106781f, -0.5f, -0.258819045f, -1.8369702e-16f, 0.258819045f, 0.5f, 0.707106781f, 0.866025404f, 0.965925826f}; return t[j]; }
    static __host__ __device__ constexpr float s(int j) { constexpr float t[24] = {0.0f, 0.258819045f, 0.5f, 0.707106781f, 0.866025404f, 0.965925826f, 1.0f, 0.965925826f, 0.866025404f, 0.707106781f, 0.5f, 0.258819045f, 1.2246468e-16f, -0.258819045f, -0.5f, -0.707106781f, -0.866025404f, -0.965925826f, -1.0f, -0.965925826f, -0.866025404f, -0.707106781f, -0.5f, -0.258819045f}; return t[j]; }
};

constexpr int kDirectThreads = 128;

template <int N1>
__global__ void __launch_bounds__(2 * kDirectThreads)
dcols_fwd_kernel(const float *__restrict__ x, const float *__restrict__ x2, int64_t rows, int64_t len, int pair,
                 float2 *__restrict__ work, int n2) {
    const int i2 = blockIdx.x * kDirectThreads + threadIdx.x;
    const int half = threadIdx.y;                          // outputs k1 = half, half + 2, ...
    const int64_t p = blockIdx.y;
    const int64_t rre = pair ? 2 * p : p, rim = pair ? 2 * p + 1 : rows;
    const float *xr = x + rre * len;
    const float *xi = rim < rows ? x + rim * len : nullptr;
    float2 z[N1];
#pragma unroll
    for (int i1 = 0; i1 < N1; ++i1) {
        const int64_t pos = (int64_t)i1 * n2 + i2;
        z[i1] = make_float2(0.f, 0.f);
        if (pos < len) {
            z[i1].x = __ldg(xr + pos);
            if (xi) z[i1].y = __ldg(xi + pos);
            if (x2) {
                z[i1].x += __ldg(x2 + rre * len + pos);
                if (xi) z[i1].y += __ldg(x2 + rim * len + pos);
            }
        }
    }
    float2 *w = work + (size_t)p * N1 * n2 + i2;
#pragma unroll
    for (int k1 = 0; k1 < N1; ++k1) {
        if ((k1 & 1) != half) continue;                    // uniform per warp (threadIdx.y)
        float re = z[0].x, im = z[0].y;
#pragma unroll
        for (int i1 = 1; i1 < N1; ++i1) {
            const float c = DirectTw<N1>::c((i1 * k1) % N1), sn = DirectTw<N1>::s((i1 * k1) % N1);   // W = c - i sn
            re = fmaf(z[i1].x, c, re);  re = fmaf(z[i1].y, sn, re);
            im = fmaf(z[i1].y, c, im);  im = fmaf(-z[i1].x, sn, im);
        }
        w[(size_t)k1 * n2] = make_float2(re, im);
    }
}

template <int N1>
__global__ void __launch_bounds__(2 * kDirectThreads)
dcols_inv_kernel(const float2 *__restrict__ work, float *__restrict__ out, int64_t rows, int64_t len, int pair,
                 int n2) {
    const int i2 = blockIdx.x * kDirectThreads + threadIdx.x;
    const int half = threadIdx.y;                          // output rows i1 = half, half + 2, ...
    const int64_t p = blockIdx.y;
    const float2 *w = work + (size_t)p * N1 * n2 + i2;
    float2 v[N1];
#pragma unroll
    for (int k1 = 0; k1 < N1; ++k1) v[k1] = w[(size_t)k1 * n2];
    const float sc = 1.0f / ((float)N1 * (float)n2);
    const int64_t rre = pair ? 2 * p : p, rim = pair ? 2 * p + 1 : rows;
    float *yr = out + rre * len;
    float *yi = rim < rows ? out + rim * len : nullptr;
#pragma unroll
    for (int i1 = 0; i1 < N1; ++i1) {
        const int64_t pos = (int64_t)i1 * n2 + i2;
        if ((i1 & 1) == half && pos < len) {               // uniform per warp except in the last row
            float re = v[0].x, im = v[0].y;
#pragma unroll
            for (int k1 = 1; k1 < N1; ++k1) {
                const float c = DirectTw<N1>::c((i1 * k1) % N1), sn = DirectTw<N1>::s((i1 * k1) % N1);   // W = c + i sn
                re = fmaf(v[k1].x, c, re);  re = fmaf(-v[k1].y, sn, re);
                im = fmaf(v[k1].y, c, im);  im = fmaf(v[k1].x, sn, im);
            }
            yr[pos] = re * sc;
            if (yi) yi[pos] = im * sc;
        }
    }
}

// ---- Reverb impulse (modules.py:21-26) -------------------------------------------------------
__device__ __forceinline__ float softplusf(float z) { return fmaxf(z, 0.f) + log1pf(expf(-fabsf(z))); }
__device__ __forceinline__ float sigmoidf_(float z) { return 1.f / (1.f + expf(-z)); }

__global__ void reverb_impulse_fwd_kernel(const float *__restrict__ noise, const float *__restrict__ decay,
                                          const float *__restrict__ wet, const float *__restrict__ t,
                                          float *__restrict__ impulse, int L) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l >= L) return;
    const float sp = softplusf(-decay[0]);
    const float sg = sigmoidf_(wet[0]);
    impulse[l] = l == 0 ? 1.f : noise[l] * expf(-sp * t[l] * 500.f) * sg;
}

// Two launches: (1) kImpBlocks CTAs write d_noise and one (d_wet, d_decay) partial pair each in double, (2) one warp
// adds the partials in index order.  Deterministic; the single-CTA version took 14 us for 16000 taps and sat at the end of
// the kernel-gradient chain of the reverb.
constexpr int kImpBlocks = 64;

__global__ void __launch_bounds__(256)
reverb_impulse_bwd_kernel(const float *__restrict__ d_imp, int Lvalid, const float *__restrict__ noise,
                          const float *__restrict__ decay, const float *__restrict__ wet,
                          const float *__restrict__ t, float *__restrict__ d_noise, double *__restrict__ partial,
                          int L) {
    __shared__ double r0[256], r1[256];
    const int tid = threadIdx.x;
    const float dec = decay[0];
    const float sp = softplusf(-dec);
    const float sg = sigmoidf_(wet[0]);
    const float sneg = sigmoidf_(-dec);                 // -d softplus(-decay)/d decay
    double aw = 0.0, ad = 0.0;
    for (int l = blockIdx.x * 256 + tid; l < L; l += kImpBlocks * 256) {
        float dn = 0.f;
        if (l >= 1 && l < Lvalid) {
            const float g = d_imp[l];
            const float env = expf(-sp * t[l] * 500.f);
            dn = g * env * sg;
            const float base = g * noise[l] * env * sg;   // g * impulse[l]
            aw += (double)(base * (1.f - sg));
            ad += (double)(base * t[l] * 500.f * sneg);
        }
        d_noise[l] = dn;
    }
    r0[tid] = aw;
    r1[tid] = ad;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if (tid < o) { r0[tid] += r0[tid + o]; r1[tid] += r1[tid + o]; }
        __syncthreads();
    }
    if (tid == 0) { partial[2 * blockIdx.x] = r0[0]; partial[2 * blockIdx.x + 1] = r1[0]; }
}

__global__ void reverb_impulse_bwd_finish_kernel(const double *__restrict__ partial, float *__restrict__ d_decay,
                                                 float *__restrict__ d_wet) {
    if (threadIdx.x == 0) {
        double aw = 0.0, ad = 0.0;
        for (int i = 0; i < kImpBlocks; ++i) { aw += partial[2 * i]; ad += partial[2 * i + 1]; }
        d_wet[0] = (float)aw;
        d_decay[0] = (float)ad;
    }
}

template <typename K>
int set_smem(K kernel, size_t bytes) {
    if (bytes > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (e != cudaSuccess) return (int)e;
    }
    return 0;
}

bool pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }
// n1 (column transform, one CTA of n1 threads per 16 columns): 64..512; n2 (row transform): 64..4096
bool direct_n1(int n1) { return n1 == 20 || n1 == 24; }          // column DFT done directly in registers
bool plan_ok(int n1, int n2) {
    if (direct_n1(n1)) return n2 == 4096;
    return pow2(n1) && pow2(n2) && n1 >= 64 && n1 <= 512 && n2 >= 64 && n2 <= 4096;
}

template <int LG> size_t col_smem() {
    return (size_t)kCols * (Plan<LG>::PITCH + 1 + Plan<LG>::N / 16 + 16) * sizeof(float2);
}
template <int LG> size_t row_smem() {
    return (size_t)RowCfg<LG>::ROWS * (Plan<LG>::PITCH + Plan<LG>::N / 16 + 16) * sizeof(float2);
}

// compile-time dispatch on log2 of a transform size (columns 64..512, rows 64..4096)
#define DDSP_LG_SWITCH_COLS(lg, CALL) \
    switch (lg) {                     \
        case 6: CALL(6); break;       \
        case 7: CALL(7); break;       \
        case 8: CALL(8); break;       \
        case 9: CALL(9); break;       \
        default: break;               \
    }
#define DDSP_LG_SWITCH_ROWS(lg, CALL) \
    switch (lg) {                     \
        case 6: CALL(6); break;       \
        case 7: CALL(7); break;       \
        case 8: CALL(8); break;       \
        case 9: CALL(9); break;       \
        case 10: CALL(10); break;     \
        case 11: CALL(11); break;     \
        case 12: CALL(12); break;     \
        default: break;               \
    }

}  // namespace

extern "C" int ddsp_b200_twiddle_table(float *table, int n, void *stream) {
    DDSP_REQUIRE(table && n > 0);
    twiddle_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<float2 *>(table), n);
    return ddsp_launch_status();
}

extern "C" int ddsp_b200_conv_plan(int64_t min_len, int *n1, int *n2) {
    DDSP_REQUIRE(n1 && n2 && min_len >= 1);
    // 5-smooth lengths between 2^16 and 2^17: 20 * 4096 and 24 * 4096 (0.625x / 0.75x the work of 2^17)
    if (min_len > 65536 && min_len <= 24 * 4096) {
        *n1 = min_len <= 20 * 4096 ? 20 : 24;
        *n2 = 4096;
        return DDSP_B200_OK;
    }
    int lg = ddsp_ilog2(min_len);
    if (lg < 12) lg = 12;
    // 128 columns x long rows measured best at 2^17 and 2^18 (swept with a since-removed split override: 2^18 bulk
    // render 10.71 ms with 512 x 512, 10.24 ms with 128 x 2048); rows are capped at 4096 points
    int lg1 = lg / 2;
    if (lg1 > 7) lg1 = 7;
    if (lg - lg1 > 12) lg1 = lg - 12;
    if (lg1 > 9) lg1 = 9;
    const int lg2 = lg - lg1;
    if (lg2 > 12) return DDSP_B200_EUNSUPPORTED;
    *n1 = 1 << lg1;
    *n2 = 1 << lg2;
    return plan_ok(*n1, *n2) ? DDSP_B200_OK : DDSP_B200_EUNSUPPORTED;
}

extern "C" int ddsp_b200_fft4_cols_fwd_sum(const float *x, const float *x2, int64_t rows, int64_t len, int pair,
                                           float *work, const float *twiddle, const float *stage1, int n1, int n2,
                                           void *stream) {
    DDSP_REQUIRE(x && work && rows > 0 && len > 0 && plan_ok(n1, n2));
    DDSP_REQUIRE(len <= (int64_t)n1 * n2);
    const int64_t slots = pair ? (rows + 1) / 2 : rows;
    DDSP_REQUIRE(slots <= 65535);
    cudaStream_t st = (cudaStream_t)stream;
    if (direct_n1(n1)) {                                 // plain column DFT in registers; twiddle applied by the row pass
        const dim3 dgrid(n2 / kDirectThreads, (unsigned)slots);
        if (n1 == 20) dcols_fwd_kernel<20><<<dgrid, dim3(kDirectThreads, 2), 0, st>>>(x, x2, rows, len, pair, reinterpret_cast<float2 *>(work), n2);
        else dcols_fwd_kernel<24><<<dgrid, dim3(kDirectThreads, 2), 0, st>>>(x, x2, rows, len, pair, reinterpret_cast<float2 *>(work), n2);
        return ddsp_launch_status();
    }
    DDSP_REQUIRE(twiddle && stage1);
    int s = DDSP_B200_EUNSUPPORTED;
    const dim3 grid(n2 / kCols, (unsigned)slots);
#define CALL(LG)                                                                                        \
    if (!(s = set_smem(cols_fwd_kernel<LG>, col_smem<LG>())))                                           \
        cols_fwd_kernel<LG><<<grid, 1 << LG, col_smem<LG>(), st>>>(                                      \
            x, x2, rows, len, pair, reinterpret_cast<float2 *>(work), reinterpret_cast<const float2 *>(twiddle), \
            reinterpret_cast<const float2 *>(stage1), n2)
    DDSP_LG_SWITCH_COLS(ddsp_ilog2(n1), CALL)
#undef CALL
    return s ? s : ddsp_launch_status();
}

extern "C" int ddsp_b200_fft4_cols_fwd(const float *x, int64_t rows, int64_t len, int pair, float *work,
                                       const float *twiddle, const float *stage1, int n1, int n2,
                                       void *stream) {
    return ddsp_b200_fft4_cols_fwd_sum(x, nullptr, rows, len, pair, work, twiddle, stage1, n1, n2, stream);
}

extern "C" int ddsp_b200_fft4_cols_inv(const float *work, float *out, int64_t rows, int64_t len, int pair,
                                       const float *stage1, int n1, int n2, void *stream) {
    DDSP_REQUIRE(work && out && rows > 0 && len > 0 && plan_ok(n1, n2));
    DDSP_REQUIRE(len <= (int64_t)n1 * n2);
    const int64_t slots = pair ? (rows + 1) / 2 : rows;
    DDSP_REQUIRE(slots <= 65535);
    cudaStream_t st = (cudaStream_t)stream;
    if (direct_n1(n1)) {
        const dim3 dgrid(n2 / kDirectThreads, (unsigned)slots);
        if (n1 == 20) dcols_inv_kernel<20><<<dgrid, dim3(kDirectThreads, 2), 0, st>>>(reinterpret_cast<const float2 *>(work), out, rows, len, pair, n2);
        else dcols_inv_kernel<24><<<dgrid, dim3(kDirectThreads, 2), 0, st>>>(reinterpret_cast<const float2 *>(work), out, rows, len, pair, n2);
        return ddsp_launch_status();
    }
    DDSP_REQUIRE(stage1);
    int s = DDSP_B200_EUNSUPPORTED;
    const dim3 grid(n2 / kCols, (unsigned)slots);
#define CALL(LG)                                                                                        \
    if (!(s = set_smem(cols_inv_kernel<LG>, col_smem<LG>())))                                           \
        cols_inv_kernel<LG><<<grid, 1 << LG, col_smem<LG>(), st>>>(                                      \
            reinterpret_cast<const float2 *>(work), out, rows, len, pair,                               \
            reinterpret_cast<const float2 *>(stage1), n2)
    DDSP_LG_SWITCH_COLS(ddsp_ilog2(n1), CALL)
#undef CALL
    return s ? s : ddsp_launch_status();
}

extern "C" int ddsp_b200_fft4_rows_spectrum(float *work, int64_t slots, const float *twiddle,
                                            const float *stage2, int n1, int n2, void *stream) {
    DDSP_REQUIRE(work && twiddle && stage2 && slots > 0 && slots <= 65535 && plan_ok(n1, n2));
    int s = DDSP_B200_EUNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if (direct_n1(n1)) {                                 // n2 = 4096, forward twiddle applied on load
        if ((s = set_smem(rows_kernel<12, 0, true>, row_smem<12>()))) return s;
        rows_kernel<12, 0, true><<<dim3(n1, (unsigned)slots), kRowThreads, row_smem<12>(), st>>>(
            reinterpret_cast<const float2 *>(work), reinterpret_cast<float2 *>(work), nullptr, 0, 0,
            reinterpret_cast<const float2 *>(twiddle), reinterpret_cast<const float2 *>(stage2), n1);
        return ddsp_launch_status();
    }
#define CALL(LG)                                                                                        \
    if (!(s = set_smem(rows_kernel<LG, 0, false>, row_smem<LG>())))                                     \
        rows_kernel<LG, 0, false><<<dim3(n1 / RowCfg<LG>::ROWS, (unsigned)slots), kRowThreads, row_smem<LG>(), st>>>( \
            reinterpret_cast<const float2 *>(work), reinterpret_cast<float2 *>(work), nullptr, 0, 0,     \
            reinterpret_cast<const float2 *>(twiddle), reinterpret_cast<const float2 *>(stage2), n1)
    DDSP_LG_SWITCH_ROWS(ddsp_ilog2(n2), CALL)
#undef CALL
    return s ? s : ddsp_launch_status();
}

extern "C" int ddsp_b200_fft4_rows_filter(const float *work, float *dst, int64_t slots, const float *hspec,
                                          int64_t h_slot_stride, int conj_h, const float *twiddle,
                                          const float *stage2, int n1, int n2, void *stream) {
    DDSP_REQUIRE(work && dst && hspec && twiddle && stage2 && slots > 0 && slots <= 65535 && plan_ok(n1, n2));
    int s = DDSP_B200_EUNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if (direct_n1(n1)) {
        if ((s = set_smem(rows_kernel<12, 1, true>, row_smem<12>()))) return s;
        rows_kernel<12, 1, true><<<dim3(n1, (unsigned)slots), kRowThreads, row_smem<12>(), st>>>(
            reinterpret_cast<const float2 *>(work), reinterpret_cast<float2 *>(dst),
            reinterpret_cast<const float2 *>(hspec), h_slot_stride, conj_h,
            reinterpret_cast<const float2 *>(twiddle), reinterpret_cast<const float2 *>(stage2), n1);
        return ddsp_launch_status();
    }
#define CALL(LG)                                                                                        \
    if (!(s = set_smem(rows_kernel<LG, 1, false>, row_smem<LG>())))                                     \
        rows_kernel<LG, 1, false><<<dim3(n1 / RowCfg<LG>::ROWS, (unsigned)slots), kRowThreads, row_smem<LG>(), st>>>( \
            reinterpret_cast<const float2 *>(work), reinterpret_cast<float2 *>(dst),                    \
            reinterpret_cast<const float2 *>(hspec), h_slot_stride, conj_h,                             \
            reinterpret_cast<const float2 *>(twiddle), reinterpret_cast<const float2 *>(stage2), n1)
    DDSP_LG_SWITCH_ROWS(ddsp_ilog2(n2), CALL)
#undef CALL
    return s ? s : ddsp_launch_status();
}

extern "C" int64_t ddsp_b200_fft4_correlate_splits(int64_t slots, int reduce) {
    if (!reduce) return slots;
    return (slots < 8 ? slots : 8) + 1;                // + the counter plane of the in-launch finish (5-smooth plans)
}

// splits for a given plan: the correlate kernel runs one CTA per SM, so (row blocks) x splits should not spill into a
// second, nearly empty wave (20 rows x 8 splits = 160 CTAs on 148 SMs did)
static int64_t corr_splits(int64_t slots, int reduce, int n1, int n2) {
    if (!reduce) return slots;
    int64_t s = slots < 8 ? slots : 8;
    if (direct_n1(n1) && n2 == 4096)
        while (s > 1 && (int64_t)n1 * s > DDSP_SM_COUNT) --s;
    return s;
}
// the reduce form on the 5-smooth plans finishes inside the correlate launch: one more scratch plane holds its row counters
static bool corr_fused_finish(int reduce, int n1, int n2) { return reduce && direct_n1(n1) && n2 == 4096; }

extern "C" int64_t ddsp_b200_fft4_correlate_splits_plan(int64_t slots, int reduce, int n1, int n2) {
    return corr_splits(slots, reduce, n1, n2) + (corr_fused_finish(reduce, n1, n2) ? 1 : 0);
}

extern "C" int ddsp_b200_fft4_rows_correlate(const float *work_g, const float *work_x, int64_t slots,
                                             int reduce, float *scratch, float *out, const float *twiddle,
                                             const float *stage2, int n1, int n2, void *stream) {
    return ddsp_b200_fft4_rows_correlate_ex(work_g, work_x, slots, reduce, scratch, out, twiddle, stage2, n1, n2, 0,
                                            stream);
}

extern "C" int64_t ddsp_b200_fft4_correlate_counter_offset(int64_t slots, int reduce, int n1, int n2) {
    return corr_fused_finish(reduce, n1, n2) ? corr_splits(slots, reduce, n1, n2) * (int64_t)n1 * n2 * 2 : -1;
}

extern "C" int ddsp_b200_fft4_rows_correlate_ex(const float *work_g, const float *work_x, int64_t slots,
                                                int reduce, float *scratch, float *out, const float *twiddle,
                                                const float *stage2, int n1, int n2, int counters_zeroed,
                                                void *stream) {
    DDSP_REQUIRE(work_g && work_x && scratch && out && twiddle && stage2 && slots > 0 && slots <= 65535);
    DDSP_REQUIRE(plan_ok(n1, n2));
    const int nsplit = (int)corr_splits(slots, reduce, n1, n2);
    const int nsum = reduce ? nsplit : 1;
    const int nout = reduce ? 1 : (int)slots;
    int s = DDSP_B200_EUNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    if (corr_fused_finish(reduce, n1, n2)) {
        if ((s = set_smem(rows_corr_kernel<12, true, true>, row_smem<12>()))) return s;
        int *counters = reinterpret_cast<int *>(scratch + (size_t)nsplit * n1 * n2 * 2);     // the extra scratch plane
        // the row counters must be zero on entry (the kernel leaves them zero).  A caller that cannot promise it gets
        // them zeroed here, by a one-warp kernel rather than cudaMemsetAsync: a memset node may be scheduled on a copy
        // engine, where it would queue behind the host->device transfer of the next batch
        if (!counters_zeroed) {
            zero_ints_kernel<<<1, 32, 0, st>>>(counters, n1);
            if ((s = ddsp_launch_status())) return s;
        }
        rows_corr_kernel<12, true, true><<<dim3(n1, nsplit), kRowThreads, row_smem<12>(), st>>>(
            reinterpret_cast<const float2 *>(work_g), reinterpret_cast<const float2 *>(work_x), slots, nsplit,
            reinterpret_cast<float2 *>(scratch), reinterpret_cast<const float2 *>(twiddle),
            reinterpret_cast<const float2 *>(stage2), n1, reinterpret_cast<float2 *>(out), counters);
        return ddsp_launch_status();
    }
    if (direct_n1(n1)) {
        if ((s = set_smem(rows_corr_kernel<12, true>, row_smem<12>())) ||
            (s = set_smem(rows_corr_finish_kernel<12>, row_smem<12>())))
            return s;
        rows_corr_kernel<12, true><<<dim3(n1, nsplit), kRowThreads, row_smem<12>(), st>>>(
            reinterpret_cast<const float2 *>(work_g), reinterpret_cast<const float2 *>(work_x), slots, nsplit,
            reinterpret_cast<float2 *>(scratch), reinterpret_cast<const float2 *>(twiddle),
            reinterpret_cast<const float2 *>(stage2), n1);
        if ((s = ddsp_launch_status())) return s;
        rows_corr_finish_kernel<12><<<dim3(n1, nout), kRowThreads, row_smem<12>(), st>>>(
            reinterpret_cast<const float2 *>(scratch), nsum, reinterpret_cast<float2 *>(out),
            reinterpret_cast<const float2 *>(twiddle), reinterpret_cast<const float2 *>(stage2), n1);
        return ddsp_launch_status();
    }
#define CALL(LG)                                                                                        \
    if (!(s = set_smem(rows_corr_kernel<LG, false>, row_smem<LG>())) &&                                 \
        !(s = set_smem(rows_corr_finish_kernel<LG>, row_smem<LG>()))) {                                 \
        rows_corr_kernel<LG, false><<<dim3(n1 / RowCfg<LG>::ROWS, nsplit), kRowThreads, row_smem<LG>(), st>>>(  \
            reinterpret_cast<const float2 *>(work_g), reinterpret_cast<const float2 *>(work_x), slots,  \
            nsplit, reinterpret_cast<float2 *>(scratch), reinterpret_cast<const float2 *>(twiddle),     \
            reinterpret_cast<const float2 *>(stage2), n1);                                              \
        if (!(s = ddsp_launch_status()))                                                                \
            rows_corr_finish_kernel<LG><<<dim3(n1 / RowCfg<LG>::ROWS, nout), kRowThreads, row_smem<LG>(), st>>>( \
                reinterpret_cast<const float2 *>(scratch), nsum, reinterpret_cast<float2 *>(out),       \
                reinterpret_cast<const float2 *>(twiddle), reinterpret_cast<const float2 *>(stage2), n1); \
    }
    DDSP_LG_SWITCH_ROWS(ddsp_ilog2(n2), CALL)
#undef CALL
    return s ? s : ddsp_launch_status();
}

extern "C" int ddsp_b200_reverb_impulse_fwd(const float *noise, const float *decay, const float *wet,
                                            const float *t, float *impulse, int L, void *stream) {
    DDSP_REQUIRE(noise && decay && wet && t && impulse && L > 0);
    reverb_impulse_fwd_kernel<<<(L + 255) / 256, 256, 0, (cudaStream_t)stream>>>(noise, decay, wet, t,
                                                                                 impulse, L);
    return ddsp_launch_status();
}

extern "C" int64_t ddsp_b200_reverb_impulse_bwd_scratch(void) { return 2 * kImpBlocks * (int64_t)sizeof(double); }

extern "C" int ddsp_b200_reverb_impulse_bwd(const float *d_impulse, int Lvalid, const float *noise,
                                            const float *decay, const float *wet, const float *t,
                                            float *d_noise, float *d_decay, float *d_wet, int L,
                                            void *scratch, void *stream) {
    DDSP_REQUIRE(d_impulse && noise && decay && wet && t && d_noise && d_decay && d_wet && scratch && L > 0);
    DDSP_REQUIRE(Lvalid >= 0 && Lvalid <= L);
    cudaStream_t st = (cudaStream_t)stream;
    reverb_impulse_bwd_kernel<<<kImpBlocks, 256, 0, st>>>(d_impulse, Lvalid, noise, decay, wet, t, d_noise,
                                                          reinterpret_cast<double *>(scratch), L);
    int s = ddsp_launch_status();
    if (s) return s;
    reverb_impulse_bwd_finish_kernel<<<1, 32, 0, st>>>(reinterpret_cast<const double *>(scratch), d_decay, d_wet);
    return ddsp_launch_status();
}

static std::atomic<unsigned long long> g_launches{0};
void ddsp_note_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
extern "C" uint64_t ddsp_b200_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

extern "C" int ddsp_b200_abi_version(void) { return 1; }

extern "C" const char *ddsp_b200_strerror(int status) {
    if (status == DDSP_B200_OK) return "ok";
    if (status == DDSP_B200_EINVAL) return "invalid argument (null pointer or bad size)";
    if (status == DDSP_B200_EUNSUPPORTED) return "shape not supported by the sm_100a kernels";
    if (status > 0) return cudaGetErrorString((cudaError_t)status);
    return "unknown ddsp_b200 status";
}
