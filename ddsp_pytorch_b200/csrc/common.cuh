// Shared device/host helpers for libddsp_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "ddsp_b200.h"

#define DDSP_SM_COUNT 148  // B200: 2 dies x 74 SMs; grids of persistent kernels are sized off this

// Launch-status helper: argument errors are negative, CUDA errors positive (header contract).
// Every successful kernel launch is also counted (ddsp_b200_launch_count: bench.py's gpu_launches).
void ddsp_note_launch();
static inline int ddsp_launch_status() {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
    ddsp_note_launch();
    return DDSP_B200_OK;
}

#define DDSP_REQUIRE(cond) \
    do {                   \
        if (!(cond)) return DDSP_B200_EINVAL; \
    } while (0)

static inline int64_t ddsp_ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Launch as the programmatic dependent of the kernel launched before it on `st`: dispatched once every CTA of that
// kernel has run griddepcontrol.launch_dependents (or exited), not when it ends.  The kernel must read nothing the
// earlier one writes (it never calls griddepcontrol.wait).
template <typename... P, typename... A>
int ddsp_launch_programmatic(void (*kernel)(P...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, A &&...args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr;
    attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr.val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = &attr;
    cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, static_cast<A &&>(args)...);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return (int)e;
    }
    return ddsp_launch_status();
}

// The oscillator bank's half of the synth pair (harmonic.cu), launched as the programmatic dependent of the filtered
// noise by ddsp_b200_synth_pair_fwd / _bwd (noise.cu).  Same arguments and results as
// ddsp_b200_harmonic_frames_raw_scan_fwd / ddsp_b200_harmonic_frames_raw_bwd.
bool ddsp_pair_bank_supported(int T, int H, int block_size);
int ddsp_pair_bank_fwd(const float *amp_raw, int64_t amp_stride, const float *dist_raw, int64_t dist_stride,
                       const float *f0, const double *phase0, uint64_t *phi, uint64_t *delta, double *phase_end,
                       float *amps, float *weights, float *audio, int B, int T, int H, int block_size,
                       double sample_rate, cudaStream_t st);
int ddsp_pair_bank_bwd(const float *g_audio, const float *amp_raw, int64_t amp_stride, const float *dist_raw,
                       int64_t dist_stride, const float *f0, const uint64_t *phi, const uint64_t *delta,
                       float *d_amp_raw, int64_t d_amp_stride, float *d_dist_raw, int64_t d_dist_stride, int B, int T,
                       int H, int block_size, float sample_rate, cudaStream_t st);

// ---------------------------------------------------------------------------------------------
// Phase arithmetic.  Phases are kept in TURNS as Q0.64 unsigned fixed point: wrap-around of the
// 64-bit integer is exactly "mod 1 turn", so k*phase for harmonic k is exact however long the
// signal (the reference's float32 k*omega loses ~4e-2 over 4 s, SURVEY 8c).
// ---------------------------------------------------------------------------------------------

// Fold a Q0.64 phase to [-1/4, 1/4) turns plus a half-turn count parity:
//   phase = psi + r/2 (mod 1),  sin(2*pi*k*phase) = (-1)^(k*r) * sin(2*pi*k*psi).
// Returns psi as a float in turns; *flip = r & 1.
__device__ __forceinline__ float ddsp_fold_quarter(uint64_t p, int *flip) {
    uint32_t r = (uint32_t)(((p >> 62) + 1) >> 1);      // round(2*p) in {0,1,2}
    uint64_t psi = p - ((uint64_t)r << 63);             // r == 2 wraps to -1 turn
    *flip = (int)(r & 1u);
    return (float)(int32_t)(psi >> 32) * 2.3283064365386963e-10f;   // * 2^-32
}

// Q0.64 (signed view) -> float turns in [-1/2, 1/2)
__device__ __forceinline__ float ddsp_turns_signed(uint64_t p) {
    return (float)(int32_t)(p >> 32) * 2.3283064365386963e-10f;
}

// sin / cos of x for |x| <= pi/4 (no range reduction; ~1 ulp).  Minimax coefficients as used by
// the usual single-precision kernels (Cephes sinf/cosf).
__device__ __forceinline__ float ddsp_sin_q(float x) {
    float z = x * x;
    float p = fmaf(z, -1.9515295891e-4f, 8.3321608736e-3f);
    p = fmaf(z, p, -1.6666654611e-1f);
    return fmaf(x * z, p, x);
}
__device__ __forceinline__ float ddsp_cos_q(float x) {
    float z = x * x;
    float p = fmaf(z, 2.443315711809948e-5f, -1.388731625493765e-3f);
    p = fmaf(z, p, 4.166664568298827e-2f);
    return fmaf(z * z, p, fmaf(z, -0.5f, 1.0f));
}

// Reinsch form of the sine recurrence, stable for |psi| <= pi/2 (cos(psi) >= 0):
//   u = -4 sin^2(psi/2);   d_{k+1} = d_k + u*s_k;   s_{k+1} = s_k + d_{k+1}
// Error grows ~1.2e-7 * steps (measured in oracle-side simulation), against ~k^2 for Chebyshev.
struct ddsp_osc {
    float s, d, u;
    __device__ __forceinline__ void step() {
        d = fmaf(u, s, d);
        s += d;
    }
};

// scale_function of the reference (ddsp/core.py:77-78): 2*sigmoid(x)^ln10 + 1e-7, and its derivative
__device__ __forceinline__ float ddsp_softplus_neg(float x) {          // log(1 + exp(-x)), stable
    return fmaxf(-x, 0.f) + log1pf(expf(-fabsf(x)));
}
__device__ __forceinline__ float ddsp_scale_core(float x) {
    return 2.f * expf(-2.302585092994046f * ddsp_softplus_neg(x));      // 2*sigmoid(x)^ln10
}
__device__ __forceinline__ float ddsp_scale_fn(float x) { return ddsp_scale_core(x) + 1e-7f; }
__device__ __forceinline__ float ddsp_scale_grad(float x) {             // ln10 * 2 sigmoid^ln10 * (1 - sigmoid)
    return 2.302585092994046f * ddsp_scale_core(x) * (1.f / (1.f + expf(x)));
}

// both at once (the backward of the controls needs the value for the normalisation and the derivative for the chain):
// one exp(-|x|), one log1p, one exp, one division instead of five exponentials, two log1p and a division
__device__ __forceinline__ void ddsp_scale_fn_grad(float x, float *fn, float *grad) {
    const float e = expf(-fabsf(x));                                    // exp(-|x|) in (0, 1]
    const float sp = fmaxf(-x, 0.f) + log1pf(e);                        // softplus(-x)
    const float core = 2.f * expf(-2.302585092994046f * sp);            // 2 sigmoid(x)^ln10
    const float r = 1.f / (1.f + e);
    const float sig_neg = x >= 0.f ? e * r : r;                         // sigmoid(-x) = 1 - sigmoid(x)
    *fn = core + 1e-7f;
    *grad = 2.302585092994046f * core * sig_neg;
}

// (mask.float() + 1e-4) of remove_above_nyquist (ddsp/core.py:73): both branches are float32 sums; the product
// f0 * k is rounded once, as the reference's float32 multiply is
__device__ __forceinline__ float ddsp_nyquist_mask(float f0, int k1, float nyq) {
    return (__fmul_rn(f0, (float)k1) < nyq) ? (1.0f + 1e-4f) : 1e-4f;
}

#define DDSP_PI_F 3.14159265358979323846f
#define DDSP_2PI_F 6.28318530717958647692f

__device__ __forceinline__ float ddsp_warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---- packed FP32 (sm_100 FFMA2 / FADD2 / FMUL2): one instruction on a 64-bit register pair of two floats.
// Measured (tools/probes/fp32_pace_probe.cu, profiles/r02_fp32_pace_probe.txt): a scalar FFMA issues every cycle
// per scheduler (128 lanes/clk/SM) and a packed one every other cycle, so the FP32 lane rate is the same; what the
// packed forms save is issue slots (and, with two transforms in the two halves, index maths and LDS/STS count).
// ptxas folds negation, a half swap (.LO_HI) and a scalar broadcast (R.F32) into the operand for free.
__device__ __forceinline__ uint64_t pk2(float a, float b) {
    uint64_t r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ void unpk2(uint64_t v, float &a, float &b) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
    uint64_t r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
