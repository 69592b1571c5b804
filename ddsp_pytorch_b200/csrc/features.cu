// K5: feature extraction for datasets: A-weighted loudness and MFCCs (SURVEY 8f, the reference's preprocessing).
//
// Reference path replaced:
//   ddsp/core.py:81-97   extract_loudness: librosa.stft(center=True) -> log(|X| + 1e-7) + A_weighting, mean over bins
//   preprocess.py        the MFCCs the autoencoder's encoder reads (encoder.py:35, librosa.feature.mfcc defaults:
//                        power mel spectrogram over 128 Slaney bands, power_to_db with top_db = 80, DCT-II ortho)
//
// Frames: F = 1 + N / hop, the signal reflect-padded by n_fft/2 on each side, the periodic Hann window, the
// unnormalised transform X[k], k = 0 .. n_fft/2 (DESIGN.md 3.7).
//
// Launch 1, one CTA per (tile of frames, row).  Each frame is one complex FFT of the register-tiled kind (regfft.cuh)
// with a zero imaginary part.  Two frames per transform (split by the mirror bins) would halve the FFT work, but
// the rounding error of each half then scales with the energy of BOTH frames: a silent frame beside a loud one gets
// |X| ~ 4e-8 instead of 0, which moves ln(|X| + 1e-7) by ~0.3 in every bin.  Alone in its transform, a frame's error
// scales with its own norm, and its spectrum depends only on its row and index, never on the tile or batch it is
// computed in.  Per batch of G frames:
//   |X|^2 of every bin goes to shared memory;
//   loudness: the sum of ln(|X| + 1e-7) + A[k] over the bins, in an order fixed per n_fft;
//   MFCC    : the 128 band sums read the staged powers through the caller's compact filterbank table (per band: first
//             bin, bin count, weights) in bin order; dB = 10 log10(max(1e-10, mel)) goes to a scratch plane and the
//             row's maximum to an order-preserving integer key (atomicMax: the maximum of a set does not depend on
//             the order it is taken in, so the result is still deterministic).
// Launch 2 clamps each row to its max - 80 dB and applies the (128 x n_mfcc) DCT table, one fixed-order dot product
// per coefficient, accumulated in double.  No sum uses atomics: outputs are bit-identical from run to run and across batch sizes.
#include "common.cuh"
#include "regfft.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int kMels = 128;
constexpr int kDctFrames = 32;          // frames per CTA of launch 2

template <int LG>
struct FeatCfg {
    using P = regfft::Plan<LG>;
    static constexpr int G = (kThreads / P::T) > 16 ? 16 : (kThreads / P::T);   // frames (transforms) per batch
    static constexpr int BINS = P::N / 2 + 1;
    static constexpr size_t SMEM = (size_t)G * P::PITCH * sizeof(float2) + (size_t)G * BINS * sizeof(float);
};

// float -> unsigned key with the same order (0 is below every float), and back
__device__ __forceinline__ unsigned int max_key(float v) {
    const unsigned int u = __float_as_uint(v);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float key_value(unsigned int k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// mel_tab: [0,128) first bin, [128,256) bin count, [256,384) offset of the band's weights, then the weights
template <int LG, bool MEL>
__global__ void __launch_bounds__(kThreads, 2)
features_frames_kernel(const float *__restrict__ signal, const float *__restrict__ window,
                       const float2 *__restrict__ tw, const float *__restrict__ a_weight,
                       const float *__restrict__ mel_tab, float *__restrict__ loud, float *__restrict__ db,
                       unsigned int *__restrict__ row_max, int64_t n, int hop, int frames, int tile_frames) {
    using namespace regfft;
    using P = Plan<LG>;
    using C = FeatCfg<LG>;
    constexpr int N = P::N, T = P::T, G = C::G, PITCH = P::PITCH, HS = N / 2, BINS = C::BINS;
    extern __shared__ __align__(16) float smem[];
    float2 *buf = reinterpret_cast<float2 *>(smem);                          // [G][PITCH]
    float *pw = reinterpret_cast<float *>(buf + (size_t)G * PITCH);          // [G][BINS]  |X|^2
    constexpr int S = G >= kWarps ? 1 : kWarps / G;                         // warps per frame in the loudness sum
    __shared__ float mx[kWarps];
    __shared__ float part[G * S];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int grp = tid / T, t = tid - grp * T;
    const bool act = grp < G;
    const int b = blockIdx.y;
    const int f0 = blockIdx.x * tile_frames;
    const int fe = min(f0 + tile_frames, frames);
    const float *x = signal + (size_t)b * n;
    const int Ni = (int)n;
    float vmax = -INFINITY;

    for (int fb = f0; fb < fe; fb += G) {
        __syncthreads();                                                     // previous batch consumed
        float2 v[16];
        float2 *bg = buf + (size_t)grp * PITCH;
        if (act) {
            // frame fb + grp in the real part; stage 0 straight from global memory
            const int f = fb + grp;
            const bool has = f < fe;
            const int base = f * hop - HS + t;
            const bool inner = f * hop - HS >= 0 && (int64_t)f * hop - HS + N <= n;
#pragma unroll
            for (int r = 0; r < 16; ++r) {
                const float w = __ldg(window + t + r * T);
                int m = base + r * T;
                if (!inner) {
                    m = m < 0 ? -m : m;
                    m = m >= Ni ? 2 * (Ni - 1) - m : m;
                }
                v[r] = make_float2(has ? __ldg(x + m) * w : 0.f, 0.f);
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

        // |X|^2 of every frame of the batch (the transforms' outputs are in natural order)
        for (int idx = tid; idx < G * BINS; idx += kThreads) {
            const int q = idx / BINS, k = idx - q * BINS;
            const float2 z = buf[(size_t)q * PITCH + pad16(k)];
            pw[idx] = fmaf(z.x, z.x, z.y * z.y);
        }
        __syncthreads();

        // loudness: S warps per frame, lane l of segment sg takes bins l + 32 (sg + S i) in order, then a fixed
        // butterfly per warp and the S segment sums in order: the same order for every frame of this n_fft
        if (loud) {
            for (int u = warp; u < G * S; u += kWarps) {
                const int q = u / S, sg = u - q * S;
                float s = 0.f;
                if (fb + q < fe) {
                    const float *pq = pw + q * BINS;
                    for (int k = lane + 32 * sg; k < BINS; k += 32 * S) s += logf(sqrtf(pq[k]) + 1e-7f) + __ldg(a_weight + k);
                }
                s = ddsp_warp_sum(s);
                if (lane == 0) part[u] = s;
            }
            __syncthreads();
            if (tid < G && fb + tid < fe) {
                float s = part[tid * S];
#pragma unroll
                for (int i = 1; i < S; ++i) s += part[tid * S + i];
                loud[(size_t)b * frames + fb + tid] = s / (float)BINS;
            }
        }

        if (MEL) {
            // band sums in bin order; lanes take consecutive bands of one frame, so the dB store coalesces
            for (int idx = tid; idx < G * kMels; idx += kThreads) {
                const int q = idx / kMels, j = idx - q * kMels;
                const int f = fb + q;
                if (f >= fe) break;
                const int k0 = (int)__ldg(mel_tab + j), cnt = (int)__ldg(mel_tab + kMels + j);
                const float *wt = mel_tab + 3 * kMels + (int)__ldg(mel_tab + 2 * kMels + j);
                const float *pq = pw + q * BINS + k0;
                float s = 0.f;
                for (int i = 0; i < cnt; ++i) s = fmaf(__ldg(wt + i), pq[i], s);
                const float d = 10.f * log10f(fmaxf(s, 1e-10f));
                db[((size_t)b * frames + f) * kMels + j] = d;
                vmax = fmaxf(vmax, d);
            }
        }
    }
    if (MEL) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
        if (lane == 0) mx[warp] = vmax;
        __syncthreads();
        if (tid == 0) {
            float m = mx[0];
            for (int w = 1; w < kWarps; ++w) m = fmaxf(m, mx[w]);
            if (m > -INFINITY) atomicMax(row_max + b, max_key(m));
        }
    }
}

// mfcc[b, f, i] = sum_j dct_t[j][i] * max(db[b, f, j], row_max[b] - 80)
__global__ void __launch_bounds__(kThreads)
features_dct_kernel(const float *__restrict__ db, const unsigned int *__restrict__ row_max,
                    const float *__restrict__ dct_t, float *__restrict__ mfcc, int frames, int n_mfcc) {
    __shared__ float s[kDctFrames][kMels];
    const int b = blockIdx.y, f0 = blockIdx.x * kDctFrames;
    const int nf = min(kDctFrames, frames - f0);
    const float floor_db = key_value(__ldg(row_max + b)) - 80.f;
    const float *src = db + ((size_t)b * frames + f0) * kMels;
    for (int i = threadIdx.x; i < nf * kMels; i += kThreads) s[i / kMels][i % kMels] = fmaxf(__ldcg(src + i), floor_db);
    __syncthreads();
    float *dst = mfcc + ((size_t)b * frames + f0) * n_mfcc;
    for (int idx = threadIdx.x; idx < nf * n_mfcc; idx += kThreads) {
        const int q = idx / n_mfcc, i = idx - q * n_mfcc;
        // in double: c_0 of a silent row is -100 sqrt(128) = -1131.4, where a float32 sum of 128 terms drifts by ~1e-3
        double acc = 0.0;
#pragma unroll 8
        for (int j = 0; j < kMels; ++j) acc = fma((double)__ldg(dct_t + j * n_mfcc + i), (double)s[q][j], acc);
        dst[idx] = (float)acc;
    }
}

struct FeatPlan {
    int lg, frames, tile_frames, tiles;
};

int feat_plan(int B, int64_t N, int n_fft, int hop, int n_mfcc, FeatPlan *p) {
    if (B < 1 || B > 65535 || n_fft < 256 || n_fft > 4096 || (n_fft & (n_fft - 1))) return DDSP_B200_EINVAL;
    if (hop < 1 || hop > (1 << 30) || N <= n_fft / 2 || N >= (1ll << 30) || n_mfcc < 1 || n_mfcc > kMels) return DDSP_B200_EINVAL;
    p->lg = 0;
    while ((1 << p->lg) < n_fft) ++p->lg;
    p->frames = 1 + (int)(N / hop);
    const int T = n_fft / 16;
    const int nf = kThreads / T > 16 ? 16 : kThreads / T;          // frames per batch
    // frames per tile, a whole number of batches: up to 4 batches, fewer while the grid is short of 4 CTAs per SM
    int batches = 4;
    while (batches > 1 && (int64_t)ddsp_ceil_div(p->frames, (int64_t)batches * nf) * B < 4 * DDSP_SM_COUNT) batches >>= 1;
    p->tile_frames = batches * nf;
    p->tiles = (int)ddsp_ceil_div(p->frames, p->tile_frames);
    return DDSP_B200_OK;
}

int64_t db_offset(int B) { return ddsp_ceil_div(B, 4) * 4; }        // the row maxima come first

template <typename K>
int allow_smem(K kernel, size_t bytes) {
    if (bytes <= 48 * 1024) return 0;
    return (int)cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

template <int LG, bool MEL>
int launch_frames(const float *signal, const float *window, const float *stage_tw, const float *a_weight,
                  const float *mel_tab, float *loud, float *db, unsigned int *row_max, int B, int64_t N, int hop,
                  const FeatPlan &p, cudaStream_t st) {
    constexpr size_t smem = FeatCfg<LG>::SMEM;
    int s;
    if ((s = allow_smem(features_frames_kernel<LG, MEL>, smem))) return s;
    features_frames_kernel<LG, MEL><<<dim3(p.tiles, B), kThreads, smem, st>>>(
        signal, window, reinterpret_cast<const float2 *>(stage_tw), a_weight, mel_tab, loud, db, row_max, N, hop,
        p.frames, p.tile_frames);
    return ddsp_launch_status();
}

template <bool MEL>
int dispatch_frames(const float *signal, const float *window, const float *stage_tw, const float *a_weight,
                    const float *mel_tab, float *loud, float *db, unsigned int *row_max, int B, int64_t N, int hop,
                    const FeatPlan &p, cudaStream_t st) {
    switch (p.lg) {
        case 8: return launch_frames<8, MEL>(signal, window, stage_tw, a_weight, mel_tab, loud, db, row_max, B, N, hop, p, st);
        case 9: return launch_frames<9, MEL>(signal, window, stage_tw, a_weight, mel_tab, loud, db, row_max, B, N, hop, p, st);
        case 10: return launch_frames<10, MEL>(signal, window, stage_tw, a_weight, mel_tab, loud, db, row_max, B, N, hop, p, st);
        case 11: return launch_frames<11, MEL>(signal, window, stage_tw, a_weight, mel_tab, loud, db, row_max, B, N, hop, p, st);
        case 12: return launch_frames<12, MEL>(signal, window, stage_tw, a_weight, mel_tab, loud, db, row_max, B, N, hop, p, st);
        default: return DDSP_B200_EINVAL;
    }
}

}  // namespace

extern "C" int64_t ddsp_b200_features_scratch(int B, int64_t N, int n_fft, int hop, int n_mfcc) {
    FeatPlan p;
    if (feat_plan(B, N, n_fft, hop, n_mfcc, &p)) return DDSP_B200_EINVAL;
    return db_offset(B) + (int64_t)B * p.frames * kMels;
}

extern "C" int ddsp_b200_features_fwd(const float *signal, const float *window, const float *stage_twiddle,
                                      const float *a_weight, const float *mel_table, const float *dct,
                                      float *loudness, float *mfcc, float *scratch, int B, int64_t N, int n_fft,
                                      int hop, int n_mfcc, void *stream) {
    DDSP_REQUIRE(signal && window && stage_twiddle && (loudness || mfcc));
    DDSP_REQUIRE(!loudness || a_weight);
    DDSP_REQUIRE(!mfcc || (mel_table && dct && scratch));
    FeatPlan p;
    int s = feat_plan(B, N, n_fft, hop, n_mfcc, &p);
    if (s) return s;
    cudaStream_t st = (cudaStream_t)stream;
    if (!mfcc)
        return dispatch_frames<false>(signal, window, stage_twiddle, a_weight, nullptr, loudness, nullptr, nullptr,
                                      B, N, hop, p, st);
    unsigned int *row_max = reinterpret_cast<unsigned int *>(scratch);
    float *db = scratch + db_offset(B);
    cudaError_t e = cudaMemsetAsync(row_max, 0, sizeof(unsigned int) * (size_t)B, st);
    if (e != cudaSuccess) return (int)e;
    if ((s = dispatch_frames<true>(signal, window, stage_twiddle, a_weight, mel_table, loudness, db, row_max, B, N,
                                   hop, p, st)))
        return s;
    features_dct_kernel<<<dim3((unsigned)ddsp_ceil_div(p.frames, kDctFrames), B), kThreads, 0, st>>>(
        db, row_max, dct, mfcc, p.frames, n_mfcc);
    return ddsp_launch_status();
}
