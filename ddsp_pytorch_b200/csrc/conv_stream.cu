// K3s: streaming causal convolution with caller-owned history (the reverb of the realtime export).
//
// Reference path extended: ddsp/models/modules.py:28-35 (Reverb.forward -> fft_convolve) convolves one whole signal
// and crops the impulse to the call's length.  Played buffer by buffer, that loses the tail: a 1024-sample buffer
// sees 1024 of the 48 000 taps and nothing carries into the next buffer.  Here the previous L-1 input samples are
// an input (history) and an output (history_out), so consecutive calls give the convolution of the whole stream:
//   u = [history | x]                        (B, L-1+N), oldest first
//   y[b,n] = sum_{k<L} h[k] * u[b, L-1+n-k]
//   history_out = last L-1 samples of u
// Direct form, B*N*L FMA: at the realtime shape (1 x 1024 x 48 000) that is 49 M FMA, a few microseconds of the
// GPU, where a transform would need >= N + 2L - 2 points and several dependent launches.
//
// Launch 1, one CTA per (chunk of TK taps, tile of kTile outputs, voice):
//   the u-window of the tile and chunk (kTile + TK floats) and the chunk's taps (reversed) are staged in shared
//   memory, the window twice: as is and shifted by one float, so that the odd-aligned pairs (w[2q+1], w[2q+2])
//   are register pairs as well.  Thread (og, ks) owns 8 consecutive outputs and a sub-chunk of TK/16 taps and
//   walks them with a register sliding window: per 4 taps two LDS.128 of window, one (broadcast) LDS.128 of
//   taps and 16 FFMA2 on output pairs, no moves.  The 16 sub-chunk sums are added in ks order through shared
//   memory.  With one chunk the CTA writes y; otherwise it writes its chunk's partial sums, and
// Launch 2 adds the chunks' partials of each output in chunk order.
// No atomics anywhere: y and history_out are bit-identical from run to run.  Launch 1 also writes history_out
// (a separate buffer from history, so no CTA can read a sample another one already overwrote).
#include "common.cuh"

namespace {

constexpr int kThreads = 256;        // 16 output groups x 16 tap sub-chunks
constexpr int kGroups = 16;
constexpr int kPerThread = 8;        // consecutive outputs per thread
constexpr int kTile = kGroups * kPerThread;      // 128 outputs per CTA
constexpr int kSub = kThreads / kGroups;         // 16 tap sub-chunks per CTA
constexpr int kMaxOdd = 47;                      // <= 64 * 47 = 3008 taps per CTA: 45 KB of shared memory
constexpr int kFinishThreads = 256;

// Taps per CTA: an odd multiple of 64, so that a sub-chunk (TK / 16 taps) is 4 mod 8 floats long and the window
// reads of the two sub-chunks in a quarter-warp fall into different 16-byte bank groups (conflict-free LDS.128).
// Chunks are sized so that the grid covers about two waves of 148 SMs.
int taps_per_cta(int B, int64_t N, int L) {
    const int64_t tiles = (int64_t)B * ddsp_ceil_div(N, kTile);
    const int64_t want = tiles >= 2 * DDSP_SM_COUNT ? 1 : ddsp_ceil_div(2 * DDSP_SM_COUNT, tiles);
    const int64_t per = ddsp_ceil_div(L, want);
    int64_t q = ddsp_ceil_div(per, 64);
    if (q % 2 == 0) ++q;
    return (int)(64 * (q < kMaxOdd ? q : kMaxOdd));
}

// lane -> (output group, tap sub-chunk): a quarter-warp holds 4 output groups x 2 sub-chunks
__device__ __forceinline__ void thread_role(int tid, int &og, int &ks) {
    const int lane = tid & 31, warp = tid >> 5;
    og = (lane & 3) | ((lane >> 3) << 2);
    ks = ((lane >> 2) & 1) | (warp << 1);
}

__device__ __forceinline__ float u_at(const float *__restrict__ hist, const float *__restrict__ x, int64_t Lm1,
                                      int64_t N, int64_t i) {
    if (i < 0 || i >= Lm1 + N) return 0.f;
    return i < Lm1 ? __ldg(hist + i) : __ldg(x + (i - Lm1));
}

__global__ void __launch_bounds__(kThreads)
conv_stream_kernel(const float *__restrict__ x, const float *__restrict__ h, const float *__restrict__ history,
                   float *__restrict__ y, float *__restrict__ history_out, float *__restrict__ partial, int64_t N,
                   int L, int TK) {
    extern __shared__ __align__(16) float smem[];
    float *win = smem;                       // [kTile + TK]   u[base + i]
    float *wsh = win + kTile + TK;           // [kTile + TK]   u[base + i + 1]
    float *hr = wsh + kTile + TK;            // [TK]           h[k0 + TK-1 - j], 0 past L
    float *red = hr + TK;                    // [kSub][kTile]  sub-chunk sums
    const int tid = threadIdx.x;
    const int chunk = blockIdx.x, chunks = gridDim.x;
    const int64_t n0 = (int64_t)blockIdx.y * kTile;
    const int b = blockIdx.z;
    const int64_t Lm1 = L - 1;
    const int64_t k0 = (int64_t)chunk * TK;
    const float *xb = x + (int64_t)b * N;
    const float *hb = history + (int64_t)b * Lm1;

    // history_out = u[N .. N+L-1), spread over every CTA of the launch
    {
        const int64_t cta = ((int64_t)b * gridDim.y + blockIdx.y) * chunks + chunk;
        const int64_t ncta = (int64_t)gridDim.x * gridDim.y * gridDim.z;
        for (int64_t j = cta * kThreads + tid; j < Lm1; j += ncta * kThreads) {
            const int64_t src = N + j;
            for (int bb = 0; bb < (int)gridDim.z; ++bb)
                history_out[bb * Lm1 + j] = src < Lm1 ? __ldg(history + bb * Lm1 + src) : __ldg(x + bb * N + (src - Lm1));
        }
    }

    // y[n0+m] gets sum_j hr[j] * win[m + j]  with  win[i] = u[base + i]
    const int64_t base = Lm1 + n0 - k0 - (TK - 1);
    for (int i = tid; i < kTile + TK; i += kThreads) {
        win[i] = u_at(hb, xb, Lm1, N, base + i);
        wsh[i] = u_at(hb, xb, Lm1, N, base + i + 1);
    }
    for (int j = tid; j < TK; j += kThreads) {
        const int64_t k = k0 + TK - 1 - j;
        hr[j] = k < L ? __ldg(h + k) : 0.f;
    }
    __syncthreads();

    int og, ks;
    thread_role(tid, og, ks);
    const int TKs = TK / kSub;
    const float *wp = win + og * kPerThread + ks * TKs;
    const float *op = wsh + og * kPerThread + ks * TKs;
    const float *hp = hr + ks * TKs;
    uint64_t acc[4] = {0, 0, 0, 0};          // (y[2p], y[2p+1]) of the thread's 8 outputs
    // e_q = (w[2q], w[2q+1]), o_q = (w[2q+1], w[2q+2]) relative to the current tap
    const ulonglong2 ea = *reinterpret_cast<const ulonglong2 *>(wp), eb = *reinterpret_cast<const ulonglong2 *>(wp + 4);
    const ulonglong2 oa = *reinterpret_cast<const ulonglong2 *>(op), ob = *reinterpret_cast<const ulonglong2 *>(op + 4);
    uint64_t e0 = ea.x, e1 = ea.y, e2 = eb.x, e3 = eb.y, o0 = oa.x, o1 = oa.y, o2 = ob.x, o3 = ob.y;
    // 3 steps = one period of the window rotation: the shifts below become register renaming (64 registers, no spill)
#pragma unroll 3
    for (int j = 0; j < TKs; j += 4) {
        const ulonglong2 en = *reinterpret_cast<const ulonglong2 *>(wp + j + 8);
        const ulonglong2 on = *reinterpret_cast<const ulonglong2 *>(op + j + 8);
        const float4 c = *reinterpret_cast<const float4 *>(hp + j);
        const uint64_t e4 = en.x, e5 = en.y, o4 = on.x, o5 = on.y;
        const uint64_t t0 = pk2(c.x, c.x), t1 = pk2(c.y, c.y), t2 = pk2(c.z, c.z), t3 = pk2(c.w, c.w);
        acc[0] = fma2(t0, e0, acc[0]); acc[1] = fma2(t0, e1, acc[1]); acc[2] = fma2(t0, e2, acc[2]); acc[3] = fma2(t0, e3, acc[3]);
        acc[0] = fma2(t1, o0, acc[0]); acc[1] = fma2(t1, o1, acc[1]); acc[2] = fma2(t1, o2, acc[2]); acc[3] = fma2(t1, o3, acc[3]);
        acc[0] = fma2(t2, e1, acc[0]); acc[1] = fma2(t2, e2, acc[1]); acc[2] = fma2(t2, e3, acc[2]); acc[3] = fma2(t2, e4, acc[3]);
        acc[0] = fma2(t3, o1, acc[0]); acc[1] = fma2(t3, o2, acc[1]); acc[2] = fma2(t3, o3, acc[2]); acc[3] = fma2(t3, o4, acc[3]);
        e0 = e2; e1 = e3; e2 = e4; e3 = e5;
        o0 = o2; o1 = o3; o2 = o4; o3 = o5;
    }
    float v[8];
#pragma unroll
    for (int p = 0; p < 4; ++p) unpk2(acc[p], v[2 * p], v[2 * p + 1]);
    float4 *dst = reinterpret_cast<float4 *>(red + ks * kTile + og * kPerThread);
    dst[0] = make_float4(v[0], v[1], v[2], v[3]);
    dst[1] = make_float4(v[4], v[5], v[6], v[7]);
    __syncthreads();
    if (tid < kTile && n0 + tid < N) {
        float s = red[tid];
#pragma unroll
        for (int k = 1; k < kSub; ++k) s += red[k * kTile + tid];
        if (chunks == 1) y[(int64_t)b * N + n0 + tid] = s;
        else partial[((int64_t)b * chunks + chunk) * N + n0 + tid] = s;
    }
}

// y[b,n] = sum over chunks, in chunk order, of partial[b][chunk][n]
__global__ void __launch_bounds__(kFinishThreads)
conv_stream_finish_kernel(const float *__restrict__ partial, float *__restrict__ y, int64_t N, int chunks) {
    const int64_t n = (int64_t)blockIdx.x * kFinishThreads + threadIdx.x;
    const int b = blockIdx.y;
    if (n >= N) return;
    const float *p = partial + (int64_t)b * chunks * N + n;
    float s = 0.f;
#pragma unroll 4
    for (int c = 0; c < chunks; ++c) s += __ldcg(p + (int64_t)c * N);
    y[(int64_t)b * N + n] = s;
}

struct StreamPlan {
    int TK, chunks;
    int64_t tiles;
};

StreamPlan stream_plan(int B, int64_t N, int L) {
    StreamPlan p;
    p.TK = taps_per_cta(B, N, L);
    p.chunks = (int)ddsp_ceil_div(L, p.TK);
    p.tiles = ddsp_ceil_div(N, kTile);
    return p;
}

}  // namespace

extern "C" int64_t ddsp_b200_conv_stream_scratch(int B, int64_t N, int L) {
    if (B < 1 || N < 1 || L < 1) return DDSP_B200_EINVAL;
    const StreamPlan p = stream_plan(B, N, L);
    return p.chunks > 1 ? (int64_t)B * p.chunks * N : 0;
}

extern "C" int ddsp_b200_conv_stream_fwd(const float *x, const float *h, const float *history, float *y,
                                         float *history_out, int B, int64_t N, int L, float *scratch,
                                         void *stream) {
    DDSP_REQUIRE(x && h && y && B >= 1 && N >= 1 && L >= 1);
    DDSP_REQUIRE(L == 1 || (history && history_out));
    const StreamPlan p = stream_plan(B, N, L);
    DDSP_REQUIRE(p.chunks == 1 || scratch);
    if (p.tiles > 65535 || B > 65535) return DDSP_B200_EUNSUPPORTED;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t smem = (size_t)(2 * kTile + 3 * p.TK + kSub * kTile) * sizeof(float);      // <= 45 KB
    conv_stream_kernel<<<dim3(p.chunks, (unsigned)p.tiles, B), kThreads, smem, st>>>(
        x, h, history, y, history_out, scratch, N, L, p.TK);
    int s = ddsp_launch_status();
    if (s || p.chunks == 1) return s;
    conv_stream_finish_kernel<<<dim3((unsigned)ddsp_ceil_div(N, kFinishThreads), B), kFinishThreads, 0, st>>>(
        scratch, y, N, p.chunks);
    return ddsp_launch_status();
}
