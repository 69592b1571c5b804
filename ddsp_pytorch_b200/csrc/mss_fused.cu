// K4L, second generation: the multi-scale spectral loss and its gradient w.r.t. the reconstruction, ALL
// scales in ONE launch (SURVEY 8a rows a11 + a12 + their backward).
//
// Reference path replaced (same as stft.cu):
//   ddsp/core.py:27-41     multiscale_fft (torch.stft per scale, reflect pad, periodic hann, normalized, abs)
//   train.py:70-76,92-103  multiscale_spec_loss (lin + log L1 per scale)
//   and the autograd backward of both.
//
// Design (DESIGN.md 3.4).  Valid for hop = n_fft/4 (overlap 0.75, the reference's only setting), n_fft = 64..4096.
//   * Work item = (scale, voice, tile of FT consecutive FRAMES); one CTA per item, items ordered by scale (largest
//     first) so the hardware block scheduler balances them over the SMs.  Every frame is transformed exactly once
//     (the first generation recomputed the 3 overlap frames of every tile: +33 % at 4096).
//   * A group of T = n_fft/16 threads owns TWO adjacent frames at a time, one per lane of the packed f32x2
//     registers (pfft.cuh): rec + i*target of frame A in lane 0, of frame B in lane 1.  Frame B's samples are frame
//     A's shifted by one hop = 4 register slots, so 20 loads per signal serve both frames.
//   * After the last forward stage the spectra stay in registers.  Bin k needs Z[k] and Z[n_fft-k]; the mirror
//     lives in thread T-t, so the upper half of each thread's bins goes through shared memory once (8 of 16 slots),
//     the loss terms and gradient spectra are computed in registers, the mirrored half of the gradient spectrum
//     goes back the same way, and the inverse transform (one complex FFT carries the real gradients of BOTH
//     frames: U_A + i U_B) starts from registers.
//   * Overlap-add stays in registers.  A tile's frames are split into contiguous RUNS, one per thread group; slot q of
//     frame f+1 is slot q+4 of frame f IN THE SAME THREAD, so a thread adds the windowed gradient frames of its run into
//     a 20-slot accumulator, stores the 8 finished slots of every pair to the scale's gradient plane P and carries 12
//     (a thread-private strip of shared memory, no barrier).  At the end of the tile a run's first 3 hops receive the
//     final carry of the previous group's run (read-modify-write of the thread's own stores); the last group's carry
//     goes to a small halo buffer that mss_combine2_kernel adds to the head of the next tile.  No atomics, every
//     position sums its frames oldest first: bit-reproducible.  80 KB of shared memory per CTA: two CTAs per SM leave
//     64 KB of L1 for the sample re-reads (a pair re-reads 12 of its predecessor's 20 slots), the window and the stage
//     twiddles.
//   * mss_combine2_kernel sums the scales in order and folds the reflect padding back.

#include "common.cuh"
#include "pfft.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kMaxScales = 8;
constexpr int kWorkBytes = kThreads * 16 * 17;           // 256 threads x 16 points x 16 B, padded 17/16

struct ScaleDesc {
    int lg, hop, frames, ft_log;       // frames per tile = 1 << ft_log
    int tiles;                          // tiles per voice
    int item0;                          // first work item of this scale
    int last_end;                       // first frame slot not finished by the last tile's batches
    int rowlen;                         // floats per voice in P (multiple of 4)
    long long p_off;                    // float offset of P      [B][rowlen]
    long long h_off;                    // float offset of halos  [B][tiles][3*hop]
    long long part_off;                 // pair offset of the loss partials [tiles][B]
    const float *window;
    const float2 *tw;
    float inv_cnt;
    int pad_;
};

struct FusedArgs {
    int n_scales, B, n_items, pad_;
    long long N;
    ScaleDesc sc[kMaxScales];
};

template <int T> __device__ __forceinline__ void gsync(int grp) {
    if (T <= 32) __syncwarp();
    else if (T == kThreads) __syncthreads();
    else if (grp == 0) asm volatile("bar.sync 1, %0;" ::"n"(T) : "memory");
    else if (grp == 1) asm volatile("bar.sync 2, %0;" ::"n"(T) : "memory");
    else if (grp == 2) asm volatile("bar.sync 3, %0;" ::"n"(T) : "memory");
    else asm volatile("bar.sync 4, %0;" ::"n"(T) : "memory");
}

// Loss terms and gradient spectra of bin k = t + Q*T (Q < 8; Q = 8 is k = n_fft/2, thread 0 only) for the two
// frames in the lanes.  x = the thread's spectra after the last forward stage, gbuf = the parked mirror bins.
// Q is a template parameter so that x[] and zi[] are indexed statically and stay in registers.  Everything except
// the four special-function evaluations per lane runs on both frames at once (packed).
//   Y2 = Z[k] + conj Z[-k] = 2 Y (rec), X2 = -i (Z[k] - conj Z[-k]) = 2 X (target): the halves are folded into rs2.
//   loss terms  |sy - sx|, |log(sy + eps) - log(sx + eps)|   with sy = |Y| / sqrt(n_fft)
//   dL/dY = (sgn(sy - sx) (1 + 1/(sy + eps)) inv_cnt / sqrt(n_fft)) Y / |Y|     (log is monotonic: one sign serves both)
// A frame that does not exist has zero input, so Y = 0 and its gradient is 0 without a test; `own` only keeps its
// log term (log(eps/eps), not exactly 0 in float) out of the sum.
template <int LG, bool GRAD, int Q>
__device__ __forceinline__ void bin_math(const pfft::C (&x)[16], pfft::V (&zi)[16], const pfft::E *gbuf, float2 *ex2,
                                         int t, pfft::V own, float rs2, float kc, pfft::V &lin, pfft::V &lgs) {
    using namespace pfft;
    constexpr int T = Plan<LG>::T;
    constexpr int q = Q;
    const C zk = x[slot_of_q<LG>(q)];
    C zm = from_e(gbuf[q < 8 ? (8 - q) * T - t : 0]);     // Z[n_fft - k]
    const bool self = (q == 0 && t == 0) || q == 8;       // k = 0 and k = n_fft/2 mirror themselves
    if (q == 0 && t == 0) zm = zk;
    const V yr = zk.re + zm.re, yi = zk.im - zm.im;
    const V xre = zk.im + zm.im, xim = zm.re - zk.re;
    const V yy = fma(yr, yr, yi * yi), xx = fma(xre, xre, xim * xim);
    float a0, a1, b0, b1;
    get(yy, a0, a1);
    get(xx, b0, b1);
    const V ry = mk(rsqrtf(fmaxf(a0, 1e-37f)), rsqrtf(fmaxf(a1, 1e-37f)));          // 1 / |Y2|
    const V rx = mk(rsqrtf(fmaxf(b0, 1e-37f)), rsqrtf(fmaxf(b1, 1e-37f)));
    const V sy = (yy * ry) * bc(rs2), sx = (xx * rx) * bc(rs2);
    const V d = sy - sx;
    const V sye = sy + bc(1e-7f);
    get(sye, a0, a1);
    const V iy = mk(__fdividef(1.0f, a0), __fdividef(1.0f, a1));
    get((sx + bc(1e-7f)) * iy, b0, b1);
    float d0, d1;
    get(d, d0, d1);
    lin = lin + mk(fabsf(d0), fabsf(d1));
    lgs = fma(own, mk(fabsf(__log2f(b0)), fabsf(__log2f(b1))), lgs);               // * ln 2 at the end
    if (GRAD) {
        // sign(d) * kc, 0 at an exact tie (torch.sign(0) = 0); interior bins carry the 1/2 of (U_A + i U_B) / 2
        const float kq = self ? kc : 0.5f * kc;
        const V sgk = mk(d0 == 0.f ? 0.f : copysignf(kq, d0), d1 == 0.f ? 0.f : copysignf(kq, d1));
        const V c = fma(sgk, iy, sgk) * ry;                                        // dL/dY2 = c * Y2
        const V ur = c * yr, ui = c * yi;                                          // U = (U_A, U_B) lanes
        float ura, urb, uia, uib;
        get(ur, ura, urb);
        get(ui, uia, uib);
        // (U_A + i U_B): real bins are (U_A, U_B); Zi[k] = (ura - uib, uia + urb), Zi[-k] = (ura + uib, urb - uia)
        zi[q] = self ? mk(ura, urb) : mk(ura - uib, uia + urb);
        if (q == 8) ex2[0] = make_float2(ura, urb);                                // keeps the read of the upper slots uniform
        else if (!self) ex2[(8 - q) * T - t] = make_float2(ura + uib, urb - uia);
    }
}

// Samples t + qT, q = 0..19, of rec and target from `start` on (reflect padding at the signal's ends): frame A uses
// slots 0..15, frame B = A + 1 hop uses slots 4..19.
// (plain cached loads: slots 8..19 are read again by the same thread for the run's next pair and then hit in L1;
// ld.global.nc.L1::no_allocate was 5 % slower here)
template <int N, int T>
__device__ __forceinline__ void load_frames(float (&r)[20], float (&g)[20], const float *__restrict__ xr,
                                            const float *__restrict__ xt, int start, int t, int Ni) {
    if (start >= 0 && start + N / 4 + N <= Ni) {
#pragma unroll
        for (int q = 0; q < 20; ++q) {
            r[q] = __ldg(xr + start + t + q * T);
            g[q] = __ldg(xt + start + t + q * T);
        }
    } else {
#pragma unroll
        for (int q = 0; q < 20; ++q) {
            int m = start + t + q * T;
            m = m < 0 ? -m : m;
            m = m >= Ni ? 2 * (Ni - 1) - m : m;
            m = min(max(m, 0), Ni - 1);                      // only frames that do not exist reach this clamp
            r[q] = __ldg(xr + m);
            g[q] = __ldg(xt + m);
        }
    }
}

template <int LG, bool GRAD>
__device__ __forceinline__ void tile_body(const ScaleDesc &sc, int b, int tile, int B, int Ni,
                                          const float *__restrict__ target, const float *__restrict__ rec,
                                          float *__restrict__ ws, float *__restrict__ partial,
                                          unsigned char *smem) {
    using namespace pfft;
    using P = Plan<LG>;
    constexpr int N = P::N, T = P::T, G = kThreads / T, HOP = N / 4, HS = N / 2;
    constexpr int GBYTES = (N + N / 16) * 16;                     // bytes of one group's work buffer
    constexpr int EX2_OFF = 13 * N;                               // mirrored gradient bins
    static_assert(kThreads % T == 0 && G * GBYTES == kWorkBytes, "work buffer layout");
    // thread-private strip (float4 [3][kThreads], conflict free): the running overlap-add carry (12 slots = 3 hops)
    float4 *cpriv = reinterpret_cast<float4 *>(smem + kWorkBytes);
    __shared__ float red[2][kThreads / 32];

    const int tid = threadIdx.x;
    const int grp = tid / T, t = tid - grp * T;
    unsigned char *gbase = smem + (size_t)grp * GBYTES;
    E *gbuf = reinterpret_cast<E *>(gbase);
    float2 *ibuf = reinterpret_cast<float2 *>(gbase);
    float2 *ex2 = reinterpret_cast<float2 *>(gbase + EX2_OFF);

    const float *xr = rec + (size_t)b * Ni;
    const float *xt = target + (size_t)b * Ni;
    const float *__restrict__ window = sc.window;
    const float2 *__restrict__ tw = sc.tw;
    // the tile's frames are split into G contiguous RUNS of RL frames, one per thread group: the overlap-add of a
    // run's frames stays inside the thread (frame f+1's sample slot q is frame f's slot q+4)
    const int rl_log = sc.ft_log - (12 - LG);                    // log2(FT / G) with G = 2^(12-LG); >= 2 (make_plan)
    const int RL = 1 << rl_log;
    const int f0 = tile << sc.ft_log;
    const int f1 = min(f0 + (1 << sc.ft_log), sc.frames);
    const int run0 = f0 + (grp << rl_log);
    // a run is taken whole or not at all; groups that share a warp take the same decision (frames past f1 are zeros)
    const int grp_w = T < 32 ? (tid & ~31) / T : grp;
    const bool active = f0 + (grp_w << rl_log) < f1;
    const float rs = rsqrtf((float)N);
    const float rs2 = 0.5f * rs;                                  // spectra are kept doubled (no 1/2 in the untangle)
    const float kc = sc.inv_cnt * rs;
    float *Pb = ws + sc.p_off + (size_t)b * sc.rowlen;

    if (GRAD) {
        const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int k = 0; k < 3; ++k) cpriv[k * kThreads + tid] = z4;
    }
    V lin = bc(0.f), lgs = bc(0.f);

    // samples of frames A (slots 0..15) and B = A + 1 (slots 4..19) of rec and target
    float r[20], g[20];

    for (int p = 0; active && p < (RL >> 1); ++p) {
        const int fA = run0 + 2 * p;
        const float mA = fA < f1 ? 1.f : 0.f, mB = fA + 1 < f1 ? 1.f : 0.f;
        load_frames<N, T>(r, g, xr, xt, fA * HOP - HS, t, Ni);
        C x[16];
        // ---- windowed frames A (lane 0) and B = A + 1 (lane 1): sample slot q of B is slot q + 4 of A
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const float w = __ldg(window + t + q * T);
            const float wa = w * mA, wb = w * mB;
            x[q].re = mk(r[q] * wa, r[q + 4] * wb);
            x[q].im = mk(g[q] * wa, g[q + 4] * wb);
        }
        // ---- forward transform of both frames; the last stage stays in registers
        stage_compute_store<LG, 0, false>(x, gbuf, t, tw);
        gsync<T>(grp);
        stage_load<LG, 1>(x, gbuf, t);
        if (P::STAGES == 3) {
            gsync<T>(grp);
            stage_compute_store<LG, 1, false>(x, gbuf, t, tw);
            gsync<T>(grp);
            stage_load<LG, 2>(x, gbuf, t);
            stage_compute_regs<LG, 2, false>(x, t, tw);
        } else {
            stage_compute_regs<LG, 1, false>(x, t, tw);
        }
        gsync<T>(grp);                                            // every load of the last stage is done
        // ---- mirror exchange: slot q >= 8 holds bin t + qT >= n_fft/2; park it at index (bin - n_fft/2)
#pragma unroll
        for (int q = 8; q < 16; ++q) gbuf[(q - 8) * T + t] = to_e(x[slot_of_q<LG>(q)]);
        gsync<T>(grp);
        // ---- per bin k = t + qT (q < 8; thread 0 also takes k = n_fft/2): loss terms and gradient spectra
        V zi[16];
        const V own = mk(mA, mB);
        bin_math<LG, GRAD, 0>(x, zi, gbuf, ex2, t, own, rs2, kc, lin, lgs);
        bin_math<LG, GRAD, 1>(x, zi, gbuf, ex2, t, own, rs2, kc, lin, lgs);
        bin_math<LG, GRAD, 2>(x, zi, gbuf, ex2, t, own, rs2, kc, lin, lgs);
        bin_math<LG, GRAD, 3>(x, zi, gbuf, ex2, t, own, rs2, kc, lin, lgs);
        bin_math<LG, GRAD, 4>(x, zi, gbuf, ex2, t, own, rs2, kc, lin, lgs);
        bin_math<LG, GRAD, 5>(x, zi, gbuf, ex2, t, own, rs2, kc, lin, lgs);
        bin_math<LG, GRAD, 6>(x, zi, gbuf, ex2, t, own, rs2, kc, lin, lgs);
        bin_math<LG, GRAD, 7>(x, zi, gbuf, ex2, t, own, rs2, kc, lin, lgs);
        if (t == 0) bin_math<LG, GRAD, 8>(x, zi, gbuf, ex2, t, own, rs2, kc, lin, lgs);
        gsync<T>(grp);                                            // mirror bins read; gradient mirror bins written
        if (GRAD) {
#pragma unroll
            for (int q = 8; q < 16; ++q) zi[q] = zfft::from_f2(ex2[(q - 8) * T + t]);
            // ---- inverse transform of U_A + i U_B, (re, im) in the lanes: one transform per thread here
            zfft::stage_compute_store<LG, 0, true>(zi, ibuf, t, tw);
            gsync<T>(grp);
            zfft::stage_load<LG, 1>(zi, ibuf, t);
            if (P::STAGES == 3) {
                gsync<T>(grp);
                zfft::stage_compute_store<LG, 1, true>(zi, ibuf, t, tw);
                gsync<T>(grp);
                zfft::stage_load<LG, 2>(zi, ibuf, t);
                gsync<T>(grp);                                    // the next pair's first stage reuses the buffer
                zfft::stage_compute_regs<LG, 2, true>(zi, t, tw);
            } else {
                gsync<T>(grp);
                zfft::stage_compute_regs<LG, 1, true>(zi, t, tw);
            }
            // ---- overlap-add in registers.  Slot s of this pair is padded position fA*HOP + t + s*T: the carry of
            // the run's earlier frames (slots 0..11), then frame A (slots 0..15), then frame B (slots 4..19): every
            // position sums its frames oldest first.  Slots 0..7 are finished, 8..19 are carried to the next pair.
            float acc[20];
            {
                const float4 c0 = cpriv[tid], c1 = cpriv[kThreads + tid], c2 = cpriv[2 * kThreads + tid];
                acc[0] = c0.x; acc[1] = c0.y; acc[2] = c0.z; acc[3] = c0.w;
                acc[4] = c1.x; acc[5] = c1.y; acc[6] = c1.z; acc[7] = c1.w;
                acc[8] = c2.x; acc[9] = c2.y; acc[10] = c2.z; acc[11] = c2.w;
#pragma unroll
                for (int s = 12; s < 20; ++s) acc[s] = 0.f;
            }
            float ub[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const float2 v = zfft::to_f2(zi[slot_of_q<LG>(q)]);
                const float w = __ldg(window + t + q * T);
                acc[q] = fmaf(w, v.x, acc[q]);
                ub[q] = w * v.y;
            }
#pragma unroll
            for (int q = 0; q < 16; ++q) acc[q + 4] += ub[q];
            // (the run's first 12 slots still miss the previous run's tail: fixed up at the end of the tile)
            float *Pp = Pb + (size_t)fA * HOP + t;
#pragma unroll
            for (int s = 0; s < 8; ++s) Pp[s * T] = acc[s];
            cpriv[tid] = make_float4(acc[8], acc[9], acc[10], acc[11]);
            cpriv[kThreads + tid] = make_float4(acc[12], acc[13], acc[14], acc[15]);
            cpriv[2 * kThreads + tid] = make_float4(acc[16], acc[17], acc[18], acc[19]);
        }
    }
    if (GRAD) {
        // ---- run boundaries: the first 3 hops of a run also get the final carry of the previous group's run (a
        // read-modify-write of this thread's own earlier stores; a run that was skipped has nothing there yet); the
        // last group's carry belongs to the head of the next tile (or to the end of the signal): halo buffer
        __syncthreads();
        if (grp > 0) {
            float *Pp = Pb + (size_t)run0 * HOP + t;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const float4 c = cpriv[k * kThreads + tid - T];
                float4 h = make_float4(0.f, 0.f, 0.f, 0.f);
                if (active) {
                    h.x = Pp[(4 * k + 0) * T]; h.y = Pp[(4 * k + 1) * T];
                    h.z = Pp[(4 * k + 2) * T]; h.w = Pp[(4 * k + 3) * T];
                }
                Pp[(4 * k + 0) * T] = h.x + c.x;
                Pp[(4 * k + 1) * T] = h.y + c.y;
                Pp[(4 * k + 2) * T] = h.z + c.z;
                Pp[(4 * k + 3) * T] = h.w + c.w;
            }
        }
        if (grp == G - 1) {
            float *Hb = ws + sc.h_off + ((size_t)b * sc.tiles + tile) * (3 * HOP) + t;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const float4 c = cpriv[k * kThreads + tid];
                Hb[(4 * k + 0) * T] = c.x;
                Hb[(4 * k + 1) * T] = c.y;
                Hb[(4 * k + 2) * T] = c.z;
                Hb[(4 * k + 3) * T] = c.w;
            }
        }
    }
    float l0, l1, g0, g1;
    get(lin, l0, l1);
    get(lgs, g0, g1);
    const float lsum = ddsp_warp_sum(l0 + l1);
    const float gsum = ddsp_warp_sum((g0 + g1) * 0.69314718055994530942f);
    if ((tid & 31) == 0) { red[0][tid >> 5] = lsum; red[1][tid >> 5] = gsum; }
    __syncthreads();
    if (tid == 0) {
        float a = 0.f, c = 0.f;
#pragma unroll
        for (int i = 0; i < kThreads / 32; ++i) { a += red[0][i]; c += red[1][i]; }
        float *pp = partial + 2 * (sc.part_off + (size_t)tile * B + b);
        pp[0] = a;
        pp[1] = c;
    }
}

template <bool GRAD>
__global__ void __launch_bounds__(kThreads, 2)
mss_fused_kernel(const float *__restrict__ target, const float *__restrict__ rec, float *__restrict__ ws,
                 float *__restrict__ partial, const __grid_constant__ FusedArgs a) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int item = blockIdx.x;
    int si = 0;
#pragma unroll
    for (int i = 1; i < kMaxScales; ++i)
        if (i < a.n_scales && item >= a.sc[i].item0) si = i;
    const ScaleDesc &sc = a.sc[si];
    const int local = item - sc.item0;
    const int tile = local / a.B, b = local - tile * a.B;
    const int Ni = (int)a.N;
    switch (sc.lg) {
        case 6: tile_body<6, GRAD>(sc, b, tile, a.B, Ni, target, rec, ws, partial, smem); break;
        case 7: tile_body<7, GRAD>(sc, b, tile, a.B, Ni, target, rec, ws, partial, smem); break;
        case 8: tile_body<8, GRAD>(sc, b, tile, a.B, Ni, target, rec, ws, partial, smem); break;
        case 9: tile_body<9, GRAD>(sc, b, tile, a.B, Ni, target, rec, ws, partial, smem); break;
        case 10: tile_body<10, GRAD>(sc, b, tile, a.B, Ni, target, rec, ws, partial, smem); break;
        case 11: tile_body<11, GRAD>(sc, b, tile, a.B, Ni, target, rec, ws, partial, smem); break;
        default: tile_body<12, GRAD>(sc, b, tile, a.B, Ni, target, rec, ws, partial, smem); break;
    }
}

// value of scale s' padded gradient at padded position i (0 outside what the tiles produced); W = 1 or 4 consecutive
// positions (i % 4 == 0: they share the frame slot, so one decision serves all four)
template <int W> struct Vec;
template <> struct Vec<1> {
    float v;
    __device__ __forceinline__ static Vec zero() { return Vec{0.f}; }
    __device__ __forceinline__ static Vec load(const float *p) { return Vec{__ldg(p)}; }
    __device__ __forceinline__ void add(const Vec &o) { v += o.v; }
};
template <> struct Vec<4> {
    float4 v;
    __device__ __forceinline__ static Vec zero() { return Vec{make_float4(0.f, 0.f, 0.f, 0.f)}; }
    __device__ __forceinline__ static Vec load(const float *p) { return Vec{__ldg(reinterpret_cast<const float4 *>(p))}; }
    __device__ __forceinline__ void add(const Vec &o) { v.x += o.v.x; v.y += o.v.y; v.z += o.v.z; v.w += o.v.w; }
};

template <int W>
__device__ __forceinline__ Vec<W> padded_grad(const ScaleDesc &sc, const float *__restrict__ ws, int b, int i) {
    const int lh = sc.lg - 2;
    const int fi = i >> lh, n0 = i & (sc.hop - 1);
    const int tl = fi >> sc.ft_log, within = fi & ((1 << sc.ft_log) - 1);
    Vec<W> v = Vec<W>::zero();
    if (fi >= sc.frames + 3) return v;               // past the last frame's tail: nothing was written there
    if (fi < sc.last_end) v = Vec<W>::load(ws + sc.p_off + (size_t)b * sc.rowlen + i);
    if (tl >= 1 && tl < sc.tiles && within < 3)
        v.add(Vec<W>::load(ws + sc.h_off + ((size_t)b * sc.tiles + (tl - 1)) * (3 * sc.hop) + within * sc.hop + n0));
    if (fi >= sc.last_end && fi < sc.last_end + 3)
        v.add(Vec<W>::load(ws + sc.h_off + ((size_t)b * sc.tiles + (sc.tiles - 1)) * (3 * sc.hop) + (fi - sc.last_end) * sc.hop + n0));
    return v;
}

// reflect-padding contributions to sample m, all scales (only samples within n_fft/2 of either end have any)
__device__ __forceinline__ float reflected_grad(const FusedArgs &a, const float *__restrict__ ws, int b, int m, int N) {
    float acc = 0.f;
    for (int k = 0; k < a.n_scales; ++k) {
        const ScaleDesc &sc = a.sc[k];
        const int hs = 2 * sc.hop;
        if (m >= 1 && m <= hs) acc += padded_grad<1>(sc, ws, b, hs - m).v;                           // left pad
        if (m <= N - 2 && m >= N - 1 - hs) acc += padded_grad<1>(sc, ws, b, 2 * (N - 1) - m + hs).v;  // right pad
    }
    return acc;
}

struct FinArgs2 {
    int n_scales;
    long long off[kMaxScales], cnt[kMaxScales];
    float inv[kMaxScales];
};

// loss = sum over scales of inv[scale] * (sum of that scale's partial pairs), by ONE block in double, fixed order
__device__ __forceinline__ void finalize_loss(const float *__restrict__ partial, float *__restrict__ loss,
                                              const FinArgs2 &fa) {
    __shared__ double red[32];
    double acc = 0.0;
    for (int i = 0; i < fa.n_scales; ++i) {
        const float *p = partial + 2 * fa.off[i];
        double s = 0.0;
        for (long long j = threadIdx.x; j < fa.cnt[i]; j += blockDim.x) s += (double)p[2 * j] + (double)p[2 * j + 1];
        acc += s * (double)fa.inv[i];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
        double v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (threadIdx.x == 0) loss[0] = (float)v;
    }
}

__global__ void __launch_bounds__(1024)
mss_finalize2_kernel(const float *__restrict__ partial, float *__restrict__ loss, const __grid_constant__ FinArgs2 fa) {
    finalize_loss(partial, loss, fa);
}

// d_rec[b, m] = sum over scales (fixed order) of the padded gradient at m + n_fft/2, then the reflections; one extra
// block reduces the loss partials (saves a launch on the critical path of the training step)
template <int W>
__global__ void __launch_bounds__(256)
mss_combine2_kernel(const float *__restrict__ ws, float *__restrict__ d_rec, const __grid_constant__ FusedArgs a,
                    int hs_max, const float *__restrict__ partial, float *__restrict__ loss,
                    const __grid_constant__ FinArgs2 fa) {
    if (blockIdx.x == gridDim.x - 1) {                  // the extra block (uniform branch)
        if (blockIdx.y == 0) finalize_loss(partial, loss, fa);
        return;
    }
    const int b = blockIdx.y;
    const int N = (int)a.N;
    for (int m = (blockIdx.x * blockDim.x + threadIdx.x) * W; m < N; m += (gridDim.x - 1) * blockDim.x * W) {
        Vec<W> acc = Vec<W>::zero();
        for (int k = 0; k < a.n_scales; ++k) acc.add(padded_grad<W>(a.sc[k], ws, b, m + 2 * a.sc[k].hop));
        const bool edge = m <= hs_max || m + W - 1 >= N - 1 - hs_max;
        if (W == 1) {
            float v = reinterpret_cast<float &>(acc);
            if (edge) v += reflected_grad(a, ws, b, m, N);
            d_rec[(size_t)b * N + m] = v;
        } else {
            float4 v = reinterpret_cast<float4 &>(acc);
            if (edge) {
                v.x += reflected_grad(a, ws, b, m, N);
                v.y += reflected_grad(a, ws, b, m + 1, N);
                v.z += reflected_grad(a, ws, b, m + 2, N);
                v.w += reflected_grad(a, ws, b, m + 3, N);
            }
            *reinterpret_cast<float4 *>(d_rec + (size_t)b * N + m) = v;
        }
    }
}

// ---- host-side plan ------------------------------------------------------------------------------------
struct Plan2 {
    FusedArgs args;
    FinArgs2 fin;
    long long ws_floats, partial_pairs;
    size_t smem;
};

int make_plan(int B, int64_t N, const int *scales, int n_scales, Plan2 *out) {
    if (B < 1 || n_scales < 1 || n_scales > kMaxScales || N >= (1ll << 30)) return DDSP_B200_EINVAL;
    FusedArgs &a = out->args;
    a.n_scales = n_scales;
    a.B = B;
    a.N = N;
    out->fin.n_scales = n_scales;
    long long off = 0, pairs = 0;
    int item = 0, max_hop = 0;
    // about 16 tiles per resident CTA slot in total, shared evenly by the scales (their work is about equal)
    const long long per_slot = 16;           // measured: 4..32 are within 2 % of each other at batch 64
    const long long want_tiles = ddsp_ceil_div(per_slot * 2 * DDSP_SM_COUNT, (long long)n_scales * B);
    for (int i = 0; i < n_scales; ++i) {
        const int s = scales[i];
        if (s < 64 || s > 4096 || (s & (s - 1))) return DDSP_B200_EUNSUPPORTED;
        if (N <= s / 2) return DDSP_B200_EUNSUPPORTED;               // reflect padding needs pad < N
        ScaleDesc &d = a.sc[i];
        d.lg = 0;
        while ((1 << d.lg) < s) ++d.lg;
        d.hop = s / 4;
        d.frames = 1 + (int)(N / d.hop);
        const int groups = kThreads / (s / 16);                      // thread groups per CTA = runs per tile
        int ft_log = 2;                                              // a run is >= 4 frames (two pairs: head + carry logic)
        while ((1 << ft_log) < 4 * groups) ++ft_log;
        while ((1 << (ft_log + 1)) <= d.frames && ddsp_ceil_div(d.frames, 1 << ft_log) > want_tiles) ++ft_log;
        d.ft_log = ft_log;
        d.tiles = (int)ddsp_ceil_div(d.frames, 1 << ft_log);
        d.item0 = item;
        item += d.tiles * B;
        d.last_end = d.tiles << ft_log;                              // every tile writes all of its FT hops
        long long rl = (long long)d.last_end * d.hop;
        if (rl < N + s) rl = N + s;
        d.rowlen = (int)((rl + 3) & ~3ll);
        d.p_off = off;
        off += (long long)B * d.rowlen;
        d.h_off = off;
        off += (long long)B * d.tiles * 3 * d.hop;
        d.part_off = pairs;
        pairs += (long long)d.tiles * B;
        d.inv_cnt = 1.0f / ((float)B * (float)(s / 2 + 1) * (float)d.frames);
        d.window = nullptr;
        d.tw = nullptr;
        d.pad_ = 0;
        out->fin.off[i] = d.part_off;
        out->fin.cnt[i] = (long long)d.tiles * B;
        out->fin.inv[i] = d.inv_cnt;
        if (d.hop > max_hop) max_hop = d.hop;
    }
    a.n_items = item;
    a.pad_ = 0;
    out->ws_floats = off;
    out->partial_pairs = pairs;
    out->smem = (size_t)kWorkBytes + 3 * kThreads * sizeof(float4);       // + the private overlap-add carry strip
    return DDSP_B200_OK;
}

}  // namespace

extern "C" int ddsp_b200_mss_fused_supported(const int *scales, const int *hops, int n_scales) {
    if (!scales || !hops || n_scales < 1 || n_scales > kMaxScales) return 0;
    for (int i = 0; i < n_scales; ++i)
        if (scales[i] < 64 || scales[i] > 4096 || (scales[i] & (scales[i] - 1)) || hops[i] * 4 != scales[i]) return 0;
    return 1;
}

extern "C" int ddsp_b200_mss_fused_sizes(int B, int64_t N, const int *scales, int n_scales, int64_t *workspace_floats,
                                         int64_t *partial_floats) {
    DDSP_REQUIRE(scales && workspace_floats && partial_floats);
    Plan2 p;
    int s = make_plan(B, N, scales, n_scales, &p);
    if (s) return s;
    *workspace_floats = p.ws_floats;
    *partial_floats = 2 * p.partial_pairs;
    return DDSP_B200_OK;
}

// The plan of one scale, for hosts that size buffers themselves and for the CPU test of the tile / run bookkeeping
// (tests/test_abi_cpu.py): out = {frames, hop, frames per tile, tiles per voice, thread groups per CTA, frames per run,
// first frame slot past the last tile, floats per voice of the gradient plane}.
extern "C" int ddsp_b200_mss_fused_plan(int B, int64_t N, const int *scales, int n_scales, int which, int64_t *out8) {
    DDSP_REQUIRE(scales && out8 && which >= 0 && which < n_scales);
    Plan2 p;
    int s = make_plan(B, N, scales, n_scales, &p);
    if (s) return s;
    const ScaleDesc &d = p.args.sc[which];
    const int groups = kThreads / (scales[which] / 16);
    out8[0] = d.frames;
    out8[1] = d.hop;
    out8[2] = 1ll << d.ft_log;
    out8[3] = d.tiles;
    out8[4] = groups;
    out8[5] = (1ll << d.ft_log) / groups;
    out8[6] = d.last_end;
    out8[7] = d.rowlen;
    return DDSP_B200_OK;
}

extern "C" int ddsp_b200_mss_fused(const float *target, const float *rec, const float *windows,
                                   const float *const *stage_twiddles, float *workspace, float *partial,
                                   float *d_rec, float *loss, int B, int64_t N, const int *scales, int n_scales,
                                   void *stream) {
    DDSP_REQUIRE(target && rec && windows && stage_twiddles && partial && loss && scales);
    DDSP_REQUIRE(!d_rec || workspace);
    DDSP_REQUIRE(B <= 65535);
    Plan2 p;
    int s = make_plan(B, N, scales, n_scales, &p);
    if (s) return s;
    int64_t woff = 0;
    for (int i = 0; i < n_scales; ++i) {
        DDSP_REQUIRE(stage_twiddles[i]);
        p.args.sc[i].window = windows + woff;
        p.args.sc[i].tw = reinterpret_cast<const float2 *>(stage_twiddles[i]);
        woff += scales[i];
    }
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e;
    if (d_rec) {
        if ((e = cudaFuncSetAttribute(mss_fused_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem)) != cudaSuccess)
            return (int)e;
        // two CTAs of 80 KB per SM: ask for the 164 KB shared-memory configuration, which leaves 64 KB of L1 for the
        // sample re-reads, the window and the stage twiddles (48 KB of tables at n_fft 4096)
        cudaFuncSetAttribute(mss_fused_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout,
                             72);
        mss_fused_kernel<true><<<p.args.n_items, kThreads, p.smem, st>>>(target, rec, workspace, partial, p.args);
    } else {
        if ((e = cudaFuncSetAttribute(mss_fused_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem)) != cudaSuccess)
            return (int)e;
        cudaFuncSetAttribute(mss_fused_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, 72);
        mss_fused_kernel<false><<<p.args.n_items, kThreads, p.smem, st>>>(target, rec, workspace, partial, p.args);
    }
    if ((s = ddsp_launch_status())) return s;
    if (!d_rec) {
        mss_finalize2_kernel<<<1, 1024, 0, st>>>(partial, loss, p.fin);
        return ddsp_launch_status();
    }
    int hs_max = 0;
    for (int i = 0; i < n_scales; ++i) hs_max = scales[i] / 2 > hs_max ? scales[i] / 2 : hs_max;
    // grid.x - 1 blocks of samples per voice + one block column whose first block reduces the loss
    if ((N & 3) == 0) {
        int gx = (int)ddsp_ceil_div(N / 4, 256);
        if (gx > 64) gx = 64;
        mss_combine2_kernel<4><<<dim3(gx + 1, B), 256, 0, st>>>(workspace, d_rec, p.args, hs_max, partial, loss, p.fin);
    } else {
        int gx = (int)ddsp_ceil_div(N, 256);
        if (gx > 64) gx = 64;
        mss_combine2_kernel<1><<<dim3(gx + 1, B), 256, 0, st>>>(workspace, d_rec, p.args, hs_max, partial, loss, p.fin);
    }
    return ddsp_launch_status();
}
