// VAE-side spectral kernel of the Audio-CALM front-end family: short-time Fourier magnitudes over the TIME axis of log-mel
// features, as AcousticVAE._stft_mag computes them for the multi-resolution STFT loss (reference models/modeling_vae.py:271-305:
// torch.stft(n_fft in {256, 128, 64}, hop n_fft / 4, periodic Hann, center=False, onesided) followed by torch.abs).
//
// One launch per resolution replaces reshape + torch.stft (framing copy, window multiply, cuFFT R2C) + abs.  A CTA stages a few
// rows [T] in shared memory once, packs every two frames (of any of its rows) into one complex FFT of n_fft = 32 R points -- R
// lanes per transform, each running the packed-FFMA2 in-register FFT-32 of the log-mel kernel (acb_fft32.cuh) over its stride-R
// samples, a twiddle, and an R-point FFT across the R lanes through a small shared-memory exchange -- separates the two real
// spectra, takes the magnitudes and writes them straight into the rows' [n_freq][frames] blocks (the 4-byte stores of a row block
// merge in L2; staging them in shared memory halved the resident CTAs and was 40 % slower).  HBM traffic is one read of the
// features and one write of the magnitudes.
#include "audiocalm_b200.h"
#include "acb_fft32.cuh"

#include <cuda_runtime.h>

#include <algorithm>
#include <string>

namespace acb {
int fail(int code, const std::string& msg);   // acb_kernels.cu: sets the thread-local message behind acb_last_error()
}

namespace acb_spectral {

using namespace acb;

constexpr int kThreads = 128;
constexpr int kStftRowsPerCta = 32;          // rows staged per CTA (upper bound)
constexpr int kStftComplexFramesPerCta = 4;  // frames per CTA of the complex STFT (Griffin-Lim), upper bound
constexpr int kIstftFramesPerCta = 4;        // frames per CTA of the inverse STFT, upper bound
constexpr int kStftBwdRowsPerCta = 16;       // rows per CTA of the backward kernel

// sqrt / reciprocal sqrt as ONE special-function instruction each (about 1 ulp / 2 ulp; the correctly rounded sqrtf and the IEEE
// division are 8-10 instructions apiece, paid twice per bin): the parity tolerance of these kernels is 1e-4 of the magnitudes
__device__ __forceinline__ float sqrt_fast(float x) {
    float y;
    asm("sqrt.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// Bank swizzle of the staged rows.  The R lanes of a group read samples base + R j + r (j = 0..31), and the 32 / R groups of a warp work on
// frames whose bases differ by multiples of the hop (8 R floats for hop = n_fft / 4) -- a multiple of 16, 32 or 64 banks: unswizzled,
// every sample load of the forward transform was an 8-way (R = 2, 4) or 4-way (R = 8) bank conflict.  XOR-ing the index of the
// 2^s-float block a sample lies in into bits [log2 R, 5) of its position spreads the groups over all 32 banks and keeps 16-byte
// groups together (R = 2 swaps their halves).  swz() is a bijection on indices (high bits into low bits only).
template <int R>
struct Swz {
    static constexpr int kL = ilog2(R);
    static constexpr int kS = R == 2 ? 5 : 3 + ilog2(R);
    static constexpr int kHm = R == 2 ? 7 : (R >= 32 ? 0 : 32 / R - 1);
    static __device__ __forceinline__ int mask_of(int n) { return ((n >> kS) & kHm) << kL; }
    static __device__ __forceinline__ int at(int n) { return n ^ mask_of(n); }
};

// Stage `n` floats of `src` at the swizzled positions of s_x (16-byte accesses when the source allows)
template <int R>
__device__ __forceinline__ void stage_rows_swizzled(float* s_x, const float* __restrict__ src, int n, int tid) {
    if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) {
        for (int i = tid; i < n / 4; i += kThreads) {
            float4 v = __ldg(reinterpret_cast<const float4*>(src) + i);
            const int p = Swz<R>::at(4 * i);
            if (p & 2) v = make_float4(v.z, v.w, v.x, v.y);          // R = 2: the halves of the group trade places
            *reinterpret_cast<float4*>(s_x + (p & ~3)) = v;
        }
        for (int i = (n & ~3) + tid; i < n; i += kThreads) s_x[Swz<R>::at(i)] = src[i];
    } else {
        for (int i = tid; i < n; i += kThreads) s_x[Swz<R>::at(i)] = src[i];
    }
}

// The windowed samples of one frame pair in the packed, bit-reversed register order fft32_packed takes (position q holds elements
// j0 = brev5(q) and j0 + 1 of the lane's stride-R sequence): frame a in pr, frame b in pi.  `blocked`: every frame starts on a multiple
// of 8 R floats, so the 8 R samples of a block share one swizzle mask (one XOR per load); frame b = frame a one hop later in the same
// row (the usual pair, hop = 8 R) then needs only 8 loads of its own: its sample j is frame a's sample j + 8.
template <int R>
__device__ __forceinline__ void load_pair_windowed(const float* s_x, int base_a, int base_b, bool valid_b, bool blocked, int r, const float (&wreg)[32],
                                                   float2 (&pr)[16], float2 (&pi)[16]) {
    const bool shared_loads = blocked && valid_b && base_b == base_a + 8 * R;       // group-uniform
    if (shared_loads) {
        float raw[40];
#pragma unroll
        for (int c = 0; c < 5; ++c) {
            const int t_c = base_a + 8 * R * c;
            const float* q_c = s_x + t_c + r;
            const int m_c = Swz<R>::mask_of(t_c);
#pragma unroll
            for (int u = 0; u < 8; ++u) raw[8 * c + u] = q_c[(R * u) ^ m_c];
        }
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const int j0 = brev5(q);
            pr[q] = make_float2(raw[j0] * wreg[2 * q], raw[j0 + 1] * wreg[2 * q + 1]);
            pi[q] = make_float2(raw[j0 + 8] * wreg[2 * q], raw[j0 + 9] * wreg[2 * q + 1]);
        }
    } else if (blocked) {                       // two unrelated frames (pairs across rows): per-block masks for each of them
        float ra[32], rb[32];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int ta = base_a + 8 * R * c, tb = base_b + 8 * R * c;
            const float* qa_c = s_x + ta + r;
            const float* qb_c = s_x + tb + r;
            const int ma = Swz<R>::mask_of(ta), mb = Swz<R>::mask_of(tb);
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                ra[8 * c + u] = qa_c[(R * u) ^ ma];
                rb[8 * c + u] = valid_b ? qb_c[(R * u) ^ mb] : 0.f;
            }
        }
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const int j0 = brev5(q);
            pr[q] = make_float2(ra[j0] * wreg[2 * q], ra[j0 + 1] * wreg[2 * q + 1]);
            pi[q] = make_float2(rb[j0] * wreg[2 * q], rb[j0 + 1] * wreg[2 * q + 1]);
        }
    } else {
#pragma unroll
        for (int q = 0; q < 16; ++q) {
            const int j0 = brev5(q);
            const int n0 = R * j0 + r, n1 = R * (j0 + 1) + r;
            pr[q] = make_float2(s_x[Swz<R>::at(base_a + n0)] * wreg[2 * q], s_x[Swz<R>::at(base_a + n1)] * wreg[2 * q + 1]);
            pi[q] = valid_b ? make_float2(s_x[Swz<R>::at(base_b + n0)] * wreg[2 * q], s_x[Swz<R>::at(base_b + n1)] * wreg[2 * q + 1])
                            : make_float2(0.f, 0.f);
        }
    }
}

struct SpectralSmem {
    int x, win, tw, buf, total_bytes;
};

__host__ __device__ inline SpectralSmem spectral_smem(int R, int rows_per_cta, int T) {
    const int N = 32 * R;
    SpectralSmem L;
    int off = 0;   // 4-byte words
    L.x = off; off += (rows_per_cta * T + 255) & ~255;           // the swizzle permutes inside aligned 256-float blocks
    L.win = off; off += N;
    L.tw = off; off += 2 * N;
    L.buf = off; off += (kThreads / R) * (2 * 33 * R);           // per lane group: N complex values, index k1 + 33 * k2
    L.total_bytes = off * 4;
    return L;
}

template <int R>
__global__ void __launch_bounds__(kThreads) stft_mag_kernel(const float* __restrict__ x, long long rows, int T, int hop, int n_frames,
                                                            const float* __restrict__ window, float* __restrict__ out, int rows_per_cta) {
    constexpr int N = 32 * R, kFreq = N / 2 + 1, kGroups = kThreads / R, kPerLane = 32 / R;
    extern __shared__ __align__(16) float smem[];
    const SpectralSmem L = spectral_smem(R, rows_per_cta, T);
    float* s_x = smem + L.x;
    float* s_win = smem + L.win;
    float2* s_tw = reinterpret_cast<float2*>(smem + L.tw);
    const int tid = threadIdx.x;
    const long long row0 = (long long)blockIdx.x * rows_per_cta;
    const int n_rows = (int)min((long long)rows_per_cta, rows - row0);

    // stage the rows (bank-swizzled), the window and the twiddles W_N^m = exp(-2 pi i m / N)
    {
        stage_rows_swizzled<R>(s_x, x + row0 * T, n_rows * T, tid);
        for (int i = tid; i < N; i += kThreads) {
            s_win[i] = window[i];
            float sn, cs;
            sincospif(2.f * (float)((i % R) * (i / R)) / (float)N, &sn, &cs);      // entry [k = i / R][r = i % R] = W_N^(r k)
            s_tw[i] = make_float2(cs, -sn);
        }
    }
    __syncthreads();

    const int g = tid / R, r = tid % R;                 // lane group (one transform) and position inside it
    float2* buf = reinterpret_cast<float2*>(smem + L.buf) + g * (33 * R);
    const int total_frames = n_rows * n_frames;
    const int n_items = (total_frames + 1) / 2;         // two frames per complex transform
    const int n_iter = (n_items + kGroups - 1) / kGroups;
    // every frame starts on a multiple of 8 R floats: the 8 R samples of a block share one swizzle mask (one XOR per load)
    const bool blocked = R < 32 && T % (8 * R) == 0 && hop % (8 * R) == 0;
    float wreg[32];                                     // this lane's window values, bit-reversed pair order (loop-invariant)
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        wreg[2 * q] = s_win[R * brev5(q) + r];
        wreg[2 * q + 1] = s_win[R * (brev5(q) + 1) + r];
    }
    for (int it = 0; it < n_iter; ++it) {
        const int item = it * kGroups + g;
        const bool valid = item < n_items;
        const int qa = 2 * item, qb = qa + 1;
        const bool valid_b = valid && qb < total_frames;
        const int row_a = valid ? qa / n_frames : 0, fa = valid ? qa - row_a * n_frames : 0;
        const int row_b = valid_b ? qb / n_frames : 0, fb = valid_b ? qb - row_b * n_frames : 0;
        if (valid) {
            const int base_a = row_a * T + fa * hop, base_b = row_b * T + fb * hop;
            float2 pr[16], pi[16];
            load_pair_windowed<R>(s_x, base_a, base_b, valid_b, blocked, r, wreg, pr, pi);
            group_fft_stage1<R>(pr, pi, buf, s_tw, r);
        }
        __syncwarp();
        if (valid) group_fft_stage2<R>(buf, r);
        __syncwarp();
        if (valid) {                                    // separate the two real spectra, magnitudes
            float* obase = out + row0 * kFreq * n_frames;
            float* oa = obase + (size_t)row_a * kFreq * n_frames + fa;
            float* ob = obase + (size_t)row_b * kFreq * n_frames + fb;
            for (int k = r; k < kFreq; k += R) {
                const int kc = (N - k) & (N - 1);
                const float2 z = buf[(k & 31) + 33 * (k >> 5)], zc = buf[(kc & 31) + 33 * (kc >> 5)];
                const float apc = z.x + zc.x, bmd = z.y - zc.y, amc = z.x - zc.x, bpd = z.y + zc.y;
                oa[(size_t)k * n_frames] = 0.5f * sqrt_fast(fmaf(apc, apc, bmd * bmd));
                if (valid_b) ob[(size_t)k * n_frames] = 0.5f * sqrt_fast(fmaf(amc, amc, bpd * bpd));
            }
        }
        __syncwarp();
    }
}

template <int R>
static int launch(const float* x, int64_t rows, int T, int hop, int n_frames, const float* window, float* out, cudaStream_t st) {
    int dev = 0, optin = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess)
        return fail(ACB_ERR_CUDA, "acb_stft_mag: cannot query the device");
    // rows per CTA: 16 (measured best for 5-13 frames per row), doubled while a CTA's frame pairs would leave lane groups idle
    // (one frame per row at n_fft = T), halved while the footprint is large
    int rpc = (int)std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(16, kStftRowsPerCta), 16384 / T));
    while (rpc < kStftRowsPerCta && (rpc * n_frames + 1) / 2 < kThreads / R && 2 * rpc <= 16384 / T) rpc <<= 1;
    while (rpc > 1 && spectral_smem(R, rpc, T).total_bytes > std::min(optin, 160 * 1024)) rpc >>= 1;
    const SpectralSmem L = spectral_smem(R, rpc, T);
    if (L.total_bytes > optin)
        return fail(ACB_ERR_UNSUPPORTED, "acb_stft_mag: a row of " + std::to_string(T) + " frames does not fit in shared memory");
    cudaError_t e = cudaFuncSetAttribute(stft_mag_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin);
    if (e != cudaSuccess) return fail(ACB_ERR_CUDA, std::string("acb_stft_mag: ") + cudaGetErrorString(e));
    const unsigned grid = (unsigned)((rows + rpc - 1) / rpc);
    stft_mag_kernel<R><<<grid, kThreads, L.total_bytes, st>>>(x, rows, T, hop, n_frames, window, out, rpc);
    e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ACB_ERR_CUDA, std::string("acb_stft_mag launch: ") + cudaGetErrorString(e));
    return ACB_OK;
}

// Backward of stft_mag: grad_x[row][n] = sum over the frames that cover n of w * Re( sum_k g[k] conj(X[k] / |X[k]|) e^(-2 pi i k n' / N) ).
// Per pair of frames: the forward transform again (X is not kept), then ONE more complex FFT of the same size: the one-sided
// sums of both frames are the real and the imaginary part of the transform of H_A + i H_B, where H is the Hermitian extension of
// h[k] = g[k] conj(X[k]) / |X[k]| (a bin with |X| = 0 passes no gradient, like torch's abs).  The windowed results are accumulated
// in a shared-memory copy of the rows' gradients (frames overlap: shared-memory atomics) and written out once.
struct SpectralBwdSmem {
    int x, gx, g, win, tw, buf, total_bytes;
};
__host__ __device__ inline SpectralBwdSmem spectral_bwd_smem(int R, int rows_per_cta, int T, int n_frames) {
    const int N = 32 * R, n_freq = N / 2 + 1;
    SpectralBwdSmem L;
    int off = 0;
    L.x = off; off += (rows_per_cta * T + 255) & ~255;
    L.gx = off; off += (rows_per_cta * T + 255) & ~255;
    L.g = off; off += (rows_per_cta * n_freq * n_frames + 3) & ~3;
    L.win = off; off += N;
    L.tw = off; off += 2 * N;
    L.buf = off; off += (kThreads / R) * (2 * 33 * R);
    L.total_bytes = off * 4;
    return L;
}

template <int R>
__global__ void __launch_bounds__(kThreads) stft_mag_backward_kernel(const float* __restrict__ x, const float* __restrict__ grad_mag, long long rows, int T,
                                                                     int hop, int n_frames, const float* __restrict__ window,
                                                                     float* __restrict__ grad_x, int rows_per_cta) {
    constexpr int N = 32 * R, kFreq = N / 2 + 1, kGroups = kThreads / R;
    extern __shared__ __align__(16) float smem[];
    const SpectralBwdSmem L = spectral_bwd_smem(R, rows_per_cta, T, n_frames);
    float* s_x = smem + L.x;
    float* s_gx = smem + L.gx;
    float* s_g = smem + L.g;
    float* s_win = smem + L.win;
    float2* s_tw = reinterpret_cast<float2*>(smem + L.tw);
    const int tid = threadIdx.x;
    const long long row0 = (long long)blockIdx.x * rows_per_cta;
    const int n_rows = (int)min((long long)rows_per_cta, rows - row0);
    stage_rows_swizzled<R>(s_x, x + row0 * T, n_rows * T, tid);               // s_x and s_gx share the bank swizzle of the forward kernel
    for (int i = tid; i < ((n_rows * T + 255) & ~255); i += kThreads) s_gx[i] = 0.f;     // the swizzle permutes inside aligned blocks: clear whole blocks
    {
        const float* gsrc = grad_mag + row0 * kFreq * n_frames;
        const int n = n_rows * kFreq * n_frames;
        if ((reinterpret_cast<uintptr_t>(gsrc) & 15) == 0) {
            for (int i = tid; i < n / 4; i += kThreads) reinterpret_cast<float4*>(s_g)[i] = __ldg(reinterpret_cast<const float4*>(gsrc) + i);
            for (int i = (n & ~3) + tid; i < n; i += kThreads) s_g[i] = gsrc[i];
        } else {
            for (int i = tid; i < n; i += kThreads) s_g[i] = gsrc[i];
        }
    }
    for (int i = tid; i < N; i += kThreads) {
        s_win[i] = window[i];
        float sn, cs;
        sincospif(2.f * (float)((i % R) * (i / R)) / (float)N, &sn, &cs);      // entry [k = i / R][r = i % R] = W_N^(r k)
        s_tw[i] = make_float2(cs, -sn);
    }
    __syncthreads();

    const int g = tid / R, r = tid % R;
    float2* buf = reinterpret_cast<float2*>(smem + L.buf) + g * (33 * R);
    const int total_frames = n_rows * n_frames;
    const int n_items = (total_frames + 1) / 2;
    const int n_iter = (n_items + kGroups - 1) / kGroups;
    const bool blocked = R < 32 && T % (8 * R) == 0 && hop % (8 * R) == 0;
    float wreg[32];                                     // this lane's window values, bit-reversed pair order (loop-invariant)
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        wreg[2 * q] = s_win[R * brev5(q) + r];
        wreg[2 * q + 1] = s_win[R * (brev5(q) + 1) + r];
    }
    for (int it = 0; it < n_iter; ++it) {
        const int item = it * kGroups + g;
        const bool valid = item < n_items;
        const int qa = 2 * item, qb = qa + 1;
        const bool valid_b = valid && qb < total_frames;
        const int row_a = valid ? qa / n_frames : 0, fa = valid ? qa - row_a * n_frames : 0;
        const int row_b = valid_b ? qb / n_frames : 0, fb = valid_b ? qb - row_b * n_frames : 0;
        float2 pr[16], pi[16];
        bool live_a = false, live_b = false;            // this lane holds a nonzero windowed sample of frame a / b
        if (valid) {                                    // forward transform of the pair, as in stft_mag_kernel
            load_pair_windowed<R>(s_x, row_a * T + fa * hop, row_b * T + fb * hop, valid_b, blocked, r, wreg, pr, pi);
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                live_a |= pr[q].x != 0.f || pr[q].y != 0.f;
                live_b |= pi[q].x != 0.f || pi[q].y != 0.f;
            }
            group_fft_stage1<R>(pr, pi, buf, s_tw, r);
        }
        // A silent frame (every windowed sample 0) has X = 0 exactly and passes no gradient, as in torch.  Packed with a sounding
        // frame, the separation below leaves that frame's rounding noise in its X instead, and g conj(X) / |X| of noise is a
        // unit-sized direction: such a frame is zeroed by the group's vote rather than by |X| = 0.
        const unsigned group_bits = (R == 32 ? 0xffffffffu : (1u << (R & 31)) - 1u) << ((tid & 31) & ~(R - 1));
        const bool silent_a = (__ballot_sync(0xffffffffu, live_a) & group_bits) == 0u;
        const bool silent_b = (__ballot_sync(0xffffffffu, live_b) & group_bits) == 0u;
        __syncwarp();
        if (valid) group_fft_stage2<R>(buf, r);
        __syncwarp();
        if (valid) {                                    // h = g conj(X) / |X| per frame; C = H_A + i H_B written over Z in place
            const float* ga = s_g + (size_t)row_a * kFreq * n_frames + fa;       // staged: reading them where they lie in global memory was measured 40 % slower
            const float* gb = s_g + (size_t)row_b * kFreq * n_frames + fb;
            for (int k = r; k < kFreq; k += R) {
                const int kc = (N - k) & (N - 1);
                const float2 z = buf[buf_index(k)], zc = buf[buf_index(kc)];
                const float xar = 0.5f * (z.x + zc.x), xai = 0.5f * (z.y - zc.y);          // X_A[k]
                const float xbr = 0.5f * (z.y + zc.y), xbi = -0.5f * (z.x - zc.x);         // X_B[k]
                const float pa = fmaf(xar, xar, xai * xai), pb = fmaf(xbr, xbr, xbi * xbi);   // |X|^2; g / |X| = g * rsqrt(|X|^2)
                const float sa = (!silent_a && pa > 0.f) ? ga[(size_t)k * n_frames] * rsqrtf(pa) : 0.f;
                const float sb = (valid_b && !silent_b && pb > 0.f) ? gb[(size_t)k * n_frames] * rsqrtf(pb) : 0.f;
                const float har = sa * xar, hai = -sa * xai;                                // h_A = g conj(X_A) / |X_A|
                const float hbr = sb * xbr, hbi = -sb * xbi;
                if (k == 0 || 2 * k == N) {
                    buf[buf_index(k)] = make_float2(har, hbr);                              // Re h_A + i Re h_B
                } else {
                    buf[buf_index(k)] = make_float2(0.5f * (har - hbi), 0.5f * (hai + hbr));        // (h_A + i h_B) / 2
                    buf[buf_index(kc)] = make_float2(0.5f * (har + hbi), 0.5f * (-hai + hbr));      // (conj h_A + i conj h_B) / 2
                }
            }
        }
        __syncwarp();
        if (valid) {                                    // second transform: the lane gathers its stride-R inputs from the buffer
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const int j0 = brev5(q);
                const float2 c0 = buf[buf_index(R * j0 + r)], c1 = buf[buf_index(R * (j0 + 1) + r)];
                pr[q] = make_float2(c0.x, c1.x);
                pi[q] = make_float2(c0.y, c1.y);
            }
        }
        __syncwarp();
        if (valid) group_fft_stage1<R>(pr, pi, buf, s_tw, r);
        __syncwarp();
        if (valid) group_fft_stage2<R>(buf, r);
        __syncwarp();
        if (valid) {                                    // windowed overlap-add into the rows' gradients (a silent frame adds exactly 0,
                                                        // not the partner's rounding noise in its half of the transform)
            const int base_a = row_a * T + fa * hop, base_b = row_b * T + fb * hop;
            for (int n = r; n < N; n += R) {
                const float2 y = buf[buf_index(n)];
                const float w = s_win[n];
                if (!silent_a) atomicAdd(s_gx + Swz<R>::at(base_a + n), w * y.x);
                if (valid_b && !silent_b) atomicAdd(s_gx + Swz<R>::at(base_b + n), w * y.y);
            }
        }
        __syncwarp();
    }
    __syncthreads();
    for (int i = tid; i < n_rows * T; i += kThreads) grad_x[row0 * T + i] = s_gx[Swz<R>::at(i)];
}

template <int R>
static int launch_backward(const float* x, const float* grad_mag, int64_t rows, int T, int hop, int n_frames, const float* window, float* grad_x,
                           cudaStream_t st) {
    int dev = 0, optin = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess)
        return fail(ACB_ERR_CUDA, "acb_stft_mag_backward: cannot query the device");
    // rows per CTA: 16, or 8 when a row has many frames (measured at T = 256: 13 frames per row run 25 % faster in one pass over 8 rows than
    // in two passes over 16 with twice the shared memory)
    int rpc = (int)std::max<int64_t>(1, std::min<int64_t>(n_frames >= 8 ? kStftBwdRowsPerCta / 2 : kStftBwdRowsPerCta, 16384 / T));
    while (rpc > 1 && spectral_bwd_smem(R, rpc, T, n_frames).total_bytes > std::min(optin, 160 * 1024)) rpc >>= 1;
    const SpectralBwdSmem L = spectral_bwd_smem(R, rpc, T, n_frames);
    if (L.total_bytes > optin)
        return fail(ACB_ERR_UNSUPPORTED, "acb_stft_mag_backward: a row of " + std::to_string(T) + " frames does not fit in shared memory");
    cudaError_t e = cudaFuncSetAttribute(stft_mag_backward_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin);
    if (e != cudaSuccess) return fail(ACB_ERR_CUDA, std::string("acb_stft_mag_backward: ") + cudaGetErrorString(e));
    const unsigned grid = (unsigned)((rows + rpc - 1) / rpc);
    stft_mag_backward_kernel<R><<<grid, kThreads, L.total_bytes, st>>>(x, grad_mag, rows, T, hop, n_frames, window, grad_x, rpc);
    e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ACB_ERR_CUDA, std::string("acb_stft_mag_backward launch: ") + cudaGetErrorString(e));
    return ACB_OK;
}

// --------------------------------------------------------------------------------------------
// Griffin-Lim building blocks (the vocoder fallback of eval/eval_calm.py:184-208 -> torchaudio GriffinLim(n_fft=1024)):
// a complex STFT with centred, reflect-padded frames (torch.stft center=True) whose epilogue can apply the phase update of one
// Griffin-Lim iteration, an inverse STFT (torch.istft: inverse transform, window, overlap-add, division by the window envelope,
// centre trimmed), both on the same group FFT; long rows are cut into chunks of frames per CTA.
// --------------------------------------------------------------------------------------------
struct ChunkSmem {
    int x, spec, y, win, tw, buf, total_bytes;
};
__host__ __device__ inline ChunkSmem chunk_smem(int R, int frames_per_cta, int hop, bool with_spec) {
    const int N = 32 * R, n_freq = N / 2 + 1;
    ChunkSmem L;
    int off = 0;
    L.x = off; off += with_spec ? 0 : (((frames_per_cta - 1) * hop + N + 3) & ~3);
    L.spec = off; off += 2 * n_freq * frames_per_cta;                                   // [k][frame of the chunk] complex: istft input / stft output
    L.y = off; off += with_spec ? (((frames_per_cta - 1) * hop + N + 3) & ~3) : 0;     // istft: the chunk's overlap-added output
    L.win = off; off += N;
    L.tw = off; off += 2 * N;
    const int groups = kThreads / R, pairs = (frames_per_cta + 1) / 2;                  // lane groups beyond the chunk's frame pairs never run a transform
    L.buf = off; off += (groups < pairs ? groups : pairs) * (2 * 33 * R);
    L.total_bytes = off * 4;
    return L;
}

template <int R>
__global__ void __launch_bounds__(kThreads) stft_complex_kernel(const float* __restrict__ x, long long length, int hop, int n_frames,
                                                                const float* __restrict__ window, float2* __restrict__ spec_out,
                                                                float2* __restrict__ tprev, const float* __restrict__ mag, float momentum,
                                                                int frames_per_cta) {
    constexpr int N = 32 * R, kFreq = N / 2 + 1, kGroups = kThreads / R;
    extern __shared__ __align__(16) float smem[];
    const ChunkSmem L = chunk_smem(R, frames_per_cta, hop, false);
    float* s_x = smem + L.x;
    float2* s_spec = reinterpret_cast<float2*>(smem + L.spec);
    float* s_win = smem + L.win;
    float2* s_tw = reinterpret_cast<float2*>(smem + L.tw);
    const int tid = threadIdx.x;
    const long long row = blockIdx.y;
    const int t0 = blockIdx.x * frames_per_cta, n_loc = min(frames_per_cta, n_frames - t0);
    const float* src = x + row * length;
    {   // the chunk's samples with torch.stft's centred reflect padding
        const long long g0 = (long long)t0 * hop - N / 2;
        const int n = (n_loc - 1) * hop + N;
        for (int i = tid; i < n; i += kThreads) {
            long long idx = g0 + i;
            if (idx < 0) idx = -idx;
            if (idx >= length) idx = 2 * (length - 1) - idx;
            s_x[i] = (idx >= 0 && idx < length) ? __ldg(src + idx) : 0.f;
        }
        for (int i = tid; i < N; i += kThreads) {
            s_win[i] = window[i];
            float sn, cs;
            sincospif(2.f * (float)((i % R) * (i / R)) / (float)N, &sn, &cs);      // entry [k = i / R][r = i % R] = W_N^(r k)
            s_tw[i] = make_float2(cs, -sn);
        }
    }
    __syncthreads();
    const int g = tid / R, r = tid % R;
    float2* buf = reinterpret_cast<float2*>(smem + L.buf) + g * (33 * R);
    const int n_items = (n_loc + 1) / 2, n_iter = (n_items + kGroups - 1) / kGroups;
    for (int it = 0; it < n_iter; ++it) {
        const int item = it * kGroups + g;
        const bool valid = item < n_items;
        const int fa = 2 * item, fb = fa + 1;
        const bool valid_b = valid && fb < n_loc;
        if (valid) {
            const float* pa = s_x + fa * hop;
            const float* pb = s_x + (valid_b ? fb : fa) * hop;
            float2 pr[16], pi[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const int j0 = brev5(q);
                const int n0 = R * j0 + r, n1 = R * (j0 + 1) + r;
                const float w0 = s_win[n0], w1 = s_win[n1];
                pr[q] = make_float2(pa[n0] * w0, pa[n1] * w1);
                pi[q] = valid_b ? make_float2(pb[n0] * w0, pb[n1] * w1) : make_float2(0.f, 0.f);
            }
            group_fft_stage1<R>(pr, pi, buf, s_tw, r);
        }
        __syncwarp();
        if (valid) group_fft_stage2<R>(buf, r);
        __syncwarp();
        if (valid) {                                    // separate the two spectra into the chunk's staged output [k][frame]
            for (int k = r; k < kFreq; k += R) {
                const int kc = (N - k) & (N - 1);
                const float2 z = buf[buf_index(k)], zc = buf[buf_index(kc)];
                s_spec[k * frames_per_cta + fa] = make_float2(0.5f * (z.x + zc.x), 0.5f * (z.y - zc.y));
                if (valid_b) s_spec[k * frames_per_cta + fb] = make_float2(0.5f * (z.y + zc.y), -0.5f * (z.x - zc.x));
            }
        }
        __syncwarp();
    }
    __syncthreads();
    // one coalesced pass over the chunk's [k][frames] block: every k row is a contiguous run of the chunk's frames in global memory
    // (four elements per thread and step, all loads issued before the first store: the read-modify-write of `previous` would
    // otherwise serialise on memory latency)
    const int total = kFreq * frames_per_cta;
    for (int i0 = tid; i0 < total; i0 += 4 * kThreads) {
        size_t o[4];
        float2 v[4], prev[4];
        float m[4];
        bool ok[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * kThreads;
            const int k = i / frames_per_cta, t = i - k * frames_per_cta;
            ok[u] = i < total && t < n_loc;
            o[u] = ((size_t)row * kFreq + k) * n_frames + t0 + t;
            v[u] = ok[u] ? s_spec[i] : make_float2(0.f, 0.f);
            if (mag != nullptr && ok[u]) { prev[u] = tprev[o[u]]; m[u] = mag[o[u]]; }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (!ok[u]) continue;
            float2 w = v[u];
            if (mag != nullptr) {      // one Griffin-Lim phase update: angles = (rebuilt - m * previous) / (|.| + 1e-16); out = angles * magnitude
                tprev[o[u]] = w;
                const float ar = fmaf(-momentum, prev[u].x, w.x), ai = fmaf(-momentum, prev[u].y, w.y);
                const float inv = __fdividef(1.f, sqrt_fast(fmaf(ar, ar, ai * ai)) + 1e-16f);     // two special-function instructions instead of ~20
                w = make_float2(ar * inv * m[u], ai * inv * m[u]);
            }
            spec_out[o[u]] = w;
        }
    }
}

template <int R>
__global__ void __launch_bounds__(kThreads) istft_kernel(const float2* __restrict__ spec, int n_frames, int hop, const float* __restrict__ window,
                                                         float* __restrict__ out, long long length, int frames_per_cta) {
    constexpr int N = 32 * R, kFreq = N / 2 + 1, kGroups = kThreads / R;
    extern __shared__ __align__(16) float smem[];
    const ChunkSmem L = chunk_smem(R, frames_per_cta, hop, true);
    float2* s_spec = reinterpret_cast<float2*>(smem + L.spec);      // [k][frame of the chunk]
    float* s_win = smem + L.win;
    float2* s_tw = reinterpret_cast<float2*>(smem + L.tw);
    const int tid = threadIdx.x;
    const long long row = blockIdx.y;
    const int t0 = blockIdx.x * frames_per_cta, n_loc = min(frames_per_cta, n_frames - t0);
    for (int i = tid; i < kFreq * frames_per_cta; i += kThreads) {
        const int k = i / frames_per_cta, t = i - k * frames_per_cta;
        s_spec[i] = t < n_loc ? spec[((size_t)row * kFreq + k) * n_frames + t0 + t] : make_float2(0.f, 0.f);
    }
    for (int i = tid; i < N; i += kThreads) {
        s_win[i] = window[i];
        float sn, cs;
        sincospif(2.f * (float)((i % R) * (i / R)) / (float)N, &sn, &cs);      // entry [k = i / R][r = i % R] = W_N^(r k)
        s_tw[i] = make_float2(cs, -sn);
    }
    __syncthreads();
    const int g = tid / R, r = tid % R;
    float2* buf = reinterpret_cast<float2*>(smem + L.buf) + g * (33 * R);
    float* dst = out + row * length;
    float* s_y = smem + L.y;                            // overlap-add of the chunk's frames: shared-memory atomics, global ones only at the chunk's rims
    const int span = (n_loc - 1) * hop + N;
    for (int i = tid; i < span; i += kThreads) s_y[i] = 0.f;
    __syncthreads();
    const float inv_n = 1.f / (float)N;
    const int n_items = (n_loc + 1) / 2, n_iter = (n_items + kGroups - 1) / kGroups;
    for (int it = 0; it < n_iter; ++it) {
        const int item = it * kGroups + g;
        const bool valid = item < n_items;
        const int fa = 2 * item, fb = fa + 1;
        const bool valid_b = valid && fb < n_loc;
        if (valid) {
            // y_A + i y_B = IFFT(X_A + i X_B) = conj(FFT(conj(D))) / N with D the Hermitian extension of both one-sided spectra
            for (int k = r; k < kFreq; k += R) {
                const float2 a = s_spec[k * frames_per_cta + fa];
                const float2 b = valid_b ? s_spec[k * frames_per_cta + fb] : make_float2(0.f, 0.f);
                if (k == 0 || 2 * k == N) {
                    buf[buf_index(k)] = make_float2(a.x, -b.x);                  // irfft ignores the imaginary part of DC / Nyquist
                } else {
                    buf[buf_index(k)] = make_float2(a.x - b.y, -(a.y + b.x));
                    buf[buf_index(N - k)] = make_float2(a.x + b.y, a.y - b.x);
                }
            }
        }
        __syncwarp();
        float2 pr[16], pi[16];
        if (valid) {
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const int j0 = brev5(q);
                const float2 c0 = buf[buf_index(R * j0 + r)], c1 = buf[buf_index(R * (j0 + 1) + r)];
                pr[q] = make_float2(c0.x, c1.x);
                pi[q] = make_float2(c0.y, c1.y);
            }
        }
        __syncwarp();
        if (valid) group_fft_stage1<R>(pr, pi, buf, s_tw, r);
        __syncwarp();
        if (valid) group_fft_stage2<R>(buf, r);
        __syncwarp();
        if (valid) {                                    // window and overlap-add inside the chunk
            for (int n = r; n < N; n += R) {
                const float2 y = buf[buf_index(n)];
                const float w = s_win[n] * inv_n;
                atomicAdd(s_y + fa * hop + n, w * y.x);
                if (valid_b) atomicAdd(s_y + fb * hop + n, -w * y.y);
            }
        }
        __syncwarp();
    }
    __syncthreads();
    {   // write the chunk out, centre trimmed (torch.istft center=True): positions that the neighbouring chunks' frames also reach
        // (the first and last N - hop samples of the span) are combined with global atomics, the rest are plain stores
        const long long base = (long long)t0 * hop - N / 2;
        const int rim = N - hop;
        const bool first = t0 == 0, last = t0 + n_loc >= n_frames;
        for (int i = tid; i < span; i += kThreads) {
            const long long pos = base + i;
            if (pos < 0 || pos >= length) continue;
            if ((i < rim && !first) || (i >= span - rim && !last)) atomicAdd(dst + pos, s_y[i]);
            else dst[pos] = s_y[i];
        }
    }
}

// division by the window envelope sum_t w^2[i + N/2 - t hop] (torch.istft; positions whose envelope is below 1e-11 are left as they are)
__global__ void __launch_bounds__(256) istft_normalize_kernel(float* __restrict__ out, long long rows, long long length, int n_fft, int hop, int n_frames,
                                                              const float* __restrict__ window) {
    const long long total = rows * length;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const long long pos = i % length + n_fft / 2;
        const long long t_hi = min((long long)n_frames - 1, pos / hop);
        const long long t_lo = max(0LL, (pos - n_fft + hop) / hop);
        float env = 0.f;
        for (long long t = t_lo; t <= t_hi; ++t) {
            const long long n = pos - t * hop;
            if (n >= 0 && n < n_fft) { const float w = __ldg(window + n); env = fmaf(w, w, env); }
        }
        if (env > 1e-11f) out[i] = out[i] / env;
    }
}

// Frames per CTA of the chunked transforms (complex STFT / inverse STFT).  Measured on 32 Griffin-Lim iterations (n_fft 1024): 1 x 20 s
// 2.8 / 1.8 / 1.6 ms, 8 x 20 s 7.3 / 4.6 / 4.1 ms, 64 x 20 s 49 / 30.6 / 29.3 ms at 16 / 8 / 4 frames per CTA (16 frames leave one CTA per SM;
// the FFT of a chunk keeps only some of its warps busy, the staging and the overlap-add all of them; with the exchange buffers sized
// by the chunk's frame pairs, 4 frames are 55 KB per CTA).  The upper bound is halved while the grid would not fill the chip.
static int chunk_frames(int upper, int n_frames, int64_t rows) {
    int dev = 0, sms = 0;   // SM count of the current device (148 on a B200)
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) sms = 148;
    int fpc = std::max(2, upper);
    while (fpc > 4 && (int64_t)((n_frames + fpc - 1) / fpc) * rows < 8 * (int64_t)sms) fpc >>= 1;
    return fpc;
}

template <int R>
static int launch_stft_complex(const float* x, int64_t rows, int64_t length, int hop, int n_frames, const float* window, float2* spec, float2* tprev,
                               const float* mag, float momentum, cudaStream_t st) {
    int dev = 0, optin = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess)
        return fail(ACB_ERR_CUDA, "acb_stft_complex: cannot query the device");
    int fpc = chunk_frames(kStftComplexFramesPerCta, n_frames, rows);
    while (fpc > 2 && chunk_smem(R, fpc, hop, false).total_bytes > std::min(optin, 160 * 1024)) fpc >>= 1;
    const ChunkSmem L = chunk_smem(R, fpc, hop, false);
    if (L.total_bytes > optin) return fail(ACB_ERR_UNSUPPORTED, "acb_stft_complex: hop too large for shared memory");
    cudaError_t e = cudaFuncSetAttribute(stft_complex_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin);
    if (e != cudaSuccess) return fail(ACB_ERR_CUDA, std::string("acb_stft_complex: ") + cudaGetErrorString(e));
    const dim3 grid((unsigned)((n_frames + fpc - 1) / fpc), (unsigned)rows);
    stft_complex_kernel<R><<<grid, kThreads, L.total_bytes, st>>>(x, length, hop, n_frames, window, spec, tprev, mag, momentum, fpc);
    e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ACB_ERR_CUDA, std::string("acb_stft_complex launch: ") + cudaGetErrorString(e));
    return ACB_OK;
}

template <int R>
static int launch_istft(const float2* spec, int64_t rows, int n_frames, int hop, const float* window, float* out, int64_t length, cudaStream_t st) {
    int dev = 0, optin = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess)
        return fail(ACB_ERR_CUDA, "acb_istft: cannot query the device");
    int fpc = chunk_frames(kIstftFramesPerCta, n_frames, rows);
    while (fpc > 2 && chunk_smem(R, fpc, hop, true).total_bytes > std::min(optin, 160 * 1024)) fpc >>= 1;
    const ChunkSmem L = chunk_smem(R, fpc, hop, true);
    if (L.total_bytes > optin) return fail(ACB_ERR_UNSUPPORTED, "acb_istft: transform too large for shared memory");
    cudaError_t e = cudaFuncSetAttribute(istft_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin);
    if (e == cudaSuccess) e = cudaMemsetAsync(out, 0, sizeof(float) * (size_t)rows * (size_t)length, st);
    if (e != cudaSuccess) return fail(ACB_ERR_CUDA, std::string("acb_istft: ") + cudaGetErrorString(e));
    const dim3 grid((unsigned)((n_frames + fpc - 1) / fpc), (unsigned)rows);
    istft_kernel<R><<<grid, kThreads, L.total_bytes, st>>>(spec, n_frames, hop, window, out, length, fpc);
    const long long total = (long long)rows * length;
    istft_normalize_kernel<<<(unsigned)std::min<long long>(4096, (total + 255) / 256), 256, 0, st>>>(out, rows, length, 32 * R, hop, n_frames, window);
    e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ACB_ERR_CUDA, std::string("acb_istft launch: ") + cudaGetErrorString(e));
    return ACB_OK;
}

}  // namespace acb_spectral

extern "C" {

int64_t acb_stft_mag_frames(int64_t length, int n_fft, int hop) {
    if (n_fft <= 0 || hop <= 0 || length < n_fft) return -1;
    return 1 + (length - n_fft) / hop;
}

int acb_stft_mag(const float* x, int64_t rows, int64_t length, int n_fft, int hop, const float* window, float* out, void* stream) {
    using namespace acb_spectral;
    if (rows <= 0) return ACB_OK;
    if (!x || !window || !out) return fail(ACB_ERR_INVALID, "acb_stft_mag: null argument");
    if (hop < 1) return fail(ACB_ERR_INVALID, "acb_stft_mag: hop must be >= 1");
    if (length < n_fft)
        return fail(ACB_ERR_INVALID, "acb_stft_mag: rows of " + std::to_string(length) + " values are shorter than n_fft = " + std::to_string(n_fft) +
                                         " (center=False: torch.stft raises)");
    if (length > (1 << 24) || rows > ((int64_t)1 << 40)) return fail(ACB_ERR_UNSUPPORTED, "acb_stft_mag: input too large");
    const int n_frames = (int)acb_stft_mag_frames(length, n_fft, hop);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (n_fft) {
        case 64: return launch<2>(x, rows, (int)length, hop, n_frames, window, out, st);
        case 128: return launch<4>(x, rows, (int)length, hop, n_frames, window, out, st);
        case 256: return launch<8>(x, rows, (int)length, hop, n_frames, window, out, st);
        case 512: return launch<16>(x, rows, (int)length, hop, n_frames, window, out, st);
        case 1024: return launch<32>(x, rows, (int)length, hop, n_frames, window, out, st);
        default:
            return fail(ACB_ERR_UNSUPPORTED, "acb_stft_mag: n_fft must be 64, 128, 256, 512 or 1024 (got " + std::to_string(n_fft) + ")");
    }
}

int acb_stft_mag_backward(const float* x, const float* grad_mag, int64_t rows, int64_t length, int n_fft, int hop, const float* window,
                          float* grad_x, void* stream) {
    using namespace acb_spectral;
    if (rows <= 0) return ACB_OK;
    if (!x || !grad_mag || !window || !grad_x) return fail(ACB_ERR_INVALID, "acb_stft_mag_backward: null argument");
    if (hop < 1 || length < n_fft) return fail(ACB_ERR_INVALID, "acb_stft_mag_backward: bad hop / length");
    if (length > (1 << 24) || rows > ((int64_t)1 << 40)) return fail(ACB_ERR_UNSUPPORTED, "acb_stft_mag_backward: input too large");
    const int n_frames = (int)acb_stft_mag_frames(length, n_fft, hop);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (n_fft) {
        case 64: return launch_backward<2>(x, grad_mag, rows, (int)length, hop, n_frames, window, grad_x, st);
        case 128: return launch_backward<4>(x, grad_mag, rows, (int)length, hop, n_frames, window, grad_x, st);
        case 256: return launch_backward<8>(x, grad_mag, rows, (int)length, hop, n_frames, window, grad_x, st);
        case 512: return launch_backward<16>(x, grad_mag, rows, (int)length, hop, n_frames, window, grad_x, st);
        case 1024: return launch_backward<32>(x, grad_mag, rows, (int)length, hop, n_frames, window, grad_x, st);
        default:
            return fail(ACB_ERR_UNSUPPORTED, "acb_stft_mag_backward: n_fft must be 64, 128, 256, 512 or 1024 (got " + std::to_string(n_fft) + ")");
    }
}

int acb_stft_complex(const float* x, int64_t rows, int64_t length, int n_fft, int hop, const float* window, float* spec, float* gl_previous,
                     const float* gl_magnitude, float gl_momentum, void* stream) {
    using namespace acb_spectral;
    if (rows <= 0) return ACB_OK;
    if (!x || !window || !spec) return fail(ACB_ERR_INVALID, "acb_stft_complex: null argument");
    if ((gl_previous == nullptr) != (gl_magnitude == nullptr)) return fail(ACB_ERR_INVALID, "acb_stft_complex: gl_previous and gl_magnitude go together");
    if (hop < 1 || length <= n_fft / 2) return fail(ACB_ERR_INVALID, "acb_stft_complex: reflect padding needs rows longer than n_fft / 2");
    if (rows > 65535) return fail(ACB_ERR_UNSUPPORTED, "acb_stft_complex: at most 65535 rows per call");
    const int n_frames = (int)(1 + length / hop);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    float2* sp = reinterpret_cast<float2*>(spec);
    float2* tp = reinterpret_cast<float2*>(gl_previous);
    switch (n_fft) {
        case 256: return launch_stft_complex<8>(x, rows, length, hop, n_frames, window, sp, tp, gl_magnitude, gl_momentum, st);
        case 512: return launch_stft_complex<16>(x, rows, length, hop, n_frames, window, sp, tp, gl_magnitude, gl_momentum, st);
        case 1024: return launch_stft_complex<32>(x, rows, length, hop, n_frames, window, sp, tp, gl_magnitude, gl_momentum, st);
        default: return fail(ACB_ERR_UNSUPPORTED, "acb_stft_complex: n_fft must be 256, 512 or 1024");
    }
}

int acb_istft(const float* spec, int64_t rows, int64_t n_frames, int n_fft, int hop, const float* window, float* out, int64_t length, void* stream) {
    using namespace acb_spectral;
    if (rows <= 0) return ACB_OK;
    if (!spec || !window || !out) return fail(ACB_ERR_INVALID, "acb_istft: null argument");
    if (hop < 1 || n_frames < 1 || length < 1) return fail(ACB_ERR_INVALID, "acb_istft: bad hop / frames / length");
    if (rows > 65535 || n_frames > (1 << 24)) return fail(ACB_ERR_UNSUPPORTED, "acb_istft: input too large");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const float2* sp = reinterpret_cast<const float2*>(spec);
    switch (n_fft) {
        case 256: return launch_istft<8>(sp, rows, (int)n_frames, hop, window, out, length, st);
        case 512: return launch_istft<16>(sp, rows, (int)n_frames, hop, window, out, length, st);
        case 1024: return launch_istft<32>(sp, rows, (int)n_frames, hop, window, out, length, st);
        default: return fail(ACB_ERR_UNSUPPORTED, "acb_istft: n_fft must be 256, 512 or 1024");
    }
}

}  // extern "C"
