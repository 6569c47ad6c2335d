// General STFT log-mel kernel of the front-end: n_fft = 32 R in {256, 512, 1024} with any hop in [1, n_fft], any fp32 window and any
// banded filterbank over bins 0..n_fft/2 (DC and Nyquist included).  (n_fft, hop) = (1024, 256) keeps its tuned kernel
// (logmel_fused_kernel, acb_kernels.cu); acb_frontend_create routes every other supported pair here.  The launch contract is the
// same acb_logmel_args: uniform and ragged batches, fused peak gain, fp32 / bf16 in both layouts, reflected pad columns, tail fill,
// scalar / per-band affine and fp64 per-band moments, with the cursor, store and fill helpers of acb_logmel_common.cuh.
// The handle's spectrogram definition (acb_stft_options) sets the framing pad p (T = 1 + (L + 2 p - n_fft) / hop), reflect or
// constant padding, and power 2 or magnitude sqrt(|X|^2 + eps); a definition other than the centred power spectrogram runs here at
// every supported (n_fft, hop), (1024, 256) included.
//
// Mapping: one CTA of 4 R threads works through a contiguous range of 8-frame tiles (acb_frames_per_tile), persistent over the grid.
// Per tile:
//   1. the tile's (8 - 1) * hop + n_fft samples, from sample f0 * hop - p on, are staged in shared memory by 4-byte cp.async copies
//      issued while the previous tile's mel phase runs.  Each copy computes its own source index: reflection about sample 0 / L - 1
//      (pad_mode="reflect"), or zeros outside [0, L) (pad_mode="constant", a cp.async of source size 0), and zero fill beyond come
//      for free, no read leaves [clip_offset, clip_offset + clip_length), and a hop that is not a multiple of 4 samples needs no
//      alignment;
//   2. lane group g (R lanes) takes frames 2g and 2g + 1 of the tile and runs ONE complex n_fft-point group FFT of A + iB
//      (acb_fft32.cuh: in-register FFT-32 per lane, twiddle, R-point FFT across the lanes through shared memory), with the whole
//      window held in registers;
//   3. the two real spectra are separated (Z[k], Z[N - k]) into 4 |X|^2 for bins 0..n_fft/2 -- with power 1 into
//      sqrt(s^2 4 |X|^2 + 4 eps) = 2 sqrt(|s X|^2 + eps), the peak gain s^2 taken under the root -- and written over the FFT buffer
//      as [bin][8 frames] (the 1/4, or 1/2, is folded into the weights);
//   4. thread (band, frame quad) sums its band's contiguous run of weights against four frames with 16-byte power loads, then
//      clamp, log, moments and affine; the tile is staged in shared memory and stored by store_tile (masking, reflected pad-to-4
//      columns, tail fill).
#include "audiocalm_b200.h"
#include "acb_fft32.cuh"
#include "acb_logmel_common.cuh"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <string>
#include <type_traits>
#include <vector>

namespace acb {

constexpr int kStftMaxWeights = 16384;   // banded weights held in shared memory (64 KB)

struct StftLogmelParams {
    LogmelParams c;            // batch, output and epilogue fields shared with logmel_fused_kernel (its table fields are unused here)
    int hop;
    int n_weights;
    const float* window;       // [N]
    const float2* twiddle;     // [32][R]: entry k * R + r = W_N^(r k)
    const float* weights;      // [n_weights] band after band, each its run of bins, times 1/4 (power 2) or 1/2 (power 1)
    const int4* band;          // [n_mels] {first bin, bins, offset in weights, 0}
    // spectrogram definition (acb_stft_options), read by the kDefinition instantiations only
    int pad;                   // samples padded on each side before framing
    int len_off;               // 2 pad - N: T = 1 + (L + len_off) / hop
    int pad_constant;          // 1: zeros outside the clip; 0: reflection about its first and last sample
    int magnitude;             // 1: power rows hold 2 sqrt(|X|^2 + eps) (power 1); 0: 4 |X|^2 (power 2)
    float eps4;                // 4 * magnitude_eps
};

struct StftSmem {
    int samples, buf, out, tw, w, band, affine, moments, total_bytes;
};

// offsets in 4-byte words, every region 16-byte aligned
__host__ __device__ inline StftSmem stft_smem(int R, int hop, int n_mels, int n_weights) {
    StftSmem L;
    int off = 0;
    L.samples = off; off += ((kTileFrames - 1) * hop + 32 * R + 3) & ~3;
    L.buf = off; off += 4 * 2 * 33 * R;                             // four group-FFT buffers of 33 R float2; then the power spectra
    L.out = off; off += (kTileFrames * out_row_stride(n_mels) + 3) & ~3;
    L.tw = off; off += 2 * 32 * R;
    L.w = off; off += (n_weights + 3) & ~3;
    L.band = off; off += 4 * n_mels;
    L.affine = off; off += 2 * ((n_mels + 1) & ~1);
    L.moments = off; off += 4 * n_mels;                             // float2 [2][n_mels]
    L.total_bytes = off * 4;
    return L;
}

// Position of bin k's 8 frames in the power buffer: rows of 8 floats with 4 floats of padding after every 4 rows, so that the 16-byte
// loads of lanes on neighbouring bins and the 8-byte stores of one lane group's bins spread over the banks.
__device__ __forceinline__ int pow_index(int k) { return 8 * k + 4 * (k >> 2); }

__device__ __forceinline__ void cp_async4(float* dst, const float* src, bool valid) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;"
                 ::"r"(static_cast<unsigned>(__cvta_generic_to_shared(dst))), "l"(src), "r"(valid ? 4 : 0) : "memory");
}

// Request the tile's samples (relative index i = sample f0 * hop - pad + i of the clip; reflected at both ends in reflect mode, zero
// beyond; zero outside the clip in constant mode).
template <int R, bool kDefinition>
__device__ __forceinline__ void stage_tile(const StftLogmelParams& sp, const ClipCursor& c, int hop, float* s_samples, int tid) {
    constexpr int N = 32 * R, kThreads = 4 * R;
    const LogmelParams& p = sp.c;
    const bool constant = kDefinition && sp.pad_constant;
    const long long g0 = (long long)c.tile_in_clip * kTileFrames * hop - (kDefinition ? sp.pad : N / 2);
    const int n = (kTileFrames - 1) * hop + N;
    const float* src = p.wav + c.wav_base;
    const long long L = c.length;
    for (int i = tid; i < n; i += kThreads) {
        long long idx = g0 + i;
        if (!constant) {
            if (idx < 0) idx = -idx;
            if (idx >= L) idx = 2 * (L - 1) - idx;
        }
        const bool ok = idx >= 0 && idx < L;
        cp_async4(s_samples + i, src + (ok ? idx : 0), ok);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
}

// kDefinition = false: the centred, reflect-padded power spectrogram (pad N/2 at compile time); true: the handle's spectrogram
// definition (acb_stft_options), read from sp
template <int R, bool kMoments, typename OutT, bool kDefinition>
__global__ void __launch_bounds__(4 * R) logmel_stft_kernel(const StftLogmelParams sp) {
    constexpr int N = 32 * R, kThreads = 4 * R, kHalf = N / 2;
    const LogmelParams& p = sp.c;
    const int len_off = kDefinition ? sp.len_off : 0;
    const bool magnitude = kDefinition && sp.magnitude;
    extern __shared__ __align__(16) float smem[];
    const int hop = sp.hop, n_mels = p.n_mels, S = out_row_stride(n_mels);
    const StftSmem L = stft_smem(R, hop, n_mels, sp.n_weights);
    const int tid = threadIdx.x;
    const int g = tid / R, r = tid % R;                      // frame pair of the tile (frames 2g, 2g + 1), lane within its group
    const bool write_out = p.out != nullptr;
    float* s_samples = smem + L.samples;
    float2* buf = reinterpret_cast<float2*>(smem + L.buf) + g * (33 * R);
    float* s_pow = smem + L.buf;
    float* s_out = smem + L.out;
    float2* s_tw = reinterpret_cast<float2*>(smem + L.tw);
    float* s_w = smem + L.w;
    int4* s_band = reinterpret_cast<int4*>(smem + L.band);
    float2* s_aff = reinterpret_cast<float2*>(smem + L.affine);
    float2* s_mom = reinterpret_cast<float2*>(smem + L.moments);

    for (int i = tid; i < N; i += kThreads) s_tw[i] = sp.twiddle[i];
    for (int i = tid; i < sp.n_weights; i += kThreads) s_w[i] = sp.weights[i];
    for (int i = tid; i < n_mels; i += kThreads) {
        s_band[i] = sp.band[i];
        float sc = 1.f, sh = 0.f;   // affine == 0: v * 1 + 0 is exact
        if (p.affine == 1) { sc = p.affine_inv_std; sh = -p.affine_mean * p.affine_inv_std; }
        else if (p.affine == 2) { sc = 1.f / __ldg(p.bin_std + i); sh = -__ldg(p.bin_mean + i) * sc; }
        s_aff[i] = make_float2(sc, sh);
    }
    if (kMoments)
        for (int i = tid; i < 2 * n_mels; i += kThreads) s_mom[i] = make_float2(0.f, 0.f);
    float wreg[32];                                          // this lane's window values, bit-reversed pair order (loop-invariant)
#pragma unroll
    for (int q = 0; q < 16; ++q) {
        wreg[2 * q] = __ldg(sp.window + R * brev5(q) + r);
        wreg[2 * q + 1] = __ldg(sp.window + R * (brev5(q) + 1) + r);
    }

    // ---- this CTA's contiguous tile range ----
    const long long t_begin = (long long)p.n_tiles * blockIdx.x / gridDim.x;
    const long long t_end = (long long)p.n_tiles * (blockIdx.x + 1) / gridDim.x;
    ClipCursor cur;
    if (t_begin < t_end) {
        cursor_init(p, cur, t_begin, hop, len_off);
        if (cur.tile_in_clip * kTileFrames < cur.frames) stage_tile<R, kDefinition>(sp, cur, hop, s_samples, tid);
    }

    for (long long tile = t_begin; tile < t_end; ++tile) {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();   // the tile's samples have landed; the previous tile's power spectra and staged output are no longer read

        const int f0 = cur.tile_in_clip * kTileFrames;
        const bool has_frames = f0 < cur.frames;             // false for pure tail-fill tiles
        const bool active = has_frames && f0 + 2 * g < cur.frames;
        float2 pr[16], pi[16];
        if (active) {
            const float* pa = s_samples + (2 * g) * hop;
            const float* pb = pa + hop;
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const int n0 = R * brev5(q) + r, n1 = n0 + R;
                pr[q] = make_float2(pa[n0] * wreg[2 * q], pa[n1] * wreg[2 * q + 1]);
                pi[q] = make_float2(pb[n0] * wreg[2 * q], pb[n1] * wreg[2 * q + 1]);
            }
        }
        __syncthreads();   // samples consumed: the next tile's copies may land

        ClipCursor nxt = cur;
        if (tile + 1 < t_end) {
            cursor_advance(p, nxt, hop, len_off);
            if (nxt.tile_in_clip * kTileFrames < nxt.frames) stage_tile<R, kDefinition>(sp, nxt, hop, s_samples, tid);
        }

        // ---- group FFT of the pair, separation into 4 |X_A|^2, 4 |X_B|^2 for bins k = r + R t <= N/2 ----
        if (active) group_fft_stage1<R>(pr, pi, buf, s_tw, r);
        __syncwarp();
        if (active) group_fft_stage2<R>(buf, r);
        __syncwarp();
        float pwa[17], pwb[17];
        if (active) {
#pragma unroll
            for (int t = 0; t <= 16; ++t) {
                const int k = r + R * t;
                if (t < 16 || k == kHalf) {
                    const int kc = (N - k) & (N - 1);
                    const float2 z = buf[buf_index(k)], zc = buf[buf_index(kc)];
                    const float apc = z.x + zc.x, bmd = z.y - zc.y, amc = z.x - zc.x, bpd = z.y + zc.y;
                    pwa[t] = fmaf(apc, apc, bmd * bmd);
                    pwb[t] = fmaf(amc, amc, bpd * bpd);
                    if (magnitude) {   // 2 sqrt(s^2 |X|^2 + eps): the peak gain s^2 goes under the root with the eps
                        pwa[t] = sqrtf(fmaf(cur.gain, pwa[t], sp.eps4));
                        pwb[t] = sqrtf(fmaf(cur.gain, pwb[t], sp.eps4));
                    }
                }
            }
        }
        __syncthreads();   // every pair's transform has been read: the buffers take the power spectra
        if (active) {
#pragma unroll
            for (int t = 0; t <= 16; ++t) {
                const int k = r + R * t;
                if (t < 16 || k == kHalf) *reinterpret_cast<float2*>(s_pow + pow_index(k) + 2 * g) = make_float2(pwa[t], pwb[t]);
            }
        }
        __syncthreads();

        // ---- banded mel projection over four frames per thread, clamp, log, moments, affine -> staged tile ----
        const float gain = magnitude ? 1.f : cur.gain;   // a magnitude spectrum took its gain before the root
        if (has_frames) {
            for (int base = 0; base < 2 * n_mels; base += kThreads) {   // uniform trip count: the moments' shuffle needs every lane
                const int item = base + tid;
                const bool valid = item < 2 * n_mels;
                const int b = valid ? item >> 1 : 0, h = item & 1;
                const int4 bd = s_band[b];
                const int nb = valid ? bd.y : 0;
                const float* pw = s_pow + 4 * h;
                const float* w = s_w + bd.z;
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
                for (int i = 0; i < nb; ++i) {
                    const float wi = w[i];
                    const float4 v = *reinterpret_cast<const float4*>(pw + pow_index(bd.x + i));
                    acc.x = fmaf(wi, v.x, acc.x);
                    acc.y = fmaf(wi, v.y, acc.y);
                    acc.z = fmaf(wi, v.z, acc.z);
                    acc.w = fmaf(wi, v.w, acc.w);
                }
                float v[4] = {acc.x * gain, acc.y * gain, acc.z * gain, acc.w * gain};
#pragma unroll
                for (int j = 0; j < 4; ++j) v[j] = (v[j] > p.clamp_min) ? lg2_normal(v[j]) * p.log_scale : p.log_floor;
                if (kMoments) {
                    // frames T-2-j (j < pad) are stored twice (reflected pad-to-4 columns) and counted twice; the two lanes of a band
                    // combine their four frames and the even one adds them to the CTA's compensated accumulators
                    const int T = cur.frames, pad = cur.frames_padded - cur.frames;
                    float s = 0.f, s2 = 0.f;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int fr = f0 + 4 * h + j;
                        if (valid && fr < T) {
                            const float cv = (fr <= T - 2 && fr > T - 2 - pad) ? 2.f * v[j] : v[j];
                            s += cv;
                            s2 = fmaf(cv, v[j], s2);
                        }
                    }
                    s += __shfl_xor_sync(0xffffffffu, s, 1);
                    s2 += __shfl_xor_sync(0xffffffffu, s2, 1);
                    if (valid && h == 0) {
                        two_sum_add(s_mom[b], s);
                        two_sum_add(s_mom[n_mels + b], s2);
                    }
                }
                if (valid) {
                    const float2 af = s_aff[b];
#pragma unroll
                    for (int j = 0; j < 4; ++j) s_out[(4 * h + j) * S + b] = fmaf(v[j], af.x, af.y);
                }
            }
        }
        __syncthreads();   // output tile staged
        if (write_out) {
            store_tile<OutT, kThreads>(p, cur, s_out, n_mels, S, tid);
            if (p.fill_tail && p.tile_start != nullptr && cur.tile_in_clip == cur.tiles_in_clip - 1) fill_row_tail<OutT, kThreads>(p, cur, n_mels, tid);
        }
        cur = nxt;
    }

    if (kMoments) {
        __syncthreads();
        for (int i = tid; i < 2 * n_mels; i += kThreads)
            p.moments_partial[(size_t)blockIdx.x * 2 * n_mels + i] = (double)s_mom[i].x + (double)s_mom[i].y;
    }
}

bool stft_logmel_supported(int n_fft, int hop) {
    return (n_fft == 256 || n_fft == 512 || n_fft == 1024) && hop >= 1 && hop <= n_fft;
}

template <int R, typename F>
static void for_each_instantiation(F&& f) {
    f(logmel_stft_kernel<R, false, float, false>);
    f(logmel_stft_kernel<R, false, __nv_bfloat16, false>);
    f(logmel_stft_kernel<R, true, float, false>);
    f(logmel_stft_kernel<R, true, __nv_bfloat16, false>);
    f(logmel_stft_kernel<R, false, float, true>);
    f(logmel_stft_kernel<R, false, __nv_bfloat16, true>);
    f(logmel_stft_kernel<R, true, float, true>);
    f(logmel_stft_kernel<R, true, __nv_bfloat16, true>);
}

template <typename F>
static void for_each_instantiation(int R, F&& f) {
    if (R == 8) for_each_instantiation<8>(f);
    else if (R == 16) for_each_instantiation<16>(f);
    else for_each_instantiation<32>(f);
}

int stft_frontend_create(acb_frontend** out, int device, int n_fft, int hop, int n_mels, const float* window_host, const float* fb_host,
                         float clamp_min, int log_kind, const acb_stft_options& opt) {
    const int R = n_fft / 32, n_freq = n_fft / 2 + 1;
    // banded form of the filterbank: each band's run from its first to its last non-zero bin; the 1/4 of the packed-pair power
    // spectrum (4 |X|^2), or the 1/2 of its magnitude (2 sqrt(|X|^2 + eps)), is folded in (exact scaling)
    const float fold = opt.power == 1 ? 0.5f : 0.25f;
    std::vector<int4> band(n_mels);
    std::vector<float> weights;
    for (int m = 0; m < n_mels; ++m) {
        int lo = -1, hi = -1;
        for (int f = 0; f < n_freq; ++f)
            if (fb_host[(size_t)f * n_mels + m] != 0.f) { if (lo < 0) lo = f; hi = f; }
        band[m] = make_int4(lo < 0 ? 0 : lo, lo < 0 ? 0 : hi - lo + 1, (int)weights.size(), 0);
        for (int f = lo; lo >= 0 && f <= hi; ++f) weights.push_back(fb_host[(size_t)f * n_mels + m] * fold);
    }
    if ((int)weights.size() > kStftMaxWeights)
        return fail(ACB_ERR_UNSUPPORTED, "acb_frontend_create: filterbank too dense (" + std::to_string(weights.size()) +
                                             " banded weights; the n_fft=" + std::to_string(n_fft) + " kernel holds at most " +
                                             std::to_string(kStftMaxWeights) + ")");
    // W_N^(r k) = exp(-2 pi i r k / N) in double, rounded once; laid out [k][r] as group_fft_stage1 reads it
    std::vector<float2> tw(n_fft);
    for (int k = 0; k < 32; ++k)
        for (int r = 0; r < R; ++r) {
            const double a = -2.0 * M_PI * (double)(r * k) / (double)n_fft;
            tw[k * R + r] = make_float2((float)cos(a), (float)sin(a));
        }

    int prev = 0;
    cudaError_t e = cudaGetDevice(&prev);
    if (e == cudaSuccess) e = cudaSetDevice(device);
    if (e != cudaSuccess) return fail(ACB_ERR_CUDA, std::string("acb_frontend_create: ") + cudaGetErrorString(e));
    auto* fe = new acb_frontend();
    fe->device = device; fe->n_fft = n_fft; fe->hop = hop; fe->n_mels = n_mels; fe->n_weights = (int)weights.size();
    fe->log_kind = log_kind; fe->clamp_min = clamp_min;
    fe->stft_r = R;
    fe->opt = opt;
    fe->groups = 1;

    size_t o = 0;
    auto take = [&](size_t bytes) { size_t q = o; o += (bytes + 255) & ~size_t(255); return q; };
    const size_t o_win = take(sizeof(float) * n_fft), o_tw = take(sizeof(float2) * n_fft),
                 o_w = take(sizeof(float) * std::max<size_t>(weights.size(), 1)), o_band = take(sizeof(int4) * n_mels), o_err = take(16);
    std::vector<unsigned char> host(o, 0);
    memcpy(host.data() + o_win, window_host, sizeof(float) * n_fft);
    memcpy(host.data() + o_tw, tw.data(), sizeof(float2) * n_fft);
    if (!weights.empty()) memcpy(host.data() + o_w, weights.data(), sizeof(float) * weights.size());
    memcpy(host.data() + o_band, band.data(), sizeof(int4) * n_mels);
    e = cudaMalloc(&fe->d_blob, o);
    if (e == cudaSuccess) e = cudaMemcpy(fe->d_blob, host.data(), o, cudaMemcpyHostToDevice);
    int optin = 0, sms = 0;
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    const StftSmem L = stft_smem(R, hop, n_mels, fe->n_weights);
    fe->smem_bytes = fe->smem_bytes_moments = L.total_bytes;
    if (e == cudaSuccess && L.total_bytes > optin) {
        cudaFree(fe->d_blob);
        delete fe;
        cudaSetDevice(prev);
        return fail(ACB_ERR_UNSUPPORTED, "acb_frontend_create: the n_fft=" + std::to_string(n_fft) + " kernel needs " + std::to_string(L.total_bytes) +
                                             " bytes of shared memory, more than the device offers");
    }
    // the attribute is per function, not per handle: raised to the opt-in maximum, the launch passes the handle's own size
    int occ = 0;
    for_each_instantiation(R, [&](auto kernel) {
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, optin);
        if (e == cudaSuccess && occ == 0) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, 4 * R, L.total_bytes);
    });
    if (e != cudaSuccess) {
        if (fe->d_blob) cudaFree(fe->d_blob);
        delete fe;
        cudaSetDevice(prev);
        return fail(ACB_ERR_CUDA, std::string("acb_frontend_create: ") + cudaGetErrorString(e));
    }
    fe->num_sms = sms;
    fe->grid = sms * std::max(occ, 1);
    auto* base = static_cast<unsigned char*>(fe->d_blob);
    fe->d_window = reinterpret_cast<const float*>(base + o_win);
    fe->d_stft_twiddle = reinterpret_cast<const float2*>(base + o_tw);
    fe->d_stft_weights = reinterpret_cast<const float*>(base + o_w);
    fe->d_stft_band = reinterpret_cast<const int4*>(base + o_band);
    fe->d_err = reinterpret_cast<int*>(base + o_err);
    cudaSetDevice(prev);
    *out = fe;
    return ACB_OK;
}

void stft_logmel_launch(const acb_frontend* fe, const LogmelParams& p, bool moments, cudaStream_t st) {
    StftLogmelParams sp{};
    sp.c = p;
    sp.hop = fe->hop;
    sp.n_weights = fe->n_weights;
    sp.window = fe->d_window;
    sp.twiddle = fe->d_stft_twiddle;
    sp.weights = fe->d_stft_weights;
    sp.band = fe->d_stft_band;
    sp.pad = fe->opt.pad;
    sp.len_off = 2 * fe->opt.pad - fe->n_fft;
    sp.pad_constant = fe->opt.pad_mode == ACB_PAD_CONSTANT;
    sp.magnitude = fe->opt.power == 1;
    sp.eps4 = 4.f * fe->opt.magnitude_eps;
    const int R = fe->stft_r;
    auto launch = [&](auto kernel) { kernel<<<fe->grid, 4 * R, fe->smem_bytes, st>>>(sp); };
    // the centred power spectrogram runs the instantiation with its framing and power fixed at compile time
    const bool definition = !(fe->opt.pad == fe->n_fft / 2 && fe->opt.pad_mode == ACB_PAD_REFLECT && fe->opt.power == 2);
    auto dispatch_def = [&](auto r_tag, auto def_tag) {
        constexpr int kR = decltype(r_tag)::value;
        constexpr bool kD = decltype(def_tag)::value;
        if (moments) { if (p.out_bf16) launch(logmel_stft_kernel<kR, true, __nv_bfloat16, kD>); else launch(logmel_stft_kernel<kR, true, float, kD>); }
        else { if (p.out_bf16) launch(logmel_stft_kernel<kR, false, __nv_bfloat16, kD>); else launch(logmel_stft_kernel<kR, false, float, kD>); }
    };
    auto dispatch = [&](auto r_tag) {
        if (definition) dispatch_def(r_tag, std::true_type{}); else dispatch_def(r_tag, std::false_type{});
    };
    if (R == 8) dispatch(std::integral_constant<int, 8>{});
    else if (R == 16) dispatch(std::integral_constant<int, 16>{});
    else dispatch(std::integral_constant<int, 32>{});
}

}  // namespace acb
