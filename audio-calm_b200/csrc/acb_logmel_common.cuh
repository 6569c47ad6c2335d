// Internal header of the log-mel front-end: the launch parameters, the clip cursor, the output store / fill helpers and the epilogue
// arithmetic shared by the tuned n_fft-1024 hop-256 kernel (logmel_fused_kernel, acb_kernels.cu) and the general STFT log-mel kernel
// (logmel_stft_kernel, acb_logmel_stft.cu), and the front-end handle both routes fill in.
#pragma once
#include "audiocalm_b200.h"

#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <mutex>
#include <string>
#include <vector>

namespace acb {

constexpr int kTileFrames = 8;                               // one tile = 4 frame pairs
constexpr int kGroupWarps = 4;
constexpr int kGroupThreads = kGroupWarps * 32;
constexpr int kMaxMels = 128;

int fail(int code, const std::string& msg);   // acb_kernels.cu: sets the thread-local message behind acb_last_error()

struct LogmelParams {
    // tables (device)
    const float* window;       // [1024]
    const float4* twiddle;     // [5][32]  seeds of the twiddle chains per lane l, W = exp(-2*pi*i/1024):
                               //          [k][l] = (Re W^kl, Re W^(k+16)l, Im W^kl, Im W^(k+16)l), k = 0..3;  [4][l] = (Re, Im W^4l, 0, 0)
    // mel plan: per (group warp, round) eight band slots with a common even trip count; weights zero-padded to the trip
    // and interleaved as [i/2][slot][2] so that a lane fetches two consecutive weights with one 8-byte load
    const float* plan_w;       // [n_plan_w]
    const int* plan_woff;      // [kGroupWarps][kMaxRounds] offset (floats) of the round's weights in plan_w
    const short* plan_trip;    // [kGroupWarps][kMaxRounds] bins per round (even, 0 = no more rounds)
    const short* plan_band;    // [kGroupWarps][kMaxRounds][kSlots] band id or -1
    const short* plan_astart;  // [kGroupWarps][kMaxRounds][kSlots] first bin (even) of the slot's run
    int n_plan_w;
    int n_mels;
    float clamp_min;
    float log_scale;           // ln(2) for ln, log10(2) for log10 (applied to log2)
    float log_floor;           // log(clamp_min) computed on the host: clamped values are exactly the reference's floor
    // batch
    const float* wav;
    const long long* clip_offset;
    const long long* clip_length;
    long long clip_stride;
    long long uniform_length;
    const int* tile_start;
    int n_clips;
    int n_tiles;
    int uniform_tiles_per_clip;
    const float* clip_peak;
    // output
    void* out;
    int out_bf16;
    int time_major;
    const long long* out_offset;
    long long out_clip_stride;
    long long frame_capacity;
    const long long* frame_capacity_per_clip;
    int pad_multiple;
    int fill_tail;
    float fill_value;
    int affine;
    float affine_mean;
    float affine_inv_std;
    const float* bin_mean;
    const float* bin_std;
    double* moments_partial;   // [gridDim.x * G][2][n_mels] or nullptr
    int* error_flag;           // set to 1 when a sample-tile barrier timed out (results invalid)
};

__host__ __device__ inline int out_row_stride(int n_mels) { return n_mels | 1; }   // odd: conflict-free both ways

// Position of a group in its contiguous tile range: which clip, which tile of the clip, and the clip's geometry.
struct ClipCursor {
    long long wav_base;    // element index of the clip's first sample in wav
    long long length;      // samples in the clip
    long long out_base;    // element offset of the clip in out
    int cap;               // frame capacity (row pitch of the mel-major layout)
    int frames;            // T
    int frames_padded;     // T4
    int clip;
    int tile_in_clip;
    int tiles_in_clip;
    float gain;            // squared waveform scale (fused peak normalisation), 1 otherwise
};

// T = 1 + (L + len_off) / hop with len_off = 2 pad - n_fft of the framing: 0 for torch.stft(center=True), a compile-time 0 in the
// tuned kernel.
__device__ __forceinline__ void cursor_load_clip(const LogmelParams& p, ClipCursor& c, int hop, int len_off = 0) {
    const int i = c.clip;
    c.wav_base = p.clip_offset ? p.clip_offset[i] : (long long)i * p.clip_stride;
    c.length = p.clip_length ? p.clip_length[i] : p.uniform_length;
    c.out_base = p.out_offset ? p.out_offset[i] : (long long)i * p.out_clip_stride;
    c.cap = (int)(p.frame_capacity_per_clip ? p.frame_capacity_per_clip[i] : p.frame_capacity);
    c.frames = 1 + (int)((c.length + len_off) / hop);
    const int rem = c.frames % p.pad_multiple;
    c.frames_padded = rem ? c.frames + (p.pad_multiple - rem) : c.frames;
    c.tiles_in_clip = p.tile_start ? (__ldg(p.tile_start + i + 1) - __ldg(p.tile_start + i)) : p.uniform_tiles_per_clip;
    c.gain = 1.f;
    if (p.clip_peak) {
        const float peak = __ldg(p.clip_peak + i);
        if (peak > 0.f) {
            const float s = 0.95f / (peak + 1e-8f);
            c.gain = s * s;
        }
    }
}

__device__ __forceinline__ void cursor_init(const LogmelParams& p, ClipCursor& c, long long tile, int hop, int len_off = 0) {
    if (p.tile_start == nullptr) {
        c.clip = (int)(tile / p.uniform_tiles_per_clip);
        c.tile_in_clip = (int)(tile - (long long)c.clip * p.uniform_tiles_per_clip);
    } else {  // largest clip with tile_start[clip] <= tile
        int lo = 0, hi = p.n_clips;
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if ((long long)__ldg(p.tile_start + mid) <= tile) lo = mid; else hi = mid;
        }
        c.clip = lo;
        c.tile_in_clip = (int)(tile - __ldg(p.tile_start + lo));
    }
    cursor_load_clip(p, c, hop, len_off);
}

__device__ __forceinline__ void cursor_advance(const LogmelParams& p, ClipCursor& c, int hop, int len_off = 0) {
    if (++c.tile_in_clip >= c.tiles_in_clip) {
        c.tile_in_clip = 0;
        do { ++c.clip; cursor_load_clip(p, c, hop, len_off); } while (c.tiles_in_clip == 0 && c.clip + 1 < p.n_clips);
    }
}

template <typename OutT>
__device__ __forceinline__ OutT to_out(float v);
template <>
__device__ __forceinline__ float to_out<float>(float v) { return v; }
template <>
__device__ __forceinline__ __nv_bfloat16 to_out<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

template <typename OutT>
__device__ __forceinline__ void store_pair(OutT* dst, float a, float b);
template <>
__device__ __forceinline__ void store_pair<float>(float* dst, float a, float b) { *reinterpret_cast<float2*>(dst) = make_float2(a, b); }
template <>
__device__ __forceinline__ void store_pair<__nv_bfloat16>(__nv_bfloat16* dst, float a, float b) {
    *reinterpret_cast<__nv_bfloat162*>(dst) = __floats2bfloat162_rn(a, b);
}

// Store one staged tile [kTileFrames][S] with the kThreads threads of a group (index tid).  Interior tiles (every frame exists and
// none is a pad-to-4 source) take loops without per-element conditions; the last tiles of a clip take the general path (masking,
// reflected columns, tail fill).
template <typename OutT, int kThreads = kGroupThreads>
__device__ __forceinline__ void store_tile(const LogmelParams& p, const ClipCursor& c, const float* s_out, int n_mels, int S, int tid) {
    OutT* out = reinterpret_cast<OutT*>(p.out) + c.out_base;
    const int lane = tid & 31, warp = tid >> 5;   // thread / warp index inside the group
    const int f0 = c.tile_in_clip * kTileFrames;
    const int T = c.frames, T4 = c.frames_padded, pad = T4 - T;
    const bool interior = (f0 + kTileFrames - 1 <= T - 2 - pad);
    if (interior) {
        if (p.time_major) {
            OutT* row0 = out + (size_t)f0 * n_mels;
            for (int f = warp; f < kTileFrames; f += kThreads / 32) {
                OutT* row = row0 + f * n_mels;
                const float* srow = s_out + f * S;
                for (int b = lane; b < n_mels; b += 32) row[b] = to_out<OutT>(srow[b]);
            }
        } else {
            OutT* col0 = out + f0;
            const int f = tid & (kTileFrames - 1);
            for (int b = tid / kTileFrames; b < n_mels; b += kThreads / kTileFrames)
                col0[(unsigned)b * (unsigned)c.cap + f] = to_out<OutT>(s_out[f * S + b]);
        }
        return;
    }
    const int n_out = kTileFrames * n_mels;
    for (int idx = tid; idx < n_out; idx += kThreads) {
        int f, b;
        if (p.time_major) { f = idx / n_mels; b = idx - f * n_mels; }
        else { b = idx / kTileFrames; f = idx - b * kTileFrames; }
        const int fr = f0 + f;
        if (fr >= c.cap) continue;
        float v;
        bool dup = false;
        if (fr < T) {
            v = s_out[f * S + b];
            dup = (fr <= T - 2) && (fr > T - 2 - pad);
        } else if (fr >= T4 && p.fill_tail) {
            v = p.fill_value;
        } else {
            continue;
        }
        const size_t e0 = p.time_major ? ((size_t)fr * n_mels + b) : ((size_t)b * c.cap + fr);
        out[e0] = to_out<OutT>(v);
        if (dup) {
            const int fd = 2 * T - 2 - fr;  // column T + j with j = T-2-fr  (out[T+j] = mel[T-2-j])
            const size_t e1 = p.time_major ? ((size_t)fd * n_mels + b) : ((size_t)b * c.cap + fd);
            out[e1] = to_out<OutT>(v);
        }
    }
}

// Fill `n` elements at `ptr` with `fv`: scalar head / tail around 16-byte stores, `nt` cooperating threads (index t)
template <typename OutT>
__device__ __forceinline__ void fill_span(OutT* ptr, long long n, OutT fv, int t, int nt) {
    constexpr int per16 = 16 / (int)sizeof(OutT);
    const long long head = min(n, (long long)(((16 - (reinterpret_cast<uintptr_t>(ptr) & 15)) & 15) / sizeof(OutT)));
    for (long long i = t; i < head; i += nt) ptr[i] = fv;
    const long long body = (n - head) / per16;
    unsigned w;
    if (sizeof(OutT) == 4) w = *reinterpret_cast<const unsigned*>(&fv);
    else { const unsigned short h = *reinterpret_cast<const unsigned short*>(&fv); w = (unsigned)h | ((unsigned)h << 16); }
    uint4* q = reinterpret_cast<uint4*>(ptr + head);
    for (long long i = t; i < body; i += nt) q[i] = make_uint4(w, w, w, w);
    for (long long i = head + body * per16 + t; i < n; i += nt) ptr[i] = fv;
}

// Padded batches with a tile plan (tiles cover only the frames that exist): the group that stores a clip's last tile also sets the
// rest of the clip's row, frames [end of the tile, frame_capacity), to the fill value -- one vectorised sweep instead of one
// near-empty tile per 8 frames.
template <typename OutT, int kThreads = kGroupThreads>
__device__ __forceinline__ void fill_row_tail(const LogmelParams& p, const ClipCursor& c, int n_mels, int tid) {
    const int f_begin = (c.tile_in_clip + 1) * kTileFrames;
    const long long n_fill = (long long)c.cap - f_begin;
    if (n_fill <= 0) return;
    OutT* out = reinterpret_cast<OutT*>(p.out) + c.out_base;
    const OutT fv = to_out<OutT>(p.fill_value);
    if (p.time_major) {
        fill_span<OutT>(out + (size_t)f_begin * n_mels, n_fill * n_mels, fv, tid, kThreads);
    } else {
        const int lane = tid & 31, warp = tid >> 5;
        for (int b = warp; b < n_mels; b += kThreads / 32) fill_span<OutT>(out + (size_t)b * c.cap + f_begin, n_fill, fv, lane, 32);
    }
}

// log2 of a value known to be a normal float (it is above the clamp): the bare MUFU.LG2, without __log2f's denormal rescue
__device__ __forceinline__ float lg2_normal(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// (hi, lo) += x with the rounding error of hi + x carried in lo (Knuth two-sum; no fast-math reassociation is enabled)
__device__ __forceinline__ void two_sum_add(float2& acc, float x) {
    const float t = __fadd_rn(acc.x, x);
    const float bb = __fsub_rn(t, acc.x);
    const float e = __fadd_rn(__fsub_rn(acc.x, __fsub_rn(t, bb)), __fsub_rn(x, bb));
    acc.y = __fadd_rn(acc.y, e);
    acc.x = t;
}

}  // namespace acb

// Device-resident tables of one front-end.  Two routes share the handle: (n_fft, hop) = (1024, 256) with the default spectrogram
// definition runs logmel_fused_kernel with its mel plan (acb_kernels.cu); every other supported (n_fft, hop), and every (n_fft, hop)
// with another definition, runs logmel_stft_kernel<R> with R = n_fft / 32 (acb_logmel_stft.cu).
struct acb_frontend {
    int device = 0;
    int n_fft = 0, hop = 0, n_mels = 0, n_weights = 0, log_kind = 0;
    float clamp_min = 0.f;
    int num_sms = 0;
    int stft_r = 0;        // 0: logmel_fused_kernel; 8, 16 or 32: logmel_stft_kernel<stft_r>
    acb_stft_options opt{};   // spectrogram definition (pad, pad mode, power, magnitude eps); only the STFT kernel takes other than the default
    int groups = 0;        // groups per CTA (template parameter G of the kernel): 4, or 2 when four do not fit in shared memory; 1 for the STFT kernel
    int grid = 0;          // persistent grid (CTAs)
    int smem_bytes = 0;
    int smem_bytes_moments = 0;
    // one device allocation holding every table
    void* d_blob = nullptr;
    const float* d_window = nullptr;
    const float4* d_twiddle = nullptr;
    const float* d_plan_w = nullptr;
    const int* d_plan_woff = nullptr;
    const short* d_plan_trip = nullptr;
    const short* d_plan_band = nullptr;
    const short* d_plan_astart = nullptr;
    int n_plan_w = 0;
    // tables of the STFT kernel: W_N^(r k) per (k, lane r), banded weights, per-band {first bin, bins, weight offset}
    const float2* d_stft_twiddle = nullptr;
    const float* d_stft_weights = nullptr;
    const int4* d_stft_band = nullptr;
    int* d_err = nullptr;  // in-kernel barrier timeout flag
    // host-path streams/events (created lazily)
    cudaStream_t s_in = nullptr, s_out = nullptr;
    std::vector<cudaEvent_t> ev;
    std::mutex mu;
};

namespace acb {
// acb_logmel_stft.cu: the general route.  stft_logmel_supported says whether (n_fft, hop) has a kernel there; stft_frontend_create
// validates the filterbank and builds the handle (n_mels, log_kind, clamp_min and the options are checked by the caller); stft_logmel_launch
// enqueues one launch of the kernel for the batch `p` describes.
bool stft_logmel_supported(int n_fft, int hop);
int stft_frontend_create(acb_frontend** out, int device, int n_fft, int hop, int n_mels, const float* window_host, const float* fb_host,
                         float clamp_min, int log_kind, const acb_stft_options& opt);
void stft_logmel_launch(const acb_frontend* fe, const LogmelParams& p, bool moments, cudaStream_t st);
}  // namespace acb
