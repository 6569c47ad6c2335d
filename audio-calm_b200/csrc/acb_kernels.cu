// B200 (sm_100a) kernels + C ABI of the Audio-CALM log-mel front-end.
//
// Hot path: acb_logmel_forward -> logmel_fused_kernel.  One persistent launch replaces, per clip,
// the ~10 library launches behind MelExtractor.forward (reference preprocess/core.py:50-61:
// reflection_pad1d, framing*window, cuFFT R2C, abs, pow, SGEMM, clamp, log) plus the optional
// pad-to-4 (preprocess/process_dataset.py:146-150), the VAE's affine normalisation
// (models/modeling_vae.py:317-319), the peak normalisation of process_audio_chunk
// (preprocess/core.py:108-110) and the statistics pass (preprocess/compute_mel_stats.py:26-27).
// Every input sample is read from HBM once (plus a 3/16 halo served by L2) and every output value is
// written once.
//
// Structure: a CTA holds G independent groups of 4 warps: 4 groups in one 512-thread CTA per SM by default, or 2 groups in
// each of 2 CTAs per SM when a large filterbank plan does not leave room for four groups' buffers.  A group owns a contiguous
// range of 8-frame tiles, its own sample buffer, scratch and named barrier, so the four groups of an SM run out of phase and
// the FMA-heavy and the shared-memory-heavy parts of different groups overlap.  Per tile a group does:
//   1. one bulk async copy (cp.async.bulk + mbarrier) brings the tile's (8+3)*256 samples into shared memory (edge tiles,
//      which need reflection, are gathered by the group);
//   2. each warp takes one pair of adjacent frames (A, B) and runs ONE complex 1024-point FFT of
//      A + iB as 32 x 32: radix-2 DIT FFT-32 in registers (FMA butterflies), twiddle, transpose through
//      a warp-private padded scratch, second FFT-32; the two real spectra are separated with warp
//      shuffles ((k, 1024-k) partners live in lane 32-j) and |X|^2 goes to the warp's scratch;
//   3. the group applies the banded mel filterbank (1001 non-zero weights instead of a 513x80 GEMM):
//      lanes = 8 bands x 4 frame pairs, warp-uniform trip counts from a host-built balanced schedule;
//      clamp, log, optional affine, optional fp64 moments; interior tiles store straight from registers;
//   4. edge tiles are staged in shared memory and stored with masking, reflected pad-to-4 columns and tail fill.
// The next tile's samples are prefetched while step 3/4 run; the first FFT-32 of the next tile runs before the barrier that
// frees the scratch, so a warp never waits for its group with nothing to do.
#include "audiocalm_b200.h"
#include "acb_fft32.cuh"
#include "acb_logmel_common.cuh"

#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <numeric>
#include <string>
#include <vector>

namespace acb {

constexpr int kNfft = 1024;
constexpr int kHop = 256;
constexpr int kBins = 512;                                   // bins 0..511 are produced; 512 (Nyquist) has zero weight
// Groups per CTA are a template parameter G: 4 groups in ONE 512-thread CTA per SM (the tables are staged once per SM and
// the 16 warps share one instruction footprint; measured 7 % faster than 2 CTAs of 2 groups), or 2 groups x 2 CTAs per SM when
// a large filterbank plan does not leave room for four groups' buffers.
constexpr int kMaxGroups = 4;
constexpr int kTileSamples = (kTileFrames + 3) * kHop;       // 2816 samples staged per tile
constexpr int kRowStride = 36;                               // floats per row of a transpose plane: 4-byte column stores and 16-byte row loads are both conflict-free
constexpr int kPlaneFloats = 32 * kRowStride;                // the real and the imaginary parts are transposed in separate planes
constexpr int kScratchFloats = 2 * kPlaneFloats + 8;         // 2312 floats / warp; == 8 (mod 32): see the mel phase
constexpr int kSlots = 8;                                    // band slots per mel round: lanes = 8 slots x 4 frame pairs
constexpr int kMaxRounds = 4;                                // mel plan: rounds of (8 bands) per warp
constexpr int kMaxWeights = 4096;
constexpr int kOutStageOffset = 2 * kBins;                   // the staged output tile lives above pair 0's power spectrum
static_assert(kScratchFloats % 32 == 8 && kScratchFloats % 4 == 0, "pair stride must be 8 (mod 32) words and 16-byte aligned");
static_assert(kOutStageOffset + kTileFrames * (kMaxMels | 1) <= kScratchFloats, "staged tile must fit above the power spectrum");

thread_local std::string g_last_error;

int fail(int code, const std::string& msg) {   // also used by acb_spectral.cu: one thread-local message for the whole library
    g_last_error = msg;
    return code;
}
static int cuda_fail(cudaError_t e, const char* what) {
    g_last_error = std::string(what) + ": " + cudaGetErrorString(e);
    return ACB_ERR_CUDA;
}
#define ACB_CUDA(call)                                  \
    do {                                                \
        cudaError_t e__ = (call);                       \
        if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
    } while (0)

// --------------------------------------------------------------------------------------------
// device helpers
// --------------------------------------------------------------------------------------------
// ---- mbarrier + 1-D bulk async copy (TMA without a tensor map): sample tiles land in shared memory without LSU work ----
__device__ __forceinline__ unsigned smem_addr(const void* p) { return static_cast<unsigned>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
// Bounded wait: a faulted bulk copy must not hang the GPU box.  Returns false after ~2^26 polls (seconds); the kernel then
// raises its error flag, which acb_frontend_check / the host-buffer paths turn into ACB_ERR_CUDA.
__device__ __forceinline__ bool mbar_wait(unsigned long long* bar, unsigned parity) {
    unsigned ok = 0;
    for (int spin = 0; spin < (1 << 26) && !ok; ++spin) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(ok) : "r"(smem_addr(bar)), "r"(parity) : "memory");
    }
    return ok != 0;
}
__device__ __forceinline__ void bulk_copy_g2s(void* smem, const void* gmem, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_addr(smem)), "l"(gmem), "r"(bytes), "r"(smem_addr(bar)) : "memory");
}

// --------------------------------------------------------------------------------------------
// fused log-mel kernel
// --------------------------------------------------------------------------------------------
struct SmemLayout {
    int samples, scratch, twiddle, window, plan_w, affine, plan_rec, mbar, moments, total_bytes;
};

// Kernels without the moment accumulators: every offset is a compile-time constant of the kernel -- the regions whose size depends on
// the filterbank are sized for kMaxMels (the per-band affine pairs) or placed last (the plan's weights) -- so that no shared-memory
// address has to be derived from kernel parameters inside the tile loop (at the 128-register cap the compiler re-derived the
// mbarrier's, the plan records' and the weights' addresses every iteration instead of keeping them: 0.4633 -> 0.4548 ms at config 2).
// The kernels WITH moments keep the parameter-dependent order: measured with the constant one, 0.545 -> 0.565 ms for the ragged
// statistics launch and 0.512 -> 0.533 ms for features + moments (the register allocation of the longer mel epilogue changes for the
// worse; tools/stats_step.py; constant addresses for the plan records and the barrier alone: 0.571 ms).
__host__ __device__ inline SmemLayout make_smem_layout(int kGroups, int n_mels, int n_plan_w, bool with_moments = false) {
    SmemLayout L;
    int off = 0;  // in 4-byte words
    L.samples = off; off += kGroups * kTileSamples;
    L.scratch = off; off += kGroups * kGroupWarps * kScratchFloats;
    L.twiddle = off; off += 5 * 32 * 4;
    L.window = off; off += 32 * 20;                               // first half only (w[n + N/2] = 1 - w[n]), per lane with a 20-float pitch
    if (!with_moments) {
        L.plan_rec = off; off += kGroupWarps * kMaxRounds * kSlots * 4;   // int4 per (warp, round, slot): the mel phase's per-lane constants
        L.mbar = off; off += 2 * kGroups;                                 // one 8-byte mbarrier per group ("sample tile landed")
        off = (off + 3) & ~3;
        L.affine = off; off += 2 * kMaxMels;                              // float2 per band
        L.plan_w = off; off += (n_plan_w + 3) & ~3;                       // last: the only region of variable size
        L.moments = off;
    } else {
        L.plan_w = off; off += (n_plan_w + 3) & ~3;
        L.affine = off; off += 2 * ((n_mels + 1) & ~1);
        off = (off + 3) & ~3;
        L.plan_rec = off; off += kGroupWarps * kMaxRounds * kSlots * 4;
        L.mbar = off; off += 2 * kGroups;
        L.moments = off; off += kGroups * 4 * n_mels;                     // float2 [kGroups][2][n_mels]
    }
    L.total_bytes = off * 4;
    return L;
}

__device__ __forceinline__ void group_sync(int grp) {   // named barrier of one 4-warp group (barrier 0 is __syncthreads)
    asm volatile("bar.sync %0, %1;" ::"r"(grp + 1), "n"(kGroupThreads) : "memory");
}

// Edge tiles (reflection about sample 0 / L - 1; torch.stft center=True, pad_mode="reflect") and unaligned clips: every thread of the
// group fetches its 22 staged positions with all loads in flight together.  Kept out of line so that its registers do not weigh
// on the hot loop's allocation; slots that belong only to frames >= T get zeros.
__device__ __noinline__ void gather_edge_tile(const float* __restrict__ src, long long g0, long long L, float* s_samples, int gt) {
    static_assert(kTileSamples % kGroupThreads == 0, "whole rounds");
    float v[kTileSamples / kGroupThreads];
#pragma unroll
    for (int k = 0; k < kTileSamples / kGroupThreads; ++k) {
        long long idx = g0 + gt + k * kGroupThreads;
        if (idx < 0) idx = -idx;
        if (idx >= L) idx = 2 * (L - 1) - idx;
        v[k] = (idx >= 0 && idx < L) ? __ldg(src + idx) : 0.f;
    }
#pragma unroll
    for (int k = 0; k < kTileSamples / kGroupThreads; ++k) s_samples[gt + k * kGroupThreads] = v[k];
}

// Stage one tile's samples; the group's mbarrier completes a phase when they have landed.  Called by all threads of the group.
// Interior tiles are ONE bulk async copy issued by one thread (the copy engine writes shared memory and counts the bytes on the
// mbarrier); edge tiles (reflection about sample 0 / L-1, torch.stft center=True pad_mode="reflect") and unaligned clips are
// gathered by the whole group, which then arrives once.
__device__ __forceinline__ void load_tile_samples(const LogmelParams& p, const ClipCursor& t, float* s_samples, int gt, int grp,
                                                  unsigned long long* full) {
    const int f0 = t.tile_in_clip * kTileFrames;
    const long long g0 = (long long)f0 * kHop - kNfft / 2;  // sample index (relative to the clip) of smem slot 0
    const float* src = p.wav + t.wav_base;
    const bool interior = (g0 >= 0) && (g0 + kTileSamples <= t.length);
    if (interior && (reinterpret_cast<uintptr_t>(src + g0) & 15) == 0) {   // group-uniform
        if (gt == 0) {
            mbar_arrive_expect_tx(full, kTileSamples * (unsigned)sizeof(float));
            bulk_copy_g2s(s_samples, src + g0, kTileSamples * (unsigned)sizeof(float), full);
        }
        return;
    }
    gather_edge_tile(src, g0, t.length, s_samples, gt);
    group_sync(grp);
    if (gt == 0) mbar_arrive(full);
}

template <int G, bool kMoments, typename OutT>
__global__ void __launch_bounds__(G * kGroupThreads, G == 4 ? 1 : 2) logmel_fused_kernel(const LogmelParams p) {
    constexpr int kGroups = G;
    constexpr int kThreads = G * kGroupThreads;
    extern __shared__ __align__(16) float smem[];
    const SmemLayout L = make_smem_layout(G, p.n_mels, p.n_plan_w, kMoments);
    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int grp = tid / kGroupThreads;          // which of the CTA's independent groups
    const int gt = tid % kGroupThreads;           // thread index inside the group
    const int gw = gt >> 5;                       // warp index inside the group = frame pair of the tile
    const int n_mels = p.n_mels;
    const int S = out_row_stride(n_mels);
    const bool write_out = p.out != nullptr;      // statistics-only launches have no feature output

    float* s_samples = smem + L.samples + grp * kTileSamples;
    float* s_scratch = smem + L.scratch + grp * kGroupWarps * kScratchFloats;
    float* s_out = s_scratch + kOutStageOffset;   // staged edge tiles: above pair 0's power spectrum, dead during the mel phase
    float4* s_tw4 = reinterpret_cast<float4*>(smem + L.twiddle);
    float* s_win = smem + L.window;
    float* s_pw = smem + L.plan_w;
    float2* s_aff = reinterpret_cast<float2*>(smem + L.affine);   // per band (scale, shift): out = v * scale + shift
    int4* s_rec = reinterpret_cast<int4*>(smem + L.plan_rec);   // {power offset (16-byte units), weight offset (8-byte units), band, trip}
    float2* s_mom = reinterpret_cast<float2*>(smem + L.moments) + grp * 2 * n_mels;   // [2][n_mels] (hi, lo) pairs per group, only when kMoments
    unsigned long long* s_full = reinterpret_cast<unsigned long long*>(smem + L.mbar) + grp;   // "sample tile landed"

    // ---- one-time table staging (whole CTA) ----
    for (int i = tid; i < 5 * 32; i += kThreads) s_tw4[i] = p.twiddle[i];
    for (int i = tid; i < kNfft / 2; i += kThreads)
        s_win[(i & 31) * 20 + (i >> 5)] = p.window[i];      // [lane][row], 20-float pitch: conflict-free 16-byte loads
    for (int i = tid; i < p.n_plan_w; i += kThreads) s_pw[i] = p.plan_w[i];
    for (int i = tid; i < kGroupWarps * kMaxRounds * kSlots; i += kThreads) {
        const int slot = i / kSlots, qq = i - slot * kSlots;
        s_rec[i] = make_int4(p.plan_astart[i] >> 1, (p.plan_woff[slot] >> 1) + qq, p.plan_band[i], p.plan_trip[slot]);
    }
    for (int i = tid; i < n_mels; i += kThreads) {
        float sc = 1.f, sh = 0.f;   // affine == 0: v * 1 + 0 is exact
        if (p.affine == 1) { sc = p.affine_inv_std; sh = -p.affine_mean * p.affine_inv_std; }
        else if (p.affine == 2) { sc = 1.f / __ldg(p.bin_std + i); sh = -__ldg(p.bin_mean + i) * sc; }
        s_aff[i] = make_float2(sc, sh);
    }
    if (kMoments)
        for (int i = gt; i < 2 * n_mels; i += kGroupThreads) s_mom[i] = make_float2(0.f, 0.f);
    if (gt == 0) {
        mbar_init(s_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    // ---- this group's contiguous tile range ----
    const long long n_groups = (long long)gridDim.x * kGroups, g_index = (long long)blockIdx.x * kGroups + grp;
    const long long t_begin = (long long)p.n_tiles * g_index / n_groups;
    const long long t_end = (long long)p.n_tiles * (g_index + 1) / n_groups;

    ClipCursor cur;
    bool staged = false;          // group-uniform: a sample tile was requested for the current tile
    unsigned full_parity = 0;
    if (t_begin < t_end) {
        cursor_init(p, cur, t_begin, kHop);
        staged = cur.tile_in_clip * kTileFrames < cur.frames;
        if (staged) load_tile_samples(p, cur, s_samples, gt, grp, s_full);
    }

    // ---- per-thread constants of the mel phase: lanes = 8 band slots x 4 frame pairs ----
    // A quarter-warp's 16-byte power loads touch 2 slots x 4 pairs.  The pair stride is 8 (mod 32) words, so one slot's four
    // pairs fall on bank groups {0, 8, 16, 24} + 4 * ((astart/2 + i) mod 2): the host plan gives the two slots of a quarter
    // opposite parity of astart/2, which makes the load conflict-free.
    const int q = lane >> 2;     // band slot within a round
    const int pl = lane & 3;     // frame pair served by this lane in the mel phase
    const float* pair_scratch = s_scratch + pl * kScratchFloats;
    float* scr = s_scratch + gw * kScratchFloats;
    float2* scr2 = reinterpret_cast<float2*>(scr);

    for (long long tile = t_begin; tile < t_end; ++tile) {
        if (staged) {             // the tile's samples have landed (bulk copy counted in, or the gathering group arrived)
            if (!mbar_wait(s_full, full_parity) && lane == 0) atomicExch(p.error_flag, 1);
            full_parity ^= 1;
        }

        const int f0 = cur.tile_in_clip * kTileFrames;
        const bool has_frames = f0 < cur.frames;  // false for pure tail-fill tiles
        const bool active = has_frames && f0 + 2 * gw < cur.frames;   // this warp's frame pair exists

        // ================= phase 1: one frame pair per warp =================
        // The first FFT-32 needs only the samples and registers, so it runs BEFORE the barrier that frees the scratch: a warp that
        // is done with the previous tile's mel phase does not wait for the slower warps of its group here.
        if (active) {
            float2 pr[16], pi[16];   // element k < 16 in .x, element k + 16 in .y (see fft32_packed)
            {
                // Hann window folded into the first radix-2 stage: positions (2j, 2j+1) of the bit-reversed order hold samples
                // n1 and n1 + 16 (x[2j] = a*wa + b*wb, x[2j+1] = a*wa - b*wb); positions 16 higher hold samples n1 + 1, so a
                // register pair is two adjacent sample rows.  Frame A is the real part, frame B (one hop later) the imaginary.
                const float* sp = s_samples + (2 * gw) * kHop + lane;
                float2 v[20];
#pragma unroll
                for (int r = 0; r < 20; ++r) v[r] = make_float2(sp[32 * (2 * r)], sp[32 * (2 * r + 1)]);
                // the lane's 16 window values, stored per lane: four 16-byte loads instead of sixteen 4-byte ones
                float4 w4[4];
                const float4* wq = reinterpret_cast<const float4*>(s_win + lane * 20);
#pragma unroll
                for (int u = 0; u < 4; ++u) w4[u] = wq[u];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int t = brev5(2 * j) >> 1;      // sample rows n1 = 2t, 2t + 1 (n1 < 16)
                    const float2 wa = (t & 1) ? make_float2(w4[t >> 1].z, w4[t >> 1].w) : make_float2(w4[t >> 1].x, w4[t >> 1].y);
                    // periodic Hann: w[n + N/2] = 1 - w[n], so b (1 - w) = b - b w is one FMA, and a w +- that another
                    const float2 br = __ffma2_rn(neg2(v[t + 8]), wa, v[t + 8]), bi = __ffma2_rn(neg2(v[t + 12]), wa, v[t + 12]);
                    pr[2 * j] = __ffma2_rn(v[t], wa, br);
                    pr[2 * j + 1] = __ffma2_rn(v[t], wa, neg2(br));
                    pi[2 * j] = __ffma2_rn(v[t + 4], wa, bi);
                    pi[2 * j + 1] = __ffma2_rn(v[t + 4], wa, neg2(bi));
                }
            }
            fft32_packed_from_stage2(pr, pi);  // over n1 -> k1 (natural order)
            group_sync(grp);  // the group is done with the previous tile's mel phase / staged store: the scratch is free
            // twiddle W_1024^(k1*lane), then transposed store plane[k1][lane].  The twiddles of a lane are powers of W^lane, kept
            // as pairs T[k] = (W^(k*lane), W^((k+16)*lane)): four chains T[k+4] = T[k] * W^(4*lane) seeded with exact values
            // (3 steps deep) cost packed FMA-pipe instructions instead of an 8-byte shared-memory load per twiddle.
            {
                float* pre = scr + lane;
                float* pim = scr + kPlaneFloats + lane;
                float2 tr[4], ti[4];
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float4 sd = s_tw4[c * 32 + lane];
                    tr[c] = make_float2(sd.x, sd.y);
                    ti[c] = make_float2(sd.z, sd.w);
                }
                const float4 w4 = s_tw4[4 * 32 + lane];
                const float2 w4r = bcast2(w4.x), w4i = bcast2(w4.y);
#pragma unroll
                for (int k = 0; k < 16; ++k) {
                    const int c = k & 3;
                    const float2 yr = __ffma2_rn(neg2(pi[k]), ti[c], __fmul2_rn(pr[k], tr[c]));
                    const float2 yi = __ffma2_rn(pr[k], ti[c], __fmul2_rn(pi[k], tr[c]));
                    pre[k * kRowStride] = yr.x;
                    pre[(k + 16) * kRowStride] = yr.y;
                    pim[k * kRowStride] = yi.x;
                    pim[(k + 16) * kRowStride] = yi.y;
                    if (k + 4 < 16) {
                        const float2 nr = __ffma2_rn(neg2(ti[c]), w4i, __fmul2_rn(tr[c], w4r));
                        ti[c] = __ffma2_rn(tr[c], w4i, __fmul2_rn(ti[c], w4r));
                        tr[c] = nr;
                    }
                }
            }
            __syncwarp();
            // lane j = k1 now owns row j: the 32 values over n2, four per 16-byte load.  Values n2 = 4h, 4h+1 go to bit-reversed
            // positions brev3(h) and brev3(h) + 16 -- one register pair -- and n2 = 4h+2, 4h+3 to the pair 8 places up.
            {
                const float4* re4 = reinterpret_cast<const float4*>(scr + lane * kRowStride);
                const float4* im4 = reinterpret_cast<const float4*>(scr + kPlaneFloats + lane * kRowStride);
#pragma unroll
                for (int h = 0; h < 8; ++h) {
                    const float4 zr = re4[h], zi = im4[h];
                    pr[brev3(h)] = make_float2(zr.x, zr.y);
                    pr[brev3(h) + 8] = make_float2(zr.z, zr.w);
                    pi[brev3(h)] = make_float2(zi.x, zi.y);
                    pi[brev3(h) + 8] = make_float2(zi.z, zi.w);
                }
            }
            __syncwarp();
            fft32_packed(pr, pi);  // over n2 -> k2 ; lane j holds Z[j + 32*k2]
            // separate the two real spectra and take |X|^2 (x4; the 1/4 is folded into the weights):
            //   Z[k] = a+ib, Z[1024-k] = c+id  =>  4|XA|^2 = (a+c)^2+(b-d)^2 , 4|XB|^2 = (a-c)^2+(b+d)^2
            // Z[1024-k] for k = j + 32m lives in lane (32-j)&31, element 31-m (element 32-m when j == 0).
            const int src_lane = (32 - lane) & 31;
#pragma unroll
            for (int m = 0; m < 16; ++m) {
                // elements 31-m and (32-m)&31: 31-m >= 16 is the high half of pair 15-m; (32-m)&31 is element 0 for m == 0
                const float alt_r = (m == 0) ? pr[0].x : pr[16 - m].y;
                const float alt_i = (m == 0) ? pi[0].x : pi[16 - m].y;
                const float offer_r = (lane == 0) ? alt_r : pr[15 - m].y;
                const float offer_i = (lane == 0) ? alt_i : pi[15 - m].y;
                const float c = __shfl_sync(0xffffffffu, offer_r, src_lane);
                const float d = __shfl_sync(0xffffffffu, offer_i, src_lane);
                const float a = pr[m].x, b = pi[m].x;
                const float apc = a + c, bmd = b - d, amc = a - c, bpd = b + d;
                const float pa = fmaf(apc, apc, bmd * bmd);
                const float pb = fmaf(amc, amc, bpd * bpd);
                scr2[lane + 32 * m] = make_float2(pa, pb);
            }
        }
        else {
            group_sync(grp);  // warps without a frame pair (tail of a clip) take part in the same barrier
        }
        // the mel phase's per-lane constants are loaded one round ahead; the first record's latency hides behind the barrier
        const int4* my_rec = s_rec + (gw * kMaxRounds) * kSlots + q;
        int4 rec_next = my_rec[0];
        group_sync(grp);  // power spectra of the group's pairs visible; sample tile is free again

        // prefetch the next tile's samples while the mel phase runs
        ClipCursor nxt = cur;
        staged = false;
        if (tile + 1 < t_end) {
            cursor_advance(p, nxt, kHop);
            staged = nxt.tile_in_clip * kTileFrames < nxt.frames;
            if (staged) load_tile_samples(p, nxt, s_samples, gt, grp, s_full);
        }

        // interior tile: every frame exists and none is a pad-to-4 source -> mel-major results go straight to global
        // memory from the mel phase (4 lanes x 2 frames = 32 contiguous bytes per band); other tiles and the
        // time-major layout are staged in shared memory and stored by store_tile().
        const int pad = cur.frames_padded - cur.frames;
        const bool direct = !p.time_major && (f0 + kTileFrames - 1 <= cur.frames - 2 - pad);

        // ================= phase 2: banded mel projection, clamp, log, affine, moments =================
        if (has_frames) {
            const int fA = f0 + 2 * pl;
            OutT* out_clip = reinterpret_cast<OutT*>(p.out) + cur.out_base;
            const bool pair_store = ((cur.cap & 1) == 0) && ((reinterpret_cast<uintptr_t>(out_clip) & (2 * sizeof(OutT) - 1)) == 0);
            for (int r = 0; r < kMaxRounds; ++r) {
                const int4 rec = rec_next;
                const int trip = rec.w;
                if (trip == 0) break;  // warp-uniform; rounds are filled in order
                if (r + 1 < kMaxRounds) rec_next = my_rec[(r + 1) * kSlots];
                const int b = rec.z;
                const float2 af = s_aff[b < 0 ? 0 : b];   // issued early: needed only after the log
                const float4* p4 = reinterpret_cast<const float4*>(pair_scratch) + rec.x;   // two bins x (A, B)
                const float2* w2 = reinterpret_cast<const float2*>(s_pw) + rec.y;
                float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
                const int half_trip = trip >> 1;
#pragma unroll 4
                for (int i = 0; i < half_trip; ++i) {
                    const float4 pw = p4[i];
                    const float2 w = w2[kSlots * i];
                    acc0 = fmaf(w.x, pw.x, acc0);
                    acc1 = fmaf(w.x, pw.y, acc1);
                    acc2 = fmaf(w.y, pw.z, acc2);
                    acc3 = fmaf(w.y, pw.w, acc3);
                }
                const float mA = (acc0 + acc2) * cur.gain, mB = (acc1 + acc3) * cur.gain;
                float vA = (mA > p.clamp_min) ? lg2_normal(mA) * p.log_scale : p.log_floor;
                float vB = (mB > p.clamp_min) ? lg2_normal(mB) * p.log_scale : p.log_floor;
                if (kMoments) {
                    // frames T-2-j (j < pad) are stored twice (reflected pad-to-4 columns) and counted twice.  The tile's 8 frames of a
                    // band are summed in fp32 (two values per lane, then the slot's 4 pair lanes by shuffle) and enter the group's
                    // accumulators once per (band, tile).  The accumulators are compensated fp32 pairs (hi, lo), exact to ~2^-46 and
                    // turned into fp64 once at the end of the kernel: vector fp64 is a scarce pipe on B200.
                    float s = 0.f, s2 = 0.f;
                    if (b >= 0 && fA < cur.frames) {
                        const float c = (fA <= cur.frames - 2 && fA > cur.frames - 2 - pad) ? 2.f : 1.f;
                        s = c * vA;
                        s2 = s * vA;
                    }
                    if (b >= 0 && fA + 1 < cur.frames) {
                        const float c = (fA + 1 <= cur.frames - 2 && fA + 1 > cur.frames - 2 - pad) ? 2.f : 1.f;
                        const float cv = c * vB;
                        s += cv;
                        s2 = fmaf(cv, vB, s2);
                    }
                    // The 4 pair lanes of a slot are a contiguous, aligned lane group (all 32 lanes take part).  Lanes 0, 1 of the group
                    // end up with the sum, lanes 2, 3 with the sum of squares: in the first step a lane hands over the value its half
                    // does not keep, so two shuffles reduce both, and ONE compensated add per round -- lane 0 into the band's sum,
                    // lane 2 into its sum of squares -- updates both accumulators.  Same additions in the same order as reducing the
                    // two values separately ((v0 + v2) + (v1 + v3)): the moments are bit-identical.
                    const bool upper = (pl & 2) != 0;
                    float keep = (upper ? s2 : s) + __shfl_xor_sync(0xffffffffu, upper ? s : s2, 2);
                    keep += __shfl_xor_sync(0xffffffffu, keep, 1);
                    if ((pl & 1) == 0 && b >= 0)   // each band has exactly one owner slot per group
                        two_sum_add(s_mom[(upper ? n_mels : 0) + b], keep);
                }
                if (b >= 0) {
                    vA = fmaf(vA, af.x, af.y);
                    vB = fmaf(vB, af.x, af.y);
                    if (direct) {
                        if (write_out) {
                            OutT* dst = out_clip + (size_t)((unsigned)b * (unsigned)cur.cap) + fA;
                            if (pair_store) {   // frames A and B in one store (the row pitch and the clip's base keep the pair aligned)
                                store_pair<OutT>(dst, vA, vB);
                            } else {
                                dst[0] = to_out<OutT>(vA);
                                dst[1] = to_out<OutT>(vB);
                            }
                        }
                    } else {
                        s_out[(2 * pl) * S + b] = vA;
                        s_out[(2 * pl + 1) * S + b] = vB;
                    }
                }
            }
        }
        if (!direct) {   // group-uniform
            group_sync(grp);  // output tile staged
            if (write_out) {
                store_tile<OutT>(p, cur, s_out, n_mels, S, gt);
                if (p.fill_tail && p.tile_start != nullptr && cur.tile_in_clip == cur.tiles_in_clip - 1) fill_row_tail<OutT>(p, cur, n_mels, gt);
            }
        }
        cur = nxt;
    }

    if (kMoments) {
        group_sync(grp);
        for (int i = gt; i < 2 * n_mels; i += kGroupThreads)
            p.moments_partial[(size_t)g_index * 2 * n_mels + i] = (double)s_mom[i].x + (double)s_mom[i].y;
    }
}

// Sum the per-group partials in a fixed order (deterministic) and add into the running accumulators: one warp per value,
// lanes stride over the partials (independent loads), then a shuffle tree.
__global__ void __launch_bounds__(256) moments_reduce_kernel(const double* __restrict__ partial, int n_parts, int n_vals, double* __restrict__ acc) {
    const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= n_vals) return;
    double s = 0.0;
    for (int k = lane; k < n_parts; k += 32) s += partial[(size_t)k * n_vals + i];
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) acc[i] += s;
}

// --------------------------------------------------------------------------------------------
// per-clip peak, process_audio_chunk
// --------------------------------------------------------------------------------------------
// max(m, |v|) that keeps a NaN once seen, like torch.max (preprocess/core.py:108: a NaN peak fails `peak > 0`, so the clip is left
// unscaled).  As a bit pattern a quiet NaN (0x7fc00000) is above every finite non-negative float, so atomicMax keeps it too.
__device__ __forceinline__ float nanmax_abs(float m, float v) {
    const float a = fabsf(v);
    return (a != a || m != m) ? __uint_as_float(0x7fc00000u) : fmaxf(m, a);
}
__device__ __forceinline__ float nanmax(float a, float b) { return (a != a || b != b) ? __uint_as_float(0x7fc00000u) : fmaxf(a, b); }

__global__ void peak_abs_kernel(const float* __restrict__ wav, const long long* __restrict__ clip_offset,
                                const long long* __restrict__ clip_length, long long clip_stride, long long uniform_length,
                                int blocks_per_clip, float* __restrict__ peak_out) {
    const int clip = blockIdx.x / blocks_per_clip;
    const int part = blockIdx.x - clip * blocks_per_clip;
    const long long base = clip_offset ? clip_offset[clip] : (long long)clip * clip_stride;
    const long long len = clip_length ? clip_length[clip] : uniform_length;
    const long long chunk = (len + blocks_per_clip - 1) / blocks_per_clip;
    const long long lo = (long long)part * chunk;
    const long long hi = min(len, lo + chunk);
    const float* src = wav + base;
    float m = 0.f;
    // scalar head until 16-byte aligned, then float4 body
    const long long head_end = min(hi, lo + ((4 - ((base + lo) & 3)) & 3));
    for (long long k = lo + threadIdx.x; k < head_end; k += blockDim.x) m = nanmax_abs(m, src[k]);
    const long long body0 = head_end;
    const long long nvec = (hi > body0 && (reinterpret_cast<uintptr_t>(src + body0) & 15) == 0) ? (hi - body0) / 4 : 0;
    const float4* v4 = reinterpret_cast<const float4*>(src + body0);
    for (long long k = threadIdx.x; k < nvec; k += blockDim.x) {
        const float4 v = __ldg(v4 + k);
        m = nanmax_abs(nanmax_abs(nanmax_abs(nanmax_abs(m, v.x), v.y), v.z), v.w);
    }
    for (long long k = body0 + nvec * 4 + threadIdx.x; k < hi; k += blockDim.x) m = nanmax_abs(m, src[k]);
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) m = nanmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    __shared__ float s_m[32];
    if ((threadIdx.x & 31) == 0) s_m[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x < 32) {
        m = (threadIdx.x < (blockDim.x >> 5)) ? s_m[threadIdx.x] : 0.f;
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) m = nanmax(m, __shfl_xor_sync(0xffffffffu, m, o));
        // non-negative floats order like their bit patterns
        if (threadIdx.x == 0) atomicMax(reinterpret_cast<unsigned int*>(peak_out + clip), __float_as_uint(m));
    }
}

// channel mean (sequential fp32 sum then divide, as torch.mean over dim 0 does) + peak.  16-byte accesses when every channel row
// is 16-byte aligned (length % 4 == 0 and aligned bases), scalar otherwise; `peak` may be null (mixdown only).
__global__ void __launch_bounds__(256) mixdown_peak_kernel(const float* __restrict__ wav_cl, int channels, long long length,
                                                           float* __restrict__ out, float* __restrict__ peak) {
    const long long stride = (long long)gridDim.x * blockDim.x, t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool vec = (length & 3) == 0 && ((reinterpret_cast<uintptr_t>(wav_cl) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
    const float inv_c = (float)channels;
    float m = 0.f;
    if (vec) {
        const long long n4 = length >> 2;
        for (long long i = t0; i < n4; i += stride) {
            float4 v = __ldg(reinterpret_cast<const float4*>(wav_cl) + i);
            if (channels > 1) {
                for (int c = 1; c < channels; ++c) {
                    const float4 u = __ldg(reinterpret_cast<const float4*>(wav_cl + (long long)c * length) + i);
                    v.x += u.x; v.y += u.y; v.z += u.z; v.w += u.w;
                }
                v.x = __fdiv_rn(v.x, inv_c); v.y = __fdiv_rn(v.y, inv_c); v.z = __fdiv_rn(v.z, inv_c); v.w = __fdiv_rn(v.w, inv_c);
            }
            reinterpret_cast<float4*>(out)[i] = v;
            m = nanmax_abs(nanmax_abs(nanmax_abs(nanmax_abs(m, v.x), v.y), v.z), v.w);
        }
    } else {
        for (long long i = t0; i < length; i += stride) {
            float v = wav_cl[i];
            if (channels > 1) {
                for (int c = 1; c < channels; ++c) v += wav_cl[(long long)c * length + i];
                v = __fdiv_rn(v, inv_c);
            }
            out[i] = v;
            m = nanmax_abs(m, v);
        }
    }
    if (peak == nullptr) return;
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) m = nanmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    __shared__ float s_m[8];
    if ((threadIdx.x & 31) == 0) s_m[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); ++w) m = nanmax(m, s_m[w]);
        atomicMax(reinterpret_cast<unsigned int*>(peak), __float_as_uint(m));   // non-negative floats order like their bit patterns
    }
}

// wav / (peak + 1e-8) * 0.95, division first (preprocess/core.py:110)
__global__ void __launch_bounds__(256) peak_scale_kernel(float* __restrict__ x, long long length, const float* __restrict__ peak) {
    const float pk = *peak;
    if (!(pk > 0.f)) return;
    const float d = pk + 1e-8f;
    const long long stride = (long long)gridDim.x * blockDim.x, t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long n4 = (reinterpret_cast<uintptr_t>(x) & 15) == 0 ? (length >> 2) : 0;
    for (long long i = t0; i < n4; i += stride) {
        float4 v = reinterpret_cast<float4*>(x)[i];
        v.x = __fmul_rn(__fdiv_rn(v.x, d), 0.95f); v.y = __fmul_rn(__fdiv_rn(v.y, d), 0.95f);
        v.z = __fmul_rn(__fdiv_rn(v.z, d), 0.95f); v.w = __fmul_rn(__fdiv_rn(v.w, d), 0.95f);
        reinterpret_cast<float4*>(x)[i] = v;
    }
    for (long long i = n4 * 4 + t0; i < length; i += stride) x[i] = __fmul_rn(__fdiv_rn(x[i], d), 0.95f);
}

// --------------------------------------------------------------------------------------------
// standalone moments over stored features, per-utterance normalisation
// --------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ float load_feat(const T* p, long long i);
template <>
__device__ __forceinline__ float load_feat<float>(const float* p, long long i) { return __ldg(p + i); }
template <>
__device__ __forceinline__ float load_feat<__nv_bfloat16>(const __nv_bfloat16* p, long long i) { return __bfloat162float(p[i]); }

// One 16-byte load of a row as floats: four fp32 or eight bf16 consecutive features.
template <typename T>
struct FeatVec;
template <>
struct FeatVec<float> {
    static constexpr int kPer = 4;
    static __device__ __forceinline__ void load(const float* p, float (&f)[4]) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(p));
        f[0] = a.x; f[1] = a.y; f[2] = a.z; f[3] = a.w;
    }
};
template <>
struct FeatVec<__nv_bfloat16> {
    static constexpr int kPer = 8;
    static __device__ __forceinline__ void load(const __nv_bfloat16* p, float (&f)[8]) {
        const uint4 a = __ldg(reinterpret_cast<const uint4*>(p));
        const unsigned w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) { f[2 * k] = __uint_as_float(w[k] << 16); f[2 * k + 1] = __uint_as_float(w[k] & 0xffff0000u); }
    }
};

// One warp per (clip, band) row; rows are dealt round-robin to the grid's warps.  Lane l takes the 16-byte group l, l + 32, ... of the
// row (every load instruction of the warp covers 512 contiguous bytes) and keeps 8 loads in flight -- 4 KB per warp, enough bytes in
// flight to cover HBM latency at 8 warps x 8 CTAs per SM.  Every value enters fp64 accumulators (B200 has full-rate fp64 units: 2 fp64
// operations per 4 bytes read are far below their rate), so the moments are exact to fp64 rounding.  Per-warp fp64 accumulators in
// shared memory, combined in a fixed order -> deterministic partial per CTA.
template <typename T>
__global__ void __launch_bounds__(256) moments_rows_kernel(const T* __restrict__ feat, int n_clips, int n_mels, long long cap,
                                                           long long clip_stride, const long long* __restrict__ frames,
                                                           double* __restrict__ partial) {
    extern __shared__ double s_acc[];  // [warps][2][n_mels]
    const int warps = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < warps * 2 * n_mels; i += blockDim.x) s_acc[i] = 0.0;
    __syncthreads();
    double* my = s_acc + (size_t)warp * 2 * n_mels;
    const long long n_rows = (long long)n_clips * n_mels;
    for (long long row = (long long)blockIdx.x * warps + warp; row < n_rows; row += (long long)gridDim.x * warps) {
        const int clip = (int)(row / n_mels), b = (int)(row - (long long)clip * n_mels);
        const long long n_fr = frames ? frames[clip] : cap;
        const T* src = feat + (long long)clip * clip_stride + (long long)b * cap;
        double sa[2] = {0.0, 0.0}, sb[2] = {0.0, 0.0};
        // scalar head up to the first 16-byte boundary, vector body, scalar tail
        constexpr int kPer = FeatVec<T>::kPer, kDeep = 8;
        const int mis = (int)((reinterpret_cast<uintptr_t>(src) & 15) / sizeof(T));
        const long long head = min(n_fr, (long long)((mis ? (16 / (int)sizeof(T)) - mis : 0)));
        for (long long i = lane; i < head; i += 32) { const double v = (double)load_feat<T>(src, i); sa[0] += v; sb[0] += v * v; }
        const long long nv = (n_fr - head) / kPer;
        const T* body = src + head;
        for (long long i = lane; i < nv; i += 32 * kDeep) {          // kDeep predicated 16-byte groups per lane and trip, all loads up front
            float f[kDeep][kPer];
#pragma unroll
            for (int k = 0; k < kDeep; ++k) {
                if (i + 32 * k < nv) {
                    FeatVec<T>::load(body + kPer * (i + 32 * k), f[k]);
                } else {
#pragma unroll
                    for (int j = 0; j < kPer; ++j) f[k][j] = 0.f;
                }
            }
#pragma unroll
            for (int k = 0; k < kDeep; ++k) {
#pragma unroll
                for (int j = 0; j < kPer; ++j) { const double v = (double)f[k][j]; sa[j & 1] += v; sb[j & 1] = fma(v, v, sb[j & 1]); }
            }
        }
        for (long long t = head + nv * kPer + lane; t < n_fr; t += 32) { const double v = (double)load_feat<T>(src, t); sa[1] += v; sb[1] += v * v; }
        double s = sa[0] + sa[1], s2 = sb[0] + sb[1];
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) {
            s += __shfl_xor_sync(0xffffffffu, s, o);
            s2 += __shfl_xor_sync(0xffffffffu, s2, o);
        }
        if (lane == 0) { my[b] += s; my[n_mels + b] += s2; }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * n_mels; i += blockDim.x) {
        double s = 0.0;
        for (int w = 0; w < warps; ++w) s += s_acc[(size_t)w * 2 * n_mels + i];
        partial[(size_t)blockIdx.x * 2 * n_mels + i] = s;
    }
}

// (x - mean_t) / max(std_t, min_std) per (clip, band) row, unbiased std (eval/eval_vae.py:80-82).
// Register form: one WARP per row, the row (up to 32 * 4 * kVecs frames) is read from HBM once with all of a lane's 16-byte loads in
// flight together and stays in registers for the mean, the variance and the write: one read + one write of the features, no barrier.
// Per-lane partial sums are fp32 (four interleaved accumulators over <= 64 values), the cross-lane reduction and the division are fp64.
template <int kVecs>
__global__ void __launch_bounds__(256) normalize_rows_warp_kernel(const float* __restrict__ feat, float* __restrict__ out, long long n_rows,
                                                                  int n_mels, long long cap, const long long* __restrict__ frames, float min_std) {
    const long long r = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r >= n_rows) return;
    const int lane = threadIdx.x & 31;
    const long long T = frames ? frames[r / n_mels] : cap;
    const float4* src = reinterpret_cast<const float4*>(feat + r * cap);
    float4* dst = reinterpret_cast<float4*>(out + r * cap);
    const int T4 = (int)((T + 3) >> 2);             // 16-byte groups that hold valid frames (cap % 4 == 0: the last one is inside the row)
    float4 v[kVecs];
#pragma unroll
    for (int k = 0; k < kVecs; ++k) {
        const int i = k * 32 + lane;
        v[k] = i < T4 ? __ldg(src + i) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    // frames beyond T inside the last group do not count
    const int last = T4 - 1, rem = (int)(T - 4LL * last);      // valid elements of the last group (1..4)
#pragma unroll
    for (int k = 0; k < kVecs; ++k)
        if (k * 32 + lane == last) {
            if (rem < 2) v[k].y = 0.f;
            if (rem < 3) v[k].z = 0.f;
            if (rem < 4) v[k].w = 0.f;
        }
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
    for (int k = 0; k < kVecs; ++k) { a0 += v[k].x; a1 += v[k].y; a2 += v[k].z; a3 += v[k].w; }
    double s = ((double)a0 + (double)a1) + ((double)a2 + (double)a3);
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    const float mean = (float)(s / (double)T);
    a0 = a1 = a2 = a3 = 0.f;
#pragma unroll
    for (int k = 0; k < kVecs; ++k) {
        const int i = k * 32 + lane;
        if (i < T4) {
            const bool is_last = i == last;
            const float dx = v[k].x - mean, dy = v[k].y - mean, dz = v[k].z - mean, dw = v[k].w - mean;
            a0 = fmaf(dx, dx, a0);
            if (!is_last || rem >= 2) a1 = fmaf(dy, dy, a1);
            if (!is_last || rem >= 3) a2 = fmaf(dz, dz, a2);
            if (!is_last || rem >= 4) a3 = fmaf(dw, dw, a3);
        }
    }
    double s2 = ((double)a0 + (double)a1) + ((double)a2 + (double)a3);
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    const float sd = fmaxf((float)sqrt(s2 / (double)(T > 1 ? T - 1 : 1)), min_std);
#pragma unroll
    for (int k = 0; k < kVecs; ++k) {
        const int i = k * 32 + lane;
        if (i < T4) {
            float4 y = make_float4(__fdiv_rn(v[k].x - mean, sd), __fdiv_rn(v[k].y - mean, sd), __fdiv_rn(v[k].z - mean, sd), __fdiv_rn(v[k].w - mean, sd));
            if (i == last && rem < 4) {              // keep what lies beyond the clip's frames untouched
                const float4 old = dst[i];
                if (rem < 2) y.y = old.y;
                if (rem < 3) y.z = old.z;
                y.w = old.w;
            }
            dst[i] = y;
        }
    }
}

// General form (any length, any alignment): one CTA per row, three passes (the re-reads hit L1 / L2), fp64 sums.
__global__ void __launch_bounds__(128) normalize_rows_kernel(const float* __restrict__ feat, float* __restrict__ out, int n_mels,
                                                             long long cap, const long long* __restrict__ frames, float min_std) {
    const int clip = blockIdx.x / n_mels;
    const long long T = frames ? frames[clip] : cap;
    const float* src = feat + (long long)blockIdx.x * cap;
    float* dst = out + (long long)blockIdx.x * cap;
    __shared__ double s_red[4];
    __shared__ float s_stat[2];
    double s = 0.0;
    for (long long i = threadIdx.x; i < T; i += blockDim.x) s += (double)src[i];
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) s_stat[0] = (float)((s_red[0] + s_red[1] + s_red[2] + s_red[3]) / (double)T);
    __syncthreads();
    const float mean = s_stat[0];
    double s2 = 0.0;
    for (long long i = threadIdx.x; i < T; i += blockDim.x) {
        const double d = (double)src[i] - (double)mean;
        s2 += d * d;
    }
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = s2;
    __syncthreads();
    if (threadIdx.x == 0) {
        const double var = (s_red[0] + s_red[1] + s_red[2] + s_red[3]) / (double)(T > 1 ? T - 1 : 1);
        s_stat[1] = fmaxf((float)sqrt(var), min_std);
    }
    __syncthreads();
    const float sd = s_stat[1];
    for (long long i = threadIdx.x; i < T; i += blockDim.x) dst[i] = __fdiv_rn(src[i] - mean, sd);
}

// --------------------------------------------------------------------------------------------
// 16-bit PCM transport: int16 samples -> fp32 in [-1, 1) exactly as torchaudio.load(normalize=True) scales them (x / 32768)
// --------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pcm16_to_float_kernel(const short* __restrict__ in, float* __restrict__ out, long long n, float scale) {
    const long long n8 = ((reinterpret_cast<uintptr_t>(in) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0) ? n / 8 : 0;
    const long long stride = (long long)gridDim.x * blockDim.x, t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (long long i = t0; i < n8; i += stride) {   // 16 bytes in, 32 bytes out per thread and step
        const int4 v = __ldg(reinterpret_cast<const int4*>(in) + i);
        const int w[4] = {v.x, v.y, v.z, v.w};
        float f[8];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            f[2 * k] = (float)(short)(w[k] & 0xffff) * scale;
            f[2 * k + 1] = (float)(w[k] >> 16) * scale;
        }
        float4* o = reinterpret_cast<float4*>(out) + 2 * i;
        o[0] = make_float4(f[0], f[1], f[2], f[3]);
        o[1] = make_float4(f[4], f[5], f[6], f[7]);
    }
    for (long long i = n8 * 8 + t0; i < n; i += stride) out[i] = (float)in[i] * scale;
}

// --------------------------------------------------------------------------------------------
// training-feed collation of stored features (train/train_vae.py:83-116, train/train_calm.py:205-215)
// --------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ T from_float(float v);
template <>
__device__ __forceinline__ float from_float<float>(float v) { return v; }
template <>
__device__ __forceinline__ __nv_bfloat16 from_float<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// out[b][d][t] = feat[b][d][start[b] + t] while start[b] + t < frames[b], else pad: the crop / zero-pad of MelDataset.__getitem__
// followed by the stack of data_collator.  One warp per (clip, band) row, rows dealt round-robin over a grid sized to the chip; a
// lane moves 4 consecutive frames per step (16-byte store when the output row allows it; the crop start is arbitrary, so the
// loads are scalar but coalesced).
template <typename T>
__global__ void __launch_bounds__(256) crop_pad_kernel(const T* __restrict__ feat, int n_clips, int n_mels, long long cap, long long clip_stride,
                                                       const long long* __restrict__ frames, const long long* __restrict__ start,
                                                       T* __restrict__ out, long long out_frames, float pad_value) {
    const int warps = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long n_rows = (long long)n_clips * n_mels;
    const T padv = from_float<T>(pad_value);
    const bool vec = sizeof(T) == 4 && (out_frames & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0;
    for (long long row = (long long)blockIdx.x * warps + warp; row < n_rows; row += (long long)gridDim.x * warps) {
        const int clip = (int)(row / n_mels), b = (int)(row - (long long)clip * n_mels);
        const long long n = frames ? frames[clip] : cap;
        const long long s0 = start ? start[clip] : 0;
        const T* src = feat + (long long)clip * clip_stride + (long long)b * cap;
        T* dst = out + row * out_frames;
        if (vec) {
            if constexpr (sizeof(T) == 4) {
                for (long long t = 4 * lane; t < out_frames; t += 128) {
                    T v[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) { const long long f = s0 + t + j; v[j] = (f >= 0 && f < n) ? src[f] : padv; }
                    *reinterpret_cast<float4*>(dst + t) = make_float4(v[0], v[1], v[2], v[3]);
                }
            }
        } else {
            for (long long t = lane; t < out_frames; t += 32) {
                const long long f = s0 + t;
                dst[t] = (f >= 0 && f < n) ? src[f] : padv;
            }
        }
    }
}

// Ragged time-major features [sum T_i][dim] -> channels-first padded batch out[b][d][t] (CalmCollator: pad_sequence of (T, D)
// items, then transpose(1, 2)), with the optional time mask of _apply_spec_augment (frames [mask_start, mask_start + mask_len)
// set to 0).  64 x 64 tiles go through shared memory: 16-byte global reads along the feature dimension, 16-byte global writes
// along time (when rows are 16-byte aligned; scalar otherwise), 16 values per thread in flight.
template <typename T>
__global__ void __launch_bounds__(256) pad_transpose_kernel(const T* __restrict__ feat, const long long* __restrict__ row_offset,
                                                            const long long* __restrict__ lens, int dim, T* __restrict__ out,
                                                            long long out_frames, float pad_value,
                                                            const long long* __restrict__ mask_start, const long long* __restrict__ mask_len) {
    constexpr int kT = 64;
    __shared__ float tile[kT][kT + 1];          // [d][t], odd pitch
    const int clip = blockIdx.z;
    const long long t0 = (long long)blockIdx.x * kT;
    const int d0 = blockIdx.y * kT;
    const long long n = lens[clip];
    const T* src = feat + row_offset[clip] * dim;
    const long long m0 = mask_start ? mask_start[clip] : 0, m1 = mask_start ? m0 + mask_len[clip] : 0;
    const int q = threadIdx.x & 15, r0 = threadIdx.x >> 4;    // 16 quads x 16 rows per pass
    const bool vec_in = sizeof(T) == 4 && (dim & 3) == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0;
#pragma unroll
    for (int pass = 0; pass < kT / 16; ++pass) {              // read: rows = time, 4 consecutive feature values per thread
        const int r = pass * 16 + r0;
        const long long t = t0 + r;
        const int d = d0 + 4 * q;
        float v[4] = {pad_value, pad_value, pad_value, pad_value};
        if (t < n) {
            const bool masked = t >= m0 && t < m1;
            if (vec_in && d + 3 < dim) {
                if constexpr (sizeof(T) == 4) {
                    const float4 u = __ldg(reinterpret_cast<const float4*>(src + t * dim + d));
                    v[0] = u.x; v[1] = u.y; v[2] = u.z; v[3] = u.w;
                }
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) if (d + j < dim) v[j] = (float)src[t * dim + d + j];
            }
            if (masked) { v[0] = v[1] = v[2] = v[3] = 0.f; }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) tile[4 * q + j][r] = v[j];
    }
    __syncthreads();
    const bool vec_out = sizeof(T) == 4 && (out_frames & 3) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0;
#pragma unroll
    for (int pass = 0; pass < kT / 16; ++pass) {              // write: rows = feature dim, 4 consecutive frames per thread
        const int r = pass * 16 + r0;
        const int d = d0 + r;
        const long long t = t0 + 4 * q;
        if (d >= dim || t >= out_frames) continue;
        T* dst = out + ((long long)clip * dim + d) * out_frames + t;
        if (vec_out && t + 3 < out_frames) {
            if constexpr (sizeof(T) == 4)
                *reinterpret_cast<float4*>(dst) = make_float4(tile[r][4 * q], tile[r][4 * q + 1], tile[r][4 * q + 2], tile[r][4 * q + 3]);
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j) if (t + j < out_frames) dst[j] = from_float<T>(tile[r][4 * q + j]);
        }
    }
}

}  // namespace acb

// ==============================================================================================
// host side: handle, planning, launches
// ==============================================================================================
using namespace acb;

extern "C" {

int acb_abi_version(void) { return ACB_ABI_VERSION; }
const char* acb_last_error(void) { return g_last_error.c_str(); }
int acb_frames_per_tile(void) { return kTileFrames; }

int64_t acb_frames_for_length(int64_t length, int n_fft, int hop) {
    if (n_fft <= 0 || hop <= 0) return -1;
    if (length <= n_fft / 2) return -1;
    return 1 + length / hop;
}

int64_t acb_padded_frames(int64_t frames, int multiple) {
    if (multiple <= 1) return frames;
    const int64_t r = frames % multiple;
    return r ? frames + (multiple - r) : frames;
}

}  // extern "C"

// ---- spectrogram definitions (acb_stft_options) ----
static acb_stft_options stft_options_or_default(const acb_stft_options* opt, int n_fft) {
    return opt ? *opt : acb_stft_options{n_fft / 2, ACB_PAD_REFLECT, 2, 0.f};
}

static bool stft_options_default(const acb_stft_options& o, int n_fft) {
    return o.pad == n_fft / 2 && o.pad_mode == ACB_PAD_REFLECT && o.power == 2;
}

// ACB_OK, or the error code with the envelope in `msg`
static int stft_options_check(const acb_stft_options& o, int n_fft, std::string& msg) {
    if (o.pad < 0 || o.pad > n_fft / 2) {
        msg = "pad must be in [0, n_fft/2] = [0, " + std::to_string(n_fft / 2) + "] (got " + std::to_string(o.pad) + ")";
        return ACB_ERR_INVALID;
    }
    if (o.pad_mode != ACB_PAD_REFLECT && o.pad_mode != ACB_PAD_CONSTANT) {
        msg = "pad_mode must be ACB_PAD_REFLECT (0) or ACB_PAD_CONSTANT (1); replicate and circular padding have no kernel (got " +
              std::to_string(o.pad_mode) + ")";
        return ACB_ERR_UNSUPPORTED;
    }
    if (o.power != 1 && o.power != 2) {
        msg = "power must be 1 (magnitude) or 2 (power) (got " + std::to_string(o.power) + ")";
        return ACB_ERR_INVALID;
    }
    if (!std::isfinite(o.magnitude_eps) || o.magnitude_eps < 0.f) {
        msg = "magnitude_eps must be finite and >= 0 (got " + std::to_string(o.magnitude_eps) + ")";
        return ACB_ERR_INVALID;
    }
    if (o.power == 2 && o.magnitude_eps != 0.f) {
        msg = "magnitude_eps applies to power 1 only; it must be 0 with power 2";
        return ACB_ERR_INVALID;
    }
    return ACB_OK;
}

// T = 1 + (L + 2 pad - n_fft) / hop, or -1 below the definition's minimum length (torch.stft / F.pad's limits)
static int64_t stft_frames(int64_t length, int n_fft, int hop, const acb_stft_options& o) {
    if (n_fft <= 0 || hop <= 0) return -1;
    if (length + 2 * (int64_t)o.pad < n_fft) return -1;
    if (o.pad_mode == ACB_PAD_REFLECT ? length <= o.pad : length < 1) return -1;
    return 1 + (length + 2 * (int64_t)o.pad - n_fft) / hop;
}

static std::string stft_minimum(int n_fft, const acb_stft_options& o) {
    if (stft_options_default(o, n_fft)) return "reflect padding needs more than " + std::to_string(n_fft / 2);
    const int64_t need = std::max<int64_t>(n_fft - 2 * (int64_t)o.pad, o.pad_mode == ACB_PAD_REFLECT ? o.pad + 1 : 1);
    return "n_fft=" + std::to_string(n_fft) + " with " + (o.pad_mode == ACB_PAD_REFLECT ? "reflect" : "constant") + " padding of " +
           std::to_string(o.pad) + " needs at least " + std::to_string(need);
}

extern "C" {

int64_t acb_stft_frames_for_length(int64_t length, int n_fft, int hop, const acb_stft_options* opt) {
    const acb_stft_options o = stft_options_or_default(opt, n_fft);
    std::string msg;
    if (stft_options_check(o, n_fft, msg) != ACB_OK) return -1;
    return stft_frames(length, n_fft, hop, o);
}

int64_t acb_plan_tiles(const int64_t* lengths_host, int32_t n_clips, int n_fft, int hop, int64_t frame_capacity,
                       int32_t* tile_start_host) {
    return acb_stft_plan_tiles(lengths_host, n_clips, n_fft, hop, nullptr, frame_capacity, tile_start_host);
}

int64_t acb_stft_plan_tiles(const int64_t* lengths_host, int32_t n_clips, int n_fft, int hop, const acb_stft_options* opt,
                            int64_t frame_capacity, int32_t* tile_start_host) {
    if (!lengths_host || !tile_start_host || n_clips < 0) return fail(ACB_ERR_INVALID, "acb_plan_tiles: null argument");
    const acb_stft_options o = stft_options_or_default(opt, n_fft);
    std::string msg;
    if (stft_options_check(o, n_fft, msg) != ACB_OK) return fail(ACB_ERR_INVALID, "acb_plan_tiles: " + msg);
    int64_t total = 0;
    for (int32_t i = 0; i < n_clips; ++i) {
        const int64_t T = stft_frames(lengths_host[i], n_fft, hop, o);
        if (T < 0) {
            return fail(ACB_ERR_INVALID, "acb_plan_tiles: clip " + std::to_string(i) + " has " + std::to_string(lengths_host[i]) +
                                             " samples; " + stft_minimum(n_fft, o));
        }
        const int64_t cover = frame_capacity > 0 ? frame_capacity : T;
        tile_start_host[i] = (int32_t)total;
        total += (cover + kTileFrames - 1) / kTileFrames;
        if (total > INT32_MAX) return fail(ACB_ERR_INVALID, "acb_plan_tiles: more than 2^31 tiles in one call");
    }
    tile_start_host[n_clips] = (int32_t)total;
    return total;
}

int acb_frontend_create(acb_frontend** out, int device, int n_fft, int hop, int n_mels, const float* window_host,
                        const float* fb_host, float clamp_min, int log_kind) {
    return acb_frontend_create_stft(out, device, n_fft, hop, n_mels, window_host, fb_host, clamp_min, log_kind, nullptr);
}

int acb_frontend_create_stft(acb_frontend** out, int device, int n_fft, int hop, int n_mels, const float* window_host,
                             const float* fb_host, float clamp_min, int log_kind, const acb_stft_options* opt) {
    if (!out || !window_host || !fb_host) return fail(ACB_ERR_INVALID, "acb_frontend_create: null argument");
    const acb_stft_options so = stft_options_or_default(opt, n_fft);
    // (1024, 256) with the default definition runs the tuned kernel below; every other supported (n_fft, hop), and every one with
    // another definition, the general STFT kernel (acb_logmel_stft.cu)
    const bool tuned = n_fft == kNfft && hop == kHop && stft_options_default(so, n_fft);
    if (!tuned && !stft_logmel_supported(n_fft, hop))
        return fail(ACB_ERR_UNSUPPORTED, "acb_frontend_create: this build has kernels for n_fft 256, 512 or 1024 with 1 <= hop <= n_fft (got n_fft=" +
                                             std::to_string(n_fft) + ", hop=" + std::to_string(hop) + ")");
    if (n_mels < 1 || n_mels > kMaxMels) return fail(ACB_ERR_UNSUPPORTED, "acb_frontend_create: n_mels must be in [1, 128]");
    if (log_kind != ACB_LOG_NATURAL && log_kind != ACB_LOG_10) return fail(ACB_ERR_INVALID, "acb_frontend_create: bad log_kind");
    if (!(clamp_min >= 1.17549435e-38f)) return fail(ACB_ERR_INVALID, "acb_frontend_create: clamp_min must be a positive normal float");
    std::string msg;
    if (const int rc = stft_options_check(so, n_fft, msg)) return fail(rc, "acb_frontend_create_stft: " + msg);
    if (!tuned) return stft_frontend_create(out, device, n_fft, hop, n_mels, window_host, fb_host, clamp_min, log_kind, so);
    // The kernel stages only w[0 .. N/2 - 1] and computes the second half as 1 - w[n] (the periodic-Hann property).  A window
    // without that property would give wrong features silently; fp32 periodic Hann deviates by 1.8e-7.
    for (int n = 0; n < kNfft / 2; ++n) {
        const double dev = std::fabs((double)window_host[n + kNfft / 2] - (1.0 - (double)window_host[n]));
        if (!(dev <= 1e-6))
            return fail(ACB_ERR_UNSUPPORTED, "acb_frontend_create: the window must have the periodic-Hann property w[n + 512] = 1 - w[n] "
                                             "(deviation " + std::to_string(dev) + " at n=" + std::to_string(n) + ")");
    }
    const int n_freq = n_fft / 2 + 1;

    // banded form of the filterbank; the 1/4 of the packed-pair power spectrum is folded in (exact scaling)
    std::vector<int> start(n_mels, 0), len(n_mels, 0), off(n_mels, 0);
    std::vector<float> weights;
    for (int m = 0; m < n_mels; ++m) {
        int lo = -1, hi = -1;
        for (int f = 0; f < n_freq; ++f)
            if (fb_host[(size_t)f * n_mels + m] != 0.f) { if (lo < 0) lo = f; hi = f; }
        off[m] = (int)weights.size();
        if (lo >= 0) {
            if (hi >= kBins) {
                // the Nyquist bin is not produced by the packed FFT; the slaney bank (f_max = sr/2) has zero weight there
                if (fb_host[(size_t)(n_freq - 1) * n_mels + m] != 0.f)
                    return fail(ACB_ERR_UNSUPPORTED, "acb_frontend_create: filterbank has weight on the Nyquist bin");
            }
            start[m] = lo;
            len[m] = hi - lo + 1;
            for (int f = lo; f <= hi; ++f) weights.push_back(fb_host[(size_t)f * n_mels + m] * 0.25f);
        }
    }
    if ((int)weights.size() > kMaxWeights) return fail(ACB_ERR_UNSUPPORTED, "acb_frontend_create: filterbank too dense");

    // mel plan: bands sorted by (even-aligned) run length, groups of 8 (one per lane slot), groups dealt to the 4 warps of a
    // group longest-processing-time first.  Within a round every slot is zero-padded to the round's trip count, so the kernel's
    // inner loop is predicate-free; runs start on an even bin so two bins are fetched with one 16-byte load.  Slots (2j, 2j+1)
    // share a quarter-warp: they get opposite parity of astart/2 (a run may start one bin pair early, on zero weights), which
    // keeps the 16-byte power loads free of bank conflicts (see the kernel).
    std::vector<int> alen(n_mels), aend(n_mels);
    for (int m = 0; m < n_mels; ++m) {
        if (len[m] == 0) { start[m] = 0; len[m] = 0; }
        aend[m] = (start[m] + std::max(len[m], 1) + 1) & ~1;
        alen[m] = aend[m] - (start[m] & ~1);
    }
    std::vector<int> order(n_mels);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return alen[a] > alen[b]; });
    const int n_rounds = (n_mels + kSlots - 1) / kSlots;
    std::vector<short> plan_band(kGroupWarps * kMaxRounds * kSlots, (short)-1), plan_astart(kGroupWarps * kMaxRounds * kSlots, (short)0),
        plan_trip(kGroupWarps * kMaxRounds, (short)0);
    std::vector<int> plan_woff(kGroupWarps * kMaxRounds, 0);
    std::vector<float> plan_w;
    std::vector<int> load(kGroupWarps, 0), rounds(kGroupWarps, 0);
    for (int g = 0; g < n_rounds; ++g) {
        int best = -1;
        for (int w = 0; w < kGroupWarps; ++w)
            if (rounds[w] < kMaxRounds && (best < 0 || load[w] < load[best])) best = w;
        if (best < 0) return fail(ACB_ERR_UNSUPPORTED, "acb_frontend_create: mel plan overflow");
        // order the round's bands so that neighbours (2j, 2j+1) have opposite parity of astart/2 where possible
        std::vector<int> par[2];
        for (int q = 0; q < kSlots && kSlots * g + q < n_mels; ++q) {
            const int m = order[kSlots * g + q];
            par[((start[m] & ~1) >> 1) & 1].push_back(m);
        }
        std::vector<int> slots;
        while (!par[0].empty() && !par[1].empty()) {
            slots.push_back(par[0].back()); par[0].pop_back();
            slots.push_back(par[1].back()); par[1].pop_back();
        }
        for (int k = 0; k < 2; ++k)
            for (int m : par[k]) slots.push_back(m);
        std::vector<int> shift(slots.size(), 0), as(slots.size(), 0);
        int trip = 2;
        for (int iter = 0; iter < 8; ++iter) {
            trip = 2;
            for (size_t i = 0; i < slots.size(); ++i) trip = std::max(trip, aend[slots[i]] - ((start[slots[i]] & ~1) - shift[i]));
            for (size_t i = 0; i < slots.size(); ++i) {
                as[i] = (start[slots[i]] & ~1) - shift[i];
                if (as[i] + trip > kBins) as[i] = std::max(0, (kBins - trip) & ~1);   // keep every 16-byte read inside the 512-bin power array
            }
            bool changed = false;
            for (size_t i = 0; i + 1 < slots.size(); i += 2) {
                if ((((as[i] >> 1) ^ (as[i + 1] >> 1)) & 1) != 0) continue;
                const size_t x = (as[i + 1] >= 2 && (start[slots[i + 1]] & ~1) - shift[i + 1] == as[i + 1]) ? i + 1
                                 : ((as[i] >= 2 && (start[slots[i]] & ~1) - shift[i] == as[i]) ? i : slots.size());
                if (x < slots.size()) { shift[x] += 2; changed = true; }
            }
            if (!changed) break;
        }
        const int slot = best * kMaxRounds + rounds[best];
        plan_trip[slot] = (short)trip;
        plan_woff[slot] = (int)plan_w.size();
        plan_w.resize(plan_w.size() + (size_t)trip * kSlots, 0.f);
        float* wbase = plan_w.data() + plan_woff[slot];
        for (size_t q = 0; q < slots.size(); ++q) {
            const int m = slots[q];
            plan_band[slot * kSlots + q] = (short)m;
            plan_astart[slot * kSlots + q] = (short)as[q];
            for (int i = 0; i < len[m]; ++i) {
                const int rel = start[m] + i - as[q];                 // bin offset inside the slot's window
                if (rel < 0 || rel >= trip) return fail(ACB_ERR_UNSUPPORTED, "acb_frontend_create: mel plan window error");
                wbase[(rel >> 1) * (2 * kSlots) + q * 2 + (rel & 1)] = weights[off[m] + i];
            }
        }
        load[best] += trip + 16;  // + fixed per-round epilogue cost
        rounds[best]++;
    }
    if ((int)plan_w.size() > kMaxWeights * 4) return fail(ACB_ERR_UNSUPPORTED, "acb_frontend_create: mel plan too large");

    // seeds of the in-register twiddle chains: W^(m*l) = exp(-2*pi*i*m*l/1024) in double, rounded once
    std::vector<float4> tw(5 * 32);
    for (int l = 0; l < 32; ++l) {
        auto wre = [&](int m) { return (float)cos(-2.0 * M_PI * (double)(m * l) / 1024.0); };
        auto wim = [&](int m) { return (float)sin(-2.0 * M_PI * (double)(m * l) / 1024.0); };
        for (int k = 0; k < 4; ++k) tw[k * 32 + l] = make_float4(wre(k), wre(k + 16), wim(k), wim(k + 16));
        tw[4 * 32 + l] = make_float4(wre(4), wim(4), 0.f, 0.f);
    }

    int prev = 0;
    ACB_CUDA(cudaGetDevice(&prev));
    ACB_CUDA(cudaSetDevice(device));
    auto* fe = new acb_frontend();
    fe->opt = so;
    fe->device = device; fe->n_fft = n_fft; fe->hop = hop; fe->n_mels = n_mels; fe->n_weights = (int)weights.size();
    fe->n_plan_w = (int)plan_w.size();
    fe->log_kind = log_kind; fe->clamp_min = clamp_min;

    // pack the blob
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += (bytes + 255) & ~size_t(255); return r; };
    const size_t o_win = take(sizeof(float) * kNfft), o_tw = take(sizeof(float4) * 160),
                 o_pw = take(sizeof(float) * std::max<size_t>(plan_w.size(), 1)), o_po = take(sizeof(int) * plan_woff.size()),
                 o_pt = take(sizeof(short) * plan_trip.size()), o_pb = take(sizeof(short) * plan_band.size()),
                 o_pa = take(sizeof(short) * plan_astart.size()), o_err = take(16);
    std::vector<unsigned char> host(o, 0);
    memcpy(host.data() + o_win, window_host, sizeof(float) * kNfft);
    memcpy(host.data() + o_tw, tw.data(), sizeof(float4) * 160);
    if (!plan_w.empty()) memcpy(host.data() + o_pw, plan_w.data(), sizeof(float) * plan_w.size());
    memcpy(host.data() + o_po, plan_woff.data(), sizeof(int) * plan_woff.size());
    memcpy(host.data() + o_pt, plan_trip.data(), sizeof(short) * plan_trip.size());
    memcpy(host.data() + o_pb, plan_band.data(), sizeof(short) * plan_band.size());
    memcpy(host.data() + o_pa, plan_astart.data(), sizeof(short) * plan_astart.size());
    cudaError_t e = cudaMalloc(&fe->d_blob, o);
    if (e == cudaSuccess) e = cudaMemcpy(fe->d_blob, host.data(), o, cudaMemcpyHostToDevice);
    cudaDeviceProp prop;
    if (e == cudaSuccess) e = cudaGetDeviceProperties(&prop, device);
    // The attribute is per function, not per handle: several front-ends (different n_mels) may live in one process, so it is
    // always raised to the device's opt-in maximum; the launch passes the handle's own size.
    const int optin = (int)prop.sharedMemPerBlockOptin;
    fe->groups = std::max(make_smem_layout(kMaxGroups, n_mels, fe->n_plan_w, true).total_bytes,
                          make_smem_layout(kMaxGroups, n_mels, fe->n_plan_w, false).total_bytes) <= optin ? kMaxGroups : 2;
    const SmemLayout L = make_smem_layout(fe->groups, n_mels, fe->n_plan_w, false);
    const SmemLayout Lm = make_smem_layout(fe->groups, n_mels, fe->n_plan_w, true);
    fe->smem_bytes = L.total_bytes;
    fe->smem_bytes_moments = Lm.total_bytes;
    if (e == cudaSuccess && std::max(L.total_bytes, Lm.total_bytes) > optin) {
        if (fe->d_blob) cudaFree(fe->d_blob);
        delete fe;
        cudaSetDevice(prev);
        return fail(ACB_ERR_UNSUPPORTED, "acb_frontend_create: filterbank plan needs more shared memory than the device offers");
    }
    int occ = 0;
    auto prepare = [&](auto kernel, int threads) {
        if (e == cudaSuccess) e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, optin);
        if (e == cudaSuccess && occ == 0) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, L.total_bytes);
    };
    if (fe->groups == 4) {
        prepare(logmel_fused_kernel<4, false, float>, 4 * kGroupThreads);
        prepare(logmel_fused_kernel<4, false, __nv_bfloat16>, 4 * kGroupThreads);
        prepare(logmel_fused_kernel<4, true, float>, 4 * kGroupThreads);
        prepare(logmel_fused_kernel<4, true, __nv_bfloat16>, 4 * kGroupThreads);
    } else {
        prepare(logmel_fused_kernel<2, false, float>, 2 * kGroupThreads);
        prepare(logmel_fused_kernel<2, false, __nv_bfloat16>, 2 * kGroupThreads);
        prepare(logmel_fused_kernel<2, true, float>, 2 * kGroupThreads);
        prepare(logmel_fused_kernel<2, true, __nv_bfloat16>, 2 * kGroupThreads);
    }
    if (e != cudaSuccess) {
        if (fe->d_blob) cudaFree(fe->d_blob);
        delete fe;
        cudaSetDevice(prev);
        return cuda_fail(e, "acb_frontend_create");
    }
    fe->num_sms = prop.multiProcessorCount;
    fe->grid = fe->num_sms * std::max(occ, 1);
    auto* base = static_cast<unsigned char*>(fe->d_blob);
    fe->d_window = reinterpret_cast<const float*>(base + o_win);
    fe->d_twiddle = reinterpret_cast<const float4*>(base + o_tw);
    fe->d_plan_w = reinterpret_cast<const float*>(base + o_pw);
    fe->d_plan_woff = reinterpret_cast<const int*>(base + o_po);
    fe->d_plan_trip = reinterpret_cast<const short*>(base + o_pt);
    fe->d_plan_band = reinterpret_cast<const short*>(base + o_pb);
    fe->d_plan_astart = reinterpret_cast<const short*>(base + o_pa);
    fe->d_err = reinterpret_cast<int*>(base + o_err);
    cudaSetDevice(prev);
    *out = fe;
    return ACB_OK;
}

int acb_frontend_destroy(acb_frontend* fe) {
    if (!fe) return ACB_OK;
    int prev = 0;
    cudaGetDevice(&prev);
    cudaSetDevice(fe->device);
    for (auto ev : fe->ev) cudaEventDestroy(ev);
    if (fe->s_in) cudaStreamDestroy(fe->s_in);
    if (fe->s_out) cudaStreamDestroy(fe->s_out);
    if (fe->d_blob) cudaFree(fe->d_blob);
    cudaSetDevice(prev);
    delete fe;
    return ACB_OK;
}

int64_t acb_moments_workspace_bytes(const acb_frontend* fe) {
    if (!fe) return fail(ACB_ERR_INVALID, "acb_moments_workspace_bytes: null handle");
    return (int64_t)fe->grid * fe->groups * 2 * fe->n_mels * (int64_t)sizeof(double);
}

int acb_logmel_forward(const acb_frontend* fe, const acb_logmel_args* a, void* stream) {
    if (!fe || !a) return fail(ACB_ERR_INVALID, "acb_logmel_forward: null argument");
    if (a->n_clips <= 0 || a->n_tiles <= 0) return ACB_OK;  // empty batch
    if (!a->wav) return fail(ACB_ERR_INVALID, "acb_logmel_forward: null wav");
    if (!a->out && !a->moments) return fail(ACB_ERR_INVALID, "acb_logmel_forward: out may be NULL only for a statistics-only launch (moments set)");
    if (a->out_dtype != ACB_F32 && a->out_dtype != ACB_BF16) return fail(ACB_ERR_INVALID, "acb_logmel_forward: bad out_dtype");
    if (a->out_layout != ACB_MEL_MAJOR && a->out_layout != ACB_TIME_MAJOR) return fail(ACB_ERR_INVALID, "acb_logmel_forward: bad out_layout");
    if (a->pad_multiple < 1) return fail(ACB_ERR_INVALID, "acb_logmel_forward: pad_multiple must be >= 1");
    // the reflected pad columns are written by the tile that holds their source frames, which needs the padded count to end on a
    // tile boundary or inside the last tile: multiples that divide the tile (1, 2, 4, 8; the reference uses 4)
    if (kTileFrames % a->pad_multiple != 0)
        return fail(ACB_ERR_UNSUPPORTED, "acb_logmel_forward: pad_multiple must divide the " + std::to_string(kTileFrames) + "-frame tile (1, 2, 4 or 8)");
    if (a->affine < 0 || a->affine > 2) return fail(ACB_ERR_INVALID, "acb_logmel_forward: bad affine mode");
    if (a->affine == 2 && (!a->bin_mean || !a->bin_std)) return fail(ACB_ERR_INVALID, "acb_logmel_forward: per-bin affine needs bin_mean/bin_std");
    if (a->affine == 1 && !(a->affine_std > 0.f)) return fail(ACB_ERR_INVALID, "acb_logmel_forward: affine_std must be > 0");
    if (a->moments && !a->moments_workspace) return fail(ACB_ERR_INVALID, "acb_logmel_forward: moments need a workspace");
    if (!a->frame_capacity_per_clip && a->frame_capacity <= 0) return fail(ACB_ERR_INVALID, "acb_logmel_forward: frame_capacity must be > 0");
    if (a->frame_capacity * (int64_t)fe->n_mels >= (int64_t)1 << 32) return fail(ACB_ERR_INVALID, "acb_logmel_forward: n_mels * frame_capacity must be < 2^32");

    LogmelParams p{};
    p.window = fe->d_window; p.twiddle = fe->d_twiddle;
    p.plan_w = fe->d_plan_w; p.plan_woff = fe->d_plan_woff; p.plan_trip = fe->d_plan_trip;
    p.plan_band = fe->d_plan_band; p.plan_astart = fe->d_plan_astart; p.n_plan_w = fe->n_plan_w;
    p.n_mels = fe->n_mels; p.clamp_min = fe->clamp_min;
    p.log_scale = fe->log_kind == ACB_LOG_10 ? 0.30102999566398120f : 0.69314718055994531f;   // log10(2) : ln(2)
    p.log_floor = fe->log_kind == ACB_LOG_10 ? log10f(fe->clamp_min) : logf(fe->clamp_min);
    p.wav = a->wav;
    p.clip_offset = reinterpret_cast<const long long*>(a->clip_offset);
    p.clip_length = reinterpret_cast<const long long*>(a->clip_length);
    p.clip_stride = a->clip_stride; p.uniform_length = a->uniform_length;
    p.tile_start = a->tile_start; p.n_clips = a->n_clips; p.n_tiles = a->n_tiles;
    p.uniform_tiles_per_clip = 1;
    if (!a->tile_start && a->clip_length) {
        // ragged clips without a tile plan: allowed for padded outputs (fill_tail), where every clip covers the whole row of
        // frame_capacity frames and the tile count per clip is uniform.  The caller vouches that no clip is shorter than
        // n_fft/2 + 1 samples and that every padded frame count fits frame_capacity (frontend.py checks both on the host).
        if (!a->fill_tail || a->frame_capacity_per_clip)
            return fail(ACB_ERR_INVALID, "acb_logmel_forward: ragged clips need tile_start (acb_plan_tiles) unless fill_tail pads every clip to frame_capacity");
        p.uniform_tiles_per_clip = (int)((a->frame_capacity + kTileFrames - 1) / kTileFrames);
        if ((int64_t)p.uniform_tiles_per_clip * a->n_clips != a->n_tiles)
            return fail(ACB_ERR_INVALID, "acb_logmel_forward: n_tiles does not match n_clips * tiles per clip");
    } else if (!a->tile_start) {
        const int64_t T = stft_frames(a->uniform_length, fe->n_fft, fe->hop, fe->opt);
        if (T < 0) return fail(ACB_ERR_INVALID, "acb_logmel_forward: clips of " + std::to_string(a->uniform_length) +
                                                    " samples are too short: " + stft_minimum(fe->n_fft, fe->opt));
        const int64_t cover = a->fill_tail ? a->frame_capacity : T;
        p.uniform_tiles_per_clip = (int)((cover + kTileFrames - 1) / kTileFrames);
        if ((int64_t)p.uniform_tiles_per_clip * a->n_clips != a->n_tiles)
            return fail(ACB_ERR_INVALID, "acb_logmel_forward: n_tiles does not match n_clips * tiles per clip");
        if (acb_padded_frames(T, a->pad_multiple) > a->frame_capacity)
            return fail(ACB_ERR_INVALID, "acb_logmel_forward: frame_capacity smaller than the padded frame count");
        if (acb_padded_frames(T, a->pad_multiple) - T >= T)   // F.pad(mode="reflect") needs pad < T (process_dataset.py:147-150)
            return fail(ACB_ERR_INVALID, "acb_logmel_forward: reflect pad to the multiple needs more frames than the clip has");
    }
    p.clip_peak = a->clip_peak;
    p.out = a->out; p.out_bf16 = a->out_dtype == ACB_BF16; p.time_major = a->out_layout == ACB_TIME_MAJOR;
    p.out_offset = reinterpret_cast<const long long*>(a->out_offset);
    p.out_clip_stride = a->out_clip_stride; p.frame_capacity = a->frame_capacity;
    p.frame_capacity_per_clip = reinterpret_cast<const long long*>(a->frame_capacity_per_clip);
    p.pad_multiple = a->pad_multiple; p.fill_tail = a->fill_tail; p.fill_value = a->fill_value;
    p.affine = a->affine; p.affine_mean = a->affine_mean;
    p.affine_inv_std = a->affine == 1 ? (float)(1.0 / (double)a->affine_std) : 1.f;
    p.bin_mean = a->bin_mean; p.bin_std = a->bin_std;
    p.moments_partial = a->moments ? static_cast<double*>(a->moments_workspace) : nullptr;
    p.error_flag = fe->d_err;

    int prev = 0;
    ACB_CUDA(cudaGetDevice(&prev));
    if (prev != fe->device) ACB_CUDA(cudaSetDevice(fe->device));
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int grid = fe->grid;  // persistent: every CTA takes a contiguous share of the tiles (possibly empty)
    // The mel projection runs on the CUDA cores: measured on B200 (256 x 30 s) this kernel runs 0.466 ms against 1.80 ms for a
    // warp-specialised variant with the projection on the tensor pipe, whose twelve FFT warps alone needed 0.437 ms
    // (profiles/r02_tc_variant.txt) -- the FFT phase, not the mel projection, bounds this path.
    const int threads = fe->groups * kGroupThreads;
    const size_t smem = a->moments ? fe->smem_bytes_moments : fe->smem_bytes;
    auto launch = [&](auto kernel) { kernel<<<grid, threads, smem, st>>>(p); };
    if (fe->stft_r) {
        stft_logmel_launch(fe, p, a->moments != nullptr, st);
    } else if (fe->groups == 4) {
        if (a->moments) { if (p.out_bf16) launch(logmel_fused_kernel<4, true, __nv_bfloat16>); else launch(logmel_fused_kernel<4, true, float>); }
        else { if (p.out_bf16) launch(logmel_fused_kernel<4, false, __nv_bfloat16>); else launch(logmel_fused_kernel<4, false, float>); }
    } else {
        if (a->moments) { if (p.out_bf16) launch(logmel_fused_kernel<2, true, __nv_bfloat16>); else launch(logmel_fused_kernel<2, true, float>); }
        else { if (p.out_bf16) launch(logmel_fused_kernel<2, false, __nv_bfloat16>); else launch(logmel_fused_kernel<2, false, float>); }
    }
    if (a->moments) {
        const int n_vals = 2 * fe->n_mels;
        moments_reduce_kernel<<<(n_vals + 7) / 8, 256, 0, st>>>(p.moments_partial, grid * fe->groups, n_vals, a->moments);
    }
    cudaError_t e = cudaGetLastError();
    if (prev != fe->device) cudaSetDevice(prev);
    if (e != cudaSuccess) return cuda_fail(e, "acb_logmel_forward launch");
    return ACB_OK;
}

int acb_frontend_set_kernel(acb_frontend* fe, int kind) {
    if (!fe) return fail(ACB_ERR_INVALID, "acb_frontend_set_kernel: null handle");
    if (kind < 0 || kind > 2) return fail(ACB_ERR_INVALID, "acb_frontend_set_kernel: kind must be 0 (automatic), 1 (CUDA-core mel) or 2 (tensor-core mel)");
    if (kind == 2) return fail(ACB_ERR_UNSUPPORTED, "acb_frontend_set_kernel: this build has only the CUDA-core mel kernel (kind 0 or 1)");
    return ACB_OK;
}

int acb_frontend_check(const acb_frontend* fe, void* stream) {
    if (!fe) return fail(ACB_ERR_INVALID, "acb_frontend_check: null handle");
    int flag = 0, prev = 0;
    ACB_CUDA(cudaGetDevice(&prev));
    if (prev != fe->device) ACB_CUDA(cudaSetDevice(fe->device));
    cudaError_t e = cudaStreamSynchronize(static_cast<cudaStream_t>(stream));
    if (e == cudaSuccess) e = cudaMemcpy(&flag, fe->d_err, sizeof(int), cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && flag) cudaMemset(fe->d_err, 0, sizeof(int));
    if (prev != fe->device) cudaSetDevice(prev);
    if (e != cudaSuccess) return cuda_fail(e, "acb_frontend_check");
    if (flag) return fail(ACB_ERR_CUDA, "acb_frontend_check: a sample-tile copy did not complete inside the kernel (results are invalid)");
    return ACB_OK;
}

// SM count of the current device (launch sizing of the small kernels); 148 on a B200
static int current_sm_count() {
    thread_local int cached_dev = -1, cached = 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (dev != cached_dev) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached_dev = dev; cached = n;
    }
    return cached;
}

int acb_peak_abs(const float* wav, const int64_t* clip_offset, const int64_t* clip_length, int64_t clip_stride,
                 int64_t uniform_length, int32_t n_clips, float* peak_out, void* stream) {
    if (n_clips <= 0) return ACB_OK;
    if (!wav || !peak_out) return fail(ACB_ERR_INVALID, "acb_peak_abs: null argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ACB_CUDA(cudaMemsetAsync(peak_out, 0, sizeof(float) * n_clips, st));
    // enough CTAs to fill the chip even for a single clip
    int blocks_per_clip = std::max(1, std::min(64, (current_sm_count() * 8 + n_clips - 1) / n_clips));
    peak_abs_kernel<<<n_clips * blocks_per_clip, 256, 0, st>>>(wav, reinterpret_cast<const long long*>(clip_offset),
                                                               reinterpret_cast<const long long*>(clip_length), clip_stride,
                                                               uniform_length, blocks_per_clip, peak_out);
    ACB_CUDA(cudaGetLastError());
    return ACB_OK;
}

int acb_process_audio_chunk(const float* wav_cl, int32_t channels, int64_t length, float* out, float* scratch_peak, void* stream) {
    if (!wav_cl || !out || !scratch_peak || channels < 1 || length < 0) return fail(ACB_ERR_INVALID, "acb_process_audio_chunk: bad argument");
    if (length == 0) return ACB_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    ACB_CUDA(cudaMemsetAsync(scratch_peak, 0, sizeof(float), st));
    const int blocks = (int)std::min<int64_t>(current_sm_count() * 8, (length + 255) / 256);
    mixdown_peak_kernel<<<blocks, 256, 0, st>>>(wav_cl, channels, length, out, scratch_peak);
    peak_scale_kernel<<<blocks, 256, 0, st>>>(out, length, scratch_peak);
    ACB_CUDA(cudaGetLastError());
    return ACB_OK;
}

// upper bound of the standalone moments grid (the workspace is sized before a device is known): 8 CTAs per SM of a 256-SM part
constexpr int kMomentsMaxCtas = 2048;

int acb_mixdown_peak(const float* wav_cl, int32_t channels, int64_t length, float* out, float* peak_out, void* stream) {
    if (!wav_cl || !out || channels < 1 || length < 0) return fail(ACB_ERR_INVALID, "acb_mixdown_peak: bad argument");
    if (length == 0) return ACB_OK;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (peak_out) ACB_CUDA(cudaMemsetAsync(peak_out, 0, sizeof(float), st));
    const int blocks = (int)std::min<int64_t>(current_sm_count() * 8, (length / 4 + 255) / 256 + 1);
    mixdown_peak_kernel<<<blocks, 256, 0, st>>>(wav_cl, channels, length, out, peak_out);
    ACB_CUDA(cudaGetLastError());
    return ACB_OK;
}

int64_t acb_moments_accumulate_workspace_bytes(int32_t n_mels) {
    return (int64_t)sizeof(double) * kMomentsMaxCtas * 2 * (int64_t)(n_mels > 0 ? n_mels : 0);
}

int acb_moments_accumulate(const void* feat, int32_t dtype, int32_t n_clips, int32_t n_mels, int64_t frame_capacity,
                           int64_t clip_stride, const int64_t* frames, double* moments, void* workspace, void* stream) {
    if (n_clips <= 0) return ACB_OK;
    if (!feat || !moments || n_mels < 1 || frame_capacity < 1) return fail(ACB_ERR_INVALID, "acb_moments_accumulate: bad argument");
    if (dtype != ACB_F32 && dtype != ACB_BF16) return fail(ACB_ERR_INVALID, "acb_moments_accumulate: bad dtype");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int warps = 8;
    const long long n_rows = (long long)n_clips * n_mels;
    // one wave of CTAs in which every warp takes the same number of rows (a ragged last trip would leave most warps idle)
    const long long max_ctas = std::min(kMomentsMaxCtas, current_sm_count() * 8);
    const long long rows_per_warp = (n_rows + max_ctas * warps - 1) / (max_ctas * warps);
    const int grid = (int)((n_rows + rows_per_warp * warps - 1) / (rows_per_warp * warps));
    double* partial = static_cast<double*>(workspace);   // caller-owned scratch (acb_moments_accumulate_workspace_bytes), or a stream-ordered one
    if (!workspace) ACB_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&partial), sizeof(double) * (size_t)grid * 2 * n_mels, st));
    const size_t smem = sizeof(double) * warps * 2 * n_mels;
    if (dtype == ACB_F32)
        moments_rows_kernel<float><<<grid, warps * 32, smem, st>>>(static_cast<const float*>(feat), n_clips, n_mels, frame_capacity,
                                                                    clip_stride, reinterpret_cast<const long long*>(frames), partial);
    else
        moments_rows_kernel<__nv_bfloat16><<<grid, warps * 32, smem, st>>>(static_cast<const __nv_bfloat16*>(feat), n_clips, n_mels,
                                                                            frame_capacity, clip_stride,
                                                                            reinterpret_cast<const long long*>(frames), partial);
    moments_reduce_kernel<<<(2 * n_mels + 7) / 8, 256, 0, st>>>(partial, grid, 2 * n_mels, moments);
    cudaError_t e = cudaGetLastError();
    if (!workspace) cudaFreeAsync(partial, st);
    if (e != cudaSuccess) return cuda_fail(e, "acb_moments_accumulate launch");
    return ACB_OK;
}

int acb_moments_finalize(const double* m, int32_t n_mels, int64_t frames, double var_floor, double* bin_mean, double* bin_std,
                         double* global_mean, double* global_std) {
    if (!m || n_mels < 1 || frames < 1) return fail(ACB_ERR_INVALID, "acb_moments_finalize: bad argument");
    double S = 0.0, S2 = 0.0;
    for (int b = 0; b < n_mels; ++b) {
        const double mean = m[b] / (double)frames;
        const double var = std::max(m[n_mels + b] / (double)frames - mean * mean, var_floor);
        if (bin_mean) bin_mean[b] = mean;
        if (bin_std) bin_std[b] = std::sqrt(var);
        S += m[b];
        S2 += m[n_mels + b];
    }
    const double N = (double)frames * (double)n_mels;  // mel.numel() summed over files (compute_mel_stats.py:28)
    const double mean = S / N;
    const double var = std::max(S2 / N - mean * mean, var_floor);
    if (global_mean) *global_mean = mean;
    if (global_std) *global_std = std::sqrt(var);
    return ACB_OK;
}

int acb_normalize_per_utterance(const float* feat, float* out, int32_t n_clips, int32_t n_mels, int64_t frame_capacity,
                                const int64_t* frames, float min_std, void* stream) {
    if (n_clips <= 0) return ACB_OK;
    if (!feat || !out || n_mels < 1 || frame_capacity < 1) return fail(ACB_ERR_INVALID, "acb_normalize_per_utterance: bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long n_rows = (long long)n_clips * n_mels;
    const long long* fr = reinterpret_cast<const long long*>(frames);
    const bool aligned = ((reinterpret_cast<uintptr_t>(feat) | reinterpret_cast<uintptr_t>(out)) & 15) == 0 && frame_capacity % 4 == 0;
    const unsigned wgrid = (unsigned)((n_rows + 7) / 8);
    if (aligned && frame_capacity <= 32 * 4 * 8)
        normalize_rows_warp_kernel<8><<<wgrid, 256, 0, st>>>(feat, out, n_rows, n_mels, frame_capacity, fr, min_std);
    else if (aligned && frame_capacity <= 32 * 4 * 16)
        normalize_rows_warp_kernel<16><<<wgrid, 256, 0, st>>>(feat, out, n_rows, n_mels, frame_capacity, fr, min_std);
    else
        normalize_rows_kernel<<<n_clips * n_mels, 128, 0, st>>>(feat, out, n_mels, frame_capacity, fr, min_std);
    ACB_CUDA(cudaGetLastError());
    return ACB_OK;
}

int acb_crop_pad(const void* feat, int32_t dtype, int32_t n_clips, int32_t n_mels, int64_t frame_capacity, int64_t clip_stride,
                 const int64_t* frames, const int64_t* start, void* out, int64_t out_frames, float pad_value, void* stream) {
    if (n_clips <= 0 || out_frames <= 0) return ACB_OK;
    if (!feat || !out || n_mels < 1 || frame_capacity < 1) return fail(ACB_ERR_INVALID, "acb_crop_pad: bad argument");
    if (dtype != ACB_F32 && dtype != ACB_BF16) return fail(ACB_ERR_INVALID, "acb_crop_pad: bad dtype");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const long long n_rows = (long long)n_clips * n_mels;
    const unsigned grid = (unsigned)std::min<long long>((long long)current_sm_count() * 8, (n_rows + 7) / 8);
    if (dtype == ACB_F32)
        crop_pad_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float*>(feat), n_clips, n_mels, frame_capacity, clip_stride,
                                                    reinterpret_cast<const long long*>(frames), reinterpret_cast<const long long*>(start),
                                                    static_cast<float*>(out), out_frames, pad_value);
    else
        crop_pad_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(feat), n_clips, n_mels, frame_capacity, clip_stride,
                                                            reinterpret_cast<const long long*>(frames), reinterpret_cast<const long long*>(start),
                                                            static_cast<__nv_bfloat16*>(out), out_frames, pad_value);
    ACB_CUDA(cudaGetLastError());
    return ACB_OK;
}

int acb_pad_transpose(const void* feat_tm, int32_t dtype, const int64_t* row_offset, const int64_t* lens, int32_t n_clips, int32_t dim,
                      void* out, int64_t out_frames, float pad_value, const int64_t* mask_start, const int64_t* mask_len, void* stream) {
    if (n_clips <= 0 || out_frames <= 0) return ACB_OK;
    if (!feat_tm || !row_offset || !lens || !out || dim < 1) return fail(ACB_ERR_INVALID, "acb_pad_transpose: bad argument");
    if ((mask_start == nullptr) != (mask_len == nullptr)) return fail(ACB_ERR_INVALID, "acb_pad_transpose: mask_start and mask_len go together");
    if (dtype != ACB_F32 && dtype != ACB_BF16) return fail(ACB_ERR_INVALID, "acb_pad_transpose: bad dtype");
    if (n_clips > 65535) return fail(ACB_ERR_INVALID, "acb_pad_transpose: at most 65535 clips per call");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const dim3 grid((unsigned)((out_frames + 63) / 64), (unsigned)((dim + 63) / 64), (unsigned)n_clips);
    if (dtype == ACB_F32)
        pad_transpose_kernel<float><<<grid, 256, 0, st>>>(static_cast<const float*>(feat_tm), reinterpret_cast<const long long*>(row_offset),
                                                          reinterpret_cast<const long long*>(lens), dim, static_cast<float*>(out), out_frames,
                                                          pad_value, reinterpret_cast<const long long*>(mask_start),
                                                          reinterpret_cast<const long long*>(mask_len));
    else
        pad_transpose_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(static_cast<const __nv_bfloat16*>(feat_tm),
                                                                  reinterpret_cast<const long long*>(row_offset),
                                                                  reinterpret_cast<const long long*>(lens), dim,
                                                                  static_cast<__nv_bfloat16*>(out), out_frames, pad_value,
                                                                  reinterpret_cast<const long long*>(mask_start),
                                                                  reinterpret_cast<const long long*>(mask_len));
    ACB_CUDA(cudaGetLastError());
    return ACB_OK;
}

int acb_pcm16_to_float(const int16_t* pcm, float* out, int64_t n, void* stream) {
    if (n <= 0) return ACB_OK;
    if (!pcm || !out) return fail(ACB_ERR_INVALID, "acb_pcm16_to_float: null argument");
    const int blocks = (int)std::min<int64_t>(current_sm_count() * 8, (n / 8 + 255) / 256 + 1);
    pcm16_to_float_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(pcm, out, n, 1.0f / 32768.0f);
    ACB_CUDA(cudaGetLastError());
    return ACB_OK;
}

// Shared body of the host-buffer paths.  dev_pcm == nullptr: wav_host holds fp32 samples; otherwise int16 PCM that is staged in
// dev_pcm and widened on the device (half the bytes over PCIe).
static int forward_host_impl(const acb_frontend* fe_c, const void* wav_host, int32_t n_clips, int64_t length, void* out_host,
                             acb_logmel_args* tmpl, int16_t* dev_pcm, float* dev_in, void* dev_out, int32_t n_chunks, void* stream) {
    // out_host may be NULL: the features stay in dev_out (a training feed consumes them on the device; no D2H at all)
    if (!fe_c || !wav_host || !tmpl || !dev_in || !dev_out) return fail(ACB_ERR_INVALID, "acb_logmel_forward_host: null argument");
    if (n_clips <= 0) return ACB_OK;
    auto* fe = const_cast<acb_frontend*>(fe_c);
    const int64_t T = stft_frames(length, fe->n_fft, fe->hop, fe->opt);
    if (T < 0) return fail(ACB_ERR_INVALID, "acb_logmel_forward_host: clips too short");
    n_chunks = std::max(1, std::min(n_chunks, n_clips));
    const int64_t cap = tmpl->frame_capacity;
    const size_t esz = tmpl->out_dtype == ACB_BF16 ? 2 : 4;
    const int64_t out_clip = (int64_t)fe->n_mels * cap;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    std::lock_guard<std::mutex> lock(fe->mu);
    int prev = 0;
    ACB_CUDA(cudaGetDevice(&prev));
    if (prev != fe->device) ACB_CUDA(cudaSetDevice(fe->device));
    if (!fe->s_in) {
        ACB_CUDA(cudaStreamCreateWithFlags(&fe->s_in, cudaStreamNonBlocking));
        ACB_CUDA(cudaStreamCreateWithFlags(&fe->s_out, cudaStreamNonBlocking));
    }
    while ((int)fe->ev.size() < 2 * n_chunks + 1) {
        cudaEvent_t e;
        ACB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        fe->ev.push_back(e);
    }
    // order the side streams after work already queued on the caller's stream
    ACB_CUDA(cudaEventRecord(fe->ev[2 * n_chunks], st));
    ACB_CUDA(cudaStreamWaitEvent(fe->s_in, fe->ev[2 * n_chunks], 0));
    const int cover_tiles = (int)(((tmpl->fill_tail ? cap : T) + kTileFrames - 1) / kTileFrames);
    // Errors inside the loop are recorded and break out: the streams are always drained and the device restored before returning.
    int rc = ACB_OK;
    cudaError_t ce = cudaSuccess;
#define ACB_TRY(call) { ce = (call); if (ce != cudaSuccess) break; }
    for (int c = 0; c < n_chunks; ++c) {
        const int c0 = (int)((int64_t)n_clips * c / n_chunks), c1 = (int)((int64_t)n_clips * (c + 1) / n_chunks);
        if (c1 == c0) continue;
        const size_t n_samples = (size_t)(c1 - c0) * length;
        if (dev_pcm) {
            ACB_TRY(cudaMemcpyAsync(dev_pcm + (int64_t)c0 * length, static_cast<const int16_t*>(wav_host) + (int64_t)c0 * length,
                                    sizeof(int16_t) * n_samples, cudaMemcpyHostToDevice, fe->s_in));
        } else {
            ACB_TRY(cudaMemcpyAsync(dev_in + (int64_t)c0 * length, static_cast<const float*>(wav_host) + (int64_t)c0 * length,
                                    sizeof(float) * n_samples, cudaMemcpyHostToDevice, fe->s_in));
        }
        ACB_TRY(cudaEventRecord(fe->ev[2 * c], fe->s_in));
        ACB_TRY(cudaStreamWaitEvent(st, fe->ev[2 * c], 0));
        if (dev_pcm) {
            rc = acb_pcm16_to_float(dev_pcm + (int64_t)c0 * length, dev_in + (int64_t)c0 * length, (int64_t)n_samples, st);
            if (rc != ACB_OK) break;
        }
        acb_logmel_args a = *tmpl;
        a.wav = dev_in + (int64_t)c0 * length;
        a.clip_offset = nullptr; a.clip_length = nullptr; a.tile_start = nullptr;
        a.clip_stride = length; a.uniform_length = length;
        a.n_clips = c1 - c0; a.n_tiles = (c1 - c0) * cover_tiles;
        a.out = static_cast<unsigned char*>(dev_out) + (size_t)c0 * out_clip * esz;
        a.out_offset = nullptr; a.out_clip_stride = out_clip; a.frame_capacity_per_clip = nullptr;
        if (a.clip_peak) a.clip_peak = tmpl->clip_peak + c0;
        rc = acb_logmel_forward(fe, &a, st);
        if (rc != ACB_OK) break;
        if (!out_host) continue;
        ACB_TRY(cudaEventRecord(fe->ev[2 * c + 1], st));
        ACB_TRY(cudaStreamWaitEvent(fe->s_out, fe->ev[2 * c + 1], 0));
        ACB_TRY(cudaMemcpyAsync(static_cast<unsigned char*>(out_host) + (size_t)c0 * out_clip * esz,
                                static_cast<unsigned char*>(dev_out) + (size_t)c0 * out_clip * esz, (size_t)(c1 - c0) * out_clip * esz,
                                cudaMemcpyDeviceToHost, fe->s_out));
    }
#undef ACB_TRY
    cudaError_t e1 = cudaStreamSynchronize(fe->s_out);
    cudaError_t e2 = cudaStreamSynchronize(st);
    cudaError_t e3 = cudaStreamSynchronize(fe->s_in);
    int flag = 0;
    cudaError_t e4 = cudaMemcpy(&flag, fe->d_err, sizeof(int), cudaMemcpyDeviceToHost);
    if (e4 == cudaSuccess && flag) cudaMemset(fe->d_err, 0, sizeof(int));
    if (prev != fe->device) cudaSetDevice(prev);
    if (rc != ACB_OK) return rc;
    if (ce != cudaSuccess) return cuda_fail(ce, "acb_logmel_forward_host");
    if (e1 != cudaSuccess) return cuda_fail(e1, "acb_logmel_forward_host sync");
    if (e2 != cudaSuccess) return cuda_fail(e2, "acb_logmel_forward_host sync");
    if (e3 != cudaSuccess) return cuda_fail(e3, "acb_logmel_forward_host sync");
    if (e4 != cudaSuccess) return cuda_fail(e4, "acb_logmel_forward_host flag");
    if (flag) return fail(ACB_ERR_CUDA, "acb_logmel_forward_host: a sample-tile copy did not complete inside the kernel (results are invalid)");
    return ACB_OK;
}

int acb_logmel_forward_host(const acb_frontend* fe, const float* wav_host, int32_t n_clips, int64_t length, void* out_host,
                            acb_logmel_args* tmpl, float* dev_in, void* dev_out, int32_t n_chunks, void* stream) {
    return forward_host_impl(fe, wav_host, n_clips, length, out_host, tmpl, nullptr, dev_in, dev_out, n_chunks, stream);
}

int acb_logmel_forward_host_pcm16(const acb_frontend* fe, const int16_t* pcm_host, int32_t n_clips, int64_t length, void* out_host,
                                  acb_logmel_args* tmpl, int16_t* dev_pcm, float* dev_in, void* dev_out, int32_t n_chunks, void* stream) {
    if (!dev_pcm) return fail(ACB_ERR_INVALID, "acb_logmel_forward_host_pcm16: null staging buffer");
    return forward_host_impl(fe, pcm_host, n_clips, length, out_host, tmpl, dev_pcm, dev_in, dev_out, n_chunks, stream);
}

}  // extern "C"
