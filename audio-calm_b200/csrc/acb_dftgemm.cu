// B200 (sm_100a) tensor-core route of the log-mel front-end: STFT as a DFT-GEMM on tcgen05 with split-fp16 operands.
//
// This is the "Whisper-style" preset BASELINE.json's north star words the path as (n_fft 400, hop 160, 80-band bank of
// models/mel_filters.npz, log10 with clamp, max-8 dynamic-range floor, (x + 4) / 4) -- what the reference runs inside the Hugging
// Face ASR pipeline that scores its TTS output (eval/eval_calm.py:548-552 -> transformers.WhisperFeatureExtractor).  The
// reference's own extractor (preprocess/core.py, n_fft 1024) stays on the CUDA-core FFT kernel in acb_kernels.cu: DESIGN.md
// section 3.1 measures why a DFT-GEMM loses there.  At n_fft = 400 the GEMM is 6.5x smaller per frame and wins.
//
// Math (one frame x[0..399], periodic symmetric window w[n] = w[400-n], xw = w * x, indices mod 400):
//   s[n] = xw[n] + xw[n+200], d[n] = xw[n] - xw[n+200]                      (radix-2 split: even / odd bins)
//   se[n] = s[n] + s[200-n], so[n] = s[n] - s[200-n], de[n] = d[n] - d[200-n], do[n] = d[n] + d[200-n],  n = 0..100
//   Re X[2m]   =  sum_n c_n se[n] cos(2 pi m n / 200)          Im X[2m]   = -sum_n so[n] sin(2 pi m n / 200)
//   Re X[2m+1] =  sum_n c_n de[n] cos(2 pi (2m+1) n / 400)     Im X[2m+1] = -sum_n c_n do[n] sin(2 pi (2m+1) n / 400)
//   (c_n = 1/2 on the self-paired rows n = 0 / 100, folded into the matrices.)
// Four real GEMMs  D_g[128 frames x 112] = A_g[128 x 112] * B_g[112 x 112]^T  replace a 400 x 402 DFT: 4x fewer flops.
// fp32 accuracy from fp16 tensor cores: A = A_hi + A_lo, B = B_hi + B_lo (fp16 pairs, 22 significant bits),
// D = A_hi B_hi + A_lo B_hi + A_hi B_lo accumulated in fp32 in TMEM (measured 2e-6 on the final features).
//
// Kernel (persistent, one CTA per SM, tiles of 128 frames of one clip; 16 worker warps + 1 MMA issuer warp + 1 loader warp, every
// hand-off an mbarrier):
//   1. loader warp: the tile's 20960 samples are staged in shared memory by 6 TMA tensor copies (the batch viewed as rows of 32
//      floats, SWIZZLE_128B: frames are 5 rows apart, so a warp's 16-byte loads of 32 different frames are conflict-free) while
//      the previous tile's epilogue runs; positions outside the clip (reflection about sample 0 / L-1) are patched by the workers;
//      batches that are not 128-byte row addressable are gathered by the workers instead;
//   2. K loop, 7 steps of 16: the first 8 worker warps (thread = frame row x k-half) build the step's A slices (window, folds, fp16
//      hi/lo split with packed conversions): the lo halves go to shared memory in the canonical K-major no-swizzle core-matrix
//      layout, the hi halves to the 64 TMEM columns the accumulators leave free (tcgen05.st; the MMAs that use them take A from
//      tensor memory); the loader streams the step's B slices (28 KB of the 200 KB DFT matrices, L2-resident) with one bulk copy;
//      the issuer's elected lane issues 12 tcgen05.mma (M 128, N 112, K 16, kind::f16) and commits to mbarriers.  A and B are
//      double-buffered: the MMAs of step k run under the CUDA-core work of step k+1;
//   3. epilogue (all 16 worker warps): tcgen05.ld of the four accumulators, |X|^2 into shared memory as [bin][frame] (the operand
//      stages are idle), then the banded mel projection with lane = 4 consecutive frames (one 16-byte load per bin) and warp = a
//      group of bands (warp-uniform weights), clamp, log, affine, 512-byte band stores, per-clip max / per-tile min by atomics;
//   4. the affine (x + 4) / 4 is applied at the store (it commutes with the floor); the kernel also records the minimum of every tile,
//      so the second kernel (dynamic-range floor, per-clip max - 8) only touches the tiles that hold values below the floor.
#include "audiocalm_b200.h"

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <string>
#include <vector>

namespace acb {
extern thread_local std::string g_last_error;
}

namespace acbg {

constexpr int kNfft = 400;
constexpr int kHop = 160;
constexpr int kBinsAll = 201;
constexpr int kTileFrames = 128;
constexpr int kAhiCols = 448;                       // first TMEM column of the A_hi stages (the 64 the accumulators leave free): [stage][gemm][8 columns = 16 fp16]
constexpr int kWorkerWarps = 16;                    // all of them run the epilogue (4 per TMEM lane quarter)
constexpr int kPrepWarps = 8;                       // the first 8 build the A slices, thread = (frame row, k-half), 16-byte stores
constexpr int kWorkerThreads = kWorkerWarps * 32;
constexpr int kThreads = kWorkerThreads + 64;      // + one MMA issuer warp + one B-slice loader warp (one elected lane each)
constexpr int kKpad = 112;                       // K of every GEMM (n = 0..100 used)
constexpr int kNpad = 112;                       // N of every GEMM (m = 0..100 used)
constexpr int kKsteps = kKpad / 16;              // 7
constexpr int kGemms = 4;
constexpr int kBlocks = kTileFrames + 3;         // hop blocks staged per tile
constexpr int kStageRows = 656;                  // staged sample tile: rows of 32 floats (128 B); 131 * 160 = 20960 samples = 655 rows
constexpr int kBoxRows = 128;                    // TMA box: 128 rows (16 KB, a multiple of the 1 KB swizzle atom); 5 of them + one of 16 rows
constexpr int kSampleFloats = kStageRows * 32;   // 20992
constexpr int kASliceBytes = 2 * kTileFrames * 16;            // two k-halves x 128 rows x 8 halves
constexpr int kAStageBytes = kGemms * 2 * kASliceBytes;       // 32768
constexpr int kBSliceBytes = kNpad * 16 * 2;                  // 3584
constexpr int kBStageBytes = kGemms * 2 * kBSliceBytes;       // 28672
constexpr int kPowBins = 224;                    // 7 chunks of 32 bins of |X|^2 staged per frame (bins 201.. are padding)
constexpr int kMaxWeights = 3072;                // packed non-zero filterbank weights (banded form)
constexpr int kTmemCols = 512;
constexpr int kMaxMels = 128;
constexpr int kBandCost = 16;                      // fixed cost of a band (logs, stores) in units of one weight, for balancing the band groups
constexpr float kPrescale = 4096.f;                // power-of-two scale of the A operands (see acb_dftgemm_create)

// shared memory carve-up (bytes)
constexpr int kOffSamples = 0;
constexpr int kOffA = (kSampleFloats * 4 + 1023) & ~1023;     // 83968
constexpr int kOffB = kOffA + 2 * kAStageBytes;               // +65536
constexpr int kOffWin = kOffB + 2 * kBStageBytes;             // +57344
constexpr int kOffBand = kOffWin + 2 * kKpad * 4;            // int4 per band: first bin, bins, weight offset
constexpr int kOffMelW = kOffBand + kMaxMels * 16;
constexpr int kOffBar = kOffMelW + kMaxWeights * 4;
constexpr int kOffPow = kOffA;                                // |X|^2 [224 bins][128 rows] fp32 reuses the A/B stages during the epilogue
static_assert(kPowBins * kTileFrames * 4 <= 2 * kAStageBytes + 2 * kBStageBytes, "power tile must fit the operand stages");
constexpr int kOffAff = kOffBar + 96;                         // float2 per band: (scale, shift) of the affine
constexpr int kOffMom = kOffAff + kMaxMels * 8;               // float2 [2][kMaxMels]: compensated per-band sums of the fused moments
constexpr int kSmemBytes = kOffMom + 2 * kMaxMels * 8;
static_assert(kOffWin % 16 == 0 && kOffBand % 16 == 0 && kOffBar % 8 == 0 && kOffAff % 8 == 0, "alignment");
static_assert(kSmemBytes <= 227 * 1024, "shared memory budget");

static int fail(int code, const std::string& msg) {
    acb::g_last_error = msg;
    return code;
}
static int cuda_fail(cudaError_t e, const char* what) {
    acb::g_last_error = std::string(what) + ": " + cudaGetErrorString(e);
    return ACB_ERR_CUDA;
}
#define ACBG_CUDA(call)                                       \
    do {                                                      \
        cudaError_t e__ = (call);                             \
        if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
    } while (0)

// ---------------------------------------------------------------------------------------------------------------------
// device helpers: mbarrier, bulk copy, tcgen05
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void worker_sync() {   // named barrier of the worker warps (barrier 0 is __syncthreads, 1 the band exchange)
    asm volatile("bar.sync 2, %0;" ::"n"(kWorkerThreads) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// Bounded wait: a wrong descriptor or a lost completion must not hang the GPU box.  try_wait carries a suspend-time hint: a waiting warp
// sleeps in hardware until the phase completes (or the hint expires) instead of polling.  Without it 45 % of the kernel's issued
// instructions were mbarrier polls of idle warps, each one an access to shared memory next to the K loop's operand traffic:
// 0.480 -> 0.463 ms per 256 x 30 s (hint 100 ns: 0.465, 1 us: 0.4634, 10 us: 0.4629).  Returns false after ~10 s.
constexpr uint32_t kWaitHintNs = 10000;
__device__ __forceinline__ bool mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok = 0;
    for (int spin = 0; spin < (1 << 20) && !ok; ++spin) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(ok) : "r"(bar), "r"(parity), "r"(kWaitHintNs) : "memory");
    }
    return ok != 0;
}
__device__ __forceinline__ void bulk_copy_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void tensor_copy_2d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, uint32_t bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
                 ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(bar) : "memory");
}
// K-major, SWIZZLE_NONE shared-memory matrix descriptor: 8-row x 16-byte core matrices (rows 16 bytes apart);
// lbo = byte distance between core matrices adjacent in K, sbo = between 8-row groups (validated on B200 by
// tools/microbench/umma_hankel.cu).
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
    d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;   // descriptor version of sm_100
    return d;
}
// kind::f16 instruction descriptor: D = f32 (bit 4), A = B = fp16 (format 0), both K-major, N >> 3 at bit 17, M >> 4 at bit 24
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N) {
    return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void mma_f16_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// A operand in tensor memory (M = 128 rows = lanes, K = 16 fp16 = 8 columns of two packed halves), B in shared memory
__device__ __forceinline__ void mma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
                 ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(r0), "r"(r1), "r"(r2), "r"(r3) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void mma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&r)[16]) {
    uint32_t u[16];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
                 : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]), "=r"(u[8]),
                   "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
                 : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 16; ++i) r[i] = __uint_as_float(u[i]);
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&r)[8]) {
    uint32_t u[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n"
                 : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7])
                 : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = __uint_as_float(u[i]);
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// (hi, lo) += x with the rounding error of hi + x carried in lo (Knuth two-sum)
__device__ __forceinline__ void two_sum_add(float2& acc, float x) {
    const float t = __fadd_rn(acc.x, x);
    const float bb = __fsub_rn(t, acc.x);
    const float e = __fadd_rn(__fsub_rn(acc.x, __fsub_rn(t, bb)), __fsub_rn(x, bb));
    acc.y = __fadd_rn(acc.y, e);
    acc.x = t;
}

__device__ __forceinline__ float lg2_normal(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// order-preserving int key of a float (atomicMax on ints)
__device__ __forceinline__ int float_key(float v) {
    const int b = __float_as_int(v);
    return b >= 0 ? b : (b ^ 0x7fffffff);
}
__host__ __device__ __forceinline__ float key_float(int k) {
    const int b = k >= 0 ? k : (k ^ 0x7fffffff);
#ifdef __CUDA_ARCH__
    return __int_as_float(b);
#else
    float f;
    std::memcpy(&f, &b, 4);
    return f;
#endif
}

struct Params {
    // tables (device)
    const uint8_t* b_slices;   // [kKsteps][kGemms][2][kBSliceBytes] fp16 DFT matrices, core-matrix layout
    const float* win_fwd;      // [112] w[n] (0 beyond n = 100)
    const float* win_rev;      // [112] w[200 - n] (0 beyond n = 100)
    const int4* bands;         // [n_mels] (first bin, bins, offset into mel_w, 0): the filterbank in banded form
    const float* mel_w;        // [n_mel_w] packed weights (with the 2^-24 of the pre-scale folded in)
    int n_mel_w;
    int band_group[kWorkerWarps + 1];   // worker warp w projects bands [band_group[w], band_group[w + 1]) (balanced by weight count)
    int n_mels;
    float clamp_min, log_scale, log_floor;
    // batch
    const float* wav;
    long long clip_stride;
    long long length;
    int n_clips;
    int tiles_per_clip;
    int frames_out;            // frames stored per clip
    // output
    void* out;                 // fp32 or bf16 [n_clips][n_mels][frame_capacity]
    int out_bf16;
    long long out_clip_stride;
    long long frame_capacity;
    int* clip_max;             // [n_clips] ordered-int keys of the per-clip maximum, or nullptr (no dynamic-range floor)
    int* tile_min;             // [n_clips * tiles_per_clip] ordered-int keys of MINUS the per-tile minimum (tiles above the floor are skipped later)
    float aff_scale, aff_shift;   // out = v * aff_scale + aff_shift (1, 0 when no affine)
    const float* bin_mean;     // per-band affine (v - bin_mean[b]) / bin_std[b] instead of the uniform pair, or nullptr
    const float* bin_std;
    const long long* clip_length;   // [n_clips] samples of every clip (<= length; rows are padded to `length`), or nullptr: uniform
    const float* clip_peak;    // [n_clips] max|x|: power-of-two pre-scale of the samples (any amplitude fits the fp16 operands) and,
    int peak_norm;             //   with peak_norm, the fused process_audio_chunk gain 0.95 / (peak + 1e-8); or nullptr
    int drop_last_frame;
    float fill_value;          // stored for frames beyond a clip's own count (ragged batches)
    double* moments_partial;   // [gridDim.x][2][n_mels] per-CTA sums of v and v^2 over the frames that exist, or nullptr
    int* error_flag;           // set to 1 when a barrier wait timed out
    int use_tma;               // the batch is 128-byte row addressable (16-byte aligned base, clip_stride % 32 == 0): tensor copies
};

// A-operand values of one thread for one K step: 8 consecutive n of its frame row, for the 4 GEMMs
struct Fold8 {
    float se[8], so[8], de[8], dd[8];
};

__device__ __forceinline__ uint32_t pack_half2(__half a, __half b) {
    return (uint32_t)__half_as_ushort(a) | ((uint32_t)__half_as_ushort(b) << 16);
}

// split 8 fp32 values into fp16 (hi, lo) (packed conversions: F2FP / HADD2.F32); the hi halves go to tensor memory, 4 columns
// (8 packed halves) of this thread's lane at `t_hi`, the lo halves to shared memory as one 16-byte core-matrix row
__device__ __forceinline__ void split_store_tmem(const float (&v)[8], uint32_t t_hi, uint8_t* dst_lo) {
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const __half2 h = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
        const float2 hf = __half22float2(h);
        const __half2 l = __floats2half2_rn(v[2 * i] - hf.x, v[2 * i + 1] - hf.y);
        hi[i] = *reinterpret_cast<const uint32_t*>(&h);
        lo[i] = *reinterpret_cast<const uint32_t*>(&l);
    }
    tmem_st4(t_hi, hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(dst_lo) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
}

// Staged float index of linear position `lin` (= 160 * row + 120 + n).  The tile is staged as rows of 32 floats in the TMA
// SWIZZLE_128B layout (the 16-byte chunk index within a 128-byte row is XORed with the row index mod 8): frames are 160 floats
// = 5 rows apart, so the 8 threads of a 16-byte load phase (8 consecutive frames) hit 8 different chunk positions -- no bank
// conflicts, and the whole tile arrives with 6 tensor copies instead of one copy per hop block.
__device__ __forceinline__ int staged_index(int lin) { return lin ^ (((lin >> 5) & 7) << 2); }

// One K step of A-operand construction for one thread: 8 consecutive n (n0 .. n0 + 7) of its frame row, for the 4 GEMMs.
// `srow` = the staged samples, `base` = 160 * row + 120 (linear staged position of the frame's sample 0).
__device__ __forceinline__ void build_a_slices(const float* __restrict__ srow, int base, int n0, const float* __restrict__ s_wf,
                                               const float* __restrict__ s_wr, uint8_t* dst, uint32_t t_hi, float pre) {
    float xa[8], xc[8], xb[8], xe[8];
    {
        const float* pa = srow + staged_index(base + n0);              // x[n0 .. n0+7]
        const float* pc = srow + staged_index(base + 200 + n0);        // x[200+n0 .. 200+n0+7]
        // the second 16-byte chunk of an aligned group of 8 sits at the swizzled index ^ 4
        const float4 a0 = *reinterpret_cast<const float4*>(pa), a1 = *reinterpret_cast<const float4*>(srow + (staged_index(base + n0) ^ 4));
        const float4 c0 = *reinterpret_cast<const float4*>(pc), c1 = *reinterpret_cast<const float4*>(srow + (staged_index(base + 200 + n0) ^ 4));
        xa[0] = a0.x; xa[1] = a0.y; xa[2] = a0.z; xa[3] = a0.w; xa[4] = a1.x; xa[5] = a1.y; xa[6] = a1.z; xa[7] = a1.w;
        xc[0] = c0.x; xc[1] = c0.y; xc[2] = c0.z; xc[3] = c0.w; xc[4] = c1.x; xc[5] = c1.y; xc[6] = c1.z; xc[7] = c1.w;
        // x[200 - n0 - i] and x[400 - n0 - i], i = 0..7: the aligned group of 8 below plus one element above
        const float* pb = srow + staged_index(base + 192 - n0);        // x[192-n0 .. 199-n0]
        const float* pb8 = srow + staged_index(base + 200 - n0);       // x[200-n0]
        const float4 b0 = *reinterpret_cast<const float4*>(pb), b1 = *reinterpret_cast<const float4*>(srow + (staged_index(base + 192 - n0) ^ 4));
        xb[0] = *pb8; xb[1] = b1.w; xb[2] = b1.z; xb[3] = b1.y; xb[4] = b1.x; xb[5] = b0.w; xb[6] = b0.z; xb[7] = b0.y;
        const float* pe = srow + staged_index(base + 392 - n0);        // x[392-n0 .. 399-n0]
        const float* pe8 = srow + staged_index(base + (n0 == 0 ? 0 : 400 - n0));   // x[400-n0], index taken mod 400
        const float4 e0 = *reinterpret_cast<const float4*>(pe), e1 = *reinterpret_cast<const float4*>(srow + (staged_index(base + 392 - n0) ^ 4));
        xe[0] = *pe8; xe[1] = e1.w; xe[2] = e1.z; xe[3] = e1.y; xe[4] = e1.x; xe[5] = e0.w; xe[6] = e0.z; xe[7] = e0.y;
    }
    Fold8 f;
    {
        const float4 wf0 = *reinterpret_cast<const float4*>(s_wf + n0), wf1 = *reinterpret_cast<const float4*>(s_wf + n0 + 4);
        const float4 wr0 = *reinterpret_cast<const float4*>(s_wr + n0), wr1 = *reinterpret_cast<const float4*>(s_wr + n0 + 4);
        float wa[8] = {wf0.x, wf0.y, wf0.z, wf0.w, wf1.x, wf1.y, wf1.z, wf1.w};
        float wb[8] = {wr0.x, wr0.y, wr0.z, wr0.w, wr1.x, wr1.y, wr1.z, wr1.w};
        if (pre != 1.f) {      // warp-uniform: the clip's power-of-two pre-scale (exact), folded into the window
#pragma unroll
            for (int i = 0; i < 8; ++i) { wa[i] *= pre; wb[i] *= pre; }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float pa = wa[i] * xa[i], pe = wa[i] * xe[i];      // w[400-n] = w[n]
            const float pb = wb[i] * xb[i], pc = wb[i] * xc[i];      // w[200+n] = w[200-n]
            const float sn = pa + pc, sr = pb + pe, dn = pa - pc, dr = pb - pe;
            f.se[i] = sn + sr;
            f.so[i] = sn - sr;
            f.de[i] = dn - dr;
            f.dd[i] = dn + dr;
        }
    }
    split_store_tmem(f.se, t_hi + 0, dst + 1 * kASliceBytes);
    split_store_tmem(f.so, t_hi + 8, dst + 3 * kASliceBytes);
    split_store_tmem(f.de, t_hi + 16, dst + 5 * kASliceBytes);
    split_store_tmem(f.dd, t_hi + 24, dst + 7 * kASliceBytes);
    tmem_st_wait();
}

// Where a tile's samples come from: clip pointer and the clip sample held by staged position 0.  Returns whether the tile is fetched by
// TMA tensor copies (the batch layout allows it; positions outside the clip are then patched with the reflection by the workers) or
// gathered entirely by the workers.
__device__ __forceinline__ bool tile_source(const Params& p, int tile, const float*& src, long long& g0) {
    const int clip = tile / p.tiles_per_clip, tic = tile - clip * p.tiles_per_clip;
    src = p.wav + (long long)clip * p.clip_stride;
    g0 = (long long)(tic * kTileFrames - 2) * kHop;
    return p.use_tma != 0;
}

// Warp roles: 16 worker warps run the epilogue and gather edge tiles, the first 8 of them (thread = frame row x k-half) also build
// the A slices; warp 16 (one elected lane) issues the MMAs, warp 17 streams the B slices and prefetches sample tiles.  All hand-offs are mbarriers: no
// CTA-wide barrier sits inside the K loop.
template <bool kMoments>
__global__ void __launch_bounds__(kThreads, 1) dftgemm_logmel_kernel(const Params p, const __grid_constant__ CUtensorMap tm_box128,
                                                                     const __grid_constant__ CUtensorMap tm_box16) {
    extern __shared__ __align__(1024) uint8_t smem[];
    float* s_samples = reinterpret_cast<float*>(smem + kOffSamples);
    uint8_t* s_a = smem + kOffA;
    uint8_t* s_b = smem + kOffB;
    float* s_wf = reinterpret_cast<float*>(smem + kOffWin);
    float* s_wr = s_wf + kKpad;
    int4* s_band = reinterpret_cast<int4*>(smem + kOffBand);
    float* s_melw = reinterpret_cast<float*>(smem + kOffMelW);
    float* s_pow = reinterpret_cast<float*>(smem + kOffPow);
    const uint32_t bar_base = smem_u32(smem + kOffBar);
    const uint32_t bar_smp = bar_base;              // sample tile landed (bulk copies, tx count)
    const uint32_t bar_bfull0 = bar_base + 8;       // [2] B slices of a stage landed (tx count)
    const uint32_t bar_afull0 = bar_base + 24;      // [2] A slices of a stage written (8 worker warps)
    const uint32_t bar_mma0 = bar_base + 40;        // [2] the MMAs reading a stage are complete (tcgen05.commit)
    const uint32_t bar_tile = bar_base + 56;        // all MMAs of the tile complete: accumulators ready
    const uint32_t bar_tfree = bar_base + 64;       // accumulators drained by the epilogue (8 worker warps)
    const uint32_t bar_sfree = bar_base + 72;       // sample tile no longer read (8 worker warps)
    uint32_t* s_tmem_slot = reinterpret_cast<uint32_t*>(smem + kOffBar + 80);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int row = ((warp & 3) << 5) | lane;     // frame row of the tile = TMEM lane (workers)
    const int hsel = (warp >> 2) & 1;             // prep warps: k-half of the K step
    const int qsel = (warp >> 2) & 3;             // power pass: which quarter of the accumulator columns of the row

    // ---- one-time setup ----
    for (int i = tid; i < kKpad; i += kThreads) { s_wf[i] = p.win_fwd[i]; s_wr[i] = p.win_rev[i]; }
    for (int i = tid; i < p.n_mels; i += kThreads) s_band[i] = p.bands[i];
    for (int i = tid; i < p.n_mel_w; i += kThreads) s_melw[i] = p.mel_w[i];
    float2* s_aff = reinterpret_cast<float2*>(smem + kOffAff);
    float2* s_mom = reinterpret_cast<float2*>(smem + kOffMom);
    for (int i = tid; i < p.n_mels; i += kThreads) {
        float sc = p.aff_scale, sh = p.aff_shift;
        if (p.bin_mean) { sc = 1.f / __ldg(p.bin_std + i); sh = -__ldg(p.bin_mean + i) * sc; }
        s_aff[i] = make_float2(sc, sh);
        s_mom[i] = make_float2(0.f, 0.f);
        s_mom[kMaxMels + i] = make_float2(0.f, 0.f);
    }
    if (tid == 0) {
        mbar_init(bar_smp, 1);
        mbar_init(bar_bfull0, 1);
        mbar_init(bar_bfull0 + 8, 1);
        mbar_init(bar_afull0, kPrepWarps);
        mbar_init(bar_afull0 + 8, kPrepWarps);
        mbar_init(bar_mma0, 1);
        mbar_init(bar_mma0 + 8, 1);
        mbar_init(bar_tile, 1);
        mbar_init(bar_tfree, kWorkerWarps);
        mbar_init(bar_sfree, kPrepWarps);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem_slot)), "r"(kTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *s_tmem_slot;
    const int n_tiles = p.n_clips * p.tiles_per_clip;
    bool ok = (smem_u32(smem) & 1023u) == 0;       // the swizzled sample tile needs a 1 KB aligned base

    if (warp == kWorkerWarps + 1) {
        // ======================================= B-slice loader =======================================
        // Streams the 28 KB of DFT-matrix slices of every K step from L2 as soon as the stage's previous MMAs have completed,
        // independently of the issuer, so the copy of step k+1 overlaps the MMAs of step k.
        // The same warp (all lanes, one 640-byte hop block each per round) fetches the next tile's samples as soon as the workers
        // have left the K loop, so no worker warp spends its time issuing copies.
        auto fetch_samples = [&](int tile) {
            const float* src;
            long long g0;
            if (!tile_source(p, tile, src, g0)) return;     // not row addressable: the workers gather the tile themselves
            const long long row0 = ((src - p.wav) + g0) >> 5;       // first 128-byte row of the tile in the batch buffer
            if (lane == 0) mbar_arrive_expect_tx(bar_smp, kStageRows * 128);
            __syncwarp();
            if (lane < 6) {
                const CUtensorMap* tm = lane < 5 ? &tm_box128 : &tm_box16;
                tensor_copy_2d(smem_u32(s_samples) + lane * (kBoxRows * 128), tm, 0, (int)(row0 + lane * kBoxRows), bar_smp);
            }
        };
        uint32_t gs = 0, tile_iter = 0;
        if ((int)blockIdx.x < n_tiles) fetch_samples(blockIdx.x);
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tile_iter) {
            if (lane == 0) {
                for (int ks = 0; ks < kKsteps; ++ks) {
                    const uint32_t st = (gs + ks) & 1u, use = (gs + ks) >> 1;
                    if (gs + ks >= 2) ok = mbar_wait(bar_mma0 + 8 * st, (use - 1) & 1u) && ok;      // the stage's previous MMAs are complete
                    // the epilogue of the previous tile keeps |X|^2 in the operand stages: wait until it is done with them
                    if (ks == 0 && tile_iter > 0) ok = mbar_wait(bar_tfree, (tile_iter - 1) & 1u) && ok;
                    mbar_arrive_expect_tx(bar_bfull0 + 8 * st, kBStageBytes);
                    bulk_copy_g2s(smem_u32(s_b + st * kBStageBytes), p.b_slices + (size_t)ks * kBStageBytes, kBStageBytes, bar_bfull0 + 8 * st);
                }
            }
            gs += kKsteps;
            __syncwarp();
            ok = mbar_wait(bar_sfree, tile_iter & 1u) && ok;      // every worker is past its last read of the sample tile
            if (tile + (int)gridDim.x < n_tiles) fetch_samples(tile + gridDim.x);
        }
    } else if (warp == kWorkerWarps) {
        // ======================================= MMA issuer =======================================
        if (lane == 0) {
            const uint32_t idesc = make_idesc_f16(kTileFrames, kNpad);
            uint32_t gs = 0, tile_iter = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++tile_iter) {
                for (int ks = 0; ks < kKsteps; ++ks, ++gs) {
                    const uint32_t st = gs & 1u, use = gs >> 1;
                    ok = mbar_wait(bar_afull0 + 8 * st, use & 1u) && ok;      // A slices written by the worker warps
                    ok = mbar_wait(bar_bfull0 + 8 * st, use & 1u) && ok;      // B slices landed (implies: accumulators drained, see the loader)
                    tc_fence_after();
                    const uint32_t a_base = smem_u32(s_a + st * kAStageBytes), b_base = smem_u32(s_b + st * kBStageBytes);
#pragma unroll
                    for (int g = 0; g < kGemms; ++g) {
                        const uint32_t a_hi = tmem + (uint32_t)(kAhiCols + st * 32 + g * 8);
                        const uint64_t a_lo = make_desc(a_base + (2 * g + 1) * kASliceBytes, kTileFrames * 16, 128);
                        const uint64_t b_hi = make_desc(b_base + (2 * g) * kBSliceBytes, 128, 256);
                        const uint64_t b_lo = make_desc(b_base + (2 * g + 1) * kBSliceBytes, 128, 256);
                        const uint32_t d = tmem + (uint32_t)(g * kNpad);
                        mma_f16_ts(d, a_hi, b_hi, idesc, ks > 0);
                        mma_f16_ss(d, a_lo, b_hi, idesc, 1);
                        mma_f16_ts(d, a_hi, b_lo, idesc, 1);
                    }
                    mma_commit(bar_mma0 + 8 * st);
                    if (ks == kKsteps - 1) mma_commit(bar_tile);
                }
            }
        }
    } else {
        // ================================================ workers ================================================
        const int wtid = tid;                       // 0..255
        uint32_t gs = 0, smp_uses = 0, tile_iter = 0;
        const int b_begin = p.band_group[warp], b_end = p.band_group[warp + 1];     // this warp's bands of the mel pass (read once: an indexed parameter load)
        const float clamp_min = p.clamp_min, log_scale = p.log_scale, log_floor = p.log_floor;
        const long long cap = p.frame_capacity;

        // sample staging of one tile: with a row-addressable batch every tile arrives by the loader warp's tensor copies (bar_smp
        // completes a phase, returns true); otherwise the workers gather it here with reflection
        auto stage_samples = [&](int tile) -> bool {
            const float* src;
            long long g0;
            if (tile_source(p, tile, src, g0)) return true;
            const long long L = p.clip_length ? __ldg(p.clip_length + tile / p.tiles_per_clip) : p.length;
#pragma unroll 8
            for (int i = wtid; i < kBlocks * kHop; i += kWorkerThreads) {
                long long idx = g0 + i;
                if (idx < 0) idx = -idx;                       // reflection about sample 0 (torch.stft center=True, pad_mode="reflect")
                if (idx >= L) idx = 2 * (L - 1) - idx;         // and about sample L - 1
                float v = 0.f;
                if (idx >= 0 && idx < L) v = __ldg(src + idx);
                s_samples[staged_index(i)] = v;
            }
            return false;
        };

        int tile = blockIdx.x;
        bool smp_async = false;
        if (tile < n_tiles) smp_async = stage_samples(tile);

        for (; tile < n_tiles; tile += gridDim.x, ++tile_iter) {
            const int clip = tile / p.tiles_per_clip, tic = tile - clip * p.tiles_per_clip;
            // geometry and scaling of this tile's clip: own length (ragged batches are rows padded to p.length), frames that exist,
            // power-of-two pre-scale of the samples and the factor that undoes it (and applies the peak-normalisation gain) on the mel powers
            const long long clip_len = p.clip_length ? __ldg(p.clip_length + clip) : p.length;
            const int clip_frames = min(p.frames_out, (int)(clip_len / kHop) + (p.drop_last_frame ? 0 : 1));
            float pre = 1.f, post = 1.f;
            if (p.clip_peak) {
                const float peak = __ldg(p.clip_peak + clip);
                if (peak > 0.f && peak < 3.0e38f) {
                    int e;
                    frexpf(peak, &e);                                   // peak = m 2^e, 0.5 <= m < 1: |x 2^-e| < 1
                    pre = exp2f((float)-e);
                    const float g = p.peak_norm ? (0.95f / (peak + 1e-8f)) * exp2f((float)e) : exp2f((float)e);
                    post = g * g;
                }
            }
            if (smp_async) {
                ok = mbar_wait(bar_smp, smp_uses & 1) && ok;
                ++smp_uses;
                // positions outside the clip (reflection about sample 0 / L - 1: torch.stft center=True, pad_mode="reflect") are
                // patched over what the tensor copy brought in; only the first and the last tiles of a clip have any
                const float* src = p.wav + (long long)clip * p.clip_stride;
                const long long g0 = (long long)(tic * kTileFrames - 2) * kHop, L = clip_len;
                const long long e0 = max(0LL, L - g0);              // first staged position beyond the clip (0: the whole tile lies beyond a short clip of a ragged batch)
                if (g0 < 0 || e0 < kBlocks * kHop) {                // CTA-uniform
                    if (g0 < 0)
                        for (int i = wtid; i < (int)-g0; i += kWorkerThreads) {
                            const long long idx = -(g0 + i);
                            s_samples[staged_index(i)] = idx < L ? __ldg(src + idx) : 0.f;
                        }
                    if (e0 < kBlocks * kHop) {                      // the 200 reflected samples the last frame needs (and a margin)
                        const int i = (int)e0 + wtid;
                        if (wtid < 256 && i < kBlocks * kHop) {
                            const long long idx = 2 * (L - 1) - (g0 + i);
                            s_samples[staged_index(i)] = idx >= 0 ? __ldg(src + idx) : 0.f;
                        }
                    }
                    worker_sync();
                }
            } else {
                worker_sync();   // gathered samples visible
            }
            // ---------------- K loop: build the A slices of each step ----------------
            const int base = kHop * row + 120;
            if (warp < kPrepWarps) {
#pragma unroll 1
                for (int ks = 0; ks < kKsteps; ++ks) {
                    const uint32_t st = (gs + ks) & 1u, use = (gs + ks) >> 1;
                    if (gs + ks >= 2) ok = mbar_wait(bar_mma0 + 8 * st, (use - 1) & 1u) && ok;   // MMAs that read this stage are complete
                    build_a_slices(s_samples, base, 16 * ks + 8 * hsel, s_wf, s_wr,
                                   s_a + st * kAStageBytes + hsel * (kTileFrames * 16) + row * 16,
                                   tmem + ((uint32_t)((warp & 3) << 5) << 16) + (uint32_t)(kAhiCols + st * 32 + hsel * 4), pre);
                    fence_async_smem();      // generic-proxy writes of A -> visible to the tensor core's async proxy
                    tc_fence_before();       // (and the tensor-memory stores of A_hi, completed by tcgen05.wait::st, ordered before the arrive)
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_afull0 + 8 * st);
                }
                // this warp is past its last read of the sample tile: tell the loader, which prefetches an interior next tile
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_sfree);
            }
            gs += kKsteps;
            // an edge next tile is gathered here by all workers once every prep warp has left the K loop
            const int next_tile = tile + gridDim.x;
            bool next_async = false;
            if (next_tile < n_tiles) {
                const float* nsrc;
                long long ng0;
                next_async = tile_source(p, next_tile, nsrc, ng0);
                if (!next_async) {
                    worker_sync();
                    stage_samples(next_tile);
                }
            }

            // ---------------- epilogue: |X|^2 -> shared memory, banded mel, log, store ----------------
            ok = mbar_wait(bar_tile, tile_iter & 1u) && ok;      // every MMA of the tile is complete: accumulators ready, stages idle
            tc_fence_after();
            {
                // power pass: the 4 warps of a lane quarter share the 14 units of 8 accumulator columns (16 bins); s_pow[bin][row]
                // (a warp writes 32 consecutive rows: conflict-free)
                const uint32_t t_row = tmem + ((uint32_t)((warp & 3) << 5) << 16);
#pragma unroll 1
                for (int u = (14 * qsel) / 4; u < (14 * (qsel + 1)) / 4; ++u) {
                    float d0[8], d1[8], d2[8], d3[8];
                    tmem_ld8(t_row + (uint32_t)(0 * kNpad + 8 * u), d0);
                    tmem_ld8(t_row + (uint32_t)(1 * kNpad + 8 * u), d1);
                    tmem_ld8(t_row + (uint32_t)(2 * kNpad + 8 * u), d2);
                    tmem_ld8(t_row + (uint32_t)(3 * kNpad + 8 * u), d3);
                    tmem_ld_wait();
                    float* dst = s_pow + (16 * u) * kTileFrames + row;
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        dst[(2 * i) * kTileFrames] = fmaf(d0[i], d0[i], d1[i] * d1[i]);          // even bin 2m
                        dst[(2 * i + 1) * kTileFrames] = fmaf(d2[i], d2[i], d3[i] * d3[i]);      // odd bin 2m + 1
                    }
                }
                tc_fence_before();
                worker_sync();       // the whole power tile is in shared memory; the accumulators are drained

                // mel pass: lane = 4 consecutive frames (one 16-byte load per bin), warp = one group of bands (weights are
                // warp-uniform broadcast loads); a warp stores 32 x 4 consecutive frames of one band = 512 contiguous bytes
                const int frame0 = tic * kTileFrames + 4 * lane;
                const int n_valid = clip_frames - frame0;             // frames of this lane that exist (<= 0: none)
                const int n_store = p.frames_out - frame0;            // frames of this lane inside the row (the rest of them get fill_value)
                long long out_col = (long long)clip * p.out_clip_stride + (long long)b_begin * cap + frame0;    // element index in out
                const int esize = p.out_bf16 ? 2 : 4;
                // four consecutive frames of a band go out as one 16-byte (fp32) / 8-byte (bf16) store when every row keeps them aligned
                const bool vec_store = n_valid >= 4 && ((reinterpret_cast<uintptr_t>(p.out) | (uintptr_t)(p.out_clip_stride * esize) | (uintptr_t)(cap * esize)) & (4 * esize - 1)) == 0;
                float vmax = -3.0e38f, vmin = 3.0e38f, chk = 0.f;
                const float clamp_eff = clamp_min / post, log_post = post == 1.f ? 0.f : log2f(post) * log_scale;
                const float4* pow4 = reinterpret_cast<const float4*>(s_pow) + lane;
                int4 bd_next = s_band[b_begin];               // a band's record is fetched while the previous band is being finished
                for (int b = b_begin; b < b_end; ++b, out_col += cap) {
                    const int4 bd = bd_next;
                    bd_next = s_band[min(b + 1, p.n_mels - 1)];
                    const float4* pp = pow4 + bd.x * (kTileFrames / 4);
                    const float* ww = s_melw + bd.z;
                    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
                    for (int i = 0; i < bd.y; ++i) {
                        const float w = ww[i];
                        const float4 q = pp[i * (kTileFrames / 4)];
                        a.x = fmaf(w, q.x, a.x);
                        a.y = fmaf(w, q.y, a.y);
                        a.z = fmaf(w, q.z, a.z);
                        a.w = fmaf(w, q.w, a.w);
                    }
                    chk += (a.x + a.y) + (a.z + a.w);          // inf / NaN powers (operand overflow) must not hide behind the clamp
                    // the factor that undoes the pre-scale / applies the peak gain moves through the log: log(a post) = log a + log post,
                    // and the clamp is compared against clamp_min / post
                    float4 v;
                    v.x = (a.x > clamp_eff) ? fmaf(lg2_normal(a.x), log_scale, log_post) : log_floor;
                    v.y = (a.y > clamp_eff) ? fmaf(lg2_normal(a.y), log_scale, log_post) : log_floor;
                    v.z = (a.z > clamp_eff) ? fmaf(lg2_normal(a.z), log_scale, log_post) : log_floor;
                    v.w = (a.w > clamp_eff) ? fmaf(lg2_normal(a.w), log_scale, log_post) : log_floor;
                    const float raw[4] = {v.x, v.y, v.z, v.w};          // un-normalised log-mel: maximum / minimum tracking, moments
                    if (kMoments) {                                     // per-band sums over the frames that exist (compiled out of the plain kernel)
                        float sm = 0.f, sq = 0.f;
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            if (j < n_valid) { sm += raw[j]; sq = fmaf(raw[j], raw[j], sq); }
#pragma unroll
                        for (int o = 16; o >= 1; o >>= 1) {
                            sm += __shfl_xor_sync(0xffffffffu, sm, o);
                            sq += __shfl_xor_sync(0xffffffffu, sq, o);
                        }
                        if (lane == 0) {                                // every band has exactly one owner warp
                            two_sum_add(s_mom[b], sm);
                            two_sum_add(s_mom[kMaxMels + b], sq);
                        }
                    }
                    // the affine is applied here; the dynamic-range floor commutes with it: max(v, M - r) * s + t = max(v s + t, (M - r) s + t)
                    const float2 af = s_aff[b];
                    v.x = fmaf(v.x, af.x, af.y);
                    v.y = fmaf(v.y, af.x, af.y);
                    v.z = fmaf(v.z, af.x, af.y);
                    v.w = fmaf(v.w, af.x, af.y);
                    if (vec_store) {
                        if (p.out_bf16) {
                            const __nv_bfloat162 lo2 = __floats2bfloat162_rn(v.x, v.y), hi2 = __floats2bfloat162_rn(v.z, v.w);
                            *reinterpret_cast<uint2*>(static_cast<__nv_bfloat16*>(p.out) + out_col) =
                                make_uint2(*reinterpret_cast<const uint32_t*>(&lo2), *reinterpret_cast<const uint32_t*>(&hi2));
                        } else {
                            *reinterpret_cast<float4*>(static_cast<float*>(p.out) + out_col) = v;
                        }
                        vmax = fmaxf(fmaxf(vmax, fmaxf(raw[0], raw[1])), fmaxf(raw[2], raw[3]));
                        vmin = fminf(fminf(vmin, fminf(raw[0], raw[1])), fminf(raw[2], raw[3]));
                    } else {
                        const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            if (j < n_store) {
                                const float o = j < n_valid ? vv[j] : p.fill_value;
                                if (p.out_bf16) static_cast<__nv_bfloat16*>(p.out)[out_col + j] = __float2bfloat16_rn(o);
                                else static_cast<float*>(p.out)[out_col + j] = o;
                                if (j < n_valid) {
                                    vmax = fmaxf(vmax, raw[j]);
                                    vmin = fminf(vmin, raw[j]);
                                }
                            }
                    }
                }
                // a sample beyond the fp16 range of the split operands (|x| >= ~4 without a pre-scale) turns into inf / NaN features:
                // flag it (bit 1) instead of returning garbage silently
                if (!(fabsf(chk) < 3.0e38f) && n_valid > 0) atomicOr(p.error_flag, 2);
                if (p.clip_max) {
#pragma unroll
                    for (int o = 16; o >= 1; o >>= 1) vmax = fmaxf(vmax, __shfl_xor_sync(0xffffffffu, vmax, o));
                    if (lane == 0 && vmax > -3.0e38f) atomicMax(p.clip_max + clip, float_key(vmax));
#pragma unroll
                    for (int o = 16; o >= 1; o >>= 1) vmin = fminf(vmin, __shfl_xor_sync(0xffffffffu, vmin, o));
                    if (lane == 0 && vmin < 3.0e38f) atomicMax(p.tile_min + tile, float_key(-vmin));   // key of -min: same initial pattern as clip_max
                }
                worker_sync();       // nobody reads the power tile any more: the operand stages may be refilled
                if (lane == 0) mbar_arrive(bar_tfree);
            }
            smp_async = next_async;
        }
    }

    if (!ok && p.error_flag) atomicOr(p.error_flag, 1);
    tc_fence_before();
    __syncthreads();
    if (kMoments) {              // per-CTA partial sums (compensated fp32 pairs -> fp64 once), combined in a fixed order afterwards
        const float2* s_mom = reinterpret_cast<const float2*>(smem + kOffMom);
        double* dst = p.moments_partial + (size_t)blockIdx.x * 2 * p.n_mels;
        for (int i = tid; i < p.n_mels; i += kThreads) {
            dst[i] = (double)s_mom[i].x + (double)s_mom[i].y;
            dst[p.n_mels + i] = (double)s_mom[kMaxMels + i].x + (double)s_mom[kMaxMels + i].y;
        }
    }
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols));
}

// Dynamic-range floor of the stored features (WhisperFeatureExtractor: maximum(x, max - 8); the affine (x + 4) / 4 has already been
// applied and commutes with it).  One CTA per 4 tiles of 128 frames; a tile whose minimum is not below the floor -- the common
// case -- is skipped after one load, so the pass costs a fraction of a read + write of the features.
constexpr int kFloorTilesPerCta = 4;
__device__ __forceinline__ float load_out(const float* q) { return *q; }
__device__ __forceinline__ float load_out(const __nv_bfloat16* q) { return __bfloat162float(*q); }
__device__ __forceinline__ void store_out(float* q, float v) { *q = v; }
__device__ __forceinline__ void store_out(__nv_bfloat16* q, float v) { *q = __float2bfloat16_rn(v); }

template <typename T>
__global__ void __launch_bounds__(256) dftgemm_floor_kernel(T* __restrict__ out, long long out_clip_stride, long long frame_capacity, int n_mels,
                                                            int frames, int tiles_per_clip, const int* __restrict__ clip_max,
                                                            const int* __restrict__ tile_min, float range, float aff_scale, float aff_shift,
                                                            const float* __restrict__ bin_mean, const float* __restrict__ bin_std,
                                                            const long long* __restrict__ clip_length, int drop_last_frame) {
    const int clip = blockIdx.y;
    const float floor_raw = key_float(__ldg(clip_max + clip)) - range;      // on the un-normalised log-mel; stored values carry the affine
    if (clip_length) frames = min(frames, (int)(__ldg(clip_length + clip) / kHop) + (drop_last_frame ? 0 : 1));
    auto floor_of = [&](int b) {
        if (bin_mean == nullptr) return fmaf(floor_raw, aff_scale, aff_shift);
        const float sc = 1.f / __ldg(bin_std + b);
        return fmaf(floor_raw, sc, -__ldg(bin_mean + b) * sc);
    };
    const int t_end = min(tiles_per_clip, (int)(blockIdx.x + 1) * kFloorTilesPerCta);
    for (int tic = blockIdx.x * kFloorTilesPerCta; tic < t_end; ++tic) {
        if (!(-key_float(__ldg(tile_min + clip * tiles_per_clip + tic)) < floor_raw)) continue;     // CTA-uniform: nothing below the floor
        const int f0 = tic * kTileFrames, nf = min(kTileFrames, frames - f0);
        T* base = out + (long long)clip * out_clip_stride + f0;
        if (sizeof(T) == 4 && nf == kTileFrames && ((reinterpret_cast<uintptr_t>(base) | (uintptr_t)(frame_capacity * 4)) & 15) == 0) {
#pragma unroll 4
            for (int i = threadIdx.x; i < n_mels * (kTileFrames / 4); i += blockDim.x) {
                const int b = i / (kTileFrames / 4), f4 = i - b * (kTileFrames / 4);
                const float floor_v = floor_of(b);
                float4* q = reinterpret_cast<float4*>(base + (long long)b * frame_capacity) + f4;
                float4 v = *q;
                if (fminf(fminf(v.x, v.y), fminf(v.z, v.w)) < floor_v) {
                    v.x = fmaxf(v.x, floor_v); v.y = fmaxf(v.y, floor_v); v.z = fmaxf(v.z, floor_v); v.w = fmaxf(v.w, floor_v);
                    *q = v;
                }
            }
        } else {
            for (int i = threadIdx.x; i < n_mels * kTileFrames; i += blockDim.x) {
                const int b = i / kTileFrames, f = i - b * kTileFrames;
                if (f < nf) {
                    const float floor_v = floor_of(b);
                    T* q = base + (long long)b * frame_capacity + f;
                    if (load_out(q) < floor_v) store_out(q, floor_v);
                }
            }
        }
    }
}

// Sum the per-CTA moment partials in a fixed order and add them into the running accumulators: one warp per value
__global__ void __launch_bounds__(256) dftgemm_moments_reduce_kernel(const double* __restrict__ partial, int n_parts, int n_vals, double* __restrict__ acc) {
    const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (i >= n_vals) return;
    double s = 0.0;
    for (int k = lane; k < n_parts; k += 32) s += partial[(size_t)k * n_vals + i];
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) acc[i] += s;
}

}  // namespace acbg

// =====================================================================================================================
// host side
// =====================================================================================================================
struct acb_dftgemm {
    int device = 0;
    int n_mels = 0;
    int log_kind = 0;
    float clamp_min = 0.f;
    int num_sms = 0;
    int band_group[acbg::kWorkerWarps + 1] = {0};
    void* d_blob = nullptr;
    const uint8_t* d_b = nullptr;
    const float* d_wf = nullptr;
    const float* d_wr = nullptr;
    const int4* d_bands = nullptr;
    const float* d_melw = nullptr;
    int n_mel_w = 0;
    int* d_err = nullptr;
};

using namespace acbg;

static uint16_t half_bits(float v) {
    const __half h = __float2half_rn(v);
    uint16_t u;
    std::memcpy(&u, &h, 2);
    return u;
}
static float half_value(uint16_t u) {
    __half h;
    std::memcpy(&h, &u, 2);
    return __half2float(h);
}

extern "C" {

int64_t acb_dftgemm_workspace_ints(int64_t length, int drop_last_frame, int32_t n_clips) {
    const int64_t T = 1 + length / kHop - (drop_last_frame ? 1 : 0);
    if (length <= kNfft / 2 || n_clips < 0) return -1;
    return (int64_t)n_clips * (1 + (T + kTileFrames - 1) / kTileFrames);
}

int64_t acb_dftgemm_frames(int64_t length, int drop_last_frame) {
    if (length <= kNfft / 2) return -1;
    return 1 + length / kHop - (drop_last_frame ? 1 : 0);
}

int acb_dftgemm_create(acb_dftgemm** out, int device, int n_fft, int hop, int n_mels, const float* window_host, const float* fb_host,
                       float clamp_min, int log_kind) {
    if (!out || !window_host || !fb_host) return fail(ACB_ERR_INVALID, "acb_dftgemm_create: null argument");
    if (n_fft != kNfft || hop != kHop)
        return fail(ACB_ERR_UNSUPPORTED, "acb_dftgemm_create: the tensor-core route is built for n_fft=400, hop=160 (got n_fft=" +
                                             std::to_string(n_fft) + ", hop=" + std::to_string(hop) + ")");
    if (n_mels < 2 || n_mels > kMaxMels) return fail(ACB_ERR_UNSUPPORTED, "acb_dftgemm_create: n_mels must be in [2, 128]");
    if (log_kind != ACB_LOG_NATURAL && log_kind != ACB_LOG_10) return fail(ACB_ERR_INVALID, "acb_dftgemm_create: bad log_kind");
    if (!(clamp_min >= 1.17549435e-38f)) return fail(ACB_ERR_INVALID, "acb_dftgemm_create: clamp_min must be a positive normal float");
    // the folds need w[n] == w[400 - n]
    for (int n = 1; n < kNfft / 2; ++n)
        if (std::fabs(window_host[n] - window_host[kNfft - n]) > 1e-6f * std::fmax(1.f, std::fabs(window_host[n])))
            return fail(ACB_ERR_UNSUPPORTED, "acb_dftgemm_create: the window is not symmetric (w[n] != w[n_fft - n])");

    // ---- DFT matrices, fp16 (hi, lo), [ks][g][hi/lo] slices in the K-major no-swizzle core-matrix layout ----
    std::vector<uint8_t> bsl((size_t)kKsteps * kBStageBytes, 0);
    const double two_pi = 6.283185307179586476925286766559;
    for (int g = 0; g < kGemms; ++g)
        for (int m = 0; m < kNpad; ++m)
            for (int n = 0; n < kKpad; ++n) {
                double v = 0.0;
                if (g == 0 && m <= 100 && n <= 100) v = std::cos(two_pi * ((m * n) % 200) / 200.0) * ((n == 0 || n == 100) ? 0.5 : 1.0);
                if (g == 1 && m <= 100 && n >= 1 && n <= 99) v = std::sin(two_pi * ((m * n) % 200) / 200.0);
                if (g == 2 && m <= 99 && n <= 99) v = std::cos(two_pi * (((2 * m + 1) * n) % 400) / 400.0) * (n == 0 ? 0.5 : 1.0);
                if (g == 3 && m <= 99 && n >= 1 && n <= 100) v = std::sin(two_pi * (((2 * m + 1) * n) % 400) / 400.0) * (n == 100 ? 0.5 : 1.0);
                const float vf = (float)v;
                const uint16_t hi = half_bits(vf);
                const uint16_t lo = half_bits((float)(v - (double)half_value(hi)));
                const int ks = n / 16, kk = n % 16;
                const size_t off = (size_t)(m / 8) * 256 + (size_t)(kk / 8) * 128 + (size_t)(m % 8) * 16 + (size_t)(kk % 8) * 2;
                uint8_t* s_hi = bsl.data() + (size_t)ks * kBStageBytes + (size_t)(2 * g) * kBSliceBytes + off;
                uint8_t* s_lo = bsl.data() + (size_t)ks * kBStageBytes + (size_t)(2 * g + 1) * kBSliceBytes + off;
                std::memcpy(s_hi, &hi, 2);
                std::memcpy(s_lo, &lo, 2);
            }

    // ---- window halves ----
    std::vector<float> wf(kKpad, 0.f), wr(kKpad, 0.f);
    // The window carries a power-of-two pre-scale (exact): fp16's narrow exponent would push the lo halves of quiet audio into the
    // subnormal range (absolute precision 2^-24); with x 4096 the split keeps 22 bits for amplitudes down to ~3e-5.  The
    // 2^-24 on the power spectrum is folded into the mel weights (exact).  Operand range: 4 |x| 4096 < 65504, i.e. |x| < 3.99.
    for (int n = 0; n <= 100; ++n) { wf[n] = window_host[n] * kPrescale; wr[n] = window_host[200 - n] * kPrescale; }

    // ---- filterbank in banded form: band b = one contiguous run of bins [start, start + len) with packed weights.  The 2^-24 of
    // the pre-scaled power spectrum is folded into the weights (exact).  Bands are split between the two k-halves of the CTA so
    // that both get about the same number of multiply-adds.
    std::vector<int> bands((size_t)n_mels * 4, 0);
    std::vector<float> melw;
    for (int b = 0; b < n_mels; ++b) {
        int lo = -1, hi = -1;
        for (int k = 0; k < kBinsAll; ++k)
            if (fb_host[(size_t)k * n_mels + b] != 0.f) { if (lo < 0) lo = k; hi = k; }
        bands[(size_t)b * 4 + 0] = lo < 0 ? 0 : lo;
        bands[(size_t)b * 4 + 1] = lo < 0 ? 0 : hi - lo + 1;
        bands[(size_t)b * 4 + 2] = (int)melw.size();
        for (int k = lo; lo >= 0 && k <= hi; ++k) melw.push_back(fb_host[(size_t)k * n_mels + b] / (kPrescale * kPrescale));
    }
    if ((int)melw.size() > kMaxWeights)
        return fail(ACB_ERR_UNSUPPORTED, "acb_dftgemm_create: filterbank too dense (" + std::to_string(melw.size()) + " banded weights, limit " +
                                             std::to_string(kMaxWeights) + ")");
    int band_group[kWorkerWarps + 1];
    {
        long long total = 0, run = 0;
        for (int b = 0; b < n_mels; ++b) total += bands[(size_t)b * 4 + 1] + kBandCost;
        int g = 0;
        band_group[0] = 0;
        for (int b = 0; b < n_mels; ++b) {      // cut after the band that reaches the next multiple of total / 8
            run += bands[(size_t)b * 4 + 1] + kBandCost;
            while (g + 1 < kWorkerWarps && run * kWorkerWarps >= total * (g + 1)) band_group[++g] = b + 1;
        }
        while (g < kWorkerWarps) band_group[++g] = n_mels;
    }
    melw.resize((melw.size() + 3) & ~(size_t)3, 0.f);

    acb_dftgemm* fe = new acb_dftgemm();
    fe->device = device;
    fe->n_mels = n_mels;
    fe->log_kind = log_kind;
    fe->clamp_min = clamp_min;
    for (int g = 0; g <= kWorkerWarps; ++g) fe->band_group[g] = band_group[g];
    int prev = 0;
    cudaGetDevice(&prev);
    auto bail = [&](int rc) { cudaSetDevice(prev); delete fe; return rc; };
    if (cudaSetDevice(device) != cudaSuccess) return bail(fail(ACB_ERR_CUDA, "acb_dftgemm_create: cudaSetDevice failed"));
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return bail(fail(ACB_ERR_CUDA, "acb_dftgemm_create: cudaGetDeviceProperties failed"));
    if (prop.major != 10) return bail(fail(ACB_ERR_UNSUPPORTED, "acb_dftgemm_create: needs an sm_100 device (tcgen05)"));
    fe->num_sms = prop.multiProcessorCount;
    const size_t b_bytes = bsl.size(), w_bytes = kKpad * 4, bd_bytes = bands.size() * 4, mw_bytes = melw.size() * 4, p_bytes = bd_bytes + mw_bytes;
    fe->n_mel_w = (int)melw.size();
    const size_t total = b_bytes + 2 * w_bytes + p_bytes + 16;
    if (cudaMalloc(&fe->d_blob, total) != cudaSuccess) return bail(fail(ACB_ERR_CUDA, "acb_dftgemm_create: cudaMalloc failed"));
    uint8_t* d = static_cast<uint8_t*>(fe->d_blob);
    fe->d_b = d;
    fe->d_wf = reinterpret_cast<const float*>(d + b_bytes);
    fe->d_wr = reinterpret_cast<const float*>(d + b_bytes + w_bytes);
    fe->d_bands = reinterpret_cast<const int4*>(d + b_bytes + 2 * w_bytes);
    fe->d_melw = reinterpret_cast<const float*>(d + b_bytes + 2 * w_bytes + bd_bytes);
    fe->d_err = reinterpret_cast<int*>(d + b_bytes + 2 * w_bytes + p_bytes);
    bool good = cudaMemcpy(d, bsl.data(), b_bytes, cudaMemcpyHostToDevice) == cudaSuccess &&
                cudaMemcpy(d + b_bytes, wf.data(), w_bytes, cudaMemcpyHostToDevice) == cudaSuccess &&
                cudaMemcpy(d + b_bytes + w_bytes, wr.data(), w_bytes, cudaMemcpyHostToDevice) == cudaSuccess &&
                cudaMemcpy(d + b_bytes + 2 * w_bytes, bands.data(), bd_bytes, cudaMemcpyHostToDevice) == cudaSuccess &&
                cudaMemcpy(d + b_bytes + 2 * w_bytes + bd_bytes, melw.data(), mw_bytes, cudaMemcpyHostToDevice) == cudaSuccess &&
                cudaMemset(fe->d_err, 0, 16) == cudaSuccess &&
                cudaFuncSetAttribute(dftgemm_logmel_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes) == cudaSuccess &&
                cudaFuncSetAttribute(dftgemm_logmel_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes) == cudaSuccess;
    if (!good) {
        cudaFree(fe->d_blob);
        return bail(fail(ACB_ERR_CUDA, std::string("acb_dftgemm_create: table upload failed: ") + cudaGetErrorString(cudaGetLastError())));
    }
    cudaSetDevice(prev);
    *out = fe;
    return ACB_OK;
}

int acb_dftgemm_destroy(acb_dftgemm* fe) {
    if (!fe) return ACB_OK;
    int prev = 0;
    cudaGetDevice(&prev);
    cudaSetDevice(fe->device);
    if (fe->d_blob) cudaFree(fe->d_blob);
    cudaSetDevice(prev);
    delete fe;
    return ACB_OK;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link against libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = [] {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) f = nullptr;
        return reinterpret_cast<EncodeTiledFn>(f);
    }();
    return fn;
}
// The batch buffer as rows of 32 floats: [rows][32], boxes of `box_rows` rows, 128-byte swizzle
static bool make_sample_map(CUtensorMap* tm, const float* base, long long rows, int box_rows) {
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) return false;
    const cuuint64_t dims[2] = {32, (cuuint64_t)rows};
    const cuuint64_t strides[1] = {128};
    const cuuint32_t box[2] = {32, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

int64_t acb_dftgemm_moments_workspace_bytes(const acb_dftgemm* fe) {
    if (!fe) return fail(ACB_ERR_INVALID, "acb_dftgemm_moments_workspace_bytes: null handle");
    return (int64_t)fe->num_sms * 2 * fe->n_mels * (int64_t)sizeof(double);
}

int acb_dftgemm_forward(const acb_dftgemm* fe, const acb_dftgemm_args* a, void* stream) {
    if (!fe || !a) return fail(ACB_ERR_INVALID, "acb_dftgemm_forward: null argument");
    if (!a->wav || !a->out) return fail(ACB_ERR_INVALID, "acb_dftgemm_forward: wav and out must be device pointers");
    if (a->out_dtype != ACB_F32 && a->out_dtype != ACB_BF16) return fail(ACB_ERR_INVALID, "acb_dftgemm_forward: out_dtype must be ACB_F32 or ACB_BF16");
    if (a->n_clips <= 0) return ACB_OK;
    const int64_t T = acb_dftgemm_frames(a->length, a->drop_last_frame);
    if (T < 0) return fail(ACB_ERR_INVALID, "acb_dftgemm_forward: clips of " + std::to_string(a->length) + " samples; reflect padding needs more than " + std::to_string(kNfft / 2));
    if (T == 0) return ACB_OK;
    if (a->frame_capacity < T) return fail(ACB_ERR_INVALID, "acb_dftgemm_forward: frame_capacity " + std::to_string(a->frame_capacity) + " < frames " + std::to_string(T));
    if (a->clip_stride < a->length) return fail(ACB_ERR_INVALID, "acb_dftgemm_forward: clip_stride < length");
    if (a->out_clip_stride < (int64_t)fe->n_mels * a->frame_capacity) return fail(ACB_ERR_INVALID, "acb_dftgemm_forward: out_clip_stride too small");
    if (a->dyn_range > 0.f && !a->clip_max) return fail(ACB_ERR_INVALID, "acb_dftgemm_forward: dyn_range needs the clip_max workspace");
    if (a->affine < 0 || a->affine > 2) return fail(ACB_ERR_INVALID, "acb_dftgemm_forward: bad affine mode");
    if (a->affine == 1 && !(a->affine_std > 0.f)) return fail(ACB_ERR_INVALID, "acb_dftgemm_forward: affine_std must be positive");
    if (a->affine == 2 && (!a->bin_mean || !a->bin_std)) return fail(ACB_ERR_INVALID, "acb_dftgemm_forward: per-bin affine needs bin_mean / bin_std");
    if (a->peak_norm && !a->clip_peak) return fail(ACB_ERR_INVALID, "acb_dftgemm_forward: peak_norm needs clip_peak (acb_peak_abs)");
    if (a->moments && !a->moments_workspace) return fail(ACB_ERR_INVALID, "acb_dftgemm_forward: moments need a workspace");
    if (a->moments && a->dyn_range > 0.f)
        return fail(ACB_ERR_UNSUPPORTED, "acb_dftgemm_forward: fused moments describe the features before the per-clip dynamic-range floor; "
                                         "with dyn_range > 0 run acb_moments_accumulate over the stored features instead");
    const int64_t tiles_per_clip = (T + kTileFrames - 1) / kTileFrames;
    if (tiles_per_clip * a->n_clips > INT32_MAX) return fail(ACB_ERR_INVALID, "acb_dftgemm_forward: more than 2^31 tiles in one call");
    cudaStream_t s = static_cast<cudaStream_t>(stream);

    Params p{};
    p.b_slices = fe->d_b;
    p.win_fwd = fe->d_wf;
    p.win_rev = fe->d_wr;
    p.bands = fe->d_bands;
    p.mel_w = fe->d_melw;
    p.n_mel_w = fe->n_mel_w;
    for (int g = 0; g <= kWorkerWarps; ++g) p.band_group[g] = fe->band_group[g];
    p.n_mels = fe->n_mels;
    p.clamp_min = fe->clamp_min;
    p.log_scale = fe->log_kind == ACB_LOG_10 ? 0.30102999566398120f : 0.69314718055994531f;
    p.log_floor = fe->log_kind == ACB_LOG_10 ? (float)std::log10((double)fe->clamp_min) : (float)std::log((double)fe->clamp_min);
    p.wav = a->wav;
    p.clip_stride = a->clip_stride;
    p.length = a->length;
    p.n_clips = a->n_clips;
    p.tiles_per_clip = (int)tiles_per_clip;
    p.frames_out = (int)T;
    p.out = a->out;
    p.out_bf16 = a->out_dtype == ACB_BF16;
    p.out_clip_stride = a->out_clip_stride;
    p.frame_capacity = a->frame_capacity;
    p.clip_max = a->dyn_range > 0.f ? a->clip_max : nullptr;
    p.tile_min = p.clip_max ? a->clip_max + a->n_clips : nullptr;
    p.aff_scale = a->affine == 1 ? 1.f / a->affine_std : 1.f;
    p.aff_shift = a->affine == 1 ? -a->affine_mean / a->affine_std : 0.f;
    p.bin_mean = a->affine == 2 ? a->bin_mean : nullptr;
    p.bin_std = a->affine == 2 ? a->bin_std : nullptr;
    p.clip_length = reinterpret_cast<const long long*>(a->clip_length);
    p.clip_peak = a->clip_peak;
    p.peak_norm = a->peak_norm;
    p.drop_last_frame = a->drop_last_frame;
    p.fill_value = a->fill_value;
    p.error_flag = fe->d_err;
    if (p.clip_max)   // one fill for both arrays: keys below every float (tile_min holds keys of the negated minimum)
        ACBG_CUDA(cudaMemsetAsync(p.clip_max, 0x80, sizeof(int) * (size_t)a->n_clips * (size_t)(1 + tiles_per_clip), s));
    const int64_t n_tiles = tiles_per_clip * a->n_clips;
    const int grid = (int)std::min<int64_t>(n_tiles, fe->num_sms);
    p.moments_partial = a->moments ? static_cast<double*>(a->moments_workspace) : nullptr;
    // tensor maps of the sample buffer: usable when every tile start is a whole 128-byte row of a 16-byte aligned buffer
    CUtensorMap tm128, tm16;
    std::memset(&tm128, 0, sizeof(tm128));
    std::memset(&tm16, 0, sizeof(tm16));
    const bool row_addressable = (reinterpret_cast<uintptr_t>(a->wav) & 15) == 0 && (a->n_clips == 1 || a->clip_stride % 32 == 0);
    if (row_addressable) {
        // rows that hold samples of the batch (a partial last row is read whole: allocations are 256-byte granular)
        const long long rows = ((long long)(a->n_clips - 1) * a->clip_stride + a->length + 31) / 32;
        p.use_tma = rows > 0 && make_sample_map(&tm128, a->wav, rows, kBoxRows) && make_sample_map(&tm16, a->wav, rows, 16);
    }
    if (a->moments) dftgemm_logmel_kernel<true><<<grid, kThreads, kSmemBytes, s>>>(p, tm128, tm16);
    else dftgemm_logmel_kernel<false><<<grid, kThreads, kSmemBytes, s>>>(p, tm128, tm16);
    ACBG_CUDA(cudaGetLastError());
    if (p.clip_max) {
        const dim3 fgrid((unsigned)((tiles_per_clip + kFloorTilesPerCta - 1) / kFloorTilesPerCta), (unsigned)a->n_clips);
        if (p.out_bf16)
            dftgemm_floor_kernel<__nv_bfloat16><<<fgrid, 256, 0, s>>>(static_cast<__nv_bfloat16*>(a->out), a->out_clip_stride, a->frame_capacity, fe->n_mels,
                                                                     (int)T, (int)tiles_per_clip, p.clip_max, p.tile_min, a->dyn_range, p.aff_scale,
                                                                     p.aff_shift, p.bin_mean, p.bin_std, p.clip_length, p.drop_last_frame);
        else
            dftgemm_floor_kernel<float><<<fgrid, 256, 0, s>>>(static_cast<float*>(a->out), a->out_clip_stride, a->frame_capacity, fe->n_mels, (int)T,
                                                             (int)tiles_per_clip, p.clip_max, p.tile_min, a->dyn_range, p.aff_scale, p.aff_shift,
                                                             p.bin_mean, p.bin_std, p.clip_length, p.drop_last_frame);
        ACBG_CUDA(cudaGetLastError());
    }
    if (a->moments) {
        const int n_vals = 2 * fe->n_mels;
        dftgemm_moments_reduce_kernel<<<(n_vals + 7) / 8, 256, 0, s>>>(p.moments_partial, grid, n_vals, a->moments);
        ACBG_CUDA(cudaGetLastError());
    }
    return ACB_OK;
}

int acb_dftgemm_check(const acb_dftgemm* fe, void* stream) {
    if (!fe) return fail(ACB_ERR_INVALID, "acb_dftgemm_check: null handle");
    int flag = 0;
    ACBG_CUDA(cudaStreamSynchronize(static_cast<cudaStream_t>(stream)));
    ACBG_CUDA(cudaMemcpy(&flag, fe->d_err, sizeof(int), cudaMemcpyDeviceToHost));
    if (flag) {
        cudaMemset(fe->d_err, 0, sizeof(int));
        if (flag & 1) return fail(ACB_ERR_CUDA, "acb_dftgemm_check: a tensor-core pipeline barrier timed out inside the kernel (results are invalid)");
        return fail(ACB_ERR_INVALID, "acb_dftgemm_check: non-finite features -- a sample beyond the fp16 operand range (|x| >= ~4) or a NaN input; "
                                     "pass clip_peak (acb_peak_abs) so that every clip is pre-scaled by a power of two");
    }
    return ACB_OK;
}

}  // extern "C"
