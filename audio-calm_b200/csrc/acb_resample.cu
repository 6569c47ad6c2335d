// Polyphase sinc resampling with torchaudio.transforms.Resample semantics (method "sinc_interp_hann"): the host-side
// resampling step of the reference's dataset driver (preprocess/process_dataset.py:135-137), moved to the device.
//
// With (O, N) = (orig, new) / gcd, output sample y[b * N + j] (block b, phase j) is
//     y[b * N + j] = sum_t w_j[t] * x[b * O + s_j + t - width]      (x = 0 outside the clip)
// where w_j is the band of non-zero fp32 coefficients of row j of torchaudio's [N][K] kernel and s_j its first column.
// Skipped taps are exact zeros, so for finite input this is torchaudio's zero-padded strided conv1d.
//
// Layout.  A CTA owns one tile of TB consecutive blocks of one row (TB * N outputs).  It stages the tile's input span in shared
// memory (16-byte vector loads where the whole vector lies inside the clip, zero fill outside it, int16 widened to x / 32768 on
// the way in), computes, stages the outputs in shared memory and writes them with coalesced stores.  A thread owns one phase
// j and R consecutive blocks of it, with the phase's band in registers (weights never come from shared memory):
//   - small O (1, 2, 3: 8/12/24/32/48 kHz -> 16 kHz): the R blocks' bands overlap in all but O samples, so the thread walks the
//     union of the R windows once ((R - 1) * O + KB shared-memory reads for R outputs) and feeds every sample to each output
//     whose band covers it (compile-time O makes every register index static);
//   - other O (22.05/44.1/88.2 kHz: O = 441): one shared-memory read per tap;
//   - bands wider than 64 taps: the weights are read from global memory (L1-resident) instead of registers.
// Tiles are spread over a persistent grid: every CTA walks the rows, takes the tiles whose running index is its own modulo the
// grid, so ragged rows of any length are balanced without a host-side plan.  The sum of every output runs t = 0, 1, ... in
// fp32 FMAs, independent of the tile and of the launch (ragged, uniform or per clip): those results are bit-identical.
#include "audiocalm_b200.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <numeric>
#include <string>
#include <vector>

namespace acb {
int fail(int code, const std::string& msg);   // acb_kernels.cu: sets the thread-local message behind acb_last_error()
}

namespace acb_rs {

using namespace acb;

constexpr int kThreads = 256;
constexpr int kMaxCoefficients = 32768;    // banded coefficients of one table
constexpr int kMaxBand = 512;              // taps of one phase's band
constexpr int kMaxRegBand = 64;            // widest band held in registers
constexpr int kSpanTarget = 16384;         // staged input samples per tile (64 KB), upper bound where a tile allows it
constexpr int kOutTarget = 8192;           // staged outputs per tile (32 KB)
constexpr int kWindowBlocks = 9;           // R of the small-O path (odd: conflict-free window reads for O = 1, 3)
constexpr int kTapBlocks = 4;              // R of the other paths (amortises the weight loads)

struct Params {
    const void* in;
    int in_dtype;                 // ACB_F32 | ACB_I16
    int vec_ok;                   // base pointer 16-byte aligned: vector staging loads allowed
    const long long* in_offset;
    const long long* in_length;
    long long in_stride, uniform_length;
    int n_rows;
    float* out;
    const long long* out_offset;
    long long out_stride;
    const float* w;               // [kb][N] tap-major, zero-padded beyond each band
    const int* start;             // [N] first tap of the band minus the smallest one
    const int* len;               // [N] band length
    int O, N, width, smin, kb, tb, span, span_alloc;
};

// torchaudio's output length: ceil(torch.as_tensor(N * L / O)) -- a Python float (fp64) rounded to fp32 before the ceil --
// capped by the conv1d length (L / O + 1) * N.
__host__ __device__ inline long long resampled_length(long long L, int O, int N) {
    if (L <= 0) return 0;
    const double q = (double)((long long)N * L) / (double)O;
    const long long c = (long long)ceilf((float)q);
    const long long conv = (L / O + 1) * (long long)N;
    return c < conv ? c : conv;
}

__device__ __forceinline__ float widen(float v) { return v; }
__device__ __forceinline__ float widen(short v) { return (float)v * (1.0f / 32768.0f); }

// xs[q] = x[lo + q] for q in [0, span), zero outside [0, L).  Vectors that lie wholly inside the clip are loaded with one 16-byte
// load; the rest element by element, so nothing outside the clip (a packed neighbour, or memory past the buffer) is read.
template <typename T>
__device__ __forceinline__ void stage(const T* __restrict__ in, long long off, long long L, long long lo, int span, int vec_ok, float* xs) {
    constexpr int V = 16 / sizeof(T);
    const long long a0 = (off + lo) & ~(long long)(V - 1);
    const long long nvec = (off + lo + span - a0 + V - 1) / V;
    for (long long v = threadIdx.x; v < nvec; v += kThreads) {
        const long long i = a0 + v * V - off;               // clip-relative index of the vector's first element
        float e[V];
        if (vec_ok && i >= 0 && i + V <= L) {
            const int4 raw = __ldg(reinterpret_cast<const int4*>(in + off + i));
            if constexpr (V == 4) {
                e[0] = __int_as_float(raw.x); e[1] = __int_as_float(raw.y); e[2] = __int_as_float(raw.z); e[3] = __int_as_float(raw.w);
            } else {
                const int u[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    e[2 * k] = widen((short)(u[k] & 0xffff));
                    e[2 * k + 1] = widen((short)(u[k] >> 16));
                }
            }
        } else {
#pragma unroll
            for (int k = 0; k < V; ++k) e[k] = (i + k >= 0 && i + k < L) ? widen(in[off + i + k]) : 0.f;
        }
#pragma unroll
        for (int k = 0; k < V; ++k) {
            const long long q = i + k - lo;
            if (q >= 0 && q < span) xs[q] = e[k];
        }
    }
}

// OC > 0: compile-time O, sliding window over R blocks; OC == 0: runtime O, one read per tap.  KB: register band (padded), or
// 0 for the wide-band path with weights from global memory.
template <int OC, int KB, int R>
__global__ void __launch_bounds__(kThreads, 2) resample_kernel(Params p) {
    extern __shared__ float smem[];
    float* xs = smem;
    float* os = smem + p.span_alloc;
    const int O = OC > 0 ? OC : p.O;
    const int N = p.N, TB = p.tb;
    const long long G = gridDim.x;
    const int n_items = N * (TB / R);
    long long prefix = 0;                                     // tiles of the rows before this one (running index)
    for (int row = 0; row < p.n_rows; ++row) {
        const long long L = p.in_length ? p.in_length[row] : p.uniform_length;
        const long long Lout = resampled_length(L, O, N);
        const long long tiles = ((Lout + N - 1) / N + TB - 1) / TB;
        long long t = ((long long)blockIdx.x - prefix) % G;
        if (t < 0) t += G;
        prefix += tiles;
        if (t >= tiles) continue;
        const long long in_off = p.in_offset ? p.in_offset[row] : row * p.in_stride;
        const long long out_off = p.out_offset ? p.out_offset[row] : row * p.out_stride;
        for (; t < tiles; t += G) {
            const long long b0 = t * TB;
            const long long lo = b0 * O + p.smin - p.width;
            if (p.in_dtype == ACB_I16)
                stage(static_cast<const short*>(p.in), in_off, L, lo, p.span, p.vec_ok, xs);
            else
                stage(static_cast<const float*>(p.in), in_off, L, lo, p.span, p.vec_ok, xs);
            __syncthreads();
            for (int k = threadIdx.x; k < n_items; k += kThreads) {
                const int j = k % N, c = k / N;
                const int s = __ldg(p.start + j);
                float acc[R];
#pragma unroll
                for (int r = 0; r < R; ++r) acc[r] = 0.f;
                if constexpr (KB > 0) {
                    float w[KB];
#pragma unroll
                    for (int i = 0; i < KB; ++i) w[i] = __ldg(p.w + i * N + j);
                    if constexpr (OC > 0) {
                        const float* xb = xs + c * R * OC + s;
#pragma unroll
                        for (int v = 0; v < (R - 1) * OC + KB; ++v) {
                            const float x = xb[v];
#pragma unroll
                            for (int r = 0; r < R; ++r) {
                                const int i = v - r * OC;
                                if (i >= 0 && i < KB) acc[r] = fmaf(w[i], x, acc[r]);
                            }
                        }
                    } else {
                        const int n = __ldg(p.len + j);
#pragma unroll
                        for (int r = 0; r < R; ++r) {
                            const float* xb = xs + (c * R + r) * O + s;
#pragma unroll
                            for (int i = 0; i < KB; ++i)
                                if (i < n) acc[r] = fmaf(w[i], xb[i], acc[r]);
                        }
                    }
                } else {
                    const int n = __ldg(p.len + j);
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        const float* xb = xs + (c * R + r) * O + s;
                        for (int i = 0; i < n; ++i) acc[r] = fmaf(__ldg(p.w + i * N + j), xb[i], acc[r]);
                    }
                }
#pragma unroll
                for (int r = 0; r < R; ++r) os[(c * R + r) * N + j] = acc[r];
            }
            __syncthreads();
            const long long first = b0 * N;
            const long long cnt = min((long long)TB * N, Lout - first);
            float* dst = p.out + out_off + first;
            for (long long e = threadIdx.x; e < cnt; e += kThreads) dst[e] = os[e];
            // the next tile's staging writes xs only, which nobody reads after the barrier above; its outputs go to os only
            // after its own staging barrier, which every thread reaches after this loop
        }
    }
}

using KernelFn = void (*)(Params);

struct Config {
    KernelFn fn;
    int oc, kb, r;
};

template <int OC, int R>
static bool pick_kb(int band, Config* c) {
    const int kbs[] = {16, 24, 32, 40, 64};
    const KernelFn fns[] = {resample_kernel<OC, 16, R>, resample_kernel<OC, 24, R>, resample_kernel<OC, 32, R>,
                            resample_kernel<OC, 40, R>, resample_kernel<OC, 64, R>};
    for (int i = 0; i < 5; ++i)
        if (band <= kbs[i]) {
            *c = Config{fns[i], OC, kbs[i], R};
            return true;
        }
    return false;
}

static Config choose(int O, int band) {
    Config c{};
    if (band <= kMaxRegBand) {
        if (O == 1 && pick_kb<1, kWindowBlocks>(band, &c)) return c;
        if (O == 2 && pick_kb<2, kWindowBlocks>(band, &c)) return c;
        if (O == 3 && pick_kb<3, kWindowBlocks>(band, &c)) return c;
        if (pick_kb<0, kTapBlocks>(band, &c)) return c;
    }
    return Config{resample_kernel<0, 0, kTapBlocks>, 0, 0, kTapBlocks};
}

}  // namespace acb_rs

using namespace acb_rs;

struct acb_resampler {
    int device = 0;
    int O = 0, N = 0, width = 0, smin = 0, kb = 0, band = 0, n_coef = 0;
    int tb = 0, span = 0, span_alloc = 0, smem_bytes = 0, grid = 0;
    Config cfg{};
    void* d_blob = nullptr;       // weights [kb][N], start [N], len [N]
    const float* d_w = nullptr;
    const int* d_start = nullptr;
    const int* d_len = nullptr;
};

extern "C" {

int64_t acb_resampled_length(int64_t length, int orig_freq, int new_freq) {
    if (length < 0 || orig_freq <= 0 || new_freq <= 0) return -1;
    if (orig_freq == new_freq) return length;
    const int g = std::gcd(orig_freq, new_freq);
    return resampled_length(length, orig_freq / g, new_freq / g);
}

int acb_resampler_create(acb_resampler** out, int device, int orig_freq, int new_freq, int width, const float* kernel_host) {
    if (!out || !kernel_host) return fail(ACB_ERR_INVALID, "acb_resampler_create: null argument");
    if (orig_freq <= 0 || new_freq <= 0 || width < 0) return fail(ACB_ERR_INVALID, "acb_resampler_create: rates must be positive and width >= 0");
    if (orig_freq == new_freq) return fail(ACB_ERR_INVALID, "acb_resampler_create: orig_freq == new_freq needs no resampler");
    const int g = std::gcd(orig_freq, new_freq);
    const int O = orig_freq / g, N = new_freq / g;
    const long long K = 2LL * width + O;
    if ((long long)N * K > (1LL << 28)) return fail(ACB_ERR_UNSUPPORTED, "acb_resampler_create: kernel table too large");
    // banded form: first .. last non-zero fp32 coefficient of each phase (zeros inside a band are kept)
    std::vector<int> st(N, 0), ln(N, 0);
    long long n_coef = 0;
    int band = 0;
    for (int j = 0; j < N; ++j) {
        long long lo = -1, hi = -1;
        for (long long k = 0; k < K; ++k)
            if (kernel_host[j * K + k] != 0.f) { if (lo < 0) lo = k; hi = k; }
        if (lo >= 0) { st[j] = (int)lo; ln[j] = (int)(hi - lo + 1); }
        n_coef += ln[j];
        band = std::max(band, ln[j]);
    }
    if (n_coef > kMaxCoefficients || band > kMaxBand)
        return fail(ACB_ERR_UNSUPPORTED, "acb_resampler_create: " + std::to_string(n_coef) + " banded coefficients with bands up to " +
                                             std::to_string(band) + " taps; this build handles at most " + std::to_string(kMaxCoefficients) +
                                             " coefficients and " + std::to_string(kMaxBand) + "-tap bands");
    int smin = INT32_MAX, smax = 0;
    for (int j = 0; j < N; ++j)
        if (ln[j]) { smin = std::min(smin, st[j]); smax = std::max(smax, st[j]); }
    if (smin == INT32_MAX) smin = 0;
    for (int j = 0; j < N; ++j) st[j] = ln[j] ? st[j] - smin : 0;
    const Config cfg = choose(O, band);
    const int kb = cfg.kb > 0 ? cfg.kb : std::max(band, 1);
    // tile: TB blocks (a multiple of R), as many chunks C = TB / R as the span and output targets allow, choosing the C that leaves
    // the fewest idle threads in the last pass over the tile's N * C items
    const int R = cfg.r;
    const long long extra = (long long)(smax - smin) + kb;
    const long long c_span = std::max<long long>(1, ((long long)kSpanTarget - extra) / ((long long)O * R));
    const long long c_out = std::max<long long>(1, (long long)kOutTarget / ((long long)N * R));
    const long long c_max = std::min(c_span, c_out);
    long long best_c = 1;
    double best_fill = 0.0;
    for (long long c = 1; c <= c_max; ++c) {
        const long long items = (long long)N * c;
        const double fill = (double)items / (double)(((items + kThreads - 1) / kThreads) * kThreads);
        if (fill >= best_fill) { best_fill = fill; best_c = c; }
    }
    const long long tb = best_c * R;
    const long long span = (tb - 1) * O + extra;
    const long long span_alloc = (span + 3) & ~3LL;
    const long long smem = (span_alloc + tb * N) * (long long)sizeof(float);

    int prev = 0;
    if (cudaGetDevice(&prev) != cudaSuccess) return fail(ACB_ERR_CUDA, "acb_resampler_create: cudaGetDevice failed");
    if (cudaSetDevice(device) != cudaSuccess) return fail(ACB_ERR_INVALID, "acb_resampler_create: bad device " + std::to_string(device));
    int optin = 0, sms = 0, occ = 0;
    cudaError_t e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    if (e != cudaSuccess) { cudaSetDevice(prev); return fail(ACB_ERR_CUDA, std::string("acb_resampler_create: ") + cudaGetErrorString(e)); }
    if (smem > optin) {
        cudaSetDevice(prev);
        return fail(ACB_ERR_UNSUPPORTED, "acb_resampler_create: a tile needs " + std::to_string(smem) + " bytes of shared memory (O = " +
                                             std::to_string(O) + ", N = " + std::to_string(N) + ")");
    }
    // the limit is per kernel and device, shared by every resampler that launches this instantiation: set it to the device maximum
    e = cudaFuncSetAttribute(cfg.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, optin);
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, cfg.fn, kThreads, (size_t)smem);
    auto* rs = new acb_resampler();
    const size_t w_bytes = (size_t)kb * N * sizeof(float), i_bytes = (size_t)N * sizeof(int);
    if (e == cudaSuccess) e = cudaMalloc(&rs->d_blob, w_bytes + 2 * i_bytes);
    if (e != cudaSuccess) {
        delete rs;
        cudaSetDevice(prev);
        return fail(ACB_ERR_CUDA, std::string("acb_resampler_create: ") + cudaGetErrorString(e));
    }
    std::vector<float> w((size_t)kb * N, 0.f);
    for (int j = 0; j < N; ++j)
        for (int t = 0; t < ln[j]; ++t) w[(size_t)t * N + j] = kernel_host[j * K + smin + st[j] + t];
    char* base = static_cast<char*>(rs->d_blob);
    e = cudaMemcpy(base, w.data(), w_bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(base + w_bytes, st.data(), i_bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(base + w_bytes + i_bytes, ln.data(), i_bytes, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) {
        cudaFree(rs->d_blob);
        delete rs;
        cudaSetDevice(prev);
        return fail(ACB_ERR_CUDA, std::string("acb_resampler_create: ") + cudaGetErrorString(e));
    }
    rs->device = device;
    rs->O = O; rs->N = N; rs->width = width; rs->smin = smin; rs->kb = kb; rs->band = band; rs->n_coef = (int)n_coef;
    rs->tb = (int)tb; rs->span = (int)span; rs->span_alloc = (int)span_alloc; rs->smem_bytes = (int)smem;
    rs->grid = std::max(1, sms) * std::max(1, occ);
    rs->cfg = cfg;
    rs->d_w = reinterpret_cast<const float*>(base);
    rs->d_start = reinterpret_cast<const int*>(base + w_bytes);
    rs->d_len = reinterpret_cast<const int*>(base + w_bytes + i_bytes);
    cudaSetDevice(prev);
    *out = rs;
    return ACB_OK;
}

int acb_resampler_destroy(acb_resampler* rs) {
    if (!rs) return ACB_OK;
    int prev = 0;
    cudaGetDevice(&prev);
    cudaSetDevice(rs->device);
    if (rs->d_blob) cudaFree(rs->d_blob);
    cudaSetDevice(prev);
    delete rs;
    return ACB_OK;
}

int acb_resample(const acb_resampler* rs, const void* in, int32_t in_dtype, const int64_t* in_offset, const int64_t* in_length,
                 int64_t in_stride, int64_t uniform_length, int32_t n_rows, float* out, const int64_t* out_offset,
                 int64_t out_stride, void* stream) {
    if (!rs) return fail(ACB_ERR_INVALID, "acb_resample: null resampler");
    if (n_rows < 0) return fail(ACB_ERR_INVALID, "acb_resample: negative row count");
    if (in_dtype != ACB_F32 && in_dtype != ACB_I16) return fail(ACB_ERR_INVALID, "acb_resample: in_dtype must be ACB_F32 or ACB_I16");
    if (!in_length && uniform_length < 0) return fail(ACB_ERR_INVALID, "acb_resample: negative uniform_length");
    if ((!in_offset && in_stride < 0) || (!out_offset && out_stride < 0)) return fail(ACB_ERR_INVALID, "acb_resample: negative stride");
    if (n_rows == 0) return ACB_OK;
    if (!in || !out) return fail(ACB_ERR_INVALID, "acb_resample: null buffer");
    Params p{};
    p.in = in;
    p.in_dtype = in_dtype;
    p.vec_ok = (reinterpret_cast<uintptr_t>(in) & 15) == 0;
    p.in_offset = reinterpret_cast<const long long*>(in_offset);
    p.in_length = reinterpret_cast<const long long*>(in_length);
    p.in_stride = in_stride;
    p.uniform_length = uniform_length;
    p.n_rows = n_rows;
    p.out = out;
    p.out_offset = reinterpret_cast<const long long*>(out_offset);
    p.out_stride = out_stride;
    p.w = rs->d_w;
    p.start = rs->d_start;
    p.len = rs->d_len;
    p.O = rs->O; p.N = rs->N; p.width = rs->width; p.smin = rs->smin; p.kb = rs->kb;
    p.tb = rs->tb; p.span = rs->span; p.span_alloc = rs->span_alloc;
    long long grid = rs->grid;
    if (!in_length) {                                          // uniform rows: no more CTAs than tiles
        const long long lout = resampled_length(uniform_length, rs->O, rs->N);
        const long long tiles = ((lout + rs->N - 1) / rs->N + rs->tb - 1) / rs->tb;
        grid = std::max(1LL, std::min(grid, tiles * n_rows));
    }
    int prev = 0;
    cudaGetDevice(&prev);
    if (prev != rs->device) cudaSetDevice(rs->device);
    rs->cfg.fn<<<(unsigned)grid, kThreads, (size_t)rs->smem_bytes, static_cast<cudaStream_t>(stream)>>>(p);
    const cudaError_t e = cudaGetLastError();
    if (prev != rs->device) cudaSetDevice(prev);
    if (e != cudaSuccess) return fail(ACB_ERR_CUDA, std::string("acb_resample launch: ") + cudaGetErrorString(e));
    return ACB_OK;
}

}  // extern "C"
