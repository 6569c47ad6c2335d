// In-register complex FFT-32 on packed fp32 (FFMA2 / FADD2, sm_100): the building block shared by the fused log-mel kernels
// (acb_kernels.cu, acb_logmel_stft.cu) and the VAE-side spectral kernels (acb_spectral.cu).
#pragma once
#include <cuda_runtime.h>

namespace acb {

__host__ __device__ constexpr int brev5(int x) {
    return ((x & 1) << 4) | ((x & 2) << 2) | (x & 4) | ((x & 8) >> 2) | ((x & 16) >> 4);
}

// cos/sin of 2*pi*j/32, j = 0..15
__device__ constexpr float kCos32[16] = {1.f, 0.98078528040323043f, 0.92387953251128674f, 0.83146961230254524f,
                                         0.70710678118654757f, 0.55557023301960229f, 0.38268343236508984f, 0.19509032201612833f,
                                         0.f, -0.19509032201612819f, -0.38268343236508973f, -0.55557023301960196f,
                                         -0.70710678118654746f, -0.83146961230254535f, -0.92387953251128674f, -0.98078528040323043f};
__device__ constexpr float kSin32[16] = {0.f, 0.19509032201612825f, 0.38268343236508978f, 0.55557023301960218f,
                                         0.70710678118654746f, 0.83146961230254524f, 0.92387953251128674f, 0.98078528040323043f,
                                         1.f, 0.98078528040323043f, 0.92387953251128674f, 0.83146961230254546f,
                                         0.70710678118654757f, 0.55557023301960218f, 0.38268343236508989f, 0.19509032201612861f};

// One radix-2 DIT butterfly with twiddle W = exp(-2*pi*i*TW/32): (u, v) -> (u + W v, u - W v).
// Generic twiddles use the 6-FMA form (sum by 4 FMAs, difference as 2u - sum).
template <int TW>
__device__ __forceinline__ void bfly(float& ur, float& ui, float& vr, float& vi) {
    if (TW == 0) {
        const float sr = ur + vr, si = ui + vi;
        vr = ur - vr; vi = ui - vi;
        ur = sr; ui = si;
    } else if (TW == 8) {  // W = -i : W v = (vi, -vr)
        const float sr = ur + vi, si = ui - vr;
        const float dr = ur - vi, di = ui + vr;
        ur = sr; ui = si; vr = dr; vi = di;
    } else {
        constexpr float wr = kCos32[TW];
        constexpr float wi = -kSin32[TW];
        const float sr = fmaf(wr, vr, fmaf(-wi, vi, ur));
        const float si = fmaf(wr, vi, fmaf(wi, vr, ui));
        vr = fmaf(2.f, ur, -sr);
        vi = fmaf(2.f, ui, -si);
        ur = sr; ui = si;
    }
}

// ---- packed fp32 (FFMA2 / FADD2 / FMUL2, new on sm_100): two butterflies per instruction ----
// The 32 complex values of an FFT-32 are held as 16 pairs (x[i], x[i + 16]) in 64-bit registers, real and imaginary parts
// in separate arrays.  Stages 1-4 of the radix-2 DIT network combine indices i and i + half with both below 16 or both above,
// and the twin butterfly 16 places up uses the same twiddle: one packed butterfly does both.  Stage 5 pairs i with i + 16,
// i.e. the two halves of one register pair, and runs as scalar code on the halves.
__device__ __forceinline__ float2 bcast2(float a) { return make_float2(a, a); }
__device__ __forceinline__ float2 neg2(float2 a) { return make_float2(-a.x, -a.y); }   // folds into the consumer's operand modifier

template <int TW>
__device__ __forceinline__ void bfly2(float2& ur, float2& ui, float2& vr, float2& vi) {
    if (TW == 0) {            // W = 1
        const float2 sr = __fadd2_rn(ur, vr), si = __fadd2_rn(ui, vi);
        vr = __fadd2_rn(ur, neg2(vr));
        vi = __fadd2_rn(ui, neg2(vi));
        ur = sr; ui = si;
    } else if (TW == 8) {     // W = -i : W v = (vi, -vr)
        const float2 sr = __fadd2_rn(ur, vi), si = __fadd2_rn(ui, neg2(vr));
        const float2 dr = __fadd2_rn(ur, neg2(vi)), di = __fadd2_rn(ui, vr);
        ur = sr; ui = si; vr = dr; vi = di;
    } else {                  // generic: s = u + W v by 4 packed FMAs, d = 2u - s by 2 more (6 for two butterflies)
        constexpr float wr = kCos32[TW];
        constexpr float wi = -kSin32[TW];
        const float2 sr = __ffma2_rn(vi, bcast2(-wi), __ffma2_rn(vr, bcast2(wr), ur));
        const float2 si = __ffma2_rn(vr, bcast2(wi), __ffma2_rn(vi, bcast2(wr), ui));
        vr = __ffma2_rn(ur, bcast2(2.f), neg2(sr));
        vi = __ffma2_rn(ui, bcast2(2.f), neg2(si));
        ur = sr; ui = si;
    }
}

template <int S, int K, int J>
struct Bfly2Loop {
    // packed stage S <= 4 (m = 2^S), group base K < 16, index J within the half-group
    static __device__ __forceinline__ void run(float2 (&pr)[16], float2 (&pi)[16]) {
        constexpr int m = 1 << S, half = m >> 1;
        bfly2<J * (32 / m)>(pr[K + J], pi[K + J], pr[K + J + half], pi[K + J + half]);
        if constexpr (J + 1 < half) {
            Bfly2Loop<S, K, J + 1>::run(pr, pi);
        } else if constexpr (K + m < 16) {
            Bfly2Loop<S, K + m, 0>::run(pr, pi);
        }
    }
};

template <int J>
struct LastStageLoop {
    // stage 5: butterfly (J, J + 16) = the two halves of pair J, twiddle W32^J, scalar code
    static __device__ __forceinline__ void run(float2 (&pr)[16], float2 (&pi)[16]) {
        bfly<J>(pr[J].x, pi[J].x, pr[J].y, pi[J].y);
        if constexpr (J + 1 < 16) LastStageLoop<J + 1>::run(pr, pi);
    }
};

// In-register complex FFT-32, decimation in time: input in bit-reversed order, output natural order
// (element k < 16 is pr[k].x, element k >= 16 is pr[k - 16].y).
__device__ __forceinline__ void fft32_packed(float2 (&pr)[16], float2 (&pi)[16]) {
    Bfly2Loop<1, 0, 0>::run(pr, pi);
    Bfly2Loop<2, 0, 0>::run(pr, pi);
    Bfly2Loop<3, 0, 0>::run(pr, pi);
    Bfly2Loop<4, 0, 0>::run(pr, pi);
    LastStageLoop<0>::run(pr, pi);
}

// Same, when stage 1 (span-1 butterflies, twiddle 1) has already been applied by the caller.
__device__ __forceinline__ void fft32_packed_from_stage2(float2 (&pr)[16], float2 (&pi)[16]) {
    Bfly2Loop<2, 0, 0>::run(pr, pi);
    Bfly2Loop<3, 0, 0>::run(pr, pi);
    Bfly2Loop<4, 0, 0>::run(pr, pi);
    LastStageLoop<0>::run(pr, pi);
}

__host__ __device__ constexpr int brev3(int x) { return ((x & 1) << 2) | (x & 2) | ((x & 4) >> 2); }

// ---- the group FFT: a complex FFT of N = 32 R points (R a power of two <= 32) on R lanes, each lane running the in-register
// FFT-32 above over its stride-R samples; shared by the spectral kernels (acb_spectral.cu) and the general log-mel kernel
// (acb_logmel_stft.cu) ----
__host__ __device__ constexpr int brev_bits(int x, int bits) {
    int r = 0;
    for (int i = 0; i < bits; ++i) r |= ((x >> i) & 1) << (bits - 1 - i);
    return r;
}
__host__ __device__ constexpr int ilog2(int x) { return x <= 1 ? 0 : 1 + ilog2(x >> 1); }

// In-register complex FFT of R points (R a power of two <= 32), natural order in and out: the cross-lane factor of the transform.
template <int R>
__device__ __forceinline__ void small_fft(float2 (&v)[R]) {
    constexpr int kLog = ilog2(R);
#pragma unroll
    for (int i = 0; i < R; ++i) {
        const int j = brev_bits(i, kLog);
        if (i < j) { const float2 t = v[i]; v[i] = v[j]; v[j] = t; }
    }
#pragma unroll
    for (int half = 1; half < R; half <<= 1) {
#pragma unroll
        for (int base = 0; base < R; base += 2 * half) {
#pragma unroll
            for (int j = 0; j < half; ++j) {
                const int tw = j * (16 / half);                       // W_(2 half)^j = W_32^tw, tw < 16
                const float wr = kCos32[tw], wi = -kSin32[tw];
                const float2 u = v[base + j], w = v[base + j + half];
                const float tr = fmaf(wr, w.x, -wi * w.y), ti = fmaf(wr, w.y, wi * w.x);
                v[base + j] = make_float2(u.x + tr, u.y + ti);
                v[base + j + half] = make_float2(u.x - tr, u.y - ti);
            }
        }
    }
}

// The complex FFT of N = 32 R points that a group of R lanes computes together.  Stage 1: the lane's 32 stride-R inputs (packed,
// bit-reversed order: see fft32_packed) -> in-register FFT-32, twiddle W_N^(r k1), hand-over to the group's exchange buffer at index
// k1 + 33 r.  Stage 2 (after a __syncwarp): an R-point FFT across the group's lanes, in place; Z[k1 + 32 k2] ends up at index k1 + 33 k2.
template <int R>
__device__ __forceinline__ void group_fft_stage1(float2 (&pr)[16], float2 (&pi)[16], float2* buf, const float2* s_tw, int r) {
    fft32_packed(pr, pi);
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        const float2 t0 = s_tw[k * R + r], t1 = s_tw[(k + 16) * R + r];     // table laid out [k][r]: a group's lanes read consecutive entries
        buf[k + 33 * r] = make_float2(fmaf(pr[k].x, t0.x, -pi[k].x * t0.y), fmaf(pr[k].x, t0.y, pi[k].x * t0.x));
        buf[k + 16 + 33 * r] = make_float2(fmaf(pr[k].y, t1.x, -pi[k].y * t1.y), fmaf(pr[k].y, t1.y, pi[k].y * t1.x));
    }
}
template <int R>
__device__ __forceinline__ void group_fft_stage2(float2* buf, int r) {
    constexpr int kPerLane = 32 / R;
#pragma unroll
    for (int t = 0; t < kPerLane; ++t) {
        const int k1 = r + R * t;             // interleaved over the lanes: the group's lanes touch consecutive 8-byte slots (a blocked r * kPerLane + t
                                              // put the 32 lanes of a warp on 4 of the 16 bank pairs)
        float2 v[R];
#pragma unroll
        for (int rr = 0; rr < R; ++rr) v[rr] = buf[k1 + 33 * rr];
        small_fft<R>(v);
#pragma unroll
        for (int rr = 0; rr < R; ++rr) buf[k1 + 33 * rr] = v[rr];
    }
}
__device__ __forceinline__ int buf_index(int k) { return (k & 31) + 33 * (k >> 5); }

}  // namespace acb
