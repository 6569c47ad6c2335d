// FLAC (RFC 9639) decoding on the device: many independent streams in one call, bit-exact.
//
// A clip is the audio-frame region of one FLAC stream (the bytes after its metadata blocks) plus the STREAMINFO fields the host
// parsed.  Three launches:
//   1. locate  (one CTA per clip): every byte position p of the region is tested for the frame sync (0xFFF8 / 0xFFF9); a sync is
//      parsed as a frame header (RFC 9639 9.1: block-size codes with the 8- and 16-bit uncommon forms, sample-rate codes with the
//      uncommon forms, channel assignments 0-10, bit-depth code, the UTF-8-style coded number of up to 7 bytes) and kept only
//      when its CRC-8 matches and its fields agree with STREAMINFO and the clip's length.  A thread tests 32 consecutive positions,
//      and a block-wide scan of the hit counts compacts the survivors into the clip's candidate list in byte order.
//   2. decode  (one thread per candidate, persistent grid): the frame is parsed twice.  Pass A reads every subframe (CONSTANT,
//      VERBATIM, FIXED 0-4, LPC 1-32, wasted bits, residual methods 0 and 1 with partition orders 0-15 and escaped partitions)
//      without predicting, records where each subframe starts, skips the byte-alignment padding and checks the frame's CRC-16.
//      Only a frame that passes is decoded again (pass B) and written: independent channels one after the other, the stereo modes
//      (left/side, side/right, mid/side; the side channel has bps + 1 bits) with both subframes decoded in lock step.  A false
//      sync inside residual data has to pass its CRC-8 and then the CRC-16 of a decode that starts from it, and even then the
//      coverage check below rejects the clip.
//   3. verify  (one thread per clip): the accepted frames, in byte order, must start at byte 0, follow each other with no gap in
//      bytes or samples, and end at sample total_samples.  Otherwise the clip's status is ACB_FLAC_NOT_TILED; other clips keep
//      their bits.
// Every read goes through a bit reader bounded by the clip's own region: a truncated or corrupt stream is a status, never a read
// outside the region.  LPC sums run in 64 bits when precision + bps + log2(order) can exceed 32 bits.  The STREAMINFO MD5 is not
// checked (it is sequential over the whole stream); the per-frame CRC-16 is.
#include "audiocalm_b200.h"

#include <cuda_runtime.h>

#include <cstdint>
#include <string>

namespace acb {
int fail(int code, const std::string& msg);   // acb_kernels.cu: sets the thread-local message behind acb_last_error()
}

namespace acb_fl {

using namespace acb;

constexpr int kLocateThreads = 256;
constexpr int kRun = 32;                 // consecutive positions one locate thread tests per sweep (one bit of a hit mask each)
constexpr int kDecodeThreads = 128;
constexpr int kMaxOrder = 32;

struct Cand {                            // one candidate frame, in byte order within its clip
    int start;                           // region-relative byte of the sync
    int end;                             // byte after the CRC-16 of an accepted frame; -1: rejected
    int bs;
    int pad;
    long long pos;                       // first sample
};

static_assert(sizeof(acb_flac_clip) == 72, "acb_flac_clip layout");

__host__ __device__ inline long long candidate_capacity(long long bytes) { return bytes / 8 + 16; }

__device__ __forceinline__ bool clip_ok(const acb_flac_clip& c) {
    return c.byte_length >= 0 && c.byte_length < (1LL << 31) && c.channels >= 1 && c.channels <= 8 && c.bps >= 4 && c.bps <= 24 &&
           c.max_block >= 1 && c.max_block <= 65536 && c.total_samples >= 0 && (c.variable == 0 || c.variable == 1);
}

__device__ void crc_tables(unsigned char* t8, unsigned short* t16) {
    for (int b = threadIdx.x; b < 256; b += blockDim.x) {
        unsigned c8 = b, c16 = (unsigned)b << 8;
        for (int i = 0; i < 8; ++i) {
            c8 = (c8 & 0x80) ? ((c8 << 1) ^ 0x07) & 0xFF : (c8 << 1) & 0xFF;
            c16 = (c16 & 0x8000) ? ((c16 << 1) ^ 0x8005) & 0xFFFF : (c16 << 1) & 0xFFFF;
        }
        t8[b] = (unsigned char)c8;
        t16[b] = (unsigned short)c16;
    }
}

struct Header {
    int bs, assignment, size;
    long long pos;
};

// The frame header at region byte p (RFC 9639 9.1), checked against STREAMINFO.  Reads only [p, min(p + 16, len)).
__device__ __forceinline__ bool parse_header(const unsigned char* __restrict__ d, long long len, long long p, const acb_flac_clip& c,
                             const unsigned char* t8, Header* h) {
    if (p + 6 > len) return false;
    // the (at most 16) header bytes in two big-endian words: every byte access below is a shift, no local memory
    const int n = (int)min(16LL, len - p);
    unsigned long long w0 = 0, w1 = 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        const unsigned long long v = i < n ? __ldg(d + p + i) : 0;
        if (i < 8) w0 |= v << (56 - 8 * i); else w1 |= v << (56 - 8 * (i - 8));
    }
    auto b = [&](int i) -> unsigned { return (unsigned)((i < 8 ? w0 >> (56 - 8 * i) : w1 >> (56 - 8 * (i - 8))) & 0xFF); };
    if (b(0) != 0xFF || (b(1) & 0xFE) != 0xF8 || (int)(b(1) & 1) != c.variable) return false;
    const int bs_code = b(2) >> 4, sr_code = b(2) & 15, asg = b(3) >> 4, bps_code = (b(3) >> 1) & 7;
    if (bs_code == 0 || sr_code == 15 || asg > 10 || bps_code == 3 || (b(3) & 1)) return false;
    int q = 4;
    const unsigned lead = b(4);
    int extra;
    unsigned long long num;
    if (lead < 0x80) {
        extra = 0; num = lead;
    } else if (lead == 0xFE) {
        extra = 6; num = 0;
    } else if (lead >= 0xC0 && lead < 0xFE) {
        extra = __clz(~(lead << 24)) - 1;                 // leading ones of the lead byte, minus one
        num = lead & (0x3Fu >> extra);
    } else {
        return false;
    }
    if (q + 1 + extra > n) return false;
    for (int i = 0; i < extra; ++i) {
        const unsigned x = b(q + 1 + i);
        if ((x & 0xC0) != 0x80) return false;
        num = (num << 6) | (x & 0x3F);
    }
    q += 1 + extra;
    int bs;
    if (bs_code == 6 || bs_code == 7) {
        if (q + bs_code - 5 > n) return false;
        bs = (int)(bs_code == 6 ? b(q) : (b(q) << 8 | b(q + 1))) + 1;
        q += bs_code - 5;
    } else if (bs_code == 1) {
        bs = 192;
    } else if (bs_code <= 5) {
        bs = 576 << (bs_code - 2);
    } else {
        bs = 256 << (bs_code - 8);
    }
    int sr = 0;
    if (sr_code >= 12) {
        const int k = sr_code == 12 ? 1 : 2;
        if (q + k > n) return false;
        const int v = (int)(k == 1 ? b(q) : (b(q) << 8 | b(q + 1)));
        sr = sr_code == 12 ? v * 1000 : (sr_code == 13 ? v : v * 10);
        q += k;
    } else if (sr_code > 0) {
        sr = sr_code == 1 ? 88200 : sr_code == 2 ? 176400 : sr_code == 3 ? 192000 : sr_code == 4 ? 8000 : sr_code == 5 ? 16000
           : sr_code == 6 ? 22050 : sr_code == 7 ? 24000 : sr_code == 8 ? 32000 : sr_code == 9 ? 44100 : sr_code == 10 ? 48000 : 96000;
    }
    if (q >= n) return false;
    unsigned crc = 0;
    for (int i = 0; i < q; ++i) crc = t8[crc ^ b(i)];
    if (crc != b(q)) return false;
    const int bps_of_code = bps_code == 1 ? 8 : bps_code == 2 ? 12 : bps_code == 4 ? 16 : bps_code == 5 ? 20 : bps_code == 6 ? 24 : 32;
    if ((asg < 8 ? asg + 1 : 2) != c.channels) return false;
    if (bps_code && bps_of_code != c.bps) return false;
    if (sr_code && sr != c.sample_rate) return false;
    if (bs > c.max_block) return false;
    if (!c.variable && num >= (1ULL << 31)) return false;
    const long long pos = c.variable ? (long long)num : (long long)num * c.max_block;
    if (pos + bs > c.total_samples) return false;
    h->bs = bs; h->assignment = asg; h->size = q + 1; h->pos = pos;
    return true;
}

// MSB-first bit reader over one clip's region [0, len): reading past len sets `bad` and returns zeros.
struct BitReader {
    const unsigned char* d;
    long long len, byte;                 // next byte to load
    unsigned long long cache;            // valid bits left-aligned, zeros below them
    int nb;
    bool bad;

    __device__ __forceinline__ void init(const unsigned char* data, long long n, long long bit) {
        d = data; len = n; byte = bit >> 3; cache = 0; nb = 0; bad = false;
        refill();
        const int skip = (int)(bit & 7);
        if (nb < skip) { bad = true; return; }
        cache <<= skip;
        nb -= skip;
    }
    __device__ __forceinline__ void refill() {
        while (nb <= 56 && byte < len) {
            cache |= (unsigned long long)__ldg(d + byte++) << (56 - nb);
            nb += 8;
        }
    }
    __device__ __forceinline__ unsigned read(int n) {        // n <= 32
        if (n == 0) return 0;
        if (nb < n) {
            refill();
            if (nb < n) { bad = true; return 0; }
        }
        const unsigned v = (unsigned)(cache >> (64 - n));
        cache = n == 64 ? 0 : cache << n;
        nb -= n;
        return v;
    }
    __device__ __forceinline__ int sread(int n) { return n ? (int)(read(n) << (32 - n)) >> (32 - n) : 0; }
    __device__ __forceinline__ unsigned unary() {
        unsigned q = 0;
        for (;;) {
            if (nb == 0) {
                refill();
                if (nb == 0) { bad = true; return 0; }
            }
            const int z = cache ? __clzll((long long)cache) : 64;
            if (z < nb) {
                cache = z == 63 ? 0 : cache << (z + 1);
                nb -= z + 1;
                return q + z;
            }
            q += nb;
            cache = 0;
            nb = 0;
            if (q > (1u << 31)) { bad = true; return 0; }
        }
    }
    __device__ __forceinline__ long long bitpos() const { return byte * 8 - nb; }
};

// One subframe (RFC 9639 9.2) producing its samples one at a time.  Predict = false only walks the bits (pass A).
struct Subframe {
    BitReader br;
    int kind;                            // 0 CONSTANT, 1 VERBATIM, 2 FIXED / LPC
    int bps, wasted, order, shift, bs, i;
    bool wide;
    int cval;
    int pbits, esc, po, part, left, k, raw;    // residual state; raw >= 0: escaped partition of `raw`-bit samples
    int coef[kMaxOrder];
    int hist[kMaxOrder];

    __device__ __forceinline__ void start_partition() {
        left = (bs >> po) - (part == 0 ? order : 0);
        k = (int)br.read(pbits);
        raw = -1;
        if (k == esc) raw = (int)br.read(5);
    }

    __device__ __forceinline__ bool init(const unsigned char* d, long long len, long long bit, int block, int sbps) {
        br.init(d, len, bit);
        bs = block; i = 0; order = 0; shift = 0; wide = false;
        if (br.read(1)) return false;
        const int type = (int)br.read(6);
        wasted = 0;
        if (br.read(1)) wasted = (int)br.unary() + 1;
        if (br.bad || wasted >= sbps) return false;
        bps = sbps - wasted;
        if (type == 0) { kind = 0; cval = br.sread(bps); return !br.bad; }
        if (type == 1) { kind = 1; return !br.bad; }
        kind = 2;
        if (type >= 8 && type <= 12) {
            order = type - 8;
            const int fixed[5][4] = {{0, 0, 0, 0}, {1, 0, 0, 0}, {2, -1, 0, 0}, {3, -3, 1, 0}, {4, -6, 4, -1}};
            for (int j = 0; j < order; ++j) coef[j] = fixed[order][j];
        } else if (type >= 32) {
            order = type - 31;
        } else {
            return false;                                      // reserved subframe type
        }
        if (order > bs) return false;
        for (int j = 0; j < order; ++j) hist[j] = br.sread(bps);
        if (type >= 32) {
            const int prec = (int)br.read(4) + 1;
            if (prec == 16) return false;
            shift = br.sread(5);
            if (shift < 0) return false;                       // RFC 9639 9.2.6: a negative shift is invalid
            for (int j = 0; j < order; ++j) coef[j] = br.sread(prec);
            wide = prec + bps + (32 - __clz(order)) > 32;
        }
        const unsigned method = br.read(2);
        if (method > 1) return false;
        pbits = method ? 5 : 4;
        esc = method ? 31 : 15;
        po = (int)br.read(4);
        if ((bs & ((1 << po) - 1)) || (bs >> po) < order) return false;
        part = 0;
        start_partition();
        return !br.bad;
    }

    template <bool Predict>
    __device__ __forceinline__ int next() {
        int v;
        if (kind == 0) {
            v = cval;
        } else if (kind == 1) {
            v = br.sread(bps);
        } else if (i < order) {
            v = hist[i];
        } else {
            while (left == 0) {
                if (++part >= (1 << po)) { br.bad = true; break; }
                start_partition();
            }
            int r;
            if (raw >= 0) {
                r = br.sread(raw);
            } else {
                const unsigned q = br.unary();
                const unsigned long long u = ((unsigned long long)q << k) | br.read(k);
                if (u >> 32) br.bad = true;
                r = (int)(unsigned)(u >> 1) ^ -(int)(u & 1);
            }
            --left;
            if (Predict) {
                if (wide) {
                    long long s = 0;
                    for (int j = 0; j < order; ++j) s += (long long)coef[j] * hist[(i - 1 - j) & (kMaxOrder - 1)];
                    v = r + (int)(s >> shift);
                } else {
                    int s = 0;
                    for (int j = 0; j < order; ++j) s += coef[j] * hist[(i - 1 - j) & (kMaxOrder - 1)];
                    v = r + (s >> shift);
                }
                hist[i & (kMaxOrder - 1)] = v;
            } else {
                v = r;
            }
        }
        ++i;
        return (int)((unsigned)v << wasted);
    }
};

__device__ __forceinline__ bool is_side(int asg, int ch) { return (asg == 8 && ch == 1) || (asg == 9 && ch == 0) || (asg == 10 && ch == 1); }

__global__ void __launch_bounds__(kLocateThreads) flac_locate_kernel(const unsigned char* __restrict__ data, const acb_flac_clip* clips,
                                                                      Cand* cands, int* counts) {
    __shared__ unsigned char t8[256];
    __shared__ unsigned short t16[256];
    __shared__ int warp_sum[kLocateThreads / 32];
    crc_tables(t8, t16);
    const acb_flac_clip c = clips[blockIdx.x];
    if (!clip_ok(c)) {
        if (threadIdx.x == 0) counts[blockIdx.x] = -1;
        return;
    }
    __syncthreads();
    const unsigned char* d = data + c.byte_offset;
    const long long len = c.byte_length, cap = candidate_capacity(len);
    Cand* out = cands + c.cand_offset;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long base = 0;
    for (long long chunk = 0; chunk < len; chunk += (long long)kLocateThreads * kRun) {
        const long long p0 = chunk + (long long)threadIdx.x * kRun;
        unsigned mask = 0;
        for (int j = 0; j < kRun; ++j) {
            const long long p = p0 + j;
            if (p + 1 < len && __ldg(d + p) == 0xFF && (__ldg(d + p + 1) & 0xFE) == 0xF8) {
                Header h;
                if (parse_header(d, len, p, c, t8, &h)) mask |= 1u << j;
            }
        }
        const int cnt = __popc(mask);
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) warp_sum[warp] = incl;
        __syncthreads();
        int wbase = 0, total = 0;
#pragma unroll
        for (int w = 0; w < kLocateThreads / 32; ++w) {
            const int s = warp_sum[w];
            wbase += w < warp ? s : 0;
            total += s;
        }
        long long idx = base + wbase + incl - cnt;
        while (mask) {
            const int j = __ffs(mask) - 1;
            mask &= mask - 1;
            if (idx < cap) out[idx] = Cand{(int)(p0 + j), -1, 0, 0, 0};
            ++idx;
        }
        base += total;
        __syncthreads();                                       // warp_sum is rewritten by the next sweep
    }
    if (threadIdx.x == 0) counts[blockIdx.x] = (int)min(base, cap + 1);   // cap + 1: the list overflowed
}

template <typename T>
__device__ __forceinline__ void store(void* out, long long idx, int v, float scale);
template <>
__device__ __forceinline__ void store<short>(void* out, long long idx, int v, float) { static_cast<short*>(out)[idx] = (short)v; }
template <>
__device__ __forceinline__ void store<float>(void* out, long long idx, int v, float scale) { static_cast<float*>(out)[idx] = (float)v * scale; }

template <typename T>
__device__ __forceinline__ void decode_frame(const unsigned char* __restrict__ d, const acb_flac_clip& c, Cand* cand, const unsigned char* t8,
                             const unsigned short* t16, void* out) {
    const long long len = c.byte_length;
    Header h;
    if (!parse_header(d, len, cand->start, c, t8, &h)) return;
    const int bs = h.bs, asg = h.assignment;
    long long sub_bit[8];
    long long bit = (cand->start + (long long)h.size) * 8;
    Subframe sf[2];                                            // pass A and independent channels use sf[0]; stereo both
    // pass A: walk every subframe, find the frame's end, check its CRC-16
    for (int ch = 0; ch < c.channels; ++ch) {
        sub_bit[ch] = bit;
        Subframe& s = sf[0];
        if (!s.init(d, len, bit, bs, c.bps + is_side(asg, ch))) return;
        for (int n = 0; n < bs; ++n) s.next<false>();
        if (s.br.bad) return;
        bit = s.br.bitpos();
    }
    const long long end = (bit + 7) >> 3;
    if (end + 2 > len) return;
    unsigned crc = 0;
    for (long long p = cand->start; p < end + 2; ++p) crc = ((crc << 8) & 0xFFFF) ^ t16[(crc >> 8) ^ __ldg(d + p)];
    if (crc != 0) return;                                      // CRC-16 over the frame and its own CRC is zero
    // pass B: decode and write
    const float scale = 1.0f / (float)(1 << (c.bps - 1));
    const long long o = c.out_offset + h.pos;
    if (asg < 8) {
        for (int ch = 0; ch < c.channels; ++ch) {
            Subframe& s = sf[0];
            s.init(d, len, sub_bit[ch], bs, c.bps);
            const long long row = o + ch * c.out_stride;
            for (int n = 0; n < bs; ++n) store<T>(out, row + n, s.next<true>(), scale);
        }
    } else {
        Subframe &a = sf[0], &b = sf[1];
        a.init(d, len, sub_bit[0], bs, c.bps + is_side(asg, 0));
        b.init(d, len, sub_bit[1], bs, c.bps + is_side(asg, 1));
        for (int n = 0; n < bs; ++n) {
            const int x = a.next<true>(), y = b.next<true>();
            int l, r;
            if (asg == 8) {
                l = x; r = x - y;
            } else if (asg == 9) {
                l = x + y; r = y;
            } else {
                const int m = (int)((unsigned)x << 1) | (y & 1);
                l = (m + y) >> 1; r = (m - y) >> 1;
            }
            store<T>(out, o + n, l, scale);
            store<T>(out, o + c.out_stride + n, r, scale);
        }
    }
    cand->end = (int)(end + 2);
    cand->bs = bs;
    cand->pos = h.pos;
}

template <typename T>
__global__ void __launch_bounds__(kDecodeThreads, 4) flac_decode_kernel(const unsigned char* __restrict__ data, const acb_flac_clip* clips,
                                                                     int n_clips, Cand* cands, const int* counts, void* out) {
    __shared__ unsigned char t8[256];
    __shared__ unsigned short t16[256];
    crc_tables(t8, t16);
    __syncthreads();
    const long long G = (long long)gridDim.x * blockDim.x, tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    long long prefix = 0;                                      // candidates of the clips before this one (running index)
    for (int ci = 0; ci < n_clips; ++ci) {
        int n = counts[ci];
        if (n <= 0) continue;
        const long long cap = candidate_capacity(clips[ci].byte_length);
        if (n > cap) continue;                                 // overflowed list: verify reports it
        long long k = (tid - prefix) % G;
        if (k < 0) k += G;
        prefix += n;
        if (k >= n) continue;
        const acb_flac_clip c = clips[ci];
        const unsigned char* d = data + c.byte_offset;
        for (; k < n; k += G) decode_frame<T>(d, c, cands + c.cand_offset + k, t8, t16, out);
    }
}

__global__ void flac_verify_kernel(const acb_flac_clip* clips, int n_clips, const Cand* cands, const int* counts, int* status) {
    const int ci = blockIdx.x * blockDim.x + threadIdx.x;
    if (ci >= n_clips) return;
    const acb_flac_clip c = clips[ci];
    const int n = counts[ci];
    if (n < 0) { status[ci] = ACB_FLAC_BAD_CLIP; return; }
    if (n > candidate_capacity(c.byte_length)) { status[ci] = ACB_FLAC_TOO_MANY_CANDIDATES; return; }
    long long eb = 0, es = 0;
    int st = ACB_FLAC_OK;
    for (int k = 0; k < n; ++k) {
        const Cand x = cands[c.cand_offset + k];
        if (x.end < 0) continue;                               // a false sync or a frame that failed its CRC-16
        if (x.start != eb || x.pos != es) { st = ACB_FLAC_NOT_TILED; break; }
        eb = x.end;
        es += x.bs;
    }
    if (st == ACB_FLAC_OK && es != c.total_samples) st = ACB_FLAC_NOT_TILED;
    status[ci] = st;
}

}  // namespace acb_fl

using namespace acb_fl;

extern "C" {

int64_t acb_flac_candidate_capacity(int64_t byte_length) { return byte_length < 0 ? -1 : candidate_capacity(byte_length); }

int64_t acb_flac_workspace_bytes(int64_t total_candidates, int32_t n_clips) {
    if (total_candidates < 0 || n_clips < 0) return -1;
    return total_candidates * (int64_t)sizeof(Cand) + (((int64_t)n_clips * 4 + 15) & ~15LL);
}

int acb_flac_decode(const uint8_t* data, const acb_flac_clip* clips, int32_t n_clips, int32_t out_dtype, void* out, int32_t* status,
                    void* workspace, int64_t total_candidates, void* stream) {
    if (n_clips < 0 || total_candidates < 0) return fail(ACB_ERR_INVALID, "acb_flac_decode: negative clip or candidate count");
    if (out_dtype != ACB_F32 && out_dtype != ACB_I16) return fail(ACB_ERR_INVALID, "acb_flac_decode: out_dtype must be ACB_F32 or ACB_I16");
    if (n_clips == 0) return ACB_OK;
    if (!data || !clips || !out || !status || !workspace) return fail(ACB_ERR_INVALID, "acb_flac_decode: null buffer");
    if (reinterpret_cast<uintptr_t>(workspace) & 15) return fail(ACB_ERR_INVALID, "acb_flac_decode: workspace must be 16-byte aligned");
    int dev = 0, sms = 0, occ = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const auto decode = out_dtype == ACB_I16 ? flac_decode_kernel<short> : flac_decode_kernel<float>;
    if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, decode, kDecodeThreads, 0);
    if (e != cudaSuccess) return fail(ACB_ERR_CUDA, std::string("acb_flac_decode: ") + cudaGetErrorString(e));
    auto* cands = static_cast<Cand*>(workspace);
    int* counts = reinterpret_cast<int*>(static_cast<char*>(workspace) + total_candidates * (int64_t)sizeof(Cand));
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    flac_locate_kernel<<<n_clips, kLocateThreads, 0, s>>>(data, clips, cands, counts);
    decode<<<sms * (occ > 0 ? occ : 1), kDecodeThreads, 0, s>>>(data, clips, n_clips, cands, counts, out);
    flac_verify_kernel<<<(n_clips + 127) / 128, 128, 0, s>>>(clips, n_clips, cands, counts, status);
    e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ACB_ERR_CUDA, std::string("acb_flac_decode launch: ") + cudaGetErrorString(e));
    return ACB_OK;
}

}  // extern "C"
