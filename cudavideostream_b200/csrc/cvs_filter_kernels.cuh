// cvs_filter_kernels.cuh -- the kernels around the fused stream kernel: noise filter, text overlay,
// binarisation pass 2, stand-alone display filters, client-side apply and the synthetic camera.
#pragma once
#include "cvs_pixel.cuh"

namespace cvs {

// ------------------------------------------------------------------------------------------------
// A10 noise filter: K x K zero-padded convolution per channel, fp32 accumulation with one FFMA per
// tap in row-major tap order, truncation to u8.   (loop structure of server/src/kernels.cu:119-134;
// nvcc contracts "acc += k*p" into FFMA, which is what reproduces REPORT/report.tex:2351-2378.)
//
// The frame is treated as an H x 3W byte image in which the horizontal neighbour of a byte is 3
// bytes away.  Fast path (3W % 4 == 0): a thread produces 4 consecutive output bytes; it fetches,
// for each of the K tap rows, the aligned words that cover bytes [x - 3(K/2), x + 3 + 3(K/2)] through
// L1 (neighbouring threads share them) and converts each byte to float once.
// ------------------------------------------------------------------------------------------------
struct ConvWeights {
    float k[81];
};

__device__ __forceinline__ uint32_t trunc_u8(float acc)
{
    // (uint8_t)acc as x86-64 compiles it: cvttss2si to a 32-bit integer, low byte.  cvttss2si gives 0x80000000 (low
    // byte 0) for NaN and for anything outside [-2^31, 2^31); F2I saturates 2^31 and above (+inf too) to 0x7fffffff,
    // whose low byte would be 0xff.  Below -2^31 it also gives 0x80000000, and NaN converts to 0.
    return acc < 2147483648.0f ? (uint32_t)__float2int_rz(acc) & 0xffu : 0u;
}

template <int K>
__global__ void __launch_bounds__(256) k_conv_rows4(const uint8_t *__restrict__ in, uint8_t *__restrict__ out,
                                                    int width, int height, size_t in_stride, size_t out_stride,
                                                    const __grid_constant__ ConvWeights w)
{
    constexpr int R = K / 2;
    constexpr int HALO = 3 * R;                      // bytes on each side
    constexpr int WL = (HALO + 3) / 4;               // whole words on each side
    constexpr int NW = 1 + 2 * WL;                   // words fetched per tap row
    const int rowbytes = 3 * width;
    const int wordsperrow = rowbytes >> 2;
    const int xw = blockIdx.x * blockDim.x + threadIdx.x; // word column
    const int row = blockIdx.y;
    const uint8_t *fin = in + (size_t)blockIdx.z * in_stride;
    uint8_t *fout = out + (size_t)blockIdx.z * out_stride;
    if (xw >= wordsperrow) return;

    float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < K; i++) {
        const int rr = row + i - R;
        uint32_t wd[NW];
        if (rr >= 0 && rr < height) {
            const uint32_t *rp = reinterpret_cast<const uint32_t *>(fin + (size_t)rr * rowbytes);
#pragma unroll
            for (int u = 0; u < NW; u++) {
                const int xi = xw + u - WL;
                wd[u] = (xi >= 0 && xi < wordsperrow) ? __ldg(rp + xi) : 0u;
            }
        } else {
#pragma unroll
            for (int u = 0; u < NW; u++) wd[u] = 0u;
        }
        // bytes at offsets [-HALO, 3 + HALO] relative to x = 4*xw  <->  byte index (4*WL - HALO) + n of wd[]
        float f[4 + 2 * HALO];
#pragma unroll
        for (int n = 0; n < 4 + 2 * HALO; n++) {
            const int bi = 4 * WL - HALO + n;
            f[n] = (float)((wd[bi >> 2] >> (8 * (bi & 3))) & 0xffu);
        }
#pragma unroll
        for (int j = 0; j < K; j++) {
            const float kw = w.k[i * K + j];
#pragma unroll
            for (int o = 0; o < 4; o++) acc[o] = __fmaf_rn(kw, f[o + 3 * j], acc[o]);
        }
    }
    uint32_t pk = trunc_u8(acc[0]) | (trunc_u8(acc[1]) << 8) | (trunc_u8(acc[2]) << 16) | (trunc_u8(acc[3]) << 24);
    reinterpret_cast<uint32_t *>(fout + (size_t)row * rowbytes)[xw] = pk;
}

// K = 3 (the reference's configuration, common.h:6) and K = 5, register-blocked: a thread produces a strip of
// 4 bytes x kConvRows rows.  Each input row is fetched once per strip (aligned words through L1), each of its
// 4 + 6*(K/2) bytes becomes a float once (PRMT into the mantissa of 2^23, one FADD) and stays in a K-row register
// window, so an output costs K*K FFMA -- in the same row-major tap order as k_conv_rows4, hence the same bits.
// NONNEG: all weights >= 0, so 0 <= acc < 2^23 and truncation is one FADD.RZ against 2^23 instead of F2I.
#ifndef CVS_CONV_ROWS
#define CVS_CONV_ROWS 8 // 12 / 16 / 24 rows per strip (fewer halo rows converted) measured the same: 6.67 / 6.66 / 6.73 vs 6.71 us per frame with the diff
#endif
constexpr int kConvRows = CVS_CONV_ROWS;

__device__ __forceinline__ float byte_to_float(uint32_t word, int b) // b: compile-time byte index
{
    return __uint_as_float(__byte_perm(word, 0x4B000000u, 0x7650u + (uint32_t)b)) - 8388608.0f;
}

// Packed pairs of floats (sm_100: FFMA2 / FADD2 work on two independent fp32 lanes held in an aligned register pair;
// each lane is rounded exactly like the scalar instruction, so the accumulation order per output byte -- and with it
// every bit -- is that of __fmaf_rn in row-major tap order).  One issue slot per two taps: the filter is FMA-pipe-bound.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi)
{
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ f32x2 pack2u(uint32_t lo, uint32_t hi)
{
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi));
    return r;
}
__device__ __forceinline__ float lo2(f32x2 v) { return __uint_as_float((uint32_t)v); }
__device__ __forceinline__ float hi2(f32x2 v) { return __uint_as_float((uint32_t)(v >> 32)); }
__device__ __forceinline__ f32x2 fma2_bcast(float a, f32x2 b, f32x2 c) // {a, a} * b + c
{
    asm("{ .reg .b64 ra;\n mov.b64 ra, {%1, %1};\n fma.rn.f32x2 %0, ra, %2, %0; }" : "+l"(c) : "f"(a), "l"(b));
    return c;
}
__device__ __forceinline__ f32x2 add2_bcast(f32x2 a, float b) // a + {b, b}, round to nearest
{
    f32x2 r;
    asm("{ .reg .b64 rb;\n mov.b64 rb, {%2, %2};\n add.rn.f32x2 %0, %1, rb; }" : "=l"(r) : "l"(a), "f"(b));
    return r;
}
__device__ __forceinline__ f32x2 add2_rz_bcast(f32x2 a, float b) // a + {b, b}, round towards zero
{
    f32x2 r;
    asm("{ .reg .b64 rb;\n mov.b64 rb, {%2, %2};\n add.rz.f32x2 %0, %1, rb; }" : "=l"(r) : "l"(a), "f"(b));
    return r;
}

template <int K, bool NONNEG, int WB>
__global__ void __launch_bounds__(128) k_conv_strip(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, int width,
                                                    int height, size_t in_stride, size_t out_stride,
                                                    const __grid_constant__ ConvWeights w)
{
    // a thread produces WB words (4*WB bytes) x kConvRows rows; WB = 2 halves the halo conversions per output byte
    constexpr int R = K / 2, HALO = 3 * R, WL = (HALO + 3) / 4, NW = WB + 2 * WL, NB = 4 * WB, NF = NB + 2 * HALO;
    static_assert(NF % 2 == 0, "the window is held as float pairs");
    constexpr int NE = NF / 2, NO = NF / 2 - 1;
    const int rowbytes = 3 * width;
    const int wordsperrow = rowbytes >> 2;
    const int xw = (blockIdx.x * blockDim.x + threadIdx.x) * WB; // first word column of this thread
    const int row0 = blockIdx.y * kConvRows;
    if (xw >= wordsperrow) return;
    const uint8_t *fin = in + (size_t)blockIdx.z * in_stride;
    uint8_t *fout = out + (size_t)blockIdx.z * out_stride;

    // window: bytes x-HALO .. x+NB-1+HALO of K consecutive input rows as floats, twice: fe[.][m] = (f[2m], f[2m+1]) and
    // fo[.][m] = (f[2m+1], f[2m+2]) -- tap j of output pair (o, o+1) reads (f[o+3j], f[o+3j+1]), which starts on an odd
    // float for odd j, and FFMA2 wants an aligned register pair.
    f32x2 fe[K][NE], fo[K][NO > 0 ? NO : 1];
    // A warp issues in order and waits at the first instruction that reads a loaded register, so the words of a row are
    // requested one output row before they are converted: fetch() only loads, convert() is the first reader.
    auto fetch = [&](int rr, uint32_t (&wd)[NW]) {
#pragma unroll
        for (int u = 0; u < NW; u++) {
            const int xi = xw + u - WL;
            wd[u] = 0u;
            if (rr >= 0 && rr < height && xi >= 0 && xi < wordsperrow)
                wd[u] = __ldg(reinterpret_cast<const uint32_t *>(fin + (size_t)rr * rowbytes) + xi);
        }
    };
    auto convert = [&](const uint32_t (&wd)[NW], f32x2 (&de)[NE], f32x2 (&dO)[NO > 0 ? NO : 1]) {
#pragma unroll
        for (int m = 0; m < NE; m++) {
            const int b0 = 4 * WL - HALO + 2 * m, b1 = b0 + 1; // byte indices inside wd[]
            // the byte lands in the mantissa of 2^23; subtracting 2^23 leaves its value (exact)
            const uint32_t u0 = __byte_perm(wd[b0 >> 2], 0x4B000000u, 0x7650u + (uint32_t)(b0 & 3));
            const uint32_t u1 = __byte_perm(wd[b1 >> 2], 0x4B000000u, 0x7650u + (uint32_t)(b1 & 3));
            de[m] = add2_bcast(pack2u(u0, u1), -8388608.0f);
        }
        // (converted again rather than copied out of de[]: two PRMT + one FADD2 land in an aligned pair directly, whereas
        // ptxas re-creates a copied pair with two MOV at each of its three uses)
#pragma unroll
        for (int m = 0; m < NO; m++) {
            const int b0 = 4 * WL - HALO + 2 * m + 1, b1 = b0 + 1;
            const uint32_t u0 = __byte_perm(wd[b0 >> 2], 0x4B000000u, 0x7650u + (uint32_t)(b0 & 3));
            const uint32_t u1 = __byte_perm(wd[b1 >> 2], 0x4B000000u, 0x7650u + (uint32_t)(b1 & 3));
            dO[m] = add2_bcast(pack2u(u0, u1), -8388608.0f);
        }
    };
    {
        uint32_t w0[K - 1][NW];
#pragma unroll
        for (int i = 0; i < K - 1; i++) fetch(row0 - R + i, w0[i]);
#pragma unroll
        for (int i = 0; i < K - 1; i++) convert(w0[i], fe[i], fo[i]);
    }
    uint32_t wn[NW]; // words of the next input row, in flight
    fetch(row0 + R, wn);
#pragma unroll
    for (int r = 0; r < kConvRows; r++) {
        const int row = row0 + r;
        if (row >= height) break;
        convert(wn, fe[(r + K - 1) % K], fo[(r + K - 1) % K]);
        if (r + 1 < kConvRows) fetch(row + 1 + R, wn);
        f32x2 acc[NB / 2];
#pragma unroll
        for (int o = 0; o < NB / 2; o++) acc[o] = 0ull;
#pragma unroll
        for (int i = 0; i < K; i++)
#pragma unroll
            for (int j = 0; j < K; j++) {
                const float kw = w.k[i * K + j];
#pragma unroll
                for (int o = 0; o < NB / 2; o++) {
                    const int s0 = 2 * o + 3 * j; // first float of the pair
                    acc[o] = fma2_bcast(kw, (s0 & 1) ? fo[(r + i) % K][s0 >> 1] : fe[(r + i) % K][s0 >> 1], acc[o]);
                }
            }
        uint32_t pk[WB];
#pragma unroll
        for (int q = 0; q < WB; q++) {
            if (NONNEG) {
                const f32x2 t0 = add2_rz_bcast(acc[2 * q], 8388608.0f), t1 = add2_rz_bcast(acc[2 * q + 1], 8388608.0f);
                const uint32_t b0 = __float_as_uint(lo2(t0)), b1 = __float_as_uint(hi2(t0)), b2 = __float_as_uint(lo2(t1)),
                               b3 = __float_as_uint(hi2(t1));
                pk[q] = __byte_perm(__byte_perm(b0, b1, 0x0040), __byte_perm(b2, b3, 0x0040), 0x5410);
            } else {
                pk[q] = trunc_u8(lo2(acc[2 * q])) | (trunc_u8(hi2(acc[2 * q])) << 8) | (trunc_u8(lo2(acc[2 * q + 1])) << 16) |
                        (trunc_u8(hi2(acc[2 * q + 1])) << 24);
            }
        }
        uint32_t *dst = reinterpret_cast<uint32_t *>(fout + (size_t)row * rowbytes) + xw;
        if (WB == 2) *reinterpret_cast<uint2 *>(dst) = make_uint2(pk[0], pk[WB - 1]); // host guarantees 8-byte alignment
        else dst[0] = pk[0];
    }
}

// generic path: any width, one output byte per thread
__global__ void __launch_bounds__(256) k_conv_bytes(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, int width,
                                                    int height, size_t in_stride, size_t out_stride, int K,
                                                    const __grid_constant__ ConvWeights w)
{
    const int rowbytes = 3 * width;
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int row = blockIdx.y;
    if (x >= rowbytes) return;
    const uint8_t *fin = in + (size_t)blockIdx.z * in_stride;
    uint8_t *fout = out + (size_t)blockIdx.z * out_stride;
    const int R = K / 2;
    float acc = 0.f;
    for (int i = 0; i < K; i++)
        for (int j = 0; j < K; j++) {
            const int rr = row + i - R, xx = x + 3 * (j - R);
            float pix = 0.f;
            if (rr >= 0 && rr < height && xx >= 0 && xx < rowbytes) pix = (float)fin[(size_t)rr * rowbytes + xx];
            acc = __fmaf_rn(w.k[i * K + j], pix, acc);
        }
    fout[(size_t)row * rowbytes + x] = (uint8_t)trunc_u8(acc);
}

// ------------------------------------------------------------------------------------------------
// text overlay: glyph idx[j] is blitted to rows [0, gh), byte columns [j*gw*3, (j+1)*gw*3)
//                                                (server/src/kernels.cu:337-348 and host loop :466-476)
// ------------------------------------------------------------------------------------------------
struct OverlayText {
    int n;
    signed char idx[252]; // glyph index per character, -1 = not in the atlas (skipped)
};

__global__ void __launch_bounds__(256) k_overlay(uint8_t *frames, size_t stride, int width, const uint8_t *__restrict__ glyphs,
                                                 int gw, int gh, const __grid_constant__ OverlayText txt)
{
    const int j = blockIdx.y; // character
    const int g = txt.idx[j];
    if (g < 0) return;
    const int mw = 3 * gw, area = mw * gh;
    const int offset = j * mw;
    if (offset + mw > 3 * width) return;
    uint8_t *f = frames + (size_t)blockIdx.z * stride;
    const uint8_t *m = glyphs + (size_t)g * area;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < area; i += gridDim.x * blockDim.x) {
        const int y = i / mw, x = offset + i - y * mw;
        f[(size_t)y * 3 * width + x] = m[i];
    }
}

// ------------------------------------------------------------------------------------------------
// A7 "two max" threshold (server/src/server.cpp:108-127).  The CPU loop keeps a running arg-max with ">=":
// index_max ends as the LAST bin that holds the global maximum and -- because sec_max is overwritten with the new
// maximum, so the else-branch can never fire -- index_sec_max ends as the running arg-max just before that, i.e.
// the previous "record" bin (a bin whose count is >= every count before it), or -1.  One 256-thread block per
// frame finds the records with a prefix maximum and picks the last two.   hist: [nframes][256]; thr: [nframes].
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_threshold(const unsigned int *__restrict__ hist, int *__restrict__ thr,
                                                   int nframes, int clamp_lo, int clamp_hi)
{
    __shared__ unsigned int wmax[8];
    __shared__ unsigned int rec[8];
    const int t = blockIdx.x, i = threadIdx.x, lane = i & 31, warp = i >> 5;
    if (t >= nframes) return;
    const unsigned int v = hist[(size_t)t * 256 + i];
    unsigned int inc = v; // inclusive prefix maximum inside the warp
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const unsigned int n = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc = max(inc, n);
    }
    if (lane == 31) wmax[warp] = inc;
    __syncthreads();
    unsigned int before = 0; // maximum of every earlier bin (0 when there is none: counts are >= 0)
    for (int w = 0; w < warp; w++) before = max(before, wmax[w]);
    const unsigned int prev = __shfl_up_sync(0xffffffffu, inc, 1);
    if (lane > 0) before = max(before, prev);
    const unsigned int b = __ballot_sync(0xffffffffu, v >= before); // bin 0 is always a record (max starts at -1)
    if (lane == 0) rec[warp] = b;
    __syncthreads();
    if (i == 0) {
        int imax = -1, isec = -1;
        for (int w = 7; w >= 0 && isec < 0; w--) {
            unsigned int m = rec[w];
            while (m && isec < 0) {
                const int bit = 31 - __clz((int)m);
                m &= ~(1u << bit);
                if (imax < 0) imax = 32 * w + bit;
                else isec = 32 * w + bit;
            }
        }
        int th = (imax + isec) / 2; // C division: (0 + -1) / 2 == 0
        if (th < clamp_lo) th = clamp_lo;
        if (th > clamp_hi) th = clamp_hi;
        thr[t] = th;
    }
}

// A6 binarize pass 2: gray1 (1 B/pixel) -> 3-channel 0/255 image   (server.cpp:129-135)
__global__ void __launch_bounds__(256) k_binarize_expand(const uint8_t *__restrict__ gray1, size_t gray_stride,
                                                         uint8_t *__restrict__ out, size_t out_stride,
                                                         const int *__restrict__ thr, uint32_t npix)
{
    const uint32_t ngroups = (npix + kGroupPixels - 1) / kGroupPixels;
    const int t = blockIdx.y;
    const int th = thr[t];
    // gray > th for all four bytes of a word at once (th is the frame's: uniform in the block).  th < 128: bit 7 of
    // (g & 0x7f) + (127 - th), or g >= 128; th >= 128: bit 7 of (g & 0x7f) + (255 - th) and g >= 128.
    const bool always = th < 0, hi = th >= 128;
    const uint32_t live = th >= 255 ? 0u : 0xffffffffu; // nothing is > 255
    const uint32_t addc = (uint32_t)((hi ? 255 - th : 127 - th) & 0x7f) * 0x01010101u;
    const uint8_t *g = gray1 + (size_t)t * gray_stride;
    uint8_t *o = out + (size_t)t * out_stride;
    for (uint32_t gi = blockIdx.x * blockDim.x + threadIdx.x; gi < ngroups; gi += gridDim.x * blockDim.x) {
        const uint32_t px0 = gi * kGroupPixels;
        const uint32_t npx = min(npix - px0, (uint32_t)kGroupPixels);
        uint32_t gw[4] = {0, 0, 0, 0};
        if (npx == (uint32_t)kGroupPixels) {
            uint4 v = *reinterpret_cast<const uint4 *>(g + px0);
            gw[0] = v.x; gw[1] = v.y; gw[2] = v.z; gw[3] = v.w;
        } else {
            for (uint32_t i = 0; i < npx; i++) gw[i >> 2] |= (uint32_t)g[px0 + i] << (8 * (i & 3));
        }
        // four pixels per word: "gray > th" as 0x80 flags with the carry-free byte compare of the diff (changed80),
        // flags -> 0xFF bytes, every byte repeated three times (B, G, R) with three PRMT: 7 instructions per 4 pixels
        uint32_t ow[kGroupWords];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            const uint32_t low = (gw[i] & 0x7f7f7f7fu) + addc;
            const uint32_t m = always ? 0xffffffffu : spread80((hi ? (low & gw[i]) : (low | gw[i])) & 0x80808080u & live);
            ow[3 * i] = __byte_perm(m, 0u, 0x1000);
            ow[3 * i + 1] = __byte_perm(m, 0u, 0x2211);
            ow[3 * i + 2] = __byte_perm(m, 0u, 0x3332);
        }
        store_group(o + (size_t)px0 * 3, ow, npx * 3);
    }
}

// ------------------------------------------------------------------------------------------------
// stand-alone display filters on a frame pair / a frame (the micro-benchmarks of tests/heat_map_*,
// tests/grayscale-*, tests/binarization).  Grid-stride over 48-byte groups.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void load_group(const uint8_t *src, uint32_t (&w)[kGroupWords], uint32_t nv)
{
    if (nv >= (uint32_t)kGroupBytes) {
        const uint4 *s = reinterpret_cast<const uint4 *>(src);
        uint4 a = __ldg(s), b = __ldg(s + 1), c = __ldg(s + 2);
        w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w;
        w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
        w[8] = c.x; w[9] = c.y; w[10] = c.z; w[11] = c.w;
    } else {
#pragma unroll
        for (int k = 0; k < kGroupWords; k++) w[k] = 0;
#pragma unroll
        for (int j = 0; j < kGroupBytes; j++)
            if ((uint32_t)j < nv) w[j >> 2] |= (uint32_t)src[j] << (8 * (j & 3));
    }
}

// OP: 0 heat map (prev, cur), 1 red map (prev, cur, threshold), 2 gray avg 3ch, 3 gray weighted 3ch,
//     4 gray avg 1ch, 5 gray weighted 1ch
template <int OP, bool HI>
__global__ void __launch_bounds__(256) k_filter(const uint8_t *__restrict__ prev, const uint8_t *__restrict__ cur,
                                                uint8_t *__restrict__ out, uint32_t nbytes, uint32_t addc,
                                                const uint32_t *__restrict__ lut_g, unsigned int *hist)
{
    __shared__ uint32_t slut[768];
    __shared__ uint32_t shist[256];
    if (OP == 0)
        for (uint32_t i = threadIdx.x; i < 766; i += blockDim.x) slut[i] = lut_g[i];
    if (OP >= 4 && hist)
        for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) shist[i] = 0;
    __syncthreads();
    const uint32_t ngroups = (nbytes + kGroupBytes - 1) / kGroupBytes;
    for (uint32_t gi = blockIdx.x * blockDim.x + threadIdx.x; gi < ngroups; gi += gridDim.x * blockDim.x) {
        const uint32_t goff = gi * kGroupBytes;
        const uint32_t nv = min(nbytes - goff, (uint32_t)kGroupBytes);
        uint32_t c[kGroupWords], o[kGroupWords];
        load_group(cur + goff, c, nv);
        if (OP == 0 || OP == 1) {
            uint32_t r[kGroupWords];
            load_group(prev + goff, r, nv);
            if (OP == 0) {
                uint32_t ad[kGroupWords];
#pragma unroll
                for (int k = 0; k < kGroupWords; k++) ad[k] = absdiff4(c[k], r[k]);
                group_heat(ad, slut, o);
            } else {
                uint32_t mk[kGroupWords];
#pragma unroll
                for (int k = 0; k < kGroupWords; k++) mk[k] = changed80<HI>(absdiff4(c[k], r[k]), addc);
                group_red<false>(mk, r, o);
            }
            store_group(out + goff, o, nv);
        } else if (OP == 2 || OP == 3) {
            group_gray3<OP == 3>(c, o);
            store_group(out + goff, o, nv);
        } else {
            uint32_t g4[4];
            group_gray1<OP == 5>(c, g4);
            const uint32_t npx = nv / 3u;
            uint8_t *gd = out + goff / 3u;
            if (npx == (uint32_t)kGroupPixels) stg_stream(gd, make_uint4(g4[0], g4[1], g4[2], g4[3]));
#pragma unroll
            for (int px = 0; px < kGroupPixels; px++)
                if ((uint32_t)px < npx) {
                    const uint32_t gv = byte_of(g4[px >> 2], px & 3);
                    if (npx != (uint32_t)kGroupPixels) gd[px] = (uint8_t)gv;
                    if (hist) atomicAdd(&shist[gv], 1u);
                }
        }
    }
    if (OP >= 4 && hist) {
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x)
            if (shist[i]) atomicAdd(hist + i, shist[i]);
    }
}

// ------------------------------------------------------------------------------------------------
// Binarisation pass 1 of a SEQUENCE (modes 5, 7): gray byte of every pixel + one 256-bin histogram per frame
// (server.cpp:96-106, tests/grayscale-weighted/cpu.cu:38-42), grid = (blocks per frame, frames).
// In a sequence this runs as a kernel of its own in front of the plain diff+compact kernel instead of inside it:
// k_stream_ws' front warps (4 per scheduler) are what the fused form waits for -- the exact weighted gray is ~15
// instructions per pixel on them, 3.7 us per 1080p frame on top of the diff -- whereas here 64 warps per SM hide the
// same arithmetic behind the frame's loads (one extra read of the frame, which HBM has room for; measured in
// profiles/README.md).  Single frames (the drop-in call) keep the fused kernel: one launch less.
//   hist: [nframes][256], zeroed by the caller; gray1: [nframes][gray_stride]
// Lane L adds to histogram copy L mod kGrayHistCopies (copy-interleaved: the copies of a bin sit in different banks).
// ------------------------------------------------------------------------------------------------
#ifndef CVS_GRAY_HIST_COPIES
#define CVS_GRAY_HIST_COPIES 1 // 4 / 8 / 16 copies measured 1-3 % slower (6.89 / 6.90 / 6.81 vs 6.72 us per frame, mode 5): not conflict-bound
#endif
constexpr int kGrayHistCopies = CVS_GRAY_HIST_COPIES;
#ifndef CVS_GRAY_HIST_GROUPS
#define CVS_GRAY_HIST_GROUPS 4
#endif
constexpr int kGrayHistGroupsPerThread = CVS_GRAY_HIST_GROUPS; // groups (16 pixels each) a thread walks: fewer histogram flushes per frame

template <bool WEIGHTED>
__global__ void __launch_bounds__(256) k_gray_hist_seq(const uint8_t *__restrict__ frames, size_t frame_stride, uint32_t nbytes,
                                                        uint8_t *__restrict__ gray1, size_t gray_stride,
                                                        unsigned int *__restrict__ hist)
{
    __shared__ uint32_t shist[256 * kGrayHistCopies];
    for (uint32_t i = threadIdx.x; i < 256u * kGrayHistCopies; i += blockDim.x) shist[i] = 0;
    __syncthreads();
    const uint32_t t = blockIdx.y;
    const uint8_t *cur = frames + (size_t)t * frame_stride;
    uint8_t *gout = gray1 + (size_t)t * gray_stride;
    const uint32_t copy = threadIdx.x & (kGrayHistCopies - 1);
    const uint32_t ngroups = (nbytes + kGroupBytes - 1) / kGroupBytes;
    for (uint32_t gi = blockIdx.x * blockDim.x + threadIdx.x; gi < ngroups; gi += gridDim.x * blockDim.x) {
        const uint32_t goff = gi * kGroupBytes;
        const uint32_t nv = min(nbytes - goff, (uint32_t)kGroupBytes);
        uint32_t c[kGroupWords], g4[4];
        load_group(cur + goff, c, nv);
        group_gray1<WEIGHTED>(c, g4);
        const uint32_t npx = nv / 3u;
        uint8_t *gd = gout + goff / 3u;
        if (npx == (uint32_t)kGroupPixels) stg_stream(gd, make_uint4(g4[0], g4[1], g4[2], g4[3]));
#pragma unroll
        for (int px = 0; px < kGroupPixels; px++)
            if ((uint32_t)px < npx) {
                const uint32_t gv = byte_of(g4[px >> 2], px & 3);
                if (npx != (uint32_t)kGroupPixels) gd[px] = (uint8_t)gv;
                atomicAdd(&shist[gv * kGrayHistCopies + copy], 1u); // server.cpp:103-106
            }
    }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) {
        uint32_t hv = 0;
#pragma unroll
        for (int k = 0; k < kGrayHistCopies; k++) hv += shist[i * kGrayHistCopies + k];
        if (hv) atomicAdd(hist + (size_t)t * 256 + i, hv);
    }
}

// ------------------------------------------------------------------------------------------------
// client side of the wire format: frame[xs[i]] += diff[i]   (client/opencv.cpp:64-66)
// xs is strictly ascending, so no two entries touch the same byte.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_client_apply(uint8_t *frame, const int *__restrict__ xs,
                                                      const uint8_t *__restrict__ diff,
                                                      const unsigned int *__restrict__ pos, size_t capacity)
{
    size_t n = *pos;
    if (n > capacity) n = capacity;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int x = xs[i];
        frame[x] = (uint8_t)(frame[x] + diff[i]);
    }
}

// ------------------------------------------------------------------------------------------------
// egress: push exactly pos payload entries from the device buffers into the caller's pinned host buffers
// (mapped into the device address space), 16 bytes per store.  Replaces the count round trip + two
// cudaMemcpyAsync of server/src/kernels.cu:507-508, 522-524.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_payload_push(const int *__restrict__ xs, const uint8_t *__restrict__ diff,
                                                      const unsigned int *__restrict__ pos, int *h_xs, uint8_t *h_diff,
                                                      size_t capacity)
{
    size_t n = *pos;
    if (n > capacity) n = capacity;
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nt = (size_t)gridDim.x * blockDim.x;
    const size_t xq = n / 4, dq = n / 16; // whole 16-byte vectors
    for (size_t i = tid; i < xq; i += nt) reinterpret_cast<uint4 *>(h_xs)[i] = reinterpret_cast<const uint4 *>(xs)[i];
    for (size_t i = tid; i < dq; i += nt) reinterpret_cast<uint4 *>(h_diff)[i] = reinterpret_cast<const uint4 *>(diff)[i];
    for (size_t i = 4 * xq + tid; i < n; i += nt) h_xs[i] = xs[i];
    for (size_t i = 16 * dq + tid; i < n; i += nt) h_diff[i] = diff[i];
}

// ------------------------------------------------------------------------------------------------
// Opt-in compact wire format "CVW1" (SURVEY.md section 8f row 3).  The reference sends, per frame, u32 pos,
// i32 xs[pos], u8 diff[pos] (server/src/threads.cpp:229-231, read back by client/opencv.cpp:52-66): 5 bytes per
// entry.  Because xs is ascending, the index can be sent as (tile, offset): the frame is cut into tiles of
// kWireTile = 192 bytes (64 pixels), a tile's entry count fits one byte (0..192) and so does the offset inside the
// tile.  Encoded frame (little endian):
//     u32 magic "CVW1", u32 pos, u32 ntiles, u32 tile            16-byte header
//     u8  count[ntiles]   (padded to a multiple of 16)
//     u8  off[pos]        (padded to a multiple of 16)            offset of entry i inside its tile
//     u8  diff[pos]                                               the reference's value bytes, unchanged
// = 16 + N/192 + 2 pos bytes instead of 4 + 5 pos.  Encoding is two small kernels over the payload the stream kernel
// left in device memory; they store 16 bytes per thread straight into the caller's (mapped, pinned) buffer.
// Decoding (client side): exclusive scan of the counts, then one warp per tile checks the offsets, then one warp per
// tile applies them.
// ------------------------------------------------------------------------------------------------
constexpr uint32_t kWireTile = 192;
constexpr uint32_t kWireMagic = 0x31575643u; // "CVW1"
constexpr uint32_t kWireHeader = 16;

__host__ __device__ __forceinline__ uint32_t wire_pad16(uint32_t v) { return (v + 15u) & ~15u; }

// starts[t] = number of entries with index < t * kWireTile, t = 0..ntiles (xs ascending: one binary search each)
__global__ void __launch_bounds__(256) k_wire_bounds(const int *__restrict__ xs, const unsigned int *__restrict__ pos,
                                                     size_t capacity, uint32_t ntiles, uint32_t *__restrict__ starts)
{
    uint32_t n = *pos;
    if (n > capacity) n = (uint32_t)capacity;
    for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t <= ntiles; t += gridDim.x * blockDim.x) {
        const int key = (int)(t * kWireTile);
        uint32_t lo = 0, hi = n;
        while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (__ldg(xs + mid) < key) lo = mid + 1;
            else hi = mid;
        }
        starts[t] = lo;
    }
}

// header, per-tile counts and the (offset, value) bytes; `out` may be mapped host memory (16-byte aligned)
__global__ void __launch_bounds__(256) k_wire_pack(const int *__restrict__ xs, const uint8_t *__restrict__ diff,
                                                   const unsigned int *__restrict__ pos, size_t capacity, uint32_t ntiles,
                                                   const uint32_t *__restrict__ starts, uint8_t *out)
{
    uint32_t n = *pos;
    if (n > capacity) n = (uint32_t)capacity;
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x, nt = gridDim.x * blockDim.x;
    if (tid == 0) *reinterpret_cast<uint4 *>(out) = make_uint4(kWireMagic, n, ntiles, kWireTile);
    uint8_t *cnt = out + kWireHeader;
    uint8_t *off = cnt + wire_pad16(ntiles);
    uint8_t *val = off + wire_pad16(n);
    // counts: 16 tiles per thread
    for (uint32_t t0 = 16 * tid; t0 < ntiles; t0 += 16 * nt) {
        uint32_t w[4] = {0, 0, 0, 0};
#pragma unroll
        for (int j = 0; j < 16; j++) {
            const uint32_t t = t0 + j;
            const uint32_t c = t < ntiles ? starts[t + 1] - starts[t] : 0u;
            w[j >> 2] |= c << (8 * (j & 3));
        }
        *reinterpret_cast<uint4 *>(cnt + t0) = make_uint4(w[0], w[1], w[2], w[3]);
    }
    // entries: 16 per thread
    for (uint32_t i0 = 16 * tid; i0 < n; i0 += 16 * nt) {
        uint32_t w[4] = {0, 0, 0, 0};
        if (i0 + 16 <= n) {
            const int4 *xp = reinterpret_cast<const int4 *>(xs + i0);
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int4 x = __ldg(xp + q);
                w[q] = ((uint32_t)x.x % kWireTile) | (((uint32_t)x.y % kWireTile) << 8) | (((uint32_t)x.z % kWireTile) << 16) |
                       (((uint32_t)x.w % kWireTile) << 24);
            }
            *reinterpret_cast<uint4 *>(val + i0) = __ldg(reinterpret_cast<const uint4 *>(diff + i0));
        } else {
            for (uint32_t j = 0; i0 + j < n; j++) {
                w[j >> 2] |= ((uint32_t)xs[i0 + j] % kWireTile) << (8 * (j & 3));
                val[i0 + j] = diff[i0 + j];
            }
        }
        *reinterpret_cast<uint4 *>(off + i0) = make_uint4(w[0], w[1], w[2], w[3]); // the off region is padded to 16
    }
}

// client: exclusive scan of the per-tile counts of one encoded frame -> starts[0..ntiles], one 1024-thread block.
// starts[ntiles + 1] = 0 when the header matches the frame geometry, no tile counts more entries than it has bytes
// (192, the last tile last_len) and the counts add up to pos (so pos <= N); else 1.
__global__ void __launch_bounds__(1024) k_wire_scan(const uint8_t *__restrict__ wire, uint32_t ntiles_expected,
                                                    uint32_t last_len, uint32_t *__restrict__ starts)
{
    __shared__ uint32_t wsum[32];
    const uint4 hd = *reinterpret_cast<const uint4 *>(wire);
    const uint32_t ntiles = ntiles_expected;
    const bool header_ok = hd.x == kWireMagic && hd.z == ntiles_expected && hd.w == kWireTile;
    const uint8_t *cnt = wire + kWireHeader;
    const uint32_t per = (ntiles + 1023u) / 1024u;
    const uint32_t t0 = threadIdx.x * per;
    uint32_t mine = 0;
    bool too_many = false;
    for (uint32_t j = 0; j < per; j++)
        if (t0 + j < ntiles) {
            const uint32_t c = cnt[t0 + j];
            too_many |= c > (t0 + j + 1 == ntiles ? last_len : kWireTile);
            mine += c;
        }
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t incl = warp_incl_scan(mine, lane);
    if (lane == 31) wsum[warp] = incl;
    too_many = __syncthreads_or(too_many);
    if (warp == 0) {
        const uint32_t v = wsum[lane];
        const uint32_t iv = warp_incl_scan(v, lane);
        wsum[lane] = iv - v;
    }
    __syncthreads();
    uint32_t run = wsum[warp] + incl - mine;
    for (uint32_t j = 0; j < per; j++)
        if (t0 + j < ntiles) {
            starts[t0 + j] = run;
            run += cnt[t0 + j];
        }
    if (threadIdx.x == 1023) {
        starts[ntiles] = run;
        starts[ntiles + 1] = (header_ok && !too_many && run == hd.y) ? 0u : 1u;
    }
}

// client: inside every tile the offsets are strictly ascending and below the tile's length (192, the last tile
// last_len), one warp per tile; a violation sets bit 1 of starts[ntiles + 1].  Runs only on a frame k_wire_scan found
// consistent, so it reads no further than the frame's cvs_wire_size.  Afterwards no two entries name the same byte.
__global__ void __launch_bounds__(256) k_wire_check(const uint8_t *__restrict__ wire, uint32_t ntiles, uint32_t last_len,
                                                    uint32_t *starts)
{
    if (starts[ntiles + 1]) return;
    const uint8_t *cnt = wire + kWireHeader;
    const uint8_t *off = cnt + wire_pad16(ntiles);
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    bool bad = false;
    for (uint32_t t = w; t < ntiles; t += nw) {
        const uint32_t c = cnt[t], s0 = starts[t], len = t + 1 == ntiles ? last_len : kWireTile;
        for (uint32_t j = lane; j < c; j += 32) {
            const uint32_t o = off[s0 + j];
            bad |= o >= len || (j > 0 && o <= off[s0 + j - 1]);
        }
    }
    if (bad) atomicOr(starts + ntiles + 1, 2u);
}

// client: frame[x] += diff (client/opencv.cpp:64-66) and/or the reference-format payload back, one warp per tile
__global__ void __launch_bounds__(256) k_wire_apply(const uint8_t *__restrict__ wire, uint32_t ntiles,
                                                    const uint32_t *__restrict__ starts, uint8_t *frame, int *xs_out,
                                                    uint8_t *diff_out, unsigned int *pos_out)
{
    if (starts[ntiles + 1]) return; // inconsistent frame: nothing is applied, the host reports it
    // (offsets checked by k_wire_check: x < N and distinct, so the plain read-modify-write of frame[x] does not race)
    const uint32_t n = starts[ntiles];
    const uint8_t *cnt = wire + kWireHeader;
    const uint8_t *off = cnt + wire_pad16(ntiles);
    const uint8_t *val = off + wire_pad16(n);
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
    if (pos_out && blockIdx.x == 0 && threadIdx.x == 0) *pos_out = n;
    for (uint32_t t = w; t < ntiles; t += nw) {
        const uint32_t c = cnt[t], s0 = starts[t];
        for (uint32_t j = lane; j < c; j += 32) {
            const uint32_t x = t * kWireTile + off[s0 + j];
            const uint8_t d = val[s0 + j];
            if (frame) frame[x] = (uint8_t)(frame[x] + d);
            if (xs_out) xs_out[s0 + j] = (int)x;
            if (diff_out) diff_out[s0 + j] = d;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// synthetic camera (SURVEY.md section 8d); numpy twin: cudavideostream_b200/synth.py
// ------------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint8_t synth_base_byte(uint64_t seed, uint32_t i, int width, int height)
{
    const uint32_t px = i / 3u, ch = i - 3u * px;
    const uint32_t x = px % (uint32_t)width, y = px / (uint32_t)width;
    const uint32_t den = (uint32_t)(width + height - 2);
    const int grad = den ? (int)(((x + y) * 255u) / den) : 0;
    const uint64_t h = splitmix64(seed + (uint64_t)i);
    int v = grad + (int)(h & 63u) - 32 + 3 * (int)ch;
    v = v < 0 ? 0 : (v > 255 ? 255 : v);
    return (uint8_t)v;
}

__host__ __device__ __forceinline__ uint8_t synth_next_byte(uint64_t key, uint32_t i, uint8_t prev, uint32_t density_ppm)
{
    const uint64_t h = splitmix64(key + (uint64_t)i);
    const uint32_t u = (uint32_t)(h & 0xFFFFFu);
    int v;
    if ((((uint64_t)u * 1000000ull) >> 20) < (uint64_t)density_ppm) {
        const int delta = 21 + (int)((h >> 20) % 60u);
        const bool up = (h >> 40) & 1u;
        v = up ? prev + delta : prev - delta;
        if (v > 255) v = prev - delta;
        if (v < 0) v = prev + delta;
    } else {
        v = (int)prev + (int)((h >> 24) % 7u) - 3;
        v = v < 0 ? 0 : (v > 255 ? 255 : v);
    }
    return (uint8_t)v;
}

__global__ void __launch_bounds__(256) k_synth_base(uint8_t *out, uint32_t nbytes, int width, int height, uint64_t seed)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nbytes; i += gridDim.x * blockDim.x)
        out[i] = synth_base_byte(seed, i, width, height);
}

__global__ void __launch_bounds__(256) k_synth_next(const uint8_t *__restrict__ prev, uint8_t *out, uint32_t nbytes,
                                                    uint64_t key, uint32_t density_ppm)
{
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < nbytes; i += gridDim.x * blockDim.x)
        out[i] = synth_next_byte(key, i, prev[i], density_ppm);
}

} // namespace cvs
