// cvs_pixel.cuh -- per-group pixel arithmetic of the filter chain.
//
// A "group" is 48 consecutive frame bytes = 16 whole BGR pixels = 12 32-bit words held in
// registers (48 is the smallest size that is both a whole number of pixels and a whole number of
// 16-byte vector accesses).  Every routine here is bit-exact with the CPU loop it cites.
#pragma once
#include "cvs_device.cuh"

namespace cvs {

constexpr int kGroupBytes = 48;
constexpr int kGroupWords = 12;
constexpr int kGroupPixels = 16;

enum Mode : int {
    kModeNone = 0,
    kModeHeat = 1,         // tests/heat_map_benchmark/cpu.cu:19-27,54-66
    kModeRedBlack = 2,     // server/src/kernels.cu:273-281 on a zeroed frame (:513)
    kModeRedOverlap = 3,   // server/src/kernels.cu:517 on the previous reference frame
    kModeGrayWeighted = 4, // tests/grayscale-weighted/cpu.cu:38-42
    kModeBinarize = 5,     // weighted gray -> histogram -> two-max -> binarize (kernels.cu:493-499)
    kModeGrayAverage = 6,  // server/src/server.cpp:96-101
    kModeBinarizeAvg = 7   // server/src/server.cpp:96-135
};

// byte j (compile-time after unrolling) of a 12-word group
__device__ __forceinline__ uint32_t gbyte(const uint32_t (&w)[kGroupWords], int j)
{
    return __byte_perm(w[j >> 2], 0u, 0x4440u + (uint32_t)(j & 3)); // one PRMT (a shift and a mask are two)
}

// (B + G + R) / 3, integer division                                   server.cpp:96-101
__device__ __forceinline__ uint32_t gray_avg(uint32_t b, uint32_t g, uint32_t r) { return (b + g + r) / 3u; }

// (uchar)(0.114*B + 0.587*G + 0.299*R): double products, left-to-right double adds, truncation
//                                                              tests/grayscale-weighted/cpu.cu:38-42
// Exact integer shortcut: with s = 114 B + 587 G + 299 R the true value is s/1000; unless s is a
// multiple of 1000 it lies >= 0.001 from an integer, far more than the < 1e-12 rounding error of
// the three double products and two adds, so trunc(double expression) == s / 1000.  When s is a
// multiple of 1000 the double expression can land just below the integer (e.g. 96.99999999999999),
// so that case evaluates the reference's expression itself with round-to-nearest, un-fused
// double operations (identical to x86-64 SSE2 code built without FMA contraction).
__device__ __forceinline__ uint32_t gray_weighted(uint32_t b, uint32_t g, uint32_t r)
{
    uint32_t s = 114u * b + 587u * g + 299u * r;
    uint32_t q = s / 1000u;
    if (s - q * 1000u == 0u) {
        double v = __dadd_rn(__dadd_rn(__dmul_rn(0.114, (double)b), __dmul_rn(0.587, (double)g)),
                             __dmul_rn(0.299, (double)r));
        q = (uint32_t)(int)v;
    }
    return q;
}

template <bool WEIGHTED>
__device__ __forceinline__ uint32_t gray_of(uint32_t b, uint32_t g, uint32_t r)
{
    return WEIGHTED ? gray_weighted(b, g, r) : gray_avg(b, g, r);
}

// byte k of a word with ONE instruction (PRMT; the shift-and-mask form costs two on the same pipe)
__device__ __forceinline__ uint32_t byte_of(uint32_t w, int k) { return __byte_perm(w, 0u, 0x4440u + (uint32_t)k); }

// Four gray values (the four pixels of twelve frame bytes w0 w1 w2), packed into one word.
// Weighted: the same values as gray_weighted(), arranged for the instruction scheduler -- the four pixels form ONE
// basic block instead of four (a test-and-branch per pixel puts the pixels' multiply chains in series, and the warps
// that run this inside k_stream_ws have few neighbours to hide them behind).  With M = 4,294,968 = ceil(2^32 / 1000)
// the 64-bit product s * M holds s / 1000 in its upper word for every s <= 255,000 (the error 0.704 s stays below
// 2^32 / 1000), and its lower word is below 1,000,000 exactly when s is a multiple of 1000 (remainder 0: <= 179,520;
// remainder >= 1: >= 4,294,967).  Only then -- one pixel in a thousand -- the reference's double expression is evaluated.
template <bool WEIGHTED>
__device__ __forceinline__ uint32_t gray4(uint32_t w0, uint32_t w1, uint32_t w2)
{
    const uint32_t b[4] = {byte_of(w0, 0), byte_of(w0, 3), byte_of(w1, 2), byte_of(w2, 1)};
    const uint32_t g[4] = {byte_of(w0, 1), byte_of(w1, 0), byte_of(w1, 3), byte_of(w2, 2)};
    const uint32_t r[4] = {byte_of(w0, 2), byte_of(w1, 1), byte_of(w2, 0), byte_of(w2, 3)};
    uint32_t q[4];
    if (!WEIGHTED) {
#pragma unroll
        for (int i = 0; i < 4; i++) q[i] = gray_avg(b[i], g[i], r[i]);
    } else {
        uint32_t s[4];
        bool multiple = false;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            s[i] = 114u * b[i] + 587u * g[i] + 299u * r[i];
            const uint64_t m = (uint64_t)s[i] * 4294968ull;
            q[i] = (uint32_t)(m >> 32);
            multiple |= (uint32_t)m < 1000000u;
        }
        if (multiple) {
#pragma unroll
            for (int i = 0; i < 4; i++)
                if (s[i] == q[i] * 1000u) q[i] = gray_weighted(b[i], g[i], r[i]);
        }
    }
    return __byte_perm(__byte_perm(q[0], q[1], 0x0040), __byte_perm(q[2], q[3], 0x0040), 0x5410);
}

// 16 gray values of a group, packed 4 per word
template <bool WEIGHTED>
__device__ __forceinline__ void group_gray1(const uint32_t (&c)[kGroupWords], uint32_t (&g)[4])
{
#pragma unroll
    for (int i = 0; i < 4; i++) g[i] = gray4<WEIGHTED>(c[3 * i], c[3 * i + 1], c[3 * i + 2]);
}

// gray replicated to the three channels: pixels 4i..4i+3 = gray bytes (g0 g0 g0 g1 | g1 g1 g2 g2 | g2 g3 g3 g3)
template <bool WEIGHTED>
__device__ __forceinline__ void group_gray3(const uint32_t (&c)[kGroupWords], uint32_t (&o)[kGroupWords])
{
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const uint32_t g = gray4<WEIGHTED>(c[3 * i], c[3 * i + 1], c[3 * i + 2]);
        o[3 * i] = __byte_perm(g, 0u, 0x1000);
        o[3 * i + 1] = __byte_perm(g, 0u, 0x2211);
        o[3 * i + 2] = __byte_perm(g, 0u, 0x3332);
    }
}

// heat map: d = |dB|+|dG|+|dR| in 0..765, colour from the 766-entry table (built on the host with
// the reference's own double-precision sin() expression, so the result is bit-exact)
//                                                     tests/heat_map_benchmark/cpu.cu:19-27,54-66
__device__ __forceinline__ void group_heat(const uint32_t (&ad)[kGroupWords], const uint32_t *lut,
                                           uint32_t (&o)[kGroupWords])
{
    // four pixels = three words: the 24-bit table entries l0..l3 are laid end to end with three PRMT (measured equal to the
    // shift-and-or form: 3.86 vs 3.87 us per frame -- after the one-PRMT gbyte the heat map no longer waits for this)
#pragma unroll
    for (int i = 0; i < kGroupPixels / 4; i++) {
        uint32_t l[4];
#pragma unroll
        for (int p = 0; p < 4; p++) {
            const int j = 12 * i + 3 * p;
            l[p] = lut[gbyte(ad, j) + gbyte(ad, j + 1) + gbyte(ad, j + 2)];
        }
        o[3 * i] = __byte_perm(l[0], l[1], 0x4210);     // B0 G0 R0 B1
        o[3 * i + 1] = __byte_perm(l[1], l[2], 0x5421); // G1 R1 B2 G2
        o[3 * i + 2] = __byte_perm(l[2], l[3], 0x6542); // R2 B3 G3 R3
    }
}

// red map: pixel with any changed channel -> (0,0,255), else `base` (zero or the old reference)
//   m80: 0x80 in every changed byte          tests/heat_map_red_benchmark/cpu.cu:38-55, kernels.cu:273-281
template <bool OVERLAP>
__device__ __forceinline__ void group_red(const uint32_t (&m80)[kGroupWords], const uint32_t (&base)[kGroupWords],
                                          uint32_t (&o)[kGroupWords])
{
#pragma unroll
    for (int k = 0; k < kGroupWords; k++) o[k] = OVERLAP ? base[k] : 0u;
#pragma unroll
    for (int p = 0; p < kGroupPixels; p++) {
        uint32_t any = gbyte(m80, 3 * p) | gbyte(m80, 3 * p + 1) | gbyte(m80, 3 * p + 2); // 0 or 0x80
        // R byte of pixel p is byte 3p+2
        const int j = 3 * p + 2;
        uint32_t ff = (any >> 7) * 0xffu;
        o[j >> 2] |= ff << (8 * (j & 3));
    }
}

// store the first nv bytes of a group (nv == 48: three 16-byte streaming stores)
__device__ __forceinline__ void store_group(uint8_t *dst, const uint32_t (&o)[kGroupWords], uint32_t nv)
{
    if (nv >= (uint32_t)kGroupBytes) {
        stg_stream(dst, make_uint4(o[0], o[1], o[2], o[3]));
        stg_stream(dst + 16, make_uint4(o[4], o[5], o[6], o[7]));
        stg_stream(dst + 32, make_uint4(o[8], o[9], o[10], o[11]));
    } else {
#pragma unroll
        for (int j = 0; j < kGroupBytes; j++)
            if ((uint32_t)j < nv) dst[j] = (uint8_t)gbyte(o, j);
    }
}

} // namespace cvs
