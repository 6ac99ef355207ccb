// cvs_yuv.cuh -- raw camera YUV (YUYV 4:2:2, NV12 / I420 4:2:0) -> packed BGR24 with OpenCV's pixels
// (cv2.cvtColor COLOR_YUV2BGR_YUYV / _NV12 / _I420: BT.601 limited range, nearest-neighbour chroma).
//
// OpenCV's fixed-point form, integer only (matched on all 2^24 (Y, U, V) triples, tests/test_yuv_oracle.py):
//     y = max(0, Y - 16) * 1220542,  u = U - 128,  v = V - 128
//     B = clamp((y + 2^19 + 2116026 u) >> 20),  G = clamp((y + 2^19 - 409993 u - 852492 v) >> 20),
//     R = clamp((y + 2^19 + 1673527 v) >> 20)
// No sum leaves int32: y < 2^29 and every chroma term is below 2^29 in magnitude.
#pragma once
#include "cvs_pixel.cuh"

namespace cvs {

enum YuvFormat { kYuyv = 1, kNv12 = 2, kI420 = 3 };

struct YuvParams {
    const uint8_t *plane[3]; // YUYV: [0]; NV12: Y, UV; I420: Y, U, V
    size_t pitch[3];         // bytes per row of each plane
    uint8_t *bgr;            // 3 * width * height bytes, rows contiguous
    int width, height;       // width even; height even for the 4:2:0 formats
    uint32_t groups;         // 16-pixel groups per row: (width + 15) / 16
};

constexpr int kYuvThreads = 256;
constexpr int kYuvPixels = 16; // pixels per thread: one 16-byte Y load, three 16-byte BGR stores

__device__ __forceinline__ uint32_t word_of(const uint4 &v, int k) { return k == 0 ? v.x : k == 1 ? v.y : k == 2 ? v.z : v.w; }
__device__ __forceinline__ uint32_t byte_of(const uint4 &v, int i) { return byte_of(word_of(v, i >> 2), i & 3); } // i: a constant after unrolling
__device__ __forceinline__ uint32_t clamp_u8(int32_t v) { return (uint32_t)min(max(v, 0), 255); }

// One thread = 16 horizontally adjacent pixels of one row (the last group of a row may hold fewer; widths are even, so
// a group always holds whole chroma pairs).  Where the sources and the destination are aligned (every group when width
// % 16 == 0 and the pitches are multiples of 16) it reads its Y / YUYV / UV bytes with 16-byte loads (I420: 8-byte U
// and V loads) and writes its 48 BGR bytes with three 16-byte stores; any other group (widths such as 1918, packed
// planes whose rows are not aligned) runs the same arithmetic on byte loads and stores.  The stores are plain: in the
// submit path the stream kernel reads the frame right behind, from L2.  Nothing outside the 3 * width * height bytes of
// p.bgr is written.
template <int FMT>
__global__ void __launch_bounds__(kYuvThreads) k_yuv_to_bgr(const YuvParams p)
{
    const uint32_t item = blockIdx.x * kYuvThreads + threadIdx.x;
    const uint32_t row = item / p.groups;
    if (row >= (uint32_t)p.height) return;
    const int x0 = (int)(item - row * p.groups) * kYuvPixels;
    const int npx = min(kYuvPixels, p.width - x0);
    const uint32_t crow = FMT == kYuyv ? row : row >> 1;
    const uint8_t *s0 = p.plane[0] + (size_t)row * p.pitch[0] + (FMT == kYuyv ? 2 * x0 : x0);
    const uint8_t *s1 = FMT == kYuyv ? nullptr : p.plane[1] + (size_t)crow * p.pitch[1] + (FMT == kNv12 ? x0 : x0 / 2);
    const uint8_t *s2 = FMT == kI420 ? p.plane[2] + (size_t)crow * p.pitch[2] + x0 / 2 : nullptr;

    uint32_t Y[kYuvPixels], U[kYuvPixels / 2], V[kYuvPixels / 2];
    bool vec = npx == kYuvPixels && (reinterpret_cast<uintptr_t>(s0) & 15u) == 0;
    if (FMT == kNv12) vec = vec && (reinterpret_cast<uintptr_t>(s1) & 15u) == 0;
    if (FMT == kI420) vec = vec && ((reinterpret_cast<uintptr_t>(s1) | reinterpret_cast<uintptr_t>(s2)) & 7u) == 0;
    if (vec) {
        if (FMT == kYuyv) { // Y0 U Y1 V per pair: pairs 0..3 in a, 4..7 in b
            const uint4 a = __ldg(reinterpret_cast<const uint4 *>(s0)), b = __ldg(reinterpret_cast<const uint4 *>(s0) + 1);
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const uint32_t w = word_of(j < 4 ? a : b, j & 3);
                Y[2 * j] = byte_of(w, 0);
                U[j] = byte_of(w, 1);
                Y[2 * j + 1] = byte_of(w, 2);
                V[j] = byte_of(w, 3);
            }
        } else {
            const uint4 y = __ldg(reinterpret_cast<const uint4 *>(s0));
#pragma unroll
            for (int i = 0; i < kYuvPixels; i++) Y[i] = byte_of(y, i);
            if (FMT == kNv12) { // U V interleaved
                const uint4 c = __ldg(reinterpret_cast<const uint4 *>(s1));
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    U[j] = byte_of(c, 2 * j);
                    V[j] = byte_of(c, 2 * j + 1);
                }
            } else {
                const uint2 u = __ldg(reinterpret_cast<const uint2 *>(s1)), v = __ldg(reinterpret_cast<const uint2 *>(s2));
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    U[j] = byte_of(j < 4 ? u.x : u.y, j & 3);
                    V[j] = byte_of(j < 4 ? v.x : v.y, j & 3);
                }
            }
        }
    } else {
#pragma unroll
        for (int j = 0; j < 8; j++) {
            Y[2 * j] = Y[2 * j + 1] = U[j] = V[j] = 0;
            if (2 * j < npx) {
                if (FMT == kYuyv) {
                    Y[2 * j] = s0[4 * j];
                    U[j] = s0[4 * j + 1];
                    Y[2 * j + 1] = s0[4 * j + 2];
                    V[j] = s0[4 * j + 3];
                } else {
                    Y[2 * j] = s0[2 * j];
                    Y[2 * j + 1] = s0[2 * j + 1];
                    U[j] = FMT == kNv12 ? s1[2 * j] : s1[j];
                    V[j] = FMT == kNv12 ? s1[2 * j + 1] : s2[j];
                }
            }
        }
    }

    // 48 output bytes B G R per pixel, packed into 12 little-endian words
    uint32_t out[12];
#pragma unroll
    for (int k = 0; k < 12; k++) out[k] = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const int32_t u = (int32_t)U[j] - 128, v = (int32_t)V[j] - 128;
        const int32_t bu = (1 << 19) + 2116026 * u, gu = (1 << 19) - 409993 * u - 852492 * v, rv = (1 << 19) + 1673527 * v;
#pragma unroll
        for (int e = 0; e < 2; e++) {
            const int32_t y = max((int32_t)Y[2 * j + e] - 16, 0) * 1220542;
            const int b = 6 * j + 3 * e; // byte index of the pixel's B
            out[b >> 2] |= clamp_u8((y + bu) >> 20) << (8 * (b & 3));
            out[(b + 1) >> 2] |= clamp_u8((y + gu) >> 20) << (8 * ((b + 1) & 3));
            out[(b + 2) >> 2] |= clamp_u8((y + rv) >> 20) << (8 * ((b + 2) & 3));
        }
    }

    uint8_t *dst = p.bgr + ((size_t)row * (size_t)p.width + (size_t)x0) * 3;
    if (npx == kYuvPixels && (reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
        uint4 *d4 = reinterpret_cast<uint4 *>(dst);
        d4[0] = make_uint4(out[0], out[1], out[2], out[3]);
        d4[1] = make_uint4(out[4], out[5], out[6], out[7]);
        d4[2] = make_uint4(out[8], out[9], out[10], out[11]);
    } else {
        const int nb = 3 * npx;
#pragma unroll
        for (int i = 0; i < 3 * kYuvPixels; i++)
            if (i < nb) dst[i] = (uint8_t)byte_of(out[i >> 2], i & 3);
    }
}

} // namespace cvs
