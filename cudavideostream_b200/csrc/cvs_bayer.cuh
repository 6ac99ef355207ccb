// cvs_bayer.cuh -- raw 8-bit Bayer mosaic (BGGR, GBRG, GRBG, RGGB) -> packed BGR24 with OpenCV's pixels
// (cv2.cvtColor COLOR_Bayer<P>2BGR, the default bilinear demosaic).
//
// OpenCV's rule, integer only (matched byte for byte, tests/test_bayer_oracle.py):
//     W < 3 or H < 3: all zero; otherwise out(y, x) = I(clamp(y, 1, H-2), clamp(x, 1, W-2)) where, at an interior
//     pixel whose mosaic colour is c:
//       channel c = raw[y][x];
//       c = G:      horizontal neighbours' colour = (left + right + 1) >> 1, vertical neighbours' = (up + down + 1) >> 1;
//       c = R or B: G = (left + right + up + down + 2) >> 2, the opposite colour = (four diagonals + 2) >> 2.
// The pattern is a parity offset: P at (y, x) is BGGR at (y + py, x + px).
#pragma once
#include "cvs_pixel.cuh"

namespace cvs {

struct BayerParams {
    const uint8_t *raw; // width * height mosaic bytes, rows `pitch` bytes apart
    size_t pitch;
    uint8_t *bgr;       // 3 * width * height bytes, rows contiguous
    int width, height;  // any positive size
    uint32_t groups;    // 16-pixel groups per row: (width + 15) / 16
    int py, px;         // the pattern's offset into BGGR
};

constexpr int kBayerThreads = 256;
constexpr int kBayerPixels = 16; // pixels per thread: one 16-byte load per source row, three 16-byte BGR stores

// (a + b + c + d + 2) >> 2 per byte: the sums need 10 bits, so even and odd bytes go through 16-bit lanes apart
__device__ __forceinline__ uint32_t avg4_u8(uint32_t a, uint32_t b, uint32_t c, uint32_t d)
{
    constexpr uint32_t K = 0x00ff00ffu;
    const uint32_t e = (a & K) + (b & K) + (c & K) + (d & K) + 0x00020002u;
    const uint32_t o = ((a >> 8) & K) + ((b >> 8) & K) + ((c >> 8) & K) + ((d >> 8) & K) + 0x00020002u;
    return ((e >> 2) & K) | ((o << 6) & ~K);
}

// One thread = 16 horizontally adjacent output pixels of row y, whose interior values centre on source row
// cy = clamp(y, 1, H-2) and read rows cy-1, cy, cy+1.  The arithmetic works on 4 pixels per 32-bit word: l / m / r[row]
// hold the bytes left of, at and right of each pixel's centre column, `colour` marks the bytes whose centre holds the
// row's R or B (the others hold G).
//   Vector path (source rows 16-byte aligned, 16 pixels in the group): one 16-byte load per row gives m; l and r are m
//   shifted by a byte, with the bytes at x0-1 and x0+16 read from L1 (the neighbouring threads' loads brought their
//   lines in).  In the first group of a row pixel 0 replicates column 1, in the last pixel 15 replicates column W-2
//   (a byte permute afterwards; the edge byte read outside the row is clamped into it and never used).
//   Byte path (any other group: a row's partial last group, rows that are not aligned): each pixel's three columns
//   around clamp(x, 1, W-2), one byte load each.
// The 48 output bytes go out as three 16-byte stores where the destination is aligned and the group full, else as bytes;
// nothing outside the 3 * width * height bytes of p.bgr is written.  The stores are plain: in the submit path the
// stream kernel reads the frame right behind, from L2.
__global__ void __launch_bounds__(kBayerThreads) k_bayer_to_bgr(const BayerParams p)
{
    const uint32_t item = blockIdx.x * kBayerThreads + threadIdx.x;
    const uint32_t y = item / p.groups;
    if (y >= (uint32_t)p.height) return;
    const int W = p.width, H = p.height;
    const int x0 = (int)(item - y * p.groups) * kBayerPixels;
    const int npx = min(kBayerPixels, W - x0);

    uint32_t B[4] = {0, 0, 0, 0}, G[4] = {0, 0, 0, 0}, R[4] = {0, 0, 0, 0};
    if (W >= 3 && H >= 3) {
        const int cy = min(max((int)y, 1), H - 2);
        const uint32_t odd_row = (uint32_t)(cy + p.py) & 1u; // 0: the row's colour is B, 1: R
        const uint8_t *src[3];
#pragma unroll
        for (int k = 0; k < 3; k++) src[k] = p.raw + (size_t)(cy - 1 + k) * p.pitch;

        uint32_t l[3][4], m[3][4], r[3][4], colour[4];
        const bool vec = npx == kBayerPixels && ((reinterpret_cast<uintptr_t>(p.raw) | p.pitch) & 15u) == 0;
        if (vec) {
            const int xl = max(x0 - 1, 0), xr = min(x0 + kBayerPixels, W - 1);
#pragma unroll
            for (int k = 0; k < 3; k++) {
                const uint4 v = __ldg(reinterpret_cast<const uint4 *>(src[k] + x0));
                const uint32_t w[6] = {(uint32_t)__ldg(src[k] + xl) << 24, v.x, v.y, v.z, v.w, (uint32_t)__ldg(src[k] + xr)};
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    m[k][j] = w[j + 1];
                    l[k][j] = __funnelshift_l(w[j], w[j + 1], 8);
                    r[k][j] = __funnelshift_r(w[j + 1], w[j + 2], 8);
                }
            }
            // x0 is even: the colour bytes are the even ones or the odd ones
            const uint32_t cm = ((odd_row ^ (uint32_t)p.px) & 1u) ? 0xff00ff00u : 0x00ff00ffu;
#pragma unroll
            for (int j = 0; j < 4; j++) colour[j] = cm;
        } else {
#pragma unroll
            for (int j = 0; j < 4; j++) {
                colour[j] = 0;
#pragma unroll
                for (int k = 0; k < 3; k++) l[k][j] = m[k][j] = r[k][j] = 0;
            }
#pragma unroll
            for (int i = 0; i < kBayerPixels; i++) {
                if (i < npx) {
                    const int c = min(max(x0 + i, 1), W - 2);
                    const int s = 8 * (i & 3);
#pragma unroll
                    for (int k = 0; k < 3; k++) {
                        l[k][i >> 2] |= (uint32_t)__ldg(src[k] + c - 1) << s;
                        m[k][i >> 2] |= (uint32_t)__ldg(src[k] + c) << s;
                        r[k][i >> 2] |= (uint32_t)__ldg(src[k] + c + 1) << s;
                    }
                    if ((((uint32_t)(c + p.px)) & 1u) == odd_row) colour[i >> 2] |= 0xffu << s;
                }
            }
        }

#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t hor = __vavgu4(l[1][j], r[1][j]), ver = __vavgu4(m[0][j], m[2][j]);
            const uint32_t cross = avg4_u8(l[1][j], r[1][j], m[0][j], m[2][j]);
            const uint32_t diag = avg4_u8(l[0][j], r[0][j], l[2][j], r[2][j]);
            const uint32_t c = colour[j];
            const uint32_t own = (m[1][j] & c) | (hor & ~c);   // the row's colour (B or R)
            const uint32_t other = (diag & c) | (ver & ~c);    // the other one
            G[j] = (cross & c) | (m[1][j] & ~c);
            B[j] = odd_row ? other : own;
            R[j] = odd_row ? own : other;
        }
        if (vec && x0 == 0) { // out(y, 0) = I(cy, 1)
            B[0] = __byte_perm(B[0], 0u, 0x3211u);
            G[0] = __byte_perm(G[0], 0u, 0x3211u);
            R[0] = __byte_perm(R[0], 0u, 0x3211u);
        }
        if (vec && x0 + kBayerPixels == W) { // out(y, W-1) = I(cy, W-2)
            B[3] = __byte_perm(B[3], 0u, 0x2210u);
            G[3] = __byte_perm(G[3], 0u, 0x2210u);
            R[3] = __byte_perm(R[3], 0u, 0x2210u);
        }
    }

    // B G R per pixel, 4 pixels -> 3 little-endian words
    uint32_t out[12];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        out[3 * j] = __byte_perm(__byte_perm(B[j], G[j], 0x1040u), R[j], 0x3410u);     // b0 g0 r0 b1
        out[3 * j + 1] = __byte_perm(__byte_perm(G[j], R[j], 0x2051u), B[j], 0x3610u); // g1 r1 b2 g2
        out[3 * j + 2] = __byte_perm(__byte_perm(R[j], B[j], 0x3072u), G[j], 0x3710u); // r2 b3 g3 r3
    }

    uint8_t *dst = p.bgr + ((size_t)y * (size_t)W + (size_t)x0) * 3;
    if (npx == kBayerPixels && (reinterpret_cast<uintptr_t>(dst) & 15u) == 0) {
        uint4 *d4 = reinterpret_cast<uint4 *>(dst);
        d4[0] = make_uint4(out[0], out[1], out[2], out[3]);
        d4[1] = make_uint4(out[4], out[5], out[6], out[7]);
        d4[2] = make_uint4(out[8], out[9], out[10], out[11]);
    } else {
        const int nb = 3 * npx;
#pragma unroll
        for (int i = 0; i < 3 * kBayerPixels; i++)
            if (i < nb) dst[i] = (uint8_t)byte_of(out[i >> 2], i & 3);
    }
}

} // namespace cvs
