/* jpeg_oracle.c -- CPU restatement of the capture-side decode.  TEST INFRASTRUCTURE ONLY (see cvs_oracle.c).
 *
 * The reference's capture thread asks the camera for MJPG and lets OpenCV decode every frame into the BGR24 buffer the
 * hot path consumes (server/src/threads.cpp:32-41: CAP_PROP_FOURCC 'MJPG' ... cap >> frame; the test programs read the
 * fixture frames the same way, tests/noise_filter_benchmark/v2.cu:195-198 imread("f1.jpg")).  The arithmetic therefore
 * lives in a third-party dependency that is not in /root/reference: OpenCV's bundled libjpeg-turbo (this image:
 * opencv-python 4.13.0 -> libjpeg-turbo 3.x; the arithmetic below has been unchanged since libjpeg 6b).  This file
 * restates the published algorithm of its default decompression path for baseline JPEG:
 *
 *   jdhuff.c   decode_mcu            Huffman decoding of an interleaved scan, DC prediction, restart intervals
 *   jpeg_idct_islow                  dequantisation + accurate integer IDCT (JDCT_ISLOW, the default) and output range
 *                                    limit, as x86-64 runs it: the SIMD code simd/x86_64/jidctint-avx2.asm, which is
 *                                    OpenCV's path (16-bit lanes: wrapping dequantisation, saturating passes), not
 *                                    jidctint.c, whose int32 arithmetic and x & 1023 range limit differ once
 *                                    dequantised coefficients leave 16 bits
 *   jdsample.c h2v1/h2v2_fancy_upsample  "fancy" (triangle filter) chroma upsampling (do_fancy_upsampling = TRUE),
 *   jdmainct.c                       with the context rows at the top / bottom of the image replicated
 *   jdcolor.c  ycc_rgb_convert       fixed-point YCbCr -> RGB tables, stored B, G, R (OpenCV's channel order)
 *
 * PINNED: tests/test_jpeg_oracle.py compares it byte for byte with cv2.imread on the reference's own camera frames
 * (digests in tests/golden/k1_f1_f2.json, made by tests/golden/make_golden.py from the reference's files) and on
 * re-encodings at other qualities / samplings / sizes / restart intervals (tests/golden/jpeg_cases.npz, made by
 * tests/golden/make_jpeg_cases.py with cv2 in the build container); tests/test_jpeg_coefficient_range.py does the same on
 * streams designed to reach the edges of the coefficient range.
 *
 * Scope: baseline sequential DCT (SOF0), 8 bit, Huffman, one interleaved scan, 3 components Y Cb Cr with luma sampling
 * 1x1, 2x1 or 2x2 and chroma 1x1 (what UVC cameras and cv2.imwrite produce), or 1 component (gray, replicated to B=G=R).
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define ORC_API __attribute__((visibility("default")))

typedef struct {
    uint8_t bits[17];
    uint8_t vals[256];
    /* jdhuff.c jpeg_make_d_derived_tbl: canonical code tables */
    int mincode[17], maxcode[18], valptr[17];
    int present;
} huff_t;

typedef struct {
    int width, height, ncomp;
    int hs[3], vs[3], tq[3], td[3], ta[3], cid[3];
    uint16_t q[4][64]; /* in zig-zag order as transmitted */
    int qpresent[4];
    huff_t dc[4], ac[4];
    int restart_interval;
    const uint8_t *scan;
    size_t scan_len;
} jpg_t;

static const uint8_t zigzag_natural[64 + 16] = {
    0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6,  7,  14, 21, 28,
    35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63,
    63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63 /* jutils.c: extra entries for safety */
};

/* ITU-T T.81 Annex K.3 (the tables a camera's MJPG frame implies when it carries no DHT segment; libjpeg-turbo jstdhuff.c) */
static const uint8_t std_dc_lum_bits[17] = {
    0x00, 0x00, 0x01, 0x05, 0x01, 0x01, 0x01, 0x01, 0x01, 0x01, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00, 0x00,
};
static const uint8_t std_dc_lum_vals[12] = {
    0x00, 0x01, 0x02, 0x03, 0x04, 0x05, 0x06, 0x07, 0x08, 0x09, 0x0a, 0x0b,
};
static const uint8_t std_dc_chrom_bits[17] = {
    0x00, 0x00, 0x03, 0x01, 0x01, 0x01, 0x01, 0x01, 0x01, 0x01, 0x01, 0x01, 0x00, 0x00, 0x00, 0x00, 0x00,
};
static const uint8_t std_dc_chrom_vals[12] = {
    0x00, 0x01, 0x02, 0x03, 0x04, 0x05, 0x06, 0x07, 0x08, 0x09, 0x0a, 0x0b,
};
static const uint8_t std_ac_lum_bits[17] = {
    0x00, 0x00, 0x02, 0x01, 0x03, 0x03, 0x02, 0x04, 0x03, 0x05, 0x05, 0x04, 0x04, 0x00, 0x00, 0x01, 0x7d,
};
static const uint8_t std_ac_lum_vals[162] = {
    0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71, 0x14, 0x32, 0x81, 0x91, 0xa1, 0x08,
    0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72, 0x82, 0x09, 0x0a, 0x16, 0x17, 0x18, 0x19, 0x1a, 0x25, 0x26, 0x27, 0x28,
    0x29, 0x2a, 0x34, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59,
    0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89,
    0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6,
    0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2,
    0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa,
};
static const uint8_t std_ac_chrom_bits[17] = {
    0x00, 0x00, 0x02, 0x01, 0x02, 0x04, 0x04, 0x03, 0x04, 0x07, 0x05, 0x04, 0x04, 0x00, 0x01, 0x02, 0x77,
};
static const uint8_t std_ac_chrom_vals[162] = {
    0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22, 0x32, 0x81, 0x08, 0x14, 0x42, 0x91,
    0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1, 0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25, 0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26,
    0x27, 0x28, 0x29, 0x2a, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58,
    0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x82, 0x83, 0x84, 0x85, 0x86, 0x87,
    0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4,
    0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda,
    0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa,
};

static void derive(huff_t *h)
{
    int code = 0, k = 0;
    for (int l = 1; l <= 16; l++) {
        h->valptr[l] = k;
        h->mincode[l] = code;
        code += h->bits[l];
        k += h->bits[l];
        h->maxcode[l] = h->bits[l] ? code - 1 : -1;
        code <<= 1;
    }
    h->maxcode[17] = 0x7fffffff;
}

static int parse(const uint8_t *d, size_t n, jpg_t *j)
{
    memset(j, 0, sizeof *j);
    if (n < 4 || d[0] != 0xFF || d[1] != 0xD8) return -1;
    /* a scan whose Huffman tables were never defined uses the standard ones (libjpeg-turbo jdhuff.c / jstdhuff.c:
     * MJPG frames of cameras carry no DHT segment): table 0 = luminance, 1 = chrominance */
    {
        const uint8_t *sb[2][2] = {{std_dc_lum_bits, std_dc_chrom_bits}, {std_ac_lum_bits, std_ac_chrom_bits}};
        const uint8_t *sv[2][2] = {{std_dc_lum_vals, std_dc_chrom_vals}, {std_ac_lum_vals, std_ac_chrom_vals}};
        const size_t sn[2][2] = {{sizeof std_dc_lum_vals, sizeof std_dc_chrom_vals}, {sizeof std_ac_lum_vals, sizeof std_ac_chrom_vals}};
        for (int tc = 0; tc < 2; tc++)
            for (int th = 0; th < 2; th++) {
                huff_t *h = tc ? &j->ac[th] : &j->dc[th];
                memcpy(h->bits, sb[tc][th], 17);
                memcpy(h->vals, sv[tc][th], sn[tc][th]);
                derive(h);
                h->present = 1;
            }
    }
    size_t i = 2;
    int sof = 0;
    while (i + 4 <= n) {
        if (d[i] != 0xFF) return -2;
        while (i < n && d[i] == 0xFF) i++; /* fill bytes */
        if (i >= n) return -2;
        const int m = d[i++];
        if (m == 0xD8 || (m >= 0xD0 && m <= 0xD7) || m == 0x01) continue;
        if (m == 0xD9) return -3;
        if (i + 2 > n) return -2;
        const size_t L = ((size_t)d[i] << 8) | d[i + 1];
        if (L < 2 || i + L > n) return -2;
        const uint8_t *p = d + i + 2;
        const size_t pl = L - 2;
        if (m == 0xDB) {
            size_t o = 0;
            while (o < pl) {
                const int pq = p[o] >> 4, tq = p[o] & 15;
                o++;
                if (tq > 3) return -4;
                if (o + (pq ? 128 : 64) > pl) return -4;
                for (int k = 0; k < 64; k++) {
                    j->q[tq][k] = pq ? (uint16_t)((p[o] << 8) | p[o + 1]) : p[o];
                    o += pq ? 2 : 1;
                }
                j->qpresent[tq] = 1;
            }
        } else if (m == 0xC4) {
            size_t o = 0;
            while (o < pl) {
                if (o + 17 > pl) return -5;
                const int tc = p[o] >> 4, th = p[o] & 15;
                if (tc > 1 || th > 3) return -5;
                huff_t *h = tc ? &j->ac[th] : &j->dc[th];
                int cnt = 0;
                h->bits[0] = 0;
                for (int l = 1; l <= 16; l++) {
                    h->bits[l] = p[o + l];
                    cnt += p[o + l];
                }
                o += 17;
                if (cnt > 256 || o + (size_t)cnt > pl) return -5;
                memcpy(h->vals, p + o, (size_t)cnt);
                o += (size_t)cnt;
                derive(h);
                h->present = 1;
            }
        } else if (m == 0xC0 || m == 0xC1) {
            if (pl < 6 || p[0] != 8) return -6;
            j->height = (p[1] << 8) | p[2];
            j->width = (p[3] << 8) | p[4];
            j->ncomp = p[5];
            if ((j->ncomp != 3 && j->ncomp != 1) || pl < 6 + 3 * (size_t)j->ncomp) return -6;
            for (int c = 0; c < j->ncomp; c++) {
                j->cid[c] = p[6 + 3 * c];
                j->hs[c] = p[7 + 3 * c] >> 4;
                j->vs[c] = p[7 + 3 * c] & 15;
                j->tq[c] = p[8 + 3 * c];
                if (j->tq[c] > 3) return -6;
            }
            sof = 1;
        } else if (m == 0xC2 || (m >= 0xC3 && m <= 0xCF && m != 0xC4 && m != 0xC8 && m != 0xCC)) {
            return -7; /* progressive, lossless, arithmetic: not the camera's format */
        } else if (m == 0xDD) {
            if (pl < 2) return -8;
            j->restart_interval = (p[0] << 8) | p[1];
        } else if (m == 0xDA) {
            if (!sof || pl < 1 || p[0] != j->ncomp || pl < 1 + 2 * (size_t)j->ncomp + 3) return -9;
            for (int c = 0; c < j->ncomp; c++) {
                if (p[1 + 2 * c] != j->cid[c]) return -9; /* scan components in another order: not covered */
                j->td[c] = p[2 + 2 * c] >> 4;
                j->ta[c] = p[2 + 2 * c] & 15;
                if (j->td[c] > 3 || j->ta[c] > 3) return -9;
            }
            j->scan = d + i + L;
            j->scan_len = n - (i + L);
            break;
        }
        i += L;
    }
    if (!j->scan || j->width <= 0 || j->height <= 0) return -10;
    if (j->ncomp == 3) {
        if (j->hs[1] != 1 || j->vs[1] != 1 || j->hs[2] != 1 || j->vs[2] != 1) return -11;
        if (!((j->hs[0] == 1 && j->vs[0] == 1) || (j->hs[0] == 2 && j->vs[0] == 1) || (j->hs[0] == 2 && j->vs[0] == 2))) return -11;
    } else {
        j->hs[0] = j->vs[0] = 1; /* a single-component scan is never interleaved: one block per MCU */
    }
    for (int c = 0; c < j->ncomp; c++)
        if (!j->qpresent[j->tq[c]] || !j->dc[j->td[c]].present || !j->ac[j->ta[c]].present) return -12;
    return 0;
}

/* ---- bit reader over the entropy-coded segment: FF 00 -> FF, markers stop the stream (zeros are fed, as jdhuff.c's
 *      jpeg_fill_bit_buffer does after "no_more_bytes") ---------------------------------------------------------------- */
typedef struct {
    const uint8_t *p, *end;
    uint32_t acc;
    int nbits;
    int hit_marker;
} bits_t;

static void fill(bits_t *b)
{
    while (b->nbits <= 24) {
        int c = 0;
        if (!b->hit_marker && b->p < b->end) {
            c = *b->p;
            if (c == 0xFF) {
                if (b->p + 1 < b->end && b->p[1] == 0x00) {
                    b->p += 2;
                } else {
                    b->hit_marker = 1; /* leave the marker in place */
                    c = 0;
                }
            } else {
                b->p++;
            }
        }
        b->acc |= (uint32_t)c << (24 - b->nbits);
        b->nbits += 8;
    }
}
static int getbits(bits_t *b, int n)
{
    if (n == 0) return 0;
    fill(b);
    const int v = (int)(b->acc >> (32 - n));
    b->acc <<= n;
    b->nbits -= n;
    return v;
}
static int decode_sym(bits_t *b, const huff_t *h)
{
    /* jdhuff.c jpeg_huff_decode: extend the code bit by bit until it is <= maxcode[l] */
    int l = 1;
    int code = getbits(b, 1);
    while (l <= 16 && code > h->maxcode[l]) {
        code = (code << 1) | getbits(b, 1);
        l++;
    }
    if (l > 16) return 0; /* "Corrupt JPEG data: bad Huffman code": libjpeg uses a zero symbol */
    return h->vals[(h->valptr[l] + code - h->mincode[l]) & 255];
}
/* HUFF_EXTEND (jdhuff.c): value of an s-bit magnitude-coded number */
static int extend(int x, int s) { return x < (1 << (s - 1)) ? x + (int)((~0u) << s) + 1 : x; }

/* ---- coefficients of every block, in scan order (MCU by MCU; inside an MCU: hs*vs luma blocks row by row, Cb, Cr),
 *      natural (row-major) order inside a block, DC prediction resolved ----------------------------------------------- */
static int decode_coefficients(const jpg_t *j, int16_t *coef, size_t nblocks_total)
{
    const int mcux = (j->width + 8 * j->hs[0] - 1) / (8 * j->hs[0]), mcuy = (j->height + 8 * j->vs[0] - 1) / (8 * j->vs[0]);
    const int bpm = j->hs[0] * j->vs[0] + (j->ncomp == 3 ? 2 : 0);
    if ((size_t)mcux * mcuy * bpm != nblocks_total) return -20;
    memset(coef, 0, nblocks_total * 64 * sizeof(int16_t));
    bits_t b = {j->scan, j->scan + j->scan_len, 0, 0, 0};
    int pred[3] = {0, 0, 0};
    int togo = j->restart_interval;
    size_t blk = 0;
    for (int m = 0; m < mcux * mcuy; m++) {
        if (j->restart_interval && togo == 0) {
            /* process_restart: drop the partial byte, skip to and over the RSTn marker, reset the predictors */
            b.acc = 0;
            b.nbits = 0;
            b.hit_marker = 0;
            while (b.p + 1 < b.end && !(b.p[0] == 0xFF && b.p[1] >= 0xD0 && b.p[1] <= 0xD7)) b.p++;
            if (b.p + 1 < b.end) b.p += 2;
            pred[0] = pred[1] = pred[2] = 0;
            togo = j->restart_interval;
        }
        for (int bi = 0; bi < bpm; bi++, blk++) {
            const int c = (j->ncomp == 1) ? 0 : (bi < bpm - 2 ? 0 : bi - (bpm - 2) + 1);
            const huff_t *dc = &j->dc[j->td[c]], *ac = &j->ac[j->ta[c]];
            int16_t *out = coef + blk * 64;
            int s = decode_sym(&b, dc);
            int diff = 0;
            if (s) {
                s &= 15; /* baseline: 0..11 */
                diff = extend(getbits(&b, s), s);
            }
            pred[c] += diff;
            out[0] = (int16_t)pred[c];
            for (int k = 1; k < 64; k++) {
                const int rs = decode_sym(&b, ac);
                const int r = rs >> 4, sz = rs & 15;
                if (sz) {
                    k += r;
                    const int v = extend(getbits(&b, sz), sz);
                    out[zigzag_natural[k]] = (int16_t)v; /* k <= 63 + 15: inside the padded table */
                } else {
                    if (r != 15) break;
                    k += 15;
                }
            }
        }
        togo--;
    }
    return 0;
}

/* ---- jpeg_idct_islow as libjpeg-turbo runs it on x86-64: simd/x86_64/jidctint-avx2.asm (jsimd_idct_islow_avx2, the
 *      path OpenCV's bundled libjpeg-turbo takes on an AVX2 CPU).  jidctint.c's algorithm in 16-bit lanes, which differs
 *      from the C code only where values leave 16 bits -- large dequantised coefficients:
 *        - dequantisation is pmullw: coef * q wrapped to int16;
 *        - the sums in0+in4, in0-in4 (even part) and in7+in3, in5+in1 (odd part's z3, z4) are paddw / psubw: wrapped to
 *          int16; every other product and sum is a pmaddwd / paddd in 32 bits, where no value of these inputs overflows;
 *        - pass 1 descales and packs with packssdw: saturated to int16;
 *        - a block whose coefficient rows 1..7 are all zero skips pass 1: every row of the workspace is the dequantised
 *          row 0 shifted left by PASS1_BITS with psllw (wrapped to int16, not saturated);
 *        - pass 2 descales, packs with packssdw and packsswb (saturated to -128..127) and adds CENTERJSAMPLE with paddb.
 *      tests/test_jpeg_coefficient_range.py states these rules in a Python reference and checks them against cv2. */
#define CONST_BITS 13
#define PASS1_BITS 2
#define DESCALE(x, n) (((x) + ((int32_t)1 << ((n)-1))) >> (n))
/* the pmaddwd constant pairs of the asm (PW_F130_F054, PW_F054_MF130, PW_MF078_F117, PW_F117_F078, PW_MF060_MF089,
 * PW_MF089_F060, PW_MF050_MF256, PW_MF256_F050): sums and differences of jidctint.c's FIX_x values */
#define F_0_541 4433                 /* FIX_0_541196100 */
#define F_1_306 (4433 + 6270)        /* FIX_0_541196100 + FIX_0_765366865 */
#define F_M1_306 (4433 - 15137)      /* FIX_0_541196100 - FIX_1_847759065 */
#define F_1_175 9633                 /* FIX_1_175875602 */
#define F_M0_785 (9633 - 16069)      /* FIX_1_175875602 - FIX_1_961570560 */
#define F_0_785 (9633 - 3196)        /* FIX_1_175875602 - FIX_0_390180644 */
#define F_M0_899 (-7373)             /* -FIX_0_899976223 */
#define F_M0_601 (2446 - 7373)       /* FIX_0_298631336 - FIX_0_899976223 */
#define F_0_601 (12299 - 7373)       /* FIX_1_501321110 - FIX_0_899976223 */
#define F_M2_562 (-20995)            /* -FIX_2_562915447 */
#define F_M0_509 (16819 - 20995)     /* FIX_2_053119869 - FIX_2_562915447 */
#define F_0_509 (25172 - 20995)      /* FIX_3_072711026 - FIX_2_562915447 */

static int32_t wrap16(int32_t x) { return (int32_t)(int16_t)(uint16_t)(uint32_t)x; }
static int16_t sat16(int32_t x) { return (int16_t)(x < -32768 ? -32768 : (x > 32767 ? 32767 : x)); }

/* one 1-D pass over eight int16 inputs, undescaled: out[0..7] as jidctint.c's tmp10+tmp3 ... tmp10-tmp3 */
static void idct8_simd(const int16_t *in, int32_t *out)
{
    /* even part: tmp3 = z2 * (0.541 + 0.765) + z3 * 0.541, tmp2 = z2 * 0.541 + z3 * (0.541 - 1.848) */
    const int32_t tmp3 = in[2] * F_1_306 + in[6] * F_0_541, tmp2 = in[2] * F_0_541 + in[6] * F_M1_306;
    const int32_t tmp0 = wrap16(in[0] + in[4]) * (1 << CONST_BITS), tmp1 = wrap16(in[0] - in[4]) * (1 << CONST_BITS);
    const int32_t tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    /* odd part: z3 = in7 + in3, z4 = in5 + in1 in 16 bits; z5 folded into the pmaddwd constants */
    const int32_t z3 = wrap16(in[7] + in[3]), z4 = wrap16(in[5] + in[1]);
    const int32_t Z3 = z3 * F_M0_785 + z4 * F_1_175, Z4 = z3 * F_1_175 + z4 * F_0_785;
    const int32_t o0 = in[7] * F_M0_601 + in[1] * F_M0_899 + Z3, o3 = in[7] * F_M0_899 + in[1] * F_0_601 + Z4;
    const int32_t o1 = in[5] * F_M0_509 + in[3] * F_M2_562 + Z4, o2 = in[5] * F_M2_562 + in[3] * F_0_509 + Z3;
    out[0] = tmp10 + o3;
    out[7] = tmp10 - o3;
    out[1] = tmp11 + o2;
    out[6] = tmp11 - o2;
    out[2] = tmp12 + o1;
    out[5] = tmp12 - o1;
    out[3] = tmp13 + o0;
    out[4] = tmp13 - o0;
}

static void idct_islow(const int16_t *in, const uint16_t *qzz, uint8_t *out, size_t pitch)
{
    int16_t dq[64], ws[64];
    int rows_zero = 1;
    for (int k = 0; k < 64; k++) dq[zigzag_natural[k]] = (int16_t)wrap16(in[zigzag_natural[k]] * (int32_t)qzz[k]);
    for (int k = 8; k < 64; k++) rows_zero &= in[k] == 0; /* tested on the quantised coefficients, before pmullw */
    for (int c = 0; c < 8; c++) {
        int16_t col[8];
        int32_t o[8];
        if (rows_zero) {
            for (int r = 0; r < 8; r++) ws[8 * r + c] = (int16_t)wrap16(dq[c] * (1 << PASS1_BITS));
            continue;
        }
        for (int r = 0; r < 8; r++) col[r] = dq[8 * r + c];
        idct8_simd(col, o);
        for (int r = 0; r < 8; r++) ws[8 * r + c] = sat16(DESCALE(o[r], CONST_BITS - PASS1_BITS));
    }
    for (int r = 0; r < 8; r++) {
        int32_t o[8];
        idct8_simd(ws + 8 * r, o);
        for (int c = 0; c < 8; c++) {
            const int32_t v = DESCALE(o[c], CONST_BITS + PASS1_BITS + 3);
            out[(size_t)r * pitch + c] = (uint8_t)((v < -128 ? -128 : (v > 127 ? 127 : v)) + 128);
        }
    }
}

static uint8_t clamp255(int v) { return (uint8_t)(v < 0 ? 0 : (v > 255 ? 255 : v)); }

/* ---- the planes: luma at full resolution, chroma at its own; blocks land where their MCU puts them ------------------ */
typedef struct {
    uint8_t *y, *cb, *cr;
    int yw, yh, cw, ch; /* padded plane sizes (multiples of the MCU) */
} planes_t;

static void planes_free(planes_t *p)
{
    free(p->y);
    free(p->cb);
    free(p->cr);
}

/* geometry of the scan; exported so that tests can size buffers */
ORC_API int orc_jpeg_info(const uint8_t *jpg, size_t n, int *width, int *height, int *hs, int *vs, int *ncomp, int *restart_interval,
                          long *nblocks)
{
    jpg_t j;
    const int e = parse(jpg, n, &j);
    if (e) return e;
    const int mcux = (j.width + 8 * j.hs[0] - 1) / (8 * j.hs[0]), mcuy = (j.height + 8 * j.vs[0] - 1) / (8 * j.vs[0]);
    *width = j.width;
    *height = j.height;
    *hs = j.hs[0];
    *vs = j.vs[0];
    *ncomp = j.ncomp;
    *restart_interval = j.restart_interval;
    *nblocks = (long)mcux * mcuy * (j.hs[0] * j.vs[0] + (j.ncomp == 3 ? 2 : 0));
    return 0;
}

/* coefficients in scan order, natural order inside the block, DC absolute (what the GPU entropy stage must produce) */
ORC_API int orc_jpeg_coefficients(const uint8_t *jpg, size_t n, int16_t *coef, long nblocks)
{
    jpg_t j;
    const int e = parse(jpg, n, &j);
    if (e) return e;
    return decode_coefficients(&j, coef, (size_t)nblocks);
}

/* the whole decode: BGR24, width*height*3 bytes, rows top to bottom (what cv2.imread / VideoCapture hand over) */
ORC_API int orc_jpeg_decode_bgr(const uint8_t *jpg, size_t n, uint8_t *bgr, int width, int height)
{
    jpg_t j;
    int e = parse(jpg, n, &j);
    if (e) return e;
    if (j.width != width || j.height != height) return -30;
    const int H = j.hs[0], V = j.vs[0];
    const int mcux = (j.width + 8 * H - 1) / (8 * H), mcuy = (j.height + 8 * V - 1) / (8 * V);
    const int bpm = H * V + (j.ncomp == 3 ? 2 : 0);
    const size_t nblocks = (size_t)mcux * mcuy * bpm;
    int16_t *coef = (int16_t *)malloc(nblocks * 64 * sizeof(int16_t));
    if (!coef) return -31;
    e = decode_coefficients(&j, coef, nblocks);
    if (e) {
        free(coef);
        return e;
    }
    planes_t P;
    P.yw = mcux * 8 * H;
    P.yh = mcuy * 8 * V;
    P.cw = mcux * 8;
    P.ch = mcuy * 8;
    P.y = (uint8_t *)malloc((size_t)P.yw * P.yh);
    P.cb = (uint8_t *)malloc((size_t)P.cw * P.ch);
    P.cr = (uint8_t *)malloc((size_t)P.cw * P.ch);
    size_t blk = 0;
    for (int my = 0; my < mcuy; my++)
        for (int mx = 0; mx < mcux; mx++) {
            for (int v = 0; v < V; v++)
                for (int h = 0; h < H; h++, blk++)
                    idct_islow(coef + blk * 64, j.q[j.tq[0]], P.y + (size_t)(my * V + v) * 8 * P.yw + (size_t)(mx * H + h) * 8, (size_t)P.yw);
            if (j.ncomp == 3) {
                idct_islow(coef + blk * 64, j.q[j.tq[1]], P.cb + (size_t)my * 8 * P.cw + (size_t)mx * 8, (size_t)P.cw);
                blk++;
                idct_islow(coef + blk * 64, j.q[j.tq[2]], P.cr + (size_t)my * 8 * P.cw + (size_t)mx * 8, (size_t)P.cw);
                blk++;
            }
        }
    free(coef);
    if (j.ncomp == 1) {
        for (int y = 0; y < height; y++)
            for (int x = 0; x < width; x++) {
                const uint8_t g = P.y[(size_t)y * P.yw + x];
                uint8_t *o = bgr + ((size_t)y * width + x) * 3;
                o[0] = o[1] = o[2] = g;
            }
        planes_free(&P);
        return 0;
    }
    /* jdcolor.c build_ycc_rgb_table */
    int cr_r[256], cb_b[256];
    int32_t cr_g[256], cb_g[256];
    for (int i = 0, x = -128; i < 256; i++, x++) {
        cr_r[i] = (int)((91881 * (int32_t)x + 32768) >> 16);  /* FIX(1.40200) */
        cb_b[i] = (int)((116130 * (int32_t)x + 32768) >> 16); /* FIX(1.77200) */
        cr_g[i] = -46802 * (int32_t)x;                        /* FIX(0.71414) */
        cb_g[i] = -22554 * (int32_t)x + 32768;                /* FIX(0.34414) + ONE_HALF */
    }
    /* real (downsampled) chroma size: jdmaster.c / jdinput.c downsampled_width = ceil(width * h_samp / max_h_samp) */
    const int dw = (width + H - 1) / H, dh = (height + V - 1) / V;
    uint8_t *ub = (uint8_t *)malloc((size_t)2 * width + 4), *ur = ub + width + 2;
    for (int y = 0; y < height; y++) {
        /* upsampled chroma of this row */
        for (int pl = 0; pl < 2; pl++) {
            const uint8_t *src = pl ? P.cr : P.cb;
            uint8_t *dst = pl ? ur : ub;
            if (H == 1 && V == 1) {
                memcpy(dst, src + (size_t)y * P.cw, (size_t)width);
            } else if (H == 2 && V == 1) {
                const uint8_t *in = src + (size_t)y * P.cw;
                if (dw > 2) { /* h2v1_fancy_upsample */
                    for (int c = 0; c < dw; c++) {
                        const int v = in[c];
                        if (2 * c < width) dst[2 * c] = (uint8_t)(c == 0 ? v : (3 * v + in[c - 1] + 1) >> 2);
                        if (2 * c + 1 < width) dst[2 * c + 1] = (uint8_t)(c == dw - 1 ? v : (3 * v + in[c + 1] + 2) >> 2);
                    }
                } else { /* h2v1_upsample */
                    for (int x = 0; x < width; x++) dst[x] = in[x >> 1];
                }
            } else { /* H == 2, V == 2 */
                const int r = y >> 1;
                if (dw > 2) { /* h2v2_fancy_upsample; context rows replicated at the image border (jdmainct.c) */
                    int rn = (y & 1) ? r + 1 : r - 1;
                    if (rn < 0) rn = 0;
                    if (rn > dh - 1) rn = dh - 1;
                    const uint8_t *in0 = src + (size_t)r * P.cw, *in1 = src + (size_t)rn * P.cw;
                    for (int c = 0; c < dw; c++) {
                        const int t = 3 * in0[c] + in1[c];
                        const int l = c > 0 ? 3 * in0[c - 1] + in1[c - 1] : 0, nx = c < dw - 1 ? 3 * in0[c + 1] + in1[c + 1] : 0;
                        if (2 * c < width) dst[2 * c] = (uint8_t)(c == 0 ? (4 * t + 8) >> 4 : (3 * t + l + 8) >> 4);
                        if (2 * c + 1 < width) dst[2 * c + 1] = (uint8_t)(c == dw - 1 ? (4 * t + 7) >> 4 : (3 * t + nx + 7) >> 4);
                    }
                } else { /* h2v2_upsample */
                    for (int x = 0; x < width; x++) dst[x] = src[(size_t)r * P.cw + (x >> 1)];
                }
            }
        }
        for (int x = 0; x < width; x++) {
            const int yy = P.y[(size_t)y * P.yw + x], cb = ub[x], cr = ur[x];
            uint8_t *o = bgr + ((size_t)y * width + x) * 3;
            o[2] = clamp255(yy + cr_r[cr]);
            o[1] = clamp255(yy + (int)((cb_g[cb] + cr_g[cr]) >> 16));
            o[0] = clamp255(yy + cb_b[cb]);
        }
    }
    free(ub);
    planes_free(&P);
    return 0;
}
