// cvs_jpeg.cuh -- capture-side decode on the GPU: baseline JPEG (the camera's MJPG frames, server/src/threads.cpp:32-41)
// -> BGR24 frame in device memory, bit for bit what OpenCV's libjpeg-turbo makes of the same bitstream (JDCT_ISLOW,
// fancy chroma upsampling, fixed-point YCbCr -> RGB), i.e. what the reference's hot path is fed.  SURVEY 8(f) row 4.
//
// A camera frame has no restart markers, so its Huffman stream is one sequential dependency chain (432 KB at 1080p).
// It is decoded in parallel through the self-synchronisation of Huffman codes:
//
//   k_entropy (one cooperative launch; phases separated by grid barriers)
//       clear    the scratch that must start as zero; FF 00 -> FF: the entropy-coded segment becomes a plain bit string of
//       unstuff  T bits (16 bytes per thread, kept bytes compacted by a two-level prefix sum)
//       The bit string is cut into subsequences of S = 1,024 bits.  The decoder state at a boundary is (bit offset of the
//       first token that starts behind it, block-in-MCU phase, zig-zag position).  A decoder started in a wrong state falls
//       into step with the true token sequence -- but only once its PHASE is right too, because the luma blocks of an MCU
//       share their tables, and the phase of a wrong guess performs a random walk (13-24 plain rounds on a camera frame).
//       X Y W    so for every boundary and every phase h one thread decodes from "a block of phase h starts here" through
//                three subsequences and notes its state at their ends: 2 * bpm candidate states per boundary
//       maps     at which candidate of boundary i does the sequence through candidate c of boundary i-1 arrive?
//       scan     the true sequence starts at candidate 0 of boundary 0; following it is a prefix scan of map compositions
//       rounds   decode from the entry state, hand the exit state to the successor, whoever received a new state decodes
//                again, until nothing changes: ONE round when the scan found every state (a camera frame; on half
//                subsequences then: the Y / W runs also note their state in the middle), as many as it takes otherwise -- exact states travel one subsequence per round at least, so every stream decodes.
//                A run also leaves the blocks completed, the DC differences summed and its state every 128 bits.
//       sums     exclusive prefix sums give every subsequence its first block index and DC predictors
//       write    one thread per 128 bits decodes once more from its exact state and stores the coefficients
//   k_unstuff_count / k_unstuff_write / k_entropy_restart   scans WITH restart intervals: the markers are dropped with the
//               stuffing, every interval starts in a known state and is decoded by one thread, no synchronisation
//   k_idct      dequantisation + the accurate integer IDCT (jpeg_idct_islow in libjpeg-turbo's x86-64 SIMD form) per
//               8x8 block -> Y / Cb / Cr planes
//   k_colour    jdsample.c's h2v1 / h2v2 "fancy" upsampling (context rows replicated at the border) + jdcolor.c's
//               fixed-point conversion, stored B, G, R
//
// The arithmetic of every stage is integer; tests compare with the CPU oracle (oracle/jpeg_oracle.c, pinned against cv2)
// and with the digests of cv2's pixels of the reference's own camera frames.
//
// The token-level functions are __host__ __device__ so that tests/host/jpeg_sim.cpp can run the very same
// synchronisation logic on the CPU (g++, no GPU).
#pragma once
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define CVS_HD __host__ __device__ __forceinline__
#else
#define CVS_HD inline
#endif

namespace cvs {
namespace jpg {

constexpr int kLutBits = 9;      // first-level look-ahead
constexpr int kLut2Bits = 7;     // second level: the remaining bits of a 16-bit code
constexpr int kLut2Tables = 8;   // second-level tables per Huffman table (the standard tables need 5)
constexpr int kMaxSplit = 8;     // write-pass threads per subsequence
constexpr int kRoundCounters = 4; // per-round change counters in rotation (see k_entropy)

// Canonical Huffman table as the decoder wants it.  A decoded token is one 32-bit entry:
//   bits 0-7 symbol (run << 4 | size), 8-12 code length, 13-18 token length (code + size bits),
//   19-25 advance of the zig-zag position (DC: 1; coefficient: run + 1; ZRL: 16; EOB: 64 = to the end of the block)
// lut[first kLutBits bits] resolves every code of that length or shorter; for a longer code it holds kEntryLevel2 | t and
// lut2[t][next kLut2Bits bits] resolves it; when a table has more than kLut2Tables long prefixes the entry is
// kEntrySlow and maxcode[] is walked as jdhuff.c's slow path does.  Codes that do not exist decode as a zero symbol of
// 16 bits (damaged data; libjpeg warns and uses zero as well).
constexpr uint32_t kEntryLevel2 = 0x80000000u, kEntrySlow = 0x40000000u;
struct HuffDev {
    uint32_t lut[1 << kLutBits];
    uint32_t lut2[kLut2Tables][1 << kLut2Bits];
    int32_t maxcode[17]; // largest code of length l (1..16), -1: none
    int32_t valoff[17];  // valptr[l] - mincode[l]
    uint8_t vals[256];
    uint32_t is_ac;
};
constexpr uint32_t kOffLut2 = sizeof(uint32_t) << kLutBits;
constexpr uint32_t kOffMaxcode = kOffLut2 + sizeof(uint32_t) * kLut2Tables * (1u << kLut2Bits);
constexpr uint32_t kOffValoff = kOffMaxcode + 17 * 4, kOffVals = kOffValoff + 17 * 4, kOffIsAc = kOffVals + 256;
static_assert(sizeof(HuffDev) == kOffIsAc + 4, "HuffDev is addressed by byte offsets");

CVS_HD uint32_t make_entry(uint32_t sym, uint32_t len, uint32_t is_ac)
{
    const uint32_t s = sym & 15u, run = sym >> 4;
    const uint32_t kadd = is_ac ? (s ? run + 1u : (run == 15u ? 16u : 64u)) : 1u;
    return sym | (len << 8) | ((len + s) << 13) | (kadd << 19);
}

struct Tables {
    HuffDev h[3][2];   // per component: [0] DC table, [1] AC table
    uint16_t q[3][64]; // per component: quantisation table in natural (row-major) order
};

// The tables as the token loop reads them: byte offsets from the start of a Tables object -- in shared memory on the
// device (explicit ld.shared: no generic-address arithmetic inside the loop), plain memory in the host build.
struct TableRef {
#if defined(__CUDA_ARCH__)
    uint32_t base;
    __device__ __forceinline__ uint32_t ld32(uint32_t off) const
    {
        uint32_t v;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(base + off));
        return v;
    }
    __device__ __forceinline__ uint32_t ld8(uint32_t off) const
    {
        uint32_t v;
        asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(base + off));
        return v;
    }
#else
    const uint8_t *base;
    uint32_t ld32(uint32_t off) const
    {
        uint32_t v;
        memcpy(&v, base + off, 4);
        return v;
    }
    uint32_t ld8(uint32_t off) const { return base[off]; }
#endif
};

struct Geometry {
    int width, height;   // image
    int H, V;            // luma sampling factors (chroma is 1x1): 1x1, 2x1, 2x2
    int ncomp;           // 3, or 1 (gray: one block per MCU, B = G = R = Y)
    int bpm;             // blocks per MCU: H*V + 2 (or 1)
    int mcux, mcuy;
    uint32_t nblocks;    // mcux * mcuy * bpm
    uint32_t sub_bits;   // S: bits per subsequence (multiple of 32)
    uint32_t nsub_max;   // subsequences the launch covers (from the raw length; the unstuffed string may be shorter)
};

// ---- entry / exit state of a subsequence, packed: bit offset of the first own token (0..31) | phase << 5 | k << 8 -------
CVS_HD uint32_t pack_state(uint32_t off, uint32_t ph, uint32_t k) { return off | (ph << 5) | (k << 8); }
constexpr uint32_t kStateUnset = 0xffffffffu;
constexpr uint32_t kNoCandidate = 15u;

// what one run over a subsequence leaves behind
struct RunResult {
    uint32_t exit_state;
    uint32_t half_state;        // HALF runs: state of the first token that starts in the second half (kStateUnset: none)
    uint32_t nblocks;           // blocks completed by tokens that start in this subsequence
    int32_t dc0, dc1, dc2;      // DC differences decoded in this subsequence, per component
};

CVS_HD uint32_t bswap32(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return __byte_perm(x, 0u, 0x0123u);
#else
    return __builtin_bswap32(x);
#endif
}

CVS_HD TableRef table_ref(const Tables *t) // device: t lives in shared memory
{
    TableRef r;
#if defined(__CUDA_ARCH__)
    r.base = (uint32_t)__cvta_generic_to_shared(t);
#else
    r.base = reinterpret_cast<const uint8_t *>(t);
#endif
    return r;
}

// 32 bits of the unstuffed string starting at bit p (big-endian bit order).  Held: the two words under the window, the
// one behind them, and the one behind that as it was loaded an iteration (or more) ago -- every call issues the load of
// word (p >> 5) + 3 and nobody reads its result before a later call, so a warp (which issues in order and waits at the
// first instruction that reads a loaded register) never waits for memory on the token chain.
// p may advance by at most 31 bits between two calls (a token is at most 16 + 15 bits long).
// (Measured and not adopted: the window as a 64-bit shift register that is shifted by the token length and refilled by
//  OR -- no selects between table entry and next window -- together with an 11-bit first-level table: X / Y / W phases
//  136 us instead of 123 us, 335 us instead of 317 us per frame.  A phase lasts as long as its slowest subsequence
//  (286 tokens in 1,024 bits against a mean of 120), i.e. ~50 dependent instructions per token on a warp that runs
//  alone on its scheduler; the look-up chain is not what it waits for.)
struct BitWindow {
    const uint32_t *words;
    uint32_t widx, hi, lo, n1, q; // n1 = word widx + 2 (as loaded), q = word widx + 3 (as loaded, possibly still in flight)
    CVS_HD void init(const uint32_t *w, uint32_t p)
    {
        words = w;
        widx = p >> 5;
        hi = bswap32(words[widx]);
        lo = bswap32(words[widx + 1]);
        n1 = words[widx + 2];
        q = words[widx + 3];
    }
    CVS_HD uint32_t peek(uint32_t p)
    {
        const uint32_t wi = p >> 5;
        const bool adv = wi != widx;
        hi = adv ? lo : hi;
        lo = adv ? bswap32(n1) : lo;
        n1 = adv ? q : n1;
        widx = wi;
        q = words[wi + 3];
        const uint32_t s = p & 31u;
#if defined(__CUDA_ARCH__)
        return __funnelshift_l(lo, hi, s);
#else
        return s ? ((hi << s) | (lo >> (32u - s))) : hi;
#endif
    }
};

// the token at the top of w (see HuffDev); toff = byte offset of the Huffman table
CVS_HD uint32_t huff_decode(const TableRef &tb, uint32_t toff, uint32_t w)
{
    uint32_t e = tb.ld32(toff + 4u * (w >> (32 - kLutBits)));
    if (e >> 30) {
        if (e & kEntryLevel2) {
            e = tb.ld32(toff + kOffLut2 + ((e & 0xffu) << (kLut2Bits + 2)) + 4u * ((w >> (32 - kLutBits - kLut2Bits)) & ((1u << kLut2Bits) - 1u)));
        } else { // a table with more long prefixes than second-level tables: canonical search (jdhuff.c slow path)
            const uint32_t is_ac = tb.ld32(toff + kOffIsAc);
            e = make_entry(0, 16, is_ac);
            for (uint32_t l = kLutBits + 1; l <= 16; l++) {
                const int32_t code = (int32_t)(w >> (32u - l));
                if (code <= (int32_t)tb.ld32(toff + kOffMaxcode + 4u * l)) {
                    e = make_entry(tb.ld8(toff + kOffVals + ((uint32_t)(code + (int32_t)tb.ld32(toff + kOffValoff + 4u * l)) & 255u)), l, is_ac);
                    break;
                }
            }
        }
    }
    return e;
}

// Where a counting run leaves the state it passes the inner boundaries of its subsequence in (every G bits), together
// with the blocks completed and the DC differences summed since the start of the subsequence: the write pass then runs
// with one thread per G bits instead of one per S bits.
struct MidRecords {
    uint32_t *state; // [nsplit * nsub]; kStateUnset: no token starts behind this boundary
    uint32_t *nblk;
    int32_t *dc;     // [3][stride]
    uint32_t stride; // nsplit * nsub_max
    uint32_t nsplit, G;
};

// One run over subsequence i: tokens that start in [i*S + off, min((i+1)*S, T)).  WRITE: store the coefficients
// (scan order, natural order inside a block, DC absolute) of blocks first_block.. with the predictors pred0..2.
// The token step is one code path for DC and AC tokens, written with selects: the lanes of a warp sit in different places
// of different blocks, divergent paths would put their latencies in series, and the chain p -> window -> table -> p is
// what the whole decode waits for.
template <bool WRITE, bool RECORD = false, bool HALF = false>
CVS_HD RunResult run_range(const TableRef &tb, const Geometry &g, const uint32_t *words, uint32_t total_bits, uint32_t begin,
                           uint32_t end_nominal, uint32_t i, uint32_t entry, const uint8_t *natural, int16_t *coef,
                           uint32_t first_block, int32_t pred0, int32_t pred1, int32_t pred2, const MidRecords *mid = nullptr)
{
    RunResult r;
    int32_t dc0 = pred0, dc1 = pred1, dc2 = pred2;
    const uint32_t end = end_nominal < total_bits ? end_nominal : total_bits;
    uint32_t p = begin + (entry & 31u), ph = (entry >> 5) & 7u, k = (entry >> 8) & 63u;
    uint32_t blk = first_block, nblocks = 0;
    const uint32_t nluma = (uint32_t)(g.bpm - (g.ncomp == 3 ? 2 : 0)), bpm = (uint32_t)g.bpm;
    uint32_t next_inner = 0, inner = 1;
    // (the fields of *mid in locals: the record stores below could alias them, and they would be re-read per token)
    uint32_t *const rec_state = RECORD ? mid->state : nullptr, *const rec_nblk = RECORD ? mid->nblk : nullptr;
    int32_t *const rec_dc = RECORD ? mid->dc : nullptr;
    const uint32_t rec_G = RECORD ? mid->G : 0u, rec_nsplit = RECORD ? mid->nsplit : 0u, rec_stride = RECORD ? mid->stride : 0u;
    if (RECORD) {
        next_inner = begin + rec_G;
        for (uint32_t j = 1; j < rec_nsplit; j++) rec_state[i * rec_nsplit + j] = kStateUnset;
    }
    const uint32_t half_at = begin + ((end_nominal - begin) >> 1);
    uint32_t half = kStateUnset;
    if (begin < total_bits && p < end) {
        BitWindow bw;
        bw.init(words, p);
        do {
            const uint32_t is_ac = k != 0 ? 1u : 0u;
            const uint32_t c = ph < nluma ? 0u : ph - nluma + 1u;
            const uint32_t w = bw.peek(p);
            const uint32_t e = huff_decode(tb, (2u * c + is_ac) * (uint32_t)sizeof(HuffDev), w);
            const uint32_t len = (e >> 8) & 31u, s = e & 15u;
            // jdhuff.c HUFF_EXTEND of the s bits behind the code (0 for s = 0)
            const uint32_t x = ((w << len) >> 1) >> (31u - s);
            const int32_t v = (int32_t)x + ((((int32_t)x - (int32_t)((1u << s) >> 1)) >> 31) & (int32_t)((0xffffffffu << s) + 1u));
            p += (e >> 13) & 63u;
            const int32_t vdc = is_ac ? 0 : v;
            dc0 += c == 0 ? vdc : 0;
            dc1 += c == 1 ? vdc : 0;
            dc2 += c == 2 ? vdc : 0;
            if (WRITE) {
                if (blk < g.nblocks) {
                    const uint32_t kk = k + ((e >> 4) & 15u); // zig-zag position of an AC coefficient
                    if (!is_ac) coef[(size_t)blk * 64] = (int16_t)(c == 0 ? dc0 : (c == 1 ? dc1 : dc2));
                    else if (s && kk < 64) coef[(size_t)blk * 64 + natural[kk]] = (int16_t)v;
                }
            }
            k += (e >> 19) & 127u;
            const bool block_end = k >= 64u;
            k = block_end ? 0u : k;
            ph = block_end ? (ph + 1 == bpm ? 0u : ph + 1) : ph;
            blk += block_end ? 1u : 0u;
            nblocks += block_end ? 1u : 0u;
            if (RECORD) {
                if (p >= next_inner && p < end) { // the first token behind an inner boundary starts at p
                    const uint32_t idx = i * rec_nsplit + inner;
                    rec_state[idx] = pack_state(p - next_inner, ph, k);
                    rec_nblk[idx] = nblocks;
                    rec_dc[idx] = dc0 - pred0;
                    rec_dc[rec_stride + idx] = dc1 - pred1;
                    rec_dc[2 * rec_stride + idx] = dc2 - pred2;
                    next_inner += rec_G;
                    inner++;
                }
            }
            if (HALF) { // the first token of the second half starts at p
                const bool hit = half == kStateUnset && p >= half_at && p < end;
                half = hit ? pack_state(p - half_at, ph, k) : half;
            }
        } while (p < end);
    }
    const uint32_t over = p > end_nominal ? p - end_nominal : 0u; // < 32: a token is at most 31 bits long
    r.exit_state = pack_state(over & 31u, ph, k);
    r.half_state = half;
    r.nblocks = nblocks;
    r.dc0 = WRITE ? dc0 : dc0 - pred0; // sums of the differences when counting
    r.dc1 = WRITE ? dc1 : dc1 - pred1;
    r.dc2 = WRITE ? dc2 : dc2 - pred2;
    return r;
}

template <bool WRITE, bool RECORD = false, bool HALF = false>
CVS_HD RunResult run_subsequence(const TableRef &tb, const Geometry &g, const uint32_t *words, uint32_t total_bits, uint32_t i,
                                 uint32_t entry, const uint8_t *natural, int16_t *coef, uint32_t first_block, int32_t pred0,
                                 int32_t pred1, int32_t pred2, const MidRecords *mid = nullptr)
{
    return run_range<WRITE, RECORD, HALF>(tb, g, words, total_bits, i * g.sub_bits, i * g.sub_bits + g.sub_bits, i, entry, natural, coef,
                                    first_block, pred0, pred1, pred2, mid);
}

} // namespace jpg
} // namespace cvs

// =====================================================================================================================
#if defined(__CUDACC__)
#include <cooperative_groups.h>
#include <stdio.h>

namespace cvs {
namespace jpg {

__constant__ uint8_t c_natural[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                      41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                      30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

constexpr int kUnstuffThreads = 256, kUnstuffBytes = 16; // bytes per thread
constexpr int kEntropyThreads = 256;

// status bits of a decode (OR-ed into the ticket's status word)
constexpr unsigned int kJpegNotConverged = 1u << 8, kJpegBlockCount = 1u << 9;

// ---- byte unstuffing ------------------------------------------------------------------------------------------------
// A byte is dropped when it is the 00 behind an FF (T.81 B.1.1.5) or part of a restart marker FF D0..D7; what remains is
// the plain bit string of the scan, restart intervals back to back (each ends padded to a byte).  raw_len is the length
// of the entropy-coded segment.  *marks: bit j set = byte j is the second byte of a restart marker.
__device__ __forceinline__ uint32_t unstuff_keep_mask(const uint8_t *raw, uint32_t raw_len, uint32_t first, uint8_t (&b)[kUnstuffBytes],
                                                      uint32_t *marks)
{
    uint32_t keep = 0, mk = 0;
    uint8_t prev = first ? raw[first - 1] : 0;
    if (first + kUnstuffBytes <= raw_len) {
        const uint4 v = *reinterpret_cast<const uint4 *>(raw + first);
        const uint32_t wv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < kUnstuffBytes; j++) b[j] = (uint8_t)(wv[j >> 2] >> (8 * (j & 3)));
    } else {
#pragma unroll
        for (int j = 0; j < kUnstuffBytes; j++) b[j] = first + j < raw_len ? raw[first + j] : 0;
    }
    const uint8_t after = first + kUnstuffBytes < raw_len ? raw[first + kUnstuffBytes] : 0;
#pragma unroll
    for (int j = 0; j < kUnstuffBytes; j++) {
        const uint8_t next = j + 1 < kUnstuffBytes ? b[j + 1 < kUnstuffBytes ? j + 1 : j] : after;
        const bool stuffed = b[j] == 0x00 && prev == 0xFF;
        const bool marker2 = (b[j] & 0xF8) == 0xD0 && prev == 0xFF;
        const bool marker1 = b[j] == 0xFF && (next & 0xF8) == 0xD0;
        if (first + j < raw_len) {
            if (!(stuffed || marker1 || marker2)) keep |= 1u << j;
            if (marker2) mk |= 1u << j;
        }
        prev = b[j];
    }
    *marks = mk;
    return keep;
}

// one block's share (block index vb of the unstuffing grid); kUnstuffThreads threads
__device__ __forceinline__ void unstuff_count_block(uint32_t vb, const uint8_t *__restrict__ raw, uint32_t raw_len, uint32_t *block_kept,
                                                    uint32_t *block_marks, uint32_t (*wsum)[kUnstuffThreads / 32])
{
    const uint32_t first = (vb * kUnstuffThreads + threadIdx.x) * kUnstuffBytes;
    uint8_t b[kUnstuffBytes];
    uint32_t mk = 0;
    uint32_t n = first < raw_len ? (uint32_t)__popc(unstuff_keep_mask(raw, raw_len, first, b, &mk)) : 0u;
    n = __reduce_add_sync(0xffffffffu, n);
    const uint32_t m = __reduce_add_sync(0xffffffffu, (uint32_t)__popc(mk));
    if ((threadIdx.x & 31) == 0) {
        wsum[0][threadIdx.x >> 5] = n;
        wsum[1][threadIdx.x >> 5] = m;
    }
    __syncthreads();
    if (threadIdx.x < 2) {
        uint32_t t = 0;
        for (int w = 0; w < kUnstuffThreads / 32; w++) t += wsum[threadIdx.x][w];
        (threadIdx.x ? block_marks : block_kept)[vb] = t;
    }
    __syncthreads();
}

// out must be zero beyond the string (the decoder looks up to 16 bytes past its end); total_bits <- 8 * kept bytes;
// seg_start[m] <- byte offset (in out) at which restart interval m starts (seg_start[0] = 0 is the caller's),
// total_marks <- number of restart markers
__device__ __forceinline__ void unstuff_write_block(uint32_t vb, uint32_t nvb, const uint8_t *__restrict__ raw, uint32_t raw_len,
                                                    const uint32_t *block_kept, const uint32_t *block_marks, uint8_t *out,
                                                    uint32_t *total_bits, uint32_t *seg_start, uint32_t seg_cap, uint32_t *total_marks,
                                                    uint32_t (*wsum)[kUnstuffThreads / 32], uint32_t *s_base)
{
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // bytes kept / markers seen by the blocks in front of this one
    uint32_t part = 0, partm = 0;
    for (uint32_t j = tid; j < vb; j += kUnstuffThreads) {
        part += __ldcg(block_kept + j);
        partm += __ldcg(block_marks + j);
    }
    part = __reduce_add_sync(0xffffffffu, part);
    partm = __reduce_add_sync(0xffffffffu, partm);
    if (lane == 0) {
        wsum[0][warp] = part;
        wsum[1][warp] = partm;
    }
    __syncthreads();
    if (tid < 2) {
        uint32_t t = 0;
        for (int w = 0; w < kUnstuffThreads / 32; w++) t += wsum[tid][w];
        s_base[tid] = t;
    }
    __syncthreads();
    const uint32_t base = s_base[0], basem = s_base[1];
    __syncthreads();
    const uint32_t first = (vb * kUnstuffThreads + tid) * kUnstuffBytes;
    uint8_t b[kUnstuffBytes];
    uint32_t mk = 0;
    const uint32_t keep = first < raw_len ? unstuff_keep_mask(raw, raw_len, first, b, &mk) : 0u;
    const uint32_t n = (uint32_t)__popc(keep), nm = (uint32_t)__popc(mk);
    uint32_t incl = n | (nm << 16); // both counts in one scan (a block keeps <= 4096 bytes and sees <= 2048 markers)
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t o = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= (uint32_t)d) incl += o;
    }
    if (lane == 31) wsum[0][warp] = incl;
    __syncthreads();
    uint32_t woff = 0;
    for (uint32_t w = 0; w < warp; w++) woff += wsum[0][w];
    const uint32_t excl = woff + incl - (n | (nm << 16));
    uint32_t o = base + (excl & 0xffffu);
    uint32_t mi = basem + (excl >> 16);
    if (keep == 0xffffu && (o & 3u) == 0) { // the common case: nothing dropped, word-aligned destination
        uint32_t *dst = reinterpret_cast<uint32_t *>(out + o);
#pragma unroll
        for (int q = 0; q < 4; q++)
            dst[q] = (uint32_t)b[4 * q] | ((uint32_t)b[4 * q + 1] << 8) | ((uint32_t)b[4 * q + 2] << 16) | ((uint32_t)b[4 * q + 3] << 24);
    } else {
#pragma unroll
        for (int j = 0; j < kUnstuffBytes; j++) {
            if (keep >> j & 1u) out[o++] = b[j];
            if (mk >> j & 1u) { // the next restart interval starts at the byte that follows
                ++mi;
                if (mi < seg_cap) seg_start[mi] = o;
            }
        }
    }
    if (vb == nvb - 1 && tid == kUnstuffThreads - 1) {
        uint32_t t = 0;
        for (int w = 0; w < kUnstuffThreads / 32; w++) t += wsum[0][w];
        *total_bits = 8u * (base + (t & 0xffffu));
        *total_marks = basem + (t >> 16);
    }
    __syncthreads();
}

// stand-alone launches (scans with restart intervals; k_entropy does the same work in its own first phases)
__global__ void __launch_bounds__(kUnstuffThreads) k_unstuff_count(const uint8_t *__restrict__ raw, uint32_t raw_len, uint32_t *block_kept,
                                                                  uint32_t *block_marks)
{
    __shared__ uint32_t wsum[2][kUnstuffThreads / 32];
    unstuff_count_block(blockIdx.x, raw, raw_len, block_kept, block_marks, wsum);
}

__global__ void __launch_bounds__(kUnstuffThreads) k_unstuff_write(const uint8_t *__restrict__ raw, uint32_t raw_len,
                                                                  const uint32_t *__restrict__ block_kept,
                                                                  const uint32_t *__restrict__ block_marks, uint8_t *out,
                                                                  uint32_t *total_bits, uint32_t *seg_start, uint32_t seg_cap,
                                                                  uint32_t *total_marks)
{
    __shared__ uint32_t wsum[2][kUnstuffThreads / 32];
    __shared__ uint32_t s_base[2];
    unstuff_write_block(blockIdx.x, gridDim.x, raw, raw_len, block_kept, block_marks, out, total_bits, seg_start, seg_cap, total_marks,
                        wsum, s_base);
}

// ---- entropy decode, scans with restart intervals: every interval starts byte-aligned in a known state (first block of
//      its MCUs, predictors zero), so one thread decodes one interval straight into the coefficients -- no
//      synchronisation, no counting pass.  (Parallel only across intervals: a camera that puts a whole MCU row into one
//      interval gets 68 sequential chains per 1080p frame, about 1 ms; intervals of a few MCUs decode in microseconds.)
struct RestartParams {
    const Tables *tables;
    Geometry g;
    const uint32_t *words;
    const uint32_t *total_bits, *total_marks;
    const uint32_t *seg_start; // [nseg]
    uint32_t nseg;             // ceil(MCUs / restart interval)
    uint32_t blocks_per_seg;   // restart interval * blocks per MCU
    int16_t *coef;
    unsigned int *status;
};

__global__ void __launch_bounds__(128) k_entropy_restart(const RestartParams p)
{
    __shared__ Tables tb;
    __shared__ uint8_t s_nat[64];
    const uint32_t tid = threadIdx.x;
    if (tid < 64) s_nat[tid] = c_natural[tid];
    {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(p.tables);
        uint32_t *dst = reinterpret_cast<uint32_t *>(&tb);
        for (uint32_t j = tid; j < sizeof(Tables) / 4; j += blockDim.x) dst[j] = src[j];
    }
    __syncthreads();
    const TableRef tbr = table_ref(&tb);
    const uint32_t T = *p.total_bits;
    if (blockIdx.x == 0 && tid == 0 && *p.total_marks + 1 != p.nseg) atomicOr(p.status, kJpegBlockCount);
    const uint32_t sgm = blockIdx.x * blockDim.x + tid;
    if (sgm >= p.nseg) return;
    const uint32_t begin = sgm ? 8u * p.seg_start[sgm] : 0u;
    uint32_t end = sgm + 1 < p.nseg ? 8u * p.seg_start[sgm + 1] : T;
    if (begin >= T || end > T || end <= begin) return; // fewer markers than intervals: reported above
    Geometry g = p.g;
    const uint32_t first = sgm * p.blocks_per_seg;
    // the interval's blocks only: a damaged interval must not spill into its neighbour's coefficients
    g.nblocks = min(p.g.nblocks, first + p.blocks_per_seg);
    const RunResult r = run_range<true>(tbr, g, p.words, end, begin, end, 0, pack_state(0, 0, 0), s_nat, p.coef, first, 0, 0, 0);
    if (first + r.nblocks < g.nblocks) atomicOr(p.status, kJpegBlockCount);
}

// ---- entropy decode -------------------------------------------------------------------------------------------------
struct EntropyParams {
    // first phases: clear the scratch, FF 00 -> FF (what k_unstuff_count / k_unstuff_write do as launches of their own)
    const uint8_t *raw;       // entropy-coded segment as received
    uint32_t raw_len;
    uint8_t *unst;            // unstuffed string (= words)
    uint32_t unst_bytes;      // bytes of it to clear (a multiple of 16, covers the string and its padding)
    uint32_t *block_kept, *block_marks, *total_marks_out, *seg_start;
    uint32_t seg_cap;
    uint32_t *total_bits_out;
    const Tables *tables;     // device copy
    Geometry g;
    const uint32_t *words;    // unstuffed string
    const uint32_t *total_bits;
    uint32_t *entry;          // [2 * nsub_max + 2] entry state of each (half) subsequence (written by its predecessor)
    uint32_t *used;           // [nsub_max] entry state of the last run
    uint32_t *nblk;           // [nsub_max] blocks completed, then (after the scan) first block index
    int32_t *dcs;             // [3][nsub_max] DC sums, then predictors at entry
    uint32_t *tile_blk;       // [ntiles] per-tile totals
    int32_t *tile_dc;         // [3][ntiles]
    MidRecords mid;           // inner-boundary records of the counting runs (write pass granularity)
    uint32_t *hx, *hy, *hw;   // [nsub_max * bpm] exit states of the phase hypotheses: fresh / followed one / two subsequences further
    uint32_t *hym, *hwm;      // [nsub_max * bpm] state of the Y / W runs in the middle of their subsequence (hym[0]: the exact run of subsequence 0)
    uint8_t *hmap;            // [nsub_max][16] successor of candidate c of boundary i-1 among the candidates of boundary i
    unsigned int *changed;    // [kRoundCounters] states changed in a round, three counters in rotation
    int16_t *coef;            // [nblocks][64], zeroed
    unsigned int *status;
};

__global__ void __launch_bounds__(kEntropyThreads) k_entropy(const EntropyParams p)
{
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ Tables tb;
    __shared__ uint32_t s_scan[4][kEntropyThreads / 32];
    __shared__ uint32_t s_tile_base[4];
    __shared__ uint8_t s_nat[64];
    __shared__ unsigned long long s_compose[kEntropyThreads];
    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < 64) s_nat[tid] = c_natural[tid];
    {
        const uint32_t *src = reinterpret_cast<const uint32_t *>(p.tables);
        uint32_t *dst = reinterpret_cast<uint32_t *>(&tb);
        for (uint32_t j = tid; j < sizeof(Tables) / 4; j += kEntropyThreads) dst[j] = src[j];
    }
    __syncthreads();
    const TableRef tbr = table_ref(&tb);
    const Geometry g = p.g;

    // ---- clear what must start as zero (round counters, entry states, coefficients, the unstuffed string's buffer) and
    //      count the bytes that stay; then compact them.  Two grid barriers instead of a memset and two launches.
    {
        static_assert(kUnstuffThreads == kEntropyThreads, "the unstuffing phases run on k_entropy's blocks");
        uint32_t(*wsum)[kUnstuffThreads / 32] = reinterpret_cast<uint32_t(*)[kUnstuffThreads / 32]>(&s_scan[0][0]);
        const uint32_t gthreads = gridDim.x * kEntropyThreads, gtid = blockIdx.x * kEntropyThreads + tid;
        const uint4 z = make_uint4(0, 0, 0, 0);
        uint4 *cz = reinterpret_cast<uint4 *>(p.coef);
        for (uint32_t j = gtid; j < g.nblocks * 8u; j += gthreads) cz[j] = z; // 128 bytes per block
        uint4 *uz = reinterpret_cast<uint4 *>(p.unst);
        for (uint32_t j = gtid; j < p.unst_bytes / 16u; j += gthreads) uz[j] = z;
        for (uint32_t j = gtid; j < 2u * g.nsub_max + 2u; j += gthreads) p.entry[j] = 0u; // first guess: a block of phase 0 starts here
        if (gtid < (uint32_t)kRoundCounters) p.changed[gtid] = 0u;
        const uint32_t nvb = (p.raw_len + kUnstuffThreads * kUnstuffBytes - 1) / (kUnstuffThreads * kUnstuffBytes);
        for (uint32_t vb = blockIdx.x; vb < nvb; vb += gridDim.x) unstuff_count_block(vb, p.raw, p.raw_len, p.block_kept, p.block_marks, wsum);
        grid.sync();
        for (uint32_t vb = blockIdx.x; vb < nvb; vb += gridDim.x)
            unstuff_write_block(vb, nvb, p.raw, p.raw_len, p.block_kept, p.block_marks, p.unst, p.total_bits_out, p.seg_start, p.seg_cap,
                                p.total_marks_out, wsum, s_tile_base);
        grid.sync();
    }
    const uint32_t T = __ldcg(p.total_bits);
    const uint32_t nsub = (T + g.sub_bits - 1) / g.sub_bits; // <= nsub_max
    const uint32_t ntiles = (nsub + kEntropyThreads - 1) / kEntropyThreads;

    // the rounds, the prefix sums and the write pass work on HALF subsequences when the hypotheses deliver the states in
    // the middle of the subsequences too (half the length of the confirming round).  (The state in the middle costs a
    // compare and a select per token.  Measured and not adopted: the state at EVERY 128-bit boundary, stored from a
    // branch -- confirming round 28 -> 8 us, but with 32 lanes crossing boundaries at different tokens the branch is
    // taken by some lane in nearly every iteration and the hypothesis phases go from 105 to 160 us.)
    const bool half = g.sub_bits % 256u == 0 && p.mid.nsplit % 2u == 0;
    const uint32_t hstep = half ? 2u : 1u;
    // ---- phase hypotheses (see the header): seed entry[] with the states the true token sequence passes through
    {
        const uint32_t B = (uint32_t)g.bpm, nh = nsub * B, gstride = gridDim.x * kEntropyThreads;
        const uint32_t first = blockIdx.x * kEntropyThreads + tid;
        // X: a block of phase h starts at the subsequence boundary; Y, W: that sequence followed through the next and the
        // next-but-one subsequence.  One thread walks the three in a row -- nobody else's result is needed in between, so
        // there is no grid barrier between them, and a thread waits for the tokens of ITS three subsequences (at most
        // 600 on the camera frame) instead of three times for the slowest subsequence of the frame (3 x 286).
        for (uint32_t idx = first; idx < nh; idx += gstride) {
            const uint32_t i = idx / B, h = idx - i * B;
            uint32_t x;
            if (idx == 0) { // the exact start: this is the decode of subsequence 0, its middle state is wanted below
                const RunResult r0 = run_subsequence<false, false, true>(tbr, g, p.words, T, 0, pack_state(0, 0, 0), s_nat, nullptr, 0, 0, 0, 0);
                x = r0.exit_state;
                p.hym[0] = r0.half_state;
            } else {
                x = run_subsequence<false>(tbr, g, p.words, T, i, pack_state(0, h, 0), s_nat, nullptr, 0, 0, 0, 0).exit_state;
            }
            p.hx[idx] = x;
            if (i == 0) p.hy[idx] = kStateUnset;
            if (i + 1 < nsub) {
                // (a Y / W run that starts from the TRUE state of its boundary is the decode of its subsequence: its state
                //  in the middle lets the rounds below work on half subsequences)
                const RunResult ry = run_subsequence<false, false, true>(tbr, g, p.words, T, i + 1, x, s_nat, nullptr, 0, 0, 0, 0);
                p.hy[idx + B] = ry.exit_state;
                p.hym[idx + B] = ry.half_state;
                if (i + 2 < nsub) {
                    const RunResult rw = run_subsequence<false, false, true>(tbr, g, p.words, T, i + 2, ry.exit_state, s_nat, nullptr, 0, 0, 0, 0);
                    p.hw[idx + 2 * B] = rw.exit_state;
                    p.hwm[idx + 2 * B] = rw.half_state;
                }
            }
        }
        grid.sync();
        // where does each candidate of boundary i-1 arrive among those of boundary i?
        for (uint32_t idx = first; idx < nh; idx += gstride) {
            const uint32_t i = idx / B, h = idx - i * B;
            uint32_t m0 = kNoCandidate, m1 = kNoCandidate;
            if (i) {
                const uint32_t y = __ldcg(p.hy + idx);
                m0 = B + h; // candidate X_h of the boundary in front arrives here as Y_h, or as a fresh sequence it fell in with
                for (uint32_t h2 = 0; h2 < B; h2++)
                    if (__ldcg(p.hx + i * B + h2) == y) {
                        m0 = h2;
                        break;
                    }
                if (i >= 2) {
                    const uint32_t w = __ldcg(p.hw + idx); // candidate Y_h of the boundary in front, followed through subsequence i
                    for (uint32_t h2 = 0; h2 < B && m1 == kNoCandidate; h2++)
                        if (__ldcg(p.hx + i * B + h2) == w) m1 = h2;
                    for (uint32_t h2 = 0; h2 < B && m1 == kNoCandidate; h2++)
                        if (__ldcg(p.hy + i * B + h2) == w) m1 = B + h2;
                }
            }
            p.hmap[(size_t)i * 16 + h] = (uint8_t)m0;
            p.hmap[(size_t)i * 16 + B + h] = (uint8_t)m1;
        }
        grid.sync();
        // follow candidate 0 of boundary 0 (the exact start) through the maps: a scan of map compositions, one block
        if (blockIdx.x == 0) {
            unsigned long long *s_f = reinterpret_cast<unsigned long long *>(&s_compose[0]);
            const uint32_t chunk = (nsub - 1 + kEntropyThreads - 1) / kEntropyThreads; // maps 1 .. nsub-1
            const uint32_t lo = 1 + tid * chunk, hi = min(lo + chunk, nsub);
            auto load_map = [&](uint32_t i) -> unsigned long long {
                const uint4 v = __ldcg(reinterpret_cast<const uint4 *>(p.hmap + (size_t)i * 16));
                const uint32_t wv[4] = {v.x, v.y, v.z, v.w};
                unsigned long long m = 0;
#pragma unroll
                for (int c = 0; c < 16; c++) m |= (unsigned long long)((wv[c >> 2] >> (8 * (c & 3))) & 15u) << (4 * c);
                return m;
            };
            auto compose = [&](unsigned long long f, unsigned long long m) -> unsigned long long { // first f, then m
                unsigned long long r = 0;
#pragma unroll
                for (int c = 0; c < 12; c++) {
                    const uint32_t x = (uint32_t)(f >> (4 * c)) & 15u;
                    const uint32_t y = x >= 12u ? kNoCandidate : (uint32_t)(m >> (4 * x)) & 15u;
                    r |= (unsigned long long)y << (4 * c);
                }
                return r;
            };
            const unsigned long long ident = 0xBA9876543210ull;
            unsigned long long f = ident;
            for (uint32_t i = lo; i < hi; i++) f = compose(f, load_map(i));
            s_f[tid] = f;
            __syncthreads();
            for (uint32_t d = 1; d < (uint32_t)kEntropyThreads; d <<= 1) { // inclusive scan (Hillis-Steele)
                unsigned long long a = ident;
                if (tid >= d) a = s_f[tid - d];
                __syncthreads();
                if (tid >= d) s_f[tid] = compose(a, s_f[tid]);
                __syncthreads();
            }
            uint32_t t = tid ? (uint32_t)(s_f[tid - 1]) & 15u : 0u; // candidate the true sequence is at boundary lo - 1
            // entry[] is filled at the granularity the rounds use: 2 * i = start of subsequence i, 2 * i + 1 = its middle
            // (hstep = 2), or just the subsequence starts (hstep = 1)
            if (tid == 0) {
                p.entry[hstep] = __ldcg(p.hx); // boundary 0: the exact run
                if (half) p.entry[1] = __ldcg(p.hym) == kStateUnset ? 0u : __ldcg(p.hym);
            }
            for (uint32_t i = lo; i < hi; i++) {
                if (half) { // subsequence i was decoded from candidate t of boundary i - 1: by its Y run (t < B) or its W run
                    uint32_t hs = kStateUnset;
                    if (t < B) hs = __ldcg(p.hym + i * B + t);
                    else if (t < 2 * B) hs = __ldcg(p.hwm + i * B + t - B);
                    p.entry[2 * i + 1] = hs == kStateUnset ? 0u : hs;
                }
                if (t < 12u) t = p.hmap[(size_t)i * 16 + t];
                uint32_t st = __ldcg(p.hx + i * B); // no candidate known: any state, the rounds below repair it
                if (t < B) st = __ldcg(p.hx + i * B + t);
                else if (t < 2 * B) st = __ldcg(p.hy + i * B + t - B);
                p.entry[hstep * (i + 1)] = st;
            }
        }
        __threadfence();
        grid.sync();
    }

    Geometry gr = g;
    MidRecords midr = p.mid;
    uint32_t nsubr = nsub, ntilesr = ntiles;
    if (half) {
        gr.sub_bits = g.sub_bits / 2u;
        gr.nsub_max = 2u * g.nsub_max;
        midr.nsplit = p.mid.nsplit / 2u; // the inner boundaries stay where they were (every G bits)
        nsubr = (T + gr.sub_bits - 1) / gr.sub_bits;
        ntilesr = (nsubr + kEntropyThreads - 1) / kEntropyThreads;
    }
    // ---- rounds: decode from the entry state, hand the exit state on, until no state changes (one round when the
    //      seeds above are all true; any number otherwise).  (Measured and not adopted: letting the Y / W runs keep their
    //      counts and inner-boundary records -- the run that started from the true state of its boundary IS the decode,
    //      so this round could go -- makes those phases 183 us instead of 123 us with six times the records to store;
    //      317 us per frame either way.)
    bool converged = false;
    // Exact states travel at least one subsequence per round, so nsubr rounds always suffice (a stream whose codes do not
    // self-synchronise at all -- every code equally long -- needs them all; a camera frame needs one).  The counter of a
    // round is one of three in rotation: the one of round r + 1 is cleared during round r, when every thread has long
    // read it for round r - 2.
    for (uint32_t round = 0; round <= nsubr; round++) {
        unsigned int *const counter = p.changed + round % 3u;
        if (blockIdx.x == 0 && tid == 0) p.changed[(round + 1u) % 3u] = 0u;
        for (uint32_t tile = blockIdx.x; tile < ntilesr; tile += gridDim.x) {
            const uint32_t i = tile * kEntropyThreads + tid;
            if (i >= nsubr) continue;
            const uint32_t e = i == 0 ? pack_state(0, 0, 0) : __ldcg(p.entry + i);
            if (round && e == p.used[i]) continue;
            const RunResult r = run_subsequence<false, true>(tbr, gr, p.words, T, i, e, s_nat, nullptr, 0, 0, 0, 0, &midr);
            p.used[i] = e;
            p.nblk[i] = r.nblocks;
            p.dcs[i] = r.dc0;
            p.dcs[gr.nsub_max + i] = r.dc1;
            p.dcs[2 * gr.nsub_max + i] = r.dc2;
            if (__ldcg(p.entry + i + 1) != r.exit_state) {
                __stcg(p.entry + i + 1, r.exit_state);
                if (i + 1 < nsubr) atomicAdd(counter, 1u);
            }
        }
        grid.sync();
        if (__ldcg(counter) == 0) {
            converged = true;
            break;
        }
    }
    if (!converged) {
        if (blockIdx.x == 0 && tid == 0) atomicOr(p.status, kJpegNotConverged);
        return;
    }

    // ---- scan: per-tile totals, then every tile sums the totals in front of it
    for (uint32_t tile = blockIdx.x; tile < ntilesr; tile += gridDim.x) {
        const uint32_t i = tile * kEntropyThreads + tid;
        uint32_t v[4] = {0, 0, 0, 0};
        if (i < nsubr) {
            v[0] = p.nblk[i];
            v[1] = (uint32_t)p.dcs[i];
            v[2] = (uint32_t)p.dcs[gr.nsub_max + i];
            v[3] = (uint32_t)p.dcs[2 * gr.nsub_max + i];
        }
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const uint32_t s = __reduce_add_sync(0xffffffffu, v[q]);
            if (lane == 0) s_scan[q][warp] = s;
        }
        __syncthreads();
        if (tid < 4) {
            uint32_t t = 0;
            for (int w = 0; w < kEntropyThreads / 32; w++) t += s_scan[tid][w];
            if (tid == 0) p.tile_blk[tile] = t;
            else p.tile_dc[(tid - 1) * ntilesr + tile] = (int32_t)t;
        }
        __syncthreads();
    }
    grid.sync();
    uint32_t total_blocks_seen = 0;
    for (uint32_t tile = blockIdx.x; tile < ntilesr; tile += gridDim.x) {
        // base of this tile
        uint32_t part[4] = {0, 0, 0, 0};
        for (uint32_t j = tid; j < tile; j += kEntropyThreads) {
            part[0] += __ldcg(p.tile_blk + j);
            part[1] += (uint32_t)__ldcg(p.tile_dc + j);
            part[2] += (uint32_t)__ldcg(p.tile_dc + ntilesr + j);
            part[3] += (uint32_t)__ldcg(p.tile_dc + 2 * ntilesr + j);
        }
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const uint32_t s = __reduce_add_sync(0xffffffffu, part[q]);
            if (lane == 0) s_scan[q][warp] = s;
        }
        __syncthreads();
        if (tid < 4) {
            uint32_t t = 0;
            for (int w = 0; w < kEntropyThreads / 32; w++) t += s_scan[tid][w];
            s_tile_base[tid] = t;
        }
        __syncthreads();
        uint32_t base[4] = {s_tile_base[0], s_tile_base[1], s_tile_base[2], s_tile_base[3]};
        __syncthreads();
        // exclusive scan inside the tile
        const uint32_t i = tile * kEntropyThreads + tid;
        uint32_t v[4] = {0, 0, 0, 0};
        if (i < nsubr) {
            v[0] = p.nblk[i];
            v[1] = (uint32_t)p.dcs[i];
            v[2] = (uint32_t)p.dcs[gr.nsub_max + i];
            v[3] = (uint32_t)p.dcs[2 * gr.nsub_max + i];
        }
        uint32_t incl[4];
#pragma unroll
        for (int q = 0; q < 4; q++) {
            incl[q] = v[q];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t o = __shfl_up_sync(0xffffffffu, incl[q], d);
                if (lane >= (uint32_t)d) incl[q] += o;
            }
            if (lane == 31) s_scan[q][warp] = incl[q];
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < 4; q++) {
            uint32_t woff = 0;
            for (uint32_t w = 0; w < warp; w++) woff += s_scan[q][w];
            base[q] += woff + incl[q] - v[q];
        }
        __syncthreads();
        // first block index and DC predictors of the subsequence (over the counts, which are not needed any more)
        if (i < nsubr) {
            if (i == nsubr - 1) total_blocks_seen = base[0] + v[0];
            p.nblk[i] = base[0];
            p.dcs[i] = (int32_t)base[1];
            p.dcs[gr.nsub_max + i] = (int32_t)base[2];
            p.dcs[2 * gr.nsub_max + i] = (int32_t)base[3];
        }
    }
    grid.sync();
    // ---- write pass: one thread per G bits, from the states the counting runs left at the inner boundaries
    {
        Geometry gw = gr;
        gw.sub_bits = midr.G;
        const uint32_t nsplit = midr.nsplit, nparts = nsubr * nsplit;
        for (uint32_t j = blockIdx.x * kEntropyThreads + tid; j < nparts; j += gridDim.x * kEntropyThreads) {
            const uint32_t i = j / nsplit, part = j - i * nsplit;
            uint32_t e = __ldcg(p.used + i), blk0 = __ldcg(p.nblk + i);
            int32_t d0 = __ldcg(p.dcs + i), d1 = __ldcg(p.dcs + gr.nsub_max + i), d2 = __ldcg(p.dcs + 2 * gr.nsub_max + i);
            if (part) {
                e = __ldcg(midr.state + j);
                if (e == kStateUnset) continue;
                blk0 += __ldcg(midr.nblk + j);
                d0 += __ldcg(midr.dc + j);
                d1 += __ldcg(midr.dc + midr.stride + j);
                d2 += __ldcg(midr.dc + 2 * midr.stride + j);
            }
            run_subsequence<true>(tbr, gw, p.words, T, j, e, s_nat, p.coef, blk0, d0, d1, d2);
        }
    }
    // the string must hold exactly the image's blocks (padding bits after the last block decode to no complete block
    // in a well-formed stream; more or fewer blocks means a damaged frame)
    if (total_blocks_seen && total_blocks_seen < gr.nblocks) atomicOr(p.status, kJpegBlockCount);
}

// ---- IDCT: jpeg_idct_islow, one thread per 8x8 block ---------------------------------------------------------------------
struct PlaneParams {
    Geometry g;
    const Tables *tables;
    const int16_t *coef;
    uint8_t *y, *cb, *cr; // planes: luma pitch = mcux*8*H, chroma pitch = mcux*8
};

// The arithmetic is libjpeg-turbo's x86-64 SIMD islow IDCT (simd/x86_64/jidctint-avx2.asm), which is what OpenCV runs;
// it differs from jidctint.c only where values leave 16 bits.  The rules, as in oracle/jpeg_oracle.c idct_islow:
// dequantisation wraps to int16 (pmullw); in0+in4, in0-in4, in7+in3 and in5+in1 wrap to int16 (paddw / psubw); all
// other products and sums are 32-bit (pmaddwd / paddd) and cannot overflow; pass 1 saturates to int16 (packssdw); a
// block whose coefficient rows 1..7 are zero skips pass 1 with row 0 << PASS1_BITS wrapped to int16 (psllw); pass 2
// saturates to -128..127 and adds 128 (packsswb, paddb).

__device__ __forceinline__ int32_t idct_wrap16(int32_t x) { return (int32_t)(int16_t)x; }

// the 1-D transform of both passes, eight int16 inputs -> eight outputs descaled by SHIFT; the constants are the
// asm's pmaddwd pairs (sums / differences of jidctint.c's FIX_x values)
template <int SHIFT>
__device__ __forceinline__ void idct8(const int32_t (&in)[8], int32_t (&out)[8])
{
    const int32_t tmp3 = in[2] * (4433 + 6270) + in[6] * 4433, tmp2 = in[2] * 4433 + in[6] * (4433 - 15137);
    const int32_t tmp0 = idct_wrap16(in[0] + in[4]) * (1 << 13), tmp1 = idct_wrap16(in[0] - in[4]) * (1 << 13);
    const int32_t tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
    const int32_t z3 = idct_wrap16(in[7] + in[3]), z4 = idct_wrap16(in[5] + in[1]);
    const int32_t Z3 = z3 * (9633 - 16069) + z4 * 9633, Z4 = z3 * 9633 + z4 * (9633 - 3196);
    const int32_t o0 = in[7] * (2446 - 7373) + in[1] * (-7373) + Z3, o3 = in[7] * (-7373) + in[1] * (12299 - 7373) + Z4;
    const int32_t o1 = in[5] * (16819 - 20995) + in[3] * (-20995) + Z4, o2 = in[5] * (-20995) + in[3] * (25172 - 20995) + Z3;
    constexpr int32_t rnd = 1 << (SHIFT - 1);
    out[0] = (tmp10 + o3 + rnd) >> SHIFT;
    out[7] = (tmp10 - o3 + rnd) >> SHIFT;
    out[1] = (tmp11 + o2 + rnd) >> SHIFT;
    out[6] = (tmp11 - o2 + rnd) >> SHIFT;
    out[2] = (tmp12 + o1 + rnd) >> SHIFT;
    out[5] = (tmp12 - o1 + rnd) >> SHIFT;
    out[3] = (tmp13 + o0 + rnd) >> SHIFT;
    out[4] = (tmp13 - o0 + rnd) >> SHIFT;
}

constexpr int kIdctThreads = 128;

__global__ void __launch_bounds__(kIdctThreads) k_idct(const PlaneParams p)
{
    __shared__ uint16_t sq[3][64];
    for (uint32_t j = threadIdx.x; j < 192; j += kIdctThreads) sq[j >> 6][j & 63] = p.tables->q[j >> 6][j & 63];
    __syncthreads();
    const Geometry g = p.g;
    const uint32_t b = blockIdx.x * kIdctThreads + threadIdx.x;
    if (b >= g.nblocks) return;
    const uint32_t m = b / (uint32_t)g.bpm, j = b - m * (uint32_t)g.bpm;
    const uint32_t my = m / (uint32_t)g.mcux, mx = m - my * (uint32_t)g.mcux;
    const uint32_t nluma = (uint32_t)(g.bpm - (g.ncomp == 3 ? 2 : 0));
    uint32_t c;
    uint8_t *dst;
    size_t pitch;
    if (j < nluma) {
        c = 0;
        pitch = (size_t)g.mcux * 8 * g.H;
        dst = p.y + ((size_t)my * g.V + j / (uint32_t)g.H) * 8 * pitch + ((size_t)mx * g.H + j % (uint32_t)g.H) * 8;
    } else {
        c = j - nluma + 1;
        pitch = (size_t)g.mcux * 8;
        dst = (c == 1 ? p.cb : p.cr) + (size_t)my * 8 * pitch + (size_t)mx * 8;
    }
    // dequantised coefficients of the block, wrapped to int16: row r in ws[r][0..7]
    int32_t ws[8][8];
    uint32_t rows_nz = 0; // OR of the quantised coefficients of rows 1..7
    const uint4 *src = reinterpret_cast<const uint4 *>(p.coef + (size_t)b * 64);
#pragma unroll
    for (int r = 0; r < 8; r++) {
        const uint4 v = __ldg(src + r);
        if (r) rows_nz |= v.x | v.y | v.z | v.w;
        const uint32_t wv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int q = 0; q < 8; q++) {
            const int32_t cf = (int32_t)(int16_t)(wv[q >> 1] >> (16 * (q & 1)));
            ws[r][q] = idct_wrap16(cf * (int32_t)sq[c][8 * r + q]);
        }
    }
    // pass 1: columns, saturated to int16; rows 1..7 all zero: row 0 << 2 wrapped to int16 in every row
#pragma unroll
    for (int col = 0; col < 8; col++) {
        int32_t in[8], out[8];
#pragma unroll
        for (int r = 0; r < 8; r++) in[r] = ws[r][col];
        idct8<13 - 2>(in, out);
        const int32_t dc_only = idct_wrap16(in[0] * 4);
#pragma unroll
        for (int r = 0; r < 8; r++) ws[r][col] = rows_nz ? min(max(out[r], -32768), 32767) : dc_only;
    }
    // pass 2: rows, saturated to -128..127, + 128
#pragma unroll
    for (int r = 0; r < 8; r++) {
        int32_t out[8];
        idct8<13 + 2 + 3>(ws[r], out);
        uint32_t lo = 0, hi = 0;
#pragma unroll
        for (int q = 0; q < 4; q++) {
            lo |= (uint32_t)(min(max(out[q], -128), 127) + 128) << (8 * q);
            hi |= (uint32_t)(min(max(out[4 + q], -128), 127) + 128) << (8 * q);
        }
        *reinterpret_cast<uint2 *>(dst + (size_t)r * pitch) = make_uint2(lo, hi);
    }
}

// ---- chroma upsampling + colour conversion: one thread per 4 horizontally adjacent pixels -------------------------------
struct ColourParams {
    Geometry g;
    const uint8_t *y, *cb, *cr;
    uint8_t *bgr; // width * height * 3, rows contiguous
};

__device__ __forceinline__ uint32_t clamp255(int32_t v) { return (uint32_t)min(max(v, 0), 255); }

constexpr int kColourThreads = 256;

__global__ void __launch_bounds__(kColourThreads) k_colour(const ColourParams p)
{
    const Geometry g = p.g;
    const int x0 = (blockIdx.x * kColourThreads + threadIdx.x) * 4;
    const int yrow = blockIdx.y;
    if (x0 >= g.width) return;
    const size_t ypitch = (size_t)g.mcux * 8 * g.H, cpitch = (size_t)g.mcux * 8;
    const uint32_t yw = *reinterpret_cast<const uint32_t *>(p.y + (size_t)yrow * ypitch + x0);
    int32_t cbv[4], crv[4];
    if (g.ncomp == 1) {
#pragma unroll
        for (int q = 0; q < 4; q++) cbv[q] = crv[q] = 128;
    } else if (g.H == 1) {
        const uint32_t b4 = *reinterpret_cast<const uint32_t *>(p.cb + (size_t)yrow * cpitch + x0);
        const uint32_t r4 = *reinterpret_cast<const uint32_t *>(p.cr + (size_t)yrow * cpitch + x0);
#pragma unroll
        for (int q = 0; q < 4; q++) {
            cbv[q] = (int32_t)((b4 >> (8 * q)) & 255u);
            crv[q] = (int32_t)((r4 >> (8 * q)) & 255u);
        }
    } else {
        const int dw = (g.width + 1) >> 1;            // downsampled_width
        const int c0 = x0 >> 1;                       // chroma columns c0, c0 + 1 cover the four pixels
        const bool fancy = dw > 2;
#pragma unroll
        for (int pl = 0; pl < 2; pl++) {
            const uint8_t *src = pl ? p.cr : p.cb;
            int32_t *dstv = pl ? crv : cbv;
            if (g.V == 1) {
                const uint8_t *in = src + (size_t)yrow * cpitch;
                if (fancy) { // h2v1_fancy_upsample (jdsample.c)
#pragma unroll
                    for (int e = 0; e < 2; e++) {
                        const int c = min(c0 + e, dw - 1);
                        const int v = in[c];
                        dstv[2 * e] = c == 0 ? v : (3 * v + in[c - 1] + 1) >> 2;
                        dstv[2 * e + 1] = c == dw - 1 ? v : (3 * v + in[c + 1] + 2) >> 2;
                    }
                } else {
#pragma unroll
                    for (int q = 0; q < 4; q++) dstv[q] = in[min((x0 + q) >> 1, dw - 1)];
                }
            } else {
                const int dh = (g.height + 1) >> 1;
                const int r = yrow >> 1;
                if (fancy) { // h2v2_fancy_upsample; the rows above the first / below the last are that row again (jdmainct.c)
                    const int rn = min(max((yrow & 1) ? r + 1 : r - 1, 0), dh - 1);
                    const uint8_t *in0 = src + (size_t)r * cpitch, *in1 = src + (size_t)rn * cpitch;
                    // column sums 3 * nearer + further for columns c0 - 1 .. c0 + 2
                    int32_t cs[4];
#pragma unroll
                    for (int e = 0; e < 4; e++) {
                        const int c = min(max(c0 - 1 + e, 0), dw - 1);
                        cs[e] = 3 * (int32_t)in0[c] + (int32_t)in1[c];
                    }
#pragma unroll
                    for (int e = 0; e < 2; e++) {
                        const int c = c0 + e;
                        const int32_t t = cs[1 + e];
                        dstv[2 * e] = c == 0 ? (4 * t + 8) >> 4 : (3 * t + cs[e] + 8) >> 4;
                        dstv[2 * e + 1] = c >= dw - 1 ? (4 * t + 7) >> 4 : (3 * t + cs[2 + e] + 7) >> 4;
                    }
                } else {
#pragma unroll
                    for (int q = 0; q < 4; q++) dstv[q] = src[(size_t)r * cpitch + min((x0 + q) >> 1, dw - 1)];
                }
            }
        }
    }
    // jdcolor.c ycc_rgb_convert with the tables of build_ycc_rgb_table written out
    uint32_t px[12];
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const int32_t yy = (int32_t)((yw >> (8 * q)) & 255u), cb = cbv[q] - 128, cr = crv[q] - 128;
        if (g.ncomp == 1) {
            px[3 * q] = px[3 * q + 1] = px[3 * q + 2] = (uint32_t)yy;
        } else {
            px[3 * q + 2] = clamp255(yy + ((91881 * cr + 32768) >> 16));
            px[3 * q + 1] = clamp255(yy + ((-22554 * cb + 32768 - 46802 * cr) >> 16));
            px[3 * q] = clamp255(yy + ((116130 * cb + 32768) >> 16));
        }
    }
    uint8_t *dst = p.bgr + ((size_t)yrow * g.width + x0) * 3;
    if (x0 + 4 <= g.width && (((size_t)yrow * g.width * 3) & 3u) == 0 && (reinterpret_cast<uintptr_t>(p.bgr) & 3u) == 0) {
        uint32_t *d4 = reinterpret_cast<uint32_t *>(dst);
#pragma unroll
        for (int q = 0; q < 3; q++) d4[q] = px[4 * q] | (px[4 * q + 1] << 8) | (px[4 * q + 2] << 16) | (px[4 * q + 3] << 24);
    } else {
        const int npx = min(4, g.width - x0);
        for (int j = 0; j < 3 * npx; j++) dst[j] = (uint8_t)px[j];
    }
}

} // namespace jpg
} // namespace cvs
#endif // __CUDACC__
