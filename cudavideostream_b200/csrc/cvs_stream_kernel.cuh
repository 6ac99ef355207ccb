// cvs_stream_kernel.cuh -- the fused hot path: thresholded difference + negative feedback +
// ordered compaction (+ one display filter), as ONE persistent launch over a sequence of frames.
//
// Replaces kernel2 (server/src/kernels.cu:289-334), its CPU twin (tests/cuda_streaming/
// test.cu:560-576) and the visualiser kernels that read the same frame pair (kernels.cu:31-95,
// 243-281).  nframes = 1 is the drop-in exec_core path; nframes = T walks a device-resident
// sequence (frame t+1 is differenced against the reference frame t left behind).
//
// The path is integer byte work: on B200 it is bound by instruction issue long before HBM, so the
// design minimises instructions per frame byte and keeps HBM traffic at its floor.
//
// Work decomposition
//   * a frame is cut into groups of 48 B = 16 BGR pixels = three 16-byte vectors (cvs_pixel.cuh); a
//     thread owns a CHUNK of two consecutive groups (96 B), which halves the per-byte cost of the
//     scans, the barrier, the look-back and the flush;
//   * the grid is G persistent blocks of 512 threads, one per SM (128 registers per thread fill the register
//     file; measured 5 % faster than two blocks of 256), all co-resident (cooperative launch).
//     A frame is covered in nseg passes ("segments") of G*cps chunks; in segment s block b owns the cps
//     consecutive chunks starting at (s*G + b)*cps and thread i of the block owns chunk i of that
//     slice -- the SAME bytes in every frame.  One (frame, segment) pair is a "step";
//   * ingest: a block streams its slice of the coming steps into a shared-memory ring (3 stages of 48 KB)
//     with 1-D bulk copies (TMA engine, cp.async.bulk + mbarrier, L2 evict-first): every byte of a frame crosses HBM -> SM exactly once,
//     as one contiguous request per slice (42 KB at 1080p), and each thread picks its 32 whole pixels
//     out of shared memory with six conflict-free LDS.128 (half the lanes keep their two pixel groups
//     in swapped order, see voff());
//   * reference: the host runs this kernel only on frames that do not fit one pass of the grid
//     (3840x2160 single frames and short sequences; k_stream_ws takes everything else), so nseg > 1
//     and a thread's chunk changes from segment to segment.  In every step each thread reloads its
//     96 reference bytes with L2 evict-last loads and, if any of them changed, stores them back (the
//     reference frame stays L2 resident; same thread, same address, so no cross-thread hazard exists);
//   * one pass over the 24 words of a chunk produces, per word: byte-SIMD |cur-ref| > T flags (the
//     eight flags of two words are gathered into one byte of the 96-bit change mask by ONE multiply),
//     the difference bytes cur-ref (parked in the thread's own 96 bytes of the ring stage) and the
//     updated reference (negative feedback).  popc of the mask is the thread's entry count;
//   * compaction: warp totals by REDUX, one block barrier per step, per-lane ranks by a shuffle scan;
//     cross-block offsets by a one-round decoupled look-back: each block publishes
//     (epoch<<32 | count) for the step and sums the descriptors of its predecessors, each read by
//     its own thread; the running total of earlier segments of the frame travels in one extra
//     descriptor.  A sparse WARP then walks the set bits of its lanes' masks, stages (index, value) in
//     its own shared-memory window in rank order and flushes it with 16-byte (xs) / 4-byte (diff)
//     coalesced streaming stores; a dense warp (more entries than the window holds) walks its chunks
//     with all lanes and stores contiguous runs straight to global memory (emit_coop) -- warps drift
//     apart freely, the last one to finish refills the stage;
//   * display filter MODE (heat map, red maps, grayscale, binarisation pass 1) is computed from the
//     same registers and written with 16-byte streaming stores;
//   * the step loop is software-pipelined: while a block runs the front half of step q (ingest ...
//     publish) the descriptors it needs for step q-1 are already in flight, and the back half of
//     step q-1 (staging and flush) follows, so the L2 round trip of the look-back stays hidden.
//
// Order, values and the new reference are bit-exact with oracle/cvs_oracle.c orc_diff_compact;
// unlike kernel2 the payload order is deterministic (ascending byte index).
#pragma once
#include "cvs_pixel.cuh"

namespace cvs {

constexpr int kThreads = 512;                         // threads per block
constexpr int kWarps = kThreads / 32;
constexpr int kWarpsPad = (kWarps + 3) / 4 * 4;       // stride of the per-warp total arrays
constexpr int kBlocksPerSM = 512 / kThreads;          // 128 registers per thread fill the register file
// look-back descriptors a thread may read: one per kThreads blocks of a B200-sized grid (the host clamps the grid
// to kLook * kThreads blocks on a larger device)
constexpr int kLook = (148 * kBlocksPerSM + kThreads - 1) / kThreads;
constexpr int kGroupsPerThread = 2;
constexpr int kChunkBytes = kGroupsPerThread * kGroupBytes;   // 96
constexpr int kChunkWords = kChunkBytes / 4;                  // 24
constexpr int kMaskWords = kChunkBytes / 32;                  // 3
constexpr int kStageBytes = kThreads * kChunkBytes;   // 49,152 B: one block slice
constexpr int kStages = 4;                            // one parked, one in process, two slices in flight
constexpr int kWarpEntries = 512;                     // payload entries a warp's staging window holds
constexpr uint32_t kWatchdogPolls = 1u << 24;         // look-back polls (>= 100 ns each) before giving up

enum StatusBits : unsigned { kStatusCapacity = 1u, kStatusWatchdog = 2u };

struct StreamParams {
    const uint8_t *frames;      // frame t at frames + t*frame_stride (16-byte aligned)
    size_t frame_stride;        // multiple of 16, >= nbytes rounded up to 16
    int nframes;
    uint8_t *ref;               // reference frame, padded to a whole number of chunks
    uint32_t nbytes;            // N = 3*W*H
    uint32_t nbytes16;          // N rounded up to 16
    uint32_t nchunks;           // ceil(N / 96)
    uint32_t nseg;              // segments per frame
    uint32_t cps;               // chunks per block per segment (<= kThreads)
    uint32_t nstages;           // ring stages in use (2..kStages); the launch pays SmemLayout::total(nstages)
    unsigned int *pos;          // [nframes]
    int *xs;                    // frame t at xs + t*cap
    uint8_t *diff;              // frame t at diff + t*cap
    size_t cap;                 // payload capacity per frame (entries)
    uint8_t *show;              // display frame t at show + t*show_stride (MODE 1,2,3,4,6)
    size_t show_stride;
    uint8_t *gray1;             // MODE 5/7: one gray byte per pixel, frame t at gray1 + t*gray_stride
    size_t gray_stride;
    unsigned int *hist;         // MODE 5/7: [nframes][256], zeroed by the host before the launch
    const uint32_t *heat_lut;   // MODE 1: 766 entries B | G<<8 | R<<16
    unsigned long long *desc;   // [nframes*nseg][G+1]
    uint32_t epoch;             // tag of this launch
    uint32_t addc;              // threshold constant for changed80<>
    unsigned int *status;       // StatusBits
    // banded launches (k_stream_ws only; 0 / nullptr otherwise): the launch covers the byte range
    // [index_base, index_base + nbytes) of larger frames -- frames, ref are already offset by the host; indices and
    // display offsets get index_base added -- and frame t's entries follow the pos_prior[t] entries of the bands before
    uint32_t index_base;
    const unsigned int *pos_prior;
};

// dynamic shared memory layout (bytes).  The small tables come first and the ring last, so the launch decides
// how many stages it pays for (total(nstages)): shared memory not used stays L1.
struct SmemLayout {
    static constexpr int kXsHalves = kWarpEntries + 8;                     // + alignment shift; 16-bit offsets in the warp's span
    static constexpr int kSdBytes = kWarpEntries + 16;
    static constexpr int lut = 0;                                          // 768 words
    static constexpr int hist = lut + 768 * 4;                             // 256 words
    static constexpr int wtot = hist + 256 * 4;                            // 2 x kWarpsPad words (by step parity)
    static constexpr int red = wtot + 2 * kWarpsPad * 4;                   // 2 x kWarpsPad words
    static constexpr int done = red + 2 * kWarpsPad * 4;                   // kStages words
    static constexpr int bar = done + 8 * 4;                               // kStages mbarriers
    static constexpr int sxs = bar + 8 * 8;                                // kWarps * kXsHalves uint16
    static constexpr int sd = sxs + kWarps * kXsHalves * 2;                // kWarps * kSdBytes bytes
    static constexpr int stage = (sd + kWarps * kSdBytes + 127) / 128 * 128; // nstages * kStageBytes
    static constexpr int total(int nstages) { return stage + nstages * kStageBytes; }
};
static_assert(kStages <= 8, "done[] / mbarrier slots");
static_assert(SmemLayout::bar % 8 == 0, "mbarrier alignment");
static_assert(SmemLayout::sd % 16 == 0 && SmemLayout::sxs % 16 == 0, "staging alignment");
static_assert((SmemLayout::kXsHalves * 2) % 16 == 0 && SmemLayout::kSdBytes % 16 == 0, "per-warp staging alignment");

// Coalesced flush by one warp of n staged entries to global rank g0.  The staging arrays were filled
// starting at element (g0 & 3), so that 16-byte vectors of xs (and 4-byte words of diff) line up
// between shared and global memory.
// A staged index is the 16-bit offset of the byte inside the warp's 3,072-byte span; wbase (the frame offset of
// the span) is added on the way out.
__device__ __forceinline__ void flush_warp(const uint16_t *sxs, const uint8_t *sd, uint32_t wbase, int *xs_out,
                                           uint8_t *df_out, size_t g0, uint32_t n, size_t cap, uint32_t lane)
{
    if (g0 >= cap) return;
    if (g0 + n > cap) n = (uint32_t)(cap - g0);
    const uint32_t sh = (uint32_t)(g0 & 3);
    // element e of the staging arrays <-> global rank (g0 - sh) + e ; valid e in [sh, sh + n)
    int *xg = xs_out + (g0 - sh);
    uint8_t *dg = df_out + (g0 - sh);
    const uint32_t end = sh + n;
    // whole quads [4i, 4i+4) go out as one 16-byte + one 4-byte store per lane
    const uint32_t q0 = (sh + 3u) & ~3u, q1 = end & ~3u;
#pragma unroll 1
    for (uint32_t e = q0 + 4 * lane; e < q1; e += 128) {
        const uint2 h = *reinterpret_cast<const uint2 *>(sxs + e); // four 16-bit offsets
        stg_stream(xg + e, make_uint4(wbase + (h.x & 0xffffu), wbase + (h.x >> 16), wbase + (h.y & 0xffffu), wbase + (h.y >> 16)));
        stg_stream_u32(dg + e, *reinterpret_cast<const uint32_t *>(sd + e));
    }
    // the (at most three + three) entries before the first and after the last whole quad: one lane each
    const uint32_t e1 = lane < 4 ? sh + lane : max(q1, q0) + (lane - 4);
    if (lane < 8 && e1 < (lane < 4 ? min(q0, end) : end)) {
        stg_stream_u32(xg + e1, wbase + sxs[e1]);
        stg_stream_u8(dg + e1, sd[e1]);
    }
}

// walks the set bits of `bits` (bit j <-> byte `jbase + j` of the chunk): index goes to sxs, the
// difference byte is fetched from the thread's parked bytes at shared address dvaddr
__device__ __forceinline__ uint32_t lds_u8(uint32_t addr)
{
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}

__device__ __forceinline__ void emit_bits(uint32_t bits, uint32_t jbase, uint32_t coff, uint32_t dvaddr, uint16_t *sxs,
                                          uint8_t *sd, uint32_t &o)
{
    // two entries per trip: half the loop overhead, and the two byte loads are in flight together.  With one bit
    // left the second load reads the byte before the thread's chunk (harmless) and nothing is stored for it.
    while (bits) {
        const uint32_t j0 = jbase + (uint32_t)__ffs((int)bits) - 1u;
        bits &= bits - 1u;
        const bool two = bits != 0u;
        const uint32_t j1 = jbase + (uint32_t)__ffs((int)bits) - 1u;
        bits &= bits - 1u;
        const uint32_t v0 = lds_u8(dvaddr + j0), v1 = lds_u8(dvaddr + j1);
        sxs[o] = (uint16_t)(coff + j0);
        sd[o] = (uint8_t)v0;
        if (two) {
            sxs[o + 1] = (uint16_t)(coff + j1);
            sd[o + 1] = (uint8_t)v1;
        }
        o += two ? 2u : 1u;
    }
}

// base + scale * i as ONE 64-bit multiply-add (the plain pointer arithmetic costs an add and a carry add per store)
__device__ __forceinline__ int *at_u32(int *base, uint32_t i)
{
    int *q;
    asm("mad.wide.u32 %0, %1, 4, %2;" : "=l"(q) : "r"(i), "l"(base));
    return q;
}
__device__ __forceinline__ uint8_t *at_u8(uint8_t *base, uint32_t i)
{
    uint8_t *q;
    asm("mad.wide.u32 %0, %1, 1, %2;" : "=l"(q) : "r"(i), "l"(base));
    return q;
}

// Dense warps (more entries than the staging window holds): the warp walks its 32 chunks one after the other
// and handles each chunk with all lanes -- lane L owns bytes L, L+32 and L+64 of the chunk, finds its rank by a
// popc over the chunk's change mask and stores straight to global memory.  Consecutive changed bytes land on
// consecutive ranks, so every store instruction writes one contiguous run (up to 128 B of indices).
// The masks and the ranks of the first entry of each 32-byte third of every chunk are exchanged through `scratch`
// (the warp's staging window, idle in a dense step): one broadcast 16-byte and one 8-byte shared load per chunk
// instead of shuffles and popcounts.  CHECK = false when the warp's whole run fits the payload capacity.
// This loop is the bulk of a dense frame's instructions.
// nchunk: chunks the warp holds (lanes >= nchunk have an empty mask); a multiple of the batch size.
template <bool CHECK>
__device__ __forceinline__ void emit_coop(const uint32_t (&m)[kMaskWords], uint32_t coff0, uint32_t dvaddr0,
                                          int *xs_out, uint8_t *df_out, uint32_t g_lane, uint32_t cap32, uint32_t lane,
                                          uint32_t scratch, uint32_t nchunk = 32)
{
    {
        const uint32_t r1 = g_lane + (uint32_t)__popc(m[0]), r2 = r1 + (uint32_t)__popc(m[1]);
        asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(scratch + 16 * lane), "r"(m[0]), "r"(m[1]), "r"(m[2]),
                     "r"(g_lane) : "memory");
        asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(scratch + 512 + 8 * lane), "r"(r1), "r"(r2) : "memory");
    }
    __syncwarp();
    const uint32_t lanebit = 1u << lane;
    const uint32_t lt = lanebit - 1u;
    constexpr int kBatch = 2; // chunks in flight: their shared loads are issued before any store
#pragma unroll 1
    for (uint32_t S0 = 0; S0 < nchunk; S0 += kBatch) {
        uint32_t sm[kBatch][kMaskWords], rk[kBatch][kMaskWords], v[kBatch][kMaskWords];
#pragma unroll
        for (int i = 0; i < kBatch; i++) {
            const uint4 a = lds128(scratch + 16 * (S0 + i));
            uint32_t b0, b1;
            asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(b0), "=r"(b1) : "r"(scratch + 512 + 8 * (S0 + i)) : "memory");
            sm[i][0] = a.x; sm[i][1] = a.y; sm[i][2] = a.z;
            rk[i][0] = a.w; rk[i][1] = b0; rk[i][2] = b1;
        }
#pragma unroll
        for (int i = 0; i < kBatch; i++)
#pragma unroll
            for (int w = 0; w < kMaskWords; w++) v[i][w] = lds_u8(dvaddr0 + (S0 + i) * kChunkBytes + lane + 32 * w);
#pragma unroll
        for (int i = 0; i < kBatch; i++) {
            const uint32_t cb = coff0 + (S0 + i) * kChunkBytes + lane;
#pragma unroll
            for (int w = 0; w < kMaskWords; w++) {
                const uint32_t g = rk[i][w] + (uint32_t)__popc(sm[i][w] & lt);
                // both stores under one predicate (no branch around two instructions)
                uint32_t on = sm[i][w] & lanebit;
                if (CHECK && g >= cap32) on = 0;
                asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.u32 p, %0, 0;\n\t"
                             "@p st.global.cs.u32 [%1], %2;\n\t"
                             "@p st.global.cs.u8 [%3], %4;\n\t}" ::"r"(on), "l"(at_u32(xs_out, g)), "r"(cb + 32 * w),
                             "l"(at_u8(df_out, g)), "r"(v[i][w])
                             : "memory");
            }
        }
    }
}

__device__ __forceinline__ uint32_t warp_add(uint32_t v) { return __reduce_add_sync(0xffffffffu, v); }

// sum of the first n and of all kWarps words at p: lane i reads word i, two warp reductions (REDUX)
__device__ __forceinline__ void sum_warps(const uint32_t *p, uint32_t n, uint32_t lane, uint32_t &first_n, uint32_t &all)
{
    static_assert(kWarps <= 32, "one lane per warp total");
    const uint32_t v = lane < (uint32_t)kWarps ? p[lane] : 0u;
    all = warp_add(v);
    first_n = warp_add(lane < n ? v : 0u);
}
__device__ __forceinline__ uint32_t sum_warps(const uint32_t *p, uint32_t lane)
{
    return warp_add(lane < (uint32_t)kWarps ? p[lane] : 0u);
}

template <int MODE, bool HI>
__global__ void __launch_bounds__(kThreads, kBlocksPerSM) k_stream(const StreamParams p)
{
    extern __shared__ __align__(128) unsigned char smem[];
    uint32_t *slut = reinterpret_cast<uint32_t *>(smem + SmemLayout::lut);
    uint32_t *shist = reinterpret_cast<uint32_t *>(smem + SmemLayout::hist);
    uint32_t *wtot = reinterpret_cast<uint32_t *>(smem + SmemLayout::wtot);
    uint32_t *red = reinterpret_cast<uint32_t *>(smem + SmemLayout::red);
    uint32_t *done = reinterpret_cast<uint32_t *>(smem + SmemLayout::done);
    const uint32_t stage_addr = smem_u32(smem + SmemLayout::stage);
    const uint32_t bar_addr = smem_u32(smem + SmemLayout::bar);

    const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t b = blockIdx.x, G = gridDim.x;
    const uint32_t N = p.nbytes;
    const uint32_t nsteps = (uint32_t)p.nframes * p.nseg;
    // ring depth in use (chosen by the host, < kStages: a deeper prefetch measured 17 % slower at 3840x2160)
    const uint32_t nstages = p.nstages;
    constexpr bool kBinarize = (MODE == kModeBinarize || MODE == kModeBinarizeAvg);
    constexpr bool kGrayW = (MODE == kModeGrayWeighted || MODE == kModeBinarize);
    // this warp's staging window
    uint16_t *sxs = reinterpret_cast<uint16_t *>(smem + SmemLayout::sxs) + warp * SmemLayout::kXsHalves;
    uint8_t *sd = smem + SmemLayout::sd + warp * SmemLayout::kSdBytes;

    uint32_t phase = 0;     // bit st: parity the next wait on stage st expects
    bool tripped = false;   // watchdog expired once: stop waiting altogether

    // slice of this block in segment s: byte offset and byte count of the bulk copy
    auto slice = [&](uint32_t s, uint32_t &off, uint32_t &bytes) {
        uint64_t c0 = ((uint64_t)s * G + b) * p.cps;
        uint64_t o = c0 * kChunkBytes;
        if (o >= p.nbytes16) { off = 0; bytes = 0; return; }
        uint64_t e = o + (uint64_t)p.cps * kChunkBytes;
        if (e > p.nbytes16) e = p.nbytes16;
        off = (uint32_t)o;
        bytes = (uint32_t)(e - o);
    };
    // one thread: refill ring stage st with the slice of step q (st == q mod nstages, tracked by the callers: the
    // ring depth is a launch parameter and a division per step would cost more than the rest of the bookkeeping)
    auto issue = [&](uint32_t q, uint32_t st) {
        const uint32_t t = q / p.nseg, s = q - t * p.nseg;
        uint32_t off, bytes;
        slice(s, off, bytes);
        if (bytes) {
            const uint64_t pol = l2_policy_evict_first();
            // the stage was last written through the generic proxy (parked difference bytes)
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            mbar_expect_tx(bar_addr + 8 * st, bytes);
            bulk_g2s(stage_addr + st * kStageBytes, p.frames + (size_t)t * p.frame_stride + off, bytes,
                     bar_addr + 8 * st, pol);
        }
    };

    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < kStages; i++) {
            mbar_init(bar_addr + 8 * i, 1);
            done[i] = 0;
        }
        for (int i = 0; i < 2 * kWarpsPad; i++) wtot[i] = red[i] = 0;
        mbar_init_fence();
    }
    if (MODE == kModeHeat)
        for (uint32_t i = tid; i < 766; i += kThreads) slut[i] = p.heat_lut[i];
    __syncthreads();
    if (tid == 0)
        for (uint32_t q = 0; q < nstages && q < nsteps; q++) issue(q, q);

    // Bank-conflict-free 16-byte shared accesses.  Chunks are 96 B apart, so with every lane on the same vector of
    // its chunk lanes L and L+4 of a quarter-warp hit the same banks (6L mod 8 takes four values).  Lanes with bit 2
    // set therefore keep their two 48-byte pixel groups in SWAPPED order in registers ("slot" order): slot vector v
    // of such a lane is vector (v+3) mod 6 of the chunk, which lands on the four odd bank groups.  Only the change
    // mask has to be put back into byte order; every address below goes through voff().
    const uint32_t sw = ((lane >> 2) & 1u) * (uint32_t)kGroupBytes; // 0 or 48
    auto voff = [&](int v) -> uint32_t { return v < 3 ? 16u * v + sw : 16u * v - sw; }; // chunk offset of slot vector v
    uint32_t r[kChunkWords];
    const uint64_t keep = l2_policy_evict_last();
    uint32_t coff = 0, nv = 0; // byte offset of this thread's chunk in the frame, valid bytes (0..96)
    uint32_t sbytes = 0;       // bytes of the block's slice in the current segment
    auto geometry = [&](uint32_t s) {
        uint32_t soff;
        slice(s, soff, sbytes);
        uint64_t c = ((uint64_t)s * G + b) * p.cps + tid;
        bool ok = tid < p.cps && c < p.nchunks;
        coff = ok ? (uint32_t)(c * kChunkBytes) : 0u;
        nv = ok ? min(N - coff, (uint32_t)kChunkBytes) : 0u;
    };
    auto load_ref = [&]() {
        if (nv) {
#pragma unroll
            for (int v = 0; v < kChunkWords / 4; v++) {
                uint4 a = ldg_keep(p.ref + coff + voff(v), keep);
                r[4 * v] = a.x; r[4 * v + 1] = a.y; r[4 * v + 2] = a.z; r[4 * v + 3] = a.w;
            }
        } else {
#pragma unroll
            for (int k = 0; k < kChunkWords; k++) r[k] = 0;
        }
    };
    auto store_ref = [&]() {
#pragma unroll
        for (int v = 0; v < kChunkWords / 4; v++)
            stg_keep(p.ref + coff + voff(v), make_uint4(r[4 * v], r[4 * v + 1], r[4 * v + 2], r[4 * v + 3]), keep);
    };

    // (every step computes its own geometry below; without this first call the compiler schedules the loop differently)
    geometry(0);

    // The loop is software-pipelined by one step: iteration q runs the FRONT half of step q (ingest, flags,
    // change mask, feedback, counts, publish) and then the BACK half of step q-1 (look-back sum, staging,
    // flush).  The predecessors' descriptors of step q-1 are fetched at the top of the iteration, so their L2
    // round trip hides behind the front half, and the single barrier of an iteration serves both the block
    // scan of step q and the look-back reduction of step q-1.
    uint32_t b_m[kMaskWords] = {0, 0, 0};
    uint32_t b_wrank = 0, b_wexc = 0, b_wtotal = 0, b_total = 0, b_coff = 0, b_myaddr = 0, b_t = 0, b_s = 0;
    bool pending = false;
    uint32_t t = 0, s = 0; // frame and segment of step q
    uint32_t st = 0, b_st = 0; // ring stage of step q / of step q-1

    for (uint32_t q = 0; q <= nsteps; q++) {
        const bool front = q < nsteps;

        // ---- back half, part 1: start fetching the look-back descriptors of step q-1.  Thread i reads
        //      predecessors i, i+256, ...; thread b%256 also reads the running total of the earlier segments
        unsigned long long pv[kLook], pv2 = 0;
        const unsigned long long *prow = p.desc + (size_t)(q ? q - 1 : 0) * (G + 1);
        const bool has2 = pending && b_s > 0 && tid == (b % kThreads);
#pragma unroll
        for (int i = 0; i < kLook; i++) {
            pv[i] = 0;
            if (pending && tid + i * kThreads < b) pv[i] = desc_peek(prow + tid + i * kThreads);
        }
        if (has2) pv2 = desc_peek(prow - 1); // slot G of the previous step

        uint32_t m[kMaskWords] = {0, 0, 0};
        uint32_t cnt = 0, incl = 0, myaddr = 0;
        if (front) {
            geometry(s);
            load_ref(); // L2 hit; issued before the wait on the frame slice
            if (kBinarize && s == 0) {
                // the thread that zeroes bin i is the one that flushed it at the end of the previous frame;
                // the barrier below orders the zeroing before this frame's atomics
                for (uint32_t i = tid; i < 256; i += kThreads) shist[i] = 0;
                __syncthreads();
            }

            // ---- 1. this thread's 32 pixels out of the ring
            if (sbytes) {
                // steps with an empty slice never touch the barrier, so the parity is tracked per stage
                if (!tripped && !mbar_wait(bar_addr + 8 * st, (phase >> st) & 1u)) {
                    tripped = true;
                    atomicOr(p.status, kStatusWatchdog);
                }
                phase ^= 1u << st;
            }
            myaddr = stage_addr + st * kStageBytes + tid * kChunkBytes;
            // The pixels are consumed straight from the ring, a few registers at a time: 16 bytes (one vector of
            // look-ahead) without a display filter, one 48-byte pixel group when a filter needs whole pixels.
            constexpr bool kStreamLoad = (MODE == kModeNone);
            // the chunk that holds the end of the frame: bytes past N never differ (slot word k of the chunk)
            auto clip_word = [&](int k, uint32_t cw) -> uint32_t {
                const int vb = (int)nv - (int)(voff(k >> 2) + 4 * (k & 3)); // valid bytes from this slot word on
                const uint32_t vm = vb >= 4 ? 0xffffffffu : (vb <= 0 ? 0u : ((1u << (8 * vb)) - 1u));
                return (cw & vm) | (r[k] & ~vm);
            };
            // ---- 3. (defined first, used per vector) one pass: flags -> 96-bit change mask, difference bytes,
            //         negative feedback: reference := changed ? current : reference        (test.cu:565-570)
            // four words (one 16-byte vector) of the chunk
            auto pass_vector = [&](int v, const uint32_t (&cv)[4]) {
                uint32_t dv[4];
#pragma unroll
                for (int h = 0; h < 4; h += 2) {
                    const int k = 4 * v + h;
                    const uint32_t f0 = changed80<HI>(absdiff4(cv[h], r[k]), p.addc);
                    const uint32_t f1 = changed80<HI>(absdiff4(cv[h + 1], r[k + 1]), p.addc);
                    // the eight flag bits of two words (7,15,23,31 and, shifted, 3,11,19,27) -> one byte of the change
                    // mask: every partial product of the multiply lands on its own bit, and bits 32..39 of the product
                    // are the flags in byte order
                    const uint32_t g8 = __umulhi(f1 + (f0 >> 4), 0x20408100u);
                    m[k >> 3] = __byte_perm(m[k >> 3], g8, ((k >> 1) & 3) == 0 ? 0x3214 : ((k >> 1) & 3) == 1 ? 0x3240
                                                          : ((k >> 1) & 3) == 2 ? 0x3410 : 0x4210);
                    dv[h] = sub4<true>(cv[h], r[k]);
                    dv[h + 1] = sub4<true>(cv[h + 1], r[k + 1]);
                    const uint32_t fm0 = spread80(f0), fm1 = spread80(f1);
                    r[k] = (cv[h] & fm0) | (r[k] & ~fm0);
                    r[k + 1] = (cv[h + 1] & fm1) | (r[k + 1] & ~fm1);
                }
                // park the difference bytes of this vector in the thread's own 96 bytes of the stage right away (needed
                // only if the chunk has entries, but 24 live registers cost more than six unconditional shared stores)
                asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(myaddr + voff(v)), "r"(dv[0]), "r"(dv[1]), "r"(dv[2]),
                             "r"(dv[3])
                             : "memory");
            };

            // ---- 2. display filter on the same registers (reference as it was BEFORE this frame)
            if (MODE != kModeNone && nv) {
#pragma unroll
                for (int g = 0; g < kGroupsPerThread; g++) {
                    const uint32_t gb = sw ? (uint32_t)(1 - g) * kGroupBytes : (uint32_t)g * kGroupBytes; // slot group -> chunk
                    const uint32_t goff = coff + gb;
                    const uint32_t gnv = nv > gb ? min(nv - gb, (uint32_t)kGroupBytes) : 0u;
                    if (gnv == 0) continue;
                    uint32_t cg[kGroupWords], rg[kGroupWords], o[kGroupWords];
#pragma unroll
                    for (int v = 0; v < kGroupWords / 4; v++) {
                        const uint4 x = lds128(myaddr + voff(g * (kGroupWords / 4) + v));
                        cg[4 * v] = x.x; cg[4 * v + 1] = x.y; cg[4 * v + 2] = x.z; cg[4 * v + 3] = x.w;
                    }
                    if (__builtin_expect(nv < (uint32_t)kChunkBytes, 0)) {
#pragma unroll
                        for (int k = 0; k < kGroupWords; k++) cg[k] = clip_word(g * kGroupWords + k, cg[k]);
                    }
#pragma unroll
                    for (int k = 0; k < kGroupWords; k++) rg[k] = r[g * kGroupWords + k];
                    if (MODE == kModeHeat) {
                        uint32_t ad[kGroupWords];
#pragma unroll
                        for (int k = 0; k < kGroupWords; k++) ad[k] = absdiff4(cg[k], rg[k]);
                        group_heat(ad, slut, o);
                        store_group(p.show + (size_t)t * p.show_stride + goff, o, gnv);
                    } else if (MODE == kModeRedBlack || MODE == kModeRedOverlap) {
                        uint32_t mk[kGroupWords];
#pragma unroll
                        for (int k = 0; k < kGroupWords; k++) mk[k] = changed80<HI>(absdiff4(cg[k], rg[k]), p.addc);
                        group_red<MODE == kModeRedOverlap>(mk, rg, o);
                        store_group(p.show + (size_t)t * p.show_stride + goff, o, gnv);
                    } else if (MODE == kModeGrayWeighted || MODE == kModeGrayAverage) {
                        group_gray3<kGrayW>(cg, o);
                        store_group(p.show + (size_t)t * p.show_stride + goff, o, gnv);
                    } else if (kBinarize) {
                        uint32_t g4[4];
                        group_gray1<kGrayW>(cg, g4);
                        const uint32_t npx = gnv / 3u; // whole pixels of this group inside the frame
                        uint8_t *gdst = p.gray1 + (size_t)t * p.gray_stride + goff / 3u;
                        if (npx == (uint32_t)kGroupPixels) stg_keep(gdst, make_uint4(g4[0], g4[1], g4[2], g4[3]), keep);
#pragma unroll
                        for (int px = 0; px < kGroupPixels; px++) {
                            if ((uint32_t)px < npx) {
                                uint32_t gv = byte_of(g4[px >> 2], px & 3);
                                if (npx != (uint32_t)kGroupPixels) gdst[px] = (uint8_t)gv;
                                atomicAdd(&shist[gv], 1u); // server.cpp:103-106
                            }
                        }
                    }
                    // the filter saw the reference as it was BEFORE this frame; now the pass over the same registers
#pragma unroll
                    for (int v = 0; v < kGroupWords / 4; v++) {
                        const uint32_t cv[4] = {cg[4 * v], cg[4 * v + 1], cg[4 * v + 2], cg[4 * v + 3]};
                        pass_vector(g * (kGroupWords / 4) + v, cv);
                    }
                }
            }

            if (kStreamLoad && nv) {
                uint4 nx = lds128(myaddr + voff(0));
#pragma unroll
                for (int v = 0; v < kChunkWords / 4; v++) {
                    uint32_t cv[4] = {nx.x, nx.y, nx.z, nx.w};
                    if (v + 1 < kChunkWords / 4) nx = lds128(myaddr + voff(v + 1));
                    if (__builtin_expect(nv < (uint32_t)kChunkBytes, 0)) {
#pragma unroll
                        for (int h = 0; h < 4; h++) cv[h] = clip_word(4 * v + h, cv[h]);
                    }
                    pass_vector(v, cv);
                }
            }
            if (sw) { // slot order -> byte order: rotate the 96-bit mask by 48
                const uint32_t n0 = __funnelshift_r(m[1], m[2], 16), n1 = __funnelshift_r(m[2], m[0], 16),
                               n2 = __funnelshift_r(m[0], m[1], 16);
                m[0] = n0; m[1] = n1; m[2] = n2;
            }
            if (__builtin_expect(nv < (uint32_t)kChunkBytes, 0)) { // bytes past the end of the frame are never entries (matters for T < 0)
#pragma unroll
                for (int w = 0; w < kMaskWords; w++) {
                    const int vb = (int)nv - 32 * w;
                    m[w] &= vb >= 32 ? 0xffffffffu : (vb <= 0 ? 0u : ((1u << vb) - 1u));
                }
            }
            if (m[0] | m[1] | m[2]) store_ref();
            cnt = (uint32_t)__popc(m[0]) + (uint32_t)__popc(m[1]) + (uint32_t)__popc(m[2]);
            // only the warp total has to cross the barrier; the per-lane ranks are scanned after it
            const uint32_t wsum = warp_add(cnt);
            if (lane == 0) wtot[(q & 1u) * kWarpsPad + warp] = wsum;
        }

        // ---- back half, part 2: the descriptors fetched at the top (retry in the rare case a predecessor
        //      had not published yet)
        if (pending) {
            auto settle = [&](unsigned long long v, const unsigned long long *d) -> uint32_t {
                uint32_t polls = 0;
                while ((uint32_t)(v >> 32) != p.epoch && !tripped) {
                    __nanosleep(64);
                    v = desc_peek(d);
                    if (++polls > kWatchdogPolls) { // each poll costs well over 100 ns: seconds, i.e. a bug
                        tripped = true;
                        atomicOr(p.status, kStatusWatchdog);
                    }
                }
                return (uint32_t)v;
            };
            uint32_t part = 0;
#pragma unroll
            for (int i = 0; i < kLook; i++)
                if (tid + i * kThreads < b) part += settle(pv[i], prow + tid + i * kThreads);
            if (has2) part += settle(pv2, prow - 1);
            // G <= kLook * kThreads is enforced by the host, so kLook reads per thread cover every predecessor
            part = warp_add(part);
            if (lane == 0) red[(q & 1u) * kWarpsPad + warp] = part;
        }

        __syncthreads(); // the one barrier of a step: warp totals of step q, look-back partial sums of step q-1

        uint32_t total = 0, wexc = 0, wtotal = 0;
        if (front) {
            sum_warps(wtot + (q & 1u) * kWarpsPad, warp, lane, wexc, total); // entries of the warps before this one / of the block
            if (tid == 0) desc_publish(p.desc + (size_t)q * (G + 1) + b, ((unsigned long long)p.epoch << 32) | total);
            incl = warp_incl_scan(cnt, lane);
            wtotal = __shfl_sync(0xffffffffu, incl, 31); // entries of this warp in step q
        }

        if (pending) {
            const uint32_t base = sum_warps(red + (q & 1u) * kWarpsPad, lane);
            if (tid == 0) {
                if (b == G - 1) {
                    desc_publish(p.desc + (size_t)(q - 1) * (G + 1) + G, ((unsigned long long)p.epoch << 32) | (base + b_total));
                    if (b_s == p.nseg - 1) p.pos[b_t] = base + b_total;
                }
                if ((size_t)base + b_total > p.cap) atomicOr(p.status, kStatusCapacity);
            }

            // ---- back half, part 3: the (index, value) entries of step q-1.  A warp whose entries fit its staging
            //      window writes them there in rank order and flushes the window coalesced; a denser warp lets every
            //      lane store its own run of entries directly.  No other warp is involved either way.
            int *xs_out = p.xs + (size_t)b_t * p.cap;
            uint8_t *df_out = p.diff + (size_t)b_t * p.cap;
            // opaque from here on: otherwise the compiler folds the frame offset into every store of the emission loops
            // and recomputes it there in 64-bit arithmetic (nine instructions per store pair instead of two)
            asm volatile("" : "+l"(xs_out), "+l"(df_out));
            const size_t g0 = (size_t)base + b_wexc; // global rank of this warp's first entry
            if (b_wtotal) {
                if (b_wtotal <= (uint32_t)kWarpEntries) {
                    uint32_t o = b_wrank + (uint32_t)(g0 & 3);
#pragma unroll
                    for (int w = 0; w < kMaskWords; w++) emit_bits(b_m[w], 32 * w, lane * kChunkBytes, b_myaddr, sxs, sd, o);
                    __syncwarp();
                    flush_warp(sxs, sd, __shfl_sync(0xffffffffu, b_coff, 0), xs_out, df_out, g0, b_wtotal, p.cap, lane);
                } else {
                    // chunk S of the warp starts 96*S bytes after lane 0's chunk (frame and ring stage alike); lane 0 holds a
                    // chunk of the frame whenever any lane of the warp does
                    // 32-bit ranks: cap32 saturates, and a run that starts beyond it is dropped entry by entry
                    const uint32_t cap32 = p.cap > 0xffffffffull ? 0xffffffffu : (uint32_t)p.cap;
                    const uint32_t wb = __shfl_sync(0xffffffffu, b_coff, 0), dv0 = b_myaddr - lane * kChunkBytes;
                    if (g0 + b_wtotal <= (size_t)cap32)
                        emit_coop<false>(b_m, wb, dv0, xs_out, df_out, (uint32_t)g0 + b_wrank, cap32, lane, smem_u32(sxs));
                    else
                        emit_coop<true>(b_m, wb, dv0, xs_out, df_out, (uint32_t)g0 + b_wrank, cap32, lane, smem_u32(sxs));
                }
            }
            // ---- this warp is done with the ring stage of step q-1 (pixels consumed before the barrier of
            //      that step, parked bytes emitted above); the last warp to get here refills the stage
            __syncwarp();
            if (lane == 0) {
                const uint32_t stq = b_st;
                __threadfence_block();
                if (atomicAdd(&done[stq], 1u) == (uint32_t)kWarps - 1u) {
                    done[stq] = 0;
                    if (q - 1 + nstages < nsteps) issue(q - 1 + nstages, stq);
                }
            }
        }

        if (front) {
            if (kBinarize && s == p.nseg - 1) {
                __syncthreads();
                for (uint32_t i = tid; i < 256; i += kThreads)
                    if (shist[i]) atomicAdd(p.hist + (size_t)t * 256 + i, shist[i]);
            }
#pragma unroll
            for (int w = 0; w < kMaskWords; w++) b_m[w] = m[w];
            b_wrank = incl - cnt; b_wexc = wexc; b_wtotal = wtotal; b_total = total;
            b_coff = coff; b_myaddr = myaddr; b_t = t; b_s = s;
            pending = true;
            if (++s == p.nseg) { s = 0; ++t; }
            b_st = st;
            if (++st == nstages) st = 0;
        } else {
            pending = false;
        }
    }
}

} // namespace cvs
