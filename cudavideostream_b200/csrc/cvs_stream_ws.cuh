// cvs_stream_ws.cuh -- the fused hot path as a WARP-SPECIALISED persistent kernel (round 2).
//
// Same work, same results and same data layout as k_stream (cvs_stream_kernel.cuh: thresholded difference +
// negative feedback + ordered compaction (+ one display filter) over a sequence of frames, replacing kernel2,
// server/src/kernels.cu:289-334, and its CPU twin tests/cuda_streaming/test.cu:560-576), but a block is split into
// two groups of warps that only meet through mbarriers:
//
//   FRONT warps (0..15)   own the reference bytes (in registers when a frame fits one pass of the grid) and run
//                         the per-word pass of step q: pixels out of the TMA ring, flags, 96-bit change mask,
//                         difference bytes parked in the thread's own 96 bytes of the ring stage, negative feedback,
//                         display filter.  They leave (mask, count) per chunk and the warp totals in shared memory,
//                         arrive on fdone[stage] and go straight on to step q+1 -- no block barrier, no look-back.
//   BACK warps (16..31)   back warp w emits the entries of front warp w's 32 chunks: it waits for fdone[stage],
//                         scans the counts, waits for the block's global offset and stages + flushes (sparse) or
//                         stores cooperatively (dense) exactly as k_stream does.  The LAST back warp also owns the
//                         cross-block exchange: it publishes the block total of the step and sums the predecessors'
//                         descriptors (one-round look-back) before it turns to its own emission.  The last back
//                         warp to finish a stage re-arms it and issues the bulk copy of step q+nstages.
//
// Why: k_stream runs one 512-thread block per SM (the frame gives an SM only 438 chunks at 1080p, and 112
// registers per thread leave room for nothing else), i.e. 3.5 warps per scheduler, and ncu shows 1.0 eligible warp
// per cycle, 52 % issue utilisation, 18 % of warp time at the one block barrier.  Splitting the step doubles the
// warps that can issue (the pass of step q+1 overlaps look-back latency and emission of step q), removes the block
// barrier, and setmaxnreg moves registers from the back warps (which need few) to the front warps.
#pragma once
#include "cvs_stream_kernel.cuh"

namespace cvs {

constexpr int kWsFrontWarps = 16;
constexpr int kWsBackWarps = 16;
constexpr int kWsThreads = 32 * (kWsFrontWarps + kWsBackWarps); // 1024
constexpr int kWsFrontThreads = 32 * kWsFrontWarps;             // chunks per block per step (= kThreads)
constexpr int kWsLook = 5;                                      // descriptors a lane of the look-back warp reads: G <= 160
#ifndef CVS_WS_FRONT_REGS
#define CVS_WS_FRONT_REGS 80
#endif
#ifndef CVS_WS_BACK_REGS
#define CVS_WS_BACK_REGS 48
#endif
// pause between two probes of an mbarrier (ns): front warps waiting for their slice / back warps waiting for the front
// or for the block's global offset
#ifndef CVS_WS_SLEEP_FULL
#define CVS_WS_SLEEP_FULL 100
#endif
#ifndef CVS_WS_SLEEP_BACK
#define CVS_WS_SLEEP_BACK 200
#endif
// binarisation histogram (modes 5, 7): copies in shared memory, lane L adds to copy L mod kWsHistCopies, which cuts the
// same-address serialisation of the shared atomics inside a warp (neighbouring pixels have similar gray values)
#ifndef CVS_WS_HIST_COPIES
#define CVS_WS_HIST_COPIES 1   // 4 copies measured 2 % SLOWER (7.29 vs 7.16 us per frame, mode 5): the atomics are not conflict-bound
#endif
constexpr int kWsHistCopies = CVS_WS_HIST_COPIES;
static_assert(kWsFrontThreads == kThreads, "front threads own one chunk each, like k_stream's threads");
static_assert(512 * CVS_WS_FRONT_REGS + 512 * CVS_WS_BACK_REGS <= 65536, "register file");

// dynamic shared memory of k_stream_ws (bytes).  Stage size and mask stride follow the chunks per block of the
// launch (cps), so four stages fit next to the mask queue at 1080p / 3840x2160 (cps = 438).
struct WsLayout {
    static constexpr int lut = 0;                                      // 768 words
    static constexpr int hist = 0;                                     // kWsHistCopies x 256 words, copy-interleaved; shares
                                                                       // the table's bytes (a launch is heat map OR binarise)
    static constexpr int bar_full = 4096;                              // kStages mbarriers: bulk copy landed
    static constexpr int bar_fdone = bar_full + 8 * 8;                 // kStages mbarriers: front warps done with the step
    static constexpr int bar_base = bar_fdone + 8 * 8;                 // 2 x kStages mbarriers: global offset of the block known
    static constexpr int done = bar_base + 8 * 8;                      // kStages words: back warps finished with the stage
    static constexpr int base = done + 8 * 4;                          // 2 x kStages words: global rank of the block's first entry
    static constexpr int fcnt = base + 8 * 4;                          // kStages words: front warps that have posted their total
    static constexpr int ftot = fcnt + 8 * 4;                          // kStages words: entries of the block in the step so far
    static constexpr int wtot = ftot + 8 * 4;                          // kStages x 16 words: entries per front warp
    static constexpr int sxs = wtot + 8 * 16 * 4;                      // kWsBackWarps * kXsHalves uint16
    static constexpr int sd = sxs + kWsBackWarps * SmemLayout::kXsHalves * 2;
    static constexpr int msk = (sd + kWsBackWarps * SmemLayout::kSdBytes + 127) / 128 * 128; // nstages * msk_stride
    static __host__ __device__ constexpr uint32_t msk_stride(uint32_t cps) { return (cps + 31u) / 32u * 32u * 16u; }
    // whole warps of chunks: the dense emission walks all 32 chunks of a warp, also those past the block's slice
    static __host__ __device__ constexpr uint32_t stage_bytes(uint32_t cps)
    {
        return ((cps + 31u) / 32u * 32u * kChunkBytes + 127u) / 128u * 128u;
    }
    static __host__ __device__ constexpr uint32_t stage0(uint32_t cps, uint32_t nstages) { return msk + nstages * msk_stride(cps); }
    static __host__ __device__ constexpr uint32_t total(uint32_t cps, uint32_t nstages)
    {
        return stage0(cps, nstages) + nstages * stage_bytes(cps);
    }
};
static_assert(kWsHistCopies * 256 * 4 <= WsLayout::bar_full && 768 * 4 <= WsLayout::bar_full, "table / histogram region");
static_assert(2 * kStages <= 8, "bar_base / base slots");
static_assert(WsLayout::bar_full % 8 == 0 && WsLayout::sxs % 16 == 0 && WsLayout::sd % 16 == 0, "alignment");

__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

// Coalesced flush by one warp of n entries staged at elements [0, n) of its window, to global ranks g0 .. g0 + n - 1.
// Unlike flush_warp (k_stream) the window was filled BEFORE g0 was known, so shared and global memory are not aligned
// to each other: the 16-byte index vector / 4-byte value word of a quad is cut out of two aligned shared loads with a
// funnel shift (the misalignment is the same for every quad of the warp).
__device__ __forceinline__ void flush_warp_shifted(const uint16_t *sxs, const uint8_t *sd, uint32_t wbase, int *xs_out,
                                                   uint8_t *df_out, size_t g0, uint32_t n, size_t cap, uint32_t lane)
{
    if (g0 >= cap) return;
    if (g0 + n > cap) n = (uint32_t)(cap - g0);
    const uint32_t a = (4u - (uint32_t)(g0 & 3)) & 3u; // elements in front of the first rank that is a multiple of 4
    const uint32_t head = min(a, n);
    const uint32_t nq = (n - head) >> 2;               // whole quads: elements head + 4k .. head + 4k + 3
    int *xg = xs_out + g0;
    uint8_t *dg = df_out + g0;
    const uint32_t sx = smem_u32(sxs), sv = smem_u32(sd);
    const uint32_t sh16 = 16u * (a & 1u), sh8 = 8u * a;
#pragma unroll 1
    for (uint32_t k = lane; k < nq; k += 32) {
        uint32_t w0, w1, w2, w3, d0, d1;
        asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(w0), "=r"(w1) : "r"(sx + 8 * k) : "memory");
        asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(w2), "=r"(w3) : "r"(sx + 8 * k + 8) : "memory");
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(d0) : "r"(sv + 4 * k) : "memory");
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(d1) : "r"(sv + 4 * k + 4) : "memory");
        if (a & 2u) { w0 = w1; w1 = w2; w2 = w3; }
        const uint32_t x = __funnelshift_r(w0, w1, sh16), y = __funnelshift_r(w1, w2, sh16);
        stg_stream(xg + head + 4 * k, make_uint4(wbase + (x & 0xffffu), wbase + (x >> 16), wbase + (y & 0xffffu), wbase + (y >> 16)));
        stg_stream_u32(dg + head + 4 * k, __funnelshift_r(d0, d1, sh8));
    }
    // the (at most three + three) entries in front of the first and behind the last whole quad: one lane each
    const uint32_t e1 = lane < 4 ? lane : head + 4 * nq + (lane - 4);
    if (lane < 8 && e1 < (lane < 4 ? head : n)) {
        stg_stream_u32(xg + e1, wbase + sxs[e1]);
        stg_stream_u8(dg + e1, sd[e1]);
    }
}

// n difference bytes that lie compacted in shared memory at `sv` (16-byte aligned) go to df_out + g0 as whole words:
// aligned 4-byte stores, the source cut out of two shared words with a funnel shift; the (at most three + three) bytes in
// front of the first and behind the last whole word one by one.  The caller has checked g0 + n <= capacity.
__device__ __forceinline__ void flush_diff_shifted(uint32_t sv, uint8_t *df_out, size_t g0, uint32_t n, uint32_t lane)
{
    const uint32_t a = (4u - (uint32_t)(g0 & 3)) & 3u; // bytes in front of the first rank that is a multiple of 4
    const uint32_t head = min(a, n);
    const uint32_t nq = (n - head) >> 2;
    uint8_t *dg = df_out + g0;
    const uint32_t sh8 = 8u * a;
#pragma unroll 2
    for (uint32_t k = lane; k < nq; k += 32) {
        uint32_t d0, d1 = 0;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(d0) : "r"(sv + 4 * k) : "memory");
        if (a) asm volatile("ld.shared.u32 %0, [%1];" : "=r"(d1) : "r"(sv + 4 * k + 4) : "memory"); // (a == 0: word k alone)
        stg_stream_u32(dg + head + 4 * k, __funnelshift_r(d0, d1, sh8));
    }
    const uint32_t e1 = lane < 4 ? lane : head + 4 * nq + (lane - 4);
    if (lane < 8 && e1 < (lane < 4 ? head : n)) stg_stream_u8(dg + e1, lds_u8(sv + e1));
}

// Batches: one frame of each of up to kMaxBatch camera streams in one launch (k_stream_ws_batch).  Step q is camera q
// (every frame fits one pass, nseg == 1); the pointers of camera q come from this table, which travels in the kernel
// parameters (kMaxBatch * 72 bytes): no upload, nothing to keep alive after the launch.
constexpr int kMaxBatch = 64;
struct BatchCam {
    const uint8_t *frame;  // the camera's frame (16-byte aligned)
    uint8_t *ref;          // its reference frame
    unsigned int *pos;     // its count
    int *xs;               // its payload (capacity StreamParams::cap)
    uint8_t *diff;
    uint8_t *show;         // its display frame (MODE 1,2,3,4,6)
    uint8_t *gray1;        // MODE 5/7: its gray bytes and histogram
    unsigned int *hist;
    unsigned int *status;  // its StatusBits
};
struct BatchTable {
    BatchCam cam[kMaxBatch];
};

// The body of k_stream_ws and of k_stream_ws_batch.  BATCH: step q is the single pass of camera q, every per-frame
// pointer comes from cams[q], and the reference goes through L2 step by step (each step is another camera's reference:
// the !REFREG reload / store, at the camera's address).
template <int MODE, bool HI, bool REFREG, bool BATCH>
__device__ __forceinline__ void ws_body(const StreamParams &p, const BatchCam *cams)
{
    static_assert(!(BATCH && REFREG), "a batch reloads the reference of every step");
    extern __shared__ __align__(128) unsigned char smem[];
    // role of a warp: the scheduler arbitrates highest-warp-id-first, so which group gets the upper half decides who
    // wins when both want an issue slot
#ifdef CVS_WS_FRONT_HIGH
    const uint32_t tid = threadIdx.x ^ (uint32_t)kWsFrontThreads; // front = hardware warps 16..31
#else
    const uint32_t tid = threadIdx.x;
#endif
    const uint32_t lane = tid & 31, warp = tid >> 5;
    const uint32_t b = blockIdx.x, G = gridDim.x;
    const uint32_t N = p.nbytes;
    const uint32_t nsteps = (uint32_t)p.nframes * p.nseg;
    const uint32_t nstages = p.nstages;
    const uint32_t smem0 = smem_u32(smem);
    const uint32_t msk_stride = WsLayout::msk_stride(p.cps), stage_bytes = WsLayout::stage_bytes(p.cps);
    const uint32_t nact = msk_stride / 16u; // front threads whose warp holds chunks (cps rounded up to whole warps)
    const uint32_t stage_addr = smem0 + WsLayout::stage0(p.cps, nstages);
    const uint32_t msk_addr = smem0 + WsLayout::msk;
    const uint32_t bar_full = smem0 + WsLayout::bar_full, bar_fdone = smem0 + WsLayout::bar_fdone,
                   bar_base = smem0 + WsLayout::bar_base;
    uint32_t *done = reinterpret_cast<uint32_t *>(smem + WsLayout::done);
    uint32_t *fcnt = reinterpret_cast<uint32_t *>(smem + WsLayout::fcnt);
    uint32_t *ftot = reinterpret_cast<uint32_t *>(smem + WsLayout::ftot);
    uint32_t *sbase = reinterpret_cast<uint32_t *>(smem + WsLayout::base);
    uint32_t *wtot = reinterpret_cast<uint32_t *>(smem + WsLayout::wtot);
    constexpr bool kBinarize = (MODE == kModeBinarize || MODE == kModeBinarizeAvg);
    constexpr bool kGrayW = (MODE == kModeGrayWeighted || MODE == kModeBinarize);

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
    // one thread: refill ring stage st with the slice of step q
    auto issue = [&](uint32_t q, uint32_t st) {
        const uint32_t t = (REFREG || BATCH) ? q : q / p.nseg, s = (REFREG || BATCH) ? 0u : q - t * p.nseg;
        uint32_t off, bytes;
        slice(s, off, bytes);
        if (bytes) {
            const uint64_t pol = l2_policy_evict_first();
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); // parked bytes were written through the generic proxy
            mbar_expect_tx(bar_full + 8 * st, bytes);
            bulk_g2s(stage_addr + st * stage_bytes, (BATCH ? cams[t].frame : p.frames + (size_t)t * p.frame_stride) + off, bytes,
                     bar_full + 8 * st, pol);
        } else {
            // a block whose slice lies past the end of the frame still hands the stage over: the front warps must not
            // run ahead of the back warps by more than the ring (fdone[st] would complete twice before it is waited for)
            mbar_arrive(bar_full + 8 * st);
        }
    };

    if (tid == 0) {
#pragma unroll
        for (int i = 0; i < kStages; i++) {
            mbar_init(bar_full + 8 * i, 1);
            mbar_init(bar_fdone + 8 * i, kWsFrontWarps);
            mbar_init(bar_base + 8 * i, 1);
            mbar_init(bar_base + 8 * (i + kStages), 1);
            done[i] = 0;
            fcnt[i] = 0;
            ftot[i] = 0;
        }
        mbar_init_fence();
    }
    if (MODE == kModeHeat) {
        uint32_t *slut = reinterpret_cast<uint32_t *>(smem + WsLayout::lut);
        for (uint32_t i = tid; i < 766; i += kWsThreads) slut[i] = p.heat_lut[i];
    }
    if (kBinarize) {
        uint32_t *shist = reinterpret_cast<uint32_t *>(smem + WsLayout::hist);
        for (uint32_t i = tid; i < 256 * kWsHistCopies; i += kWsThreads) shist[i] = 0;
    }
    __syncthreads();
    if (tid == 0)
        for (uint32_t q = 0; q < nstages && q < nsteps; q++) issue(q, q);

    // a spin wait that gave up once stops every later wait of the thread (the launch must terminate); the status word
    // tells the host
    bool tripped = false;
    auto wait_bar = [&](uint32_t bar, uint32_t parity, uint32_t sleep_ns) {
        if (!tripped && !mbar_wait(bar, parity, sleep_ns)) {
            tripped = true;
            atomicOr(p.status, kStatusWatchdog);
        }
    };

    if (warp < (uint32_t)kWsFrontWarps) {
        // =====================================================================================================
        // FRONT: the per-word pass
        // =====================================================================================================
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(CVS_WS_FRONT_REGS));
        uint32_t *slut = reinterpret_cast<uint32_t *>(smem + WsLayout::lut);
        uint32_t *shist = reinterpret_cast<uint32_t *>(smem + WsLayout::hist);
        // bank-conflict-free 16-byte shared accesses: lanes with bit 2 set keep their two 48-byte pixel groups in
        // swapped order ("slot" order), see k_stream
        const uint32_t sw = ((lane >> 2) & 1u) * (uint32_t)kGroupBytes;
        auto voff = [&](int v) -> uint32_t { return v < 3 ? 16u * v + sw : 16u * v - sw; };
        uint32_t r[kChunkWords];
        const uint64_t keep = l2_policy_evict_last();
        bool dirty = false;
        uint32_t coff = 0, nv = 0, sbytes = 0;
        auto geometry = [&](uint32_t s) {
            uint32_t soff;
            slice(s, soff, sbytes);
            uint64_t c = ((uint64_t)s * G + b) * p.cps + tid;
            bool ok = tid < p.cps && c < p.nchunks;
            coff = ok ? (uint32_t)(c * kChunkBytes) : 0u;
            nv = ok ? min(N - coff, (uint32_t)kChunkBytes) : 0u;
        };
        // rb: the reference frame of the step's camera (p.ref unless BATCH)
        auto load_ref = [&](uint8_t *rb) {
            if (nv) {
#pragma unroll
                for (int v = 0; v < kChunkWords / 4; v++) {
                    uint4 a = ldg_keep(rb + coff + voff(v), keep);
                    r[4 * v] = a.x; r[4 * v + 1] = a.y; r[4 * v + 2] = a.z; r[4 * v + 3] = a.w;
                }
            } else {
#pragma unroll
                for (int k = 0; k < kChunkWords; k++) r[k] = 0;
            }
        };
        auto store_ref = [&](uint8_t *rb) {
#pragma unroll
            for (int v = 0; v < kChunkWords / 4; v++)
                stg_keep(rb + coff + voff(v), make_uint4(r[4 * v], r[4 * v + 1], r[4 * v + 2], r[4 * v + 3]), keep);
        };
        geometry(0);
        if (REFREG) load_ref(p.ref);

        uint32_t phase = 0, st = 0, t = 0, s = 0;
        for (uint32_t q = 0; q < nsteps; q++) {
            if (!REFREG) {
                if (!BATCH) geometry(s);
                // a batch has one geometry for all its steps; opaque here, so that what derives from it is recomputed per
                // step instead of being held (spilled) across the loop
                else asm volatile("" : "+r"(coff), "+r"(nv));
                load_ref(BATCH ? cams[q].ref : p.ref); // L2 hit (a batch: the camera's reference, from HBM unless
                                                       // recently used); issued before the wait on the frame slice
            }
            wait_bar(bar_full + 8 * st, (phase >> st) & 1u, CVS_WS_SLEEP_FULL); // completes at once for an empty slice (see issue())
            phase ^= 1u << st;
            const uint32_t myaddr = stage_addr + st * stage_bytes + tid * kChunkBytes;
            uint32_t m[kMaskWords] = {0, 0, 0};
            constexpr bool kStreamLoad = (MODE == kModeNone);
            // the chunk that holds the end of the frame: bytes past N never differ (slot word k of the chunk)
            auto clip_word = [&](int k, uint32_t cw) -> uint32_t {
                const int vb = (int)nv - (int)(voff(k >> 2) + 4 * (k & 3));
                const uint32_t vm = vb >= 4 ? 0xffffffffu : (vb <= 0 ? 0u : ((1u << (8 * vb)) - 1u));
                return (cw & vm) | (r[k] & ~vm);
            };
            // one 16-byte vector of the chunk: flags -> change mask, difference bytes (parked), negative feedback
            //                                                                              (test.cu:565-570)
            auto pass_vector = [&](int v, const uint32_t (&cv)[4]) {
                uint32_t dv[4];
#pragma unroll
                for (int h = 0; h < 4; h += 2) {
                    const int k = 4 * v + h;
                    const uint32_t f0 = changed80<HI>(absdiff4(cv[h], r[k]), p.addc);
                    const uint32_t f1 = changed80<HI>(absdiff4(cv[h + 1], r[k + 1]), p.addc);
                    const uint32_t g8 = __umulhi(f1 + (f0 >> 4), 0x20408100u);
                    m[k >> 3] = __byte_perm(m[k >> 3], g8, ((k >> 1) & 3) == 0 ? 0x3214 : ((k >> 1) & 3) == 1 ? 0x3240
                                                          : ((k >> 1) & 3) == 2 ? 0x3410 : 0x4210);
                    dv[h] = sub4<true>(cv[h], r[k]);
                    dv[h + 1] = sub4<true>(cv[h + 1], r[k + 1]);
                    const uint32_t fm0 = spread80(f0), fm1 = spread80(f1);
                    r[k] = (cv[h] & fm0) | (r[k] & ~fm0);
                    r[k + 1] = (cv[h + 1] & fm1) | (r[k + 1] & ~fm1);
                }
                asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(myaddr + voff(v)), "r"(dv[0]), "r"(dv[1]), "r"(dv[2]),
                             "r"(dv[3])
                             : "memory");
            };

            // display filter on the same registers (reference as it was BEFORE this frame), then the pass
            if (MODE != kModeNone && nv) {
#pragma unroll
                for (int g = 0; g < kGroupsPerThread; g++) {
                    const uint32_t gb = sw ? (uint32_t)(1 - g) * kGroupBytes : (uint32_t)g * kGroupBytes;
                    const uint32_t goff = p.index_base + coff + gb; // byte offset of the group in the whole frame
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
                        store_group((BATCH ? cams[q].show : p.show + (size_t)t * p.show_stride) + goff, o, gnv);
                    } else if (MODE == kModeRedBlack || MODE == kModeRedOverlap) {
                        uint32_t mk[kGroupWords];
#pragma unroll
                        for (int k = 0; k < kGroupWords; k++) mk[k] = changed80<HI>(absdiff4(cg[k], rg[k]), p.addc);
                        group_red<MODE == kModeRedOverlap>(mk, rg, o);
                        store_group((BATCH ? cams[q].show : p.show + (size_t)t * p.show_stride) + goff, o, gnv);
                    } else if (MODE == kModeGrayWeighted || MODE == kModeGrayAverage) {
                        group_gray3<kGrayW>(cg, o);
                        store_group((BATCH ? cams[q].show : p.show + (size_t)t * p.show_stride) + goff, o, gnv);
                    } else if (kBinarize) {
                        uint32_t g4[4];
                        group_gray1<kGrayW>(cg, g4);
                        const uint32_t npx = gnv / 3u;
                        uint8_t *gdst = (BATCH ? cams[q].gray1 : p.gray1 + (size_t)t * p.gray_stride) + goff / 3u;
                        if (npx == (uint32_t)kGroupPixels) stg_keep(gdst, make_uint4(g4[0], g4[1], g4[2], g4[3]), keep);
#pragma unroll
                        for (int px = 0; px < kGroupPixels; px++) {
                            if ((uint32_t)px < npx) {
                                uint32_t gv = byte_of(g4[px >> 2], px & 3);
                                if (npx != (uint32_t)kGroupPixels) gdst[px] = (uint8_t)gv;
#ifndef CVS_EXP_NO_HIST // (timing experiment: the atomics are 0.68 of mode 5's 7.87 us per frame; the weighted gray of
                        //  32 pixels per thread, ~15 instructions each, is what mode 5 costs over mode 0)
                                atomicAdd(&shist[gv * kWsHistCopies + (lane & (kWsHistCopies - 1))], 1u); // server.cpp:103-106
#endif
                            }
                        }
                    }
#pragma unroll
                    for (int v = 0; v < kGroupWords / 4; v++) {
                        const uint32_t cv[4] = {cg[4 * v], cg[4 * v + 1], cg[4 * v + 2], cg[4 * v + 3]};
                        pass_vector(g * (kGroupWords / 4) + v, cv);
                    }
                }
            }
#ifdef CVS_PROFILING
            if (p.debug & 4u) nv = 0; // timing experiment: ingest only (results wrong by construction)
#endif
            if (kStreamLoad && nv == (uint32_t)kChunkBytes) {
                // the common case as ONE basic block (no per-vector test for the end of the frame), two vectors of look-ahead:
                // the scheduler can interleave the six independent vector passes, which is what hides the ALU latency with
                // only 3.5 front warps per scheduler
                uint4 n0 = lds128(myaddr + voff(0)), n1 = lds128(myaddr + voff(1));
#pragma unroll
                for (int v = 0; v < kChunkWords / 4; v++) {
                    const uint32_t cv[4] = {n0.x, n0.y, n0.z, n0.w};
                    n0 = n1;
                    if (v + 2 < kChunkWords / 4) n1 = lds128(myaddr + voff(v + 2));
                    pass_vector(v, cv);
                }
            } else if (kStreamLoad && nv) {
                // the chunk that holds the end of the frame
#pragma unroll 1
                for (int pass = 0; pass < 1; pass++) {
#pragma unroll
                    for (int v = 0; v < kChunkWords / 4; v++) {
                        const uint4 nx = lds128(myaddr + voff(v));
                        uint32_t cv[4] = {nx.x, nx.y, nx.z, nx.w};
#pragma unroll
                        for (int h = 0; h < 4; h++) cv[h] = clip_word(4 * v + h, cv[h]);
                        pass_vector(v, cv);
                    }
                }
            }
            if (sw) { // slot order -> byte order: rotate the 96-bit mask by 48
                const uint32_t n0 = __funnelshift_r(m[1], m[2], 16), n1 = __funnelshift_r(m[2], m[0], 16),
                               n2 = __funnelshift_r(m[0], m[1], 16);
                m[0] = n0; m[1] = n1; m[2] = n2;
            }
            if (__builtin_expect(nv < (uint32_t)kChunkBytes, 0)) { // bytes past the end of the frame are never entries
#pragma unroll
                for (int w = 0; w < kMaskWords; w++) {
                    const int vb = (int)nv - 32 * w;
                    m[w] &= vb >= 32 ? 0xffffffffu : (vb <= 0 ? 0u : ((1u << vb) - 1u));
                }
            }
            if (m[0] | m[1] | m[2]) {
                if (REFREG) dirty = true;
                else store_ref(BATCH ? cams[q].ref : p.ref);
            }
            const uint32_t cnt = (uint32_t)__popc(m[0]) + (uint32_t)__popc(m[1]) + (uint32_t)__popc(m[2]);
            // hand the step to the back warps: (mask, count) per chunk, entries of this warp
            if (tid < nact)
                asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(msk_addr + st * msk_stride + 16 * tid), "r"(m[0]),
                             "r"(m[1]), "r"(m[2]), "r"(cnt)
                             : "memory");
            const uint32_t wsum = warp_add(cnt);
            if (lane == 0) {
                wtot[st * 16 + warp] = wsum;
#ifndef CVS_WS_SCAN_PUBLISH
                // the block total of the step goes out to the other blocks as early as possible: the last front warp to
                // get here publishes it (the back warps' look-back then rarely has to wait for a predecessor).  Publishing
                // from the look-back warp instead (CVS_WS_SCAN_PUBLISH) makes the pass alone 4 % faster (1.58 vs 1.65 us per
                // frame) and the whole kernel 4 % slower at 1 % density (2.28 vs 2.19): the look-backs start later.
                atomicAdd(&ftot[st], wsum);
                __threadfence_block();
                if (atomicAdd(&fcnt[st], 1u) == (uint32_t)kWsFrontWarps - 1u) {
                    __threadfence_block();
                    const uint32_t total = atomicExch(&ftot[st], 0u);
                    fcnt[st] = 0;
                    desc_publish(p.desc + (size_t)q * (G + 1) + b, ((unsigned long long)p.epoch << 32) | total);
                }
#endif
            }
            if (kBinarize && (BATCH || s == p.nseg - 1)) {
                // histogram of the frame complete: flush and clear (front warps only: named barrier 1)
                asm volatile("bar.sync 1, %0;" ::"n"(kWsFrontThreads) : "memory");
                for (uint32_t i = tid; i < 256; i += kWsFrontThreads) {
                    uint32_t hv = 0;
#pragma unroll
                    for (int c = 0; c < kWsHistCopies; c++) {
                        hv += shist[i * kWsHistCopies + c];
                        shist[i * kWsHistCopies + c] = 0;
                    }
                    if (hv) atomicAdd((BATCH ? cams[q].hist : p.hist + (size_t)t * 256) + i, hv);
                }
                asm volatile("bar.sync 1, %0;" ::"n"(kWsFrontThreads) : "memory");
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_fdone + 8 * st); // release: the warp's shared stores above are visible to the waiters
            if (REFREG || BATCH) ++t;
            else if (++s == p.nseg) { s = 0; ++t; }
            if (++st == nstages) st = 0;
        }
        if (REFREG && dirty) store_ref(p.ref);
    } else {
        // =====================================================================================================
        // BACK: block scan, cross-block look-back, emission of the (index, value) entries
        // =====================================================================================================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(CVS_WS_BACK_REGS));
        // back warp w emits the chunks front warp w holds.  Measured and rejected (round 2, us per 1080p frame at
        // 1 / 10 / 50 % against 2.18 / 2.97 / 5.72): dealing the block's chunks out evenly to all sixteen back warps (28
        // each instead of 32 for 13.7 warps) 2.31 / 3.25 / 5.67 -- the look-back warp then has entries of its own and
        // starts the next look-back late; letting the front warp store the upper half of its own chunks in dense steps
        // (ranks scanned by the front, posted in the mask queue) 2.36 / 2.88 / 7.53 -- the front then waits for the
        // global offset and its next pass starts late, so pass and emission no longer overlap; a LAZY difference for
        // sparse warps (the front parks current ^ reference, 7 instead of 10 ALU instructions per word, and the back warp
        // rebuilds the few difference bytes from the frame in global memory) 3.20 / 3.08 / 5.68 -- the pass alone drops
        // from 1.65 to 1.41 us per frame, but the scattered byte loads from L2 / HBM put more than a microsecond of
        // latency into every step of a back warp.
        const uint32_t bw = warp - kWsFrontWarps;
        const uint32_t per = 32;
        const uint32_t c0 = per * bw;                 // first chunk (= front thread) of this warp
        const uint32_t ftid = c0 + lane;              // front thread whose chunk this lane emits
        const bool has_chunk = ftid < nact;
        const bool scan_warp = bw == (uint32_t)kWsBackWarps - 1;
        uint16_t *sxs = reinterpret_cast<uint16_t *>(smem + WsLayout::sxs) + bw * SmemLayout::kXsHalves;
        uint8_t *sd = smem + WsLayout::sd + bw * SmemLayout::kSdBytes;
        const uint32_t cap32 = p.cap > 0xffffffffull ? 0xffffffffu : (uint32_t)p.cap;

        uint32_t ph_f = 0, ph_b = 0, st = 0, t = 0, s = 0;
        for (uint32_t q = 0; q < nsteps; q++) {
            if (BATCH) asm volatile("" : "+l"(sxs), "+l"(sd)); // (as the front's geometry: recomputed, not spilled)
            // byte offset of lane 0's chunk in the frame (chunk S of the warp starts 96*S bytes later)
            const uint32_t wcoff = p.index_base + (uint32_t)((((uint64_t)s * G + b) * p.cps + c0) * kChunkBytes);
            // global-offset slot of the step: 2 x nstages slots, because a sparse warp lets its stage go before it waits
            // for the offset, so the look-back warp may be up to nstages steps ahead of it (not more: the bulk copy of
            // step q + nstages + 1 needs this warp's release of step q + 1)
            const uint32_t bslot = q & (2u * kStages - 1u);
            wait_bar(bar_fdone + 8 * st, (ph_f >> st) & 1u, CVS_WS_SLEEP_BACK);
            ph_f ^= 1u << st;
            uint32_t m[kMaskWords] = {0, 0, 0}, cnt = 0;
            if (has_chunk)
                asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];"
                             : "=r"(m[0]), "=r"(m[1]), "=r"(m[2]), "=r"(cnt)
                             : "r"(msk_addr + st * msk_stride + 16 * ftid)
                             : "memory");
            uint32_t wexc, total; // entries of the block in front of this warp's chunks / of the whole block
            {
                const uint32_t v = lane < (uint32_t)kWsFrontWarps ? wtot[st * 16 + lane] : 0u;
                total = warp_add(v);
                wexc = warp_add(lane < bw ? v : 0u);
            }
#ifdef CVS_WS_SCAN_PUBLISH
            if (scan_warp && lane == 0)
                desc_publish(p.desc + (size_t)q * (G + 1) + b, ((unsigned long long)p.epoch << 32) | total);
#endif
            const uint32_t incl = warp_incl_scan(cnt, lane);
            const uint32_t wtotal = __shfl_sync(0xffffffffu, incl, 31);
            const uint32_t wrank = incl - cnt;
            const uint32_t dv0 = stage_addr + st * stage_bytes + c0 * kChunkBytes; // parked bytes of lane 0's chunk
            // this warp is done with the ring stage; the last warp to say so refills it
            auto release_stage = [&]() {
                __syncwarp();
                if (lane == 0) {
                    __threadfence_block();
                    if (atomicAdd(&done[st], 1u) == (uint32_t)kWsBackWarps - 1u) {
                        done[st] = 0;
                        if (q + nstages < nsteps) issue(q + nstages, st);
                    }
                }
            };
            // A warp whose entries fit its window copies them out of the stage NOW, in rank order, and lets the stage
            // go before it waits for the block's global offset: the look-back latency is then outside the stage's
            // lifetime (bulk copy -> pass -> this copy), which is what bounds the step rate with four stages.
            const bool sparse = wtotal <= (uint32_t)kWarpEntries;
#ifdef CVS_PROFILING
            if (p.debug & 2u) { // timing experiment: no emission at all (results wrong by construction)
                release_stage();
                ph_b ^= 1u << bslot;
                if (REFREG || BATCH) ++t;
                else if (++s == p.nseg) { s = 0; ++t; }
                if (++st == nstages) st = 0;
                continue;
            }
#endif
            if (sparse) {
                if (wtotal) {
                    uint32_t o = wrank;
#pragma unroll
                    for (int w = 0; w < kMaskWords; w++)
                        emit_bits(m[w], 32 * w, lane * kChunkBytes, dv0 + lane * kChunkBytes, sxs, sd, o);
                }
                release_stage();
            }
            if (scan_warp) {
                // (after this warp has let go of the stage: the look-back must not sit inside the stage's lifetime)
                // ---- cross-block exchange of the step: sum the predecessors' totals (each lane reads up to kWsLook
                //      descriptors, all in flight together: one L2 round trip)
                unsigned long long *row = p.desc + (size_t)q * (G + 1); // (the block's own total was published by the front)
                unsigned long long pv[kWsLook], pv2 = 0;
                const bool has2 = !REFREG && s > 0 && lane == 31;
#pragma unroll
                for (int i = 0; i < kWsLook; i++) {
                    pv[i] = 0;
                    if (lane + 32 * i < b) pv[i] = desc_peek(row + lane + 32 * i);
                }
                if (has2) pv2 = desc_peek(row - 1); // running total of the earlier segments: slot G of the previous step
                uint32_t prior = 0;                 // entries of the frame that earlier bands (launches) produced
                if (p.pos_prior && lane == 0) prior = p.pos_prior[t];
                auto settle = [&](unsigned long long v, const unsigned long long *d) -> uint32_t {
                    uint32_t polls = 0;
                    while ((uint32_t)(v >> 32) != p.epoch && !tripped) {
                        __nanosleep(32);
                        v = desc_peek(d);
                        if (++polls > kWatchdogPolls) {
                            tripped = true;
                            atomicOr(p.status, kStatusWatchdog);
                        }
                    }
                    return (uint32_t)v;
                };
                uint32_t part = prior;
#pragma unroll
                for (int i = 0; i < kWsLook; i++)
                    if (lane + 32 * i < b) part += settle(pv[i], row + lane + 32 * i);
                if (has2) part += settle(pv2, row - 1);
                const uint32_t base = warp_add(part);
                if (lane == 0) {
                    sbase[bslot] = base;
                    if (b == G - 1) {
                        if (!REFREG && !BATCH) desc_publish(row + G, ((unsigned long long)p.epoch << 32) | (base + total));
                        if (BATCH) *cams[q].pos = base + total;
                        else if (REFREG || s == p.nseg - 1) p.pos[t] = base + total;
                    }
                    if ((size_t)base + total > p.cap) atomicOr(BATCH ? cams[q].status : p.status, kStatusCapacity);
                    mbar_arrive(bar_base + 8 * bslot);
                }
            }
            if (wtotal) {
                wait_bar(bar_base + 8 * bslot, (ph_b >> bslot) & 1u, CVS_WS_SLEEP_BACK);
                const uint32_t base = *reinterpret_cast<volatile uint32_t *>(sbase + bslot);
                int *xs_out = BATCH ? cams[q].xs : p.xs + (size_t)t * p.cap;
                uint8_t *df_out = BATCH ? cams[q].diff : p.diff + (size_t)t * p.cap;
                asm volatile("" : "+l"(xs_out), "+l"(df_out)); // keep the frame offset out of the emission loops
                const size_t g0 = (size_t)base + wexc;
                if (sparse) {
                    flush_warp_shifted(sxs, sd, wcoff, xs_out, df_out, g0, wtotal, p.cap, lane);
                    __syncwarp(); // the window is refilled by the next step
                } else if (g0 + wtotal <= (size_t)cap32) {
#ifdef CVS_WS_DENSE_STAGED
                    // Measured and rejected (round 2, bit-exact): indices straight to global memory, difference bytes
                    // compacted in place in the stage and flushed as whole words instead of one st.global.u8 per entry --
                    // 6.38 instead of 5.75 us per frame at 50 % (3.21 / 2.96 at 10 % from the larger kernel): the dense
                    // emission is bound by the instructions it issues, not by its byte stores.
                    emit_coop<false, true>(m, wcoff, dv0, xs_out, df_out, (uint32_t)g0 + wrank, cap32, lane, smem_u32(sxs), per,
                                           (uint32_t)g0);
                    __syncwarp();
                    flush_diff_shifted(dv0, df_out, g0, wtotal, lane);
#else
                    emit_coop<false>(m, wcoff, dv0, xs_out, df_out, (uint32_t)g0 + wrank, cap32, lane, smem_u32(sxs), per);
#endif
                } else {
                    emit_coop<true>(m, wcoff, dv0, xs_out, df_out, (uint32_t)g0 + wrank, cap32, lane, smem_u32(sxs), per);
                }
            }
            ph_b ^= 1u << bslot; // every step completes its bar_base slot exactly once, waited for or not
            if (!sparse) release_stage(); // a dense warp stores straight out of the stage
            if (REFREG || BATCH) ++t;
            else if (++s == p.nseg) { s = 0; ++t; }
            if (++st == nstages) st = 0;
        }
    }
    // (a batch's watchdog bits go to the first camera's word during the launch: the later steps of a thread that gave
    // up are not run, so every camera is told)
    if (BATCH && tripped)
        for (uint32_t i = 0; i < nsteps; i++) atomicOr(cams[i].status, kStatusWatchdog);
}

template <int MODE, bool HI, bool REFREG>
__global__ void __launch_bounds__(kWsThreads, 1) k_stream_ws(const StreamParams p)
{
    ws_body<MODE, HI, REFREG, false>(p, nullptr);
}

// one frame of each of p.nframes cameras (p.nseg == 1; p.frames, ref, pos, xs, diff, show, gray1, hist unused: see cams)
template <int MODE, bool HI>
__global__ void __launch_bounds__(kWsThreads, 1) k_stream_ws_batch(const StreamParams p, const __grid_constant__ BatchTable tbl)
{
    ws_body<MODE, HI, false, true>(p, tbl.cam);
}

} // namespace cvs
