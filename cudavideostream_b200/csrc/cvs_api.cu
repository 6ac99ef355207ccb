// cvs_api.cu -- host side of libcvs_b200.so: the C ABI declared in include/cvs_b200.h.
//
// Replaces the host orchestration of diff::cuda::CUDACore (server/src/kernels.cu:377-536).  There is
// no CPU fallback anywhere in this file: without an sm_100 device every entry point that would
// compute returns CVS_ERR_NODEVICE.
#include "../../include/cvs_b200.h"

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nvjpeg.h>
#include <vector>
#include <cooperative_groups.h>

#include <algorithm>
#include <atomic>
#include <cassert>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <mutex>
#include <string>
#include <type_traits>

#include "cvs_bayer.cuh"
#include "cvs_filter_kernels.cuh"
#include "cvs_jpeg_host.hpp"
#include "cvs_stream_kernel.cuh"
#include "cvs_stream_ws.cuh"
#include "cvs_yuv.cuh"

namespace {

thread_local char g_err[512] = "";

cvs_status fail(cvs_status st, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return st;
}

#define CU_TRY(expr)                                                                                                   \
    do {                                                                                                               \
        cudaError_t e_ = (expr);                                                                                       \
        if (e_ != cudaSuccess)                                                                                         \
            return fail(CVS_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__);     \
    } while (0)

#define CVS_TRY(expr)                                                                                                  \
    do {                                                                                                               \
        const cvs_status s_ = (expr);                                                                                  \
        if (s_ != CVS_OK) return s_;                                                                                   \
    } while (0)

inline size_t round_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

inline uintptr_t addr_bits(const void *p) { return (uintptr_t)p; }
inline uintptr_t addr_bits(size_t v) { return v; }
// true when every pointer and stride is a multiple of 16 bytes (the kernels' vector loads and stores)
template <class... T>
bool aligned16(T... v)
{
    return ((addr_bits(v) & 15) | ...) == 0;
}

// Device memory owned by the handle (or one of its slots): freed with it.  Grow-only: a buffer that is too small is
// freed and allocated anew, after a synchronise, because earlier launches may still use it.
template <class T>
struct DevBuf {
    T *p = nullptr;
    size_t bytes = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { cudaFree(p); }
    operator T *() const { return p; }

    // any stream of the device may use the buffer: the whole device is synchronised; zero: the new buffer is cleared
    cvs_status grow(size_t need, const char *what, bool zero = false)
    {
        if (need <= bytes) return CVS_OK;
        if (p) CU_TRY(cudaDeviceSynchronize());
        CVS_TRY(replace(need, what));
        if (zero) CU_TRY(cudaMemset(p, 0, need));
        return CVS_OK;
    }
    // only stream `user` uses the buffer: it alone is synchronised
    cvs_status grow_on(cudaStream_t user, size_t need, const char *what)
    {
        if (need <= bytes) return CVS_OK;
        if (p) CU_TRY(cudaStreamSynchronize(user));
        return replace(need, what);
    }

  private:
    cvs_status replace(size_t need, const char *what)
    {
        // forget the old buffer before anything can fail: a later call (or the destructor) must not free it again
        cudaFree(p);
        p = nullptr;
        bytes = 0;
        const cudaError_t e = cudaMalloc(&p, need);
        if (e != cudaSuccess) {
            cudaGetLastError();
            p = nullptr;
            return fail(CVS_ERR_NOMEM, "%s: %zu bytes of device memory do not fit (%s)", what, need, cudaGetErrorString(e));
        }
        bytes = need;
        return CVS_OK;
    }
};

// one word of pinned host memory that a count or status word is copied back into
struct PinnedWord {
    unsigned int *p = nullptr;
    PinnedWord() = default;
    PinnedWord(const PinnedWord &) = delete;
    PinnedWord &operator=(const PinnedWord &) = delete;
    ~PinnedWord() { cudaFreeHost(p); }
    operator unsigned int *() const { return p; }
    cvs_status alloc()
    {
        CU_TRY(cudaHostAlloc(&p, sizeof *p, cudaHostAllocDefault));
        *p = 0;
        return CVS_OK;
    }
};

bool device_is_sm100(int dev)
{
    int major = 0;
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return false;
    return major == 10;
}

// threshold constant for changed80<HI>
void threshold_consts(int thr, bool &hi, uint32_t &addc)
{
    if (thr < -1) thr = -1;   // everything changes
    if (thr > 255) thr = 255; // nothing changes
    hi = thr >= 128;
    uint32_t a = hi ? (uint32_t)(255 - thr) : (uint32_t)(127 - thr);
    addc = a * 0x01010101u;
}

// heat-map colour table: the reference's getHeatPixel evaluated for every possible d
// (tests/heat_map_benchmark/cpu.cu:19-27); entry = B | G<<8 | R<<16
void build_heat_lut(uint32_t *lut)
{
    for (int d = 0; d < 766; d++) {
        float diff1 = d / (255.0 * 2.0);
        int r = (int)fmin(fmax(sin(M_PI * diff1 - M_PI / 2.0) * 255.0, 0.0), 255.0);
        int g = (int)fmin(fmax(sin(M_PI * diff1) * 255.0, 0.0), 255.0);
        int b = (int)fmin(fmax(sin(M_PI * diff1 + M_PI / 2.0) * 255.0, 0.0), 255.0);
        lut[d] = (uint32_t)(b & 255) | ((uint32_t)(g & 255) << 8) | ((uint32_t)(r & 255) << 16);
    }
    lut[766] = lut[767] = 0;
}

// per-device constant tables for the stand-alone filter entry points
std::mutex g_lut_mutex;
uint32_t *g_dev_lut[64] = {nullptr};

cvs_status device_heat_lut(uint32_t **out)
{
    int dev = 0;
    CU_TRY(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) return fail(CVS_ERR_INVALID, "device ordinal %d out of range", dev);
    std::lock_guard<std::mutex> lk(g_lut_mutex);
    if (!g_dev_lut[dev]) {
        uint32_t host[768];
        build_heat_lut(host);
        uint32_t *d = nullptr;
        CU_TRY(cudaMalloc(&d, sizeof host));
        CU_TRY(cudaMemcpy(d, host, sizeof host, cudaMemcpyHostToDevice));
        g_dev_lut[dev] = d;
    }
    *out = g_dev_lut[dev];
    return CVS_OK;
}

int grid_for(size_t items, int block, int sms)
{
    size_t blocks = (items + block - 1) / block;
    size_t cap = (size_t)sms * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

// ---------------------------------------------------------------------------------------------------------------
// nvJPEG, loaded on first use (dlopen: libcvs_b200.so has no link-time dependency on it).  Used by cvs_submit_jpeg /
// cvs_decode_jpeg_device: the capture side of the reference delivers MJPG (server/src/threads.cpp:32-41) and decodes
// it on the CPU; decoding on the GPU replaces the 6.2 MB host-to-device copy of a raw 1080p frame by the ~0.4 MB
// bitstream.  The decode itself is the library's (like calling cuBLAS); everything after it is this library's path.
// ---------------------------------------------------------------------------------------------------------------
struct NvJpegApi {
    void *lib = nullptr;
    nvjpegStatus_t (*CreateEx)(nvjpegBackend_t, nvjpegDevAllocator_t *, nvjpegPinnedAllocator_t *, unsigned int, nvjpegHandle_t *) = nullptr;
    nvjpegStatus_t (*CreateSimple)(nvjpegHandle_t *) = nullptr;
    nvjpegStatus_t (*Destroy)(nvjpegHandle_t) = nullptr;
    nvjpegStatus_t (*StateCreate)(nvjpegHandle_t, nvjpegJpegState_t *) = nullptr;
    nvjpegStatus_t (*StateDestroy)(nvjpegJpegState_t) = nullptr;
    nvjpegStatus_t (*GetImageInfo)(nvjpegHandle_t, const unsigned char *, size_t, int *, nvjpegChromaSubsampling_t *, int *, int *) = nullptr;
    nvjpegStatus_t (*Decode)(nvjpegHandle_t, nvjpegJpegState_t, const unsigned char *, size_t, nvjpegOutputFormat_t, nvjpegImage_t *,
                             cudaStream_t) = nullptr;
    nvjpegStatus_t (*BatchedInit)(nvjpegHandle_t, nvjpegJpegState_t, int, int, nvjpegOutputFormat_t) = nullptr;
    nvjpegStatus_t (*Batched)(nvjpegHandle_t, nvjpegJpegState_t, const unsigned char *const *, const size_t *, nvjpegImage_t *,
                              cudaStream_t) = nullptr;
    bool ok = false;
};
std::mutex g_nvjpeg_mutex;
NvJpegApi g_nvjpeg;

const NvJpegApi *nvjpeg_api()
{
    std::lock_guard<std::mutex> lk(g_nvjpeg_mutex);
    NvJpegApi &a = g_nvjpeg;
    if (a.ok) return &a;
    if (!a.lib) {
        for (const char *name : {"libnvjpeg.so.12", "libnvjpeg.so", "/usr/local/cuda/lib64/libnvjpeg.so.12"}) {
            a.lib = dlopen(name, RTLD_NOW | RTLD_LOCAL);
            if (a.lib) break;
        }
    }
    if (!a.lib) return nullptr;
    a.CreateEx = (decltype(a.CreateEx))dlsym(a.lib, "nvjpegCreateEx");
    a.CreateSimple = (decltype(a.CreateSimple))dlsym(a.lib, "nvjpegCreateSimple");
    a.Destroy = (decltype(a.Destroy))dlsym(a.lib, "nvjpegDestroy");
    a.StateCreate = (decltype(a.StateCreate))dlsym(a.lib, "nvjpegJpegStateCreate");
    a.StateDestroy = (decltype(a.StateDestroy))dlsym(a.lib, "nvjpegJpegStateDestroy");
    a.GetImageInfo = (decltype(a.GetImageInfo))dlsym(a.lib, "nvjpegGetImageInfo");
    a.Decode = (decltype(a.Decode))dlsym(a.lib, "nvjpegDecode");
    a.BatchedInit = (decltype(a.BatchedInit))dlsym(a.lib, "nvjpegDecodeBatchedInitialize");
    a.Batched = (decltype(a.Batched))dlsym(a.lib, "nvjpegDecodeBatched");
    a.ok = a.CreateSimple && a.Destroy && a.StateCreate && a.StateDestroy && a.GetImageInfo && a.Decode;
    return a.ok ? &a : nullptr;
}

constexpr int kSlots = 4; // tickets that may be outstanding per stream

// scratch of the GPU JPEG decoder (cvs_jpeg.cuh), one set per handle: decodes of a handle are ordered on one stream
struct JpegDecoder {
    DevBuf<uint8_t> arena;        // every d_* below points into this one allocation (carve)
    size_t raw_cap = 0, block_cap = 0; // entropy-coded bytes and blocks the arena is carved for
    size_t zero_bytes_fixed = 0;  // bytes in front of the coefficients that every decode clears
    uint8_t *d_raw = nullptr, *d_unst = nullptr; // entropy-coded segment as received / unstuffed (zero-padded)
    uint32_t *d_block_kept = nullptr, *d_block_marks = nullptr, *d_total_bits = nullptr, *d_total_marks = nullptr, *d_seg_start = nullptr;
    uint32_t seg_cap = 0;
    cvs::jpg::Tables *d_tables = nullptr;
    cvs::jpg::Parsed parsed;       // header of the last frame ...
    std::vector<uint8_t> header;   // ... and its bytes up to the scan (a camera repeats them: no table rebuild per frame)
    cvs::jpg::Tables tables_host;  // what d_tables holds
    bool tables_valid = false;
    uint32_t *d_entry = nullptr, *d_used = nullptr, *d_nblk = nullptr, *d_tile_blk = nullptr, *d_hx = nullptr, *d_hy = nullptr, *d_hw = nullptr, *d_hym = nullptr, *d_hwm = nullptr;
    uint8_t *d_hmap = nullptr;
    uint32_t *d_mid_state = nullptr, *d_mid_nblk = nullptr;
    int32_t *d_mid_dc = nullptr;
    int32_t *d_dcs = nullptr, *d_tile_dc = nullptr;
    unsigned int *d_changed = nullptr;
    int16_t *d_coef = nullptr;
    uint8_t *d_planes = nullptr;
    int coop_blocks_per_sm = 0;
    uint32_t sub_bits = 1024;

    // Lays the scratch for raw_cap entropy-coded bytes and block_cap blocks out from `base` and returns its size;
    // base == nullptr only sizes it (the pointers are then null).
    size_t carve(uint8_t *base, size_t raw_cap, size_t block_cap)
    {
        namespace J = cvs::jpg;
        const size_t nsub = (raw_cap * 8 + sub_bits - 1) / sub_bits + 1;
        const size_t nhalf = 2 * nsub, ntile = nhalf / J::kEntropyThreads + 2; // the rounds may work on half subsequences
        const size_t nunstuff = raw_cap / (J::kUnstuffThreads * J::kUnstuffBytes) + 1;
        size_t off = 0;
        auto take = [&](auto *&ptr, size_t count) {
            using T = std::remove_reference_t<decltype(*ptr)>;
            ptr = base ? reinterpret_cast<T *>(base + off) : nullptr;
            off += round_up(count * sizeof(T), 256);
        };
        take(d_changed, J::kRoundCounters);
        take(d_entry, nhalf + 2);
        take(d_unst, raw_cap);
        take(d_coef, block_cap * 64);
        take(d_raw, raw_cap);
        take(d_block_kept, nunstuff);
        take(d_block_marks, nunstuff);
        take(d_seg_start, block_cap + 2);
        take(d_total_bits, 2);
        take(d_tables, 1);
        take(d_used, nhalf);
        take(d_nblk, nhalf);
        take(d_dcs, 3 * nhalf);
        take(d_tile_blk, ntile);
        take(d_tile_dc, 3 * ntile);
        take(d_hx, 6 * nsub);
        take(d_hy, 6 * nsub);
        take(d_hw, 6 * nsub);
        take(d_hym, 6 * nsub);
        take(d_hwm, 6 * nsub);
        take(d_hmap, 16 * nsub);
        take(d_mid_state, J::kMaxSplit * nsub);
        take(d_mid_nblk, J::kMaxSplit * nsub);
        take(d_mid_dc, 3 * J::kMaxSplit * nsub);
        take(d_planes, block_cap * 64 + 256);
        d_total_marks = d_total_bits ? d_total_bits + 1 : nullptr;
        seg_cap = (uint32_t)block_cap + 2;
        if (base) {
            // a decode with restart intervals clears [base, base + zero_bytes_fixed + nblocks * 128) with one memset, so
            // what it must clear besides the coefficients (round counters, entry states, unstuffed string) lies in front
            const uint8_t *coef = reinterpret_cast<uint8_t *>(d_coef);
            zero_bytes_fixed = (size_t)(coef - base);
            assert(reinterpret_cast<uint8_t *>(d_changed + J::kRoundCounters) <= coef &&
                   reinterpret_cast<uint8_t *>(d_entry + nhalf + 2) <= coef && d_unst + raw_cap <= coef);
        }
        return off;
    }
};

// decoder sets of a handle: tickets of cvs_submit_jpeg alternate between two, each decoding on a stream of its own
// (consecutive frames decode side by side); cvs_decode_jpeg_device decodes with the third on the caller's stream
enum JpegSet { kJpegTicketEven, kJpegTicketOdd, kJpegCallerStream, kJpegSets };

struct Slot {
    DevBuf<uint8_t> d_in;      // raw frame as uploaded
    DevBuf<int> d_xs;
    DevBuf<uint8_t> d_diff;
    DevBuf<unsigned int> d_pos;
    DevBuf<uint8_t> d_show;
    PinnedWord h_pos;
    DevBuf<uint32_t> d_starts;        // compact wire format: entries before each tile (ntiles + 2 words), on first use
    DevBuf<uint8_t> d_wire;           // compact wire format: encoded frame when the caller's buffer is not mapped
    nvjpegJpegState_t jpeg_state = nullptr; // cvs_submit_jpeg: decoder state of this slot (on first use)
    DevBuf<uint8_t> d_cam;            // cvs_submit_yuv / _bayer: the camera's raw frame as uploaded (on first use)
    uint8_t *u_wire = nullptr;        // caller's buffer of a cvs_submit_wire ticket (nullptr: reference-format ticket)
    DevBuf<unsigned int> d_status;    // StatusBits of this ticket's launches (cleared at submit)
    PinnedWord h_status;              // copy of d_status, valid once ev_pos has fired
    cudaEvent_t ev_h2d0 = nullptr, ev_h2d1 = nullptr, ev_k0 = nullptr, ev_k1 = nullptr, ev_pos = nullptr,
                ev_p0 = nullptr, ev_done = nullptr;
    bool busy = false;
    bool copied = false; // payload fetched with cudaMemcpyAsync in cvs_wait (ev_done is valid)
    bool pushed = false; // payload already written to the caller's pinned buffers by k_payload_push
    uint32_t spec = 0;   // entries copied speculatively behind the count (cvs_submit_io); 0 = none
    uint64_t ticket = 0;
    uint8_t *u_frame = nullptr;
    int *u_xs = nullptr;
    unsigned int *u_pos = nullptr;
};

double host_us()
{
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e6 + ts.tv_nsec * 1e-3;
}

// true when `host` is pinned host memory the current device can write through `*dev`
bool mapped_device_pointer(const void *host, void **dev)
{
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, host) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    if (attr.type != cudaMemoryTypeHost || !attr.devicePointer) return false;
    *dev = attr.devicePointer;
    return true;
}

// the stream kernels: k_stream (one warp group; walks a frame in segments with the reference through L2), k_stream_ws
// (front / back warp groups; a frame or band in one pass with the reference in registers), k_stream_ws_batch (k_stream_ws
// over one frame of each of several handles)
enum Family { kFamStream, kFamWs, kFamBatch, kFamilies };
typedef void (*StreamKernel)(const cvs::StreamParams);
typedef void (*BatchKernel)(const cvs::StreamParams, const cvs::BatchTable);

// every variant of a stream kernel, by display mode and threshold form: [mode][hi]
#define CVS_BY_MODE(K)                                                                                                 \
    {{K<0, false>, K<0, true>}, {K<1, false>, K<1, true>}, {K<2, false>, K<2, true>}, {K<3, false>, K<3, true>},     \
     {K<4, false>, K<4, true>}, {K<5, false>, K<5, true>}, {K<6, false>, K<6, true>}, {K<7, false>, K<7, true>}}
const StreamKernel kStreamKernels[8][2] = CVS_BY_MODE(cvs::k_stream);
const StreamKernel kWsKernels[8][2] = CVS_BY_MODE(cvs::k_stream_ws);
const BatchKernel kBatchKernels[8][2] = CVS_BY_MODE(cvs::k_stream_ws_batch);
#undef CVS_BY_MODE
static_assert(cvs::kMaxBatch == CVS_MAX_BATCH, "batch table and public limit");

} // namespace

struct cvs_stream_s {
    int width = 0, height = 0, threshold = 20, mode = 0, noise_filter = 0, ksize = 3, device = 0;
    int max_sequence = 512;
    uint32_t N = 0, N16 = 0, nchunks = 0, npix = 0;
    size_t Npad = 0, P16 = 0;
    bool hi = false;
    uint32_t addc = 0;
    bool trace = false;
    cudaEvent_t ev_base = nullptr;
    uint32_t pred = 0;        // predicted entries of the next frame (previous count + margin)
    cvs::ConvWeights weights;
    int sms = 0;
    // glyph atlas
    DevBuf<uint8_t> d_glyphs;
    int glyph_w = 0, glyph_h = 0;
    std::string glyph_chars;
    // device state
    DevBuf<uint8_t> d_ref;
    DevBuf<uint32_t> d_lut;
    DevBuf<unsigned int> d_status;
    PinnedWord h_status;
    DevBuf<unsigned long long> d_desc;  // look-back descriptors of the stream kernels
    JpegDecoder jd[kJpegSets];          // the library's own decoder (cvs_jpeg.cuh), scratch allocated on first use
    cudaStream_t s_jpg[kJpegCallerStream] = {}; // decode streams of the cvs_submit_jpeg sets (on first use)
    bool jpeg_own_only = false;         // own decoder only: refuse the forms it does not cover instead of using nvJPEG
    nvjpegHandle_t jpeg = nullptr;      // cvs_submit_jpeg / cvs_decode_jpeg_device: nvJPEG handle (on first use)
    bool jpeg_batched = false;          // the handle's backend wants the batched entry points (hardware engine / GPU Huffman)
    nvjpegJpegState_t jpeg_state = nullptr; // decoder state of cvs_decode_jpeg_device
    uint32_t epoch = 0;
    // scratch that grows with the longest piece seen
    DevBuf<unsigned int> d_band_pos; // banded launches: two arrays of per-frame counts so far (ping-pong)
    DevBuf<uint8_t> d_work;      // filtered / overlaid frames
    DevBuf<uint8_t> d_gray1;     // binarise: 1 B per pixel per frame
    DevBuf<unsigned int> d_hist;
    DevBuf<int> d_thr;
    cudaStream_t s_comp = nullptr, s_h2d = nullptr, s_d2h = nullptr, s_pay = nullptr;
    Slot slot[kSlots];
    int last_slot = -1; // slot of the most recently completed ticket (for cvs_get_timing)
    int occ[kFamilies][8][2] = {}; // co-resident blocks per SM of each stream-kernel variant (0 = not queried yet)
    uint64_t next_ticket = 1;
    uint64_t launches = 0;
    float t_h2d = 0, t_kernel = 0, t_d2h = 0;
};

namespace {

cvs_status launch_conv(const uint8_t *in, uint8_t *out, int width, int height, size_t in_stride, size_t out_stride,
                       int nframes, int K, const cvs::ConvWeights &w, cudaStream_t st)
{
    const int rowbytes = 3 * width;
    const bool fast = (rowbytes % 4 == 0) && (in_stride % 4 == 0) && (out_stride % 4 == 0) &&
                      ((uintptr_t)in % 4 == 0) && ((uintptr_t)out % 4 == 0) && (K == 1 || K == 3 || K == 5);
    // K = 1 keeps the one-row kernel; K >= 7 falls to the byte kernel (a K-row float window no longer fits in registers)
    if (fast && (K == 3 || K == 5)) {
        // non-negative weights with a modest sum keep every accumulator inside [0, 2^23): cheap truncation
        bool nonneg = true;
        float sum = 0.f;
        for (int i = 0; i < K * K; i++) { nonneg = nonneg && w.k[i] >= 0.f; sum += w.k[i]; }
        nonneg = nonneg && sum <= 16384.f;
        // two words per thread when every row and frame starts 8-byte aligned (K = 3 only: the K = 5 window would not
        // fit in registers)
        const bool wide = K == 3 && rowbytes % 8 == 0 && in_stride % 8 == 0 && out_stride % 8 == 0 &&
                          (uintptr_t)in % 8 == 0 && (uintptr_t)out % 8 == 0;
        const int wb = wide ? 2 : 1;
        dim3 block(128), grid((rowbytes / (4 * wb) + 127) / 128, (height + cvs::kConvRows - 1) / cvs::kConvRows, nframes);
        if (wide) {
            if (nonneg) cvs::k_conv_strip<3, true, 2><<<grid, block, 0, st>>>(in, out, width, height, in_stride, out_stride, w);
            else cvs::k_conv_strip<3, false, 2><<<grid, block, 0, st>>>(in, out, width, height, in_stride, out_stride, w);
        } else if (K == 3) {
            if (nonneg) cvs::k_conv_strip<3, true, 1><<<grid, block, 0, st>>>(in, out, width, height, in_stride, out_stride, w);
            else cvs::k_conv_strip<3, false, 1><<<grid, block, 0, st>>>(in, out, width, height, in_stride, out_stride, w);
        } else {
            if (nonneg) cvs::k_conv_strip<5, true, 1><<<grid, block, 0, st>>>(in, out, width, height, in_stride, out_stride, w);
            else cvs::k_conv_strip<5, false, 1><<<grid, block, 0, st>>>(in, out, width, height, in_stride, out_stride, w);
        }
    } else if (fast) {
        dim3 block(256), grid((rowbytes / 4 + 255) / 256, height, nframes);
        cvs::k_conv_rows4<1><<<grid, block, 0, st>>>(in, out, width, height, in_stride, out_stride, w);
    } else {
        dim3 block(256), grid((rowbytes + 255) / 256, height, nframes);
        cvs::k_conv_bytes<<<grid, block, 0, st>>>(in, out, width, height, in_stride, out_stride, K, w);
    }
    CU_TRY(cudaGetLastError());
    return CVS_OK;
}

// glyph indices of the overlay text (kernels.cu:466-473); characters outside the atlas are skipped
cvs::OverlayText overlay_text(cvs_handle h, const char *text)
{
    cvs::OverlayText txt;
    txt.n = 0;
    if (text && text[0] && h->d_glyphs && h->glyph_h <= h->height) {
        int n = (int)strlen(text);
        if (n > (int)sizeof txt.idx) n = (int)sizeof txt.idx;
        for (int j = 0; j < n; j++) {
            size_t at = h->glyph_chars.find(text[j]);
            txt.idx[j] = (at == std::string::npos || at > 126) ? (signed char)-1 : (signed char)at;
        }
        txt.n = n;
    }
    return txt;
}

// Pre-pass of `piece` frames in front of the stream kernel: the noise filter writes a private copy of the frames; the
// overlay is blitted into that copy, into a plain copy, or (frames_private) into the frames themselves.  On return
// frames / fstride say where the stream kernel reads.  binarize: the histograms of the piece are cleared.
cvs_status pre_pass(cvs_handle h, const uint8_t *&frames, size_t &fstride, int piece, const cvs::OverlayText &txt,
                    bool frames_private, bool binarize, cudaStream_t st)
{
    if (h->noise_filter) {
        cvs_status s = launch_conv(frames, h->d_work, h->width, h->height, fstride, h->Npad, piece, h->ksize, h->weights, st);
        if (s) return s;
        h->launches++;
        frames = h->d_work;
        fstride = h->Npad;
    } else if (txt.n && !frames_private) {
        CU_TRY(cudaMemcpy2DAsync(h->d_work, h->Npad, frames, fstride, h->N, piece, cudaMemcpyDeviceToDevice, st));
        frames = h->d_work;
        fstride = h->Npad;
    }
    if (txt.n) {
        const int area = 3 * h->glyph_w * h->glyph_h;
        dim3 grid((area + 255) / 256, txt.n, piece);
        cvs::k_overlay<<<grid, 256, 0, st>>>(const_cast<uint8_t *>(frames), fstride, h->width, h->d_glyphs, h->glyph_w,
                                             h->glyph_h, txt);
        CU_TRY(cudaGetLastError());
        h->launches++;
    }
    if (binarize) CU_TRY(cudaMemsetAsync(h->d_hist, 0, (size_t)piece * 256 * sizeof(unsigned int), st));
    return CVS_OK;
}

// binarisation pass 2 of `piece` frames (modes 5, 7): threshold from the histograms, then the 0 / 255 display frames
cvs_status binarize_pass(cvs_handle h, int piece, uint8_t *d_show, size_t show_stride, cudaStream_t st)
{
    cvs::k_threshold<<<piece, 256, 0, st>>>(h->d_hist, h->d_thr, piece, 50, 200);
    CU_TRY(cudaGetLastError());
    dim3 grid(grid_for((h->npix + 15) / 16, 256, h->sms), piece);
    cvs::k_binarize_expand<<<grid, 256, 0, st>>>(h->d_gray1, h->P16, d_show, show_stride, h->d_thr, h->npix);
    CU_TRY(cudaGetLastError());
    h->launches += 2;
    return CVS_OK;
}

// scratch for pieces of `frames` frames: the pre-pass's private copy (noise filter, or an overlay that may not be
// blitted into the frames themselves) and binarisation's gray bytes, histograms and thresholds
cvs_status ensure_scratch(cvs_handle h, size_t frames, const cvs::OverlayText &txt, bool frames_private, bool binarize)
{
    if (h->noise_filter || (txt.n && !frames_private)) CVS_TRY(h->d_work.grow(frames * h->Npad + 64, "pre-pass frames", true));
    if (binarize) {
        CVS_TRY(h->d_gray1.grow(frames * h->P16 + 64, "binarisation gray bytes"));
        CVS_TRY(h->d_hist.grow(frames * 256 * sizeof(unsigned int), "binarisation histograms"));
        CVS_TRY(h->d_thr.grow(frames * sizeof(int), "binarisation thresholds"));
    }
    return CVS_OK;
}

// What a stream-kernel launch needs: the kernel, G co-resident blocks, each owning the same cps consecutive chunks of
// every frame (or band) in each of nseg segments, the ring stages and the shared memory they take.
struct LaunchPlan {
    bool per_handle = false; // batch only: run the handles one by one through run_frames instead
    Family fam = kFamWs;
    const void *kern = nullptr;
    int G = 0, block = 0, nbands = 1, nstages = 0, smem = 0;
    uint32_t cps = 0, nseg = 0;

    // The blocks only ever wait for blocks of LOWER index of the same step (look-back), never at a grid barrier, and
    // G <= the blocks the device can hold, so a plain launch cannot deadlock (blocks are dispatched in index order); a
    // cooperative launch additionally waits until the WHOLE grid fits at once.  Sequences keep that (every block starts
    // together: the timings of DESIGN 4.1); a single frame of the submit / exec path is launched plain, so that its
    // blocks start as SMs become free instead of draining the device first -- with several camera streams on a GPU,
    // whose decode kernels (cvs_jpeg.cuh) and payload pushes would otherwise run strictly one after the other: 3 JPEG
    // streams 3.8 k -> 7.1 k frames/s, raw streams unchanged.  (Frames walked in several segments wait for the totals of
    // ALL blocks of the previous segment: cooperative.)  A batch is launched plain, as the single frames it replaces.
    bool cooperative(int piece) const { return fam != kFamBatch && (piece > 1 || nseg > 1); }
};

// The launch plan of the stream kernel over pieces of `piece` frames of h (batch: one frame of each of `piece` handles
// shaped like h) in display mode kmode.
// k_stream_ws (front / back warp groups) wherever the reference can stay in registers.  Frames that do not fit one pass
// of the grid (3840x2160): a SEQUENCE is walked band by band -- every band is a byte range of the frame that does fit,
// and one k_stream_ws launch takes that band through all frames of the piece with its reference bytes in registers;
// frame t's entries of band j are appended behind those of the bands before it (counts handed from launch to launch).
// Same payload, 1.3-1.8x faster than walking the frame in segments with the reference going through L2, which is what
// single frames (the drop-in call) still do, with the one-group kernel k_stream (k_stream_ws measured 25 against 17 us
// per 4K frame there).  A batch of such frames, or a batch of one, runs handle by handle (see run_batch).
cvs_status plan_launch(cvs_handle h, bool batch, int kmode, int piece, LaunchPlan &lp)
{
    lp = LaunchPlan();
    const int g0 = std::min(h->sms, 32 * cvs::kWsLook);
    const bool one_pass = h->nchunks <= (size_t)g0 * cvs::kThreads;
    if (batch && (piece == 1 || !one_pass)) {
        lp.per_handle = true;
        return CVS_OK;
    }
    lp.fam = batch ? kFamBatch : (one_pass || piece >= 4) ? kFamWs : kFamStream;
    const bool ws = lp.fam != kFamStream;
    if (!one_pass && ws) lp.nbands = (int)((h->nchunks + (size_t)g0 * cvs::kThreads - 1) / ((size_t)g0 * cvs::kThreads));
    const uint32_t chunks = (h->nchunks + lp.nbands - 1) / lp.nbands; // of a frame or band
    const int look_max = ws ? 32 * cvs::kWsLook : cvs::kLook * cvs::kThreads; // predecessors the look-back can read
    lp.G = std::min({ws ? h->sms : cvs::kBlocksPerSM * h->sms, look_max, (int)chunks});
    auto split = [&] {
        lp.nseg = (uint32_t)((chunks + (size_t)lp.G * cvs::kThreads - 1) / ((size_t)lp.G * cvs::kThreads));
        lp.cps = (uint32_t)((chunks + (size_t)lp.G * lp.nseg - 1) / ((size_t)lp.G * lp.nseg));
    };
    split();
    // k_stream_ws keeps the reference in registers, so it takes a frame (or a band) in one pass; k_stream walks the
    // frame in segments
    if ((lp.nseg == 1) != ws)
        return fail(CVS_ERR_INTERNAL, "%s launch geometry has %u passes per frame", ws ? "k_stream_ws" : "k_stream", lp.nseg);
    const bool hi = h->hi;
    lp.kern = lp.fam == kFamBatch ? (const void *)kBatchKernels[kmode][hi]
              : ws                ? (const void *)kWsKernels[kmode][hi]
                                  : (const void *)kStreamKernels[kmode][hi];
    lp.block = ws ? cvs::kWsThreads : cvs::kThreads;
    // ring depth: all four stages for k_stream_ws (measured +5 % at 1080p), three for k_stream (a deeper prefetch
    // measured 17 % slower at 3840x2160); fewer if shared memory is short
    int smem_max = 0;
    CU_TRY(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device));
    auto smem_need = [&](int ns) { return ws ? (int)cvs::WsLayout::total(lp.cps, (uint32_t)ns) : cvs::SmemLayout::total(ns); };
    lp.nstages = ws ? cvs::kStages : cvs::kStages - 1;
    while (lp.nstages > 2 && smem_need(lp.nstages) > smem_max) lp.nstages--;
    lp.smem = smem_need(lp.nstages);
    if (lp.smem > smem_max) return fail(CVS_ERR_INTERNAL, "stream kernel needs %d bytes of shared memory, device has %d", lp.smem, smem_max);
    int &occ = h->occ[lp.fam][kmode][hi];
    if (occ == 0) { // first launch of this variant on this handle
        CU_TRY(cudaFuncSetAttribute(lp.kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
        CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, lp.kern, lp.block, lp.smem));
    }
    if (occ < 1) return fail(CVS_ERR_INTERNAL, "stream kernel does not fit on an SM");
    if (lp.G > occ * h->sms) { // fewer co-resident blocks than planned: recompute
        const uint32_t nseg = lp.nseg;
        lp.G = occ * h->sms;
        split();
        if (lp.nseg != nseg) return fail(CVS_ERR_INTERNAL, "occupancy changed the segment count");
    }
    return CVS_OK;
}

// The parameters of a launch of h that come from the handle and the plan, under a fresh epoch tag of h's descriptors;
// the caller adds the frames, the outputs and, for a band, its byte range.
cvs_status stream_params(cvs_handle h, const LaunchPlan &lp, size_t cap, unsigned int *status, cudaStream_t st,
                         cvs::StreamParams &p)
{
    h->epoch++;
    if (h->epoch == 0) { // tag wrapped: stale descriptors could alias
        CU_TRY(cudaMemsetAsync(h->d_desc, 0, h->d_desc.bytes, st));
        h->epoch = 1;
    }
    memset(&p, 0, sizeof p);
    p.nbytes = h->N;
    p.nbytes16 = h->N16;
    p.nchunks = h->nchunks;
    p.nseg = lp.nseg;
    p.cps = lp.cps;
    p.nstages = (uint32_t)lp.nstages;
    p.cap = cap;
    p.heat_lut = h->d_lut;
    p.desc = h->d_desc;
    p.epoch = h->epoch;
    p.addc = h->addc;
    p.status = status;
    return CVS_OK;
}

cvs_status launch(cvs_handle h, const LaunchPlan &lp, void **args, int piece, cudaStream_t st)
{
    if (lp.cooperative(piece))
        CU_TRY(cudaLaunchCooperativeKernel(lp.kern, dim3(lp.G), dim3(lp.block), args, (size_t)lp.smem, st));
    else
        CU_TRY(cudaLaunchKernel(lp.kern, dim3(lp.G), dim3(lp.block), args, (size_t)lp.smem, st));
    h->launches++;
    return CVS_OK;
}

// One pass of the whole hot path over nframes device-resident frames (A11, kernels.cu:455-520).
// Long sequences are walked in pieces of at most max_sequence frames; every piece runs the complete chain (noise
// filter / overlay pre-pass, fused stream kernel, binarisation pass 2), so the scratch buffers are sized by the piece
// and no launch dimension grows with the length of the sequence.
//   frames_private: d_frames is a buffer of this library (a slot's upload buffer) that may be modified in place --
//                   the text overlay is then blitted straight into it instead of into a copy.
cvs_status run_frames(cvs_handle h, const uint8_t *d_frames, size_t stride, int nframes, unsigned int *d_pos, int *d_xs,
                      uint8_t *d_diff, size_t cap, uint8_t *d_show, size_t show_stride, const char *text,
                      cudaStream_t st, bool frames_private, unsigned int *d_status)
{
    if (nframes <= 0) return CVS_OK;

    const cvs::OverlayText txt = overlay_text(h, text);

    const int mode = h->mode;
    const bool binarize = (mode == 5 || mode == 7) && d_show;
    // A sequence in a binarising mode computes the gray byte and the histograms in a kernel of its own in front of the
    // plain stream kernel (k_gray_hist_seq: why, and what it measured); a single frame keeps the fused kernel.
    const bool split_gray = binarize && nframes >= 2;
    const int kmode = d_show && !split_gray ? mode : 0; // without a display buffer only the payload is produced
    const int piece_max = h->max_sequence < nframes ? h->max_sequence : nframes;
    CVS_TRY(ensure_scratch(h, (size_t)piece_max, txt, frames_private, binarize));
    LaunchPlan lp;
    CVS_TRY(plan_launch(h, false, kmode, piece_max, lp));
    if (lp.nbands > 1) CVS_TRY(h->d_band_pos.grow(2 * (size_t)piece_max * sizeof(unsigned int), "band counts"));

    int done = 0;
    while (done < nframes) {
        int piece = nframes - done;
        if (piece > h->max_sequence) piece = h->max_sequence;
        const uint8_t *frames = d_frames + (size_t)done * stride;
        size_t fstride = stride;

        CVS_TRY(pre_pass(h, frames, fstride, piece, txt, frames_private, binarize, st));
        if (split_gray) { // gray byte + histogram of the frames as the diff will see them (filtered, overlay blitted)
            const size_t groups = ((size_t)h->N + cvs::kGroupBytes - 1) / cvs::kGroupBytes;
            dim3 grid(grid_for((groups + cvs::kGrayHistGroupsPerThread - 1) / cvs::kGrayHistGroupsPerThread, 256, h->sms), piece);
            if (mode == 5) cvs::k_gray_hist_seq<true><<<grid, 256, 0, st>>>(frames, fstride, h->N, h->d_gray1, h->P16, h->d_hist);
            else cvs::k_gray_hist_seq<false><<<grid, 256, 0, st>>>(frames, fstride, h->N, h->d_gray1, h->P16, h->d_hist);
            CU_TRY(cudaGetLastError());
            h->launches++;
        }

        CVS_TRY(h->d_desc.grow((size_t)piece * lp.nseg * (lp.G + 1) * sizeof(unsigned long long), "stream-kernel descriptors", true));
        const size_t band_bytes = (size_t)lp.G * lp.cps * cvs::kChunkBytes; // bytes of a band (the last one may be shorter)
        for (int band = 0; band < lp.nbands; band++) {
            const bool banded = lp.nbands > 1;
            const size_t boff = banded ? (size_t)band * band_bytes : 0;
            if (boff >= h->N) break;
            const uint32_t bbytes = banded ? (uint32_t)((h->N - boff) < band_bytes ? (h->N - boff) : band_bytes) : h->N;
            const bool last_band = !banded || boff + band_bytes >= h->N;
            cvs::StreamParams p;
            CVS_TRY(stream_params(h, lp, cap, d_status, st, p));
            p.frames = frames + boff;
            p.frame_stride = fstride;
            p.nframes = piece;
            p.ref = h->d_ref + boff;
            p.nbytes = bbytes;
            p.nbytes16 = banded ? (uint32_t)round_up(bbytes, 16) : h->N16;
            p.nchunks = (bbytes + cvs::kChunkBytes - 1) / cvs::kChunkBytes;
            p.pos = last_band ? d_pos + done : h->d_band_pos + (size_t)(band & 1) * piece_max;
            p.pos_prior = band ? h->d_band_pos + (size_t)((band - 1) & 1) * piece_max : nullptr;
            p.index_base = (uint32_t)boff;
            p.xs = d_xs + (size_t)done * cap;
            p.diff = d_diff + (size_t)done * cap;
            p.show = d_show ? d_show + (size_t)done * show_stride : nullptr;
            p.show_stride = show_stride;
            p.gray1 = binarize && !split_gray ? h->d_gray1.p : nullptr;
            p.gray_stride = h->P16;
            p.hist = binarize && !split_gray ? h->d_hist.p : nullptr;
            void *args[] = {&p};
            CVS_TRY(launch(h, lp, args, piece, st));
        }

        if (binarize) CVS_TRY(binarize_pass(h, piece, d_show + (size_t)done * show_stride, show_stride, st));
        done += piece;
    }
    return CVS_OK;
}

// One frame of each of n cameras (hs[i] device-resident at frames[i], N bytes readable up to N16) through one
// k_stream_ws_batch launch on `st`, step i = camera i; outputs of camera i at pos[i], xs[i], diff[i], show[i] (show: all
// NULL or all set), status bits at status[i].  Pre- and post-passes (noise filter, overlay, binarisation pass 2) stay per
// camera.  Frames that k_stream_ws does not take in one pass (3840x2160: k_stream, segments) are run camera by camera
// through run_frames, and so is a batch of one: its reference stays in registers there (1080p, scripts/batch_probe.py:
// 19-24 us per frame against 22-28 for a batch of one; from two cameras on the batch is faster).  The handles were
// checked by check_batch.
cvs_status run_batch(const cvs_handle *hs, int n, const uint8_t *const *frames, unsigned int *const *pos, int *const *xs,
                     uint8_t *const *diff, size_t cap, uint8_t *const *show, const char *const *texts, cudaStream_t st,
                     bool frames_private, unsigned int *const *status)
{
    cvs_handle h0 = hs[0];
    const bool binarize = (h0->mode == 5 || h0->mode == 7) && show;
    LaunchPlan lp;
    CVS_TRY(plan_launch(h0, true, show ? h0->mode : 0, n, lp));
    if (lp.per_handle) {
        for (int i = 0; i < n; i++)
            CVS_TRY(run_frames(hs[i], frames[i], hs[i]->Npad, 1, pos[i], xs[i], diff[i], cap, show ? show[i] : nullptr,
                               hs[i]->Npad, texts ? texts[i] : nullptr, st, frames_private, status[i]));
        return CVS_OK;
    }

    cvs::BatchTable tbl; // (copied into the launch's parameters by cudaLaunchKernel)
    for (int i = 0; i < n; i++) {
        cvs_handle h = hs[i];
        const cvs::OverlayText txt = overlay_text(h, texts ? texts[i] : nullptr);
        CVS_TRY(ensure_scratch(h, 1, txt, frames_private, binarize));
        const uint8_t *f = frames[i];
        size_t fstride = h->Npad;
        CVS_TRY(pre_pass(h, f, fstride, 1, txt, frames_private, binarize, st));
        tbl.cam[i] = {f, h->d_ref, pos[i], xs[i], diff[i], show ? show[i] : nullptr, binarize ? h->d_gray1.p : nullptr,
                      binarize ? h->d_hist.p : nullptr, status[i]};
    }
    CVS_TRY(h0->d_desc.grow((size_t)n * (lp.G + 1) * sizeof(unsigned long long), "stream-kernel descriptors", true));
    cvs::StreamParams p;
    CVS_TRY(stream_params(h0, lp, cap, status[0], st, p));
    p.nframes = n;
    void *args[] = {&p, &tbl};
    CVS_TRY(launch(h0, lp, args, n, st));
    if (binarize)
        for (int i = 0; i < n; i++) CVS_TRY(binarize_pass(hs[i], 1, show[i], hs[i]->Npad, st));
    return CVS_OK;
}

cvs_status check_handle(cvs_handle h)
{
    if (!h) return fail(CVS_ERR_INVALID, "null handle");
    int cur = -1;
    if (cudaGetDevice(&cur) != cudaSuccess || cur != h->device) CU_TRY(cudaSetDevice(h->device));
    return CVS_OK;
}

cvs_status status_word(unsigned int w)
{
    if (w & cvs::kStatusWatchdog) return fail(CVS_ERR_INTERNAL, "device watchdog tripped (status 0x%x)", w);
    if (w & cvs::kStatusCapacity) return fail(CVS_ERR_CAPACITY, "payload capacity exceeded");
    if (w & (cvs::jpg::kJpegNotConverged | cvs::jpg::kJpegBlockCount))
        return fail(CVS_ERR_INVALID, "damaged JPEG bitstream (decoder status 0x%x): the frame's payload is not valid", w);
    return CVS_OK;
}

} // namespace

namespace {
cvs_status init_device_state(cvs_handle h, const cvs_config *cfg);
}

extern "C" {

const char *cvs_last_error(void) { return g_err; }
int cvs_abi_version(void) { return CVS_ABI_VERSION; }

int cvs_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    int ok = 0;
    for (int i = 0; i < n; i++)
        if (device_is_sm100(i)) ok++;
    return ok;
}

void cvs_config_default(cvs_config *cfg)
{
    if (!cfg) return;
    memset(cfg, 0, sizeof *cfg);
    cfg->width = 1920;  // server/src/threads.cpp:37-38
    cfg->height = 1080;
    cfg->threshold = 20; // LR_THRESHOLDS, common.h:14
    cfg->mode = 0;
    cfg->noise_filter = 0;
    cfg->ksize = 3; // K, common.h:6
    cfg->max_sequence = 512;
}

cvs_status cvs_create(const cvs_config *cfg, cvs_handle *out)
{
    if (!cfg || !out) return fail(CVS_ERR_INVALID, "null argument");
    *out = nullptr;
    if (cfg->width <= 0 || cfg->height <= 0) return fail(CVS_ERR_INVALID, "bad frame size %dx%d", cfg->width, cfg->height);
    if ((uint64_t)cfg->width * cfg->height * 3 > 0x7fffffffull - 64)
        return fail(CVS_ERR_INVALID, "frame too large for 32-bit byte indices");
    if (cfg->mode < 0 || cfg->mode > 7) return fail(CVS_ERR_INVALID, "bad mode %d", cfg->mode);
    if (cfg->noise_filter && (cfg->ksize < 1 || cfg->ksize > 9 || !(cfg->ksize & 1) || !cfg->kweights))
        return fail(CVS_ERR_INVALID, "noise filter needs an odd ksize in 1..9 and weights");
    if (!cfg->base_frame) return fail(CVS_ERR_INVALID, "base_frame is required");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || cfg->device < 0 || cfg->device >= ndev) {
        cudaGetLastError();
        return fail(CVS_ERR_NODEVICE, "CUDA device %d not available (there is no CPU fallback)", cfg->device);
    }
    if (!device_is_sm100(cfg->device))
        return fail(CVS_ERR_NODEVICE, "device %d is not sm_100 (there is no CPU fallback)", cfg->device);
    CU_TRY(cudaSetDevice(cfg->device));

    cvs_handle h = new cvs_stream_s();
    h->width = cfg->width;
    h->height = cfg->height;
    h->threshold = cfg->threshold;
    h->mode = cfg->mode;
    h->noise_filter = cfg->noise_filter ? 1 : 0;
    h->ksize = cfg->ksize;
    h->device = cfg->device;
    h->max_sequence = cfg->max_sequence > 0 ? cfg->max_sequence : 512;
    h->npix = (uint32_t)cfg->width * (uint32_t)cfg->height;
    h->N = 3u * h->npix;
    h->N16 = (uint32_t)round_up(h->N, 16);
    h->nchunks = (h->N + cvs::kChunkBytes - 1) / cvs::kChunkBytes;
    h->Npad = (size_t)h->nchunks * cvs::kChunkBytes;
    h->P16 = round_up(h->npix, 16);
    threshold_consts(cfg->threshold, h->hi, h->addc);
    if (const char *tr = getenv("CVS_TRACE")) h->trace = atoi(tr) != 0; // instrumentation only: timelines on stderr
    // own decoder only (refuse, do not fall back to nvJPEG): part of the documented interface
    if (const char *jd = getenv("CVS_JPEG_DECODER")) h->jpeg_own_only = !strcmp(jd, "own");
    // subsequence length of the parallel Huffman decode: tests reach 128-bit subsequences (whole-subsequence rounds) only here
    if (const char *sb = getenv("CVS_JPEG_SUB_BITS")) {
        const int v = atoi(sb);
        if (v >= 64 && v <= 65536 && v % 32 == 0) h->jd[0].sub_bits = h->jd[1].sub_bits = h->jd[2].sub_bits = (uint32_t)v;
    }
    memset(&h->weights, 0, sizeof h->weights);
    if (cfg->noise_filter) memcpy(h->weights.k, cfg->kweights, sizeof(float) * cfg->ksize * cfg->ksize);
    const cvs_status st = init_device_state(h, cfg);
    if (st != CVS_OK) { // g_err already holds the reason; release whatever was allocated
        cvs_destroy(h);
        return st;
    }
    *out = h;
    return CVS_OK;
}

} // extern "C"

namespace {

// device-side half of cvs_create: streams, events, the reference frame, per-slot buffers
cvs_status init_device_state(cvs_handle h, const cvs_config *cfg)
{
    CU_TRY(cudaDeviceGetAttribute(&h->sms, cudaDevAttrMultiProcessorCount, cfg->device));

    CU_TRY(cudaStreamCreateWithFlags(&h->s_comp, cudaStreamNonBlocking));
    CU_TRY(cudaStreamCreateWithFlags(&h->s_h2d, cudaStreamNonBlocking));
    CU_TRY(cudaStreamCreateWithFlags(&h->s_d2h, cudaStreamNonBlocking));
    CU_TRY(cudaStreamCreateWithFlags(&h->s_pay, cudaStreamNonBlocking));
    CVS_TRY(h->d_ref.grow(h->Npad + 64, "reference frame", true));
    CU_TRY(cudaMemcpy(h->d_ref, cfg->base_frame, h->N, cudaMemcpyHostToDevice)); // kernels.cu:406
    {
        uint32_t lut[768];
        build_heat_lut(lut);
        CVS_TRY(h->d_lut.grow(sizeof lut, "heat-map table"));
        CU_TRY(cudaMemcpy(h->d_lut, lut, sizeof lut, cudaMemcpyHostToDevice));
    }
    CVS_TRY(h->d_status.grow(sizeof(unsigned int), "status word", true));
    CVS_TRY(h->h_status.alloc());
    if (cfg->glyphs && cfg->glyph_w > 0 && cfg->glyph_h > 0 && cfg->glyph_chars) {
        h->glyph_chars = cfg->glyph_chars;
        h->glyph_w = cfg->glyph_w;
        h->glyph_h = cfg->glyph_h;
        size_t bytes = h->glyph_chars.size() * 3 * (size_t)cfg->glyph_w * cfg->glyph_h;
        CVS_TRY(h->d_glyphs.grow(bytes + 16, "glyph atlas"));
        CU_TRY(cudaMemcpy(h->d_glyphs, cfg->glyphs, bytes, cudaMemcpyHostToDevice));
    }
    const size_t cap = round_up(h->N, 4);
    for (Slot &s : h->slot) {
        CVS_TRY(s.d_in.grow(h->Npad + 64, "upload frame", true));
        CVS_TRY(s.d_xs.grow(cap * sizeof(int), "payload indices"));
        CVS_TRY(s.d_diff.grow(cap, "payload bytes"));
        CVS_TRY(s.d_pos.grow(sizeof(unsigned int), "payload count"));
        if (h->mode) CVS_TRY(s.d_show.grow(h->Npad + 64, "display frame"));
        CVS_TRY(s.h_pos.alloc());
        CVS_TRY(s.d_status.grow(sizeof(unsigned int), "status word", true));
        CVS_TRY(s.h_status.alloc());
        cudaEvent_t *evs[] = {&s.ev_h2d0, &s.ev_h2d1, &s.ev_k0, &s.ev_k1, &s.ev_pos, &s.ev_p0, &s.ev_done};
        for (cudaEvent_t *e : evs) CU_TRY(cudaEventCreate(e));
    }
    {   // CVS_TRACE timelines of all handles of the process share one origin
        static cudaEvent_t g_trace_base = nullptr;
        static std::mutex g_trace_mutex;
        std::lock_guard<std::mutex> lk(g_trace_mutex);
        if (!g_trace_base) {
            CU_TRY(cudaEventCreate(&g_trace_base));
            CU_TRY(cudaEventRecord(g_trace_base, h->s_h2d));
        }
        h->ev_base = g_trace_base;
    }
    CU_TRY(cudaDeviceSynchronize());
    return CVS_OK;
}

} // namespace

extern "C" {

cvs_status cvs_destroy(cvs_handle h)
{
    if (!h) return CVS_OK;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    for (Slot &s : h->slot) {
        if (s.jpeg_state && g_nvjpeg.ok) g_nvjpeg.StateDestroy(s.jpeg_state);
        cudaEvent_t evs[] = {s.ev_h2d0, s.ev_h2d1, s.ev_k0, s.ev_k1, s.ev_pos, s.ev_p0, s.ev_done};
        for (cudaEvent_t e : evs)
            if (e) cudaEventDestroy(e);
    }
    for (cudaStream_t js : h->s_jpg)
        if (js) cudaStreamDestroy(js);
    if (h->jpeg_state && g_nvjpeg.ok) g_nvjpeg.StateDestroy(h->jpeg_state);
    if (h->jpeg && g_nvjpeg.ok) g_nvjpeg.Destroy(h->jpeg);
    if (h->s_comp) cudaStreamDestroy(h->s_comp);
    if (h->s_h2d) cudaStreamDestroy(h->s_h2d);
    if (h->s_d2h) cudaStreamDestroy(h->s_d2h);
    if (h->s_pay) cudaStreamDestroy(h->s_pay);
    delete h; // device and pinned memory: freed by the buffers of the handle and its slots
    return CVS_OK;
}

cvs_status cvs_reset(cvs_handle h, const uint8_t *base_frame)
{
    cvs_status s = check_handle(h);
    if (s) return s;
    if (!base_frame) return fail(CVS_ERR_INVALID, "null base frame");
    CU_TRY(cudaDeviceSynchronize());
    CU_TRY(cudaMemcpy(h->d_ref, base_frame, h->N, cudaMemcpyHostToDevice));
    return CVS_OK;
}

cvs_status cvs_alloc_host(void **ptr, size_t bytes)
{
    if (!ptr) return fail(CVS_ERR_INVALID, "null argument");
    *ptr = nullptr;
    if (cvs_device_count() == 0) return fail(CVS_ERR_NODEVICE, "no sm_100 device (there is no CPU fallback)");
    CU_TRY(cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocPortable));
    return CVS_OK;
}

cvs_status cvs_free_host(void *ptr)
{
    if (!ptr) return CVS_OK;
    CU_TRY(cudaFreeHost(ptr));
    return CVS_OK;
}

// common body of cvs_submit / cvs_submit_io (reference-format payload into diff_out / xs / pos) and cvs_submit_wire
// (wire_out != nullptr: compact "CVW1" frame, see cvs_filter_kernels.cuh)
// decode one baseline JPEG of the stream's frame size into d_out (BGR interleaved, pitch 3*width), asynchronously on `st`
static cvs_status jpeg_decode_nvjpeg(cvs_handle h, nvjpegJpegState_t *state, const uint8_t *jpeg, size_t jpeg_bytes, uint8_t *d_out,
                                     cudaStream_t st)
{
    const NvJpegApi *nj = nvjpeg_api();
    if (!nj) return fail(CVS_ERR_NODEVICE, "libnvjpeg could not be loaded: %s", dlerror());
    if (!h->jpeg) {
        // Backend, in order of preference: the hardware JPEG engine, GPU-assisted Huffman decoding (both through the
        // batched entry points, batch of one), the library's default single-image decode.  Chroma is upsampled WITH
        // interpolation, as libjpeg-turbo (OpenCV, the reference's decoder) does by default: on the reference's fixture
        // frames that brings the decoded pixels from max |d| 26 / 63 % of the bytes differing to max |d| 5 / 55 %, and the
        // K1 count from 404,321 to 370,732 (OpenCV: 369,350).
        const unsigned flags = NVJPEG_FLAGS_UPSAMPLING_WITH_INTERPOLATION;
        nvjpegStatus_t e = NVJPEG_STATUS_NOT_INITIALIZED;
        const bool can_batch = nj->CreateEx && nj->BatchedInit && nj->Batched;
        if (can_batch) {
            e = nj->CreateEx(NVJPEG_BACKEND_HARDWARE, nullptr, nullptr, flags, &h->jpeg);
            h->jpeg_batched = e == NVJPEG_STATUS_SUCCESS;
        }
        if (e != NVJPEG_STATUS_SUCCESS && can_batch) {
            e = nj->CreateEx(NVJPEG_BACKEND_GPU_HYBRID, nullptr, nullptr, flags, &h->jpeg);
            h->jpeg_batched = e == NVJPEG_STATUS_SUCCESS;
        }
        if (e != NVJPEG_STATUS_SUCCESS && nj->CreateEx) e = nj->CreateEx(NVJPEG_BACKEND_DEFAULT, nullptr, nullptr, flags, &h->jpeg);
        if (e != NVJPEG_STATUS_SUCCESS) e = nj->CreateSimple(&h->jpeg);
        if (e != NVJPEG_STATUS_SUCCESS) return fail(CVS_ERR_CUDA, "nvjpegCreate failed (%d)", (int)e);
    }
    if (!*state) {
        nvjpegStatus_t e = nj->StateCreate(h->jpeg, state);
        if (e != NVJPEG_STATUS_SUCCESS) return fail(CVS_ERR_CUDA, "nvjpegJpegStateCreate failed (%d)", (int)e);
        if (h->jpeg_batched) {
            e = nj->BatchedInit(h->jpeg, *state, 1, 1, NVJPEG_OUTPUT_BGRI);
            if (e != NVJPEG_STATUS_SUCCESS) return fail(CVS_ERR_CUDA, "nvjpegDecodeBatchedInitialize failed (%d)", (int)e);
        }
    }
    int ncomp = 0, widths[NVJPEG_MAX_COMPONENT] = {0}, heights[NVJPEG_MAX_COMPONENT] = {0};
    nvjpegChromaSubsampling_t sub;
    nvjpegStatus_t e = nj->GetImageInfo(h->jpeg, jpeg, jpeg_bytes, &ncomp, &sub, widths, heights);
    if (e != NVJPEG_STATUS_SUCCESS) return fail(CVS_ERR_INVALID, "not a decodable JPEG (nvjpegGetImageInfo %d)", (int)e);
    if (widths[0] != h->width || heights[0] != h->height)
        return fail(CVS_ERR_INVALID, "JPEG is %dx%d, the stream is %dx%d", widths[0], heights[0], h->width, h->height);
    nvjpegImage_t img;
    memset(&img, 0, sizeof img);
    img.channel[0] = d_out;
    img.pitch[0] = (size_t)3 * h->width;
    if (h->jpeg_batched) {
        const unsigned char *data[1] = {jpeg};
        const size_t lengths[1] = {jpeg_bytes};
        e = nj->Batched(h->jpeg, *state, data, lengths, &img, st);
    } else {
        e = nj->Decode(h->jpeg, *state, jpeg, jpeg_bytes, NVJPEG_OUTPUT_BGRI, &img, st);
    }
    if (e != NVJPEG_STATUS_SUCCESS) return fail(CVS_ERR_CUDA, "nvjpeg decode failed (%d)", (int)e);
    return CVS_OK;
}

// The library's own decoder (cvs_jpeg.cuh): bit for bit the pixels OpenCV / libjpeg-turbo produce.  `status` receives the
// decoder's status bits (device word, OR-ed).  *unsupported is set when the bitstream is a JPEG this decoder does not
// cover (restart intervals, progressive, other samplings); nothing has been enqueued then.
static cvs_status jpeg_decode_own(cvs_handle h, JpegDecoder &jd, const uint8_t *jpeg, size_t jpeg_bytes, uint8_t *d_out,
                                  cudaStream_t st, unsigned int *d_status, bool *unsupported)
{
    namespace J = cvs::jpg;
    *unsupported = false;
    J::Parsed &P = jd.parsed;
    if (!J::reparse_same_header(jpeg, jpeg_bytes, jd.header.data(), jd.header.size(), jd.sub_bits, &P)) {
        jd.header.clear();
        const J::ParseStatus ps = J::parse(jpeg, jpeg_bytes, jd.sub_bits, &P);
        if (ps == J::kParseUnsupported) {
            *unsupported = true;
            return CVS_OK;
        }
        if (ps != J::kParseOk) return fail(CVS_ERR_INVALID, "not a decodable baseline JPEG");
        jd.header.assign(jpeg, jpeg + P.scan_offset); // the next frame of the camera starts with the same bytes
    }
    const J::Geometry &g = P.g;
    if (g.width != h->width || g.height != h->height)
        return fail(CVS_ERR_INVALID, "JPEG is %dx%d, the stream is %dx%d", g.width, g.height, h->width, h->height);

    // ---- scratch: one arena, carved (JpegDecoder::carve), grown by half again when a frame needs more
    const size_t raw_pad = round_up(P.scan_bytes, 4096) + 4096;
    const size_t luma_bytes = (size_t)g.mcux * 8 * g.H * g.mcuy * 8 * g.V, chroma_bytes = (size_t)g.mcux * 8 * g.mcuy * 8;
    if (raw_pad > jd.raw_cap || g.nblocks > jd.block_cap) {
        const size_t raw_cap = std::max(jd.raw_cap, raw_pad + raw_pad / 2), block_cap = std::max<size_t>(jd.block_cap, g.nblocks);
        jd.raw_cap = jd.block_cap = 0; // until the arena holds the new layout
        CVS_TRY(jd.arena.grow_on(st, jd.carve(nullptr, raw_cap, block_cap), "JPEG decoder scratch"));
        jd.carve(jd.arena, raw_cap, block_cap);
        jd.raw_cap = raw_cap;
        jd.block_cap = block_cap;
        jd.tables_valid = false;
    }
    if (!jd.tables_valid || memcmp(&jd.tables_host, &P.t, sizeof(J::Tables)) != 0) {
        // rare (a camera sends the same tables with every frame); the pageable source is staged before the call returns
        CU_TRY(cudaMemcpyAsync(jd.d_tables, &P.t, sizeof(J::Tables), cudaMemcpyHostToDevice, st));
        memcpy(&jd.tables_host, &P.t, sizeof(J::Tables));
        jd.tables_valid = true;
    }

    // ---- the entropy-coded segment crosses PCIe (0.4 MB instead of the 6.2 MB frame), FF 00 -> FF
    const uint32_t raw_len = (uint32_t)P.scan_bytes;
    CU_TRY(cudaMemcpyAsync(jd.d_raw, jpeg + P.scan_offset, raw_len, cudaMemcpyHostToDevice, st));
    const uint32_t ublocks = (raw_len + J::kUnstuffThreads * J::kUnstuffBytes - 1) / (J::kUnstuffThreads * J::kUnstuffBytes);

    if (P.restart_interval) {
        // ---- scratch cleared, FF 00 -> FF and FF Dn dropped (launches of their own on this path)
        CU_TRY(cudaMemsetAsync(jd.arena, 0, jd.zero_bytes_fixed + (size_t)g.nblocks * 64 * sizeof(int16_t), st));
        J::k_unstuff_count<<<ublocks, J::kUnstuffThreads, 0, st>>>(jd.d_raw, raw_len, jd.d_block_kept, jd.d_block_marks);
        J::k_unstuff_write<<<ublocks, J::kUnstuffThreads, 0, st>>>(jd.d_raw, raw_len, jd.d_block_kept, jd.d_block_marks, jd.d_unst,
                                                                     jd.d_total_bits, jd.d_seg_start, jd.seg_cap, jd.d_total_marks);
        // ---- Huffman decode of a scan with restart intervals: one thread per interval (k_entropy_restart)
        J::RestartParams rp;
        rp.tables = jd.d_tables;
        rp.g = g;
        rp.words = reinterpret_cast<const uint32_t *>(jd.d_unst);
        rp.total_bits = jd.d_total_bits;
        rp.total_marks = jd.d_total_marks;
        rp.seg_start = jd.d_seg_start;
        const uint32_t mcus = (uint32_t)g.mcux * (uint32_t)g.mcuy;
        rp.nseg = (mcus + P.restart_interval - 1) / P.restart_interval;
        rp.blocks_per_seg = P.restart_interval * (uint32_t)g.bpm;
        rp.coef = jd.d_coef;
        rp.status = d_status;
        if (rp.nseg + 1 > jd.seg_cap) return fail(CVS_ERR_INTERNAL, "restart interval table too small");
        J::k_entropy_restart<<<(rp.nseg + 127) / 128, 128, 0, st>>>(rp);
    } else {
    // ---- one cooperative launch: scratch cleared, FF 00 -> FF, Huffman decode (hypotheses, rounds, prefix sums, write)
    if (!jd.coop_blocks_per_sm) {
        CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&jd.coop_blocks_per_sm, J::k_entropy, J::kEntropyThreads, 0));
        if (jd.coop_blocks_per_sm < 1) return fail(CVS_ERR_INTERNAL, "k_entropy does not fit an SM");
    }
    J::EntropyParams ep;
    ep.raw = jd.d_raw;
    ep.raw_len = raw_len;
    ep.unst = jd.d_unst;
    ep.unst_bytes = (uint32_t)std::min(jd.raw_cap, round_up(raw_len, 4096) + 4096);
    ep.block_kept = jd.d_block_kept;
    ep.block_marks = jd.d_block_marks;
    ep.total_marks_out = jd.d_total_marks;
    ep.seg_start = jd.d_seg_start;
    ep.seg_cap = jd.seg_cap;
    ep.total_bits_out = jd.d_total_bits;
    ep.tables = jd.d_tables;
    ep.g = g;
    ep.words = reinterpret_cast<const uint32_t *>(jd.d_unst);
    ep.total_bits = jd.d_total_bits;
    ep.entry = jd.d_entry;
    ep.used = jd.d_used;
    ep.nblk = jd.d_nblk;
    ep.dcs = jd.d_dcs;
    ep.tile_blk = jd.d_tile_blk;
    ep.tile_dc = jd.d_tile_dc;
    // the write pass runs with one thread per G bits: S/8 or S/4 when that is a multiple of 32 bits
    ep.mid.nsplit = jd.sub_bits % 256 == 0 ? 8u : (jd.sub_bits % 128 == 0 ? 4u : 1u);
    ep.mid.G = jd.sub_bits / ep.mid.nsplit;
    ep.mid.stride = ep.mid.nsplit * g.nsub_max;
    ep.mid.state = jd.d_mid_state;
    ep.mid.nblk = jd.d_mid_nblk;
    ep.mid.dc = jd.d_mid_dc;
    ep.hx = jd.d_hx;
    ep.hy = jd.d_hy;
    ep.hw = jd.d_hw;
    ep.hym = jd.d_hym;
    ep.hwm = jd.d_hwm;
    ep.hmap = jd.d_hmap;
    ep.changed = jd.d_changed;
    ep.coef = jd.d_coef;
    ep.status = d_status;
    // one thread per subsequence and phase hypothesis in the first phases, one per subsequence afterwards
    const uint32_t ntiles = (g.nsub_max * (uint32_t)g.bpm + J::kEntropyThreads - 1) / J::kEntropyThreads;
    const uint32_t egrid = std::max(1u, std::min(ntiles, (uint32_t)(jd.coop_blocks_per_sm * h->sms)));
    void *eargs[] = {&ep};
    CU_TRY(cudaLaunchCooperativeKernel((const void *)J::k_entropy, dim3(egrid), dim3(J::kEntropyThreads), eargs, 0, st));
    }

    // ---- IDCT -> planes -> upsampling + colour conversion -> BGR24
    J::PlaneParams pp;
    pp.g = g;
    pp.tables = jd.d_tables;
    pp.coef = jd.d_coef;
    pp.y = jd.d_planes;
    pp.cb = jd.d_planes + luma_bytes;
    pp.cr = jd.d_planes + luma_bytes + chroma_bytes;
    J::k_idct<<<(g.nblocks + J::kIdctThreads - 1) / J::kIdctThreads, J::kIdctThreads, 0, st>>>(pp);
    J::ColourParams cp;
    cp.g = g;
    cp.y = pp.y;
    cp.cb = pp.cb;
    cp.cr = pp.cr;
    cp.bgr = d_out;
    const dim3 cgrid((unsigned)((g.width + 4 * J::kColourThreads - 1) / (4 * J::kColourThreads)), (unsigned)g.height);
    J::k_colour<<<cgrid, J::kColourThreads, 0, st>>>(cp);
    CU_TRY(cudaGetLastError());
    return CVS_OK;
}

// decode one baseline JPEG of the stream's frame size into d_out (BGR interleaved, pitch 3*width), asynchronously on `st`
static cvs_status jpeg_decode(cvs_handle h, JpegSet set, nvjpegJpegState_t *state, const uint8_t *jpeg, size_t jpeg_bytes,
                              uint8_t *d_out, cudaStream_t st, unsigned int *d_status)
{
    bool unsupported = false;
    const cvs_status e = jpeg_decode_own(h, h->jd[set], jpeg, jpeg_bytes, d_out, st, d_status, &unsupported);
    if (e || !unsupported) return e;
    if (h->jpeg_own_only) return fail(CVS_ERR_INVALID, "JPEG form not covered by the built-in decoder (CVS_JPEG_DECODER=own)");
    return jpeg_decode_nvjpeg(h, state, jpeg, jpeg_bytes, d_out, st);
}

// Egress of a ticket whose stream kernel has been enqueued (s.ev_k1 recorded behind it), on h->s_d2h; marks the slot
// busy under the next ticket number of h.  Shared by submit_common and cvs_submit_io_batch.
static cvs_status egress(cvs_handle h, Slot &s, const uint8_t *frame, uint8_t *diff_out, uint8_t *show, uint8_t *dshow,
                         unsigned int *pos, int *xs, uint8_t *wire_out)
{
    const size_t cap = round_up(h->N, 4);
    const uint32_t ntiles = (h->N + cvs::kWireTile - 1) / cvs::kWireTile;
    // D2H of the count (kernels.cu:507) and of the display frame.  When the caller's payload buffers are
    // pinned (cvs_alloc_host) a copy kernel that reads the count on the device pushes exactly pos entries
    // into them, so no host round trip separates the count from the payload (kernels.cu:507-508 + :522-524).
    CU_TRY(cudaStreamWaitEvent(h->s_d2h, s.ev_k1, 0));
    CU_TRY(cudaEventRecord(s.ev_p0, h->s_d2h));
    // Egress.  (a) separate output buffer (cvs_submit_io) and a mid-sized payload expected: the copy engine fetches
    //     a PREDICTED number of entries (previous count + margin) right behind the count -- no host round trip and
    //     no SM time (the copy kernel of (b) delays the next frame's cooperative launch), and the D2H engine runs
    //     beside the next frame's H2D; cvs_wait fetches the remainder in the rare case the frame had more.  Bytes
    //     past *pos of diff_out / xs are unspecified on that entry point, so the over-copy is invisible.  Measured
    //     (1080p, one stream, frames/s at 1 / 10 / 50 % density): 7,559 / 6,776 / 2,572 against 7,794 / 5,856 / 3,042
    //     for (b): small payloads do not repay the extra copy calls and large ones not the over-copy, hence the
    //     window.  (Round 2, three interleaved streams per GPU: taking the copy engine for the 50 % stream as well
    //     measured 4,680 frames/s against 5,260 with the push -- the path is bound by the PCIe link's combined
    //     traffic of both directions, about 62 GB/s on the pool's boxes, and the over-copy only adds to it.)
    // (b) otherwise, and always in-place (cvs_submit / cvs_exec: "rest of the frame untouched"): a copy kernel that
    //     reads the count on the device pushes exactly pos entries into the caller's pinned buffers, or (c) count
    //     round trip + exact copies in cvs_wait when the buffers are not mapped.
    void *dev_diff = nullptr, *dev_xs = nullptr;
    s.spec = 0;
    s.pushed = false;
    s.u_wire = wire_out;
    if (wire_out) {
        // compact wire format: two small kernels turn the payload into (tile counts, offsets, values) and store the
        // encoded frame -- its size depends on the count, which only the device knows yet -- straight into the
        // caller's pinned buffer; a pageable buffer gets the bytes from s.d_wire in cvs_wait
        void *dev_wire = nullptr;
        s.pushed = mapped_device_pointer(wire_out, &dev_wire) && aligned16(dev_wire);
        cvs::k_wire_bounds<<<(ntiles + 256) / 256, 256, 0, h->s_d2h>>>(s.d_xs, s.d_pos, cap, ntiles, s.d_starts);
        CU_TRY(cudaGetLastError());
        cvs::k_wire_pack<<<2 * h->sms, 256, 0, h->s_d2h>>>(s.d_xs, s.d_diff, s.d_pos, cap, ntiles, s.d_starts,
                                                         s.pushed ? (uint8_t *)dev_wire : s.d_wire);
        CU_TRY(cudaGetLastError());
        h->launches += 2;
    }
    const uint32_t spec_lo = h->N / 64u < 262144u ? h->N / 64u : 262144u; // ~1.3 MB of payload at 1080p
    // only with a prediction from a previous frame, and never more entries than the caller's buffers hold (N)
    if (wire_out) {
        // nothing else to fetch: the encoded frame carries the count
    } else if (diff_out != frame && h->pred != 0 && h->pred >= spec_lo && h->pred <= h->N / 4u) {
        const size_t guess = round_up(h->pred, 4);
        s.spec = (uint32_t)(guess > h->N ? h->N : guess);
    } else {
        s.pushed = mapped_device_pointer(diff_out, &dev_diff) && mapped_device_pointer(xs, &dev_xs) && aligned16(dev_diff, dev_xs);
    }
    if (s.pushed && !wire_out) {
        cvs::k_payload_push<<<h->sms, 256, 0, h->s_d2h>>>(s.d_xs, s.d_diff, s.d_pos, (int *)dev_xs, (uint8_t *)dev_diff, cap);
        CU_TRY(cudaGetLastError());
        h->launches++;
    }
    CU_TRY(cudaMemcpyAsync(s.h_pos, s.d_pos, sizeof(unsigned int), cudaMemcpyDeviceToHost, h->s_d2h));
    CU_TRY(cudaMemcpyAsync(s.h_status, s.d_status, sizeof(unsigned int), cudaMemcpyDeviceToHost, h->s_d2h));
    if (s.spec) {
        CU_TRY(cudaMemcpyAsync(diff_out, s.d_diff, s.spec, cudaMemcpyDeviceToHost, h->s_d2h));
        CU_TRY(cudaMemcpyAsync(xs, s.d_xs, (size_t)s.spec * sizeof(int), cudaMemcpyDeviceToHost, h->s_d2h));
    }
    if (dshow) CU_TRY(cudaMemcpyAsync(show, dshow, h->N, cudaMemcpyDeviceToHost, h->s_d2h));
    CU_TRY(cudaEventRecord(s.ev_pos, h->s_d2h));
    s.busy = true;
    s.ticket = h->next_ticket++;
    s.u_frame = diff_out;
    s.u_xs = xs;
    s.u_pos = pos;
    return CVS_OK;
}

// k_yuv_to_bgr<format> on `st`: planes / pitches as cvs_yuv_to_bgr_device takes them, already checked
static cvs_status yuv_launch(int format, const uint8_t *const *planes, const size_t *pitches, uint8_t *d_out, int width,
                             int height, cudaStream_t st)
{
    cvs::YuvParams p;
    const int nplanes = format == CVS_YUV_YUYV ? 1 : format == CVS_YUV_NV12 ? 2 : 3;
    for (int i = 0; i < 3; i++) {
        p.plane[i] = i < nplanes ? planes[i] : nullptr;
        p.pitch[i] = i < nplanes ? pitches[i] : 0;
    }
    p.bgr = d_out;
    p.width = width;
    p.height = height;
    p.groups = (uint32_t)(width + cvs::kYuvPixels - 1) / cvs::kYuvPixels;
    const unsigned blocks = (unsigned)(((size_t)p.groups * (size_t)height + cvs::kYuvThreads - 1) / cvs::kYuvThreads);
    if (format == CVS_YUV_YUYV) cvs::k_yuv_to_bgr<cvs::kYuyv><<<blocks, cvs::kYuvThreads, 0, st>>>(p);
    else if (format == CVS_YUV_NV12) cvs::k_yuv_to_bgr<cvs::kNv12><<<blocks, cvs::kYuvThreads, 0, st>>>(p);
    else cvs::k_yuv_to_bgr<cvs::kI420><<<blocks, cvs::kYuvThreads, 0, st>>>(p);
    CU_TRY(cudaGetLastError());
    return CVS_OK;
}

// the planes of a packed frame as cvs_submit_yuv receives it (rows without padding, planes back to back)
static void yuv_packed_planes(int format, const uint8_t *base, int width, int height, const uint8_t *planes[3], size_t pitches[3])
{
    const size_t luma = (size_t)width * (size_t)height;
    planes[0] = base;
    pitches[0] = format == CVS_YUV_YUYV ? 2 * (size_t)width : (size_t)width;
    planes[1] = base + luma;
    pitches[1] = format == CVS_YUV_NV12 ? (size_t)width : (size_t)width / 2;
    planes[2] = base + luma + luma / 4;
    pitches[2] = (size_t)width / 2;
}

// k_bayer_to_bgr on `st`: arguments as cvs_bayer_to_bgr_device takes them, already checked
static cvs_status bayer_launch(int pattern, const uint8_t *raw, size_t pitch, uint8_t *d_out, int width, int height,
                               cudaStream_t st)
{
    cvs::BayerParams p;
    p.raw = raw;
    p.pitch = pitch;
    p.bgr = d_out;
    p.width = width;
    p.height = height;
    p.groups = (uint32_t)(width + cvs::kBayerPixels - 1) / cvs::kBayerPixels;
    p.py = (pattern - CVS_BAYER_BGGR) >> 1; // BGGR, GBRG, GRBG, RGGB: (py, px) = (0, 0), (0, 1), (1, 0), (1, 1)
    p.px = (pattern - CVS_BAYER_BGGR) & 1;
    const unsigned blocks = (unsigned)(((size_t)p.groups * (size_t)height + cvs::kBayerThreads - 1) / cvs::kBayerThreads);
    cvs::k_bayer_to_bgr<<<blocks, cvs::kBayerThreads, 0, st>>>(p);
    CU_TRY(cudaGetLastError());
    return CVS_OK;
}

// The camera format of a submitted frame: 0 for a BGR frame (or a JPEG bitstream), a cvs_yuv_format, or kCamBayer plus a
// cvs_bayer_pattern.  A raw camera frame is uploaded as packed rows into the slot's staging buffer s.d_cam and converted
// to BGR on the compute stream in front of the stream kernel.
constexpr int kCamBayer = 16;

// bytes of a packed raw camera frame (cam != 0, checked by the caller)
static size_t cam_frame_bytes(int cam, int width, int height)
{
    return cam > kCamBayer ? (size_t)width * (size_t)height : cvs_yuv_frame_bytes(cam, width, height);
}

// the packed raw camera frame at `src` (device) -> BGR at d_out, on `st`
static cvs_status cam_to_bgr(int cam, const uint8_t *src, uint8_t *d_out, int width, int height, cudaStream_t st)
{
    if (cam > kCamBayer) return bayer_launch(cam - kCamBayer, src, (size_t)width, d_out, width, height, st);
    const uint8_t *planes[3];
    size_t pitches[3];
    yuv_packed_planes(cam, src, width, height, planes, pitches);
    return yuv_launch(cam, planes, pitches, d_out, width, height, st);
}

// H2D of a ticket's frame into s.d_in (kernels.cu:461) between the slot's timing events: the N-byte BGR frame, or
// (cam != 0) a raw camera frame into s.d_cam, converted on the compute stream later, or (jpeg_bytes != 0) the
// camera's JPEG bitstream, decoded on the device.  JPEG tickets alternate between two decode streams with their own
// scratch: frame t+1 is decoded beside frame t (a decode is a latency chain that leaves most of the GPU idle); the
// stream kernel still takes the frames in ticket order.  The compute stream waits for the frame and marks ev_k0.
static cvs_status ingest(cvs_handle h, Slot &s, const uint8_t *frame, size_t jpeg_bytes = 0, int cam = 0)
{
    cudaStream_t s_in = h->s_h2d;
    const JpegSet jset = (h->next_ticket & 1) ? kJpegTicketOdd : kJpegTicketEven;
    if (jpeg_bytes) {
        if (!h->s_jpg[jset]) CU_TRY(cudaStreamCreateWithFlags(&h->s_jpg[jset], cudaStreamNonBlocking));
        s_in = h->s_jpg[jset];
    }
    CU_TRY(cudaEventRecord(s.ev_h2d0, s_in));
    if (jpeg_bytes) {
        // (the ticket's status word is cleared here, in front of the decoder that may raise bits in it)
        CU_TRY(cudaMemsetAsync(s.d_status, 0, sizeof(unsigned int), s_in));
        CVS_TRY(jpeg_decode(h, jset, &s.jpeg_state, frame, jpeg_bytes, s.d_in, s_in, s.d_status));
    } else if (cam) {
        CU_TRY(cudaMemcpyAsync(s.d_cam, frame, cam_frame_bytes(cam, h->width, h->height), cudaMemcpyHostToDevice, h->s_h2d));
    } else {
        CU_TRY(cudaMemcpyAsync(s.d_in, frame, h->N, cudaMemcpyHostToDevice, h->s_h2d));
    }
    CU_TRY(cudaEventRecord(s.ev_h2d1, s_in));
    CU_TRY(cudaStreamWaitEvent(h->s_comp, s.ev_h2d1, 0));
    CU_TRY(cudaEventRecord(s.ev_k0, h->s_comp));
    return CVS_OK;
}

// jpeg_bytes != 0: `frame` is the camera's JPEG bitstream; cam != 0: `frame` is a raw camera frame of that format
// (checked by the caller); otherwise the N-byte BGR frame
static cvs_status submit_common(cvs_handle h, const uint8_t *frame, uint8_t *diff_out, uint8_t *show, const char *text,
                                unsigned int *pos, int *xs, uint8_t *wire_out, uint64_t *ticket, size_t jpeg_bytes = 0,
                                int cam = 0)
{
    cvs_status st = check_handle(h);
    if (st) return st;
    if (!frame || !ticket || (!wire_out && (!diff_out || !pos || !xs))) return fail(CVS_ERR_INVALID, "null argument");
    Slot &s = h->slot[h->next_ticket % kSlots];
    if (s.busy) return fail(CVS_ERR_INVALID, "%d tickets are already outstanding; cvs_wait the oldest first", kSlots);
    if (wire_out) {
        const uint32_t ntiles = (h->N + cvs::kWireTile - 1) / cvs::kWireTile;
        CVS_TRY(s.d_starts.grow((size_t)(ntiles + 2) * sizeof(uint32_t), "wire tile starts"));
        CVS_TRY(s.d_wire.grow(cvs_wire_bound(h->width, h->height), "wire frame"));
    }
    // sized for the largest layout (YUYV, 2WH), so tickets of every format share it
    if (cam) CVS_TRY(s.d_cam.grow(round_up(2 * (size_t)h->width * (size_t)h->height, 16), "camera frame"));

    const double th0 = h->trace ? host_us() : 0;
    CVS_TRY(ingest(h, s, frame, jpeg_bytes, cam));
    const size_t cap = round_up(h->N, 4);
    uint8_t *dshow = (h->mode && show) ? s.d_show.p : nullptr;
    const double th1 = h->trace ? host_us() : 0;
    if (!jpeg_bytes) CU_TRY(cudaMemsetAsync(s.d_status, 0, sizeof(unsigned int), h->s_comp));
    if (cam) { // (inside ev_k0 .. ev_k1: cvs_get_timing counts the conversion as kernel time)
        st = cam_to_bgr(cam, s.d_cam, s.d_in, h->width, h->height, h->s_comp);
        if (st) return st;
        h->launches++;
    }
    st = run_frames(h, s.d_in, h->Npad, 1, s.d_pos, s.d_xs, s.d_diff, cap, dshow, h->Npad, text, h->s_comp,
                    /*frames_private=*/true, s.d_status);
    if (st) return st;
    const double th2 = h->trace ? host_us() : 0;
    CU_TRY(cudaEventRecord(s.ev_k1, h->s_comp));
    st = egress(h, s, frame, diff_out, show, dshow, pos, xs, wire_out);
    if (st) return st;
    if (h->trace)
        fprintf(stderr, "submit host us: h2d %.1f run_frames %.1f d2h %.1f\n", th1 - th0, th2 - th1, host_us() - th2);
    *ticket = s.ticket;
    return CVS_OK;
}

cvs_status cvs_submit_io(cvs_handle h, const uint8_t *frame, uint8_t *diff_out, uint8_t *show, const char *text,
                         unsigned int *pos, int *xs, uint64_t *ticket)
{
    return submit_common(h, frame, diff_out, show, text, pos, xs, nullptr, ticket);
}

// the handles of a batch: 1..CVS_MAX_BATCH of them, none NULL or repeated, all on one device with one geometry, mode and
// threshold (the stream kernel's template and its launch-wide threshold); makes their device current
static cvs_status check_batch(const cvs_handle *hs, int n)
{
    if (n < 1 || n > CVS_MAX_BATCH) return fail(CVS_ERR_INVALID, "batch of %d streams (1..%d)", n, CVS_MAX_BATCH);
    if (!hs) return fail(CVS_ERR_INVALID, "null argument");
    for (int i = 0; i < n; i++) {
        const cvs_handle h = hs[i];
        if (!h) return fail(CVS_ERR_INVALID, "null handle at %d", i);
        for (int j = 0; j < i; j++)
            if (hs[j] == h) return fail(CVS_ERR_INVALID, "handle at %d repeats the one at %d", i, j);
        if (h->device != hs[0]->device || h->width != hs[0]->width || h->height != hs[0]->height || h->mode != hs[0]->mode ||
            h->threshold != hs[0]->threshold)
            return fail(CVS_ERR_INVALID, "stream %d differs from stream 0 in device, size, mode or threshold", i);
    }
    return check_handle(hs[0]);
}

cvs_status cvs_submit_io_batch(const cvs_handle *hs, int n, const uint8_t *const *frames, uint8_t *const *diff_out,
                               uint8_t *const *show, const char *const *texts, unsigned int *const *pos, int *const *xs,
                               uint64_t *tickets)
{
    cvs_status st = check_batch(hs, n);
    if (st) return st;
    if (!frames || !diff_out || !pos || !xs || !tickets) return fail(CVS_ERR_INVALID, "null argument");
    bool any_show = false;
    for (int i = 0; i < n; i++) {
        if (!frames[i] || !diff_out[i] || !pos[i] || !xs[i]) return fail(CVS_ERR_INVALID, "null entry at %d", i);
        if (hs[i]->slot[hs[i]->next_ticket % kSlots].busy)
            return fail(CVS_ERR_INVALID, "stream %d: %d tickets are already outstanding; cvs_wait the oldest first", i, kSlots);
        any_show = any_show || (show && show[i]);
    }
    any_show = any_show && hs[0]->mode;
    cvs_handle L = hs[0]; // the leader: its compute stream, descriptors and epoch carry the launch
    const uint8_t *d_frames[CVS_MAX_BATCH];
    unsigned int *d_pos[CVS_MAX_BATCH], *d_status[CVS_MAX_BATCH];
    int *d_xs[CVS_MAX_BATCH];
    uint8_t *d_diff[CVS_MAX_BATCH], *d_show[CVS_MAX_BATCH];
    for (int i = 0; i < n; i++) {
        cvs_handle h = hs[i];
        Slot &s = h->slot[h->next_ticket % kSlots];
        // upload on the stream's own copy stream; its compute stream then marks the point behind the upload and behind
        // the stream's earlier tickets (which updated the reference this batch starts from)
        CVS_TRY(ingest(h, s, frames[i]));
        CU_TRY(cudaStreamWaitEvent(L->s_comp, s.ev_k0, 0));
        d_frames[i] = s.d_in;
        d_pos[i] = s.d_pos;
        d_xs[i] = s.d_xs;
        d_diff[i] = s.d_diff;
        d_show[i] = any_show ? s.d_show.p : nullptr; // (a camera without a show buffer still gets its frame: not copied out)
        d_status[i] = s.d_status;
        CU_TRY(cudaMemsetAsync(s.d_status, 0, sizeof(unsigned int), L->s_comp));
    }
    st = run_batch(hs, n, d_frames, d_pos, d_xs, d_diff, round_up(L->N, 4), any_show ? d_show : nullptr, texts, L->s_comp,
                   /*frames_private=*/true, d_status);
    if (st) return st;
    for (int i = 0; i < n; i++) {
        cvs_handle h = hs[i];
        Slot &s = h->slot[h->next_ticket % kSlots];
        // later work of the stream (its next tickets, this ticket's egress) is ordered behind the batch
        CU_TRY(cudaEventRecord(s.ev_k1, L->s_comp));
        CU_TRY(cudaStreamWaitEvent(h->s_comp, s.ev_k1, 0));
        uint8_t *sh = show ? show[i] : nullptr;
        st = egress(h, s, frames[i], diff_out[i], sh, sh && any_show ? s.d_show.p : nullptr, pos[i], xs[i], nullptr);
        if (st) return st;
        tickets[i] = s.ticket;
    }
    return CVS_OK;
}

cvs_status cvs_submit_jpeg(cvs_handle h, const uint8_t *jpeg, size_t jpeg_bytes, uint8_t *diff_out, uint8_t *show,
                           const char *text, unsigned int *pos, int *xs, uint64_t *ticket)
{
    if (!jpeg || jpeg_bytes == 0) return fail(CVS_ERR_INVALID, "null argument");
    return submit_common(h, jpeg, diff_out, show, text, pos, xs, nullptr, ticket, jpeg_bytes);
}

cvs_status cvs_submit_jpeg_wire(cvs_handle h, const uint8_t *jpeg, size_t jpeg_bytes, uint8_t *wire_out, uint8_t *show,
                                const char *text, uint64_t *ticket)
{
    if (!jpeg || jpeg_bytes == 0 || !wire_out) return fail(CVS_ERR_INVALID, "null argument");
    return submit_common(h, jpeg, nullptr, show, text, nullptr, nullptr, wire_out, ticket, jpeg_bytes);
}

cvs_status cvs_decode_jpeg_device(cvs_handle h, const uint8_t *jpeg, size_t jpeg_bytes, uint8_t *d_out, void *cuda_stream)
{
    cvs_status st = check_handle(h);
    if (st) return st;
    if (!jpeg || jpeg_bytes == 0 || !d_out) return fail(CVS_ERR_INVALID, "null argument");
    // (status bits of the decoder go to the handle's own status word: cvs_decode_status reads it)
    st = jpeg_decode(h, kJpegCallerStream, &h->jpeg_state, jpeg, jpeg_bytes, d_out, (cudaStream_t)cuda_stream, h->d_status);
    if (st) return st;
    CU_TRY(cudaMemcpyAsync(h->h_status, h->d_status, sizeof(unsigned int), cudaMemcpyDeviceToHost, (cudaStream_t)cuda_stream));
    return CVS_OK;
}

// a YUV submission that cvs_submit_yuv / cvs_submit_yuv_wire refuse before anything is enqueued
static cvs_status check_yuv_submit(cvs_handle h, int format, const uint8_t *yuv)
{
    cvs_status st = check_handle(h);
    if (st) return st;
    if (format < CVS_YUV_YUYV || format > CVS_YUV_I420) return fail(CVS_ERR_INVALID, "unknown YUV format %d", format);
    if (!cvs_yuv_frame_bytes(format, h->width, h->height))
        return fail(CVS_ERR_INVALID, "a %dx%d stream cannot take YUV format %d (odd %s)", h->width, h->height, format,
                    format == CVS_YUV_YUYV ? "width" : "width or height");
    if (!yuv) return fail(CVS_ERR_INVALID, "null argument");
    return CVS_OK;
}

cvs_status cvs_submit_yuv(cvs_handle h, int format, const uint8_t *yuv, uint8_t *diff_out, uint8_t *show, const char *text,
                          unsigned int *pos, int *xs, uint64_t *ticket)
{
    cvs_status st = check_yuv_submit(h, format, yuv);
    if (st) return st;
    return submit_common(h, yuv, diff_out, show, text, pos, xs, nullptr, ticket, 0, format);
}

cvs_status cvs_submit_yuv_wire(cvs_handle h, int format, const uint8_t *yuv, uint8_t *wire_out, uint8_t *show,
                               const char *text, uint64_t *ticket)
{
    cvs_status st = check_yuv_submit(h, format, yuv);
    if (st) return st;
    if (!wire_out) return fail(CVS_ERR_INVALID, "null argument");
    return submit_common(h, yuv, nullptr, show, text, nullptr, nullptr, wire_out, ticket, 0, format);
}

// a Bayer submission that cvs_submit_bayer / cvs_submit_bayer_wire refuse before anything is enqueued (every frame size
// is accepted, as cv2.cvtColor does)
static cvs_status check_bayer_submit(cvs_handle h, int pattern, const uint8_t *raw)
{
    cvs_status st = check_handle(h);
    if (st) return st;
    if (pattern < CVS_BAYER_BGGR || pattern > CVS_BAYER_RGGB) return fail(CVS_ERR_INVALID, "unknown Bayer pattern %d", pattern);
    if (!raw) return fail(CVS_ERR_INVALID, "null argument");
    return CVS_OK;
}

cvs_status cvs_submit_bayer(cvs_handle h, int pattern, const uint8_t *raw, uint8_t *diff_out, uint8_t *show,
                            const char *text, unsigned int *pos, int *xs, uint64_t *ticket)
{
    cvs_status st = check_bayer_submit(h, pattern, raw);
    if (st) return st;
    return submit_common(h, raw, diff_out, show, text, pos, xs, nullptr, ticket, 0, kCamBayer + pattern);
}

cvs_status cvs_submit_bayer_wire(cvs_handle h, int pattern, const uint8_t *raw, uint8_t *wire_out, uint8_t *show,
                                 const char *text, uint64_t *ticket)
{
    cvs_status st = check_bayer_submit(h, pattern, raw);
    if (st) return st;
    if (!wire_out) return fail(CVS_ERR_INVALID, "null argument");
    return submit_common(h, raw, nullptr, show, text, nullptr, nullptr, wire_out, ticket, 0, kCamBayer + pattern);
}

cvs_status cvs_submit_wire(cvs_handle h, const uint8_t *frame, uint8_t *wire_out, uint8_t *show, const char *text,
                           uint64_t *ticket)
{
    if (!wire_out) return fail(CVS_ERR_INVALID, "null argument");
    return submit_common(h, frame, nullptr, show, text, nullptr, nullptr, wire_out, ticket);
}

cvs_status cvs_submit(cvs_handle h, uint8_t *frame, uint8_t *show, const char *text, unsigned int *pos, int *xs,
                      uint64_t *ticket)
{
    return cvs_submit_io(h, frame, frame, show, text, pos, xs, ticket);
}

cvs_status cvs_wait(cvs_handle h, uint64_t ticket)
{
    cvs_status st = check_handle(h);
    if (st) return st;
    Slot &s = h->slot[ticket % kSlots];
    if (!s.busy || s.ticket != ticket) return fail(CVS_ERR_INVALID, "unknown ticket %llu", (unsigned long long)ticket);
    CU_TRY(cudaEventSynchronize(s.ev_pos));
    st = status_word(*s.h_status);
    if (st == CVS_ERR_INTERNAL) {
        s.busy = false; // the ticket is consumed: its launch gave up, there is nothing to deliver
        return st;
    }
    const unsigned int n = *s.h_pos;
    // payload (kernels.cu:522-523): diff bytes over the head of the frame buffer, then the indices
    // (on their own stream: s_d2h already holds the work of the younger tickets, and anything queued behind
    // it would make this call wait for them)
    const unsigned int have = s.spec; // entries already on the host
    if (s.u_wire) {
        s.copied = !s.pushed;
        if (s.copied) { // pageable buffer: the encoded frame waits in device memory
            const size_t cap_n = n > h->N ? h->N : n;
            const size_t bytes = cvs::kWireHeader + cvs::wire_pad16((h->N + cvs::kWireTile - 1) / cvs::kWireTile) +
                                 cvs::wire_pad16((uint32_t)cap_n) + cap_n;
            CU_TRY(cudaMemcpyAsync(s.u_wire, s.d_wire, bytes, cudaMemcpyDeviceToHost, h->s_pay));
            CU_TRY(cudaEventRecord(s.ev_done, h->s_pay));
            CU_TRY(cudaEventSynchronize(s.ev_done));
        }
    } else if ((s.copied = n > have && !s.pushed)) {
        CU_TRY(cudaMemcpyAsync(s.u_frame + have, s.d_diff + have, n - have, cudaMemcpyDeviceToHost, h->s_pay));
        CU_TRY(cudaMemcpyAsync(s.u_xs + have, s.d_xs + have, (size_t)(n - have) * sizeof(int), cudaMemcpyDeviceToHost, h->s_pay));
        CU_TRY(cudaEventRecord(s.ev_done, h->s_pay));
        CU_TRY(cudaEventSynchronize(s.ev_done));
    }
    s.busy = false; // from here on nothing can fail: the slot may be reused
    if (s.u_pos) *s.u_pos = n;
    h->pred = n + (n / 16 > 16384 ? n / 16 : 16384); // change density is strongly correlated from frame to frame
    h->last_slot = (int)(ticket % kSlots);
    if (h->trace) { // CVS_TRACE=1: device timeline of every ticket on stderr (debug aid)
        float t[6] = {0, 0, 0, 0, 0, 0};
        cudaEvent_t ev[6] = {s.ev_h2d0, s.ev_h2d1, s.ev_k0, s.ev_k1, s.ev_pos, s.copied ? s.ev_done : s.ev_pos};
        for (int i = 0; i < 6; i++) cudaEventElapsedTime(&t[i], h->ev_base, ev[i]);
        fprintf(stderr, "stream %p ticket %llu h2d %.1f-%.1f kern %.1f-%.1f pos %.1f done %.1f us n %u %s\n", (void *)h,
                (unsigned long long)ticket, t[0] * 1e3, t[1] * 1e3, t[2] * 1e3, t[3] * 1e3, t[4] * 1e3, t[5] * 1e3, n,
                s.pushed ? "push" : (s.spec ? "spec" : "copy"));
    }
    // a capacity overflow or a damaged JPEG bitstream: the ticket is consumed and whatever the frame produced has been
    // delivered, but the caller must know (after a damaged frame the reference holds its pixels: cvs_reset re-seeds it)
    return st;
}

cvs_status cvs_exec(cvs_handle h, uint8_t *frame, uint8_t *show, const char *text, unsigned int *pos, int *xs)
{
    uint64_t ticket = 0;
    cvs_status st = cvs_submit(h, frame, show, text, pos, xs, &ticket);
    if (st) return st;
    return cvs_wait(h, ticket);
}

cvs_status cvs_get_timing(cvs_handle h, float *h2d_us, float *kernel_us, float *d2h_us)
{
    if (!h) return fail(CVS_ERR_INVALID, "null handle");
    if (h->last_slot >= 0) { // the events of the last completed ticket are read on demand, not per frame
        Slot &s = h->slot[h->last_slot];
        // the slot's events may already have been re-recorded by a younger ticket that is still in flight
        // (cudaErrorNotReady): keep the previous values then
        float a = 0, b = 0, c = 0, d = 0;
        cudaError_t e = cudaEventElapsedTime(&a, s.ev_h2d0, s.ev_h2d1);
        if (e == cudaSuccess) e = cudaEventElapsedTime(&b, s.ev_k0, s.ev_k1);
        if (e == cudaSuccess) e = cudaEventElapsedTime(&c, s.ev_p0, s.ev_pos);
        if (e == cudaSuccess && s.copied) e = cudaEventElapsedTime(&d, s.ev_pos, s.ev_done);
        if (e == cudaSuccess) {
            h->t_h2d = a * 1000.f;
            h->t_kernel = b * 1000.f;
            h->t_d2h = (c + d) * 1000.f;
        } else if (e == cudaErrorNotReady) {
            cudaGetLastError();
        } else {
            return fail(CVS_ERR_CUDA, "cudaEventElapsedTime failed: %s", cudaGetErrorString(e));
        }
    }
    if (h2d_us) *h2d_us = h->t_h2d;
    if (kernel_us) *kernel_us = h->t_kernel;
    if (d2h_us) *d2h_us = h->t_d2h;
    return CVS_OK;
}

cvs_status cvs_get_reference(cvs_handle h, uint8_t *out)
{
    cvs_status st = check_handle(h);
    if (st) return st;
    if (!out) return fail(CVS_ERR_INVALID, "null argument");
    CU_TRY(cudaDeviceSynchronize());
    CU_TRY(cudaMemcpy(out, h->d_ref, h->N, cudaMemcpyDeviceToHost));
    return CVS_OK;
}

cvs_status cvs_reference_device(cvs_handle h, void **dptr)
{
    if (!h || !dptr) return fail(CVS_ERR_INVALID, "null argument");
    *dptr = h->d_ref;
    return CVS_OK;
}

cvs_status cvs_run_sequence_device(cvs_handle h, const uint8_t *d_frames, size_t frame_stride, int nframes,
                                   unsigned int *d_pos, int *d_xs, uint8_t *d_diff, size_t payload_capacity,
                                   uint8_t *d_show, size_t show_stride, const char *text, void *cuda_stream)
{
    cvs_status st = check_handle(h);
    if (st) return st;
    if (nframes < 0 || !d_frames || !d_pos || !d_xs || !d_diff) return fail(CVS_ERR_INVALID, "null argument");
    if (!aligned16(d_frames, frame_stride, d_xs, d_diff) || (d_show && !aligned16(d_show, show_stride)))
        return fail(CVS_ERR_ALIGN, "device pointers and strides must be 16-byte aligned");
    if (frame_stride < h->N16) return fail(CVS_ERR_INVALID, "frame_stride %zu < %u", frame_stride, h->N16);
    if (d_show && show_stride < h->N) return fail(CVS_ERR_INVALID, "show_stride too small");
    if (payload_capacity == 0 || (payload_capacity & 3))
        return fail(CVS_ERR_INVALID, "payload_capacity must be a positive multiple of 4");
    cudaStream_t s = (cudaStream_t)cuda_stream;
    st = run_frames(h, d_frames, frame_stride, nframes, d_pos, d_xs, d_diff, payload_capacity, d_show, show_stride, text, s,
                    /*frames_private=*/false, h->d_status);
    if (st) return st;
    CU_TRY(cudaMemcpyAsync(h->h_status, h->d_status, sizeof(unsigned int), cudaMemcpyDeviceToHost, s));
    return CVS_OK;
}

cvs_status cvs_run_batch_device(const cvs_handle *hs, int n, const uint8_t *const *d_frames, unsigned int *d_pos, int *d_xs,
                                uint8_t *d_diff, size_t payload_capacity, uint8_t *d_show, size_t show_stride,
                                const char *const *texts, void *cuda_stream)
{
    cvs_status st = check_batch(hs, n);
    if (st) return st;
    if (!d_frames || !d_pos || !d_xs || !d_diff) return fail(CVS_ERR_INVALID, "null argument");
    for (int i = 0; i < n; i++)
        if (!d_frames[i]) return fail(CVS_ERR_INVALID, "null frame at %d", i);
    bool aligned = aligned16(d_xs, d_diff) && (!d_show || aligned16(d_show, show_stride));
    for (int i = 0; i < n; i++) aligned = aligned && aligned16(d_frames[i]);
    if (!aligned)
        return fail(CVS_ERR_ALIGN, "device pointers and strides must be 16-byte aligned");
    if (d_show && show_stride < hs[0]->N) return fail(CVS_ERR_INVALID, "show_stride too small");
    if (payload_capacity == 0 || (payload_capacity & 3))
        return fail(CVS_ERR_INVALID, "payload_capacity must be a positive multiple of 4");
    unsigned int *pos[CVS_MAX_BATCH], *status[CVS_MAX_BATCH];
    int *xs[CVS_MAX_BATCH];
    uint8_t *diff[CVS_MAX_BATCH], *show[CVS_MAX_BATCH];
    for (int i = 0; i < n; i++) {
        pos[i] = d_pos + i;
        xs[i] = d_xs + (size_t)i * payload_capacity;
        diff[i] = d_diff + (size_t)i * payload_capacity;
        show[i] = d_show ? d_show + (size_t)i * show_stride : nullptr;
        status[i] = hs[i]->d_status;
    }
    cudaStream_t s = (cudaStream_t)cuda_stream;
    st = run_batch(hs, n, d_frames, pos, xs, diff, payload_capacity, d_show ? show : nullptr, texts, s,
                   /*frames_private=*/false, status);
    if (st) return st;
    for (int i = 0; i < n; i++)
        CU_TRY(cudaMemcpyAsync(hs[i]->h_status, hs[i]->d_status, sizeof(unsigned int), cudaMemcpyDeviceToHost, s));
    return CVS_OK;
}

cvs_status cvs_sequence_status(cvs_handle h)
{
    cvs_status st = check_handle(h);
    if (st) return st;
    st = status_word(*h->h_status);
    if (*h->h_status) { // sticky bits are cleared once reported
        CU_TRY(cudaMemset(h->d_status, 0, sizeof(unsigned int)));
        *h->h_status = 0;
    }
    return st;
}

uint64_t cvs_launch_count(cvs_handle h) { return h ? h->launches : 0; }

// ---------------------------------------------------------------------------------------------
// stand-alone filters on device buffers (current device)
// ---------------------------------------------------------------------------------------------
static cvs_status filter_common(int &sms)
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || !device_is_sm100(dev)) {
        cudaGetLastError();
        return fail(CVS_ERR_NODEVICE, "no sm_100 device (there is no CPU fallback)");
    }
    CU_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    return CVS_OK;
}

cvs_status cvs_heat_map_device(const uint8_t *d_prev, const uint8_t *d_cur, uint8_t *d_out, int width, int height,
                               void *cuda_stream)
{
    int sms = 0;
    cvs_status st = filter_common(sms);
    if (st) return st;
    if (!d_prev || !d_cur || !d_out || width <= 0 || height <= 0) return fail(CVS_ERR_INVALID, "bad argument");
    if (!aligned16(d_prev, d_cur, d_out)) return fail(CVS_ERR_ALIGN, "16-byte alignment required");
    uint32_t *lut = nullptr;
    st = device_heat_lut(&lut);
    if (st) return st;
    const uint32_t n = 3u * (uint32_t)width * (uint32_t)height;
    cvs::k_filter<0, false><<<grid_for((n + 47) / 48, 256, sms), 256, 0, (cudaStream_t)cuda_stream>>>(d_prev, d_cur, d_out, n, 0, lut, nullptr);
    CU_TRY(cudaGetLastError());
    return CVS_OK;
}

cvs_status cvs_red_map_device(const uint8_t *d_prev, const uint8_t *d_cur, uint8_t *d_out, int width, int height,
                              int threshold, void *cuda_stream)
{
    int sms = 0;
    cvs_status st = filter_common(sms);
    if (st) return st;
    if (!d_prev || !d_cur || !d_out || width <= 0 || height <= 0) return fail(CVS_ERR_INVALID, "bad argument");
    if (!aligned16(d_prev, d_cur, d_out)) return fail(CVS_ERR_ALIGN, "16-byte alignment required");
    bool hi;
    uint32_t addc;
    threshold_consts(threshold, hi, addc);
    const uint32_t n = 3u * (uint32_t)width * (uint32_t)height;
    const int grid = grid_for((n + 47) / 48, 256, sms);
    if (hi) cvs::k_filter<1, true><<<grid, 256, 0, (cudaStream_t)cuda_stream>>>(d_prev, d_cur, d_out, n, addc, nullptr, nullptr);
    else cvs::k_filter<1, false><<<grid, 256, 0, (cudaStream_t)cuda_stream>>>(d_prev, d_cur, d_out, n, addc, nullptr, nullptr);
    CU_TRY(cudaGetLastError());
    return CVS_OK;
}

static cvs_status gray_launch(const uint8_t *d_frame, uint8_t *d_out, uint32_t n, int weighted, int channels,
                              unsigned int *d_hist, int sms, cudaStream_t s)
{
    const int grid = grid_for((n + 47) / 48, 256, sms);
    if (channels == 3) {
        if (weighted) cvs::k_filter<3, false><<<grid, 256, 0, s>>>(nullptr, d_frame, d_out, n, 0, nullptr, nullptr);
        else cvs::k_filter<2, false><<<grid, 256, 0, s>>>(nullptr, d_frame, d_out, n, 0, nullptr, nullptr);
    } else {
        if (weighted) cvs::k_filter<5, false><<<grid, 256, 0, s>>>(nullptr, d_frame, d_out, n, 0, nullptr, d_hist);
        else cvs::k_filter<4, false><<<grid, 256, 0, s>>>(nullptr, d_frame, d_out, n, 0, nullptr, d_hist);
    }
    CU_TRY(cudaGetLastError());
    return CVS_OK;
}

cvs_status cvs_grayscale_device(const uint8_t *d_frame, uint8_t *d_out, int width, int height, int weighted,
                                int channels, void *cuda_stream)
{
    int sms = 0;
    cvs_status st = filter_common(sms);
    if (st) return st;
    if (!d_frame || !d_out || width <= 0 || height <= 0 || (channels != 1 && channels != 3))
        return fail(CVS_ERR_INVALID, "bad argument");
    if (!aligned16(d_frame, d_out)) return fail(CVS_ERR_ALIGN, "16-byte alignment required");
    return gray_launch(d_frame, d_out, 3u * (uint32_t)width * (uint32_t)height, weighted, channels, nullptr, sms,
                       (cudaStream_t)cuda_stream);
}

cvs_status cvs_binarize_device(const uint8_t *d_frame, uint8_t *d_out, uint8_t *d_gray, int *d_hist_thr, int width,
                               int height, int weighted, int clamp_lo, int clamp_hi, void *cuda_stream)
{
    int sms = 0;
    cvs_status st = filter_common(sms);
    if (st) return st;
    if (!d_frame || !d_out || !d_gray || !d_hist_thr || width <= 0 || height <= 0)
        return fail(CVS_ERR_INVALID, "bad argument");
    if (!aligned16(d_frame, d_out, d_gray))
        return fail(CVS_ERR_ALIGN, "16-byte alignment required");
    cudaStream_t s = (cudaStream_t)cuda_stream;
    const uint32_t npix = (uint32_t)width * (uint32_t)height;
    CU_TRY(cudaMemsetAsync(d_hist_thr, 0, 257 * sizeof(int), s));
    st = gray_launch(d_frame, d_gray, 3u * npix, weighted, 1, (unsigned int *)d_hist_thr, sms, s);
    if (st) return st;
    cvs::k_threshold<<<1, 256, 0, s>>>((const unsigned int *)d_hist_thr, d_hist_thr + 256, 1, clamp_lo, clamp_hi);
    CU_TRY(cudaGetLastError());
    cvs::k_binarize_expand<<<dim3(grid_for((npix + 15) / 16, 256, sms), 1), 256, 0, s>>>(d_gray, 0, d_out, 0,
                                                                                        d_hist_thr + 256, npix);
    CU_TRY(cudaGetLastError());
    return CVS_OK;
}

cvs_status cvs_noise_filter_device(const uint8_t *d_frame, uint8_t *d_out, int width, int height, int ksize,
                                   const float *h_weights, void *cuda_stream)
{
    int sms = 0;
    cvs_status st = filter_common(sms);
    if (st) return st;
    if (!d_frame || !d_out || !h_weights || width <= 0 || height <= 0 || ksize < 1 || ksize > 9 || !(ksize & 1))
        return fail(CVS_ERR_INVALID, "bad argument");
    if (d_frame == d_out) return fail(CVS_ERR_INVALID, "the noise filter is not in-place");
    cvs::ConvWeights w;
    memset(&w, 0, sizeof w);
    memcpy(w.k, h_weights, sizeof(float) * ksize * ksize);
    const size_t n = (size_t)3 * width * height;
    return launch_conv(d_frame, d_out, width, height, n, n, 1, ksize, w, (cudaStream_t)cuda_stream);
}

cvs_status cvs_client_apply_device(uint8_t *d_frame, const int *d_xs, const uint8_t *d_diff, const unsigned int *d_pos,
                                   size_t capacity, void *cuda_stream)
{
    int sms = 0;
    cvs_status st = filter_common(sms);
    if (st) return st;
    if (!d_frame || !d_xs || !d_diff || !d_pos) return fail(CVS_ERR_INVALID, "null argument");
    cvs::k_client_apply<<<sms * 4, 256, 0, (cudaStream_t)cuda_stream>>>(d_frame, d_xs, d_diff, d_pos, capacity);
    CU_TRY(cudaGetLastError());
    return CVS_OK;
}

size_t cvs_wire_bound(int width, int height)
{
    if (width <= 0 || height <= 0) return 0;
    const uint64_t n = (uint64_t)3 * (uint64_t)width * (uint64_t)height;
    const uint64_t ntiles = (n + cvs::kWireTile - 1) / cvs::kWireTile;
    return (size_t)(cvs::kWireHeader + ((ntiles + 15) & ~15ull) + ((n + 15) & ~15ull) + n);
}

size_t cvs_wire_size(const uint8_t *wire)
{
    if (!wire) return 0;
    uint32_t hd[4];
    memcpy(hd, wire, sizeof hd);
    if (hd[0] != cvs::kWireMagic || hd[3] != cvs::kWireTile) return 0;
    // in 64 bits: ntiles and pos come from the sender, and near 2^32 their padding would wrap in 32
    const uint64_t ntiles = hd[2], pos = hd[1];
    return (size_t)(cvs::kWireHeader + ((ntiles + 15) & ~15ull) + ((pos + 15) & ~15ull) + pos);
}

cvs_status cvs_wire_encode_device(const int *d_xs, const uint8_t *d_diff, const unsigned int *d_pos, size_t capacity,
                                  int width, int height, uint32_t *d_scratch, uint8_t *d_wire, void *cuda_stream)
{
    int sms = 0;
    cvs_status st = filter_common(sms);
    if (st) return st;
    if (!d_xs || !d_diff || !d_pos || !d_scratch || !d_wire || width <= 0 || height <= 0)
        return fail(CVS_ERR_INVALID, "bad argument");
    if (!aligned16(d_xs, d_diff, d_wire)) return fail(CVS_ERR_ALIGN, "16-byte alignment required");
    const uint32_t n = 3u * (uint32_t)width * (uint32_t)height, ntiles = (n + cvs::kWireTile - 1) / cvs::kWireTile;
    cudaStream_t s = (cudaStream_t)cuda_stream;
    cvs::k_wire_bounds<<<(ntiles + 256) / 256, 256, 0, s>>>(d_xs, d_pos, capacity, ntiles, d_scratch);
    CU_TRY(cudaGetLastError());
    cvs::k_wire_pack<<<2 * sms, 256, 0, s>>>(d_xs, d_diff, d_pos, capacity, ntiles, d_scratch, d_wire);
    CU_TRY(cudaGetLastError());
    return CVS_OK;
}

cvs_status cvs_wire_decode_device(const uint8_t *d_wire, uint32_t *d_scratch, uint8_t *d_frame, int *d_xs, uint8_t *d_diff,
                                  unsigned int *d_pos, int width, int height, void *cuda_stream)
{
    int sms = 0;
    cvs_status st = filter_common(sms);
    if (st) return st;
    if (!d_wire || !d_scratch || width <= 0 || height <= 0) return fail(CVS_ERR_INVALID, "bad argument");
    if (!aligned16(d_wire)) return fail(CVS_ERR_ALIGN, "16-byte alignment required");
    const uint32_t n = 3u * (uint32_t)width * (uint32_t)height, ntiles = (n + cvs::kWireTile - 1) / cvs::kWireTile;
    const uint32_t last_len = n - (ntiles - 1) * cvs::kWireTile;
    cudaStream_t s = (cudaStream_t)cuda_stream;
    // header, counts and sum; then the offsets of a frame that passed; then the frame, unless one of the two refused it
    cvs::k_wire_scan<<<1, 1024, 0, s>>>(d_wire, ntiles, last_len, d_scratch);
    CU_TRY(cudaGetLastError());
    cvs::k_wire_check<<<4 * sms, 256, 0, s>>>(d_wire, ntiles, last_len, d_scratch);
    CU_TRY(cudaGetLastError());
    cvs::k_wire_apply<<<4 * sms, 256, 0, s>>>(d_wire, ntiles, d_scratch, d_frame, d_xs, d_diff, d_pos);
    CU_TRY(cudaGetLastError());
    return CVS_OK;
}

cvs_status cvs_wire_decode_status(const uint32_t *d_scratch, int width, int height, void *cuda_stream)
{
    if (!d_scratch || width <= 0 || height <= 0) return fail(CVS_ERR_INVALID, "bad argument");
    const uint32_t n = 3u * (uint32_t)width * (uint32_t)height, ntiles = (n + cvs::kWireTile - 1) / cvs::kWireTile;
    uint32_t flag = 0;
    CU_TRY(cudaMemcpyAsync(&flag, d_scratch + ntiles + 1, sizeof flag, cudaMemcpyDeviceToHost, (cudaStream_t)cuda_stream));
    CU_TRY(cudaStreamSynchronize((cudaStream_t)cuda_stream));
    if (flag) return fail(CVS_ERR_INVALID, "encoded frame is inconsistent (magic, tile or geometry, a tile count above its tile's length, counts that do not "
                                       "add up to pos, or offsets out of range or not ascending): nothing was applied");
    return CVS_OK;
}

size_t cvs_yuv_frame_bytes(int format, int width, int height)
{
    if (width <= 0 || height <= 0 || (width & 1)) return 0;
    const uint64_t luma = (uint64_t)width * (uint64_t)height;
    if (format == CVS_YUV_YUYV) return (size_t)(2 * luma);
    if ((format == CVS_YUV_NV12 || format == CVS_YUV_I420) && !(height & 1)) return (size_t)(luma + luma / 2);
    return 0;
}

cvs_status cvs_yuv_to_bgr_device(int format, const uint8_t *const *planes, const size_t *pitches, uint8_t *d_out, int width,
                                 int height, void *cuda_stream)
{
    // arguments first: a refusal needs no device
    if (format < CVS_YUV_YUYV || format > CVS_YUV_I420) return fail(CVS_ERR_INVALID, "unknown YUV format %d", format);
    if (!cvs_yuv_frame_bytes(format, width, height))
        return fail(CVS_ERR_INVALID, "%dx%d: not a size YUV format %d takes (positive, width even; 4:2:0 height even)", width,
                    height, format);
    if (!planes || !pitches || !d_out) return fail(CVS_ERR_INVALID, "null argument");
    const int nplanes = format == CVS_YUV_YUYV ? 1 : format == CVS_YUV_NV12 ? 2 : 3;
    const size_t row_bytes[3] = {format == CVS_YUV_YUYV ? 2 * (size_t)width : (size_t)width,
                                 format == CVS_YUV_NV12 ? (size_t)width : (size_t)width / 2, (size_t)width / 2};
    bool aligned = aligned16(d_out);
    for (int i = 0; i < nplanes; i++) {
        if (!planes[i]) return fail(CVS_ERR_INVALID, "null plane %d", i);
        if (pitches[i] < row_bytes[i]) return fail(CVS_ERR_INVALID, "pitch of plane %d is %zu, its rows hold %zu bytes", i, pitches[i], row_bytes[i]);
        aligned = aligned && aligned16(planes[i], pitches[i]);
    }
    if (!aligned) return fail(CVS_ERR_ALIGN, "planes, pitches and d_out must be 16-byte aligned");
    int sms = 0;
    cvs_status st = filter_common(sms);
    if (st) return st;
    return yuv_launch(format, planes, pitches, d_out, width, height, (cudaStream_t)cuda_stream);
}

cvs_status cvs_bayer_to_bgr_device(int pattern, const uint8_t *d_raw, size_t pitch, uint8_t *d_out, int width, int height,
                                   void *cuda_stream)
{
    // arguments first: a refusal needs no device
    if (pattern < CVS_BAYER_BGGR || pattern > CVS_BAYER_RGGB) return fail(CVS_ERR_INVALID, "unknown Bayer pattern %d", pattern);
    if (width <= 0 || height <= 0) return fail(CVS_ERR_INVALID, "%dx%d: not a frame size", width, height);
    if (!d_raw || !d_out) return fail(CVS_ERR_INVALID, "null argument");
    if (pitch < (size_t)width) return fail(CVS_ERR_INVALID, "pitch %zu is less than the width %d", pitch, width);
    if (!aligned16(d_raw, pitch, d_out)) return fail(CVS_ERR_ALIGN, "d_raw, pitch and d_out must be 16-byte aligned");
    int sms = 0;
    cvs_status st = filter_common(sms);
    if (st) return st;
    return bayer_launch(pattern, d_raw, pitch, d_out, width, height, (cudaStream_t)cuda_stream);
}

cvs_status cvs_synth_base_device(uint8_t *d_out, int width, int height, uint64_t seed, void *cuda_stream)
{
    int sms = 0;
    cvs_status st = filter_common(sms);
    if (st) return st;
    if (!d_out || width <= 0 || height <= 0) return fail(CVS_ERR_INVALID, "bad argument");
    const uint32_t n = 3u * (uint32_t)width * (uint32_t)height;
    cvs::k_synth_base<<<grid_for(n, 256, sms), 256, 0, (cudaStream_t)cuda_stream>>>(d_out, n, width, height, seed);
    CU_TRY(cudaGetLastError());
    return CVS_OK;
}

cvs_status cvs_synth_next_device(const uint8_t *d_prev, uint8_t *d_out, int width, int height, uint64_t seed,
                                 uint32_t frame_index, uint32_t density_ppm, void *cuda_stream)
{
    int sms = 0;
    cvs_status st = filter_common(sms);
    if (st) return st;
    if (!d_prev || !d_out || width <= 0 || height <= 0) return fail(CVS_ERR_INVALID, "bad argument");
    const uint32_t n = 3u * (uint32_t)width * (uint32_t)height;
    const uint64_t key = cvs::splitmix64(seed ^ ((uint64_t)(frame_index + 1) * 0xD6E8FEB86659FD93ull));
    cvs::k_synth_next<<<grid_for(n, 256, sms), 256, 0, (cudaStream_t)cuda_stream>>>(d_prev, d_out, n, key, density_ppm);
    CU_TRY(cudaGetLastError());
    return CVS_OK;
}

} // extern "C"
