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

#include <atomic>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <mutex>
#include <string>

#include "cvs_filter_kernels.cuh"
#include "cvs_jpeg_host.hpp"
#include "cvs_stream_kernel.cuh"
#include "cvs_stream_ws.cuh"

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

inline size_t round_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

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
    uint8_t *d_arena = nullptr;   // everything below points into this one allocation
    size_t zero_bytes_fixed = 0;  // bytes in front of the coefficients that every decode clears
    uint8_t *d_raw = nullptr, *d_unst = nullptr; // entropy-coded segment as received / unstuffed (zero-padded)
    size_t raw_cap = 0;
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
    size_t sub_cap = 0;
    unsigned int *d_changed = nullptr;
    int16_t *d_coef = nullptr;
    uint8_t *d_planes = nullptr;
    size_t block_cap = 0;
    int coop_blocks_per_sm = 0;
    uint32_t sub_bits = 1024;
    void release() { cudaFree(d_arena); }
};

struct Slot {
    uint8_t *d_in = nullptr;   // raw frame as uploaded
    int *d_xs = nullptr;
    uint8_t *d_diff = nullptr;
    unsigned int *d_pos = nullptr;
    uint8_t *d_show = nullptr;
    unsigned int *h_pos = nullptr; // pinned
    uint32_t *d_starts = nullptr;     // compact wire format: entries before each tile (ntiles + 2 words), on first use
    uint8_t *d_wire = nullptr;        // compact wire format: encoded frame when the caller's buffer is not mapped
    nvjpegJpegState_t jpeg_state = nullptr; // cvs_submit_jpeg: decoder state of this slot (on first use)
    uint8_t *u_wire = nullptr;        // caller's buffer of a cvs_submit_wire ticket (nullptr: reference-format ticket)
    unsigned int *d_status = nullptr; // StatusBits of this ticket's launches (cleared at submit)
    unsigned int *h_status = nullptr; // pinned copy, valid once ev_pos has fired
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

typedef void (*StreamKernel)(const cvs::StreamParams);

template <int MODE>
StreamKernel pick_hr(bool hi, bool refreg)
{
    if (hi) return refreg ? cvs::k_stream<MODE, true, true> : cvs::k_stream<MODE, true, false>;
    return refreg ? cvs::k_stream<MODE, false, true> : cvs::k_stream<MODE, false, false>;
}
StreamKernel pick_kernel(int mode, bool hi, bool refreg)
{
    switch (mode) {
    case 1: return pick_hr<1>(hi, refreg);
    case 2: return pick_hr<2>(hi, refreg);
    case 3: return pick_hr<3>(hi, refreg);
    case 4: return pick_hr<4>(hi, refreg);
    case 5: return pick_hr<5>(hi, refreg);
    case 6: return pick_hr<6>(hi, refreg);
    case 7: return pick_hr<7>(hi, refreg);
    default: return pick_hr<0>(hi, refreg);
    }
}

template <int MODE>
StreamKernel pick_ws_hr(bool hi, bool refreg)
{
    if (hi) return refreg ? cvs::k_stream_ws<MODE, true, true> : cvs::k_stream_ws<MODE, true, false>;
    return refreg ? cvs::k_stream_ws<MODE, false, true> : cvs::k_stream_ws<MODE, false, false>;
}
StreamKernel pick_ws_kernel(int mode, bool hi, bool refreg)
{
    switch (mode) {
    case 1: return pick_ws_hr<1>(hi, refreg);
    case 2: return pick_ws_hr<2>(hi, refreg);
    case 3: return pick_ws_hr<3>(hi, refreg);
    case 4: return pick_ws_hr<4>(hi, refreg);
    case 5: return pick_ws_hr<5>(hi, refreg);
    case 6: return pick_ws_hr<6>(hi, refreg);
    case 7: return pick_ws_hr<7>(hi, refreg);
    default: return pick_ws_hr<0>(hi, refreg);
    }
}

typedef void (*BatchKernel)(const cvs::StreamParams, const cvs::BatchTable);

template <int MODE>
BatchKernel pick_batch_h(bool hi)
{
    return hi ? cvs::k_stream_ws_batch<MODE, true> : cvs::k_stream_ws_batch<MODE, false>;
}
BatchKernel pick_batch_kernel(int mode, bool hi)
{
    switch (mode) {
    case 1: return pick_batch_h<1>(hi);
    case 2: return pick_batch_h<2>(hi);
    case 3: return pick_batch_h<3>(hi);
    case 4: return pick_batch_h<4>(hi);
    case 5: return pick_batch_h<5>(hi);
    case 6: return pick_batch_h<6>(hi);
    case 7: return pick_batch_h<7>(hi);
    default: return pick_batch_h<0>(hi);
    }
}
static_assert(cvs::kMaxBatch == CVS_MAX_BATCH, "batch table and public limit");

} // namespace

struct cvs_stream_s {
    int width = 0, height = 0, threshold = 20, mode = 0, noise_filter = 0, ksize = 3, device = 0;
    int max_sequence = 512;
    uint32_t N = 0, N16 = 0, nchunks = 0, npix = 0;
    size_t Npad = 0, P16 = 0;
    bool hi = false;
    uint32_t addc = 0;
    uint32_t debug = 0; // CVS_DEBUG_FLAGS (profiling experiments only)
    int stages = 0;     // CVS_STAGES: ring depth override (0 = default)
    bool trace = false;
    cudaEvent_t ev_base = nullptr;
    uint32_t pred = 0;        // predicted entries of the next frame (previous count + margin)
    cvs::ConvWeights weights;
    int sms = 0;
    // glyph atlas
    uint8_t *d_glyphs = nullptr;
    int glyph_w = 0, glyph_h = 0;
    std::string glyph_chars;
    // device state
    uint8_t *d_ref = nullptr;
    uint32_t *d_lut = nullptr;
    unsigned int *d_status = nullptr;
    unsigned int *h_status = nullptr; // pinned
    unsigned long long *d_desc = nullptr;
    size_t desc_words = 0;
    JpegDecoder jd[3];                  // the library's own decoder (cvs_jpeg.cuh), scratch allocated on first use: sets 0 / 1
                                        // for cvs_submit_jpeg on two streams (consecutive frames decode side by side),
                                        // set 2 for cvs_decode_jpeg_device on the caller's stream
    cudaStream_t s_jpg[2] = {nullptr, nullptr};
    bool jpeg_own_only = false;         // own decoder only: refuse the forms it does not cover instead of using nvJPEG
    nvjpegHandle_t jpeg = nullptr;      // cvs_submit_jpeg / cvs_decode_jpeg_device: nvJPEG handle (on first use)
    bool jpeg_batched = false;          // the handle's backend wants the batched entry points (hardware engine / GPU Huffman)
    nvjpegJpegState_t jpeg_state = nullptr; // decoder state of cvs_decode_jpeg_device
    unsigned int *d_band_pos = nullptr; // banded launches: two arrays of per-frame counts so far (ping-pong)
    size_t band_frames = 0;
    uint32_t epoch = 0;
    // scratch that grows with the longest sequence seen
    uint8_t *d_work = nullptr;   // filtered / overlaid frames
    size_t work_frames = 0;
    uint8_t *d_gray1 = nullptr;  // binarise: 1 B per pixel per frame
    unsigned int *d_hist = nullptr;
    int *d_thr = nullptr;
    size_t bin_frames = 0;
    // geometry of the persistent launch (per kernel variant)
    cudaStream_t s_comp = nullptr, s_h2d = nullptr, s_d2h = nullptr, s_pay = nullptr;
    Slot slot[kSlots];
    int last_slot = -1; // slot of the most recently completed ticket (for cvs_get_timing)
    int occ_cache[8][2][2] = {}; // co-resident blocks per SM of each k_stream variant (0 = not queried yet)
    int occ_ws[8][2][2] = {};    // same for k_stream_ws
    int occ_batch[8][2] = {};    // same for k_stream_ws_batch
    bool use_ws = true;          // CVS_STREAM_KERNEL=v1 selects the one-group kernel (k_stream) for A/B measurements
    bool force_ws = false;       // CVS_STREAM_KERNEL=ws: k_stream_ws also for multi-pass frames
    uint64_t next_ticket = 1;
    uint64_t launches = 0;
    float t_h2d = 0, t_kernel = 0, t_d2h = 0;
    cvs_status seq_status = CVS_OK;
};

namespace {

cvs_status ensure_desc(cvs_handle h, size_t words)
{
    if (h->desc_words >= words) return CVS_OK;
    if (h->d_desc) {
        CU_TRY(cudaDeviceSynchronize());
        CU_TRY(cudaFree(h->d_desc));
        h->d_desc = nullptr;
        h->desc_words = 0;
    }
    CU_TRY(cudaMalloc(&h->d_desc, words * sizeof(unsigned long long)));
    CU_TRY(cudaMemset(h->d_desc, 0, words * sizeof(unsigned long long)));
    h->desc_words = words;
    return CVS_OK;
}

cvs_status ensure_work(cvs_handle h, size_t frames)
{
    if (h->work_frames >= frames) return CVS_OK;
    if (h->d_work) {
        CU_TRY(cudaDeviceSynchronize());
        CU_TRY(cudaFree(h->d_work));
        h->d_work = nullptr;
        h->work_frames = 0;
    }
    CU_TRY(cudaMalloc(&h->d_work, frames * h->Npad + 64));
    CU_TRY(cudaMemset(h->d_work, 0, frames * h->Npad + 64));
    h->work_frames = frames;
    return CVS_OK;
}

cvs_status ensure_bin(cvs_handle h, size_t frames)
{
    if (h->bin_frames >= frames) return CVS_OK;
    if (h->d_gray1 || h->d_hist || h->d_thr) {
        CU_TRY(cudaDeviceSynchronize());
        // forget the pointers before anything below can fail: a later call (or cvs_destroy) must not free them again
        uint8_t *g = h->d_gray1;
        unsigned int *hi = h->d_hist;
        int *th = h->d_thr;
        h->d_gray1 = nullptr;
        h->d_hist = nullptr;
        h->d_thr = nullptr;
        h->bin_frames = 0;
        cudaFree(g);
        cudaFree(hi);
        cudaFree(th);
    }
    uint8_t *g = nullptr;
    unsigned int *hi = nullptr;
    int *th = nullptr;
    if (cudaMalloc(&g, frames * h->P16 + 64) != cudaSuccess || cudaMalloc(&hi, frames * 256 * sizeof(unsigned int)) != cudaSuccess ||
        cudaMalloc(&th, frames * sizeof(int)) != cudaSuccess) {
        cudaGetLastError();
        cudaFree(g);
        cudaFree(hi);
        cudaFree(th);
        return fail(CVS_ERR_NOMEM, "binarisation scratch for %zu frames does not fit", frames);
    }
    h->d_gray1 = g;
    h->d_hist = hi;
    h->d_thr = th;
    h->bin_frames = frames;
    return CVS_OK;
}

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
    const bool need_work = h->noise_filter || (txt.n && !frames_private);
    if (need_work) {
        cvs_status s = ensure_work(h, (size_t)piece_max);
        if (s) return s;
    }
    if (binarize) {
        cvs_status s = ensure_bin(h, (size_t)piece_max);
        if (s) return s;
    }

    // ---- geometry of the persistent launch: G co-resident blocks, each owning the same cps consecutive chunks of
    //      every frame.  k_stream_ws (front / back warp groups) wherever the reference can stay in registers.
    // Frames that do not fit one pass of the grid (3840x2160): a SEQUENCE is walked band by band -- every band is a
    // byte range of the frame that does fit, and one k_stream_ws launch takes that band through all frames of the
    // piece with its reference bytes in registers; frame t's entries of band j are appended behind those of the bands
    // before it (counts handed from launch to launch).  Same payload, 1.3-1.8x faster than walking the frame in
    // segments with the reference going through L2, which is what single frames (the drop-in call) still do, with
    // the one-group kernel k_stream (k_stream_ws measured 25 against 17 us per 4K frame there).
    bool ws = h->use_ws;
    int nbands = 1;
    {
        const int g0 = h->sms < 32 * cvs::kWsLook ? h->sms : 32 * cvs::kWsLook;
        if (ws && h->nchunks > (size_t)g0 * cvs::kThreads) {
            if (piece_max >= 4 && !h->force_ws)
                nbands = (int)((h->nchunks + (size_t)g0 * cvs::kThreads - 1) / ((size_t)g0 * cvs::kThreads));
            else if (!h->force_ws)
                ws = false; // k_stream (segments, reference through L2)
        }
    }
    const size_t band_chunks_total = (h->nchunks + nbands - 1) / nbands; // chunks per band before rounding to the grid
    const uint32_t geo_chunks = nbands > 1 ? (uint32_t)band_chunks_total : h->nchunks;
    int G = ws ? h->sms : cvs::kBlocksPerSM * h->sms;
    const int look_max = ws ? 32 * cvs::kWsLook : cvs::kLook * cvs::kThreads; // predecessors the look-back can read
    if (G > look_max) G = look_max;
    if ((uint32_t)G > geo_chunks) G = (int)geo_chunks;
    uint32_t nseg = (uint32_t)((geo_chunks + (size_t)G * cvs::kThreads - 1) / ((size_t)G * cvs::kThreads));
    uint32_t cps = (uint32_t)((geo_chunks + (size_t)G * nseg - 1) / ((size_t)G * nseg));
    const bool refreg = nseg == 1;
    if (nbands > 1 && !refreg) return fail(CVS_ERR_INTERNAL, "band geometry does not fit one pass");
    StreamKernel kern = ws ? pick_ws_kernel(kmode, h->hi, refreg) : pick_kernel(kmode, h->hi, refreg);
    const int block_threads = ws ? cvs::kWsThreads : cvs::kThreads;
    // ring depth: all four stages when the reference lives in registers (measured +5 % at 1080p), three when it goes
    // through L2 (a deeper prefetch measured 17 % slower at 3840x2160 with k_stream); fewer if shared memory is short
    int nstages = refreg ? cvs::kStages : cvs::kStages - 1;
#ifdef CVS_PROFILING
    if (h->stages >= 2 && h->stages <= cvs::kStages) nstages = h->stages;
#endif
    int smem_max = 0;
    CU_TRY(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device));
    auto smem_need = [&](int ns) { return ws ? (int)cvs::WsLayout::total(cps, (uint32_t)ns) : cvs::SmemLayout::total(ns); };
    while (nstages > 2 && smem_need(nstages) > smem_max) nstages--;
    const int smem_bytes = smem_need(nstages);
    if (smem_bytes > smem_max) return fail(CVS_ERR_INTERNAL, "stream kernel needs %d bytes of shared memory, device has %d", smem_bytes, smem_max);
    int &occ = ws ? h->occ_ws[kmode][h->hi ? 1 : 0][refreg ? 1 : 0] : h->occ_cache[kmode][h->hi ? 1 : 0][refreg ? 1 : 0];
    if (occ == 0) { // first launch of this variant on this handle
        CU_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
        CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, block_threads, smem_bytes));
    }
    if (occ < 1) return fail(CVS_ERR_INTERNAL, "stream kernel does not fit on an SM");
    if (G > occ * h->sms) { // fewer co-resident blocks than planned: recompute
        G = occ * h->sms;
        nseg = (uint32_t)((geo_chunks + (size_t)G * cvs::kThreads - 1) / ((size_t)G * cvs::kThreads));
        cps = (uint32_t)((geo_chunks + (size_t)G * nseg - 1) / ((size_t)G * nseg));
        if ((nseg == 1) != refreg) return fail(CVS_ERR_INTERNAL, "occupancy changed the segment count");
    }
    if (nbands > 1 && h->band_frames < (size_t)piece_max) {
        if (h->d_band_pos) {
            CU_TRY(cudaDeviceSynchronize());
            cudaFree(h->d_band_pos);
            h->d_band_pos = nullptr;
            h->band_frames = 0;
        }
        CU_TRY(cudaMalloc(&h->d_band_pos, 2 * (size_t)piece_max * sizeof(unsigned int)));
        h->band_frames = (size_t)piece_max;
    }

    int done = 0;
    while (done < nframes) {
        int piece = nframes - done;
        if (piece > h->max_sequence) piece = h->max_sequence;
        const uint8_t *frames = d_frames + (size_t)done * stride;
        size_t fstride = stride;

        {
            cvs_status s = pre_pass(h, frames, fstride, piece, txt, frames_private, binarize, st);
            if (s) return s;
        }
        if (split_gray) { // gray byte + histogram of the frames as the diff will see them (filtered, overlay blitted)
            const size_t groups = ((size_t)h->N + cvs::kGroupBytes - 1) / cvs::kGroupBytes;
            dim3 grid(grid_for((groups + cvs::kGrayHistGroupsPerThread - 1) / cvs::kGrayHistGroupsPerThread, 256, h->sms), piece);
            if (mode == 5) cvs::k_gray_hist_seq<true><<<grid, 256, 0, st>>>(frames, fstride, h->N, h->d_gray1, h->P16, h->d_hist);
            else cvs::k_gray_hist_seq<false><<<grid, 256, 0, st>>>(frames, fstride, h->N, h->d_gray1, h->P16, h->d_hist);
            CU_TRY(cudaGetLastError());
            h->launches++;
        }

        cvs_status s = ensure_desc(h, (size_t)piece * nseg * (G + 1));
        if (s) return s;
        const size_t band_bytes = (size_t)G * cps * cvs::kChunkBytes; // bytes of a band (the last one may be shorter)
        for (int band = 0; band < nbands; band++) {
            const size_t boff = nbands > 1 ? (size_t)band * band_bytes : 0;
            if (boff >= h->N) break;
            const uint32_t bbytes = nbands > 1 ? (uint32_t)((h->N - boff) < band_bytes ? (h->N - boff) : band_bytes) : h->N;
            h->epoch++;
            if (h->epoch == 0) { // tag wrapped: stale descriptors could alias
                CU_TRY(cudaMemsetAsync(h->d_desc, 0, h->desc_words * sizeof(unsigned long long), st));
                h->epoch = 1;
            }
            const bool last_band = nbands == 1 || boff + band_bytes >= h->N;
            cvs::StreamParams p;
            p.frames = frames + boff;
            p.frame_stride = fstride;
            p.nframes = piece;
            p.ref = h->d_ref + boff;
            p.nbytes = bbytes;
            p.nbytes16 = nbands > 1 ? (uint32_t)round_up(bbytes, 16) : h->N16;
            p.nchunks = (bbytes + cvs::kChunkBytes - 1) / cvs::kChunkBytes;
            p.nseg = nseg;
            p.cps = cps;
            p.nstages = (uint32_t)nstages;
            p.pos = last_band ? d_pos + done : h->d_band_pos + (size_t)(band & 1) * h->band_frames;
            p.pos_prior = band ? h->d_band_pos + (size_t)((band - 1) & 1) * h->band_frames : nullptr;
            p.index_base = (uint32_t)boff;
            p.xs = d_xs + (size_t)done * cap;
            p.diff = d_diff + (size_t)done * cap;
            p.cap = cap;
            p.show = d_show ? d_show + (size_t)done * show_stride : nullptr;
            p.show_stride = show_stride;
            p.gray1 = binarize && !split_gray ? h->d_gray1 : nullptr;
            p.gray_stride = h->P16;
            p.hist = binarize && !split_gray ? h->d_hist : nullptr;
            p.heat_lut = h->d_lut;
            p.desc = h->d_desc;
            p.epoch = h->epoch;
            p.addc = h->addc;
            p.debug = h->debug;
            p.status = d_status;
            void *args[] = {&p};
            // The blocks only ever wait for blocks of LOWER index of the same step (look-back), never at a grid barrier, and
            // G <= the blocks the device can hold, so a plain launch cannot deadlock (blocks are dispatched in index
            // order); a cooperative launch additionally waits until the WHOLE grid fits at once.  Sequences keep that
            // (every block starts together: the timings of DESIGN 4.1); a single frame of the submit / exec path is
            // launched plain, so that its blocks start as SMs become free instead of draining the device first -- with
            // several camera streams on a GPU, whose decode kernels (cvs_jpeg.cuh) and payload pushes would otherwise
            // run strictly one after the other: 3 JPEG streams 3.8 k -> 7.1 k frames/s, raw streams unchanged.
            // (frames walked in several segments wait for the totals of ALL blocks of the previous segment: cooperative)
            if (piece > 1 || nseg > 1)
                CU_TRY(cudaLaunchCooperativeKernel((const void *)kern, dim3(G), dim3(block_threads), args, (size_t)smem_bytes, st));
            else
                CU_TRY(cudaLaunchKernel((const void *)kern, dim3(G), dim3(block_threads), args, (size_t)smem_bytes, st));
            h->launches++;
        }

        if (binarize) {
            cvs_status s = binarize_pass(h, piece, d_show + (size_t)done * show_stride, show_stride, st);
            if (s) return s;
        }
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
    const int G = std::min(std::min(h0->sms, 32 * cvs::kWsLook), (int)h0->nchunks);
    if (n == 1 || !h0->use_ws || h0->nchunks > (size_t)G * cvs::kThreads) {
        for (int i = 0; i < n; i++) {
            cvs_status s = run_frames(hs[i], frames[i], hs[i]->Npad, 1, pos[i], xs[i], diff[i], cap, show ? show[i] : nullptr,
                                      hs[i]->Npad, texts ? texts[i] : nullptr, st, frames_private, status[i]);
            if (s) return s;
        }
        return CVS_OK;
    }
    const int mode = h0->mode;
    const bool binarize = (mode == 5 || mode == 7) && show;
    const int kmode = show ? mode : 0;
    const uint32_t cps = (h0->nchunks + G - 1) / G;
    const BatchKernel kern = pick_batch_kernel(kmode, h0->hi);
    int smem_max = 0;
    CU_TRY(cudaDeviceGetAttribute(&smem_max, cudaDevAttrMaxSharedMemoryPerBlockOptin, h0->device));
    int nstages = cvs::kStages;
    while (nstages > 2 && (int)cvs::WsLayout::total(cps, (uint32_t)nstages) > smem_max) nstages--;
    const int smem_bytes = (int)cvs::WsLayout::total(cps, (uint32_t)nstages);
    if (smem_bytes > smem_max) return fail(CVS_ERR_INTERNAL, "stream kernel needs %d bytes of shared memory, device has %d", smem_bytes, smem_max);
    int &occ = h0->occ_batch[kmode][h0->hi ? 1 : 0];
    if (occ == 0) {
        CU_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
        CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, cvs::kWsThreads, smem_bytes));
    }
    if (occ < 1) return fail(CVS_ERR_INTERNAL, "stream kernel does not fit on an SM");

    cvs::BatchTable tbl; // (copied into the launch's parameters by cudaLaunchKernel)
    for (int i = 0; i < n; i++) {
        cvs_handle h = hs[i];
        const cvs::OverlayText txt = overlay_text(h, texts ? texts[i] : nullptr);
        if (h->noise_filter || (txt.n && !frames_private)) {
            cvs_status s = ensure_work(h, 1);
            if (s) return s;
        }
        if (binarize) {
            cvs_status s = ensure_bin(h, 1);
            if (s) return s;
        }
        const uint8_t *f = frames[i];
        size_t fstride = h->Npad;
        cvs_status s = pre_pass(h, f, fstride, 1, txt, frames_private, binarize, st);
        if (s) return s;
        tbl.cam[i] = {f, h->d_ref, pos[i], xs[i], diff[i], show ? show[i] : nullptr, binarize ? h->d_gray1 : nullptr,
                      binarize ? h->d_hist : nullptr, status[i]};
    }
    cvs_status s = ensure_desc(h0, (size_t)n * (G + 1));
    if (s) return s;
    h0->epoch++;
    if (h0->epoch == 0) { // tag wrapped: stale descriptors could alias
        CU_TRY(cudaMemsetAsync(h0->d_desc, 0, h0->desc_words * sizeof(unsigned long long), st));
        h0->epoch = 1;
    }
    cvs::StreamParams p;
    memset(&p, 0, sizeof p);
    p.nframes = n;
    p.nbytes = h0->N;
    p.nbytes16 = h0->N16;
    p.nchunks = h0->nchunks;
    p.nseg = 1;
    p.cps = cps;
    p.nstages = (uint32_t)nstages;
    p.cap = cap;
    p.heat_lut = h0->d_lut;
    p.desc = h0->d_desc;
    p.epoch = h0->epoch;
    p.addc = h0->addc;
    p.debug = h0->debug;
    p.status = status[0];
    void *args[] = {&p, &tbl};
    // plain launch, as for the single frames it replaces: blocks only wait for blocks of lower index (look-back)
    CU_TRY(cudaLaunchKernel((const void *)kern, dim3(G), dim3(cvs::kWsThreads), args, (size_t)smem_bytes, st));
    h0->launches++;
    if (binarize)
        for (int i = 0; i < n; i++) {
            s = binarize_pass(hs[i], 1, show[i], hs[i]->Npad, st);
            if (s) return s;
        }
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
#ifdef CVS_PROFILING
    // timing experiments only (results are wrong by construction): compiled into profiling builds, never into the
    // library a server links -- a stray environment variable must not be able to corrupt a stream
    if (const char *dbg = getenv("CVS_DEBUG_FLAGS")) h->debug = (uint32_t)atoi(dbg);
    if (const char *sg = getenv("CVS_STAGES")) h->stages = atoi(sg);
#endif
    // both stream kernels are bit-exact; the tests use this to run each kernel on geometries the default does not give it
    if (const char *kk = getenv("CVS_STREAM_KERNEL")) {
        h->use_ws = strcmp(kk, "v1") != 0;
        h->force_ws = strcmp(kk, "ws") == 0;
    }
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
    CU_TRY(cudaMalloc(&h->d_ref, h->Npad + 64));
    CU_TRY(cudaMemset(h->d_ref, 0, h->Npad + 64));
    CU_TRY(cudaMemcpy(h->d_ref, cfg->base_frame, h->N, cudaMemcpyHostToDevice)); // kernels.cu:406
    {
        uint32_t lut[768];
        build_heat_lut(lut);
        CU_TRY(cudaMalloc(&h->d_lut, sizeof lut));
        CU_TRY(cudaMemcpy(h->d_lut, lut, sizeof lut, cudaMemcpyHostToDevice));
    }
    CU_TRY(cudaMalloc(&h->d_status, sizeof(unsigned int)));
    CU_TRY(cudaMemset(h->d_status, 0, sizeof(unsigned int)));
    CU_TRY(cudaHostAlloc(&h->h_status, sizeof(unsigned int), cudaHostAllocDefault));
    *h->h_status = 0;
    if (cfg->glyphs && cfg->glyph_w > 0 && cfg->glyph_h > 0 && cfg->glyph_chars) {
        h->glyph_chars = cfg->glyph_chars;
        h->glyph_w = cfg->glyph_w;
        h->glyph_h = cfg->glyph_h;
        size_t bytes = h->glyph_chars.size() * 3 * (size_t)cfg->glyph_w * cfg->glyph_h;
        CU_TRY(cudaMalloc(&h->d_glyphs, bytes + 16));
        CU_TRY(cudaMemcpy(h->d_glyphs, cfg->glyphs, bytes, cudaMemcpyHostToDevice));
    }
    const size_t cap = round_up(h->N, 4);
    for (Slot &s : h->slot) {
        CU_TRY(cudaMalloc(&s.d_in, h->Npad + 64));
        CU_TRY(cudaMemset(s.d_in, 0, h->Npad + 64));
        CU_TRY(cudaMalloc(&s.d_xs, cap * sizeof(int)));
        CU_TRY(cudaMalloc(&s.d_diff, cap));
        CU_TRY(cudaMalloc(&s.d_pos, sizeof(unsigned int)));
        if (h->mode) CU_TRY(cudaMalloc(&s.d_show, h->Npad + 64));
        CU_TRY(cudaHostAlloc(&s.h_pos, sizeof(unsigned int), cudaHostAllocDefault));
        CU_TRY(cudaMalloc(&s.d_status, sizeof(unsigned int)));
        CU_TRY(cudaMemset(s.d_status, 0, sizeof(unsigned int)));
        CU_TRY(cudaHostAlloc(&s.h_status, sizeof(unsigned int), cudaHostAllocDefault));
        *s.h_status = 0;
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
        cudaFree(s.d_in); cudaFree(s.d_xs); cudaFree(s.d_diff); cudaFree(s.d_pos); cudaFree(s.d_show);
        cudaFreeHost(s.h_pos);
        cudaFree(s.d_status);
        cudaFreeHost(s.h_status);
        cudaFree(s.d_starts);
        cudaFree(s.d_wire);
        if (s.jpeg_state && g_nvjpeg.ok) g_nvjpeg.StateDestroy(s.jpeg_state);
        cudaEvent_t evs[] = {s.ev_h2d0, s.ev_h2d1, s.ev_k0, s.ev_k1, s.ev_pos, s.ev_p0, s.ev_done};
        for (cudaEvent_t e : evs)
            if (e) cudaEventDestroy(e);
    }
    cudaFree(h->d_ref); cudaFree(h->d_lut); cudaFree(h->d_status); cudaFreeHost(h->h_status);
    cudaFree(h->d_band_pos);
    for (JpegDecoder &jd : h->jd) jd.release();
    for (cudaStream_t js : h->s_jpg)
        if (js) cudaStreamDestroy(js);
    if (h->jpeg_state && g_nvjpeg.ok) g_nvjpeg.StateDestroy(h->jpeg_state);
    if (h->jpeg && g_nvjpeg.ok) g_nvjpeg.Destroy(h->jpeg);
    cudaFree(h->d_desc); cudaFree(h->d_work); cudaFree(h->d_gray1); cudaFree(h->d_hist); cudaFree(h->d_thr);
    cudaFree(h->d_glyphs);
    if (h->s_comp) cudaStreamDestroy(h->s_comp);
    if (h->s_h2d) cudaStreamDestroy(h->s_h2d);
    if (h->s_d2h) cudaStreamDestroy(h->s_d2h);
    if (h->s_pay) cudaStreamDestroy(h->s_pay);
    delete h;
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

    // ---- scratch: one arena, carved; the part every decode needs zeroed (round counters, entry states, the unstuffed
    //      string's padding, the coefficients) sits in front so that one memset clears it
    const size_t raw_pad = round_up(P.scan_bytes, 4096) + 4096;
    const size_t luma_bytes = (size_t)g.mcux * 8 * g.H * g.mcuy * 8 * g.V, chroma_bytes = (size_t)g.mcux * 8 * g.mcuy * 8;
    if (raw_pad > jd.raw_cap || g.nblocks > jd.block_cap) {
        const size_t raw_cap = std::max(jd.raw_cap, raw_pad + raw_pad / 2), block_cap = std::max<size_t>(jd.block_cap, g.nblocks);
        CU_TRY(cudaStreamSynchronize(st));
        cudaFree(jd.d_arena);
        jd.d_arena = nullptr;
        jd.raw_cap = jd.block_cap = jd.sub_cap = 0;
        const size_t nsub_cap = (raw_cap * 8 + jd.sub_bits - 1) / jd.sub_bits + 1;
        const size_t nhalf_cap = 2 * nsub_cap, ntile_cap = nhalf_cap / J::kEntropyThreads + 2; // the rounds may work on half subsequences
        size_t off = 0;
        auto carve = [&](size_t bytes) {
            const size_t o = off;
            off += round_up(bytes, 256);
            return o;
        };
        const size_t o_changed = carve(J::kRoundCounters * sizeof(unsigned int)), o_entry = carve((nhalf_cap + 2) * sizeof(uint32_t)),
                     o_unst = carve(raw_cap), o_coef = carve(block_cap * 64 * sizeof(int16_t));
        jd.zero_bytes_fixed = o_coef; // + nblocks * 128 of the coefficients
        const size_t o_raw = carve(raw_cap), o_kept = carve((raw_cap / (J::kUnstuffThreads * J::kUnstuffBytes) + 1) * sizeof(uint32_t)),
                     o_marks = carve((raw_cap / (J::kUnstuffThreads * J::kUnstuffBytes) + 1) * sizeof(uint32_t)),
                     o_seg = carve((block_cap + 2) * sizeof(uint32_t)), o_total = carve(2 * sizeof(uint32_t)), o_tables = carve(sizeof(J::Tables)), o_used = carve(nhalf_cap * sizeof(uint32_t)),
                     o_nblk = carve(nhalf_cap * sizeof(uint32_t)), o_dcs = carve(3 * nhalf_cap * sizeof(int32_t)),
                     o_tile_blk = carve(ntile_cap * sizeof(uint32_t)), o_tile_dc = carve(3 * ntile_cap * sizeof(int32_t)),
                     o_hx = carve(6 * nsub_cap * sizeof(uint32_t)), o_hy = carve(6 * nsub_cap * sizeof(uint32_t)),
                     o_hw = carve(6 * nsub_cap * sizeof(uint32_t)), o_hym = carve(6 * nsub_cap * sizeof(uint32_t)),
                     o_hwm = carve(6 * nsub_cap * sizeof(uint32_t)),
                     o_hmap = carve(16 * nsub_cap), o_mid_state = carve(J::kMaxSplit * nsub_cap * sizeof(uint32_t)),
                     o_mid_nblk = carve(J::kMaxSplit * nsub_cap * sizeof(uint32_t)),
                     o_mid_dc = carve(3 * J::kMaxSplit * nsub_cap * sizeof(int32_t)), o_planes = carve(block_cap * 64 + 256);
        CU_TRY(cudaMalloc(&jd.d_arena, off));
        uint8_t *a = jd.d_arena;
        jd.d_changed = reinterpret_cast<unsigned int *>(a + o_changed);
        jd.d_entry = reinterpret_cast<uint32_t *>(a + o_entry);
        jd.d_unst = a + o_unst;
        jd.d_coef = reinterpret_cast<int16_t *>(a + o_coef);
        jd.d_raw = a + o_raw;
        jd.d_block_kept = reinterpret_cast<uint32_t *>(a + o_kept);
        jd.d_block_marks = reinterpret_cast<uint32_t *>(a + o_marks);
        jd.d_seg_start = reinterpret_cast<uint32_t *>(a + o_seg);
        jd.seg_cap = (uint32_t)block_cap + 2;
        jd.d_total_bits = reinterpret_cast<uint32_t *>(a + o_total);
        jd.d_total_marks = jd.d_total_bits + 1;
        jd.d_tables = reinterpret_cast<J::Tables *>(a + o_tables);
        jd.d_used = reinterpret_cast<uint32_t *>(a + o_used);
        jd.d_nblk = reinterpret_cast<uint32_t *>(a + o_nblk);
        jd.d_dcs = reinterpret_cast<int32_t *>(a + o_dcs);
        jd.d_tile_blk = reinterpret_cast<uint32_t *>(a + o_tile_blk);
        jd.d_tile_dc = reinterpret_cast<int32_t *>(a + o_tile_dc);
        jd.d_hx = reinterpret_cast<uint32_t *>(a + o_hx);
        jd.d_hy = reinterpret_cast<uint32_t *>(a + o_hy);
        jd.d_hw = reinterpret_cast<uint32_t *>(a + o_hw);
        jd.d_hym = reinterpret_cast<uint32_t *>(a + o_hym);
        jd.d_hwm = reinterpret_cast<uint32_t *>(a + o_hwm);
        jd.d_hmap = a + o_hmap;
        jd.d_mid_state = reinterpret_cast<uint32_t *>(a + o_mid_state);
        jd.d_mid_nblk = reinterpret_cast<uint32_t *>(a + o_mid_nblk);
        jd.d_mid_dc = reinterpret_cast<int32_t *>(a + o_mid_dc);
        jd.d_planes = a + o_planes;
        jd.raw_cap = raw_cap;
        jd.block_cap = block_cap;
        jd.sub_cap = nsub_cap;
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
        CU_TRY(cudaMemsetAsync(jd.d_arena, 0, jd.zero_bytes_fixed + (size_t)g.nblocks * 64 * sizeof(int16_t), st));
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
static cvs_status jpeg_decode(cvs_handle h, int set, nvjpegJpegState_t *state, const uint8_t *jpeg, size_t jpeg_bytes,
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
        s.pushed = mapped_device_pointer(wire_out, &dev_wire) && ((uintptr_t)dev_wire % 16 == 0);
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
        s.pushed = mapped_device_pointer(diff_out, &dev_diff) && mapped_device_pointer(xs, &dev_xs) &&
                   ((uintptr_t)dev_diff % 16 == 0) && ((uintptr_t)dev_xs % 16 == 0);
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

static cvs_status submit_common(cvs_handle h, const uint8_t *frame, uint8_t *diff_out, uint8_t *show, const char *text,
                                unsigned int *pos, int *xs, uint8_t *wire_out, uint64_t *ticket, size_t jpeg_bytes = 0)
{
    cvs_status st = check_handle(h);
    if (st) return st;
    if (!frame || !ticket || (!wire_out && (!diff_out || !pos || !xs))) return fail(CVS_ERR_INVALID, "null argument");
    Slot &s = h->slot[h->next_ticket % kSlots];
    if (s.busy) return fail(CVS_ERR_INVALID, "%d tickets are already outstanding; cvs_wait the oldest first", kSlots);
    const uint32_t ntiles = (h->N + cvs::kWireTile - 1) / cvs::kWireTile;
    if (wire_out && !s.d_starts) {
        CU_TRY(cudaMalloc(&s.d_starts, (size_t)(ntiles + 2) * sizeof(uint32_t)));
        CU_TRY(cudaMalloc(&s.d_wire, cvs_wire_bound(h->width, h->height)));
    }

    const double th0 = h->trace ? host_us() : 0;
    // H2D (kernels.cu:461) -- of the raw frame, or of the camera's JPEG bitstream, decoded on the device.  JPEG tickets
    // alternate between two decode streams with their own scratch: frame t+1 is decoded beside frame t (a decode is a
    // latency chain that leaves most of the GPU idle); the stream kernel below still takes the frames in ticket order.
    cudaStream_t s_in = h->s_h2d;
    const int jset = (int)(h->next_ticket & 1);
    if (jpeg_bytes) {
        if (!h->s_jpg[jset]) CU_TRY(cudaStreamCreateWithFlags(&h->s_jpg[jset], cudaStreamNonBlocking));
        s_in = h->s_jpg[jset];
    }
    CU_TRY(cudaEventRecord(s.ev_h2d0, s_in));
    if (jpeg_bytes) {
        // (the ticket's status word is cleared here, in front of the decoder that may raise bits in it)
        CU_TRY(cudaMemsetAsync(s.d_status, 0, sizeof(unsigned int), s_in));
        st = jpeg_decode(h, jset, &s.jpeg_state, frame, jpeg_bytes, s.d_in, s_in, s.d_status);
        if (st) return st;
    } else {
        CU_TRY(cudaMemcpyAsync(s.d_in, frame, h->N, cudaMemcpyHostToDevice, h->s_h2d));
    }
    CU_TRY(cudaEventRecord(s.ev_h2d1, s_in));
    // kernels
    CU_TRY(cudaStreamWaitEvent(h->s_comp, s.ev_h2d1, 0));
    CU_TRY(cudaEventRecord(s.ev_k0, h->s_comp));
    const size_t cap = round_up(h->N, 4);
    uint8_t *dshow = (h->mode && show) ? s.d_show : nullptr;
    const double th1 = h->trace ? host_us() : 0;
    if (!jpeg_bytes) CU_TRY(cudaMemsetAsync(s.d_status, 0, sizeof(unsigned int), h->s_comp));
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
        CU_TRY(cudaEventRecord(s.ev_h2d0, h->s_h2d));
        CU_TRY(cudaMemcpyAsync(s.d_in, frames[i], h->N, cudaMemcpyHostToDevice, h->s_h2d));
        CU_TRY(cudaEventRecord(s.ev_h2d1, h->s_h2d));
        CU_TRY(cudaStreamWaitEvent(h->s_comp, s.ev_h2d1, 0));
        CU_TRY(cudaEventRecord(s.ev_k0, h->s_comp));
        CU_TRY(cudaStreamWaitEvent(L->s_comp, s.ev_k0, 0));
        d_frames[i] = s.d_in;
        d_pos[i] = s.d_pos;
        d_xs[i] = s.d_xs;
        d_diff[i] = s.d_diff;
        d_show[i] = any_show ? s.d_show : nullptr; // (a camera without a show buffer still gets its frame: not copied out)
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
        st = egress(h, s, frames[i], diff_out[i], sh, sh && any_show ? s.d_show : nullptr, pos[i], xs[i], nullptr);
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
    st = jpeg_decode(h, 2, &h->jpeg_state, jpeg, jpeg_bytes, d_out, (cudaStream_t)cuda_stream, h->d_status);
    if (st) return st;
    CU_TRY(cudaMemcpyAsync(h->h_status, h->d_status, sizeof(unsigned int), cudaMemcpyDeviceToHost, (cudaStream_t)cuda_stream));
    return CVS_OK;
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
    if (((uintptr_t)d_frames & 15) || (frame_stride & 15) || ((uintptr_t)d_xs & 15) || ((uintptr_t)d_diff & 15) ||
        (d_show && (((uintptr_t)d_show & 15) || (show_stride & 15))))
        return fail(CVS_ERR_ALIGN, "device pointers and strides must be 16-byte aligned");
    if (frame_stride < h->N16) return fail(CVS_ERR_INVALID, "frame_stride %zu < %u", frame_stride, h->N16);
    if (d_show && show_stride < h->N) return fail(CVS_ERR_INVALID, "show_stride too small");
    if (payload_capacity == 0 || (payload_capacity & 3))
        return fail(CVS_ERR_INVALID, "payload_capacity must be a positive multiple of 4");
    h->seq_status = CVS_OK;
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
    for (int i = 0; i < n; i++)
        if ((uintptr_t)d_frames[i] & 15) return fail(CVS_ERR_ALIGN, "device pointers and strides must be 16-byte aligned");
    if (((uintptr_t)d_xs & 15) || ((uintptr_t)d_diff & 15) || (d_show && (((uintptr_t)d_show & 15) || (show_stride & 15))))
        return fail(CVS_ERR_ALIGN, "device pointers and strides must be 16-byte aligned");
    if (d_show && show_stride < hs[0]->N) return fail(CVS_ERR_INVALID, "show_stride too small");
    if (payload_capacity == 0 || (payload_capacity & 3))
        return fail(CVS_ERR_INVALID, "payload_capacity must be a positive multiple of 4");
    unsigned int *pos[CVS_MAX_BATCH], *status[CVS_MAX_BATCH];
    int *xs[CVS_MAX_BATCH];
    uint8_t *diff[CVS_MAX_BATCH], *show[CVS_MAX_BATCH];
    for (int i = 0; i < n; i++) {
        hs[i]->seq_status = CVS_OK;
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
    if (((uintptr_t)d_prev | (uintptr_t)d_cur | (uintptr_t)d_out) & 15) return fail(CVS_ERR_ALIGN, "16-byte alignment required");
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
    if (((uintptr_t)d_prev | (uintptr_t)d_cur | (uintptr_t)d_out) & 15) return fail(CVS_ERR_ALIGN, "16-byte alignment required");
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
    if (((uintptr_t)d_frame | (uintptr_t)d_out) & 15) return fail(CVS_ERR_ALIGN, "16-byte alignment required");
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
    if (((uintptr_t)d_frame | (uintptr_t)d_out | (uintptr_t)d_gray) & 15)
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
    if (((uintptr_t)d_xs | (uintptr_t)d_diff | (uintptr_t)d_wire) & 15) return fail(CVS_ERR_ALIGN, "16-byte alignment required");
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
    if ((uintptr_t)d_wire & 15) return fail(CVS_ERR_ALIGN, "16-byte alignment required");
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
