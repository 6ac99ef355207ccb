/*
 * cvs_b200.h -- C ABI of libcvs_b200.so: the B200-native (sm_100a) replacement for the per-pixel
 * hot path of MatteoBattilana/CUDAVideoStream's server.
 *
 * The reference exposes this path as the C++ class diff::cuda::CUDACore
 * (server/include/kernels.cuh:13-43; implementation server/src/kernels.cu:377-536).  Its four
 * public members are re-implemented, with unchanged signatures, by include/cvs_cuda_core.hpp +
 * cudavideostream_b200/csrc/cvs_shim.cu, which are thin calls into the functions declared here.
 * Every entry point below names the reference interface it replaces.  Plain pointers and sizes
 * only; no CUDA, torch or OpenCV types appear in any signature (a cudaStream_t is passed as void*).
 *
 * Error convention: every function returns a cvs_status; cvs_last_error() gives a message for the
 * calling thread.  (The reference prints and exit()s inside CUDA_CHECK, kernels.cu:11-22; the C++
 * shim converts a non-zero status into exactly that behaviour.)
 *
 * Pixel layout everywhere: packed row-major BGR24 ("RGB24" in OpenCV byte order), no row padding,
 * N = 3*width*height bytes per frame.
 *
 * Which of the reference's two implementations is the contract: the CPU loops (SURVEY.md section 8, A1-A10).  Where
 * the reference's CUDA kernels compute something else, this library follows the CPU loop, and a server that switches
 * from kernels.cu to this library sees the CPU result:
 *   - weighted gray (modes 4, 5): double products, left-to-right double adds, truncation
 *     (tests/grayscale-weighted/cpu.cu:38-42); kernels.cu:67-95 accumulates the same products in a float;
 *   - binarisation threshold (modes 5, 7): the CPU "two max" loop with its quirk (server.cpp:108-127: the previous
 *     running arg-max, clamp [50,200]); kernels.cu:176-206 compute_max takes the arg-max of the even and of the odd bins;
 *   - noise filter: float accumulator -> (uint8_t) as x86-64 converts it (cvttss2si, low byte: out-of-range values
 *     wrap modulo 256 while the accumulator is inside [-2^31, 2^31); NaN, infinities and anything outside give 0);
 *     CUDA's float-to-u8 conversion in kernels.cu:134 saturates.  With the reference's non-negative,
 *     normalised weights the accumulator never leaves [0, 255] and both agree.
 *
 * Threading: a cvs_handle is NOT thread-safe -- one host thread at a time may call into a given handle (the reference
 * calls exec_core from its main thread only, server.cpp:139).  Different handles may be used from different threads
 * concurrently.  Tickets of one handle complete in submission order and must be waited for in that order.
 */
#ifndef CVS_B200_H_
#define CVS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

#define CVS_ABI_VERSION 1

typedef enum cvs_status {
    CVS_OK = 0,
    CVS_ERR_INVALID = 1,   /* bad argument                                                    */
    CVS_ERR_CUDA = 2,      /* a CUDA runtime call failed (message in cvs_last_error)          */
    CVS_ERR_NOMEM = 3,
    CVS_ERR_ALIGN = 4,     /* device pointer / stride not 16-byte aligned                     */
    CVS_ERR_CAPACITY = 5,  /* payload_capacity too small for a frame of the sequence          */
    CVS_ERR_NODEVICE = 6,  /* no sm_100 device: there is no CPU fallback                      */
    CVS_ERR_INTERNAL = 7   /* device-side watchdog tripped (look-back did not resolve)        */
} cvs_status;

/* NOISE_VISUALIZER values of server/include/common.h:9-10, plus two extensions (6, 7) that expose
 * the average-grayscale variants of server/src/server.cpp:96-135. */
typedef enum cvs_mode {
    CVS_MODE_NONE = 0,
    CVS_MODE_HEAT_MAP = 1,          /* kernels.cu:243-270 / tests/heat_map_benchmark/cpu.cu        */
    CVS_MODE_RED_BLACK = 2,         /* kernels.cu:273-281 on a zeroed frame (kernels.cu:513-515)   */
    CVS_MODE_RED_OVERLAP = 3,       /* kernels.cu:517 on the previous reference frame              */
    CVS_MODE_GRAY_WEIGHTED = 4,     /* kernels.cu:67-95 / tests/grayscale-weighted/cpu.cu:38-42    */
    CVS_MODE_BINARIZE = 5,          /* kernels.cu:493-499: weighted gray, hist, two-max, binarize  */
    CVS_MODE_GRAY_AVERAGE = 6,      /* server.cpp:96-101                                           */
    CVS_MODE_BINARIZE_AVERAGE = 7   /* server.cpp:96-135 (the CPU branch, average gray)            */
} cvs_mode;

/* Runtime form of the compile-time switches in server/include/common.h:4-18 plus the constructor
 * arguments of CUDACore (kernels.cuh:38).  Fill with cvs_config_default() first. */
typedef struct cvs_config {
    int width;                 /* frameSz.width                                               */
    int height;                /* frameSz.height                                              */
    int threshold;             /* LR_THRESHOLDS (common.h:14), default 20; changed <=> |df| > threshold */
    int mode;                  /* cvs_mode                                                    */
    int noise_filter;          /* NOISE_FILTER (common.h:5): 1 = K x K convolution before the diff */
    int ksize;                 /* K (common.h:6): odd, 1..9                                   */
    const float *kweights;     /* ksize*ksize weights, row major (CUDACore ctor `k`)          */
    int device;                /* CUDA device ordinal (the reference hard-codes 0)            */
    const uint8_t *base_frame; /* first reference frame, N bytes, host (sampleMatData)        */
    const uint8_t *glyphs;     /* glyph atlas charsPx: nglyphs x (glyph_h x glyph_w x 3) bytes, or NULL */
    int glyph_w, glyph_h;      /* charsSz                                                     */
    const char *glyph_chars;   /* CHARS_STR (common.h:13): character of glyph i              */
    int max_sequence;          /* largest nframes a cvs_run_sequence_device call will use (default 512) */
} cvs_config;

typedef struct cvs_stream_s *cvs_handle; /* one camera stream = one reference-frame state */

const char *cvs_last_error(void);
int cvs_abi_version(void);
/* number of visible sm_100 devices (0 => nothing in this library can run) */
int cvs_device_count(void);

void cvs_config_default(cvs_config *cfg);

/* replaces CUDACore::CUDACore (kernels.cu:377-428): allocates device state, uploads base frame */
cvs_status cvs_create(const cvs_config *cfg, cvs_handle *out);
cvs_status cvs_destroy(cvs_handle h);
/* re-seed the reference frame (the reference has no resync, SURVEY.md section 5) */
cvs_status cvs_reset(cvs_handle h, const uint8_t *base_frame);

/* replaces CUDACore::alloc_arrays (kernels.cu:531-536): pinned host memory */
cvs_status cvs_alloc_host(void **ptr, size_t bytes);
cvs_status cvs_free_host(void *ptr);

/* replaces CUDACore::exec_core (kernels.cu:430-525), synchronous.
 *   frame : in  N-byte frame (pinned or pageable host memory)
 *           out frame[0..*pos) = diff bytes (df & 0xFF), rest untouched   (kernels.cu:522)
 *   show  : out N-byte visualisation frame when mode != 0 (may be NULL)   (showReadyNData)
 *   text  : overlay string over glyph_chars, may be NULL/empty            (kernels.cu:466-476)
 *   pos   : out number of changed bytes                                   (kernels.cu:507)
 *   xs    : out xs[0..*pos) ascending byte indices, capacity N ints       (kernels.cu:523)
 */
cvs_status cvs_exec(cvs_handle h, uint8_t *frame, uint8_t *show, const char *text,
                    unsigned int *pos, int *xs);

/* Pipelined form of the same call: cvs_submit enqueues H2D + kernels + D2H on the stream's
 * double-buffered slots and returns a ticket; cvs_wait blocks until that frame's outputs are on
 * the host.  At most 4 tickets may be outstanding; they complete in submission order.  Host buffers must be pinned (cvs_alloc_host)
 * for the copies to overlap. */
cvs_status cvs_submit(cvs_handle h, uint8_t *frame, uint8_t *show, const char *text,
                      unsigned int *pos, int *xs, uint64_t *ticket);
cvs_status cvs_wait(cvs_handle h, uint64_t ticket);
/* cvs_submit with the payload bytes written to a separate buffer instead of over the head of the input
 * frame (which is then left untouched): for callers that keep captured frames in a pinned ring.
 * diff_out (capacity N bytes) and xs (capacity N ints) hold the payload in [0, *pos); what lies past *pos is
 * unspecified on this entry point: the copy engine fetches a predicted number of entries right behind the
 * count instead of waiting for the host to read it. */
cvs_status cvs_submit_io(cvs_handle h, const uint8_t *frame, uint8_t *diff_out, uint8_t *show,
                         const char *text, unsigned int *pos, int *xs, uint64_t *ticket);

/* device times of the most recent completed cvs_exec / cvs_wait, microseconds (CUDA events):
 * host-to-device copy, kernels, device-to-host copies -- reported separately, as the
 * reference's report does (REPORT/report.tex:922-926). */
cvs_status cvs_get_timing(cvs_handle h, float *h2d_us, float *kernel_us, float *d2h_us);

/* copy the current reference frame (client-reconstructed image) to host memory, N bytes */
cvs_status cvs_get_reference(cvs_handle h, uint8_t *out);
/* device pointer of the reference frame (16-byte aligned, N bytes valid) */
cvs_status cvs_reference_device(cvs_handle h, void **dptr);

/* Device-resident sequence: the whole hot path over `nframes` consecutive frames that are already
 * in device memory, one persistent launch, asynchronous on `cuda_stream` (a cudaStream_t, NULL =
 * default stream).  This is the path bench.py times for `value` (inputs resident in HBM).
 *   d_frames        frame t at d_frames + t*frame_stride; base and stride 16-byte aligned,
 *                   stride >= N rounded up to 16
 *   d_pos           [nframes] changed-byte count per frame
 *   d_xs, d_diff    frame t's payload at d_xs + t*payload_capacity (ints) and
 *                   d_diff + t*payload_capacity (bytes); payload_capacity entries per frame.
 *                   Entries beyond the capacity are dropped and the call's completion status
 *                   (cvs_sequence_status) reports CVS_ERR_CAPACITY; d_pos still holds the true count.
 *   d_show          NULL, or frame t's visualisation at d_show + t*show_stride (mode != 0)
 * Noise filter and text overlay are applied per frame exactly as in cvs_exec (text fixed for the call).
 */
cvs_status cvs_run_sequence_device(cvs_handle h, const uint8_t *d_frames, size_t frame_stride,
                                   int nframes, unsigned int *d_pos, int *d_xs, uint8_t *d_diff,
                                   size_t payload_capacity, uint8_t *d_show, size_t show_stride,
                                   const char *text, void *cuda_stream);
/* after the stream has been synchronised: status word the last sequence launch left behind */
cvs_status cvs_sequence_status(cvs_handle h);
/* how many kernels of this library the handle has launched so far (bench.py's gpu_launches).  A batch's stream-kernel
 * launch counts once, on hs[0]; its per-camera pre- and post-passes count on their own handles. */
uint64_t cvs_launch_count(cvs_handle h);

/* ---------------------------------------------------------------------------------------------------------------
 * Batches: one frame of each of n camera streams (n handles) in ONE stream-kernel launch.  A single frame costs a
 * fixed launch-and-drain time on top of its pass (DESIGN.md section 9); a server with many cameras on one GPU pays it
 * once per batch instead of once per camera.
 *   - hs[0..n): 1 <= n <= CVS_MAX_BATCH distinct handles that share device, width, height, mode and threshold.  Noise
 *     filter and weights, glyph atlas, overlay text and max_sequence may differ.
 *   - Every output is bit for bit what n separate calls produce, in any order of the handles: payload, counts,
 *     display frames, and each handle's reference afterwards.
 *   - A refused batch (CVS_ERR_INVALID: n out of range, a NULL array or entry, a repeated handle, handles that differ
 *     in device, size, mode or threshold; CVS_ERR_ALIGN as cvs_run_sequence_device) has enqueued nothing.
 *   - Frames that do not fit one pass of the stream kernel (3840x2160 on a B200) run handle by handle through the
 *     single-frame path: same results, n stream-kernel launches (cvs_launch_count shows them).  So does a batch of one,
 *     which is faster there (the single-frame launch keeps the reference in registers).
 *   - Noise filter, text overlay and the binarisation's second pass (modes 5, 7) stay per camera, in front of and
 *     behind the one launch.
 * --------------------------------------------------------------------------------------------------------------- */
#define CVS_MAX_BATCH 64
/* one frame of each of n streams, device-resident (d_frames[i]: 16-byte aligned, N bytes, readable up to N rounded up to
 * 16), asynchronous on cuda_stream.  Outputs are laid out like a sequence indexed by camera: d_pos[i],
 * d_xs + i*payload_capacity, d_diff + i*payload_capacity, d_show + i*show_stride (d_show may be NULL).  texts may be
 * NULL or hold n entries (a NULL entry: no overlay).  Completion: cvs_sequence_status(hs[i]) after the stream has been
 * synchronised; a capacity overflow of camera i is reported by hs[i] alone. */
cvs_status cvs_run_batch_device(const cvs_handle *hs, int n, const uint8_t *const *d_frames,
                                unsigned int *d_pos, int *d_xs, uint8_t *d_diff, size_t payload_capacity,
                                uint8_t *d_show, size_t show_stride, const char *const *texts, void *cuda_stream);
/* cvs_submit_io for one frame of each of n streams: tickets[i] belongs to hs[i] and is completed with
 * cvs_wait(hs[i], tickets[i]); tickets of a handle still complete in submission order, batched or not.  show and texts
 * may be NULL or hold n entries (NULL entries allowed).  Each frame is uploaded on its own handle's copy stream; the
 * launch runs on hs[0]'s compute stream behind every handle's earlier tickets, and every handle's later tickets run
 * behind it.  A handle with 4 outstanding tickets refuses the whole batch (nothing is enqueued for any camera). */
cvs_status cvs_submit_io_batch(const cvs_handle *hs, int n, const uint8_t *const *frames, uint8_t *const *diff_out,
                               uint8_t *const *show, const char *const *texts, unsigned int *const *pos,
                               int *const *xs, uint64_t *tickets);

/* Stand-alone filters on device buffers (config 4 of BASELINE.json and the micro-benchmarks of
 * tests/heat_map_benchmark, tests/heat_map_red_benchmark, tests/grayscale-*, tests/binarization,
 * tests/noise_filter_benchmark).  All pointers are device pointers, 16-byte aligned; asynchronous
 * on `cuda_stream`.  `device` selects the GPU.                                                  */
cvs_status cvs_heat_map_device(const uint8_t *d_prev, const uint8_t *d_cur, uint8_t *d_out,
                               int width, int height, void *cuda_stream);
cvs_status cvs_red_map_device(const uint8_t *d_prev, const uint8_t *d_cur, uint8_t *d_out,
                              int width, int height, int threshold, void *cuda_stream);
/* weighted != 0: 0.114 B + 0.587 G + 0.299 R (double, truncated); else (B+G+R)/3.
 * channels = 1 (P bytes out) or 3 (value replicated, N bytes out). */
cvs_status cvs_grayscale_device(const uint8_t *d_frame, uint8_t *d_out, int width, int height,
                                int weighted, int channels, void *cuda_stream);
/* gray (weighted or average) -> 256-bin histogram -> two-max threshold clamped to
 * [clamp_lo, clamp_hi] -> 3-channel 0/255 image  (server.cpp:96-135, tests/binarization/cpu.cu).
 * d_gray: width*height bytes (rounded up to 16) of scratch/out, the 1-channel gray image;
 * d_hist_thr: 257 ints of scratch/out (histogram[256], threshold). */
cvs_status cvs_binarize_device(const uint8_t *d_frame, uint8_t *d_out, uint8_t *d_gray, int *d_hist_thr,
                               int width, int height, int weighted, int clamp_lo, int clamp_hi,
                               void *cuda_stream);
/* K x K zero-padded convolution, fp32 FMA accumulation in row-major tap order, truncation */
cvs_status cvs_noise_filter_device(const uint8_t *d_frame, uint8_t *d_out, int width, int height,
                                   int ksize, const float *h_weights, void *cuda_stream);
/* client side of the wire format (client/opencv.cpp:64-66): frame[xs[i]] += diff[i] */
cvs_status cvs_client_apply_device(uint8_t *d_frame, const int *d_xs, const uint8_t *d_diff,
                                   const unsigned int *d_pos, size_t capacity, void *cuda_stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Opt-in compact wire format "CVW1" (SURVEY.md section 8f row 3).  The reference transmits, per frame, u32 pos,
 * i32 xs[pos], u8 diff[pos] (server/src/threads.cpp:229-231; read back by client/opencv.cpp:52-66): 5 bytes per
 * entry.  xs is ascending, so the index can travel as (tile, offset-in-tile) with tiles of CVS_WIRE_TILE bytes:
 *     u32 magic "CVW1", u32 pos, u32 ntiles, u32 tile      16-byte header (little endian)
 *     u8  count[ntiles]   padded to a multiple of 16       entries per tile (0..192)
 *     u8  off[pos]        padded to a multiple of 16       offset of entry i inside its tile
 *     u8  diff[pos]                                        value bytes, exactly the reference's
 * = 16 + N/192 + 2*pos bytes instead of 4 + 5*pos (1080p: 157 KB instead of 311 KB at 1 % density, 1.28 MB instead of
 * 3.11 MB at 10 %, 6.3 MB instead of 15.6 MB at 50 %).  The default everywhere stays the reference's format; a server
 * and a client have to opt in together.
 * --------------------------------------------------------------------------------------------------------------- */
#define CVS_WIRE_TILE 192
#define CVS_WIRE_MAGIC 0x31575643u
/* largest encoded frame for this geometry: size wire_out buffers with it */
size_t cvs_wire_bound(int width, int height);
/* total bytes of an encoded frame, read from its header (host memory); 0 if the header is not CVW1.  Computed in 64
 * bits from the sender's ntiles and pos, so it can be far larger than any real frame: a client refuses a frame whose
 * cvs_wire_size exceeds cvs_wire_bound(width, height) before it reads (or receives) the frame's body. */
size_t cvs_wire_size(const uint8_t *wire);
/* cvs_submit_io that delivers the frame's payload as one CVW1 frame in wire_out (capacity cvs_wire_bound; pinned
 * memory from cvs_alloc_host lets the device store it directly).  Complete it with cvs_wait(ticket); the count is
 * the header's pos field. */
cvs_status cvs_submit_wire(cvs_handle h, const uint8_t *frame, uint8_t *wire_out, uint8_t *show,
                           const char *text, uint64_t *ticket);
/* device-resident payload (as cvs_run_sequence_device leaves it for one frame) -> CVW1 frame in d_wire.
 * d_scratch: (ntiles + 2) 32-bit words, ntiles = ceil(3*width*height / CVS_WIRE_TILE). */
cvs_status cvs_wire_encode_device(const int *d_xs, const uint8_t *d_diff, const unsigned int *d_pos,
                                  size_t capacity, int width, int height, uint32_t *d_scratch,
                                  uint8_t *d_wire, void *cuda_stream);
/* client side: decodes one CVW1 frame that lies in device memory.  Any of the outputs may be NULL:
 *   d_frame : frame[x] += diff for every entry (client/opencv.cpp:64-66)
 *   d_xs, d_diff, d_pos : the reference-format payload back (ascending indices)
 * d_scratch as above.  d_wire holds at least cvs_wire_size bytes of the frame and at least 16 + ntiles rounded up to
 * 16 (what a cvs_wire_bound-sized buffer holds).  An inconsistent frame is not applied at all: no output is written,
 * and cvs_wire_decode_status (synchronises the stream) returns CVS_ERR_INVALID.  Inconsistent means any of
 *   - a magic other than CVW1, a tile other than CVS_WIRE_TILE, or ntiles other than this geometry's;
 *   - a tile count above the tile's length (192; the last tile holds N - 192 * (ntiles - 1) bytes);
 *   - counts that do not add up to pos (so pos <= N);
 *   - inside a tile, an offset at or past the tile's length, or offsets that are not strictly ascending.
 * The offsets are read only after the header and counts have passed, so never past cvs_wire_size bytes.  Pad bytes
 * after the counts and after the offsets are ignored. */
cvs_status cvs_wire_decode_device(const uint8_t *d_wire, uint32_t *d_scratch, uint8_t *d_frame, int *d_xs,
                                  uint8_t *d_diff, unsigned int *d_pos, int width, int height,
                                  void *cuda_stream);
cvs_status cvs_wire_decode_status(const uint32_t *d_scratch, int width, int height, void *cuda_stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Capture-side decode on the GPU (SURVEY.md section 8f row 4).  The reference's camera delivers MJPG and OpenCV
 * decodes it on the CPU before exec_core sees the frame (server/src/threads.cpp:32-41; "read 37 ms",
 * REPORT/report.tex:914).  cvs_submit_jpeg takes the camera's JPEG bitstream instead of the decoded frame: ~0.4 MB
 * cross PCIe instead of 6.2 MB (1080p), the library's own kernels (csrc/cvs_jpeg.cuh) decode it into the slot's
 * upload buffer and the rest of the path is unchanged.
 *   The decoder reproduces OpenCV's (libjpeg-turbo's default) arithmetic -- sequential-DCT Huffman decoding, the
 *   accurate integer IDCT (jidctint.c), "fancy" chroma upsampling with replicated border rows (jdsample.c /
 *   jdmainct.c), fixed-point YCbCr -> RGB (jdcolor.c) -- so the pixels are bit for bit the ones the reference's
 *   capture thread would have produced: on the reference's own f1.jpg / f2.jpg the payload is the reference's, K1 =
 *   369,350 (tests/test_jpeg_ingest.py; oracle: oracle/jpeg_oracle.c, pinned against cv2).
 *   Covered: baseline (SOF0/SOF1 Huffman, 8 bit), one interleaved scan, Y Cb Cr with luma sampling 1x1 / 2x1 / 2x2
 *   and chroma 1x1 (what UVC cameras and cv2.imwrite produce), or one gray component; with or without restart
 *   intervals (one thread per interval then); frames without a DHT segment use the standard tables (MJPG).
 *   Other forms (progressive, arithmetic coding, other samplings) go to nvJPEG (loaded with dlopen on first use), whose pixels
 *   are close to but not identical with libjpeg-turbo's (<= 5 apart on the fixture frames); CVS_JPEG_DECODER=own
 *   refuses them instead.
 *   A damaged entropy-coded segment never writes outside the frame; when the decoder notices (the stream holds
 *   fewer blocks than the image) cvs_wait / cvs_sequence_status return CVS_ERR_INVALID for that frame.  Every
 *   well-formed stream decodes, however unfriendly its code: the parallel decode falls back to as many rounds as it
 *   needs (a stream whose codes are all equally long does not self-synchronise and decodes at sequential speed).
 *   1080p camera frame (432 KB): 0.30 ms per decode on one stream, ~11,000 decodes/s with four streams of a GPU
 *   (nvJPEG on the same box: 205/s) -- profiles/README.md.
 * --------------------------------------------------------------------------------------------------------------- */
cvs_status cvs_submit_jpeg(cvs_handle h, const uint8_t *jpeg, size_t jpeg_bytes, uint8_t *diff_out, uint8_t *show,
                           const char *text, unsigned int *pos, int *xs, uint64_t *ticket);
/* both opt-ins together: the camera's JPEG bitstream in, one compact CVW1 frame (cvs_submit_wire) out -- the fewest
 * bytes across PCIe in either direction (1080p camera frame: 0.43 MB up, 16 + N/192 + 2*pos bytes down) */
cvs_status cvs_submit_jpeg_wire(cvs_handle h, const uint8_t *jpeg, size_t jpeg_bytes, uint8_t *wire_out, uint8_t *show,
                                const char *text, uint64_t *ticket);
/* the decode alone: baseline JPEG of the stream's frame size -> BGR24 frame in device memory (N bytes) */
cvs_status cvs_decode_jpeg_device(cvs_handle h, const uint8_t *jpeg, size_t jpeg_bytes, uint8_t *d_out,
                                  void *cuda_stream);

/* Synthetic camera used by bench.py and the parity tests (SURVEY.md section 8d): counter-based
 * splitmix64 so that the numpy twin in cudavideostream_b200/synth.py produces identical bytes.
 *   cvs_synth_base_device   : base frame (diagonal gradient + noise)
 *   cvs_synth_next_device   : frame t from frame t-1; each byte changes by +-U[21,80] with
 *                             probability density_ppm/1e6, otherwise drifts by U[-3,3]
 */
cvs_status cvs_synth_base_device(uint8_t *d_out, int width, int height, uint64_t seed,
                                 void *cuda_stream);
cvs_status cvs_synth_next_device(const uint8_t *d_prev, uint8_t *d_out, int width, int height,
                                 uint64_t seed, uint32_t frame_index, uint32_t density_ppm,
                                 void *cuda_stream);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* CVS_B200_H_ */
