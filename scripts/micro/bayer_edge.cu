// bayer_edge.cu -- micro-benchmark: where should k_bayer_to_bgr take the byte on each side of its 16-pixel group from?
// From L1 (the library's kernel: the neighbouring threads' loads brought the lines in) or from the neighbouring lanes
// by shuffle.  Both kernels over an L2-cold ring in a CUDA graph, alternated, CUDA events; outputs compared.
// build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -I ../../include -o bayer_edge bayer_edge.cu
// run on the GPU box
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "../../cudavideostream_b200/csrc/cvs_bayer.cuh"

// k_bayer_to_bgr with the bytes at x0-1 and x0+16 taken from the neighbouring lanes' 16-byte loads (shuffles) where
// those lanes hold the adjacent group of the same row, from L1 otherwise
namespace cvs {
__global__ void __launch_bounds__(kBayerThreads) k_bayer_shfl(const BayerParams p)
{
    const uint32_t item = blockIdx.x * kBayerThreads + threadIdx.x;
    const uint32_t y0 = item / p.groups;
    const bool live = y0 < (uint32_t)p.height;
    const uint32_t y = live ? y0 : (uint32_t)p.height - 1;
    const unsigned lane = threadIdx.x & 31u;
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
        const bool vec = live && npx == kBayerPixels && ((reinterpret_cast<uintptr_t>(p.raw) | p.pitch) & 15u) == 0;
        uint4 vv[3];
        const bool nb_vec = __shfl_down_sync(0xffffffffu, vec, 1);
        const bool left_ok = lane > 0 && x0 > 0, right_ok = lane < 31 && x0 + kBayerPixels < W && nb_vec;
#pragma unroll
        for (int k = 0; k < 3; k++) vv[k] = vec ? __ldg(reinterpret_cast<const uint4 *>(src[k] + x0)) : make_uint4(0, 0, 0, 0);
        uint32_t lb[3], rb[3];
#pragma unroll
        for (int k = 0; k < 3; k++) {
            lb[k] = __shfl_up_sync(0xffffffffu, vv[k].w, 1) >> 24;
            rb[k] = __shfl_down_sync(0xffffffffu, vv[k].x, 1) & 0xffu;
        }
        if (vec) {
            const int xl = max(x0 - 1, 0), xr = min(x0 + kBayerPixels, W - 1);
#pragma unroll
            for (int k = 0; k < 3; k++) {
                const uint4 v = vv[k];
                const uint32_t w[6] = {(left_ok ? lb[k] : (uint32_t)__ldg(src[k] + xl)) << 24, v.x, v.y, v.z, v.w,
                                       right_ok ? rb[k] : (uint32_t)__ldg(src[k] + xr)};
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

    if (!live) return;
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
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e)); exit(1); } } while (0)
template <class F> float graph_us(F launch, int K, cudaStream_t st) {
    cudaGraph_t g; cudaGraphExec_t ge;
    for (int i = 0; i < K; i++) launch(i, st);
    CK(cudaStreamSynchronize(st));
    CK(cudaStreamBeginCapture(st, cudaStreamCaptureModeGlobal));
    for (int i = 0; i < K; i++) launch(i, st);
    CK(cudaStreamEndCapture(st, &g));
    CK(cudaGraphInstantiate(&ge, g, 0));
    CK(cudaGraphLaunch(ge, st));
    CK(cudaStreamSynchronize(st));
    cudaEvent_t a, b; cudaEventCreate(&a); cudaEventCreate(&b);
    int reps = 3000 / K + 4;
    cudaEventRecord(a, st);
    for (int r = 0; r < reps; r++) cudaGraphLaunch(ge, st);
    cudaEventRecord(b, st);
    CK(cudaEventSynchronize(b));
    float ms; cudaEventElapsedTime(&ms, a, b);
    cudaGraphExecDestroy(ge); cudaGraphDestroy(g);
    return ms * 1e3f / (reps * K);
}
int main() {
    cudaStream_t st; CK(cudaStreamCreate(&st));
    int sizes[][2] = {{1920, 1080}, {3840, 2160}, {1918, 1078}};
    for (auto &wh : sizes) {
        int w = wh[0], h = wh[1];
        size_t pitch = (w + 15) / 16 * 16, fin = pitch * h, fout = ((size_t)3 * w * h + 15) / 16 * 16;
        int K = (int)(3 * (126u << 20) / (fin + fout)) + 1;
        uint8_t *src, *d1, *d2;
        CK(cudaMalloc(&src, K * fin)); CK(cudaMalloc(&d1, K * fout)); CK(cudaMalloc(&d2, K * fout));
        std::vector<uint8_t> hs(K * fin);
        for (auto &c : hs) c = (uint8_t)rand();
        CK(cudaMemcpy(src, hs.data(), hs.size(), cudaMemcpyHostToDevice));
        auto params = [&](int i, uint8_t *d) {
            cvs::BayerParams p; p.raw = src + i * fin; p.pitch = pitch; p.bgr = d + i * fout; p.width = w; p.height = h;
            p.groups = (w + 15) / 16; p.py = 1; p.px = 1; return p; };
        unsigned blocks = (unsigned)(((size_t)((w + 15) / 16) * h + 255) / 256);
        float t[2][3];
        for (int r = 0; r < 3; r++) { // alternated
            t[0][r] = graph_us([&](int i, cudaStream_t s) { cvs::k_bayer_to_bgr<<<blocks, 256, 0, s>>>(params(i, d1)); }, K, st);
            t[1][r] = graph_us([&](int i, cudaStream_t s) { cvs::k_bayer_shfl<<<blocks, 256, 0, s>>>(params(i, d2)); }, K, st);
        }
        std::vector<uint8_t> o1(K * fout), o2(K * fout);
        CK(cudaMemcpy(o1.data(), d1, o1.size(), cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(o2.data(), d2, o2.size(), cudaMemcpyDeviceToHost));
        size_t diff = 0;
        for (size_t i = 0; i < o1.size(); i++) diff += o1[i] != o2[i];
        printf("%dx%d pitch %zu ring %d: edge bytes from L1 %.2f %.2f %.2f us | from neighbouring lanes %.2f %.2f %.2f us | outputs differ in %zu bytes\n",
               w, h, pitch, K, t[0][0], t[0][1], t[0][2], t[1][0], t[1][1], t[1][2], diff);
        cudaFree(src); cudaFree(d1); cudaFree(d2);
    }
    return 0;
}
