/*
 * rv_yuv.cu -- YUV 4:2:0 decoder output (NV12, I420) to BGR, as cv2.cvtColor(COLOR_YUV2BGR_NV12 / COLOR_YUV2BGR_I420) computes it.
 * Hardware decoders (NVDEC, V4L2 M2M, VA-API, GStreamer `appsink format=NV12`) produce NV12, software decoders (libavcodec yuv420p)
 * produce I420.  Taking those frames as they are halves the bytes a host-fed batch moves over PCIe (1.5 bytes per pixel against 3)
 * and spares the host its own colour conversion.
 *
 * What cv2 computes (ITU-R BT.601 video range, 20-bit fixed point; every term fits in int32; rv_yuv_px.cuh, shared with rv_yuv422.cu):
 *   u = U - 128, v = V - 128, one (U, V) pair per 2 x 2 block of Y
 *   ruv = 2^19 + CVR v,  guv = 2^19 + CVG v + CUG u,  buv = 2^19 + CUB u,  y = max(0, Y - 16) CY
 *   B, G, R = sat_u8((y + buv) >> 20), sat_u8((y + guv) >> 20), sat_u8((y + ruv) >> 20)
 * Layouts (cv2's single-array form, 3h/2 rows of `pitch` bytes per frame):
 *   NV12  h rows of Y, then h/2 rows of interleaved U, V bytes (U first), both planes at the same pitch
 *   I420  the Y plane, then w h / 4 bytes of U, then w h / 4 bytes of V, packed back to back (pitch == w)
 *
 * k_yuv420_to_bgr<LAYOUT> writes packed BGR rows into a BGR buffer -- in the chunked host pipeline (rv_b200.cu, chain_pipe) the
 * 16-byte-pitched workspace on which the unchanged 3-channel chain then runs.  A thread converts 8 x 2 pixels (four chroma pairs)
 * with 8-byte loads of both Y rows and of the chroma (NV12; 4-byte U and V loads for I420) and 8-byte stores of the 2 x 24 output
 * bytes.  Unaligned buffers (odd pitches, offset device pointers, I420 frames whose width is not a multiple of 8) take a byte-wise
 * path with its own thread mapping, which keeps the warp's accesses contiguous; the ragged right edge is converted byte by byte.
 */
#include "../../include/rv_b200.h"

#include <cuda_runtime.h>

#include <algorithm>

#include "rv_internal.h"
#include "rv_yuv_px.cuh"

using namespace rv;
using namespace rv::yuv;

namespace {

__device__ __forceinline__ int byte_of(uint2 v, int k) { return (int)(((k < 4 ? v.x : v.y) >> (8 * (k & 3))) & 0xFFu); }

// the 2 x 2 block whose left column is x, one byte at a time (da / db: the block's two output rows)
template <int LAYOUT>
__device__ __forceinline__ void block_scalar(const uint8_t *ya, const uint8_t *yb, const uint8_t *c, size_t vofs, int x, uint8_t *da,
                                             uint8_t *db)
{
    int buv, guv, ruv;
    if constexpr (LAYOUT == RV_YUV_NV12) chroma_terms(c[x], c[x + 1], buv, guv, ruv);
    else chroma_terms(c[x / 2], c[vofs + x / 2], buv, guv, ruv);
    #pragma unroll
    for (int k = 0; k < 2; ++k) {
        uint32_t p[3];
        bgr_px(ya[x + k], buv, guv, ruv, p);
        #pragma unroll
        for (int ch = 0; ch < 3; ++ch) da[3 * k + ch] = (uint8_t)p[ch];
        bgr_px(yb[x + k], buv, guv, ruv, p);
        #pragma unroll
        for (int ch = 0; ch < 3; ++ch) db[3 * k + ch] = (uint8_t)p[ch];
    }
}

// frame f of `src` starts at f * sfstride (= spitch * H * 3 / 2); vec: every load and store address below is 8-byte aligned.
// The x threads of the grid are sized for 8 pixels each.  vec: thread t converts pixels [8t, 8t + 8) with vector loads and stores
// (the ragged right edge byte by byte).  Otherwise thread t converts the 2 x 2 blocks t, t + T, t + 2T, t + 3T (T threads), so that a
// warp's byte loads and stores stay contiguous; with 8 pixels per thread they would be 24 bytes apart, and the
// pass took 1.42 ms instead of 0.33 ms per 1080p x 64 batch (B200).
template <int LAYOUT>
__global__ void __launch_bounds__(256) k_yuv420_to_bgr(const uint8_t *__restrict__ src, size_t spitch, size_t sfstride,
                                                       uint8_t *__restrict__ dst, size_t dpitch, size_t dfstride, int H, int W, int vec)
{
    const int f = blockIdx.z, t = blockIdx.x * blockDim.x + threadIdx.x, T = gridDim.x * blockDim.x, x0 = 8 * t;
    if (vec && x0 >= W) return;
    const uint8_t *fr = src + (size_t)f * sfstride;
    // chroma row cy: NV12 U at uv[2i], V at uv[2i + 1]; I420 U at uv[i], V at uv[vofs + i]
    const uint8_t *uv = fr + (size_t)H * (LAYOUT == RV_YUV_NV12 ? spitch : (size_t)W);
    const size_t cpitch = LAYOUT == RV_YUV_NV12 ? spitch : (size_t)(W / 2), vofs = (size_t)(H / 2) * (W / 2);
    for (int cy = blockIdx.y; cy < H / 2; cy += gridDim.y) {
        const uint8_t *ya = fr + (size_t)(2 * cy) * spitch, *yb = ya + spitch, *c = uv + (size_t)cy * cpitch;
        uint8_t *ra = dst + (size_t)f * dfstride + (size_t)(2 * cy) * dpitch, *rb = ra + dpitch;
        if (!vec) {
            for (int q = t; q < W / 2; q += T) block_scalar<LAYOUT>(ya, yb, c, vofs, 2 * q, ra + 6 * q, rb + 6 * q);
        } else if (x0 + 8 <= W) {
            const uint2 va = *reinterpret_cast<const uint2 *>(ya + x0), vb = *reinterpret_cast<const uint2 *>(yb + x0);
            int U[4], V[4];
            if constexpr (LAYOUT == RV_YUV_NV12) {
                const uint2 cw = *reinterpret_cast<const uint2 *>(c + x0);
                #pragma unroll
                for (int i = 0; i < 4; ++i) { U[i] = byte_of(cw, 2 * i); V[i] = byte_of(cw, 2 * i + 1); }
            } else {
                const uint32_t cu = *reinterpret_cast<const uint32_t *>(c + x0 / 2), cv = *reinterpret_cast<const uint32_t *>(c + vofs + x0 / 2);
                #pragma unroll
                for (int i = 0; i < 4; ++i) { U[i] = (cu >> (8 * i)) & 0xFF; V[i] = (cv >> (8 * i)) & 0xFF; }
            }
            uint32_t oa[24], ob[24];
            #pragma unroll
            for (int i = 0; i < 4; ++i) {
                int buv, guv, ruv;
                chroma_terms(U[i], V[i], buv, guv, ruv);
                #pragma unroll
                for (int k = 0; k < 2; ++k) {
                    bgr_px(byte_of(va, 2 * i + k), buv, guv, ruv, &oa[3 * (2 * i + k)]);
                    bgr_px(byte_of(vb, 2 * i + k), buv, guv, ruv, &ob[3 * (2 * i + k)]);
                }
            }
            store24(ra + 3 * x0, oa);
            store24(rb + 3 * x0, ob);
        } else {
            for (int x = x0; x < W; x += 2) block_scalar<LAYOUT>(ya, yb, c, vofs, x, ra + 3 * x, rb + 3 * x);
        }
    }
}

}  // namespace

int rv::check_yuv(rv_ctx *ctx, const void *in, const void *out, int n, int h, int w, size_t ipitch, size_t opitch, int in_layout,
                  int out_layout)
{
    if (!ctx) return RV_ERR_ARG;
    if (in_layout != 0 && !is_yuv420(in_layout) && !is_yuv422(in_layout)) return fail(ctx, RV_ERR_ARG, "bad YUV layout %d", in_layout);
    if (out_layout != 0 && !is_yuv420(out_layout)) return fail(ctx, RV_ERR_ARG, "bad YUV layout %d", out_layout);
    if (!in_layout && !out_layout) return fail(ctx, RV_ERR_ARG, "bad YUV layout 0");
    const int ib = !in_layout ? 3 : is_yuv422(in_layout) ? 2 : 1, ob = out_layout ? 1 : 3;
    // without a frame output (a tensor-only job) the input stands in for it
    RV_TRY(check_frames(ctx, in, out ? out : in, n, h, w, ipitch, out ? opitch : (size_t)ob * w, ib, ob, 1));
    if ((is_yuv420(in_layout) || out_layout) && (h < 2 || w < 2 || ((h | w) & 1)))
        return fail(ctx, RV_ERR_ARG, "4:2:0 frames need an even height and width of at least 2, got %dx%d", w, h);
    if (is_yuv422(in_layout) && (w & 1)) return fail(ctx, RV_ERR_ARG, "4:2:2 frames need an even width, got %d", w);
    if (in_layout == RV_YUV_I420 && ipitch != (size_t)w) return fail(ctx, RV_ERR_ARG, "I420 frames need in_pitch == w (packed planes)");
    if (out && out_layout == RV_YUV_I420 && opitch != (size_t)w)
        return fail(ctx, RV_ERR_ARG, "I420 frames need out_pitch == w (packed planes)");
    if (out && n > 0) {
        const uintptr_t a0 = (uintptr_t)in, a1 = a0 + (size_t)n * ipitch * frame_rows(in_layout, h);
        const uintptr_t b0 = (uintptr_t)out, b1 = b0 + (size_t)n * opitch * frame_rows(out_layout, h);
        if (a0 < b1 && b0 < a1) return fail(ctx, RV_ERR_ARG, "input and output ranges overlap");
    }
    return RV_OK;
}

int rv::launch_yuv420(rv_ctx *ctx, int layout, const uint8_t *src, size_t sp, uint8_t *dst, size_t dp, int n, int h, int w,
                      cudaStream_t st)
{
    const size_t sfs = sp * frame_rows(layout, h), dfs = dp * h;
    const int vec = (((uintptr_t)src | sp | sfs | (uintptr_t)dst | dp | dfs) % 8) == 0;
    const int groups = (w + 7) / 8;
    for (int f0 = 0; f0 < n; f0 += MAX_FRAMES_PER_LAUNCH) {
        const dim3 grid((groups + 255) / 256, std::min(h / 2, 1024), std::min(MAX_FRAMES_PER_LAUNCH, n - f0));
        if (layout == RV_YUV_NV12)
            k_yuv420_to_bgr<RV_YUV_NV12><<<grid, 256, 0, st>>>(src + (size_t)f0 * sfs, sp, sfs, dst + (size_t)f0 * dfs, dp, dfs, h, w, vec);
        else
            k_yuv420_to_bgr<RV_YUV_I420><<<grid, 256, 0, st>>>(src + (size_t)f0 * sfs, sp, sfs, dst + (size_t)f0 * dfs, dp, dfs, h, w, vec);
        rv_internal_count_launches(ctx, 1);
    }
    CK(cudaGetLastError());
    return RV_OK;
}

int rv::launch_convert(rv_ctx *ctx, int in_layout, int out_layout, const uint8_t *src, size_t sp, uint8_t *dst, size_t dp, int n, int h,
                       int w, cudaStream_t st)
{
    if (is_yuv420(in_layout)) return launch_yuv420(ctx, in_layout, src, sp, dst, dp, n, h, w, st);
    if (is_yuv422(in_layout)) return launch_yuv422(ctx, in_layout, src, sp, dst, dp, n, h, w, st);
    return launch_bgr420(ctx, out_layout, src, sp, dst, dp, n, h, w, st);
}

int rv::convert_frames(rv_ctx *ctx, const uint8_t *in, uint8_t *out, int n, int h, int w, size_t in_pitch, size_t out_pitch,
                       int in_layout, int out_layout, int mem_kind, void *stream)
{
    RV_TRY(check_yuv(ctx, in, out, n, h, w, in_pitch, out_pitch, in_layout, out_layout));
    RV_TRY(check_kind(ctx, mem_kind));
    if (n == 0) return RV_OK;
    CK(cudaSetDevice(rv_internal_device(ctx)));
    if (mem_kind == RV_MEM_DEVICE) {
        cudaStream_t st = stream ? (cudaStream_t)stream : (cudaStream_t)rv_internal_stream(ctx);
        RV_TRY(launch_convert(ctx, in_layout, out_layout, in, in_pitch, out, out_pitch, n, h, w, st));
        if (!stream) CK(cudaStreamSynchronize(st));
        return RV_OK;
    }
    // host frames, group by group: H2D at a pitch the vector paths can read, conversion into a pitch they can write, D2H at the
    // caller's pitch
    ChWs &c = rv_internal_ch(ctx);
    cudaStream_t st = (cudaStream_t)rv_internal_stream(ctx);
    RV_TRY(ws_acquire(ctx, c.sync, st));
    const size_t irows = frame_rows(in_layout, h), ip = stage_pitch(in_layout, w);
    const size_t orows = frame_rows(out_layout, h), op = stage_pitch(out_layout, w);
    const int G = (int)group_frames(stage_pitch(0, w) * h);
    for (int f0 = 0; f0 < n; f0 += G) {
        const int g = std::min(G, n - f0);
        RV_TRY(ensure(ctx, c.din, ip * irows * g));
        RV_TRY(ensure(ctx, c.dout, op * orows * g));
        RV_TRY(copy_rows(ctx, c.din.p, ip, in + (size_t)f0 * in_pitch * irows, in_pitch, row_bytes(in_layout, w), irows * g,
                         cudaMemcpyHostToDevice, st));
        RV_TRY(launch_convert(ctx, in_layout, out_layout, (const uint8_t *)c.din.p, ip, (uint8_t *)c.dout.p, op, g, h, w, st));
        RV_TRY(copy_rows(ctx, out + (size_t)f0 * out_pitch * orows, out_pitch, c.dout.p, op, row_bytes(out_layout, w), orows * g,
                         cudaMemcpyDeviceToHost, st));
    }
    RV_TRY(ws_release(ctx, c.sync, st));
    CK(cudaStreamSynchronize(st));
    return RV_OK;
}

extern "C" {

int rv_yuv420_to_bgr(rv_ctx *ctx, const uint8_t *in, uint8_t *out, int n, int h, int w, size_t in_pitch, size_t out_pitch, int layout,
                     int mem_kind, void *stream)
{
    if (!ctx) return RV_ERR_ARG;
    if (!out) return fail(ctx, RV_ERR_ARG, "null frame pointer");      // check_yuv takes a null `out` for a tensor-only job
    if (is_yuv422(layout)) return fail(ctx, RV_ERR_ARG, "bad YUV layout %d (4:2:2 frames: rv_yuv422_to_bgr)", layout);
    return convert_frames(ctx, in, out, n, h, w, in_pitch, out_pitch, layout, 0, mem_kind, stream);
}

}  // extern "C"
