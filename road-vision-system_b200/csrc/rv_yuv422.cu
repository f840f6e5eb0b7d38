/*
 * rv_yuv422.cu -- packed YUV 4:2:2 camera frames (YUY2, UYVY) to BGR, as cv2.cvtColor(COLOR_YUV2BGR_YUY2 / COLOR_YUV2BGR_UYVY)
 * computes it.  YUY2 (V4L2's YUYV) is the uncompressed output of UVC / USB cameras; UYVY is what GMSL / FPD-Link serializers and SDI
 * capture cards deliver.  Taking those frames as they are cuts the bytes a host-fed batch moves over PCIe to 2/3 (2 bytes per pixel
 * against 3) and spares the host its own colour conversion.
 *
 * The arithmetic is the 4:2:0 conversion's (rv_yuv_px.cuh) with one (U, V) pair per horizontal pixel pair.  A frame is cv2's (H, W, 2)
 * array: H rows of `pitch` bytes, each holding W/2 groups of 4 bytes, one per pixel pair (x = 2i, 2i + 1):
 *   YUY2  Y0 U Y1 V          UYVY  U Y0 V Y1
 * No row pairing is needed, so H may be odd; W is even (cv2 raises for an odd one: a pair is never split).
 *
 * k_yuv422_to_bgr<LAYOUT> has the structure of k_yuv420_to_bgr.  On aligned buffers a thread converts 8 pixels of one row: one 16-byte
 * load of four pixel pairs, the chroma terms computed 4 times, three 8-byte stores of the 24 output bytes; the thread that owns the
 * ragged right edge (W not a multiple of 8) converts it byte by byte.  Unaligned buffers (odd pitches, offset device pointers) take a
 * byte-wise path that maps pixel pair t, t + T, ... to thread t, so that a warp's accesses stay contiguous.
 *
 * The kernel has a translation unit of its own so that its SASS lines cannot re-pad cuobjdump's listing of the kernels in rv_yuv.cu
 * (rv_yuv_out.cu says why that would change their SASS hashes).
 */
#include "../../include/rv_b200.h"

#include <cuda_runtime.h>

#include <algorithm>

#include "rv_internal.h"
#include "rv_yuv_px.cuh"

using namespace rv;
using namespace rv::yuv;

namespace {

// byte offsets of Y0, U, Y1, V in a pixel pair's 4-byte group
template <int LAYOUT> struct Pair;
template <> struct Pair<RV_YUV_YUY2> { static constexpr int Y0 = 0, U = 1, Y1 = 2, V = 3; };
template <> struct Pair<RV_YUV_UYVY> { static constexpr int Y0 = 1, U = 0, Y1 = 3, V = 2; };

// the pixel pair whose 4-byte group starts at s, one byte at a time, into the 6 bytes at d
template <int LAYOUT>
__device__ __forceinline__ void pair_scalar(const uint8_t *s, uint8_t *d)
{
    using P = Pair<LAYOUT>;
    int buv, guv, ruv;
    chroma_terms(s[P::U], s[P::V], buv, guv, ruv);
    uint32_t p[6];
    bgr_px(s[P::Y0], buv, guv, ruv, p);
    bgr_px(s[P::Y1], buv, guv, ruv, p + 3);
    #pragma unroll
    for (int k = 0; k < 6; ++k) d[k] = (uint8_t)p[k];
}

// frame f of `src` starts at f * sfstride (= spitch * H); vec: every load address below is 16-byte aligned and every store address
// 8-byte aligned.  The x threads of the grid are sized for 8 pixels each.  vec: thread t converts pixels [8t, 8t + 8) of a row (the
// ragged right edge byte by byte).  Otherwise thread t converts the pixel pairs t, t + T, t + 2T, t + 3T (T threads) of a row, so
// that a warp's byte loads and stores stay contiguous.
template <int LAYOUT>
__global__ void __launch_bounds__(256) k_yuv422_to_bgr(const uint8_t *__restrict__ src, size_t spitch, size_t sfstride,
                                                       uint8_t *__restrict__ dst, size_t dpitch, size_t dfstride, int H, int W, int vec)
{
    using P = Pair<LAYOUT>;
    const int f = blockIdx.z, t = blockIdx.x * blockDim.x + threadIdx.x, T = gridDim.x * blockDim.x, x0 = 8 * t;
    if (vec && x0 >= W) return;
    for (int y = blockIdx.y; y < H; y += gridDim.y) {
        const uint8_t *s = src + (size_t)f * sfstride + (size_t)y * spitch;
        uint8_t *d = dst + (size_t)f * dfstride + (size_t)y * dpitch;
        if (!vec) {
            for (int q = t; q < W / 2; q += T) pair_scalar<LAYOUT>(s + 4 * q, d + 6 * q);
        } else if (x0 + 8 <= W) {
            const uint4 v = *reinterpret_cast<const uint4 *>(s + 2 * x0);
            const uint32_t g[4] = {v.x, v.y, v.z, v.w};
            uint32_t o[24];
            #pragma unroll
            for (int i = 0; i < 4; ++i) {
                int buv, guv, ruv;
                chroma_terms((g[i] >> (8 * P::U)) & 0xFF, (g[i] >> (8 * P::V)) & 0xFF, buv, guv, ruv);
                bgr_px((g[i] >> (8 * P::Y0)) & 0xFF, buv, guv, ruv, &o[6 * i]);
                bgr_px((g[i] >> (8 * P::Y1)) & 0xFF, buv, guv, ruv, &o[6 * i + 3]);
            }
            store24(d + 3 * x0, o);
        } else {
            for (int x = x0; x < W; x += 2) pair_scalar<LAYOUT>(s + 2 * x, d + 3 * x);
        }
    }
}

}  // namespace

int rv::launch_yuv422(rv_ctx *ctx, int layout, const uint8_t *src, size_t sp, uint8_t *dst, size_t dp, int n, int h, int w,
                      cudaStream_t st)
{
    const size_t sfs = sp * frame_rows(layout, h), dfs = dp * h;
    const int vec = (((uintptr_t)src | sp) % 16) == 0 && (((uintptr_t)dst | dp | dfs) % 8) == 0;
    const int groups = (w + 7) / 8;
    for (int f0 = 0; f0 < n; f0 += MAX_FRAMES_PER_LAUNCH) {
        const dim3 grid((groups + 255) / 256, std::min(h, 65535), std::min(MAX_FRAMES_PER_LAUNCH, n - f0));
        if (layout == RV_YUV_YUY2)
            k_yuv422_to_bgr<RV_YUV_YUY2><<<grid, 256, 0, st>>>(src + (size_t)f0 * sfs, sp, sfs, dst + (size_t)f0 * dfs, dp, dfs, h, w, vec);
        else
            k_yuv422_to_bgr<RV_YUV_UYVY><<<grid, 256, 0, st>>>(src + (size_t)f0 * sfs, sp, sfs, dst + (size_t)f0 * dfs, dp, dfs, h, w, vec);
        rv_internal_count_launches(ctx, 1);
    }
    CK(cudaGetLastError());
    return RV_OK;
}

extern "C" {

int rv_yuv422_to_bgr(rv_ctx *ctx, const uint8_t *in, uint8_t *out, int n, int h, int w, size_t in_pitch, size_t out_pitch, int layout,
                     int mem_kind, void *stream)
{
    if (!ctx) return RV_ERR_ARG;
    if (!out) return fail(ctx, RV_ERR_ARG, "null frame pointer");      // check_yuv takes a null `out` for a tensor-only job
    if (!is_yuv422(layout)) return fail(ctx, RV_ERR_ARG, "bad YUV 4:2:2 layout %d", layout);
    return convert_frames(ctx, in, out, n, h, w, in_pitch, out_pitch, layout, 0, mem_kind, stream);
}

}  // extern "C"
