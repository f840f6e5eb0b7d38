/*
 * rv_yuv_out.cu -- processed BGR frames to YUV 4:2:0 (NV12, I420) for a video encoder, as cv2.cvtColor(COLOR_BGR2YUV_I420)
 * computes it.  NVENC and GStreamer encoders take NV12, libavcodec / x264 take yuv420p (I420).  Returning 4:2:0 halves the bytes a
 * host-fed batch copies back over PCIe (1.5 bytes per pixel against 3) and spares the host its own colour conversion.
 *
 * What cv2 computes (ITU-R BT.601 video range, 20-bit fixed point; every term fits in int32):
 *   Y = (CRY r + CGY g + CBY b + 2^19 + (16 << 20)) >> 20                     every pixel
 *   U = (CRU r + CGU g + CBU b + 2^19 + (128 << 20)) >> 20                    the top-left pixel of each 2 x 2 block only
 *   V = (CBU r + CGV g + CBV b + 2^19 + (128 << 20)) >> 20                    (not an average of the block)
 * Y lands in [16, 235] and U, V in [16, 240]: nothing saturates.  Layouts are those rv_yuv.cu reads: cv2's I420 array (the Y plane,
 * w h / 4 bytes of U, w h / 4 bytes of V, packed), and NV12 as that array with U and V interleaved (U first) in h/2 rows at the Y
 * pitch.
 *
 * k_bgr_to_yuv420<LAYOUT> has the structure of k_yuv420_to_bgr.  A thread converts 8 x 2 pixels: two rows of 24 bytes read with
 * 8-byte loads, two 8-byte Y stores and one 8-byte UV store (NV12) or 4-byte U and V stores (I420); the chroma arithmetic runs on
 * pixels 0, 2, 4, 6 of the top row only.  Unaligned buffers (odd pitches, offset device pointers, I420 frames whose width is not a
 * multiple of 8) take a byte-wise path that maps 2 x 2 blocks to consecutive threads, so that a warp's accesses stay contiguous.
 *
 * The kernel has a translation unit of its own: cuobjdump pads every line of a cubin's SASS listing to its longest instruction, and
 * the compiler materialises some of the coefficients below with HFMA2 moves whose operands print longer than any instruction of
 * rv_yuv.cu.  Compiled there, it would re-pad k_yuv420_to_bgr's listing and change that kernel's SASS hash (kernel_sass_hashes)
 * without any change to its machine code.
 */
#include "../../include/rv_b200.h"

#include <cuda_runtime.h>

#include <algorithm>

#include "rv_internal.h"

using namespace rv;

namespace {

constexpr int CRY = 269484, CGY = 528482, CBY = 102760, CRU = -155188, CGU = -305135, CBU = 460324, CGV = -385875, CBV = -74448;
constexpr int YBIAS = (1 << 19) + (16 << 20), CBIAS = (1 << 19) + (128 << 20);

__device__ __forceinline__ uint32_t y_of(int b, int g, int r) { return (uint32_t)((CRY * r + CGY * g + CBY * b + YBIAS) >> 20); }
__device__ __forceinline__ uint32_t u_of(int b, int g, int r) { return (uint32_t)((CRU * r + CGU * g + CBU * b + CBIAS) >> 20); }
__device__ __forceinline__ uint32_t v_of(int b, int g, int r) { return (uint32_t)((CBU * r + CGV * g + CBV * b + CBIAS) >> 20); }

__device__ __forceinline__ int byte_of(const uint32_t (&v)[6], int k) { return (int)((v[k >> 2] >> (8 * (k & 3))) & 0xFFu); }

// the 2 x 2 block whose left column is x, one byte at a time (sa / sb: its two BGR rows, at pixel x)
template <int LAYOUT>
__device__ __forceinline__ void block_scalar(const uint8_t *sa, const uint8_t *sb, uint8_t *ya, uint8_t *yb, uint8_t *c, size_t vofs,
                                             int x)
{
    #pragma unroll
    for (int k = 0; k < 2; ++k) {
        ya[x + k] = (uint8_t)y_of(sa[3 * k], sa[3 * k + 1], sa[3 * k + 2]);
        yb[x + k] = (uint8_t)y_of(sb[3 * k], sb[3 * k + 1], sb[3 * k + 2]);
    }
    const uint8_t U = (uint8_t)u_of(sa[0], sa[1], sa[2]), V = (uint8_t)v_of(sa[0], sa[1], sa[2]);
    if constexpr (LAYOUT == RV_YUV_NV12) { c[x] = U; c[x + 1] = V; }
    else { c[x / 2] = U; c[vofs + x / 2] = V; }
}

// frame f of `src` (BGR) starts at f * sfstride, frame f of `dst` at f * dfstride (= dpitch * H * 3 / 2); vec: every load and store
// address below is 8-byte aligned.  The thread mapping is k_yuv420_to_bgr's: with vec, thread t converts pixels [8t, 8t + 8) of both
// rows (the ragged right edge byte by byte); otherwise the 2 x 2 blocks t, t + T, ... (T threads).
template <int LAYOUT>
__global__ void __launch_bounds__(256) k_bgr_to_yuv420(const uint8_t *__restrict__ src, size_t spitch, size_t sfstride,
                                                       uint8_t *__restrict__ dst, size_t dpitch, size_t dfstride, int H, int W, int vec)
{
    const int f = blockIdx.z, t = blockIdx.x * blockDim.x + threadIdx.x, T = gridDim.x * blockDim.x, x0 = 8 * t;
    if (vec && x0 >= W) return;
    uint8_t *fr = dst + (size_t)f * dfstride;
    // chroma row cy: NV12 U at uv[2i], V at uv[2i + 1]; I420 U at uv[i], V at uv[vofs + i]
    uint8_t *uv = fr + (size_t)H * (LAYOUT == RV_YUV_NV12 ? dpitch : (size_t)W);
    const size_t cpitch = LAYOUT == RV_YUV_NV12 ? dpitch : (size_t)(W / 2), vofs = (size_t)(H / 2) * (W / 2);
    for (int cy = blockIdx.y; cy < H / 2; cy += gridDim.y) {
        const uint8_t *sa = src + (size_t)f * sfstride + (size_t)(2 * cy) * spitch, *sb = sa + spitch;
        uint8_t *ya = fr + (size_t)(2 * cy) * dpitch, *yb = ya + dpitch, *c = uv + (size_t)cy * cpitch;
        if (!vec) {
            for (int q = t; q < W / 2; q += T) block_scalar<LAYOUT>(sa + 6 * q, sb + 6 * q, ya, yb, c, vofs, 2 * q);
        } else if (x0 + 8 <= W) {
            uint32_t wa[6], wb[6];
            #pragma unroll
            for (int i = 0; i < 3; ++i) {
                const uint2 a = reinterpret_cast<const uint2 *>(sa + 3 * x0)[i], b = reinterpret_cast<const uint2 *>(sb + 3 * x0)[i];
                wa[2 * i] = a.x; wa[2 * i + 1] = a.y; wb[2 * i] = b.x; wb[2 * i + 1] = b.y;
            }
            uint32_t oa[2] = {0, 0}, ob[2] = {0, 0}, cu = 0, cv = 0;
            #pragma unroll
            for (int p = 0; p < 8; ++p) {
                oa[p >> 2] |= y_of(byte_of(wa, 3 * p), byte_of(wa, 3 * p + 1), byte_of(wa, 3 * p + 2)) << (8 * (p & 3));
                ob[p >> 2] |= y_of(byte_of(wb, 3 * p), byte_of(wb, 3 * p + 1), byte_of(wb, 3 * p + 2)) << (8 * (p & 3));
            }
            #pragma unroll
            for (int i = 0; i < 4; ++i) {                   // chroma of pixels 0, 2, 4, 6 of the top row
                const int b = byte_of(wa, 6 * i), g = byte_of(wa, 6 * i + 1), r = byte_of(wa, 6 * i + 2);
                cu |= u_of(b, g, r) << (8 * i);
                cv |= v_of(b, g, r) << (8 * i);
            }
            *reinterpret_cast<uint2 *>(ya + x0) = make_uint2(oa[0], oa[1]);
            *reinterpret_cast<uint2 *>(yb + x0) = make_uint2(ob[0], ob[1]);
            if constexpr (LAYOUT == RV_YUV_NV12) {
                // U0 V0 U1 V1 | U2 V2 U3 V3
                *reinterpret_cast<uint2 *>(c + x0) = make_uint2(__byte_perm(cu, cv, 0x5140), __byte_perm(cu, cv, 0x7362));
            } else {
                *reinterpret_cast<uint32_t *>(c + x0 / 2) = cu;
                *reinterpret_cast<uint32_t *>(c + vofs + x0 / 2) = cv;
            }
        } else {
            for (int x = x0; x < W; x += 2) block_scalar<LAYOUT>(sa + 3 * x, sb + 3 * x, ya, yb, c, vofs, x);
        }
    }
}

}  // namespace

int rv::launch_bgr420(rv_ctx *ctx, int layout, const uint8_t *src, size_t sp, uint8_t *dst, size_t dp, int n, int h, int w,
                      cudaStream_t st)
{
    const size_t sfs = sp * h, dfs = dp * frame_rows(layout, h);
    const int vec = (((uintptr_t)src | sp | (uintptr_t)dst | dp) % 8) == 0;       // (then both frame strides are multiples of 8)
    const int groups = (w + 7) / 8;
    for (int f0 = 0; f0 < n; f0 += MAX_FRAMES_PER_LAUNCH) {
        const dim3 grid((groups + 255) / 256, std::min(h / 2, 1024), std::min(MAX_FRAMES_PER_LAUNCH, n - f0));
        if (layout == RV_YUV_NV12)
            k_bgr_to_yuv420<RV_YUV_NV12><<<grid, 256, 0, st>>>(src + (size_t)f0 * sfs, sp, sfs, dst + (size_t)f0 * dfs, dp, dfs, h, w, vec);
        else
            k_bgr_to_yuv420<RV_YUV_I420><<<grid, 256, 0, st>>>(src + (size_t)f0 * sfs, sp, sfs, dst + (size_t)f0 * dfs, dp, dfs, h, w, vec);
        rv_internal_count_launches(ctx, 1);
    }
    CK(cudaGetLastError());
    return RV_OK;
}

extern "C" {

int rv_bgr_to_yuv420(rv_ctx *ctx, const uint8_t *in, uint8_t *out, int n, int h, int w, size_t in_pitch, size_t out_pitch, int layout,
                     int mem_kind, void *stream)
{
    if (!ctx) return RV_ERR_ARG;
    if (!out) return fail(ctx, RV_ERR_ARG, "null frame pointer");      // check_yuv takes a null `out` for a tensor-only job
    return convert_frames(ctx, in, out, n, h, w, in_pitch, out_pitch, 0, layout, mem_kind, stream);
}

}  // extern "C"
