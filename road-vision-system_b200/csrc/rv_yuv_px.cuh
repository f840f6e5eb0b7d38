/*
 * rv_yuv_px.cuh -- cv2's per-pixel YUV -> BGR arithmetic (ITU-R BT.601 video range, 20-bit fixed point; every term fits in int32),
 * shared by the 4:2:0 (rv_yuv.cu) and the 4:2:2 (rv_yuv422.cu) conversions:
 *   u = U - 128, v = V - 128
 *   ruv = 2^19 + CVR v,  guv = 2^19 + CVG v + CUG u,  buv = 2^19 + CUB u,  y = max(0, Y - 16) CY
 *   B, G, R = sat_u8((y + buv) >> 20), sat_u8((y + guv) >> 20), sat_u8((y + ruv) >> 20)
 */
#pragma once
#include <cstdint>

// a namespace of their own: rv::sat8 (rv_common.cuh) is the chain's saturation of an unshifted value
namespace rv::yuv {

constexpr int CY = 1220542, CUB = 2116026, CUG = -409993, CVG = -852492, CVR = 1673527, HALF = 1 << 19;

__device__ __forceinline__ uint32_t sat8(int v) { return (uint32_t)min(max(v >> 20, 0), 255); }

// the B, G, R bytes of one pixel from its Y and the chroma terms of its (U, V) pair
__device__ __forceinline__ void bgr_px(int Y, int buv, int guv, int ruv, uint32_t *b)
{
    const int y = max(0, Y - 16) * CY;
    b[0] = sat8(y + buv);
    b[1] = sat8(y + guv);
    b[2] = sat8(y + ruv);
}

__device__ __forceinline__ void chroma_terms(int U, int V, int &buv, int &guv, int &ruv)
{
    const int u = U - 128, v = V - 128;
    buv = HALF + CUB * u;
    guv = HALF + CVG * v + CUG * u;
    ruv = HALF + CVR * v;
}

// packs 24 output bytes (one per word) and writes them with three 8-byte stores (d 8-byte aligned)
__device__ __forceinline__ void store24(uint8_t *d, const uint32_t (&b)[24])
{
    uint32_t o[6];
    #pragma unroll
    for (int i = 0; i < 6; ++i) o[i] = b[4 * i] | (b[4 * i + 1] << 8) | (b[4 * i + 2] << 16) | (b[4 * i + 3] << 24);
    #pragma unroll
    for (int i = 0; i < 3; ++i) reinterpret_cast<uint2 *>(d)[i] = make_uint2(o[2 * i], o[2 * i + 1]);
}

}  // namespace rv::yuv
