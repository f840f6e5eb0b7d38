/*
 * rv_u16.cu -- the stock chain on 16-bit frames: CLAHEDehaze (YCrCb) -> MedianDerain (k = 3 / 5) on uint16 BGR, as cv2 runs it on
 * CV_16U input (reference: src/preprocess/ops/clahe_dehaze.py:13-32, ops/median_derain.py:10-14, pipeline.py:24-30).  HDR road
 * cameras and raw frames read with cv2.IMREAD_ANYDEPTH deliver such frames; the reference hands them to cv2 unchanged.
 *
 * cv2's 16-bit arithmetic (the CPU restatement and its pins against cv2 are in the test suite, tests/test_u16.py):
 *   BGR2YCrCb   Y = D(1868 B + 9617 G + 4899 R), Cr = sat16(D((R - Y) 11682 + (32768 << 14))), Cb likewise with 9241 and B;
 *               D(x) = (x + 8192) >> 14
 *   YCrCb2BGR   B = sat16(Y + D((Cb - 32768) 29049)), G = sat16(Y + D((Cb - 32768)(-5636) + (Cr - 32768)(-11698))),
 *               R = sat16(Y + D((Cr - 32768) 22987))
 *   BGR2GRAY    (3735 B + 19235 G + 9798 R + 16384) >> 15 (the 8-bit coefficients), for the low-contrast gate
 *   CLAHE       SURVEY.md A.3 with 65,536 bins: clip = max(1, int(clip_limit * area / 65536)), batch = clipped / 65536,
 *               step = max(65536 / residual, 1), lutScale = float32(65535) / float32(area), 16-bit saturation
 *   medianBlur  exact k x k median per channel, BORDER_REPLICATE
 *
 * Kernels (none of them shares code with the 8-bit k_chain / k_luma_hist / k_build_lut, whose machine code is unchanged):
 *   k_u16_hist_lut    one CTA per (tile, frame): the tile's 65,536-bin histogram is built in shared memory one value half
 *                     (32,768 int32 bins, 128 KB) at a time -- half 0, half 1, half 0 again -- so that no counter can overflow
 *                     (a constant 4K tile at grid 8 has 129,600 pixels of one value) and nothing but the u16 LUT is ever
 *                     written to global memory.  Clip / redistribute / scan are warp-parallel; the redistribution is the
 *                     closed form of A.3 (bin i gets +1 iff i % step == 0 and i / step < residual).
 *   k_u16_apply       per pixel: Y, four LUT gathers (L2: a frame group's LUTs are sized to stay resident), the float32 blend
 *                     of A.3 without FMA, inverse YCrCb, u16 BGR out
 *   k_u16_median<K>   k = 3 / 5 with the generated selection networks of rv_median_net.h on u16x2 lanes (two output rows), in
 *                     their ALU form only (__vminu2 / __vmaxu2): the FMA-pipe form of the 8-bit kernel relies on values below
 *                     0x400 and is wrong for 16-bit data
 *   k_u16_gray_minmax, k_u16_gate_copy   the low-contrast gate; its decision is the 8-bit path's k_gate_flags (launch_gate_flags)
 *
 * The host side is the 8-bit path's (rv_internal.h): argument checks, CLAHE geometry, the gate threshold, workspaces and their
 * ordering between streams.
 */
#include "../../include/rv_b200.h"

#include <cuda_runtime.h>

#include <algorithm>

#include "rv_common.cuh"        // Geo, reflect101
#include "rv_internal.h"
#include "rv_median_net.h"      // RV_CEX is not overridden here: every compare-exchange is __vminu2 / __vmaxu2

using namespace rv;

namespace {

constexpr int U16_MAX_GRID = 64;            // a dense grid-64 LUT set is 512 MB per frame
constexpr int HALF_BINS = 32768;
constexpr int HL_THREADS = 1024;
constexpr size_t LUT_GROUP_BYTES = (size_t)48 << 20;    // LUTs of one frame group: well inside the 126 MB L2 of a B200

__device__ __forceinline__ int d14(int x) { return (x + 8192) >> 14; }
__device__ __forceinline__ int sat16(int v) { return min(max(v, 0), 65535); }
__device__ __forceinline__ int y16(int b, int g, int r) { return d14(1868 * b + 9617 * g + 4899 * r); }
__device__ __forceinline__ int gray16(int b, int g, int r) { return (3735 * b + 19235 * g + 9798 * r + 16384) >> 15; }

// Histogram + clip + redistribute + scan of one tile of one frame.  lut: [frame][tile][65536] u16.
__global__ void __launch_bounds__(HL_THREADS) k_u16_hist_lut(const uint16_t *__restrict__ src, size_t spitch, size_t sfstride, Geo g,
                                                             int clip, float lut_scale, uint16_t *__restrict__ lut,
                                                             const int32_t *__restrict__ flags)
{
    extern __shared__ int32_t hist[];                       // HALF_BINS counters, then per-warp partials
    int32_t *wsum = hist + HALF_BINS;                       // [32] capped sums
    int32_t *wclip = wsum + 32;                             // [32] clipped excess
    const int f = blockIdx.y, tile = blockIdx.x;
    if (flags && !flags[f]) return;
    const int ty = tile / g.grid, tx = tile % g.grid;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint16_t *fr = src + (size_t)f * (sfstride / 2);
    const size_t pitch = spitch / 2;
    uint16_t *tl = lut + ((size_t)f * g.grid * g.grid + tile) * 65536;

    int S0 = 0, clipped_total = 0, batch = 0, residual = 0, step = 1;
    for (int pass = 0; pass < 3; ++pass) {
        const int half = pass == 1 ? 1 : 0;
        for (int i = threadIdx.x; i < HALF_BINS; i += HL_THREADS) hist[i] = 0;
        __syncthreads();
        for (int r = warp; r < g.th; r += HL_THREADS / 32) {
            const uint16_t *row = fr + (size_t)reflect101(ty * g.th + r, g.H) * pitch;
            for (int c = lane; c < g.tw; c += 32) {
                const uint16_t *px = row + 3 * reflect101(tx * g.tw + c, g.W);
                const int Y = y16(px[0], px[1], px[2]);
                if ((Y >> 15) == half) atomicAdd(&hist[Y & (HALF_BINS - 1)], 1);
            }
        }
        __syncthreads();
        // warp w owns bins [1024 w, 1024 w + 1024) of this half, 32 consecutive bins per step
        const int base = warp * 1024;
        int capped_sum = 0, excess = 0;
        for (int k = 0; k < 32; ++k) {
            const int h = hist[base + 32 * k + lane];
            const int c = clip > 0 ? min(h, clip) : h;
            capped_sum += c;
            excess += h - c;
        }
        #pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            capped_sum += __shfl_xor_sync(0xffffffffu, capped_sum, o);
            excess += __shfl_xor_sync(0xffffffffu, excess, o);
        }
        if (lane == 0) { wsum[warp] = capped_sum; wclip[warp] = excess; }
        __syncthreads();
        int carry = 0, half_sum = 0, half_clip = 0;
        for (int w = 0; w < 32; ++w) {
            if (w == warp) carry = half_sum;
            half_sum += wsum[w];
            half_clip += wclip[w];
        }
        if (pass == 0) {
            S0 = half_sum;
            clipped_total = half_clip;
            __syncthreads();                                // wsum / wclip are rewritten by the next pass
            continue;
        }
        if (pass == 1) {
            clipped_total += half_clip;
            if (clip > 0) {
                batch = clipped_total / 65536;
                residual = clipped_total - batch * 65536;
                step = residual ? max(65536 / residual, 1) : 1;
            }
        }
        // LUT of this half, written over the counters (each lane reads its bin before it writes it)
        int run = (half ? S0 : 0) + carry;
        for (int k = 0; k < 32; ++k) {
            const int j = base + 32 * k + lane;
            const int h = hist[j];
            int x = clip > 0 ? min(h, clip) : h;
            #pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, x, o);
                if (lane >= o) x += t;
            }
            const int v = half * HALF_BINS + j;
            int s = run + x + batch * (v + 1);
            if (residual) s += min(v / step + 1, residual);
            run += __shfl_sync(0xffffffffu, x, 31);
            hist[j] = sat16(__float2int_rn(__fmul_rn(__int2float_rn(s), lut_scale)));
        }
        __syncthreads();
        uint32_t *dst = reinterpret_cast<uint32_t *>(tl + half * HALF_BINS);
        for (int i = threadIdx.x; i < HALF_BINS / 2; i += HL_THREADS)
            dst[i] = (uint32_t)hist[2 * i] | ((uint32_t)hist[2 * i + 1] << 16);
        __syncthreads();
    }
}

// CLAHE apply + inverse YCrCb, one pixel per thread.
__global__ void __launch_bounds__(256) k_u16_apply(const uint16_t *__restrict__ src, size_t spitch, size_t sfstride, uint16_t *__restrict__ dst,
                                                   size_t dpitch, size_t dfstride, Geo g, const uint16_t *__restrict__ lut,
                                                   const int32_t *__restrict__ flags)
{
    const int f = blockIdx.z, y = blockIdx.y, x = blockIdx.x * blockDim.x + threadIdx.x;
    if (x >= g.W || (flags && !flags[f])) return;
    const uint16_t *px = src + (size_t)f * (sfstride / 2) + (size_t)y * (spitch / 2) + 3 * x;
    const int B = px[0], G = px[1], R = px[2];
    const int Y = y16(B, G, R);
    const int Cr = sat16(d14((R - Y) * 11682 + (32768 << 14))) - 32768;
    const int Cb = sat16(d14((B - Y) * 9241 + (32768 << 14))) - 32768;

    // A.3 geometry and blend, every multiply and add rounded on its own (no FMA), xa from the unclamped tx1
    const float tyf = __fadd_rn(__fmul_rn((float)y, g.inv_th), -0.5f);
    int ty1 = (int)floorf(tyf);
    const float ya = __fsub_rn(tyf, (float)ty1), ya1 = __fsub_rn(1.0f, ya);
    const int ty2 = min(ty1 + 1, g.grid - 1);
    ty1 = max(ty1, 0);
    const float txf = __fadd_rn(__fmul_rn((float)x, g.inv_tw), -0.5f);
    int tx1 = (int)floorf(txf);
    const float xa = __fsub_rn(txf, (float)tx1), xa1 = __fsub_rn(1.0f, xa);
    const int tx2 = min(tx1 + 1, g.grid - 1);
    tx1 = max(tx1, 0);
    const uint16_t *L = lut + (size_t)f * g.grid * g.grid * 65536 + Y;
    const float l00 = (float)__ldg(L + ((size_t)(ty1 * g.grid + tx1) << 16)), l01 = (float)__ldg(L + ((size_t)(ty1 * g.grid + tx2) << 16));
    const float l10 = (float)__ldg(L + ((size_t)(ty2 * g.grid + tx1) << 16)), l11 = (float)__ldg(L + ((size_t)(ty2 * g.grid + tx2) << 16));
    const float top = __fadd_rn(__fmul_rn(l00, xa1), __fmul_rn(l01, xa));
    const float bot = __fadd_rn(__fmul_rn(l10, xa1), __fmul_rn(l11, xa));
    const int Yn = sat16(__float2int_rn(__fadd_rn(__fmul_rn(top, ya1), __fmul_rn(bot, ya))));

    uint16_t *o = dst + (size_t)f * (dfstride / 2) + (size_t)y * (dpitch / 2) + 3 * x;
    o[0] = (uint16_t)sat16(Yn + d14(Cb * 29049));
    o[1] = (uint16_t)sat16(Yn + d14(Cb * -5636 + Cr * -11698));
    o[2] = (uint16_t)sat16(Yn + d14(Cr * 22987));
}

// k x k median, k = 3 / 5.  A CTA covers MT_W x MT_H output pixels of one frame; its input box (with a k/2 halo, coordinates
// clamped = BORDER_REPLICATE) is staged in shared memory as three planes.  One task = one channel, one pair of output rows
// (r, r + MT_H / 2) in the two u16 lanes, M consecutive output columns.
constexpr int MT_W = 48, MT_H = 16, MT_HALF = MT_H / 2;

template <int K> struct U16Median;
template <> struct U16Median<3> { static constexpr int M = RV_MEDIAN3_M; };
template <> struct U16Median<5> { static constexpr int M = RV_MEDIAN5_M; };

template <int K>
__global__ void __launch_bounds__(3 * MT_HALF * (MT_W / U16Median<K>::M))
k_u16_median(const uint16_t *__restrict__ src, size_t spitch, size_t sfstride, uint16_t *__restrict__ dst, size_t dpitch, size_t dfstride,
             int H, int W, const int32_t *__restrict__ flags)
{
    constexpr int R = K / 2, M = U16Median<K>::M, NC = M + K - 1, SW = MT_W + K - 1, SH = MT_H + K - 1, GROUPS = MT_W / M;
    static_assert(MT_W % M == 0, "median tile width");
    __shared__ uint16_t s[3][SH][SW];
    const int f = blockIdx.z, x0 = blockIdx.x * MT_W, y0 = blockIdx.y * MT_H;
    if (flags && !flags[f]) return;
    const uint16_t *fr = src + (size_t)f * (sfstride / 2);
    const size_t sp = spitch / 2;
    for (int e = threadIdx.x; e < SH * SW * 3; e += blockDim.x) {
        const int r = e / (SW * 3), rem = e - r * (SW * 3), p = rem / 3, c = rem - 3 * p;
        const int gy = min(max(y0 - R + r, 0), H - 1), gx = min(max(x0 - R + p, 0), W - 1);
        s[c][r][p] = fr[(size_t)gy * sp + 3 * gx + c];
    }
    __syncthreads();
    const int t = threadIdx.x, c = t / (MT_HALF * GROUPS), rem = t - c * (MT_HALF * GROUPS), rp = rem / GROUPS, cg = rem - rp * GROUPS;
    uint32_t v[NC][K];
    #pragma unroll
    for (int j = 0; j < NC; ++j)
        #pragma unroll
        for (int k = 0; k < K; ++k)
            v[j][k] = (uint32_t)s[c][rp + k][cg * M + j] | ((uint32_t)s[c][rp + MT_HALF + k][cg * M + j] << 16);
    uint32_t out[M];
    if constexpr (K == 3) rv_median3_net(v, out);
    else rv_median5_net(v, out);
    uint16_t *fo = dst + (size_t)f * (dfstride / 2);
    const size_t dp = dpitch / 2;
    const int ya = y0 + rp, yb = ya + MT_HALF;
    #pragma unroll
    for (int o = 0; o < M; ++o) {
        const int x = x0 + cg * M + o;
        if (x >= W) break;
        if (ya < H) fo[(size_t)ya * dp + 3 * x + c] = (uint16_t)(out[o] & 0xFFFFu);
        if (yb < H) fo[(size_t)yb * dp + 3 * x + c] = (uint16_t)(out[o] >> 16);
    }
}

__global__ void k_u16_init_minmax(int32_t *mm, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { mm[2 * i] = 65535; mm[2 * i + 1] = 0; }
}

// gray min / max of every frame (pipeline.py:24-30): grid-stride over rows, one atomic pair per warp
__global__ void __launch_bounds__(256) k_u16_gray_minmax(const uint16_t *__restrict__ src, size_t spitch, size_t sfstride, int H, int W,
                                                         int32_t *__restrict__ mm)
{
    const int f = blockIdx.z;
    const uint16_t *fr = src + (size_t)f * (sfstride / 2);
    int lo = 65535, hi = 0;
    for (int y = blockIdx.y; y < H; y += gridDim.y) {
        const uint16_t *row = fr + (size_t)y * (spitch / 2);
        for (int x = blockIdx.x * blockDim.x + threadIdx.x; x < W; x += gridDim.x * blockDim.x) {
            const int gv = gray16(row[3 * x], row[3 * x + 1], row[3 * x + 2]);
            lo = min(lo, gv);
            hi = max(hi, gv);
        }
    }
    #pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMin(&mm[2 * f], lo);
        atomicMax(&mm[2 * f + 1], hi);
    }
}

// frames the gate skipped are passed through unchanged
__global__ void k_u16_gate_copy(const uint8_t *__restrict__ src, size_t spitch, size_t sfstride, uint8_t *__restrict__ dst, size_t dpitch,
                                size_t dfstride, int H, int rowbytes, const int32_t *__restrict__ flags)
{
    const int f = blockIdx.z;
    if (flags[f]) return;
    for (int y = blockIdx.y; y < H; y += gridDim.y) {
        const uint16_t *s = reinterpret_cast<const uint16_t *>(src + (size_t)f * sfstride + (size_t)y * spitch);
        uint16_t *d = reinterpret_cast<uint16_t *>(dst + (size_t)f * dfstride + (size_t)y * dpitch);
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < rowbytes / 2; i += gridDim.x * blockDim.x) d[i] = s[i];
    }
}

}  // namespace

// ------------------------------------------------------------------------------------------------ host side
namespace rv {

int check_params_u16(rv_ctx *ctx, const rv_params *p)
{
    if (!p) return fail(ctx, RV_ERR_ARG, "null params");
    if (p->space == RV_SPACE_LAB) return fail(ctx, RV_ERR_ARG, "LAB has no 16-bit path (cv2.cvtColor BGR2LAB rejects CV_16U)");
    if (p->space != RV_SPACE_YCRCB) return fail(ctx, RV_ERR_ARG, "bad space %d", p->space);
    if (p->clahe && (p->grid < 2 || p->grid > U16_MAX_GRID))
        return fail(ctx, RV_ERR_ARG, "tile grid %d out of range [2,%d] for 16-bit frames", p->grid, U16_MAX_GRID);
    if (!(p->ksize == 0 || p->ksize == 3 || p->ksize == 5))
        return fail(ctx, RV_ERR_ARG, "ksize %d not in {0,3,5} for 16-bit frames (cv2.medianBlur has no 16-bit k > 5)", p->ksize);
    if (!p->clahe && p->ksize == 0) return fail(ctx, RV_ERR_ARG, "nothing to do (no CLAHE, no median)");
    return RV_OK;
}

long group_frames_u16(const rv_params *p, int h, int w)
{
    long g = group_frames((size_t)6 * w * h);
    if (p->clahe) {
        const size_t lb = (size_t)p->grid * p->grid * 65536 * 2;
        g = std::min<long>(g, std::max<long>(1, (long)(LUT_GROUP_BYTES / lb)));
    }
    return g;
}

static int launch_median(rv_ctx *ctx, int k, const uint16_t *src, size_t sp, size_t sfs, uint16_t *dst, size_t dp, size_t dfs, int n, int h,
                  int w, const int32_t *flags, cudaStream_t st)
{
    for (int f0 = 0; f0 < n; f0 += MAX_FRAMES_PER_LAUNCH) {
        const int nf = std::min(MAX_FRAMES_PER_LAUNCH, n - f0);
        const dim3 grid((w + MT_W - 1) / MT_W, (h + MT_H - 1) / MT_H, nf);
        const uint16_t *s = (const uint16_t *)((const uint8_t *)src + (size_t)f0 * sfs);
        uint16_t *d = (uint16_t *)((uint8_t *)dst + (size_t)f0 * dfs);
        const int32_t *fl = flags ? flags + f0 : nullptr;
        if (k == 3)
            k_u16_median<3><<<grid, 3 * MT_HALF * (MT_W / U16Median<3>::M), 0, st>>>(s, sp, sfs, d, dp, dfs, h, w, fl);
        else
            k_u16_median<5><<<grid, 3 * MT_HALF * (MT_W / U16Median<5>::M), 0, st>>>(s, sp, sfs, d, dp, dfs, h, w, fl);
        rv_internal_count_launches(ctx, 1);
    }
    CK(cudaGetLastError());
    return RV_OK;
}

static int launch_gray(rv_ctx *ctx, U16Ws &s, const uint16_t *src, size_t sp, size_t sfs, int n, int h, int w, cudaStream_t st)
{
    RV_TRY(ensure(ctx, s.mm, (size_t)n * 8));
    int32_t *mm = (int32_t *)s.mm.p;
    k_u16_init_minmax<<<(n + 127) / 128, 128, 0, st>>>(mm, n);
    for (int f0 = 0; f0 < n; f0 += MAX_FRAMES_PER_LAUNCH) {
        const int nf = std::min(MAX_FRAMES_PER_LAUNCH, n - f0);
        const dim3 grid((unsigned)std::min(4, (w + 255) / 256), (unsigned)std::min(h, 32), nf);
        k_u16_gray_minmax<<<grid, 256, 0, st>>>((const uint16_t *)((const uint8_t *)src + (size_t)f0 * sfs), sp, sfs, h, w, mm + 2 * f0);
    }
    rv_internal_count_launches(ctx, 1 + (n + MAX_FRAMES_PER_LAUNCH - 1) / MAX_FRAMES_PER_LAUNCH);
    CK(cudaGetLastError());
    return RV_OK;
}

// The chain on one group of frames that are on the device.  Returns the device gate flags (or nullptr) through flags_out.
int run_group_u16(rv_ctx *ctx, U16Ws &s, const uint16_t *din, size_t ip, size_t ifs, uint16_t *dout, size_t op, size_t ofs, int n,
                  int h, int w, const rv_params *p, cudaStream_t st, const int32_t **flags_out, bool copy_skipped)
{
    const int32_t *flags = nullptr;
    if (p->gate_enable) {
        RV_TRY(launch_gray(ctx, s, din, ip, ifs, n, h, w, st));
        RV_TRY(ensure(ctx, s.flags, (size_t)n * 4));
        launch_gate_flags(ctx, (const int32_t *)s.mm.p, n, p->gate_thresh, (int32_t *)s.flags.p, st);
        flags = (const int32_t *)s.flags.p;
    }
    if (p->clahe) {
        const Geo g = make_geo(h, w, p->grid);
        const int tiles = g.grid * g.grid;
        RV_TRY(ensure(ctx, s.lut, (size_t)n * tiles * 65536 * 2));
        if (!s.attr_set) {
            CK(cudaFuncSetAttribute(k_u16_hist_lut, cudaFuncAttributeMaxDynamicSharedMemorySize, (HALF_BINS + 64) * 4));
            s.attr_set = true;
        }
        // clahe.cpp: clipLimit = max(int(clip * tileArea / histSize), 1) when clip > 0
        const int area = g.tw * g.th;
        int clip = 0;
        if (p->clip_limit > 0.0) clip = std::max((int)(p->clip_limit * (double)area / 65536.0), 1);
        const float lut_scale = 65535.0f / (float)area;
        uint16_t *lut = (uint16_t *)s.lut.p;
        k_u16_hist_lut<<<dim3(tiles, n), HL_THREADS, (HALF_BINS + 64) * 4, st>>>(din, ip, ifs, g, clip, lut_scale, lut, flags);
        uint16_t *ao = dout;
        size_t aop = op, aofs = ofs;
        if (p->ksize) {
            aop = (size_t)6 * w;
            aofs = aop * h;
            RV_TRY(ensure(ctx, s.mid, aofs * n));
            ao = (uint16_t *)s.mid.p;
        }
        k_u16_apply<<<dim3((w + 255) / 256, h, n), 256, 0, st>>>(din, ip, ifs, ao, aop, aofs, g, lut, flags);
        rv_internal_count_launches(ctx, 2);
        CK(cudaGetLastError());
        if (p->ksize) RV_TRY(launch_median(ctx, p->ksize, ao, aop, aofs, dout, op, ofs, n, h, w, flags, st));
    } else {
        RV_TRY(launch_median(ctx, p->ksize, din, ip, ifs, dout, op, ofs, n, h, w, flags, st));
    }
    if (flags && copy_skipped) {
        k_u16_gate_copy<<<dim3(4, std::min(h, 64), n), 256, 0, st>>>((const uint8_t *)din, ip, ifs, (uint8_t *)dout, op, ofs, h, 6 * w,
                                                                     flags);
        rv_internal_count_launches(ctx, 1);
        CK(cudaGetLastError());
    }
    *flags_out = flags;
    return RV_OK;
}

static int host_flags(rv_ctx *ctx, U16Ws &s, int n)
{
    if (s.hflags_cap >= (size_t)n) return RV_OK;
    if (s.hflags) CK(cudaFreeHost(s.hflags));
    s.hflags = nullptr;
    s.hflags_cap = 0;
    CK(cudaHostAlloc((void **)&s.hflags, (size_t)std::max(n, 64) * 4, cudaHostAllocDefault));
    s.hflags_cap = (size_t)std::max(n, 64);
    return RV_OK;
}

}  // namespace rv

extern "C" {

int rv_chain_u16(rv_ctx *ctx, const uint16_t *in, uint16_t *out, int n, int h, int w, size_t in_pitch, size_t out_pitch,
                 const rv_params *p, int mem_kind, int32_t *processed, void *stream)
{
    RV_TRY(check_frames(ctx, in, out, n, h, w, in_pitch, out_pitch, 6));
    RV_TRY(check_params_u16(ctx, p));
    RV_TRY(check_kind(ctx, mem_kind));
    if (in == out) return fail(ctx, RV_ERR_ARG, "in-place operation is not supported (tiles read their neighbours' halo)");
    if (n == 0) return RV_OK;
    CK(cudaSetDevice(rv_internal_device(ctx)));
    U16Ws &s = rv_internal_u16(ctx);
    const bool dev = mem_kind == RV_MEM_DEVICE;
    cudaStream_t st = (dev && stream) ? (cudaStream_t)stream : (cudaStream_t)rv_internal_stream(ctx);
    RV_TRY(ws_acquire(ctx, s.sync, st));
    if (processed && p->gate_enable) RV_TRY(host_flags(ctx, s, n));
    const long G = group_frames_u16(p, h, w);
    const size_t fb = (size_t)6 * w * h;
    for (int f0 = 0; f0 < n; f0 += (int)G) {
        const int g = (int)std::min<long>(G, n - f0);
        const uint16_t *gin;
        uint16_t *gout;
        size_t ip = in_pitch, op = out_pitch;
        if (dev) {
            gin = (const uint16_t *)((const uint8_t *)in + (size_t)f0 * h * in_pitch);
            gout = (uint16_t *)((uint8_t *)out + (size_t)f0 * h * out_pitch);
        } else {
            // host frames: one group at a time through packed device buffers (allocated once per shape, then reused)
            RV_TRY(ensure(ctx, s.din, fb * g));
            RV_TRY(ensure(ctx, s.dout, fb * g));
            CK(cudaMemcpy2DAsync(s.din.p, (size_t)6 * w, (const uint8_t *)in + (size_t)f0 * h * in_pitch, in_pitch, (size_t)6 * w,
                                 (size_t)h * g, cudaMemcpyHostToDevice, st));
            gin = (const uint16_t *)s.din.p;
            gout = (uint16_t *)s.dout.p;
            ip = op = (size_t)6 * w;
        }
        const int32_t *flags = nullptr;
        RV_TRY(run_group_u16(ctx, s, gin, ip, ip * h, gout, op, op * h, g, h, w, p, st, &flags));
        if (!dev)
            CK(cudaMemcpy2DAsync((uint8_t *)out + (size_t)f0 * h * out_pitch, out_pitch, s.dout.p, (size_t)6 * w, (size_t)6 * w,
                                 (size_t)h * g, cudaMemcpyDeviceToHost, st));
        if (processed && flags) CK(cudaMemcpyAsync(s.hflags + f0, flags, (size_t)g * 4, cudaMemcpyDeviceToHost, st));
    }
    RV_TRY(ws_release(ctx, s.sync, st));
    if (!dev || !stream || (processed && p->gate_enable)) CK(cudaStreamSynchronize(st));
    if (processed)
        for (int i = 0; i < n; ++i) processed[i] = p->gate_enable ? s.hflags[i] : 1;
    return RV_OK;
}

int rv_gray_span_u16(rv_ctx *ctx, const uint16_t *in, int n, int h, int w, size_t pitch, int32_t *span, int mem_kind)
{
    RV_TRY(check_frames(ctx, in, in, n, h, w, pitch, pitch, 6));
    RV_TRY(check_kind(ctx, mem_kind));
    if (!span) return fail(ctx, RV_ERR_ARG, "null span");
    if (n == 0) return RV_OK;
    CK(cudaSetDevice(rv_internal_device(ctx)));
    U16Ws &s = rv_internal_u16(ctx);
    cudaStream_t st = (cudaStream_t)rv_internal_stream(ctx);
    RV_TRY(ws_acquire(ctx, s.sync, st));
    RV_TRY(host_flags(ctx, s, 2 * n));
    const size_t fb = (size_t)6 * w * h;
    const int G = (int)group_frames(fb);
    for (int f0 = 0; f0 < n; f0 += G) {
        const int g = std::min(G, n - f0);
        const uint16_t *gin = (const uint16_t *)((const uint8_t *)in + (size_t)f0 * h * pitch);
        size_t ip = pitch;
        if (mem_kind != RV_MEM_DEVICE) {
            RV_TRY(ensure(ctx, s.din, fb * g));
            CK(cudaMemcpy2DAsync(s.din.p, (size_t)6 * w, gin, pitch, (size_t)6 * w, (size_t)h * g, cudaMemcpyHostToDevice, st));
            gin = (const uint16_t *)s.din.p;
            ip = (size_t)6 * w;
        }
        RV_TRY(launch_gray(ctx, s, gin, ip, ip * h, g, h, w, st));
        CK(cudaMemcpyAsync(s.hflags + 2 * (size_t)f0, s.mm.p, (size_t)g * 8, cudaMemcpyDeviceToHost, st));
    }
    RV_TRY(ws_release(ctx, s.sync, st));
    CK(cudaStreamSynchronize(st));
    return write_spans(ctx, s.hflags, n, span, mem_kind);
}

}  // extern "C"
