/*
 * rv_channels.cu -- CLAHEDehaze, MedianDerain and the low-contrast gate on 4-channel (BGRA / BGRx) and single-channel frames, at 8
 * and 16 bits, as cv2 treats them (the reference hands whatever array it gets to cv2: src/preprocess/ops/clahe_dehaze.py:19-30,
 * ops/median_derain.py:14, pipeline.py:24-30).  BGRA frames come from cv2.imread(..., IMREAD_UNCHANGED) on PNGs with alpha and from
 * video decoders / converters (BGRx, RGBA surfaces); single-channel ones from monochrome, NIR and thermal cameras.
 *
 * What cv2 computes:
 *   CLAHE      cvtColor BGR2YCrCb / BGR2LAB read B, G, R of a 4-channel frame and ignore the fourth; the inverse conversion gives 3
 *              channels.  So CLAHEDehaze (and the fused CLAHE -> median pair) on BGRA is the 3-channel chain on the frame without its
 *              alpha.  LAB has no 16-bit path; one channel has no colour conversion at all (RV_ERR_ARG).
 *   median     every channel on its own, BORDER_REPLICATE, alpha included: k 3 / 5 / 7 / 9 at 8 bits, 3 / 5 at 16 bits.
 *   gate       BGR2GRAY of B, G, R, (3735 B + 19235 G + 9798 R + 16384) >> 15 at both depths, alpha ignored; no single channel.
 *
 * Kernels (the 3-channel kernels elsewhere are not touched; this file launches none of them itself):
 *   k_strip_alpha<T>        BGRA -> packed BGR in a 16-byte-pitched group workspace, four pixels per thread (16 / 32 bytes in,
 *                           12 / 24 bytes out); the 3-channel chains of rv_b200.cu (chain_device: histogram, LUT, k_chain with
 *                           TMA staging) and rv_u16.cu (run_group_u16) then run on that workspace unchanged.
 *   k_ch_median<T, K, CH>   k x k median of every channel of 1- or CH = 4-channel frames with the generated selection networks of
 *                           rv_median_net.h on u16x2 lanes.  8 bits: the two-row networks with a share of the compare-exchanges on
 *                           the FMA pipe, as k_chain; 16 bits: the one-row networks in ALU form, as k_u16_median.  A frame the gate
 *                           skips is copied through.
 *   k_ch_gray_minmax<T>     gray min / max of every 4-channel frame for the gate; the decision is launch_gate_flags'.
 *
 * Host frames go group by group: H2D into a packed buffer, the kernels, D2H.  Device frames are read and written in place.
 */
#include "../../include/rv_b200.h"

#include <cuda_runtime.h>

#include <algorithm>

#include <cuda_fp16.h>

#include "rv_common.cuh"        // RV_CHECK_IDX
#include "rv_internal.h"

// Median compare-exchange forms, as in rv_chain.cuh.  The two-row networks (RV_CEX*X2) serve 8-bit planes only, whose 0x00vv lanes are
// also exact IEEE half subnormals, so a share of their compare-exchanges runs on the FMA pipe (s = relu(b - a); max = a + s;
// min = b - s).  The one-row networks keep the ALU form (__vminu2 / __vmaxu2), which 16-bit planes need.
__device__ __forceinline__ void ch_ce_fma(uint32_t a, uint32_t b, uint32_t &lo, uint32_t &hi)
{
    const __half2 x = *reinterpret_cast<const __half2 *>(&a), y = *reinterpret_cast<const __half2 *>(&b);
    const uint32_t m1bits = 0xBC00BC00u;                       // (-1, -1)
    const __half2 m1 = *reinterpret_cast<const __half2 *>(&m1bits);
    const __half2 sd = __hfma2_relu(x, m1, y);                 // relu(y - x)
    const __half2 h = __hadd2(x, sd), l = __hsub2(y, sd);
    hi = *reinterpret_cast<const uint32_t *>(&h);
    lo = *reinterpret_cast<const uint32_t *>(&l);
}
#define CH_CEX_MIX(num, den, n, lo, hi, a, b)                      \
    uint32_t lo, hi;                                               \
    if constexpr (((n) % (den)) < (num)) ch_ce_fma(a, b, lo, hi);  \
    else { lo = __vminu2(a, b); hi = __vmaxu2(a, b); }
// shares on the FMA pipe: k_chain's measured ones (1/2 for k5, 3/7 where the kernel is nothing but the median), not retuned here
#define RV_CEX3X2(n, lo, hi, a, b) CH_CEX_MIX(1, 2, n, lo, hi, a, b)
#define RV_CEX5X2(n, lo, hi, a, b) CH_CEX_MIX(1, 2, n, lo, hi, a, b)
#define RV_CEX7X2(n, lo, hi, a, b) CH_CEX_MIX(3, 7, n, lo, hi, a, b)
#define RV_CEX9X2(n, lo, hi, a, b) CH_CEX_MIX(3, 7, n, lo, hi, a, b)
#include "rv_median_net.h"

using namespace rv;

namespace {

template <typename T> struct Word;                  // one 4-sample pixel as one load
template <> struct Word<uint8_t> { using type = uint32_t; };
template <> struct Word<uint16_t> { using type = uint2; };

// Three output words (12 samples) from four BGRA pixels, alpha dropped.
__device__ __forceinline__ void pack3(const uint32_t (&p)[4], uint32_t (&o)[3])
{
    o[0] = __byte_perm(p[0], p[1], 0x4210);
    o[1] = __byte_perm(p[1], p[2], 0x5421);
    o[2] = __byte_perm(p[2], p[3], 0x6542);
}
__device__ __forceinline__ void pack3(const uint2 (&p)[4], uint2 (&o)[3])
{
    o[0] = make_uint2(p[0].x, __byte_perm(p[0].y, p[1].x, 0x5410));
    o[1] = make_uint2(__byte_perm(p[1].x, p[1].y, 0x5432), p[2].x);
    o[2] = make_uint2(__byte_perm(p[2].y, p[3].x, 0x5410), __byte_perm(p[3].x, p[3].y, 0x5432));
}

// BGRA -> BGR, four pixels per thread.  vec: the source pixels are word aligned (one load per pixel); the destination always is.
template <typename T>
__global__ void __launch_bounds__(256) k_strip_alpha(const uint8_t *__restrict__ src, size_t spitch, size_t sfstride, uint8_t *__restrict__ dst,
                                                     size_t dpitch, size_t dfstride, int H, int W, int vec)
{
    using Wd = typename Word<T>::type;
    const int f = blockIdx.z, x0 = 4 * (blockIdx.x * blockDim.x + threadIdx.x);
    if (x0 >= W) return;
    for (int y = blockIdx.y; y < H; y += gridDim.y) {
        const T *s = reinterpret_cast<const T *>(src + (size_t)f * sfstride + (size_t)y * spitch) + 4 * x0;
        T *d = reinterpret_cast<T *>(dst + (size_t)f * dfstride + (size_t)y * dpitch) + 3 * x0;
        if (vec && x0 + 4 <= W) {
            Wd p[4], o[3];
            #pragma unroll
            for (int i = 0; i < 4; ++i) p[i] = reinterpret_cast<const Wd *>(s)[i];
            pack3(p, o);
            #pragma unroll
            for (int i = 0; i < 3; ++i) reinterpret_cast<Wd *>(d)[i] = o[i];
        } else {
            for (int i = 0; i < 4 && x0 + i < W; ++i)
                #pragma unroll
                for (int c = 0; c < 3; ++c) d[3 * i + c] = s[4 * i + c];
        }
    }
}

__global__ void k_ch_init_minmax(int32_t *mm, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { mm[2 * i] = 65535; mm[2 * i + 1] = 0; }
}

// gray min / max of every 4-channel frame (pipeline.py:24-30): grid-stride over rows, one atomic pair per warp
template <typename T>
__global__ void __launch_bounds__(256) k_ch_gray_minmax(const uint8_t *__restrict__ src, size_t spitch, size_t sfstride, int H, int W,
                                                        int32_t *__restrict__ mm)
{
    const int f = blockIdx.z;
    int lo = 65535, hi = 0;
    for (int y = blockIdx.y; y < H; y += gridDim.y) {
        const T *row = reinterpret_cast<const T *>(src + (size_t)f * sfstride + (size_t)y * spitch);
        for (int x = blockIdx.x * blockDim.x + threadIdx.x; x < W; x += gridDim.x * blockDim.x) {
            const int gv = (3735 * (int)row[4 * x] + 19235 * (int)row[4 * x + 1] + 9798 * (int)row[4 * x + 2] + 16384) >> 15;
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

// k x k median of each of the CH channels.  A CTA covers MT_W x MT_H output pixels of one frame; its input box (k/2 halo, clamped
// coordinates = BORDER_REPLICATE) is staged in shared memory as CH planes.  The two u16 lanes of a task hold output rows r and
// r + MT_H / 2.  8 bits: one task = two adjacent row pairs (the two-row networks share the K - 1 middle window rows); 16 bits: one row
// pair.  M consecutive output columns per task; a thread runs its task on every channel in turn.
constexpr int MT_W = 48, MT_H = 32, MT_HALF = MT_H / 2;

template <typename T, int K> struct ChMedian;       // M: output columns per task; ROWS: output rows per lane and task
template <int K> struct ChMedian<uint8_t, K> {
    static constexpr int M = K == 3 ? RV_MEDIAN3X2_M : K == 5 ? RV_MEDIAN5X2_M : K == 7 ? RV_MEDIAN7X2_M : RV_MEDIAN9X2_M, ROWS = 2;
};
template <int K> struct ChMedian<uint16_t, K> { static constexpr int M = K == 3 ? RV_MEDIAN3_M : RV_MEDIAN5_M, ROWS = 1; };

template <typename T, int K> constexpr int ch_median_threads()
{
    return MT_HALF / ChMedian<T, K>::ROWS * (MT_W / ChMedian<T, K>::M);
}

template <typename T, int K, int CH>
__global__ void __launch_bounds__(ch_median_threads<T, K>())
k_ch_median(const uint8_t *__restrict__ src, size_t spitch, size_t sfstride, uint8_t *__restrict__ dst, size_t dpitch, size_t dfstride,
            int H, int W, const int32_t *__restrict__ flags)
{
    constexpr int R = K / 2, M = ChMedian<T, K>::M, ROWS = ChMedian<T, K>::ROWS, NC = M + K - 1, NR = K + ROWS - 1;
    constexpr int SW = MT_W + K - 1, SH = MT_H + K - 1, GROUPS = MT_W / M;
    static_assert(MT_W % M == 0 && MT_HALF % ROWS == 0, "median tile");
    __shared__ T s[CH * SH * SW];
    const int f = blockIdx.z, x0 = blockIdx.x * MT_W, y0 = blockIdx.y * MT_H;
    const uint8_t *fr = src + (size_t)f * sfstride;
    uint8_t *fo = dst + (size_t)f * dfstride;
    if (flags && !flags[f]) {
        // the gate skipped this frame: its tile is copied through
        for (int e = threadIdx.x; e < MT_H * MT_W * CH; e += blockDim.x) {
            const int r = e / (MT_W * CH), q = e - r * (MT_W * CH), y = y0 + r;
            if (y < H && x0 * CH + q < W * CH)
                reinterpret_cast<T *>(fo + (size_t)y * dpitch)[x0 * CH + q] = reinterpret_cast<const T *>(fr + (size_t)y * spitch)[x0 * CH + q];
        }
        return;
    }
    for (int e = threadIdx.x; e < SH * SW * CH; e += blockDim.x) {
        const int r = e / (SW * CH), rem = e - r * (SW * CH), p = rem / CH, c = rem - CH * p;
        const int gy = min(max(y0 - R + r, 0), H - 1), gx = min(max(x0 - R + p, 0), W - 1);
        RV_CHECK_IDX((c * SH + r) * SW + p, CH * SH * SW, "k_ch_median staging");
        s[(c * SH + r) * SW + p] = reinterpret_cast<const T *>(fr + (size_t)gy * spitch)[CH * gx + c];
    }
    __syncthreads();
    const int rp = ROWS * (threadIdx.x / GROUPS), cg = threadIdx.x - (rp / ROWS) * GROUPS;
    if (y0 + rp >= H || x0 + cg * M >= W) return;
    #pragma unroll 1
    for (int c = 0; c < CH; ++c) {
        const T *pl = s + c * SH * SW;
        uint32_t v[NC][NR];
        #pragma unroll
        for (int j = 0; j < NC; ++j)
            #pragma unroll
            for (int k = 0; k < NR; ++k) {
                RV_CHECK_IDX((rp + MT_HALF + k) * SW + cg * M + j, SH * SW, "k_ch_median window");
                v[j][k] = (uint32_t)pl[(rp + k) * SW + cg * M + j] | ((uint32_t)pl[(rp + MT_HALF + k) * SW + cg * M + j] << 16);
            }
        uint32_t out[ROWS][M];
        if constexpr (ROWS == 2) {
            if constexpr (K == 3) rv_median3x2_net(v, out);
            else if constexpr (K == 5) rv_median5x2_net(v, out);
            else if constexpr (K == 7) rv_median7x2_net(v, out);
            else rv_median9x2_net(v, out);
        } else {
            if constexpr (K == 3) rv_median3_net(v, out[0]);
            else rv_median5_net(v, out[0]);
        }
        #pragma unroll
        for (int r = 0; r < ROWS; ++r) {
            const int ya = y0 + rp + r, yb = ya + MT_HALF;
            #pragma unroll
            for (int o = 0; o < M; ++o) {
                const int x = x0 + cg * M + o;
                if (x >= W) break;
                if (ya < H) reinterpret_cast<T *>(fo + (size_t)ya * dpitch)[CH * x + c] = (T)(out[r][o] & 0xFFFFu);
                if (yb < H) reinterpret_cast<T *>(fo + (size_t)yb * dpitch)[CH * x + c] = (T)(out[r][o] >> 16);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------ host side
// Every launch covers one frame group (group_frames: at most 256 frames), so frames always fit on gridDim.z in one launch.
template <typename T>
int launch_strip(rv_ctx *ctx, const uint8_t *src, size_t sp, size_t sfs, uint8_t *dst, size_t dp, size_t dfs, int n, int h, int w,
                 cudaStream_t st)
{
    const int vec = (((uintptr_t)src | sp | sfs) % (4 * sizeof(T))) == 0;
    const int quads = (w + 3) / 4;
    k_strip_alpha<T><<<dim3((quads + 255) / 256, std::min(h, 1024), n), 256, 0, st>>>(src, sp, sfs, dst, dp, dfs, h, w, vec);
    rv_internal_count_launches(ctx, 1);
    CK(cudaGetLastError());
    return RV_OK;
}

// gray (min, max) pairs of n 4-channel device frames into c.mm
template <typename T>
int launch_gray(rv_ctx *ctx, ChWs &c, const uint8_t *src, size_t sp, size_t sfs, int n, int h, int w, cudaStream_t st)
{
    RV_TRY(ensure(ctx, c.mm, (size_t)n * 8));
    int32_t *mm = (int32_t *)c.mm.p;
    k_ch_init_minmax<<<(n + 127) / 128, 128, 0, st>>>(mm, n);
    const dim3 grid((unsigned)std::min(4, (w + 255) / 256), (unsigned)std::min(h, 32), n);
    k_ch_gray_minmax<T><<<grid, 256, 0, st>>>(src, sp, sfs, h, w, mm);
    rv_internal_count_launches(ctx, 2);
    CK(cudaGetLastError());
    return RV_OK;
}

template <typename T, int K, int CH>
void launch_median_k(const uint8_t *s, size_t sp, size_t sfs, uint8_t *d, size_t dp, size_t dfs, int nf, int h, int w, const int32_t *fl,
                     cudaStream_t st)
{
    const dim3 grid((w + MT_W - 1) / MT_W, (h + MT_H - 1) / MT_H, nf);
    k_ch_median<T, K, CH><<<grid, ch_median_threads<T, K>(), 0, st>>>(s, sp, sfs, d, dp, dfs, h, w, fl);
}

template <typename T, int CH>
int launch_median(rv_ctx *ctx, int k, const uint8_t *src, size_t sp, size_t sfs, uint8_t *dst, size_t dp, size_t dfs, int n, int h, int w,
                  const int32_t *flags, cudaStream_t st)
{
    if (k == 3) launch_median_k<T, 3, CH>(src, sp, sfs, dst, dp, dfs, n, h, w, flags, st);
    else if (k == 5) launch_median_k<T, 5, CH>(src, sp, sfs, dst, dp, dfs, n, h, w, flags, st);
    else if constexpr (sizeof(T) == 1) {        // cv2.medianBlur has k 7 / 9 at 8 bits only
        if (k == 7) launch_median_k<T, 7, CH>(src, sp, sfs, dst, dp, dfs, n, h, w, flags, st);
        else launch_median_k<T, 9, CH>(src, sp, sfs, dst, dp, dfs, n, h, w, flags, st);
    }
    rv_internal_count_launches(ctx, 1);
    CK(cudaGetLastError());
    return RV_OK;
}

template <typename T>
int launch_median_ch(rv_ctx *ctx, int channels, int k, const uint8_t *src, size_t sp, size_t sfs, uint8_t *dst, size_t dp, size_t dfs,
                     int n, int h, int w, const int32_t *flags, cudaStream_t st)
{
    if (channels == 1) return launch_median<T, 1>(ctx, k, src, sp, sfs, dst, dp, dfs, n, h, w, flags, st);
    return launch_median<T, 4>(ctx, k, src, sp, sfs, dst, dp, dfs, n, h, w, flags, st);
}

int host_flags(rv_ctx *ctx, ChWs &c, size_t n)
{
    if (c.hflags_cap >= n) return RV_OK;
    if (c.hflags) CK(cudaFreeHost(c.hflags));
    c.hflags = nullptr;
    c.hflags_cap = 0;
    CK(cudaHostAlloc((void **)&c.hflags, std::max<size_t>(n, 64) * 4, cudaHostAllocDefault));
    c.hflags_cap = std::max<size_t>(n, 64);
    return RV_OK;
}

int check_depth(rv_ctx *ctx, int bits, int channels)
{
    if (!ctx) return RV_ERR_ARG;
    if (bits != 8 && bits != 16) return fail(ctx, RV_ERR_ARG, "bits %d not in {8,16}", bits);
    if (channels != 1 && channels != 3 && channels != 4) return fail(ctx, RV_ERR_ARG, "channels %d not in {1,3,4}", channels);
    return RV_OK;
}

}  // namespace

extern "C" {

int rv_chain_ex(rv_ctx *ctx, const void *in, void *out, int n, int h, int w, size_t in_pitch, size_t out_pitch, int bits, int channels,
                const rv_params *p, int mem_kind, int32_t *processed, void *stream)
{
    RV_TRY(check_depth(ctx, bits, channels));
    if (channels == 3)
        return bits == 8 ? rv_chain_u8(ctx, (const uint8_t *)in, (uint8_t *)out, n, h, w, in_pitch, out_pitch, p, mem_kind, processed, stream)
                         : rv_chain_u16(ctx, (const uint16_t *)in, (uint16_t *)out, n, h, w, in_pitch, out_pitch, p, mem_kind, processed,
                                        stream);
    if (!p) return fail(ctx, RV_ERR_ARG, "null params");
    const int sb = bits / 8, oc = p->clahe ? 3 : channels;
    RV_TRY(check_frames(ctx, in, out, n, h, w, in_pitch, out_pitch, channels * sb, oc * sb, sb));
    RV_TRY(bits == 8 ? check_params_u8(ctx, p) : check_params_u16(ctx, p));
    if (!p->clahe && p->ksize == 0) return fail(ctx, RV_ERR_ARG, "nothing to do (no CLAHE, no median)");
    if (channels == 1 && p->clahe)
        return fail(ctx, RV_ERR_ARG, "CLAHE needs 3- or 4-channel frames (cv2.cvtColor BGR2YCrCb / BGR2LAB reject one channel)");
    if (channels == 1 && p->gate_enable)
        return fail(ctx, RV_ERR_ARG, "the gate needs 3- or 4-channel frames (cv2.cvtColor BGR2GRAY rejects one channel)");
    if (p->clahe && p->gate_enable && !processed)
        return fail(ctx, RV_ERR_ARG, "the gate with CLAHE on 4-channel frames needs `processed` (skipped frames are not written)");
    RV_TRY(check_kind(ctx, mem_kind));
    if (in == out) return fail(ctx, RV_ERR_ARG, "in-place operation is not supported (tiles read their neighbours' halo)");
    if (n == 0) return RV_OK;
    CK(cudaSetDevice(rv_internal_device(ctx)));
    ChWs &c = rv_internal_ch(ctx);
    U16Ws &u = rv_internal_u16(ctx);
    const bool dev = mem_kind == RV_MEM_DEVICE, u16_clahe = bits == 16 && p->clahe;
    cudaStream_t st = (dev && stream) ? (cudaStream_t)stream : (cudaStream_t)rv_internal_stream(ctx);
    RV_TRY(ws_acquire(ctx, c.sync, st));
    if (u16_clahe) RV_TRY(ws_acquire(ctx, u.sync, st));
    if (processed && p->gate_enable) RV_TRY(host_flags(ctx, c, (size_t)n));
    const size_t ib = (size_t)channels * sb * w, ob = (size_t)oc * sb * w;     // packed row bytes of the host path
    const size_t pp = ((size_t)3 * sb * w + 15) & ~(size_t)15;                 // row pitch of the BGR workspace
    long G = group_frames(ib * h);
    if (u16_clahe) G = std::min(G, group_frames_u16(p, h, w));
    for (int f0 = 0; f0 < n; f0 += (int)G) {
        const int g = (int)std::min<long>(G, n - f0);
        const uint8_t *gin;
        uint8_t *gout;
        size_t ip = in_pitch, op = out_pitch;
        if (dev) {
            gin = (const uint8_t *)in + (size_t)f0 * h * in_pitch;
            gout = (uint8_t *)out + (size_t)f0 * h * out_pitch;
        } else {
            RV_TRY(ensure(ctx, c.din, ib * h * g));
            RV_TRY(ensure(ctx, c.dout, ob * h * g));
            CK(cudaMemcpy2DAsync(c.din.p, ib, (const uint8_t *)in + (size_t)f0 * h * in_pitch, in_pitch, ib, (size_t)h * g,
                                 cudaMemcpyHostToDevice, st));
            gin = (const uint8_t *)c.din.p;
            gout = (uint8_t *)c.dout.p;
            ip = ib;
            op = ob;
        }
        const int32_t *flags = nullptr;
        if (p->clahe) {
            RV_TRY(ensure(ctx, c.pack, pp * h * g));
            uint8_t *pk = (uint8_t *)c.pack.p;
            if (bits == 8) {
                RV_TRY(launch_strip<uint8_t>(ctx, gin, ip, ip * h, pk, pp, pp * h, g, h, w, st));
                // with the gate, chain_device writes the decisions to processed[] and synchronises
                RV_TRY(chain_device(ctx, pk, gout, g, h, w, pp, op, p, processed ? processed + f0 : nullptr, st, false));
            } else {
                RV_TRY(launch_strip<uint16_t>(ctx, gin, ip, ip * h, pk, pp, pp * h, g, h, w, st));
                RV_TRY(run_group_u16(ctx, u, (const uint16_t *)pk, pp, pp * h, (uint16_t *)gout, op, op * h, g, h, w, p, st, &flags, false));
            }
        } else {
            if (p->gate_enable) {
                RV_TRY(bits == 8 ? launch_gray<uint8_t>(ctx, c, gin, ip, ip * h, g, h, w, st)
                                 : launch_gray<uint16_t>(ctx, c, gin, ip, ip * h, g, h, w, st));
                RV_TRY(ensure(ctx, c.flags, (size_t)g * 4));
                launch_gate_flags(ctx, (const int32_t *)c.mm.p, g, p->gate_thresh, (int32_t *)c.flags.p, st);
                flags = (const int32_t *)c.flags.p;
            }
            RV_TRY(bits == 8 ? launch_median_ch<uint8_t>(ctx, channels, p->ksize, gin, ip, ip * h, gout, op, op * h, g, h, w, flags, st)
                             : launch_median_ch<uint16_t>(ctx, channels, p->ksize, gin, ip, ip * h, gout, op, op * h, g, h, w, flags, st));
        }
        if (processed && flags) CK(cudaMemcpyAsync(c.hflags + f0, flags, (size_t)g * 4, cudaMemcpyDeviceToHost, st));
        if (!dev) {
            uint8_t *hout = (uint8_t *)out + (size_t)f0 * h * out_pitch;
            if (p->clahe && p->gate_enable) {
                // only the frames the gate processed come back; the others stay as the caller left them
                CK(cudaStreamSynchronize(st));
                const int32_t *hf = bits == 8 ? processed + f0 : c.hflags + f0;
                for (int i = 0; i < g;) {
                    if (!hf[i]) { ++i; continue; }
                    int j = i;
                    while (j < g && hf[j]) ++j;
                    CK(cudaMemcpy2DAsync(hout + (size_t)i * h * out_pitch, out_pitch, gout + (size_t)i * h * ob, ob, ob, (size_t)h * (j - i),
                                         cudaMemcpyDeviceToHost, st));
                    i = j;
                }
            } else {
                CK(cudaMemcpy2DAsync(hout, out_pitch, gout, ob, ob, (size_t)h * g, cudaMemcpyDeviceToHost, st));
            }
        }
    }
    RV_TRY(ws_release(ctx, c.sync, st));
    if (u16_clahe) RV_TRY(ws_release(ctx, u.sync, st));
    if (!dev || !stream || (processed && p->gate_enable)) CK(cudaStreamSynchronize(st));
    if (processed && !(bits == 8 && p->clahe))
        for (int i = 0; i < n; ++i) processed[i] = p->gate_enable ? c.hflags[i] : 1;
    return RV_OK;
}

int rv_gray_span_ex(rv_ctx *ctx, const void *in, int n, int h, int w, size_t pitch, int bits, int channels, int32_t *span, int mem_kind)
{
    RV_TRY(check_depth(ctx, bits, channels));
    if (channels == 3)
        return bits == 8 ? rv_gray_span(ctx, (const uint8_t *)in, n, h, w, pitch, span, mem_kind)
                         : rv_gray_span_u16(ctx, (const uint16_t *)in, n, h, w, pitch, span, mem_kind);
    if (channels == 1) return fail(ctx, RV_ERR_ARG, "the gray span needs 3- or 4-channel frames (cv2.cvtColor BGR2GRAY rejects one channel)");
    const int sb = bits / 8;
    RV_TRY(check_frames(ctx, in, in, n, h, w, pitch, pitch, 4 * sb, 4 * sb, sb));
    RV_TRY(check_kind(ctx, mem_kind));
    if (!span) return fail(ctx, RV_ERR_ARG, "null span");
    if (n == 0) return RV_OK;
    CK(cudaSetDevice(rv_internal_device(ctx)));
    ChWs &c = rv_internal_ch(ctx);
    cudaStream_t st = (cudaStream_t)rv_internal_stream(ctx);
    RV_TRY(ws_acquire(ctx, c.sync, st));
    RV_TRY(host_flags(ctx, c, 2 * (size_t)n));
    const size_t ib = (size_t)4 * sb * w;
    const int G = (int)group_frames(ib * h);
    for (int f0 = 0; f0 < n; f0 += G) {
        const int g = std::min(G, n - f0);
        const uint8_t *gin = (const uint8_t *)in + (size_t)f0 * h * pitch;
        size_t ip = pitch;
        if (mem_kind != RV_MEM_DEVICE) {
            RV_TRY(ensure(ctx, c.din, ib * h * g));
            CK(cudaMemcpy2DAsync(c.din.p, ib, gin, pitch, ib, (size_t)h * g, cudaMemcpyHostToDevice, st));
            gin = (const uint8_t *)c.din.p;
            ip = ib;
        }
        RV_TRY(bits == 8 ? launch_gray<uint8_t>(ctx, c, gin, ip, ip * h, g, h, w, st) : launch_gray<uint16_t>(ctx, c, gin, ip, ip * h, g, h, w, st));
        CK(cudaMemcpyAsync(c.hflags + 2 * (size_t)f0, c.mm.p, (size_t)g * 8, cudaMemcpyDeviceToHost, st));
    }
    RV_TRY(ws_release(ctx, c.sync, st));
    CK(cudaStreamSynchronize(st));
    return write_spans(ctx, c.hflags, n, span, mem_kind);
}

}  // extern "C"
