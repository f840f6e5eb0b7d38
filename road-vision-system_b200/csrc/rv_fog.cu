/*
 * rv_fog.cu -- fog synthesis on the GPU (SURVEY.md 8 f4): the full-frame work of the reference's
 * EnhancedFogSynthesizer.synthesize (/root/reference/src/augment/fog.py:227-299), the generator behind tools/fog_batch.py:7-34
 * that makes the hot path's test and benchmark inputs.
 *
 * Split of the work.  Everything that is O(1) per frame or needs the reference's exact random stream stays on the host
 * (road-vision-system_b200/augment/fog.py draws every random number with numpy's RandomState in the reference's order: fog
 * density, noise lattices, tints, glow / contrast / gamma / sensor-noise decisions; it also takes the 0.9-quantile of the top
 * band for the airlight colour, fog.py:120-131).  Per geometry the host builds the depth prior and the sky weight once
 * (fog.py:144-170).  Everything that touches every pixel of every frame runs here, in float32 like numpy:
 *
 *   k_fog_noise      multi-octave bilinear value noise (rand_perlin, fog.py:8-46) + global min / max
 *   k_fog_trans      beta map (fog.py:173-176) and transmission t = clip(exp(-beta d), 0.05, 1) (fog.py:179-185)
 *   k_bilateral_f32  cv2.bilateralFilter on float planes (the fallback of _guided_filter, fog.py:55-67): transmission, airlight
 *   k_fog_airlight   airlight map A = vgrad * A_rgb * xgrad (fog.py:133-137)
 *   k_fog_compose    I = J t + A (1 - t), global veil (fog.py:266-270), after scaling A to its target mean (fog.py:258-259)
 *   k_fog_gray_stats / k_fog_hard   glow mask from the gray mean / std (fog.py:188-192)
 *   k_gauss_rows / k_gauss_cols     separable cv2.GaussianBlur on float data, BORDER_REFLECT_101 (fog.py:193-197, 215-217)
 *   k_fog_glow, k_fog_band_mask, k_fog_band_mix   glow blend (fog.py:198) and the three-band depth blur (fog.py:201-221)
 *   k_fog_to_ycc, k_bilateral_u8, k_fog_finish    local contrast fade in YCrCb (fog.py:224-231), tint / gamma / sensor noise /
 *                                                 rounding to u8 (fog.py:284-293)
 *
 * Parity is statistical by nature (float pipeline, library exp / pow, OpenCV's SIMD summation order): tests compare with
 * frames the reference itself produced from the same seeds (tests/golden/fog_small.npz) within the tolerances written there.
 */
#include "../../include/rv_b200.h"

#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <new>
#include <vector>

#include "rv_internal.h"

using namespace rv;

namespace {

constexpr int MAX_TAPS = 95;                 // largest Gaussian kernel (k2 of the glow at 4K x heavy fog is 47)
constexpr int MAX_OCT = 4;

struct Taps { int n; float w[MAX_TAPS]; };
struct Lattices { int n; int gh[MAX_OCT], gw[MAX_OCT], off[MAX_OCT]; double amp[MAX_OCT]; float norm; };

struct FogState {
    int h = 0, w = 0;
    float *depth = nullptr, *sky = nullptr, *vgrad = nullptr, *xgrad = nullptr;     // per geometry
    float *f3[4] = {};                       // 3-channel float planes (interleaved BGR like the frame)
    float *p1[6] = {};                       // 1-channel float planes
    uint8_t *u8[5] = {};                     // frame in / out, Y, Cr, Cb (+ smoothed Y in p1 slot reuse is avoided: own plane)
    uint8_t *ysm = nullptr;
    float *lat = nullptr; size_t lat_cap = 0;
    double *red = nullptr;                   // reductions: [0] min bits, [1] max bits (as ints), [2] sum A, [3] sum gray, [4] sum gray^2
    float *noise = nullptr;
    size_t cap_px = 0;
};

__device__ __forceinline__ int refl101(int p, int len)
{
    if (len == 1) return 0;
    while (p < 0 || p >= len) p = p < 0 ? -p : 2 * (len - 1) - p;
    return p;
}

// ---- value noise ------------------------------------------------------------------------------------------------------
// rand_perlin: per octave, a (gh+1) x (gw+1) lattice of uniforms is sampled bilinearly at ys = linspace(0, gh, h, endpoint=False)
// (float64 in numpy), scaled by the octave amplitude and accumulated into a float32 image.
__global__ void k_fog_noise(const float *__restrict__ lat, Lattices L, int h, int w, float *__restrict__ base, int *__restrict__ mm)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    float v = 0.f;
    const bool in = x < w && y < h;
    if (in) {
        for (int o = 0; o < L.n; ++o) {
            const int gh = L.gh[o], gw = L.gw[o];
            const double ys = (double)y * ((double)gh / (double)h), xs = (double)x * ((double)gw / (double)w);
            const int y0 = (int)floor(ys), x0 = (int)floor(xs);
            const int y1 = min(y0 + 1, gh), x1 = min(x0 + 1, gw);
            const double wy = ys - y0, wx = xs - x0;
            const float *g = lat + L.off[o];
            const int pitch = gw + 1;
            const double top = (double)g[y0 * pitch + x0] * (1.0 - wx) + (double)g[y0 * pitch + x1] * wx;
            const double bot = (double)g[y1 * pitch + x0] * (1.0 - wx) + (double)g[y1 * pitch + x1] * wx;
            const double val = top * (1.0 - wy) + bot * wy;
            v = (float)((double)v + L.amp[o] * val);               // base += amp * val  (float32 accumulator)
        }
        v = __fdiv_rn(v, fmaxf(1e-6f, L.norm));
        base[(size_t)y * w + x] = v;
    }
    // block min / max -> global (values are >= 0: integer order of the bit patterns equals float order)
    float lo = in ? v : 3.0e38f, hi = in ? v : 0.f;
    for (int o = 16; o; o >>= 1) {
        lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if (((threadIdx.y * blockDim.x + threadIdx.x) & 31) == 0) {
        atomicMin(&mm[0], __float_as_int(lo));
        atomicMax(&mm[1], __float_as_int(hi));
    }
}

__global__ void k_fog_trans(const float *__restrict__ base, const int *__restrict__ mm, const float *__restrict__ depth, float base_beta,
                            size_t n, float *__restrict__ beta, float *__restrict__ t)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float mn = __int_as_float(mm[0]), mx = __int_as_float(mm[1]);
    const float nz = __fdiv_rn(__fsub_rn(base[i], mn), fmaxf(1e-6f, __fsub_rn(mx, mn)));
    const float b = __fmul_rn(base_beta, __fadd_rn(0.85f, __fmul_rn(0.35f, nz)));
    beta[i] = b;
    t[i] = fminf(fmaxf(expf(-__fmul_rn(b, depth[i])), 0.05f), 1.0f);
}

// ---- cv2.bilateralFilter, CV_32FC1, BORDER_REFLECT_101 ------------------------------------------------------------------
// weights: exp(-r^2 / (2 sigma_s^2)) over the disc r <= radius, times exp(-(v - v0)^2 / (2 sigma_c^2)); then clip.
// One block = 32 x 8 outputs; the (32 + 2R) x (8 + 2R) source patch is staged in shared memory.
// The weight of a tap is ONE ex2 of  r^2 cs log2(e) + (v - v0)^2 cc log2(e): the first term depends only on the tap and comes from a
// (2R + 1)^2 table in shared memory (every lane reads the same word: a broadcast), and each row of the disc is a contiguous run
// [-hw(dy), hw(dy)], so the inner loop is two loads, five float operations and the ex2, without an integer-to-float conversion
// (which shares the MUFU pipe with ex2) and without a test per tap.  Arguments stay in [-(R^2 + d^2) / 200, 0]: no range handling.
// Taps are visited in the order of the plain double loop (RV_FOG_BILATERAL_V1 keeps that first version for comparison: same
// frames to within the last bit of the weights, 2.3x the time).
__global__ void k_bilateral_f32(const float *__restrict__ src, int sstride, float *__restrict__ dst, int dstride, int h, int w, int radius,
                                float cs, float cc, float lo, float hi)
{
    extern __shared__ float tile[];
    const int pw = 32 + 2 * radius, ph = 8 + 2 * radius;
    const int bx = blockIdx.x * 32, by = blockIdx.y * 8;
    const int tid = threadIdx.y * 32 + threadIdx.x;
    for (int i = tid; i < pw * ph; i += 256) {
        const int ty = i / pw, tx = i - ty * pw;
        const int gy = refl101(by + ty - radius, h), gx = refl101(bx + tx - radius, w);
        tile[i] = src[((size_t)gy * w + gx) * sstride];
    }
#ifndef RV_FOG_BILATERAL_V1
    const int D = 2 * radius + 1;
    float *sw = tile + pw * ph;                  // [D][D] spatial exponents, scaled by log2(e)
    int *hw = reinterpret_cast<int *>(sw + D * D);   // [D] half-width of the disc's row
    constexpr float LOG2E = 1.4426950408889634f;
    const float csl = cs * LOG2E, ccl = cc * LOG2E;
    for (int i = tid; i < D * D; i += 256) {
        const int dy = i / D - radius, dx = i - (i / D) * D - radius;
        sw[i] = (float)(dy * dy + dx * dx) * csl;
    }
    if (tid < D) {
        const int dy = tid - radius, rem = radius * radius - dy * dy;
        int q = (int)sqrtf((float)rem);
        while (q * q > rem) --q;
        while ((q + 1) * (q + 1) <= rem) ++q;
        hw[tid] = q;
    }
    __syncthreads();
    const int x = bx + threadIdx.x, y = by + threadIdx.y;
    if (x >= w || y >= h) return;
    const float v0 = tile[(threadIdx.y + radius) * pw + threadIdx.x + radius];
    float sum = 0.f, wsum = 0.f;
    for (int j = 0; j < D; ++j) {
        const int q = hw[j];
        const float *row = tile + (threadIdx.y + j) * pw + threadIdx.x + radius;
        const float *srow = sw + j * D + radius;
#pragma unroll 4
        for (int dx = -q; dx <= q; ++dx) {
            const float v = row[dx];
            const float d = v - v0;
            float wgt;
            asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(wgt) : "f"(fmaf(d * d, ccl, srow[dx])));
            sum = fmaf(v, wgt, sum);
            wsum += wgt;
        }
    }
    dst[((size_t)y * w + x) * dstride] = fminf(fmaxf(sum / wsum, lo), hi);
#else
    __syncthreads();
    const int x = bx + threadIdx.x, y = by + threadIdx.y;
    if (x >= w || y >= h) return;
    const float v0 = tile[(threadIdx.y + radius) * pw + threadIdx.x + radius];
    float sum = 0.f, wsum = 0.f;
    const int r2 = radius * radius;
    for (int dy = -radius; dy <= radius; ++dy) {
        const float *row = tile + (threadIdx.y + radius + dy) * pw + threadIdx.x + radius;
        for (int dx = -radius; dx <= radius; ++dx) {
            const int rr = dy * dy + dx * dx;
            if (rr > r2) continue;
            const float v = row[dx];
            const float d = v - v0;
            const float wgt = __expf((float)rr * cs + d * d * cc);
            sum += v * wgt;
            wsum += wgt;
        }
    }
    dst[((size_t)y * w + x) * dstride] = fminf(fmaxf(sum / wsum, lo), hi);
#endif
}

// shared memory of k_bilateral_f32: the patch, the (2R + 1)^2 spatial table and the 2R + 1 row half-widths
static inline size_t bilateral_f32_smem(int R) { return ((size_t)(32 + 2 * R) * (8 + 2 * R) + (size_t)(2 * R + 1) * (2 * R + 1) + (2 * R + 1)) * 4; }

// ---- cv2.bilateralFilter, CV_8UC1 ----------------------------------------------------------------------------------------
__global__ void k_bilateral_u8(const uint8_t *__restrict__ src, uint8_t *__restrict__ dst, int h, int w, int radius, float cs, float cc)
{
    extern __shared__ float tile[];              // staged as bytes
    __shared__ float cw[256];
    uint8_t *tb = reinterpret_cast<uint8_t *>(tile);
    const int pw = 32 + 2 * radius, ph = 8 + 2 * radius;
    const int bx = blockIdx.x * 32, by = blockIdx.y * 8;
    const int tid = threadIdx.y * 32 + threadIdx.x;
    cw[tid] = expf((float)(tid * tid) * cc);
    for (int i = tid; i < pw * ph; i += 256) {
        const int ty = i / pw, tx = i - ty * pw;
        tb[i] = src[(size_t)refl101(by + ty - radius, h) * w + refl101(bx + tx - radius, w)];
    }
    __syncthreads();
    const int x = bx + threadIdx.x, y = by + threadIdx.y;
    if (x >= w || y >= h) return;
    const int v0 = tb[(threadIdx.y + radius) * pw + threadIdx.x + radius];
    float sum = 0.f, wsum = 0.f;
    const int r2 = radius * radius;
    for (int dy = -radius; dy <= radius; ++dy) {
        const uint8_t *row = tb + (threadIdx.y + radius + dy) * pw + threadIdx.x + radius;
        for (int dx = -radius; dx <= radius; ++dx) {
            const int rr = dy * dy + dx * dx;
            if (rr > r2) continue;
            const int v = row[dx];
            const float wgt = expf((float)rr * cs) * cw[abs(v - v0)];
            sum += (float)v * wgt;
            wsum += wgt;
        }
    }
    dst[(size_t)y * w + x] = (uint8_t)min(max(__float2int_rn(sum / wsum), 0), 255);
}

// ---- airlight map, composition ---------------------------------------------------------------------------------------------
__global__ void k_fog_airlight(const float *__restrict__ vgrad, const float *__restrict__ xgrad, float a0, float a1, float a2, int h, int w,
                               float *__restrict__ A)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= w || y >= h) return;
    const float v = vgrad[y], g = xgrad[x];
    float *o = A + ((size_t)y * w + x) * 3;
    o[0] = __fmul_rn(__fmul_rn(v, a0), g);
    o[1] = __fmul_rn(__fmul_rn(v, a1), g);
    o[2] = __fmul_rn(__fmul_rn(v, a2), g);
}

__global__ void k_sum(const float *__restrict__ a, size_t n, double *__restrict__ out)
{
    double s = 0.0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) s += (double)a[i];
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(out, s);
}

// A <- clip(A * scale, 0.75, 1);  hazy = J t + A (1 - t);  hazy = clip(hazy (1 - gv) + A gv, 0, 1), gv = veil (0.6 + 0.4 sky)
__global__ void k_fog_compose(const uint8_t *__restrict__ bgr, const float *__restrict__ t, float *__restrict__ A, const double *__restrict__ sumA,
                              float a_target, float veil, const float *__restrict__ sky, size_t npx, float *__restrict__ hazy)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npx) return;
    const float meanA = (float)(*sumA / (double)(3 * npx));
    const float scale = __fdiv_rn(a_target, fmaxf(1e-6f, meanA));
    const float tt = t[i], omt = __fsub_rn(1.0f, tt);
    const float gv = __fmul_rn(veil, __fadd_rn(0.6f, __fmul_rn(0.4f, sky[i])));
    const float omg = __fsub_rn(1.0f, gv);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float a = fminf(fmaxf(__fmul_rn(A[3 * i + c], scale), 0.75f), 1.0f);
        A[3 * i + c] = a;
        const float img = __fdiv_rn((float)bgr[3 * i + c], 255.0f);
        float hz = __fadd_rn(__fmul_rn(img, tt), __fmul_rn(a, omt));
        hz = __fadd_rn(__fmul_rn(hz, omg), __fmul_rn(a, gv));
        hazy[3 * i + c] = fminf(fmaxf(hz, 0.f), 1.f);
    }
}

// ---- glow -------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int u8_trunc(float v) { return (int)(__fmul_rn(v, 255.0f)); }      // (x * 255).astype(uint8), x in [0, 1]

__global__ void k_fog_gray_stats(const float *__restrict__ img, size_t npx, float *__restrict__ gray, double *__restrict__ sums)
{
    double s = 0.0, s2 = 0.0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < npx; i += (size_t)gridDim.x * blockDim.x) {
        const int B = u8_trunc(img[3 * i]), G = u8_trunc(img[3 * i + 1]), R = u8_trunc(img[3 * i + 2]);
        const float g = __fdiv_rn((float)((3735 * B + 19235 * G + 9798 * R + 16384) >> 15), 255.0f);
        gray[i] = g;
        s += (double)g;
        s2 += (double)g * (double)g;
    }
    for (int o = 16; o; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
    if ((threadIdx.x & 31) == 0) { atomicAdd(&sums[0], s); atomicAdd(&sums[1], s2); }
}

__global__ void k_fog_hard(const float *__restrict__ gray, const double *__restrict__ sums, size_t npx, float *__restrict__ hard)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npx) return;
    const double mean = sums[0] / (double)npx;
    const double var = fmax(sums[1] / (double)npx - mean * mean, 0.0);
    const float thr = fminf(fmaxf(__fadd_rn((float)mean, __fmul_rn(0.6f, (float)sqrt(var))), 0.65f), 0.9f);
    hard[i] = gray[i] > thr ? 1.0f : 0.0f;
}

// separable Gaussian, float, interleaved channels (nc = 1 or 3), BORDER_REFLECT_101
__global__ void k_gauss_rows(const float *__restrict__ src, float *__restrict__ dst, int h, int w, int nc, Taps tp)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= w) return;
    const int r = tp.n / 2;
    const float *row = src + (size_t)y * w * nc;
    float acc[3] = {0.f, 0.f, 0.f};
    for (int k = 0; k < tp.n; ++k) {
        const int xx = refl101(x + k - r, w);
        for (int c = 0; c < nc; ++c) acc[c] += row[xx * nc + c] * tp.w[k];
    }
    for (int c = 0; c < nc; ++c) dst[((size_t)y * w + x) * nc + c] = acc[c];
}

__global__ void k_gauss_cols(const float *__restrict__ src, float *__restrict__ dst, int h, int w, int nc, Taps tp, float lo, float hi)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= w) return;
    const int r = tp.n / 2;
    float acc[3] = {0.f, 0.f, 0.f};
    for (int k = 0; k < tp.n; ++k) {
        const int yy = refl101(y + k - r, h);
        for (int c = 0; c < nc; ++c) acc[c] += src[((size_t)yy * w + x) * nc + c] * tp.w[k];
    }
    for (int c = 0; c < nc; ++c) dst[((size_t)y * w + x) * nc + c] = fminf(fmaxf(acc[c], lo), hi);
}

// out = clip(img (1 - soft) + (img + s blur) soft, 0, 1)
__global__ void k_fog_glow(const float *__restrict__ img, const float *__restrict__ blur, const float *__restrict__ soft, float s, size_t npx,
                           float *__restrict__ out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npx) return;
    const float sf = soft[i], oms = __fsub_rn(1.0f, sf);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float v = img[3 * i + c];
        const float lit = __fadd_rn(v, __fmul_rn(s, blur[3 * i + c]));
        out[3 * i + c] = fminf(fmaxf(__fadd_rn(__fmul_rn(v, oms), __fmul_rn(lit, sf)), 0.f), 1.f);
    }
}

__global__ void k_fog_band_mask(const float *__restrict__ depth, float lo, float hi, size_t npx, float *__restrict__ mask)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < npx) mask[i] = (depth[i] >= lo && depth[i] < hi) ? 1.0f : 0.0f;
}

// out = out (1 - m) + blurred m
__global__ void k_fog_band_mix(float *__restrict__ out, const float *__restrict__ blurred, const float *__restrict__ m, size_t npx)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npx) return;
    const float mm = m[i], omm = __fsub_rn(1.0f, mm);
#pragma unroll
    for (int c = 0; c < 3; ++c) out[3 * i + c] = __fadd_rn(__fmul_rn(out[3 * i + c], omm), __fmul_rn(blurred[3 * i + c], mm));
}

// ---- local contrast fade + sensor model ------------------------------------------------------------------------------------------
__global__ void k_fog_to_ycc(const float *__restrict__ img, size_t npx, uint8_t *__restrict__ Y, uint8_t *__restrict__ Cr, uint8_t *__restrict__ Cb)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npx) return;
    const int B = u8_trunc(fminf(fmaxf(img[3 * i], 0.f), 1.f)), G = u8_trunc(fminf(fmaxf(img[3 * i + 1], 0.f), 1.f)),
              R = u8_trunc(fminf(fmaxf(img[3 * i + 2], 0.f), 1.f));
    const int y = (4899 * R + 9617 * G + 1868 * B + 8192) >> 14;
    Y[i] = (uint8_t)y;
    Cr[i] = (uint8_t)min(max(((R - y) * 11682 + ((128 << 14) + 8192)) >> 14, 0), 255);
    Cb[i] = (uint8_t)min(max(((B - y) * 9241 + ((128 << 14) + 8192)) >> 14, 0), 255);
}

__device__ __forceinline__ uint32_t fog_hash(uint32_t x)
{
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}

struct Finish { float amount, tint[3], gamma, noise_sigma; uint32_t seed; };

// y_mix = addWeighted(y, 1 - a, y_smooth, a); YCrCb -> BGR; / 255; * tint; ** gamma; + noise; (x * 255 + 0.5) -> u8
__global__ void k_fog_finish(const uint8_t *__restrict__ Y, const uint8_t *__restrict__ Ys, const uint8_t *__restrict__ Cr,
                             const uint8_t *__restrict__ Cb, Finish f, const float *__restrict__ noise, size_t npx, uint8_t *__restrict__ out)
{
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npx) return;
    const float a1 = __fsub_rn(1.0f, f.amount);
    const int ym = min(max(__float2int_rn(__fadd_rn(__fmul_rn((float)Y[i], a1), __fmul_rn((float)Ys[i], f.amount))), 0), 255);
    const int cb = Cb[i] - 128, cr = Cr[i] - 128;
    int c3[3];
    c3[0] = min(max(ym + ((cb * 29049 + 8192) >> 14), 0), 255);
    c3[1] = min(max(ym + ((cb * -5636 + cr * -11698 + 8192) >> 14), 0), 255);
    c3[2] = min(max(ym + ((cr * 22987 + 8192) >> 14), 0), 255);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        float v = __fdiv_rn((float)c3[c], 255.0f);
        v = fminf(fmaxf(__fmul_rn(v, f.tint[c]), 0.f), 1.f);
        if (f.gamma > 0.f) v = fminf(fmaxf(powf(v, f.gamma), 0.f), 1.f);
        if (f.noise_sigma > 0.f) {
            float nz;
            if (noise != nullptr) {
                nz = noise[3 * i + c];
            } else {                                     // device generator: Box-Muller over two hashed counters
                const uint32_t k = (uint32_t)(3 * i + c);
                const float u1 = ((fog_hash(k * 2u + f.seed) >> 8) + 1) * (1.0f / 16777217.0f);
                const float u2 = (fog_hash(k * 2u + 1u + f.seed * 0x9E3779B9u) >> 8) * (1.0f / 16777216.0f);
                nz = f.noise_sigma * sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
            }
            v = fminf(fmaxf(__fadd_rn(v, nz), 0.f), 1.f);
        }
        out[3 * i + c] = (uint8_t)(__fadd_rn(__fmul_rn(v, 255.0f), 0.5f));
    }
}

// ---- host ------------------------------------------------------------------------------------------------------------------------
Taps gaussian_taps(int k, double sigma)
{
    // cv2.getGaussianKernel(k, sigma, CV_32F): exp(-x^2 / (2 sigma^2)) in double, normalised, stored as float
    Taps t;
    t.n = k;
    std::vector<double> v(k);
    double sum = 0.0;
    for (int i = 0; i < k; ++i) {
        const double x = i - (k - 1) * 0.5;
        v[i] = exp(-0.5 / (sigma * sigma) * x * x);
        sum += v[i];
    }
    for (int i = 0; i < k; ++i) t.w[i] = (float)(v[i] / sum);
    for (int i = k; i < MAX_TAPS; ++i) t.w[i] = 0.f;
    return t;
}

void fog_free(FogState *s)
{
    if (!s) return;
    float *fl[] = {s->depth, s->sky, s->vgrad, s->xgrad, s->f3[0], s->f3[1], s->f3[2], s->f3[3], s->p1[0], s->p1[1], s->p1[2], s->p1[3], s->p1[4],
                   s->p1[5], s->lat, s->noise};
    for (float *p : fl)
        if (p) cudaFree(p);
    for (uint8_t *p : s->u8)
        if (p) cudaFree(p);
    if (s->ysm) cudaFree(s->ysm);
    if (s->red) cudaFree(s->red);
    delete s;
}

void fog_destroy_hook(void *p) { fog_free(static_cast<FogState *>(p)); }

int gauss(rv_ctx *ctx, cudaStream_t st, const float *src, float *tmp, float *dst, int h, int w, int nc, int k, double sigma, float lo, float hi)
{
    if (k > MAX_TAPS) return fail(ctx, RV_ERR_ARG, "Gaussian kernel %d larger than %d taps", k, MAX_TAPS);
    const Taps tp = gaussian_taps(k, sigma);
    dim3 grid((w + 127) / 128, h);
    k_gauss_rows<<<grid, 128, 0, st>>>(src, tmp, h, w, nc, tp);
    k_gauss_cols<<<grid, 128, 0, st>>>(tmp, dst, h, w, nc, tp, lo, hi);
    rv_internal_count_launches(ctx, 2);
    return RV_OK;
}

}  // namespace

extern "C" {

int rv_fog_set_geometry(rv_ctx *ctx, int h, int w, const float *depth, const float *sky_weight, const float *vgrad, const float *xgrad)
{
    if (!ctx) return RV_ERR_ARG;
    if (h < 1 || w < 1 || h > 32768 || w > 32768 || !depth || !sky_weight || !vgrad || !xgrad)
        return fail(ctx, RV_ERR_ARG, "bad fog geometry arguments");
    CK(cudaSetDevice(rv_internal_device(ctx)));
    CK(cudaDeviceSynchronize());
    fog_free(static_cast<FogState *>(rv_internal_get_fog(ctx)));
    rv_internal_set_fog(ctx, nullptr, nullptr);
    FogState *s = new (std::nothrow) FogState();
    if (!s) return RV_ERR_NOMEM;
    rv_internal_set_fog(ctx, s, fog_destroy_hook);
    const size_t npx = (size_t)h * w;
    s->h = h; s->w = w; s->cap_px = npx;
    CK(cudaMalloc(&s->depth, npx * 4));
    CK(cudaMalloc(&s->sky, npx * 4));
    CK(cudaMalloc(&s->vgrad, (size_t)h * 4));
    CK(cudaMalloc(&s->xgrad, (size_t)w * 4));
    for (float *&p : s->f3) CK(cudaMalloc(&p, npx * 12));
    for (float *&p : s->p1) CK(cudaMalloc(&p, npx * 4));
    for (int i = 0; i < 5; ++i) CK(cudaMalloc(&s->u8[i], i < 2 ? npx * 3 : npx));
    CK(cudaMalloc(&s->ysm, npx));
    CK(cudaMalloc(&s->red, 8 * sizeof(double)));
    CK(cudaMemcpy(s->depth, depth, npx * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(s->sky, sky_weight, npx * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(s->vgrad, vgrad, (size_t)h * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(s->xgrad, xgrad, (size_t)w * 4, cudaMemcpyHostToDevice));
    return RV_OK;
}

int rv_fog_u8(rv_ctx *ctx, const uint8_t *in, uint8_t *out, int h, int w, const rv_fog_frame *f, const float *lattice, const float *noise,
              float *t_out, float *beta_out, float *airlight_out)
{
    if (!ctx) return RV_ERR_ARG;
    FogState *s = static_cast<FogState *>(rv_internal_get_fog(ctx));
    if (!s || s->h != h || s->w != w) return fail(ctx, RV_ERR_ARG, "rv_fog_set_geometry(%d, %d) has not been called", h, w);
    if (!in || !out || !f || !lattice) return fail(ctx, RV_ERR_ARG, "null pointer");
    if (f->octaves < 1 || f->octaves > MAX_OCT) return fail(ctx, RV_ERR_ARG, "octaves %d not in [1,%d]", f->octaves, MAX_OCT);
    CK(cudaSetDevice(rv_internal_device(ctx)));
    cudaStream_t st = (cudaStream_t)rv_internal_stream(ctx);
    const size_t npx = (size_t)h * w;
    const int TB = 256;
    const unsigned gpx = (unsigned)((npx + TB - 1) / TB);
    dim3 b2(32, 8), g2((w + 31) / 32, (h + 7) / 8);

    // lattices
    Lattices L;
    memset(&L, 0, sizeof L);
    L.n = f->octaves;
    size_t lat_floats = 0;
    double amp = 1.0, norm = 0.0;
    for (int o = 0; o < L.n; ++o) {
        if (f->lat_gh[o] < 1 || f->lat_gw[o] < 1) return fail(ctx, RV_ERR_ARG, "bad lattice size");
        L.gh[o] = f->lat_gh[o]; L.gw[o] = f->lat_gw[o]; L.off[o] = (int)lat_floats; L.amp[o] = amp;
        lat_floats += (size_t)(L.gh[o] + 1) * (L.gw[o] + 1);
        norm += amp;
        amp *= f->persistence;
    }
    L.norm = (float)norm;
    if (s->lat_cap < lat_floats) {
        if (s->lat) CK(cudaFree(s->lat));
        s->lat = nullptr; s->lat_cap = 0;
        CK(cudaMalloc(&s->lat, lat_floats * 4));
        s->lat_cap = lat_floats;
    }
    CK(cudaMemcpyAsync(s->lat, lattice, lat_floats * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(s->u8[0], in, npx * 3, cudaMemcpyHostToDevice, st));
    const float *dnoise = nullptr;
    if (noise && f->noise_sigma > 0.f) {
        if (!s->noise) CK(cudaMalloc(&s->noise, npx * 12));
        CK(cudaMemcpyAsync(s->noise, noise, npx * 12, cudaMemcpyHostToDevice, st));
        dnoise = s->noise;
    }
    // reductions: min / max bit patterns, sum(A), sum(gray), sum(gray^2)
    {
        int mm[4] = {0x7f7fffff, 0, 0, 0};
        CK(cudaMemsetAsync(s->red, 0, 8 * sizeof(double), st));
        CK(cudaMemcpyAsync(s->red + 6, mm, sizeof mm, cudaMemcpyHostToDevice, st));
    }
    int *mm = reinterpret_cast<int *>(s->red + 6);
    float *base = s->p1[0], *beta = s->p1[1], *t0 = s->p1[2], *t = s->p1[3];
    float *A0 = s->f3[0], *A = s->f3[1], *hazy = s->f3[2];

    k_fog_noise<<<g2, b2, 0, st>>>(s->lat, L, h, w, base, mm);
    k_fog_trans<<<gpx, TB, 0, st>>>(base, mm, s->depth, f->base_beta, npx, beta, t0);
    rv_internal_count_launches(ctx, 2);
    if (beta_out) CK(cudaMemcpyAsync(beta_out, beta, npx * 4, cudaMemcpyDeviceToHost, st));      // the plane is reused below
    const float cs = (float)(-0.5 / (12.0 * 12.0)), cc = cs;
    if (f->edge_guided) {
        const int R = 8;
        k_bilateral_f32<<<g2, b2, bilateral_f32_smem(R), st>>>(t0, 1, t, 1, h, w, R, cs, cc, 0.05f, 1.0f);
        rv_internal_count_launches(ctx, 1);
    } else {
        t = t0;
    }
    // airlight: ramp map, per-channel bilateral (radius 16), clip to [0.7, 1], mean -> scale (inside k_fog_compose)
    k_fog_airlight<<<g2, b2, 0, st>>>(s->vgrad, s->xgrad, f->A_bgr[0], f->A_bgr[1], f->A_bgr[2], h, w, A0);
    {
        const int R = 16;
        for (int c = 0; c < 3; ++c)
            k_bilateral_f32<<<g2, b2, bilateral_f32_smem(R), st>>>(A0 + c, 3, A + c, 3, h, w, R, cs, cc, 0.7f, 1.0f);
    }
    k_sum<<<592, TB, 0, st>>>(A, npx * 3, s->red + 2);
    k_fog_compose<<<gpx, TB, 0, st>>>(s->u8[0], t, A, s->red + 2, f->a_target, f->global_veil, s->sky, npx, hazy);
    rv_internal_count_launches(ctx, 6);

    // glow (fog.py:188-198)
    float *gray = s->p1[0], *hard = s->p1[1], *soft = s->p1[4], *tmp1 = s->p1[5];
    float *blur = s->f3[0], *tmp3 = s->f3[3], *glow = s->f3[1];          // A0 and A are free from here on
    if (airlight_out) CK(cudaMemcpyAsync(airlight_out, A, npx * 12, cudaMemcpyDeviceToHost, st));
    k_fog_gray_stats<<<592, TB, 0, st>>>(hazy, npx, gray, s->red + 3);
    k_fog_hard<<<gpx, TB, 0, st>>>(gray, s->red + 3, npx, hard);
    rv_internal_count_launches(ctx, 2);
    {
        // k = int(9 + 20 s) | 1 and k2 = int(max(7, (h + w)(0.003 + 0.01 s))) | 1 come from the host (evaluated there in double)
        const int k = f->glow_k, k2 = f->glow_k2;
        if (k < 1 || k2 < 1 || !(k & 1) || !(k2 & 1)) return fail(ctx, RV_ERR_ARG, "bad glow kernel sizes %d, %d", k, k2);
        RV_TRY(gauss(ctx, st, hard, tmp1, soft, h, w, 1, k, k * 0.35, 0.f, 1.f));
        RV_TRY(gauss(ctx, st, hazy, tmp3, blur, h, w, 3, k2, k2 * 0.25, -3.0e38f, 3.0e38f));
    }
    k_fog_glow<<<gpx, TB, 0, st>>>(hazy, blur, soft, f->glow, npx, glow);
    rv_internal_count_launches(ctx, 1);

    // depth blur in three bands (fog.py:201-221): every band blurs the glow image, not the running result
    float *outp = s->f3[2];
    CK(cudaMemcpyAsync(outp, glow, npx * 12, cudaMemcpyDeviceToDevice, st));
    {
        const float edges[4] = {0.0f, 0.33f, 0.66f, 1.0f};
        for (int b = 0; b < 3; ++b) {
            const int rad = f->band_rad[b];
            if (rad <= 1) continue;
            float *mask = s->p1[0], *m = s->p1[1];
            k_fog_band_mask<<<gpx, TB, 0, st>>>(s->depth, edges[b], edges[b + 1], npx, mask);
            RV_TRY(gauss(ctx, st, glow, tmp3, blur, h, w, 3, rad, rad * 0.5, -3.0e38f, 3.0e38f));
            RV_TRY(gauss(ctx, st, mask, tmp1, m, h, w, 1, rad | 1, rad * 0.5, -3.0e38f, 3.0e38f));
            k_fog_band_mix<<<gpx, TB, 0, st>>>(outp, blur, m, npx);
            rv_internal_count_launches(ctx, 2);
        }
    }
    // local contrast fade + sensor model
    k_fog_to_ycc<<<gpx, TB, 0, st>>>(outp, npx, s->u8[2], s->u8[3], s->u8[4]);
    {
        const int d = f->fade_d;                   // int(5 + 20 a) | 1, from the host
        if (d < 1 || d > 63) return fail(ctx, RV_ERR_ARG, "bad fade kernel size %d", d);
        const int R = d / 2;
        const double sg = (double)f->fade_sigma;   // 25 + 50 a
        const float c2 = (float)(-0.5 / (sg * sg));
        k_bilateral_u8<<<g2, b2, (size_t)(32 + 2 * R) * (8 + 2 * R), st>>>(s->u8[2], s->ysm, h, w, R, c2, c2);
    }
    Finish fin;
    fin.amount = f->cdrop;
    for (int c = 0; c < 3; ++c) fin.tint[c] = f->tint[c];
    fin.gamma = f->gamma; fin.noise_sigma = f->noise_sigma; fin.seed = f->noise_seed;
    k_fog_finish<<<gpx, TB, 0, st>>>(s->u8[2], s->ysm, s->u8[3], s->u8[4], fin, dnoise, npx, s->u8[1]);
    rv_internal_count_launches(ctx, 3);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, s->u8[1], npx * 3, cudaMemcpyDeviceToHost, st));
    if (t_out) CK(cudaMemcpyAsync(t_out, t, npx * 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return RV_OK;
}

}  // extern "C"
