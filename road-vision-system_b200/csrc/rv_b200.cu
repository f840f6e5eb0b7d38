/*
 * rv_b200.cu -- C ABI (include/rv_b200.h) over the sm_100a kernels in rv_kernels.cuh (rv_common / rv_colour / rv_hist_lut / rv_chain).
 *
 * Host-side logic of the drop-in boundary: parameter validation, CLAHE geometry
 * (clahe.cpp semantics, SURVEY.md A.3), workspaces, the hist -> lut -> apply+median launch
 * sequence in frame groups sized for L2 residency, and the chunked H2D / compute / D2H
 * pipeline for host buffers.  No CPU fallback anywhere: if CUDA fails the call fails.
 */
#include "../../include/rv_b200.h"

#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <mutex>
#include <new>
#include <thread>
#include <vector>

#include "rv_kernels.cuh"
#include "rv_internal.h"
#include "rv_ycc_g.h"

using namespace rv;

namespace {

#ifndef RV_NPIPE
#define RV_NPIPE 3
#endif
constexpr int NPIPE = RV_NPIPE;          // streams (and buffer sets) of the chunked host pipeline
constexpr int NWS = NPIPE + 3;               // workspace sets: [0, NPIPE) host pipeline, NPIPE / NPIPE+1 device path, NPIPE+2 single-frame path
constexpr int WS_FRAME = NPIPE + 2;

struct TimedLaunch {
    cudaEvent_t a, b;
    int which;                              // 0 k_luma_hist, 1 k_build_lut, 2 k_chain
};

// Read-only device tables that depend on the frame geometry only; built once per geometry, uploaded on the stream that
// first needs them from a page-locked host copy that lives as long as the entry, never rewritten afterwards.
struct ColTab {                             // k_chain column records for (W, tile width)
    int w = 0, tw = 0;
    float *dev = nullptr, *host = nullptr;
    cudaEvent_t ready = nullptr;
    cudaStream_t up = nullptr;
};
struct LbTab {                              // cv2.resize tables of k_letterbox for (h, w) -> (nh, nw)
    int h = 0, w = 0, nh = 0, nw = 0;
    uint8_t *dev = nullptr, *host = nullptr;
    size_t o_yofs = 0, o_xa = 0, o_ya = 0;
    cudaEvent_t ready = nullptr;
    cudaStream_t up = nullptr;
};
constexpr int MAX_TABS = 32;
constexpr int MAX_FRAME_GRAPHS = 16;
                // geometries cached per context before the cache is flushed

}  // namespace

// One instantiated CUDA graph per (frame shape, parameters) for the per-frame plugin contract `proc = pipeline(raw)`
// (main_preview.py:94): histogram (+ gate) -> LUT -> k_chain (-> gate copy, flag read-back) replayed with one launch between
// the H2D copy of the frame and the D2H copy of the result, which are issued around it because their host pointers change.
struct FrameGraph {
    int h = 0, w = 0;
    rv_params p = {};
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    void *bufs[6] = {};                     // the device buffers the graph was captured on (a reallocation invalidates it)
    long kernels = 0;                       // kernel nodes in the graph (launch accounting)
};

struct HostBuf {
    uint8_t *p = nullptr;
    size_t cap = 0;
};

// Helper threads that stage a PAGEABLE input frame into page-locked memory for the single-frame path: the frame is cut into slices,
// the caller and the helpers copy slices concurrently, and the caller issues the H2D DMA of each slice as soon as it is staged, so
// the CPU copy of later slices overlaps the DMA of earlier ones.  Helpers sleep on a condition variable between frames.
// MEASURED NEGATIVE (profiles/r2_g_latency.jsonl): with three helpers a 1080p call from pageable memory takes 0.95 ms (p50; best
// 0.63 ms) against 0.47 ms when the driver stages the frame itself (one cudaMemcpyAsync from pageable memory, ~19 GB/s): waking
// the helpers and their cold-cache memcpy cost more than they save.  Kept behind option "stage_threads" (default 0 = off).
struct StagePool {
    static constexpr int MAX_SLICES = 16;
    std::vector<std::thread> threads;
    std::mutex m;
    std::condition_variable cv;
    unsigned long gen = 0;
    bool quit = false;
    const uint8_t *src = nullptr;
    uint8_t *dst = nullptr;
    size_t bytes = 0, slice = 0;
    int nslices = 0;
    std::atomic<int> next{0};
    std::atomic<int> active{0};             // helpers currently inside a job; a new job is published only when it is 0
    std::atomic<int> done[MAX_SLICES];

    void copy_some()
    {
        for (;;) {
            const int s = next.fetch_add(1, std::memory_order_relaxed);
            if (s >= nslices) return;
            const size_t off = (size_t)s * slice, len = std::min(slice, bytes - off);
            memcpy(dst + off, src + off, len);
            done[s].store(1, std::memory_order_release);
        }
    }
    void copy_some_one()
    {
        const int s = next.fetch_add(1, std::memory_order_relaxed);
        if (s >= nslices) return;
        const size_t off = (size_t)s * slice, len = std::min(slice, bytes - off);
        memcpy(dst + off, src + off, len);
        done[s].store(1, std::memory_order_release);
    }
    void worker()
    {
        unsigned long seen = 0;
        for (;;) {
            {
                std::unique_lock<std::mutex> lk(m);
                cv.wait(lk, [&] { return quit || gen != seen; });
                if (quit) return;
                seen = gen;
                active.fetch_add(1, std::memory_order_relaxed);     // under the lock: the job's fields are final and stay so
            }
            copy_some();
            active.fetch_sub(1, std::memory_order_release);
        }
    }
    void start(int n)
    {
        for (int i = 0; i < n; ++i) threads.emplace_back([this] { worker(); });
    }
    void stop()
    {
        {
            std::lock_guard<std::mutex> lk(m);
            quit = true;
        }
        cv.notify_all();
        for (std::thread &t : threads) t.join();
        threads.clear();
    }
};

struct rv_ctx {
    int device = -1;
    int sm_count = 0;
    cudaStream_t stream = nullptr;          // main stream (device buffers, stage-level calls)
    cudaStream_t pipe[NPIPE] = {};          // H2D / compute / D2H pipeline for host buffers
    Buf hist[NWS], quads[NWS], lut[NWS], flags[NWS], mm[NWS];
    Buf din[NWS], dout[NWS];
    Buf dlb[NPIPE];                         // detector tensors of the host pipeline's chunks
    Buf dyuv[NPIPE];                        // 4:2:0 input chunks of the host pipeline (rv_submit_io_yuv), before the conversion
    WsSync wsync[NWS];
    cudaStream_t fstream = nullptr;         // single-frame path (per-frame plugin contract): its own stream, workspace set and graphs
    std::vector<struct FrameGraph> fgraphs;
    int32_t *fflag = nullptr;               // page-locked: gate decision of the single-frame path
    void *fog = nullptr;                    // state of rv_fog.cu (fog synthesis), destroyed through fog_destroy
    void (*fog_destroy)(void *) = nullptr;
    U16Ws u16;                              // workspaces of rv_u16.cu (16-bit frames)
    ChWs ch;                                // workspaces of rv_channels.cu (1- and 4-channel frames)
    StagePool *stage = nullptr;             // helper threads + page-locked staging frame for pageable single-frame input
    HostBuf fstage;                         // page-locked staging frame of the optional helper-thread upload
    long stage_threads = 0;                 // option "stage_threads": helpers next to the caller; 0 (default) = the driver stages pageable
                                            // input itself, which measured 2x faster on B200 hosts (0.47 ms against 0.95 ms per 1080p call)
    long frame_graphs = 1;                  // option "frame_graphs": 0 = the single-frame path launches directly (no CUDA graph)
    std::vector<ColTab> coltabs;
    std::vector<LbTab> lbtabs;
    cudaStream_t aux = nullptr;             // high-priority stream: histogram/LUT of the next group under the current k_chain
    cudaEvent_t ev_entry = nullptr, ev_pre[2] = {}, ev_chain[2] = {};
    long overlap_groups = 0;                // device path: split a batch into this many groups (0/1 = no overlap); measured
                                            // slower on B200 (k_chain leaves no SM resources for co-resident CTAs), kept as an option
    Buf scratch;                            // stage-level calls
    Buf lbfull;                             // full-resolution intermediate of the unfused letterbox (device path, set NPIPE)
    long launches = 0;
    long group_frames = 0, chunk_frames = 0;
    long chunk_taper = 1;                   // option "chunk_taper" (default on): smaller chunks at both ends of a host job (see chain_pipe)
    long prefetch_ctas_per_sm = 0;          // L2 prefetch distance of k_chain in CTAs per SM, option "prefetch_ctas" (0 = off, the
                                            // default: distances 2..9 measured 0.8 % slower -- the staging wait is already hidden)
    long use_tma = 1;                       // stage k_chain's box with TMA when the source buffer is 16-byte aligned
    long kernel_timing = 0;                 // bracket hist / lut / chain launches with events
    std::vector<TimedLaunch> timed;         // pending (not yet read) event pairs
    std::vector<cudaEvent_t> ev_pool;
    double k_ms[3] = {0, 0, 0};
    long k_n[3] = {0, 0, 0};
    char err[512] = {0};
};

namespace {

// Chroma round-trip tables of k_chain (layout: rv_colour.cuh, YccTabs).  Same integer formulas as A.1.
void build_ycc_table(YccTabs &y)
{
    memset(&y, 0, sizeof y);
    auto clamp8 = [](int v) { return v < 0 ? 0 : (v > 255 ? 255 : v); };
    for (int i = 0; i <= 510; ++i) {
        const int d = i - 255;
        // >> on negative ints is arithmetic here (gcc/nvcc host), as in the oracle
        const int cb = clamp8((d * 9241 + ((128 << 14) + 8192)) >> 14) - 128;
        const int cr = clamp8((d * 11682 + ((128 << 14) + 8192)) >> 14) - 128;
        const int fB = (cb * 29049 + 8192) >> 14, fR = (cr * 22987 + 8192) >> 14;
#if RV_YCC16
        y.e[i] = ((uint32_t)RV_YCC_GB[cb + 128] << 16) | (uint32_t)(fB + 256);
        y.e[512 + i] = ((uint32_t)RV_YCC_GR[cr + 128] << 16) | (uint32_t)(fR + 256);
#else
        const int tB = cb * -5636 / 2, tR = cr * -11698 / 2 + 4096 + (1 << 21);      // both products are even
        y.e[i] = ((uint32_t)(fB + 256) << 22) | ((uint32_t)tB & 0x3FFFFFu);
        y.e[512 + i] = ((uint32_t)(fR + 256) << 22) | ((uint32_t)tR & 0x3FFFFFu);
#endif
    }
}

// Histogram-pass LAB luminance tables (layout: rv_colour.cuh, LabHistTabs), from the same gamma and cube-root tables.
void build_lab_hist_table(LabHistTabs &t)
{
    memset(&t, 0, sizeof t);
    for (int v = 0; v < 256; ++v) {
        t.pm[0][v] = 871u * RV_LAB_G8[v];
        t.pm[1][v] = 2929u * RV_LAB_G8[v];
        t.pm[2][v] = 296u * RV_LAB_G8[v] + 2048u;
    }
    const int ncb = (int)(sizeof RV_LAB_CB / sizeof RV_LAB_CB[0]);
    for (int i = 0; i < 2048; ++i) {
        const int fy = i < ncb ? RV_LAB_CB[i] : RV_LAB_CB[ncb - 1];      // indices past the table are unreachable
        const int L = (296 * fy - 1336934 + 16384) >> 15;
        t.lq[i] = (uint8_t)(L < 0 ? 0 : (L > 255 ? 255 : L));
    }
}

}  // namespace

// ---- the host toolkit declared in rv_internal.h (shared with rv_fog.cu and rv_u16.cu) ------------------------------------
namespace rv {

int fail(rv_ctx *c, int code, const char *fmt, ...)
{
    if (c) {
        va_list ap;
        va_start(ap, fmt);
        vsnprintf(c->err, sizeof c->err, fmt, ap);
        va_end(ap);
    }
    return code;
}

int ensure(rv_ctx *ctx, Buf &b, size_t bytes)
{
    if (b.cap >= bytes) return RV_OK;
    if (b.p) CK(cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
    size_t want = (bytes + 255) & ~(size_t)255;
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) return fail(ctx, RV_ERR_NOMEM, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
    b.cap = want;
    return RV_OK;
}

int ws_acquire(rv_ctx *ctx, WsSync &w, cudaStream_t st)
{
    if (w.used && w.last != st) CK(cudaStreamWaitEvent(st, w.ev, 0));
    return RV_OK;
}

// (re-)arm the ordering event of a workspace set after the last work queued on `st` that touches it
int ws_release(rv_ctx *ctx, WsSync &w, cudaStream_t st)
{
    CK(cudaEventRecord(w.ev, st));
    w.last = st;
    w.used = true;
    return RV_OK;
}

int check_frames(rv_ctx *ctx, const void *in, const void *out, int n, int h, int w, size_t ipitch, size_t opitch, int in_bpp,
                 int out_bpp, int sample_bytes)
{
    if (!ctx) return RV_ERR_ARG;
    if (!in || !out) return fail(ctx, RV_ERR_ARG, "null frame pointer");
    if (n < 0 || h < 1 || w < 1) return fail(ctx, RV_ERR_ARG, "bad frame shape n=%d h=%d w=%d", n, h, w);
    if (h > 32768 || w > 32768) return fail(ctx, RV_ERR_ARG, "frame too large (%dx%d)", w, h);
    if (ipitch < (size_t)in_bpp * w) return fail(ctx, RV_ERR_ARG, "pitch smaller than %d*w", in_bpp);
    if (opitch < (size_t)out_bpp * w) return fail(ctx, RV_ERR_ARG, "pitch smaller than %d*w", out_bpp);
    if (sample_bytes == 2) {
        if ((ipitch | opitch) & 1) return fail(ctx, RV_ERR_ARG, "16-bit frames need even pitches");
        if (((uintptr_t)in | (uintptr_t)out) & 1) return fail(ctx, RV_ERR_ARG, "16-bit frames need 2-byte aligned buffers");
    }
    if (in != out && n > 0) {
        // unified addressing: host and device ranges never coincide, so a numeric overlap is a real one.  Tiles read their
        // neighbours' halo, so partially overlapping buffers would race exactly like in-place operation.
        const uintptr_t a0 = (uintptr_t)in, a1 = a0 + (size_t)n * h * ipitch, b0 = (uintptr_t)out, b1 = b0 + (size_t)n * h * opitch;
        if (a0 < b1 && b0 < a1) return fail(ctx, RV_ERR_ARG, "input and output ranges overlap");
    }
    return RV_OK;
}

int check_kind(rv_ctx *ctx, int kind)
{
    if (kind != RV_MEM_HOST && kind != RV_MEM_HOST_PINNED && kind != RV_MEM_DEVICE) return fail(ctx, RV_ERR_ARG, "bad memory kind %d", kind);
    return RV_OK;
}

// pipeline.py:24-30 compares an integer span with a Python float: span < t  <=>  span < ceil(t) for integer spans.  The
// decision is taken in integers on the device so that it can never differ from the per-frame path at the boundary.  A gray
// span is at most 65535 (16-bit frames), so every threshold above 65536 decides like 65536.
static int gate_thresh_int(double t)
{
    if (!(t == t)) return -1;                               // NaN: every comparison is false, nothing is processed
    const double c = ceil(t);
    if (c > 65536.0) return 65536;
    if (c < -1.0) return -1;
    return (int)c;
}

void launch_gate_flags(rv_ctx *ctx, const int32_t *mm, int n, double thresh, int32_t *flags, cudaStream_t st)
{
    k_gate_flags<<<(n + 127) / 128, 128, 0, st>>>(mm, n, gate_thresh_int(thresh), flags);
    ctx->launches++;
}

int write_spans(rv_ctx *ctx, const int32_t *mm, int n, int32_t *span, int mem_kind)
{
    int32_t *tmp = mem_kind == RV_MEM_DEVICE ? new (std::nothrow) int32_t[n] : span;
    if (!tmp) return fail(ctx, RV_ERR_NOMEM, "host alloc");
    for (int i = 0; i < n; ++i) tmp[i] = mm[2 * i + 1] - mm[2 * i];
    if (mem_kind == RV_MEM_DEVICE) {
        const cudaError_t e = cudaMemcpy(span, tmp, (size_t)n * 4, cudaMemcpyHostToDevice);
        delete[] tmp;
        if (e != cudaSuccess) return fail(ctx, RV_ERR_CUDA, "gray span copy: %s", cudaGetErrorString(e));
    }
    return RV_OK;
}

}  // namespace rv

namespace {

cudaEvent_t get_event(rv_ctx *ctx)
{
    if (!ctx->ev_pool.empty()) {
        cudaEvent_t e = ctx->ev_pool.back();
        ctx->ev_pool.pop_back();
        return e;
    }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}

struct ScopedTiming {                       // records an event pair around one launch when kernel_timing is on
    rv_ctx *ctx; cudaStream_t st; TimedLaunch t; bool on;
    ScopedTiming(rv_ctx *c, cudaStream_t s, int which) : ctx(c), st(s), on(c->kernel_timing != 0)
    {
        if (on) { t.a = get_event(c); t.b = get_event(c); t.which = which; cudaEventRecord(t.a, st); }
    }
    ~ScopedTiming()
    {
        if (on) { cudaEventRecord(t.b, st); ctx->timed.push_back(t); }
    }
};

int clip_int(double clip_limit, const Geo &g)
{
    if (!(clip_limit > 0.0)) return 0;
    int c = (int)(clip_limit * (double)(g.tw * g.th) / 256.0);
    return std::max(c, 1);
}

}  // namespace

int rv::check_params_u8(rv_ctx *ctx, const rv_params *p)
{
    if (!p) return fail(ctx, RV_ERR_ARG, "null params");
    if (p->space != RV_SPACE_YCRCB && p->space != RV_SPACE_LAB) return fail(ctx, RV_ERR_ARG, "bad space %d", p->space);
    if (p->clahe && (p->grid < 2 || p->grid > 256)) return fail(ctx, RV_ERR_ARG, "tile grid %d out of range [2,256]", p->grid);
    if (!(p->ksize == 0 || p->ksize == 3 || p->ksize == 5 || p->ksize == 7 || p->ksize == 9))
        return fail(ctx, RV_ERR_ARG, "ksize %d not in {0,3,5,7,9}", p->ksize);
    return RV_OK;
}

namespace {

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled()
{
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

// Tensor map over the source frames as u32 words: dims (3W/4, H, n), box (A_STRIDE/4 = 100, box_h, 1).  Returns false when the
// buffer does not meet TMA's alignment rules (the kernel then stages with ordinary loads).
bool make_src_map(const ChainArgs &a, int n, int box_h, CUtensorMap *map)
{
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return false;
    const uintptr_t base = reinterpret_cast<uintptr_t>(a.src);
    if ((base & 15) || (a.spitch & 15) || (a.sfstride & 15) || (3 * a.g.W) % 4) return false;
    if (3 * a.g.W / 4 < A_STRIDE / 4 || a.g.H < box_h) return false;
    cuuint64_t dims[3] = {(cuuint64_t)(3 * a.g.W / 4), (cuuint64_t)a.g.H, (cuuint64_t)n};
    cuuint64_t strides[2] = {(cuuint64_t)a.spitch, (cuuint64_t)(n > 1 ? a.sfstride : a.spitch * a.g.H)};
    cuuint32_t box[3] = {(cuuint32_t)(A_STRIDE / 4), (cuuint32_t)box_h, 1};
    cuuint32_t es[3] = {1, 1, 1};
    return enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, const_cast<uint8_t *>(a.src), dims, strides, box, es,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int MODE, int K>
int launch_chain_t(rv_ctx *ctx, const ChainArgs &a0, int n, cudaStream_t st)
{
    using S = ChainSmem<MODE, K>;
    ChainArgs a = a0;
    CUtensorMap tmap;
    memset(&tmap, 0, sizeof tmap);
    a.use_tma = (ctx->use_tma && make_src_map(a, n, S::BOX_H, &tmap)) ? 1 : 0;
    // the CTA that takes this one's place on its SM is (SMs x resident CTAs per SM) block ids ahead
    a.prefetch_dist = a.use_tma ? (int)(ctx->prefetch_ctas_per_sm * ctx->sm_count) : 0;
    static bool configured[64] = {};
    if (!configured[ctx->device & 63]) {
        CK(cudaFuncSetAttribute(k_chain<MODE, K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)S::total));
        configured[ctx->device & 63] = true;
    }
    dim3 grid((a.g.W + TILE_W - 1) / TILE_W, (a.g.H + TILE_H - 1) / TILE_H, n);
    {
        ScopedTiming tm(ctx, st, 2);
        k_chain<MODE, K><<<grid, CHAIN_THREADS, S::total, st>>>(a, tmap);
    }
    ctx->launches++;
    CK(cudaGetLastError());
    return RV_OK;
}

// frames ride on gridDim.z: very large batches of small frames go out in several launches
template <int MODE, int K>
int launch_chain_groups(rv_ctx *ctx, const ChainArgs &a0, int n, cudaStream_t st)
{
    if (n <= MAX_FRAMES_PER_LAUNCH) return launch_chain_t<MODE, K>(ctx, a0, n, st);
    for (int f0 = 0; f0 < n; f0 += MAX_FRAMES_PER_LAUNCH) {
        ChainArgs a = a0;
        a.src += (size_t)f0 * a.sfstride;
        a.dst += (size_t)f0 * a.dfstride;
        if (a.quads) a.quads += (size_t)f0 * (a.g.grid + 1) * (a.g.grid + 1) * 256;
        if (a.flags) a.flags += f0;
        if (a.lb_out) a.lb_out += (size_t)f0 * 3 * a.lb_S * a.lb_S;
        RV_TRY((launch_chain_t<MODE, K>(ctx, a, std::min(MAX_FRAMES_PER_LAUNCH, n - f0), st)));
    }
    return RV_OK;
}

template <int MODE>
int launch_chain_k(rv_ctx *ctx, const ChainArgs &a, int n, int k, cudaStream_t st)
{
    switch (k) {
        case 0: return launch_chain_groups<MODE, 0>(ctx, a, n, st);
        case 3: return launch_chain_groups<MODE, 3>(ctx, a, n, st);
        case 5: return launch_chain_groups<MODE, 5>(ctx, a, n, st);
        case 7: return launch_chain_groups<MODE, 7>(ctx, a, n, st);
        case 9: return launch_chain_groups<MODE, 9>(ctx, a, n, st);
    }
    return fail(ctx, RV_ERR_ARG, "bad ksize %d", k);
}

int launch_chain(rv_ctx *ctx, int mode, const ChainArgs &a, int n, int k, cudaStream_t st)
{
    if (mode == 0) return launch_chain_k<0>(ctx, a, n, k, st);
    if (mode == 1) return launch_chain_k<1>(ctx, a, n, k, st);
    if (k == 0) return fail(ctx, RV_ERR_ARG, "nothing to do (no CLAHE, no median)");
    return launch_chain_k<2>(ctx, a, n, k, st);
}

int launch_hist(rv_ctx *ctx, const uint8_t *src, size_t pitch, size_t fstride, const Geo &g, int space, int n,
                int32_t *hist, uint8_t *luma, int32_t *mm, cudaStream_t st)
{
    const int tiles = g.grid * g.grid;
    if (mm) {
        k_init_minmax<<<(n + 127) / 128, 128, 0, st>>>(mm, n);
        ctx->launches++;
    }
    // enough CTAs to fill the machine a few times over; slices of a tile accumulate with global atomics
    int slices = 1;
    const long want = 4L * ctx->sm_count;
    if ((long)tiles * n < want) slices = (int)std::min<long>((want + (long)tiles * n - 1) / ((long)tiles * n), std::max(1, g.th / 8));
    const int rps = (g.th + slices - 1) / slices;
    slices = (g.th + rps - 1) / rps;
    if (slices > 1) CK(cudaMemsetAsync(hist, 0, (size_t)n * tiles * 256 * sizeof(int32_t), st));
    // tiles on gridDim.x (up to 256 x 256 of them), slices on y, frames on z in groups
    for (int f0 = 0; f0 < n; f0 += MAX_FRAMES_PER_LAUNCH) {
        const int nf = std::min(MAX_FRAMES_PER_LAUNCH, n - f0);
        dim3 grid(tiles, slices, nf);
        const uint8_t *s0 = src + (size_t)f0 * fstride;
        int32_t *h0 = hist + (size_t)f0 * tiles * 256;
        uint8_t *l0 = luma ? luma + (size_t)f0 * g.H * g.W : nullptr;
        int32_t *m0 = mm ? mm + 2 * (size_t)f0 : nullptr;
        ScopedTiming tm(ctx, st, 0);
        const bool extra = luma != nullptr || mm != nullptr;
        if (space == RV_SPACE_LAB) {
            if (extra) k_luma_hist<1, true><<<grid, HIST_THREADS, 0, st>>>(s0, pitch, fstride, g, rps, h0, l0, m0);
            else k_luma_hist<1, false><<<grid, HIST_THREADS, 0, st>>>(s0, pitch, fstride, g, rps, h0, l0, m0);
        } else {
            if (extra) k_luma_hist<0, true><<<grid, HIST_THREADS, 0, st>>>(s0, pitch, fstride, g, rps, h0, l0, m0);
            else k_luma_hist<0, false><<<grid, HIST_THREADS, 0, st>>>(s0, pitch, fstride, g, rps, h0, l0, m0);
        }
        ctx->launches++;
    }
    CK(cudaGetLastError());
    return RV_OK;
}

int launch_lut(rv_ctx *ctx, const int32_t *hist, const Geo &g, double clip_limit, int n, uint8_t *lut, uint32_t *quads,
               cudaStream_t st)
{
    const int clip = clip_int(clip_limit, g);
    const float lut_scale = 255.0f / (float)(g.tw * g.th);
    const size_t tiles = (size_t)g.grid * g.grid, nq = (size_t)(g.grid + 1) * (g.grid + 1);
    for (int f0 = 0; f0 < n; f0 += MAX_FRAMES_PER_LAUNCH) {
        const int nf = std::min(MAX_FRAMES_PER_LAUNCH, n - f0);
        const int32_t *h0 = hist + (size_t)f0 * tiles * 256;
        uint8_t *l0 = lut ? lut + (size_t)f0 * tiles * 256 : nullptr;
        uint32_t *q0 = quads + (size_t)f0 * nq * 256;
        ScopedTiming tm(ctx, st, 1);
        if (g.grid <= LUT_ROWS_MAX_GRID)
            k_build_lut_rows<<<dim3(g.grid + 1, nf), 64 * g.grid, 0, st>>>(h0, g.grid, clip, lut_scale, l0, q0);
        else
            k_build_lut<<<dim3((g.grid + 1) * (g.grid + 1), nf), 128, 0, st>>>(h0, g.grid, clip, lut_scale, l0, q0);
        ctx->launches++;
    }
    CK(cudaGetLastError());
    return RV_OK;
}

// A geometry table is uploaded on the stream that first needs it (page-locked host copy kept with the entry) and is read-only
// afterwards; other streams wait for the upload event.  Nothing synchronises the device.
void drop_frame_graphs(rv_ctx *ctx)
{
    for (FrameGraph &g : ctx->fgraphs) {
        if (g.exec) cudaGraphExecDestroy(g.exec);
        if (g.graph) cudaGraphDestroy(g.graph);
    }
    ctx->fgraphs.clear();
}

int flush_tables(rv_ctx *ctx)
{
    CK(cudaDeviceSynchronize());            // rare: more than MAX_TABS geometries seen by one context
    drop_frame_graphs(ctx);                 // they reference the column records
    for (ColTab &t : ctx->coltabs) { cudaFree(t.dev); cudaFreeHost(t.host); cudaEventDestroy(t.ready); }
    for (LbTab &t : ctx->lbtabs) { cudaFree(t.dev); cudaFreeHost(t.host); cudaEventDestroy(t.ready); }
    ctx->coltabs.clear();
    ctx->lbtabs.clear();
    return RV_OK;
}

// Column records for k_chain (A.3 horizontal terms), built once per (W, tile width).  Record r describes
// the four pixels 4*(r-1) .. 4*(r-1)+3 (clamped into the frame): xa, xa1 = 1 - xa, -2^23*xa, -2^23*xa1, quad column.
// Every value is produced by single IEEE-754 binary32 operations, exactly as the kernel used to compute them.
int get_colparams(rv_ctx *ctx, const Geo &g, cudaStream_t st, const float **out, bool capturing = false)
{
    for (ColTab &t : ctx->coltabs)
        if (t.w == g.W && t.tw == g.tw) {
            // (while capturing, the same stream has already waited for the upload in the direct run that precedes the capture)
            if (t.up != st && !capturing) CK(cudaStreamWaitEvent(st, t.ready, 0));
            *out = t.dev;
            return RV_OK;
        }
    if ((int)ctx->coltabs.size() >= MAX_TABS) RV_TRY(flush_tables(ctx));
    const int ngroups = (TILE_W / 4) * ((g.W + TILE_W - 1) / TILE_W) + 34;
    const size_t bytes = (size_t)ngroups * 20 * 4;
    ColTab t;
    t.w = g.W; t.tw = g.tw; t.up = st;
    CK(cudaHostAlloc((void **)&t.host, bytes, cudaHostAllocDefault));
    if (cudaMalloc((void **)&t.dev, bytes) != cudaSuccess) { cudaFreeHost(t.host); return fail(ctx, RV_ERR_NOMEM, "cudaMalloc(column records)"); }
    if (cudaEventCreateWithFlags(&t.ready, cudaEventDisableTiming) != cudaSuccess) { cudaFree(t.dev); cudaFreeHost(t.host); return fail(ctx, RV_ERR_CUDA, "cudaEventCreate"); }
    for (int r = 0; r < ngroups; ++r)
        for (int j = 0; j < 4; ++j) {
            const int cx = std::min(std::max(4 * (r - 1) + j, 0), g.W - 1);
            volatile float tt = (float)cx * g.inv_tw;
            volatile float txf = tt - 0.5f;
            const float fl = floorf(txf);
            volatile float xa = txf - fl;
            volatile float xa1 = 1.0f - xa;
            float *rec = &t.host[(size_t)r * 20];
            rec[j] = xa; rec[4 + j] = xa1; rec[8 + j] = -8388608.0f * xa; rec[12 + j] = -8388608.0f * xa1;
            const int q = (int)fl + 1;
            memcpy(&rec[16 + j], &q, 4);
        }
    ctx->coltabs.push_back(t);
    CK(cudaMemcpyAsync(t.dev, t.host, bytes, cudaMemcpyHostToDevice, st));
    CK(cudaEventRecord(t.ready, st));
    *out = t.dev;
    return RV_OK;
}

// one group of frames, everything on device, on stream `st`, using workspace set `ws`
struct LbFused {            // fused detector-input stage of one group (integer down-scale only)
    uint16_t *out; int scale, S, top, left, write_full;
};

int run_group(rv_ctx *ctx, int ws, const uint8_t *din, size_t ipitch, size_t ifs, uint8_t *dout, size_t opitch, size_t ofs,
              int n, int h, int w, const rv_params *p, cudaStream_t st, int32_t **flags_out, const LbFused *lb = nullptr,
              cudaStream_t st_pre = nullptr, cudaEvent_t ev_pre = nullptr, bool capturing = false, bool copy_skipped = true)
{
    // capturing: `st` is in stream capture (single-frame graph): nothing may allocate, wait for or record outside events; the
    // set WS_FRAME is only ever used on that one stream, so it needs no cross-stream ordering
    // st_pre (optional): histogram / LUT / gate flags run there and `st` waits for them before k_chain
    cudaStream_t sp = st_pre ? st_pre : st;
    // the previous user of this workspace set may have been on another stream (two caller streams, or a stage-level call)
    WsSync &wsy = ctx->wsync[ws];
    if (!capturing) {
        RV_TRY(ws_acquire(ctx, wsy, sp));
        if (st != sp) RV_TRY(ws_acquire(ctx, wsy, st));
    }
    ChainArgs a;
    a.src = din; a.spitch = ipitch; a.sfstride = ifs;
    a.dst = dout; a.dpitch = opitch; a.dfstride = ofs;
    a.quads = nullptr; a.flags = nullptr; a.use_tma = 0; a.prefetch_dist = 0; a.colp = nullptr;
    a.lb_out = lb ? lb->out : nullptr; a.lb_scale = lb ? lb->scale : 0; a.lb_S = lb ? lb->S : 0;
    a.lb_top = lb ? lb->top : 0; a.lb_left = lb ? lb->left : 0; a.write_full = lb ? lb->write_full : 1;
    if (flags_out) *flags_out = nullptr;
    if (!p->clahe) {
        a.g = make_geo(h, w, 2);
        // gate without CLAHE: still needs the gray span
        if (p->gate_enable) {
            RV_TRY(ensure(ctx, ctx->hist[ws], (size_t)n * 4 * 256 * 4));
            RV_TRY(ensure(ctx, ctx->mm[ws], (size_t)n * 8));
            RV_TRY(ensure(ctx, ctx->flags[ws], (size_t)n * 4));
            RV_TRY(launch_hist(ctx, din, ipitch, ifs, a.g, RV_SPACE_YCRCB, n, (int32_t *)ctx->hist[ws].p, nullptr,
                               (int32_t *)ctx->mm[ws].p, sp));
            launch_gate_flags(ctx, (int32_t *)ctx->mm[ws].p, n, p->gate_thresh, (int32_t *)ctx->flags[ws].p, sp);
            a.flags = (int32_t *)ctx->flags[ws].p;
        }
        RV_TRY(launch_chain(ctx, 2, a, n, p->ksize, st));
    } else {
        const Geo g = make_geo(h, w, p->grid);
        a.g = g;
        const size_t tiles = (size_t)g.grid * g.grid, nq = (size_t)(g.grid + 1) * (g.grid + 1);
        RV_TRY(ensure(ctx, ctx->hist[ws], (size_t)n * tiles * 256 * 4));
        RV_TRY(ensure(ctx, ctx->quads[ws], (size_t)n * nq * 256 * 4));
        int32_t *mm = nullptr;
        if (p->gate_enable) {
            RV_TRY(ensure(ctx, ctx->mm[ws], (size_t)n * 8));
            RV_TRY(ensure(ctx, ctx->flags[ws], (size_t)n * 4));
            mm = (int32_t *)ctx->mm[ws].p;
        }
        RV_TRY(launch_hist(ctx, din, ipitch, ifs, g, p->space, n, (int32_t *)ctx->hist[ws].p, nullptr, mm, sp));
        RV_TRY(launch_lut(ctx, (int32_t *)ctx->hist[ws].p, g, p->clip_limit, n, nullptr, (uint32_t *)ctx->quads[ws].p, sp));
        if (p->gate_enable) {
            launch_gate_flags(ctx, mm, n, p->gate_thresh, (int32_t *)ctx->flags[ws].p, sp);
            a.flags = (int32_t *)ctx->flags[ws].p;
        }
        a.quads = (uint32_t *)ctx->quads[ws].p;
        if (st_pre) {
            CK(cudaEventRecord(ev_pre, st_pre));
            CK(cudaStreamWaitEvent(st, ev_pre, 0));
        }
        RV_TRY(get_colparams(ctx, g, st, &a.colp, capturing));
        RV_TRY(launch_chain(ctx, p->space == RV_SPACE_LAB ? 1 : 0, a, n, p->ksize, st));
    }
    if (a.flags) {
        for (int f0 = 0; copy_skipped && f0 < n; f0 += MAX_FRAMES_PER_LAUNCH) {
            dim3 grid(4, std::min(h, 64), std::min(MAX_FRAMES_PER_LAUNCH, n - f0));
            k_gate_copy<<<grid, 256, 0, st>>>(din + (size_t)f0 * ifs, ipitch, ifs, dout + (size_t)f0 * ofs, opitch, ofs, h, 3 * w,
                                              a.flags + f0);
            ctx->launches++;
        }
        if (flags_out) *flags_out = (int32_t *)ctx->flags[ws].p;
    }
    CK(cudaGetLastError());
    if (capturing) return RV_OK;
    return ws_release(ctx, wsy, st);        // (a caller that reads the flags afterwards releases the set again)
}

long auto_group(const rv_ctx *ctx, int h, int w)
{
    if (ctx->group_frames > 0) return ctx->group_frames;
    // The chain is instruction-bound, not DRAM-bound (profiles/), so a group is as large as the
    // workspaces comfortably allow: three launches per batch, no tail effects between small groups.
    const size_t fb = (size_t)3 * w * h;
    return std::max<long>(1, std::min<long>(256, (long)(((size_t)1 << 30) / fb)));
}

long auto_chunk(const rv_ctx *ctx, int h, int w)
{
    if (ctx->chunk_frames > 0) return ctx->chunk_frames;
    const size_t fb = (size_t)3 * w * h;
    return std::max<long>(1, (long)((24u << 20) / fb));
}

}  // namespace

int rv::chain_device(rv_ctx *ctx, const uint8_t *in, uint8_t *out, int n, int h, int w, size_t ipitch, size_t opitch,
                     const rv_params *p, int32_t *processed_host, cudaStream_t st, bool copy_skipped)
{
    const size_t ifs = ipitch * h, ofs = opitch * h;
    // Overlap: the batch is cut into a few groups; histogram + LUT of group i+1 run on a high-priority side stream while
    // k_chain of group i (instruction bound, memory system idle) owns the SMs.  Two workspace sets alternate.
    const bool overlap = ctx->overlap_groups > 1 && p->clahe && !p->gate_enable && !processed_host && n >= 2 * ctx->overlap_groups &&
                         ctx->group_frames == 0;
    if (overlap) {
        const int ng = (int)ctx->overlap_groups;
        const int per = (n + ng - 1) / ng;
        CK(cudaEventRecord(ctx->ev_entry, st));
        CK(cudaStreamWaitEvent(ctx->aux, ctx->ev_entry, 0));
        int gi = 0;
        for (int f0 = 0; f0 < n; f0 += per, ++gi) {
            const int g = std::min(per, n - f0);
            const int ws = NPIPE + (gi & 1);
            if (gi >= 2) CK(cudaStreamWaitEvent(ctx->aux, ctx->ev_chain[gi & 1], 0));      // workspace `ws` free again
            RV_TRY(run_group(ctx, ws, in + (size_t)f0 * ifs, ipitch, ifs, out + (size_t)f0 * ofs, opitch, ofs, g, h, w, p, st, nullptr,
                             nullptr, ctx->aux, ctx->ev_pre[gi & 1]));
            CK(cudaEventRecord(ctx->ev_chain[gi & 1], st));
        }
        return RV_OK;
    }
    const long G = auto_group(ctx, h, w);
    for (int f0 = 0; f0 < n; f0 += (int)G) {
        const int g = (int)std::min<long>(G, n - f0);
        int32_t *flags = nullptr;
        RV_TRY(run_group(ctx, NPIPE, in + (size_t)f0 * ifs, ipitch, ifs, out + (size_t)f0 * ofs, opitch, ofs, g, h, w, p, st, &flags,
                         nullptr, nullptr, nullptr, false, copy_skipped));
        if (processed_host) {
            if (flags) {
                CK(cudaMemcpyAsync(processed_host + f0, flags, (size_t)g * 4, cudaMemcpyDeviceToHost, st));
                CK(cudaStreamSynchronize(st));      // the workspace is reused by the next group
            } else {
                for (int i = 0; i < g; ++i) processed_host[f0 + i] = 1;
            }
        }
    }
    return RV_OK;
}

namespace {

int wait_all(rv_ctx *ctx)
{
    for (int i = 0; i < NPIPE; ++i) CK(cudaStreamSynchronize(ctx->pipe[i]));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaStreamSynchronize(ctx->aux));
    if (ctx->fstream) CK(cudaStreamSynchronize(ctx->fstream));
    return RV_OK;
}

// stage-level helper: bring an input to the device if it is on the host
struct Staged {
    rv_ctx *ctx;
    void *dev = nullptr;
    bool owned = false;
    ~Staged() { if (owned && dev) cudaFree(dev); }
};

int stage_in(rv_ctx *ctx, Staged &s, const void *p, size_t bytes, int mem_kind)
{
    s.ctx = ctx;
    if (mem_kind == RV_MEM_DEVICE) { s.dev = const_cast<void *>(p); return RV_OK; }
    CK(cudaMalloc(&s.dev, std::max<size_t>(bytes, 16)));
    s.owned = true;
    CK(cudaMemcpyAsync(s.dev, p, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return RV_OK;
}

int stage_out(rv_ctx *ctx, Staged &s, void *p, size_t bytes, int mem_kind)
{
    s.ctx = ctx;
    if (mem_kind == RV_MEM_DEVICE) { s.dev = p; return RV_OK; }
    CK(cudaMalloc(&s.dev, std::max<size_t>(bytes, 16)));
    s.owned = true;
    return RV_OK;
}

int finish_out(rv_ctx *ctx, Staged &s, void *p, size_t bytes, int mem_kind)
{
    if (mem_kind != RV_MEM_DEVICE && p) CK(cudaMemcpyAsync(p, s.dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return RV_OK;
}

// ---- detector-input stage (SURVEY.md 8f-1) ------------------------------------------------------------
struct LbGeo { int S, nw, nh, top, left, scale; };    // scale > 0: exact integer down-scale (fusable)

// ultralytics-style square letterbox: r = min(S/h, S/w); new = round(w r) x round(h r) (Python round = half to even);
// padding split with the -0.1 / +0.1 rounding so odd remainders put the extra row/column at the bottom/right.
LbGeo lb_geometry(int h, int w, int S)
{
    LbGeo g;
    g.S = S;
    const double r = std::min((double)S / h, (double)S / w);
    g.nw = std::max(1, (int)nearbyint(w * r));
    g.nh = std::max(1, (int)nearbyint(h * r));
    const double dw = (S - g.nw) / 2.0, dh = (S - g.nh) / 2.0;
    g.top = (int)nearbyint(dh - 0.1);
    g.left = (int)nearbyint(dw - 0.1);
    g.scale = 0;
    if (w % g.nw == 0 && h % g.nh == 0 && w / g.nw == h / g.nh) {
        const int sc = w / g.nw;
        const bool x_ok = TILE_W % sc == 0;
        const bool y_ok = (sc & 1) || TILE_H % sc == 0 || (((sc >> 1) - 1) & 1) == 0;
        if (sc >= 1 && x_ok && y_ok) g.scale = sc;
    }
    return g;
}

// cv2.resize(INTER_LINEAR) tables for 8-bit data (resize.cpp): x clamps with the fraction forced to 0,
// y keeps the fraction and clips the two row indices; coefficients are cvRound(c * 2048) as shorts.
void lb_tables(int ssize, int dsize, bool is_x, int32_t *ofs, int16_t *coef)
{
    const double scale = 1.0 / ((double)dsize / ssize);
    for (int d = 0; d < dsize; ++d) {
        float f = (float)((d + 0.5) * scale - 0.5);
        int sidx = (int)floorf(f);
        f -= (float)sidx;
        if (is_x) {
            if (sidx < 0) { sidx = 0; f = 0.f; }
            if (sidx >= ssize - 1) { sidx = ssize - 1; f = 0.f; }
            ofs[d] = sidx;
        } else {
            ofs[2 * d] = std::min(std::max(sidx, 0), ssize - 1);
            ofs[2 * d + 1] = std::min(std::max(sidx + 1, 0), ssize - 1);
        }
        coef[2 * d] = (int16_t)lrintf((1.f - f) * 2048.f);
        coef[2 * d + 1] = (int16_t)lrintf(f * 2048.f);
    }
}

// the four resize tables of one (h, w) -> (nh, nw) geometry, cached like the column records (see get_colparams)
int get_lbtab(rv_ctx *ctx, int h, int w, const LbGeo &g, cudaStream_t st, const LbTab **out)
{
    for (LbTab &t : ctx->lbtabs)
        if (t.h == h && t.w == w && t.nh == g.nh && t.nw == g.nw) {
            if (t.up != st) CK(cudaStreamWaitEvent(st, t.ready, 0));
            *out = &t;
            return RV_OK;
        }
    if ((int)ctx->lbtabs.size() >= MAX_TABS) RV_TRY(flush_tables(ctx));
    auto up16 = [](size_t v) { return (v + 15) & ~(size_t)15; };
    LbTab t;
    t.h = h; t.w = w; t.nh = g.nh; t.nw = g.nw; t.up = st;
    t.o_yofs = up16((size_t)g.nw * 4);
    t.o_xa = t.o_yofs + up16((size_t)2 * g.nh * 4);
    t.o_ya = t.o_xa + up16((size_t)2 * g.nw * 2);
    const size_t bytes = t.o_ya + up16((size_t)2 * g.nh * 2);
    CK(cudaHostAlloc((void **)&t.host, bytes, cudaHostAllocDefault));
    if (cudaMalloc((void **)&t.dev, bytes) != cudaSuccess) { cudaFreeHost(t.host); return fail(ctx, RV_ERR_NOMEM, "cudaMalloc(letterbox tables)"); }
    if (cudaEventCreateWithFlags(&t.ready, cudaEventDisableTiming) != cudaSuccess) { cudaFree(t.dev); cudaFreeHost(t.host); return fail(ctx, RV_ERR_CUDA, "cudaEventCreate"); }
    memset(t.host, 0, bytes);
    lb_tables(w, g.nw, true, (int32_t *)t.host, (int16_t *)(t.host + t.o_xa));
    lb_tables(h, g.nh, false, (int32_t *)(t.host + t.o_yofs), (int16_t *)(t.host + t.o_ya));
    ctx->lbtabs.push_back(t);
    CK(cudaMemcpyAsync(t.dev, t.host, bytes, cudaMemcpyHostToDevice, st));
    CK(cudaEventRecord(t.ready, st));
    *out = &ctx->lbtabs.back();
    return RV_OK;
}

int launch_letterbox(rv_ctx *ctx, const uint8_t *src, size_t pitch, size_t fstride, int n, int h, int w, const LbGeo &g,
                     int pad, bool only_pad, uint16_t *out, cudaStream_t st)
{
    LbArgs a;
    a.src = src; a.spitch = pitch; a.sfstride = fstride; a.out = out;
    a.H = h; a.W = w; a.S = g.S; a.nw = g.nw; a.nh = g.nh; a.top = g.top; a.left = g.left; a.pad = pad; a.only_pad = only_pad ? 1 : 0;
    a.xofs = nullptr; a.xa = nullptr; a.yofs = nullptr; a.ya = nullptr;
    if (!only_pad) {
        const LbTab *t = nullptr;
        RV_TRY(get_lbtab(ctx, h, w, g, st, &t));
        a.xofs = (const int32_t *)t->dev; a.yofs = (const int32_t *)(t->dev + t->o_yofs);
        a.xa = (const int16_t *)(t->dev + t->o_xa); a.ya = (const int16_t *)(t->dev + t->o_ya);
    }
    for (int f0 = 0; f0 < n; f0 += MAX_FRAMES_PER_LAUNCH) {
        LbArgs b = a;
        if (b.src) b.src += (size_t)f0 * fstride;
        b.out += (size_t)f0 * 3 * g.S * g.S;
        dim3 grid((g.S + 31) / 32, (g.S + 7) / 8, std::min(MAX_FRAMES_PER_LAUNCH, n - f0)), block(32, 8);
        k_letterbox<<<grid, block, 0, st>>>(b);
        ctx->launches++;
    }
    CK(cudaGetLastError());
    return RV_OK;
}

// ---- the chunked pipeline for jobs that touch host memory ----------------------------------------------------
// Chunks of frames flow  H2D -> kernels -> D2H  on NPIPE streams, so the copies of consecutive chunks overlap with each other
// and with the kernels.  Every end of the job may independently live on the host or on the device: a device input skips the
// H2D, a device output / tensor skips its D2H (results that the next stage consumes on the same GPU never cross PCIe).
struct PipeJob {
    const uint8_t *in = nullptr; int in_kind = RV_MEM_HOST; size_t ipitch = 0;
    int yuv = 0;                            // RV_YUV_NV12 / RV_YUV_I420: 4:2:0 frames in, converted into the BGR workspace first; 0 = BGR
    uint8_t *out = nullptr; int out_kind = RV_MEM_HOST; size_t opitch = 0;      // full-resolution result; nullptr = not wanted
    uint16_t *lb = nullptr; int lb_kind = RV_MEM_HOST; int S = 0, pad = 114;     // detector tensor; nullptr = none
    bool lb_rows_only = false;              // host tensor whose padding rows the caller already holds: copy back the image rows only
    int32_t *processed = nullptr;                                               // host, optional
};

// Frames in chunk number `chunk` of a host job of n frames cut into chunks of at most C, `left` frames still to go (see the comment
// on the schedule in chain_pipe; rv_chunk_schedule exposes it to the CPU tests).
long chunk_frames_at(long C, bool taper, long n, int chunk, long left)
{
    long want = C;
    if (taper && C >= 2 && n > 3 * C) {
        const long Cs = std::max<long>(1, C / 3);
        if (chunk == 0) want = Cs;
        else if (chunk == 1) want = std::max<long>(Cs, 2 * C / 3);
        else if (left > Cs && left <= C + Cs) want = left - Cs;          // the last two chunks: (rest - C/3, C/3)
    }
    return std::min<long>(want, left);
}

int chain_pipe(rv_ctx *ctx, const PipeJob &j, int n, int h, int w, const rv_params *p)
{
    const long C = std::min<long>(std::min<long>(auto_chunk(ctx, h, w), std::max(1, n)), 4096);
    const size_t rowb = (size_t)3 * w;
    const size_t dpitch = (rowb + 15) & ~(size_t)15;
    const size_t dfs = dpitch * h;
    const bool in_dev = j.in_kind == RV_MEM_DEVICE, out_dev = j.out_kind == RV_MEM_DEVICE, lb_dev = j.lb_kind == RV_MEM_DEVICE;
    LbGeo lg = {};
    size_t lbf = 0;                                         // halves per frame of the detector tensor
    if (j.lb) {
        lg = lb_geometry(h, w, j.S);
        lbf = (size_t)3 * j.S * j.S;
    }
    const bool fused = j.lb && lg.scale > 0;
    const bool need_dfull = (j.out && !out_dev) || (j.lb && !fused && !(j.out && out_dev));   // a device staging copy of the full result
    // 4:2:0 chunks are uploaded at a pitch that k_yuv420_to_bgr's vector path can read (I420 planes stay packed)
    const size_t ypitch = j.yuv == RV_YUV_NV12 ? ((size_t)w + 7) & ~(size_t)7 : (size_t)w, yfs = ypitch * h * 3 / 2;
    for (int i = 0; i < NPIPE; ++i) {
        if (!in_dev || j.yuv) RV_TRY(ensure(ctx, ctx->din[i], dfs * C));
        if (j.yuv && !in_dev) RV_TRY(ensure(ctx, ctx->dyuv[i], yfs * C));
        if (need_dfull) RV_TRY(ensure(ctx, ctx->dout[i], dfs * C));
        if (j.lb && !lb_dev) RV_TRY(ensure(ctx, ctx->dlb[i], lbf * 2 * C));
    }
    // Chunk schedule.  Uniform chunks of C frames leave the D2H engine idle while the first chunk is uploaded and processed, and the
    // H2D engine idle while the last one comes back; with option "chunk_taper" the job starts and ends with smaller chunks
    // (C/3, 2C/3, C, ..., C, rest - C/3, C/3) so that both ends of the pipeline fill and drain in a third of the time.  Measured at
    // 64 x 1080p: +0.3 % full frames back, +0.8 % tensor rows back, +0.5 % nothing back (profiles/r2_ac_chunk_taper.jsonl) -- small,
    // because the legs sit at the PCIe link's duplex rate (43 GB/s each way), but consistent and free.
    const bool taper = ctx->chunk_taper != 0;
    int chunk = 0;
    for (int f0 = 0, g = 0; f0 < n; f0 += g, ++chunk) {
        const int s = chunk % NPIPE;
        g = (int)chunk_frames_at(C, taper, n, chunk, n - f0);
        cudaStream_t st = ctx->pipe[s];
        // input
        const uint8_t *di;
        size_t dip, difs;
        if (j.yuv) {
            const uint8_t *src = j.in + (size_t)f0 * j.ipitch * h * 3 / 2;
            size_t sp = j.ipitch;
            if (!in_dev) {
                uint8_t *y = (uint8_t *)ctx->dyuv[s].p;
                if (j.ipitch == ypitch)
                    CK(cudaMemcpyAsync(y, src, yfs * g, cudaMemcpyHostToDevice, st));
                else
                    CK(cudaMemcpy2DAsync(y, ypitch, src, j.ipitch, w, (size_t)h * 3 / 2 * g, cudaMemcpyHostToDevice, st));
                src = y; sp = ypitch;
            }
            RV_TRY(launch_yuv420(ctx, j.yuv, src, sp, (uint8_t *)ctx->din[s].p, dpitch, dfs, g, h, w, st));
            di = (const uint8_t *)ctx->din[s].p; dip = dpitch; difs = dfs;
        } else if (in_dev) {
            di = j.in + (size_t)f0 * j.ipitch * h; dip = j.ipitch; difs = j.ipitch * h;
        } else {
            uint8_t *d = (uint8_t *)ctx->din[s].p;
            if (j.ipitch == dpitch)
                CK(cudaMemcpyAsync(d, j.in + (size_t)f0 * j.ipitch * h, dfs * g, cudaMemcpyHostToDevice, st));
            else
                CK(cudaMemcpy2DAsync(d, dpitch, j.in + (size_t)f0 * j.ipitch * h, j.ipitch, rowb, (size_t)h * g, cudaMemcpyHostToDevice, st));
            di = d; dip = dpitch; difs = dfs;
        }
        // where the kernels write
        uint8_t *dfull = nullptr;
        size_t dop = dpitch, dofs = dfs;
        if (j.out && out_dev) { dfull = j.out + (size_t)f0 * j.opitch * h; dop = j.opitch; dofs = j.opitch * h; }
        else if (need_dfull) dfull = (uint8_t *)ctx->dout[s].p;
        uint16_t *dl = nullptr;
        if (j.lb) dl = lb_dev ? j.lb + (size_t)f0 * lbf : (uint16_t *)ctx->dlb[s].p;
        int32_t *flags = nullptr;
        if (fused) {
            LbFused lb = {dl, lg.scale, j.S, lg.top, lg.left, j.out ? 1 : 0};
            RV_TRY(launch_letterbox(ctx, nullptr, 0, 0, g, h, w, lg, j.pad, true, dl, st));
            RV_TRY(run_group(ctx, s, di, dip, difs, j.out ? dfull : (uint8_t *)dl, j.out ? dop : dip, j.out ? dofs : difs, g, h, w, p, st,
                             &flags, &lb));
        } else {
            RV_TRY(run_group(ctx, s, di, dip, difs, dfull, dop, dofs, g, h, w, p, st, &flags));
            if (j.lb) RV_TRY(launch_letterbox(ctx, dfull, dop, dofs, g, h, w, lg, j.pad, false, dl, st));
        }
        // results
        if (j.out && !out_dev) {
            if (j.opitch == dpitch)
                CK(cudaMemcpyAsync(j.out + (size_t)f0 * j.opitch * h, dfull, dfs * g, cudaMemcpyDeviceToHost, st));
            else
                CK(cudaMemcpy2DAsync(j.out + (size_t)f0 * j.opitch * h, j.opitch, dfull, dpitch, rowb, (size_t)h * g, cudaMemcpyDeviceToHost, st));
        }
        if (j.lb && !lb_dev) {
            if (j.lb_rows_only && lg.nh < j.S) {
                // rows [top, top + nh) of each of the 3 g planes are one contiguous run: a strided copy skips the constant padding rows
                // (44 % of a 1080p -> 640 x 640 tensor), which the caller's buffer already holds
                const size_t plane = (size_t)j.S * j.S * 2, off = (size_t)lg.top * j.S;
                CK(cudaMemcpy2DAsync(j.lb + (size_t)f0 * lbf + off, plane, dl + off, plane, (size_t)lg.nh * j.S * 2, (size_t)3 * g,
                                     cudaMemcpyDeviceToHost, st));
            } else {
                CK(cudaMemcpyAsync(j.lb + (size_t)f0 * lbf, dl, lbf * 2 * g, cudaMemcpyDeviceToHost, st));
            }
        }
        if (j.processed) {
            if (flags) CK(cudaMemcpyAsync(j.processed + f0, flags, (size_t)g * 4, cudaMemcpyDeviceToHost, st));
            else for (int i = 0; i < g; ++i) j.processed[f0 + i] = 1;
        }
        RV_TRY(ws_release(ctx, ctx->wsync[s], st));
    }
    return RV_OK;
}

// ---- the single-frame path: `proc = pipeline(raw)` (main_preview.py:94), one frame in flight, lowest latency --------------
// Host rows are contiguous (pitch 3w).  H2D copy, one graph launch (or the direct launches), D2H copy, one synchronisation.
int frame_kernels(rv_ctx *ctx, int h, int w, const rv_params *p, bool capturing)
{
    cudaStream_t st = ctx->fstream;
    const size_t pitch = (size_t)3 * w, fs = pitch * h;
    int32_t *flags = nullptr;
    RV_TRY(run_group(ctx, WS_FRAME, (const uint8_t *)ctx->din[WS_FRAME].p, pitch, fs, (uint8_t *)ctx->dout[WS_FRAME].p, pitch, fs, 1, h, w, p,
                     st, &flags, nullptr, nullptr, nullptr, capturing));
    if (flags) CK(cudaMemcpyAsync(ctx->fflag, flags, 4, cudaMemcpyDeviceToHost, st));
    return RV_OK;
}

void frame_bufs(rv_ctx *ctx, void *(&b)[6])
{
    b[0] = ctx->din[WS_FRAME].p; b[1] = ctx->dout[WS_FRAME].p; b[2] = ctx->hist[WS_FRAME].p;
    b[3] = ctx->quads[WS_FRAME].p; b[4] = ctx->mm[WS_FRAME].p; b[5] = ctx->flags[WS_FRAME].p;
}

// H2D of the frame of the single-frame path.  Page-locked input: one DMA.  Pageable input of at least 1.5 MB: staged through a
// page-locked frame by the caller and the helper threads, slice by slice, each slice's DMA issued as soon as it is staged.
int frame_upload(rv_ctx *ctx, const uint8_t *in, size_t fb, cudaStream_t st)
{
    uint8_t *din = (uint8_t *)ctx->din[WS_FRAME].p;
    bool pageable = false;
    if (ctx->stage_threads > 0 && fb >= (1536u << 10)) {
        cudaPointerAttributes attr;
        if (cudaPointerGetAttributes(&attr, in) == cudaSuccess) pageable = attr.type == cudaMemoryTypeUnregistered;
        else (void)cudaGetLastError();
    }
    if (!pageable) {
        CK(cudaMemcpyAsync(din, in, fb, cudaMemcpyHostToDevice, st));
        return RV_OK;
    }
    if (ctx->fstage.cap < fb) {
        CK(cudaStreamSynchronize(st));
        if (ctx->fstage.p) CK(cudaFreeHost(ctx->fstage.p));
        ctx->fstage.p = nullptr; ctx->fstage.cap = 0;
        cudaError_t e = cudaHostAlloc((void **)&ctx->fstage.p, fb, cudaHostAllocDefault);
        if (e != cudaSuccess) return fail(ctx, RV_ERR_NOMEM, "cudaHostAlloc(%zu): %s", fb, cudaGetErrorString(e));
        ctx->fstage.cap = fb;
    }
    if (!ctx->stage) {
        ctx->stage = new (std::nothrow) StagePool();
        if (!ctx->stage) return fail(ctx, RV_ERR_NOMEM, "staging pool");
        ctx->stage->start((int)std::min<long>(ctx->stage_threads, 15));
    }
    StagePool &sp = *ctx->stage;
    // (the previous frame's DMAs out of the staging frame finished: every call ends with a stream synchronisation)
    const int nsl = (int)std::min<size_t>(StagePool::MAX_SLICES, std::max<size_t>(2, fb / (768u << 10)));
    for (;;) {
        std::unique_lock<std::mutex> lk(sp.m);
        if (sp.active.load(std::memory_order_acquire) != 0) {           // a helper is still leaving the previous job's loop
            lk.unlock();
            std::this_thread::yield();
            continue;
        }
        sp.src = in; sp.dst = ctx->fstage.p; sp.bytes = fb;
        sp.slice = ((fb + nsl - 1) / nsl + 63) & ~(size_t)63;
        sp.nslices = (int)((fb + sp.slice - 1) / sp.slice);
        for (int i = 0; i < sp.nslices; ++i) sp.done[i].store(0, std::memory_order_relaxed);
        sp.next.store(0, std::memory_order_relaxed);
        ++sp.gen;
        break;
    }
    sp.cv.notify_all();
    cudaError_t err = cudaSuccess;
    for (int s = 0; s < sp.nslices; ++s) {
        while (!sp.done[s].load(std::memory_order_acquire)) {
            if (sp.next.load(std::memory_order_relaxed) < sp.nslices) sp.copy_some_one();
            else std::this_thread::yield();
        }
        // after a failed DMA the loop only waits for the helpers: they read the caller's frame until every slice is staged
        const size_t off = (size_t)s * sp.slice, len = std::min(sp.slice, fb - off);
        if (err == cudaSuccess) err = cudaMemcpyAsync(din + off, ctx->fstage.p + off, len, cudaMemcpyHostToDevice, st);
    }
    if (err != cudaSuccess) return fail(ctx, RV_ERR_CUDA, "staged upload failed: %s", cudaGetErrorString(err));
    return RV_OK;
}

int chain_frame(rv_ctx *ctx, const uint8_t *in, uint8_t *out, int h, int w, const rv_params *p, int32_t *processed)
{
    cudaStream_t st = ctx->fstream;
    const size_t fb = (size_t)3 * w * h;
    RV_TRY(ensure(ctx, ctx->din[WS_FRAME], fb));
    RV_TRY(ensure(ctx, ctx->dout[WS_FRAME], fb));
    RV_TRY(frame_upload(ctx, in, fb, st));
    *ctx->fflag = 1;
    FrameGraph *fg = nullptr;
    const bool use_graph = ctx->frame_graphs != 0 && ctx->kernel_timing == 0;
    if (use_graph) {
        void *cur[6];
        frame_bufs(ctx, cur);
        for (size_t i = 0; i < ctx->fgraphs.size(); ++i) {
            FrameGraph &g = ctx->fgraphs[i];
            if (g.h == h && g.w == w && memcmp(&g.p, p, sizeof *p) == 0) {
                if (memcmp(g.bufs, cur, sizeof cur) == 0) { fg = &g; break; }
                cudaGraphExecDestroy(g.exec);            // a workspace was reallocated since the capture: stale pointers
                cudaGraphDestroy(g.graph);
                ctx->fgraphs.erase(ctx->fgraphs.begin() + i);
                break;
            }
        }
    }
    if (fg) {
        CK(cudaGraphLaunch(fg->exec, st));
        ctx->launches += fg->kernels;
    } else {
        // first frame of this (shape, parameters): direct launches (they size the workspaces and upload the tables) ...
        RV_TRY(frame_kernels(ctx, h, w, p, false));
    }
    CK(cudaMemcpyAsync(out, ctx->dout[WS_FRAME].p, fb, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (processed) *processed = *ctx->fflag;
    if (!fg && use_graph) {
        // ... then the same sequence is captured for the frames that follow (nothing allocates or waits any more)
        if ((int)ctx->fgraphs.size() >= MAX_FRAME_GRAPHS) drop_frame_graphs(ctx);
        FrameGraph g;
        g.h = h; g.w = w; g.p = *p;
        if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
            const long launches = ctx->launches;
            const int rc = frame_kernels(ctx, h, w, p, true);
            g.kernels = ctx->launches - launches;
            ctx->launches = launches;                                   // captured, not launched
            cudaError_t e = cudaStreamEndCapture(st, &g.graph);
            if (rc == RV_OK && e == cudaSuccess && g.graph && cudaGraphInstantiate(&g.exec, g.graph, 0) == cudaSuccess) {
                frame_bufs(ctx, g.bufs);
                ctx->fgraphs.push_back(g);
            } else {
                if (g.graph) cudaGraphDestroy(g.graph);
                (void)cudaGetLastError();                               // the direct path keeps working without a graph
            }
        } else {
            (void)cudaGetLastError();
        }
    }
    return RV_OK;
}

int check_lb_args(rv_ctx *ctx, const void *tensor, int S, int pad_value)
{
    if (!tensor || S < 1 || S > 8192 || pad_value < 0 || pad_value > 255) return fail(ctx, RV_ERR_ARG, "bad letterbox arguments");
    return RV_OK;
}

}  // namespace

int rv_internal_device(const rv_ctx *ctx) { return ctx->device; }
void *rv_internal_stream(rv_ctx *ctx) { return ctx->stream; }
void rv_internal_count_launches(rv_ctx *ctx, long n) { ctx->launches += n; }
void *rv_internal_get_fog(rv_ctx *ctx) { return ctx->fog; }
void rv_internal_set_fog(rv_ctx *ctx, void *state, void (*destroy)(void *)) { ctx->fog = state; ctx->fog_destroy = destroy; }
U16Ws &rv_internal_u16(rv_ctx *ctx) { return ctx->u16; }
ChWs &rv_internal_ch(rv_ctx *ctx) { return ctx->ch; }

extern "C" {

const char *rv_version(void) { return "rv_b200 0.1 (sm_100a)"; }

int rv_ycc_table(uint32_t *out1024)
{
    if (!out1024) return RV_ERR_ARG;
    YccTabs y;
    build_ycc_table(y);
    memcpy(out1024, y.e, sizeof y.e);
    return RV_OK;
}

int rv_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int rv_create(int device, rv_ctx **out)
{
    if (!out) return RV_ERR_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return RV_ERR_NODEV;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return RV_ERR_NODEV;
    if (prop.major != 10) return RV_ERR_NODEV;              // sm_100a code only; no other backend, no CPU fallback
    if (cudaSetDevice(device) != cudaSuccess) return RV_ERR_CUDA;
    rv_ctx *ctx = new (std::nothrow) rv_ctx();
    if (!ctx) return RV_ERR_NOMEM;
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return RV_ERR_CUDA; }
    for (int i = 0; i < NPIPE; ++i)
        if (cudaStreamCreateWithFlags(&ctx->pipe[i], cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return RV_ERR_CUDA; }
    {
        int lo = 0, hi = 0;
        cudaDeviceGetStreamPriorityRange(&lo, &hi);
        if (cudaStreamCreateWithPriority(&ctx->aux, cudaStreamNonBlocking, hi) != cudaSuccess) { delete ctx; return RV_ERR_CUDA; }
        cudaEvent_t *evs[] = {&ctx->ev_entry, &ctx->ev_pre[0], &ctx->ev_pre[1], &ctx->ev_chain[0], &ctx->ev_chain[1]};
        for (cudaEvent_t *e : evs)
            if (cudaEventCreateWithFlags(e, cudaEventDisableTiming) != cudaSuccess) { delete ctx; return RV_ERR_CUDA; }
        for (WsSync &w : ctx->wsync)
            if (cudaEventCreateWithFlags(&w.ev, cudaEventDisableTiming) != cudaSuccess) { delete ctx; return RV_ERR_CUDA; }
        if (cudaEventCreateWithFlags(&ctx->u16.sync.ev, cudaEventDisableTiming) != cudaSuccess) { delete ctx; return RV_ERR_CUDA; }
        if (cudaEventCreateWithFlags(&ctx->ch.sync.ev, cudaEventDisableTiming) != cudaSuccess) { delete ctx; return RV_ERR_CUDA; }
        if (cudaStreamCreateWithFlags(&ctx->fstream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return RV_ERR_CUDA; }
        if (cudaHostAlloc((void **)&ctx->fflag, 64, cudaHostAllocDefault) != cudaSuccess) { delete ctx; return RV_ERR_NOMEM; }
    }
    // LAB tables
    LabTabs *t = new (std::nothrow) LabTabs();
    if (!t) { delete ctx; return RV_ERR_NOMEM; }
    memset(t, 0, sizeof *t);
    memcpy(t->g8, RV_LAB_G8, sizeof RV_LAB_G8);
    memcpy(t->yt, RV_LAB_YT, sizeof RV_LAB_YT);
    for (int i = 0; i < 256; ++i) t->ft[i] = (uint16_t)(RV_LAB_FT[i] + RV_LAB_FT_BIAS);     // <= 16384 + 10484
    memcpy(t->cb, RV_LAB_CB, sizeof RV_LAB_CB);
    memcpy(t->ig, RV_LAB_IG, sizeof RV_LAB_IG);
    cudaError_t e = cudaMemcpyToSymbol(g_lab, t, sizeof *t);
    delete t;
    if (e != cudaSuccess) { delete ctx; return RV_ERR_CUDA; }
    {
        LabHistTabs lh;
        build_lab_hist_table(lh);
        if (cudaMemcpyToSymbol(g_labh, &lh, sizeof lh) != cudaSuccess) { delete ctx; return RV_ERR_CUDA; }
    }
    {
        YccTabs y;
        build_ycc_table(y);
        if (cudaMemcpyToSymbol(g_ycc, &y, sizeof y) != cudaSuccess) { delete ctx; return RV_ERR_CUDA; }
    }
    *out = ctx;
    return RV_OK;
}

void rv_destroy(rv_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    Buf *sets[] = {ctx->hist, ctx->quads, ctx->lut, ctx->flags, ctx->mm, ctx->din, ctx->dout};
    for (Buf *set : sets)
        for (int i = 0; i < NWS; ++i)
            if (set[i].p) cudaFree(set[i].p);
    for (Buf &b : ctx->dlb)
        if (b.p) cudaFree(b.p);
    for (Buf &b : ctx->dyuv)
        if (b.p) cudaFree(b.p);
    for (Buf *b : {&ctx->u16.lut, &ctx->u16.mid, &ctx->u16.din, &ctx->u16.dout, &ctx->u16.mm, &ctx->u16.flags})
        if (b->p) cudaFree(b->p);
    if (ctx->u16.hflags) cudaFreeHost(ctx->u16.hflags);
    for (Buf *b : {&ctx->ch.pack, &ctx->ch.din, &ctx->ch.dout, &ctx->ch.mm, &ctx->ch.flags})
        if (b->p) cudaFree(b->p);
    if (ctx->ch.hflags) cudaFreeHost(ctx->ch.hflags);
    if (ctx->scratch.p) cudaFree(ctx->scratch.p);
    if (ctx->lbfull.p) cudaFree(ctx->lbfull.p);
    for (ColTab &t : ctx->coltabs) { cudaFree(t.dev); cudaFreeHost(t.host); cudaEventDestroy(t.ready); }
    for (LbTab &t : ctx->lbtabs) { cudaFree(t.dev); cudaFreeHost(t.host); cudaEventDestroy(t.ready); }
    for (WsSync &w : ctx->wsync)
        if (w.ev) cudaEventDestroy(w.ev);
    if (ctx->u16.sync.ev) cudaEventDestroy(ctx->u16.sync.ev);
    if (ctx->ch.sync.ev) cudaEventDestroy(ctx->ch.sync.ev);
    drop_frame_graphs(ctx);
    if (ctx->stage) { ctx->stage->stop(); delete ctx->stage; }
    if (ctx->fstage.p) cudaFreeHost(ctx->fstage.p);
    if (ctx->fog && ctx->fog_destroy) ctx->fog_destroy(ctx->fog);
    if (ctx->fstream) cudaStreamDestroy(ctx->fstream);
    if (ctx->fflag) cudaFreeHost(ctx->fflag);
    for (const TimedLaunch &t : ctx->timed) { cudaEventDestroy(t.a); cudaEventDestroy(t.b); }
    for (cudaEvent_t e : ctx->ev_pool) cudaEventDestroy(e);
    for (int i = 0; i < NPIPE; ++i)
        if (ctx->pipe[i]) cudaStreamDestroy(ctx->pipe[i]);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    if (ctx->aux) cudaStreamDestroy(ctx->aux);
    cudaEvent_t evs[] = {ctx->ev_entry, ctx->ev_pre[0], ctx->ev_pre[1], ctx->ev_chain[0], ctx->ev_chain[1]};
    for (cudaEvent_t e : evs)
        if (e) cudaEventDestroy(e);
    delete ctx;
}

const char *rv_last_error(const rv_ctx *ctx) { return ctx ? ctx->err : "null context"; }

int rv_set_option(rv_ctx *ctx, const char *name, long value)
{
    if (!ctx || !name) return RV_ERR_ARG;
    if (strcmp(name, "group_frames") == 0) { ctx->group_frames = value; return RV_OK; }
    if (strcmp(name, "chunk_frames") == 0) { ctx->chunk_frames = value; return RV_OK; }
    if (strcmp(name, "chunk_taper") == 0) { ctx->chunk_taper = value; return RV_OK; }
    if (strcmp(name, "kernel_timing") == 0) { ctx->kernel_timing = value; return RV_OK; }
    if (strcmp(name, "use_tma") == 0) { ctx->use_tma = value; return RV_OK; }
    if (strcmp(name, "prefetch_ctas") == 0) { ctx->prefetch_ctas_per_sm = value < 0 ? 0 : value; return RV_OK; }
    if (strcmp(name, "overlap_groups") == 0) { ctx->overlap_groups = value; return RV_OK; }
    if (strcmp(name, "frame_graphs") == 0) { ctx->frame_graphs = value; return RV_OK; }
    if (strcmp(name, "stage_threads") == 0) { ctx->stage_threads = value < 0 ? 0 : value; return RV_OK; }
    return fail(ctx, RV_ERR_ARG, "unknown option '%s'", name);
}

long rv_launch_count(const rv_ctx *ctx) { return ctx ? ctx->launches : 0; }

int rv_chunk_schedule(int n, int chunk_frames, int taper, int *out, int cap)
{
    if (n < 0 || chunk_frames < 1 || (cap > 0 && !out)) return RV_ERR_ARG;
    int chunk = 0;
    for (long f0 = 0; f0 < n; ++chunk) {
        const long g = chunk_frames_at(chunk_frames, taper != 0, n, chunk, n - f0);
        if (chunk < cap) out[chunk] = (int)g;
        f0 += g;
    }
    return chunk;
}

int rv_alloc_pinned(rv_ctx *ctx, size_t bytes, void **out)
{
    if (!ctx || !out) return RV_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaError_t e = cudaHostAlloc(out, std::max<size_t>(bytes, 16), cudaHostAllocPortable);
    if (e != cudaSuccess) return fail(ctx, RV_ERR_NOMEM, "cudaHostAlloc(%zu): %s", bytes, cudaGetErrorString(e));
    return RV_OK;
}

int rv_free_pinned(rv_ctx *ctx, void *p)
{
    if (!ctx) return RV_ERR_ARG;
    if (p) CK(cudaFreeHost(p));
    return RV_OK;
}

int rv_host_register(rv_ctx *ctx, void *p, size_t bytes)
{
    if (!ctx || !p || bytes == 0) return RV_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaError_t e = cudaHostRegister(p, bytes, cudaHostRegisterPortable);
    if (e != cudaSuccess) return fail(ctx, RV_ERR_CUDA, "cudaHostRegister(%zu): %s", bytes, cudaGetErrorString(e));
    return RV_OK;
}

int rv_host_unregister(rv_ctx *ctx, void *p)
{
    if (!ctx || !p) return RV_ERR_ARG;
    CK(cudaHostUnregister(p));
    return RV_OK;
}

int rv_alloc_device(rv_ctx *ctx, size_t bytes, void **out)
{
    if (!ctx || !out) return RV_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaError_t e = cudaMalloc(out, std::max<size_t>(bytes, 16));
    if (e != cudaSuccess) return fail(ctx, RV_ERR_NOMEM, "cudaMalloc(%zu): %s", bytes, cudaGetErrorString(e));
    return RV_OK;
}

int rv_free_device(rv_ctx *ctx, void *p)
{
    if (!ctx) return RV_ERR_ARG;
    if (p) CK(cudaFree(p));
    return RV_OK;
}

int rv_memcpy(rv_ctx *ctx, void *dst, const void *src, size_t bytes, int kind)
{
    if (!ctx) return RV_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    const cudaMemcpyKind k = kind == 0 ? cudaMemcpyHostToDevice : kind == 1 ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    CK(cudaMemcpyAsync(dst, src, bytes, k, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return RV_OK;
}

int rv_sync(rv_ctx *ctx)
{
    if (!ctx) return RV_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    return wait_all(ctx);
}

int rv_kernel_time(rv_ctx *ctx, int which, double *ms_total, long *launches)
{
    if (!ctx || which < 0 || which > 2) return RV_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    if (!ctx->timed.empty()) {
        RV_TRY(wait_all(ctx));
        for (const TimedLaunch &t : ctx->timed) {
            float ms = 0.f;
            CK(cudaEventSynchronize(t.b));
            CK(cudaEventElapsedTime(&ms, t.a, t.b));
            ctx->k_ms[t.which] += ms;
            ctx->k_n[t.which] += 1;
            ctx->ev_pool.push_back(t.a);
            ctx->ev_pool.push_back(t.b);
        }
        ctx->timed.clear();
    }
    if (ms_total) *ms_total = ctx->k_ms[which];
    if (launches) *launches = ctx->k_n[which];
    return RV_OK;
}

int rv_kernel_time_reset(rv_ctx *ctx)
{
    if (!ctx) return RV_ERR_ARG;
    double d; long l;
    RV_TRY(rv_kernel_time(ctx, 0, &d, &l));
    for (int i = 0; i < 3; ++i) { ctx->k_ms[i] = 0; ctx->k_n[i] = 0; }
    return RV_OK;
}

namespace {
int check_chain_call(rv_ctx *ctx, const uint8_t *in, uint8_t *out, int n, int h, int w, size_t in_pitch, size_t out_pitch, const rv_params *p)
{
    RV_TRY(check_frames(ctx, in, out, n, h, w, in_pitch, out_pitch, 3));
    RV_TRY(check_params_u8(ctx, p));
    if (!p->clahe && p->ksize == 0) return fail(ctx, RV_ERR_ARG, "nothing to do (no CLAHE, no median)");
    if (in == out) return fail(ctx, RV_ERR_ARG, "in-place operation is not supported (tiles read their neighbours' halo)");
    return RV_OK;
}
}  // namespace

int rv_submit(rv_ctx *ctx, const uint8_t *in, uint8_t *out, int n, int h, int w, size_t in_pitch, size_t out_pitch,
              const rv_params *p, int mem_kind, void *stream)
{
    RV_TRY(check_chain_call(ctx, in, out, n, h, w, in_pitch, out_pitch, p));
    RV_TRY(check_kind(ctx, mem_kind));
    if (n == 0) return RV_OK;
    CK(cudaSetDevice(ctx->device));
    if (mem_kind == RV_MEM_DEVICE)
        return chain_device(ctx, in, out, n, h, w, in_pitch, out_pitch, p, nullptr, stream ? (cudaStream_t)stream : ctx->stream);
    PipeJob j;
    j.in = in; j.in_kind = mem_kind; j.ipitch = in_pitch;
    j.out = out; j.out_kind = mem_kind; j.opitch = out_pitch;
    return chain_pipe(ctx, j, n, h, w, p);
}

namespace {
// rv_submit_io (BGR frames in) and rv_submit_io_yuv (yuv: 4:2:0 frames of `layout` in)
int submit_io(rv_ctx *ctx, const rv_io *io, bool yuv, int layout, int n, int h, int w, const rv_params *p)
{
    if (!io) return fail(ctx, RV_ERR_ARG, "null rv_io");
    if (!io->in) return fail(ctx, RV_ERR_ARG, "null frame pointer");
    if (!io->out && !io->tensor) return fail(ctx, RV_ERR_ARG, "neither a frame output nor a tensor output was given");
    RV_TRY(check_kind(ctx, io->in_kind));
    if (yuv)
        RV_TRY(check_yuv(ctx, io->in, io->out, n, h, w, io->in_pitch, io->out_pitch, layout));
    else    // with no frame output the input stands in for it in the shape / pitch checks
        RV_TRY(check_frames(ctx, io->in, io->out ? io->out : io->in, n, h, w, io->in_pitch, io->out ? io->out_pitch : io->in_pitch, 3));
    RV_TRY(check_params_u8(ctx, p));
    if (!p->clahe && p->ksize == 0) return fail(ctx, RV_ERR_ARG, "nothing to do (no CLAHE, no median)");
    if (io->out) {
        RV_TRY(check_kind(ctx, io->out_kind));
        if (io->in == io->out) return fail(ctx, RV_ERR_ARG, "in-place operation is not supported (tiles read their neighbours' halo)");
    }
    if (io->tensor) {
        RV_TRY(check_kind(ctx, io->tensor_kind));
        RV_TRY(check_lb_args(ctx, io->tensor, io->tensor_size, io->pad_value));
        if (p->gate_enable) return fail(ctx, RV_ERR_ARG, "the gate is not supported together with the letterbox stage");
    }
    if (n == 0) return RV_OK;
    CK(cudaSetDevice(ctx->device));
    PipeJob j;
    j.in = io->in; j.in_kind = io->in_kind; j.ipitch = io->in_pitch;
    j.out = io->out; j.out_kind = io->out_kind; j.opitch = io->out_pitch;
    j.lb = io->tensor; j.lb_kind = io->tensor_kind; j.S = io->tensor_size; j.pad = io->pad_value;
    j.lb_rows_only = (io->tensor_flags & RV_TENSOR_PADDING_PRESENT) != 0;
    j.processed = io->processed;
    j.yuv = yuv ? layout : 0;
    return chain_pipe(ctx, j, n, h, w, p);
}
}  // namespace

int rv_submit_io(rv_ctx *ctx, const rv_io *io, int n, int h, int w, const rv_params *p)
{
    if (!ctx) return RV_ERR_ARG;
    return submit_io(ctx, io, false, 0, n, h, w, p);
}

int rv_submit_io_yuv(rv_ctx *ctx, const rv_io *io, int layout, int n, int h, int w, const rv_params *p)
{
    if (!ctx) return RV_ERR_ARG;
    return submit_io(ctx, io, true, layout, n, h, w, p);
}

int rv_wait(rv_ctx *ctx) { return rv_sync(ctx); }

int rv_chain_u8(rv_ctx *ctx, const uint8_t *in, uint8_t *out, int n, int h, int w, size_t in_pitch, size_t out_pitch,
                const rv_params *p, int mem_kind, int32_t *processed, void *stream)
{
    RV_TRY(check_chain_call(ctx, in, out, n, h, w, in_pitch, out_pitch, p));
    RV_TRY(check_kind(ctx, mem_kind));
    if (n == 0) return RV_OK;
    CK(cudaSetDevice(ctx->device));
    if (mem_kind == RV_MEM_DEVICE) {
        cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
        RV_TRY(chain_device(ctx, in, out, n, h, w, in_pitch, out_pitch, p, processed, st));
        CK(cudaStreamSynchronize(st));
        return RV_OK;
    }
    if (n == 1 && in_pitch == (size_t)3 * w && out_pitch == (size_t)3 * w)
        return chain_frame(ctx, in, out, h, w, p, processed);
    PipeJob j;
    j.in = in; j.in_kind = mem_kind; j.ipitch = in_pitch;
    j.out = out; j.out_kind = mem_kind; j.opitch = out_pitch;
    j.processed = processed;
    RV_TRY(chain_pipe(ctx, j, n, h, w, p));
    return wait_all(ctx);
}

int rv_luma_hist(rv_ctx *ctx, const uint8_t *in, int n, int h, int w, size_t pitch, int space, int grid, int32_t *hist,
                 uint8_t *luma, int32_t *gray_minmax, int mem_kind)
{
    RV_TRY(check_frames(ctx, in, in, n, h, w, pitch, pitch, 3));
    if (!hist) return fail(ctx, RV_ERR_ARG, "null hist");
    if (grid < 1 || grid > 256) return fail(ctx, RV_ERR_ARG, "bad grid %d", grid);
    if (n == 0) return RV_OK;
    CK(cudaSetDevice(ctx->device));
    const Geo g = make_geo(h, w, grid);
    const size_t hb = (size_t)n * grid * grid * 256 * 4, lb = (size_t)n * h * w, mb = (size_t)n * 8;
    Staged si, sh, sl, sm;
    RV_TRY(stage_in(ctx, si, in, pitch * h * n, mem_kind));
    RV_TRY(stage_out(ctx, sh, hist, hb, mem_kind));
    if (luma) RV_TRY(stage_out(ctx, sl, luma, lb, mem_kind));
    if (gray_minmax) RV_TRY(stage_out(ctx, sm, gray_minmax, mb, mem_kind));
    RV_TRY(launch_hist(ctx, (const uint8_t *)si.dev, pitch, pitch * h, g, space, n, (int32_t *)sh.dev,
                       luma ? (uint8_t *)sl.dev : nullptr, gray_minmax ? (int32_t *)sm.dev : nullptr, ctx->stream));
    RV_TRY(finish_out(ctx, sh, hist, hb, mem_kind));
    if (luma) RV_TRY(finish_out(ctx, sl, luma, lb, mem_kind));
    if (gray_minmax) RV_TRY(finish_out(ctx, sm, gray_minmax, mb, mem_kind));
    CK(cudaStreamSynchronize(ctx->stream));
    return RV_OK;
}

int rv_build_lut(rv_ctx *ctx, const int32_t *hist, int n, int h, int w, int grid, double clip_limit, uint8_t *lut, int mem_kind)
{
    if (!ctx) return RV_ERR_ARG;
    if (!hist || !lut) return fail(ctx, RV_ERR_ARG, "null pointer");
    if (n < 0 || h < 1 || w < 1 || grid < 1 || grid > 256) return fail(ctx, RV_ERR_ARG, "bad shape");
    if (n == 0) return RV_OK;
    CK(cudaSetDevice(ctx->device));
    const Geo g = make_geo(h, w, grid);
    const size_t hb = (size_t)n * grid * grid * 256 * 4, lb = (size_t)n * grid * grid * 256;
    Staged sh, sl;
    RV_TRY(stage_in(ctx, sh, hist, hb, mem_kind));
    RV_TRY(stage_out(ctx, sl, lut, lb, mem_kind));
    RV_TRY(ensure(ctx, ctx->scratch, (size_t)n * (grid + 1) * (grid + 1) * 256 * 4));
    RV_TRY(launch_lut(ctx, (const int32_t *)sh.dev, g, clip_limit, n, (uint8_t *)sl.dev, (uint32_t *)ctx->scratch.p, ctx->stream));
    RV_TRY(finish_out(ctx, sl, lut, lb, mem_kind));
    CK(cudaStreamSynchronize(ctx->stream));
    return RV_OK;
}

int rv_clahe_dehaze(rv_ctx *ctx, const uint8_t *in, uint8_t *out, int n, int h, int w, size_t in_pitch, size_t out_pitch,
                    int space, double clip_limit, int grid, int mem_kind)
{
    rv_params p;
    memset(&p, 0, sizeof p);
    p.space = space; p.grid = grid; p.ksize = 0; p.clahe = 1; p.clip_limit = clip_limit;
    return rv_chain_u8(ctx, in, out, n, h, w, in_pitch, out_pitch, &p, mem_kind, nullptr, nullptr);
}

int rv_median(rv_ctx *ctx, const uint8_t *in, uint8_t *out, int n, int h, int w, size_t in_pitch, size_t out_pitch, int ksize,
              int mem_kind)
{
    rv_params p;
    memset(&p, 0, sizeof p);
    p.space = RV_SPACE_YCRCB; p.grid = 2; p.ksize = ksize; p.clahe = 0;
    if (ksize == 0) return fail(ctx, RV_ERR_ARG, "ksize 0");
    return rv_chain_u8(ctx, in, out, n, h, w, in_pitch, out_pitch, &p, mem_kind, nullptr, nullptr);
}

int rv_letterbox_geometry(int h, int w, int S, int32_t *new_w, int32_t *new_h, int32_t *top, int32_t *left, int32_t *fused_scale)
{
    if (h < 1 || w < 1 || S < 1) return RV_ERR_ARG;
    const LbGeo g = lb_geometry(h, w, S);
    if (new_w) *new_w = g.nw;
    if (new_h) *new_h = g.nh;
    if (top) *top = g.top;
    if (left) *left = g.left;
    if (fused_scale) *fused_scale = g.scale;
    return RV_OK;
}

int rv_letterbox_f16(rv_ctx *ctx, const uint8_t *in, int n, int h, int w, size_t pitch, uint16_t *out, int S, int pad_value, int mem_kind)
{
    RV_TRY(check_frames(ctx, in, in, n, h, w, pitch, pitch, 3));
    if (!out || S < 1 || S > 8192 || pad_value < 0 || pad_value > 255) return fail(ctx, RV_ERR_ARG, "bad letterbox arguments");
    if (n == 0) return RV_OK;
    CK(cudaSetDevice(ctx->device));
    const LbGeo g = lb_geometry(h, w, S);
    const size_t ob = (size_t)n * 3 * S * S * 2;
    Staged si, so;
    RV_TRY(stage_in(ctx, si, in, pitch * h * n, mem_kind));
    RV_TRY(stage_out(ctx, so, out, ob, mem_kind));
    RV_TRY(launch_letterbox(ctx, (const uint8_t *)si.dev, pitch, pitch * h, n, h, w, g, pad_value, false, (uint16_t *)so.dev, ctx->stream));
    RV_TRY(finish_out(ctx, so, out, ob, mem_kind));
    CK(cudaStreamSynchronize(ctx->stream));
    return RV_OK;
}

int rv_chain_letterbox_f16(rv_ctx *ctx, const uint8_t *in, int n, int h, int w, size_t in_pitch, const rv_params *p,
                           uint16_t *out, int S, int pad_value, uint8_t *full_out, size_t full_pitch, int mem_kind, void *stream)
{
    RV_TRY(check_frames(ctx, in, full_out ? full_out : in, n, h, w, in_pitch, full_out ? full_pitch : in_pitch, 3));
    RV_TRY(check_params_u8(ctx, p));
    RV_TRY(check_kind(ctx, mem_kind));
    if (!p->clahe && p->ksize == 0) return fail(ctx, RV_ERR_ARG, "nothing to do (no CLAHE, no median)");
    if (p->gate_enable) return fail(ctx, RV_ERR_ARG, "the gate is not supported together with the letterbox stage");
    RV_TRY(check_lb_args(ctx, out, S, pad_value));
    if (full_out && in == full_out) return fail(ctx, RV_ERR_ARG, "in-place operation is not supported (tiles read their neighbours' halo)");
    if (n == 0) return RV_OK;
    CK(cudaSetDevice(ctx->device));
    if (mem_kind != RV_MEM_DEVICE) {
        // host buffers: the chunked H2D / kernels / D2H pipeline; only the tensor (and the frames, if asked for) come back
        PipeJob j;
        j.in = in; j.in_kind = mem_kind; j.ipitch = in_pitch;
        j.out = full_out; j.out_kind = mem_kind; j.opitch = full_pitch;
        j.lb = out; j.lb_kind = mem_kind; j.S = S; j.pad = pad_value;
        RV_TRY(chain_pipe(ctx, j, n, h, w, p));
        return wait_all(ctx);
    }
    const LbGeo g = lb_geometry(h, w, S);
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
    uint8_t *dfull = full_out;
    size_t dpitch = full_pitch;
    if (!full_out && g.scale == 0) {
        dpitch = ((size_t)3 * w + 15) & ~(size_t)15;        // unfused: the resize reads a full-resolution intermediate
        RV_TRY(ws_acquire(ctx, ctx->wsync[NPIPE], st));     // lbfull belongs to workspace set NPIPE
        RV_TRY(ensure(ctx, ctx->lbfull, dpitch * h * n));
        dfull = (uint8_t *)ctx->lbfull.p;
    }
    if (g.scale > 0) {
        LbFused lb = {out, g.scale, S, g.top, g.left, dfull ? 1 : 0};
        RV_TRY(launch_letterbox(ctx, nullptr, 0, 0, n, h, w, g, pad_value, true, out, st));
        RV_TRY(run_group(ctx, NPIPE, in, in_pitch, in_pitch * h, dfull ? dfull : (uint8_t *)out, dfull ? dpitch : in_pitch,
                         dfull ? dpitch * h : in_pitch * h, n, h, w, p, st, nullptr, &lb));
    } else {
        RV_TRY(run_group(ctx, NPIPE, in, in_pitch, in_pitch * h, dfull, dpitch, dpitch * h, n, h, w, p, st, nullptr, nullptr));
        RV_TRY(launch_letterbox(ctx, dfull, dpitch, dpitch * h, n, h, w, g, pad_value, false, out, st));
        RV_TRY(ws_release(ctx, ctx->wsync[NPIPE], st));
    }
    if (!stream) CK(cudaStreamSynchronize(st));
    return RV_OK;
}

int rv_gray_span(rv_ctx *ctx, const uint8_t *in, int n, int h, int w, size_t pitch, int32_t *span, int mem_kind)
{
    RV_TRY(check_frames(ctx, in, in, n, h, w, pitch, pitch, 3));
    if (!span) return fail(ctx, RV_ERR_ARG, "null span");
    if (n == 0) return RV_OK;
    CK(cudaSetDevice(ctx->device));
    const Geo g = make_geo(h, w, 2);
    Staged si;
    RV_TRY(stage_in(ctx, si, in, pitch * h * n, mem_kind));
    RV_TRY(ws_acquire(ctx, ctx->wsync[NPIPE], ctx->stream));
    RV_TRY(ensure(ctx, ctx->hist[NPIPE], (size_t)n * 4 * 256 * 4));
    RV_TRY(ensure(ctx, ctx->mm[NPIPE], (size_t)n * 8));
    RV_TRY(launch_hist(ctx, (const uint8_t *)si.dev, pitch, pitch * h, g, RV_SPACE_YCRCB, n, (int32_t *)ctx->hist[NPIPE].p, nullptr,
                       (int32_t *)ctx->mm[NPIPE].p, ctx->stream));
    int32_t *mm = new (std::nothrow) int32_t[2 * (size_t)n];
    if (!mm) return fail(ctx, RV_ERR_NOMEM, "host alloc");
    cudaError_t e = cudaMemcpyAsync(mm, ctx->mm[NPIPE].p, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaEventRecord(ctx->wsync[NPIPE].ev, ctx->stream);
    ctx->wsync[NPIPE].last = ctx->stream;
    ctx->wsync[NPIPE].used = true;
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { delete[] mm; return fail(ctx, RV_ERR_CUDA, "gray span: %s", cudaGetErrorString(e)); }
    const int rc = write_spans(ctx, mm, n, span, mem_kind);
    delete[] mm;
    return rc;
}

}  // extern "C"
