/*
 * rv_internal.h -- the host toolkit shared by the translation units of librv_b200.so (rv_b200.cu, rv_fog.cu, rv_u16.cu,
 * rv_channels.cu, rv_yuv.cu, rv_yuv422.cu, rv_yuv_out.cu): error
 * recording, device buffers, workspace ordering between streams, and the argument rules and CLAHE geometry that every entry must
 * apply alike.  What is not defined here is defined once, in rv_b200.cu, which owns the context.  Not part of the C ABI
 * (include/rv_b200.h).
 */
#pragma once
#include <cuda_runtime.h>

#include <algorithm>

#include "../../include/rv_b200.h"
#include "rv_common.cuh"        // Geo

namespace rv {

constexpr int MAX_FRAMES_PER_LAUNCH = 32768;    // frames ride on gridDim.z / gridDim.y (limit 65535)

struct Buf {
    void *p = nullptr;
    size_t cap = 0;
};

// Ordering of a workspace set between streams: the event is recorded after the last kernel that touches the set; the next
// user on a different stream waits for it first (two batches submitted on different caller streams never overlap on a set).
struct WsSync {
    cudaEvent_t ev = nullptr;
    cudaStream_t last = nullptr;
    bool used = false;
};

// Workspaces of the 16-bit path (rv_u16.cu) of one context, used on whichever stream a call runs on.
struct U16Ws {
    Buf lut, mid, din, dout, mm, flags;
    int32_t *hflags = nullptr;                  // page-locked copy of the gate decisions
    size_t hflags_cap = 0;
    WsSync sync;
    bool attr_set = false;                      // k_u16_hist_lut's dynamic shared-memory limit is raised
};

// Workspaces of the 1- and 4-channel path (rv_channels.cu) and of the host path of convert_frames (rv_yuv.cu; din / dout) of one
// context, used on whichever stream a call runs on.
struct ChWs {
    Buf pack, din, dout, mm, flags;             // pack: BGR without alpha, the input of the 3-channel chains
    int32_t *hflags = nullptr;                  // page-locked copy of the gate decisions / gray min-max pairs
    size_t hflags_cap = 0;
    WsSync sync;
};

int fail(rv_ctx *ctx, int code, const char *fmt, ...);     // records the message, returns code

#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess)                                                                           \
            return rv::fail(ctx, RV_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

#define RV_TRY(call)              \
    do {                          \
        int rc_ = (call);         \
        if (rc_ != RV_OK) return rc_; \
    } while (0)

int ensure(rv_ctx *ctx, Buf &b, size_t bytes);              // b holds at least `bytes` (reallocated, contents lost, if not)
int ws_acquire(rv_ctx *ctx, WsSync &w, cudaStream_t st);    // `st` waits for the set's last user on another stream
int ws_release(rv_ctx *ctx, WsSync &w, cudaStream_t st);    // after the last work queued on `st` that touches the set

// Shape, pitch and overlap rules of frame arguments: pitches of at least in_bpp * w (input) and out_bpp * w (output) bytes;
// 2-byte samples (16-bit frames) also need even pitches and 2-byte aligned buffers.
int check_frames(rv_ctx *ctx, const void *in, const void *out, int n, int h, int w, size_t ipitch, size_t opitch, int in_bpp,
                 int out_bpp, int sample_bytes);
// BGR frames: bytes_per_pixel 3 (uint8) or 6 (uint16)
inline int check_frames(rv_ctx *ctx, const void *in, const void *out, int n, int h, int w, size_t ipitch, size_t opitch,
                        int bytes_per_pixel)
{
    return check_frames(ctx, in, out, n, h, w, ipitch, opitch, bytes_per_pixel, bytes_per_pixel, bytes_per_pixel == 6 ? 2 : 1);
}
int check_kind(rv_ctx *ctx, int kind);

// clahe.cpp geometry (A.3): both dimensions are padded when either is not divisible by the grid
inline Geo make_geo(int h, int w, int grid)
{
    Geo g;
    g.H = h; g.W = w; g.grid = grid;
    int eh = h, ew = w;
    if (w % grid != 0 || h % grid != 0) {
        ew = w + (grid - w % grid);
        eh = h + (grid - h % grid);
    }
    g.tw = ew / grid;
    g.th = eh / grid;
    g.inv_tw = 1.0f / (float)g.tw;
    g.inv_th = 1.0f / (float)g.th;
    return g;
}

// The low-contrast gate's decision on the device: flags[i] = 1 (process frame i) iff its gray span mm[2i+1] - mm[2i] < thresh.
void launch_gate_flags(rv_ctx *ctx, const int32_t *mm, int n, double thresh, int32_t *flags, cudaStream_t st);

// span[i] = mm[2i+1] - mm[2i] for host (min, max) pairs; span is device memory when mem_kind is RV_MEM_DEVICE
int write_spans(rv_ctx *ctx, const int32_t *mm, int n, int32_t *span, int mem_kind);

// The chains' parameter rules: 8-bit (rv_b200.cu) and 16-bit (rv_u16.cu, which also rejects "nothing to do").
int check_params_u8(rv_ctx *ctx, const rv_params *p);
int check_params_u16(rv_ctx *ctx, const rv_params *p);

// rv_b200.cu: the 8-bit chain over n device frames on stream `st`, group by group on the device path's workspace set.  With the
// gate, processed_host (optional, host) receives the decisions and the frames it skips are copied through if copy_skipped.
int chain_device(rv_ctx *ctx, const uint8_t *in, uint8_t *out, int n, int h, int w, size_t ipitch, size_t opitch,
                 const rv_params *p, int32_t *processed_host, cudaStream_t st, bool copy_skipped = true);

// rv_u16.cu: frames per group of the 16-bit chain, and the chain on one group of device frames (workspaces `s`, which the caller
// has acquired for `st`).  *flags_out receives the device gate flags or nullptr.
long group_frames_u16(const rv_params *p, int h, int w);
int run_group_u16(rv_ctx *ctx, U16Ws &s, const uint16_t *din, size_t ip, size_t ifs, uint16_t *dout, size_t op, size_t ofs, int n,
                  int h, int w, const rv_params *p, cudaStream_t st, const int32_t **flags_out, bool copy_skipped = true);

// Frames per group of a pass that works group by group: as many frames of `frame_bytes` as fit in 1 GiB, at least 1, at most 256.
inline long group_frames(size_t frame_bytes) { return std::max<long>(1, std::min<long>(256, (long)(((size_t)1 << 30) / frame_bytes))); }

// `rows` rows of `rowb` bytes from src (pitch spitch) to dst (pitch dpitch) on `st`: one linear copy when the pitches are equal,
// else a 2D copy of the row bytes.
inline int copy_rows(rv_ctx *ctx, void *dst, size_t dpitch, const void *src, size_t spitch, size_t rowb, size_t rows,
                     cudaMemcpyKind dir, cudaStream_t st)
{
    if (dpitch == spitch) CK(cudaMemcpyAsync(dst, src, spitch * rows, dir, st));
    else CK(cudaMemcpy2DAsync(dst, dpitch, src, spitch, rowb, rows, dir, st));
    return RV_OK;
}

// Frame layouts: 0 is BGR, else enum rv_yuv (4:2:0) or enum rv_yuv422 (4:2:2).
inline bool is_yuv420(int layout) { return layout == RV_YUV_NV12 || layout == RV_YUV_I420; }
inline bool is_yuv422(int layout) { return layout == RV_YUV_YUY2 || layout == RV_YUV_UYVY; }
// rows of one frame: 4:2:0 frames are 3h/2 rows of their pitch, BGR and 4:2:2 frames h rows
inline size_t frame_rows(int layout, int h) { return is_yuv420(layout) ? (size_t)h * 3 / 2 : (size_t)h; }
// bytes of one row: 3w for BGR pixels, w for 4:2:0 planes, 2w for 4:2:2 pixel pairs
inline size_t row_bytes(int layout, int w) { return (size_t)(!layout ? 3 : is_yuv422(layout) ? 2 : 1) * w; }
// the row pitch of frames staged on the device: one that the chains and the conversions' vector paths can use (16 bytes for BGR
// and 4:2:2 rows, 8 for NV12; I420 planes stay packed)
inline size_t stage_pitch(int layout, int w)
{
    if (layout == RV_YUV_NV12) return ((size_t)w + 7) & ~(size_t)7;
    return layout == RV_YUV_I420 ? (size_t)w : (row_bytes(layout, w) + 15) & ~(size_t)15;
}

// rv_yuv.cu: the argument rules of a job with YUV frames on either side (in_layout: RV_YUV_NV12, RV_YUV_I420, RV_YUV_YUY2,
// RV_YUV_UYVY or 0 for BGR; out_layout: RV_YUV_NV12, RV_YUV_I420 or 0; not both 0; out: nullptr = none).
int check_yuv(rv_ctx *ctx, const void *in, const void *out, int n, int h, int w, size_t ipitch, size_t opitch, int in_layout,
              int out_layout);
// rv_yuv.cu: the conversion of n frames of in_layout at pitch sp into frames of out_layout at pitch dp on `st` (one side BGR; frame
// f of either side starts at f * pitch * frame_rows).  It takes the launcher of its family: launch_yuv420 (rv_yuv.cu),
// launch_yuv422 (rv_yuv422.cu) or launch_bgr420 (rv_yuv_out.cu), `layout` being the YUV side's.
int launch_convert(rv_ctx *ctx, int in_layout, int out_layout, const uint8_t *src, size_t sp, uint8_t *dst, size_t dp, int n, int h,
                   int w, cudaStream_t st);
int launch_yuv420(rv_ctx *ctx, int layout, const uint8_t *src, size_t sp, uint8_t *dst, size_t dp, int n, int h, int w, cudaStream_t st);
int launch_yuv422(rv_ctx *ctx, int layout, const uint8_t *src, size_t sp, uint8_t *dst, size_t dp, int n, int h, int w, cudaStream_t st);
int launch_bgr420(rv_ctx *ctx, int layout, const uint8_t *src, size_t sp, uint8_t *dst, size_t dp, int n, int h, int w, cudaStream_t st);
// rv_yuv.cu: the checked job of rv_yuv420_to_bgr, rv_yuv422_to_bgr and rv_bgr_to_yuv420 -- check_yuv, check_kind, then device frames
// converted on `stream` (or, without one, synchronously on the context's stream), host frames group by group through the context's
// ChWs din / dout at stage_pitch.
int convert_frames(rv_ctx *ctx, const uint8_t *in, uint8_t *out, int n, int h, int w, size_t in_pitch, size_t out_pitch, int in_layout,
                   int out_layout, int mem_kind, void *stream);

}  // namespace rv

int rv_internal_device(const rv_ctx *ctx);
void *rv_internal_stream(rv_ctx *ctx);                                  /* the context's main cudaStream_t */
void rv_internal_count_launches(rv_ctx *ctx, long n);
rv::U16Ws &rv_internal_u16(rv_ctx *ctx);
rv::ChWs &rv_internal_ch(rv_ctx *ctx);
void *rv_internal_get_fog(rv_ctx *ctx);
void rv_internal_set_fog(rv_ctx *ctx, void *state, void (*destroy)(void *));
