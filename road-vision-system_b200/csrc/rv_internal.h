/*
 * rv_internal.h -- the host toolkit shared by the translation units of librv_b200.so (rv_b200.cu, rv_fog.cu, rv_u16.cu): error
 * recording, device buffers, workspace ordering between streams, and the argument rules and CLAHE geometry that every entry must
 * apply alike.  What is not defined here is defined once, in rv_b200.cu, which owns the context.  Not part of the C ABI
 * (include/rv_b200.h).
 */
#pragma once
#include <cuda_runtime.h>

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

// Shape, pitch and overlap rules of frame arguments; bytes_per_pixel 3 (uint8 BGR) or 6 (uint16 BGR, which also needs even
// pitches and 2-byte aligned buffers).
int check_frames(rv_ctx *ctx, const void *in, const void *out, int n, int h, int w, size_t ipitch, size_t opitch,
                 int bytes_per_pixel);
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

}  // namespace rv

int rv_internal_device(const rv_ctx *ctx);
void *rv_internal_stream(rv_ctx *ctx);                                  /* the context's main cudaStream_t */
void rv_internal_count_launches(rv_ctx *ctx, long n);
rv::U16Ws &rv_internal_u16(rv_ctx *ctx);
void *rv_internal_get_fog(rv_ctx *ctx);
void rv_internal_set_fog(rv_ctx *ctx, void *state, void (*destroy)(void *));
