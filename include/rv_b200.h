/*
 * rv_b200.h -- C ABI of the B200-native road-vision preprocessing chain.
 *
 * Drop-in boundary for the reference's `src/preprocess` plugin chain.  The reference has no
 * FFI of its own (it is pure Python calling OpenCV), so every entry point below cites the
 * reference *Python* interface it replaces (paths relative to /root/reference):
 *
 *   rv_chain_u8        PreprocessPipeline.__call__            src/preprocess/pipeline.py:32-45
 *                      = CLAHEDehaze.__call__                 src/preprocess/ops/clahe_dehaze.py:13-32
 *                      + MedianDerain.__call__                src/preprocess/ops/median_derain.py:10-14
 *                      (+ the low-contrast gate               src/preprocess/pipeline.py:24-30,37-40)
 *   rv_luma_hist       cv2.cvtColor(BGR2LAB|BGR2YCrCb)+split  clahe_dehaze.py:22-23 / :27-28, and the
 *                      histogram stage of clahe.apply          clahe_dehaze.py:24 / :29
 *   rv_build_lut       clip/redistribute/CDF stage of cv2.createCLAHE(...).apply   clahe_dehaze.py:19,24,29
 *   rv_clahe_dehaze    CLAHEDehaze.__call__ alone             clahe_dehaze.py:13-32
 *   rv_median          MedianDerain.__call__ alone            median_derain.py:10-14
 *   rv_gray_span       PreprocessPipeline._low_contrast       pipeline.py:24-30
 *   rv_chain_u16       rv_chain_u8 for uint16 frames: the same PreprocessPipeline.__call__ / CLAHEDehaze.__call__ /
 *                      MedianDerain.__call__ (pipeline.py:32-45, clahe_dehaze.py:13-32, median_derain.py:10-14) when the
 *                      reference is handed a 16-bit frame, which it passes to cv2's CV_16U path unchanged
 *   rv_gray_span_u16   PreprocessPipeline._low_contrast on a 16-bit frame   pipeline.py:24-30
 *   rv_chain_ex        rv_chain_u8 / rv_chain_u16 for 1-, 3- and 4-channel frames (gray; BGR; BGRA / BGRx) at either depth, as
 *                      cv2 treats the arrays the reference hands it unchanged
 *   rv_gray_span_ex    rv_gray_span / rv_gray_span_u16 for 3- and 4-channel frames
 *   rv_yuv420_to_bgr   (new) cv2.cvtColor(COLOR_YUV2BGR_NV12 / COLOR_YUV2BGR_I420), the host-side step a user of the reference runs on a
 *                      decoder's 4:2:0 output before pipeline(frame)
 *   rv_submit/rv_wait  (new) batched multi-frame entry fed from pinned host buffers; no reference
 *                      counterpart (the reference loop is one frame in flight, main_preview.py:88-142)
 *   rv_submit_io       (new) the same with every end of the job placed independently: what src/io_video/capture.py:18-21
 *                      captured on the host goes in, the processed frames and / or the detector's input tensor
 *                      (main_preview.py:99 -> src/detect/yolo_ultralytics.py:28-35) come out on the host or stay on the GPU
 *   rv_submit_io_yuv   (new) rv_submit_io on NV12 / I420 frames: the YUV bytes cross PCIe and are converted to BGR on the GPU
 *
 * Conventions: plain C types only; every function returns 0 on success or a negative rv_status;
 * rv_last_error(ctx) gives the message.  A context is bound to one CUDA device, owns its streams and
 * workspaces, and is not thread-safe: one host thread at a time may call into a context; different contexts may be used
 * from different threads.  Within that thread, work may be enqueued on several caller streams (`stream` arguments): every use of
 * a context workspace is ordered after the previous one with CUDA events, so submissions on different streams serialise on the
 * GPU where they share a workspace instead of racing (use one context per stream for concurrency).
 * There is NO CPU fallback: without a usable sm_100 device rv_create fails.
 *
 * Frames are uint8 BGR, interleaved, `h` rows of `w` pixels, `pitch` bytes between rows
 * (pitch >= 3*w), `n` frames h*pitch bytes apart.  `in` and `out` must not alias (in-place is rejected).
 */
#ifndef RV_B200_H
#define RV_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct rv_ctx rv_ctx;

enum rv_status {
    RV_OK = 0,
    RV_ERR_ARG = -1,      /* bad argument (shape, pitch, ksize, ...) */
    RV_ERR_CUDA = -2,     /* a CUDA runtime call or kernel failed */
    RV_ERR_NODEV = -3,    /* no usable sm_100 device */
    RV_ERR_NOMEM = -4
};

enum rv_space { RV_SPACE_YCRCB = 0, RV_SPACE_LAB = 1 };

/* where `in`/`out` live */
enum rv_mem { RV_MEM_HOST = 0, RV_MEM_HOST_PINNED = 1, RV_MEM_DEVICE = 2 };

/* Parameters after the reference's coercions (clahe_dehaze.py:14-17, median_derain.py:11-13):
 * space exactly "LAB" -> RV_SPACE_LAB else YCrCb; grid = max(2, int(tile_grid));
 * ksize in {0 (no median), 3, 5, 7, 9}; clip_limit <= 0 disables clipping (plain AHE). */
typedef struct rv_params {
    int32_t space;
    int32_t grid;
    int32_t ksize;
    int32_t clahe;          /* 0: skip CLAHEDehaze (median only), 1: run it */
    double clip_limit;
    int32_t gate_enable;    /* pipeline.py:37-40: run the chain only if gray span < gate_thresh */
    int32_t reserved;
    double gate_thresh;
} rv_params;

const char *rv_version(void);
int rv_device_count(void);

/* Host-only (no GPU needed): copies the 1024-word YCrCb chroma round-trip table that rv_create uploads for k_chain into
 * out1024 (layout: csrc/rv_colour.cuh, YccTabs).  It replaces, per pixel, the Cr/Cb arithmetic of cv2.cvtColor
 * (COLOR_BGR2YCrCb / COLOR_YCrCb2BGR; reference: src/preprocess/ops/clahe_dehaze.py:27-30); exposed so that the CPU test
 * suite can check it exhaustively against the oracle.  Returns RV_OK. */
int rv_ycc_table(uint32_t *out1024);

int rv_create(int device, rv_ctx **out);
void rv_destroy(rv_ctx *ctx);
const char *rv_last_error(const rv_ctx *ctx);

/* tuning knobs: "group_frames" (frames per hist->lut->apply pass, sized for L2 residency),
 * "chunk_frames" (frames per H2D/compute/D2H pipeline stage for host memory), 0 = automatic;
 * "chunk_taper" (default 1: a host job starts and ends with smaller chunks so that the pipeline fills and drains faster; 0 = uniform);
 * "kernel_timing" (0/1, see rv_kernel_time); "use_tma" (default 1; 0 forces the plain-load staging path);
 * "prefetch_ctas" (default 0 = off: k_chain also prefetches into L2 the box of the CTA that many resident-CTA generations
 * ahead; measured 0.8 % slower on B200, the staging wait is already hidden by the co-resident CTAs);
 * "overlap_groups" (default 0 = off: device batches cut into this many groups so that the histogram/LUT pass of
 * the next group runs on a high-priority side stream under the current group's k_chain; measured 1-6 % slower on
 * B200 because k_chain leaves no SM resources for co-resident CTAs);
 * "frame_graphs" (default 1: single-frame host calls -- rv_chain_u8 with n = 1 and contiguous rows, i.e. the per-frame plugin
 * contract -- replay one captured CUDA graph per (shape, parameters) between the two copies; 0 = direct launches);
 * "stage_threads" (default 0 = pageable single-frame input is left to the driver's own staged copy; n > 0: n helper threads and the
 * caller stage a pageable frame of >= 1.5 MB into page-locked memory slice by slice while earlier slices are already being uploaded
 * -- measured 2x SLOWER than the driver on B200 hosts, kept as an option). */
int rv_set_option(rv_ctx *ctx, const char *name, long value);
/* kernels launched by this context since creation (for bench accounting) */
long rv_launch_count(const rv_ctx *ctx);

/* The chunk schedule of the host pipeline (pure host arithmetic, no context, no GPU: for tests and for callers that size their rings):
 * a job of n frames with at most chunk_frames per chunk; taper != 0 = the default schedule with smaller chunks at both ends (option
 * "chunk_taper").  Writes the first min(count, cap) chunk sizes to out and returns the number of chunks (RV_ERR_ARG on bad arguments).
 * No reference counterpart: the reference processes one frame per call (main_preview.py:94). */
int rv_chunk_schedule(int n, int chunk_frames, int taper, int *out, int cap);
/* With option "kernel_timing" = 1 every k_luma_hist (which=0), k_build_lut (1) and k_chain (2) launch is
 * bracketed by CUDA events on its own stream; this returns the summed device time and launch count
 * since the last reset (synchronises first). */
int rv_kernel_time(rv_ctx *ctx, int which, double *ms_total, long *launches);
int rv_kernel_time_reset(rv_ctx *ctx);

/* pinned host memory for the batched entry */
int rv_alloc_pinned(rv_ctx *ctx, size_t bytes, void **out);
int rv_free_pinned(rv_ctx *ctx, void *p);
/* page-lock memory the caller owns (e.g. a capture library's frame buffers, or huge-page backed memory) so that copies from /
 * to it are plain DMA; unregister before freeing it */
int rv_host_register(rv_ctx *ctx, void *p, size_t bytes);
int rv_host_unregister(rv_ctx *ctx, void *p);
/* device memory helpers (so that Python callers do not need torch/cupy) */
int rv_alloc_device(rv_ctx *ctx, size_t bytes, void **out);
int rv_free_device(rv_ctx *ctx, void *p);
int rv_memcpy(rv_ctx *ctx, void *dst, const void *src, size_t bytes, int kind /*0 h2d,1 d2h,2 d2d*/);
int rv_sync(rv_ctx *ctx);

/* The whole chain, synchronous.  `processed` (optional, host, n ints) receives 1 for frames the chain
 * ran on and 0 for frames the gate skipped (those are copied through unchanged).
 * `stream` (optional) is a cudaStream_t used for RV_MEM_DEVICE buffers; NULL = the context's stream. */
int rv_chain_u8(rv_ctx *ctx, const uint8_t *in, uint8_t *out, int n, int h, int w,
                size_t in_pitch, size_t out_pitch, const rv_params *p, int mem_kind,
                int32_t *processed, void *stream);

/* Asynchronous form for device or pinned buffers: enqueue, return immediately; rv_wait blocks until
 * everything submitted on this context's own streams has finished.  `stream` (optional cudaStream_t,
 * RV_MEM_DEVICE only) enqueues on the caller's stream instead, which the caller synchronises. */
int rv_submit(rv_ctx *ctx, const uint8_t *in, uint8_t *out, int n, int h, int w,
              size_t in_pitch, size_t out_pitch, const rv_params *p, int mem_kind, void *stream);
int rv_wait(rv_ctx *ctx);

/* General asynchronous job (host memory goes through the context's chunked H2D / kernels / D2H pipeline streams; rv_wait
 * blocks until it is finished).  Every end has its own rv_mem kind:
 *   in        frames, host (pageable or pinned) or device
 *   out       processed full-resolution frames, host or device; NULL = not wanted (only legal with `tensor`)
 *   tensor    detector input as rv_chain_letterbox_f16 produces it (n*3*S*S halves), host or device; NULL = none
 *   processed optional host array of n ints (gate decisions, as rv_chain_u8)
 * A device `in` must be complete before the call (the pipeline streams do not wait for other streams); device outputs are
 * complete after rv_wait.  Results that stay on the GPU never cross PCIe: pinned frames in, device frames / tensor out is
 * the path for a detector on the same GPU (main_preview.py:94,99). */
typedef struct rv_io {
    const uint8_t *in;
    size_t in_pitch;
    uint8_t *out;
    size_t out_pitch;
    uint16_t *tensor;
    int32_t *processed;
    int32_t in_kind, out_kind, tensor_kind;
    int32_t tensor_size;    /* S of the S x S letterbox */
    int32_t pad_value;      /* 114 in ultralytics */
    int32_t tensor_flags;   /* RV_TENSOR_PADDING_PRESENT: a HOST tensor buffer already holds the padding rows (written once, e.g. with
                             * pad_value / 255 as a half): only the image rows [top, top + new_h) of every plane are copied back, which
                             * is 56 % of a 1080p -> 640 x 640 tensor; rv_letterbox_geometry gives top and new_h */
} rv_io;
enum { RV_TENSOR_PADDING_PRESENT = 1 };
int rv_submit_io(rv_ctx *ctx, const rv_io *io, int n, int h, int w, const rv_params *p);

/* Stage-level entry points (parity tests). All synchronous; mem_kind applies to every pointer. */
/* hist: n*grid*grid*256 int32; luma (optional): n*h*w bytes, packed; span (optional): n*2 int32 {min,max} of gray */
int rv_luma_hist(rv_ctx *ctx, const uint8_t *in, int n, int h, int w, size_t pitch, int space, int grid,
                 int32_t *hist, uint8_t *luma, int32_t *gray_minmax, int mem_kind);
/* lut: n*grid*grid*256 bytes */
int rv_build_lut(rv_ctx *ctx, const int32_t *hist, int n, int h, int w, int grid, double clip_limit,
                 uint8_t *lut, int mem_kind);
int rv_clahe_dehaze(rv_ctx *ctx, const uint8_t *in, uint8_t *out, int n, int h, int w,
                    size_t in_pitch, size_t out_pitch, int space, double clip_limit, int grid, int mem_kind);
int rv_median(rv_ctx *ctx, const uint8_t *in, uint8_t *out, int n, int h, int w,
              size_t in_pitch, size_t out_pitch, int ksize, int mem_kind);
/* ---- detector-input stage (SURVEY.md 8f-1, the step right after the chain: detector.infer(proc), main_preview.py:99 ->
 * ultralytics' LetterBox + BGR->RGB + HWC->CHW + /255 + half inside model.predict, src/detect/yolo_ultralytics.py:28-35).
 * Square letterbox to S x S: r = min(S/h, S/w), new size round(w r) x round(h r), centred (extra row/column at the
 * bottom/right), constant padding, cv2.resize(INTER_LINEAR) 8-bit arithmetic.  out: n*3*S*S IEEE halves (RGB planes).
 * ultralytics is not installed here and unpinned in the reference: the geometry is this documented spec ("parity
 * unpinned" for it); the resize arithmetic is pinned bit-exactly against cv2.resize. */
int rv_letterbox_geometry(int h, int w, int S, int32_t *new_w, int32_t *new_h, int32_t *top, int32_t *left, int32_t *fused_scale);
int rv_letterbox_f16(rv_ctx *ctx, const uint8_t *in, int n, int h, int w, size_t pitch, uint16_t *out, int S, int pad_value, int mem_kind);
/* chain + detector input in one call.  full_out (optional) also receives the full-resolution BGR result; when it is NULL
 * and the down-scale is an exact integer (1080p -> 640: 3) the full-resolution frame is never written at all (the
 * resize is fused into the chain kernel's store phase).  stream: as rv_submit (RV_MEM_DEVICE: asynchronous if given). */
int rv_chain_letterbox_f16(rv_ctx *ctx, const uint8_t *in, int n, int h, int w, size_t in_pitch, const rv_params *p,
                           uint16_t *out, int S, int pad_value, uint8_t *full_out, size_t full_pitch, int mem_kind, void *stream);

/* ---- fog synthesis (SURVEY.md 8 f4): the per-pixel work of EnhancedFogSynthesizer.synthesize (src/augment/fog.py:227-299, driven by
 * tools/fog_batch.py:7-34), the generator of the hot path's inputs.  The host side (road-vision-system_b200/augment/fog.py) draws
 * every random number in the reference's order and builds the per-geometry maps; these two calls do the full-frame work on the GPU.
 * rv_fog_set_geometry: depth prior and sky weight (h*w floats each, fog.py:144-170), the airlight ramps vgrad (h) and xgrad (w)
 * (fog.py:133-134); host pointers, copied.  rv_fog_u8: one BGR frame in, one fogged BGR frame out (host pointers); `lattice` holds the
 * octaves' (gh+1)*(gw+1) uniform lattices back to back (rand_perlin, fog.py:8-46); `noise` (optional, h*w*3 floats) is the sensor
 * noise field when the host drew it, else the device generates one; t_out / beta_out / airlight_out (optional, host) receive the
 * transmission map, the beta map (h*w floats each) and the scaled airlight map (h*w*3), the reference's `meta`. */
typedef struct rv_fog_frame {
    double persistence;     /* octave amplitude ratio of the value noise (0.5) */
    float base_beta;        /* fog density drawn for this frame */
    float A_bgr[3];         /* airlight colour after tint and clip (fog.py:120-131) */
    float a_target;         /* mean the airlight map is scaled to (fog.py:258) */
    float global_veil;
    float glow;             /* glow strength */
    float cdrop;            /* local contrast fade amount */
    float tint[3];
    float gamma;            /* 0 = no gamma step */
    float noise_sigma;      /* 0 = no sensor noise */
    uint32_t noise_seed;    /* device generator, used when `noise` is NULL */
    int32_t octaves;        /* 1..4 */
    int32_t lat_gh[4], lat_gw[4];
    int32_t band_rad[3];    /* Gaussian sizes of the three depth-blur bands, <= 1 = band skipped (fog.py:207-216) */
    int32_t glow_k, glow_k2;/* Gaussian sizes of the glow mask and the glow blur (fog.py:193, 196) */
    int32_t fade_d;         /* bilateral diameter of the contrast fade (fog.py:227) */
    float fade_sigma;       /* its sigma, 25 + 50 * cdrop */
    int32_t edge_guided;
} rv_fog_frame;
int rv_fog_set_geometry(rv_ctx *ctx, int h, int w, const float *depth, const float *sky_weight, const float *vgrad, const float *xgrad);
int rv_fog_u8(rv_ctx *ctx, const uint8_t *in, uint8_t *out, int h, int w, const rv_fog_frame *f, const float *lattice, const float *noise,
              float *t_out, float *beta_out, float *airlight_out);

/* span: n ints = max(gray) - min(gray) per frame */
int rv_gray_span(rv_ctx *ctx, const uint8_t *in, int n, int h, int w, size_t pitch, int32_t *span, int mem_kind);

/* ---- 16-bit frames (uint16 BGR, e.g. HDR automotive sensors or cv2.imread(..., IMREAD_ANYDEPTH)).  The chain as cv2 computes it on
 * CV_16U: cvtColor BGR2YCrCb / YCrCb2BGR in 16-bit fixed point, CLAHE with 65,536-bin histograms, medianBlur k = 3 / 5
 * (reference: pipeline.py:32-45, clahe_dehaze.py:13-32, median_derain.py:10-14; arithmetic in csrc/rv_u16.cu).
 * rv_chain_u16 behaves like rv_chain_u8 except:
 *   - pitches are in bytes, even, and >= 6*w; buffers are 2-byte aligned;
 *   - RV_SPACE_LAB, a ksize outside {0, 3, 5} (cv2 has neither at 16 bits), "nothing to do" or a tile grid outside [2, 64] (a dense
 *     grid-64 LUT set is already 512 MB per frame) -> RV_ERR_ARG;
 *   - RV_MEM_DEVICE with a `stream` is asynchronous on that stream (as rv_chain_letterbox_f16) unless `processed` is asked for together
 *     with the gate; host memory and device memory without a stream are synchronous.
 * The gate compares the span of cv2's 16-bit BGR2GRAY, (3735 B + 19235 G + 9798 R + 16384) >> 15, with gate_thresh. */
int rv_chain_u16(rv_ctx *ctx, const uint16_t *in, uint16_t *out, int n, int h, int w, size_t in_pitch, size_t out_pitch,
                 const rv_params *p, int mem_kind, int32_t *processed, void *stream);
/* span: n ints = max(gray) - min(gray) per 16-bit frame (synchronous) */
int rv_gray_span_u16(rv_ctx *ctx, const uint16_t *in, int n, int h, int w, size_t pitch, int32_t *span, int mem_kind);

/* ---- 1-, 3- and 4-channel frames at 8 and 16 bits: gray (monochrome, NIR and thermal cameras, IMREAD_GRAYSCALE), BGR, and BGRA / BGRx
 * (IMREAD_UNCHANGED on PNGs with alpha, video decoder and converter surfaces), as cv2 computes on them (arithmetic in csrc/rv_channels.cu):
 *   - CLAHE reads B, G, R and returns 3 channels (cv2.cvtColor ignores alpha and drops it): output channels are 3 when p->clahe,
 *     else `channels`; the median filters every channel on its own, alpha included; the gate's gray ignores alpha.
 *   - channels == 3 is exactly rv_chain_u8 (bits 8) / rv_chain_u16 (bits 16), launch for launch.
 *   - pitches are in bytes: in_pitch >= channels * w * bits / 8, out_pitch >= out_channels * w * bits / 8; 16-bit frames need even
 *     pitches and 2-byte aligned buffers; the rules of rv_chain_u8 / rv_chain_u16 apply otherwise (LAB and ksize 7 / 9 only at 8 bits).
 *   - RV_ERR_ARG: bits not in {8, 16}, channels not in {1, 3, 4}, CLAHE or the gate on one channel (cv2.cvtColor rejects it), and the gate
 *     with CLAHE on 4 channels without `processed` -- those frames it skips are left unwritten in `out` (their result would have 4
 *     channels, not 3).  A median-only pass copies skipped frames through.
 *   - host memory goes group by group through device buffers (synchronous); RV_MEM_DEVICE with a `stream` is asynchronous on it unless
 *     `processed` is asked for together with the gate. */
int rv_chain_ex(rv_ctx *ctx, const void *in, void *out, int n, int h, int w, size_t in_pitch, size_t out_pitch, int bits, int channels,
                const rv_params *p, int mem_kind, int32_t *processed, void *stream);
/* span: n ints = max(gray) - min(gray) per 3- or 4-channel frame (synchronous; one channel -> RV_ERR_ARG) */
int rv_gray_span_ex(rv_ctx *ctx, const void *in, int n, int h, int w, size_t pitch, int bits, int channels, int32_t *span, int mem_kind);

/* ---- YUV 4:2:0 frames (NV12 from hardware decoders: NVDEC, V4L2 M2M, VA-API, GStreamer `appsink format=NV12`; I420 from libavcodec
 * yuv420p), converted to BGR exactly as cv2.cvtColor(COLOR_YUV2BGR_NV12 / COLOR_YUV2BGR_I420) does (arithmetic in csrc/rv_yuv.cu).
 * A frame is cv2's single array of 3h/2 rows of `in_pitch` bytes: h rows of Y, then
 *   RV_YUV_NV12  h/2 rows of interleaved U, V bytes (U first), at the same pitch;
 *   RV_YUV_I420  w*h/4 bytes of U, then w*h/4 bytes of V, packed (in_pitch must equal w).
 * Frame f starts at f * in_pitch * h * 3 / 2.  h and w are the BGR frame's, even and >= 2.  RV_ERR_ARG also for a bad layout,
 * in_pitch < w, out_pitch < 3*w and overlapping buffers. */
enum rv_yuv { RV_YUV_NV12 = 1, RV_YUV_I420 = 2 };
/* The conversion alone into n BGR frames at out_pitch.  Host memory goes group by group and is synchronous; RV_MEM_DEVICE with a
 * `stream` is asynchronous on that stream, without one synchronous on the context's stream. */
int rv_yuv420_to_bgr(rv_ctx *ctx, const uint8_t *in, uint8_t *out, int n, int h, int w, size_t in_pitch, size_t out_pitch, int layout,
                     int mem_kind, void *stream);
/* rv_submit_io with 4:2:0 frames in io->in (host or device): each chunk's YUV bytes are uploaded (or read in place on the device),
 * converted into the BGR workspace, and the chain, gate, letterbox and result copies run exactly as for BGR input.  Results equal
 * rv_submit_io on the frames rv_yuv420_to_bgr gives. */
int rv_submit_io_yuv(rv_ctx *ctx, const rv_io *io, int layout, int n, int h, int w, const rv_params *p);

#ifdef __cplusplus
}
#endif
#endif /* RV_B200_H */
