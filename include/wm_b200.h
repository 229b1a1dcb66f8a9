/*
 * wm_b200.h — C ABI of the B200-native watermark hot path (libwm_b200.so).
 *
 * This is the drop-in boundary for kar-dim/Watermarking-GPU's `Watermark`
 * class (reference: Watermark_GPU/Watermark.hpp:62-71) and its per-frame
 * video driver (Watermark_GPU/videoprocessingcontext.hpp:13-29,
 * Watermark_GPU/main.cpp:319-410).  Plain pointers and sizes only: no torch,
 * ArrayFire or CUDA types appear in any signature.  ArrayFire arrays enter
 * through `array.device<float>()` device pointers (wm_image.data), never as
 * af::array.  Every call runs hand-written sm_100a kernels; there is no CPU,
 * ArrayFire, OpenCL or library fallback behind any entry point.
 *
 * Image convention: an image is `rows x cols` (x channels planes).
 *   WM_COL_MAJOR : element (r,c) at data[c*ld + r]   (ArrayFire, ld >= rows)
 *   WM_ROW_MAJOR : element (r,c) at data[r*ld + c]   (video planes, ld >= cols)
 * `ld` is in elements.  W is always handed over row-major rows x cols, the
 * layout of the reference's watermark file (Watermark.cpp:72-74).
 *
 * Packed 8-bit colour images, as decoders hand them over (PIL / nvJPEG: R G B R G B ...; OpenCV / ffmpeg bgr24: B G R ...; PIL RGBA,
 * OpenCV IMREAD_UNCHANGED BGRA, ffmpeg rgba / bgra / rgb0 / bgr0, B8G8R8A8 surfaces, CUDA uchar4 images: 4 bytes per pixel):
 *   WM_PACKED_RGB / WM_PACKED_BGR : channel k of pixel (r,c) at data[r*ld + 3*c + k], channels in R,G,B / B,G,R order.
 *   WM_PACKED_RGBA / WM_PACKED_BGRA : channel k of pixel (r,c) at data[r*ld + 4*c + k], the first three in R,G,B / B,G,R order, then
 *   a fourth byte (alpha or padding) that takes no part in the gray, the masks or the correlation.
 *   dtype must be WM_U8 and channels the bytes per pixel (3 or 4); `ld` is in BYTES (>= channels*cols, 0 = dense channels*cols);
 *   plane_stride is ignored; batch strides are in bytes (0 = dense, rows*ld).  The gray of a pixel is (0.299f*R + 0.587f*G) + 0.114f*B,
 *   every operation rounded in f32: af::rgb2gray with the reference's weights (main.cpp:154), bit for bit what wm_rgb2gray gives on the
 *   widened planes.
 *   Taken by wm_embed*, wm_embed_host*, wm_embed_verify_host_batch and wm_detect*, wm_detect_host*:
 *     embed: in_gray = the packed image (its gray is computed on the device), base = NULL or the same image (pointer, layout, ld,
 *            stride), out = a packed u8 image of the same layout value, not overlapping in.  out[k] = (uint8_t)clamp(in[k] + a.mask.W,
 *            0, 255) for the three colour channels (the reference's RGB makeWatermark + .as(u8)); a comes from the gray.  The fourth byte
 *            of a 4-byte pixel is copied from in unchanged.  WM_SINGULAR / WM_ZERO_MASK: out receives all of in's bytes.
 *            wm_embed_verify_host_batch detects on the gray of the truncated u8 output.
 *     detect: the correlation of the image's gray.
 *   Every other entry point (wm_rgb2gray, wm_debug_plane, wm_debug_detect_planes) refuses them with WM_ERR_ARG, as does any mix of a
 *   packed input with a planar or gray base / out, or with a packed base / out of another layout (3 / 4 bytes, RGB / BGR order).
 *   ARGB / ABGR orders are not taken.
 *   Video frames (wm_process_frames*) are Y planes unless wm_video_ctx.layout names one of these layouts; packed frames then get, frame by
 *   frame, what wm_embed / wm_detect give the packed image with the ME mask (see wm_video_ctx).
 *
 * Packed 8-bit 4:2:2 YUV images, as raw video sources hand them over (V4L2 / UVC YUYV, Media Foundation YUY2, DeckLink 2vuy, ffmpeg
 * yuyv422 / uyvy422 / yvyu422):
 *   WM_PACKED_YUYV / WM_PACKED_UYVY : the luma of pixel (r,c) at data[r*ld + 2*c + k], k = 0 (YUYV) or 1 (UYVY); the other byte of each
 *   pixel is chroma.  The chroma takes no part in the masks or the correlation and its order does not matter, so WM_PACKED_YUYV also
 *   takes YVYU and WM_PACKED_UYVY also takes VYUY.
 *   dtype must be WM_U8, channels 2 and cols even (4:2:2 pairs pixels); `ld` is in BYTES (>= 2*cols, 0 = dense 2*cols); batch strides
 *   are in bytes.  Taken by the same entry points as the packed colour layouts:
 *     embed: in_gray = the packed image, base = NULL or the same image, out = a packed image of the same layout, not overlapping in.
 *            The luma of out is (uint8_t)clamp(Y + a.mask.W, 0, 255), computed exactly as for a u8 Y plane holding the same luma;
 *            the chroma bytes are copied from in without arithmetic.  WM_SINGULAR / WM_ZERO_MASK: out receives all of in's bytes.
 *     detect: the correlation of the luma.
 *   A mix of YUYV and UYVY, or of a 4:2:2 layout with a colour or planar layout, is refused with WM_ERR_ARG, as are wm_rgb2gray,
 *   wm_debug_plane and wm_debug_detect_planes.
 */
#ifndef WM_B200_H
#define WM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Watermark.hpp:10-14 — enum MASK_TYPE { ME, NVF } */
enum { WM_MASK_ME = 0, WM_MASK_NVF = 1 };
enum { WM_COL_MAJOR = 0, WM_ROW_MAJOR = 1, WM_PACKED_RGB = 2, WM_PACKED_BGR = 3, WM_PACKED_RGBA = 4, WM_PACKED_BGRA = 5, WM_PACKED_YUYV = 6,
       WM_PACKED_UYVY = 7 };
enum { WM_F32 = 0, WM_U8 = 1 };

/* return codes: 0 ok; >0 non-fatal (mirrors the reference's fall-backs); <0 errors */
enum {
    WM_OK = 0,
    WM_SINGULAR = 1,      /* Watermark.cpp:164-165,205-208,246-247: unsolvable system -> out = base / corr = 0 */
    WM_ZERO_MASK = 2,     /* ||mask.W|| == 0 (reference: a = inf, NaN image; here: out = base, a = inf) */
    WM_ERR_BAD_P = -1,    /* Watermark.cpp:24-25 */
    WM_ERR_W_FILE = -2,   /* Watermark.cpp:65-66 */
    WM_ERR_W_SIZE = -3,   /* Watermark.cpp:70-71 */
    WM_ERR_DIMS = -4,     /* image dims differ from the ctx dims / unsupported */
    WM_ERR_ARG = -5,
    WM_ERR_CUDA = -6,
    WM_ERR_NO_DEVICE = -7
};

typedef struct wm_ctx wm_ctx;

typedef struct wm_image {
    void *data;            /* DEVICE pointer (wm_*_host entry points take HOST pointers instead) */
    int64_t rows, cols;
    int64_t ld;            /* leading dimension in elements, bytes for packed images (0 = dense) */
    int32_t channels;      /* 1, or 3 for the RGB base/out of makeWatermark (Watermark.cpp:171); bytes per pixel (2, 3 or 4) for packed images */
    int32_t layout;        /* WM_COL_MAJOR | WM_ROW_MAJOR | WM_PACKED_RGB | WM_PACKED_BGR | WM_PACKED_RGBA | WM_PACKED_BGRA | WM_PACKED_YUYV |
                              WM_PACKED_UYVY */
    int32_t dtype;         /* WM_F32 | WM_U8 */
    int32_t reserved;
    int64_t plane_stride;  /* elements between channel planes (0 = dense) */
} wm_image;

/* options for wm_set_option */
enum {
    WM_OPT_FP16_PRODUCTS = 1, /* 1 (default): Rx/rx products rounded to fp16 as kernels/me_p3.hpp:10-20 does; 0: f32 */
    WM_OPT_KERNEL_TIMING = 2, /* 1: bracket every kernel with CUDA events (wm_get_kernel_times) */
    WM_OPT_USE_TMA = 3,       /* 1 (default): TMA tile loads when the shape allows; 0: always the plain loader */
    WM_OPT_SERIAL_SLOTS = 4,  /* 1: the video driver uses one slot (kernels do not overlap: per-kernel timing) */
    WM_OPT_CUDA_GRAPHS = 5,   /* 1 (default): wm_embed / wm_detect replay a captured CUDA graph when called again with the same arguments */
    WM_OPT_SPLIT_COST = 7,    /* tile-times one more launch is assumed to cost (default 8: launch gap, pipeline ramp, second stage + solve tail) when a batch whose size does not divide
                                 the resident CTA count is launched as better-balanced sub-batches; < 0: never split */
    WM_OPT_MMA_ACCUM = 6,     /* 1 (default): the fp16-rounded Rx/rx products are summed on the tensor pipe (HMMA with a 0/1 selector
                                 matrix = four mixed-precision adds per lane); 0: FHADD chain.  Same bits for integer-valued pixels */
    WM_OPT_TMA_STORE = 10,    /* 1 (default): where base = input and the output is gray, dense enough and 16-byte aligned, the apply kernel's output leaves through
                                 TMA stores (cp.async.bulk.tensor smem -> global) instead of per-thread vector stores; same bits, +8..10 % on that kernel
                                 (profiles/r2_tma_store_ab.md); 0: always per-thread stores */
    WM_OPT_PDL = 11,          /* 1 (default): the 2nd / 3rd kernel of an op is launched with programmatic stream serialization: it becomes resident, initialises
                                 its barriers and issues its first tile loads while the previous kernel's last block still reduces / solves, and executes
                                 griddepcontrol.wait before reading that kernel's results; 0: plain stream order */
    WM_OPT_FUSED_SINGLE = 12, /* 0 (default): every op is 2-3 kernels chained with programmatic dependent launch; 1: a synchronous wm_detect on one f32 image
                                 whose tiles fit the resident CTAs' shared memory (e.g. 1080p) runs as ONE cooperative kernel (k_detect1) that keeps its tiles in
                                 shared memory across sweep -> solve -> detector.  Same results; measured 3 us SLOWER per op at 1080p (profiles/r2_latency.md:
                                 the grid-wide hand-over costs more than the second launch it saves), kept as an experiment */
    WM_OPT_PADDED_UPLOAD = 13, /* 1 (default): wm_process_frames uploads a HOST frame whose row padding is small (<= width / 8) and whose linesize is a multiple
                                 of 16 together with its padding, as one linear copy, and reads it in place with ld = linesize; 0: the padding is always dropped on
                                 the way up by a 2-D copy (the reference's row-by-row repack, main.cpp:348-353) */
    WM_OPT_NARROW_U8 = 14,    /* 1 (default): the stats / apply kernels of u8 frames (TMA path) run on 128-thread CTAs, 4 warps x 8 lines of a tile, four CTAs per SM,
                                 like the sweep; 0: 256-thread CTAs, 8 warps x 4 lines, three per SM.  Same bits */
    WM_OPT_RUN_MB = 15,       /* frames of one run (one batched launch sequence) of wm_process_frames on DEVICE frames fill at most this many MB (default 136, at most
                                 32 frames; packed frames count their packed bytes): large enough to amortise a launch's ramp and tail, small enough that a run's watermarked frames are still in L2 when
                                 the detector's kernels read them back */
    WM_OPT_HOST_RUN_FRAMES = 9, /* frames per run (one batched launch sequence + its copies) of wm_process_frames when frames are in HOST memory; default 4 */
    WM_OPT_F32_SOLVE = 8      /* 0 (default): the 8x8 system is summed and solved in f64 (pivot cut 1e-12 max|Rx|); 1: Rx / rx are rounded to f32
                                 and solved by an f32 LU (pivot cut 1e-6 max|Rx|) like af::solve on the reference's f32 arrays
                                 (Watermark.cpp:203) — the mode to use when pinning against a real ArrayFire run */
};

/* ---- lifetime: Watermark ctor / copy-ctor / reinitialize / dtor (Watermark.cpp:21-85) ----
 * p: 3, 5, 7 or 9 like the reference's constructor (anything else: WM_ERR_BAD_P, "Wrong p parameter: <p>!").  p is the NVF
 * window (kernels/nvf.hpp:14-17); the prediction-error mask and the detector are 3 x 3 for every p, as in the reference. */
int wm_create(wm_ctx **out, int64_t rows, int64_t cols, const float *w_host_rowmajor, int p, float psnr,
              int device, void *cuda_stream /* cudaStream_t or NULL = own stream */);
int wm_create_from_file(wm_ctx **out, int64_t rows, int64_t cols, const char *w_path, int p, float psnr,
                        int device, void *cuda_stream);
int wm_clone(const wm_ctx *src, wm_ctx **out);                 /* shares W, owns workspace + stream */
int wm_reinitialize(wm_ctx *ctx, int64_t rows, int64_t cols, const float *w_host_rowmajor);
int wm_reinitialize_from_file(wm_ctx *ctx, int64_t rows, int64_t cols, const char *w_path);
void wm_destroy(wm_ctx *ctx);
int wm_set_option(wm_ctx *ctx, int option, int value);
const char *wm_last_error(const wm_ctx *ctx);                  /* ctx may be NULL: last creation error */
float wm_strength_factor(const wm_ctx *ctx);                   /* Watermark.cpp:22 */

/* ---- hot path, device pointers, synchronous like the reference (scalars valid on return) ---- */
/* Watermark::makeWatermark (Watermark.cpp:156-172).  in: gray, 1 channel.  base/out: 1 or 3 channels,
 * same rows/cols/layout; out may alias base.  *a_host receives watermarkStrength. */
int wm_embed(wm_ctx *ctx, const wm_image *in_gray, const wm_image *base, wm_image *out, int mask_type,
             float *a_host);
/* Watermark::detectWatermark (Watermark.cpp:234-250) */
int wm_detect(wm_ctx *ctx, const wm_image *img, int mask_type, float *corr_host);

/* ---- batched / pipelined form (BASELINE config 5; the video driver's inner loop) ----
 * `batch` equal-size images, image b at data + b*batch_stride elements (in/base/out each).
 * One launch sequence covers the whole batch; results land in a_host/corr_host/status_host[batch]
 * (status may be NULL).  Asynchronous on `slot` (0..wm_num_slots-1, each its own stream + workspace): calls on one
 * slot queue up in stream order (no host wait between them); results are valid after wm_sync(ctx, slot). */
int wm_num_slots(const wm_ctx *ctx);
void *wm_get_stream(const wm_ctx *ctx, int slot); /* the slot's cudaStream_t: order your own copies on it */
int wm_embed_batch(wm_ctx *ctx, int slot, const wm_image *in_gray, const wm_image *base, wm_image *out,
                   int64_t in_stride, int64_t base_stride, int64_t out_stride, int batch, int mask_type,
                   float *a_host, int *status_host);
int wm_detect_batch(wm_ctx *ctx, int slot, const wm_image *img, int64_t img_stride, int batch, int mask_type,
                    float *corr_host, int *status_host);
int wm_sync(wm_ctx *ctx, int slot /* -1 = all */);

/* ---- host-buffer form: H2D copy, compute, D2H copy inside the call (main.cpp:355-357,379-381,405) ---- */
int wm_embed_host(wm_ctx *ctx, const wm_image *in_gray_host, const wm_image *base_host, wm_image *out_host,
                  int mask_type, float *a_host);
int wm_detect_host(wm_ctx *ctx, const wm_image *img_host, int mask_type, float *corr_host);

/* Pipelined host-buffer form: `batch` host images (element strides as in the device batch API, 0 = dense) are staged with 2-D copies on the
 * slot's stream, processed as one batched launch sequence and copied back; the call returns at once, results (and the output images) are
 * valid after wm_sync(ctx, slot).  Strided host views are honoured: only the images' own pixels are read or written. */
int wm_embed_host_batch(wm_ctx *ctx, int slot, const wm_image *in_gray_host, const wm_image *base_host, wm_image *out_host,
                        int64_t in_stride, int64_t base_stride, int64_t out_stride, int batch, int mask_type,
                        float *a_host, int *status_host);
int wm_detect_host_batch(wm_ctx *ctx, int slot, const wm_image *img_host, int64_t img_stride, int batch, int mask_type,
                         float *corr_host, int *status_host);
/* embed + verify: wm_embed_host_batch, then detectWatermark on each watermarked image while it is still in the slot's device staging buffer
 * (gray output of the input's dtype): the embed / detect pair of the reference's testForImage flow (main.cpp:178-217) with one upload and one
 * download per image.  corr_host[b] = correlation of image b. */
int wm_embed_verify_host_batch(wm_ctx *ctx, int slot, const wm_image *in_gray_host, const wm_image *base_host, wm_image *out_host,
                               int64_t in_stride, int64_t base_stride, int64_t out_stride, int batch, int mask_type,
                               float *a_host, float *corr_host, int *status_host);

/* ---- af::rgb2gray(rgb, wr, wg, wb) of the reference's image flow (main.cpp:142-154,196-197): planar f32 RGB -> gray ---- */
int wm_rgb2gray(wm_ctx *ctx, const wm_image *rgb, wm_image *gray, float wr, float wg, float wb);

/* ---- parity access to the class's private intermediates (Watermark.hpp:52-58) ----
 * Valid after the last synchronous wm_embed / wm_detect.  dst is HOST memory.
 *   WM_DBG_RX     64 doubles  Rx (reference neighbour order, full symmetric)      Watermark.cpp:148
 *   WM_DBG_RXVEC   8 doubles  rx                                                  Watermark.cpp:149
 *   WM_DBG_COEFFS  8 floats   prediction coefficients                             Watermark.cpp:203
 *   WM_DBG_SCALARS 8 doubles  {status, a, max|e|, sum (|mask|W)^2, dot, |ez|^2, |eu|^2, corr}
 *   WM_DBG_PHASES  8 doubles  timeline of the last Rx sweep's last CTA, ns since that CTA started: [1] tiles done, [2] frame
 *                             ring done, [3] elected last, [4] second-stage sums done, [5] 8x8 system solved (profiling aid)
 * wm_debug_set_coeffs injects coefficients: the next call skips the Rx sweep + solve (staged parity, SURVEY H1).
 * wm_debug_plane computes e_z (WM_DBG_ERRSEQ), the NVF mask (WM_DBG_MASK_NVF) or the prediction-error mask |e| / max|e|
 * (WM_DBG_MASK_ME, Watermark.cpp:213-214) of an image into dst_dev.
 * wm_debug_detect_planes runs detectWatermark's own kernel on an f32 image and also writes the two planes it never materialises:
 * u = mask.W (Watermark.cpp:248; for the ME mask the kernel's u is |e_z|.W — the 1 / max|e| scale cancels in the correlation and is
 * dropped) and e_u = u - prediction(u) with u clamped to the edge (Watermark.cpp:221-225), dense, same layout as the image. */
enum { WM_DBG_RX = 0, WM_DBG_RXVEC = 1, WM_DBG_COEFFS = 2, WM_DBG_SCALARS = 3, WM_DBG_ERRSEQ = 4, WM_DBG_MASK_NVF = 5, WM_DBG_PHASES = 6, WM_DBG_MASK_ME = 7 };
int wm_debug_get(wm_ctx *ctx, int what, void *dst_host);
int wm_debug_set_coeffs(wm_ctx *ctx, const float *coeffs8_or_null);
int wm_debug_plane(wm_ctx *ctx, const wm_image *img, int what, float *dst_dev /* same layout, dense */);
int wm_debug_detect_planes(wm_ctx *ctx, const wm_image *img, int mask_type, float *u_dev, float *eu_dev, float *corr_host);

/* per-kernel device time (ms) accumulated since the last reset, when WM_OPT_KERNEL_TIMING is on.
 * names: 0 rx_sweep(+solve) 1 me_stats 2 nvf_stats 3 me_apply 4 me_detect 5 nvf_apply 6 nvf_detect.  Returns the number of timed brackets
 * (one per op call: all sub-batch launches of that kernel family). */
enum { WM_K_SWEEP = 0, WM_K_ME_STATS = 1, WM_K_NVF_STATS = 2, WM_K_APPLY = 3, WM_K_DETECT = 4, WM_K_APPLY_NVF = 5, WM_K_DETECT_NVF = 6, WM_K_COUNT = 7 };
int64_t wm_get_kernel_times(wm_ctx *ctx, int kernel, double *total_ms, int reset);
int64_t wm_launch_count(const wm_ctx *ctx); /* kernels launched by this ctx since creation */

/* ---- video driver: VideoProcessingContext + processFrames / embedWatermarkFrame / detectFrameWatermark
 * (videoprocessingcontext.hpp:13-29, main.cpp:319-410).  By default frames are Y planes, u8 row-major height x width with
 * row stride `linesize` (>= width); ffmpeg decode/encode is outside this library (frames come from memory).
 * Packed colour frames (layout = WM_PACKED_RGB / BGR / RGBA / BGRA: cv2.VideoCapture's BGR, ffmpeg's rgb24 / bgr24 / rgba / bgra /
 * rgb0 / bgr0, B8G8R8A8 screen captures): height rows of bpp * width bytes (bpp = 3 or 4), `linesize` is the row pitch in BYTES
 * (ffmpeg's linesize[0]; >= bpp * width, 0 = dense) and `out` receives dense frames of height x (bpp * width) bytes.  A gated frame gets
 * what wm_embed / wm_detect give that packed image with the ME mask: `a` from its gray, the watermark added to the three colour bytes,
 * the fourth byte copied unchanged, DETECT / EMBED_VERIFY correlate the gray.  Gated-off frames are copied through, all bytes of a pixel.
 * Packed 4:2:2 frames (layout = WM_PACKED_YUYV / UYVY: V4L2 YUYV, YUY2, 2vuy, ffmpeg yuyv422 / uyvy422): height rows of 2 * width bytes
 * (width even), `linesize` the row pitch in bytes (>= 2 * width, 0 = dense), `out` dense height x (2 * width) frames.  A gated frame gets
 * what wm_embed / wm_detect give it: `a` and the watermark from the luma (the bits of the Y-plane driver on the same luma), the chroma
 * copied unchanged, DETECT / EMBED_VERIFY correlate the luma.  Gated-off frames are copied through, both bytes of a pixel. */
typedef struct wm_video_ctx {
    wm_ctx *watermark;        /* watermarkObj (non-owning) */
    int32_t height, width;
    int32_t watermark_interval;
    int32_t linesize;         /* frame->linesize[0] in bytes; rows are repacked when != width * bytes per pixel (main.cpp:348-353) */
    int64_t frame_stride;     /* bytes between consecutive frames in `frames` */
    int32_t frames_on_device; /* 1: `frames`/`out` are device pointers; 0: host (pinned recommended) */
    int32_t layout;           /* 0 or WM_ROW_MAJOR: Y planes; WM_PACKED_RGB | WM_PACKED_BGR | WM_PACKED_RGBA | WM_PACKED_BGRA: packed u8
                                 colour frames; WM_PACKED_YUYV | WM_PACKED_UYVY: packed 4:2:2 frames; anything else is refused with WM_ERR_ARG */
} wm_video_ctx;
enum { WM_VIDEO_EMBED = 0, WM_VIDEO_DETECT = 1, WM_VIDEO_EMBED_VERIFY = 2 };
/* Processes frames [first_index, first_index + n_frames) of a stream: frame i is gated by
 * (i % watermark_interval == 0) exactly as main.cpp:346,395 (global index, so shards agree).
 * EMBED: out receives every frame (Y plane or packed frame, contiguous and without row padding; gated-off frames are copied
 * through), scalars[i] = a (NaN for gated-off and for unsolvable frames).  DETECT: scalars[i] = correlation (NaN for gated-off frames).  out may be NULL
 * for DETECT.
 * EMBED_VERIFY: EMBED, then DETECT on each frame just written while it is still on the device (no second upload): scalars_host has
 * 2 * n_frames entries, [i] = a, [n_frames + i] = correlation.  Returns the number of frames processed or a negative error. */
int64_t wm_process_frames(const wm_video_ctx *v, int mode, const uint8_t *frames, uint8_t *out,
                          int64_t first_index, int64_t n_frames, float *scalars_host);

/* Multi-GPU form (SURVEY.md 8e; the gate of main.cpp:346,395 is on the GLOBAL frame index): the range [first_index, first_index + n_frames)
 * is cut into `ngpus` contiguous chunks by wm_shard_frames; chunk g is processed by v[g] (a wm_video_ctx whose watermark lives on the device
 * that should do the work; several contexts may share a device) on its own host thread.  chunk_frames[g] / chunk_out[g] point at the FIRST frame
 * of chunk g (host or device memory according to v[g]->frames_on_device), so device-resident chunks need no common address space.
 * scalars_host[i] belongs to global frame first_index + i.  No collective: only these scalars leave a GPU.  Returns frames processed. */
void wm_shard_frames(int64_t n_frames, int rank, int world, int64_t *first, int64_t *count);
int64_t wm_process_frames_multi(const wm_video_ctx *const *v, int ngpus, int mode, const uint8_t *const *chunk_frames,
                                uint8_t *const *chunk_out, int64_t first_index, int64_t n_frames, float *scalars_host);

/* ---- small device-memory helpers for FFI hosts without a CUDA binding (tests, ctypes) ---- */
void *wm_dev_alloc(wm_ctx *ctx, int64_t bytes);
void wm_dev_free(wm_ctx *ctx, void *p);
int wm_dev_upload(wm_ctx *ctx, void *dst_dev, const void *src_host, int64_t bytes);
int wm_dev_download(wm_ctx *ctx, void *dst_host, const void *src_dev, int64_t bytes);
void *wm_host_alloc_pinned(int64_t bytes);
void wm_host_free_pinned(void *p);
int wm_device_count(void);
const char *wm_version(void);

#ifdef __cplusplus
}
#endif
#endif /* WM_B200_H */
