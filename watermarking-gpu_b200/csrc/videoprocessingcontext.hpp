// videoprocessingcontext.hpp — the per-frame video driver of the reference (videoprocessingcontext.hpp:13-29,
// main.cpp:319-410) over the B200 path.  ffmpeg demux/decode/encode stays outside (SURVEY.md §8: out of scope);
// frames arrive as wm::VideoFrame, the three fields of AVFrame the reference's driver actually reads.
#pragma once
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <functional>
#include <iostream>
#include <vector>

#include "Watermark.hpp"

namespace wm {
// AVFrame subset (main.cpp:348-386,398-405): Y, U, V planes with their row strides
struct VideoFrame {
    uint8_t* data[3];
    int linesize[3];
    int height;
};
}  // namespace wm

// Struct to hold common data for video watermarking and detection
// holds pointers and references, does not own any resources
struct VideoProcessingContext {
    void* inputFormatCtx;   // AVFormatContext* in the reference; opaque here
    void* inputDecoderCtx;  // AVCodecContext*
    const int videoStreamIndex;
    const Watermark* watermarkObj;
    const int height;
    const int width;
    const int watermarkInterval;
    uint8_t* frameFlatPinned;  // width*height bytes of pinned host memory (wm_host_alloc_pinned)

    VideoProcessingContext(void* inputCtx, void* decoderCtx, const int streamIdx, const Watermark* watermark, const int h,
                           const int w, const int interval, uint8_t* pinnedMem)
        : inputFormatCtx(inputCtx), inputDecoderCtx(decoderCtx), videoStreamIndex(streamIdx), watermarkObj(watermark), height(h),
          width(w), watermarkInterval(interval), frameFlatPinned(pinnedMem)
    {
    }
};

// main.cpp:319-340 — the frame loop; `nextFrame` stands in for av_read_frame + the decoder (returns false at EOF)
inline int processFrames(const VideoProcessingContext& data, const std::function<bool(wm::VideoFrame&)>& nextFrame,
                         const std::function<void(wm::VideoFrame*, int&)>& processFrame)
{
    (void)data;
    wm::VideoFrame frame{};
    int framesCount = 0;
    while (nextFrame(frame)) processFrame(&frame, framesCount);
    return framesCount;
}

// main.cpp:343-389 — embed into the Y plane of every watermarkInterval-th frame (u8 -> f32 -> ME embed -> truncating u8),
// then write Y, U, V to the encoder pipe.  The u8<->f32 casts and the transpose of the reference (af::array(width, height,
// ptr).T().as(f32) ... .as(u8).T()) happen inside the kernels: frames go in and out as row-major u8.
inline void embedWatermarkFrame(const VideoProcessingContext& data, int& framesCount, wm::VideoFrame* frame, FILE* ffmpegPipe)
{
    float watermarkStrength = 0.0f;
    const bool embedWatermark = framesCount % data.watermarkInterval == 0;
    const size_t ySize = (size_t)data.width * frame->height;
    if (embedWatermark) {
        wm_image in{};
        in.data = frame->data[0]; in.rows = data.height; in.cols = data.width; in.ld = frame->linesize[0];  // strided read: no repack pass
        in.channels = 1; in.layout = WM_ROW_MAJOR; in.dtype = WM_U8;
        wm_image out = in;
        out.data = data.frameFlatPinned; out.ld = data.width;
        const int rc = wm_embed_host(data.watermarkObj->handle(), &in, &in, &out, WM_MASK_ME, &watermarkStrength);
        if (rc < 0) throw std::runtime_error(std::string(wm_last_error(data.watermarkObj->handle())) + "\n");
        if (ffmpegPipe) fwrite(data.frameFlatPinned, 1, ySize, ffmpegPipe);
    } else if (ffmpegPipe) {
        for (int y = 0; y < data.height; y++) fwrite(frame->data[0] + (size_t)y * frame->linesize[0], 1, data.width, ffmpegPipe);
    }
    if (ffmpegPipe) {  // always write UV planes as-is
        for (int pl = 1; pl <= 2; pl++)
            for (int y = 0; y < data.height / 2; y++)
                fwrite(frame->data[pl] + (size_t)y * frame->linesize[pl], 1, data.width / 2, ffmpegPipe);
    }
    framesCount++;
}

// main.cpp:392-410
inline float detectFrameWatermark(const VideoProcessingContext& data, int& framesCount, wm::VideoFrame* frame, bool print = true)
{
    float correlation = 0.0f;
    if (framesCount % data.watermarkInterval == 0) {
        wm_image in{};
        in.data = frame->data[0]; in.rows = data.height; in.cols = data.width; in.ld = frame->linesize[0];
        in.channels = 1; in.layout = WM_ROW_MAJOR; in.dtype = WM_U8;
        const int rc = wm_detect_host(data.watermarkObj->handle(), &in, WM_MASK_ME, &correlation);
        if (rc < 0) throw std::runtime_error(std::string(wm_last_error(data.watermarkObj->handle())) + "\n");
        if (print) std::cout << "Correlation for frame: " << framesCount << ": " << correlation << "\n";
    }
    framesCount++;
    return correlation;
}

// Batched form of the two frame functions for frames that already sit in HOST memory (a decoded clip): every
// watermarkInterval-th frame of [firstIndex, firstIndex + nFrames) goes through ME embed (mode WM_VIDEO_EMBED), detection
// (WM_VIDEO_DETECT) or both (WM_VIDEO_EMBED_VERIFY: scalars[i] = strength, scalars[nFrames + i] = correlation) in runs of several
// frames per launch sequence with copies and kernels overlapped, on ONE GPU (one Watermark object) or SEVERAL (one object per
// device: contiguous chunks of the global frame index, one host thread per device, the gate of main.cpp:346,395 on the global
// index).  `out` receives the Y planes without row padding (gated-off frames copied through), as embedWatermarkFrame writes them.
// layout 0 (Y planes), a packed colour layout (WM_PACKED_RGB / BGR / RGBA / BGRA, e.g. the BGR frames of cv2.VideoCapture) or a packed
// 4:2:2 layout (WM_PACKED_YUYV / UYVY, e.g. a V4L2 webcam's YUYV) or a 10-bit luma layout (WM_Y10 / WM_Y10_MSB: the Y plane of
// yuv420p10le / P010, 2 bytes per pixel) or v210 (WM_PACKED_V210, e.g. a DeckLink's bmdFormat10BitYUV): `linesize` is then the row pitch in
// bytes and `out` receives dense height x (bytes per pixel * width) frames, v210 frames at the format's pitch WM_V210_PITCH(width)
// (wm_video_ctx in wm_b200.h).
inline int64_t processFramesInMemory(const std::vector<const Watermark*>& watermarkPerGpu, const int height, const int width,
                                     const int watermarkInterval, const int linesize, const int mode, const uint8_t* frames,
                                     uint8_t* out, const int64_t firstIndex, const int64_t nFrames, float* scalars, const int layout = 0)
{
    const int64_t bpp = layout == WM_PACKED_RGB || layout == WM_PACKED_BGR     ? 3
                        : layout == WM_PACKED_RGBA || layout == WM_PACKED_BGRA ? 4
                        : layout == WM_PACKED_YUYV || layout == WM_PACKED_UYVY ? 2
                        : layout == WM_Y10 || layout == WM_Y10_MSB             ? 2
                                                                               : 1;
    const int64_t rowb = layout == WM_PACKED_V210 ? WM_V210_PITCH(width) : bpp * width;  // bytes of an `out` row
    const int ngpus = (int)watermarkPerGpu.size();
    if (ngpus < 1) throw std::runtime_error("processFramesInMemory: no Watermark object\n");
    if (mode == WM_VIDEO_EMBED_VERIFY && ngpus > 1) throw std::runtime_error("processFramesInMemory: EMBED_VERIFY runs on one GPU per call\n");
    std::vector<wm_video_ctx> ctx((size_t)ngpus);
    std::vector<const wm_video_ctx*> pc;
    std::vector<const uint8_t*> in;
    std::vector<uint8_t*> ou;
    for (int g = 0; g < ngpus; g++) {
        int64_t first = 0, count = 0;
        wm_shard_frames(nFrames, g, ngpus, &first, &count);
        ctx[(size_t)g] = wm_video_ctx{watermarkPerGpu[(size_t)g]->handle(), height, width, watermarkInterval, linesize, 0, 0, layout};
        pc.push_back(&ctx[(size_t)g]);
        in.push_back(frames + first * (int64_t)height * linesize);
        ou.push_back(out ? out + first * (int64_t)height * rowb : nullptr);
    }
    const int64_t n = ngpus == 1 ? wm_process_frames(pc[0], mode, in[0], ou[0], firstIndex, nFrames, scalars)
                                 : wm_process_frames_multi(pc.data(), ngpus, mode, in.data(), out ? ou.data() : nullptr, firstIndex, nFrames, scalars);
    if (n < 0) {
        for (int g = 0; g < ngpus; g++) {
            const char* msg = wm_last_error(watermarkPerGpu[(size_t)g]->handle());
            if (msg && *msg) throw std::runtime_error(std::string(msg) + "\n");
        }
        throw std::runtime_error("processFramesInMemory failed\n");
    }
    return n;
}
