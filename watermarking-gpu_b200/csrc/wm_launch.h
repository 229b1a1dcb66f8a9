// wm_launch.h — launch dispatchers, one translation unit per kernel family so the build compiles them in parallel.
#pragma once
#include "wm_kernels.cuh"

namespace wm {
void launch_sweep(int dtype, int acc, bool tma, dim3 grid, cudaStream_t st, const CUtensorMap& tmI, const SweepArgs& a);
void launch_stats(int dtype, int mask, bool tr, bool tma, bool narrow, dim3 grid, cudaStream_t st, const CUtensorMap& tmI, const CUtensorMap& tmW, const EmbedArgs& a);
void launch_apply(int in_dtype, int out_dtype, int mask, bool tr, bool tma, dim3 grid, cudaStream_t st, const CUtensorMap& tmI,
                  const CUtensorMap& tmW, const EmbedArgs& a);
void launch_apply_ts(int dtype, int mask, bool tr, bool narrow, dim3 grid, cudaStream_t st, const CUtensorMap& tmI, const CUtensorMap& tmW, const CUtensorMap& tmO,
                     const EmbedArgs& a);
void launch_detect(int dtype, int mask, bool tr, bool tma, bool narrow, dim3 grid, cudaStream_t st, const CUtensorMap& tmZ, const CUtensorMap& tmW, const DetectArgs& a);
// single-image fused detect (cooperative launch): false when the grid cannot be co-resident or the launch fails (the caller falls back)
bool launch_detect1(int mask, bool tr, int grid_x, cudaStream_t st, const CUtensorMap& tmZ, const CUtensorMap& tmW, const SweepArgs& sa,
                    const DetectArgs& a, unsigned* gen, int sms);
void launch_nvfp(int dtype, int pw, bool tr, dim3 grid, cudaStream_t st, const NvfpArgs& a);
void launch_plane(int dtype, int what_errseq, bool tr, dim3 grid, cudaStream_t st, const PlaneArgs& a);
void launch_mask_from_errseq(float* plane, long long n, unsigned* scratch, cudaStream_t st);
void launch_transpose(const float* src, float* dst, int rows, int cols, cudaStream_t st);
void launch_rgb2gray(const float* r, const float* g, const float* b, float* gray, long long ld_in, long long ld_out, int L, int P,
                     float wr, float wg, float wb, int blocks, cudaStream_t st);
// packed 8-bit batch of 3 (RGB / BGR) or 4 (RGBA / BGRA) bytes per pixel (byte ld / stride) -> dense f32 gray planes [batch][L x P];
// align: 2 = src, ld and bstride are multiples of 16 bytes, 1 = of 4 bytes, 0 = neither
void launch_packed_gray(const uint8_t* src, long long ld, long long bstride, int batch, int pixel_bytes, bool bgr, float* gray, int L, int P,
                        int align, int blocks, cudaStream_t st);
// packed 4:2:2 batch (byte ld / stride; luma at byte `luma` of a pixel: 0 YUYV, 1 UYVY; P even) -> u8 luma planes [batch][L x lp], lp a
// multiple of 16; align as above
void launch_packed_luma(const uint8_t* src, long long ld, long long bstride, int batch, int luma, uint8_t* dst, long long lp, int L, int P,
                        int align, int blocks, cudaStream_t st);
// apply kernel of a packed image: input = its gray (f32, dense) or, for 4:2:2 images (pixel_bytes 2), its u8 luma plane; base / out = the
// packed image and the packed output (a.base_vec_ok / a.out_vec_ok: their alignment levels, as for launch_packed_gray; 4:2:2 images: level 2
// means 8-byte aligned)
void launch_apply_packed(int mask, int pixel_bytes, int luma, bool tma, dim3 grid, cudaStream_t st, const CUtensorMap& tmI, const CUtensorMap& tmW,
                         const EmbedArgs& a);
}  // namespace wm

// dtype / mask codes shared with include/wm_b200.h
#ifndef WM_B200_H
enum { WM_MASK_ME = 0, WM_MASK_NVF = 1 };
enum { WM_F32 = 0, WM_U8 = 1 };
#endif

// Every kernel goes through cudaLaunchKernelEx so that the 2nd / 3rd kernel of an op can be launched with programmatic stream
// serialization (PDL): it becomes resident while its predecessor's last block is still reducing / solving, initialises its barriers and
// issues its first TMA loads (the op's input image and W: nothing the predecessor writes), and only then executes
// griddepcontrol.wait before it reads the predecessor's results.  wm::pdl_next() is set by the host code for exactly those launches.
namespace wm {
bool& pdl_next();
}
#define WM_LAUNCH_T(KERNEL, THREADS, SMEM, ...)                        \
    do {                                                               \
        static bool done_[64] = {false};                               \
        int dev_ = 0;                                                  \
        cudaGetDevice(&dev_);                                          \
        if (!done_[dev_ & 63]) { cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM); done_[dev_ & 63] = true; } \
        cudaLaunchConfig_t cfg_ = {};                                  \
        cfg_.gridDim = grid; cfg_.blockDim = dim3(THREADS); cfg_.dynamicSmemBytes = SMEM; cfg_.stream = st; \
        cudaLaunchAttribute at_[1];                                    \
        at_[0].id = cudaLaunchAttributeProgrammaticStreamSerialization; \
        at_[0].val.programmaticStreamSerializationAllowed = 1;         \
        cfg_.attrs = at_; cfg_.numAttrs = wm::pdl_next() ? 1 : 0;      \
        cudaLaunchKernelEx(&cfg_, KERNEL, __VA_ARGS__);                \
    } while (0)
#define WM_LAUNCH(KERNEL, SMEM, ...) WM_LAUNCH_T(KERNEL, NT, SMEM, __VA_ARGS__)
