// wm_k_detect.cu — instantiations + dispatch of one kernel family (see wm_launch.h)
#include "wm_launch.h"

namespace wm {

template <typename PixT, bool TMA>
void launch_detect_t(int mask, bool tr, dim3 grid, cudaStream_t st, const CUtensorMap& tmZ, const CUtensorMap& tmW, const DetectArgs& a)
{
    if (mask == 2) { if (tr) WM_LAUNCH((k_detect<PixT, 2, true, TMA>), detect_smem(TMA, sizeof(PixT) == 1), tmZ, tmW, a); else WM_LAUNCH((k_detect<PixT, 2, false, TMA>), detect_smem(TMA, sizeof(PixT) == 1), tmZ, tmW, a); }  // NVF plane (p > 3)
    else if (mask == WM_MASK_ME) { if (tr) WM_LAUNCH((k_detect<PixT, 0, true, TMA>), detect_smem(TMA, sizeof(PixT) == 1), tmZ, tmW, a); else WM_LAUNCH((k_detect<PixT, 0, false, TMA>), detect_smem(TMA, sizeof(PixT) == 1), tmZ, tmW, a); }
    else { if (tr) WM_LAUNCH((k_detect<PixT, 1, true, TMA>), detect_smem(TMA, sizeof(PixT) == 1), tmZ, tmW, a); else WM_LAUNCH((k_detect<PixT, 1, false, TMA>), detect_smem(TMA, sizeof(PixT) == 1), tmZ, tmW, a); }
}
// debug instantiations (f32, 3x3 masks): the same kernel also writes its u and e_u planes
template <bool TMA>
static void launch_detect_dbg(int mask, bool tr, dim3 grid, cudaStream_t st, const CUtensorMap& tmZ, const CUtensorMap& tmW, const DetectArgs& a)
{
    if (mask == WM_MASK_ME) { if (tr) WM_LAUNCH((k_detect<float, 0, true, TMA, true>), detect_smem(TMA, false), tmZ, tmW, a); else WM_LAUNCH((k_detect<float, 0, false, TMA, true>), detect_smem(TMA, false), tmZ, tmW, a); }
    else { if (tr) WM_LAUNCH((k_detect<float, 1, true, TMA, true>), detect_smem(TMA, false), tmZ, tmW, a); else WM_LAUNCH((k_detect<float, 1, false, TMA, true>), detect_smem(TMA, false), tmZ, tmW, a); }
}
// u8 TMA frames on 128-thread CTAs (8 lines per thread, u in place over the W tile, 4 CTAs per SM)
static void launch_detect_u8n(int mask, bool tr, dim3 grid, cudaStream_t st, const CUtensorMap& tmZ, const CUtensorMap& tmW, const DetectArgs& a)
{
    constexpr int SM = detect_smem_u8n();
    if (mask == 2) { if (tr) WM_LAUNCH_T((k_detect<uint8_t, 2, true, true, false, ENT_U8>), ENT_U8, SM, tmZ, tmW, a); else WM_LAUNCH_T((k_detect<uint8_t, 2, false, true, false, ENT_U8>), ENT_U8, SM, tmZ, tmW, a); }
    else if (mask == WM_MASK_ME) { if (tr) WM_LAUNCH_T((k_detect<uint8_t, 0, true, true, false, ENT_U8>), ENT_U8, SM, tmZ, tmW, a); else WM_LAUNCH_T((k_detect<uint8_t, 0, false, true, false, ENT_U8>), ENT_U8, SM, tmZ, tmW, a); }
    else { if (tr) WM_LAUNCH_T((k_detect<uint8_t, 1, true, true, false, ENT_U8>), ENT_U8, SM, tmZ, tmW, a); else WM_LAUNCH_T((k_detect<uint8_t, 1, false, true, false, ENT_U8>), ENT_U8, SM, tmZ, tmW, a); }
}
void launch_detect(int dtype, int mask, bool tr, bool tma, bool narrow, dim3 grid, cudaStream_t st, const CUtensorMap& tmZ, const CUtensorMap& tmW, const DetectArgs& a)
{
    if (narrow && tma && dtype != WM_F32 && !a.dbg_u) { launch_detect_u8n(mask, tr, grid, st, tmZ, tmW, a); return; }
    if (a.dbg_u) { if (tma) launch_detect_dbg<true>(mask, tr, grid, st, tmZ, tmW, a); else launch_detect_dbg<false>(mask, tr, grid, st, tmZ, tmW, a); return; }
    if (dtype == WM_F32) { if (tma) launch_detect_t<float, true>(mask, tr, grid, st, tmZ, tmW, a); else launch_detect_t<float, false>(mask, tr, grid, st, tmZ, tmW, a); }
    else { if (tma) launch_detect_t<uint8_t, true>(mask, tr, grid, st, tmZ, tmW, a); else launch_detect_t<uint8_t, false>(mask, tr, grid, st, tmZ, tmW, a); }
}

// cooperative launch of a single-image fused kernel: every CTA must be resident at once (they hand over through a spin-wait)
template <typename K, typename... Args>
static bool launch_coop(K kernel, int threads, int smem, int grid_x, int sms, cudaStream_t st, Args... args)
{
    // (set on every call: these launches are captured into a CUDA graph once per image, and K is the same type for every instantiation)
    cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem) != cudaSuccess || per_sm * sms < grid_x) { cudaGetLastError(); return false; }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid_x); cfg.blockDim = dim3(threads); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative;
    at[0].val.cooperative = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    if (cudaLaunchKernelEx(&cfg, kernel, args...) != cudaSuccess) { cudaGetLastError(); return false; }
    return true;
}
bool launch_detect1(int mask, bool tr, int grid_x, cudaStream_t st, const CUtensorMap& tmZ, const CUtensorMap& tmW, const SweepArgs& sa,
                    const DetectArgs& a, unsigned* gen, int sms)
{
    const int smem = detect_smem(true, false);
    if (mask == WM_MASK_ME) return tr ? launch_coop(k_detect1<0, true>, NT, smem, grid_x, sms, st, tmZ, tmW, sa, a, gen) : launch_coop(k_detect1<0, false>, NT, smem, grid_x, sms, st, tmZ, tmW, sa, a, gen);
    return tr ? launch_coop(k_detect1<1, true>, NT, smem, grid_x, sms, st, tmZ, tmW, sa, a, gen) : launch_coop(k_detect1<1, false>, NT, smem, grid_x, sms, st, tmZ, tmW, sa, a, gen);
}

void launch_plane(int dtype, int what_errseq, bool tr, dim3 grid, cudaStream_t st, const PlaneArgs& a)
{
#define WM_PLANE(PIX)                                                                                             \
    if (what_errseq) { if (tr) k_plane<PIX, 0, true><<<grid, NT, 0, st>>>(a); else k_plane<PIX, 0, false><<<grid, NT, 0, st>>>(a); } \
    else { if (tr) k_plane<PIX, 1, true><<<grid, NT, 0, st>>>(a); else k_plane<PIX, 1, false><<<grid, NT, 0, st>>>(a); }
    if (dtype == WM_F32) { WM_PLANE(float) } else { WM_PLANE(uint8_t) }
#undef WM_PLANE
}

void launch_mask_from_errseq(float* plane, long long n, unsigned* scratch, cudaStream_t st)
{
    cudaMemsetAsync(scratch, 0, sizeof(unsigned), st);
    k_absmax<<<256, 256, 0, st>>>(plane, n, scratch);
    k_scale_abs<<<256, 256, 0, st>>>(plane, n, scratch);
}

void launch_rgb2gray(const float* r, const float* g, const float* b, float* gray, long long ld_in, long long ld_out, int L, int P,
                     float wr, float wg, float wb, int blocks, cudaStream_t st)
{
    k_rgb2gray<<<blocks, 256, 0, st>>>(r, g, b, gray, ld_in, ld_out, L, P, wr, wg, wb);
}

void launch_packed_gray(const uint8_t* src, long long ld, long long bstride, int batch, int pixel_bytes, bool bgr, float* gray, int L, int P,
                        int align, int blocks, cudaStream_t st)
{
    const dim3 grid((unsigned)(blocks > batch ? blocks / batch : 1), (unsigned)batch);
    if (pixel_bytes == 4) {
        if (bgr) k_packed_gray<4, true><<<grid, 256, 0, st>>>(src, ld, bstride, gray, L, P, align);
        else k_packed_gray<4, false><<<grid, 256, 0, st>>>(src, ld, bstride, gray, L, P, align);
    } else {
        if (bgr) k_packed_gray<3, true><<<grid, 256, 0, st>>>(src, ld, bstride, gray, L, P, align);
        else k_packed_gray<3, false><<<grid, 256, 0, st>>>(src, ld, bstride, gray, L, P, align);
    }
}

void launch_packed_luma(const uint8_t* src, long long ld, long long bstride, int batch, int luma, uint8_t* dst, long long lp, int L, int P,
                        int align, int blocks, cudaStream_t st)
{
    const dim3 grid((unsigned)(blocks > batch ? blocks / batch : 1), (unsigned)batch);
    if (luma) k_packed_luma<1><<<grid, 256, 0, st>>>(src, ld, bstride, dst, lp, L, P, align);
    else k_packed_luma<0><<<grid, 256, 0, st>>>(src, ld, bstride, dst, lp, L, P, align);
}

void launch_packed_y10(const uint8_t* src, long long ld, long long bstride, int batch, int shift, float* x, int L, int P, int align, int blocks,
                       cudaStream_t st)
{
    const dim3 grid((unsigned)(blocks > batch ? blocks / batch : 1), (unsigned)batch);
    if (shift) k_packed_y10<6><<<grid, 256, 0, st>>>(src, ld, bstride, x, L, P, align);
    else k_packed_y10<0><<<grid, 256, 0, st>>>(src, ld, bstride, x, L, P, align);
}

void launch_packed_v210(const uint8_t* src, long long ld, long long bstride, int batch, float* x, int L, int P, int align, int blocks, cudaStream_t st)
{
    const dim3 grid((unsigned)(blocks > batch ? blocks / batch : 1), (unsigned)batch);
    if (align == 2) k_packed_v210<true><<<grid, 256, 0, st>>>(src, ld, bstride, x, L, P);
    else k_packed_v210<false><<<grid, 256, 0, st>>>(src, ld, bstride, x, L, P);
}

void launch_transpose(const float* src, float* dst, int rows, int cols, cudaStream_t st)
{
    const dim3 blk(32, 8), grd((unsigned)((cols + 31) / 32), (unsigned)((rows + 31) / 32));
    k_transpose<<<grd, blk, 0, st>>>(src, dst, rows, cols);
}

}  // namespace wm
