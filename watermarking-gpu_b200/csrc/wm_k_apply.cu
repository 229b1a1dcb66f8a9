// wm_k_apply.cu — instantiations + dispatch of one kernel family (see wm_launch.h)
#include "wm_launch.h"

namespace wm {

template <typename PixT, typename OutT, bool TMA, bool SB>
void launch_apply_s(int mask, bool tr, dim3 grid, cudaStream_t st, const CUtensorMap& tmI, const CUtensorMap& tmW, const EmbedArgs& a)
{
    if (mask == 2) { WM_LAUNCH((k_apply<PixT, OutT, 2, false, TMA, SB>), embed_smem(TMA, sizeof(PixT) == 1), tmI, tmW, a); }  // NVF plane (p > 3)
    else if (mask == WM_MASK_ME) { if (tr) WM_LAUNCH((k_apply<PixT, OutT, 0, true, TMA, SB>), embed_smem(TMA, sizeof(PixT) == 1), tmI, tmW, a); else WM_LAUNCH((k_apply<PixT, OutT, 0, false, TMA, SB>), embed_smem(TMA, sizeof(PixT) == 1), tmI, tmW, a); }
    else { if (tr) WM_LAUNCH((k_apply<PixT, OutT, 1, true, TMA, SB>), embed_smem(TMA, sizeof(PixT) == 1), tmI, tmW, a); else WM_LAUNCH((k_apply<PixT, OutT, 1, false, TMA, SB>), embed_smem(TMA, sizeof(PixT) == 1), tmI, tmW, a); }
}
template <typename PixT, typename OutT, bool TMA>
void launch_apply_t(int mask, bool tr, dim3 grid, cudaStream_t st, const CUtensorMap& tmI, const CUtensorMap& tmW, const EmbedArgs& a)
{
    if (a.same_base) launch_apply_s<PixT, OutT, TMA, true>(mask, tr, grid, st, tmI, tmW, a);
    else launch_apply_s<PixT, OutT, TMA, false>(mask, tr, grid, st, tmI, tmW, a);
}
// A/B variant with TMA stores (gray, same base, TMA loads, 3x3 masks)
void launch_apply_ts(int dtype, int mask, bool tr, bool narrow, dim3 grid, cudaStream_t st, const CUtensorMap& tmI, const CUtensorMap& tmW, const CUtensorMap& tmO, const EmbedArgs& a)
{
    if (narrow && dtype != WM_F32) {  // u8 frames on 128-thread CTAs (8 lines per thread, 4 CTAs per SM)
        constexpr int SM = embed_smem(true, true, ENT_U8) + 2 * TL * TP;
        if (mask == WM_MASK_ME) { if (tr) WM_LAUNCH_T((k_apply_ts<uint8_t, 0, true, ENT_U8>), ENT_U8, SM, tmI, tmW, tmO, a); else WM_LAUNCH_T((k_apply_ts<uint8_t, 0, false, ENT_U8>), ENT_U8, SM, tmI, tmW, tmO, a); }
        else { if (tr) WM_LAUNCH_T((k_apply_ts<uint8_t, 1, true, ENT_U8>), ENT_U8, SM, tmI, tmW, tmO, a); else WM_LAUNCH_T((k_apply_ts<uint8_t, 1, false, ENT_U8>), ENT_U8, SM, tmI, tmW, tmO, a); }
        return;
    }
#define WM_TS(PIX, SM)                                                                                                                 \
    if (mask == WM_MASK_ME) { if (tr) WM_LAUNCH((k_apply_ts<PIX, 0, true>), SM, tmI, tmW, tmO, a); else WM_LAUNCH((k_apply_ts<PIX, 0, false>), SM, tmI, tmW, tmO, a); } \
    else { if (tr) WM_LAUNCH((k_apply_ts<PIX, 1, true>), SM, tmI, tmW, tmO, a); else WM_LAUNCH((k_apply_ts<PIX, 1, false>), SM, tmI, tmW, tmO, a); }
    if (dtype == WM_F32) { WM_TS(float, embed_smem(true, false)) } else { WM_TS(uint8_t, embed_smem(true, true) + 2 * TL * TP) }
#undef WM_TS
}

void launch_apply_packed(int mask, int pixel_bytes, int luma, bool tma, dim3 grid, cudaStream_t st, const CUtensorMap& tmI, const CUtensorMap& tmW,
                         const EmbedArgs& a)
{
#define WM_PK(PIX, TMA, PB, OFF)                                                                                                       \
    if (mask == 2) WM_LAUNCH((k_apply<PIX, uint8_t, 2, false, TMA, false, PB, OFF>), embed_smem(TMA, sizeof(PIX) == 1), tmI, tmW, a);   \
    else if (mask == WM_MASK_ME) WM_LAUNCH((k_apply<PIX, uint8_t, 0, false, TMA, false, PB, OFF>), embed_smem(TMA, sizeof(PIX) == 1), tmI, tmW, a); \
    else WM_LAUNCH((k_apply<PIX, uint8_t, 1, false, TMA, false, PB, OFF>), embed_smem(TMA, sizeof(PIX) == 1), tmI, tmW, a);
    if (pixel_bytes == 2) {  // 4:2:2: the input is the u8 luma plane
        if (luma) { if (tma) { WM_PK(uint8_t, true, 2, 1) } else { WM_PK(uint8_t, false, 2, 1) } }
        else { if (tma) { WM_PK(uint8_t, true, 2, 0) } else { WM_PK(uint8_t, false, 2, 0) } }
    }
    else if (pixel_bytes == 4) { if (tma) { WM_PK(float, true, 4, 0) } else { WM_PK(float, false, 4, 0) } }
    else { if (tma) { WM_PK(float, true, 3, 0) } else { WM_PK(float, false, 3, 0) } }
#undef WM_PK
}

void launch_apply(int in_dtype, int out_dtype, int mask, bool tr, bool tma, dim3 grid, cudaStream_t st, const CUtensorMap& tmI,
                  const CUtensorMap& tmW, const EmbedArgs& a)
{
    if (in_dtype == WM_F32) {
        if (out_dtype == WM_F32) { if (tma) launch_apply_t<float, float, true>(mask, tr, grid, st, tmI, tmW, a); else launch_apply_t<float, float, false>(mask, tr, grid, st, tmI, tmW, a); }
        else { if (tma) launch_apply_t<float, uint8_t, true>(mask, tr, grid, st, tmI, tmW, a); else launch_apply_t<float, uint8_t, false>(mask, tr, grid, st, tmI, tmW, a); }
    } else {
        if (out_dtype == WM_F32) { if (tma) launch_apply_t<uint8_t, float, true>(mask, tr, grid, st, tmI, tmW, a); else launch_apply_t<uint8_t, float, false>(mask, tr, grid, st, tmI, tmW, a); }
        else { if (tma) launch_apply_t<uint8_t, uint8_t, true>(mask, tr, grid, st, tmI, tmW, a); else launch_apply_t<uint8_t, uint8_t, false>(mask, tr, grid, st, tmI, tmW, a); }
    }
}

}  // namespace wm
