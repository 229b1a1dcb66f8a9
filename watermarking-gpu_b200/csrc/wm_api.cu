// wm_api.cu — context, launch orchestration and the C ABI declared in include/wm_b200.h.
//
// Mirrors the reference's Watermark object (Watermark_GPU/Watermark.{hpp,cpp}): a ctx owns W, the strength
// factor and per-slot workspaces (the reference owns one staging texture => one object per concurrent caller;
// here each slot has its own stream + workspace so one ctx can pipeline frames).  There is no CPU fallback.
#include "../../include/wm_b200.h"
#include "wm_launch.h"

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

using namespace wm;

#define WM_VERSION_STR "wm_b200 0.1 (sm_100a)"

namespace {

constexpr int NSLOTS = 8;
thread_local std::string g_create_error;

struct WShared {  // W is shared between clones, like the ref-counted af::array (Watermark.cpp:31)
    int device = 0;
    float* row_major = nullptr;  // rows x cols
    float* col_major = nullptr;  // lazily transposed copy for WM_COL_MAJOR images
    std::mutex mu;
    ~WShared()
    {
        cudaSetDevice(device);
        if (row_major) cudaFree(row_major);
        if (col_major) cudaFree(col_major);
    }
};

struct TimedLaunch { int kernel; cudaEvent_t e0, e1; };

struct Slot {
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int batch_cap = 0;
    size_t part_cap = 0;     // doubles
    double* part = nullptr;  // sweep partials, then stats/detect partials (separate regions)
    unsigned* counters = nullptr;  // [3][batch_cap]
    Scal* scal = nullptr;
    ScalDbg* dbg = nullptr;
    Scal* scal_host = nullptr;  // pinned
    // results in flight on this slot's stream, delivered in order by finish_slot (several ops may be queued)
    struct Pending { int kind; int batch; float* scalar; int* status; size_t off; int64_t sstride; };  // kind 1 embed, 2 detect
    std::vector<Pending> queue;
    size_t host_cap = 0, host_used = 0;  // pinned result ring, in Scal units
    // staging for the host-buffer API / video driver
    void* stage_in = nullptr; size_t stage_in_cap = 0;
    void* stage_base = nullptr; size_t stage_base_cap = 0;
    void* stage_out = nullptr; size_t stage_out_cap = 0;
    void* maskp = nullptr; size_t maskp_cap = 0;  // NVF mask planes of a batch when p > 3 (k_nvfp)
    void* gray = nullptr; size_t gray_cap = 0;    // gray planes of a packed batch: f32 (k_packed_gray) or the u8 luma of 4:2:2 (k_packed_luma)
    std::vector<TimedLaunch> timed;
    // direct delivery of synchronous single-image ops (slot 0 only): mapped pinned result + device sequence / completion counters
    HostResult* hres = nullptr;      // pinned host memory
    HostResult* hres_dev = nullptr;  // its device alias
    unsigned* dl_words = nullptr;    // device: [0] apply completion counter, [1] generation word of the fused single-image kernels' hand-over
};

}  // namespace

struct wm_ctx {
    int device = 0, sms = 148;
    int64_t rows = 0, cols = 0;
    int p = 3;
    float psnr = 0.f, strength = 0.f;
    std::shared_ptr<WShared> w;
    Slot slots[NSLOTS];
    int opt_fp16 = 1, opt_timing = 0, opt_tma = 1, opt_serial = 0, opt_mma = 1, opt_f32_solve = 0;
    int opt_pdl = 1;         // WM_OPT_PDL: 2nd / 3rd kernel of an op launched with programmatic stream serialization
    int opt_run_mb = 136;       // WM_OPT_RUN_MB: frames of a run of the video driver (device frames) fill at most this many MB (4K u8: 17 frames)
    int opt_narrow_u8 = 1;      // WM_OPT_NARROW_U8: stats / apply of u8 TMA frames on 128-thread CTAs (8 lines per thread), four per SM
    int opt_padded_upload = 1;  // WM_OPT_PADDED_UPLOAD: host video frames with a small row padding are uploaded with it (one linear copy per frame)
    int opt_fused = 0;       // WM_OPT_FUSED_SINGLE: synchronous single-image detect as one cooperative kernel where the image fits (measured slower: off)
    int fused_failures = 0;  // cooperative launches that were refused (the op then takes the multi-kernel path)
    int opt_tma_store = 1;   // WM_OPT_TMA_STORE: apply kernel output through TMA stores where the shape allows (+8..10 % on the apply kernel)
    int opt_host_run = 4;    // frames per run of the video driver's host-frame path (WM_OPT_HOST_RUN_FRAMES)
    int opt_split_cost = 8;  // tile-times one more launch is assumed to cost when a batch is partitioned (WM_OPT_SPLIT_COST)
    bool inject_coef = false;
    float injected[8];
    std::string err;
    double ktime_ms[WM_K_COUNT] = {0};
    int64_t kcount[WM_K_COUNT] = {0};
    int64_t launches = 0;
    std::vector<cudaEvent_t> event_pool;
    // CUDA-graph cache of the synchronous single-image calls (the reference's loops_for_test protocol calls the same
    // arrays over and over: main.cpp:175-222): key = every argument the launch sequence depends on
    struct GraphEntry { std::string key; int seen; cudaGraphExec_t exec; int launches; };
    std::vector<GraphEntry> graphs;
    int opt_graphs = 1;
};

namespace {

struct PdlScope {  // launches inside the scope carry the programmatic-serialization attribute (wm_launch.h)
    bool prev;
    explicit PdlScope(bool on) : prev(wm::pdl_next()) { wm::pdl_next() = on; }
    ~PdlScope() { wm::pdl_next() = prev; }
};

int fail(wm_ctx* c, int code, const std::string& msg)
{
    if (c) c->err = msg; else g_create_error = msg;
    return code;
}
#define CU(call)                                                                                      \
    do {                                                                                              \
        cudaError_t e_ = (call);                                                                      \
        if (e_ != cudaSuccess)                                                                        \
            return fail(ctx, WM_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));        \
    } while (0)

// The packed 8-bit layouts: bytes per pixel (0 = not a packed layout), whether B comes before R, the byte of a pixel that holds its
// luma (-1: a colour layout, whose RGB gray is computed) and the bytes the packed apply kernel moves in one aligned access of a thread's
// four pixels.  Every other place reads these facts from here, so a packed layout is described once.
struct PackedFmt { int bytes; bool bgr; int luma; int apply_vec; const char* name; };
constexpr PackedFmt PLANAR = {0, false, -1, 0, ""};
PackedFmt packed_fmt(int layout)
{
    switch (layout) {
    case WM_PACKED_RGB: return {3, false, -1, 16, "RGB"};
    case WM_PACKED_BGR: return {3, true, -1, 16, "BGR"};
    case WM_PACKED_RGBA: return {4, false, -1, 16, "RGBA"};
    case WM_PACKED_BGRA: return {4, true, -1, 16, "BGRA"};
    case WM_PACKED_YUYV: return {2, false, 0, 8, "YUYV"};
    case WM_PACKED_UYVY: return {2, false, 1, 8, "UYVY"};
    default: return PLANAR;
    }
}
// bytes of the gray plane one image of a packed layout fills in a slot: f32 L x P for the RGB gray; for 4:2:2 the u8 luma at a pitch of
// round_up(P, 16), so that its rows are TMA-loadable like a caller's Y plane at that pitch
long long luma_pitch(int P) { return ((long long)P + 15) / 16 * 16; }
size_t gray_plane_bytes(const PackedFmt& f, int L, int P)
{
    return f.luma >= 0 ? (size_t)L * (size_t)luma_pitch(P) : (size_t)L * (size_t)P * sizeof(float);
}
// An image reduced to planes of L lines x P pixels; ld and pstride are in elements.  A packed image is one plane of L = rows lines of
// P = cols pixels, ld in bytes, dtype u8 and channels = bytes per pixel.
struct View {
    void* ptr; int L, P; long long ld, pstride; int channels; int dtype; bool transposed;
    int layout; PackedFmt fmt;  // fmt.bytes == 0: a planar image
    bool packed() const { return fmt.bytes != 0; }
    long long elem() const { return dtype == WM_F32 ? 4 : 1; }
    int planes() const { return packed() ? 1 : channels; }
    long long row_bytes() const { return (long long)P * (packed() ? fmt.bytes : elem()); }  // of a line's pixels, without its padding
    long long pitch() const { return ld * elem(); }
    long long plane_bytes() const { return pstride * elem(); }
    long long extent() const { return (planes() - 1) * plane_bytes() + (L - 1) * pitch() + row_bytes(); }  // first byte to past the last pixel
};

// Compares an image on the device with the watermark's dims, before make_view checks the rest of it.  A host image is compared once it
// is staged, so its descriptor is checked first.
int check_dims(wm_ctx* ctx, const wm_image* im)
{
    if (!im || !im->data) return fail(ctx, WM_ERR_ARG, "null image");
    if (im->rows != ctx->rows || im->cols != ctx->cols)
        return fail(ctx, WM_ERR_DIMS, "image dims " + std::to_string(im->rows) + "x" + std::to_string(im->cols) +
                                          " != watermark dims " + std::to_string(ctx->rows) + "x" + std::to_string(ctx->cols));
    return WM_OK;
}
// Checks an image descriptor and reduces it to a View.  allow_rgb: three planes are taken (base / out).  allow_packed: packed 8-bit
// images are taken (the embed and detect entry points).  channels_from_layout: a packed image's channels field is not read but implied
// by its layout (the video driver's frames, which have no such field).
int make_view(wm_ctx* ctx, const wm_image* im, View* v, bool allow_rgb, bool allow_packed = false, bool channels_from_layout = false)
{
    if (!im || !im->data) return fail(ctx, WM_ERR_ARG, "null image");
    if (im->rows < 1 || im->cols < 1) return fail(ctx, WM_ERR_ARG, "image rows and cols must be positive");
    v->ptr = im->data;
    v->layout = im->layout;
    v->fmt = packed_fmt(im->layout);
    if (v->packed()) {
        const PackedFmt& f = v->fmt;
        const std::string what = std::string("a packed ") + f.name + " image";
        if (!allow_packed) return fail(ctx, WM_ERR_ARG, std::string("packed ") + f.name + " images are taken by the wm_embed* and wm_detect* entry points only");
        if (im->dtype != WM_U8 || (im->channels != f.bytes && !channels_from_layout))
            return fail(ctx, WM_ERR_ARG, what + " has dtype WM_U8 and " + std::to_string(f.bytes) + " channels");
        v->transposed = false;
        v->L = (int)im->rows;
        v->P = (int)im->cols;
        v->channels = f.bytes;
        v->dtype = WM_U8;
        v->ld = im->ld > 0 ? im->ld : v->row_bytes();
        if (v->ld < v->row_bytes()) return fail(ctx, WM_ERR_ARG, what + ": ld (bytes) smaller than " + std::to_string(f.bytes) + " * cols");
        if (f.luma >= 0 && im->cols % 2) return fail(ctx, WM_ERR_ARG, what + " has an even number of cols (4:2:2 pairs pixels)");
        v->pstride = (long long)v->L * v->ld;
        return WM_OK;
    }
    if (im->layout != WM_COL_MAJOR && im->layout != WM_ROW_MAJOR) return fail(ctx, WM_ERR_ARG, "bad layout");
    if (im->dtype != WM_F32 && im->dtype != WM_U8) return fail(ctx, WM_ERR_ARG, "bad dtype");
    const int ch = im->channels <= 0 ? 1 : im->channels;
    if (ch != 1 && !(allow_rgb && ch == 3)) return fail(ctx, WM_ERR_ARG, "channels must be 1 (or 3 for base/out)");
    v->transposed = im->layout == WM_COL_MAJOR;
    v->L = (int)(v->transposed ? im->cols : im->rows);
    v->P = (int)(v->transposed ? im->rows : im->cols);
    v->ld = im->ld > 0 ? im->ld : v->P;
    if (v->ld < v->P) return fail(ctx, WM_ERR_ARG, "ld smaller than the contiguous dimension");
    v->pstride = im->plane_stride > 0 ? im->plane_stride : (long long)v->L * v->ld;
    v->channels = ch;
    v->dtype = im->dtype;
    return WM_OK;
}

bool vec_ok(const void* p, long long ld, long long bstride, long long pstride, int dtype)
{
    const uintptr_t al = dtype == WM_F32 ? 16 : 4;
    return ((uintptr_t)p % al == 0) && (ld % 4 == 0) && (bstride % 4 == 0) && (pstride % 4 == 0);
}
// alignment level of a packed image's rows (launch_packed_gray): 2 = pointer, ld and batch stride are multiples of `vec` bytes (16; 8 for the
// 4:2:2 apply, whose thread accesses 8 bytes), 1 = of 4 bytes, 0
int packed_align(const void* p, long long ld, long long bstride, long long vec = 16)
{
    auto al = [&](long long m) { return (uintptr_t)p % (uintptr_t)m == 0 && ld % m == 0 && bstride % m == 0; };
    return al(vec) ? 2 : al(4) ? 1 : 0;
}


// batch stride conventions (include/wm_b200.h): 0 means dense (plane_stride * channels, i.e. L * ld * channels for dense planes); a stride
// smaller than one image would make the images of a batch overlap.  Resolved once, so the tensor maps, the plain loaders and the
// apply kernel's base / out addressing all see the same number.
int resolve_stride(wm_ctx* ctx, const View& v, int batch, int64_t* stride, const char* what)
{
    // elements spanned by one image, the padding of its last line included
    const long long one = v.pstride * (v.planes() - 1) + (long long)v.L * v.ld;
    if (*stride == 0) *stride = v.pstride * v.planes();
    if (batch > 1 && *stride < one) return fail(ctx, WM_ERR_ARG, std::string(what) + " batch stride smaller than one image");
    return WM_OK;
}
// [first, last) bytes touched by a batch
void byte_range(const View& v, int64_t stride, int batch, uintptr_t* lo, uintptr_t* hi)
{
    *lo = (uintptr_t)v.ptr;
    *hi = (uintptr_t)v.ptr + (uintptr_t)((long long)(batch - 1) * stride * v.elem() + v.extent());
}

int finish_slot(wm_ctx* ctx, Slot& s);
void clear_graphs(wm_ctx* ctx)
{
    for (auto& g : ctx->graphs) if (g.exec) cudaGraphExecDestroy(g.exec);
    ctx->graphs.clear();
}

int ensure_slot(wm_ctx* ctx, Slot& s, int batch, int gx_max, int nsweep, int nframe)
{
    const size_t need_part = (size_t)batch * ((size_t)nsweep * NTOT + (size_t)gx_max * 3 + (size_t)SMAXG * NTOT);
    if (batch > s.batch_cap || need_part > s.part_cap) clear_graphs(ctx);  // cached graphs point into these buffers
    if ((batch > s.batch_cap || need_part > s.part_cap) && !s.queue.empty()) {
        const int r = finish_slot(ctx, s);  // buffers in use by queued work are about to be replaced
        if (r < 0) return r;
    }
    if (batch > s.batch_cap) {
        if (s.counters) cudaFree(s.counters);
        if (s.scal) cudaFree(s.scal);
        if (s.dbg) cudaFree(s.dbg);
        if (s.scal_host) cudaFreeHost(s.scal_host);
        s.counters = nullptr; s.scal = nullptr; s.dbg = nullptr; s.scal_host = nullptr;
        CU(cudaMalloc(&s.counters, sizeof(unsigned) * (3 + SMAXG) * batch));  // [3][batch] last-block counters + [batch][SMAXG] group counters of the sweep
        CU(cudaMemsetAsync(s.counters, 0, sizeof(unsigned) * (3 + SMAXG) * batch, s.stream));
        CU(cudaMalloc(&s.scal, sizeof(Scal) * batch));
        CU(cudaMemsetAsync(s.scal, 0, sizeof(Scal) * batch, s.stream));
        CU(cudaMalloc(&s.dbg, sizeof(ScalDbg) * batch));
        CU(cudaMemsetAsync(s.dbg, 0, sizeof(ScalDbg) * batch, s.stream));
        s.host_cap = (size_t)std::max(batch * 16, 256);  // 16 ops of this batch size may be queued before a delivery is forced
        s.host_used = 0;
        CU(cudaMallocHost(&s.scal_host, sizeof(Scal) * s.host_cap));
        s.batch_cap = batch;
    }
    const size_t need = need_part;
    (void)nframe;
    if (need > s.part_cap) {
        if (s.part) cudaFree(s.part);
        s.part = nullptr;
        CU(cudaMalloc(&s.part, need * sizeof(double)));
        s.part_cap = need;
    }
    return WM_OK;
}

int ensure_stage(wm_ctx* ctx, void** p, size_t* cap, size_t bytes)
{
    if (bytes > *cap) {
        if (*p) cudaFree(*p);
        *p = nullptr;
        CU(cudaMalloc(p, bytes));
        *cap = bytes;
    }
    return WM_OK;
}

const float* w_for(wm_ctx* ctx, bool transposed, cudaStream_t st, int* rc)
{
    *rc = WM_OK;
    WShared& w = *ctx->w;
    if (!transposed) return w.row_major;
    std::lock_guard<std::mutex> g(w.mu);
    if (!w.col_major) {
        if (cudaMalloc(&w.col_major, sizeof(float) * ctx->rows * ctx->cols) != cudaSuccess) {
            *rc = fail(ctx, WM_ERR_CUDA, "cudaMalloc(W col-major)");
            return nullptr;
        }
        launch_transpose(w.row_major, w.col_major, (int)ctx->rows, (int)ctx->cols, st);
        cudaStreamSynchronize(st);  // other slots/clones may use it right away
    }
    return w.col_major;
}

struct Geo { int L, P, tiles_p, tiles_l, ntiles; };
Geo geo(int L, int P)
{
    Geo g;
    g.L = L; g.P = P;
    g.tiles_p = (P + TP - 1) / TP;
    g.tiles_l = (L + TL - 1) / TL;
    g.ntiles = g.tiles_p * g.tiles_l;
    return g;
}

// One launch = at most ONE wave of resident CTAs (persistent tile loops; a partial second wave would leave most SMs idle for
// a whole tile loop): 2 per SM for the detector, SWEEP_CTAS_PER_SM / EMBED_CTAS_PER_SM for the sweep and stats / apply.  The
// wave is split over the images of the launch as evenly as possible: image b gets base + (b < extra) CTAs, gridDim.x is the
// larger of the two and the surplus CTAs exit at once.  When that split is uneven (64 images on 444 CTAs: 60 get 7, 4 get 6
// and set the pace), the batch is launched as sub-batches whose own splits are even enough to pay for the extra launch —
// images are independent and every per-image buffer is indexed by the global image number (kernel argument b0).
struct SubBatch { int b0, nb, base, extra; };
struct Plan {
    std::vector<SubBatch> sweep, embed, detect;
    int nsweep, nframe, gx_stats, gx_detect;  // partial rows per image (strides) of the three families
};
void split_wave(int cap, int batch, int ntiles, int* base, int* extra)
{
    *base = cap / batch; *extra = cap % batch;
    if (*base < 1) { *base = 1; *extra = 0; }
    if (*base >= ntiles) { *base = ntiles; *extra = 0; }
}
// duration of one wave of `cap` CTAs over m images, in tile-times of the slowest CTA
int wave_cost(int cap, int m, int ntiles)
{
    if (m >= cap) return ((m + cap - 1) / cap) * ntiles;
    const int base = cap / m;
    return base >= ntiles ? 1 : (ntiles + base - 1) / base;
}
// a split must promise at least 8 % (the model ignores second-order effects; measured: a 4 % promise lost 10 %)
static bool worth(long long split, long long single) { return split * 100 < single * 92; }
// split_cost: what one more launch costs (launch gap + ramp / tail of one more wave), in tile-times
std::vector<SubBatch> partition(int cap, int batch, int ntiles, int split_cost)
{
    std::vector<SubBatch> out;
    int b0 = 0, rest = batch;
    while (rest > 0) {
        int take = rest;
        if (rest > cap && rest % cap != 0) {
            // more images than CTAs: whole waves of one CTA per image first, the remainder shares a wave of its own
            const int full = (rest / cap) * cap;
            if (worth(wave_cost(cap, full, ntiles) + split_cost + wave_cost(cap, rest - full, ntiles), wave_cost(cap, rest, ntiles))) take = full;
        } else if (rest > 1 && rest < cap && cap % rest != 0) {
            const int single = wave_cost(cap, rest, ntiles);
            int best = single;
            for (int na = 1; na < rest; na++) {
                const int c = wave_cost(cap, na, ntiles) + split_cost + wave_cost(cap, rest - na, ntiles);
                if (c < best && worth(c, single)) { best = c; take = na; }
            }
        }
        SubBatch sb;
        sb.b0 = b0; sb.nb = take;
        split_wave(cap, take, ntiles, &sb.base, &sb.extra);
        out.push_back(sb);
        b0 += take; rest -= take;
    }
    return out;
}
int max_rows(const std::vector<SubBatch>& v)
{
    int m = 1;
    for (const SubBatch& sb : v) m = std::max(m, sb.base + (sb.extra > 0 ? 1 : 0));
    return m;
}
// narrow: stats / apply of u8 TMA frames run on 128-thread CTAs, four per SM (WM_OPT_NARROW_U8)
Plan plan(const wm_ctx* ctx, const Geo& g, int batch, int dtype, bool narrow = false)
{
    Plan p;
    p.detect = partition((narrow ? DETECT_CTAS_PER_SM_U8N : detect_ctas_per_sm(dtype == WM_U8)) * ctx->sms, batch, g.ntiles, ctx->opt_split_cost);
    p.embed = partition((narrow ? EMBED_CTAS_PER_SM_U8 : EMBED_CTAS_PER_SM) * ctx->sms, batch, g.ntiles, ctx->opt_split_cost);
    p.sweep = partition(SWEEP_CTAS_PER_SM * ctx->sms, batch, g.ntiles, ctx->opt_split_cost);
    p.nframe = 0;  // the frame ring is shared by the sweep blocks
    p.nsweep = max_rows(p.sweep);
    p.gx_detect = max_rows(p.detect);
    p.gx_stats = max_rows(p.embed);
    return p;
}

// ---- timing brackets ----
cudaEvent_t get_event(wm_ctx* ctx)
{
    if (!ctx->event_pool.empty()) {
        cudaEvent_t e = ctx->event_pool.back();
        ctx->event_pool.pop_back();
        return e;
    }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}
struct KTimer {
    wm_ctx* ctx; Slot& s; int k; cudaEvent_t e0 = nullptr, e1 = nullptr;
    KTimer(wm_ctx* c, Slot& sl, int kernel) : ctx(c), s(sl), k(kernel)
    {
        ctx->launches++;
        if (ctx->opt_timing) { e0 = get_event(ctx); e1 = get_event(ctx); cudaEventRecord(e0, s.stream); }
    }
    ~KTimer()
    {
        if (e0) { cudaEventRecord(e1, s.stream); s.timed.push_back({k, e0, e1}); }
    }
};
void drain_timers(wm_ctx* ctx, Slot& s)
{
    for (auto& t : s.timed) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, t.e0, t.e1) == cudaSuccess) { ctx->ktime_ms[t.kernel] += ms; ctx->kcount[t.kernel]++; }
        ctx->event_pool.push_back(t.e0);
        ctx->event_pool.push_back(t.e1);
    }
    s.timed.clear();
}

// ---- TMA tensor maps (cuTensorMapEncodeTiled through the runtime's driver entry point: no libcuda link) ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_fn()
{
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return (EncodeTiledFn)p;
    }();
    return fn;
}
// f32 / u8 tensor (pixel, line, image) with a (boxP x boxL x 1) box; out-of-bounds elements are zero-filled.
// boxP is given in f32 terms (SW or TP); u8 image boxes are U8_ROW (144) pixels wide so that the row is 16-byte sized.
bool make_tmap(CUtensorMap* tm, int dtype, const void* ptr, int P, int L, int B, long long ld, long long bstride, int boxP, int boxL, int u8_box = U8_ROW)
{
    EncodeTiledFn fn = encode_fn();
    if (!fn) return false;
    const int es = dtype == WM_F32 ? 4 : 1;
    const cuuint64_t dims[3] = {(cuuint64_t)P, (cuuint64_t)L, (cuuint64_t)std::max(B, 1)};
    const long long bs = (B > 1 && bstride > 0) ? bstride : (long long)L * ld;
    const cuuint64_t strides[2] = {(cuuint64_t)ld * es, (cuuint64_t)bs * es};
    const cuuint32_t box[3] = {(cuuint32_t)(dtype == WM_F32 ? boxP : u8_box), (cuuint32_t)boxL, 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    return fn(tm, dtype == WM_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void*>(ptr), dims,
              strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
bool tma_ok(const wm_ctx* ctx, const View& v, long long bstride, int batch)
{
    const long long al = v.dtype == WM_F32 ? 4 : 16;  // strides must be multiples of 16 bytes
    return ctx->opt_tma && ((uintptr_t)v.ptr % 16 == 0) && (v.ld % al == 0) && (v.P % 4 == 0) &&
           (batch == 1 || bstride % al == 0) && encode_fn() != nullptr;
}

// copy the op's per-image scalars into the slot's pinned ring (in stream order) and queue their delivery
int push_result(wm_ctx* ctx, Slot& s, int kind, int batch)
{
    if (s.host_used + (size_t)batch > s.host_cap || s.queue.size() >= 32) {
        const int r = finish_slot(ctx, s);  // ring full: deliver what is queued (the kernels of this op are already enqueued)
        if (r < 0) return r;
    }
    CU(cudaMemcpyAsync(s.scal_host + s.host_used, s.scal, sizeof(Scal) * batch, cudaMemcpyDeviceToHost, s.stream));
    s.queue.push_back({kind, batch, nullptr, nullptr, s.host_used, 1});
    s.host_used += (size_t)batch;
    return WM_OK;
}

SweepArgs sweep_args(wm_ctx* ctx, Slot& s, const View& v, long long bstride, int batch, const Geo& g, const Plan& pl)
{
    SweepArgs a;
    memset(&a, 0, sizeof a);
    a.img = v.ptr; a.ld = v.ld; a.bstride = bstride;
    a.L = g.L; a.P = g.P; a.tiles_p = g.tiles_p; a.ntiles = g.ntiles;
    a.nsweep = pl.nsweep; a.nframe = pl.nframe;
    a.vec_ok = vec_ok(v.ptr, v.ld, bstride, 0, v.dtype);
    a.transposed = v.transposed;
    a.solve_f32 = ctx->opt_f32_solve;
    a.part = s.part;
    a.counter = s.counters;
    a.gcounter = s.counters + 3 * (size_t)s.batch_cap;
    a.gpart = s.part + (size_t)batch * ((size_t)pl.nsweep * NTOT + (size_t)std::max(pl.gx_stats, pl.gx_detect) * 3);
    a.scal = s.scal; a.dbg = s.dbg;
    return a;
}

// Single-image fused kernels (wm_kernels.cuh: k_detect1, k_embed1): `grid` CTAs keep at most `nst` tiles each in shared memory, and their
// frame-ring slices must stay in the one-warp-per-pixel mode (<= 96 ring pixels per CTA; the per-thread mode needs more scratch than they have)
bool fused_fits(const Geo& g, int grid, int nst, bool with_ring)
{
    if (grid < 1 || (long long)g.ntiles > (long long)nst * grid) return false;
    if (!with_ring) return true;
    const long long L = g.L, P = g.P;
    const long long ntop = std::min(2LL, L), lbot = std::max(2LL, L - 2), nbot = std::max(0LL, L - lbot), nmid = std::max(0LL, L - 4);
    const long long ncl = std::min(2LL, P), pright = std::max(2LL, P - 2), ncr = std::max(0LL, P - pright);
    const long long count = (ntop + nbot) * P + nmid * (ncl + ncr);
    const int nlong = g.ntiles % grid;
    const bool light_only = nlong != 0 && 2 * (grid - nlong) >= grid;
    const int nring = light_only ? grid - nlong : grid;
    return (count + nring - 1) / nring <= 96;
}

// enqueue the Rx sweep (+ solve), or the injection of debug coefficients
int enqueue_sweep(wm_ctx* ctx, Slot& s, const View& v, long long bstride, int batch, const Geo& g, const Plan& pl)
{
    if (ctx->inject_coef) {
        for (int b = 0; b < batch; b++) {
            Scal h;
            memset(&h, 0, sizeof h);
            memcpy(h.coef, ctx->injected, sizeof h.coef);
            CU(cudaMemcpyAsync(s.scal + b, &h, sizeof h, cudaMemcpyHostToDevice, s.stream));
            CU(cudaStreamSynchronize(s.stream));  // h is a stack temporary
        }
        return WM_OK;
    }
    SweepArgs a = sweep_args(ctx, s, v, bstride, batch, g, pl);
    CUtensorMap tmI;
    memset(&tmI, 0, sizeof tmI);
    bool tma = tma_ok(ctx, v, bstride, batch);
    if (tma) tma = make_tmap(&tmI, v.dtype, v.ptr, g.P, g.L, batch, v.ld, bstride, SW, TL + 2);
    {
        KTimer t(ctx, s, WM_K_SWEEP);
        for (const SubBatch& sb : pl.sweep) {
            a.b0 = sb.b0; a.nblk_base = sb.base; a.nblk_extra = sb.extra;
            launch_sweep(v.dtype, ctx->opt_fp16 ? (ctx->opt_mma ? 2 : 1) : 0, tma, dim3(sb.base + (sb.extra > 0 ? 1 : 0), sb.nb), s.stream, tmI, a);
        }
    }
    CU(cudaGetLastError());
    return WM_OK;
}

// NVF mask with a p x p window, p > 3 (Watermark.cpp:96-114 with -Dp=5/7/9): one dense L x P plane per image of the batch
int enqueue_nvf_planes(wm_ctx* ctx, Slot& s, const View& v, long long bstride, int batch, const Geo& g, float* dst = nullptr)
{
    const size_t plane = (size_t)g.L * g.P;
    if (!dst) {
        const size_t need = plane * batch * sizeof(float);
        if (need > s.maskp_cap) {
            if (!s.queue.empty()) { const int r = finish_slot(ctx, s); if (r < 0) return r; }
            CU(cudaStreamSynchronize(s.stream));
            clear_graphs(ctx);
            int rc;
            if ((rc = ensure_stage(ctx, &s.maskp, &s.maskp_cap, need))) return rc;
        }
        dst = (float*)s.maskp;
    }
    NvfpArgs a;
    a.img = v.ptr; a.ld = v.ld; a.bstride = bstride;
    a.L = g.L; a.P = g.P; a.tiles_p = g.tiles_p; a.ntiles = g.ntiles;
    a.vec_ok = vec_ok(v.ptr, v.ld, bstride, 0, v.dtype);
    a.dst = dst; a.dst_bstride = (long long)plane;
    const int gx = std::max(1, std::min(g.ntiles, (4 * ctx->sms + batch - 1) / batch));
    launch_nvfp(v.dtype, ctx->p, v.transposed, dim3(gx, batch), s.stream, a);
    CU(cudaGetLastError());
    return WM_OK;
}

// the slot's f32 gray planes hold at least `need` bytes
int reserve_gray(wm_ctx* ctx, Slot& s, size_t need)
{
    if (need > s.gray_cap) {  // queued work and captured graphs may still read the old planes
        if (!s.queue.empty()) { const int r = finish_slot(ctx, s); if (r < 0) return r; }
        CU(cudaStreamSynchronize(s.stream));
        clear_graphs(ctx);
        const int rc = ensure_stage(ctx, &s.gray, &s.gray_cap, need);
        if (rc) return rc;
    }
    return WM_OK;
}
// Packed batch: its gray goes into the slot's planes, and *v / *stride become that gray batch.
// Colour layouts: the RGB gray, dense f32, so the op runs on it exactly as on a caller's dense f32 gray batch (same tiles, launch plan and
// partial sums: the scalars of the composed path).  4:2:2 layouts: the luma, u8 at a pitch of round_up(P, 16), so the op runs on it exactly
// as on a caller's u8 Y plane at that pitch (the same u8 kernels, narrow where TMA holds, and plan: the Y-plane bits).
int enqueue_packed_gray(wm_ctx* ctx, Slot& s, View* v, int64_t* stride, int batch)
{
    const PackedFmt& f = v->fmt;
    const size_t plane = gray_plane_bytes(f, v->L, v->P);
    const int rc = reserve_gray(ctx, s, plane * batch);
    if (rc) return rc;
    const int al = packed_align(v->ptr, v->ld, *stride);
    if (f.luma >= 0) {
        const long long lp = luma_pitch(v->P);
        launch_packed_luma((const uint8_t*)v->ptr, v->ld, *stride, batch, f.luma, (uint8_t*)s.gray, lp, v->L, v->P, al, 8 * ctx->sms, s.stream);
        v->ld = lp; v->dtype = WM_U8;
    } else {
        launch_packed_gray((const uint8_t*)v->ptr, v->ld, *stride, batch, f.bytes, f.bgr, (float*)s.gray, v->L, v->P, al, 8 * ctx->sms, s.stream);
        v->ld = v->P; v->dtype = WM_F32;
    }
    ctx->launches++;
    CU(cudaGetLastError());
    v->ptr = s.gray; v->pstride = (long long)v->L * v->ld; v->channels = 1;
    v->layout = WM_ROW_MAJOR;
    v->fmt = PLANAR;
    *stride = (int64_t)v->pstride;
    return WM_OK;
}

size_t stats_part_offset(const Plan& pl, int batch) { return (size_t)batch * (size_t)pl.nsweep * NTOT; }

// the pieces of a slot that direct delivery needs (created on first use)
int ensure_direct(wm_ctx* ctx, Slot& s)
{
    if (s.hres) return WM_OK;
    CU(cudaHostAlloc(&s.hres, sizeof(HostResult), cudaHostAllocMapped));
    memset(s.hres, 0, sizeof(HostResult));
    CU(cudaHostGetDevicePointer((void**)&s.hres_dev, s.hres, 0));
    CU(cudaMalloc(&s.dl_words, 2 * sizeof(unsigned)));
    CU(cudaMemset(s.dl_words, 0, 2 * sizeof(unsigned)));
    return WM_OK;
}
Deliver deliver_args(Slot& s, bool direct)
{
    Deliver d;
    d.host = direct ? s.hres_dev : nullptr;
    d.done = direct ? s.dl_words : nullptr;
    return d;
}

int do_embed(wm_ctx* ctx, int slot, const wm_image* in, const wm_image* base, wm_image* out, int64_t in_stride,
             int64_t base_stride, int64_t out_stride, int batch, int mask, bool direct = false)
{
    if (!ctx) return WM_ERR_ARG;
    if (slot < 0 || slot >= NSLOTS) return fail(ctx, WM_ERR_ARG, "bad slot");
    if (mask != WM_MASK_ME && mask != WM_MASK_NVF) return fail(ctx, WM_ERR_ARG, "bad mask type");
    if (batch < 1 || batch > 65535) return fail(ctx, WM_ERR_ARG, "batch must be 1..65535");
    View vi, vb, vo;
    int rc;
    if ((rc = check_dims(ctx, in)) || (rc = make_view(ctx, in, &vi, false, true))) return rc;
    if ((rc = check_dims(ctx, base ? base : in)) || (rc = make_view(ctx, base ? base : in, &vb, true, true))) return rc;
    if ((rc = check_dims(ctx, out)) || (rc = make_view(ctx, out, &vo, true, true))) return rc;
    // a packed input: base and out are packed images of its layout, so the apply kernel reads its format from them
    const bool packed = vi.packed();
    if (packed || vb.packed() || vo.packed()) {
        if (!packed) return fail(ctx, WM_ERR_ARG, "a packed base or output needs the same packed image as the input");
        if (vb.layout != vi.layout || vb.ptr != vi.ptr || vb.ld != vi.ld)
            return fail(ctx, WM_ERR_ARG, "with a packed input, base must be NULL or the same image (pointer, layout, ld)");
        if (vo.layout != vi.layout) return fail(ctx, WM_ERR_ARG, "with a packed input, out must be a packed image of the same layout");
        if (!base) base_stride = in_stride;  // NULL base: the input batch itself
    }
    if (vb.transposed != vi.transposed || vo.transposed != vi.transposed) return fail(ctx, WM_ERR_ARG, "in/base/out layouts differ");
    if (vb.dtype != vi.dtype) return fail(ctx, WM_ERR_ARG, "base dtype must equal input dtype");
    if (vo.channels != vb.channels) return fail(ctx, WM_ERR_ARG, "out channels != base channels");
    if ((rc = resolve_stride(ctx, vi, batch, &in_stride, "in"))) return rc;
    if ((rc = resolve_stride(ctx, vb, batch, &base_stride, "base"))) return rc;
    if ((rc = resolve_stride(ctx, vo, batch, &out_stride, "out"))) return rc;
    if (packed && batch > 1 && base_stride != in_stride) return fail(ctx, WM_ERR_ARG, "with a packed input, base must be the same batch (stride)");
    {
        uintptr_t ilo, ihi, olo, ohi;
        byte_range(vi, in_stride, batch, &ilo, &ihi);
        byte_range(vo, out_stride, batch, &olo, &ohi);
        if (olo < ihi && ilo < ohi) return fail(ctx, WM_ERR_ARG, "out must not overlap the gray input (neighbour reads race with stores)");
    }
    CU(cudaSetDevice(ctx->device));
    Slot& s = ctx->slots[slot];
    if (packed && (rc = enqueue_packed_gray(ctx, s, &vi, &in_stride, batch))) return rc;
    const Geo g = geo(vi.L, vi.P);
    const bool narrow = ctx->opt_narrow_u8 && vi.dtype == WM_U8 && tma_ok(ctx, vi, in_stride, batch);
    const Plan pl = plan(ctx, g, batch, vi.dtype, narrow);
    if ((rc = ensure_slot(ctx, s, batch, std::max(pl.gx_stats, pl.gx_detect), pl.nsweep, pl.nframe))) return rc;
    const float* W = w_for(ctx, vi.transposed, s.stream, &rc);
    if (rc) return rc;
    if (mask == WM_MASK_ME) {
        if ((rc = enqueue_sweep(ctx, s, vi, in_stride, batch, g, pl))) return rc;
    }
    EmbedArgs ea;
    memset(&ea, 0, sizeof ea);
    ea.img = vi.ptr; ea.ld = vi.ld; ea.bstride = in_stride;
    ea.W = W;
    ea.L = g.L; ea.P = g.P; ea.tiles_p = g.tiles_p; ea.ntiles = g.ntiles;
    ea.vec_ok = vec_ok(vi.ptr, vi.ld, in_stride, 0, vi.dtype);
    ea.w_vec_ok = (g.P % 4 == 0);
    ea.strength = ctx->strength;
    ea.pstride = pl.gx_stats;
    const bool planes = mask == WM_MASK_NVF && ctx->p != 3;  // larger NVF windows: the mask comes from k_nvfp's planes
    const int kmask = planes ? 2 : mask;
    ea.maskp = nullptr; ea.mask_bstride = (long long)g.L * g.P;
    ea.part = s.part + stats_part_offset(pl, batch);
    ea.counter = s.counters + s.batch_cap;
    ea.scal = s.scal; ea.dbg = s.dbg;
    ea.base = vb.ptr; ea.base_ld = vb.ld; ea.base_bstride = base_stride; ea.base_pstride = vb.pstride;
    ea.out = vo.ptr; ea.out_ld = vo.ld; ea.out_bstride = out_stride; ea.out_pstride = vo.pstride;
    ea.channels = vb.channels;
    ea.same_base = (vb.ptr == vi.ptr && vb.ld == vi.ld && base_stride == in_stride && vb.channels == 1);
    ea.dl = deliver_args(s, direct && batch == 1);
    // packed base / out: alignment levels (the apply kernel's vector access, word or byte accesses)
    ea.base_vec_ok = packed ? packed_align(vb.ptr, vb.ld, base_stride, vb.fmt.apply_vec) : vec_ok(vb.ptr, vb.ld, base_stride, vb.channels > 1 ? vb.pstride : 0, vb.dtype);
    ea.out_vec_ok = packed ? packed_align(vo.ptr, vo.ld, out_stride, vo.fmt.apply_vec) : vec_ok(vo.ptr, vo.ld, out_stride, vo.channels > 1 ? vo.pstride : 0, vo.dtype);
    CUtensorMap tmI, tmW;
    memset(&tmI, 0, sizeof tmI);
    memset(&tmW, 0, sizeof tmW);
    bool tma = tma_ok(ctx, vi, in_stride, batch);
    if (tma) tma = make_tmap(&tmI, vi.dtype, vi.ptr, g.P, g.L, batch, vi.ld, in_stride, SW, TL + 2) &&
                   make_tmap(&tmW, WM_F32, W, g.P, g.L, 1, g.P, 0, TP, TL);
    {
        KTimer t(ctx, s, mask == WM_MASK_ME ? WM_K_ME_STATS : WM_K_NVF_STATS);
        if (planes) {
            if ((rc = enqueue_nvf_planes(ctx, s, vi, in_stride, batch, g))) return rc;
            ea.maskp = (const float*)s.maskp;
        }
        PdlScope pdl(ctx->opt_pdl && mask == WM_MASK_ME && !ctx->opt_timing && !ctx->inject_coef);  // the Rx sweep of this op precedes
        for (const SubBatch& sb : pl.embed) {
            ea.b0 = sb.b0; ea.nblk_base = sb.base; ea.nblk_extra = sb.extra;
            launch_stats(vi.dtype, kmask, vi.transposed, tma, narrow, dim3(sb.base + (sb.extra > 0 ? 1 : 0), sb.nb), s.stream, tmI, tmW, ea);
        }
    }
    CU(cudaGetLastError());
    {
        KTimer t(ctx, s, mask == WM_MASK_ME ? WM_K_APPLY : WM_K_APPLY_NVF);
        // WM_OPT_TMA_STORE (default on): gray output of the same dtype, base = input, TMA-loadable input and a TMA-storable output
        CUtensorMap tmO;
        memset(&tmO, 0, sizeof tmO);
        PdlScope pdl(ctx->opt_pdl && !ctx->opt_timing && !planes);  // the stats pass of this op precedes
        bool ts = ctx->opt_tma_store && tma && ea.same_base && vo.dtype == vi.dtype && vo.channels == 1 && !planes && tma_ok(ctx, vo, out_stride, batch);
        if (ts) ts = make_tmap(&tmO, vo.dtype, vo.ptr, g.P, g.L, batch, vo.ld, out_stride, TP, TL, TP);
        // the packed apply runs NT-thread CTAs, EMBED_CTAS_PER_SM per SM: a plan made for the narrow u8 kernels (4:2:2 luma) is resized for it
        std::vector<SubBatch> wide;
        if (packed && narrow) wide = partition(EMBED_CTAS_PER_SM * ctx->sms, batch, g.ntiles, ctx->opt_split_cost);
        const std::vector<SubBatch>& apply_sb = wide.empty() ? pl.embed : wide;
        for (const SubBatch& sb : apply_sb) {
            ea.b0 = sb.b0; ea.nblk_base = sb.base; ea.nblk_extra = sb.extra;
            const dim3 grid(sb.base + (sb.extra > 0 ? 1 : 0), sb.nb);
            if (ts) launch_apply_ts(vi.dtype, kmask, vi.transposed, narrow, grid, s.stream, tmI, tmW, tmO, ea);
            else if (packed) launch_apply_packed(kmask, vo.fmt.bytes, vo.fmt.luma, tma, grid, s.stream, tmI, tmW, ea);
            else launch_apply(vi.dtype, vo.dtype, kmask, vi.transposed, tma, grid, s.stream, tmI, tmW, ea);
        }
    }
    CU(cudaGetLastError());
    if (direct && batch == 1) return WM_OK;  // the apply kernel's last CTA publishes the scalars itself
    return push_result(ctx, s, 1, batch);
}

int do_detect(wm_ctx* ctx, int slot, const wm_image* img, int64_t img_stride, int batch, int mask, float* dbg_u = nullptr, float* dbg_eu = nullptr,
              bool direct = false)
{
    if (!ctx) return WM_ERR_ARG;
    if (slot < 0 || slot >= NSLOTS) return fail(ctx, WM_ERR_ARG, "bad slot");
    if (mask != WM_MASK_ME && mask != WM_MASK_NVF) return fail(ctx, WM_ERR_ARG, "bad mask type");
    if (batch < 1 || batch > 65535) return fail(ctx, WM_ERR_ARG, "batch must be 1..65535");
    View v;
    int rc;
    if ((rc = check_dims(ctx, img)) || (rc = make_view(ctx, img, &v, false, true))) return rc;
    if ((rc = resolve_stride(ctx, v, batch, &img_stride, "image"))) return rc;
    CU(cudaSetDevice(ctx->device));
    Slot& s = ctx->slots[slot];
    if (v.packed() && (rc = enqueue_packed_gray(ctx, s, &v, &img_stride, batch))) return rc;
    const Geo g = geo(v.L, v.P);
    bool tma = tma_ok(ctx, v, img_stride, batch);
    const bool narrow = ctx->opt_narrow_u8 && v.dtype == WM_U8 && tma && !dbg_u;
    const Plan pl = plan(ctx, g, batch, v.dtype, narrow);
    if ((rc = ensure_slot(ctx, s, batch, std::max(pl.gx_stats, pl.gx_detect), pl.nsweep, pl.nframe))) return rc;
    const float* W = w_for(ctx, v.transposed, s.stream, &rc);
    if (rc) return rc;
    const bool planes = mask == WM_MASK_NVF && ctx->p != 3;
    // synchronous single image: sweep + solve + detector as ONE cooperative kernel with the tiles kept in shared memory
    const int fgrid = std::min(g.ntiles, detect_ctas_per_sm(false) * ctx->sms);
    const bool fuse = direct && batch == 1 && ctx->opt_fused && tma && v.dtype == WM_F32 && !planes && ctx->opt_fp16 && ctx->opt_mma &&
                      !ctx->inject_coef && !ctx->opt_timing && !dbg_u && fused_fits(g, fgrid, DETECT_NST, true);
    if (!fuse && (rc = enqueue_sweep(ctx, s, v, img_stride, batch, g, pl))) return rc;
    DetectArgs da;
    da.img = v.ptr; da.ld = v.ld; da.bstride = img_stride;
    da.W = W;
    da.L = g.L; da.P = g.P; da.tiles_p = g.tiles_p; da.ntiles = g.ntiles;
    da.vec_ok = vec_ok(v.ptr, v.ld, img_stride, 0, v.dtype);
    da.w_vec_ok = (g.P % 4 == 0);
    da.pstride = pl.gx_detect;
    da.maskp = nullptr; da.mask_bstride = (long long)g.L * g.P;
    da.part = s.part + stats_part_offset(pl, batch);
    da.counter = s.counters + 2 * s.batch_cap;
    da.scal = s.scal; da.dbg = s.dbg;
    da.dbg_u = dbg_u; da.dbg_eu = dbg_eu;
    da.dl = deliver_args(s, direct && batch == 1);
    CUtensorMap tmZ, tmW;
    memset(&tmZ, 0, sizeof tmZ);
    memset(&tmW, 0, sizeof tmW);
    if (tma) tma = make_tmap(&tmZ, v.dtype, v.ptr, g.P, g.L, batch, v.ld, img_stride, SW, TL + 4) &&
                   make_tmap(&tmW, WM_F32, W, g.P, g.L, 1, g.P, 0, SW, TL + 2);
    if (fuse) {
        da.b0 = 0; da.nblk_base = fgrid; da.nblk_extra = 0;
        const SweepArgs sa = sweep_args(ctx, s, v, img_stride, batch, g, pl);
        if (tma && launch_detect1(mask, v.transposed, fgrid, s.stream, tmZ, tmW, sa, da, s.dl_words + 1, ctx->sms)) {
            ctx->launches++;
            CU(cudaGetLastError());
            return WM_OK;  // the kernel's last CTA publishes the result itself
        }
        ctx->fused_failures++;
        if ((rc = enqueue_sweep(ctx, s, v, img_stride, batch, g, pl))) return rc;
    }
    {
        KTimer t(ctx, s, mask == WM_MASK_ME ? WM_K_DETECT : WM_K_DETECT_NVF);
        if (planes) {
            if ((rc = enqueue_nvf_planes(ctx, s, v, img_stride, batch, g))) return rc;
            da.maskp = (const float*)s.maskp;
        }
        PdlScope pdl(ctx->opt_pdl && !ctx->opt_timing && !planes && !ctx->inject_coef);  // the Rx sweep of this op precedes
        for (const SubBatch& sb : pl.detect) {
            da.b0 = sb.b0; da.nblk_base = sb.base; da.nblk_extra = sb.extra;
            launch_detect(v.dtype, planes ? 2 : mask, v.transposed, tma, narrow, dim3(sb.base + (sb.extra > 0 ? 1 : 0), sb.nb), s.stream, tmZ, tmW, da);
        }
    }
    CU(cudaGetLastError());
    if (direct && batch == 1) return WM_OK;  // k_detect's last CTA publishes the scalars itself
    return push_result(ctx, s, 2, batch);
}

// wait for a slot and deliver the scalars of every queued op; returns the first non-zero status (or error)
int finish_slot(wm_ctx* ctx, Slot& s)
{
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(s.stream));
    drain_timers(ctx, s);
    int rc = WM_OK;
    for (const Slot::Pending& q : s.queue) {
        for (int b = 0; b < q.batch; b++) {
            const Scal& h = s.scal_host[q.off + b];
            if (q.scalar) {
                float* dst = q.scalar + (int64_t)b * q.sstride;
                if (q.kind == 1) { if (h.status != WM_SINGULAR) *dst = h.a; }  // untouched when unsolvable (Watermark.cpp:164-165)
                else *dst = h.status == 0 ? h.corr : 0.0f;                    // Watermark.cpp:246-247
            }
            if (q.status) q.status[b] = h.status;
            if (h.status != 0 && rc == WM_OK) rc = h.status;
        }
    }
    s.queue.clear();
    s.host_used = 0;
    return rc;
}

int load_w_file(wm_ctx* ctx, const char* path, int64_t rows, int64_t cols, std::vector<float>* w)
{
    // Watermark.cpp:62-75
    FILE* f = path ? fopen(path, "rb") : nullptr;
    if (!f) return fail(ctx, WM_ERR_W_FILE, std::string("Error opening '") + (path ? path : "(null)") + "' file for Random noise W array");
    fseek(f, 0, SEEK_END);
    const long long bytes = ftell(f);
    fseek(f, 0, SEEK_SET);
    if ((long long)(rows * cols * (int64_t)sizeof(float)) != bytes) {
        fclose(f);
        return fail(ctx, WM_ERR_W_SIZE, "Error: W file total elements != image dimensions! W file total elements: " +
                                            std::to_string(bytes / (long long)sizeof(float)) + ", Image width: " + std::to_string(cols) +
                                            ", Image height: " + std::to_string(rows));
    }
    w->resize((size_t)(rows * cols));
    const size_t got = fread(w->data(), sizeof(float), w->size(), f);
    fclose(f);
    if (got != w->size()) return fail(ctx, WM_ERR_W_FILE, "short read on W file");
    return WM_OK;
}

int upload_w(wm_ctx* ctx, int64_t rows, int64_t cols, const float* w_host)
{
    auto ws = std::make_shared<WShared>();
    ws->device = ctx->device;
    CU(cudaSetDevice(ctx->device));
    CU(cudaMalloc(&ws->row_major, sizeof(float) * rows * cols));
    CU(cudaMemcpy(ws->row_major, w_host, sizeof(float) * rows * cols, cudaMemcpyHostToDevice));
    ctx->w = ws;
    ctx->rows = rows;
    ctx->cols = cols;
    return WM_OK;
}

int init_slots(wm_ctx* ctx, void* user_stream)
{
    CU(cudaSetDevice(ctx->device));
    for (int i = 0; i < NSLOTS; i++) {
        Slot& s = ctx->slots[i];
        if (i == 0 && user_stream) { s.stream = (cudaStream_t)user_stream; s.own_stream = false; }
        else { CU(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking)); s.own_stream = true; }
    }
    return WM_OK;
}

void free_slot(Slot& s)
{
    if (s.part) cudaFree(s.part);
    if (s.counters) cudaFree(s.counters);
    if (s.scal) cudaFree(s.scal);
    if (s.dbg) cudaFree(s.dbg);
    if (s.scal_host) cudaFreeHost(s.scal_host);
    if (s.stage_in) cudaFree(s.stage_in);
    if (s.stage_base) cudaFree(s.stage_base);
    if (s.stage_out) cudaFree(s.stage_out);
    if (s.maskp) cudaFree(s.maskp);
    if (s.gray) cudaFree(s.gray);
    if (s.hres) cudaFreeHost(s.hres);
    if (s.dl_words) cudaFree(s.dl_words);
    for (auto& t : s.timed) { cudaEventDestroy(t.e0); cudaEventDestroy(t.e1); }
    if (s.own_stream && s.stream) cudaStreamDestroy(s.stream);
    s = Slot();
}

int create_common(wm_ctx** out, int64_t rows, int64_t cols, int p, float psnr, int device, void* stream, wm_ctx** made)
{
    wm_ctx* ctx = nullptr;
    if (!out) return fail(nullptr, WM_ERR_ARG, "null out");
    *out = nullptr;
    // Watermark.cpp:24-25
    if (p != 3 && p != 5 && p != 7 && p != 9) return fail(nullptr, WM_ERR_BAD_P, "Wrong p parameter: " + std::to_string(p) + "!");
    if (!(psnr > 0.0f)) return fail(nullptr, WM_ERR_ARG, "psnr must be > 0 (main.cpp:96)");
    if (rows < 3 || cols < 3 || rows > (1 << 30) / 4 || cols > (1 << 30) / 4) return fail(nullptr, WM_ERR_DIMS, "unsupported image dims");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail(nullptr, WM_ERR_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(nullptr, WM_ERR_NO_DEVICE, "invalid device " + std::to_string(device));
    ctx = new wm_ctx();
    ctx->device = device;
    ctx->p = p;
    ctx->psnr = psnr;
    ctx->strength = 255.0f / sqrtf(powf(10.0f, psnr / 10.0f));  // Watermark.cpp:22
    cudaSetDevice(device);
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->sms = prop.multiProcessorCount;
    const int rc = init_slots(ctx, stream);
    if (rc) { g_create_error = ctx->err; wm_destroy(ctx); return rc; }
    *made = ctx;
    (void)rows; (void)cols;
    return WM_OK;
}

// Synchronous single-image calls.  The second call with identical arguments captures the launch sequence (kernels +
// the scalar read-back) into a CUDA graph; from the third on the graph is replayed: one launch instead of 3-4.
std::string image_key(const wm_image* im)
{
    char b[160];
    if (!im) return "-";
    snprintf(b, sizeof b, "%p,%lld,%lld,%lld,%d,%d,%d,%lld;", im->data, (long long)im->rows, (long long)im->cols, (long long)im->ld,
             im->channels, im->layout, im->dtype, (long long)im->plane_stride);
    return b;
}
// direct delivery: the host clears the token, launches, and polls the token; the stream is only consulted every few thousand polls so that a
// failed launch cannot spin forever
void arm_direct(Slot& s)
{
    s.hres->token = 0;
    std::atomic_thread_fence(std::memory_order_release);
}
int wait_direct(wm_ctx* ctx, Slot& s, int kind, float* scalar_host)
{
    volatile unsigned* tok = &s.hres->token;
    for (unsigned spins = 0; *tok == 0; spins++) {
        if ((spins & 0x3fff) == 0x3fff) {
            const cudaError_t q = cudaStreamQuery(s.stream);
            if (q == cudaSuccess) { if (*tok == 0) return fail(ctx, WM_ERR_CUDA, "direct delivery: the op finished without publishing its result"); break; }
            if (q != cudaErrorNotReady) return fail(ctx, WM_ERR_CUDA, std::string("direct delivery: ") + cudaGetErrorString(q));
        }
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    const volatile HostResult* hr = s.hres;
    const float a = hr->a, corr = hr->corr;
    const int status = hr->status;
    if (scalar_host) {
        if (kind == 1) { if (status != WM_SINGULAR) *scalar_host = a; }  // untouched when unsolvable (Watermark.cpp:164-165)
        else *scalar_host = status == 0 ? corr : 0.0f;                  // Watermark.cpp:246-247
    }
    return status;
}

// Synchronous single-image calls.  The second call with identical arguments captures the launch sequence into a CUDA graph; from the
// third on the graph is replayed: one launch instead of 3-4, and the result comes back through direct delivery (no copy node, no
// stream synchronisation).  enqueue(direct) issues the op's kernels.
template <typename Enqueue>
int run_sync(wm_ctx* ctx, const std::string& key, int kind, float* scalar_host, Enqueue enqueue)
{
    Slot& s = ctx->slots[0];
    if (!s.queue.empty()) { const int r = finish_slot(ctx, s); if (r < 0) return r; }
    const bool eligible = ctx->opt_graphs && !ctx->opt_timing && !ctx->inject_coef;
    wm_ctx::GraphEntry* ge = nullptr;
    if (eligible) {
        for (auto& g : ctx->graphs) if (g.key == key) { ge = &g; break; }
        if (!ge) {
            if (ctx->graphs.size() >= 32) clear_graphs(ctx);
            ctx->graphs.push_back({key, 0, nullptr, 0});
            ge = &ctx->graphs.back();
        }
    }
    if (ge && ge->exec) {  // replay
        CU(cudaSetDevice(ctx->device));
        arm_direct(s);
        CU(cudaGraphLaunch(ge->exec, s.stream));
        ctx->launches += ge->launches;
        return wait_direct(ctx, s, kind, scalar_host);
    }
    if (ge && ge->seen >= 1) {  // second sighting: buffers exist, attributes are set -> capture
        CU(cudaSetDevice(ctx->device));
        int rc = ensure_direct(ctx, s);
        if (rc) return rc;
        const int64_t l0 = ctx->launches;
        cudaGraph_t graph = nullptr;
        if (cudaStreamBeginCapture(s.stream, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
            rc = enqueue(true);
            const cudaError_t ce = cudaStreamEndCapture(s.stream, &graph);
            s.queue.clear();
            s.host_used = 0;
            if (rc == WM_OK && ce == cudaSuccess && graph && cudaGraphInstantiate(&ge->exec, graph, 0) == cudaSuccess) {
                ge->launches = (int)(ctx->launches - l0);
                ctx->launches = l0;
            } else {
                ge->exec = nullptr;
                ge->seen = -1000000;  // do not try again for this key
                cudaGetLastError();
            }
            if (graph) cudaGraphDestroy(graph);
            if (rc < 0) return rc;
        }
        if (ge->exec) {
            arm_direct(s);
            CU(cudaGraphLaunch(ge->exec, s.stream));
            ctx->launches += ge->launches;
            return wait_direct(ctx, s, kind, scalar_host);
        }
    }
    if (ge) ge->seen++;
    const int rc = enqueue(false);
    if (rc) return rc;
    s.queue.back().scalar = scalar_host;
    return finish_slot(ctx, s);
}

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

const char* wm_version(void) { return WM_VERSION_STR; }

int wm_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

int wm_create(wm_ctx** out, int64_t rows, int64_t cols, const float* w_host, int p, float psnr, int device, void* stream)
{
    wm_ctx* ctx = nullptr;
    int rc = create_common(out, rows, cols, p, psnr, device, stream, &ctx);
    if (rc) return rc;
    if (!w_host) { wm_destroy(ctx); return fail(nullptr, WM_ERR_ARG, "null W"); }
    rc = upload_w(ctx, rows, cols, w_host);
    if (rc) { g_create_error = ctx->err; wm_destroy(ctx); return rc; }
    *out = ctx;
    return WM_OK;
}

int wm_create_from_file(wm_ctx** out, int64_t rows, int64_t cols, const char* w_path, int p, float psnr, int device, void* stream)
{
    wm_ctx* ctx = nullptr;
    int rc = create_common(out, rows, cols, p, psnr, device, stream, &ctx);
    if (rc) return rc;
    std::vector<float> w;
    rc = load_w_file(ctx, w_path, rows, cols, &w);
    if (!rc) rc = upload_w(ctx, rows, cols, w.data());
    if (rc) { g_create_error = ctx->err; wm_destroy(ctx); return rc; }
    *out = ctx;
    return WM_OK;
}

int wm_clone(const wm_ctx* src, wm_ctx** out)
{
    if (!src || !out) return WM_ERR_ARG;
    wm_ctx* ctx = new wm_ctx();
    ctx->device = src->device; ctx->sms = src->sms;
    ctx->rows = src->rows; ctx->cols = src->cols;
    ctx->p = src->p; ctx->psnr = src->psnr; ctx->strength = src->strength;
    ctx->w = src->w;
    ctx->opt_fp16 = src->opt_fp16; ctx->opt_mma = src->opt_mma; ctx->opt_split_cost = src->opt_split_cost; ctx->opt_timing = src->opt_timing; ctx->opt_tma = src->opt_tma;
    ctx->opt_serial = src->opt_serial; ctx->opt_graphs = src->opt_graphs; ctx->opt_f32_solve = src->opt_f32_solve; ctx->opt_host_run = src->opt_host_run; ctx->opt_tma_store = src->opt_tma_store; ctx->opt_pdl = src->opt_pdl; ctx->opt_fused = src->opt_fused; ctx->opt_padded_upload = src->opt_padded_upload; ctx->opt_narrow_u8 = src->opt_narrow_u8; ctx->opt_run_mb = src->opt_run_mb;
    const int rc = init_slots(ctx, nullptr);
    if (rc) { g_create_error = ctx->err; wm_destroy(ctx); return rc; }
    *out = ctx;
    return WM_OK;
}

int wm_reinitialize(wm_ctx* ctx, int64_t rows, int64_t cols, const float* w_host)
{
    if (!ctx || !w_host) return WM_ERR_ARG;
    if (rows < 3 || cols < 3) return fail(ctx, WM_ERR_DIMS, "unsupported image dims");
    wm_sync(ctx, -1);
    clear_graphs(ctx);
    return upload_w(ctx, rows, cols, w_host);
}

int wm_reinitialize_from_file(wm_ctx* ctx, int64_t rows, int64_t cols, const char* w_path)
{
    if (!ctx) return WM_ERR_ARG;
    std::vector<float> w;
    const int rc = load_w_file(ctx, w_path, rows, cols, &w);
    if (rc) return rc;
    return wm_reinitialize(ctx, rows, cols, w.data());
}

void wm_destroy(wm_ctx* ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    for (int i = 0; i < NSLOTS; i++) {
        if (ctx->slots[i].stream) cudaStreamSynchronize(ctx->slots[i].stream);
        free_slot(ctx->slots[i]);
    }
    for (auto e : ctx->event_pool) cudaEventDestroy(e);
    clear_graphs(ctx);
    delete ctx;
}

int wm_set_option(wm_ctx* ctx, int option, int value)
{
    if (!ctx) return WM_ERR_ARG;
    switch (option) {
    case WM_OPT_FP16_PRODUCTS: ctx->opt_fp16 = value != 0; return WM_OK;
    case WM_OPT_KERNEL_TIMING: ctx->opt_timing = value != 0; return WM_OK;
    case WM_OPT_USE_TMA: ctx->opt_tma = value != 0; return WM_OK;
    case WM_OPT_SERIAL_SLOTS: ctx->opt_serial = value != 0; return WM_OK;
    case WM_OPT_CUDA_GRAPHS: ctx->opt_graphs = value != 0; return WM_OK;
    case WM_OPT_MMA_ACCUM: ctx->opt_mma = value != 0; return WM_OK;
    case WM_OPT_HOST_RUN_FRAMES: ctx->opt_host_run = std::max(1, std::min(value, 64)); return WM_OK;
    case WM_OPT_TMA_STORE: ctx->opt_tma_store = value != 0; clear_graphs(ctx); return WM_OK;
    case WM_OPT_PDL: ctx->opt_pdl = value != 0; clear_graphs(ctx); return WM_OK;
    case WM_OPT_FUSED_SINGLE: ctx->opt_fused = value != 0; clear_graphs(ctx); return WM_OK;
    case WM_OPT_PADDED_UPLOAD: ctx->opt_padded_upload = value != 0; return WM_OK;
    case WM_OPT_NARROW_U8: ctx->opt_narrow_u8 = value != 0; clear_graphs(ctx); return WM_OK;
    case WM_OPT_RUN_MB: ctx->opt_run_mb = std::max(1, std::min(value, 4096)); return WM_OK;
    case WM_OPT_F32_SOLVE: ctx->opt_f32_solve = value != 0; clear_graphs(ctx); return WM_OK;
    case WM_OPT_SPLIT_COST: ctx->opt_split_cost = value < 0 ? 1 << 28 : value; return WM_OK;
    default: return fail(ctx, WM_ERR_ARG, "unknown option");
    }
}

const char* wm_last_error(const wm_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }
float wm_strength_factor(const wm_ctx* ctx) { return ctx ? ctx->strength : 0.0f; }
int wm_num_slots(const wm_ctx*) { return NSLOTS; }
void* wm_get_stream(const wm_ctx* ctx, int slot) { return (ctx && slot >= 0 && slot < NSLOTS) ? (void*)ctx->slots[slot].stream : nullptr; }

int wm_sync(wm_ctx* ctx, int slot)
{
    if (!ctx) return WM_ERR_ARG;
    if (slot >= NSLOTS) return fail(ctx, WM_ERR_ARG, "bad slot");
    int rc = WM_OK;
    for (int i = (slot < 0 ? 0 : slot); i < (slot < 0 ? NSLOTS : slot + 1); i++) {
        const int r = finish_slot(ctx, ctx->slots[i]);
        if (r < 0) return r;
        if (r && !rc) rc = r;
    }
    return rc;
}

int wm_embed_batch(wm_ctx* ctx, int slot, const wm_image* in, const wm_image* base, wm_image* out, int64_t in_stride,
                   int64_t base_stride, int64_t out_stride, int batch, int mask, float* a_host, int* status_host)
{
    if (!ctx) return WM_ERR_ARG;
    if (slot < 0 || slot >= NSLOTS) return fail(ctx, WM_ERR_ARG, "bad slot");
    const int rc = do_embed(ctx, slot, in, base, out, in_stride, base_stride, out_stride, batch, mask);
    if (rc) return rc;
    ctx->slots[slot].queue.back().scalar = a_host;
    ctx->slots[slot].queue.back().status = status_host;
    return WM_OK;
}

int wm_detect_batch(wm_ctx* ctx, int slot, const wm_image* img, int64_t img_stride, int batch, int mask, float* corr_host, int* status_host)
{
    if (!ctx) return WM_ERR_ARG;
    if (slot < 0 || slot >= NSLOTS) return fail(ctx, WM_ERR_ARG, "bad slot");
    const int rc = do_detect(ctx, slot, img, img_stride, batch, mask);
    if (rc) return rc;
    ctx->slots[slot].queue.back().scalar = corr_host;
    ctx->slots[slot].queue.back().status = status_host;
    return WM_OK;
}

int wm_embed(wm_ctx* ctx, const wm_image* in, const wm_image* base, wm_image* out, int mask, float* a_host)
{
    if (!ctx) return WM_ERR_ARG;
    const std::string key = "E" + std::to_string(mask) + image_key(in) + image_key(base) + image_key(out) + std::to_string(ctx->opt_fp16 + 2 * ctx->opt_mma + 4 * ctx->opt_f32_solve) +
                            std::to_string(ctx->opt_tma);
    return run_sync(ctx, key, 1, a_host, [&](bool direct) { return do_embed(ctx, 0, in, base, out, 0, 0, 0, 1, mask, direct); });
}

int wm_detect(wm_ctx* ctx, const wm_image* img, int mask, float* corr_host)
{
    if (!ctx) return WM_ERR_ARG;
    const std::string key = "D" + std::to_string(mask) + image_key(img) + std::to_string(ctx->opt_fp16 + 2 * ctx->opt_mma + 4 * ctx->opt_f32_solve) + std::to_string(ctx->opt_tma);
    return run_sync(ctx, key, 2, corr_host, [&](bool direct) { return do_detect(ctx, 0, img, 0, 1, mask, nullptr, nullptr, direct); });
}

// ---- host-buffer form.  Host images may be strided views (ld > contiguous dimension, padded planes): every plane is staged
// DENSELY on the device with one 2-D copy (width = the contiguous dimension, source pitch = ld), exactly the repack the reference does
// row by row (main.cpp:348-353), and results are copied back the same way, so neither copy touches a byte outside the image's
// pixels — the caller's row and plane padding stays as it was.
static size_t dense_bytes(const View& v) { return (size_t)(v.L * v.row_bytes() * v.planes()); }
// dense device planes <-> strided host planes
static cudaError_t copy_planes(void* dev, void* host, const View& v, bool to_device, cudaStream_t st)
{
    const size_t rb = (size_t)v.row_bytes(), plane = (size_t)v.L * rb;
    for (int c = 0; c < v.planes(); c++) {
        char* d = (char*)dev + (size_t)c * plane;
        char* h = (char*)host + (size_t)c * (size_t)v.plane_bytes();
        if ((size_t)v.pitch() == rb) {  // dense rows: one linear copy (a 2-D copy is programmed row by row)
            const cudaError_t e1 = to_device ? cudaMemcpyAsync(d, h, plane, cudaMemcpyHostToDevice, st) : cudaMemcpyAsync(h, d, plane, cudaMemcpyDeviceToHost, st);
            if (e1 != cudaSuccess) return e1;
            continue;
        }
        const cudaError_t e = to_device ? cudaMemcpy2DAsync(d, rb, h, (size_t)v.pitch(), rb, (size_t)v.L, cudaMemcpyHostToDevice, st)
                                        : cudaMemcpy2DAsync(h, (size_t)v.pitch(), d, rb, rb, (size_t)v.L, cudaMemcpyDeviceToHost, st);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}
static wm_image dense_desc(const wm_image* im, void* dev)
{
    wm_image d = *im;
    d.data = dev; d.ld = 0; d.plane_stride = 0;
    return d;
}

// staging of a batch: image b of a strided host batch <-> image b of a dense device batch
static cudaError_t copy_batch(void* dev, const View& v, int64_t host_stride, int batch, bool to_device, cudaStream_t st)
{
    const size_t n = dense_bytes(v);
    const long long hs = (host_stride > 0 ? host_stride : v.pstride * v.planes()) * v.elem();  // bytes between host images
    if (v.pitch() == v.row_bytes() && v.plane_bytes() == v.L * v.row_bytes() && (size_t)hs == n) {  // the whole batch is dense on the host too: one copy
        return to_device ? cudaMemcpyAsync(dev, v.ptr, n * batch, cudaMemcpyHostToDevice, st) : cudaMemcpyAsync(v.ptr, dev, n * batch, cudaMemcpyDeviceToHost, st);
    }
    for (int b = 0; b < batch; b++) {
        const cudaError_t e = copy_planes((char*)dev + (size_t)b * n, (char*)v.ptr + (size_t)b * (size_t)hs, v, to_device, st);
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}
// a slot's staging buffer may only be replaced when nothing queued on the slot still uses it
static int grow_stage(wm_ctx* ctx, Slot& s, void** p, size_t* cap, size_t bytes)
{
    if (bytes <= *cap) return WM_OK;
    if (!s.queue.empty()) { const int r = finish_slot(ctx, s); if (r < 0) return r; }
    CU(cudaStreamSynchronize(s.stream));
    return ensure_stage(ctx, p, cap, bytes);
}

int wm_embed_host_batch(wm_ctx* ctx, int slot, const wm_image* in, const wm_image* base, wm_image* out, int64_t in_stride, int64_t base_stride,
                        int64_t out_stride, int batch, int mask, float* a_host, int* status_host)
{
    if (!ctx || !in || !out || !in->data || !out->data) return WM_ERR_ARG;
    if (slot < 0 || slot >= NSLOTS) return fail(ctx, WM_ERR_ARG, "bad slot");
    if (batch < 1 || batch > 65535) return fail(ctx, WM_ERR_ARG, "batch must be 1..65535");
    CU(cudaSetDevice(ctx->device));
    Slot& s = ctx->slots[slot];
    const wm_image* b = base ? base : in;
    View vi, vb, vo;
    int rc;
    if ((rc = make_view(ctx, in, &vi, false, true)) || (rc = make_view(ctx, b, &vb, true, true)) || (rc = make_view(ctx, out, &vo, true, true))) return rc;
    if ((rc = grow_stage(ctx, s, &s.stage_in, &s.stage_in_cap, dense_bytes(vi) * batch))) return rc;
    if ((rc = grow_stage(ctx, s, &s.stage_out, &s.stage_out_cap, dense_bytes(vo) * batch))) return rc;
    const bool base_is_in = vb.ptr == vi.ptr && vb.planes() == 1 && vb.ld == vi.ld && vb.dtype == vi.dtype && vb.layout == vi.layout &&
                            (batch == 1 || base_stride == in_stride);
    if (!base_is_in && (rc = grow_stage(ctx, s, &s.stage_base, &s.stage_base_cap, dense_bytes(vb) * batch))) return rc;
    CU(copy_batch(s.stage_in, vi, in_stride, batch, true, s.stream));
    wm_image din = dense_desc(in, s.stage_in), dbase, dout = dense_desc(out, s.stage_out);
    if (base_is_in) dbase = din;
    else {
        CU(copy_batch(s.stage_base, vb, base_stride, batch, true, s.stream));
        dbase = dense_desc(b, s.stage_base);
    }
    rc = do_embed(ctx, slot, &din, &dbase, &dout, 0, 0, 0, batch, mask);
    if (rc) return rc;
    s.queue.back().scalar = a_host;
    s.queue.back().status = status_host;
    CU(copy_batch(s.stage_out, vo, out_stride, batch, false, s.stream));
    return WM_OK;
}

// embed + verify for host images: wm_embed_host_batch, then detectWatermark on each watermarked image while it still lies in the slot's
// device staging buffer (gray outputs only) — the pair of operations of the reference's testForImage flow (main.cpp:178-217) with one upload
// and one download per image instead of a second upload of the watermarked image
int wm_embed_verify_host_batch(wm_ctx* ctx, int slot, const wm_image* in, const wm_image* base, wm_image* out, int64_t in_stride,
                               int64_t base_stride, int64_t out_stride, int batch, int mask, float* a_host, float* corr_host, int* status_host)
{
    if (!ctx || !out) return WM_ERR_ARG;
    View vo;
    int rc = make_view(ctx, out, &vo, true, true);
    if (rc) return rc;
    // a packed output is verified through its gray, like the reference's detection on the gray of the saved image
    if (!vo.packed() && (vo.channels > 1 || vo.dtype != (in ? in->dtype : vo.dtype)))
        return fail(ctx, WM_ERR_ARG, "embed + verify needs a gray output of the input's dtype (detectWatermark takes the gray image)");
    rc = wm_embed_host_batch(ctx, slot, in, base, out, in_stride, base_stride, out_stride, batch, mask, a_host, status_host);
    if (rc) return rc;
    Slot& s = ctx->slots[slot];
    wm_image d = dense_desc(out, s.stage_out);
    rc = do_detect(ctx, slot, &d, 0, batch, mask);
    if (rc) return rc;
    s.queue.back().scalar = corr_host;
    return WM_OK;
}

int wm_detect_host_batch(wm_ctx* ctx, int slot, const wm_image* img, int64_t img_stride, int batch, int mask, float* corr_host, int* status_host)
{
    if (!ctx || !img || !img->data) return WM_ERR_ARG;
    if (slot < 0 || slot >= NSLOTS) return fail(ctx, WM_ERR_ARG, "bad slot");
    if (batch < 1 || batch > 65535) return fail(ctx, WM_ERR_ARG, "batch must be 1..65535");
    CU(cudaSetDevice(ctx->device));
    Slot& s = ctx->slots[slot];
    View v;
    int rc;
    if ((rc = make_view(ctx, img, &v, false, true))) return rc;
    if ((rc = grow_stage(ctx, s, &s.stage_in, &s.stage_in_cap, dense_bytes(v) * batch))) return rc;
    CU(copy_batch(s.stage_in, v, img_stride, batch, true, s.stream));
    wm_image d = dense_desc(img, s.stage_in);
    rc = do_detect(ctx, slot, &d, 0, batch, mask);
    if (rc) return rc;
    s.queue.back().scalar = corr_host;
    s.queue.back().status = status_host;
    return WM_OK;
}

int wm_embed_host(wm_ctx* ctx, const wm_image* in, const wm_image* base, wm_image* out, int mask, float* a_host)
{
    if (!ctx) return WM_ERR_ARG;
    Slot& s = ctx->slots[0];
    if (!s.queue.empty()) { const int r = finish_slot(ctx, s); if (r < 0) return r; }
    const int rc = wm_embed_host_batch(ctx, 0, in, base, out, 0, 0, 0, 1, mask, a_host, nullptr);
    if (rc) return rc;
    return finish_slot(ctx, s);
}

int wm_detect_host(wm_ctx* ctx, const wm_image* img, int mask, float* corr_host)
{
    if (!ctx) return WM_ERR_ARG;
    Slot& s = ctx->slots[0];
    if (!s.queue.empty()) { const int r = finish_slot(ctx, s); if (r < 0) return r; }
    const int rc = wm_detect_host_batch(ctx, 0, img, 0, 1, mask, corr_host, nullptr);
    if (rc) return rc;
    return finish_slot(ctx, s);
}

int wm_rgb2gray(wm_ctx* ctx, const wm_image* rgb, wm_image* gray, float wr, float wg, float wb)
{
    if (!ctx) return WM_ERR_ARG;
    View vi, vo;
    int rc;
    if ((rc = check_dims(ctx, rgb)) || (rc = make_view(ctx, rgb, &vi, true))) return rc;
    if ((rc = check_dims(ctx, gray)) || (rc = make_view(ctx, gray, &vo, false))) return rc;
    if (vi.channels != 3 || vi.dtype != WM_F32 || vo.dtype != WM_F32 || vi.transposed != vo.transposed)
        return fail(ctx, WM_ERR_ARG, "rgb2gray needs a 3-channel f32 input and a 1-channel f32 output of the same layout");
    CU(cudaSetDevice(ctx->device));
    Slot& s = ctx->slots[0];
    const float* p0 = (const float*)vi.ptr;
    launch_rgb2gray(p0, p0 + vi.pstride, p0 + 2 * vi.pstride, (float*)vo.ptr, vi.ld, vo.ld, vi.L, vi.P, wr, wg, wb, 4 * ctx->sms, s.stream);
    ctx->launches++;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(s.stream));
    return WM_OK;
}

int wm_debug_get(wm_ctx* ctx, int what, void* dst)
{
    if (!ctx || !dst) return WM_ERR_ARG;
    CU(cudaSetDevice(ctx->device));
    Slot& s = ctx->slots[0];
    if (!s.scal) return fail(ctx, WM_ERR_ARG, "no call made yet");
    CU(cudaStreamSynchronize(s.stream));
    Scal h;
    ScalDbg d;
    CU(cudaMemcpy(&h, s.scal, sizeof h, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(&d, s.dbg, sizeof d, cudaMemcpyDeviceToHost));
    switch (what) {
    case WM_DBG_RX: memcpy(dst, d.Rx, sizeof d.Rx); return WM_OK;
    case WM_DBG_RXVEC: memcpy(dst, d.rx, sizeof d.rx); return WM_OK;
    case WM_DBG_COEFFS: memcpy(dst, h.coef, sizeof h.coef); return WM_OK;
    case WM_DBG_SCALARS: {
        double* o = (double*)dst;
        o[0] = h.status; o[1] = h.a; o[2] = h.emax; o[3] = d.sum2; o[4] = d.dot; o[5] = d.nz; o[6] = d.nu; o[7] = h.corr;
        return WM_OK;
    }
    case WM_DBG_PHASES: {
        double* o = (double*)dst;
        for (int i = 0; i < 8; i++) o[i] = (i >= 1 && d.ts[i] != 0) ? (double)(long long)(d.ts[i] - d.ts[0]) : 0.0;
        return WM_OK;
    }
    default: return fail(ctx, WM_ERR_ARG, "unknown debug item");
    }
}

int wm_debug_set_coeffs(wm_ctx* ctx, const float* c)
{
    if (!ctx) return WM_ERR_ARG;
    ctx->inject_coef = c != nullptr;
    if (c) memcpy(ctx->injected, c, sizeof ctx->injected);
    return WM_OK;
}

int wm_debug_detect_planes(wm_ctx* ctx, const wm_image* img, int mask, float* u_dev, float* eu_dev, float* corr_host)
{
    if (!ctx || !img || !u_dev || !eu_dev) return WM_ERR_ARG;
    View v;
    int rc;
    if ((rc = make_view(ctx, img, &v, false))) return rc;  // gray images only: packed images are refused here
    if (v.dtype != WM_F32 || (mask == WM_MASK_NVF && ctx->p != 3)) return fail(ctx, WM_ERR_ARG, "detector planes: f32 images, 3x3 masks");
    Slot& s = ctx->slots[0];
    if (!s.queue.empty()) { const int r = finish_slot(ctx, s); if (r < 0) return r; }
    rc = do_detect(ctx, 0, img, 0, 1, mask, u_dev, eu_dev);
    if (rc) return rc;
    s.queue.back().scalar = corr_host;
    return finish_slot(ctx, s);
}

int wm_debug_plane(wm_ctx* ctx, const wm_image* img, int what, float* dst_dev)
{
    if (!ctx || !dst_dev) return WM_ERR_ARG;
    if (what != WM_DBG_ERRSEQ && what != WM_DBG_MASK_NVF && what != WM_DBG_MASK_ME) return fail(ctx, WM_ERR_ARG, "plane must be ERRSEQ, MASK_NVF or MASK_ME");
    View v;
    int rc;
    if ((rc = check_dims(ctx, img)) || (rc = make_view(ctx, img, &v, false))) return rc;
    CU(cudaSetDevice(ctx->device));
    Slot& s = ctx->slots[0];
    if (!s.queue.empty()) { const int r = finish_slot(ctx, s); if (r < 0) return r; }
    const Geo g = geo(v.L, v.P);
    const Plan pl = plan(ctx, g, 1, v.dtype);
    if ((rc = ensure_slot(ctx, s, 1, std::max(pl.gx_stats, pl.gx_detect), pl.nsweep, pl.nframe))) return rc;
    if (what == WM_DBG_ERRSEQ || what == WM_DBG_MASK_ME) {
        if ((rc = enqueue_sweep(ctx, s, v, 0, 1, g, pl))) return rc;
    }
    if (what == WM_DBG_MASK_NVF && ctx->p != 3) {  // the p x p window goes through k_nvfp, straight into the caller's plane
        if ((rc = enqueue_nvf_planes(ctx, s, v, 0, 1, g, dst_dev))) return rc;
        ctx->launches++;
        CU(cudaStreamSynchronize(s.stream));
        return WM_OK;
    }
    PlaneArgs pa;
    pa.img = v.ptr; pa.ld = v.ld;
    pa.L = g.L; pa.P = g.P; pa.tiles_p = g.tiles_p; pa.ntiles = g.ntiles;
    pa.vec_ok = vec_ok(v.ptr, v.ld, 0, 0, v.dtype);
    pa.scal = s.scal;
    pa.dst = dst_dev;
    const dim3 grid(std::min(g.ntiles, 3 * ctx->sms));
    launch_plane(v.dtype, what != WM_DBG_MASK_NVF, v.transposed, grid, s.stream, pa);
    ctx->launches++;
    if (what == WM_DBG_MASK_ME) {  // mask = |e| / max|e| (Watermark.cpp:213-214); the counters' first word doubles as the max scratch and is zero again afterwards
        launch_mask_from_errseq(dst_dev, (long long)g.L * g.P, s.counters, s.stream);
        CU(cudaMemsetAsync(s.counters, 0, sizeof(unsigned), s.stream));
        ctx->launches += 2;
    }
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(s.stream));
    return WM_OK;
}

int64_t wm_get_kernel_times(wm_ctx* ctx, int kernel, double* total_ms, int reset)
{
    if (!ctx || kernel < 0 || kernel >= WM_K_COUNT) return -1;
    const int64_t n = ctx->kcount[kernel];
    if (total_ms) *total_ms = ctx->ktime_ms[kernel];
    if (reset) { ctx->kcount[kernel] = 0; ctx->ktime_ms[kernel] = 0.0; }
    return n;
}

int64_t wm_launch_count(const wm_ctx* ctx) { return ctx ? ctx->launches : 0; }

// ---- video driver (videoprocessingcontext.hpp:13-29, main.cpp:319-410) ----
int64_t wm_process_frames(const wm_video_ctx* v, int mode, const uint8_t* frames, uint8_t* out, int64_t first_index,
                          int64_t n_frames, float* scalars)
{
    if (!v || !v->watermark || !frames) return WM_ERR_ARG;
    wm_ctx* ctx = v->watermark;
    if (mode != WM_VIDEO_EMBED && mode != WM_VIDEO_DETECT && mode != WM_VIDEO_EMBED_VERIFY) return fail(ctx, WM_ERR_ARG, "bad mode");
    const bool embed_mode = mode != WM_VIDEO_DETECT;
    if (v->height != ctx->rows || v->width != ctx->cols) return fail(ctx, WM_ERR_DIMS, "frame dims != watermark dims");
    if (v->watermark_interval < 1) return fail(ctx, WM_ERR_ARG, "watermark_interval must be >= 1");
    if (embed_mode && !out) return fail(ctx, WM_ERR_ARG, "embed needs an output buffer");
    // a frame as an image: a Y plane (layout 0 or WM_ROW_MAJOR) or a packed frame, rows of linesize bytes (0 = dense)
    wm_image frame;
    memset(&frame, 0, sizeof frame);
    frame.data = (void*)frames; frame.rows = v->height; frame.cols = v->width; frame.dtype = WM_U8;
    frame.layout = v->layout ? v->layout : WM_ROW_MAJOR; frame.ld = v->linesize;
    View fv;
    int rc;
    if ((rc = make_view(ctx, &frame, &fv, false, true, true))) return fail(ctx, rc, "frames (ld = linesize): " + ctx->err);
    frame.channels = fv.channels;
    const int64_t H = v->height;
    const int64_t rowb = fv.row_bytes();  // bytes of a frame row without padding
    const int64_t linesize = fv.pitch();
    const int64_t fstride = v->frame_stride > 0 ? v->frame_stride : H * linesize;
    const int64_t ostride = H * rowb;
    CU(cudaSetDevice(ctx->device));
    for (int i = 0; i < NSLOTS; i++)
        if (!ctx->slots[i].queue.empty()) { const int r = finish_slot(ctx, ctx->slots[i]); if (r < 0) return r; }
    const float nanv = nanf("");
    const int64_t K = v->watermark_interval;
    const int64_t i0 = (K - first_index % K) % K;  // first gated frame: (first_index + i) % K == 0 (main.cpp:346,395: global index)
    const int64_t ngated = i0 < n_frames ? (n_frames - i0 + K - 1) / K : 0;
    const cudaMemcpyKind through = v->frames_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToHost;
    // every scalar starts as NaN: frames between the gated ones have none, and an unsolvable frame leaves `a` untouched
    // (Watermark.cpp:164-165) — the caller sees NaN there, never an uninitialised float
    if (scalars) for (int64_t i = 0; i < (mode == WM_VIDEO_EMBED_VERIFY ? 2 * n_frames : n_frames); i++) scalars[i] = nanv;
    // frames between the gated ones: copied through without the row padding (main.cpp:362-366)
    for (int64_t i = 0; i < n_frames; i++) {
        if ((first_index + i) % K == 0) continue;
        if (embed_mode)
            CU(cudaMemcpy2DAsync(out + i * ostride, rowb, frames + i * fstride, linesize, rowb, H, through, ctx->slots[i % NSLOTS].stream));
    }
    // gated frames: equally spaced in memory, so a run of them is ONE batched launch sequence (image index in
    // blockIdx.y); runs go round-robin over the slots so copies, kernels and the per-frame solves of different runs overlap
    const int64_t fbytes = H * rowb;
    // frames per run: big enough to amortise a launch's ramp and second-stage tail, small enough that several runs are in
    // flight on different slots (round 1, 4K u8: 4 / 7 / 10 / 19 / 37 frames per run gave 17.1k / 18.2k / 19.0k / 18.5k / 18.2k frames/s; with the
    // round-2 kernels 7 / 9 / 11 / 13 / 16 / 24 / 32 frames per run give 25.2k / 25.2k / 25.5k / 25.6k / 25.8k / 25.8k / 25.8k: WM_OPT_RUN_MB = 136).
    // Packed frames count their packed bytes only, not the 4 B/px of gray planes a run also fills: EMBED_VERIFY on a B200 at 1080p / 4K,
    // BGR / BGRA, gave 3-6 % more frames/s than counting packed + gray bytes (22 vs 9 frames per run at 1080p BGR, 5 vs 2 at 4K BGR)
    int64_t B = v->frames_on_device ? std::max<int64_t>(1, std::min<int64_t>(32, ((int64_t)ctx->opt_run_mb << 20) / fbytes)) : ctx->opt_host_run;
    // even runs (37 frames at 7 per run: 7,6,6,6,6,6 rather than 7,7,7,7,7,2)
    const int64_t nruns = ngated > 0 ? (ngated + B - 1) / B : 0;
    // packed frames: each slot that takes a run computes its gray (or luma) into its own planes.  They are sized once for the longest run
    // these options allow, so calls whose even runs differ by a frame (other frame counts, first indices) do not regrow them with a stream sync
    if (fv.packed())
        for (int64_t r = 0; r < std::min<int64_t>(nruns, ctx->opt_serial ? 1 : NSLOTS); r++)
            if ((rc = reserve_gray(ctx, ctx->slots[r], gray_plane_bytes(fv.fmt, fv.L, fv.P) * (size_t)B))) return rc;
    const int64_t run_base = nruns ? ngated / nruns : 0, run_extra = nruns ? ngated % nruns : 0;
    B = run_base + (run_extra ? 1 : 0);
    for (int64_t g = 0, run = 0, nbr = 0; run < nruns; g += nbr, run++) {
        nbr = run_base + (run < run_extra ? 1 : 0);
        const int nb = (int)nbr;
        const int si = ctx->opt_serial ? 0 : (int)(run % NSLOTS);
        Slot& s = ctx->slots[si];
        const int64_t i = i0 + g * K;
        wm_image fin = frame;
        int64_t in_stride;
        if (v->frames_on_device) {
            fin.data = (void*)(frames + i * fstride); fin.ld = linesize;  // strided reads: no repack pass needed
            in_stride = K * fstride;
        } else {
            // H2D.  The reference repacks a decoded frame row by row to drop ffmpeg's row padding (main.cpp:348-353).  Here a frame whose
            // padding is small and whose linesize keeps the rows 16-byte aligned goes up WITH its padding as one linear copy (a 2-D copy is
            // programmed row by row) and the kernels read it in place with ld = linesize, as they do for frames that are already on the
            // device; other paddings are dropped by a 2-D copy.
            const bool keep_pad = ctx->opt_padded_upload && linesize != rowb && linesize % 16 == 0 && (linesize - rowb) * 8 <= rowb;
            const int64_t sbytes = keep_pad ? H * linesize : fbytes;  // bytes of one staged frame
            if (sbytes * nb > (int64_t)s.stage_in_cap && !s.queue.empty()) { const int r = finish_slot(ctx, s); if (r < 0) return r; }
            if ((rc = ensure_stage(ctx, &s.stage_in, &s.stage_in_cap, (size_t)(sbytes * B)))) return rc;
            if ((linesize == rowb || keep_pad) && K * fstride == sbytes)  // the frames of the run are contiguous on the host too: one copy
                CU(cudaMemcpyAsync(s.stage_in, frames + i * fstride, (size_t)(sbytes * nb), cudaMemcpyHostToDevice, s.stream));
            else for (int j = 0; j < nb; j++) {
                const uint8_t* src = frames + (i + j * K) * fstride;
                if (linesize == rowb || keep_pad) CU(cudaMemcpyAsync((uint8_t*)s.stage_in + j * sbytes, src, (size_t)sbytes, cudaMemcpyHostToDevice, s.stream));
                else CU(cudaMemcpy2DAsync((uint8_t*)s.stage_in + j * sbytes, rowb, src, linesize, rowb, H, cudaMemcpyHostToDevice, s.stream));
            }
            fin.data = s.stage_in; fin.ld = keep_pad ? linesize : rowb;
            in_stride = sbytes;
        }
        if (embed_mode) {
            wm_image fout = fin;
            fout.ld = rowb;
            int64_t out_stride;
            if (v->frames_on_device) { fout.data = out + i * ostride; out_stride = K * ostride; }
            else {
                if (fbytes * nb > (int64_t)s.stage_out_cap && !s.queue.empty()) { const int r = finish_slot(ctx, s); if (r < 0) return r; }
                if ((rc = ensure_stage(ctx, &s.stage_out, &s.stage_out_cap, (size_t)(fbytes * B)))) return rc;
                fout.data = s.stage_out; out_stride = fbytes;
            }
            rc = do_embed(ctx, si, &fin, &fin, &fout, in_stride, in_stride, out_stride, nb, WM_MASK_ME);  // main.cpp:356,380
            if (rc) return rc;
            s.queue.back().scalar = scalars ? scalars + i : nullptr;
            s.queue.back().sstride = K;
            if (!v->frames_on_device) {
                if (K == 1) CU(cudaMemcpyAsync(out + i * ostride, s.stage_out, (size_t)(fbytes * nb), cudaMemcpyDeviceToHost, s.stream));
                else for (int j = 0; j < nb; j++)
                    CU(cudaMemcpyAsync(out + (i + j * K) * ostride, (uint8_t*)s.stage_out + j * fbytes, (size_t)fbytes,
                                       cudaMemcpyDeviceToHost, s.stream));
            }
            if (mode == WM_VIDEO_EMBED_VERIFY) {  // detect on the frame just written, where it lies on the device
                rc = do_detect(ctx, si, &fout, out_stride, nb, WM_MASK_ME);
                if (rc) return rc;
                s.queue.back().scalar = scalars ? scalars + n_frames + i : nullptr;
                s.queue.back().sstride = K;
            }
            continue;
        } else {
            rc = do_detect(ctx, si, &fin, in_stride, nb, WM_MASK_ME);  // main.cpp:406
            if (rc) return rc;
        }
        s.queue.back().scalar = scalars ? scalars + i : nullptr;
        s.queue.back().sstride = K;
    }
    for (int i = 0; i < NSLOTS; i++) { const int r = finish_slot(ctx, ctx->slots[i]); if (r < 0) return r; }
    return n_frames;
}


// ---- multi-GPU video driver (SURVEY.md 8e): frames are independent, so the global index range is cut into contiguous chunks, one
// per context / device, each driven by its own host thread; the interval gate sees the GLOBAL index (main.cpp:346,395), every scalar
// lands in one array indexed by (global frame - first_index).  No collective: nothing but per-frame scalars leaves a GPU.
void wm_shard_frames(int64_t n_frames, int rank, int world, int64_t* first, int64_t* count)
{
    if (world < 1) world = 1;
    const int64_t base = n_frames / world, rem = n_frames % world;
    if (first) *first = rank * base + std::min<int64_t>(rank, rem);
    if (count) *count = base + (rank < rem ? 1 : 0);
}

int64_t wm_process_frames_multi(const wm_video_ctx* const* v, int ngpus, int mode, const uint8_t* const* chunk_frames, uint8_t* const* chunk_out,
                                int64_t first_index, int64_t n_frames, float* scalars)
{
    if (!v || ngpus < 1 || !chunk_frames) return WM_ERR_ARG;
    for (int g = 0; g < ngpus; g++)
        if (!v[g] || !v[g]->watermark) return WM_ERR_ARG;
    std::vector<int64_t> done((size_t)ngpus, 0);
    std::vector<std::thread> th;
    th.reserve((size_t)ngpus);
    for (int g = 0; g < ngpus; g++) {
        th.emplace_back([&, g]() {
            int64_t first = 0, count = 0;
            wm_shard_frames(n_frames, g, ngpus, &first, &count);
            if (count == 0) { done[(size_t)g] = 0; return; }
            done[(size_t)g] = wm_process_frames(v[g], mode, chunk_frames[g], chunk_out ? chunk_out[g] : nullptr, first_index + first, count,
                                                scalars ? scalars + first : nullptr);
        });
    }
    for (auto& t : th) t.join();
    int64_t total = 0;
    for (int g = 0; g < ngpus; g++) {
        if (done[(size_t)g] < 0) return done[(size_t)g];  // the failing context keeps the message (wm_last_error)
        total += done[(size_t)g];
    }
    return total;
}

// ---- helpers ----
void* wm_dev_alloc(wm_ctx* ctx, int64_t bytes)
{
    if (ctx) cudaSetDevice(ctx->device);
    void* p = nullptr;
    if (cudaMalloc(&p, (size_t)bytes) != cudaSuccess) return nullptr;
    return p;
}
void wm_dev_free(wm_ctx* ctx, void* p)
{
    if (ctx) cudaSetDevice(ctx->device);
    if (p) cudaFree(p);
}
int wm_dev_upload(wm_ctx* ctx, void* dst, const void* src, int64_t bytes)
{
    if (ctx) cudaSetDevice(ctx->device);
    return cudaMemcpy(dst, src, (size_t)bytes, cudaMemcpyHostToDevice) == cudaSuccess ? WM_OK : WM_ERR_CUDA;
}
int wm_dev_download(wm_ctx* ctx, void* dst, const void* src, int64_t bytes)
{
    if (ctx) cudaSetDevice(ctx->device);
    return cudaMemcpy(dst, src, (size_t)bytes, cudaMemcpyDeviceToHost) == cudaSuccess ? WM_OK : WM_ERR_CUDA;
}
void* wm_host_alloc_pinned(int64_t bytes)
{
    void* p = nullptr;
    if (cudaMallocHost(&p, (size_t)bytes) != cudaSuccess) return nullptr;
    return p;
}
void wm_host_free_pinned(void* p) { if (p) cudaFreeHost(p); }

}  // extern "C"
