/*
 * wm_oracle.c — CPU restatement of the kar-dim/Watermarking-GPU hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under watermarking-gpu_b200/ (the product)
 * may include, link or call this file.  Only tests/, __graft_entry__.smoke()
 * and bench.py's cpu_baseline / --impl reference legs load it, and only as
 * the checker or the CPU baseline — never as the thing shipped.
 *
 * PARITY STATUS: the reference ships no tests, no golden vectors and no
 * recorded outputs (SURVEY.md §4, §8c) and cannot be built offline (ArrayFire
 * un-vendored, no OpenCL platform).  The three OpenCL kernels are PINNED: the
 * reference's own kernel source runs on the CPU under an OpenCL-C shim
 * (oracle/clshim -> oracle/_ref, see oracle/README.md) and
 * tests/test_oracle_vs_reference_kernels.py requires bit-for-bit agreement.
 * The ArrayFire library calls between them (sum, solve, norm, dot, max,
 * clamp) are restated from their documented semantics => for those
 * "parity unpinned".
 *
 * Conventions: all images are ROW-MAJOR (rows x cols) float arrays,
 * img[r*cols + c], i.e. the logical (row, col) indexing of the reference's
 * column-major af::array.  Neighbour order k=0..7 is the raster order of the
 * 3x3 window minus the centre (kernels/me_p3.hpp:46-54).  Out-of-image reads
 * clamp to the edge (CLK_ADDRESS_CLAMP_TO_EDGE, kernels/nvf.hpp:9).
 *
 * Where the reference's arithmetic is unspecified (ArrayFire reduction tree,
 * af::solve internals, -cl-mad-enable contraction) the oracle exposes the
 * choice as an option so tests can report the reference's own spread:
 *   fp16_products : 1 = products rounded to fp16 before summation
 *                       (kernels/me_p3.hpp:10-20), 0 = plain f32 products
 *   sum_f32       : 0 = cross-group / global sums in f64 (canonical),
 *                   1 = f32 pairwise tree
 *   solve_f32     : 0 = f64 LU (canonical), 1 = f32 LU, both partial pivoting
 *   contract      : 1 = a*b+c fused where -cl-mad-enable permits (canonical,
 *                       NVIDIA OpenCL behaviour), 0 = separately rounded
 *   p             : NVF window size (3 unless stated; the ME parts are p = 3 only,
 *                   as in the reference)
 *   rx_f64        : 0 = wmo_rx sums each 64-pixel group in f32 (the reference's
 *                       work-groups), 1 = every term is added in f64 — RN16(RN32(x*y))
 *                       with fp16_products, the exact x*y without — so the sums carry
 *                       no f32 rounding of their own (a reference to bound f32 sums by)
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#ifdef _OPENMP
#include <omp.h>
#endif

typedef struct {
    int fp16_products;
    int sum_f32;
    int solve_f32;
    int contract;
    int p;              /* NVF window size 3, 5, 7 or 9 (Watermark.cpp:24, kernels/nvf.hpp:14-17); 0 = 3 */
    int rx_f64;
} wmo_opts;

enum { WMO_ME = 0, WMO_NVF = 1 }; /* Watermark.hpp:10-14 */

static const int DY[8] = {-1, -1, -1, 0, 0, 1, 1, 1};
static const int DX[8] = {-1, 0, 1, -1, 1, -1, 0, 1};

static inline int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

static inline float px(const float *img, int rows, int cols, int r, int c)
{
    return img[(size_t)clampi(r, 0, rows - 1) * cols + clampi(c, 0, cols - 1)];
}

static inline float round_fp16(float v) { return (float)(_Float16)v; } /* vstore_half: RTE */

int wmo_num_threads(void)
{
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

/* Watermark.cpp:22 — strengthFactor = 255 / sqrt(10^(psnr/10)), float overloads */
float wmo_strength(float psnr) { return 255.0f / sqrtf(powf(10.0f, psnr / 10.0f)); }

/* f32 pairwise tree (one admissible instance of af::sum's unspecified order) */
static float pairwise_f32(const float *v, size_t n, size_t stride)
{
    if (n <= 8) {
        float s = 0.0f;
        for (size_t i = 0; i < n; i++) s += v[i * stride];
        return s;
    }
    size_t h = n / 2;
    return pairwise_f32(v, h, stride) + pairwise_f32(v + h * stride, n - h, stride);
}

static double reduce_f32_array(const float *v, size_t n, int sum_f32)
{
    if (sum_f32) return (double)pairwise_f32(v, n, 1);
    double s = 0.0;
    for (size_t i = 0; i < n; i++) s += (double)v[i];
    return s;
}

/* kernels/nvf.hpp:14-50 — NVF mask over the replicated p x p window (the kernel is compiled with -Dp, main.cpp:106) */
void wmo_nvf(const float *img, int rows, int cols, float *mask, const wmo_opts *o)
{
    const int contract = o->contract;
    const int pw = o->p ? o->p : 3, pad = pw / 2;
    const float psq = (float)(pw * pw); /* kernels/nvf.hpp:15,47: int pSquared, sum / pSquared */
#pragma omp parallel for schedule(static)
    for (int r = 0; r < rows; r++) {
        for (int c = 0; c < cols; c++) {
            float sum = 0.0f, sumSq = 0.0f;
            for (int i = -pad; i <= pad; i++)
                for (int j = -pad; j <= pad; j++) {
                    float v = px(img, rows, cols, r + i, c + j);
                    sum += v;
                    sumSq = contract ? fmaf(v, v, sumSq) : sumSq + v * v;
                }
            float mean = sum / psq;
            float q = sumSq / psq;
            float var = contract ? fmaf(-mean, mean, q) : q - mean * mean;
            mask[(size_t)r * cols + c] = var / (1.0f + var);
        }
    }
}

/*
 * kernels/me_p3.hpp:23-83 + Watermark.cpp:140-151,176-199.
 * Work-group = 64 consecutive columns of one row (global size align64(cols) x rows);
 * per pixel 8 rx products and 36 Rx products (upper triangle, RxMappings
 * Watermark.hpp:29-39), each rounded to fp16; per-group sums are sequential
 * f32 sums over the 64 work-items in ascending order (me_p3.hpp:61-68,76-82);
 * padded columns contribute 0.  Groups are then summed by af::sum.
 * Output: Rx[8*8] (full symmetric), rx[8] as doubles (holding f32 values when
 * sum_f32 is set).
 */
/* rx_f64: the same 44 terms per pixel (same neighbours, same clamp to the edge), each added in f64: one f64 partial per
 * row, rows added in ascending order (the same bits for any thread count) */
static void rx_terms_f64(const float *img, int rows, int cols, int fp16, double *tot)
{
    double *part = (double *)calloc((size_t)rows * 44, sizeof(double));
#pragma omp parallel for schedule(static)
    for (int r = 0; r < rows; r++) {
        double acc[44];
        for (int t = 0; t < 44; t++) acc[t] = 0.0;
        for (int c = 0; c < cols; c++) {
            float n[8];
            for (int k = 0; k < 8; k++) n[k] = px(img, rows, cols, r + DY[k], c + DX[k]);
            const float cur = img[(size_t)r * cols + c];
            int t = 0;
            for (int k = 0; k < 8; k++, t++)
                acc[t] += fp16 ? (double)round_fp16(n[k] * cur) : (double)n[k] * (double)cur;
            for (int i = 0; i < 8; i++)
                for (int j = i; j < 8; j++, t++)
                    acc[t] += fp16 ? (double)round_fp16(n[i] * n[j]) : (double)n[i] * (double)n[j];
        }
        for (int t = 0; t < 44; t++) part[(size_t)r * 44 + t] = acc[t];
    }
    for (int t = 0; t < 44; t++) tot[t] = 0.0;
    for (int r = 0; r < rows; r++)
        for (int t = 0; t < 44; t++) tot[t] += part[(size_t)r * 44 + t];
    free(part);
}

void wmo_rx(const float *img, int rows, int cols, const wmo_opts *o, double *Rx, double *rx)
{
    if (o->rx_f64) {
        double tot[44];
        rx_terms_f64(img, rows, cols, o->fp16_products, tot);
        for (int k = 0; k < 8; k++) rx[k] = tot[k];
        int t = 8;
        for (int i = 0; i < 8; i++)
            for (int j = i; j < 8; j++, t++) Rx[i * 8 + j] = Rx[j * 8 + i] = tot[t];
        return;
    }
    const int gpr = (cols + 63) / 64; /* groups per row */
    const size_t ngroups = (size_t)rows * gpr;
    float *part = (float *)malloc(ngroups * 44 * sizeof(float)); /* [44][ngroups] */
    const int fp16 = o->fp16_products;
#pragma omp parallel for schedule(static)
    for (int r = 0; r < rows; r++) {
        for (int g = 0; g < gpr; g++) {
            float acc[44];
            for (int t = 0; t < 44; t++) acc[t] = 0.0f;
            const int c0 = g * 64, c1 = c0 + 64 < cols ? c0 + 64 : cols;
            for (int c = c0; c < c1; c++) {
                float n[8];
                for (int k = 0; k < 8; k++) n[k] = px(img, rows, cols, r + DY[k], c + DX[k]);
                const float cur = img[(size_t)r * cols + c];
                int t = 0;
                for (int k = 0; k < 8; k++, t++) {
                    float p = n[k] * cur;
                    acc[t] += fp16 ? round_fp16(p) : p;
                }
                for (int i = 0; i < 8; i++)
                    for (int j = i; j < 8; j++, t++) {
                        float p = n[i] * n[j];
                        acc[t] += fp16 ? round_fp16(p) : p;
                    }
            }
            const size_t gi = (size_t)r * gpr + g;
            for (int t = 0; t < 44; t++) part[(size_t)t * ngroups + gi] = acc[t];
        }
    }
    double tot[44];
#pragma omp parallel for schedule(static)
    for (int t = 0; t < 44; t++) tot[t] = reduce_f32_array(part + (size_t)t * ngroups, ngroups, o->sum_f32);
    free(part);
    for (int k = 0; k < 8; k++) rx[k] = tot[k];
    int t = 8;
    for (int i = 0; i < 8; i++)
        for (int j = i; j < 8; j++, t++) Rx[i * 8 + j] = Rx[j * 8 + i] = tot[t];
}

/* Watermark.cpp:203 — af::solve(Rx, rx): general square system, LU with partial
 * pivoting.  Returns 0 ok, 1 singular (the reference's af::exception branch,
 * Watermark.cpp:205-208).  Singularity rule (reference undefined, SURVEY App. A):
 * |pivot| <= 1e-12 * max|Rx| (f64) or 1e-6 * max|Rx| (f32). */
int wmo_solve8(const double *Rx, const double *rx, int solve_f32, double *c)
{
    double amax = 0.0;
    for (int i = 0; i < 64; i++) amax = fmax(amax, fabs(Rx[i]));
    if (!(amax > 0.0) || !isfinite(amax)) return 1;
    if (solve_f32) {
        float A[8][9];
        for (int i = 0; i < 8; i++) {
            for (int j = 0; j < 8; j++) A[i][j] = (float)Rx[i * 8 + j];
            A[i][8] = (float)rx[i];
        }
        const float tol = 1e-6f * (float)amax;
        for (int k = 0; k < 8; k++) {
            int piv = k;
            for (int i = k + 1; i < 8; i++)
                if (fabsf(A[i][k]) > fabsf(A[piv][k])) piv = i;
            if (!(fabsf(A[piv][k]) > tol)) return 1;
            if (piv != k)
                for (int j = 0; j < 9; j++) { float t = A[k][j]; A[k][j] = A[piv][j]; A[piv][j] = t; }
            for (int i = k + 1; i < 8; i++) {
                float f = A[i][k] / A[k][k];
                for (int j = k; j < 9; j++) A[i][j] -= f * A[k][j];
            }
        }
        for (int i = 7; i >= 0; i--) {
            float s = A[i][8];
            for (int j = i + 1; j < 8; j++) s -= A[i][j] * (float)c[j];
            c[i] = (double)(s / A[i][i]);
        }
        return 0;
    }
    double A[8][9];
    for (int i = 0; i < 8; i++) {
        for (int j = 0; j < 8; j++) A[i][j] = Rx[i * 8 + j];
        A[i][8] = rx[i];
    }
    const double tol = 1e-12 * amax;
    for (int k = 0; k < 8; k++) {
        int piv = k;
        for (int i = k + 1; i < 8; i++)
            if (fabs(A[i][k]) > fabs(A[piv][k])) piv = i;
        if (!(fabs(A[piv][k]) > tol)) return 1;
        if (piv != k)
            for (int j = 0; j < 9; j++) { double t = A[k][j]; A[k][j] = A[piv][j]; A[piv][j] = t; }
        for (int i = k + 1; i < 8; i++) {
            double f = A[i][k] / A[k][k];
            for (int j = k; j < 9; j++) A[i][j] -= f * A[k][j];
        }
    }
    for (int i = 7; i >= 0; i--) {
        double s = A[i][8];
        for (int j = i + 1; j < 8; j++) s -= A[i][j] * c[j];
        c[i] = s / A[i][i];
    }
    return 0;
}

/* kernels/scaled_neighbors_p3.hpp:34-43 — dot = sum_k coeffs[k]*n_k, k ascending, f32 */
void wmo_scaled_neighbors(const float *img, int rows, int cols, const float *coef, float *out,
                          const wmo_opts *o)
{
    const int contract = o->contract;
#pragma omp parallel for schedule(static)
    for (int r = 0; r < rows; r++)
        for (int c = 0; c < cols; c++) {
            float dot = 0.0f;
            for (int k = 0; k < 8; k++) {
                float v = px(img, rows, cols, r + DY[k], c + DX[k]);
                dot = contract ? fmaf(coef[k], v, dot) : dot + coef[k] * v;
            }
            out[(size_t)r * cols + c] = dot;
        }
}

/* af::max<float>(abs(e)) */
static float max_abs(const float *e, size_t n)
{
    float m = 0.0f;
#pragma omp parallel for reduction(max : m) schedule(static)
    for (size_t i = 0; i < n; i++) {
        float a = fabsf(e[i]);
        if (a > m) m = a;
    }
    return m;
}

/* sum over elements of a[i]*b[i], products in f32 (ArrayFire element-wise mul
 * node), summed in f64 (canonical) or f32 pairwise. */
static double sum_prod(const float *a, const float *b, size_t n, int sum_f32)
{
    if (sum_f32) {
        float *t = (float *)malloc(n * sizeof(float));
#pragma omp parallel for schedule(static)
        for (size_t i = 0; i < n; i++) t[i] = a[i] * b[i];
        double s = (double)pairwise_f32(t, n, 1);
        free(t);
        return s;
    }
    /* deterministic: per-row-block f64 partials summed in order */
    const size_t B = 4096, nb = (n + B - 1) / B;
    double *pb = (double *)malloc(nb * sizeof(double));
#pragma omp parallel for schedule(static)
    for (size_t k = 0; k < nb; k++) {
        double s = 0.0;
        size_t e = (k + 1) * B < n ? (k + 1) * B : n;
        for (size_t i = k * B; i < e; i++) s += (double)(a[i] * b[i]);
        pb[k] = s;
    }
    double s = 0.0;
    for (size_t k = 0; k < nb; k++) s += pb[k];
    free(pb);
    return s;
}

/*
 * Watermark.cpp:176-218 — computePredictionErrorMask.
 * e (rows*cols) and coef[8] always written when solvable; mask written when
 * mask != NULL (maskNeeded).  Returns 0 ok, 1 unsolvable.
 * dbg_Rx (64) / dbg_rx (8) optional.
 */
int wmo_pred_error_mask(const float *img, int rows, int cols, const wmo_opts *o, float *e,
                        float *coef, float *mask, double *dbg_Rx, double *dbg_rx)
{
    double Rx[64], rx[8], c[8];
    wmo_rx(img, rows, cols, o, Rx, rx);
    if (dbg_Rx) memcpy(dbg_Rx, Rx, sizeof Rx);
    if (dbg_rx) memcpy(dbg_rx, rx, sizeof rx);
    if (wmo_solve8(Rx, rx, o->solve_f32, c)) return 1;
    for (int k = 0; k < 8; k++) coef[k] = (float)c[k];
    const size_t n = (size_t)rows * cols;
    wmo_scaled_neighbors(img, rows, cols, coef, e, o);
#pragma omp parallel for schedule(static)
    for (size_t i = 0; i < n; i++) e[i] = img[i] - e[i]; /* Watermark.cpp:210 */
    if (mask) {
        const float m = max_abs(e, n); /* Watermark.cpp:213-214 */
#pragma omp parallel for schedule(static)
        for (size_t i = 0; i < n; i++) mask[i] = fabsf(e[i]) / m;
    }
    return 0;
}

/*
 * Watermark.cpp:171 — out = clamp(base + u*a, 0, 255) over n pixels of one plane.
 * ArrayFire JIT fuses clamp(out + u*a) into one OpenCL kernel; FP_CONTRACT defaults ON in
 * OpenCL C, so the mul-add may fuse (`contract`: one rounding, fmaf).  Exposed on its own so
 * that tests can apply a strength and a u plane taken from the GPU.
 */
void wmo_apply(const float *base, const float *u, size_t n, float a, int contract, float *out)
{
#pragma omp parallel for schedule(static)
    for (size_t i = 0; i < n; i++) {
        float v = contract ? fmaf(u[i], a, base[i]) : base[i] + u[i] * a;
        out[i] = v < 0.0f ? 0.0f : (v > 255.0f ? 255.0f : v);
    }
}

/*
 * Watermark.cpp:156-172 — makeWatermark.
 * in: gray rows*cols; base/out: channels planes of rows*cols (channels 1 or 3;
 * the reference broadcasts u*a over the RGB planes, Watermark.cpp:171).
 * Returns 0 ok, 1 unsolvable (out = base unchanged, *a untouched,
 * Watermark.cpp:164-165), 2 zero-norm mask (reference undefined: inf/NaN;
 * oracle defines out = base, *a = inf).
 * Optional debug outputs: mask_out, u_out (rows*cols each), coef_out[8].
 */
int wmo_embed(const float *in, const float *base, int channels, int rows, int cols, const float *W,
              float psnr, int mask_type, const wmo_opts *o, float *out, float *a, float *mask_out,
              float *u_out, float *coef_out)
{
    const size_t n = (size_t)rows * cols;
    float *mask = mask_out ? mask_out : (float *)malloc(n * sizeof(float));
    float *u = u_out ? u_out : (float *)malloc(n * sizeof(float));
    int status = 0;
    if (mask_type == WMO_ME) {
        float *e = (float *)malloc(n * sizeof(float));
        float coef[8];
        status = wmo_pred_error_mask(in, rows, cols, o, e, coef, mask, NULL, NULL);
        if (!status && coef_out) memcpy(coef_out, coef, sizeof coef);
        free(e);
    } else {
        wmo_nvf(in, rows, cols, mask, o);
    }
    if (status) {
        memcpy(out, base, n * channels * sizeof(float));
    } else {
#pragma omp parallel for schedule(static)
        for (size_t i = 0; i < n; i++) u[i] = mask[i] * W[i]; /* Watermark.cpp:169 */
        /* af::norm(u): sqrt in double of the f32-typed sum of squares */
        const double nrm = sqrt(sum_prod(u, u, n, o->sum_f32));
        const float sf = wmo_strength(psnr);
        const float av = sf / (float)(nrm / sqrt((double)n)); /* Watermark.cpp:170 */
        *a = av;
        if (!(nrm > 0.0)) {
            memcpy(out, base, n * channels * sizeof(float));
            status = 2;
        } else {
            for (int ch = 0; ch < channels; ch++)
                wmo_apply(base + (size_t)ch * n, u, n, av, o->contract, out + (size_t)ch * n);
        }
    }
    if (!mask_out) free(mask);
    if (!u_out) free(u);
    return status;
}

/*
 * Watermark.cpp:234-250 (+221-231) — detectWatermark.
 * Returns 0 ok (corr written), 1 unsolvable (corr = 0, Watermark.cpp:246-247).
 * Optional debug outputs ez_out, u_out, eu_out (rows*cols), coef_out[8].
 */
int wmo_detect(const float *img, int rows, int cols, const float *W, int mask_type,
               const wmo_opts *o, float *corr, float *ez_out, float *u_out, float *eu_out,
               float *coef_out)
{
    const size_t n = (size_t)rows * cols;
    float *ez = ez_out ? ez_out : (float *)malloc(n * sizeof(float));
    float *u = u_out ? u_out : (float *)malloc(n * sizeof(float));
    float *eu = eu_out ? eu_out : (float *)malloc(n * sizeof(float));
    float *mask = (float *)malloc(n * sizeof(float));
    float coef[8];
    int status;
    if (mask_type == WMO_NVF) {
        status = wmo_pred_error_mask(img, rows, cols, o, ez, coef, NULL, NULL, NULL);
        if (!status) wmo_nvf(img, rows, cols, mask, o);
    } else {
        status = wmo_pred_error_mask(img, rows, cols, o, ez, coef, mask, NULL, NULL);
    }
    *corr = 0.0f;
    if (!status) {
        if (coef_out) memcpy(coef_out, coef, sizeof coef);
#pragma omp parallel for schedule(static)
        for (size_t i = 0; i < n; i++) u[i] = mask[i] * W[i]; /* Watermark.cpp:248 */
        /* computeErrorSequence (Watermark.cpp:221-225): u is staged into the texture,
         * so neighbour reads of u clamp on u's own frame */
        wmo_scaled_neighbors(u, rows, cols, coef, eu, o);
#pragma omp parallel for schedule(static)
        for (size_t i = 0; i < n; i++) eu[i] = u[i] - eu[i];
        /* computeCorrelation (Watermark.cpp:228-231) */
        const float dot = (float)sum_prod(eu, ez, n, o->sum_f32);
        const double nz = sqrt(sum_prod(ez, ez, n, o->sum_f32));
        const double nu = sqrt(sum_prod(eu, eu, n, o->sum_f32));
        *corr = dot / (float)(nz * nu);
    }
    free(mask);
    if (!ez_out) free(ez);
    if (!u_out) free(u);
    if (!eu_out) free(eu);
    return status;
}

/*
 * Video frame path, main.cpp:343-389 / 392-410: Y plane u8 row-major (height x
 * width, row stride `linesize`), repacked when linesize != width, cast to f32,
 * makeWatermark(frame, frame, a, ME), `.as(u8)` = truncation of the clamped
 * f32, written back contiguous.
 */
int wmo_embed_frame_u8(const uint8_t *y_in, int linesize, int height, int width, const float *W,
                       float psnr, int mask_type, const wmo_opts *o, uint8_t *y_out, float *a)
{
    const size_t n = (size_t)height * width;
    float *f = (float *)malloc(n * sizeof(float));
    float *g = (float *)malloc(n * sizeof(float));
    for (int r = 0; r < height; r++)
        for (int c = 0; c < width; c++) f[(size_t)r * width + c] = (float)y_in[(size_t)r * linesize + c];
    int st = wmo_embed(f, f, 1, height, width, W, psnr, mask_type, o, g, a, NULL, NULL, NULL);
    for (size_t i = 0; i < n; i++) y_out[i] = (uint8_t)g[i];
    free(f);
    free(g);
    return st;
}

int wmo_detect_frame_u8(const uint8_t *y_in, int linesize, int height, int width, const float *W,
                        int mask_type, const wmo_opts *o, float *corr)
{
    const size_t n = (size_t)height * width;
    float *f = (float *)malloc(n * sizeof(float));
    for (int r = 0; r < height; r++)
        for (int c = 0; c < width; c++) f[(size_t)r * width + c] = (float)y_in[(size_t)r * linesize + c];
    int st = wmo_detect(f, height, width, W, mask_type, o, corr, NULL, NULL, NULL, NULL);
    free(f);
    return st;
}

/* main.cpp:142-154 — af::rgb2gray(rgb, 0.299, 0.587, 0.114) on planar f32 0..255 */
void wmo_rgb2gray(const float *rgb, size_t n, float *gray)
{
    for (size_t i = 0; i < n; i++)
        gray[i] = (0.299f * rgb[i] + 0.587f * rgb[n + i]) + 0.114f * rgb[2 * n + i];
}
