"""References and error bounds for checking the 8-bit kernels one by one at full frame sizes (test_gpu_u8_kernels_full_size.py).

Every reference is built from the GPU's own inputs to the kernel under test (its mask plane, its `a`, its output bytes), so the
rounding of one stage never enters the check of the next.  Pixels are integers throughout: the Rx sweep, the masks, the prediction
error and the apply step are exact functions of their inputs, and the stats and detector sums have the short bounds derived below.
test_u8_exact_checks.py shows on the CPU that the byte check and these bounds catch the defects they target.
"""
import math
import os
import re

import numpy as np

import util

U32 = 2.0 ** -24  # unit roundoff of f32 round-to-nearest
U64 = 2.0 ** -53  # ... of f64

# (rows, cols, row pitch in bytes): HD, the reference's odd-size samples (1078 x 1918, 2160 x 3872), 4K, and two small frames whose
# tiles overhang the image (67 x 131) or whose rows are padded (130 x 264 in rows of 272 bytes)
SIZES = [(1080, 1920, 1920), (1078, 1918, 1918), (2160, 3840, 3840), (2160, 3872, 3872), (67, 131, 131), (130, 264, 272)]
SEGMENT = 128  # pixels of one line of a tile: what a thread group sums together (TP in wm_kernels.cuh)

_KERNELS = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "watermarking-gpu_b200", "csrc", "wm_kernels.cuh")


def _tile_lines():
    with open(_KERNELS) as f:
        return int(re.search(r"constexpr int TL = (\d+);", f.read()).group(1))


TL = _tile_lines()


def chain_len(threads):
    """f32 terms one thread of a stats or detector CTA of `threads` threads adds up in a tile before the sum goes to f64.

    A thread owns 4 pixels of each of LPT = TL / (threads / 32) lines of a tile (wm_kernels.cuh: k_stats, detect_tile) and folds the
    term of each pixel into one f32 register: 4 * LPT terms.  The narrow u8 kernels (WM_OPT_NARROW_U8, 128 threads) add 32, the
    256-thread ones 16."""
    return 4 * TL // (threads // 32)


def narrow_u8(opts, ld, cols, bstride=None):
    """Whether a u8 image (rows `ld` bytes apart, batch stride `bstride` bytes, device pointer 16-byte aligned) runs the narrow
    128-thread stats / detector: WM_OPT_NARROW_U8 and TMA loads (wm_api.cu: tma_ok).  opts: the options set away from their defaults."""
    return (opts.get("NARROW_U8", 1) and opts.get("USE_TMA", 1) and ld % 16 == 0 and cols % 4 == 0
            and (bstride is None or bstride % 16 == 0))


def gamma(n, u):
    """gamma_n = n u / (1 - n u): the relative error bound of n roundings (Higham, Accuracy and Stability of Numerical Algorithms, 3.1)."""
    return n * u / (1.0 - n * u)


def sum_rel_bound(k, n, u=U32):
    """Bound on |S_gpu / S_ref - 1| for S = sum of n nonnegative terms t = x^2 of f32 values x (the stats kernel's sum2 = sum (m.W)^2,
    the detector's |e_z|^2 and |e_u|^2).

    Kernel: each thread folds its k terms of a tile into one f32 register, s = fma(x, x, s) from 0: the product is exact, each of the
    k additions rounds once, and because every term is >= 0 the chain ends within gamma_k(2^-24) of its exact sum.  The chains go to
    f64 exactly and are added there in some tree of at most n values: another gamma_n(2^-53) of the total.
    Reference: the f64 sum of the exact squares (x^2 of an f32 x has 48 significant bits): within gamma_n(2^-53) of the exact sum.
    Together |S_gpu - S_ref| <= (gamma_k(2^-24) + 3 gamma_n(2^-53)) S_exact, and S_exact <= S_ref / (1 - gamma_n(2^-53)).
    k = 32 (narrow u8 kernels): 1.91e-6.  u: the relative error of one step of the chain where it is not an f32 round-to-nearest
    addition (f32_exact.U_MMA: one step of the tensor pipe's accumulation)."""
    g = gamma(n, U64)
    return (gamma(k, u) + 3 * g) / (1 - g)


def dot_abs_bound(k, n, nz_ref, nu_ref):
    """Bound on |dot_gpu - dot_ref| for dot = sum e_u e_z over n pixels, k terms per f32 chain as in sum_rel_bound.

    Terms of both signs: a chain of k fma steps ends within gamma_k(2^-24) sum |e_u e_z| of its exact value, the f64 stages and the
    reference add gamma_n(2^-53) sum |e_u e_z| each, and by Cauchy-Schwarz sum |e_u e_z| <= sqrt(|e_z|^2 |e_u|^2), taken from the
    reference norms with their own f64 error."""
    g = gamma(n, U64)
    return (gamma(k, U32) + 3 * g) * math.sqrt(nz_ref * nu_ref) / (1 - g)


def a_rel_bound(k, n):
    """Bound on |a_gpu / a_ref - 1| for the strength a = strength / (sqrt(S) [/ max|e|] / sqrt(N)) (Watermark.cpp:170).

    Kernel (k_stats, last block): the norm in f64 from its sum2 (a few f64 roundings), rounded to f32, then one f32 division:
    a_gpu = strength / d64 * (1 + d1) / (1 + d2) with |d1|, |d2| <= 2^-24.  Reference: the same formula in f64 from S_ref and the
    same max|e|.  With |S_gpu / S_ref - 1| <= eps (sum_rel_bound), sqrt(S_ref / S_gpu) lies in [1 / sqrt(1 + eps), 1 / sqrt(1 - eps)];
    eight f64 roundings on both sides cover the rest.  k = 32: 1.07e-6, k = 16: 5.9e-7."""
    e = sum_rel_bound(k, n)
    f64 = (1 + U64) ** 8
    hi = (1 / math.sqrt(1 - e)) * (1 + U32) / (1 - U32) * f64 - 1
    lo = 1 - (1 / math.sqrt(1 + e)) * (1 - U32) / (1 + U32) / f64
    return max(hi, lo)


def corr_abs_bound(k, n, dot_ref, nz_ref, nu_ref):
    """Bound on |corr_gpu - corr_ref|, corr = dot / (|e_z| |e_u|) (Watermark.cpp:228-231).

    Kernel (k_detect, last block): corr = RN32(RN32(dot) / RN32(sqrt(nz) sqrt(nu))), the square roots and their product in f64.
    Its sums lie in dot_ref +- dot_abs_bound and nz_ref, nu_ref (1 +- sum_rel_bound); the quotient is monotonic in each, so the
    extreme values lie at the corners of that box, times the three f32 roundings (and three f64 ones) at their extremes.  The
    reference correlation itself carries a few f64 roundings."""
    ed = dot_abs_bound(k, n, nz_ref, nu_ref)
    es = sum_rel_bound(k, n)
    ref = dot_ref / math.sqrt(nz_ref * nu_ref)
    fmin = (1 - U32) ** 2 / (1 + U32) / (1 + U64) ** 3
    fmax = (1 + U32) ** 2 / (1 - U32) / (1 - U64) ** 3
    worst = 0.0
    for d in (dot_ref - ed, dot_ref + ed):
        for z in (nz_ref * (1 - es), nz_ref * (1 + es)):
            for u in (nu_ref * (1 - es), nu_ref * (1 + es)):
                for f in (fmin, fmax):
                    worst = max(worst, abs(d / math.sqrt(z * u) * f - ref))
    return worst + 4 * U64 * abs(ref)


def unequal_bytes(got, want):
    """Number of pixels where the 8-bit output differs from its reference: the check allows none."""
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape and got.dtype == np.uint8 and want.dtype == np.uint8, (got.shape, got.dtype, want.shape, want.dtype)
    return int(np.count_nonzero(got != want))


def apply_ref(oracle, base, mask, W, a):
    """The apply kernel's output for the GPU's own mask plane and strength: u = RN32(mask W), clamp(fma(u, a, base), 0, 255) in f32
    (oracle.apply).  -> (f32 output, u8 output = its truncation, like `.as(u8)`)."""
    u = np.asarray(mask, np.float32) * np.asarray(W, np.float32)
    out = oracle.apply(np.asarray(base, np.float32), u, a)
    return out, out.astype(np.uint8)


def clamps_fired(base, mask, W, a):
    """(pixels clamped at 0, pixels clamped at 255) by the apply step: base + u a outside [0, 255]."""
    v = np.asarray(base, np.float64) + (np.asarray(mask, np.float32) * np.asarray(W, np.float32)).astype(np.float64) * float(a)
    return int(np.count_nonzero(v < 0)), int(np.count_nonzero(v > 255))


def frame(rows, cols, seed):
    """A natural 8-bit frame with a patch near 255 in its top half and one near 0 in its bottom half.  The patches carry +-2 of noise
    so that they do not make the prediction system singular, and they make the apply step clamp at both ends."""
    img = util.natural_image(rows, cols, seed=seed, integer=True)
    rng = np.random.default_rng(seed + 1)
    ph, pw = max(rows // 8, 4), max(cols // 8, 4)
    for level, lo in ((255, 0), (0, rows // 2)):
        r0 = int(rng.integers(lo, lo + rows // 2 - ph + 1))
        c0 = int(rng.integers(0, cols - pw + 1))
        img[r0:r0 + ph, c0:c0 + pw] = np.clip(level + rng.integers(-2, 3, (ph, pw)), 0, 255)
    return img
