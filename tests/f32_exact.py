"""References and error bounds for checking the f32 kernels one by one at full frame sizes (test_gpu_f32_kernels_full_size.py).

The f32 path differs from the 8-bit one (u8_exact.py) in one place: real-valued pixels make the Rx sweep inexact.  Its terms are
RN16(RN32(x y)) (the exact x y with WM_OPT_FP16_PRODUCTS = 0) and their f32 sums round, so Rx and rx get a bound of their own
(rx_rel_bound), against the oracle's rx_f64 mode, which adds the same terms in f64.  Every later stage is an exact function of the
GPU's own inputs to it — the coefficients are the f64 (or f32) LU of the GPU's Rx, the planes follow from the coefficients, the output
from the mask plane and `a` — and is checked bit for bit; the stats and detector sums keep the bounds of u8_exact.py with the chain of
the 256-thread kernels.  test_f32_exact_checks.py shows on the CPU that these bounds hold for simulated accumulators and that the
output check rejects the defects it targets.
"""
import math
import os
import re

import numpy as np

import util
from u8_exact import SEGMENT, TL, U32, U64, a_rel_bound, apply_ref, chain_len, corr_abs_bound, dot_abs_bound, gamma, sum_rel_bound  # noqa: F401

# (rows, cols, ld in elements of a ROW_MAJOR image; 0 = dense): HD, the reference's odd-size samples, 4K, a frame whose tiles overhang
# it and one with padded rows.  COL_MAJOR images of these sizes keep the same padding: ld = rows + (ld - cols).
SIZES = [(1080, 1920, 0), (1078, 1918, 0), (2160, 3840, 0), (2160, 3872, 0), (67, 131, 0), (130, 264, 272)]

_KERNELS = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "watermarking-gpu_b200", "csrc", "wm_kernels.cuh")


def _source():
    with open(_KERNELS) as f:
        return f.read()


def _int(pattern):
    return int(re.search(pattern, _source()).group(1))


SNT = _int(r"constexpr int SNT = (\d+)")                       # threads of a sweep CTA
SLPT = TL // (SNT // 32)                                        # lines of a tile one sweep thread takes
FLUSH = _int(r"if \(\(k & (\d+)\) == \1\) flush\(\);") + 1      # tiles between two flushes of the f32 (HMMA / FHADD) lag accumulators
RING = _int(r"\+\+chunks == (\d+)\)")                           # ring chunks one thread sums in f32 before its block sum (per-thread mode)
SWEEP_CTAS_PER_SM = _int(r"constexpr int SWEEP_CTAS_PER_SM = (\d+);")
FUSED_NST = _int(r"DETECT_NST = (\d+);")                       # resident tiles per CTA of k_detect1 (NST = DETECT_NST there)
FUSED_LPT = _int(r"sweep_tile_mma<true, (\d+), 2>")             # lines per thread of k_detect1's sweep phase

# One step of the HMMA accumulation (mma_acc4: mma.sync m16n8k16, f16 x f16 + f32, B a 0/1 selector) adds two fp16 addends t1, t2
# (products by 1.0 are exact; every other product of the row is 0) to the f32 accumulator c.  Its alignment and normalisation are not
# documented as round-to-nearest, and published measurements on earlier NVIDIA tensor cores (Fasi, Higham, Mikaitis, Pranesh,
# "Numerical behavior of NVIDIA tensor cores", PeerJ Comput. Sci. 2021) found truncation.  Model: the three addends, all >= 0 here, are
# aligned to the exponent E of the largest with a 24-bit significand, the bits shifted out are dropped, the aligned values are added
# exactly, and the sum is truncated to 24 bits.  The largest addend loses nothing; each of the two others loses less than 2^(E-23)
# <= 2^-23 s (s = c + t1 + t2, every addend >= 0); the truncation of the sum loses less than 2^-23 s.  So one step gives s (1 - theta),
# 0 <= theta < 3 * 2^-23, and a chain of k steps from 0 ends within 1 - (1 - U_MMA)^k <= gamma_k(U_MMA) of its exact sum.  Round to
# nearest, or guard bits in the alignment, only make the error smaller.  Six times the unit roundoff of an f32 addition.
U_MMA = 3 * 2.0 ** -23


def mode_of(opts):
    """Sweep accumulation of a synchronous embed / detect with the options `opts` set away from their defaults -> (embed, detect)."""
    if not opts.get("FP16_PRODUCTS", 1):
        return "ffma", "ffma"
    if not opts.get("MMA_ACCUM", 1):
        return "fhadd", "fhadd"
    return "hmma", ("fused" if opts.get("FUSED_SINGLE", 0) else "hmma")


def sweep_chains(mode):
    """The f32 chains an Rx / rx entry of the sweep is made of, as (steps, unit) with every step's relative error below `unit`.

    k_sweep (SNT-thread CTAs, SLPT lines of a tile per thread, 4 px per line): a thread's lag accumulators go to f64 every FLUSH tiles.
      hmma  (default): lags 0..11: two HMMA steps per line (pixel pairs 0-1 and 2-3), 2 SLPT FLUSH = 64 steps of U_MMA; lag 12: one step
            per two lines, SLPT / 2 FLUSH = 16 steps, then two f32 additions (c12 + c13) + (c14 + c15).
      fhadd (WM_OPT_MMA_ACCUM = 0): add.rn.f32.f16 rounds to nearest: the even / odd accumulator takes 2 SLPT FLUSH = 64 terms, then
            one addition e0 + e1: 65 roundings of U32.
      ffma  (WM_OPT_FP16_PRODUCTS = 0): the same chain with fma(x, y, e): exact products, 65 roundings.
    frame ring (sweep_ring): per-thread mode adds one product per chunk in f32, RING chunks before the block sum in f64 (FHADD or an f32
      addition: RN); the products of ffma are rounded to f32 there (one more rounding).  The one-warp-per-pixel mode adds in f64.
    fused (k_detect1, WM_OPT_FUSED_SINGLE): FUSED_NST resident tiles, FUSED_LPT lines per thread, nothing flushed in between:
      2 FUSED_LPT FUSED_NST HMMA steps for lags 0..11, FUSED_LPT / 2 FUSED_NST steps + 2 additions for lag 12; its ring adds in f64.
    An addition that rounds to nearest is counted as a step of the larger unit U_MMA where it ends an HMMA chain."""
    tile = 2 * SLPT * FLUSH
    if mode == "hmma":
        return [(tile, U_MMA), (SLPT // 2 * FLUSH + 2, U_MMA), (RING, U32)]
    if mode == "fhadd":
        return [(tile + 1, U32), (RING, U32)]
    if mode == "ffma":
        return [(tile + 1, U32), (RING + 1, U32)]
    if mode == "fused":
        return [(2 * FUSED_LPT * FUSED_NST, U_MMA), (FUSED_LPT // 2 * FUSED_NST + 2, U_MMA)]
    raise ValueError(mode)


def rx_rel_bound(mode, n):
    """Bound on |Rx_gpu / Rx_ref - 1| for every entry of Rx and rx of an image of n pixels, Rx_ref = oracle.rx(rx_f64=1).

    Pixels are >= 0 (at most 255, or 255.75 for 10-bit samples / 4), so every term is >= 0 and an entry is a sum of nonnegative terms: the f32 chain that ends furthest from its
    exact sum (sweep_chains) bounds the relative error of the whole entry.  The GPU adds its chains in f64 (per thread, per CTA, per
    group of CTAs, core + frame ring: fewer than 2 n values) and the reference adds its terms in f64: sum_rel_bound with 2 n f64 values.
    hmma: 2.29e-5, fhadd and ffma: 3.87e-6, fused: 5.72e-6."""
    return max(sum_rel_bound(k, 2 * n, u) for k, u in sweep_chains(mode))


def rx_size_limit(mode):
    """The largest frame (pixels) at which rx_rel_bound stays below half the change one missing 128-pixel segment of average terms
    makes to an Rx entry (SEGMENT / n of it).  Above it, only the exact check on integer-valued pixels sees a missing segment."""
    lo, hi = 1, 1 << 40
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if rx_rel_bound(mode, mid) < 0.5 * SEGMENT / mid else (lo, mid)
    return lo


def frame(rows, cols, seed):
    """A real-valued natural frame (no pixel is an integer but by chance) with a patch of uniform values in [251, 255) in its top half
    and one in [0, 4) in its bottom half (noisy, so that the prediction system stays regular): the apply step clamps at both ends."""
    img = util.natural_image(rows, cols, seed=seed)
    rng = np.random.default_rng(seed + 1)
    ph, pw = max(rows // 8, 4), max(cols // 8, 4)
    for lo_level, r_lo in ((251.0, 0), (0.0, rows // 2)):
        r0 = int(rng.integers(r_lo, r_lo + rows // 2 - ph + 1))
        c0 = int(rng.integers(0, cols - pw + 1))
        img[r0:r0 + ph, c0:c0 + pw] = lo_level + rng.uniform(0.0, 4.0, (ph, pw)).astype(np.float32)
    return img


def error_plane(oracle, f, c):
    """e = I - pred with the coefficients c (scaled_neighbors_p3: k ascending, fused): the kernels' DBG_ERRSEQ for those coefficients."""
    f = np.asarray(f, np.float32)
    return f - oracle.scaled_neighbors(f, np.asarray(c, np.float32))


def me_mask(e):
    """|e| / max|e|, correctly rounded (Watermark.cpp:213-214)."""
    a = np.abs(e)
    return a / a.max()


def mask_plane(oracle, f, c, mask, p=3):
    """The mask plane the embed applies: ME from the coefficients c, NVF of a p x p window."""
    return me_mask(error_plane(oracle, f, c)) if mask == oracle.ME else oracle.nvf(f, oracle.opts(p=p))


def stats_input(oracle, f, c, mask, p=3):
    """The plane whose (x W)^2 the stats kernel sums: |e| for ME (the 1 / max|e| comes after), the NVF mask for NVF -> (x, e or None)."""
    if mask == oracle.ME:
        e = error_plane(oracle, f, c)
        return np.abs(e), e
    return oracle.nvf(f, oracle.opts(p=p)), None


def detect_planes(oracle, z, c, W, mask, p=3):
    """The detector's planes of z for the coefficients c: e_z, u = m W (ME: m = |e_z|, the 1 / max|e_z| scale cancels in the
    correlation and the kernels drop it), e_u = u - pred(u) with u clamped on its own frame (Watermark.cpp:221-225)."""
    ez = error_plane(oracle, z, c)
    m = np.abs(ez) if mask == oracle.ME else oracle.nvf(np.asarray(z, np.float32), oracle.opts(p=p))
    u = m * np.asarray(W, np.float32)
    return ez, u, error_plane(oracle, u, c)


def unequal(got, want):
    """Number of values whose bits differ (f32 planes and outputs, 16-bit words): the exact checks allow none."""
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape and got.dtype == want.dtype, (got.shape, got.dtype, want.shape, want.dtype)
    if got.dtype == np.float32:
        got, want = got.view(np.uint32), want.view(np.uint32)
    return int(np.count_nonzero(got != want))


def clamps(base, m, W, a):
    """(values clamped at 0, values clamped at 255) by the apply step on every plane of base."""
    u = (np.asarray(m, np.float32) * np.asarray(W, np.float32)).astype(np.float64) * float(a)
    v = np.asarray(base, np.float64) + u
    return int(np.count_nonzero(v < 0)), int(np.count_nonzero(v > 255))


def y10_words(y):
    """The 10-bit word the WM_Y10 apply stores for an f32 output y in [0, 255]: (uint16) clamp(4 y, 0, 1023), truncating."""
    return np.minimum(np.float32(4.0) * np.asarray(y, np.float32), np.float32(1023.0)).astype(np.uint16)


def sweep_ctas(batch, ntiles, sms, split_cost=8):
    """CTAs the Rx sweep gives each image of a batch of `batch` images of `ntiles` tiles (wm_api.cu: partition, split_wave, with
    SWEEP_CTAS_PER_SM CTAs per SM).  The bits of an image's Rx depend on its pixels and this count only."""
    cap = SWEEP_CTAS_PER_SM * sms

    def wave_cost(m):
        if m >= cap:
            return -(-m // cap) * ntiles
        base = cap // m
        return 1 if base >= ntiles else -(-ntiles // base)

    def worth(split, single):
        return split * 100 < single * 92

    out, rest = [], batch
    while rest > 0:
        take = rest
        if rest > cap and rest % cap != 0:
            full = (rest // cap) * cap
            if worth(wave_cost(full) + split_cost + wave_cost(rest - full), wave_cost(rest)):
                take = full
        elif 1 < rest < cap and cap % rest != 0:
            single = best = wave_cost(rest)
            for na in range(1, rest):
                c = wave_cost(na) + split_cost + wave_cost(rest - na)
                if c < best and worth(c, single):
                    best, take = c, na
        base, extra = cap // take, cap % take
        if base < 1:
            base, extra = 1, 0
        if base >= ntiles:
            base, extra = ntiles, 0
        out += [base + (1 if i < extra else 0) for i in range(take)]
        rest -= take
    return out


def ntiles(rows, cols, layout_col_major):
    L, P = (cols, rows) if layout_col_major else (rows, cols)
    return -(-L // TL) * -(-P // 128)


def replay_batch(nblk, sms):
    """A batch size whose image 0 is swept by exactly `nblk` CTAs (one sub-batch, no image with one CTA more), or None."""
    cap = SWEEP_CTAS_PER_SM * sms
    return cap // nblk if cap % nblk == 0 else None


def rx_change_of_segment(n):
    """Relative change one missing 128-pixel line segment of average terms makes to an Rx entry of an n-pixel frame."""
    return SEGMENT / n


def a_change_of_segment(n):
    return 1 / math.sqrt(1 - SEGMENT / n) - 1
