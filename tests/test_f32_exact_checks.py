"""CPU side of the f32 kernel checks at full frame sizes (test_gpu_f32_kernels_full_size.py): the oracle's rx_f64 mode is the sum it
claims to be, the Rx bound holds for simulated HMMA (truncating) and FHADD (round-to-nearest) accumulators, the bounds resolve one
missing 128-pixel line segment where the file relies on them for that, and the f32 output check rejects the apply defects it targets."""
import numpy as np
import pytest

import f32_exact as X
import util

DY = [-1, -1, -1, 0, 0, 1, 1, 1]
DX = [-1, 0, 1, -1, 1, -1, 0, 1]


def _rx_numpy(img, fp16):
    """Rx, rx restated in numpy: the 8 neighbours of every pixel clamped to the edge, each term RN16(RN32(x y)) or the exact x y, all
    added in f64."""
    img = np.asarray(img, np.float32)
    rows, cols = img.shape
    rr, cc = np.arange(rows)[:, None], np.arange(cols)[None, :]
    nb = [img[np.clip(rr + dy, 0, rows - 1), np.clip(cc + dx, 0, cols - 1)] for dy, dx in zip(DY, DX)]

    def term(a, b):
        if fp16:
            return (a * b).astype(np.float16).astype(np.float64)
        return a.astype(np.float64) * b.astype(np.float64)

    rx = np.array([term(nb[k], img).sum() for k in range(8)])
    Rx = np.array([[term(nb[i], nb[j]).sum() for j in range(8)] for i in range(8)])
    return Rx, rx


@pytest.mark.parametrize("rows,cols", [(1, 1), (2, 3), (5, 7), (31, 67), (67, 131)])
@pytest.mark.parametrize("fp16", [1, 0])
def test_rx_f64_matches_a_numpy_restatement(oracle, rows, cols, fp16):
    img = util.natural_image(rows, cols, seed=rows + cols)
    Rx, rx = oracle.rx(img, oracle.opts(fp16_products=fp16, rx_f64=1))
    nRx, nrx = _rx_numpy(img, fp16)
    # the same terms, added in another order in f64: equal to within a few units of the last place of the f64 sum
    tol = 8 * img.size * X.U64
    assert np.all(np.abs(Rx - nRx) <= tol * np.abs(nRx)), np.abs(Rx / nRx - 1).max()
    assert np.all(np.abs(rx - nrx) <= tol * np.abs(nrx)), np.abs(rx / nrx - 1).max()
    assert np.array_equal(Rx, Rx.T)


@pytest.mark.parametrize("rows,cols", [(64, 64), (67, 131), (130, 264), (512, 512)])
def test_rx_f64_equals_faithful_on_integer_pixels(oracle, rows, cols):
    """Integer-valued pixels: every term is an integer and every partial sum of either mode is exact, so the bits are equal."""
    img = np.rint(util.natural_image(rows, cols, seed=7)).astype(np.float32)
    for fp16, o in ((1, oracle.FAITHFUL), (0, oracle.EXACT)):
        a = oracle.rx(img, o)
        b = oracle.rx(img, oracle.opts(fp16_products=fp16, rx_f64=1))
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_rx_f64_leaves_the_other_modes_alone(oracle):
    """The new field defaults to 0: EXACT still rounds products of real-valued pixels to f32 and sums groups of 64 in f32, which
    differs from the f64 sum of the exact products.  (The fp16-rounded products of these pixels are coarse enough that FAITHFUL's f32
    group sums are mostly exact.)"""
    img = util.natural_image(96, 160, seed=3)
    assert oracle.FAITHFUL.rx_f64 == 0 and oracle.EXACT.rx_f64 == 0
    assert not np.array_equal(oracle.rx(img, oracle.EXACT)[0], oracle.rx(img, oracle.opts(fp16_products=0, rx_f64=1))[0])


# ---------------------------------------------------------------------------------------------------
# the Rx bound against simulated accumulators
# ---------------------------------------------------------------------------------------------------
def _trunc24(x):
    """x >= 0 truncated to a 24-bit significand."""
    x = np.asarray(x, np.float64)
    e = np.floor(np.log2(np.where(x > 0, x, 1.0)))
    q = 2.0 ** (e - 23)
    return np.where(x > 0, np.floor(x / q) * q, 0.0)


def _hmma_step(c, t1, t2):
    """One mma.sync step of the model in f32_exact.U_MMA: align c, t1, t2 (>= 0) to the largest with 24 bits, dropping the bits shifted
    out, add exactly, truncate the sum to 24 bits.  Every value here is a multiple of 2^(E-23) below 2^(E+3): exact in f64."""
    m = np.maximum(np.maximum(c, t1), t2)
    e = np.floor(np.log2(np.where(m > 0, m, 1.0)))
    q = 2.0 ** (e - 23)
    s = np.floor(c / q) * q + np.floor(t1 / q) * q + np.floor(t2 / q) * q
    return _trunc24(s)


def _tile_terms(rng, chains, k):
    """k fp16-rounded products per chain of real-valued pixels in [0, 255], some near 0 and some near 255."""
    x = rng.uniform(0, 255, (chains, k, 2)).astype(np.float32)
    x[: chains // 4] *= np.float32(0.01)
    y = rng.uniform(0, 255, (chains, k, 2)).astype(np.float32)
    return (x * y).astype(np.float16).astype(np.float64)


def test_rx_bound_holds_for_a_truncating_hmma_chain():
    rng = np.random.default_rng(11)
    steps = X.sweep_chains("hmma")[0][0]
    t = _tile_terms(rng, 4000, steps)
    c = np.zeros(t.shape[0])
    for s in range(steps):
        c = _hmma_step(c, t[:, s, 0], t[:, s, 1])
    exact = t.sum(axis=(1, 2))
    err = np.abs(c - exact) / exact
    bound = X.gamma(steps, X.U_MMA)
    assert np.all(c <= exact) and err.max() <= bound, (err.max(), bound)
    # the model does lose bits (always downwards), but typical chains stay far inside the worst case
    assert np.count_nonzero(c < exact) > t.shape[0] // 2
    assert X.rx_rel_bound("hmma", 1) >= bound


def test_rx_bound_holds_for_a_round_to_nearest_chain():
    rng = np.random.default_rng(12)
    steps = X.sweep_chains("fhadd")[0][0] - 1  # terms per accumulator, then e0 + e1
    t = _tile_terms(rng, 4000, steps)
    e = np.zeros((t.shape[0], 2), np.float32)
    for s in range(steps):
        e = (e + t[:, s, :].astype(np.float32)).astype(np.float32)  # add.rn.f32.f16: the fp16 value is exact in f32
    c = (e[:, 0] + e[:, 1]).astype(np.float32).astype(np.float64)
    exact = t.sum(axis=(1, 2))
    err = np.abs(c - exact) / exact
    assert err.max() <= X.gamma(steps + 1, X.U32), err.max()
    assert X.rx_rel_bound("fhadd", 1) >= X.gamma(steps + 1, X.U32)


def test_chain_lengths_follow_the_kernel_source():
    assert (X.SNT, X.SLPT, X.FLUSH, X.RING) == (128, 8, 4, 64)
    assert X.sweep_chains("hmma")[0] == (64, X.U_MMA) and X.sweep_chains("fhadd")[0] == (65, X.U32)
    assert X.sweep_chains("fused")[0] == (16, X.U_MMA)
    assert X.chain_len(256) == 16  # f32 stats and detector CTAs


# ---------------------------------------------------------------------------------------------------
# the bounds against one missing 128-pixel line segment
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rows,cols,ld", X.SIZES)
def test_bounds_resolve_one_line_segment(rows, cols, ld):
    """The detector, stats and `a` bounds stay below half the change one missing segment of average terms makes at every size of the
    GPU file; the Rx bound does under FHADD / FFMA / the fused kernel at every size, under HMMA up to rx_size_limit (2.8 Mpx: 1080p
    yes, 4K no).  Above that size the exact check on integer-valued pixels is the one that sees a missing tile line."""
    n = rows * cols
    seg = X.rx_change_of_segment(n)
    k = X.chain_len(256)
    assert X.sum_rel_bound(k, n) < 0.5 * seg and X.a_rel_bound(k, n) < 0.5 * X.a_change_of_segment(n)
    for mode in ("fhadd", "ffma", "fused"):
        assert X.rx_rel_bound(mode, n) < 0.5 * seg, mode
    assert (X.rx_rel_bound("hmma", n) < 0.5 * seg) == (n <= X.rx_size_limit("hmma"))


def test_hmma_rx_bound_stops_resolving_a_segment_between_1080p_and_4k():
    assert 1080 * 1920 < X.rx_size_limit("hmma") < 2160 * 3840
    assert X.rx_rel_bound("hmma", 1080 * 1920) < 0.5 * X.rx_change_of_segment(1080 * 1920)


# ---------------------------------------------------------------------------------------------------
# the f32 output check against wrong apply kernels
# ---------------------------------------------------------------------------------------------------
def test_output_check_rejects_the_apply_defects(oracle):
    """The reference output (u8_exact.apply_ref on the mask plane and `a`) against four wrong apply kernels: the multiply-add rounded
    twice, a clamp at 254.99, u computed as mask (W a), and the prediction with two neighbour coefficients swapped (the transposed
    layout's neighbour order mixed up).  Each must change some output bits."""
    rows, cols = 96, 256
    f = X.frame(rows, cols, seed=9)
    W = util.normal_w(rows, cols)
    c = oracle.pred_error_mask(f)["coef"]
    m = X.mask_plane(oracle, f, c, oracle.ME)
    a = oracle.embed(f, W, 40.0, oracle.ME)["a"]
    ref, _ = X.apply_ref(oracle, f, m, W, a)
    lo, hi = X.clamps(f, m, W, a)
    assert lo > 0 and hi > 0
    assert np.array_equal(ref.view(np.uint32), oracle.embed(f, W, 40.0, oracle.ME)["out"].view(np.uint32))
    u = m * W
    a32 = np.float32(a)
    unfused = np.clip(f + u * a32, 0, 255).astype(np.float32)
    clamp_low = np.minimum(ref, np.float32(254.99))
    wa = np.clip(f + m * (W * a32), 0, 255).astype(np.float32)
    cs = c.copy()
    cs[[1, 3]] = cs[[3, 1]]
    swapped, _ = X.apply_ref(oracle, f, X.mask_plane(oracle, f, cs, oracle.ME), W, a)
    assert X.unequal(ref, ref) == 0
    for name, bad in (("unfused", unfused), ("clamp 254.99", clamp_low), ("mask (W a)", wa), ("swapped coefficients", swapped)):
        assert X.unequal(bad.astype(np.float32), ref) > 0, name


def test_frames_are_real_valued_and_clamp_at_both_ends(oracle):
    f = X.frame(130, 264, seed=31)
    assert np.count_nonzero(f != np.rint(f)) > 0.99 * f.size
    W = util.normal_w(130, 264)
    o = oracle.embed(f, W, 40.0, oracle.NVF)
    lo, hi = X.clamps(f, o["mask"], W, o["a"])
    assert lo > 0 and hi > 0


def test_y10_words_truncate(oracle):
    y = np.array([0.0, 0.2499, 0.25, 100.1, 254.999, 255.0], np.float32)
    assert X.y10_words(y).tolist() == [0, 0, 1, 400, 1019, 1020]
