"""CPU side of the 8-bit kernel checks at full frame sizes (test_gpu_u8_kernels_full_size.py): the oracle's apply step is exactly
clamp(RN32(u a + base), 0, 255), the byte check rejects the apply defects it is meant to catch, and every bound on a sum is tight
enough to see one 128-pixel line segment go missing or be counted twice at every frame size that file uses."""
import math
from fractions import Fraction

import numpy as np
import pytest

import u8_exact as X
import util


def _rn32(q):
    """The f32 nearest to the rational q, ties to even (no double rounding: the f64 guess is corrected exactly)."""
    x = np.float32(float(q))
    best = None
    for c in (np.nextafter(x, np.float32(-np.inf)), x, np.nextafter(x, np.float32(np.inf))):
        d = abs(Fraction(float(c)) - q)
        key = (d, int(np.array(c, np.float32).view(np.uint32)) & 1)
        if best is None or key < best[0]:
            best = (key, c)
    return np.float32(best[1])


def _exact_apply(u, a, b):
    v = _rn32(Fraction(float(u)) * Fraction(float(a)) + Fraction(float(b)))
    return np.float32(min(max(v, np.float32(0)), np.float32(255)))


def test_apply_is_an_exact_fused_multiply_add(oracle):
    """oracle.apply against exact rational arithmetic on seeded (u, a, base) triples, a third of them placed so that u a + base lies
    within an ulp or two of an integer, of 0 or of 255: where a rounding or truncation mistake would change the output byte."""
    rng = np.random.default_rng(2024)
    n = 10000
    a = rng.uniform(0.5, 60.0, n).astype(np.float32)
    b = rng.integers(0, 256, n).astype(np.float32)
    u = rng.standard_normal(n).astype(np.float32) * np.float32(3)
    near = rng.random(n) < 1 / 3
    tgt = np.where(rng.random(n) < 0.5, rng.integers(0, 256, n), rng.choice([0, 255], n)).astype(np.float64)
    for i in np.flatnonzero(near):  # u = (target - base) / a, then a few ulps either way
        x = np.float32((tgt[i] - b[i]) / a[i])
        for _ in range(int(rng.integers(-2, 3))):
            x = np.nextafter(x, np.float32(np.inf if rng.random() < 0.5 else -np.inf))
        u[i] = x
    got = np.array([oracle.apply(b[i:i + 1], u[i:i + 1], float(a[i]))[0] for i in range(n)], np.float32)
    want = np.array([_exact_apply(u[i], a[i], b[i]) for i in range(n)], np.float32)
    bad = np.flatnonzero(got.view(np.uint32) != want.view(np.uint32))
    assert bad.size == 0, [(float(u[i]), float(a[i]), float(b[i]), float(got[i]), float(want[i])) for i in bad[:5]]
    # the near-integer triples do land within an ulp of an integer, and the clamps fire at both ends
    exact = np.array([float(Fraction(float(u[i])) * Fraction(float(a[i])) + Fraction(float(b[i]))) for i in np.flatnonzero(near)])
    assert np.count_nonzero(np.abs(exact - np.rint(exact)) <= np.spacing(np.float32(np.maximum(np.abs(exact), 1)))) > 1000
    assert np.count_nonzero(want == 0) > 100 and np.count_nonzero(want == 255) > 100


def test_apply_is_the_embed_step(oracle):
    """oracle.apply with embed()'s own u and a gives embed()'s output, bit for bit."""
    img = X.frame(96, 160, seed=5).astype(np.float32)
    W = util.normal_w(96, 160)
    for mask in (oracle.ME, oracle.NVF):
        o = oracle.embed(img, W, 40.0, mask)
        assert o["status"] == 0
        assert np.array_equal(oracle.apply(img, o["u"], o["a"]).view(np.uint32), o["out"].view(np.uint32))


def test_byte_check_rejects_the_apply_defects(oracle):
    """The reference frame of the byte check against four wrong apply kernels: rounding to nearest instead of truncating, a clamp at
    254, one group of 4 pixels read one column off, one 128-pixel line segment left at its input value.  Each must be rejected."""
    rows, cols = 96, 256
    img = X.frame(rows, cols, seed=9)
    W = util.normal_w(rows, cols)
    pe = oracle.pred_error_mask(img.astype(np.float32))
    a = oracle.embed(img.astype(np.float32), W, 40.0, oracle.ME)["a"]
    v, ref = X.apply_ref(oracle, img, pe["mask"], W, a)
    lo, hi = X.clamps_fired(img, pe["mask"], W, a)
    assert lo > 0 and hi > 0
    assert X.unequal_bytes(ref, ref) == 0
    # the reference is the oracle's own u8 frame path
    assert X.unequal_bytes(ref, oracle.embed_frame_u8(img, W, 40.0, oracle.ME)[1]) == 0
    rounded = np.floor(v.astype(np.float64) + 0.5).astype(np.uint8)
    clamp254 = np.minimum(ref, 254)
    shifted = ref.copy()
    shifted[40, 64:68] = ref[40, 65:69]
    stale = ref.copy()
    stale[57, 128:256] = img[57, 128:256]
    for name, bad in (("round", rounded), ("clamp254", clamp254), ("shifted group", shifted), ("stale segment", stale)):
        assert X.unequal_bytes(bad, ref) > 0, name


@pytest.mark.parametrize("rows,cols,ls", X.SIZES)
def test_bounds_resolve_one_line_segment(rows, cols, ls):
    """Each bound on a, sum2, |e_z|^2 and |e_u|^2 must stay below half the change that dropping one 128-pixel line segment of average
    energy makes to the f64 reference: otherwise a kernel that skipped a segment, or counted one twice, could pass."""
    n = rows * cols
    s_ref = float(n)  # unit energy per pixel: the ratios below do not depend on the scale
    seg = s_ref * X.SEGMENT / n
    k = X.chain_len(128)  # the longest chain any path takes (the narrow u8 kernels)
    assert k >= X.chain_len(256)
    bound = X.sum_rel_bound(k, n) * s_ref  # sum2, |e_z|^2 and |e_u|^2 alike: sums of squares
    assert bound < 0.5 * seg, (rows, cols, bound, seg)
    # a = strength sqrt(N) / |u|: a segment less moves it by 1 / sqrt(1 - 128 / N) - 1
    da = 1 / math.sqrt(1 - X.SEGMENT / n) - 1
    assert X.a_rel_bound(k, n) < 0.5 * da, (rows, cols, X.a_rel_bound(k, n), da)


def test_chain_lengths_follow_the_tile_shape():
    assert X.chain_len(128) == 32 and X.chain_len(256) == 16
