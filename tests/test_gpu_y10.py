"""10-bit luma planes (WM_Y10: the sample in bits 0-9 of a little-endian word; WM_Y10_MSB: in bits 6-15) through the embed and detect
entry points, the host forms, the video driver and the C++ façade.

The reference is the f32 path on the 8-bit-equivalent scale: wm_embed_batch / wm_detect_batch on a dense f32 plane holding x = v * 0.25
(base = in, f32 out), with the same batch.  `a`, the correlation and the statuses must be that run's, bit for bit, and the output words
np.clip(4 * y, 0, 1023).astype(np.uint16) << shift of its f32 output y.  The ignored bits of the input words are seeded random.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import util
from test_gpu_packed_rgb import dev_get, dev_raw, f32bits
from test_gpu_packed_video import check, references, run_driver

pytestmark = pytest.mark.gpu

PSNR = 40.0
SHAPES = [(1080, 1920), (121, 203), (600, 27)]  # full HD; cols % 4 != 0 (plain loaders); tall and thin


def layouts(wmb):
    return [wmb.Y10, wmb.Y10_MSB]


def shift_of(wmb, layout):
    return {wmb.Y10: 0, wmb.Y10_MSB: 6}[layout]


def ignored_mask(wmb, layout):
    return 0xFC00 if layout == wmb.Y10 else 0x003F


def samples(rows, cols, seed=0):
    """10-bit samples (0..1023) with natural statistics: a natural 8-bit image scaled by 4 plus seeded noise of a few codes"""
    rng = np.random.default_rng(300 + seed)
    v = util.natural_image(rows, cols, seed=seed) * 4.0 + rng.integers(-2, 3, (rows, cols))
    v = np.clip(np.rint(v), 0, 1023).astype(np.uint16)
    v[0, 0], v[-1, -1] = 0, 1023
    return v


def words(wmb, v, layout, junk_seed=None):
    """the words of samples v in `layout`; junk_seed: the ignored bits are seeded random instead of zero"""
    w = (v.astype(np.uint16) << shift_of(wmb, layout)).astype(np.uint16)
    if junk_seed is not None:
        junk = np.random.default_rng(junk_seed).integers(0, 1 << 16, v.shape, dtype=np.uint16)
        w |= junk & np.uint16(ignored_mask(wmb, layout))
    return w


def quantise(wmb, y, layout):
    return (np.clip(4.0 * y.astype(np.float32), 0, 1023).astype(np.uint16) << shift_of(wmb, layout)).astype(np.uint16)


def sample_of(wmb, w, layout):
    return ((w >> shift_of(wmb, layout)) & 0x3FF).astype(np.uint16)


def x_of(v):
    return v.astype(np.float32) * np.float32(0.25)


def f32_path(wmb, wm, x, mask):
    """wm_embed_batch (base = in, f32 out) on dense f32 planes x (batch, rows, cols), then wm_detect_batch on x itself
    -> (y, a, status, corr of x, detect status)"""
    batch, rows, cols = x.shape
    pin, pout = dev_raw(wmb, wm, np.ascontiguousarray(x, np.float32)), dev_raw(wmb, wm, np.zeros(x.shape, np.float32))
    desc = lambda p: wmb.image_desc(p, rows, cols, wmb.ROW_MAJOR, wmb.F32, 0, 1)
    a, st = np.full(batch, np.nan, np.float32), np.zeros(batch, np.int32)
    corr, st2 = np.zeros(batch, np.float32), np.zeros(batch, np.int32)
    wm.embed_batch(0, desc(pin), desc(pin), desc(pout), 0, 0, 0, batch, mask, a, st)
    wm.detect_batch(0, desc(pin), 0, batch, mask, corr, st2)
    wm.sync(0)
    y = dev_get(wmb, wm, pout, (batch, rows, cols * 4)).view(np.float32)
    for p in (pin, pout):
        wmb.lib().wm_dev_free(wm._h, p)
    return y, a, st, corr, st2


def f32_detect(wmb, wm, x, mask):
    batch, rows, cols = x.shape
    p = dev_raw(wmb, wm, np.ascontiguousarray(x, np.float32))
    corr, st = np.zeros(batch, np.float32), np.zeros(batch, np.int32)
    wm.detect_batch(0, wmb.image_desc(p, rows, cols, wmb.ROW_MAJOR, wmb.F32, 0, 1), 0, batch, mask, corr, st)
    wm.sync(0)
    wmb.lib().wm_dev_free(wm._h, p)
    return corr, st


def y10_path(wmb, wm, w, layout, mask, ld=0, stride=0):
    """wm_embed_batch (base = in) and wm_detect_batch on the input and on the output, words w (batch, rows, cols) placed at a row pitch of
    `ld` bytes and a batch stride of `stride` bytes -> (out words, a, status, corr of in, detect status, corr of out, detect status)"""
    batch, rows, cols = w.shape
    ldb = ld or 2 * cols
    sb = stride or rows * ldb
    buf = np.zeros(batch * sb, np.uint8)
    for b in range(batch):
        buf[b * sb:b * sb + rows * ldb].reshape(rows, ldb)[:, :2 * cols] = w[b].astype("<u2").view(np.uint8).reshape(rows, 2 * cols)
    pin, pout = dev_raw(wmb, wm, buf), dev_raw(wmb, wm, np.full(buf.shape, 0xA5, np.uint8))
    desc = lambda p: wmb.image_desc(p, rows, cols, layout, wmb.U8, ld, 2)
    a, st = np.full(batch, np.nan, np.float32), np.zeros(batch, np.int32)
    ci, sti, co, sto = np.zeros(batch, np.float32), np.zeros(batch, np.int32), np.zeros(batch, np.float32), np.zeros(batch, np.int32)
    wm.embed_batch(0, desc(pin), desc(pin), desc(pout), stride, stride, stride, batch, mask, a, st)
    wm.detect_batch(0, desc(pin), stride, batch, mask, ci, sti)
    wm.detect_batch(0, desc(pout), stride, batch, mask, co, sto)
    wm.sync(0)
    ob = dev_get(wmb, wm, pout, buf.shape)
    assert np.array_equal(dev_get(wmb, wm, pin, buf.shape), buf)  # the input is only read
    for p in (pin, pout):
        wmb.lib().wm_dev_free(wm._h, p)
    out = np.empty(w.shape, np.uint16)
    written = np.zeros(buf.shape, bool)
    for b in range(batch):
        rowsb = ob[b * sb:b * sb + rows * ldb].reshape(rows, ldb)
        out[b] = np.ascontiguousarray(rowsb[:, :2 * cols]).view("<u2")
        written[b * sb:b * sb + rows * ldb].reshape(rows, ldb)[:, :2 * cols] = True
    assert np.all(ob[~written] == 0xA5)  # row padding and the gaps between images are not written
    return out, a, st, ci, sti, co, sto


def wm_for(wmb, rows, cols, p, W=None):
    return wmb.Watermark(rows, cols, util.normal_w(rows, cols) if W is None else W, p, PSNR)


CASES = [("ME", 3), ("NVF", 3), ("NVF", 5)]


def assert_equal_to_f32(wmb, wm, v, w, layout, mask, ld=0, stride=0, what=""):
    """the 10-bit path on words w (batch, rows, cols) against the f32 path on x = v / 4"""
    out, a, st, ci, sti, co, sto = y10_path(wmb, wm, w, layout, mask, ld, stride)
    y, ra, rst, rci, rsti = f32_path(wmb, wm, x_of(v), mask)
    q = quantise(wmb, y, layout)
    rco, rsto = f32_detect(wmb, wm, x_of(sample_of(wmb, q, layout)), mask)
    print("%s: a=%r corr(in)=%r corr(out)=%r differing words=%d" % (what, a[0], ci[0], co[0], int(np.count_nonzero(out != q))))
    assert np.array_equal(st, rst) and np.array_equal(sti, rsti) and np.array_equal(sto, rsto), what
    assert np.array_equal(a.view(np.uint32), ra.view(np.uint32)), what
    assert np.array_equal(ci.view(np.uint32), rci.view(np.uint32)), what
    assert np.array_equal(co.view(np.uint32), rco.view(np.uint32)), what
    assert np.array_equal(out, q), what
    assert np.all(out & np.uint16(ignored_mask(wmb, layout)) == 0), what
    return out, a


# ---- 1. bit equality with the f32 path on x = v / 4 ----
@pytest.mark.parametrize("rows,cols", SHAPES)
def test_equal_to_f32_path(wmb, rows, cols):
    v = samples(rows, cols, seed=rows + cols)
    for name, p in CASES:
        wm = wm_for(wmb, rows, cols, p)
        mask = wmb.ME if name == "ME" else wmb.NVF
        for layout in layouts(wmb):
            w = words(wmb, v, layout, junk_seed=rows)
            assert_equal_to_f32(wmb, wm, v[None], w[None], layout, mask, what="%dx%d %s p=%d layout=%d" % (rows, cols, name, p, layout))
        wm.close()


@pytest.mark.parametrize("rows,cols", [(1080, 1920), (121, 203)])
def test_padded_rows_and_strided_batch(wmb, rows, cols):
    """rows at a pitch of 2 * cols + 64 bytes; a batch of 3 with a byte stride larger than one image (and not a multiple of 16)"""
    vs = np.stack([samples(rows, cols, seed=40 + b) for b in range(3)])
    ld = 2 * cols + 64
    for name, p in CASES:
        wm = wm_for(wmb, rows, cols, p)
        mask = wmb.ME if name == "ME" else wmb.NVF
        for layout in layouts(wmb):
            w = np.stack([words(wmb, vs[b], layout, junk_seed=b) for b in range(3)])
            what = "%dx%d %s p=%d layout=%d" % (rows, cols, name, p, layout)
            assert_equal_to_f32(wmb, wm, vs[:1], w[:1], layout, mask, ld=ld, what="ld+64 " + what)
            assert_equal_to_f32(wmb, wm, vs, w, layout, mask, ld=ld, stride=rows * ld + 34, what="batch 3 " + what)
        wm.close()


# ---- 2. ignored bits ----
@pytest.mark.parametrize("rows,cols", [(270, 480), (121, 203)])
def test_ignored_bits(wmb, rows, cols):
    v = samples(rows, cols, seed=2)
    wm = wm_for(wmb, rows, cols, 3)
    for layout in layouts(wmb):
        for mask in (wmb.ME, wmb.NVF):
            clean = y10_path(wmb, wm, words(wmb, v, layout)[None], layout, mask)
            noisy = y10_path(wmb, wm, words(wmb, v, layout, junk_seed=9)[None], layout, mask)
            assert np.array_equal(clean[0], noisy[0]), (layout, mask)
            assert np.all(noisy[0] & np.uint16(ignored_mask(wmb, layout)) == 0)
            for k in range(1, 7):
                assert np.array_equal(np.asarray(clean[k]).view(np.uint32), np.asarray(noisy[k]).view(np.uint32)), (layout, mask, k)
    wm.close()


# ---- 3. against the CPU oracle at 1080p on x ----
def test_against_oracle(wmb, oracle):
    rows, cols = 1080, 1920
    v = samples(rows, cols, seed=5)
    x = x_of(v)
    W = util.normal_w(rows, cols)
    wm = wm_for(wmb, rows, cols, 3, W)
    for mask in (wmb.ME, wmb.NVF):
        o = oracle.embed(x, W, PSNR, mask)
        for layout in layouts(wmb):
            out, a, st, ci, sti, co, sto = y10_path(wmb, wm, words(wmb, v, layout, junk_seed=5)[None], layout, mask)
            ref_words = np.clip(4.0 * np.asarray(o["out"], np.float64), 0, 1023).astype(np.int64) << shift_of(wmb, layout)
            dw = int(np.abs(out[0].astype(np.int64) - ref_words).max())
            od = oracle.detect(x_of(sample_of(wmb, out[0], layout)), W, mask)
            di = oracle.detect(x, W, mask)
            ra, rc, ri = util.rel(a[0], o["a"]), util.rel(co[0], od["corr"]), util.rel(ci[0], di["corr"])
            print("oracle mask=%d layout=%d: a rel %.3g corr(out) rel %.3g corr(in) rel %.3g max word diff %d" % (mask, layout, ra, rc, ri, dw))
            assert st[0] == 0 and sto[0] == 0 and sti[0] == 0
            assert ra <= 1e-3 and rc <= 1e-3 and ri <= 1e-3
            assert dw <= 1 << shift_of(wmb, layout)
    wm.close()


# ---- 4. singular and zero-mask cases: out = every input word ----
def test_singular_and_zero_mask(wmb):
    rows, cols = 270, 480
    wm = wm_for(wmb, rows, cols, 3)
    wz = wm_for(wmb, rows, cols, 3, np.zeros((rows, cols), np.float32))  # W = 0: mask.W is exactly 0
    flat = np.full((rows, cols), 469, np.uint16)  # constant image: the ME system is unsolvable
    v = samples(rows, cols, seed=8)
    for layout in layouts(wmb):
        w = words(wmb, flat, layout, junk_seed=1)[None]
        out, a, st, ci, sti, co, sto = y10_path(wmb, wm, w, layout, wmb.ME)
        assert st[0] == wmb.SINGULAR and np.isnan(a[0]) and np.array_equal(out, w) and sti[0] == wmb.SINGULAR
        _, ra, rst, _, rsti = f32_path(wmb, wm, x_of(flat)[None], wmb.ME)
        assert (rst[0], rsti[0]) == (st[0], sti[0]) and np.isnan(ra[0])
        w = words(wmb, v, layout, junk_seed=2)[None]
        for mask in (wmb.ME, wmb.NVF):
            out, a, st, ci, sti, co, sto = y10_path(wmb, wz, w, layout, mask)
            assert st[0] == wmb.ZERO_MASK and np.isinf(a[0]) and np.array_equal(out, w), (layout, mask, st[0])
            y, ra, rst, _, _ = f32_path(wmb, wz, x_of(v)[None], mask)
            assert rst[0] == st[0] and f32bits(a[0]) == f32bits(ra[0])
    wz.close()
    wm.close()


# ---- 5. rows ending at the allocation end: the conversion reads nothing past 2 * cols bytes of a row ----
@pytest.mark.parametrize("cols,extra", [(200, 0), (203, 0), (121, 2), (130, 6), (1366, 0)])
def test_rows_ending_at_the_allocation_end(wmb, cols, extra):
    rows = 67
    ld = 2 * cols + extra
    v = samples(rows, cols, seed=cols)
    wm = wm_for(wmb, rows, cols, 3)
    L = wmb.lib()
    for layout in layouts(wmb):
        w = words(wmb, v, layout, junk_seed=cols)
        wb = w.astype("<u2").view(np.uint8).reshape(rows, 2 * cols)
        buf = np.zeros((rows - 1) * ld + 2 * cols, np.uint8)  # the last row ends at the last byte
        buf[:(rows - 1) * ld].reshape(rows - 1, ld)[:, :2 * cols] = wb[:-1]
        buf[(rows - 1) * ld:] = wb[-1]
        for mask in (wmb.ME, wmb.NVF):
            y, ra, rst, rci, _ = f32_path(wmb, wm, x_of(v)[None], mask)
            pin, pout = dev_raw(wmb, wm, buf), dev_raw(wmb, wm, np.zeros_like(buf))
            desc = lambda p: wmb.image_desc(p, rows, cols, layout, wmb.U8, ld, 2)
            a, st, corr, st2 = np.full(1, np.nan, np.float32), np.zeros(1, np.int32), np.zeros(1, np.float32), np.zeros(1, np.int32)
            wm.embed_batch(0, desc(pin), desc(pin), desc(pout), 0, 0, 0, 1, mask, a, st)
            wm.detect_batch(0, desc(pin), 0, 1, mask, corr, st2)
            wm.sync(0)
            o = dev_get(wmb, wm, pout, buf.shape)
            for p in (pin, pout):
                L.wm_dev_free(wm._h, p)
            got = np.empty((rows, 2 * cols), np.uint8)
            got[:-1] = o[:(rows - 1) * ld].reshape(rows - 1, ld)[:, :2 * cols]
            got[-1] = o[(rows - 1) * ld:]
            assert np.array_equal(np.ascontiguousarray(got).view("<u2"), quantise(wmb, y[0], layout)), (cols, extra, layout, mask)
            assert st[0] == rst[0] and f32bits(a[0]) == f32bits(ra[0]) and f32bits(corr[0]) == f32bits(rci[0])
    wm.close()


# ---- 6. host forms equal the device forms ----
def test_host_forms_equal_device_forms(wmb):
    rows, cols, batch = 121, 203, 3
    wm = wm_for(wmb, rows, cols, 3)
    L = wmb.lib()
    vs = np.stack([samples(rows, cols, seed=60 + b) for b in range(batch)])
    for layout in layouts(wmb):
        w = np.stack([words(wmb, vs[b], layout, junk_seed=60 + b) for b in range(batch)])
        for mask in (wmb.ME, wmb.NVF):
            refs = [y10_path(wmb, wm, w[b:b + 1], layout, mask) for b in range(batch)]
            # single images, rows of a pitched host buffer (2 * cols + 64 bytes)
            big = np.zeros((rows, cols + 32), np.uint16)
            big[:, :cols] = w[0]
            out = np.zeros((rows, cols + 32), np.uint16)
            a, st = wm.make_watermark_host(big[:, :cols], None, out[:, :cols], mask, layout=layout)
            corr, st2 = wm.detect_watermark_host(big[:, :cols], mask, layout=layout)
            assert np.array_equal(out[:, :cols], refs[0][0][0]) and np.all(out[:, cols:] == 0)
            assert f32bits(a) == f32bits(refs[0][1][0]) and st == refs[0][2][0]
            assert f32bits(corr) == f32bits(refs[0][3][0]) and st2 == refs[0][4][0]
            # batches in pinned memory
            nb = rows * 2 * cols
            hp = [L.wm_host_alloc_pinned(batch * nb) for _ in range(2)]
            hin, hout = [np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint16)), (batch, rows, cols)) for p in hp]
            hin[:] = w
            desc = lambda p: wmb.image_desc(p, rows, cols, layout, wmb.U8, 0, 2)
            a, st, corr, st2 = (np.full(batch, np.nan, np.float32), np.zeros(batch, np.int32), np.zeros(batch, np.float32), np.zeros(batch, np.int32))
            wm.embed_host_batch(1, desc(hp[0]), desc(hp[0]), desc(hp[1]), 0, 0, 0, batch, mask, a, st)
            wm.sync(1)
            for b in range(batch):
                assert np.array_equal(hout[b], refs[b][0][0]) and f32bits(a[b]) == f32bits(refs[b][1][0]) and st[b] == refs[b][2][0]
            hout[:] = 0
            a[:] = np.nan
            wm.embed_verify_host_batch(2, desc(hp[0]), desc(hp[0]), desc(hp[1]), 0, 0, 0, batch, mask, a, corr, st)
            wm.sync(2)
            for b in range(batch):
                assert np.array_equal(hout[b], refs[b][0][0]) and st[b] == refs[b][2][0] and f32bits(a[b]) == f32bits(refs[b][1][0])
                # the verify detects on x' = v' / 4 of the written words
                rc, _ = f32_detect(wmb, wm, x_of(sample_of(wmb, refs[b][0], layout)), mask)
                assert f32bits(corr[b]) == f32bits(rc[0]) == f32bits(refs[b][5][0])
            corr[:] = 0
            wm.detect_host_batch(3, desc(hp[0]), 0, batch, mask, corr, st2)
            wm.sync(3)
            for b in range(batch):
                assert f32bits(corr[b]) == f32bits(refs[b][3][0]) and st2[b] == refs[b][4][0]
            for p in hp:
                L.wm_host_free_pinned(p)
    wm.close()


# ---- 7. the video driver ----
# 270 x 480 frames have 36 tiles, fewer than the CTAs each image of a run of up to 8 frames gets, so a frame's partial sums are grouped
# the same way whatever run it shares: the driver's results are the per-frame wm_embed_batch / wm_detect_batch results bit for bit.
VROWS, VCOLS = 270, 480


def video_frames(wmb, layout, n, seed=0):
    """n frames of `layout` as (n, rows, cols, 2) bytes (the words, little-endian), ignored bits random"""
    f = np.stack([words(wmb, np.roll(samples(VROWS, VCOLS, seed=seed + i % 3), 11 * i, axis=1), layout, junk_seed=seed + i) for i in range(n)])
    return np.ascontiguousarray(f.astype("<u2")).view(np.uint8).reshape(n, VROWS, VCOLS, 2)


@pytest.mark.parametrize("on_device", [False, True])
def test_video_driver(wmb, on_device):
    n, first, interval = 10, 2, 3
    ls = 2 * VCOLS + 64
    wm = wm_for(wmb, VROWS, VCOLS, 3)
    for layout in layouts(wmb):
        frames = video_frames(wmb, layout, n, seed=30)
        refs = references(wmb, wm, frames, layout, first, interval)
        what = "layout=%d device=%d" % (layout, on_device)
        out, a = run_driver(wmb, wm, frames, layout, wmb.VIDEO_EMBED, interval, first, on_device, linesize=ls)
        _, corr = run_driver(wmb, wm, out, layout, wmb.VIDEO_DETECT, interval, first, on_device, linesize=ls)
        check(frames, first, interval, out, a, corr, refs, True, "embed/detect " + what)  # gated-off frames: byte-identical copies
        o2, s2 = run_driver(wmb, wm, frames, layout, wmb.VIDEO_EMBED_VERIFY, interval, first, on_device, linesize=ls)
        assert np.array_equal(o2, out), what
        check(frames, first, interval, o2, s2[:n], s2[n:], refs, True, "embed_verify " + what)
        # the driver's detection of the input frames: the f32 path's correlation of x
        _, cin = run_driver(wmb, wm, frames, layout, wmb.VIDEO_DETECT, interval, first, on_device, linesize=ls)
        for i in range(n):
            if (first + i) % interval == 0:
                wi = np.ascontiguousarray(frames[i]).view("<u2").reshape(VROWS, VCOLS)
                rc, _ = f32_detect(wmb, wm, x_of(sample_of(wmb, wi, layout))[None], wmb.ME)
                assert f32bits(cin[i]) == f32bits(rc[0]), (what, i)
    wm.close()


@pytest.mark.parametrize("on_device", [False, True])
def test_video_multi_equals_single(wmb, on_device):
    n, first, interval = 11, 1, 3
    ls = 2 * VCOLS + 64
    wm = wm_for(wmb, VROWS, VCOLS, 3)
    clones = [wm.clone(), wm.clone()]
    for layout in layouts(wmb):
        frames = video_frames(wmb, layout, n, seed=50)
        o1, a1 = run_driver(wmb, wm, frames, layout, wmb.VIDEO_EMBED, interval, first, on_device, linesize=ls)
        o2, a2 = run_driver(wmb, wm, frames, layout, wmb.VIDEO_EMBED, interval, first, on_device, linesize=ls, ctxs=clones)
        assert np.array_equal(o1, o2) and np.array_equal(a1.view(np.uint32), a2.view(np.uint32))
        _, c1 = run_driver(wmb, wm, o1, layout, wmb.VIDEO_DETECT, interval, first, on_device)
        _, c2 = run_driver(wmb, wm, o1, layout, wmb.VIDEO_DETECT, interval, first, on_device, ctxs=clones)
        assert np.array_equal(c1.view(np.uint32), c2.view(np.uint32))
    for c in clones:
        c.close()
    wm.close()


def test_video_rejections(wmb):
    rows, cols, n = 67, 131, 2
    wm = wm_for(wmb, rows, cols, 3)
    frames = np.zeros(n * rows * (2 * cols + 8) + 8, np.uint8)
    out = np.zeros_like(frames)
    scal = np.zeros(2 * n, np.float32)
    for layout in layouts(wmb):
        for ls, fstride, off in ((2 * cols - 2, 0, 0), (2 * cols + 1, 0, 0), (0, rows * 2 * cols + 1, 0), (0, 0, 1)):
            v = wmb.VideoProcessingContext(wm, rows, cols, 1, linesize=ls, frame_stride=fstride, layout=layout)
            with pytest.raises(wmb.WatermarkError) as e:
                wmb.process_frames(v, wmb.VIDEO_EMBED, frames.ctypes.data + off, out.ctypes.data, 0, n, scal)
            print("layout %d linesize %d frame_stride %d offset %d: %s" % (layout, ls, fstride, off, e.value))
            assert e.value.code == -5
    assert np.all(out == 0)
    # odd widths are taken
    v = wmb.VideoProcessingContext(wm, rows, cols, 1, layout=wmb.Y10)
    assert wmb.process_frames(v, wmb.VIDEO_EMBED, frames.ctypes.data, out.ctypes.data, 0, n, scal) == n
    wm.close()


# ---- 8. refusals ----
def test_rejections(wmb):
    rows, cols = 67, 130
    wm = wm_for(wmb, rows, cols, 3)
    L = wmb.lib()
    v = samples(rows, cols)
    d = wmb.DeviceArray.from_numpy(wm, words(wmb, v, wmb.Y10), wmb.Y10)
    assert np.array_equal(d.numpy(), words(wmb, v, wmb.Y10))
    out = wmb.DeviceArray(wm, rows, cols, wmb.Y10)
    outm = wmb.DeviceArray(wm, rows, cols, wmb.Y10_MSB)
    outy = wmb.DeviceArray(wm, rows, cols, wmb.PACKED_YUYV)
    out3 = wmb.DeviceArray(wm, rows, cols, wmb.PACKED_RGB)
    gray = wmb.DeviceArray(wm, rows, cols, wmb.ROW_MAJOR, wmb.F32, 1)
    y8 = wmb.DeviceArray(wm, rows, cols, wmb.ROW_MAJOR, wmb.U8, 1)
    big = wmb.lib().wm_dev_alloc(wm._h, 4 * rows * (2 * cols + 8))
    a = C.c_float(0)

    def desc(p, layout=wmb.Y10, dtype=wmb.U8, ld=0, ch=2):
        return wmb.image_desc(p, rows, cols, layout, dtype, ld, ch)

    def embed_rc(i, b, o):
        return L.wm_embed(wm._h, C.byref(i), C.byref(b) if b is not None else None, C.byref(o), wmb.ME, C.byref(a))

    def detect_rc(i):
        return L.wm_detect(wm._h, C.byref(i), wmb.ME, C.byref(a))

    def refused(rc, what):
        msg = L.wm_last_error(wm._h).decode()
        print("%s: %d %s" % (what, rc, msg))
        assert rc == -5 and msg, what

    for layout, o in ((wmb.Y10, out), (wmb.Y10_MSB, outm)):
        refused(embed_rc(desc(d.ptr, layout, dtype=wmb.F32), None, o.desc()), "f32 dtype %d" % layout)
        refused(embed_rc(desc(d.ptr, layout, ch=1), None, o.desc()), "1 channel %d" % layout)
        refused(detect_rc(desc(d.ptr, layout, ch=4)), "detect 4 channels %d" % layout)
        refused(detect_rc(desc(big, layout, ld=2 * cols + 1)), "odd ld %d" % layout)
        refused(embed_rc(desc(big, layout, ld=2 * cols + 1), None, desc(big + 2 * rows * (2 * cols + 8), layout)), "embed odd ld %d" % layout)
        refused(detect_rc(desc(d.ptr, layout, ld=2 * cols - 2)), "ld < 2 cols %d" % layout)
        refused(detect_rc(desc(big + 1, layout)), "misaligned pointer %d" % layout)
        refused(embed_rc(desc(d.ptr, layout), None, desc(big + 2 * rows * (2 * cols + 8) + 1, layout)), "misaligned out %d" % layout)
        corr, st = np.zeros(2, np.float32), np.zeros(2, np.int32)
        refused(L.wm_detect_batch(wm._h, 0, C.byref(desc(big, layout)), rows * 2 * cols + 1, 2, wmb.ME,
                                  corr.ctypes.data_as(C.POINTER(C.c_float)), st.ctypes.data_as(C.POINTER(C.c_int))), "odd batch stride %d" % layout)
        refused(L.wm_rgb2gray(wm._h, C.byref(desc(d.ptr, layout)), C.byref(gray.desc()), 0.299, 0.587, 0.114), "rgb2gray %d" % layout)
        refused(L.wm_debug_plane(wm._h, C.byref(desc(d.ptr, layout)), wmb.DBG_ERRSEQ, gray.ptr), "debug_plane %d" % layout)
        refused(L.wm_debug_detect_planes(wm._h, C.byref(desc(d.ptr, layout)), wmb.ME, gray.ptr, gray.ptr, C.byref(a)), "debug_detect_planes %d" % layout)
    refused(embed_rc(d.desc(), None, outm.desc()), "Y10 in, Y10_MSB out")
    refused(embed_rc(desc(d.ptr, wmb.Y10_MSB), None, out.desc()), "Y10_MSB in, Y10 out")
    refused(embed_rc(d.desc(), desc(d.ptr, wmb.Y10_MSB), out.desc()), "Y10 in, Y10_MSB base (same pointer)")
    refused(embed_rc(d.desc(), None, outy.desc()), "Y10 in, YUYV out")
    refused(embed_rc(desc(d.ptr, wmb.PACKED_YUYV), None, out.desc()), "YUYV in, Y10 out")
    refused(embed_rc(d.desc(), None, out3.desc()), "Y10 in, RGB out")
    refused(embed_rc(d.desc(), y8.desc(), out.desc()), "Y-plane base")
    refused(embed_rc(d.desc(), None, y8.desc()), "Y-plane out")
    refused(embed_rc(d.desc(), None, gray.desc()), "gray out")
    refused(embed_rc(y8.desc(), None, out.desc()), "Y-plane input, Y10 out")
    refused(embed_rc(gray.desc(), d.desc(), gray.desc()), "gray input, Y10 base")
    refused(embed_rc(d.desc(), None, desc(d.ptr + 2)), "out overlaps in")
    # host forms
    h = words(wmb, v, wmb.Y10)
    o = np.zeros_like(h)
    hd = lambda arr, layout, ld=0, ch=2, off=0: wmb.image_desc(arr.ctypes.data + off, rows, cols, layout, wmb.U8, ld, ch)
    refused(L.wm_embed_host(wm._h, C.byref(hd(h, wmb.Y10)), None, C.byref(hd(o, wmb.Y10_MSB)), wmb.ME, C.byref(a)), "host Y10 in, MSB out")
    refused(L.wm_detect_host(wm._h, C.byref(hd(h, wmb.Y10, ld=2 * cols + 1)), wmb.ME, C.byref(a)), "host odd ld")
    refused(L.wm_detect_host(wm._h, C.byref(hd(h, wmb.Y10_MSB, ch=3)), wmb.ME, C.byref(a)), "host 3 channels")
    hb = np.zeros(2 * rows * cols * 2 + 8, np.uint8)
    corr, st = np.zeros(2, np.float32), np.zeros(2, np.int32)
    refused(L.wm_detect_host_batch(wm._h, 0, C.byref(wmb.image_desc(hb.ctypes.data, rows, cols, wmb.Y10, wmb.U8, 0, 2)), rows * 2 * cols + 1, 2,
                                   wmb.ME, corr.ctypes.data_as(C.POINTER(C.c_float)), st.ctypes.data_as(C.POINTER(C.c_int))), "host odd batch stride")
    refused(L.wm_detect_host(wm._h, C.byref(wmb.image_desc(hb.ctypes.data + 1, rows, cols, wmb.Y10, wmb.U8, 0, 2)), wmb.ME, C.byref(a)),
            "host misaligned pointer")
    assert np.all(o == 0)
    with pytest.raises(TypeError):
        wm.make_watermark_host(np.zeros((rows, cols, 2), np.uint8), None, o, wmb.ME, layout=wmb.Y10)
    for x in (d, out, outm, outy, out3, gray, y8):
        x.free()
    L.wm_dev_free(wm._h, big)
    wm.close()


# ---- 9. the C++ façade: processFramesInMemory on WM_Y10 frames, one and two Watermark objects ----
def test_cpp_process_frames_in_memory_y10(wmb, tmp_path):
    b = wmb.build()
    exe = b.build_video_y10_test()
    assert exe and os.path.exists(exe)
    n, interval = 7, 2
    ls = 2 * VCOLS + 24
    W = util.normal_w(VROWS, VCOLS)
    frames = video_frames(wmb, wmb.Y10, n, seed=70)
    buf = np.full((n, VROWS, ls), 0x77, np.uint8)
    buf[:, :, :2 * VCOLS] = frames.reshape(n, VROWS, 2 * VCOLS)
    buf.tofile(tmp_path / "frames.u8")
    W.tofile(tmp_path / "w.dat")
    r = subprocess.run([exe, str(tmp_path / "w.dat"), str(VROWS), str(VCOLS), str(tmp_path / "frames.u8"), str(n), str(ls), str(interval),
                        str(tmp_path / "out.u8")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    got = dict(line.split(None, 1) for line in r.stdout.strip().splitlines())
    assert got["frames"].split() == [str(n), str(n)]
    assert got["equal_pixels"].strip() == "1" and got["equal_a"].strip() == "1" and got["nan_where_gated_off"].strip() == "1"
    assert float(got["corr_max_rel"]) == 0.0
    # the façade's one-object run is the Python driver's run
    wm = wmb.Watermark(VROWS, VCOLS, W, 3, PSNR)
    out, a = run_driver(wmb, wm, frames, wmb.Y10, wmb.VIDEO_EMBED, interval, 0, False, linesize=ls)
    _, corr = run_driver(wmb, wm, out, wmb.Y10, wmb.VIDEO_DETECT, interval, 0, False)
    assert np.array_equal(np.fromfile(tmp_path / "out.u8", np.uint8).reshape(out.shape), out)
    for i in range(n):
        assert np.array_equal(np.float32(got["a_%d" % i]), a[i], equal_nan=True)
        assert np.array_equal(np.float32(got["corr_%d" % i]), corr[i], equal_nan=True)
    wm.close()
