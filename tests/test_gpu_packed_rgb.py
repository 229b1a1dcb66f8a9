"""Packed 8-bit RGB / BGR images (WM_PACKED_RGB / WM_PACKED_BGR) through the embed and detect entry points.

The reference's colour flow (main.cpp:142-154, 175-222): gray = rgb2gray(0.299, 0.587, 0.114), makeWatermark(gray, rgb) on all three
channels, saved as u8, detectWatermark on the gray of the saved image.  A caller of the planar API composes it by hand: widen to planar
f32 -> wm_rgb2gray -> wm_embed with a 3-plane base and u8 planar output -> interleave; detect: widen -> wm_rgb2gray -> wm_detect.
The packed path must give exactly those bytes and the bits of `a` and of the correlation.
"""
import ctypes as C

import numpy as np
import pytest

import util

pytestmark = pytest.mark.gpu

PSNR = 40.0
SIZES = [(270, 480), (67, 131), (1080, 1920), (1078, 1918), (2160, 3840)]


def color_image(rows, cols, seed=0):
    """Natural-statistics colour image of any size: 512.png mirrored-tiled, shifted and lightly noised, rounded to u8."""
    from PIL import Image
    g = np.asarray(Image.open(util.PNG512_PATH).convert("RGB"), np.float32)
    g = np.concatenate([g, g[:, ::-1]], 1)
    g = np.concatenate([g, g[::-1, :]], 0)
    rng = np.random.default_rng(seed)
    oy, ox = rng.integers(0, 1024, 2)
    yy = (np.arange(rows) + oy) % 1024
    xx = (np.arange(cols) + ox) % 1024
    img = g[np.ix_(yy, xx)] + rng.uniform(-1.5, 1.5, (rows, cols, 3))
    return np.clip(np.rint(img), 0, 255).astype(np.uint8)


def fixture_512():
    from PIL import Image
    return np.ascontiguousarray(np.asarray(Image.open(util.PNG512_PATH).convert("RGB"), np.uint8))


def planar_f32(img):
    return np.ascontiguousarray(img.transpose(2, 0, 1)).astype(np.float32)


def composed(wmb, wm, img, mask):
    """What a caller of the planar API does today -> (packed u8 output, a, status, corr, detect status)."""
    d = wmb.DeviceArray.from_numpy(wm, planar_f32(img), wmb.ROW_MAJOR)
    gray = wm.rgb2gray(d)
    out, a, st = wm.makeWatermark(gray, d, mask, out_dtype=wmb.U8)
    o = np.ascontiguousarray(out.numpy().transpose(1, 2, 0))
    d2 = wmb.DeviceArray.from_numpy(wm, planar_f32(o), wmb.ROW_MAJOR)
    corr, st2 = wm.detectWatermark(wm.rgb2gray(d2), mask)
    for x in (d, gray, out, d2):
        x.free()
    return o, a, st, corr, st2


def packed(wmb, wm, img, layout, mask):
    d = wmb.DeviceArray.from_numpy(wm, img, layout)
    out, a, st = wm.makeWatermark(d, None, mask)
    corr, st2 = wm.detectWatermark(out, mask)
    o = out.numpy()
    d.free()
    out.free()
    return o, a, st, corr, st2


def f32bits(x):
    return np.float32(x).view(np.uint32)


def assert_same(p, c, what):
    po, pa, pst, pcorr, pst2 = p
    co, ca, cst, ccorr, cst2 = c
    print("%s: a=%r corr=%r differing bytes=%d" % (what, pa, pcorr, int(np.count_nonzero(po != co))))
    assert pst == cst and pst2 == cst2, what
    assert np.array_equal(po, co), what
    assert f32bits(pa) == f32bits(ca), (what, pa, ca)
    assert f32bits(pcorr) == f32bits(ccorr), (what, pcorr, ccorr)


def both_layouts(wmb, img):
    """(layout, packed bytes, how to map an RGB-ordered result to it): BGR input = the RGB bytes swapped."""
    return [(wmb.PACKED_RGB, img, lambda x: x), (wmb.PACKED_BGR, np.ascontiguousarray(img[..., ::-1]), lambda x: np.ascontiguousarray(x[..., ::-1]))]


def run_equal_to_composed(wmb, img):
    rows, cols = img.shape[:2]
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    for mask in (wmb.ME, wmb.NVF):
        ref = composed(wmb, wm, img, mask)
        for layout, src, to_layout in both_layouts(wmb, img):
            got = packed(wmb, wm, src, layout, mask)
            assert_same(got, (to_layout(ref[0]),) + ref[1:], "%dx%d mask=%d layout=%d" % (rows, cols, mask, layout))
    wm.close()


def test_equal_to_composed_512_fixture(wmb):
    run_equal_to_composed(wmb, fixture_512())


@pytest.mark.parametrize("rows,cols", SIZES)
def test_equal_to_composed(wmb, rows, cols):
    run_equal_to_composed(wmb, color_image(rows, cols, seed=rows + cols))


@pytest.mark.parametrize("which", ["512", "1080p"])
def test_against_oracle(wmb, oracle, which):
    img = fixture_512() if which == "512" else color_image(1080, 1920, seed=5)
    rows, cols = img.shape[:2]
    W = util.normal_w(rows, cols)
    wm = wmb.Watermark(rows, cols, W, 3, PSNR)
    rgb = planar_f32(img)
    for mask in (wmb.ME, wmb.NVF):
        e = oracle.embed(oracle.rgb2gray(rgb), W, PSNR, mask, base=rgb)
        trunc = e["out"].astype(np.uint8)  # values are clamped to 0..255: .as(u8) truncates
        corr_ref = oracle.detect(oracle.rgb2gray(trunc.astype(np.float32)), W, mask)["corr"]
        for layout, src, to_layout in both_layouts(wmb, img):
            o, a, st, corr, _ = packed(wmb, wm, src, layout, mask)
            dpx = np.abs(o.astype(int) - to_layout(trunc.transpose(1, 2, 0)).astype(int)).max()
            ra, rc = util.rel(a, e["a"]), util.rel(corr, corr_ref)
            print("oracle %s mask=%d layout=%d: a rel %.3g corr rel %.3g max pixel diff %d" % (which, mask, layout, ra, rc, dpx))
            assert st == 0 and e["status"] == 0
            assert ra <= 1e-3 and rc <= 1e-3 and dpx <= 1
    wm.close()


@pytest.mark.parametrize("rows,cols", [(1080, 1920), (2160, 3840)])
def test_tma_and_plain_loaders_agree(wmb, rows, cols):
    img = color_image(rows, cols, seed=11)
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    for mask in (wmb.ME, wmb.NVF):
        res = []
        for tma in (1, 0):
            wm.set_option(wmb.OPT_USE_TMA, tma)
            res.append(packed(wmb, wm, img, wmb.PACKED_RGB, mask))
        assert_same(res[1], res[0], "plain vs TMA %dx%d mask=%d" % (rows, cols, mask))
    wm.close()


# ---- row pitch: the caller's padding bytes are neither read into the result nor written ----
def dev_raw(wmb, wm, buf):
    p = wmb.lib().wm_dev_alloc(wm._h, buf.nbytes)
    assert p and wmb.lib().wm_dev_upload(wm._h, p, buf.ctypes.data, buf.nbytes) == 0
    return p


def dev_get(wmb, wm, p, shape):
    buf = np.empty(shape, np.uint8)
    assert wmb.lib().wm_dev_download(wm._h, buf.ctypes.data, p, buf.nbytes) == 0
    return buf


def pitched(img, ld, fill):
    rows, cols = img.shape[:2]
    big = np.full((rows, ld), fill, np.uint8)
    big[:, :3 * cols] = img.reshape(rows, 3 * cols)
    return big


@pytest.mark.parametrize("extra", [64, 5])
def test_row_pitch(wmb, extra):
    rows, cols = 270, 480
    img = color_image(rows, cols, seed=3)
    ld = 3 * cols + extra
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    L = wmb.lib()
    for mask in (wmb.ME, wmb.NVF):
        ref = packed(wmb, wm, img, wmb.PACKED_RGB, mask)
        # device
        pin, pout = dev_raw(wmb, wm, pitched(img, ld, 7)), dev_raw(wmb, wm, np.full((rows, ld), 0xA5, np.uint8))
        din = wmb.image_desc(pin, rows, cols, wmb.PACKED_RGB, wmb.U8, ld, 3)
        dout = wmb.image_desc(pout, rows, cols, wmb.PACKED_RGB, wmb.U8, ld, 3)
        a, corr = C.c_float(np.nan), C.c_float(0)
        st = wm._check(L.wm_embed(wm._h, C.byref(din), None, C.byref(dout), mask, C.byref(a)))
        st2 = wm._check(L.wm_detect(wm._h, C.byref(dout), mask, C.byref(corr)))
        o = dev_get(wmb, wm, pout, (rows, ld))
        assert np.all(o[:, 3 * cols:] == 0xA5)
        assert_same((np.ascontiguousarray(o[:, :3 * cols].reshape(rows, cols, 3)), a.value, st, corr.value, st2), ref, "device ld=%d" % ld)
        L.wm_dev_free(wm._h, pin)
        L.wm_dev_free(wm._h, pout)
        # host
        hin, hout = pitched(img, ld, 7), np.full((rows, ld), 0xA5, np.uint8)
        view = lambda b: np.lib.stride_tricks.as_strided(b, (rows, cols, 3), (ld, 3, 1))
        a, st = wm.make_watermark_host(view(hin), None, view(hout), mask, layout=wmb.PACKED_RGB)
        corr, st2 = wm.detect_watermark_host(view(hout), mask, layout=wmb.PACKED_RGB)
        assert np.all(hout[:, 3 * cols:] == 0xA5)
        assert_same((np.ascontiguousarray(view(hout)), a, st, corr, st2), ref, "host ld=%d" % ld)
    wm.close()


# ---- batches: every image equals its single-image run ----
def batch_images(rows, cols, n):
    base = [color_image(rows, cols, seed=100 + k) for k in range(4)]
    return np.stack([np.roll(base[b % 4], 7 * b, axis=1) for b in range(n)])


@pytest.mark.parametrize("rows,cols,batch,stride_extra", [(1080, 1920, 148, 0), (1080, 1920, 150, 0), (270, 480, 5, 4099)])
def test_batches(wmb, rows, cols, batch, stride_extra):
    """148 1080p images; 150 (uneven share of a wave: launched as sub-batches); an explicit stride larger than one image."""
    imgs = batch_images(rows, cols, batch)
    one = rows * 3 * cols
    stride = one + stride_extra
    buf = np.zeros((batch, stride), np.uint8)
    buf[:, :one] = imgs.reshape(batch, one)
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    L = wmb.lib()
    arg = stride if stride_extra else 0
    for mask in (wmb.ME, wmb.NVF):
        pin, pout, pone = dev_raw(wmb, wm, buf), dev_raw(wmb, wm, buf), dev_raw(wmb, wm, buf)
        desc = lambda p: wmb.image_desc(p, rows, cols, wmb.PACKED_RGB, wmb.U8, 0, 3)
        a, st, corr, st2 = (np.full(batch, np.nan, np.float32), np.zeros(batch, np.int32), np.zeros(batch, np.float32), np.zeros(batch, np.int32))
        wm.embed_batch(0, desc(pin), desc(pin), desc(pout), arg, arg, arg, batch, mask, a, st)
        wm.detect_batch(0, desc(pout), arg, batch, mask, corr, st2)
        wm.sync(0)
        a1, st1, c1, s21 = (np.full(batch, np.nan, np.float32), np.zeros(batch, np.int32), np.zeros(batch, np.float32), np.zeros(batch, np.int32))
        for b in range(batch):
            wm.embed_batch(0, desc(pin + b * stride), desc(pin + b * stride), desc(pone + b * stride), 0, 0, 0, 1, mask, a1[b:], st1[b:])
            wm.detect_batch(0, desc(pone + b * stride), 0, 1, mask, c1[b:], s21[b:])
        wm.sync(0)
        ob, o1 = dev_get(wmb, wm, pout, buf.shape), dev_get(wmb, wm, pone, buf.shape)
        for p in (pin, pout, pone):
            L.wm_dev_free(wm._h, p)
        # a batch launch gives each image fewer CTAs than a single-image launch, so the f64 partial sums are grouped differently: the
        # correlation may differ in its last f32 bits (as for gray batches); pixels and `a` come out identical
        rc = float(np.max(np.abs(corr.astype(np.float64) - c1) / np.abs(c1)))
        print("batch %d %dx%d mask=%d: differing bytes %d, corr max rel %.3g" % (batch, rows, cols, mask, int(np.count_nonzero(ob != o1)), rc))
        assert np.array_equal(ob, o1)
        assert np.array_equal(st, st1) and np.array_equal(st2, s21)
        assert np.array_equal(a.view(np.uint32), a1.view(np.uint32))
        assert rc <= 1e-6
        if stride_extra:
            assert np.all(ob[:, one:] == 0)  # the gap between strided images is not written
    wm.close()


def test_host_forms_equal_device_forms(wmb):
    rows, cols, batch = 270, 480, 5
    imgs = batch_images(rows, cols, batch)
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    L = wmb.lib()
    one = rows * 3 * cols
    for layout in (wmb.PACKED_RGB, wmb.PACKED_BGR):
        for mask in (wmb.ME, wmb.NVF):
            refs = [packed(wmb, wm, imgs[b], layout, mask) for b in range(batch)]
            # single-image host forms
            for b in (0, batch - 1):
                out = np.empty_like(imgs[b])
                a, st = wm.make_watermark_host(imgs[b], None, out, mask, layout=layout)
                corr, st2 = wm.detect_watermark_host(out, mask, layout=layout)
                assert_same((out, a, st, corr, st2), refs[b], "host single b=%d layout=%d mask=%d" % (b, layout, mask))
            # pinned batch forms
            hp = [L.wm_host_alloc_pinned(batch * one) for _ in range(2)]
            hin, hout = [np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), (batch, rows, cols, 3)) for p in hp]
            hin[:] = imgs
            desc = lambda p: wmb.image_desc(p, rows, cols, layout, wmb.U8, 0, 3)
            a, st, corr, st2 = (np.full(batch, np.nan, np.float32), np.zeros(batch, np.int32), np.zeros(batch, np.float32), np.zeros(batch, np.int32))
            wm.embed_host_batch(1, desc(hp[0]), desc(hp[0]), desc(hp[1]), 0, 0, 0, batch, mask, a, st)
            wm.sync(1)
            for b in range(batch):
                assert np.array_equal(hout[b], refs[b][0]) and f32bits(a[b]) == f32bits(refs[b][1])
            hout[:] = 0
            wm.embed_verify_host_batch(2, desc(hp[0]), desc(hp[0]), desc(hp[1]), 0, 0, 0, batch, mask, a, corr, st)
            wm.sync(2)
            for b in range(batch):
                assert_same((hout[b], a[b], st[b], corr[b], 0), refs[b][:4] + (0,), "verify b=%d layout=%d mask=%d" % (b, layout, mask))
            corr[:] = 0
            wm.detect_host_batch(3, desc(hp[1]), 0, batch, mask, corr, st2)
            wm.sync(3)
            for b in range(batch):
                assert f32bits(corr[b]) == f32bits(refs[b][3]) and st2[b] == refs[b][4]
            for p in hp:
                L.wm_host_free_pinned(p)
    wm.close()


def test_singular_and_zero_mask(wmb):
    rows, cols = 270, 480
    img = np.empty((rows, cols, 3), np.uint8)
    img[:] = (10, 200, 31)
    black = np.zeros((rows, cols, 3), np.uint8)  # gray exactly 0: the NVF mask is exactly 0 (a non-integer constant gray leaves rounding noise)
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    for layout in (wmb.PACKED_RGB, wmb.PACKED_BGR):
        o, a, st, corr, st2 = packed(wmb, wm, img, layout, wmb.ME)
        assert st == wmb.SINGULAR and np.isnan(a) and np.array_equal(o, img)  # `a` untouched, the image returned unchanged
        assert st2 == wmb.SINGULAR and corr == 0.0
        o, a, st, corr, st2 = packed(wmb, wm, black, layout, wmb.NVF)
        assert st == wmb.ZERO_MASK and np.isinf(a) and np.array_equal(o, black)
        assert_same((o, a, st, corr, st2), composed(wmb, wm, black, wmb.NVF), "zero mask layout=%d" % layout)
    wm.close()


@pytest.mark.parametrize("rows,cols", [(270, 480), (67, 131)])
def test_nvf_p5(wmb, rows, cols):
    img = color_image(rows, cols, seed=9)
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 5, PSNR)
    ref = composed(wmb, wm, img, wmb.NVF)
    for layout, src, to_layout in both_layouts(wmb, img):
        assert_same(packed(wmb, wm, src, layout, wmb.NVF), (to_layout(ref[0]),) + ref[1:], "NVF p=5 %dx%d layout=%d" % (rows, cols, layout))
    wm.close()


def test_rejections(wmb):
    rows, cols = 67, 131
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    L = wmb.lib()
    img = color_image(rows, cols)
    d = wmb.DeviceArray.from_numpy(wm, img, wmb.PACKED_RGB)
    out = wmb.DeviceArray(wm, rows, cols, wmb.PACKED_RGB)
    outb = wmb.DeviceArray(wm, rows, cols, wmb.PACKED_BGR)
    gray = wmb.DeviceArray(wm, rows, cols, wmb.ROW_MAJOR, wmb.F32, 1)
    rgb = wmb.DeviceArray(wm, rows, cols, wmb.ROW_MAJOR, wmb.U8, 3)
    big = wmb.DeviceArray(wm, rows, cols, wmb.PACKED_RGB, ld=3 * cols + 16)
    a = C.c_float(0)

    def desc(p, layout=wmb.PACKED_RGB, dtype=wmb.U8, ld=0, ch=3):
        return wmb.image_desc(p, rows, cols, layout, dtype, ld, ch)

    def embed_rc(i, b, o):
        return L.wm_embed(wm._h, C.byref(i), C.byref(b) if b is not None else None, C.byref(o), wmb.ME, C.byref(a))

    def refused(rc, what):
        msg = L.wm_last_error(wm._h).decode()
        print("%s: %d %s" % (what, rc, msg))
        assert rc == -5 and msg, what

    refused(embed_rc(desc(d.ptr, dtype=wmb.F32), None, out.desc()), "f32 packed")
    refused(embed_rc(desc(d.ptr, ch=1), None, out.desc()), "channels 1")
    refused(embed_rc(desc(d.ptr, ld=3 * cols - 1), None, out.desc()), "ld < 3 cols")
    refused(L.wm_detect(wm._h, C.byref(desc(d.ptr, ld=3 * cols - 1)), wmb.ME, C.byref(a)), "detect ld < 3 cols")
    refused(embed_rc(d.desc(), rgb.desc(), out.desc()), "planar base")
    refused(embed_rc(d.desc(), gray.desc(), out.desc()), "gray base")
    refused(embed_rc(d.desc(), None, rgb.desc()), "planar out")
    refused(embed_rc(d.desc(), None, gray.desc()), "gray out")
    refused(embed_rc(d.desc(), None, outb.desc()), "out of the other packed layout")
    refused(embed_rc(d.desc(), big.desc(), out.desc()), "base is another packed image")
    refused(embed_rc(gray.desc(), rgb.desc(), out.desc()), "gray input, packed out")
    refused(embed_rc(gray.desc(), d.desc(), rgb.desc()), "gray input, packed base")
    refused(embed_rc(d.desc(), None, desc(d.ptr + 3)), "out overlaps in")
    refused(L.wm_rgb2gray(wm._h, C.byref(d.desc()), C.byref(gray.desc()), 0.299, 0.587, 0.114), "rgb2gray")
    refused(L.wm_debug_plane(wm._h, C.byref(d.desc()), wmb.DBG_ERRSEQ, gray.ptr), "debug_plane")
    refused(L.wm_debug_detect_planes(wm._h, C.byref(d.desc()), wmb.ME, gray.ptr, gray.ptr, C.byref(a)), "debug_detect_planes")
    for x in (d, out, outb, gray, rgb, big):
        x.free()
    wm.close()
