"""Packed 8-bit images with a fourth byte per pixel (WM_PACKED_RGBA / WM_PACKED_BGRA) through the embed and detect entry points.

The reference is the packed RGB / BGR path (itself pinned to the composed planar path and to the CPU oracle by test_gpu_packed_rgb.py)
run on the same image with the fourth byte removed.  The three colour bytes of the output, `a`, the correlation and the statuses must be
those of that run, bit for bit; the fourth byte of the output must be the input's.  Alpha planes are seeded random and contain 0 and 255.
"""
import ctypes as C

import numpy as np
import pytest

import util
from test_gpu_packed_rgb import color_image, dev_get, dev_raw, f32bits, fixture_512

pytestmark = pytest.mark.gpu

PSNR = 40.0
SIZES = [(270, 480), (67, 131), (1080, 1920), (1078, 1918), (2160, 3840)]


def alpha_plane(rows, cols, seed=0):
    a = np.random.default_rng(1000 + seed).integers(0, 256, (rows, cols), dtype=np.uint8)
    a[0, 0], a[-1, -1] = 0, 255
    return a


def with_alpha(rgb, alpha):
    return np.ascontiguousarray(np.concatenate([rgb, alpha[..., None]], -1))


def three_byte(wmb, layout):
    return {wmb.PACKED_RGBA: wmb.PACKED_RGB, wmb.PACKED_BGRA: wmb.PACKED_BGR}[layout]


def both_layouts(wmb, img, alpha):
    """(4-byte layout, its bytes): BGRA = the RGB bytes swapped, then alpha."""
    return [(wmb.PACKED_RGBA, with_alpha(img, alpha)), (wmb.PACKED_BGRA, with_alpha(np.ascontiguousarray(img[..., ::-1]), alpha))]


def packed(wmb, wm, img, layout, mask):
    """device round trip -> (packed u8 output, a, status, corr, detect status)"""
    d = wmb.DeviceArray.from_numpy(wm, img, layout)
    out, a, st = wm.makeWatermark(d, None, mask)
    corr, st2 = wm.detectWatermark(out, mask)
    o = out.numpy()
    d.free()
    out.free()
    return o, a, st, corr, st2


def rgb_ref(wmb, wm, src4, layout, mask):
    """the packed RGB / BGR path on the same pixels without their fourth byte"""
    return packed(wmb, wm, np.ascontiguousarray(src4[..., :3]), three_byte(wmb, layout), mask)


def assert_like_rgb(got, ref, src4, what):
    o, a, st, corr, st2 = got
    ro, ra, rst, rcorr, rst2 = ref
    print("%s: a=%r corr=%r differing colour bytes=%d alpha bytes changed=%d" % (
        what, a, corr, int(np.count_nonzero(o[..., :3] != ro)), int(np.count_nonzero(o[..., 3] != src4[..., 3]))))
    assert st == rst and st2 == rst2, what
    assert np.array_equal(o[..., :3], ro), what
    assert np.array_equal(o[..., 3], src4[..., 3]), what
    assert f32bits(a) == f32bits(ra), (what, a, ra)
    assert f32bits(corr) == f32bits(rcorr), (what, corr, rcorr)


def run_equal_to_rgb(wmb, img, seed):
    rows, cols = img.shape[:2]
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    alpha = alpha_plane(rows, cols, seed)
    for mask in (wmb.ME, wmb.NVF):
        for layout, src in both_layouts(wmb, img, alpha):
            got = packed(wmb, wm, src, layout, mask)
            assert_like_rgb(got, rgb_ref(wmb, wm, src, layout, mask), src, "%dx%d mask=%d layout=%d" % (rows, cols, mask, layout))
    wm.close()


def test_equal_to_rgb_512_fixture(wmb):
    run_equal_to_rgb(wmb, fixture_512(), 0)


@pytest.mark.parametrize("rows,cols", SIZES)
def test_equal_to_rgb(wmb, rows, cols):
    run_equal_to_rgb(wmb, color_image(rows, cols, seed=rows + cols), rows + cols)


@pytest.mark.parametrize("which", ["512", "1080p"])
def test_against_oracle(wmb, oracle, which):
    img = fixture_512() if which == "512" else color_image(1080, 1920, seed=5)
    rows, cols = img.shape[:2]
    W = util.normal_w(rows, cols)
    wm = wmb.Watermark(rows, cols, W, 3, PSNR)
    rgb = np.ascontiguousarray(img.transpose(2, 0, 1)).astype(np.float32)
    alpha = alpha_plane(rows, cols, 5)
    for mask in (wmb.ME, wmb.NVF):
        e = oracle.embed(oracle.rgb2gray(rgb), W, PSNR, mask, base=rgb)
        trunc = e["out"].astype(np.uint8)  # values are clamped to 0..255: .as(u8) truncates
        corr_ref = oracle.detect(oracle.rgb2gray(trunc.astype(np.float32)), W, mask)["corr"]
        ref = trunc.transpose(1, 2, 0)
        for layout, src in both_layouts(wmb, img, alpha):
            o, a, st, corr, _ = packed(wmb, wm, src, layout, mask)
            colour = o[..., :3] if layout == wmb.PACKED_RGBA else o[..., 2::-1]
            dpx = np.abs(colour.astype(int) - ref.astype(int)).max()
            ra, rc = util.rel(a, e["a"]), util.rel(corr, corr_ref)
            print("oracle %s mask=%d layout=%d: a rel %.3g corr rel %.3g max pixel diff %d" % (which, mask, layout, ra, rc, dpx))
            assert st == 0 and e["status"] == 0
            assert ra <= 1e-3 and rc <= 1e-3 and dpx <= 1
            assert np.array_equal(o[..., 3], alpha)
    wm.close()


@pytest.mark.parametrize("rows,cols", [(1080, 1920), (2160, 3840)])
def test_tma_and_plain_loaders_agree(wmb, rows, cols):
    src = with_alpha(color_image(rows, cols, seed=11), alpha_plane(rows, cols, 11))
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    for mask in (wmb.ME, wmb.NVF):
        res = []
        for tma in (1, 0):
            wm.set_option(wmb.OPT_USE_TMA, tma)
            res.append(packed(wmb, wm, src, wmb.PACKED_RGBA, mask))
        po, pa, pst, pc, pst2 = res[1]
        to, ta, tst, tc, tst2 = res[0]
        print("plain vs TMA %dx%d mask=%d: differing bytes %d" % (rows, cols, mask, int(np.count_nonzero(po != to))))
        assert pst == tst and pst2 == tst2 and np.array_equal(po, to)
        assert f32bits(pa) == f32bits(ta) and f32bits(pc) == f32bits(tc)
    wm.close()


# ---- alignment: row pitch +64 (16-byte accesses), +4 (one word per pixel), +5 (bytes); images 4 bytes past an aligned address.
# The caller's padding, and every byte around the image, is neither read into the result nor written.
def placed(img, ld, off, fill):
    """a raw buffer holding img with row pitch ld at byte offset off, every other byte = fill"""
    rows, cols, n = img.shape
    buf = np.full(off + rows * ld + 16, fill, np.uint8)
    buf[off:off + rows * ld].reshape(rows, ld)[:, :n * cols] = img.reshape(rows, n * cols)
    return buf


def image_of(buf, rows, cols, ld, off):
    return np.ascontiguousarray(buf[off:off + rows * ld].reshape(rows, ld)[:, :4 * cols].reshape(rows, cols, 4))


def untouched(buf, rows, cols, ld, off, fill):
    m = np.ones(buf.shape, bool)
    m[off:off + rows * ld].reshape(rows, ld)[:, :4 * cols] = False
    return bool(np.all(buf[m] == fill))


@pytest.mark.parametrize("extra,in_off,out_off", [(64, 0, 0), (4, 0, 0), (5, 0, 0), (64, 4, 4), (64, 4, 0), (64, 0, 4)])
def test_alignment_paths(wmb, extra, in_off, out_off):
    rows, cols = 270, 480
    src = with_alpha(color_image(rows, cols, seed=3), alpha_plane(rows, cols, 3))
    ld = 4 * cols + extra
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    L = wmb.lib()
    for mask in (wmb.ME, wmb.NVF):
        ref = packed(wmb, wm, src, wmb.PACKED_RGBA, mask)  # dense rows, 16-byte aligned
        what = "ld=%d in+%d out+%d mask=%d" % (ld, in_off, out_off, mask)
        # device
        hin, hout = placed(src, ld, in_off, 7), np.full(out_off + rows * ld + 16, 0xA5, np.uint8)
        pin, pout = dev_raw(wmb, wm, hin), dev_raw(wmb, wm, hout)
        din = wmb.image_desc(pin + in_off, rows, cols, wmb.PACKED_RGBA, wmb.U8, ld, 4)
        dout = wmb.image_desc(pout + out_off, rows, cols, wmb.PACKED_RGBA, wmb.U8, ld, 4)
        a, corr = C.c_float(np.nan), C.c_float(0)
        st = wm._check(L.wm_embed(wm._h, C.byref(din), None, C.byref(dout), mask, C.byref(a)))
        st2 = wm._check(L.wm_detect(wm._h, C.byref(dout), mask, C.byref(corr)))
        o = dev_get(wmb, wm, pout, hout.shape)
        assert np.array_equal(dev_get(wmb, wm, pin, hin.shape), hin), what  # the input is only read
        assert untouched(o, rows, cols, ld, out_off, 0xA5), what
        got = (image_of(o, rows, cols, ld, out_off), a.value, st, corr.value, st2)
        assert np.array_equal(got[0], ref[0]) and f32bits(got[1]) == f32bits(ref[1]) and f32bits(got[3]) == f32bits(ref[3]), "device " + what
        assert got[2] == ref[2] and got[4] == ref[4]
        L.wm_dev_free(wm._h, pin)
        L.wm_dev_free(wm._h, pout)
        # host
        hout = np.full(out_off + rows * ld + 16, 0xA5, np.uint8)
        view = lambda b, off: np.lib.stride_tricks.as_strided(b[off:], (rows, cols, 4), (ld, 4, 1))
        a, st = wm.make_watermark_host(view(hin, in_off), None, view(hout, out_off), mask, layout=wmb.PACKED_RGBA)
        corr, st2 = wm.detect_watermark_host(view(hout, out_off), mask, layout=wmb.PACKED_RGBA)
        assert untouched(hout, rows, cols, ld, out_off, 0xA5), what
        got = (image_of(hout, rows, cols, ld, out_off), a, st, corr, st2)
        assert np.array_equal(got[0], ref[0]) and f32bits(a) == f32bits(ref[1]) and f32bits(corr) == f32bits(ref[3]), "host " + what
        assert st == ref[2] and st2 == ref[4]
    wm.close()


# ---- batches: every image equals its single-image run ----
def batch_images(rows, cols, n):
    base = [with_alpha(color_image(rows, cols, seed=100 + k), alpha_plane(rows, cols, 100 + k)) for k in range(4)]
    return np.stack([np.roll(base[b % 4], 7 * b, axis=1) for b in range(n)])


@pytest.mark.parametrize("rows,cols,batch,stride_extra", [(1080, 1920, 148, 0), (1080, 1920, 150, 0), (270, 480, 5, 4099)])
def test_batches(wmb, rows, cols, batch, stride_extra):
    """148 1080p images; 150 (uneven share of a wave: launched as sub-batches); an explicit stride larger than one image."""
    imgs = batch_images(rows, cols, batch)
    one = rows * 4 * cols
    stride = one + stride_extra
    buf = np.zeros((batch, stride), np.uint8)
    buf[:, :one] = imgs.reshape(batch, one)
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    L = wmb.lib()
    arg = stride if stride_extra else 0
    desc = lambda p: wmb.image_desc(p, rows, cols, wmb.PACKED_RGBA, wmb.U8, 0, 4)
    for mask in (wmb.ME, wmb.NVF):
        pin, pout, pone = dev_raw(wmb, wm, buf), dev_raw(wmb, wm, buf), dev_raw(wmb, wm, buf)
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
        # correlation may differ in its last f32 bits (as for gray and RGB batches); pixels and `a` come out identical
        rc = float(np.max(np.abs(corr.astype(np.float64) - c1) / np.abs(c1)))
        print("batch %d %dx%d mask=%d: differing bytes %d, corr max rel %.3g" % (batch, rows, cols, mask, int(np.count_nonzero(ob != o1)), rc))
        assert np.array_equal(ob, o1)
        assert np.array_equal(ob[:, :one].reshape(imgs.shape)[..., 3], imgs[..., 3])
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
    one = rows * 4 * cols
    for layout in (wmb.PACKED_RGBA, wmb.PACKED_BGRA):
        for mask in (wmb.ME, wmb.NVF):
            refs = [packed(wmb, wm, imgs[b], layout, mask) for b in range(batch)]
            for b in range(batch):
                assert_like_rgb(refs[b], rgb_ref(wmb, wm, imgs[b], layout, mask), imgs[b], "device b=%d layout=%d mask=%d" % (b, layout, mask))
            # single-image host forms
            for b in (0, batch - 1):
                out = np.empty_like(imgs[b])
                a, st = wm.make_watermark_host(imgs[b], None, out, mask, layout=layout)
                corr, st2 = wm.detect_watermark_host(out, mask, layout=layout)
                assert np.array_equal(out, refs[b][0]) and (st, st2) == (refs[b][2], refs[b][4])
                assert f32bits(a) == f32bits(refs[b][1]) and f32bits(corr) == f32bits(refs[b][3])
            # pinned batch forms
            hp = [L.wm_host_alloc_pinned(batch * one) for _ in range(2)]
            hin, hout = [np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), (batch, rows, cols, 4)) for p in hp]
            hin[:] = imgs
            desc = lambda p: wmb.image_desc(p, rows, cols, layout, wmb.U8, 0, 4)
            a, st, corr, st2 = (np.full(batch, np.nan, np.float32), np.zeros(batch, np.int32), np.zeros(batch, np.float32), np.zeros(batch, np.int32))
            wm.embed_host_batch(1, desc(hp[0]), desc(hp[0]), desc(hp[1]), 0, 0, 0, batch, mask, a, st)
            wm.sync(1)
            for b in range(batch):
                assert np.array_equal(hout[b], refs[b][0]) and f32bits(a[b]) == f32bits(refs[b][1]) and st[b] == refs[b][2]
            hout[:] = 0
            a[:] = np.nan
            wm.embed_verify_host_batch(2, desc(hp[0]), desc(hp[0]), desc(hp[1]), 0, 0, 0, batch, mask, a, corr, st)
            wm.sync(2)
            for b in range(batch):
                assert np.array_equal(hout[b], refs[b][0]) and st[b] == refs[b][2]
                assert f32bits(a[b]) == f32bits(refs[b][1]) and f32bits(corr[b]) == f32bits(refs[b][3])
            corr[:] = 0
            wm.detect_host_batch(3, desc(hp[1]), 0, batch, mask, corr, st2)
            wm.sync(3)
            for b in range(batch):
                assert f32bits(corr[b]) == f32bits(refs[b][3]) and st2[b] == refs[b][4]
            for p in hp:
                L.wm_host_free_pinned(p)
    wm.close()


def test_graph_replay(wmb):
    """Repeated synchronous calls replay a captured CUDA graph from the third call on; an RGB call on the same pointers afterwards is
    a different launch sequence and must give RGB results."""
    rows, cols = 270, 480
    src = with_alpha(color_image(rows, cols, seed=21), alpha_plane(rows, cols, 21))
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    L = wmb.lib()
    rgb = color_image(rows, cols, seed=22)
    for mask in (wmb.ME, wmb.NVF):
        ref4 = packed(wmb, wm, src, wmb.PACKED_RGBA, mask)
        ref3 = packed(wmb, wm, rgb, wmb.PACKED_RGB, mask)
        pin, pout = dev_raw(wmb, wm, src), dev_raw(wmb, wm, np.zeros_like(src))
        for layout, img, ref, n in ((wmb.PACKED_RGBA, src, ref4, 4), (wmb.PACKED_RGB, rgb, ref3, 3)):
            if n == 3:
                assert wmb.lib().wm_dev_upload(wm._h, pin, img.ctypes.data, img.nbytes) == 0
            din = wmb.image_desc(pin, rows, cols, layout, wmb.U8, 0, n)
            dout = wmb.image_desc(pout, rows, cols, layout, wmb.U8, 0, n)
            for call in range(4):
                a, corr = C.c_float(np.nan), C.c_float(0)
                st = wm._check(L.wm_embed(wm._h, C.byref(din), None, C.byref(dout), mask, C.byref(a)))
                st2 = wm._check(L.wm_detect(wm._h, C.byref(dout), mask, C.byref(corr)))
                o = dev_get(wmb, wm, pout, (rows, cols, n))
                what = "call %d layout=%d mask=%d" % (call, layout, mask)
                assert np.array_equal(o, ref[0]) and (st, st2) == (ref[2], ref[4]), what
                assert f32bits(a.value) == f32bits(ref[1]) and f32bits(corr.value) == f32bits(ref[3]), what
        L.wm_dev_free(wm._h, pin)
        L.wm_dev_free(wm._h, pout)
    wm.close()


def test_singular_and_zero_mask(wmb):
    rows, cols = 270, 480
    alpha = alpha_plane(rows, cols, 8)
    flat = np.empty((rows, cols, 3), np.uint8)
    flat[:] = (10, 200, 31)
    black = np.zeros((rows, cols, 3), np.uint8)  # gray exactly 0: the NVF mask is exactly 0
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    for layout in (wmb.PACKED_RGBA, wmb.PACKED_BGRA):
        img = with_alpha(flat, alpha)
        o, a, st, corr, st2 = got = packed(wmb, wm, img, layout, wmb.ME)
        assert st == wmb.SINGULAR and np.isnan(a) and np.array_equal(o, img)  # `a` untouched, all four bytes returned unchanged
        assert st2 == wmb.SINGULAR and corr == 0.0
        assert_like_rgb(got, rgb_ref(wmb, wm, img, layout, wmb.ME), img, "singular layout=%d" % layout)
        img = with_alpha(black, alpha)
        o, a, st, corr, st2 = got = packed(wmb, wm, img, layout, wmb.NVF)
        assert st == wmb.ZERO_MASK and np.isinf(a) and np.array_equal(o, img)
        assert_like_rgb(got, rgb_ref(wmb, wm, img, layout, wmb.NVF), img, "zero mask layout=%d" % layout)
    wm.close()


@pytest.mark.parametrize("rows,cols", [(270, 480), (67, 131)])
def test_nvf_p5(wmb, rows, cols):
    img = color_image(rows, cols, seed=9)
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 5, PSNR)
    for layout, src in both_layouts(wmb, img, alpha_plane(rows, cols, 9)):
        assert_like_rgb(packed(wmb, wm, src, layout, wmb.NVF), rgb_ref(wmb, wm, src, layout, wmb.NVF), src,
                        "NVF p=5 %dx%d layout=%d" % (rows, cols, layout))
    wm.close()


def test_rejections(wmb):
    rows, cols = 67, 131
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    L = wmb.lib()
    src = with_alpha(color_image(rows, cols), alpha_plane(rows, cols))
    d = wmb.DeviceArray.from_numpy(wm, src, wmb.PACKED_RGBA)
    out = wmb.DeviceArray(wm, rows, cols, wmb.PACKED_RGBA)
    outb = wmb.DeviceArray(wm, rows, cols, wmb.PACKED_BGRA)
    out3 = wmb.DeviceArray(wm, rows, cols, wmb.PACKED_RGB)
    d3 = wmb.DeviceArray.from_numpy(wm, np.ascontiguousarray(src[..., :3]), wmb.PACKED_RGB)
    gray = wmb.DeviceArray(wm, rows, cols, wmb.ROW_MAJOR, wmb.F32, 1)
    rgb = wmb.DeviceArray(wm, rows, cols, wmb.ROW_MAJOR, wmb.U8, 3)
    a = C.c_float(0)

    def desc(p, layout=wmb.PACKED_RGBA, dtype=wmb.U8, ld=0, ch=4):
        return wmb.image_desc(p, rows, cols, layout, dtype, ld, ch)

    def embed_rc(i, b, o):
        return L.wm_embed(wm._h, C.byref(i), C.byref(b) if b is not None else None, C.byref(o), wmb.ME, C.byref(a))

    def refused(rc, what):
        msg = L.wm_last_error(wm._h).decode()
        print("%s: %d %s" % (what, rc, msg))
        assert rc == -5 and msg, what

    refused(embed_rc(desc(d.ptr, dtype=wmb.F32), None, out.desc()), "f32 RGBA")
    refused(embed_rc(desc(d.ptr, ch=3), None, out.desc()), "RGBA with 3 channels")
    refused(embed_rc(desc(d.ptr, ch=1), None, out.desc()), "RGBA with 1 channel")
    refused(embed_rc(desc(d.ptr, layout=wmb.PACKED_BGRA, ch=3), None, outb.desc()), "BGRA with 3 channels")
    refused(embed_rc(desc(d3.ptr, layout=wmb.PACKED_RGB, ch=4), None, out3.desc()), "RGB with 4 channels")
    refused(embed_rc(desc(d.ptr, ld=4 * cols - 1), None, out.desc()), "ld < 4 cols")
    refused(embed_rc(desc(d.ptr, ld=3 * cols), None, out.desc()), "ld = 3 cols")
    refused(L.wm_detect(wm._h, C.byref(desc(d.ptr, ld=4 * cols - 1)), wmb.ME, C.byref(a)), "detect ld < 4 cols")
    refused(L.wm_detect(wm._h, C.byref(desc(d.ptr, ch=3)), wmb.ME, C.byref(a)), "detect RGBA with 3 channels")
    refused(embed_rc(d.desc(), None, out3.desc()), "RGBA in, RGB out")
    refused(embed_rc(d3.desc(), None, out.desc()), "RGB in, RGBA out")
    refused(embed_rc(d.desc(), None, outb.desc()), "RGBA in, BGRA out")
    refused(embed_rc(desc(d.ptr, layout=wmb.PACKED_BGRA), None, out.desc()), "BGRA in, RGBA out")
    refused(embed_rc(d.desc(), desc(d.ptr, layout=wmb.PACKED_RGB, ch=3), out.desc()), "RGBA in, RGB base (same pointer)")
    refused(embed_rc(d.desc(), desc(d.ptr, layout=wmb.PACKED_BGRA), out.desc()), "RGBA in, BGRA base (same pointer)")
    refused(embed_rc(d.desc(), rgb.desc(), out.desc()), "planar base")
    refused(embed_rc(d.desc(), gray.desc(), out.desc()), "gray base")
    refused(embed_rc(d.desc(), None, rgb.desc()), "planar out")
    refused(embed_rc(d.desc(), None, gray.desc()), "gray out")
    refused(embed_rc(gray.desc(), None, out.desc()), "gray input, RGBA out")
    refused(embed_rc(gray.desc(), d.desc(), rgb.desc()), "gray input, RGBA base")
    refused(embed_rc(d.desc(), None, desc(d.ptr + 4)), "out overlaps in")
    refused(L.wm_rgb2gray(wm._h, C.byref(d.desc()), C.byref(gray.desc()), 0.299, 0.587, 0.114), "rgb2gray")
    refused(L.wm_debug_plane(wm._h, C.byref(d.desc()), wmb.DBG_ERRSEQ, gray.ptr), "debug_plane")
    refused(L.wm_debug_detect_planes(wm._h, C.byref(d.desc()), wmb.ME, gray.ptr, gray.ptr, C.byref(a)), "debug_detect_planes")
    # host forms
    h4, h3 = np.array(src), np.ascontiguousarray(src[..., :3])
    hd = lambda arr, layout, ld=0, ch=4: wmb.image_desc(arr.ctypes.data, rows, cols, layout, wmb.U8, ld, ch)
    o4 = np.zeros_like(h4)
    refused(L.wm_embed_host(wm._h, C.byref(hd(h4, wmb.PACKED_RGBA)), None, C.byref(hd(h3, wmb.PACKED_RGB, ch=3)), wmb.ME, C.byref(a)),
            "host RGBA in, RGB out")
    refused(L.wm_embed_host(wm._h, C.byref(hd(h4, wmb.PACKED_RGBA)), None, C.byref(hd(o4, wmb.PACKED_BGRA)), wmb.ME, C.byref(a)),
            "host RGBA in, BGRA out")
    refused(L.wm_embed_host(wm._h, C.byref(hd(h4, wmb.PACKED_RGBA, ld=4 * cols - 1)), None, C.byref(hd(o4, wmb.PACKED_RGBA)), wmb.ME,
                            C.byref(a)), "host ld < 4 cols")
    refused(L.wm_detect_host(wm._h, C.byref(hd(h4, wmb.PACKED_RGBA, ch=3)), wmb.ME, C.byref(a)), "host detect RGBA with 3 channels")
    assert np.all(o4 == 0)
    with pytest.raises(TypeError):
        wm.make_watermark_host(h3, None, o4, wmb.ME, layout=wmb.PACKED_RGBA)
    for x in (d, out, outb, out3, d3, gray, rgb):
        x.free()
    wm.close()
