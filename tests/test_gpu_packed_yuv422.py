"""Packed 4:2:2 images (WM_PACKED_YUYV / WM_PACKED_UYVY) through the embed and detect entry points.

The reference is the Y-plane path: wm_embed_batch / wm_detect_batch on a WM_ROW_MAJOR u8 plane holding the same luma at a pitch of
round_up(cols, 16), so that both runs have the same tiles and CTA split.  The luma bytes of the output, `a`, the correlation and the
statuses must be those of that run, bit for bit; the chroma bytes of the output must be the input's.  The chroma is seeded random and
contains 0 and 255.
"""
import ctypes as C

import numpy as np
import pytest

import util
from test_gpu_packed_rgb import dev_get, dev_raw, f32bits

pytestmark = pytest.mark.gpu

PSNR = 40.0
SIZES = [(270, 480), (67, 130), (1080, 1920), (1078, 1918), (2160, 3840)]


def luma_image(rows, cols, seed=0):
    return util.natural_image(rows, cols, seed=seed, integer=True)


def fixture_512_luma():
    from PIL import Image
    return np.asarray(Image.open(util.PNG512_PATH).convert("L"), np.uint8).copy()


def chroma_plane(rows, cols, seed=0):
    c = np.random.default_rng(2000 + seed).integers(0, 256, (rows, cols), dtype=np.uint8)
    c[0, 0], c[-1, -1] = 0, 255
    return c


def koff(wmb, layout):
    """byte of a pixel holding the luma"""
    return {wmb.PACKED_YUYV: 0, wmb.PACKED_UYVY: 1}[layout]


def pack(wmb, y, c, layout):
    """(rows, cols, 2) 4:2:2 image: luma at byte koff(layout), chroma in the other byte"""
    img = np.empty(y.shape + (2,), np.uint8)
    k = koff(wmb, layout)
    img[..., k], img[..., 1 - k] = y, c
    return img


def layouts(wmb):
    return [wmb.PACKED_YUYV, wmb.PACKED_UYVY]


def round16(n):
    return (n + 15) // 16 * 16


def one(wmb, wm, pin, pout, rows, cols, layout, ch, ld, mask):
    """wm_embed_batch (base = in) + wm_detect_batch with batch 1 on device buffers -> (a, status, corr, detect status)"""
    desc = lambda p: wmb.image_desc(p, rows, cols, layout, wmb.U8, ld, ch)
    a, st, corr, st2 = np.full(1, np.nan, np.float32), np.zeros(1, np.int32), np.zeros(1, np.float32), np.zeros(1, np.int32)
    wm.embed_batch(0, desc(pin), desc(pin), desc(pout), 0, 0, 0, 1, mask, a, st)
    wm.detect_batch(0, desc(pout), 0, 1, mask, corr, st2)
    wm.sync(0)
    return a[0], st[0], corr[0], st2[0]


def yplane(wmb, wm, y, mask):
    """the Y-plane path on luma y at a pitch of round_up(cols, 16) -> (out luma, a, status, corr, detect status)"""
    rows, cols = y.shape
    ld = round16(cols)
    buf = np.zeros((rows, ld), np.uint8)
    buf[:, :cols] = y
    pin, pout = dev_raw(wmb, wm, buf), dev_raw(wmb, wm, np.zeros_like(buf))
    a, st, corr, st2 = one(wmb, wm, pin, pout, rows, cols, wmb.ROW_MAJOR, 1, ld, mask)
    o = dev_get(wmb, wm, pout, buf.shape)[:, :cols].copy()
    for p in (pin, pout):
        wmb.lib().wm_dev_free(wm._h, p)
    return o, a, st, corr, st2


def packed(wmb, wm, img, layout, mask):
    """the packed path on a dense 4:2:2 image -> (packed output, a, status, corr, detect status)"""
    rows, cols = img.shape[:2]
    pin, pout = dev_raw(wmb, wm, img), dev_raw(wmb, wm, np.zeros_like(img))
    a, st, corr, st2 = one(wmb, wm, pin, pout, rows, cols, layout, 2, 0, mask)
    o = dev_get(wmb, wm, pout, img.shape)
    for p in (pin, pout):
        wmb.lib().wm_dev_free(wm._h, p)
    return o, a, st, corr, st2


def assert_like_y(wmb, got, ref, src, layout, what):
    o, a, st, corr, st2 = got
    ro, ra, rst, rcorr, rst2 = ref
    k = koff(wmb, layout)
    print("%s: a=%r corr=%r differing luma bytes=%d chroma bytes changed=%d" % (
        what, a, corr, int(np.count_nonzero(o[..., k] != ro)), int(np.count_nonzero(o[..., 1 - k] != src[..., 1 - k]))))
    assert st == rst and st2 == rst2, what
    assert np.array_equal(o[..., k], ro), what
    assert np.array_equal(o[..., 1 - k], src[..., 1 - k]), what
    assert f32bits(a) == f32bits(ra), (what, a, ra)
    assert f32bits(corr) == f32bits(rcorr), (what, corr, rcorr)


def run_equal_to_yplane(wmb, y, seed):
    rows, cols = y.shape
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    c = chroma_plane(rows, cols, seed)
    for mask in (wmb.ME, wmb.NVF):
        ref = yplane(wmb, wm, y, mask)
        assert ref[2] == 0
        for layout in layouts(wmb):
            src = pack(wmb, y, c, layout)
            assert_like_y(wmb, packed(wmb, wm, src, layout, mask), ref, src, layout, "%dx%d mask=%d layout=%d" % (rows, cols, mask, layout))
    wm.close()


# ---- 1. equal to the Y-plane path ----
def test_equal_to_yplane_512_fixture(wmb):
    run_equal_to_yplane(wmb, fixture_512_luma(), 0)


@pytest.mark.parametrize("rows,cols", SIZES)
def test_equal_to_yplane(wmb, rows, cols):
    run_equal_to_yplane(wmb, luma_image(rows, cols, seed=rows + cols), rows + cols)


# ---- 2. against the CPU oracle ----
@pytest.mark.parametrize("which", ["512", "1080p"])
def test_against_oracle(wmb, oracle, which):
    y = fixture_512_luma() if which == "512" else luma_image(1080, 1920, seed=5)
    rows, cols = y.shape
    W = util.normal_w(rows, cols)
    wm = wmb.Watermark(rows, cols, W, 3, PSNR)
    c = chroma_plane(rows, cols, 5)
    for mask in (wmb.ME, wmb.NVF):
        est, eo, ea = oracle.embed_frame_u8(y, W, PSNR, mask)
        dst, dcorr = oracle.detect_frame_u8(eo, W, mask)
        for layout in layouts(wmb):
            k = koff(wmb, layout)
            o, a, st, corr, _ = packed(wmb, wm, pack(wmb, y, c, layout), layout, mask)
            dpx = np.abs(o[..., k].astype(int) - eo.astype(int)).max()
            ra, rc = util.rel(a, ea), util.rel(corr, dcorr)
            print("oracle %s mask=%d layout=%d: a rel %.3g corr rel %.3g max luma diff %d" % (which, mask, layout, ra, rc, dpx))
            assert st == 0 and est == 0 and dst == 0
            assert ra <= 1e-3 and rc <= 1e-3 and dpx <= 1
            assert np.array_equal(o[..., 1 - k], c)
    wm.close()


# ---- 3. TMA against the plain loaders ----
@pytest.mark.parametrize("rows,cols", [(1080, 1920), (2160, 3840)])
def test_tma_and_plain_loaders_agree(wmb, rows, cols):
    y, c = luma_image(rows, cols, seed=11), chroma_plane(rows, cols, 11)
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    for layout in layouts(wmb):
        src = pack(wmb, y, c, layout)
        for mask in (wmb.ME, wmb.NVF):
            res = []
            for tma in (1, 0):
                wm.set_option(wmb.OPT_USE_TMA, tma)
                res.append(packed(wmb, wm, src, layout, mask))
            wm.set_option(wmb.OPT_USE_TMA, 1)
            to, ta, tst, tc, tst2 = res[0]
            po, pa, pst, pc, pst2 = res[1]
            print("plain vs TMA %dx%d layout=%d mask=%d: differing bytes %d" % (rows, cols, layout, mask, int(np.count_nonzero(po != to))))
            assert pst == tst and pst2 == tst2 and np.array_equal(po, to)
            assert f32bits(pa) == f32bits(ta) and f32bits(pc) == f32bits(tc)
    wm.close()


# ---- 4. row pitches: +64 (8- and 16-byte accesses), +4 (words), +2 and +1 (bytes); images 2 bytes past an aligned address.
# The caller's padding, and every byte around the image, is neither read into the result nor written.
def placed(img, ld, off, fill):
    rows, cols, n = img.shape
    buf = np.full(off + rows * ld + 16, fill, np.uint8)
    buf[off:off + rows * ld].reshape(rows, ld)[:, :n * cols] = img.reshape(rows, n * cols)
    return buf


def image_of(buf, rows, cols, ld, off):
    return np.ascontiguousarray(buf[off:off + rows * ld].reshape(rows, ld)[:, :2 * cols].reshape(rows, cols, 2))


def untouched(buf, rows, cols, ld, off, fill):
    m = np.ones(buf.shape, bool)
    m[off:off + rows * ld].reshape(rows, ld)[:, :2 * cols] = False
    return bool(np.all(buf[m] == fill))


@pytest.mark.parametrize("extra,in_off,out_off", [(64, 0, 0), (4, 0, 0), (2, 0, 0), (1, 0, 0), (64, 2, 2), (64, 2, 0), (64, 0, 2)])
def test_row_pitch_and_alignment(wmb, extra, in_off, out_off):
    rows, cols = 270, 482
    ld = 2 * cols + extra
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    L = wmb.lib()
    y, c = luma_image(rows, cols, seed=3), chroma_plane(rows, cols, 3)
    for layout in layouts(wmb):
        src = pack(wmb, y, c, layout)
        for mask in (wmb.ME, wmb.NVF):
            ref = packed(wmb, wm, src, layout, mask)  # dense rows, 16-byte aligned
            what = "ld=%d in+%d out+%d layout=%d mask=%d" % (ld, in_off, out_off, layout, mask)
            # device
            hin, hout = placed(src, ld, in_off, 7), np.full(out_off + rows * ld + 16, 0xA5, np.uint8)
            pin, pout = dev_raw(wmb, wm, hin), dev_raw(wmb, wm, hout)
            din = wmb.image_desc(pin + in_off, rows, cols, layout, wmb.U8, ld, 2)
            dout = wmb.image_desc(pout + out_off, rows, cols, layout, wmb.U8, ld, 2)
            a, corr = C.c_float(np.nan), C.c_float(0)
            st = wm._check(L.wm_embed(wm._h, C.byref(din), None, C.byref(dout), mask, C.byref(a)))
            st2 = wm._check(L.wm_detect(wm._h, C.byref(dout), mask, C.byref(corr)))
            o = dev_get(wmb, wm, pout, hout.shape)
            assert np.array_equal(dev_get(wmb, wm, pin, hin.shape), hin), what  # the input is only read
            assert untouched(o, rows, cols, ld, out_off, 0xA5), what
            got = image_of(o, rows, cols, ld, out_off)
            assert np.array_equal(got, ref[0]) and f32bits(a.value) == f32bits(ref[1]) and f32bits(corr.value) == f32bits(ref[3]), "device " + what
            assert st == ref[2] and st2 == ref[4]
            L.wm_dev_free(wm._h, pin)
            L.wm_dev_free(wm._h, pout)
            # host
            hout = np.full(out_off + rows * ld + 16, 0xA5, np.uint8)
            view = lambda b, off: np.lib.stride_tricks.as_strided(b[off:], (rows, cols, 2), (ld, 2, 1))
            a, st = wm.make_watermark_host(view(hin, in_off), None, view(hout, out_off), mask, layout=layout)
            corr, st2 = wm.detect_watermark_host(view(hout, out_off), mask, layout=layout)
            assert untouched(hout, rows, cols, ld, out_off, 0xA5), what
            got = image_of(hout, rows, cols, ld, out_off)
            assert np.array_equal(got, ref[0]) and f32bits(a) == f32bits(ref[1]) and f32bits(corr) == f32bits(ref[3]), "host " + what
            assert st == ref[2] and st2 == ref[4]
    wm.close()


# widths that are not multiples of 16 (the last 16-pixel chunk of a row is partial: 4, 12 and 16 bytes short of a full one at 958, 854 and 200),
# each image in a device buffer that ends with its last row, without padding: dense 16-byte rows (200), word-aligned pitches (+4) and
# byte-aligned ones (+2).  Results only: equal to the Y-plane path.
@pytest.mark.parametrize("cols,extra", [(200, 0), (958, 0), (854, 4), (130, 2), (1366, 0)])
def test_rows_ending_at_the_allocation_end(wmb, cols, extra):
    rows = 67
    ld = 2 * cols + extra
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    L = wmb.lib()
    y, c = luma_image(rows, cols, seed=cols), chroma_plane(rows, cols, cols)
    for layout in layouts(wmb):
        src = pack(wmb, y, c, layout)
        buf = np.zeros((rows - 1) * ld + 2 * cols, np.uint8)  # the last row ends at the last byte
        buf[:(rows - 1) * ld].reshape(rows - 1, ld)[:, :2 * cols] = src[:-1].reshape(rows - 1, 2 * cols)
        buf[(rows - 1) * ld:] = src[-1].reshape(-1)
        for mask in (wmb.ME, wmb.NVF):
            ref = yplane(wmb, wm, y, mask)
            pin, pout = dev_raw(wmb, wm, buf), dev_raw(wmb, wm, np.zeros_like(buf))
            a, st, corr, st2 = one(wmb, wm, pin, pout, rows, cols, layout, 2, ld, mask)
            o = dev_get(wmb, wm, pout, buf.shape)
            for p in (pin, pout):
                L.wm_dev_free(wm._h, p)
            got = np.empty_like(src)
            got[:-1] = o[:(rows - 1) * ld].reshape(rows - 1, ld)[:, :2 * cols].reshape(rows - 1, cols, 2)
            got[-1] = o[(rows - 1) * ld:].reshape(cols, 2)
            assert_like_y(wmb, (got, a, st, corr, st2), ref, src, layout, "%dx%d ld=%d layout=%d mask=%d" % (rows, cols, ld, layout, mask))
    wm.close()


# ---- 5. batches: every image equals its single-image run ----
def batch_images(wmb, rows, cols, n, layout):
    base = [pack(wmb, luma_image(rows, cols, seed=100 + k), chroma_plane(rows, cols, 100 + k), layout) for k in range(4)]
    return np.stack([np.roll(base[b % 4], 7 * b, axis=1) for b in range(n)])


@pytest.mark.parametrize("rows,cols,batch,stride_extra", [(1080, 1920, 148, 0), (1080, 1920, 150, 0), (270, 480, 5, 4098)])
def test_batches(wmb, rows, cols, batch, stride_extra):
    """148 1080p images; 150 (uneven share of a wave: launched as sub-batches); an explicit stride larger than one image."""
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    L = wmb.lib()
    one_b = rows * 2 * cols
    stride = one_b + stride_extra
    arg = stride if stride_extra else 0
    for layout in layouts(wmb):
        imgs = batch_images(wmb, rows, cols, batch, layout)
        buf = np.zeros((batch, stride), np.uint8)
        buf[:, :one_b] = imgs.reshape(batch, one_b)
        desc = lambda p: wmb.image_desc(p, rows, cols, layout, wmb.U8, 0, 2)
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
            # a batch launch gives each image fewer CTAs than a single-image launch: the correlation's f64 partial sums are grouped
            # differently and may differ in their last f32 bits; bytes and `a` come out identical
            rc = float(np.max(np.abs(corr.astype(np.float64) - c1) / np.abs(c1)))
            print("batch %d %dx%d layout=%d mask=%d: differing bytes %d, corr max rel %.3g" % (
                batch, rows, cols, layout, mask, int(np.count_nonzero(ob != o1)), rc))
            k = koff(wmb, layout)
            assert np.array_equal(ob, o1)
            assert np.array_equal(ob[:, :one_b].reshape(imgs.shape)[..., 1 - k], imgs[..., 1 - k])
            assert np.array_equal(st, st1) and np.array_equal(st2, s21)
            assert np.array_equal(a.view(np.uint32), a1.view(np.uint32))
            assert rc <= 1e-6
            if stride_extra:
                assert np.all(ob[:, one_b:] == 0)  # the gap between strided images is not written
    wm.close()


# ---- 6. every host form equals the device path ----
def test_host_forms_equal_device_forms(wmb):
    rows, cols, batch = 270, 480, 5
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    L = wmb.lib()
    one_b = rows * 2 * cols
    for layout in layouts(wmb):
        imgs = batch_images(wmb, rows, cols, batch, layout)
        for mask in (wmb.ME, wmb.NVF):
            refs = [packed(wmb, wm, imgs[b], layout, mask) for b in range(batch)]
            for b in (0, batch - 1):
                out = np.empty_like(imgs[b])
                a, st = wm.make_watermark_host(imgs[b], None, out, mask, layout=layout)
                corr, st2 = wm.detect_watermark_host(out, mask, layout=layout)
                assert np.array_equal(out, refs[b][0]) and (st, st2) == (refs[b][2], refs[b][4])
                assert f32bits(a) == f32bits(refs[b][1]) and f32bits(corr) == f32bits(refs[b][3])
            hp = [L.wm_host_alloc_pinned(batch * one_b) for _ in range(2)]
            hin, hout = [np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), (batch, rows, cols, 2)) for p in hp]
            hin[:] = imgs
            desc = lambda p: wmb.image_desc(p, rows, cols, layout, wmb.U8, 0, 2)
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


# ---- 7. CUDA-graph replay ----
def test_graph_replay(wmb):
    """Repeated synchronous calls replay a captured CUDA graph from the third call on; a UYVY call on the same pointers and bytes
    afterwards reads the other byte of each pixel as the luma and must give the UYVY result, not a replay of the YUYV one."""
    rows, cols = 270, 480
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    L = wmb.lib()
    src = pack(wmb, luma_image(rows, cols, seed=21), luma_image(rows, cols, seed=22), wmb.PACKED_YUYV)  # both bytes natural images
    for mask in (wmb.ME, wmb.NVF):
        refs = {layout: packed(wmb, wm, src, layout, mask) for layout in layouts(wmb)}
        assert not np.array_equal(refs[wmb.PACKED_YUYV][0], refs[wmb.PACKED_UYVY][0])
        pin, pout = dev_raw(wmb, wm, src), dev_raw(wmb, wm, np.zeros_like(src))
        for layout in layouts(wmb):
            ref = refs[layout]
            din = wmb.image_desc(pin, rows, cols, layout, wmb.U8, 0, 2)
            dout = wmb.image_desc(pout, rows, cols, layout, wmb.U8, 0, 2)
            for call in range(4):
                a, corr = C.c_float(np.nan), C.c_float(0)
                st = wm._check(L.wm_embed(wm._h, C.byref(din), None, C.byref(dout), mask, C.byref(a)))
                st2 = wm._check(L.wm_detect(wm._h, C.byref(dout), mask, C.byref(corr)))
                o = dev_get(wmb, wm, pout, src.shape)
                what = "call %d layout=%d mask=%d" % (call, layout, mask)
                assert np.array_equal(o, ref[0]) and (st, st2) == (ref[2], ref[4]), what
                assert f32bits(a.value) == f32bits(ref[1]) and f32bits(corr.value) == f32bits(ref[3]), what
        L.wm_dev_free(wm._h, pin)
        L.wm_dev_free(wm._h, pout)
    wm.close()


# ---- 8. singular and zero-mask cases: out = every input byte ----
def test_singular_and_zero_mask(wmb):
    rows, cols = 270, 480
    flat = np.full((rows, cols), 117, np.uint8)  # constant luma: the ME system is unsolvable
    c = chroma_plane(rows, cols, 8)
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    wz = wmb.Watermark(rows, cols, np.zeros((rows, cols), np.float32), 3, PSNR)  # W = 0: mask.W is exactly 0
    y = luma_image(rows, cols, seed=8)
    for layout in layouts(wmb):
        img = pack(wmb, flat, c, layout)
        o, a, st, corr, st2 = got = packed(wmb, wm, img, layout, wmb.ME)
        assert st == wmb.SINGULAR and np.isnan(a) and np.array_equal(o, img)
        assert st2 == wmb.SINGULAR
        assert_like_y(wmb, got, yplane(wmb, wm, flat, wmb.ME), img, layout, "singular layout=%d" % layout)
        img = pack(wmb, y, c, layout)
        for mask in (wmb.ME, wmb.NVF):
            o, a, st, corr, st2 = got = packed(wmb, wz, img, layout, mask)
            assert st == wmb.ZERO_MASK and np.isinf(a) and np.array_equal(o, img), (layout, mask, st)
            assert_like_y(wmb, got, yplane(wmb, wz, y, mask), img, layout, "zero mask layout=%d mask=%d" % (layout, mask))
    wz.close()
    wm.close()


# ---- 9. NVF with a 5 x 5 window ----
@pytest.mark.parametrize("rows,cols", [(270, 480), (67, 130)])
def test_nvf_p5(wmb, rows, cols):
    y, c = luma_image(rows, cols, seed=9), chroma_plane(rows, cols, 9)
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 5, PSNR)
    ref = yplane(wmb, wm, y, wmb.NVF)
    for layout in layouts(wmb):
        src = pack(wmb, y, c, layout)
        assert_like_y(wmb, packed(wmb, wm, src, layout, wmb.NVF), ref, src, layout, "NVF p=5 %dx%d layout=%d" % (rows, cols, layout))
    wm.close()


# ---- 10. rejections ----
def test_rejections(wmb):
    rows, cols = 67, 130
    wm = wmb.Watermark(rows, cols, util.normal_w(rows, cols), 3, PSNR)
    L = wmb.lib()
    src = pack(wmb, luma_image(rows, cols), chroma_plane(rows, cols), wmb.PACKED_YUYV)
    d = wmb.DeviceArray.from_numpy(wm, src, wmb.PACKED_YUYV)
    out = wmb.DeviceArray(wm, rows, cols, wmb.PACKED_YUYV)
    outu = wmb.DeviceArray(wm, rows, cols, wmb.PACKED_UYVY)
    out3 = wmb.DeviceArray(wm, rows, cols, wmb.PACKED_RGB)
    out4 = wmb.DeviceArray(wm, rows, cols, wmb.PACKED_BGRA)
    d4 = wmb.DeviceArray.from_numpy(wm, np.zeros((rows, cols, 4), np.uint8), wmb.PACKED_RGBA)
    gray = wmb.DeviceArray(wm, rows, cols, wmb.ROW_MAJOR, wmb.F32, 1)
    y8 = wmb.DeviceArray(wm, rows, cols, wmb.ROW_MAJOR, wmb.U8, 1)
    a = C.c_float(0)

    def desc(p, layout=wmb.PACKED_YUYV, dtype=wmb.U8, ld=0, ch=2):
        return wmb.image_desc(p, rows, cols, layout, dtype, ld, ch)

    def embed_rc(i, b, o):
        return L.wm_embed(wm._h, C.byref(i), C.byref(b) if b is not None else None, C.byref(o), wmb.ME, C.byref(a))

    def refused(rc, what, ctx=wm):
        msg = L.wm_last_error(ctx._h).decode()
        print("%s: %d %s" % (what, rc, msg))
        assert rc == -5 and msg, what

    refused(embed_rc(desc(d.ptr, dtype=wmb.F32), None, out.desc()), "f32 YUYV")
    refused(embed_rc(desc(d.ptr, ch=1), None, out.desc()), "YUYV with 1 channel")
    refused(embed_rc(desc(d.ptr, ch=3), None, out.desc()), "YUYV with 3 channels")
    refused(embed_rc(desc(d.ptr, layout=wmb.PACKED_UYVY, ch=4), None, outu.desc()), "UYVY with 4 channels")
    refused(embed_rc(desc(d.ptr, ld=2 * cols - 1), None, out.desc()), "ld < 2 cols")
    refused(L.wm_detect(wm._h, C.byref(desc(d.ptr, ld=2 * cols - 1)), wmb.ME, C.byref(a)), "detect ld < 2 cols")
    refused(L.wm_detect(wm._h, C.byref(desc(d.ptr, ch=1)), wmb.ME, C.byref(a)), "detect YUYV with 1 channel")
    refused(L.wm_detect(wm._h, C.byref(desc(d.ptr, layout=wmb.PACKED_UYVY, dtype=wmb.F32)), wmb.ME, C.byref(a)), "detect f32 UYVY")
    refused(embed_rc(d.desc(), None, outu.desc()), "YUYV in, UYVY out")
    refused(embed_rc(desc(d.ptr, layout=wmb.PACKED_UYVY), None, out.desc()), "UYVY in, YUYV out")
    refused(embed_rc(d.desc(), desc(d.ptr, layout=wmb.PACKED_UYVY), out.desc()), "YUYV in, UYVY base (same pointer)")
    refused(embed_rc(d.desc(), None, out3.desc()), "YUYV in, RGB out")
    refused(embed_rc(d.desc(), None, out4.desc()), "YUYV in, BGRA out")
    refused(embed_rc(d4.desc(), None, out.desc()), "RGBA in, YUYV out")
    refused(embed_rc(d.desc(), d4.desc(), out.desc()), "YUYV in, RGBA base")
    refused(embed_rc(d.desc(), y8.desc(), out.desc()), "Y-plane base")
    refused(embed_rc(d.desc(), None, y8.desc()), "Y-plane out")
    refused(embed_rc(d.desc(), None, gray.desc()), "gray out")
    refused(embed_rc(y8.desc(), None, out.desc()), "Y-plane input, YUYV out")
    refused(embed_rc(y8.desc(), d.desc(), y8.desc()), "Y-plane input, YUYV base")
    refused(embed_rc(d.desc(), None, desc(d.ptr + 2)), "out overlaps in")
    refused(L.wm_rgb2gray(wm._h, C.byref(d.desc()), C.byref(gray.desc()), 0.299, 0.587, 0.114), "rgb2gray")
    refused(L.wm_debug_plane(wm._h, C.byref(d.desc()), wmb.DBG_ERRSEQ, gray.ptr), "debug_plane")
    refused(L.wm_debug_detect_planes(wm._h, C.byref(d.desc()), wmb.ME, gray.ptr, gray.ptr, C.byref(a)), "debug_detect_planes")
    for layout in (8, 9, -1):
        refused(embed_rc(desc(d.ptr, layout=layout), None, desc(out.ptr, layout=layout)), "layout %d" % layout)
    # host forms
    h2 = np.array(src)
    o2 = np.zeros_like(h2)
    hd = lambda arr, layout, ld=0, ch=2: wmb.image_desc(arr.ctypes.data, rows, cols, layout, wmb.U8, ld, ch)
    refused(L.wm_embed_host(wm._h, C.byref(hd(h2, wmb.PACKED_YUYV)), None, C.byref(hd(o2, wmb.PACKED_UYVY)), wmb.ME, C.byref(a)),
            "host YUYV in, UYVY out")
    refused(L.wm_embed_host(wm._h, C.byref(hd(h2, wmb.PACKED_YUYV, ld=2 * cols - 1)), None, C.byref(hd(o2, wmb.PACKED_YUYV)), wmb.ME,
                            C.byref(a)), "host ld < 2 cols")
    refused(L.wm_detect_host(wm._h, C.byref(hd(h2, wmb.PACKED_UYVY, ch=3)), wmb.ME, C.byref(a)), "host detect UYVY with 3 channels")
    assert np.all(o2 == 0)
    with pytest.raises(TypeError):
        wm.make_watermark_host(np.zeros((rows, cols, 3), np.uint8), None, o2, wmb.ME, layout=wmb.PACKED_YUYV)
    for x in (d, out, outu, out3, out4, d4, gray, y8):
        x.free()
    # odd cols: 4:2:2 pairs pixels
    wo = wmb.Watermark(rows, 131, util.normal_w(rows, 131), 3, PSNR)
    po = dev_raw(wmb, wo, np.zeros(rows * 2 * 131 * 2, np.uint8))
    di = wmb.image_desc(po, rows, 131, wmb.PACKED_YUYV, wmb.U8, 0, 2)
    do = wmb.image_desc(po + rows * 2 * 131, rows, 131, wmb.PACKED_YUYV, wmb.U8, 0, 2)
    refused(L.wm_embed(wo._h, C.byref(di), None, C.byref(do), wmb.ME, C.byref(a)), "odd cols", wo)
    refused(L.wm_detect(wo._h, C.byref(di), wmb.ME, C.byref(a)), "detect odd cols", wo)
    hodd = np.zeros((rows, 131, 2), np.uint8)
    refused(L.wm_detect_host(wo._h, C.byref(wmb.image_desc(hodd.ctypes.data, rows, 131, wmb.PACKED_UYVY, wmb.U8, 0, 2)), wmb.ME, C.byref(a)),
            "host detect odd cols", wo)
    L.wm_dev_free(wo._h, po)
    wo.close()
    wm.close()
